"""Parity at the shapes that are actually benchmarked (VERDICT r1, "what's weak"): a K=30 trajectory at BASELINE config-5
dimensions, the production gate kernel (`gates_tc_pair_kernel<2,2,4>`, hidden_dim 800) at its production batch of 256
instances, K=100 against the UNMODIFIED reference modules running on the same GPU, a config-3-shaped gradient check and
the 0.25 double-tie clip gradient (SURVEY.md section 7, hard parts)."""
import os
import sys

import pytest
import torch

from helpers import (rel_err, assert_parity, oracle_pair, load_golden, K100_SHAPE, K100_ROWS, k100_inputs, k100_record,
                     k100_reference_record)

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def make_model(prm, h, K, mode="tc_f16f8", dev=DEV):
    import iadmm_b200 as ia
    model = ia.LSTM(None, 2, h, K, dev, gate_mode=mode)
    with torch.no_grad():
        for k, v in prm.items():
            getattr(model, k).copy_(v.to(dev))
    return model.eval()


def test_config5_k30_trajectory_vs_oracle():
    """BASELINE config 5 (n=5000, 2500+2500, hidden_dim=800, --scaling): 30 iterations of one instance against the oracle in
    the reference's fp32 arithmetic -- five 1024-column chunks x 40 row chunks per matrix, 79 row tiles x 13 unit tiles in the
    gate kernel: an accumulation-order bug would show late, not after K=2.  x, y, z and both residual traces <= 1e-4
    (y falls back to the reference's own fp32 noise floor if its early-iterate rounding noise exceeds the bar)."""
    import iadmm_b200 as ia
    from oracle import iadmm_oracle as orc
    B, n, mi, me, h, K = 1, 5000, 2500, 2500, 800, 30
    g = torch.Generator().manual_seed(91)
    qp = dict(Q=torch.diag_embed(torch.rand((B, n), generator=g)), p=torch.rand((B, n, 1), generator=g),
              A0=torch.randn((B, mi + me, n), generator=g))
    bnd = torch.rand((B, mi + me, 1), generator=g)
    qp["zl"] = torch.cat((torch.full((B, mi, 1), float("-inf")), bnd[:, mi:]), 1)
    qp["zu"] = torch.cat((bnd[:, :mi] + 1.0, bnd[:, mi:]), 1)
    prm = orc.lstm_parameters(h, K, seed=91)
    ref32, ref64, _, _ = oracle_pair(prm, K, mi, me, qp, h)
    sc = ia.Scaling(n, mi + me, 10, DEV)
    data = sc.scale_data(*(qp[k].to(DEV) for k in ("Q", "p", "A0", "zl", "zu")))
    model = make_model(prm, h, K)
    with torch.no_grad():
        r = model.solve(K, mi, me, *data, 6e-6, scaling=sc)
    torch.cuda.synchronize()
    rep = {}
    for k in ("x", "y", "z", "pri", "dual"):
        rep[k] = assert_parity(k, getattr(r, k), getattr(ref32, k), getattr(ref64, k))
    print("config-5 K=30", {k: f"{v[0]:.1e} ({v[1]})" for k, v in rep.items()})


def test_production_kernel_at_production_batch_bit_exact():
    """hidden_dim 800 and 256 instances (512000 rows: the grid bench.py times, 148 SMs x 176 tiles each) -- sampled
    instances must be bit-identical to solving them alone (B=1: 104 tiles on 74 clusters), for the iterates AND the residual
    traces: no cross-instance arithmetic, no dependence of any rounding on the tile an instance's rows fall into."""
    from bench import device_qp_batch
    import iadmm_b200 as ia
    B, n, mi, me, h, K = 256, 1000, 500, 500, 800, 3
    torch.manual_seed(5)
    model = ia.LSTM(None, 2, h, K, DEV).eval()
    Q, p, A0, zl, zu = device_qp_batch(B, n, mi, me, 3, DEV)
    sc = ia.Scaling(n, mi + me, 10, DEV)
    data = sc.scale_data(Q, p, A0, zl, zu)
    with torch.no_grad():
        full = model.solve(K, mi, me, *data, 6e-6, scaling=sc)
        assert bool(torch.isfinite(full.x).all() and torch.isfinite(full.H).all() and torch.isfinite(full.pri).all())
        for i in (0, 101, 255):
            sc1 = ia.Scaling(n, mi + me, 10, DEV)
            d1 = sc1.scale_data(*(t_[i:i + 1].contiguous() for t_ in (Q, p, A0, zl, zu)))
            one = model.solve(K, mi, me, *d1, 6e-6, scaling=sc1)
            for k in ("x", "y", "z", "xv", "H", "C"):
                assert torch.equal(getattr(full, k)[i:i + 1], getattr(one, k)), (i, k)
            for k in ("pri", "dual", "pri_unscaled", "dual_unscaled"):
                assert torch.equal(getattr(full, k)[:, i:i + 1], getattr(one, k)), (i, k)
            assert torch.equal(full.metrics[:, :, i:i + 1], one.metrics), i


def test_k100_config2_vs_unmodified_reference_on_this_gpu():
    """The like-for-like oracle of SURVEY section 8(c/d): the reference's OWN modules (baseline/_ref, unmodified) with
    device='cuda' -- stock PyTorch fp32 kernels, TF32 off -- against the drop-in on the same GPU, same inputs, same weights:
    K=100, n=1000, 500+500, hidden_dim=800, --scaling, 16 instances.  x^K, y^K, z^K and the residual traces within 1e-4; the
    Ruiz diagonals, the scaled p, zl, zu and two rows of the scaled Q and A0 within 1e-6.  Without the reference's modules in
    baseline/_ref, the reference side is the stored outputs of the same computation (tests/golden/k100_config2.npz, written by
    tests/golden/make_k100_config2_golden.py; its `source` says what produced them)."""
    sys.path.insert(0, ROOT)
    from baseline import ref_arm
    import iadmm_b200 as ia
    s = K100_SHAPE
    B, n, mi, me, h, K = (s[k] for k in ("B", "n", "mi", "me", "h", "K"))
    if ref_arm.available():
        ref, source = k100_reference_record(DEV)
    else:
        g = load_golden("k100_config2")
        assert [int(v) for v in g["meta"]] == [s[k] for k in ("B", "n", "mi", "me", "h", "K", "seed")]
        assert tuple(int(v) for v in g["rows"]) == K100_ROWS
        ref, source = {k: torch.from_numpy(v) for k, v in g.items() if k not in ("source", "meta", "rows")}, str(g["source"])
    qp, prm = k100_inputs(DEV)
    sc = ia.Scaling(n, mi + me, 10, DEV)
    data = sc.scale_data(qp["Q"], qp["p"], qp["A0"], qp["zl"], qp["zu"])
    model = make_model(prm, h, K)
    with torch.no_grad():
        r = model.solve(K, mi, me, *data, 6e-6, scaling=sc)
    torch.cuda.synchronize()
    ours = k100_record(data, sc.d, sc.e, sc.c_vec, r.x, r.y, r.z, r.pri, r.dual)
    assert sorted(ours) == sorted(ref)
    for k in ("d", "e", "c", "p", "zl", "zu", "Q_rows", "A0_rows"):     # Ruiz: the reference's O(n^3) dense-diag form on the GPU
        assert rel_err(ours[k], ref[k]) < 1e-6, k
    errs = {k: rel_err(ours[k], ref[k]) for k in ("x", "y", "z", "pri", "dual")}
    # per instance too: the worst instance, not only the batch norm
    worst = {k: max(rel_err(ours[k][i], ref[k][i]) for i in range(B)) for k in ("x", "y", "z")}
    print("K=100 config-2 vs", source, {k: f"{v:.1e}" for k, v in errs.items()}, "worst instance", {k: f"{v:.1e}" for k, v in worst.items()})
    for k, v in errs.items():
        assert v <= 1e-4, (k, v)
    for k, v in worst.items():
        assert v <= 1e-4, ("worst instance", k, v)


def test_window_gradients_at_config3_shape():
    """BASELINE config 3 dimensions (n=1000, 500+500, hidden_dim=800, --scaling): one instance, a 2-iteration window,
    every parameter gradient against float64 autograd through the oracle.  Exercises the tensor-core forward, the
    tcgen05 NT-GEMMs of the backward at K=4h=3200 / M=2000 and the training KKT chunking at n=1000."""
    from oracle import iadmm_oracle as orc
    from test_gpu_training import oracle_window, our_window
    B, n, mi, me, h, TL = 1, 1000, 500, 500, 800, 2
    outer_T = 100
    qp = orc.qp_instances(B, n, mi, me, seed=67)
    Qs, ps, As, zls, zus, _ = orc.ruiz_equilibrate(qp["Q"], qp["p"], qp["A0"], qp["zl"], qp["zu"], 10)
    qps = dict(Q=Qs, p=ps, A0=As, zl=zls, zu=zus)
    prm = orc.lstm_parameters(h, outer_T, seed=67)
    ref_loss, ref_g, _ = oracle_window(prm, qps, mi, me, h, TL, outer_T)
    loss, g, _, _ = our_window(prm, qps, mi, me, h, TL, outer_T, mode="tc_f16f8")
    assert abs(loss - ref_loss) <= 2e-5 * abs(ref_loss)
    errs = {k: rel_err(g[k], ref_g[k]) for k in ref_g if float(ref_g[k].abs().max()) > 0}
    print("config-3 shape gradients", {k: f"{v:.1e}" for k, v in errs.items()})
    for k, v in errs.items():
        assert v < 1e-3, (k, v)


def test_clip_gradient_at_an_exact_double_tie():
    """SURVEY.md section 7: equality rows have zl == zu, and torch's binary max/min split the gradient at an exact tie, so
    through max(min(a, zu), zl) the derivative w.r.t. a is 0.25 when a == zl == zu (0 or 1 elsewhere).  With W_h = b_h = 0
    the cell cannot move xv, so from (y, z) = 0 and xv = 0 on some equality rows the clip argument is EXACTLY 0 = zl = zu in
    fp32 and in fp64: a robust double tie.  All state adjoints of one iteration against float64 autograd through the oracle."""
    import iadmm_b200 as ia
    from oracle import iadmm_oracle as orc
    B, n, mi, me, h = 2, 16, 4, 8, 16
    m = mi + me
    qp = orc.qp_instances(B, n, mi, me, seed=73)
    tie = [mi + 1, mi + 4, mi + 6]                                 # equality rows that tie; the others clip normally
    gen = torch.Generator().manual_seed(74)
    xv0 = torch.randn((B, n + m, 1), generator=gen)
    for i in tie:
        qp["zl"][:, i] = 0.0; qp["zu"][:, i] = 0.0
        xv0[:, n + i] = 0.0
    prm = orc.lstm_parameters(h, 3, seed=73, scale=3.0)
    prm["W_h"] = torch.zeros_like(prm["W_h"]); prm["b_h"] = torch.zeros_like(prm["b_h"])
    x0 = torch.randn((B, n, 1), generator=gen)
    H0 = torch.tanh(torch.randn((B, n + m, h), generator=gen)); C0 = torch.randn((B, n + m, h), generator=gen)
    wts = [torch.randn(s, generator=gen) for s in ((B, n, 1), (B, m, 1), (B, m, 1), (B, n + m, 1))]

    def run(step, dev, dt):
        leaves = [v.to(dt).to(dev).requires_grad_(True) for v in (x0, torch.zeros((B, m, 1)), torch.zeros((B, m, 1)), xv0)]
        outs = step(*leaves, H0.to(dt).to(dev), C0.to(dt).to(dev))
        sum((o * w.to(dt).to(dev)).sum() for o, w in zip(outs[:4], wts)).backward()
        return [l.grad.detach().cpu().double() for l in leaves]

    p64 = {k: v.double() for k, v in prm.items()}
    d64 = {k: qp[k].double() for k in ("Q", "p", "A0", "zl", "zu")}
    ref = run(lambda x, y, z, xv, H, C: orc.lstm_step(p64, 1, mi, me, x, y, z, xv, 6e-6, H, C, d64["Q"], d64["p"], d64["A0"],
                                                     d64["zl"], d64["zu"], form="block")[:4], "cpu", torch.float64)
    model = ia.LSTM(None, 2, h, 3, DEV, gate_mode="simt_fp32")
    with torch.no_grad():
        for k, v in prm.items():
            getattr(model, k).copy_(v.to(DEV))
    dd = {k: qp[k].to(DEV) for k in ("Q", "p", "A0", "zl", "zu")}
    ours = run(lambda x, y, z, xv, H, C: model(1, mi, me, x, y, z, xv, 6e-6, H, C, Q=dd["Q"], p=dd["p"], A0=dd["A0"], lb=None,
                                               ub=None, zl=dd["zl"], zu=dd["zu"])[:4], DEV, torch.float32)
    # (gy is exactly zero in exact arithmetic here -- y cancels out of both z' and y' -- so errors are measured against the
    # largest adjoint, not against each adjoint's own norm)
    scale = max(float(b.norm()) for b in ref)
    for name, a, b in zip(("gx", "gy", "gz", "gxv"), ours, ref):
        err = float((a - b).norm()) / scale
        assert err < 1e-4, (name, err)
    # the tie rows really carry the QUARTER gradient: with the tie made one-sided (zu or zl moved away, derivative 0.5)
    # the reference gradient is a different one
    for delta in (-1.0, 1.0):
        d_alt = {k: v.clone() for k, v in d64.items()}
        for i in tie:
            d_alt["zu"][:, i] = delta if delta > 0 else 0.0
            d_alt["zl"][:, i] = 0.0 if delta > 0 else delta
        alt = run(lambda x, y, z, xv, H, C: orc.lstm_step(p64, 1, mi, me, x, y, z, xv, 6e-6, H, C, d_alt["Q"], d_alt["p"],
                                                         d_alt["A0"], d_alt["zl"], d_alt["zu"], form="block")[:4], "cpu", torch.float64)
        assert rel_err(alt[3], ref[3]) > 1e-3      # a one-sided tie (0.5) is a different gradient than the double tie (0.25)


@pytest.mark.parametrize("h", [200, 208, 384, 400])
def test_hidden200_k100_vs_fp32_path(h):
    """configs/QP.yaml's default hidden_dim 200 (% 16 == 8: half-padded last operand group), 208 and 384: the 16-epilogue-warp
    kernel with the shared-reciprocal activations (gates_tc_pair_kernel<2,2,9>, hidden_dim <= 384); 400 (scripts/Synthetic.sh's
    QP_RHS size): the first size on the 8-warp kernel <2,2,4>.  K=100 at n=1000, 500+500, --scaling
    against the fp32 CUDA-core path on the same inputs and weights (which matches the reference's fp32 run to <= 2e-6,
    test_gpu_parity): worst INSTANCE within north_star's 1e-4 on x, y, z, batch norm within 1e-4 on the residual traces."""
    from bench import device_qp_batch
    import iadmm_b200 as ia
    B, n, mi, me, K = 4, 1000, 500, 500, 100
    Q, p, A0, zl, zu = device_qp_batch(B, n, mi, me, 21, DEV)
    sc = ia.Scaling(n, mi + me, 10, DEV)
    data = sc.scale_data(Q, p, A0, zl, zu)
    torch.manual_seed(21)
    ref_model = ia.LSTM(None, 2, h, K, DEV, gate_mode="simt_fp32").eval()
    model = ia.LSTM(None, 2, h, K, DEV, gate_mode="tc_f16f8").eval()
    model.load_state_dict(ref_model.state_dict())
    with torch.no_grad():
        ref = ref_model.solve(K, mi, me, *data, 6e-6, scaling=sc)
        r = model.solve(K, mi, me, *data, 6e-6, scaling=sc)
    worst = {k: max(rel_err(getattr(r, k)[i], getattr(ref, k)[i]) for i in range(B)) for k in ("x", "y", "z")}
    tr = {k: rel_err(getattr(r, k), getattr(ref, k)) for k in ("pri", "dual", "pri_unscaled", "dual_unscaled")}
    print(f"hidden {h}, K=100: worst instance", {k: f"{v:.1e}" for k, v in worst.items()}, "traces", {k: f"{v:.1e}" for k, v in tr.items()})
    for k, v in {**worst, **tr}.items():
        assert v <= 1e-4, (k, v)
