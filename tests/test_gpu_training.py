"""GPU tests of the training path (SURVEY.md section 8 rows a15/a16): one truncated-BPTT window driven exactly
like main.py:336-358 through the drop-in LSTM.forward + primal_dual_loss, gradients compared with
torch.autograd through the CPU oracle in float64."""
import pytest
import torch

from helpers import rel_err

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def oracle_window(prm, qp, mi, me, h, TL, outer_T, state=None, dtype=torch.float64):
    from oracle import iadmm_oracle as orc
    p64 = {k: v.detach().to(dtype).clone().requires_grad_(True) for k, v in prm.items()}
    Q, p, A0, zl, zu = (qp[k].to(dtype) for k in ("Q", "p", "A0", "zl", "zu"))
    B, n = Q.shape[0], Q.shape[1]
    m = mi + me
    if state is None:
        st = [torch.zeros((B, n, 1), dtype=dtype), torch.zeros((B, m, 1), dtype=dtype), torch.zeros((B, m, 1), dtype=dtype),
              torch.zeros((B, n + m, 1), dtype=dtype), torch.zeros((B, n + m, h), dtype=dtype), torch.zeros((B, n + m, h), dtype=dtype)]
    else:
        st = [s.to(dtype) for s in state]
    x, y, z, xv, H, C = st
    loss = 0.0
    for t in range(TL):      # t restarts at 0 every window (main.py:338)
        x, y, z, xv, H, C, _ = orc.lstm_step(p64, t, mi, me, x, y, z, xv, 6e-6, H, C, Q, p, A0, zl, zu, form="block")
        pr, du, tot = orc.primal_dual_residuals(x, y, z, Q, p, A0)
        loss = loss + tot.mean() / outer_T
    loss.backward()
    return float(loss.detach()), {k: v.grad for k, v in p64.items()}, [s.detach() for s in (x, y, z, xv, H, C)]


def our_window(prm, qp, mi, me, h, TL, outer_T, state=None, mode="simt_fp32"):
    import iadmm_b200 as ia
    model = ia.LSTM(None, 2, h, outer_T, DEV, gate_mode=mode)
    with torch.no_grad():
        for k, v in prm.items():
            getattr(model, k).copy_(v.to(DEV))
    Q, p, A0, zl, zu = (qp[k].to(DEV) for k in ("Q", "p", "A0", "zl", "zu"))
    B, n = Q.shape[0], Q.shape[1]
    m = mi + me
    if state is None:
        st = [torch.zeros((B, n, 1), device=DEV), torch.zeros((B, m, 1), device=DEV), torch.zeros((B, m, 1), device=DEV),
              torch.zeros((B, n + m, 1), device=DEV), torch.zeros((B, n + m, h), device=DEV), torch.zeros((B, n + m, h), device=DEV)]
    else:
        st = [s.float().to(DEV) for s in state]
    x, y, z, xv, H, C = st
    loss = 0.0
    for t in range(TL):
        x, y, z, xv, H, C, _, _, _ = model(t, mi, me, x, y, z, xv, 6e-6, H, C, Q=Q, p=p, A0=A0, lb=None, ub=None, zl=zl, zu=zu)
        pr, du, tot = ia.primal_dual_loss(x, y, z, Q, p, A0)
        loss = loss + tot.mean() / outer_T
    model.zero_grad()
    loss.backward()
    torch.cuda.synchronize()
    return float(loss), {k: getattr(model, k).grad for k in prm}, [s.detach() for s in (x, y, z, xv, H, C)], model


@pytest.mark.parametrize("mode", ["simt_fp32", "tc_f16f8"])
@pytest.mark.parametrize("shape", [(2, 12, 5, 7, 8, 4, 1.0), (3, 40, 12, 16, 32, 5, 3.0), (2, 100, 50, 50, 64, 6, 1.0),
                                   (2, 24, 10, 0, 16, 4, 2.0), (2, 30, 9, 8, 40, 4, 1.0)])
def test_window_gradients_match_autograd(shape, mode):
    from oracle import iadmm_oracle as orc
    B, n, mi, me, h, TL, wscale = shape
    outer_T = TL + 2
    qp = orc.qp_instances(B, n, mi, me, seed=61)
    if me == 0:
        qp["zl"][:] = -0.7                     # two-sided inequality rows exercise both clip branches
    prm = orc.lstm_parameters(h, outer_T, seed=61, scale=wscale)
    ref_loss, ref_g, ref_state = oracle_window(prm, qp, mi, me, h, TL, outer_T)
    loss, g, state, _ = our_window(prm, qp, mi, me, h, TL, outer_T, mode=mode)
    assert abs(loss - ref_loss) <= 2e-5 * abs(ref_loss)
    errs = {k: rel_err(g[k], ref_g[k]) for k in ref_g if float(ref_g[k].abs().max()) > 0}
    print(shape, mode, {k: f"{v:.1e}" for k, v in errs.items()})
    # The bias gradients b_u and b_h are sums over all B*N coordinates and TL iterations that cancel to ~1e-3 of their terms:
    # the REFERENCE's own fp32 autograd misses the float64 value by 1e-4 ... 3e-4 there.  That floor is measured here (the
    # oracle in float32 against the oracle in float64, same inputs) and an fp32 implementation is held to the fixed bound or
    # 3x the floor, whichever is larger.
    _, g32, _ = oracle_window(prm, qp, mi, me, h, TL, outer_T, dtype=torch.float32)
    floor = {k: rel_err(g32[k].double(), ref_g[k]) for k in errs}
    for k, v in errs.items():
        assert v < max(2e-4 if mode == "simt_fp32" else 5e-4, 3.0 * floor[k]), (k, v, floor[k])
    # rows >= TL of the schedule never receive gradient (main.py:338 restarts t at 0)
    assert float(g["rho"][TL:].abs().max()) == 0.0 and float(g["alpha"][TL:].abs().max()) == 0.0
    # fp32 state vs the fp64 run; y = y + rho (z~ - z) cancels catastrophically on equality rows, so its fp32
    # value carries ~rho * ulp(z) of rounding noise (the reference's own fp32-vs-fp64 drift, BASELINE.md)
    for a, b, k in zip(state, ref_state, ("x", "y", "z", "xv", "H", "C")):
        assert rel_err(a, b) < (2e-2 if k == "y" else 2e-5), k


def test_second_window_from_detached_state_and_adam_step():
    """main.py:349-358: backward, Adam step, detach, next window continues from the carried state."""
    from oracle import iadmm_oracle as orc
    B, n, mi, me, h, TL = 2, 30, 10, 12, 16, 3
    outer_T = 2 * TL
    qp = orc.qp_instances(B, n, mi, me, seed=71)
    prm = orc.lstm_parameters(h, outer_T, seed=71, scale=2.0)
    _, _, state1 = oracle_window(prm, qp, mi, me, h, TL, outer_T)
    state1 = [s.float() for s in state1]
    # From a carried (non-zero) state the gradient of rho is dominated by y_bar * (z~ - z'), a catastrophically
    # cancelling difference in fp32: the reference's own fp32 autograd differs from fp64 by 5 % here (measured).
    # The kernels reproduce the reference's fp32 rounding, so compare with the fp32 run; fp64 bounds the rest.
    ref_loss, ref_g, _ = oracle_window(prm, qp, mi, me, h, TL, outer_T, state=state1, dtype=torch.float32)
    _, ref_g64, _ = oracle_window(prm, qp, mi, me, h, TL, outer_T, state=state1)
    loss, g, _, model = our_window(prm, qp, mi, me, h, TL, outer_T, state=state1)
    assert abs(loss - ref_loss) <= 2e-5 * abs(ref_loss)
    for k in ref_g:
        if float(ref_g[k].abs().max()) > 0:
            assert rel_err(g[k], ref_g[k]) < 1e-3, k
            if k != "rho":
                assert rel_err(g[k], ref_g64[k]) < 1e-3, k
    opt = torch.optim.Adam(model.parameters(), lr=1e-3)
    before = model.U_i.detach().clone()
    opt.step()
    assert not torch.equal(before, model.U_i.detach())
    # the packed weights follow the parameter update (re-packed on version change)
    with torch.no_grad():
        r = model.solve(2, mi, me, *(qp[k].to(DEV) for k in ("Q", "p", "A0", "zl", "zu")), 6e-6)
    prm2 = {k: getattr(model, k).detach().cpu() for k in prm}
    ref = orc.solve(prm2, 2, mi, me, qp["Q"], qp["p"], qp["A0"], qp["zl"], qp["zu"], 6e-6, h, form="block")
    assert rel_err(r.x, ref.x) < 1e-5


def test_residual_gradients():
    import iadmm_b200 as ia
    from oracle import iadmm_oracle as orc
    B, n, mi, me = 3, 37, 9, 11
    qp = orc.qp_instances(B, n, mi, me, seed=81)
    gen = torch.Generator().manual_seed(82)
    x = torch.randn((B, n, 1), generator=gen); y = torch.randn((B, mi + me, 1), generator=gen); z = torch.randn((B, mi + me, 1), generator=gen)
    Qd = qp["Q"] + 0.1 * torch.randn((B, n, n), generator=gen)
    xr, yr, zr = (v.double().requires_grad_(True) for v in (x, y, z))
    pr, du, _ = orc.primal_dual_residuals(xr, yr, zr, Qd.double(), qp["p"].double(), qp["A0"].double())
    wts = torch.rand((B, 1, 1), generator=gen).double()
    (pr * wts + 2.0 * du * (1 - wts)).sum().backward()
    xg, yg, zg = (v.to(DEV).requires_grad_(True) for v in (x, y, z))
    gp, gd, _ = ia.primal_dual_loss(xg, yg, zg, Qd.to(DEV), qp["p"].to(DEV), qp["A0"].to(DEV))
    w = wts.float().to(DEV)
    (gp * w + 2.0 * gd * (1 - w)).sum().backward()
    assert rel_err(xg.grad, xr.grad) < 1e-5 and rel_err(yg.grad, yr.grad) < 1e-5 and rel_err(zg.grad, zr.grad) < 1e-5


@pytest.mark.parametrize("mode", ["simt_fp32", "tc_f16f8", "tc_f16f8u"])
@pytest.mark.parametrize("shape", [(3, 24, 7, 9, 16, 6), (2, 37, 9, 11, 48, 5), (2, 20, 0, 0, 16, 4)])
def test_fused_window_equals_per_iteration_autograd(shape, mode):
    """iadmm_train_window (one call per window) against the per-iteration autograd path it replaces: same kernels in
    the same order, so loss, end state and every parameter gradient agree to rounding of the loss seed."""
    import iadmm_b200 as ia
    from oracle import iadmm_oracle as orc
    B, n, mi, me, h, TL = shape
    outer_T = 2 * TL
    if mi + me:
        qp = orc.qp_instances(B, n, mi, me, seed=71)
    else:
        g = torch.Generator().manual_seed(71)
        M = torch.randn(B, n, n, generator=g)
        qp = dict(Q=M @ M.transpose(1, 2) / n + 0.1 * torch.eye(n), p=torch.randn(B, n, 1, generator=g),
                  A0=torch.zeros(B, 0, n), zl=torch.zeros(B, 0, 1), zu=torch.zeros(B, 0, 1))
    prm = orc.lstm_parameters(h, outer_T, seed=71)
    loss_a, grads_a, state_a, model = our_window(prm, qp, mi, me, h, TL, outer_T, mode=mode)
    # second window from the state the first one left, both ways
    loss_a2, grads_a2, state_a2, _ = our_window(prm, qp, mi, me, h, TL, outer_T, state=state_a, mode=mode)
    m = mi + me
    Q, p, A0, zl, zu = (qp[k].to(DEV) for k in ("Q", "p", "A0", "zl", "zu"))
    st = [torch.zeros((B, n, 1), device=DEV), torch.zeros((B, m, 1), device=DEV), torch.zeros((B, m, 1), device=DEV),
          torch.zeros((B, n + m, 1), device=DEV), torch.zeros((B, n + m, h), device=DEV), torch.zeros((B, n + m, h), device=DEV)]
    model.zero_grad()
    loss_f, st1 = model.train_window(TL, mi, me, Q, p, A0, zl, zu, 6e-6, st, t0=0, loss_scale=1.0 / outer_T)
    grads_f = {k: getattr(model, k).grad.clone() for k in prm}
    model.zero_grad()
    loss_f2, st2 = model.train_window(TL, mi, me, Q, p, A0, zl, zu, 6e-6, st1, t0=0, loss_scale=1.0 / outer_T)
    grads_f2 = {k: getattr(model, k).grad.clone() for k in prm}
    assert abs(float(loss_f) - loss_a) <= 1e-6 * abs(loss_a) and abs(float(loss_f2) - loss_a2) <= 1e-6 * abs(loss_a2)
    for a, f in zip(state_a + state_a2, list(st1) + list(st2)):
        assert torch.equal(a.reshape(-1), f.reshape(-1))
    for ga, gf in ((grads_a, grads_f), (grads_a2, grads_f2)):
        for k in prm:
            if k in ("rho", "alpha"):
                assert torch.allclose(ga[k], gf[k], rtol=1e-4, atol=1e-7 * float(ga[k].abs().max() + 1e-30)), k
            else:
                assert rel_err(gf[k], ga[k]) < 1e-5, (k, rel_err(gf[k], ga[k]))


def test_fused_window_accumulates_into_existing_grads():
    import iadmm_b200 as ia
    from oracle import iadmm_oracle as orc
    B, n, mi, me, h, TL = 2, 20, 5, 6, 16, 3
    qp = {k: v.to(DEV) for k, v in orc.qp_instances(B, n, mi, me, seed=3).items()}
    model = ia.LSTM(None, 2, h, TL, DEV)
    m = mi + me
    st = [torch.zeros((B, n, 1), device=DEV), torch.zeros((B, m, 1), device=DEV), torch.zeros((B, m, 1), device=DEV),
          torch.zeros((B, n + m, 1), device=DEV), torch.zeros((B, n + m, h), device=DEV), torch.zeros((B, n + m, h), device=DEV)]
    args = (TL, mi, me, qp["Q"], qp["p"], qp["A0"], qp["zl"], qp["zu"], 6e-6, st)
    model.train_window(*args)
    g1 = model.U_i.grad.clone()
    model.train_window(*args)
    assert torch.allclose(model.U_i.grad, 2 * g1, rtol=1e-6, atol=0)
    assert all(torch.count_nonzero(s) == 0 for s in st)          # the caller's state is not modified unless inplace=True


@pytest.mark.parametrize("mode", ["simt_fp32", "tc_f16f8"])
def test_recomputed_gates_give_identical_gradients(mode):
    """IADMM_TRAIN_RECOMPUTE_GATES (SURVEY.md section 7 step 6): the backward re-runs the forward's gate kernel on the saved
    H, C, xv, g instead of reading activations kept over the window -- same kernel, same inputs, so loss, end state and
    every parameter gradient are bit-identical, with a 3x smaller window workspace."""
    import ctypes
    import iadmm_b200 as ia
    from iadmm_b200 import _lib
    from oracle import iadmm_oracle as orc
    B, n, mi, me, h, TL = 3, 40, 12, 14, 48, 5
    qp = {k: v.to(DEV) for k, v in orc.qp_instances(B, n, mi, me, seed=83).items()}
    prm = orc.lstm_parameters(h, TL, seed=83, scale=2.0)
    m = mi + me
    out = []
    for rec in (False, True):
        model = ia.LSTM(None, 2, h, TL, DEV, gate_mode=mode)
        with torch.no_grad():
            for k, v in prm.items():
                getattr(model, k).copy_(v.to(DEV))
        st = [torch.zeros(s, device=DEV) for s in ((B, n, 1), (B, m, 1), (B, m, 1), (B, n + m, 1), (B, n + m, h), (B, n + m, h))]
        loss, st1 = model.train_window(TL, mi, me, qp["Q"], qp["p"], qp["A0"], qp["zl"], qp["zu"], 6e-6, st, recompute_gates=rec)
        loss2, st2 = model.train_window(TL, mi, me, qp["Q"], qp["p"], qp["A0"], qp["zl"], qp["zu"], 6e-6, st1, recompute_gates=rec)
        assert model.last_window_flags == (1 if rec else 0)
        out.append((loss, loss2, st2, {k: getattr(model, k).grad.clone() for k in prm}))
    assert torch.equal(out[0][0], out[1][0]) and torch.equal(out[0][1], out[1][1])
    for a, b in zip(out[0][2], out[1][2]):
        assert torch.equal(a, b)
    for k in prm:
        assert torch.equal(out[0][3][k], out[1][3][k]), k
    nb = [ctypes.c_size_t(), ctypes.c_size_t()]
    for f, v in zip((0, 1), nb):
        _lib.check(_lib.lib().iadmm_window_workspace_bytes(32, 1000, 1000, 800, 100, f, ctypes.byref(v)))
    assert nb[1].value < 0.45 * nb[0].value          # 129 GB -> < 58 GB at config 3, batch 32


def test_forward_under_autograd_returns_the_kkt_tuple():
    """models/lstm.py:96 always returns A_tild, b_tild, rho_vec; the training path returns them too (detached), A_tild only
    when `materialize_kkt` asks for the dense matrix (ADVICE r1)."""
    import iadmm_b200 as ia
    from oracle import iadmm_oracle as orc
    B, n, mi, me, h = 2, 12, 4, 5, 16
    m = mi + me
    qp = {k: v.to(DEV) for k, v in orc.qp_instances(B, n, mi, me, seed=87).items()}
    model = ia.LSTM(None, 2, h, 3, DEV)
    gen = torch.Generator().manual_seed(88)
    st = [torch.randn(s, generator=gen).to(DEV) for s in ((B, n, 1), (B, m, 1), (B, m, 1), (B, n + m, 1))]
    H = torch.tanh(torch.randn((B, n + m, h), generator=gen)).to(DEV); C = torch.randn((B, n + m, h), generator=gen).to(DEV)
    kw = dict(Q=qp["Q"], p=qp["p"], A0=qp["A0"], lb=None, ub=None, zl=qp["zl"], zu=qp["zu"])
    with torch.no_grad():
        ref = model(1, mi, me, *st, 6e-6, H, C, **kw)
    out = model(1, mi, me, *st, 6e-6, H, C, **kw)                   # grad mode: parameters require grad -> autograd node
    assert out[0].requires_grad and out[6] is not None
    for a, b in zip(out[6:], ref[6:]):
        assert torch.equal(a, b) and not a.requires_grad
    model.materialize_kkt = False
    out = model(1, mi, me, *st, 6e-6, H, C, **kw)
    assert out[6] is None and torch.equal(out[7], ref[7]) and torch.equal(out[8], ref[8])


def test_invalidate_packed_after_an_edit_through_param_data():
    """The packed-weight cache is keyed by (data_ptr, _version); an edit through `.data` bumps neither (ADVICE r1):
    `invalidate_packed()` is the documented way to make the kernels see it."""
    import iadmm_b200 as ia
    from oracle import iadmm_oracle as orc
    B, n, mi, me, h, K = 2, 16, 4, 4, 16, 3
    qp = {k: v.to(DEV) for k, v in orc.qp_instances(B, n, mi, me, seed=89).items()}
    args = (K, mi, me, qp["Q"], qp["p"], qp["A0"], qp["zl"], qp["zu"], 6e-6)
    model = ia.LSTM(None, 2, h, K, DEV).eval()
    with torch.no_grad():
        a = model.solve(*args)
        model.W_h.data.mul_(3.0)                                     # no version bump
        model.invalidate_packed()
        b = model.solve(*args)
        model.W_h.mul_(1.0 / 3.0)                                    # in-place op: version bump, noticed automatically
        c = model.solve(*args)
    assert not torch.equal(a.x, b.x)
    assert rel_err(c.x, a.x) < 1e-5
