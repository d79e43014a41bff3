"""The tensor-core GEMMs of the training backward (csrc/gemm_tc.cu, called from iadmm_step_bwd) against float64 autograd
through the oracle, at the shapes where their work decomposition changes:

    H_bar = D U^T    M = rows = B (n + m), N = h,  K = 4h
    U_bar = H^T D    M = h,  N = 4h,  K = rows, split over K by tc_gemm_pick_splits

One differentiable iteration (LSTM.forward under autograd: iadmm_step_fwd / iadmm_step_bwd) from a carried, non-zero state,
all six outputs driven by independent random cotangents, so that gH checks H_bar, the U_* gradients check U_bar, and the
state adjoints and every other parameter gradient are checked as well.  Bars are max(fixed, 3 x floor), the floor being the
oracle in float32 against the oracle in float64 on the same inputs (test_gpu_training).

At 10 to 16 splits the factor need not divide the K blocks: 125 blocks in 15 splits of 9 leave the 15th split without any.
launch_tc_gemm_nt launches only the splits that cover K blocks; before it did, such a unit stored a tensor-memory accumulator
that nothing in its launch had written, and split-K reduction added it into U_bar (U_* gradients off by 6e-2 ... 1.1 at the
four empty-split shapes below, and different from run to run).  Errors recorded below were measured on a B200 (148 SMs)."""
import pytest
import torch

from helpers import rel_err
from oracle import iadmm_oracle as orc

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
LENGTH, T = 3, 1                                   # a mid-schedule iteration
SIGMA = 6e-6
STATE = ("x", "y", "z", "xv", "H", "C")
QP_KEYS = ("Q", "p", "A0", "zl", "zu")
GM_BM, GM_BN, GM_BK, MAX_SPLITS = 128, 256, 64, 16      # kTcBM, kGmBN, kGmBK, kMaxSplitK


def cdiv(a, b):
    return -(-a // b)


def backward_gemm_regime(h, rows, num_sms):
    """What the training backward does with its two GEMMs at hidden_dim h and `rows` rows on `num_sms` SMs: the restated
    arithmetic of tc_gemm_pick_splits and launch_tc_gemm_nt (CTA-pair kernel, 256 x 256 tiles, one unit per pair of SMs)."""
    if h % 16 != 0:
        return dict(tc=False)
    pairs = num_sms // 2
    tiles = cdiv(h, 2 * GM_BM) * cdiv(4 * h, GM_BN)
    k_blocks = cdiv(rows, GM_BK)
    splits, best_eff = 1, 0.0
    if tiles < 4 * pairs:
        s = 1
        while s <= MAX_SPLITS and k_blocks // s >= 8:
            units = tiles * s
            eff = units / (cdiv(units, pairs) * pairs)
            if eff > best_eff + 1e-9:
                best_eff, splits = eff, s
            s += 1
    kb_per_split = cdiv(k_blocks, splits)
    covered = cdiv(k_blocks, kb_per_split)                 # splits that own at least one K block
    return dict(tc=True, rows_pad=rows % 8 != 0, k_tail=rows % GM_BK, ubar_tiles=tiles, splits=splits,
                empty_splits=splits - covered, ubar_units=tiles * covered, pairs=pairs,
                m_tail=h % (2 * GM_BM), n_tail=(4 * h) % GM_BN, hbar_units=cdiv(rows, 2 * GM_BM) * cdiv(h, GM_BN))


# (B, n, mi, me, h) and the regime each shape is there for (checked against backward_gemm_regime on the device's SM count)
SHAPES = {
    "rows_pad_k_tail": ((3, 301, 50, 50, 16), dict(rows_pad=True, k_tail=51, splits=2, empty_splits=0)),
    "m_tail_12_tiles": ((1, 1000, 500, 500, 384), dict(ubar_tiles=12, m_tail=128, splits=4, empty_splits=0)),
    "split10_empty": ((3, 1200, 264, 264, 64), dict(splits=10, empty_splits=1)),
    "split15_empty_h64": ((4, 1000, 500, 500, 64), dict(splits=15, empty_splits=1)),
    "split16_empty": ((41, 100, 50, 50, 128), dict(splits=16, empty_splits=1, k_tail=8)),
    "split15_empty_h208": ((4, 1000, 500, 500, 208), dict(splits=15, empty_splits=1, n_tail=64)),
    "h800_rounds": ((2, 1000, 500, 500, 800), dict(splits=7, empty_splits=0, ubar_units=364, m_tail=32, n_tail=128)),
    "hbar_second_round": ((12, 300, 50, 50, 800), dict(hbar_units=76, empty_splits=0)),
    "sgemm_h40": ((2, 300, 100, 100, 40), dict(tc=False)),
}
EMPTY_SPLIT = ("split10_empty", "split15_empty_h64", "split16_empty", "split15_empty_h208")


def check_regime(name):
    (B, n, mi, me, h), want = SHAPES[name]
    sms = torch.cuda.get_device_properties(DEV).multi_processor_count
    got = backward_gemm_regime(h, B * (n + mi + me), sms)
    assert {k: got[k] for k in want} == want, (name, sms, got)
    if name == "h800_rounds":
        assert got["ubar_units"] > 2 * got["pairs"]        # several units per pair: both accumulators, phase flips
    if name == "hbar_second_round":
        assert got["hbar_units"] > got["pairs"]


def make_case(B, n, mi, me, h, seed):
    """QP instances, parameters, a carried state and one cotangent per output.  The vector state is scaled by 4/sqrt(n+m) so
    that the least-squares gradient feature stays O(10) and the gate pre-activations O(1): no saturated gates, a dense D.
    H = tanh(.) stays inside (-1, 1) like the cell's output (the backward keeps H * 2^14 in fp16)."""
    m, N = mi + me, n + mi + me
    qp = orc.qp_instances(B, n, mi, me, seed=seed)
    qp = {k: qp[k] for k in QP_KEYS}
    prm = orc.lstm_parameters(h, LENGTH, seed=seed, scale=2.0)
    gen = torch.Generator().manual_seed(seed + 1)
    s = 4.0 / N ** 0.5
    state = [s * torch.randn(shape, generator=gen) for shape in ((B, n, 1), (B, m, 1), (B, m, 1), (B, N, 1))]
    state += [torch.tanh(torch.randn((B, N, h), generator=gen)), torch.randn((B, N, h), generator=gen)]
    cots = [torch.randn(v.shape, generator=gen) for v in state]
    return qp, prm, state, cots


def oracle_grads(qp, prm, state, cots, mi, me, dtype):
    p = {k: v.detach().to(dtype).clone().requires_grad_(True) for k, v in prm.items()}
    leaves = [v.detach().to(dtype).clone().requires_grad_(True) for v in state]
    d = [qp[k].to(dtype) for k in QP_KEYS]
    x, y, z, xv, H, C = leaves
    outs = orc.lstm_step(p, T, mi, me, x, y, z, xv, SIGMA, H, C, *d, form="block")[:6]
    torch.autograd.backward(outs, [c.to(dtype) for c in cots])
    return {**{"g" + k: v.grad for k, v in zip(STATE, leaves)}, **{k: v.grad for k, v in p.items()}}


def make_model(prm, h, mode, length=LENGTH):
    import iadmm_b200 as ia
    model = ia.LSTM(None, 2, h, length, DEV, gate_mode=mode)
    with torch.no_grad():
        for k, v in prm.items():
            getattr(model, k).copy_(v.to(DEV))
    model.materialize_kkt = False
    return model


def our_grads(model, qp, state, cots, mi, me):
    leaves = [v.detach().to(DEV).clone().requires_grad_(True) for v in state]
    d = {k: qp[k].to(DEV) for k in QP_KEYS}
    x, y, z, xv, H, C = leaves
    model.zero_grad(set_to_none=True)
    outs = model(T, mi, me, x, y, z, xv, SIGMA, H, C, lb=None, ub=None, **d)[:6]
    torch.autograd.backward(outs, [c.to(DEV) for c in cots])
    torch.cuda.synchronize()
    return {**{"g" + k: v.grad.detach().cpu() for k, v in zip(STATE, leaves)},
            **{k: getattr(model, k).grad.detach().cpu() for k in orc.PARAM_ORDER}}


def compare(label, shape, mode, fixed, seed):
    B, n, mi, me, h = shape
    qp, prm, state, cots = make_case(B, n, mi, me, h, seed)
    ref = oracle_grads(qp, prm, state, cots, mi, me, torch.float64)
    ref32 = oracle_grads(qp, prm, state, cots, mi, me, torch.float32)
    ours = our_grads(make_model(prm, h, mode), qp, state, cots, mi, me)
    assert sorted(ours) == sorted(ref)
    errs = {k: rel_err(ours[k], ref[k]) for k in ref if float(ref[k].abs().max()) > 0}
    floor = {k: rel_err(ref32[k].double(), ref[k]) for k in errs}
    bars = {k: max(fixed, 3.0 * floor[k]) for k in errs}
    worst = max(errs, key=lambda k: errs[k] / bars[k])
    print(f"\n{label} {shape} {mode}: worst {worst} {errs[worst]:.1e} (bar {bars[worst]:.1e});",
          " ".join(f"{k} {v:.1e}/{floor[k]:.0e}" for k, v in errs.items()))
    bad = {k: (errs[k], bars[k]) for k in errs if not errs[k] < bars[k]}
    assert not bad, bad
    # rows of the schedule other than T receive no gradient
    for k in ("rho", "alpha"):
        assert float(ours[k][torch.arange(LENGTH) != T].abs().max()) == 0.0, k


@pytest.mark.parametrize("name", list(SHAPES))
def test_backward_gemms_vs_float64(name):
    """The backward in isolation: the fp32 CUDA-core forward is bit-stable, so every error is the backward's.  Worst measured:
    gH (H_bar) 1.1e-5 at hidden_dim 800 -- its error grows with K = 4h: 9.5e-7 at 64, 3.0e-6 at 208, 5.4e-6 at 384 -- and
    gx 1.0e-5 (floor 1e-5); U_* 1.8e-6 ... 2.5e-6 at every shape (5.7e-7 through the fp32 sgemm backward at hidden_dim 40)."""
    check_regime(name)
    compare(name, SHAPES[name][0], "simt_fp32", 2e-5, seed=101)


@pytest.mark.parametrize("mode", ["tc_3xfp16", "tc_f16f8", "tc_1xfp16"])
@pytest.mark.parametrize("name", ["split15_empty_h64", "h800_rounds"])
def test_tensor_core_forward_modes(name, mode):
    """The training gate kernels of the tensor-core forward modes (<3,2,3>, <2,2,3>, <1,2,0>) ahead of the same backward.
    Worst measured: gx 2.2e-4 at hidden_dim 800 in all three modes (floor 6e-5: the same in every mode, so not the gate kernel's);
    otherwise <= 1.2e-5 for tc_3xfp16 / tc_f16f8 and <= 1.2e-4 for tc_1xfp16."""
    check_regime(name)
    compare(name, SHAPES[name][0], mode, 5e-3 if mode == "tc_1xfp16" else 5e-4, seed=103)


@pytest.mark.parametrize("name", EMPTY_SPLIT)
def test_backward_is_deterministic_across_foreign_tensor_memory(name):
    """The same backward twice, with a tensor-core solve at another hidden_dim in between: the gradients are bit-identical.
    The solve leaves its own values in tensor memory; a GEMM unit that stored an accumulator no MMA of its launch wrote would
    show them, whatever their size.  (The H_bar GEMM of the backward runs first and writes only N = h columns of each
    256-column accumulator, so the U_bar tile's other columns are still the solve's.)"""
    import iadmm_b200 as ia
    check_regime(name)
    B, n, mi, me, h = SHAPES[name][0]
    qp, prm, state, cots = make_case(B, n, mi, me, h, seed=107)
    model = make_model(prm, h, "simt_fp32")
    first = our_grads(model, qp, state, cots, mi, me)
    Bo, no, mio, meo, ho = 2, 1000, 500, 500, 800
    other = ia.LSTM(None, 2, ho, 2, DEV, gate_mode="tc_f16f8").eval()
    oqp = {k: v.to(DEV) for k, v in orc.qp_instances(Bo, no, mio, meo, seed=109).items()}
    with torch.no_grad():
        r = other.solve(2, mio, meo, *(oqp[k] for k in QP_KEYS), SIGMA, traces=False)
    torch.cuda.synchronize()
    assert bool(torch.isfinite(r.H).all())
    second = our_grads(model, qp, state, cots, mi, me)
    diff = {k: float((first[k] - second[k]).abs().max()) for k in first if not torch.equal(first[k], second[k])}
    assert not diff, diff


@pytest.mark.parametrize("recompute", [False, True])
def test_fused_window_at_empty_split_shape(recompute):
    """iadmm_train_window at a 15-split shape (hidden_dim 64, 8000 rows), TL = 2 from a carried state, with the gate
    activations kept and recomputed, against float64 autograd through the oracle (bars of test_window_gradients_match_autograd).
    Measured: every gradient within 2x of its floor, worst U_f 8.7e-5 (floor 9e-5)."""
    from test_gpu_training import oracle_window
    check_regime("split15_empty_h64")
    B, n, mi, me, h = SHAPES["split15_empty_h64"][0]
    TL, outer_T = 2, 4
    qp, _, state, _ = make_case(B, n, mi, me, h, seed=113)
    prm = orc.lstm_parameters(h, outer_T, seed=113, scale=2.0)
    ref_loss, ref_g, _ = oracle_window(prm, qp, mi, me, h, TL, outer_T, state=state)
    _, g32, _ = oracle_window(prm, qp, mi, me, h, TL, outer_T, state=state, dtype=torch.float32)
    model = make_model(prm, h, "simt_fp32", length=outer_T)
    model.zero_grad(set_to_none=True)
    loss, _ = model.train_window(TL, mi, me, *(qp[k].to(DEV) for k in QP_KEYS), SIGMA, [v.to(DEV) for v in state],
                                 loss_scale=1.0 / outer_T, recompute_gates=recompute)
    torch.cuda.synchronize()
    assert model.last_window_flags == (1 if recompute else 0)
    assert abs(float(loss) - ref_loss) <= 2e-5 * abs(ref_loss)
    errs = {k: rel_err(getattr(model, k).grad, ref_g[k]) for k in ref_g if float(ref_g[k].abs().max()) > 0}
    floor = {k: rel_err(g32[k].double(), ref_g[k]) for k in errs}
    print(f"\nfused window recompute={recompute}:", " ".join(f"{k} {v:.1e}/{floor[k]:.0e}" for k, v in errs.items()))
    bad = {k: (v, floor[k]) for k, v in errs.items() if not v < max(2e-4, 3.0 * floor[k])}
    assert not bad, bad
