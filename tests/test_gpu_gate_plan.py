"""The gate-path table that plan_gates (csrc/gates_tc.cu) decides, seen from the outside: where IADMM_GATES_TC_F16F8U runs the
same arithmetic as IADMM_GATES_TC_F16F8 and where it drops the H-rounding correction, and that an unknown mode is rejected by the
training entry points as it is by the solve."""
import ctypes

import pytest
import torch

from helpers import rel_err

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
SIGMA = 6e-6
STATE = ("x", "y", "z", "xv", "H", "C")


def make(h, K, mode, seed=5):
    import iadmm_b200 as ia
    from oracle import iadmm_oracle as orc
    model = ia.LSTM(None, 2, h, K, DEV, gate_mode=mode)
    with torch.no_grad():
        for k, v in orc.lstm_parameters(h, K, seed=seed).items():
            getattr(model, k).copy_(v.to(DEV))
    return model


def scaled_qp(B, n, mi, me, seed=9):
    import iadmm_b200 as ia
    from oracle import iadmm_oracle as orc
    d = orc.qp_instances(B, n, mi, me, seed=seed)
    return ia.Scaling(n, mi + me, 10, DEV).scale_data(*(d[k].to(DEV) for k in ("Q", "p", "A0", "zl", "zu")))


def solve_both(h, B, n, mi, me, K, streaming):
    data = scaled_qp(B, n, mi, me)
    with torch.no_grad():
        return [make(h, K, mode).solve(K, mi, me, *data, SIGMA, traces=False, streaming=streaming) for mode in ("tc_f16f8", "tc_f16f8u")]


def test_f16f8u_is_f16f8_on_the_resident_solve():
    """n + m <= 256 at hidden_dim 64 runs the on-chip-resident kernel, which keeps both correction products in F16F8U."""
    a, b = solve_both(64, 3, 40, 12, 14, 6, streaming=False)
    for k in STATE:
        assert torch.equal(getattr(a, k), getattr(b, k)), k


@pytest.mark.parametrize("h", [64, 320, 400])
def test_f16f8u_drops_the_h_correction_on_the_streaming_solve(h):
    """K >= 2 on the streaming path runs the row-interleaved kernels, where F16F8U does not issue the H-rounding correction: the
    results differ from F16F8 by that rounding only.  At hidden_dim 64 and 320 F16F8 runs 16 epilogue warps and F16F8U 8, so the
    tail sums 4 and 2 head partials per unit tile respectively; a wrong count would not stay this close."""
    a, b = solve_both(h, 3, 40, 12, 14, 6, streaming=True)
    assert not torch.equal(a.H, b.H)
    for k in ("x", "xv", "H", "C"):
        assert rel_err(getattr(b, k), getattr(a, k)) < 1e-3, (k, rel_err(getattr(b, k), getattr(a, k)))


def test_f16f8u_is_f16f8_in_a_training_window():
    """Training keeps both correction products in both modes: loss, end state and gradients are bit-identical."""
    B, n, mi, me, h, TL = 2, 24, 7, 9, 16, 4
    Q, p, A0, zl, zu = scaled_qp(B, n, mi, me)
    m = mi + me
    out = []
    for mode in ("tc_f16f8", "tc_f16f8u"):
        model = make(h, TL, mode)
        st = [torch.zeros((B, n, 1), device=DEV), torch.zeros((B, m, 1), device=DEV), torch.zeros((B, m, 1), device=DEV),
              torch.zeros((B, n + m, 1), device=DEV), torch.zeros((B, n + m, h), device=DEV), torch.zeros((B, n + m, h), device=DEV)]
        loss, st1 = model.train_window(TL, mi, me, Q, p, A0, zl, zu, SIGMA, st)
        out.append((loss, st1, [prm.grad for prm in model.parameters()]))
    (la, sa, ga), (lb, sb, gb) = out
    assert torch.equal(la, lb)
    for a, b in zip(list(sa) + ga, list(sb) + gb):
        assert torch.equal(a, b)


def test_unknown_mode_is_rejected_by_training():
    """An unknown mode at hidden_dim % 8 != 0 used to run fp32 in training while the solve rejected it."""
    import iadmm_b200 as ia
    from iadmm_b200 import _lib
    L = ia.lib()
    B, n, mi, me, h, length = 1, 4, 1, 1, 60, 2
    m, rows = mi + me, B * (n + mi + me)
    nb = ctypes.c_size_t()
    _lib.check(L.iadmm_weights_bytes(h, length, ctypes.byref(nb)))
    packed = torch.zeros(nb.value, dtype=torch.uint8, device=DEV)
    Q, p, A0, zl, zu = (torch.zeros(s, device=DEV) for s in ((B, n, n), (B, n), (B, m, n), (B, m), (B, m)))
    x, y, z, xv, H, C = (torch.zeros(s, device=DEV) for s in ((B, n), (B, m), (B, m), (rows,), (rows, h), (rows, h)))
    outs = [torch.zeros_like(v) for v in (x, y, z, xv, H, C)]
    g_save, w_save = torch.zeros(rows, device=DEV), torch.zeros(rows, device=DEV)
    ws = torch.zeros(1 << 20, dtype=torch.uint8, device=DEV)
    P = _lib.ptr
    rc = L.iadmm_step_fwd(P(packed), P(Q), P(p), P(A0), P(zl), P(zu), *map(P, (x, y, z, xv, H, C)), *map(P, outs), P(g_save),
                          P(w_save), None, B, n, mi, me, h, length, 0, SIGMA, 77, P(ws), ws.numel(), _lib.stream_ptr())
    assert rc == -6                                    # IADMM_EMODE
    assert b"unknown gate mode 77" in L.iadmm_last_error()
    grad, loss = torch.zeros(1 << 16, device=DEV), torch.zeros(1, device=DEV)
    rc = L.iadmm_train_window(P(packed), P(Q), P(p), P(A0), P(zl), P(zu), *map(P, (x, y, z, xv, H, C)), P(grad), P(loss),
                              B, n, mi, me, h, length, 0, 1, SIGMA, 1.0, 77, 0, P(ws), ws.numel(), _lib.stream_ptr())
    assert rc == -6
    assert b"unknown gate mode 77" in L.iadmm_last_error()
    torch.cuda.synchronize()
