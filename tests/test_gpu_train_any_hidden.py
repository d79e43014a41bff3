"""Training at hidden_dim % 4 != 0: the library runs such a model as the model of width hp = hidden_dim rounded up to 4 whose
extra units have zero parameters and a zero state (include/iadmm.h, training).  Those units stay exactly zero and feed nothing
into the real ones, so every output, adjoint and gradient must equal the explicitly padded model's bit for bit.  hp lands on
each regime of the training path: 4 (fp32 gates and backward), 32 (fp16+fp8 tensor-core forward, tcgen05 backward), 52 (fp32),
200 (three-product forward at hidden_dim % 16 == 8, fp32 backward)."""
import ctypes
import os

import numpy as np
import pytest
import torch

from helpers import load_golden, rel_err

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
SIGMA = 6e-6
STATE = ("x", "y", "z", "xv", "H", "C")
QP_KEYS = ("Q", "p", "A0", "zl", "zu")
B, N_VAR, MI, ME = 2, 24, 7, 9
HIDDEN = [1, 3, 30, 50, 199]


def ceil4(h):
    return -(-h // 4) * 4


def lib():
    import iadmm_b200 as ia
    return ia.lib()


def check(rc):
    from iadmm_b200 import _lib
    _lib.check(rc)


def P(t):
    from iadmm_b200 import _lib
    return _lib.ptr(t)


def S():
    from iadmm_b200 import _lib
    return _lib.stream_ptr()


def mode_id(mode):
    from iadmm_b200 import _lib
    return _lib.GATE_MODES[mode]


def pad_params(prm, h, hp):
    """The parameters of the width-hp model whose units h..hp-1 are zero."""
    out = {}
    for k, v in prm.items():
        if k.startswith("W_") and k != "W_h":
            w = torch.zeros((v.shape[0], hp)); w[:, :h] = v
        elif k.startswith("U_"):
            w = torch.zeros((hp, hp)); w[:h, :h] = v
        elif k.startswith("b_") and k != "b_h":
            w = torch.zeros(hp); w[:h] = v
        elif k == "W_h":
            w = torch.zeros((hp, 1)); w[:h] = v
        else:
            w = v.clone()
        out[k] = w
    return out


def pad_cols(t, hp):
    out = torch.zeros((t.shape[0], hp), device=t.device)
    out[:, :t.shape[1]] = t
    return out


def pack(prm, h, length):
    from oracle import iadmm_oracle as orc
    nb = ctypes.c_size_t()
    check(lib().iadmm_weights_bytes(h, length, ctypes.byref(nb)))
    buf = torch.zeros(nb.value, dtype=torch.uint8, device=DEV)
    dev = [prm[k].to(DEV).contiguous() for k in orc.PARAM_ORDER]
    check(lib().iadmm_pack_weights(*map(P, dev), h, length, P(buf), S()))
    return buf


def grads_by_name(flat, h, length):
    """The flat gradient buffer split into the 16 parameter tensors (state_dict order and shapes)."""
    from oracle import iadmm_oracle as orc
    shapes = {"W": (2, h), "U": (h, h), "b": (h,)}
    out, off = {}, 0
    for k in orc.PARAM_ORDER:
        shp = {"W_h": (h, 1), "b_h": (1,), "rho": (length, 1), "alpha": (length, 1)}.get(k) or shapes[k[0]]
        cnt = int(np.prod(shp))
        out[k] = flat[off:off + cnt].view(shp)
        off += cnt
    assert off == flat.numel()
    return out


def trim(g, h):
    """A gradient of the padded model restricted to the real units."""
    return {k: (v[:, :h] if (k.startswith("W_") and k != "W_h") else v[:h, :h] if k.startswith("U_")
                else v[:h] if (k.startswith("b_") and k != "b_h") or k == "W_h" else v) for k, v in g.items()}


def make_case(h, length, seed):
    from oracle import iadmm_oracle as orc
    qp = orc.qp_instances(B, N_VAR, MI, ME, seed=seed)
    qp = {k: qp[k].to(DEV).contiguous() for k in QP_KEYS}
    prm = orc.lstm_parameters(h, length, seed=seed, scale=2.0)
    m, rows = MI + ME, B * (N_VAR + MI + ME)
    gen = torch.Generator().manual_seed(seed + 1)
    s = 4.0 / (N_VAR + m) ** 0.5
    st = [s * torch.randn(shape, generator=gen) for shape in ((B, N_VAR), (B, m), (B, m), (rows,))]
    st += [torch.tanh(torch.randn((rows, h), generator=gen)), torch.randn((rows, h), generator=gen)]
    cots = [torch.randn(v.shape, generator=gen) for v in st]
    return qp, prm, [v.to(DEV) for v in st], [v.to(DEV) for v in cots]


def train_ws_bytes(h):
    nb = ctypes.c_size_t()
    check(lib().iadmm_train_workspace_bytes(B, N_VAR, MI + ME, h, ctypes.byref(nb)))
    return nb.value


def step(packed, qp, st, cots, h, length, t, mode, ws=None, fill=0):
    """iadmm_step_fwd + iadmm_step_bwd with a cotangent on each of the six outputs; returns the outputs, the saved gate
    activations, the input adjoints, the flat gradient and the workspace."""
    L = lib()
    rows = st[3].numel()
    if ws is None:
        ws = torch.full((train_ws_bytes(h),), fill, dtype=torch.uint8, device=DEV)
    outs = [torch.empty_like(v) for v in st]
    g_save, w_save = torch.empty(rows, device=DEV), torch.empty(rows, device=DEV)
    gates = torch.empty((rows, 4 * ceil4(h)), device=DEV)
    Q, p, A0, zl, zu = (qp[k] for k in QP_KEYS)
    check(L.iadmm_step_fwd(P(packed), P(Q), P(p), P(A0), P(zl), P(zu), *map(P, st), *map(P, outs), P(g_save), P(w_save), P(gates),
                           B, N_VAR, MI, ME, h, length, t, SIGMA, mode_id(mode), P(ws), ws.numel(), S()))
    fwd_ws = ws.clone()
    cnt = ctypes.c_size_t()
    check(L.iadmm_param_count(h, length, ctypes.byref(cnt)))
    flat = torch.zeros(cnt.value, device=DEV)
    gin = [torch.empty_like(v) for v in st]
    check(L.iadmm_step_bwd(P(packed), P(Q), P(p), P(A0), P(zl), P(zu), *map(P, st), P(outs[3]), P(outs[4]), P(g_save), P(w_save),
                           P(gates), *map(P, cots), *map(P, gin), P(flat), B, N_VAR, MI, ME, h, length, t, SIGMA,
                           P(ws), ws.numel(), S()))
    torch.cuda.synchronize()
    return outs, gates, gin, flat, fwd_ws


def window_ws_bytes(h, TL, flags):
    nb = ctypes.c_size_t()
    check(lib().iadmm_window_workspace_bytes(B, N_VAR, MI + ME, h, TL, flags, ctypes.byref(nb)))
    return nb.value


def window(packed, qp, st, h, length, t0, TL, mode, flags, fill=0):
    L = lib()
    ws = torch.full((window_ws_bytes(h, TL, flags),), fill, dtype=torch.uint8, device=DEV)
    st = [v.clone() for v in st]
    cnt = ctypes.c_size_t()
    check(L.iadmm_param_count(h, length, ctypes.byref(cnt)))
    flat, loss = torch.empty(cnt.value, device=DEV), torch.empty(1, device=DEV)
    Q, p, A0, zl, zu = (qp[k] for k in QP_KEYS)
    check(L.iadmm_train_window(P(packed), P(Q), P(p), P(A0), P(zl), P(zu), *map(P, st), P(flat), P(loss), B, N_VAR, MI, ME, h, length,
                               t0, TL, SIGMA, 0.25, mode_id(mode), flags, P(ws), ws.numel(), S()))
    torch.cuda.synchronize()
    return loss, st, flat, ws


def padded_image(prm, h, hp, t_first, count):
    """What the library's padded weight image must be: iadmm_pack_weights of the zero-padded parameters, with the schedule
    rows t_first .. t_first+count-1 of the call."""
    q = pad_params(prm, h, hp)
    q["rho"], q["alpha"] = q["rho"][t_first:t_first + count], q["alpha"][t_first:t_first + count]
    return pack(q, hp, count)


@pytest.mark.parametrize("mode", ["tc_f16f8", "simt_fp32"])
@pytest.mark.parametrize("h", HIDDEN)
def test_step_is_the_padded_model_bit_for_bit(h, mode):
    hp, length, t = ceil4(h), 4, 2
    qp, prm, st, cots = make_case(h, length, seed=200 + h)
    outs, gates, gin, flat, fwd_ws = step(pack(prm, h, length), qp, st, cots, h, length, t, mode)
    pst = st[:4] + [pad_cols(v, hp) for v in st[4:]]
    pcots = cots[:4] + [pad_cols(v, hp) for v in cots[4:]]
    pouts, pgates, pgin, pflat, _ = step(pack(pad_params(prm, h, hp), hp, length), qp, pst, pcots, hp, length, t, mode)
    # the padded weight image sits at the front of the step workspace
    want = padded_image(prm, h, hp, t, 1)
    assert torch.equal(fwd_ws[:want.numel()], want)
    for k, a, b in zip(STATE, outs, pouts):
        assert torch.equal(a, b[:, :h] if k in ("H", "C") else b), k
    for k in ("H", "C"):
        assert int(torch.count_nonzero(pouts[STATE.index(k)][:, h:])) == 0, k       # zero units stay zero
    assert torch.equal(gates, pgates)
    for k, a, b in zip(STATE, gin, pgin):
        assert torch.equal(a, b[:, :h] if k in ("H", "C") else b), "g" + k
    g, pg = grads_by_name(flat, h, length), trim(grads_by_name(pflat, hp, length), h)
    for k in g:
        assert torch.equal(g[k], pg[k]), k
    assert all(bool(torch.isfinite(v).all()) for v in outs + gin + [flat])


@pytest.mark.parametrize("recompute", [False, True])
@pytest.mark.parametrize("h", HIDDEN)
def test_window_is_the_padded_model_bit_for_bit(h, recompute):
    hp, length, t0, TL = ceil4(h), 6, 1, 3
    qp, prm, st, _ = make_case(h, length, seed=300 + h)
    flags = 1 if recompute else 0
    loss, st1, flat, ws = window(pack(prm, h, length), qp, st, h, length, t0, TL, "tc_f16f8", flags)
    pst = st[:4] + [pad_cols(v, hp) for v in st[4:]]
    ploss, pst1, pflat, _ = window(pack(pad_params(prm, h, hp), hp, length), qp, pst, hp, length, t0, TL, "tc_f16f8", flags)
    want = padded_image(prm, h, hp, t0, TL)
    assert torch.equal(ws[:want.numel()], want)
    assert torch.equal(loss, ploss)
    for k, a, b in zip(STATE, st1, pst1):
        assert torch.equal(a, b[:, :h] if k in ("H", "C") else b), k
    for k in ("H", "C"):
        assert int(torch.count_nonzero(pst1[STATE.index(k)][:, h:])) == 0, k
    g, pg = grads_by_name(flat, h, length), trim(grads_by_name(pflat, hp, length), h)
    for k in g:
        assert torch.equal(g[k], pg[k]), k
    assert float(g["U_i"].abs().max()) > 0


@pytest.mark.parametrize("h", [50, 30])
def test_one_iteration_vs_float64(h):
    """LSTM.forward under autograd from a carried state, all six outputs driven by random cotangents, against float64 autograd
    through the oracle, with the bars of test_gpu_train_gemm_edges.  LSTM runs simt_fp32 gates at hidden_dim % 8 != 0; the
    backward GEMMs are fp32 at 50 (hp = 52) and tcgen05 at 30 (hp = 32)."""
    from test_gpu_train_gemm_edges import compare
    compare(f"h{h}", (3, 301, 50, 50, h), "simt_fp32", 2e-5, seed=131)


def test_per_iteration_autograd_equals_train_window_h50():
    """The literal loop of main.py:336-358 through LSTM.forward + primal_dual_loss under autograd, and LSTM.train_window, at
    hidden_dim 50: the same kernels in the same order.  The rho / alpha gradients and the loss keep the tolerances of
    test_gpu_training.test_fused_window_equals_per_iteration_autograd (double accumulations)."""
    from oracle import iadmm_oracle as orc
    from test_gpu_training import our_window
    Bw, n, mi, me, h, TL = 2, 37, 9, 11, 50, 3
    outer_T = 2 * TL
    qp = orc.qp_instances(Bw, n, mi, me, seed=71)
    prm = orc.lstm_parameters(h, outer_T, seed=71)
    loss_a, grads_a, state_a, model = our_window(prm, qp, mi, me, h, TL, outer_T, mode="tc_f16f8")
    m = mi + me
    Q, p, A0, zl, zu = (qp[k].to(DEV) for k in QP_KEYS)
    st = [torch.zeros(s, device=DEV) for s in ((Bw, n, 1), (Bw, m, 1), (Bw, m, 1), (Bw, n + m, 1), (Bw, n + m, h), (Bw, n + m, h))]
    model.zero_grad()
    loss_f, st1 = model.train_window(TL, mi, me, Q, p, A0, zl, zu, SIGMA, st, t0=0, loss_scale=1.0 / outer_T)
    assert abs(float(loss_f) - loss_a) <= 1e-6 * abs(loss_a)
    for k, a, f in zip(STATE, state_a, st1):
        assert torch.equal(a.reshape(-1), f.reshape(-1)), k
    for k in prm:
        gf = getattr(model, k).grad
        if k in ("rho", "alpha"):
            assert torch.allclose(grads_a[k], gf, rtol=1e-4, atol=1e-7 * float(grads_a[k].abs().max() + 1e-30)), k
        else:
            assert torch.equal(grads_a[k], gf), (k, rel_err(gf, grads_a[k]))


def test_workspace_contents_do_not_matter_h50():
    h, length, t, TL = 50, 4, 1, 3
    qp, prm, st, cots = make_case(h, length, seed=401)
    packed = pack(prm, h, length)
    a = step(packed, qp, st, cots, h, length, t, "simt_fp32", fill=0)
    b = step(packed, qp, st, cots, h, length, t, "simt_fp32", fill=0xFF)
    for x, y in zip(a[0] + a[2] + [a[1], a[3]], b[0] + b[2] + [b[1], b[3]]):
        assert torch.equal(x, y) and bool(torch.isfinite(x).all())
    for flags in (0, 1):
        a = window(packed, qp, st, h, length, 0, TL, "simt_fp32", flags, fill=0)
        b = window(packed, qp, st, h, length, 0, TL, "simt_fp32", flags, fill=0xFF)
        for x, y in zip([a[0], a[2]] + a[1], [b[0], b[2]] + b[1]):
            assert torch.equal(x, y) and bool(torch.isfinite(x).all())


def test_workspace_one_byte_short_h50():
    L = lib()
    h, length, TL = 50, 4, 2
    qp, prm, st, cots = make_case(h, length, seed=403)
    packed = pack(prm, h, length)
    rows = st[3].numel()
    nbytes = train_ws_bytes(h)
    assert nbytes > train_ws_bytes(52)               # the padded weights and state come on top of the width-52 workspace
    ws = torch.zeros(nbytes, dtype=torch.uint8, device=DEV)
    Q, p, A0, zl, zu = (qp[k] for k in QP_KEYS)
    outs = [torch.empty_like(v) for v in st]
    g_save, w_save, gates = torch.empty(rows, device=DEV), torch.empty(rows, device=DEV), torch.empty((rows, 4 * 52), device=DEV)
    rc = L.iadmm_step_fwd(P(packed), P(Q), P(p), P(A0), P(zl), P(zu), *map(P, st), *map(P, outs), P(g_save), P(w_save), P(gates),
                          B, N_VAR, MI, ME, h, length, 0, SIGMA, 0, P(ws), nbytes - 1, S())
    assert rc == -5 and b"workspace too small" in L.iadmm_last_error()
    flat = torch.zeros(20000, device=DEV)
    gin = [torch.empty_like(v) for v in st]
    rc = L.iadmm_step_bwd(P(packed), P(Q), P(p), P(A0), P(zl), P(zu), *map(P, st), P(outs[3]), P(outs[4]), P(g_save), P(w_save),
                          P(gates), *map(P, cots), *map(P, gin), P(flat), B, N_VAR, MI, ME, h, length, 0, SIGMA, P(ws), nbytes - 1, S())
    assert rc == -5
    wb = window_ws_bytes(h, TL, 0)
    wws = torch.zeros(wb, dtype=torch.uint8, device=DEV)
    loss = torch.zeros(1, device=DEV)
    rc = L.iadmm_train_window(P(packed), P(Q), P(p), P(A0), P(zl), P(zu), *map(P, st), P(flat), P(loss), B, N_VAR, MI, ME, h, length,
                              0, TL, SIGMA, 1.0, 0, 0, P(wws), wb - 1, S())
    assert rc == -5
    torch.cuda.synchronize()


def test_main_py_training_branch_at_hidden_dim_50(tmp_path):
    """main.py's training branch as written, with --hidden_dim 50 (it stopped at the first iteration before)."""
    from oracle import iadmm_oracle as orc
    from main_py_runner import run_main_py
    from test_gpu_main_py import REF, REF_FILES, printed_numbers
    if not all(os.path.exists(os.path.join(REF, f)) for f in REF_FILES):
        pytest.skip("needs the reference project's main.py and utils.py in baseline/_ref, which the repository does not contain")
    g = load_golden("main_py_train_QP")
    _, K, epochs, TL, _ = (int(v) for v in g["meta"])
    h = 50
    prm = orc.lstm_parameters(h, K, seed=17)
    ck, out = run_main_py("QP", "dropin", REF, str(tmp_path), prm, h, K, "cuda:0", scaling=True,
                          train=dict(epochs=epochs, lr=float(g["lr"]), TL=TL))
    torch.cuda.synchronize()
    assert {k: tuple(v.shape) for k, v in ck.items()} == {k: tuple(v.shape) for k, v in prm.items()}
    assert all(bool(torch.isfinite(v).all()) for v in ck.values())
    assert any(not torch.equal(ck[k].cpu(), prm[k]) for k in prm)
    rows, nums = printed_numbers(out)
    assert rows and nums.size and np.isfinite(nums).all(), out[-2000:]
