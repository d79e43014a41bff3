"""torch.autograd bindings of the training entry points (iadmm_step_fwd/bwd, iadmm_residuals_fwd/bwd).

The reference trains by truncated BPTT through its Python loop (main.py:336-358): `model(t, ...)` and
`primal_dual_loss(...)` are recorded on the autograd tape.  Here each of the two is ONE autograd node whose
forward and backward are library calls, so main.py's training loop runs unchanged (Adam included) while
the tape holds, per iteration, only the small vectors, the gate activations [B*(n+m), 4h] and references
to the state tensors -- not the dense KKT matrix and the ~20 intermediates of the reference.
"""
from ctypes import byref, c_size_t

import torch

from . import _lib

PARAM_ORDER = ("W_i", "U_i", "b_i", "W_f", "U_f", "b_f", "W_o", "U_o", "b_o",
               "W_u", "U_u", "b_u", "W_h", "b_h", "rho", "alpha")


def _c(t):
    return None if t is None else t.contiguous()


def _train_ws(model, B, n, m, dev):
    nbytes = c_size_t()
    _lib.check(_lib.lib().iadmm_train_workspace_bytes(B, n, m, model.hidden_dim, byref(nbytes)))
    ws = getattr(model, "_train_ws", None)
    if ws is None or ws.numel() < nbytes.value or ws.device != dev:
        model._train_ws = None
        ws = model._train_ws = _lib.workspace(nbytes.value, dev)
    return ws


class StepFunction(torch.autograd.Function):
    """One I-ADMM-LSTM iteration (models/lstm.py:47-96) as a single differentiable node."""

    @staticmethod
    def forward(ctx, model, t, num_ineq, num_eq, sigma, Q, p, A0, zl, zu, x, y, z, xv, H, C, *params):
        L = _lib.lib()
        dev = Q.device
        Q, p, A0, zl, zu, x, y, z, xv, H, C = (_lib.f32(v, dev) for v in (Q, p, A0, zl, zu, x, y, z, xv, H, C))
        B, n = Q.shape[0], Q.shape[1]
        m = num_ineq + num_eq
        h = model.hidden_dim
        rows = B * (n + m)
        outs = [torch.empty_like(v) for v in (x, y, z, xv, H, C)]
        g_save = torch.empty((rows,), device=dev)
        w_save = torch.empty((rows,), device=dev)
        hp = -(-h // 4) * 4            # the training kernels run hidden_dim rounded up to 4 (include/iadmm.h)
        gates = torch.empty((rows, 4 * hp), device=dev)
        packed = model.packed_weights()
        ws = _train_ws(model, B, n, m, dev)
        with torch.cuda.device(dev):
            _lib.check(L.iadmm_step_fwd(_lib.ptr(packed), _lib.ptr(Q), _lib.ptr(p), _lib.ptr(A0), _lib.ptr(zl), _lib.ptr(zu),
                                        _lib.ptr(x), _lib.ptr(y), _lib.ptr(z), _lib.ptr(xv), _lib.ptr(H), _lib.ptr(C),
                                        *[_lib.ptr(o) for o in outs], _lib.ptr(g_save), _lib.ptr(w_save), _lib.ptr(gates),
                                        B, n, int(num_ineq), int(num_eq), h, model.length, int(t), float(sigma), model._mode(),
                                        _lib.ptr(ws), ws.numel(), _lib.stream_ptr()))
        ctx.model, ctx.meta = model, (int(t), int(num_ineq), int(num_eq), float(sigma), B, n, m, h)
        ctx.save_for_backward(Q, p, A0, zl, zu, x, y, z, xv, H, C, outs[3], outs[4], g_save, w_save, gates)
        ctx.n_params = len(params)
        return tuple(outs)

    @staticmethod
    def backward(ctx, gx_o, gy_o, gz_o, gxv_o, gH_o, gC_o):
        L = _lib.lib()
        model = ctx.model
        t, num_ineq, num_eq, sigma, B, n, m, h = ctx.meta
        Q, p, A0, zl, zu, x, y, z, xv, H, C, xv_o, H_o, g_save, w_save, gates = ctx.saved_tensors
        dev = Q.device
        gin = [_c(g) for g in (gx_o, gy_o, gz_o, gxv_o, gH_o, gC_o)]
        gout = [torch.empty_like(v) for v in (x, y, z, xv, H, C)]
        count = c_size_t()
        _lib.check(L.iadmm_param_count(h, model.length, byref(count)))
        flat = torch.zeros((count.value,), device=dev)
        packed = model.packed_weights()
        ws = _train_ws(model, B, n, m, dev)
        with torch.cuda.device(dev):
            _lib.check(L.iadmm_step_bwd(_lib.ptr(packed), _lib.ptr(Q), _lib.ptr(p), _lib.ptr(A0), _lib.ptr(zl), _lib.ptr(zu),
                                        _lib.ptr(x), _lib.ptr(y), _lib.ptr(z), _lib.ptr(xv), _lib.ptr(H), _lib.ptr(C),
                                        _lib.ptr(xv_o), _lib.ptr(H_o), _lib.ptr(g_save), _lib.ptr(w_save), _lib.ptr(gates),
                                        *[_lib.ptr(g) for g in gin], *[_lib.ptr(g) for g in gout], _lib.ptr(flat),
                                        B, n, num_ineq, num_eq, h, model.length, t, sigma,
                                        _lib.ptr(ws), ws.numel(), _lib.stream_ptr()))
        pgrads, off = [], 0
        for name in PARAM_ORDER:
            prm = getattr(model, name)
            k = prm.numel()
            pgrads.append(flat[off:off + k].view(prm.shape))
            off += k
        return (None,) * 10 + tuple(gout) + tuple(pgrads)


class ResidualFunction(torch.autograd.Function):
    """primal_dual_loss (utils.py:68-71): returns (pri, dual) as [B] tensors."""

    @staticmethod
    def forward(ctx, x, y, z, Q, p, A0):
        L = _lib.lib()
        dev = Q.device
        x, y, z, Q, p, A0 = (_lib.f32(v, dev) for v in (x, y, z, Q, p, A0))
        B, n, m = Q.shape[0], Q.shape[1], A0.shape[1]
        pri = torch.empty((B,), device=dev); dual = torch.empty((B,), device=dev)
        rp = torch.empty((B, m), device=dev); rd = torch.empty((B, n), device=dev)
        nbytes = c_size_t()
        _lib.check(L.iadmm_residuals_train_workspace_bytes(B, n, m, byref(nbytes)))
        ws = _lib.workspace(nbytes.value, dev)
        with torch.cuda.device(dev):
            _lib.check(L.iadmm_residuals_fwd(_lib.ptr(x), _lib.ptr(y), _lib.ptr(z), _lib.ptr(Q), _lib.ptr(p), _lib.ptr(A0),
                                             _lib.ptr(pri), _lib.ptr(dual), _lib.ptr(rp), _lib.ptr(rd), B, n, m,
                                             _lib.ptr(ws), ws.numel(), _lib.stream_ptr()))
        ctx.save_for_backward(Q, A0, pri, dual, rp, rd)
        ctx.shapes = (x.shape, y.shape, z.shape)
        return pri, dual

    @staticmethod
    def backward(ctx, gpri, gdual):
        L = _lib.lib()
        Q, A0, pri, dual, rp, rd = ctx.saved_tensors
        dev = Q.device
        B, n, m = Q.shape[0], Q.shape[1], A0.shape[1]
        gx = torch.empty((B, n), device=dev); gy = torch.empty((B, m), device=dev); gz = torch.empty((B, m), device=dev)
        nbytes = c_size_t()
        _lib.check(L.iadmm_residuals_train_workspace_bytes(B, n, m, byref(nbytes)))
        ws = _lib.workspace(nbytes.value, dev)
        with torch.cuda.device(dev):
            _lib.check(L.iadmm_residuals_bwd(_lib.ptr(Q), _lib.ptr(A0), _lib.ptr(pri), _lib.ptr(dual), _lib.ptr(rp), _lib.ptr(rd),
                                             _lib.ptr(_c(gpri)), _lib.ptr(_c(gdual)), _lib.ptr(gx), _lib.ptr(gy), _lib.ptr(gz),
                                             B, n, m, _lib.ptr(ws), ws.numel(), _lib.stream_ptr()))
        sx, sy, sz = ctx.shapes
        return gx.view(sx), gy.view(sy), gz.view(sz), None, None, None
