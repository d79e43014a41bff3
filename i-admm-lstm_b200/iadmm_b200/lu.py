"""Drop-in for the reference's `models/lu.py` (class `LU`, the optional Stage-II "feasibility restoration").

Stage II is OUTSIDE the accelerated path (SURVEY.md section 8 row f1): it is exact OSQP-style ADMM, one dense LU of
the KKT matrix and a triangular solve per iteration.  This module keeps `main.py --feas_rest` working on a B200
next to the drop-in `LSTM`/`Scaling`.  The factorisation (`iadmm_lu_factor`, csrc/lu.cu: register-resident
16-column panels, partial pivoting with LAPACK's first-maximum rule, N <= 4096; above that `iadmm_lu_factor_blocked`:
128-column blocks, cluster-wide pivot search and a 3xTF32 tensor-core trailing update, N <= 32768) and the
per-iteration triangular solves (`iadmm_lu_solve`) are the library's own kernels; the K matrix comes from `LSTM.forward`'s return tuple
(`iadmm_build_kkt`).  `lu`/`piv` in the return tuple are opaque to the caller exactly as in the reference
(main.py only hands them back): `lu` is the packed L\\U factor [B,N,N], `piv` an int32 tensor [2,B,N] holding
the interchange sequence and the row permutation derived from it.
"""
from ctypes import byref, c_size_t

import torch
import torch.nn as nn

from . import _lib

REGISTER_PANEL_MAX_N = 4096          # iadmm_lu_factor's limit: one CTA holds a 16-column panel in registers


def lu_factor(K):
    """Batched LU of K [B,N,N] (fp32, CUDA), N <= 4096.  Returns (lu, piv, info): see include/iadmm.h.
    Larger systems (up to N = 32768): `lu_factor_blocked`, same outputs."""
    _lib.require_cuda(K)
    B, N = K.shape[0], K.shape[1]
    lu = K.detach().to(torch.float32).contiguous().clone()
    piv = torch.empty(2, B, N, dtype=torch.int32, device=K.device)
    info = torch.empty(B, dtype=torch.int32, device=K.device)
    with torch.cuda.device(K.device):
        _lib.check(_lib.lib().iadmm_lu_factor(_lib.ptr(lu), _lib.ptr(piv[0]), _lib.ptr(piv[1]), _lib.ptr(info), B, N,
                                              _lib.stream_ptr()))
    return lu, piv, info


def lu_factor_blocked(K):
    """Batched LU of K [B,N,N] (fp32, CUDA) for N <= 32768: blocked, cluster-wide pivot search, 3xTF32 tensor-core
    trailing update.  Returns (lu, piv, info) in `lu_factor`'s format (`lu_solve` takes them unchanged)."""
    _lib.require_cuda(K)
    B, N = K.shape[0], K.shape[1]
    lu = K.detach().to(torch.float32).contiguous().clone()
    piv = torch.empty(2, B, N, dtype=torch.int32, device=K.device)
    info = torch.empty(B, dtype=torch.int32, device=K.device)
    L = _lib.lib()
    nbytes = c_size_t()
    _lib.check(L.iadmm_lu_factor_blocked_workspace_bytes(B, N, byref(nbytes)))
    ws = _lib.workspace(nbytes.value, K.device)
    with torch.cuda.device(K.device):
        _lib.check(L.iadmm_lu_factor_blocked(_lib.ptr(lu), _lib.ptr(piv[0]), _lib.ptr(piv[1]), _lib.ptr(info), B, N,
                                             _lib.ptr(ws), nbytes.value, _lib.stream_ptr()))
    return lu, piv, info


def lu_solve(lu, piv, rhs):
    """Solves K x = rhs with the factors of `lu_factor`; rhs [B,N] or [B,N,1]; returns x with rhs's shape."""
    _lib.require_cuda(lu)
    B, N = lu.shape[0], lu.shape[1]
    x = rhs.detach().to(torch.float32).reshape(B, N).contiguous().clone()
    with torch.cuda.device(lu.device):
        _lib.check(_lib.lib().iadmm_lu_solve(_lib.ptr(lu), _lib.ptr(piv[1]), _lib.ptr(x), B, N, _lib.stream_ptr()))
    return x.reshape(rhs.shape)


class LU(nn.Module):
    def __init__(self, device):
        super(LU, self).__init__()
        self.device = device

    def name(self):
        return 'torch_solver'

    def forward(self, rho_vec, x, y, z, xv, sigma, A_tild, lu, piv, **kwargs):
        """Same contract as models/lu.py:13-47: returns (x, y, z, xv, A_tild, b_tild, lu, piv)."""
        p, zl, zu = kwargs['p'], kwargs['zl'], kwargs['zu']
        inv_rho = 1 / rho_vec
        relax = 1.6                                         # models/lu.py:24
        b_tild = torch.cat((sigma * x - p, z - inv_rho * y), dim=1)
        if lu is None and piv is None:
            if A_tild is None:                              # assemble K as models/lu.py:28-29 does
                Q, A0 = kwargs['Q'], kwargs['A0']
                n, m = Q.shape[1], A0.shape[1]
                top = torch.cat((Q + sigma * torch.eye(n, device=Q.device), A0.transpose(1, 2)), dim=2)
                bot = torch.cat((A0, torch.diag_embed(-inv_rho.squeeze(-1))), dim=2)
                A_tild = torch.cat((top, bot), dim=1)
            if A_tild.shape[-1] <= REGISTER_PANEL_MAX_N:
                lu, piv, _ = lu_factor(A_tild)
            else:
                lu, piv, _ = lu_factor_blocked(A_tild)
        xv = lu_solve(lu, piv, b_tild)
        n = x.shape[1]
        x_tild, v = xv[:, :n, :], xv[:, n:, :]
        z_tild = z + inv_rho * (v - y)
        x = relax * x_tild + (1 - relax) * x
        z_rel = relax * z_tild + (1 - relax) * z
        z = torch.max(torch.min(z_rel + inv_rho * y, zu), zl)
        y = y + rho_vec * (z_rel - z)
        return x, y, z, xv, A_tild, b_tild, lu, piv
