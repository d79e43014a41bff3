"""Blocked Stage-II factorisation (`iadmm_lu_factor_blocked`, csrc/lu.cu) for systems above the register-resident limit
of `iadmm_lu_factor` (N = 4096) up to N = 32768: LAPACK getrf semantics checked by P K = L U reconstruction in fp64, the
pivot sequence against torch.linalg.lu_factor and against the register-resident factor, ties across the CTAs of the
panel cluster, KKT solves through the unchanged `lu_solve`, singular input, workspace independence and determinism,
the C-ABI errors, and `LU.forward` at N > 4096 against the oracle's exact ADMM.
"""
import ctypes

import pytest
import torch

from helpers import rel_err
from test_gpu_lu import _kkt_like, _unpack

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
EWORK, EALIGN, EMODE = -5, -2, -6


def _separated(B, N, seed):
    """Rows of a diagonally dominant matrix in random order: every column's pivot is the row holding the diagonal
    entry, by a wide margin, so the interchange sequence is non-trivial but not sensitive to rounding."""
    g = torch.Generator(device=DEV).manual_seed(seed)
    K = torch.randn(B, N, N, generator=g, device=DEV) / N ** 0.5 + 4 * torch.eye(N, device=DEV)
    perm = torch.stack([torch.randperm(N, generator=g, device=DEV) for _ in range(B)])
    return torch.gather(K, 1, perm[:, :, None].expand(B, N, N)).contiguous()


def _reconstruction_error(K, lu, piv):
    B, N = K.shape[0], K.shape[1]
    L, U = _unpack(lu)
    perm = piv[1].long()
    PK = torch.gather(K.double(), 1, perm[:, :, None].expand(B, N, N))
    return float((L @ U - PK).abs().max() / K.abs().max())


@pytest.mark.parametrize("B,N", [(3, 1), (2, 17), (2, 130), (2, 1000), (1, 4097), (1, 5000), (1, 6001), (1, 10000)])
def test_factor_reconstructs_permuted_matrix(B, N):
    import iadmm_b200.lu as lum
    g = torch.Generator(device=DEV).manual_seed(N)
    K = torch.randn(B, N, N, generator=g, device=DEV)
    lu, piv, info = lum.lu_factor_blocked(K)
    assert int(info.abs().max()) == 0
    perm = piv[1].long()
    ar = torch.arange(N, device=DEV)
    assert all(torch.equal(torch.sort(perm[b]).values, ar) for b in range(B))
    err = _reconstruction_error(K, lu, piv)
    assert err < 2e-6 * max(1, N) ** 0.5, err
    assert float(torch.tril(lu, -1).abs().max()) <= 1.0 + 1e-6          # partial pivoting: |L| <= 1


@pytest.mark.parametrize("N", [64, 300, 4500])
def test_pivot_sequence_is_lapacks(N):
    import iadmm_b200.lu as lum
    K = _separated(2, N, seed=7 + N)
    _, piv, _ = lum.lu_factor_blocked(K)
    _, ref = torch.linalg.lu_factor(K.double())
    agree = (piv[0] == (ref - 1)).float().mean()
    assert float(agree) > 0.99, float(agree)


def test_first_maximum_across_cluster_ctas():
    """|-7| at row 100 (first CTA of the panel cluster) ties |+7| at row 4200 (second CTA): isamax takes row 100."""
    import iadmm_b200.lu as lum
    N = 4300
    g = torch.Generator(device=DEV).manual_seed(5)
    K = torch.rand(1, N, N, generator=g, device=DEV) * 2 - 1
    K[0, 100, 0] = -7.0
    K[0, 4200, 0] = 7.0
    _, piv, _ = lum.lu_factor_blocked(K)
    assert piv[0, 0, 0].item() == 100
    K[0, 100, 0] = 6.5                                   # and the larger magnitude wins from the second CTA
    _, piv, _ = lum.lu_factor_blocked(K)
    assert piv[0, 0, 0].item() == 4200


@pytest.mark.parametrize("N", [200, 2000, 4096])
def test_matches_register_resident_factor(N):
    import iadmm_b200.lu as lum
    K = _separated(2, N, seed=N)
    lu_r, piv_r, info_r = lum.lu_factor(K)
    lu_b, piv_b, info_b = lum.lu_factor_blocked(K)
    assert torch.equal(piv_r, piv_b) and torch.equal(info_r, info_b)
    err = float((lu_b.double() - lu_r.double()).abs().max() / lu_r.double().abs().max())
    assert err < 1e-5, err


@pytest.mark.parametrize("B,n,m", [(2, 2500, 2500), (1, 5000, 5000)])
def test_solve_on_kkt_systems(B, n, m):
    """The error bar of test_gpu_lu.py::test_solve_on_kkt_systems (5x torch's fp32 error against fp64).  Its fixed 1e-4
    residual bar is out of reach for any fp32 LU at these sizes: on a B200 torch.linalg.lu_factor/lu_solve leave
    2.9e-4 at N = 5000 and 8.1e-4 at N = 10000 (this path 2.0e-4 and 4.7e-4; at N = 4000 already torch 2.0e-4 and
    the register-resident factor 1.3e-4).  So the residual is held to torch's own on the same system."""
    import iadmm_b200.lu as lum
    K = _kkt_like(B, n, m, seed=n)
    N = n + m
    g = torch.Generator().manual_seed(3)
    rhs = torch.randn(B, N, 1, generator=g).to(DEV)
    lu, piv, info = lum.lu_factor_blocked(K)
    assert int(info.abs().max()) == 0
    x = lum.lu_solve(lu, piv, rhs)
    x64 = torch.linalg.solve(K.double(), rhs.double())
    lib = torch.linalg.lu_solve(*torch.linalg.lu_factor(K), rhs)
    err = float((x.double() - x64).norm() / x64.norm())
    err_lib = float((lib.double() - x64).norm() / x64.norm())
    res = float((K.double() @ x.double() - rhs.double()).norm() / rhs.double().norm())
    res_lib = float((K.double() @ lib.double() - rhs.double()).norm() / rhs.double().norm())
    assert res < res_lib, (res, res_lib)
    assert err < 5 * err_lib + 1e-6, (err, err_lib)


def test_singular_matrix_reports_info():
    import iadmm_b200.lu as lum
    g = torch.Generator(device=DEV).manual_seed(11)
    K = torch.randn(2, 4100, 4100, generator=g, device=DEV)
    K[1, :, 3000] = 0.0
    _, _, info = lum.lu_factor_blocked(K)
    assert info[0].item() == 0 and info[1].item() == 3001


def _call(K, ws, nbytes=None, Kptr=None):
    from iadmm_b200 import _lib
    B, N = K.shape[0], K.shape[1]
    lu = K.clone()
    piv = torch.empty(2, B, N, dtype=torch.int32, device=DEV)
    info = torch.empty(B, dtype=torch.int32, device=DEV)
    rc = _lib.lib().iadmm_lu_factor_blocked(_lib.ptr(lu) if Kptr is None else Kptr, _lib.ptr(piv[0]), _lib.ptr(piv[1]),
                                            _lib.ptr(info), B, N, _lib.ptr(ws), ws.numel() if nbytes is None else nbytes,
                                            _lib.stream_ptr())
    torch.cuda.synchronize()
    return rc, lu, piv, info


def _ws_bytes(B, N):
    from iadmm_b200 import _lib
    n = ctypes.c_size_t()
    _lib.check(_lib.lib().iadmm_lu_factor_blocked_workspace_bytes(B, N, ctypes.byref(n)))
    return n.value


@pytest.mark.parametrize("B,N", [(2, 1000), (2, 4500)])
def test_workspace_contents_do_not_matter_and_runs_repeat(B, N):
    g = torch.Generator(device=DEV).manual_seed(B * N)
    K = torch.randn(B, N, N, generator=g, device=DEV)
    nbytes = _ws_bytes(B, N)
    ws = torch.zeros(nbytes, dtype=torch.uint8, device=DEV)
    rc0, lu0, piv0, info0 = _call(K, ws)
    ws.fill_(0xFF)
    rc1, lu1, piv1, info1 = _call(K, ws)
    rc2, lu2, piv2, info2 = _call(K, ws)
    assert rc0 == rc1 == rc2 == 0
    for a, b in ((lu0, lu1), (lu1, lu2)):
        assert torch.equal(a.view(torch.int32), b.view(torch.int32))
    assert torch.equal(piv0, piv1) and torch.equal(piv1, piv2)
    assert torch.equal(info0, info1) and torch.equal(info1, info2)


def test_errors_through_the_c_abi():
    from iadmm_b200 import _lib
    L = _lib.lib()
    n = ctypes.c_size_t()
    assert L.iadmm_lu_factor_blocked_workspace_bytes(1, 32769, ctypes.byref(n)) == EMODE
    dummy = torch.zeros(64, device=DEV)
    assert L.iadmm_lu_factor_blocked(_lib.ptr(dummy), _lib.ptr(dummy), _lib.ptr(dummy), None, 1, 32769, _lib.ptr(dummy), 256,
                                     _lib.stream_ptr()) == EMODE
    assert b"32768" in L.iadmm_last_error()
    K = torch.randn(1, 300, 300, device=DEV)
    nbytes = _ws_bytes(1, 300)
    ws = torch.zeros(nbytes, dtype=torch.uint8, device=DEV)
    rc, _, _, _ = _call(K, ws, nbytes=nbytes - 1)
    assert rc == EWORK
    rc, _, _, _ = _call(K, ws, Kptr=ctypes.c_void_p(0))
    assert rc == EALIGN
    rc, lu, piv, _ = _call(K, ws)
    assert rc == 0 and _reconstruction_error(K, lu, piv) < 2e-6 * 300 ** 0.5


def test_stage2_lu_dropin_above_the_register_panel_limit():
    """main.py --feas_rest at N = n + m = 4200 (> 4096): LU.forward factors with the blocked path and its exact-ADMM
    iterates follow the oracle's float64 run."""
    import iadmm_b200 as ia
    from oracle import iadmm_oracle as orc
    from test_gpu_parity import make_model
    B, n, mi, me, h, K = 2, 2600, 900, 700, 16, 3
    qp = {k: v.to(DEV) for k, v in orc.qp_instances(B, n, mi, me, seed=97).items()}
    prm = orc.lstm_parameters(h, K, seed=97)
    model = make_model(prm, h, K, "tc_f16f8")
    m = mi + me
    st = [torch.zeros((B, n, 1), device=DEV), torch.zeros((B, m, 1), device=DEV), torch.zeros((B, m, 1), device=DEV),
          torch.zeros((B, n + m, 1), device=DEV), torch.zeros((B, n + m, h), device=DEV), torch.zeros((B, n + m, h), device=DEV)]
    kw = dict(Q=qp["Q"], p=qp["p"], A0=qp["A0"], lb=None, ub=None, zl=qp["zl"], zu=qp["zu"])
    with torch.no_grad():
        for tt in range(K):
            x, y, z, xv, H, C, A_tild, b_tild, rho_vec = model(tt, mi, me, *st[:4], 6e-6, st[4], st[5], **kw)
            st = [x, y, z, xv, H, C]
        assert A_tild.shape[-1] == 4200
        stage2 = ia.LU(DEV)
        lu = piv = None
        xr, yr, zr = (v.cpu().double() for v in (x, y, z))
        for _ in range(20):
            x, y, z, xv, A_tild, b_tild, lu, piv = stage2(rho_vec, x, y, z, xv, 6e-6, A_tild, lu, piv, **kw)
        ref = orc.exact_admm(*(qp[k].cpu().double() for k in ("Q", "p", "A0", "zl", "zu")), rho_vec.cpu().double(), 6e-6, 20,
                             state=(xr, yr, zr))
    assert rel_err(x, ref[0]) < 1e-3 and rel_err(z, ref[2]) < 1e-3


def test_lu_forward_selects_the_factor_by_size(monkeypatch):
    import iadmm_b200 as ia
    import iadmm_b200.lu as lum

    def refuse(K):
        raise AssertionError("lu_factor_blocked called at N <= 4096")

    def run(N):
        g = torch.Generator(device=DEV).manual_seed(N)
        n = N // 2
        x, xv = torch.zeros(1, n, 1, device=DEV), torch.zeros(1, N, 1, device=DEV)
        y = z = torch.zeros(1, N - n, 1, device=DEV)
        K = _separated(1, N, seed=N)
        kw = dict(p=torch.randn(1, n, 1, generator=g, device=DEV), zl=torch.full((1, N - n, 1), -1.0, device=DEV),
                  zu=torch.ones(1, N - n, 1, device=DEV))
        with torch.no_grad():
            return ia.LU(DEV)(torch.ones(1, N - n, 1, device=DEV), x, y, z, xv, 6e-6, K, None, None, **kw)

    real = lum.lu_factor_blocked
    monkeypatch.setattr(lum, "lu_factor_blocked", refuse)
    for N in (100, 4096):
        run(N)
    calls = []
    monkeypatch.setattr(lum, "lu_factor_blocked", lambda K: calls.append(K.shape[-1]) or real(K))
    run(4097)
    assert calls == [4097]
