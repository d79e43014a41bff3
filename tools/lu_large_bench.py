"""Stage-II factorisation above the register-resident limit: `lu_factor_blocked` (csrc/lu.cu) against
`torch.linalg.lu_factor` (what the reference's `torch.lu` runs) on the same tensors, plus `lu_solve` at these sizes.

    python tools/lu_large_bench.py [--B 1 8 24] [--N 5000 10000] [--reps 3] [--out FILE]

Per (matrix kind, B, N):
  - factor time of both paths (CUDA events, mean of --reps after one warm-up call), and TFLOP/s over the 2/3 N^3 B
    logical flop;
  - the blocked path split by phase, from a separate torch.profiler pass (kernel times summed by name):
      panel      the 16-column sub-panels on their clusters and the in-block swaps, TRSM and rank-16 band updates
      swap_trsm  the per-block row interchanges outside the block (laswp) and U12 = L11^-1 A12
      update     the tf32 hi/lo operand splits and the tensor-core trailing update A22 -= L21 U12
      perm       pivot sequence -> permutation
  - lu_solve time (one CTA per instance) and torch.linalg.lu_solve's;
  - residuals ||K x - b|| / ||b|| in fp64 of both solves, and the relative error against an fp64 solve for B = 1.
Matrix kinds: "kkt" (quasi-definite KKT matrices as LSTM.forward hands them to Stage II, built on the GPU) and
"random" (standard normal).  Writes one JSON document with the card's name and power limit.
"""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "i-admm-lstm_b200"))

DEV = "cuda:0"
PHASES = {
    "panel": ("lu_panel_cluster_kernel", "lu_swap_band_kernel", "lu_trsm_nb_kernel<16>", "lu_update_band_kernel"),
    "swap_trsm": ("lu_swap_kernel", "lu_trsm_nb_kernel<128>"),
    "update": ("lu_split_l_kernel", "lu_split_ut_kernel", "lu_tf32_update_kernel"),
    "perm": ("lu_perm_kernel",),
}


def kkt_like(B, n, m, seed):
    """Same construction as tests/test_gpu_lu.py::_kkt_like, generated on the GPU."""
    g = torch.Generator(device=DEV).manual_seed(seed)
    K = torch.empty(B, n + m, n + m, device=DEV)
    for b in range(B):
        M = torch.randn(n, n, generator=g, device=DEV) * (torch.rand(n, n, generator=g, device=DEV) < 0.15)
        Q = M @ M.T / n + 6e-6 * torch.eye(n, device=DEV)
        A = torch.randn(m, n, generator=g, device=DEV) * (torch.rand(m, n, generator=g, device=DEV) < 0.15)
        rho = torch.full((m,), 0.5, device=DEV)
        rho[m // 2:] *= 1e3
        K[b, :n, :n] = Q
        K[b, :n, n:] = A.T
        K[b, n:, :n] = A
        K[b, n:, n:] = torch.diag(-1 / rho)
    return K


def timed(fn, reps):
    fn()
    torch.cuda.synchronize()
    t = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        t.append(e0.elapsed_time(e1))
    return sum(t) / len(t), t


def phase_split(fn):
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    out = {k: 0.0 for k in PHASES}
    out["other"] = 0.0
    for ev in prof.key_averages():
        us = getattr(ev, "device_time_total", None)
        if us is None:
            us = ev.cuda_time_total
        if us <= 0:
            continue
        ph = next((ph for ph, names in PHASES.items() if any(n in ev.key for n in names)), "other")
        out[ph] += us / 1e3
    return out


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60).stdout.strip().splitlines()[0]
    except Exception as e:   # noqa: BLE001
        q = f"nvidia-smi unavailable: {e}"
    return {"nvidia_smi": q, "torch_name": torch.cuda.get_device_name(0)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--B", type=int, nargs="+", default=[1, 8, 24])
    ap.add_argument("--N", type=int, nargs="+", default=[5000, 10000])
    ap.add_argument("--kinds", nargs="+", default=["kkt", "random"])
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("lu_large_bench: no CUDA device (the measurement has no CPU form)")
    import iadmm_b200.lu as lum
    doc = {"card": card(), "torch": torch.__version__, "reps": a.reps, "results": []}
    for kind in a.kinds:
        for N in a.N:
            for B in a.B:
                K = kkt_like(B, N // 2, N - N // 2, seed=N + B) if kind == "kkt" else \
                    torch.randn(B, N, N, generator=torch.Generator(device=DEV).manual_seed(N + B), device=DEV)
                rhs = torch.randn(B, N, 1, generator=torch.Generator(device=DEV).manual_seed(1), device=DEV)
                flop = 2.0 / 3.0 * N ** 3 * B
                t_ours, t_ours_all = timed(lambda: lum.lu_factor_blocked(K), a.reps)
                t_torch, t_torch_all = timed(lambda: torch.linalg.lu_factor(K), a.reps)
                phases = phase_split(lambda: lum.lu_factor_blocked(K))
                lu, piv, info = lum.lu_factor_blocked(K)
                LUt, pvt = torch.linalg.lu_factor(K)
                t_solve, _ = timed(lambda: lum.lu_solve(lu, piv, rhs), a.reps)
                t_tsolve, _ = timed(lambda: torch.linalg.lu_solve(LUt, pvt, rhs), a.reps)
                x = lum.lu_solve(lu, piv, rhs).double()
                xt = torch.linalg.lu_solve(LUt, pvt, rhs).double()
                Kd, bd = K.double(), rhs.double()
                res = float(((Kd @ x - bd).norm(dim=(1, 2)) / bd.norm(dim=(1, 2))).max())
                res_t = float(((Kd @ xt - bd).norm(dim=(1, 2)) / bd.norm(dim=(1, 2))).max())
                r = dict(kind=kind, B=B, N=N, info_max=int(info.abs().max()),
                         factor_ms=t_ours, factor_ms_reps=t_ours_all, factor_tflops=flop / (t_ours * 1e-3) / 1e12,
                         torch_factor_ms=t_torch, torch_factor_ms_reps=t_torch_all,
                         torch_factor_tflops=flop / (t_torch * 1e-3) / 1e12,
                         speedup_vs_torch=t_torch / t_ours, phases_ms=phases,
                         solve_ms=t_solve, torch_solve_ms=t_tsolve, residual=res, torch_residual=res_t)
                if B == 1:
                    x64 = torch.linalg.solve(Kd, bd)
                    r["err_vs_fp64"] = float((x - x64).norm() / x64.norm())
                    r["torch_err_vs_fp64"] = float((xt - x64).norm() / x64.norm())
                    del x64
                doc["results"].append(r)
                print(json.dumps(r), flush=True)
                if a.out:                                 # rewritten after every shape: a cut-short run keeps what it measured
                    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
                    with open(a.out, "w") as f:
                        json.dump(doc, f, indent=1)
                del K, lu, piv, LUt, pvt, Kd, x, xt
                torch.cuda.empty_cache()
    print(json.dumps(doc["card"]))


if __name__ == "__main__":
    main()
