#!/usr/bin/env python
"""Benchmark of the I-ADMM-LSTM unrolled solve path on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference|reference-gpu] [--workload W] [--gate-mode M] [--batch B]
                    [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Workloads (`--workload`; the default `solve` is the headline BASELINE config 2, the line the driver records):
    solve     config 2: n=1000, 500+500, hidden_dim=800, --scaling, K=100, batch 256 per GPU
    config5   config 5: n=5000, 2500+2500, hidden_dim=800, K=100, batch 24 per GPU
    hidden200 configs/QP.yaml's default hidden_dim 200 (% 16 == 8: half-padded last operand group): HBM-bound regime
    train     config 3: one truncated-BPTT window (TL=100) forward + backward + NCCL gradient all-reduce + Adam per step
    sparse    a sparse family of generate_data.py:96-228 (--family Random_QP | Equality_QP | SVM) at n=1000: Q / A0 streamed in the
              bitmap-slab form (--sparse auto) or densified like main.py:243-296 (--sparse off)

One "step" = the hot path over one batch of synthetic QPs: Ruiz equilibration (10 its) + K=100 unrolled
I-ADMM-LSTM iterations + the per-iteration primal/dual residual traces, for `batch` instances per GPU of
BASELINE config 2 (n=1000, 500 ineq + 500 eq, hidden_dim=800, --scaling).  The batch shards by instance
across GPUs with no collective (weak scaling: every rank solves its own `batch` instances).

Prints ONE JSON line (rank 0).  `value` = solves/s with inputs resident in HBM; `e2e` = the same through
the public API with pinned HOST buffers, H2D/D2H copies inside the timed region; `roofline` = the gate
kernel (tensor-bound) measured live with CUDA events through the library's profile hooks, plus
`roofline_kkt` for the HBM-bound KKT phase; `cpu_baseline` = the oracle port of the reference's torch
path on the host cores (bounded sample).  `--impl reference` times the CPU path alone: the UNMODIFIED reference modules from the git-ignored
baseline/_ref (kind "reference") when that copy travelled with the snapshot, else the oracle port (kind "port").
`--impl reference-gpu` runs the same unmodified reference modules on the B200 itself (stock PyTorch fp32, TF32 off,
device-timed): the like-for-like "what torch gives you on this GPU" number, also reported as `gpu_reference` in our line.
"""
import argparse
import dataclasses
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for _p in (ROOT, os.path.join(ROOT, "i-admm-lstm_b200")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

import torch  # noqa: E402

N_VAR, N_INEQ, N_EQ, HIDDEN, K_ITERS, SIGMA, RUIZ_ITS = 1000, 500, 500, 800, 100, 6e-6, 10
METRIC = "QP solves/sec (K=100, n=1000, m=1000)"
UNIT = "solves/s"
WORKLOAD = ("config2: dense QP n=1000, 500 ineq + 500 eq, hidden_dim=800, --scaling (10 Ruiz its), K=100 "
            "unrolled iterations + per-iteration residual traces, random-init LSTM")


_REAL_STDOUT = None


def quiet_stdout():
    """Point fd 1 at stderr for the rest of the run (NCCL prints its version banner to stdout from C, whatever NCCL_DEBUG
    says on some boxes); the ONE JSON line goes to the real stdout through emit()."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)


def emit(line):
    out = _REAL_STDOUT or sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference", "reference-gpu"])
    ap.add_argument("--workload", default="solve", choices=["solve", "config5", "hidden200", "train", "sparse"])
    ap.add_argument("--family", default="Random_QP", choices=["Random_QP", "Equality_QP", "SVM"],
                    help="sparse workload: problem family of generate_data.py:96-228")
    ap.add_argument("--sparse", default="off", choices=["auto", "off"],
                    help="Q / A0 in the library's sparse forms where measured density / block structure allow (SparseBatch.auto), or streamed "
                         "dense like the reference's densified tensors (the default, also for the headline workload)")
    ap.add_argument("--gate-mode", default="tc_f16f8", choices=["tc_3xfp16", "tc_f16f8", "tc_f16f8u", "tc_1xfp16", "simt_fp32"])
    ap.add_argument("--batch", type=int, default=None, help="instances per GPU (default: 256 solve, 24 config5, 2 train)")
    ap.add_argument("--iters", type=int, default=K_ITERS, help="unrolled iterations per solve (metric is quoted at 100)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-balance", action="store_true",
                    help="N > 1: keep equal shards instead of sharding the N*batch instances by each GPU's measured rate")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--cpu-batch", type=int, default=4, help="instances per CPU step of the reference arm (~0.8 s each on 16 cores)")
    ap.add_argument("--nvar", type=int, default=N_VAR, help="variables per QP (the metric is quoted at 1000; 5000 = BASELINE config 5, "
                                                             "with num_ineq = num_eq = nvar/2)")
    ap.add_argument("--hidden", type=int, default=HIDDEN, help="hidden_dim (the metric is quoted at 800; 200 is configs/QP.yaml's default)")
    ap.add_argument("--no-literal-loop", action="store_true", help="skip the reference's literal per-iteration loop through the drop-in modules")
    ap.add_argument("--no-gpu-reference", action="store_true", help="skip the stock-PyTorch-on-this-GPU sample in our line")
    ap.add_argument("--gpu-ref-batch", type=int, default=32, help="instances per step of the stock-PyTorch GPU arm")
    ap.add_argument("--tl", type=int, default=100, help="train: truncated_length of the window")
    ap.add_argument("--recompute", action="store_true", help="train: recompute the gate activations in the backward (3x less memory)")
    ap.add_argument("--abi-allreduce", action="store_true", help="train, N > 1: issue the gradient all-reduce through the library's own "
                                                                  "iadmm_allreduce_grads (raw NCCL communicator) instead of torch.distributed")
    ap.add_argument("--graph", action="store_true", help="train: capture scale_data + the window (forward, loss, backward) in ONE CUDA graph "
                                                          "and replay it per step (the library only enqueues on the caller's stream)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step returned as DIR/<name>.npy (rank 0's instances; "
                         "at most 64 MB in all, larger outputs as a fixed seeded sample of their rows, see dump_outputs; implies --no-balance)")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    if a.workload == "config5":
        a.nvar = 5000
    if a.workload == "hidden200":
        a.hidden = 200
    if a.batch is None:
        a.batch = {"solve": 256, "config5": 24, "hidden200": 256, "train": 2, "sparse": 128}[a.workload]
    return a


# ---------------------------------------------------------------------------------------------------
# synthetic inputs: generate_data.py:67-76 restated on the device (main.py:718 doubles Q on load)
# ---------------------------------------------------------------------------------------------------
def device_qp_batch(B, n, mi, me, seed, dev):
    from iadmm_b200.data import generate_qp_batch
    d = generate_qp_batch(B, n, mi, me, seed, dev)
    return d["Q"], d["p"], d["A0"], d["zl"], d["zu"]


# ---------------------------------------------------------------------------------------------------
# --dump-outputs: the arrays of the last timed step, for comparing two builds output for output
# ---------------------------------------------------------------------------------------------------
DUMP_BYTES = 64 * 10**6
NPY_HEADER = 256          # bytes reserved per .npy file for its header


def dump_outputs(outdir, arrays):
    """Write each tensor of `arrays` (name -> tensor) as outdir/<name>.npy, float64 if it is float64 else float32, within
    DUMP_BYTES in all.  Smallest first, each array gets an equal share of what the ones before it left; an array larger than
    its share is viewed as rows of its last dimension and stored as a sample of them, drawn by a generator with a fixed seed,
    so every run and every build at the same shape picks the same rows.  Their indices go to <name>_rows.npy (float64)."""
    import numpy as np
    os.makedirs(outdir, exist_ok=True)
    items = sorted(((k, v.detach()) for k, v in arrays.items() if v is not None), key=lambda kv: (kv[1].numel(), kv[0]))
    left = DUMP_BYTES - 2 * NPY_HEADER * len(items)
    for i, (name, t) in enumerate(items):
        dt = torch.float64 if t.dtype == torch.float64 else torch.float32
        esize = 8 if dt == torch.float64 else 4
        share = left // (len(items) - i)
        if t.numel() * esize <= share:
            out = t.to(dt).cpu()
        else:
            rows = t.reshape(-1, t.shape[-1] if t.dim() > 1 else 1)
            keep = share // (rows.shape[1] * esize + 8)
            if keep < 1:
                raise RuntimeError(f"--dump-outputs: one row of {name} {tuple(t.shape)} does not fit its share of {DUMP_BYTES} bytes")
            idx = torch.randperm(rows.shape[0], generator=torch.Generator().manual_seed(0))[:keep].sort().values
            out = rows[idx.to(rows.device)].to(dt).cpu()
            np.save(os.path.join(outdir, name + "_rows.npy"), idx.numpy().astype(np.float64))
            left -= idx.numel() * 8
        np.save(os.path.join(outdir, name + ".npy"), out.numpy())
        left -= out.numel() * esize


# ---------------------------------------------------------------------------------------------------
# clocks during the timed region
# ---------------------------------------------------------------------------------------------------
class ClockSampler:
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")
    NAMES = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")

    def __init__(self, dev):
        self.proc = None
        self.path = None
        try:
            uuid = str(torch.cuda.get_device_properties(dev).uuid)
            self.gpu_id = uuid if uuid.startswith("GPU-") else "GPU-" + uuid
        except Exception:
            self.gpu_id = str(torch.device(dev).index or 0)

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(["nvidia-smi", "-i", self.gpu_id, "--query-gpu=" + self.FIELDS,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.proc is None:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        clocks, mx, reasons, power = [], None, set(), []
        try:
            for line in open(self.path):
                f = [s.strip() for s in line.split(",")]
                if len(f) < 7:
                    continue
                try:
                    clocks.append(float(f[0])); mx = float(f[1]); power.append(float(f[2]))
                except ValueError:
                    continue
                for name, v in zip(self.NAMES, f[3:7]):
                    if v == "Active":
                        reasons.add(name)
            os.unlink(self.path)
        except Exception:
            pass
        if clocks:
            out.update(sm_mhz=statistics.median(clocks), sm_max_mhz=mx, reasons=sorted(reasons), samples=len(clocks),
                       power_w_max=max(power) if power else None)
        return out


# ---------------------------------------------------------------------------------------------------
# the reference arms: the unmodified reference modules (baseline/_ref) on the host cores or on the GPU; the oracle port
# of the same torch CPU path when the copy is not there
# ---------------------------------------------------------------------------------------------------
def _ref_inputs(batch, n, mi, me, h, iters, device):
    from oracle import iadmm_oracle as orc          # input generators only (qp_instances / lstm_parameters)
    qp = orc.qp_instances(batch, n, mi, me, seed=17)
    prm = orc.lstm_parameters(h, iters, seed=17)
    return {k: v.to(device) for k, v in qp.items()}, prm


def cpu_reference_solves_per_s(steps, warmup, cpu_batch, iters, n=N_VAR, h=HIDDEN):
    """Ruiz + K iterations + residual per iteration on the host cores.  What main.py times: scale_data (:825-834) + the K
    model() calls (:881-890); residuals as in :955."""
    from baseline import ref_arm
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    mi = me = n // 2
    qp, prm = _ref_inputs(cpu_batch, n, mi, me, h, iters, "cpu")
    if ref_arm.available():
        kind = "reference"
        model = ref_arm.make_model(prm, h, iters, "cpu")

        def one_step():
            ref_arm.solve(model, iters, mi, me, qp["Q"], qp["p"], qp["A0"], qp["zl"], qp["zu"], SIGMA, RUIZ_ITS)
        how = "UNMODIFIED reference modules (models/lstm.py, methods/scaling.py incl. its O(n^3) dense-diag Ruiz, utils.py) from baseline/_ref"
    else:
        from oracle import iadmm_oracle as orc
        kind = "port"

        def one_step():
            Qs, ps, As, zls, zus, sc = orc.ruiz_equilibrate(qp["Q"], qp["p"], qp["A0"], qp["zl"], qp["zu"], RUIZ_ITS)
            orc.solve(prm, iters, mi, me, Qs, ps, As, zls, zus, SIGMA, h, scaling=sc,
                      original=(qp["Q"], qp["p"], qp["A0"]), form="dense")
        how = ("oracle port (dense-KKT form like models/lstm.py:67-72; NOTE its Ruiz is O(n^2) where the reference's dense-diag "
               "bmm's are O(n^3), 0.32 s/instance in BASELINE.md: the port is slightly FASTER than the reference)")
    with torch.no_grad():
        for _ in range(warmup):
            one_step()
        t0 = time.perf_counter()
        for _ in range(steps):
            one_step()
        dt = time.perf_counter() - t0
    sample = (f"{steps} x ({cpu_batch} instance(s) of the same workload, Ruiz + K={iters}), {how}, "
              f"torch {torch.__version__} CPU fp32, {cores} threads")
    return cpu_batch * steps / dt, dt / steps * 1e3, cores, sample, kind


def gpu_reference_solves_per_s(steps, warmup, batch, iters, dev, n=N_VAR, h=HIDDEN):
    """The unmodified reference modules with device='cuda' (stock PyTorch fp32 kernels, TF32 off like torch's default),
    timed on the device around scale_data + K x (model() + primal_dual_loss).  None when baseline/_ref is absent."""
    from baseline import ref_arm
    if not ref_arm.available():
        return None
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    mi = me = n // 2
    qp, prm = _ref_inputs(batch, n, mi, me, h, iters, dev)
    model = ref_arm.make_model(prm, h, iters, dev)

    def one_step():
        return ref_arm.solve(model, iters, mi, me, qp["Q"], qp["p"], qp["A0"], qp["zl"], qp["zu"], SIGMA, RUIZ_ITS)

    for _ in range(warmup):
        one_step()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        r = one_step()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    del r
    torch.cuda.empty_cache()
    return {"value": batch * steps / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms / steps, "batch_per_step": batch,
            "steps": steps, "warmup": warmup,
            "what": ("UNMODIFIED reference modules (baseline/_ref: models/lstm.py, methods/scaling.py, utils.py) on this GPU, "
                     "device='cuda', stock PyTorch %s fp32 (TF32 off), same workload: Ruiz + K=%d x (model() + primal_dual_loss), "
                     "device-timed with CUDA events" % (torch.__version__, iters))}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    steps, warmup = args.steps, max(0, args.warmup)
    n, h = args.nvar, args.hidden
    workload = workload_name(args)
    if args.impl == "reference-gpu":
        dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0")))
        torch.cuda.set_device(dev)
        g = gpu_reference_solves_per_s(steps, max(1, warmup), args.gpu_ref_batch, args.iters, dev, n, h)
        if g is None:
            emit({"impl": "reference-gpu", "unavailable": "baseline/_ref is not in this snapshot (run build() in the build container)"})
            return
        line = {"impl": "reference-gpu", "metric": METRIC, "value": g["value"], "unit": UNIT, "n_gpus": 1, "steps": steps,
                "warmup": max(1, warmup), "ms_per_step": g["ms_per_step"], "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": {"workload": workload, "batch_per_step": args.gpu_ref_batch, "iters": args.iters},
                "gpu_reference": g, "gpu_launches": 0}
        emit(line)
        return
    val, ms, cores, sample, kind = cpu_reference_solves_per_s(steps, warmup, args.cpu_batch, args.iters, n, h)
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": steps,
            "warmup": warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload, "batch_per_step": args.cpu_batch, "iters": args.iters},
            "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample},
            "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    emit(line)


def workload_name(args):
    n, h = args.nvar, args.hidden
    if args.workload == "sparse":
        return ("sparse family %s of generate_data.py:96-228 at num_var=%d (densified on load like main.py:243-296), hidden_dim=%d, "
                "--scaling, K=%d; Q / A0 %s (NOT the headline workload)"
                % (args.family, n, h, args.iters, "streamed in the bitmap-slab sparse form where below 0.3 %% density" if args.sparse == "auto"
                   else "streamed dense"))
    if args.workload == "train":
        return ("config3: TBPTT training window, dense QP n=%d, %d ineq + %d eq, hidden_dim=%d, --scaling, truncated_length=%d, "
                "forward + backward + gradient all-reduce + Adam" % (n, n // 2, n // 2, h, args.tl))
    if n == N_VAR:
        return WORKLOAD if h == HIDDEN else WORKLOAD.replace("hidden_dim=800", "hidden_dim=%d" % h) + " (NOT the headline hidden_dim)"
    return ("config5: dense QP n=%d, %d ineq + %d eq, hidden_dim=%d, --scaling, K=%d (NOT the headline workload)"
            % (n, n // 2, n // 2, h, args.iters))


# ---------------------------------------------------------------------------------------------------
# our arm
# ---------------------------------------------------------------------------------------------------
def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        d = json.load(open(path))
        return d.get("hbm_gbs", 6650.0), d.get("bf16_tflops_sustained", 1400.0), d.get("bf16_tflops", 1590.0), "measured"
    return 6650.0, 1400.0, 1590.0, "fallback"


def ncu_traffic(kind, batch, mode, headline=True, suffix=""):
    """DRAM bytes per launch from the committed ncu --set full capture of this config, if any."""
    if not headline:
        return None
    path = os.path.join(ROOT, "profiles", "roofline_traffic.json")
    if os.path.exists(path):
        try:
            d = json.load(open(path))
            return d.get(f"{kind}:{mode}:B{batch}{suffix}")
        except Exception:
            return None
    return None


def run_ours(args):
    import torch.distributed as dist
    import iadmm_b200 as ia
    from ctypes import byref, c_double, c_int

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("NCCL_DEBUG", "WARN")
        quiet_stdout()                                       # keep NCCL's version banner off stdout (one JSON line only)
        dist.init_process_group("nccl", device_id=dev)
    n_gpus = world
    B, n, mi, me, h, K = args.batch, args.nvar, args.nvar // 2, args.nvar // 2, args.hidden, args.iters
    m, N = mi + me, n + mi + me
    steps, warmup = args.steps, max(3, args.warmup)
    L = ia.lib()

    torch.manual_seed(17)                                    # identical random-init weights on every rank
    model = ia.LSTM(None, 2, h, K, dev, gate_mode=args.gate_mode).eval()
    # N > 1: the job is N*B independent instances.  GPUs of one box differ by several per cent under the power cap, so after
    # the warm-up the instances are re-sharded in proportion to each GPU's measured rate (iadmm_b200.dist.balance_by_rate: one
    # all-gather of a float per rank at set-up; the solve itself has no collective).  Every rank generates some spare instances.
    # (not with --dump-outputs: rank 0's share, and so the shapes it dumps, must follow from the arguments alone)
    balance = world > 1 and not args.no_balance and not args.dump_outputs
    B_cap = B + max(8, B // 8) if balance else B
    sparse_mode = args.workload == "sparse"
    if sparse_mode and "--sparse" not in sys.argv:
        args.sparse = "auto"
    if sparse_mode:
        from iadmm_b200.data import generate_family_batch
        fam = generate_family_batch(args.family, B_cap, n if args.family != "SVM" else n // 2, num_ineq=n if args.family == "Random_QP" else n // 2,
                                    num_eq=n, seed=17 + rank, device=dev)
        Q, p, A0, zl, zu = (fam[k] for k in ("Q", "p", "A0", "zl", "zu"))
        n, mi, me = fam["num_var"], fam["num_ineq"], fam["num_eq"]
        m, N = mi + me, n + mi + me
    else:
        Q, p, A0, zl, zu = device_qp_batch(B_cap, n, mi, me, 17 + rank, dev)
    full_inputs = (Q, p, A0, zl, zu)
    Q, p, A0, zl, zu = (t[:B] for t in full_inputs)
    shares = [B] * world
    scaling = ia.Scaling(n, m, RUIZ_ITS, dev)

    sp_caps = {}

    def hot_step():
        Qs, ps, As, zls, zus = scaling.scale_data(Q, p, A0, zl, zu)
        if args.sparse == "auto":
            # the first call measures density / block occupancy (host syncs) and decides per matrix; later calls rebuild the
            # chosen form without synchronising (it is part of the step: it has to follow the Ruiz scaling)
            if not sp_caps:
                for key, M_ in (("q", Qs), ("a", As)):
                    sb = ia.SparseBatch.auto(M_)
                    sp_caps[key] = None if sb is None else (sb.kind, sb.cap, sb.density if sb.kind == "slabs" else sb.occupancy,
                                                            sb.bytes_per_instance)
            pair = tuple(None if sp_caps[key] is None else
                         (ia.SparseBatch.pack(M_, cap=sp_caps[key][1]) if sp_caps[key][0] == "slabs" else ia.SparseBatch.blocks(M_))
                         for key, M_ in (("q", Qs), ("a", As)))
            if pair[0] is not None or pair[1] is not None:
                return model.solve(K, mi, me, Qs, ps, As, zls, zus, SIGMA, scaling=scaling, sparse=pair)
        return model.solve(K, mi, me, Qs, ps, As, zls, zus, SIGMA, scaling=scaling, streaming=sparse_mode)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    with torch.no_grad():
        for _ in range(warmup):
            r = hot_step()
        barrier()
        if balance:
            from iadmm_b200.dist import balance_by_rate
            w0, w1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            w0.record()
            for _ in range(2):
                r = hot_step()
            w1.record()
            torch.cuda.synchronize()
            B_mine, shares = balance_by_rate(world * B, 2 * B / (w0.elapsed_time(w1) * 1e-3), cap=B_cap)
            Q, p, A0, zl, zu = (t[:B_mine] for t in full_inputs)
            r = hot_step()                                   # workspace for the new share, untimed
            B = B_mine
            barrier()
        sampler = ClockSampler(dev) if rank == 0 else None
        if sampler:
            sampler.start()
        ia._lib.check(L.iadmm_profile_begin(steps * K))
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        torch.cuda.profiler.start()      # `ncu --profile-from-start off` captures exactly the timed region
        e0.record()
        for _ in range(steps):
            r = hot_step()
        e1.record()
        barrier()
        torch.cuda.profiler.stop()
        ms = e0.elapsed_time(e1)
        kkt_ms, gate_ms, tail_ms, nit = c_double(), c_double(), c_double(), c_int()
        ia._lib.check(L.iadmm_profile_end(byref(kkt_ms), byref(gate_ms), byref(tail_ms), byref(nit)))
        clocks = sampler.stop() if sampler else None
        finite = bool(torch.isfinite(r.x).all() and torch.isfinite(r.pri).all())
        if args.dump_outputs and rank == 0:
            dump_outputs(args.dump_outputs, {f.name: getattr(r, f.name) for f in dataclasses.fields(r)})

        # ---- e2e: same step through the public API from pinned host buffers --------------------------
        e2e = None
        if not args.no_e2e:
            host_in = [t.cpu().pin_memory() for t in (Q, p, A0, zl, zu)]
            # two device input buffers: the H2D copy of step i+1 (copy stream) overlaps the solve of step i
            dev_in = [[torch.empty_like(t) for t in (Q, p, A0, zl, zu)] for _ in range(2)]
            host_out = None
            copy_stream = torch.cuda.Stream()
            copied = [torch.cuda.Event(), torch.cuda.Event()]
            consumed = [torch.cuda.Event(), torch.cuda.Event()]

            def upload(i):
                with torch.cuda.stream(copy_stream):
                    copy_stream.wait_event(consumed[i % 2])          # buffer free again?
                    for d_, h_ in zip(dev_in[i % 2], host_in):
                        d_.copy_(h_, non_blocking=True)
                    copied[i % 2].record(copy_stream)

            def e2e_step(i, last):
                nonlocal host_out
                cur = torch.cuda.current_stream()
                cur.wait_event(copied[i % 2])
                Qs, ps, As, zls, zus = scaling.scale_data(*dev_in[i % 2])
                consumed[i % 2].record(cur)                          # scale_data has read the raw inputs
                if not last:
                    upload(i + 1)
                rr = model.solve(K, mi, me, Qs, ps, As, zls, zus, SIGMA, scaling=scaling)
                outs = (rr.x, rr.y, rr.z, rr.pri, rr.dual, rr.pri_unscaled, rr.dual_unscaled, rr.metrics)
                if host_out is None:
                    host_out = [torch.empty(o.shape, dtype=o.dtype).pin_memory() for o in outs]
                for h_, o in zip(host_out, outs):
                    h_.copy_(o, non_blocking=True)
                return outs

            for ev in consumed:
                ev.record(torch.cuda.current_stream())
            upload(0)
            for i in range(2):
                outs = e2e_step(i, i == 1)
            barrier()
            t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0.record()
            upload(2)                                    # every timed step's H2D copy is inside the timed region
            for i in range(2, 2 + steps):
                outs = e2e_step(i, i == 1 + steps)
            t1.record()
            barrier()
            e2e_ms = t0.elapsed_time(t1)
            h2d = sum(t.numel() * t.element_size() for t in host_in)
            d2h = sum(o.numel() * o.element_size() for o in outs)
            e2e = (e2e_ms, h2d, d2h)

    # max over ranks
    times = torch.tensor([ms, e2e[0] if e2e else 0.0], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(times, op=dist.ReduceOp.MAX)
    ms, e2e_ms = float(times[0]), float(times[1])

    if rank == 0:
        hbm_gbs, tf_sus, tf_burst, peak_kind = measured_peaks()
        rows = B * N
        nit_v = max(1, nit.value)
        gate_avg_ms = gate_ms.value / nit_v
        kkt_avg_ms = kkt_ms.value / nit_v
        gate_flops = 8.0 * rows * h * h                      # logical fp32 flops of H@U (no credit for the 3-way split)
        gate_tflops = gate_flops / (gate_avg_ms * 1e-3) / 1e12 if gate_avg_ms > 0 else 0.0
        gate_gbs = 16.0 * rows * h / (gate_avg_ms * 1e-3) / 1e9 if gate_avg_ms > 0 else 0.0      # H and C read once, written once
        kkt_bytes = 8.0 * B * (n * n + m * n)                # Q and A0 streamed once per pass, two passes
        kkt_dense_bytes = kkt_bytes
        sparse_info = None
        if args.sparse == "auto":
            per_pass = (sp_caps["q"][3] if sp_caps.get("q") else 4.0 * n * n) + (sp_caps["a"][3] if sp_caps.get("a") else 4.0 * m * n)
            kkt_bytes = 2.0 * B * per_pass

            def info(v):
                return None if not v else {"form": v[0], "density" if v[0] == "slabs" else "block_occupancy": v[2], "bytes_per_pass": v[3]}
            sparse_info = {"Q": info(sp_caps.get("q")), "A0": info(sp_caps.get("a")),
                           "dense_bytes_per_pass": 4.0 * (n * n + m * n), "stored_bytes_per_pass": per_pass,
                           "note": "opt-in (--sparse auto): structural zeros of Q / A0 are not streamed; results are bit-identical to the dense path"}
        kkt_gbs = kkt_bytes / (kkt_avg_ms * 1e-3) / 1e9 if kkt_avg_ms > 0 else 0.0
        iter_bytes = kkt_bytes + 16.0 * rows * h + 64.0 * rows       # SURVEY section 8(d) bytes per iteration
        step_s = ms / steps * 1e-3
        hbm_frac_whole = (iter_bytes * K / step_s / 1e9) / hbm_gbs
        # the step also runs scale_data and the trailing residual pass; SURVEY section 8(d) counts their algorithmic bytes per solve
        # (Ruiz: RUIZ_ITS read passes + one write pass of the dense Q and A0 = its 11 x 4 (n^2 + mn); one more read pass for the residuals of
        # the last iterate)
        solve_bytes = iter_bytes * K + (RUIZ_ITS + 1) * 4.0 * B * (n * n + m * n) + kkt_bytes / 2
        hbm_frac_solve = (solve_bytes / step_s / 1e9) / hbm_gbs
        launches_per_step = K * 6 + 2 + (3 + 2 * RUIZ_ITS)
        line = {
            "metric": METRIC, "value": sum(shares) * steps / (ms * 1e-3), "unit": UNIT, "n_gpus": n_gpus,
            "steps": steps, "warmup": warmup, "ms_per_step": ms / steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload_name(args),
                       "matrix_form": ("dense streaming of Q and A0 (the reference's densified tensors)" if args.sparse != "auto" else
                                       "OPT-IN --sparse auto: structural zeros not streamed (per matrix: bitmap slabs / block skipping / dense "
                                       "by measured density and block occupancy); results bit-identical to dense streaming"),
                       "batch_per_gpu": args.batch, "instances_per_gpu": shares, "iters": K, "gate_mode": args.gate_mode,
                       "gate_arithmetic": {"tc_3xfp16": "tcgen05 fp16 hi/lo split, 3 MMAs, fp32 accumulate",
                                           "tc_f16f8": "tcgen05 fp16 MMA + 2 e4m3 correction MMAs, fp32 accumulate",
                                           "tc_f16f8u": "tcgen05 fp16 MMA + 1 e4m3 correction MMA (weights rounding only), fp32 accumulate",
                                           "tc_1xfp16": "tcgen05 single fp16 MMA, fp32 accumulate",
                                           "simt_fp32": "fp32 FMA"}[args.gate_mode],
                       "cache": "inputs larger than L2: Q+A0 %.2f GB and LSTM state %.2f GB per GPU per iteration vs 126 MB L2"
                                % (kkt_bytes / 2 / 1e9, 16.0 * rows * h / 1e9),
                       "parallelism": ("%d x %d independent instances sharded over %d GPU(s)%s, no collective in the solve"
                                       % (n_gpus, args.batch, n_gpus, " in proportion to each GPU's measured warm-up rate" if balance else "")),
                       "results_finite": finite},
            "gpu_launches": steps * launches_per_step,
            # the gate kernel against the roofline that binds it: tensor at hidden_dim 800 (8 h^2 flops per row against 16 h bytes of
            # state), HBM for hidden_dim <~ 256 (SURVEY section 8d); both fractions are in the line, `bound` names the larger
            "roofline": {"kernel": "gates_tc_pair_kernel" if args.gate_mode != "simt_fp32" else "gates_simt_kernel",
                         **({"bound": "tensor", "achieved": gate_tflops, "peak": tf_sus, "unit": "TFLOP/s", "frac": gate_tflops / tf_sus}
                            if gate_tflops / tf_sus >= gate_gbs / hbm_gbs else
                            {"bound": "hbm", "achieved": gate_gbs, "peak": hbm_gbs, "unit": "GB/s", "frac": gate_gbs / hbm_gbs}),
                         "tensor_frac": gate_tflops / tf_sus, "hbm_frac": gate_gbs / hbm_gbs, "state_bytes_per_launch": 16.0 * rows * h,
                         "traffic": ncu_traffic("gates", B, args.gate_mode, (h == HIDDEN or h == 200) and n == N_VAR, "" if h == HIDDEN else ":h%d" % h),
                         "traffic_source": "profiles/roofline_traffic.json: dram__bytes_read+write of one committed ncu --set full "
                                           "capture of this kernel at this shape (not measured in this run)",
                         "peak_kind": ("%s bf16_tflops_sustained (kernel timed inside a long step)" if gate_tflops / tf_sus >= gate_gbs / hbm_gbs
                                       else "%s hbm_gbs") % peak_kind,
                         "flops_per_launch": gate_flops, "ms_per_launch": gate_avg_ms,
                         "share_of_step": gate_ms.value / ms,
                         "issued_frac": gate_tflops * {"tc_3xfp16": 3, "tc_f16f8": 2}.get(args.gate_mode, 1) / tf_sus,
                         "note": "logical fp32 flops 8*rows*h^2; the operand split issues %dx that in fp16-equivalent MMA work "
                                 "(tc_3xfp16: 3 fp16 products, tc_f16f8: 1 fp16 + 2 e4m3 at twice the rate; issued rate %.1f TFLOP/s "
                                 "= issued_frac of the peak); the kernel runs at the board power cap (see clocks), DESIGN.md section 4"
                                 % ({"tc_3xfp16": 3, "tc_f16f8": 2}.get(args.gate_mode, 1),
                                    gate_tflops * {"tc_3xfp16": 3, "tc_f16f8": 2}.get(args.gate_mode, 1))},
            "roofline_kkt": {"kernel": "kkt_pass1+combine1+pass2+combine2", "bound": "hbm", "achieved": kkt_gbs,
                             "peak": hbm_gbs, "unit": "GB/s", "frac": kkt_gbs / hbm_gbs,
                             "traffic": ncu_traffic("kkt", B, args.gate_mode, n == N_VAR),
                             "bytes_per_iteration": kkt_bytes, "dense_bytes_per_iteration": kkt_dense_bytes, "sparse": sparse_info,
                             "ms_per_iteration": kkt_avg_ms,
                             "share_of_step": kkt_ms.value / ms, "peak_kind": "%s hbm_gbs" % peak_kind},
            "hbm_roofline_frac_whole_path": hbm_frac_whole,
            "hbm_roofline_frac_whole_solve": hbm_frac_solve,     # same, with the algorithmic bytes of scale_data and the trailing residual pass
            "phase_ms_per_iteration": {"kkt": kkt_avg_ms, "gates": gate_avg_ms, "tail": tail_ms.value / nit_v},
            "clocks": clocks,
        }
        if e2e:
            line["e2e"] = {"value": sum(shares) * steps / (e2e_ms * 1e-3), "unit": UNIT,
                           "h2d_bytes_per_step": e2e[1], "d2h_bytes_per_step": e2e[2], "ms_per_step": e2e_ms / steps}
        if n_gpus == 1 and not args.no_literal_loop and not sparse_mode:
            # the reference's LITERAL loop (main.py:837-843, 874-887, 955) through the drop-in modules: K Python-level calls of
            # model(t, ...) with the returned state fed back + primal_dual_loss per iteration, nine fresh tensors per call
            # (incl. the dense A_tild) -- what a user gets who only swaps the imports.  Informational; `value` is the fused call.
            def literal():
                Qs, ps, As, zls, zus = scaling.scale_data(Q, p, A0, zl, zu)
                st = [torch.zeros((B, d_, w_), device=dev) for d_, w_ in ((n, 1), (m, 1), (m, 1), (N, 1), (N, h), (N, h))]
                for t_ in range(K):
                    st = list(model(t_, mi, me, st[0], st[1], st[2], st[3], SIGMA, st[4], st[5], Q=Qs, p=ps, A0=As, lb=None, ub=None,
                                    zl=zls, zu=zus)[:6])
                    ia.primal_dual_loss(st[0], st[1], st[2], Qs, ps, As)
                return st
            with torch.no_grad():
                literal()
                l0, l1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                torch.cuda.synchronize()
                l0.record()
                st_l = literal()
                l1.record()
                torch.cuda.synchronize()
            line["literal_loop"] = {"value": B / (l0.elapsed_time(l1) * 1e-3), "unit": UNIT, "ms_per_step": l0.elapsed_time(l1),
                                    "resumed_calls": model.resumed_calls, "x_equals_fused": bool(torch.equal(st_l[0], r.x)),
                                    "what": "K x { model(t, ...) ; primal_dual_loss(...) } as main.py:874-887,955 writes it, state fed "
                                            "back, fresh dense A_tild per call; 1 timed run after 1 warm-up"}
            del st_l
        if n_gpus == 1 and not args.no_gpu_reference and not sparse_mode:
            # stock PyTorch on the same B200 (SURVEY section 8d): bounded sample, after our timed regions
            try:
                line["gpu_reference"] = gpu_reference_solves_per_s(1, 1, min(args.gpu_ref_batch, 32 if n <= 1000 else 2), K, dev, n, h) or \
                    {"unavailable": "baseline/_ref is not in this snapshot"}
            except Exception as exc:                                              # never lose the bench line to the side arm
                line["gpu_reference"] = {"unavailable": "%s: %s" % (type(exc).__name__, str(exc)[:200])}
        if n_gpus == 1 and not args.no_cpu_baseline and not sparse_mode:
            cb = 4 if n <= 1000 else 1
            val, cms, cores, sample, kind = cpu_reference_solves_per_s(3 if n <= 1000 else 1, 1 if n <= 1000 else 0, cb, K, n, h)
            # ~12 instances, 10-20 s of CPU work; batches of 4 are the CPU path's best operating point at n=1000
            # (measured 1.3 solves/s at batch 1-4, 0.56 at batch 12: the dense KKT build falls out of cache)
            line["cpu_baseline"] = {"value": val, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample}
        emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


# ---------------------------------------------------------------------------------------------------
# training workload (BASELINE config 3): one truncated-BPTT window per step, main.py:336-358 through the drop-in modules
# ---------------------------------------------------------------------------------------------------
def run_train(args):
    import torch.distributed as dist
    import iadmm_b200 as ia
    from iadmm_b200.dist import allreduce_gradients
    from ctypes import c_double, c_int

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("NCCL_DEBUG", "WARN")
        quiet_stdout()
        dist.init_process_group("nccl", device_id=dev)
    B, n, mi, me, h, TL = args.batch, args.nvar, args.nvar // 2, args.nvar // 2, args.hidden, args.tl
    m, N = mi + me, n + mi + me
    steps, warmup = args.steps, max(3, args.warmup)
    L = ia.lib()
    torch.manual_seed(17)                                    # identical initial weights on every rank
    model = ia.LSTM(None, 2, h, TL, dev, gate_mode=args.gate_mode)
    opt = torch.optim.Adam(model.parameters(), lr=5e-5, weight_decay=0.0)          # main.py:191
    Q, p, A0, zl, zu = device_qp_batch(B, n, mi, me, 17 + rank, dev)
    scaling = ia.Scaling(n, m, RUIZ_ITS, dev)
    ar_ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    comm = None
    if world > 1 and args.abi_allreduce:
        from iadmm_b200.dist import nccl_comm
        comm = nccl_comm()

    def zero_state():
        return (torch.zeros((B, n, 1), device=dev), torch.zeros((B, m, 1), device=dev), torch.zeros((B, m, 1), device=dev),
                torch.zeros((B, N, 1), device=dev), torch.zeros((B, N, h), device=dev), torch.zeros((B, N, h), device=dev))

    def train_step(raw, timed_idx=None):
        # main.py:306-358 for one batch with outer_T == truncated_length: scale_data, zero state, ONE window, Adam
        Qs, ps, As, zls, zus = scaling.scale_data(*raw)
        opt.zero_grad(set_to_none=True)
        loss, _ = model.train_window(TL, mi, me, Qs, ps, As, zls, zus, SIGMA, zero_state(), loss_scale=1.0 / TL, inplace=True,
                                     recompute_gates=True if args.recompute else None)
        if world > 1:
            if timed_idx is not None:
                ar_ev[timed_idx][0].record()
            allreduce_gradients(model, local_batch=B, comm=comm)   # ONE NCCL all-reduce of the flat gradient buffer per window
            if timed_idx is not None:
                ar_ev[timed_idx][1].record()
        opt.step()
        return loss

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    raw = (Q, p, A0, zl, zu)
    for _ in range(warmup):
        loss = train_step(raw)
    barrier()
    graph = None
    if args.graph:
        # Static buffers in, gradients out: the ~6000 launches of a window become one graph launch (at 2 instances per GPU the
        # per-iteration kernels take 0.5 ms and their launches another 0.13 ms).  The weight re-pack is captured too, so a
        # replay always sees the parameters Adam just updated; `.grad` tensors are allocated during capture and rewritten by
        # every replay (so no zero_grad(set_to_none=True) between replays).
        static_in = [t.clone() for t in raw]
        static_loss = torch.zeros((), device=dev)
        opt.zero_grad(set_to_none=True)
        model.invalidate_packed()
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, stream=side):
            Qs, ps, As, zls, zus = scaling.scale_data(*static_in)
            ls, _ = model.train_window(TL, mi, me, Qs, ps, As, zls, zus, SIGMA, zero_state(), loss_scale=1.0 / TL, inplace=True,
                                       recompute_gates=True if args.recompute else False)
            static_loss.copy_(ls)
        torch.cuda.current_stream().wait_stream(side)

        def train_step(raw_, timed_idx=None):                                     # noqa: F811  (graph-replay form of the step)
            for d_, s_ in zip(static_in, raw_):
                if d_.data_ptr() != s_.data_ptr():
                    d_.copy_(s_, non_blocking=True)
            graph.replay()
            if world > 1:
                if timed_idx is not None:
                    ar_ev[timed_idx][0].record()
                allreduce_gradients(model, local_batch=B, comm=comm)
                if timed_idx is not None:
                    ar_ev[timed_idx][1].record()
            opt.step()
            return static_loss

        raw = tuple(static_in)
        for _ in range(2):
            loss = train_step(raw)
        barrier()
    sampler = ClockSampler(dev) if rank == 0 else None
    if sampler:
        sampler.start()
    ia._lib.check(L.iadmm_profile_begin(steps * TL * 2))
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    torch.cuda.profiler.start()
    e0.record()
    for i in range(steps):
        loss = train_step(raw, i)
    e1.record()
    barrier()
    torch.cuda.profiler.stop()
    ms = e0.elapsed_time(e1)
    kinds = 7
    pms, pcnt = (c_double * kinds)(), (c_int * kinds)()
    ia._lib.check(L.iadmm_profile_end_kinds(pms, pcnt, kinds))
    clocks = sampler.stop() if sampler else None
    ar_ms = sum(a.elapsed_time(b) for a, b in ar_ev) if world > 1 else 0.0
    if args.dump_outputs and rank == 0:
        # the window's loss, the gradients it left in .grad and the weights after the Adam step
        outs = {"loss": loss.reshape(-1)}
        for name, prm in model.named_parameters():
            outs[name], outs["grad_" + name] = prm, prm.grad
        dump_outputs(args.dump_outputs, outs)
    loss_v = float(loss)
    mem_gb = torch.cuda.max_memory_allocated() / 1e9

    # ---- e2e: the batch arrives from pinned host memory every step, the loss goes back to the host -----------------
    host_in = [t.cpu().pin_memory() for t in raw]
    dev_in = [torch.empty_like(t) for t in raw]
    host_loss = torch.empty((1,), dtype=torch.float32).pin_memory()

    def e2e_step():
        for d_, h_ in zip(dev_in, host_in):
            d_.copy_(h_, non_blocking=True)
        ls = train_step(tuple(dev_in))
        host_loss.copy_(ls.reshape(1), non_blocking=True)

    e2e_step()
    barrier()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(steps):
        e2e_step()
    t1.record()
    barrier()
    e2e_ms = t0.elapsed_time(t1)
    h2d = sum(t.numel() * t.element_size() for t in host_in)

    # weights must stay identical across ranks (same all-reduced gradient, same Adam state)
    chk = torch.stack([prm.detach().double().sum() for prm in model.parameters()]).sum()
    same = True
    times = torch.tensor([ms, e2e_ms, ar_ms], device=dev, dtype=torch.float64)
    if world > 1:
        lo, hi = chk.clone(), chk.clone()
        dist.all_reduce(lo, op=dist.ReduceOp.MIN); dist.all_reduce(hi, op=dist.ReduceOp.MAX)
        same = bool(lo == hi)
        dist.all_reduce(times, op=dist.ReduceOp.MAX)
    ms, e2e_ms, ar_ms = (float(v) for v in times)

    if rank == 0:
        hbm_gbs, tf_sus, tf_burst, peak_kind = measured_peaks()
        rows = B * N
        its = max(1, pcnt[4])
        gemm_ms = pms[4] / its
        gemm_flops = 16.0 * rows * h * h                      # H_bar = D U^T and U_bar = H^T D: 2 x (2 * rows * h * 4h)
        gemm_tflops = gemm_flops / (gemm_ms * 1e-3) / 1e12 if gemm_ms > 0 else 0.0
        line = {
            "metric": "training instances/sec (TBPTT window TL=%d, n=%d, m=%d)" % (TL, n, m),
            "value": world * B * steps / (ms * 1e-3), "unit": "instances/s", "n_gpus": world, "steps": steps, "warmup": warmup,
            "ms_per_step": ms / steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic",
            "config": {"workload": workload_name(args), "batch_per_gpu": B, "truncated_length": TL, "gate_mode": args.gate_mode,
                       "cache": "inputs larger than L2: saved states %.1f GB per window" % (2 * (TL + 1) * rows * h * 4 / 1e9),
                       "parallelism": "data parallel over %d GPU(s): one NCCL all-reduce of the flat gradient buffer (%d floats) per window (%s), "
                                      "then the reference's Adam on every rank" % (world, sum(p_.numel() for p_ in model.parameters()),
                                                                                    "iadmm_allreduce_grads of the C ABI" if comm is not None else "torch.distributed"),
                       "weights_identical_across_ranks": same, "loss": loss_v, "peak_mem_GB": mem_gb,
                       "gate_activations": "recomputed in the backward" if getattr(model, "last_window_flags", 0) & 1 else "kept over the window",
                       "launch": "one CUDA graph per step (scale_data + window)" if graph is not None else "eager (the library enqueues ~60 launches per iteration)"},
            "gpu_launches": steps * TL * 60,
            "allreduce": {"ms_per_step": ar_ms / steps, "share_of_step": ar_ms / ms if ms > 0 else 0.0,
                          "bytes": 4 * (sum(p_.numel() for p_ in model.parameters()) + 1)},
            "roofline": {"kernel": "tc_gemm_nt_kernel x2 (+ fp16 hi/lo operand splits)", "bound": "tensor", "achieved": gemm_tflops,
                         "peak": tf_sus, "unit": "TFLOP/s", "frac": gemm_tflops / tf_sus, "traffic": None,
                         "flops_per_launch": gemm_flops, "ms_per_launch": gemm_ms, "share_of_step": pms[4] / ms,
                         "peak_kind": "%s bf16_tflops_sustained" % peak_kind,
                         "note": "logical fp32 flops of the two gate-product adjoints per iteration (16*rows*h^2); each runs as 3 fp16 "
                                 "MMAs (hi/lo split of both operands)"},
            "phase_ms_per_iteration": {"fwd_gates": pms[3] / max(1, pcnt[3]), "bwd_gemms": gemm_ms,
                                       "kkt_fwd_and_adjoint": pms[5] / its, "bwd_cell_and_small_adjoints": pms[6] / max(1, pcnt[6])},
            "clocks": clocks,
            "e2e": {"value": world * B * steps / (e2e_ms * 1e-3), "unit": "instances/s", "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": 4, "ms_per_step": e2e_ms / steps},
        }
        emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    a = parse_args()
    quiet_stdout()        # libraries (NCCL banner, MAGMA's batched-solve warning at n=5000) print to stdout from C: keep it to ONE JSON line
    if a.impl != "ours":
        run_reference(a)
    elif a.workload == "train":
        run_train(a)
    else:
        run_ours(a)
