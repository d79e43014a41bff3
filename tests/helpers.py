"""Shared helpers for the test-suite (fixture loading, error metrics)."""
import os

import numpy as np
import torch

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
GATES = ("i", "f", "o", "u")


def load_golden(name):
    z = np.load(os.path.join(GOLDEN, name + ".npz"), allow_pickle=False)
    return {k: z[k] for k in z.files}


def t(a, dtype=torch.float32, device="cpu"):
    return torch.as_tensor(np.asarray(a)).to(dtype).to(device).contiguous()


def golden_params(blob, dtype=torch.float32, device="cpu"):
    return {k[4:]: t(v, dtype, device) for k, v in blob.items() if k.startswith("prm_")}


def golden_qp(blob, dtype=torch.float32, device="cpu"):
    return {k[3:]: t(v, dtype, device) for k, v in blob.items() if k.startswith("qp_")}


def rel_err(a, b):
    """||a-b||_2 / ||b||_2 over the whole tensor (per-quantity relative error of north_star)."""
    a = torch.as_tensor(np.asarray(a)).double().cpu() if not torch.is_tensor(a) else a.double().cpu()
    b = torch.as_tensor(np.asarray(b)).double().cpu() if not torch.is_tensor(b) else b.double().cpu()
    fin = torch.isfinite(b)
    assert torch.equal(torch.isfinite(a), fin), "non-finite pattern differs"
    if not bool(fin.all()):
        assert torch.equal(a[~fin], b[~fin])
    a, b = a[fin], b[fin]
    den = float(torch.linalg.vector_norm(b))
    num = float(torch.linalg.vector_norm(a - b))
    return num / den if den > 0 else num


def assert_parity(name, ours, ref32, ref64=None, bar=1e-4, c=4.0):
    """north_star's statement: rel <= 1e-4 against the reference's fp32 result.  Where the reference's own fp32 result is
    not determined that well -- its deviation from the same computation in float64, e32 = err(ref32, ref64), is itself of
    the order of the bar (early iterates of y = y + rho (z~ - z): |y| small, rho * ulp(z) of absolute rounding noise) --
    the comparable statement is "as close to the exact result as the reference is": err(ours, ref64) <= c * e32.
    Returns (err vs ref32, which assertion held)."""
    e = rel_err(ours, ref32)
    if e <= bar:
        return e, "bar"
    assert ref64 is not None, (name, e, "above the bar and no float64 run to measure the reference's own noise floor")
    e32 = rel_err(ref32, ref64)
    e64 = rel_err(ours, ref64)
    assert e64 <= c * e32, (name, f"ours-vs-fp64 {e64:.2e} > {c} x reference-fp32-vs-fp64 {e32:.2e} (ours-vs-fp32 {e:.2e})")
    return e, "noise-floor"


def oracle_pair(prm, K, mi, me, qp, h, scaling_ites=10, sigma=6e-6, form="block"):
    """The CPU oracle's solve in float32 (the reference's arithmetic) and float64 (the tie-breaker) on the same inputs;
    Ruiz-scaled when `scaling_ites`.  Returns (ref32, ref64, scaled fp32 data, fp32 scaling)."""
    from oracle import iadmm_oracle as orc
    out = []
    for dt in (torch.float32, torch.float64):
        d = {k: qp[k].to(dt) for k in ("Q", "p", "A0", "zl", "zu")}
        sc = None
        if scaling_ites:
            Qs, ps, As, zls, zus, sc = orc.ruiz_equilibrate(d["Q"], d["p"], d["A0"], d["zl"], d["zu"], scaling_ites)
        else:
            Qs, ps, As, zls, zus = (d[k] for k in ("Q", "p", "A0", "zl", "zu"))
        r = orc.solve({k: v.to(dt) for k, v in prm.items()}, K, mi, me, Qs, ps, As, zls, zus, sigma, h, form=form)
        out.append((r, (Qs, ps, As, zls, zus), sc))
    return out[0][0], out[1][0], out[0][1], out[0][2]


# K=100 at the headline shape against the reference's fp32 computation on the GPU (test_gpu_production_shapes and
# tests/golden/make_k100_config2_golden.py): inputs from the oracle's generators, seed 43
K100_SHAPE = dict(B=16, n=1000, mi=500, me=500, h=800, K=100, seed=43)
K100_ROWS = (137, 712)                  # sampled rows of the scaled Q and A0: one inequality, one equality row


def k100_inputs(device):
    from oracle import iadmm_oracle as orc
    s = K100_SHAPE
    qp = orc.qp_instances(s["B"], s["n"], s["mi"], s["me"], seed=s["seed"])
    return ({k: qp[k].to(device) for k in ("Q", "p", "A0", "zl", "zu")},
            orc.lstm_parameters(s["h"], s["K"], seed=s["seed"]))


def k100_record(data, d, e, c, x, y, z, pri, dual):
    """What the K=100 comparison looks at, as float32 CPU tensors: the Ruiz diagonals d [B,n], e [B,m], c [B], the scaled
    p, zl, zu and rows K100_ROWS of the scaled Q and A0, the final x, y, z and the [K,B] residual traces."""
    Q, p, A0, zl, zu = data
    rows = list(K100_ROWS)
    rec = dict(d=d, e=e, c=c.reshape(-1), p=p, zl=zl, zu=zu, Q_rows=Q[:, rows], A0_rows=A0[:, rows],
               x=x, y=y, z=z, pri=pri, dual=dual)
    return {k: v.detach().float().cpu().contiguous() for k, v in rec.items()}


def k100_reference_record(device):
    """The reference's computation of the K=100 case in stock PyTorch fp32 on `device` (TF32 off): Ruiz scaling
    (methods/scaling.py), K calls of the cell with the dense KKT matrix (models/lstm.py:47-96), primal_dual_loss after each
    (utils.py:68-71).  Runs the reference's own modules when baseline/_ref holds them, else the oracle's restatement of them
    (form="dense"; test_oracle_golden pins it to outputs of the reference's modules).  Returns (k100_record, source)."""
    from baseline import ref_arm
    from oracle import iadmm_oracle as orc
    torch.backends.cuda.matmul.allow_tf32 = False
    s = K100_SHAPE
    qp, prm = k100_inputs(device)
    raw = [qp[k] for k in ("Q", "p", "A0", "zl", "zu")]
    if ref_arm.available():
        r = ref_arm.solve(ref_arm.make_model(prm, s["h"], s["K"], device), s["K"], s["mi"], s["me"], *raw, ref_arm.SIGMA, 10)
        sc = r["scaling"]
        d, e = (torch.diagonal(M, dim1=1, dim2=2) for M in (sc.D, sc.E))
        rec = k100_record(r["data"], d, e, sc.c, *(r[k] for k in ("x", "y", "z", "pri", "dual")))
        source = "the reference's modules (baseline/_ref)"
    else:
        default = torch.get_default_device()
        torch.set_default_device(device)          # the oracle allocates its work tensors without naming a device
        try:
            Qs, ps, As, zls, zus, sc = orc.ruiz_equilibrate(*raw, 10)
            r = orc.solve({k: v.to(device) for k, v in prm.items()}, s["K"], s["mi"], s["me"], Qs, ps, As, zls, zus, 6e-6, s["h"],
                          form="dense")
        finally:
            torch.set_default_device(default)
        rec = k100_record((Qs, ps, As, zls, zus), sc.d, sc.e, sc.c, r.x, r.y, r.z, r.pri, r.dual)
        source = "the oracle's restatement of the reference's modules (oracle/iadmm_oracle.py, form='dense')"
    where = torch.cuda.get_device_name(device) if torch.device(device).type == "cuda" else "CPU"
    return rec, f"{source} on {where}, torch {torch.__version__}, fp32, TF32 off"
