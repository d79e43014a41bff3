"""The reference's LITERAL per-iteration loop (main.py:874-887: `x, y, z, xv, H, C, A_tild, b_tild, rho_vec = model(t, ...)`
with the returned state fed back) through the drop-in `LSTM.forward`.  From the second call on `forward` resumes from the
operand planes the previous call left in the workspace (IADMM_F_RESUME of include/iadmm.h) instead of converting H and C on
every call; these tests hold that path bit for bit to the fused `LSTM.solve` of the same iterations, and check every way out
of it (edited state, another batch in between, a `solve` in between), the dense A_tild / b_tild / rho_vec of every call against
the oracle's restatement of models/lstm.py:61-69, and the `materialize_kkt = "shared"` buffer against the fresh one.
"""
import pytest
import torch

from oracle import iadmm_oracle as orc

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
SIGMA = 6e-6
STATE = ("x", "y", "z", "xv", "H", "C")


def make(h, K, mode="tc_f16f8", seed=5):
    import iadmm_b200 as ia
    prm = orc.lstm_parameters(h, K, seed=seed)
    model = ia.LSTM(None, 2, h, K, DEV, gate_mode=mode)
    with torch.no_grad():
        for k, v in prm.items():
            getattr(model, k).copy_(v.to(DEV))
    return model.eval(), prm


def scaled_qp(B, n, mi, me, seed):
    import iadmm_b200 as ia
    qp = orc.qp_instances(B, n, mi, me, seed=seed)
    sc = ia.Scaling(n, mi + me, 10, DEV)
    return sc.scale_data(*(qp[k].to(DEV) for k in ("Q", "p", "A0", "zl", "zu")))


def zero_state(B, n, m, h):
    N = n + m
    return [torch.zeros((B, n, 1), device=DEV), torch.zeros((B, m, 1), device=DEV), torch.zeros((B, m, 1), device=DEV),
            torch.zeros((B, N, 1), device=DEV), torch.zeros((B, N, h), device=DEV), torch.zeros((B, N, h), device=DEV)]


def poison_allocator(nbytes):
    """Leave NaN-filled free blocks in the caching allocator so an output that is not fully written shows."""
    junk = [torch.full((nbytes // 4,), float("nan"), device=DEV) for _ in range(3)]
    del junk


def call(model, t, mi, me, st, data):
    Q, p, A0, zl, zu = data
    return model(t, mi, me, st[0], st[1], st[2], st[3], SIGMA, st[4], st[5], Q=Q, p=p, A0=A0, lb=None, ub=None, zl=zl, zu=zu)


# hidden_dim 400: the 8-warp production kernel <2,2,4> (hidden_dim > 384); 320: the 16-warp kernel <2,2,9>; 200: its padded last
# operand group (hidden_dim % 16 == 8); 64 with n + m > 256: the 16-warp kernel on the streaming path.  tc_f16f8u drops the
# H-rounding correction on the row-interleaved path, which both the single steps and the fused solve take (8-warp kernel <2,2,4>)
@pytest.mark.parametrize("mode", ["tc_f16f8", "tc_f16f8u"])
@pytest.mark.parametrize("h,n,mi,me", [(400, 70, 13, 29), (320, 48, 16, 16), (200, 64, 32, 32), (64, 200, 60, 60)])
def test_forward_loop_equals_fused_solve(h, n, mi, me, mode):
    B, K, m = 3, 6, mi + me
    model, prm = make(h, K, mode)
    data = scaled_qp(B, n, mi, me, seed=31)
    with torch.no_grad():
        fused = model.solve(K, mi, me, *data, SIGMA, traces=False)
        poison_allocator(B * (n + m) * h * 4)
        st = zero_state(B, n, m, h)
        for t in range(K):
            before = [v.clone() for v in st]
            out = call(model, t, mi, me, st, data)
            for a, b in zip(before, st):                      # pure-functional like the reference: inputs untouched
                assert torch.equal(a, b)
            # the tuple of models/lstm.py:61-69 for the iterate BEFORE the update, against the oracle's restatement
            rho_vec, _ = orc.penalty_schedule(prm, t, mi, me, B)
            Kmat, rhs = orc.kkt_system(data[0].cpu(), data[1].cpu(), data[2].cpu(), st[0].cpu(), st[1].cpu(), st[2].cpu(),
                                       rho_vec, SIGMA)
            assert torch.allclose(out[8].cpu(), rho_vec, rtol=1e-6, atol=0)
            A_ref = Kmat.clone()
            idx = torch.arange(n, n + m)
            A_ref[:, idx, idx] = -(1 / out[8][:, :, 0].cpu())      # (rho_vec itself is held to 1e-6 above)
            assert torch.equal(out[6].cpu(), A_ref)
            assert float(torch.linalg.vector_norm(out[7].cpu() - rhs) / torch.linalg.vector_norm(rhs)) < 1e-5
            st = list(out[:6])
        torch.cuda.synchronize()
    assert model.resumed_calls == K - 1
    for k, a in zip(STATE, st):
        assert torch.equal(a, getattr(fused, k)), k


def test_every_way_out_of_the_resumed_path():
    """An in-place edit of H, a second batch driven alternately through the same model, and a fused `solve` in between all
    fall back to the converting path and give the results of an undisturbed run."""
    h, n, mi, me, B = 320, 48, 16, 16, 2
    m = mi + me
    model, _ = make(h, 8)
    dA, dB = scaled_qp(B, n, mi, me, seed=3), scaled_qp(B, n, mi, me, seed=4)
    with torch.no_grad():
        # (1) edited state: 2 iterations, H *= 0.5 in place, 2 more == solve(2) from the same edited state
        st = zero_state(B, n, m, h)
        for t in range(2):
            st = list(call(model, t, mi, me, st, dA)[:6])
        st[4].mul_(0.5)
        edited = [v.clone() for v in st]
        for t in range(2, 4):
            st = list(call(model, t, mi, me, st, dA)[:6])
        assert model.resumed_calls == 2          # calls 1 and 3; call 2 saw the edit
        ref = model.solve(2, mi, me, *dA, SIGMA, state=edited, t0=2, traces=False)
        for k, a in zip(STATE, st):
            assert torch.equal(a, getattr(ref, k)), k
        # (2) two batches alternately, and (3) a solve of something else between two calls
        refA = model.solve(4, mi, me, *dA, SIGMA, traces=False)
        refB = model.solve(4, mi, me, *dB, SIGMA, traces=False)
        sA, sB = zero_state(B, n, m, h), zero_state(B, n, m, h)
        for t in range(4):
            sA = list(call(model, t, mi, me, sA, dA)[:6])
            sB = list(call(model, t, mi, me, sB, dB)[:6])
            if t == 1:
                model.solve(3, mi, me, *dB, SIGMA, traces=False)
        assert model.resumed_calls == 2          # nothing resumes while two batches alternate
        for k, a, b in zip(STATE, sA, sB):
            assert torch.equal(a, getattr(refA, k)), k
            assert torch.equal(b, getattr(refB, k)), k
        torch.cuda.synchronize()


def test_shared_kkt_buffer_equals_fresh_one():
    h, n, mi, me, B, K = 64, 70, 13, 29, 2, 4
    m = mi + me
    model, _ = make(h, K)
    data = scaled_qp(B, n, mi, me, seed=9)
    with torch.no_grad():
        st, fresh = zero_state(B, n, m, h), []
        for t in range(K):
            out = call(model, t, mi, me, st, data)
            fresh.append(out[6].clone())
            st = list(out[:6])
        model.materialize_kkt = "shared"
        st, ptrs = zero_state(B, n, m, h), set()
        for t in range(K):
            out = call(model, t, mi, me, st, data)
            assert torch.equal(out[6], fresh[t]), t
            ptrs.add(out[6].data_ptr())
            st = list(out[:6])
        assert len(ptrs) == 1
        # other data: a new buffer, the right matrix
        other = scaled_qp(B, n, mi, me, seed=10)
        model.materialize_kkt = True
        want = call(model, 0, mi, me, zero_state(B, n, m, h), other)[6]
        model.materialize_kkt = "shared"
        got = call(model, 0, mi, me, zero_state(B, n, m, h), other)[6]
        assert torch.equal(got, want)
        model.materialize_kkt = False
        assert call(model, 0, mi, me, zero_state(B, n, m, h), other)[6] is None
        torch.cuda.synchronize()


# ---- dataset files written by the reference's own generate_data.py, with the counts main.py derives from them ------------
FAMILY_DIRS = {"QP": "QP_12_5_4", "QP_RHS": "QP_RHS_12_5_4", "Random_QP": "Random_QP_10_6", "Equality_QP": "Equality_QP_10_4",
               "SVM": "SVM_10_4"}


@pytest.mark.parametrize("mode", ["simt_fp32", "tc_f16f8"])
@pytest.mark.parametrize("family", list(FAMILY_DIRS))
def test_dataset_files_through_the_dropin_modules(family, mode):
    """load_batch (pinned staging -> device) + Scaling + the literal loop and the fused solve, called with main.py's
    (num_ineq, num_eq) -- for Random_QP (12 + 0 vs 6 rows of A0) and SVM (4 + 0 vs 14 rows) they do not add up to the rows of
    A0, and models/lstm.py:61-62 only slices with them -- against the reference's outputs on the same files
    (tests/golden/dataset_<family>.npz, make_dataset_golden.py)."""
    import os
    import iadmm_b200 as ia
    from iadmm_b200 import data
    from helpers import load_golden, golden_params, rel_err
    g = load_golden(f"dataset_{family}")
    B, n, num_ineq, num_eq, m, h, K, ites = (int(v) for v in g["meta"])
    prm = golden_params(g)
    d = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "datasets", FAMILY_DIRS[family])
    batch, sizes = data.load_batch(d, family, [0, 1, 2], DEV)
    assert (sizes["num_ineq"], sizes["num_eq"]) == (num_ineq, num_eq)
    model = ia.LSTM(None, 2, h, K, DEV, gate_mode=mode).eval()
    with torch.no_grad():
        for k, v in prm.items():
            getattr(model, k).copy_(v.to(DEV))
    sc = ia.Scaling(n, m, ites, DEV)
    scaled = sc.scale_data(*(batch[k] for k in ("Q", "p", "A0", "zl", "zu")))
    tol = {"simt_fp32": 2e-5, "tc_f16f8": 5e-5}[mode]
    with torch.no_grad():
        st, pri, dual = zero_state(B, n, m, h), [], []
        for t in range(K):
            out = call(model, t, num_ineq, num_eq, st, scaled)
            st = list(out[:6])
            pr, du, _ = ia.primal_dual_loss(st[0], st[1], st[2], scaled[0], scaled[1], scaled[2])
            pri.append(pr.reshape(B)); dual.append(du.reshape(B))
        fused = model.solve(K, num_ineq, num_eq, *scaled, float(g["sigma"]))
        torch.cuda.synchronize()
    for k, v in zip(STATE, st):
        assert rel_err(v, g["out_" + k]) < tol, (k, rel_err(v, g["out_" + k]))
        assert rel_err(getattr(fused, k), g["out_" + k]) < tol, ("fused", k)
    assert rel_err(torch.stack(pri), g["out_pri"]) < tol and rel_err(torch.stack(dual), g["out_dual"]) < tol
    assert rel_err(fused.pri, g["out_pri"]) < tol and rel_err(fused.dual, g["out_dual"]) < tol
    assert rel_err(out[8], g["out_rho_vec"]) < 1e-6
    assert rel_err(out[6], g["out_K"]) < 1e-5 and rel_err(out[7], g["out_rhs"]) < 1e-4


def test_forward_under_inference_mode_takes_the_converting_path():
    """Inference tensors have no version counter, so an in-place edit between two calls could not be noticed: `forward` then
    never resumes, and still equals the fused solve."""
    h, n, mi, me, B, K = 320, 48, 16, 16, 2, 3
    m = mi + me
    model, _ = make(h, K)
    data = scaled_qp(B, n, mi, me, seed=12)
    with torch.no_grad():
        fused = model.solve(K, mi, me, *data, SIGMA, traces=False)
    import iadmm_b200 as ia
    with torch.inference_mode():
        data_i = scaled_qp(B, n, mi, me, seed=12)                 # Scaling, too, on inference tensors
        st = zero_state(B, n, m, h)
        model.materialize_kkt = "shared"
        for t in range(K):
            out = call(model, t, mi, me, st, data_i)
            st = list(out[:6])
            pri, dual, tot = ia.primal_dual_loss(st[0], st[1], st[2], data_i[0], data_i[1], data_i[2])
        fused_i = model.solve(K, mi, me, *data_i, SIGMA)
        torch.cuda.synchronize()
    assert model.resumed_calls == 0
    for a, b in zip(data, data_i):
        assert torch.equal(a, b)
    for k, a in zip(STATE, st):
        assert torch.equal(a, getattr(fused, k)), k
        assert torch.equal(getattr(fused_i, k), getattr(fused, k)), k
    assert torch.allclose(pri.reshape(-1), fused_i.pri[-1], rtol=1e-6) and torch.allclose(dual.reshape(-1), fused_i.dual[-1], rtol=1e-6)
