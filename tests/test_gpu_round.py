"""-m gpu: TT rounding of TT input and truncated_svd through the drop-in API, against golden vectors."""
import os

import numpy as np
import pytest
import torch

from gpu_util import ranks_of, relerr64
from oracle import cases

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), "golden")


@pytest.mark.parametrize("name", list(cases.ROUND_CASES))
def test_round_tt_matches_reference(name):
    import tntorch_b200 as tnb

    g = np.load(os.path.join(GOLD, "round_tt.npz"))
    spec = cases.ROUND_CASES[name]
    cores = cases.make_tt(spec)
    dense = cases.tt_full(cores)
    t = tnb.Tensor([torch.as_tensor(c).cuda() for c in cores])
    kw = {k: spec[k] for k in ("eps", "rmax") if k in spec}
    t2 = tnb.round_tt(t, **kw)
    assert ranks_of(t2.cores) == list(g[f"{name}/svd/ranks"])
    tol = 1e-5
    assert abs(relerr64(dense, t2.cores) - float(g[f"{name}/svd/relerr"])) <= tol
    # round_tt(t) must not touch t (round.py:7-19 clones first)
    assert ranks_of(t.cores) == [1] + [c.shape[2] for c in cores]


@pytest.mark.parametrize("name", list(cases.TSVD_CASES))
@pytest.mark.parametrize("lo", [True, False])
def test_truncated_svd_matches_reference(name, lo):
    import tntorch_b200 as tnb

    g = np.load(os.path.join(GOLD, "truncated_svd.npz"))
    spec = cases.TSVD_CASES[name]
    M = cases.make_matrix(spec)
    kw = {k: spec[k] for k in ("eps", "delta", "rmax") if k in spec}
    left, right = tnb.truncated_svd(torch.as_tensor(M).cuda(), left_ortho=lo, **kw)
    key = f"{name}/svd/{'L' if lo else 'R'}"
    assert left.shape[1] == int(g[key + "/rank"])
    prod = (left.double() @ right.double()).cpu().numpy()
    ref = g[f"{name}/svd/left"].astype(np.float64) @ g[f"{name}/svd/right"].astype(np.float64)
    tol = 1e-4 if M.dtype == np.float32 else 1e-7
    np.testing.assert_allclose(prod, ref, atol=tol * max(1.0, np.abs(M).max()))
    if not spec.get("zero"):
        r = left.shape[1]
        eye = torch.eye(r, device="cuda", dtype=left.dtype)
        orth = (left.T @ left - eye) if lo else (right @ right.T - eye)
        assert orth.abs().max().item() < (1e-4 if M.dtype == np.float32 else 1e-8)


def test_orthogonalization_preserves_tensor():
    """tests/test_round.py:7-18: left_/right_/orthogonalize leave the tensor unchanged (<= 1e-7) and produce
    orthonormal unfoldings."""
    import tntorch_b200 as tnb

    cores = cases.random_tt((6, 5, 7, 4, 6), 5, seed=77)
    gt = cases.tt_full(cores)
    t = tnb.Tensor([torch.as_tensor(c).cuda() for c in cores])
    R = t.left_orthogonalize(1)
    assert R.shape[0] == t.cores[1].shape[-1]
    assert relerr64(gt, t.cores) <= 1e-7
    L = t.right_orthogonalize(3)
    assert L.shape[1] == t.cores[3].shape[0]
    assert relerr64(gt, t.cores) <= 1e-7
    t.orthogonalize(2)
    assert relerr64(gt, t.cores) <= 1e-7
    for k in (0, 1):
        M = t.cores[k].reshape(-1, t.cores[k].shape[-1])
        assert (M.T @ M - torch.eye(M.shape[1], device="cuda", dtype=M.dtype)).abs().max().item() < 1e-10
    for k in (3, 4):
        M = t.cores[k].reshape(t.cores[k].shape[0], -1)
        assert (M @ M.T - torch.eye(M.shape[0], device="cuda", dtype=M.dtype)).abs().max().item() < 1e-10
    with pytest.raises(AssertionError):
        t.left_orthogonalize(4)


def test_cp_cores_round_trip_through_round_tt():
    """reference tests/test_tensor.py:361-392: a CP-format tensor (plain and batched) survives round_tt(eps=1e-8); the
    CP factors are turned into TT cores with diagonal slices first (tensor.py:1717-1762)."""
    import tntorch_b200 as tnb

    rng = np.random.default_rng(5)
    fac = [torch.as_tensor(rng.standard_normal((s, 3))).cuda() for s in (10, 5, 6)]
    a = tnb.Tensor([f.clone() for f in fac])
    b = a.torch()
    assert torch.allclose(b, torch.einsum("ar,br,cr->abc", *fac))
    a.round_tt(eps=1e-8)
    assert all(c.dim() == 3 for c in a.cores) and max(a.ranks_tt) <= 3
    assert float(torch.linalg.vector_norm(b - a.torch())) < 1e-8
    facb = [torch.as_tensor(rng.standard_normal((4, s, 3))).cuda() for s in (10, 5, 6)]
    ab = tnb.Tensor([f.clone() for f in facb], batch=True)
    bb = ab.torch()
    ab.round_tt(eps=1e-8)
    assert float(torch.linalg.vector_norm(bb - ab.torch())) < 1e-8
    # orthogonalize() on CP cores (tensor.py:1898: _cp_to_tt first)
    c = tnb.Tensor([f.clone() for f in fac])
    c.orthogonalize(1)
    assert float(torch.linalg.vector_norm(b - c.torch())) < 1e-8 * float(torch.linalg.vector_norm(b))


def test_factor_orthogonalize_and_batched_orthogonalisation():
    """tensor.py:1771-1798 (Tucker factor = Q R, R pushed into the core) and the batch branches of
    left_/right_orthogonalize (tensor.py:1818-1878): the tensor is unchanged, factors / unfoldings orthonormal."""
    import tntorch_b200 as tnb

    rng = np.random.default_rng(6)
    cores = [torch.as_tensor(c).cuda() for c in cases.random_tt((4, 5, 3, 6), 3, seed=78)]
    Us = [torch.as_tensor(rng.standard_normal((I, c.shape[1]))).cuda() for I, c in zip((7, 9, 5, 8), cores)]
    t = tnb.Tensor([c.clone() for c in cores], Us=[u.clone() for u in Us])
    gt = t.torch()
    assert list(t.shape) == [7, 9, 5, 8]
    t.factor_orthogonalize(1)
    U = t.Us[1]
    assert (U.T @ U - torch.eye(U.shape[1], device="cuda", dtype=U.dtype)).abs().max().item() < 1e-10
    assert float(torch.linalg.vector_norm(gt - t.torch())) < 1e-10 * float(torch.linalg.vector_norm(gt))
    t.orthogonalize(2)  # pushes the factors of cores 0, 1, 3 as well
    assert float(torch.linalg.vector_norm(gt - t.torch())) < 1e-9 * float(torch.linalg.vector_norm(gt))
    t.round_tt(eps=1e-10)
    assert float(torch.linalg.vector_norm(gt - t.torch())) < 1e-8 * float(torch.linalg.vector_norm(gt))
    # batched TT
    B = 3
    bc = [torch.as_tensor(rng.standard_normal((B,) + c.shape)).cuda() for c in cores]
    tb = tnb.Tensor([c.clone() for c in bc], batch=True)
    gtb = tb.torch()
    R = tb.left_orthogonalize(0)
    assert R.shape == (B, 3, 3)
    L = tb.right_orthogonalize(3)
    assert L.shape == (B, 3, 3)
    tb.orthogonalize(1)
    assert float(torch.linalg.vector_norm(gtb - tb.torch())) < 1e-9 * float(torch.linalg.vector_norm(gtb))
    M = tb.cores[0].reshape(B, -1, tb.cores[0].shape[-1])
    assert (M.transpose(1, 2) @ M - torch.eye(M.shape[2], device="cuda", dtype=M.dtype)).abs().max().item() < 1e-10
