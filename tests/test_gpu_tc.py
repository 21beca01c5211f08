"""-m gpu: the tcgen05/TMA Gram kernel against an fp64 reference (TF32 inputs, fp32 accumulate)."""
import pytest
import torch

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("shape", [(8192, 128), (10000, 64), (4096, 256), (5000, 320), (3001, 100), (2048, 2048), (70000, 32),
                                   (16384, 512), (3000, 640), (5000, 1000)])
def test_gram_tc_matches_fp64(shape):
    from tntorch_b200 import ops

    if not ops.has_tensorcore_path():
        pytest.fail("tensor-core path unavailable on this device (needs sm_100)")
    g = torch.Generator().manual_seed(7)
    A = torch.randn(*shape, generator=g, dtype=torch.float32).cuda()
    G = ops.gram(A, tensorcore=True)
    torch.cuda.synchronize()
    ref = A.double().T @ A.double()
    # TF32 truncation of both operands: relative 2^-10 per product, random sign -> ~1e-3/sqrt(K) of the diagonal scale
    scale = ref.diagonal().max().item()
    err = (G - ref).abs().max().item() / scale
    assert err < 2e-3, err
    assert torch.equal(G, G.T)
    # the mean truncation bias shrinks the diagonal by < 2^-10
    d = (G.diagonal() / ref.diagonal())
    assert d.min().item() > 1 - 2e-3 and d.max().item() <= 1 + 1e-6


def test_gram_tc_structured_exact():
    """Inputs exactly representable in TF32 must give the exact Gram (catches layout/descriptor errors
    that random data would hide behind the tolerance)."""
    from tntorch_b200 import ops

    for rows, n in ((4096 + 37, 384), (2048 + 5, 1024), (1000, 768)):
        _exact_case(rows, n)


def _exact_case(rows, n):
    from tntorch_b200 import ops

    i = torch.arange(rows, dtype=torch.float64)[:, None]
    j = torch.arange(n, dtype=torch.float64)[None, :]
    A = (((i * 7 + j * 13) % 17) - 8).float().cuda()  # small integers
    G = ops.gram(A, tensorcore=True)
    ref = A.double().T @ A.double()
    assert torch.equal(G, ref)


@pytest.mark.parametrize("shape", [(2048, 2048, 64), (1000, 300, 36), (4096, 128, 256), (777, 2048, 128)])
def test_atb_tc_matches_fp64(shape):
    """General A^T B on the tensor cores (the subspace-iteration filter product) incl. the fused epilogue."""
    from tntorch_b200 import ops

    K, m, n = shape
    g = torch.Generator().manual_seed(11)
    A = torch.randn(K, m, generator=g).cuda()
    B = torch.randn(K, n, generator=g).cuda()
    D = torch.randn(m, n, generator=g).cuda()
    C = ops.atb_tensorcore(A, B, alpha=0.5, D=D, beta=-2.0)
    ref = 0.5 * (A.double().T @ B.double()) - 2.0 * D.double()
    err = (C.double() - ref).abs().max().item() / (A.double().T @ B.double()).abs().max().item()
    assert err < 3e-3, err
    # exact on TF32-representable integers
    Ai = torch.randint(-8, 9, (K, m), generator=g).float().cuda()
    Bi = torch.randint(-8, 9, (K, n), generator=g).float().cuda()
    Ci = ops.atb_tensorcore(Ai, Bi)
    assert torch.equal(Ci.double(), Ai.double().T @ Bi.double())


@pytest.mark.parametrize("shape", [(16384, 64, 32), (20000, 2048, 32), (4096 + 77, 96, 17), (70000, 64, 64), (1000, 32, 8),
                                   # V resident beyond 32 KB: stages handed back by the split warps (CP-ALS projections)
                                   (300000 + 5, 256, 50), (40000, 128, 64), (50000, 512, 32), (33000, 256, 64)])
def test_project_tc_fp32_accuracy(shape):
    """3xTF32 projection on the tensor cores keeps fp32 accuracy (a 1xTF32 product would be ~2^-11)."""
    from tntorch_b200 import ops

    rows, n, r = shape
    g = torch.Generator().manual_seed(5)
    A = torch.randn(rows, n, generator=g).cuda()
    V = torch.randn(n, r, generator=g).cuda()
    C = ops.project(A, V, tensorcore=True)
    ref = A.double() @ V.double()
    err = (C.double() - ref).abs().max().item() / ref.abs().max().item()
    assert err < 4e-6, err  # truncating TMEM accumulation is bounded by slabs of 256 columns
    Cf = ops.project(A, V)  # FFMA kernel for comparison
    errf = (Cf.double() - ref).abs().max().item() / ref.abs().max().item()
    assert err < 20 * max(errf, 1e-7)


@pytest.mark.parametrize("n,b,steps", [(256, 32, 3), (512, 64, 5), (1024, 64, 17), (2048, 64, 40), (1536, 40, 7)])
@pytest.mark.parametrize("dsmem", [True, False])
def test_resident_chebyshev_filter(n, b, steps, dsmem, monkeypatch):
    """cheb_filter.cuh: the whole three-term recurrence in one cooperative kernel vs fp64 torch; partial tiles
    reduced through distributed shared memory (clusters of 8) or through L2 (forced here for every size)."""
    from tntorch_b200 import ops

    if not dsmem:
        monkeypatch.setenv("TNB_FILTER_NO_DSMEM", "1")

    gen = torch.Generator().manual_seed(n + b)
    A = torch.randn(n, n, generator=gen, dtype=torch.float64)
    G = (A @ A.T / n).cuda()
    Y0 = torch.randn(n, b, generator=gen, dtype=torch.float64).cuda()
    lam = float(torch.linalg.matrix_norm(G, 2))
    # a damped recurrence (|a lam| + |bc| + |g| < 1.5) so that 40 steps stay O(1)
    a = [0.9 / lam] * steps
    bc = [-0.3] * steps
    g = [0.0] + [-0.25] * (steps - 1)
    out = ops.cheb_filter(G.float(), Y0.float(), a, bc, g)
    prev, cur = None, Y0
    for s in range(steps):
        nxt = a[s] * (G @ cur) + bc[s] * cur + (g[s] * prev if prev is not None else 0)
        prev, cur = cur, nxt
    err = float((out.double() - cur).norm() / cur.norm())
    assert err < 1e-3 * max(steps, 5), err  # TF32 operand truncation accumulates over the steps


def test_sweep_uses_resident_filter():
    from oracle import cases
    from tntorch_b200 import ops

    spec = cases.TTSVD_CASES["randn64x4_r32_f32"]
    X = torch.as_tensor(cases.make_dense(spec)).cuda()
    _, info = ops.ttsvd(X, rmax=spec["ranks_tt"], return_info=True)
    assert info["fused_filters"] >= 1, info


@pytest.mark.parametrize("name", ["twin32x5_r32_f32", "randn64x4_r32_f32"])
def test_concurrent_flag_same_result(name):
    """TNB_FLAG_CONCURRENT only changes scheduling (whole-GPU kernels chained across streams and sized to leave
    the reserved SMs free, no resident filter kernel): ranks and error must match the golden vectors just the same."""
    import os

    import numpy as np
    from gpu_util import ranks_of, relerr64
    from oracle import cases
    from tntorch_b200 import ops

    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "ttsvd.npz"))
    spec = cases.TTSVD_CASES[name]
    X = cases.make_dense(spec)
    cores, info = ops.ttsvd(torch.as_tensor(X).cuda(), rmax=spec["ranks_tt"], return_info=True, concurrent=True)
    alg = "svd" if f"{name}/svd/relerr" in g.files else "eig"
    assert ranks_of(cores) == list(g[f"{name}/{alg}/ranks"])
    assert abs(relerr64(X, cores) - float(g[f"{name}/{alg}/relerr"])) <= 1e-5
    assert info["fused_filters"] == 0 or info["speculative"] == 1  # the single-synchronisation sweep always uses the resident filter


def test_concurrent_threads_match_golden():
    """Three decompositions in flight on three streams / host threads with TNB_FLAG_CONCURRENT (the bench's
    schedule: event-chained whole-GPU kernels, reserved SMs): every one must still match the golden vectors."""
    import os
    from concurrent.futures import ThreadPoolExecutor

    import numpy as np
    from gpu_util import ranks_of, relerr64
    from oracle import cases
    from tntorch_b200 import ops

    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "ttsvd.npz"))
    names = ["twin32x5_r32_f32", "randn64x4_r32_f32", "randn32x5_r32_f32"]
    Xs = [cases.make_dense(cases.TTSVD_CASES[n]) for n in names]
    Xd = [torch.as_tensor(x).cuda() for x in Xs]
    streams = [torch.cuda.Stream() for _ in names]
    ops.set_reserved_sms(4)
    try:
        def run(i):
            torch.cuda.set_device(0)
            out = None
            with torch.cuda.stream(streams[i]):
                for _ in range(3):
                    out = ops.ttsvd(Xd[i], rmax=cases.TTSVD_CASES[names[i]]["ranks_tt"], concurrent=True)
                streams[i].synchronize()
            return out

        with ThreadPoolExecutor(len(names)) as pool:
            res = list(pool.map(run, range(len(names))))
    finally:
        ops.set_reserved_sms(0)
    for n, x, cores in zip(names, Xs, res):
        alg = "svd" if f"{n}/svd/relerr" in g.files else "eig"
        assert ranks_of(cores) == list(g[f"{n}/{alg}/ranks"])
        assert abs(relerr64(x, cores) - float(g[f"{n}/{alg}/relerr"])) <= 1e-5
