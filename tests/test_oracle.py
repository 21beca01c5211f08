"""The oracle (oracle/tt_oracle.py) pinned against golden vectors taken from the real
reference (oracle/gen_golden.py, run in the build container)."""
import os

import numpy as np
import pytest

from oracle import cases
from oracle import tt_oracle as orc

GOLD = os.path.join(os.path.dirname(__file__), "golden")


def _g(name):
    return np.load(os.path.join(GOLD, name))


@pytest.mark.parametrize("name", [k for k, v in cases.TTSVD_CASES.items() if not v.get("big") and "analytic" not in k and v.get("eps") is None])
@pytest.mark.parametrize("alg", ["svd", "eig"])
def test_ttsvd_oracle_matches_reference(name, alg):
    g = _g("ttsvd.npz")
    spec = cases.TTSVD_CASES[name]
    X = cases.make_dense(spec)
    cores = orc.tt_svd(X, ranks_tt=spec["ranks_tt"], algorithm=alg)
    ranks = [1] + [c.shape[2] for c in cores]
    assert ranks == list(g[f"{name}/{alg}/ranks"])
    if spec["kind"] == "zeros":
        assert all(np.all(c == 0) for c in cores)
        return
    ref = float(g[f"{name}/{alg}/relerr"])
    tol = 1e-6 if X.dtype == np.float32 else 1e-12
    if name == "smooth_f32_r6":
        tol = 2e-5  # fp32 LAPACK noise on a 1e-7-level error (the reference's own svd/eig differ by 4e-5)
    assert abs(orc.relative_error(X, cores) - ref) <= tol
    key = f"{name}/{alg}/core"
    if key + "0" in g.files and X.dtype == np.float64 and spec["kind"] != "randn":
        recon = orc.tt_reconstruct([g[f"{key}{k}"] for k in range(len(cores))])
        np.testing.assert_allclose(orc.tt_reconstruct(cores), recon, atol=1e-9 * np.abs(recon).max())


def test_tutorial_known_answers():
    """docs/tutorials/decompositions.ipynb:68 (0.0005) and :361 (ranks 1-4-6-1, 8.3358e-06)."""
    X = cases.analytic_field_128()
    cores = orc.tt_svd(X, ranks_tt=3)
    assert abs(orc.relative_error(X, cores) - 0.000512298) < 1e-8
    cores = orc.round_tt(orc.full_rank_tt(X), eps=1e-5)
    assert [c.shape[2] for c in cores] == [4, 6, 1]
    assert abs(orc.relative_error(X, cores) - 8.335824e-06) < 1e-10


@pytest.mark.parametrize("name", list(cases.ROUND_CASES))
@pytest.mark.parametrize("alg", ["svd", "eig"])
def test_round_tt_oracle_matches_reference(name, alg):
    g = _g("round_tt.npz")
    spec = cases.ROUND_CASES[name]
    cores = cases.make_tt(spec)
    kw = {k: spec[k] for k in ("eps", "rmax") if k in spec}
    out = orc.round_tt([c.copy() for c in cores], algorithm=alg, **kw)
    ranks = [1] + [c.shape[2] for c in out]
    if not (alg == "eig" and "doubled" in name):  # 'eig' ranks on exactly rank-deficient input are LAPACK-noise dependent
        assert ranks == list(g[f"{name}/{alg}/ranks"])
    ref = float(g[f"{name}/{alg}/relerr"])
    tol = 1e-5 if cores[0].dtype == np.float32 else 1e-9
    if int(np.prod([c.shape[1] for c in cores])) > 50_000_000:
        # 32^6: the dense tensor is 8.6 GB; ||A - B||^2 = <A,A> + <B,B> - 2<A,B> from TT inner products instead
        # (the error here is O(1), so the cancellation costs nothing)
        def dot(a, b):
            m = np.ones((1, 1))
            for x, y in zip(a, b):
                m = np.einsum("ab,aic,bid->cd", m, x.astype(np.float64), y.astype(np.float64), optimize=True)
            return float(m[0, 0])

        aa, bb, ab = dot(cores, cores), dot(out, out), dot(cores, out)
        err = np.sqrt(max(aa + bb - 2 * ab, 0.0) / aa)
    else:
        err = orc.relative_error(cases.tt_full(cores), out)
    assert abs(err - ref) <= tol


@pytest.mark.parametrize("name", list(cases.TSVD_CASES))
@pytest.mark.parametrize("alg", ["svd", "eig"])
@pytest.mark.parametrize("lo", [True, False])
def test_truncated_svd_oracle_matches_reference(name, alg, lo):
    g = _g("truncated_svd.npz")
    spec = cases.TSVD_CASES[name]
    M = cases.make_matrix(spec)
    kw = {k: spec[k] for k in ("eps", "delta", "rmax") if k in spec}
    left, right = orc.truncated_svd(M, left_ortho=lo, algorithm=alg, **kw)
    key = f"{name}/{alg}/{'L' if lo else 'R'}"
    if not (alg == "eig" and name == "lowrank_60x80"):
        assert left.shape[1] == int(g[key + "/rank"])
        tol = 1e-4 if M.dtype == np.float32 else 1e-8
        ref = g[f"{name}/{alg}/left"].astype(np.float64) @ g[f"{name}/{alg}/right"].astype(np.float64)
        np.testing.assert_allclose(left.astype(np.float64) @ right.astype(np.float64), ref, atol=tol * max(1.0, np.abs(M).max()))


def test_truncated_svd_errors():
    with pytest.raises(ValueError):
        orc.truncated_svd(np.eye(3), delta=1.0, eps=1.0)


@pytest.mark.parametrize("name", list(cases.MAXVOL_CASES))
def test_maxvol_oracle_matches_reference(name):
    g = _g("maxvol.npz")
    A = cases.make_matrix(cases.MAXVOL_CASES[name])
    idx, C = orc.py_maxvol(A)
    assert list(idx) == list(g[f"{name}/index"])
    assert abs(np.abs(C).max() - float(g[f"{name}/absmax"])) < 1e-9


@pytest.mark.parametrize("name", list(cases.RECT_MAXVOL_CASES))
def test_rect_maxvol_oracle_matches_reference(name):
    """maxvol.py:30-111: index sets bit-exact, coefficient matrix to rounding."""
    g = _g("rect_maxvol.npz")
    spec, kw = cases.RECT_MAXVOL_CASES[name]
    idx, C = orc.py_rect_maxvol(cases.make_matrix(spec), **kw)
    assert list(idx) == list(g[f"{name}/index"])
    np.testing.assert_allclose(C, g[f"{name}/C"], atol=1e-12)


# ---- §8(f)-3 callers: the reference's outputs (callers.npz) against the oracle's own primitives
@pytest.mark.parametrize("name", list(cases.HADAMARD_SUM_CASES))
def test_hadamard_sum_golden_is_the_dense_sum(name):
    """metrics.hadamard_sum: the reference's exact and re-rounded values against the dense elementwise product."""
    g = _g("callers.npz")
    ops64 = cases.hadamard_operands(cases.HADAMARD_SUM_CASES[name])
    dense = np.prod(np.stack([orc.tt_reconstruct(c) for c in ops64]), axis=0).sum()
    assert abs(float(g[f"{name}/exact"]) - dense) <= 1e-12 * abs(dense)
    assert abs(float(g[f"{name}/svd"]) - dense) <= 1e-6 * abs(dense)


@pytest.mark.parametrize("name", list(cases.SHIFT_MODE_CASES))
def test_shift_mode_golden(name):
    """tools.shift_mode (tools.py:650-697) restated on the oracle's orthogonalisation + truncated_svd."""
    g = _g("callers.npz")
    spec, n, shift, eps = cases.SHIFT_MODE_CASES[name]
    cores = [c.copy() for c in cases.shift_mode_input(spec)]
    # orthogonalize(n)
    for mu in range(n):
        orc.left_orthogonalize(cores, mu)
    for mu in range(len(cores) - 1, n, -1):
        orc.right_orthogonalize(cores, mu)
    sign = 1 if shift > 0 else -1
    for i in range(n, n + shift, sign):
        c1, c2, lo = (i, i + 1, True) if sign == 1 else (i - 1, i, False)
        R1, I1, R2 = cores[c1].shape
        _, I2, R3 = cores[c2].shape
        sc = np.einsum("iaj,jbk->ibak", cores[c1], cores[c2]).reshape(R1 * I2, I1 * R3)
        kw = dict(eps=0, rmax=R2) if eps == "same" else dict(eps=eps / np.sqrt(abs(shift)))
        left, right = orc.truncated_svd(sc, left_ortho=lo, **kw)
        cores[c1], cores[c2] = left.reshape(R1, I2, -1), right.reshape(-1, I1, R3)
    got = orc.tt_reconstruct(cores)
    ref = g[f"{name}/full"]
    assert got.shape == ref.shape
    assert [1] + [c.shape[2] for c in cores] == g[f"{name}/ranks"].tolist()
    assert np.linalg.norm(got - ref) <= 1e-9 * np.linalg.norm(ref)


@pytest.mark.parametrize("name", list(cases.TTMATRIX_CASES))
def test_ttmatrix_golden(name):
    """TTMatrix.__init__ (matrix.py:96): permute to (i_k o_k) modes, then the oracle's TT-SVD with the rank caps."""
    g = _g("callers.npz")
    spec = cases.TTMATRIX_CASES[name]
    M = cases.ttmatrix_input(spec)
    idims, odims, d = spec["input_dims"], spec["output_dims"], len(spec["input_dims"])
    samples = M if spec["batch"] else M[None]
    outs = []
    for S in samples:
        X = S.reshape(idims + odims).transpose([k + s * d for k in range(d) for s in (0, 1)])
        X = X.reshape([idims[k] * odims[k] for k in range(d)])
        full = orc.tt_reconstruct(orc.tt_svd(X, ranks_tt=spec["ranks"]))
        full = full.reshape([s for k in range(d) for s in (idims[k], odims[k])])
        outs.append(full.transpose([2 * k for k in range(d)] + [2 * k + 1 for k in range(d)]).reshape(S.shape))
    got = np.stack(outs) if spec["batch"] else outs[0]
    np.testing.assert_allclose(got, g[f"{name}/full"], atol=1e-9 * np.abs(M).max())
