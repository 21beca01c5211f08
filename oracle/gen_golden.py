"""Generate golden vectors from the REAL reference (rballester/tntorch @ /root/reference).

Run in the build container only (the GPU box has no /root/reference):

    cd /tmp && python /root/repo/oracle/gen_golden.py

Writes ``tests/golden/*.npz``.  Inputs are produced by ``oracle/cases.py`` (NumPy
``default_rng`` streams, bit-identical on every machine), so tests regenerate the
inputs and only the reference's outputs (ranks, relative errors, singular values,
small TT cores and truncated-SVD factors, maxvol index sets) are stored.
"""
import os
import sys
import warnings

import numpy as np

warnings.filterwarnings("ignore")
HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(HERE)
sys.path.insert(0, "/root/reference")
sys.path.insert(0, REPO)

import torch  # noqa: E402
import tntorch as tn  # noqa: E402  (the real reference)
from tntorch.maxvol import py_maxvol as ref_maxvol  # noqa: E402

from oracle import cases  # noqa: E402

OUT = os.path.join(REPO, "tests", "golden")
os.makedirs(OUT, exist_ok=True)
torch.set_num_threads(os.cpu_count())


def rel_err64(X, t):
    X64 = torch.as_tensor(X, dtype=torch.float64)
    return float(torch.norm(X64 - t.torch().double()) / torch.norm(X64))


def gen_ttsvd():
    out = {}
    for name, spec in cases.TTSVD_CASES.items():
        X = cases.make_dense(spec)
        for alg in ("svd", "eig"):
            if spec.get("big") and alg == "svd":
                continue
            kw = dict(algorithm=alg)
            if spec.get("eps") is not None:
                kw["eps"] = spec["eps"]
            else:
                kw["ranks_tt"] = spec["ranks_tt"]
            # the reference's zero-matrix branch (round.py:137-145) allocates in the DEFAULT dtype
            torch.set_default_dtype(torch.float64 if X.dtype == np.float64 else torch.float32)
            t = tn.Tensor(torch.as_tensor(X), **kw)
            torch.set_default_dtype(torch.float32)
            out[f"{name}/{alg}/ranks"] = np.asarray(t.ranks_tt, dtype=np.int64)
            out[f"{name}/{alg}/relerr"] = np.float64(rel_err64(X, t))
            # the reconstruction is compared for structured fp64 inputs only; it is stored as the reference's TT
            # cores (a few KB) rather than the dense tensor, and tests rebuild it with tt_oracle.tt_reconstruct
            if X.size <= 70000 and X.dtype == np.float64 and spec["kind"] not in ("randn", "zeros") and "eps" not in kw:
                for k, c in enumerate(t.cores):
                    out[f"{name}/{alg}/core{k}"] = c.numpy()
            print(name, alg, list(t.ranks_tt), out[f"{name}/{alg}/relerr"], flush=True)
    np.savez_compressed(os.path.join(OUT, "ttsvd.npz"), **out)


def gen_lownoise():
    """fp32 inputs with a discarded tail far below the TF32 noise floor (oracle/cases.py LOWNOISE_CASES)."""
    out = {}
    for name, spec in cases.LOWNOISE_CASES.items():
        X = cases.make_dense(spec)
        for alg in ("svd", "eig"):
            t = tn.Tensor(torch.as_tensor(X), ranks_tt=spec["ranks_tt"], algorithm=alg)
            out[f"{name}/{alg}/ranks"] = np.asarray(t.ranks_tt, dtype=np.int64)
            out[f"{name}/{alg}/relerr"] = np.float64(rel_err64(X, t))
            print(name, alg, list(t.ranks_tt), out[f"{name}/{alg}/relerr"], flush=True)
    np.savez_compressed(os.path.join(OUT, "lownoise.npz"), **out)


def gen_round():
    out = {}
    for name, spec in cases.ROUND_CASES.items():
        cores = cases.make_tt(spec)
        dense = cases.tt_full(cores)
        for alg in ("svd", "eig"):
            t = tn.Tensor([torch.as_tensor(c.copy()) for c in cores])
            kw = dict(algorithm=alg)
            if "eps" in spec:
                kw["eps"] = spec["eps"]
            if "rmax" in spec:
                kw["rmax"] = spec["rmax"]
            t.round_tt(**kw)
            out[f"{name}/{alg}/ranks"] = np.asarray(t.ranks_tt, dtype=np.int64)
            out[f"{name}/{alg}/relerr"] = np.float64(rel_err64(dense, t))
            print(name, alg, list(t.ranks_tt), out[f"{name}/{alg}/relerr"], flush=True)
    np.savez_compressed(os.path.join(OUT, "round_tt.npz"), **out)


def gen_truncsvd():
    out = {}
    for name, spec in cases.TSVD_CASES.items():
        M = cases.make_matrix(spec)
        for alg in ("svd", "eig"):
            prods = []
            for lo in (True, False):
                kw = {k: spec[k] for k in ("eps", "delta", "rmax") if k in spec}
                left, right = tn.truncated_svd(torch.as_tensor(M), left_ortho=lo, algorithm=alg, **kw)
                key = f"{name}/{alg}/{'L' if lo else 'R'}"
                out[key + "/rank"] = np.int64(left.shape[1])
                prods.append(left.double().numpy() @ right.double().numpy())
                if lo:
                    # the product left @ right is stored as its factors (kilobytes instead of megabytes), once per
                    # algorithm: both orientations of the split give the same matrix to rounding (checked below)
                    out[f"{name}/{alg}/left"] = left.numpy()
                    out[f"{name}/{alg}/right"] = right.numpy()
                out[key + "/orth"] = np.float64(
                    float(torch.dist(left.T @ left, torch.eye(left.shape[1], dtype=left.dtype)))
                    if lo
                    else float(torch.dist(right @ right.T, torch.eye(left.shape[1], dtype=left.dtype)))
                )
                print(key, int(left.shape[1]), flush=True)
            rounding = 1e-5 if M.dtype == np.float32 else 1e-12
            assert np.abs(prods[0] - prods[1]).max() <= rounding * max(1.0, np.abs(M).max()), (name, alg)
    np.savez_compressed(os.path.join(OUT, "truncated_svd.npz"), **out)


def gen_maxvol():
    out = {}
    for name, spec in cases.MAXVOL_CASES.items():
        A = cases.make_matrix(spec)
        idx, C = ref_maxvol(A)
        out[f"{name}/index"] = np.asarray(idx, dtype=np.int64)
        out[f"{name}/absmax"] = np.float64(np.abs(C).max())
        print(name, idx[:6], np.abs(C).max(), flush=True)
    np.savez_compressed(os.path.join(OUT, "maxvol.npz"), **out)


def gen_rect_maxvol():
    from tntorch.maxvol import py_rect_maxvol as ref_rect

    out = {}
    for name, (spec, kw) in cases.RECT_MAXVOL_CASES.items():
        A = cases.make_matrix(spec)
        idx, C = ref_rect(A, **kw)
        out[f"{name}/index"] = np.asarray(idx, dtype=np.int64)
        out[f"{name}/C"] = np.asarray(C, dtype=np.float64)
        print(name, len(idx), idx[-4:], flush=True)
    np.savez_compressed(os.path.join(OUT, "rect_maxvol.npz"), **out)


def gen_cross_batch():
    """config 5: the reference has no batch mode (cross.py:256-258): B problems = B sequential calls from one seed."""
    import time as _t

    res = {}
    torch.set_default_dtype(torch.float64)
    for name, spec in cases.CROSS_BATCH_CASES.items():
        np.random.seed(spec["seed"])
        torch.manual_seed(spec["seed"])
        domain = [torch.linspace(spec["lo"], spec["hi"], spec["I"], dtype=torch.float64) for _ in range(spec["N"])]
        out = {"val_eps": [], "nsamples": [], "iters": [], "probe": []}
        probe_idx = np.random.default_rng(7).integers(0, spec["I"], size=(50, spec["N"]))
        kw = {k: spec[k] for k in ("ranks_tt", "max_iter", "eps") if k in spec}
        t0 = _t.perf_counter()
        for b in range(spec["nproblems"]):
            fn = cases.cross_family_function(b, spec["family"])
            t, info = tn.cross(fn, domain=domain, verbose=False, return_info=True, suppress_warnings=True, **kw)
            out["val_eps"].append(float(info["val_eps"]))
            out["nsamples"].append(int(info["nsamples"]))
            out["iters"].append(len(info["val_epss"]))
            out["probe"].append(t[[torch.as_tensor(probe_idx[:, k]) for k in range(spec["N"])]].torch().numpy())
            print(name, b, float(info["val_eps"]), info["nsamples"], len(info["val_epss"]), flush=True)
        dt = _t.perf_counter() - t0
        res[f"{name}/val_eps"] = np.array(out["val_eps"])
        res[f"{name}/nsamples"] = np.array(out["nsamples"])
        res[f"{name}/iters"] = np.array(out["iters"])
        res[f"{name}/probe"] = np.stack(out["probe"])
        res[f"{name}/probe_idx"] = probe_idx
        res[f"{name}/seconds_per_problem_{os.cpu_count()}cores"] = np.float64(dt / spec["nproblems"])
    torch.set_default_dtype(torch.float32)
    np.savez_compressed(os.path.join(OUT, "cross_batch.npz"), **res)


def gen_cpals():
    out = {}
    for name, spec in cases.CP_CASES.items():
        X = cases.make_cp_dense(spec)
        torch.manual_seed(0)
        t = tn.Tensor(torch.as_tensor(X), ranks_cp=spec["R"], max_iter=spec["sweeps"], tol=float("-inf"))
        out[f"{name}/relerr"] = np.float64(rel_err64(X, t))
        print(name, out[f"{name}/relerr"], flush=True)
    np.savez_compressed(os.path.join(OUT, "cp_als.npz"), **out)


def gen_tucker():
    out = {}
    torch.set_default_dtype(torch.float64)
    for name, c in cases.TUCKER_CASES.items():
        if c["kind"] == "dense":
            X = cases.make_dense(c["spec"])
            kw = {k: c[k] for k in ("ranks_tucker", "eps") if k in c}
            t = tn.Tensor(torch.as_tensor(X), **kw)
            dense = X
        else:
            cores = cases.make_tt(c["spec"])
            dense = cases.tt_full(cores)
            t = tn.Tensor([torch.as_tensor(x.copy()) for x in cores])
            if "round_tucker" in c:
                t.round_tucker(**c["round_tucker"])
            else:
                t.round(**c["round"])
        out[f"{name}/ranks_tt"] = np.asarray(t.ranks_tt, dtype=np.int64)
        out[f"{name}/ranks_tucker"] = np.asarray(t.ranks_tucker, dtype=np.int64)
        out[f"{name}/relerr"] = np.float64(rel_err64(dense, t))
        print(name, list(t.ranks_tt), list(t.ranks_tucker), out[f"{name}/relerr"], flush=True)
    torch.set_default_dtype(torch.float32)
    np.savez_compressed(os.path.join(OUT, "tucker.npz"), **out)


def gen_cross():
    out = {}
    torch.set_default_dtype(torch.float64)
    for name, spec in cases.CROSS_CASES.items():
        np.random.seed(spec["seed"])
        torch.manual_seed(spec["seed"])
        domain = [torch.linspace(spec["lo"], spec["hi"], spec["I"], dtype=torch.float64) for _ in range(spec["N"])]
        kw = {k: spec[k] for k in ("ranks_tt", "kickrank", "eps", "max_iter") if k in spec}
        fn = cases.cross_function(spec.get("shift", 0.0), spec.get("fn"))
        if spec.get("minimize"):
            kw["_minimize"] = True
        t, info = tn.cross(fn, domain=domain, verbose=False, return_info=True, suppress_warnings=True, **kw)
        if spec.get("minimize"):
            out[f"{name}/min"] = np.float64(float(info["min"]))
            out[f"{name}/argmin"] = np.asarray(info["argmin"], dtype=np.int64)
            print(name, "min", float(info["min"]), "argmin", info["argmin"], flush=True)
        if spec.get("forward"):
            tf = tn.cross_forward(info, fn, domain=domain)
            out[f"{name}/forward_full"] = tf.torch().double().numpy()
            out[f"{name}/cross_full"] = t.torch().double().numpy()
        full_err = None
        if spec["I"] ** spec["N"] <= 40_000_000 and not spec.get("minimize"):
            grids = torch.meshgrid(*domain, indexing="ij")
            gt = fn(*grids)
            full_err = float(torch.norm(gt - t.torch()) / torch.norm(gt))
            out[f"{name}/full_relerr"] = np.float64(full_err)
        out[f"{name}/val_eps"] = np.float64(float(info["val_eps"]))
        out[f"{name}/nsamples"] = np.int64(info["nsamples"])
        out[f"{name}/Rs"] = np.asarray(info["Rs"], dtype=np.int64)
        out[f"{name}/lset_last"] = np.asarray(info["lsets"][-1], dtype=np.int64)
        print(name, float(info["val_eps"]), info["nsamples"], list(info["Rs"]), full_err, flush=True)
    torch.set_default_dtype(torch.float32)
    np.savez_compressed(os.path.join(OUT, "cross.npz"), **out)


if __name__ == "__main__":
    which = sys.argv[1:] or ["ttsvd", "round", "tsvd", "maxvol", "cp", "cross", "tucker", "lownoise", "rect", "crossbatch"]
    if "ttsvd" in which:
        gen_ttsvd()
    if "lownoise" in which:
        gen_lownoise()
    if "rect" in which:
        gen_rect_maxvol()
    if "crossbatch" in which:
        gen_cross_batch()
    if "round" in which:
        gen_round()
    if "tsvd" in which:
        gen_truncsvd()
    if "maxvol" in which:
        gen_maxvol()
    if "cp" in which:
        gen_cpals()
    if "cross" in which:
        gen_cross()
    if "tucker" in which:
        gen_tucker()
