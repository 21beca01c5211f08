#!/usr/bin/env python
"""bench.py — TT-SVD GElements/s on B200 (BASELINE.json metric), one JSON line on rank 0.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--shape 64,64,64,64,64] [--rank 32]
                    [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 ... bench.py --gpus N ...

A "step" = one tnb_ttsvd_batch call per GPU: the complete TT-SVD (tn.Tensor(X[B, ...], ranks_tt=r, batch=True)) of
--per-gpu-batch dense fp32 tensors.
Workload: BASELINE.json configs[1] names 64^8 (2^48 elements = 1.1 PB) which cannot exist on any
machine; the stand-in is the largest 64^d that fits one GPU, randn(64,64,64,64,64) fp32 (4 GiB),
target TT-rank 32 (SURVEY.md §0.4 / §8d, BASELINE.md §2).  Multi-GPU: weak scaling, the batch dimension
shards over the ranks, no data-path collective, one NCCL all-gather of the final cores per step.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

REPO = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, REPO)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--shape", default="64,64,64,64,64")
    ap.add_argument("--rank", type=int, default=32)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-tc", action="store_true", help="generic CUDA-core kernels only (A/B runs)")
    ap.add_argument("--cpu-shape", default="32,32,32,32,32", help="bounded sample timed on the host cores")
    ap.add_argument("--reserve-sms", type=int, default=-1, help="SMs left free by the persistent kernels (measured: no gain on B200, default 0)")
    ap.add_argument("--per-gpu-batch", type=int, default=8,
                    help="independent tensors per GPU and step, decomposed by ONE tnb_ttsvd_batch call (the library keeps "
                         "them in flight on internal streams: the latency-bound eigen chains of one tensor run beside the "
                         "bandwidth-bound Gram/projection kernels of another)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the TT cores of the last step as DIR/tensor<i>_core<k>.npy "
                         "(inputs are seeded, so two builds run with the same arguments can be compared file by file)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    return args


METRIC = "TT-SVD GElements/s"
_json_out = sys.stdout  # replaced in __main__ by a duplicate of the real fd 1 (everything else goes to stderr)
DUMP_BUDGET_BYTES = 64 << 20  # all files written by one process's --dump-outputs together


def dump_outputs(directory, arrays, budget=DUMP_BUDGET_BYTES):
    """Write `arrays` (name -> torch tensor or NumPy array, float32 or float64) as DIR/<name>.npy.  When they are larger
    than `budget` in all, each array is cut to the same fixed, seeded sample of its flattened elements, so that two runs
    with the same arguments still write comparable files."""
    import numpy as np

    host = {n: a.detach().cpu().numpy() if hasattr(a, "detach") else np.asarray(a) for n, a in arrays.items()}
    total = sum(x.nbytes for x in host.values())
    keep = min(1.0, budget / total) if total else 1.0
    os.makedirs(directory, exist_ok=True)
    for name, x in host.items():
        if keep < 1.0:
            flat = x.reshape(-1)
            x = flat[np.sort(np.random.default_rng(0).choice(flat.size, int(flat.size * keep), replace=False))]
        np.save(os.path.join(directory, name + ".npy"), x)


# ------------------------------------------------------------------------------------------------
# CPU arm: the REAL reference (rballester/tntorch, staged unmodified into oracle/_ref/ by __graft_entry__.build())
# timed on the box's host cores; the NumPy port (oracle/tt_oracle.py) only when the staged copy is missing.
# ------------------------------------------------------------------------------------------------
def cpu_threads():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def cpu_model():
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                return line.split(":", 1)[1].strip()
    except Exception:
        pass
    return "unknown"


def workload_config(args):
    """The `config` both arms print (nothing run-dependent in it, so the two lines carry the same dict)."""
    shape = [int(s) for s in args.shape.split(",")]
    return {"workload": f"TT-SVD randn{shape} fp32 -> TT-rank {args.rank} (stand-in for the infeasible 64^8: 1.1 PB)",
            "per_gpu_batch": max(1, args.per_gpu_batch),
            "parallelism": "batch-sharded over the GPUs (independent tensors), all-gather of the final cores",
            "l2": "input 4 GiB >> 126 MB L2 (no flush needed)"}


class CpuArm:
    """tn.Tensor(X, ranks_tt=r, algorithm=...) of the reference on a bounded sample of the workload."""

    def __init__(self, shape, rank):
        import numpy as np

        self.shape, self.rank = tuple(shape), rank
        self.n = int(np.prod(shape))
        self.tn = None
        try:
            from oracle import stage_ref

            self.tn = stage_ref.load()
        except Exception:
            self.tn = None
        self.kind = "reference" if self.tn is not None else "port"
        self.algorithm = "eig"
        self.threads = cpu_threads()

    def make_input(self, seed=0):
        import numpy as np

        return np.random.default_rng(seed).standard_normal(self.shape, dtype=np.float32)

    def step(self, X, algorithm=None):
        """One decomposition; returns (seconds, cores as numpy arrays)."""
        alg = algorithm or self.algorithm
        if self.tn is not None:
            import torch

            Xt = torch.from_numpy(X)
            t0 = time.perf_counter()
            t = self.tn.Tensor(Xt, ranks_tt=self.rank, algorithm=alg)
            dt = time.perf_counter() - t0
            return dt, [c.numpy() for c in t.cores]
        from oracle import tt_oracle as orc

        t0 = time.perf_counter()
        cores = orc.tt_svd(X, ranks_tt=self.rank, algorithm=alg)
        return time.perf_counter() - t0, cores

    def tune(self):
        """LAPACK/BLAS on these shapes does not scale to every core of a 100+ core host (and torchrun exports
        OMP_NUM_THREADS=1): try a few thread counts and both reference algorithms on the actual sample, keep the
        fastest combination (the reference's default 'svd' computes and discards a full Vh; 'eig' is its Gram form)."""
        avail = cpu_threads()
        X = self.make_input(0)
        best = (float("inf"), avail, "eig")
        for n in sorted({min(avail, c) for c in (8, 16, 32, 64, avail)}):
            self.set_threads(n)
            for alg in ("eig", "svd"):
                dt, _ = self.step(X, alg)
                if dt < best[0]:
                    best = (dt, n, alg)
        _, self.threads, self.algorithm = best
        self.set_threads(self.threads)
        return best

    def set_threads(self, n):
        if self.tn is not None:
            import torch

            torch.set_num_threads(int(n))
        else:
            try:
                from threadpoolctl import threadpool_limits

                self._lim = threadpool_limits(limits=int(n))
            except Exception:
                pass

    def describe(self, steps):
        what = ("rballester/tntorch tn.Tensor(X, ranks_tt=%d, algorithm='%s') from oracle/_ref" % (self.rank, self.algorithm)
                if self.tn is not None else "oracle/tt_oracle.py::tt_svd (NumPy port; oracle/_ref was not staged)")
        return (f"randn{list(self.shape)} fp32 r={self.rank} (bounded sample of the 64^5 workload), {what}, {steps} step(s), "
                f"threads and algorithm picked among 8/16/32/64/all x eig/svd; CPU: {cpu_model()}")


def run_reference(args):
    """`--impl reference`: the reference's own CPU implementation on a bounded sample of the workload."""
    rank_env = int(os.environ.get("RANK", "0"))
    if rank_env != 0:
        return
    shape = tuple(int(s) for s in args.cpu_shape.split(","))
    arm = CpuArm(shape, args.rank)
    arm.tune()
    for i in range(min(args.warmup, 1)):
        arm.step(arm.make_input(100 + i))
    times = []
    for i in range(args.steps):
        X = arm.make_input(i)
        dt, cores = arm.step(X)
        times.append(dt)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {f"tensor0_core{k}": c for k, c in enumerate(cores)})
    tot = sum(times)
    value = arm.n * args.steps / tot / 1e9
    out = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "GElements/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": tot / args.steps * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args),
        "cpu_baseline": {"value": value, "unit": "GElements/s", "cores": arm.threads, "cores_available": cpu_threads(),
                         "kind": arm.kind, "cpu_model": cpu_model(), "algorithm": arm.algorithm,
                         "sample": arm.describe(args.steps)},
        "e2e": {"value": value, "unit": "GElements/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(out), file=_json_out, flush=True)


# ------------------------------------------------------------------------------------------------
class ClockSampler:
    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits",
                                          "-i", str(self.index), "-lms", "100"], stdout=subprocess.PIPE, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, smax, reasons = [], [], set()
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                smax.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def algorithmic_bytes(shape, rank, esz=4):
    """SURVEY §8d: exact R->L TT-SVD reads the tensor twice and reads+writes every later carry once."""
    n = 1
    for s in shape:
        n *= s
    N = len(shape)
    total = 2 * n
    rows = n // shape[-1]
    r = 1
    carries = []
    for mu in range(N - 1, 0, -1):
        cols = shape[mu] * r
        r = min(rank, rows, cols)
        carries.append(rows * r)
        rows //= shape[mu - 1]
    total += 2 * sum(carries)
    return total * esz, carries


def tf32_peak_tflops(peaks):
    """Dense TF32 tcgen05 peak: measured on the box by scripts/measure_tf32_peak.py when its result is committed
    (profiles/r02_tf32_peak.json), else half the measured burst bf16 cuBLAS rate (the kernel is timed alone)."""
    try:
        d = json.load(open(os.path.join(REPO, "profiles", "r02_tf32_peak.json")))
        return float(d["tf32_tflops"]), "measured TF32 tcgen05 peak (profiles/r02_tf32_peak.json: " + d.get("how", "") + ")"
    except Exception:
        pass
    return float(peaks.get("bf16_tflops", 1700.0)) / 2, "TF32 dense peak taken as half the measured burst bf16 cuBLAS rate (kernel timed alone)"


def ncu_traffic_from_profiles(kind, step):
    """dram bytes per launch of the dominant kernels, read at run time from the committed ncu summary (never pasted)."""
    try:
        d = json.load(open(os.path.join(REPO, "profiles", "r02_ncu_traffic.json")))
        return d.get(f"{kind}{step}")
    except Exception:
        return None


def run_ours(args):
    import numpy as np
    import torch
    import torch.distributed as dist

    from tntorch_b200 import ops

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank_id = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world > 1:
        raise SystemExit(f"WORLD_SIZE={world} but --gpus {args.gpus}")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    shape = tuple(int(s) for s in args.shape.split(","))
    numel = int(np.prod(shape))
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(REPO, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "measured (MEASURED_PEAKS.json)" if "hbm_gbs" in peaks else "fallback (B200_PROFILING.md)"
    bf16_burst = float(peaks.get("bf16_tflops", 1700.0))

    # ---- the batch of this rank: PB independent tensors, decomposed by ONE library call per step (tnb_ttsvd_batch:
    # ---- the same entry point tn.Tensor(X[B, ...], ranks_tt=r, batch=True) and dist.ttsvd_batch_sharded go through)
    PB = max(1, args.per_gpu_batch)
    free_b, _ = torch.cuda.mem_get_info(dev)
    probe = ops.TTSVDBatchPlan(shape, torch.float32, 1, rmax=args.rank, device=dev, inflight=1, use_tensorcore=not args.no_tc)
    per_tensor = numel * 4 + probe.per_tensor_bytes + int(probe.cap) * 4
    del probe
    PB = max(1, min(PB, int(0.6 * free_b // per_tensor)))  # bounded by free HBM (inputs + workspaces), never grown
    reserve = args.reserve_sms if args.reserve_sms >= 0 else (4 if PB > 1 else 0)
    ops.set_reserved_sms(reserve)
    Xb = torch.empty((PB,) + shape, device=dev, dtype=torch.float32)  # PB x 4 GiB >> 126 MB L2
    for b in range(PB):
        g = torch.Generator(device=dev).manual_seed(1234 + rank_id * 16 + b)
        Xb[b].copy_(torch.randn(shape, generator=g, device=dev, dtype=torch.float32))
    plan = ops.TTSVDBatchPlan(shape, torch.float32, PB, rmax=args.rank, device=dev, inflight=PB, use_tensorcore=not args.no_tc)
    gather_out = None
    if world > 1:
        gather_out = torch.empty(world * plan.cores_buf.numel(), dtype=torch.float32, device=dev)

    def step():
        cores_list = plan.run(Xb)
        if world > 1:  # the final factor broadcast (north_star): one all-gather of every rank's cores
            dist.all_gather_into_tensor(gather_out, plan.cores_buf.view(-1))
        return cores_list

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        step()
    # ---- timed region: K steps, CUDA events on the launching stream, barrier + sync on both sides ----
    sampler = ClockSampler(local)
    barrier()
    if rank_id == 0:
        sampler.start()
    l0 = ops.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for _ in range(args.steps):
        cores_list = step()
    e1.record()
    barrier()
    ms_total = e0.elapsed_time(e1)
    launches = ops.launch_count() - l0
    clocks = sampler.stop() if rank_id == 0 else None
    t = torch.tensor([ms_total], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total = float(t.item())
    ms_step = ms_total / args.steps
    if args.dump_outputs:
        # every rank writes its own tensors under their global batch index, within its share of the budget
        dump_outputs(args.dump_outputs, {f"tensor{rank_id * PB + b}_core{k}": c
                                         for b, tcores in enumerate(cores_list) for k, c in enumerate(tcores)},
                     budget=DUMP_BUDGET_BYTES // world)
    value = world * PB * numel / (ms_step * 1e-3) / 1e9
    cores = cores_list[0]
    ranks = [1] + [int(c.shape[2]) for c in cores]
    spec_accepted = int(sum(plan.spec))
    X = Xb[0]

    # ---- one tensor, one call in flight (latency of a single tn.Tensor(X, ranks_tt=r)) + per-phase device timings
    # ---- (CUDA events inside the library on the launching stream, TNB_FLAG_PROFILE) ----
    single = ops.TTSVDPlan(shape, torch.float32, rmax=args.rank, device=dev, use_tensorcore=not args.no_tc)
    single.ws = plan.ws[: single.ws.numel()] if plan.ws.numel() >= single.ws.numel() else single.ws
    for _ in range(2):
        single.run(X)
    s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s0.record()
    nsingle = 5
    for _ in range(nsingle):
        single.run(X)
    s1.record()
    torch.cuda.synchronize()
    single_ms = s0.elapsed_time(s1) / nsingle
    prof_plan = ops.TTSVDPlan(shape, torch.float32, rmax=args.rank, device=dev, use_tensorcore=not args.no_tc, profile=True)
    prof_plan.ws = single.ws
    prof_plan.cores_buf = single.cores_buf
    phase = {"gram_ms": [], "eig_ms": [], "factor_ms": []}
    nprof = 3
    acc = np.zeros(32)
    prof_plan.run(X)
    for _ in range(nprof):
        prof_plan.run(X)
        acc += np.array(list(prof_plan.info))
    acc /= nprof
    nsteps = int(round(acc[7]))
    for s in range(nsteps):
        phase["gram_ms"].append(round(float(acc[8 + 3 * s]), 4))
        phase["eig_ms"].append(round(float(acc[9 + 3 * s]), 4))
        phase["factor_ms"].append(round(float(acc[10 + 3 * s]), 4))
    # dominant kernel = the largest single-kernel phase (Gram and projection phases are ONE kernel each; the eigen
    # phases are chains of small launches and are reported as a share in phases_ms)
    cand = []
    B_alg, carries = algorithmic_bytes(shape, args.rank)
    for s in range(nsteps):
        cand.append((phase["gram_ms"][s], f"Gram of step {s}", s, "gram"))
        cand.append((phase["factor_ms"][s], f"project_tc_kernel (3xTF32 projection of step {s})", s, "factor"))
    cand.sort(reverse=True)
    top_ms, top_name, top_s, top_kind = cand[0]
    rows = numel // shape[-1]
    r_prev = 1
    dims = []
    for mu in range(len(shape) - 1, 0, -1):
        cols = shape[mu] * r_prev
        r = ranks[mu]
        dims.append((rows, cols, r))
        r_prev = r
        rows //= shape[mu - 1]
    tf32_peak = tf32_peak_tflops(peaks)
    tf32_note = tf32_peak[1]
    tf32_peak = tf32_peak[0]

    def kernel_roof(ms_k, name_k, s_k, kind_k):
        rws_k, cls_k, rr_k = dims[s_k]
        if kind_k == "gram" and cls_k > 512:  # compute-bound symmetric Gram: rows*cols*(cols+1) flops on the upper triangle
            fl = rws_k * cls_k * (cls_k + 1)
            return {"kernel": "gram_tc2_kernel, cta_group::2 (" + name_k + ")", "bound": "tensor", "achieved": fl / ms_k / 1e9,
                    "peak": tf32_peak, "unit": "TFLOP/s", "alg_flops": fl, "peak_note": tf32_note, "ms": ms_k}
        by = rws_k * cls_k * 4 + (rws_k * rr_k * 4 if kind_k == "factor" else 0)
        return {"kernel": ("gram_tc_kernel (" + name_k + ")") if kind_k == "gram" else name_k, "bound": "hbm",
                "achieved": by / ms_k / 1e6, "peak": hbm_peak, "unit": "GB/s", "alg_bytes": by, "ms": ms_k}

    roof = kernel_roof(top_ms, top_name, top_s, top_kind)
    roof["frac"] = roof["achieved"] / roof["peak"]
    roof["traffic"] = ncu_traffic_from_profiles(top_kind, top_s) if list(shape) == [64] * 5 and args.rank == 32 and not args.no_tc else None
    roof["traffic_source"] = "profiles/r02_ncu_traffic.json (ncu --set full, dram__bytes_read.sum + dram__bytes_write.sum per launch)" if roof["traffic"] else None
    roof["peak_source"] = peak_src
    others = []
    for ms_k, name_k, s_k, kind_k in cand[:4]:
        o = kernel_roof(ms_k, name_k, s_k, kind_k)
        others.append({"kernel": o["kernel"], "ms": ms_k, "bound": o["bound"], "frac": o["achieved"] / o["peak"]})
    roof["kernels"] = others
    sweep_roof = {"alg_bytes_per_tensor": B_alg, "achieved_GBps": PB * B_alg / ms_step / 1e6, "peak_GBps": hbm_peak,
                  "frac": PB * B_alg / ms_step / 1e6 / hbm_peak,
                  "single_call_ms": single_ms, "single_call_GElements_per_s": numel / single_ms / 1e6,
                  "single_call_frac": B_alg / single_ms / 1e6 / hbm_peak}

    # ---- parity of what was just timed (device-side fp64 error kernel; not in the timed region) ----
    relerr = ops.tt_relative_error(X, cores)
    # the structured twin (SURVEY §8d: random Gaussian data is incompressible, its error says little): a random
    # TT-rank-32 tensor of the same shape + 1e-2 relative noise, built on the device, decomposed by the same call
    relerr_twin = None
    if rank_id == 0 and len(shape) >= 3:
        gt = torch.Generator(device=dev).manual_seed(99)
        rk = [1] + [min(args.rank, 32)] * (len(shape) - 1) + [1]
        f = torch.ones(1, 1, device=dev)
        for k, sk in enumerate(shape):
            ck = torch.randn(rk[k], sk * rk[k + 1], generator=gt, device=dev)
            f = (f @ ck).reshape(-1, rk[k + 1])
        tw = f.reshape(shape)
        tw.add_(torch.randn(shape, generator=gt, device=dev), alpha=1e-2 * float(tw.std()))
        ctw = single.run(tw)
        relerr_twin = {"value": ops.tt_relative_error(tw, ctw), "noise": 1e-2,
                       "note": "same call on randn TT-rank-32 signal + 1e-2 sigma noise; reference on the NumPy twin of this "
                               "construction: 0.01022974 (tests/golden/full.npz, tests/test_gpu_fullgolden.py)"}
        del tw, f
    del prof_plan, single

    # ---- e2e: HOST buffers through the same batch entry point, H2D + D2H inside the timed region ----
    e2e = None
    if not args.no_e2e:
        # two tensors per step on one GPU (8 GiB of pinned host memory is enough to be PCIe-bound); one per rank when several
        # ranks share the host, so that N ranks pin N x 4 GiB, not N x 8 GiB
        EB = min(PB, 2 if world == 1 else 1)
        hplan = ops.TTSVDBatchPlan(shape, torch.float32, EB, rmax=args.rank, device=dev, inflight=EB,
                                   use_tensorcore=not args.no_tc, host_io=True)
        hplan.ws = plan.ws  # share the workspace (EB <= PB slices)
        xh = torch.empty((EB,) + shape, dtype=torch.float32, pin_memory=True)
        xh.copy_(Xb[:EB])

        def e2e_step():
            hc = hplan.run_host(xh)
            return float(hc[0][0][0, 0, 0])  # the result is on the host

        for _ in range(2):
            e2e_step()
        barrier()
        f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        f0.record()
        ksteps = max(2, min(args.steps, 5))
        for _ in range(ksteps):
            e2e_step()
        f1.record()
        barrier()
        tt = torch.tensor([f0.elapsed_time(f1)], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        ems = float(tt.item()) / ksteps
        e2e = {"value": world * EB * numel / (ems * 1e-3) / 1e9, "unit": "GElements/s", "ms_per_step": ems,
               "h2d_bytes_per_step": EB * numel * 4, "d2h_bytes_per_step": EB * int(hplan.cap) * 4, "steps": ksteps,
               "tensors_per_step": EB,
               "note": "pinned host tensors -> tnb_ttsvd_batch -> cores in pinned host memory; bound by the PCIe link (4 GiB per tensor)"}
        del hplan, xh
        torch.cuda.empty_cache()

    cpu = None
    same_sample = None
    if rank_id == 0 and world == 1 and not args.no_cpu_baseline:  # N = 1 only (the other ranks would idle at the teardown)
        # the e2e buffers are freed by now: the CPU leg needs host RAM and cores, not HBM
        cshape = tuple(int(s) for s in args.cpu_shape.split(","))
        arm = CpuArm(cshape, args.rank)
        arm.tune()
        CX = arm.make_input(0)
        dt, ccores = arm.step(CX)
        v = arm.n / dt / 1e9
        cpu = {"value": v, "unit": "GElements/s", "cores": arm.threads, "cores_available": cpu_threads(), "kind": arm.kind,
               "cpu_model": cpu_model(), "algorithm": arm.algorithm, "sample": arm.describe(1) + f"; 1 pass = {dt:.2f} s"}
        # the SAME sample through our path: device-resident and end to end from host memory (same_config ratios)
        Xs_dev = torch.from_numpy(CX).to(dev)
        splan = ops.TTSVDPlan(cshape, torch.float32, rmax=args.rank, device=dev, use_tensorcore=not args.no_tc)
        for _ in range(3):
            scores = splan.run(Xs_dev)
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        reps = 10
        s0.record()
        for _ in range(reps):
            scores = splan.run(Xs_dev)
        s1.record()
        torch.cuda.synchronize()
        ms_dev = s0.elapsed_time(s1) / reps
        hplan = ops.TTSVDPlan(cshape, torch.float32, rmax=args.rank, device=dev, use_tensorcore=not args.no_tc, host_io=True)
        xh = torch.from_numpy(CX).pin_memory()
        hplan.run_host(xh)
        t0 = time.perf_counter()
        for _ in range(reps):
            hplan.run_host(xh)
        torch.cuda.synchronize()
        ms_host = (time.perf_counter() - t0) * 1e3 / reps
        import numpy as _np

        from oracle import tt_oracle as orc  # checker only: the error of both results against the same input

        e_ref = orc.relative_error(CX, ccores)
        e_ours = ops.tt_relative_error(Xs_dev, scores)
        same_sample = {"shape": list(cshape), "cpu_ms": dt * 1e3, "ours_device_ms": ms_dev, "ours_e2e_ms": ms_host,
                       "same_config_ratio_device": dt * 1e3 / ms_dev, "same_config_ratio_e2e": dt * 1e3 / ms_host,
                       "rel_error_reference": float(e_ref), "rel_error_ours": float(e_ours),
                       "note": "one tensor, one call in flight; the same bounded sample the CPU arm is timed on"}
        del Xs_dev, splan, hplan, xh

    if rank_id == 0:
        out = {
            "metric": METRIC, "value": value, "unit": "GElements/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32 (Gram: tcgen05 kind::tf32, fp32 TMEM accumulation; projections: 3xTF32 on tcgen05 = fp32 accuracy; Gram matrices, eigenproblems and rank rule in fp64)"
            if not args.no_tc else "f32 (fp64-accumulated Gram, fp32 projections)",
            "data": "synthetic",
            "config": workload_config(args),
            "run": {"per_gpu_batch_used": PB, "reserved_sms": reserve, "ranks": ranks,
                    "entry_point": "tnb_ttsvd_batch (ops.TTSVDBatchPlan.run): one call per step and GPU, one host thread, one synchronisation",
                    "speculative_sweeps_accepted": spec_accepted, "world": world},
            "rel_error": relerr,
            "rel_error_twin": relerr_twin,
            "gpu_launches": int(launches),
            "clocks": clocks,
            "roofline": roof,
            "sweep_roofline": sweep_roof,
            "phases_ms": phase,
            "e2e": e2e,
            "cpu_baseline": cpu,
            "same_sample": same_sample,
        }
        print(json.dumps(out), file=_json_out, flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    a = parse()
    # stdout carries exactly ONE JSON line: anything libraries print there (NCCL's version banner at communicator
    # creation, torchrun notices) is routed to stderr by pointing fd 1 at fd 2 for the whole run
    _json_out = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    sys.stdout = sys.stderr
    if a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)
