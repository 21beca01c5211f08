"""Thin torch-tensor wrappers over the C-ABI (device pointers in, torch tensors out).

PyTorch is plumbing here: device memory (caching allocator), the current stream and
``torch.distributed``.  All arithmetic happens inside libtnb200.so.
"""
from __future__ import annotations

import ctypes as C
from typing import List, Optional, Sequence, Tuple

import torch

from . import _lib
from ._lib import check, i32, i64, lib

_DT = {torch.float32: _lib.TNB_F32, torch.float64: _lib.TNB_F64}


def _dtype_code(t: torch.Tensor) -> int:
    if t.dtype not in _DT:
        raise ValueError(f"tntorch_b200 supports float32/float64 tensors, got {t.dtype}")
    return _DT[t.dtype]


def _require_cuda(t: torch.Tensor, what: str):
    if not t.is_cuda:
        raise RuntimeError(f"{what}: tensor must live on a CUDA device (tntorch_b200 has no CPU path)")


def _stream() -> C.c_void_p:
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _ws(nbytes: int, device) -> torch.Tensor:
    return torch.empty(max(int(nbytes), 256), dtype=torch.uint8, device=device)


def _ptr(t: Optional[torch.Tensor]) -> C.c_void_p:
    return C.c_void_p(0 if t is None else t.data_ptr())


def _rmax_list(rmax, nbonds: int) -> List[int]:
    """Reference convention (tensor.py:2027-2029): scalar or list of N-1; None = no cap."""
    if not hasattr(rmax, "__len__"):
        rmax = [rmax] * nbonds
    assert len(rmax) == nbonds
    out = []
    for r in rmax:
        if r is None:
            out.append(0)
        else:
            r = int(r)
            assert r >= 1
            out.append(min(r, 2**31 - 1))
    return out


def launch_count() -> int:
    return int(lib().tnb_launch_count())


def set_reserved_sms(n: int) -> None:
    """Leave n SMs free in the persistent kernels (useful with several decompositions in flight on different streams)."""
    lib().tnb_set_reserved_sms(int(n))


def measure_tf32_peak(reps: int = 200, per_commit: int = 64, trials: int = 5):
    """Dense TF32 tcgen05 peak of the current GPU in TFLOP/s (csrc/peak_tf32.cuh)."""
    tf, ms = (C.c_double * 1)(), (C.c_double * 1)()
    check(lib().tnb_measure_tf32_peak(int(reps), int(per_commit), int(trials), tf, ms, _stream()))
    return float(tf[0]), float(ms[0])


def has_tensorcore_path() -> bool:
    return bool(lib().tnb_has_tensorcore_path())


# --------------------------------------------------------------------------------------
def ttsvd(data: torch.Tensor, rmax=None, eps: float = 1e-14, batch_mode: bool = False, use_tensorcore: bool = True,
          return_info: bool = False, concurrent: bool = False, speculate: bool = True):
    """Dense tensor -> list of TT cores [r_{k-1}, I_k, r_k] (tn.Tensor(data, ranks_tt=...), tensor.py:401-408)."""
    _require_cuda(data, "ttsvd")
    data = data.contiguous()
    code = _dtype_code(data)
    N = data.dim()
    shape = list(data.shape)
    rm = _rmax_list(rmax, max(N - 1, 0))
    flags = ((0 if use_tensorcore else _lib.FLAG_NO_TENSORCORE) | (_lib.FLAG_BATCH_MODE if batch_mode else 0) |
             (_lib.FLAG_CONCURRENT if concurrent else 0) | (0 if speculate else _lib.FLAG_NO_SPECULATE))
    L = lib()
    sh = i64(shape)
    rmc = i32(rm) if N > 1 else i32([0])
    offs = (C.c_int64 * N)()
    cap = L.tnb_ttsvd_cores_capacity(N, sh, rmc, offs)
    if cap < 0:
        check(_lib.ERR_INVALID)
    wsb = L.tnb_ttsvd_workspace_bytes(code, N, sh, rmc, flags)
    if wsb == 0:
        check(_lib.ERR_UNSUPPORTED if L.tnb_last_error() else _lib.ERR_INVALID)
    ws = _ws(wsb, data.device)
    cores_buf = torch.empty(int(cap), dtype=data.dtype, device=data.device)
    ranks = (C.c_int32 * (N + 1))()
    info = (C.c_double * 32)()
    with torch.cuda.device(data.device):
        check(L.tnb_ttsvd(code, _ptr(data), N, sh, rmc, float(eps), flags, _ptr(ws), ws.numel(), _ptr(cores_buf), cap,
                          ranks, info, _stream()))
    cores = []
    for k in range(N):
        r0, r1 = ranks[k], ranks[k + 1]
        cores.append(cores_buf[offs[k]: offs[k] + r0 * shape[k] * r1].view(r0, shape[k], r1))
    if return_info:
        return cores, dict(norm=info[0], eig_solves=int(info[1]), chfsi_products=int(info[2]), tc_grams=int(info[3]),
                           fused_filters=int(info[31]), rr_sweeps=int(info[29]), outer_iterations=int(info[30]),
                           speculative=int(info[26]), spec_flags=int(info[27]))
    return cores


class TTSVDPlan:
    """Pre-allocated buffers for repeated decompositions of one shape (bench.py, serving loops)."""

    def __init__(self, shape: Sequence[int], dtype: torch.dtype, rmax=None, device="cuda", use_tensorcore: bool = True,
                 host_io: bool = False, profile: bool = False, concurrent: bool = False, speculate: bool = True):
        self.shape = [int(s) for s in shape]
        self.N = len(self.shape)
        self.dtype = dtype
        self.device = torch.device(device)
        self.code = _DT[dtype]
        self.rm = _rmax_list(rmax, max(self.N - 1, 0))
        # concurrent: several plans run at once on different streams (TNB_FLAG_CONCURRENT, include/tnb200.h)
        self.flags = ((0 if use_tensorcore else _lib.FLAG_NO_TENSORCORE) | (_lib.FLAG_PROFILE if profile else 0) |
                      (_lib.FLAG_CONCURRENT if concurrent else 0) | (0 if speculate else _lib.FLAG_NO_SPECULATE))
        L = lib()
        self._sh = i64(self.shape)
        self._rm = i32(self.rm) if self.N > 1 else i32([0])
        self._offs = (C.c_int64 * self.N)()
        self.cap = L.tnb_ttsvd_cores_capacity(self.N, self._sh, self._rm, self._offs)
        wsb = L.tnb_ttsvd_workspace_bytes(self.code, self.N, self._sh, self._rm, self.flags)
        if self.cap < 0 or wsb == 0:
            check(_lib.ERR_UNSUPPORTED)
        self.ws = _ws(wsb, self.device)
        self.cores_buf = torch.empty(int(self.cap), dtype=dtype, device=self.device)
        self.ranks = (C.c_int32 * (self.N + 1))()
        self.info = (C.c_double * 32)()
        self.numel = 1
        for s in self.shape:
            self.numel *= s
        self.dev_in = None
        self.cores_host = None
        if host_io:
            self.dev_in = torch.empty(self.numel, dtype=dtype, device=self.device)
            self.cores_host = torch.empty(int(self.cap), dtype=dtype, pin_memory=True)

    def run(self, data: torch.Tensor, eps: float = 1e-14):
        with torch.cuda.device(self.device):
            check(lib().tnb_ttsvd(self.code, _ptr(data), self.N, self._sh, self._rm, float(eps), self.flags,
                                  _ptr(self.ws), self.ws.numel(), _ptr(self.cores_buf), self.cap, self.ranks, self.info,
                                  _stream()))
        return self._views(self.cores_buf)

    def run_host(self, data_host: torch.Tensor, eps: float = 1e-14):
        """End-to-end call on HOST buffers: H2D of the tensor, decomposition, D2H of the cores."""
        assert self.dev_in is not None, "construct the plan with host_io=True"
        with torch.cuda.device(self.device):
            check(lib().tnb_ttsvd_host(self.code, _ptr(data_host), self.N, self._sh, self._rm, float(eps), self.flags,
                                       _ptr(self.dev_in), _ptr(self.ws), self.ws.numel(), _ptr(self.cores_buf), self.cap,
                                       _ptr(self.cores_host), self.ranks, self.info, _stream()))
        return self._views(self.cores_host)

    def _views(self, buf):
        out = []
        for k in range(self.N):
            r0, r1 = self.ranks[k], self.ranks[k + 1]
            out.append(buf[self._offs[k]: self._offs[k] + r0 * self.shape[k] * r1].view(r0, self.shape[k], r1))
        return out


class TTSVDBatchPlan:
    """Pre-allocated buffers for decomposing batches of `batch` dense tensors of one shape through tnb_ttsvd_batch
    (tn.Tensor(X[B, ...], ranks_tt=r, batch=True); bench.py; dist.ttsvd_batch_sharded).  Up to `inflight` tensors are
    in flight at once inside the library (internal streams, one enqueueing thread, one synchronisation)."""

    def __init__(self, shape: Sequence[int], dtype: torch.dtype, batch: int, rmax=None, device="cuda", inflight: int = 8,
                 use_tensorcore: bool = True, batch_mode: bool = False, host_io: bool = False):
        self.shape = [int(s) for s in shape]
        self.N = len(self.shape)
        self.batch = int(batch)
        self.dtype = dtype
        self.device = torch.device(device)
        self.code = _DT[dtype]
        self.rm = _rmax_list(rmax, max(self.N - 1, 0))
        self.flags = (0 if use_tensorcore else _lib.FLAG_NO_TENSORCORE) | (_lib.FLAG_BATCH_MODE if batch_mode else 0)
        L = lib()
        self._sh = i64(self.shape)
        self._rm = i32(self.rm) if self.N > 1 else i32([0])
        self._offs = (C.c_int64 * self.N)()
        self.cap = L.tnb_ttsvd_cores_capacity(self.N, self._sh, self._rm, self._offs)
        one = C.c_size_t(0)
        L.tnb_ttsvd_batch_workspace_bytes(self.code, self.batch, self.N, self._sh, self._rm, self.flags, C.byref(one))
        if self.cap < 0 or one.value == 0:
            check(_lib.ERR_UNSUPPORTED)
        self.per_tensor_bytes = int(one.value)
        self.inflight = max(1, min(int(inflight), self.batch, 8))
        self.ws = _ws(self.per_tensor_bytes * self.inflight, self.device)
        self.cores_buf = torch.empty(self.batch, int(self.cap), dtype=dtype, device=self.device)
        self.ranks = (C.c_int32 * (self.batch * (self.N + 1)))()
        self.norms = (C.c_double * self.batch)()
        self.spec = (C.c_int32 * self.batch)()
        self.numel = 1
        for s in self.shape:
            self.numel *= s
        self._cores_ptrs = (C.c_void_p * self.batch)(*[self.cores_buf[i].data_ptr() for i in range(self.batch)])
        self.dev_in = None
        self.cores_host = None
        if host_io:
            self.dev_in = torch.empty(self.batch, self.numel, dtype=dtype, device=self.device)
            self.cores_host = torch.empty(self.batch, int(self.cap), dtype=dtype, pin_memory=True)

    def run(self, tensors, eps: float = 1e-14):
        """tensors: a [batch, ...] tensor or a sequence of `batch` contiguous device tensors.  Returns, per tensor, the
        list of its cores (views of the plan's buffers: valid until the next run)."""
        if isinstance(tensors, torch.Tensor):
            tensors = [tensors[i] for i in range(tensors.shape[0])]
        assert len(tensors) == self.batch
        keep = [t if t.is_contiguous() else t.contiguous() for t in tensors]
        ptrs = (C.c_void_p * self.batch)(*[t.data_ptr() for t in keep])
        with torch.cuda.device(self.device):
            check(lib().tnb_ttsvd_batch(self.code, ptrs, self.batch, self.N, self._sh, self._rm, float(eps), self.flags,
                                        _ptr(self.ws), self.ws.numel(), self._cores_ptrs, self.cap, self.ranks, self.norms,
                                        self.spec, _stream()))
        return [self._views(self.cores_buf[i], i) for i in range(self.batch)]

    def run_host(self, tensors_host: torch.Tensor, eps: float = 1e-14):
        """End to end on HOST buffers: `tensors_host` [batch, ...] in (pinned) host memory -> device, decomposition,
        cores back to pinned host memory.  The copy of tensor i+1 overlaps nothing here (one stream): the PCIe link is
        the bound either way."""
        assert self.dev_in is not None, "construct the plan with host_io=True"
        flat = tensors_host.reshape(self.batch, self.numel)
        self.dev_in.copy_(flat, non_blocking=True)
        self.run(self.dev_in.view([self.batch] + self.shape), eps)
        self.cores_host.copy_(self.cores_buf, non_blocking=True)
        torch.cuda.current_stream().synchronize()
        return [self._views(self.cores_host[i], i) for i in range(self.batch)]

    def _views(self, buf, i):
        out = []
        base = i * (self.N + 1)
        for k in range(self.N):
            r0, r1 = self.ranks[base + k], self.ranks[base + k + 1]
            out.append(buf[self._offs[k]: self._offs[k] + r0 * self.shape[k] * r1].view(r0, self.shape[k], r1))
        return out


def ttsvd_batch(tensors, rmax=None, eps: float = 1e-14, batch_mode: bool = False, inflight: int = 8,
                use_tensorcore: bool = True, return_info: bool = False):
    """Decompose a batch of dense tensors of one shape (a [B, ...] tensor or a sequence): tn.Tensor(..., batch=True)
    and every caller that decomposes many tensors.  Returns a list (per tensor) of lists of cores (fresh tensors)."""
    if isinstance(tensors, torch.Tensor):
        tensors = [tensors[i] for i in range(tensors.shape[0])]
    if len(tensors) == 0:
        return ([], dict(speculative=[])) if return_info else []
    t0 = tensors[0]
    _require_cuda(t0, "ttsvd_batch")
    for t in tensors:
        if t.shape != t0.shape or t.dtype != t0.dtype or t.device != t0.device:
            raise ValueError("ttsvd_batch: all tensors must share shape, dtype and device")
    plan = TTSVDBatchPlan(t0.shape, t0.dtype, len(tensors), rmax=rmax, device=t0.device, inflight=inflight,
                          use_tensorcore=use_tensorcore, batch_mode=batch_mode)
    views = plan.run(tensors, eps)
    out = [[c.clone() for c in cores] for cores in views]
    if return_info:
        return out, dict(speculative=[int(x) for x in plan.spec], norms=[float(x) for x in plan.norms])
    return out


# --------------------------------------------------------------------------------------
def tt_round(cores: Sequence[torch.Tensor], eps: float = 1e-14, rmax=None, batch_mode: bool = False, speculate: bool = True):
    """Tensor.round_tt on device cores (tensor.py:2008-2083). Returns new cores.  speculate=False takes the host-driven
    sweeps even where the single-synchronisation path could run (TNB_FLAG_NO_SPECULATE)."""
    N = len(cores)
    for c in cores:
        _require_cuda(c, "tt_round")
        if c.dim() != 3:
            raise ValueError("tt_round expects TT cores of shape [r, I, r']")
    dt = cores[0].dtype
    cores = [c.contiguous() for c in cores]
    code = _dtype_code(cores[0])
    shape = [c.shape[1] for c in cores]
    rin = [cores[0].shape[0]] + [c.shape[2] for c in cores]
    for k in range(N - 1):
        if cores[k].shape[2] != cores[k + 1].shape[0]:
            raise ValueError("Core ranks do not match")
    rm = _rmax_list(rmax, max(N - 1, 0))
    L = lib()
    sh, rinc = i64(shape), i32(rin)
    rmc = i32(rm) if N > 1 else i32([0])
    offs = (C.c_int64 * N)()
    cap = L.tnb_tt_round_cores_capacity(N, sh, rinc, rmc, offs)
    if cap < 0:
        check(_lib.ERR_INVALID)
    wsb = L.tnb_tt_round_workspace_bytes(code, N, sh, rinc, rmc)
    if wsb == 0:
        check(_lib.ERR_UNSUPPORTED)
    dev = cores[0].device
    ws = _ws(wsb, dev)
    out = torch.empty(int(cap), dtype=dt, device=dev)
    ranks = (C.c_int32 * (N + 1))()
    ptrs = (C.c_void_p * N)(*[c.data_ptr() for c in cores])
    flags = (_lib.FLAG_BATCH_MODE if batch_mode else 0) | (0 if speculate else _lib.FLAG_NO_SPECULATE)
    with torch.cuda.device(dev):
        check(L.tnb_tt_round(code, ptrs, N, sh, rinc, rmc, float(eps), flags, _ptr(ws), ws.numel(), _ptr(out), cap, ranks,
                             _stream()))
    res = []
    for k in range(N):
        r0, r1 = ranks[k], ranks[k + 1]
        res.append(out[offs[k]: offs[k] + r0 * shape[k] * r1].view(r0, shape[k], r1))
    return res


def tt_round_batch(batch_cores: Sequence[Sequence[torch.Tensor]], eps: float = 1e-14, rmax=None, batch_mode: bool = False,
                   inflight: int = 8, return_info: bool = False):
    """Round a batch of TT tensors that share shape and input ranks: ONE library call, several tensors in flight
    (tnb_tt_round_batch).  batch_cores: per tensor, its list of cores [r, I, r'].  Returns per tensor the new cores."""
    B = len(batch_cores)
    if B == 0:
        return []
    N = len(batch_cores[0])
    dt, dev = batch_cores[0][0].dtype, batch_cores[0][0].device
    cs = [[c.contiguous() for c in cores] for cores in batch_cores]
    shape = [c.shape[1] for c in cs[0]]
    rin = [cs[0][0].shape[0]] + [c.shape[2] for c in cs[0]]
    for cores in cs:
        if [c.shape for c in cores] != [c.shape for c in cs[0]]:
            raise ValueError("tt_round_batch: all tensors must share their core shapes")
    code = _DT[dt]
    rm = _rmax_list(rmax, max(N - 1, 0))
    L = lib()
    sh, rinc = i64(shape), i32(rin)
    rmc = i32(rm) if N > 1 else i32([0])
    offs = (C.c_int64 * N)()
    cap = L.tnb_tt_round_cores_capacity(N, sh, rinc, rmc, offs)
    one = C.c_size_t(0)
    total = L.tnb_tt_round_batch_workspace_bytes(code, B, N, sh, rinc, rmc, C.byref(one))
    if cap < 0 or one.value == 0:
        check(_lib.ERR_UNSUPPORTED)
    k = max(1, min(int(inflight), B, 8))
    ws = _ws(one.value * k, dev)
    out = torch.empty(B, int(cap), dtype=dt, device=dev)
    ranks = (C.c_int32 * (B * (N + 1)))()
    spec = (C.c_int32 * B)()
    pin = (C.c_void_p * (B * N))(*[c.data_ptr() for cores in cs for c in cores])
    pout = (C.c_void_p * B)(*[out[i].data_ptr() for i in range(B)])
    flags = _lib.FLAG_BATCH_MODE if batch_mode else 0
    with torch.cuda.device(dev):
        check(L.tnb_tt_round_batch(code, pin, B, N, sh, rinc, rmc, float(eps), flags, _ptr(ws), ws.numel(), pout, cap, ranks, spec,
                                   _stream()))
    res = []
    for i in range(B):
        base = i * (N + 1)
        res.append([out[i, offs[n]: offs[n] + ranks[base + n] * shape[n] * ranks[base + n + 1]].view(ranks[base + n], shape[n], ranks[base + n + 1])
                    for n in range(N)])
    if return_info:
        return res, dict(speculative=[int(x) for x in spec])
    return res


def _tt_operands(operands):
    """operands: list of lists of TT cores [r, I, r'] (same shape, dtype, device) -> pointers / ranks for the C-ABI."""
    K = len(operands)
    N = len(operands[0])
    dt, dev = operands[0][0].dtype, operands[0][0].device
    ops_c = [[c.contiguous() for c in cores] for cores in operands]
    shape = [c.shape[1] for c in ops_c[0]]
    for cores in ops_c:
        if len(cores) != N or [c.shape[1] for c in cores] != shape:
            raise ValueError("TT operands must share their shape")
        for c in cores:
            _require_cuda(c, "tt_sum")
            if c.dim() != 3 or c.dtype != dt:
                raise ValueError("TT operands must be lists of [r, I, r'] cores of one dtype")
    ranks = []
    for cores in ops_c:
        ranks += [cores[0].shape[0]] + [c.shape[2] for c in cores]
    ptrs = (C.c_void_p * (K * N))(*[c.data_ptr() for cores in ops_c for c in cores])
    return ops_c, K, N, shape, ranks, ptrs, dt, dev


def tt_sum(operands, alpha=None):
    """sum_k alpha_k T_k as block TT cores (Tensor.__add__, tensor.py:445-520); no rounding."""
    ops_c, K, N, shape, ranks, ptrs, dt, dev = _tt_operands(operands)
    L = lib()
    rsum = (C.c_int32 * (N + 1))()
    offs = (C.c_int64 * N)()
    cap = L.tnb_tt_sum_cores_capacity(K, N, i64(shape), i32(ranks), rsum, offs)
    if cap < 0:
        check(_lib.ERR_INVALID)
    out = torch.empty(int(cap), dtype=dt, device=dev)
    al = None if alpha is None else (C.c_double * K)(*[float(a) for a in alpha])
    with torch.cuda.device(dev):
        check(L.tnb_tt_sum(_dtype_code(ops_c[0][0]), ptrs, K, al, N, i64(shape), i32(ranks), _ptr(out), cap, _stream()))
    return [out[offs[n]: offs[n] + rsum[n] * shape[n] * rsum[n + 1]].view(rsum[n], shape[n], rsum[n + 1]) for n in range(N)]


def tt_sum_round(operands, alpha=None, eps: float = 1e-14, rmax=None):
    """round_tt(sum_k alpha_k T_k) in ONE library call: block cores assembled in the workspace, then the rounding sweeps
    (the `tn.round(function(a, b))` step of tools.reduce, tools.py:460-512)."""
    ops_c, K, N, shape, ranks, ptrs, dt, dev = _tt_operands(operands)
    L = lib()
    rm = _rmax_list(rmax, max(N - 1, 0))
    rmc = i32(rm) if N > 1 else i32([0])
    offs = (C.c_int64 * N)()
    cap = L.tnb_tt_sum_round_cores_capacity(K, N, i64(shape), i32(ranks), rmc, offs)
    if cap < 0:
        check(_lib.ERR_INVALID)
    code = _dtype_code(ops_c[0][0])
    wsb = L.tnb_tt_sum_round_workspace_bytes(code, K, N, i64(shape), i32(ranks), rmc)
    if wsb == 0:
        check(_lib.ERR_UNSUPPORTED)
    ws = _ws(wsb, dev)
    out = torch.empty(int(cap), dtype=dt, device=dev)
    rk = (C.c_int32 * (N + 1))()
    al = None if alpha is None else (C.c_double * K)(*[float(a) for a in alpha])
    with torch.cuda.device(dev):
        check(L.tnb_tt_sum_round(code, ptrs, K, al, N, i64(shape), i32(ranks), rmc, float(eps), 0, _ptr(ws), ws.numel(), _ptr(out),
                                 cap, rk, _stream()))
    return [out[offs[n]: offs[n] + rk[n] * shape[n] * rk[n + 1]].view(rk[n], shape[n], rk[n + 1]) for n in range(N)]


def tt_hadamard(a_cores, b_cores):
    """Elementwise product of two TT tensors: Kronecker cores (Tensor.__mul__, tensor.py:560-640)."""
    ops_c, K, N, shape, ranks, ptrs, dt, dev = _tt_operands([a_cores, b_cores])
    ra, rb = ranks[: N + 1], ranks[N + 1:]
    outs = [torch.empty(ra[n] * rb[n], shape[n], ra[n + 1] * rb[n + 1], dtype=dt, device=dev) for n in range(N)]
    pa = (C.c_void_p * N)(*[c.data_ptr() for c in ops_c[0]])
    pb = (C.c_void_p * N)(*[c.data_ptr() for c in ops_c[1]])
    po = (C.c_void_p * N)(*[c.data_ptr() for c in outs])
    with torch.cuda.device(dev):
        check(lib().tnb_tt_hadamard(_dtype_code(ops_c[0][0]), pa, pb, N, i64(shape), i32(ra), i32(rb), po, _stream()))
    return outs


def truncated_svd(M: torch.Tensor, delta=None, eps=None, rmax=None, left_ortho=True, batch_mode: bool = False,
                  return_zero_flag: bool = False):
    """tn.truncated_svd (round.py:52-187) of one matrix.  batch_mode = the reference's rank rule for one sample of a
    batch (round.py:149-150); return_zero_flag additionally returns whether the sample was numerically zero."""
    if delta is not None and eps is not None:
        raise ValueError("Provide either `delta` or `eps`")
    _require_cuda(M, "truncated_svd")
    if M.dim() != 2:
        raise ValueError("truncated_svd expects a matrix")
    M = M.contiguous()
    code = _dtype_code(M)
    m, n = M.shape
    if rmax is None:
        rm = 0
    else:
        assert rmax >= 1
        rm = int(min(rmax, 2**31 - 1))
    L = lib()
    wsb = L.tnb_truncated_svd_workspace_bytes(code, m, n)
    if wsb == 0:
        check(_lib.ERR_UNSUPPORTED)
    ws = _ws(wsb, M.device)
    k = min(m, n)
    left = torch.empty(m * k, dtype=M.dtype, device=M.device)
    right = torch.empty(k * n, dtype=M.dtype, device=M.device)
    rank = (C.c_int32 * 1)()
    with torch.cuda.device(M.device):
        check(L.tnb_truncated_svd(code, _ptr(M), m, n, -1.0 if delta is None else float(delta),
                                  -1.0 if eps is None else float(eps), rm, (1 if left_ortho else 0) | (2 if batch_mode else 0),
                                  _ptr(ws), ws.numel(), _ptr(left), _ptr(right), rank, _stream()))
    r = abs(rank[0])
    out = left[: m * r].view(m, r), right[: r * n].view(r, n)
    return out + (rank[0] < 0,) if return_zero_flag else out


def cp_als(data: torch.Tensor, R: int, max_iter: int = 25, tol: float = 1e-4, return_info: bool = False, init=None):
    """CP-ALS on the device (tn.Tensor(data, ranks_cp=R, max_iter=, tol=), tensor.py:210-400).
    Returns the list of factor matrices [I_n, R].  init: optional list of starting factors [I_n, R] (CP on a Tucker
    core starts from random factors, tensor.py:278-302); default: the HOSVD initialisation of tensor.py:217-277."""
    _require_cuda(data, "cp_als")
    data = data.contiguous()
    code = _dtype_code(data)
    N = data.dim()
    shape = list(data.shape)
    L = lib()
    sh = i64(shape)
    offs = (C.c_int64 * N)()
    cap = L.tnb_cp_als_factors_capacity(N, sh, int(R), offs)
    if cap < 0:
        check(_lib.ERR_INVALID if N >= 2 else _lib.ERR_UNSUPPORTED)
    wsb = L.tnb_cp_als_workspace_bytes(code, N, sh, int(R))
    if wsb == 0:
        check(_lib.ERR_UNSUPPORTED)
    ws = _ws(wsb, data.device)
    fac = torch.zeros(int(cap), dtype=data.dtype, device=data.device)
    errs = (C.c_double * max(int(max_iter), 1))()
    iters = (C.c_int32 * 1)()
    entry = L.tnb_cp_als
    if init is not None:
        assert len(init) == N
        for n in range(N):
            assert tuple(init[n].shape) == (shape[n], int(R))
            fac[offs[n]: offs[n] + shape[n] * R].copy_(init[n].to(device=data.device, dtype=data.dtype).reshape(-1))
        entry = L.tnb_cp_als_from
    with torch.cuda.device(data.device):
        check(entry(code, _ptr(data), N, sh, int(R), int(max_iter), float(tol), _ptr(ws), ws.numel(), _ptr(fac), cap,
                    errs, iters, _stream()))
    factors = [fac[offs[n]: offs[n] + shape[n] * R].view(shape[n], R) for n in range(N)]
    if return_info:
        return factors, dict(errors=[errs[i] for i in range(iters[0])], iters=int(iters[0]))
    return factors


def maxvol(A: torch.Tensor, tol: float = 1.05, max_iters: int = 100, return_iters: bool = False):
    """Device maxvol (tntorch/maxvol.py:114-170).  A: [N, r] or a batch [B, N, r].  Returns (index int32 [.., min(N,r)],
    C [.., N, r] = A inv(A[index])) as device tensors; nothing is copied to the host."""
    _require_cuda(A, "maxvol")
    batched = A.dim() == 3
    A3 = (A if batched else A[None]).contiguous().double()
    B, N, r = A3.shape
    L = lib()
    ws = _ws(L.tnb_maxvol_workspace_bytes(B, N, r), A.device)
    index = torch.empty(B, r, dtype=torch.int32, device=A.device)
    Cm = torch.empty(B, N, r, dtype=torch.float64, device=A.device)
    iters = (C.c_int32 * B)() if return_iters else None
    with torch.cuda.device(A.device):
        check(L.tnb_maxvol(_ptr(A3), B, N, r, float(tol), int(max_iters), _ptr(ws), ws.numel(), _ptr(index), _ptr(Cm), iters,
                           _stream()))
    if N <= r:  # maxvol.py:126-127
        index, Cm = index[:, :N], Cm[:, :, :N]
    if not batched:
        index, Cm = index[0], Cm[0]
    if return_iters:
        return index, Cm, [int(x) for x in iters]
    return index, Cm


def rect_maxvol(A: torch.Tensor, tol: float = 1.0, maxK=None, min_add_K=None, minK=None, start_maxvol_iters: int = 10):
    """Device rect_maxvol (tntorch/maxvol.py:30-111).  A: [N, r] or a batch [B, N, r].  Returns (index, C) like the
    reference: the chosen rows (int32) and the coefficient matrix [N, K] with identity rows at the chosen positions; for
    a batch, lists of per-problem results (K is data dependent)."""
    _require_cuda(A, "rect_maxvol")
    batched = A.dim() == 3
    A3 = (A if batched else A[None]).contiguous().double()
    B, N, r = A3.shape
    if N <= r:  # maxvol.py:52-53
        out = [(torch.arange(N, dtype=torch.int32, device=A.device), torch.eye(N, dtype=torch.float64, device=A.device))
               for _ in range(B)]
        return out if batched else out[0]
    # parameter normalisation of maxvol.py:54-66
    if maxK is None or maxK > N:
        maxK = N
    if maxK < r:
        maxK = r
    if minK is None or minK < r:
        minK = r
    if minK > N:
        minK = N
    if min_add_K is not None:
        minK = max(minK, r + min_add_K)
    if minK > maxK:
        minK = maxK
    L = lib()
    ws = _ws(L.tnb_rect_maxvol_workspace_bytes(B, N, r, int(maxK)), A.device)
    index = torch.empty(B, int(maxK), dtype=torch.int32, device=A.device)
    Cm = torch.empty(B, N, int(maxK), dtype=torch.float64, device=A.device)
    Kd = torch.empty(B, dtype=torch.int32, device=A.device)
    with torch.cuda.device(A.device):
        check(L.tnb_rect_maxvol(_ptr(A3), B, N, r, float(tol), int(minK), int(maxK), int(start_maxvol_iters), _ptr(ws),
                                ws.numel(), _ptr(index), _ptr(Cm), _ptr(Kd), _stream()))
    Ks = Kd.tolist()
    out = [(index[b, : Ks[b]], Cm[b, :, : Ks[b]]) for b in range(B)]
    return out if batched else out[0]


# ---- batched TT-cross plumbing (cross_batch.py) -----------------------------------------------------------------------
def cross_gather_coords(lsets: torch.Tensor, rsets: torch.Tensor, grid: torch.Tensor, N: int, j: int, I: int):
    """lsets [B, Rl, j] / rsets [B, Rr, N-j-1] int32, grid [N, Imax] fp64 -> N coordinate vectors of length B*Rl*I*Rr."""
    B, Rl, Rr = lsets.shape[0], lsets.shape[1], rsets.shape[1]
    X = torch.empty(N, B * Rl * I * Rr, dtype=torch.float64, device=grid.device)
    lsets, rsets = lsets.contiguous(), rsets.contiguous()
    with torch.cuda.device(grid.device):
        check(lib().tnb_cross_gather_coords(_ptr(lsets), _ptr(rsets), _ptr(grid), grid.shape[1], B, N, j, Rl, I, Rr, _ptr(X),
                                            _stream()))
    return [X[k] for k in range(N)]


def cross_update_lsets(lsets: torch.Tensor, local: torch.Tensor, I: int, active=None, old=None):
    B, Rl, j = lsets.shape
    Rn = local.shape[1]
    out = old if (old is not None and active is not None) else torch.empty(B, Rn, j + 1, dtype=torch.int32, device=local.device)
    lsets, local = lsets.contiguous(), local.contiguous()
    with torch.cuda.device(local.device):
        check(lib().tnb_cross_update_lsets(_ptr(lsets), _ptr(local), B, j, Rl, I, Rn, _ptr(active) if old is not None else _ptr(None),
                                           _ptr(out), _stream()))
    return out


def cross_update_rsets(rsets: torch.Tensor, local: torch.Tensor, Rr: int, active=None, old=None):
    B, _, ln = rsets.shape  # suffix of modes j+1..N-1
    Rp = local.shape[1]
    out = old if (old is not None and active is not None) else torch.empty(B, Rp, ln + 1, dtype=torch.int32, device=local.device)
    rsets, local = rsets.contiguous(), local.contiguous()
    # N and j only enter through N - j - 1 = ln: pass (N, j) = (ln + 2, 1)
    I = 0
    with torch.cuda.device(local.device):
        check(lib().tnb_cross_update_rsets(_ptr(rsets), _ptr(local), B, ln + 2, 1, 1 << 30, Rr, Rp,
                                           _ptr(active) if old is not None else _ptr(None), _ptr(out), _stream()))
    return out


def cross_tt_eval(cores: Sequence[torch.Tensor], idx: torch.Tensor) -> torch.Tensor:
    """cores: N tensors [B, r, I, r'] fp64; idx: [P, N] (shared) or [B, P, N] int32 -> values [B, P]."""
    N = len(cores)
    B = cores[0].shape[0]
    per = idx.dim() == 3
    P = idx.shape[-2]
    cs = [c.contiguous() for c in cores]
    idx = idx.contiguous()
    out = torch.empty(B, P, dtype=torch.float64, device=cs[0].device)
    ptrs = (C.c_void_p * N)(*[c.data_ptr() for c in cs])
    ranks = i32([cs[0].shape[1]] + [c.shape[3] for c in cs])
    shape = i32([c.shape[2] for c in cs])
    with torch.cuda.device(cs[0].device):
        check(lib().tnb_cross_tt_eval(ptrs, N, ranks, shape, _ptr(idx), B, P, 1 if per else 0, _ptr(out), _stream()))
    return out


def matmul(A: torch.Tensor, B: torch.Tensor) -> torch.Tensor:
    """Row-major A @ B on the library's own GEMM (no cuBLAS)."""
    _require_cuda(A, "matmul")
    A, B = A.contiguous(), B.contiguous()
    assert A.dtype == B.dtype and A.shape[1] == B.shape[0]
    M, K = A.shape
    N = B.shape[1]
    Cm = torch.empty(M, N, dtype=A.dtype, device=A.device)
    with torch.cuda.device(A.device):
        check(lib().tnb_matmul(_dtype_code(A), _ptr(A), _ptr(B), _ptr(Cm), M, N, K, _stream()))
    return Cm


def qr(A: torch.Tensor, return_r: bool = False):
    """Householder QR on the device (torch.linalg.qr semantics, reduced): A [rows, n] or batch [B, rows, n], fp64."""
    _require_cuda(A, "qr")
    batched = A.dim() == 3
    A3 = (A if batched else A[None]).contiguous().double()
    B, rows, n = A3.shape
    k = min(rows, n)
    L = lib()
    ws = _ws(L.tnb_qr_workspace_bytes(B, rows, n), A.device)
    Q = torch.empty(B, rows, k, dtype=torch.float64, device=A.device)
    R = torch.empty(B, k, n, dtype=torch.float64, device=A.device) if return_r else None
    with torch.cuda.device(A.device):
        check(L.tnb_qr_householder(_ptr(A3), B, rows, n, _ptr(ws), ws.numel(), _ptr(Q), _ptr(R), _stream()))
    if not batched:
        Q = Q[0]
        R = R[0] if return_r else None
    return (Q, R) if return_r else Q


def gram(A: torch.Tensor, tensorcore: bool = False) -> torch.Tensor:
    """fp64 Gram matrix A^T A of a (rows x n) matrix; tensorcore=True uses the tcgen05/TMA kernel (fp32 only)."""
    _require_cuda(A, "gram")
    A = A.contiguous()
    rows, n = A.shape
    G = torch.empty(n, n, dtype=torch.float64, device=A.device)
    L = lib()
    with torch.cuda.device(A.device):
        if tensorcore:
            if A.dtype != torch.float32:
                raise ValueError("tensor-core Gram needs float32 input")
            wsb = L.tnb_gram_tc_workspace_bytes(rows, n)
            if wsb == 0:
                check(_lib.ERR_UNSUPPORTED)
            ws = _ws(wsb, A.device)
            check(L.tnb_gram_tc_f32(_ptr(A), rows, n, _ptr(G), _ptr(ws), ws.numel(), _stream()))
        else:
            code = _dtype_code(A)
            ws = _ws(L.tnb_gram_workspace_bytes(code, rows, n), A.device)
            check(L.tnb_gram(code, _ptr(A), rows, n, _ptr(G), _ptr(ws), ws.numel(), _stream()))
    return G


def atb_tensorcore(A: torch.Tensor, B: torch.Tensor, alpha: float = 1.0, D: Optional[torch.Tensor] = None,
                   beta: float = 0.0) -> torch.Tensor:
    """alpha * A^T B + beta * D on the tcgen05 kernel (A: K x m, B: K x n, fp32)."""
    _require_cuda(A, "atb_tensorcore")
    A, B = A.contiguous(), B.contiguous()
    K, m = A.shape
    n = B.shape[1]
    L = lib()
    wsb = L.tnb_atb_tc_workspace_bytes(K, m, n)
    if wsb == 0:
        check(_lib.ERR_UNSUPPORTED)
    ws = _ws(wsb, A.device)
    out = torch.empty(m, n, dtype=torch.float32, device=A.device)
    with torch.cuda.device(A.device):
        check(L.tnb_atb_tc_f32(_ptr(A), K, m, _ptr(B), n, _ptr(out), float(alpha), _ptr(D), float(beta), _ptr(ws),
                               ws.numel(), _stream()))
    return out


def cheb_filter(G: torch.Tensor, Y0: torch.Tensor, a, bc, g) -> torch.Tensor:
    """len(a) three-term filter products Y_s = a_s G Y_{s-1} + bc_s Y_{s-1} + g_s Y_{s-2} as one resident
    cluster kernel (csrc/cheb_filter.cuh); fp32 blocks, TF32 products."""
    _require_cuda(G, "cheb_filter")
    n, b = Y0.shape
    steps = len(a)
    bufs = [Y0.contiguous().clone(), torch.empty_like(Y0), torch.empty_like(Y0)]
    wsb = lib().tnb_cheb_filter_workspace_bytes(n, b)
    if wsb == 0:
        check(_lib.ERR_UNSUPPORTED)
    ws = _ws(wsb, G.device)
    fa, fb, fg = ((C.c_float * steps)(*[float(v) for v in x]) for x in (a, bc, g))
    with torch.cuda.device(G.device):
        check(lib().tnb_cheb_filter_f32(_ptr(G.contiguous()), n, b, _ptr(bufs[0]), _ptr(bufs[1]), _ptr(bufs[2]), steps,
                                        fa, fb, fg, _ptr(ws), ws.numel(), _stream()))
    return bufs[steps % 3]


def project(A: torch.Tensor, V: torch.Tensor, tensorcore: bool = False) -> torch.Tensor:
    _require_cuda(A, "project")
    A, V = A.contiguous(), V.contiguous()
    rows, n = A.shape
    assert V.shape[0] == n and V.dtype == A.dtype
    r = V.shape[1]
    Cc = torch.empty(rows, r, dtype=A.dtype, device=A.device)
    if tensorcore:
        L = lib()
        wsb = L.tnb_project_tc_workspace_bytes(n, r)
        if wsb == 0 or A.dtype != torch.float32:
            check(_lib.ERR_UNSUPPORTED)
        ws = _ws(wsb, A.device)
        with torch.cuda.device(A.device):
            check(L.tnb_project_tc_f32(_ptr(A), rows, n, _ptr(V), r, _ptr(Cc), _ptr(ws), ws.numel(), _stream()))
        return Cc
    with torch.cuda.device(A.device):
        check(lib().tnb_project(_dtype_code(A), _ptr(A), rows, n, _ptr(V), r, _ptr(Cc), _stream()))
    return Cc


def eigh_jacobi(G: torch.Tensor, return_sweeps: bool = False):
    _require_cuda(G, "eigh_jacobi")
    G = G.contiguous().double()
    n = G.shape[0]
    w = torch.empty(n, dtype=torch.float64, device=G.device)
    V = torch.empty(n, n, dtype=torch.float64, device=G.device)
    L = lib()
    wsb = L.tnb_eigh_workspace_bytes(n)
    if wsb == 0:
        check(_lib.ERR_UNSUPPORTED)
    ws = _ws(wsb, G.device)
    with torch.cuda.device(G.device):
        check(L.tnb_eigh_jacobi(_ptr(G), n, _ptr(w), _ptr(V), _ptr(ws), ws.numel(), _stream()))
    if return_sweeps:  # the kernel leaves its sweep count right behind the (256-byte aligned) scratch matrices
        npad = n + (n & 1)
        off = (2 * npad * (npad + 8) * 8 + 255) // 256 * 256
        return w, V, int(ws[off: off + 4].view(torch.int32).item())
    return w, V


def eig_topk(G: torch.Tensor, k: int, b: int = 0, tol: float = 1e-6):
    _require_cuda(G, "eig_topk")
    G = G.contiguous().double()
    n = G.shape[0]
    L = lib()
    wsb = L.tnb_eig_topk_workspace_bytes(n, k, b)
    ws = _ws(wsb, G.device)
    bb = b if b > 0 else min(n, min(256, max(2 * k, k + 16)))
    w = torch.empty(bb, dtype=torch.float64, device=G.device)
    V = torch.empty(n, bb, dtype=torch.float64, device=G.device)
    info = (C.c_double * 4)()
    with torch.cuda.device(G.device):
        check(L.tnb_eig_topk(_ptr(G), n, k, b, float(tol), _ptr(w), _ptr(V), _ptr(ws), ws.numel(), info, _stream()))
    return w, V, dict(products=int(info[0]), outer=int(info[1]), converged=int(info[2]))


def tt_relative_error(data: torch.Tensor, cores: Sequence[torch.Tensor]) -> float:
    """‖data − TT(cores)‖_F / ‖data‖_F, fp64 accumulation on the device (metrics.py:135-151)."""
    _require_cuda(data, "tt_relative_error")
    data = data.contiguous()
    cores = [c.contiguous() for c in cores]
    N = data.dim()
    code = _dtype_code(data)
    ranks = [cores[0].shape[0]] + [c.shape[2] for c in cores]
    L = lib()
    sh, rk = i64(list(data.shape)), i32(ranks)
    wsb = L.tnb_tt_relative_error_workspace_bytes(code, N, sh, rk)
    if wsb == 0:
        check(_lib.ERR_UNSUPPORTED)
    ws = _ws(wsb, data.device)
    ptrs = (C.c_void_p * N)(*[c.data_ptr() for c in cores])
    res = (C.c_double * 1)()
    with torch.cuda.device(data.device):
        check(L.tnb_tt_relative_error(code, _ptr(data), ptrs, N, sh, rk, _ptr(ws), ws.numel(), res, _stream()))
    return float(res[0])
