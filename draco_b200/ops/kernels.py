"""Python launchers for the sm_100a step-path kernels (thin: build the argument struct, launch on the current stream).

Every function takes either torch CUDA tensors or raw device addresses (``int``) -- peer-mapped and multicast pointers
coming from the symmetric-memory runtime are plain integers.  Nothing here falls back to PyTorch ops: if the CUDA
library is missing the call raises (see ``_native.cuda``).
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional, Sequence, Union

import torch

from .. import _native as N
from ..parallel.arena import ArenaLayout

Addr = Union[int, torch.Tensor, None]

_sm_count = {}


def addr(x: Addr) -> Optional[int]:
    if x is None:
        return None
    if isinstance(x, torch.Tensor):
        return x.data_ptr()
    return int(x)


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def sm_count(device=None) -> int:
    dev = torch.cuda.current_device() if device is None else torch.device(device).index
    if dev not in _sm_count:
        _sm_count[dev] = torch.cuda.get_device_properties(dev).multi_processor_count
    return _sm_count[dev]


def stream_grid(layout: ArenaLayout, ctas_per_sm: int = 8) -> int:
    return max(1, min(layout.ntiles, sm_count() * ctas_per_sm))


def _flag_list(flags: Sequence[Addr]) -> N.FlagList:
    fl = N.FlagList()
    assert len(flags) <= N.MAX_DST
    for i, f in enumerate(flags):
        fl.ptr[i] = addr(f)
    fl.n = len(flags)
    return fl


# ------------------------------------------------------------------------------------------------ push (K1/K2/K11)
def push_encode(layout: ArenaLayout, g32: Sequence[Addr], g16: Sequence[Addr], dst: Addr, *, step_ptr: Addr,
                worker: int, done_counter: Addr, flag: Addr = None, coef: Optional[Sequence[complex]] = None,
                adv_bitmap: Addr = None, adv_len: int = 0, attack: int = 0, magnitude: float = -100.0, seed: int = 428,
                local_copy: Addr = None, grid: Optional[int] = None, tile_range: Optional[tuple] = None,
                src_table: Addr = None) -> None:
    """Fused encode + adversary + store into ``dst`` (a peer pointer) + release flag.  ``coef`` given => cyclic encode
    of ``len(coef)`` gradient streams into an interleaved complex64 slot.  ``tile_range=(t0, t1)`` pushes one bucket."""
    a = N.PushArgs()
    if src_table is not None:
        # zero-copy mode: `src_table` is a device int64 [R, ntensors] table of per-tensor gradient pointers
        R = len(coef) if coef is not None else 1
        a.src_table = addr(src_table)
    else:
        R = len(g32)
        needs_bf16 = any(sp.is_bf16 for sp in layout.specs)
        for k in range(R):
            a.g32[k] = addr(g32[k])
            a.g16[k] = addr(g16[k]) if g16 and g16[k] is not None else None
            if needs_bf16 and not a.g16[k]:
                raise ValueError("layout has bf16 tensors: push_encode needs the bf16 gradient arena of every stream")
    assert 1 <= R <= N.MAX_R
    a.R = R
    a.cyclic = 1 if coef is not None else 0
    if coef is not None:
        assert len(coef) == R
        for k, c in enumerate(coef):
            a.coef_re[k] = float(complex(c).real)
            a.coef_im[k] = float(complex(c).imag)
    a.dst = addr(dst)
    dev = torch.device("cuda", torch.cuda.current_device())
    a.tv = layout.tile_view(dev)
    a.adv_bitmap = addr(adv_bitmap)
    a.adv_len = adv_len if adv_bitmap is not None else 0
    a.step_ptr = addr(step_ptr)
    a.worker = worker
    a.attack = attack
    a.magnitude = magnitude
    a.seed = seed
    a.done_counter = addr(done_counter)
    a.flag = addr(flag)
    a.local_copy = addr(local_copy)
    ntiles = layout.ntiles
    if tile_range is not None:
        a.tile_begin, a.tile_end = int(tile_range[0]), int(tile_range[1])
        ntiles = a.tile_end - a.tile_begin
    N.check(N.cuda().drc_push_encode(C.byref(a), grid or max(1, min(ntiles, sm_count() * 8)), _stream()), "push_encode")


def omniscient(grad_in: Addr, slot_stride: int, honest_mask: int, worker: int, magnitude: float, total: int, *,
               step_ptr: Addr, done_counter: Addr, flag: Addr = None) -> None:
    a = N.OmniArgs(addr(grad_in), slot_stride, honest_mask, worker, magnitude, total, addr(done_counter), addr(flag),
                   addr(step_ptr))
    grid = max(1, min(sm_count() * 8, total // (N.THREADS * 4)))
    N.check(N.cuda().drc_omniscient(C.byref(a), grid, _stream()), "omniscient")


def collude(layout: ArenaLayout, grad_in: Addr, slot_stride: int, P: int, adv_bitmap: Addr, adv_len: int, step_ptr: Addr,
            mode: int, param: float, tile_range: Optional[tuple] = None) -> None:
    """Colluding attack at the PS (csrc/cuda/collude.cu): the slots set in ``adv_bitmap[*step_ptr % adv_len]`` are all
    overwritten with ``mu - param * sigma`` (``mode`` = ATTACK_ALIE) or ``-param * mu`` (ATTACK_IPM) of the other slots.
    ``tile_range=(t0, t1)`` processes one bucket; an empty one launches nothing (tile_end 0 means "to the end" in the kernel)."""
    dev = torch.device("cuda", torch.cuda.current_device())
    t0, t1 = tile_range if tile_range is not None else (0, 0)
    if tile_range is not None and t1 <= t0:
        return
    a = N.CollusionArgs(addr(grad_in), slot_stride, P, layout.tile_view(dev), int(t0), int(t1), addr(adv_bitmap), adv_len,
                        addr(step_ptr), mode, param)
    ntiles = (t1 - t0) if tile_range is not None else layout.ntiles
    N.check(N.cuda().drc_collude(C.byref(a), max(1, min(ntiles, sm_count() * 8)), _stream()), "collude")


# ------------------------------------------------------------------------------------------------ vote (K3)
def vote(layout: ArenaLayout, grad_in: Addr, slot_stride: int, group_table: torch.Tensor, neq_mask: torch.Tensor,
         winner_slot: torch.Tensor, winner_member: Optional[torch.Tensor] = None, tile_range: Optional[tuple] = None,
         tensor_range: Optional[tuple] = None) -> None:
    """Exact-equality majority vote.  ``group_table``: int32 [G, max_r] worker slots (-1 padded); ``neq_mask``: zeroed
    uint32/int32 [G, T] scratch (left zeroed again on return); ``winner_slot``: int32 [G, T] out."""
    G, max_r = group_table.shape
    dev = group_table.device
    t0, t1 = tile_range if tile_range is not None else (0, 0)
    va = N.VoteArgs(addr(grad_in), slot_stride, group_table.data_ptr(), G, max_r, layout.tile_view(dev), neq_mask.data_ptr(),
                    int(t0), int(t1))
    ntiles = (t1 - t0) if tile_range is not None else layout.ntiles
    N.check(N.cuda().drc_vote_compare(C.byref(va), max(1, min(ntiles, sm_count() * 8)), _stream()), "vote_compare")
    q0, q1 = tensor_range if tensor_range is not None else (0, 0)
    ra = N.ResolveArgs(neq_mask.data_ptr(), group_table.data_ptr(), G, max_r, layout.ntensors, winner_slot.data_ptr(),
                       addr(winner_member), neq_mask.data_ptr(), int(q0), int(q1))
    N.check(N.cuda().drc_vote_resolve(C.byref(ra), _stream()), "vote_resolve")


# ------------------------------------------------------------------------------------------------ update (K7/K8/K9)
def aggregate_update(layout: ArenaLayout, grad_in: Addr, slot_stride: int, *, params: Addr, momentum: Addr, hp: Addr,
                     step_ptr: Addr, done_counter: Addr, K: int, scale: float, select: Addr = None,
                     recomb: Addr = None, first_step: int = 1, grad_out: Addr = None, mc_params: Addr = None,
                     dst: Sequence[Addr] = (), flags: Sequence[Addr] = (), grid: Optional[int] = None,
                     tile_range: Optional[tuple] = None, weights: Addr = None, exp_avg_sq: Addr = None,
                     max_exp_avg_sq: Addr = None, trim: Optional[int] = None) -> None:
    """Fused aggregate (select-sum, cyclic recombination, real per-tensor ``weights`` [T, K], or with ``trim`` the coordinate-wise
    trimmed sum: per element, the K slot values sorted ascending (NaN last) without the ``trim`` lowest and highest, summed) +
    optimizer step (SGD-momentum, or Adam / AMSGrad when the hyper-parameter block says so: ``momentum`` = first moment,
    ``exp_avg_sq`` / ``max_exp_avg_sq`` = second moment / its running maximum) + parameter broadcast + flags.  Everything is
    multiplied by ``scale`` before the optimizer step: 1 / (K - 2 trim) makes the trimmed sum a trimmed mean / median."""
    a = N.UpdateArgs()
    a.mode = 1 if recomb is not None else (2 if weights is not None else (3 if trim is not None else 0))
    if weights is not None:
        assert recomb is None and select is None and trim is None
        recomb = weights
    if trim is not None:
        assert recomb is None and select is None
        a.trim = trim
    a.grad_in = addr(grad_in)
    a.slot_stride = slot_stride
    a.select = addr(select)
    a.K = K
    a.scale = scale
    a.recomb = addr(recomb)
    dev = torch.device("cuda", torch.cuda.current_device())
    a.tv = layout.tile_view(dev)
    a.params = addr(params)
    a.momentum = addr(momentum)
    a.exp_avg_sq = addr(exp_avg_sq)
    a.max_exp_avg_sq = addr(max_exp_avg_sq)
    a.hp = addr(hp)
    a.step_ptr = addr(step_ptr)
    a.first_step = first_step
    a.grad_out = addr(grad_out)
    a.mc_params = addr(mc_params)
    assert len(dst) <= N.MAX_DST
    for i, d in enumerate(dst):
        a.dst[i] = addr(d)
    a.ndst = len(dst)
    a.done_counter = addr(done_counter)
    a.flags = _flag_list(flags)
    ntiles = layout.ntiles
    if tile_range is not None:
        a.tile_begin, a.tile_end = int(tile_range[0]), int(tile_range[1])
        ntiles = a.tile_end - a.tile_begin
    N.check(N.cuda().drc_aggregate_update(C.byref(a), grid or max(1, min(ntiles, sm_count() * 8)), _stream()), "aggregate_update")


def stream_push(src: Addr, dst: Addr, nbytes: Addr, nbytes_out: Addr = None, *, step_ptr: Addr, done_counter: Addr, flag: Addr = None,
                grid: int = 16) -> None:
    """Store ``*nbytes`` bytes (device scalar) of a packed stream into a peer buffer and raise the step-stamped flag
    (compressed push of the fused transport, csrc/cuda/codec.cu)."""
    a = N.StreamPushArgs(addr(src), addr(dst), addr(nbytes), addr(nbytes_out), addr(step_ptr), addr(done_counter), addr(flag))
    lib = N.cuda()
    if not getattr(lib, "_stream_push_ready", False):
        lib.drc_stream_push.argtypes = [C.c_void_p, C.c_int, N.ptr]
        lib.drc_stream_push.restype = C.c_int
        lib._stream_push_ready = True
    N.check(lib.drc_stream_push(C.byref(a), int(grid), _stream()), "stream_push")


def cast_params(layout: ArenaLayout, src: Addr, dst: Addr) -> None:
    dev = torch.device("cuda", torch.cuda.current_device())
    a = N.CastArgs(addr(src), addr(dst), layout.tile_view(dev))
    N.check(N.cuda().drc_cast_params(C.byref(a), stream_grid(layout), _stream()), "cast_params")


# ------------------------------------------------------------------------------------------------ flags
def wait_flags(flags: Sequence[Addr], step_ptr: Addr, addend: int, error: Addr, timeout_s: float = 30.0,
               stamps: Addr = None) -> None:
    a = N.WaitArgs()
    a.stamps = addr(stamps)
    assert len(flags) <= N.MAX_WORKERS
    for i, f in enumerate(flags):
        a.flags[i] = addr(f)
    a.n = len(flags)
    a.step_ptr = addr(step_ptr)
    a.addend = addend
    a.timeout_ns = int(timeout_s * 1e9)
    a.error = addr(error)
    N.check(N.cuda().drc_wait_flags(C.byref(a), _stream()), "wait_flags")


def set_flags(flags: Sequence[Addr], step_ptr: Addr, addend: int) -> None:
    a = N.SetFlagArgs(_flag_list(flags), addr(step_ptr), addend)
    N.check(N.cuda().drc_set_flags(C.byref(a), _stream()), "set_flags")


def stamp(ring: Addr, step_ptr: Addr, col: int) -> None:
    """ring[(step & 63)][col] = %globaltimer (ring: int64 [64, 8])."""
    lib = N.cuda()
    if not getattr(lib, "_stamp_ready", False):
        lib.drc_stamp.argtypes = [N.ptr, N.ptr, C.c_int, N.ptr]
        lib.drc_stamp.restype = C.c_int
        lib._stamp_ready = True
    N.check(lib.drc_stamp(addr(ring), addr(step_ptr), int(col), _stream()), "stamp")


def step_add(step_ptr: Addr, delta: int = 1) -> None:
    N.check(N.cuda().drc_step_add(addr(step_ptr), delta, _stream()), "step_add")


# ------------------------------------------------------------------------------------------------ cyclic decode (K4)
_epart_cache = {}


def cyclic_project(layout: ArenaLayout, R: Addr, slot_stride: int, n: int, f: Addr, E: torch.Tensor) -> None:
    """E[T, n, 2] (fp64) = R_i . f per tensor: per-tile partials, then a fixed-order fold per tensor (deterministic)."""
    key = (E.device, layout.ntiles, n)
    if key not in _epart_cache:
        _epart_cache[key] = torch.empty(layout.ntiles, n, 2, dtype=torch.float64, device=E.device)
    a = N.ProjectArgs(addr(R), slot_stride, n, addr(f), layout.tile_view(E.device), E.data_ptr(), _epart_cache[key].data_ptr())
    N.check(N.cuda().drc_cyclic_project(C.byref(a), stream_grid(layout), _stream()), "cyclic_project")


def cyclic_locate(E: torch.Tensor, n: int, s: int, recomb: torch.Tensor, healthy: Optional[torch.Tensor] = None,
                  flagged: Optional[torch.Tensor] = None, rel_tol: float = 1e-4) -> None:
    a = N.LocateArgs(E.data_ptr(), E.shape[0], n, s, rel_tol, recomb.data_ptr(), addr(healthy), addr(flagged))
    N.check(N.cuda().drc_cyclic_locate(C.byref(a), _stream()), "cyclic_locate")


# ------------------------------------------------------------------------------------------------ robust baselines (K5/K6)
class GeoMedianWorkspace:
    def __init__(self, layout: ArenaLayout, P: int, device):
        T = layout.ntensors
        self.median = layout.new_arena(device)
        self.weights = torch.zeros(T, P, dtype=torch.float32, device=device)
        self.done = torch.zeros(T, dtype=torch.int32, device=device)
        self.dist2 = torch.zeros(T, P, dtype=torch.float64, device=device)
        self.move2 = torch.zeros(T, 2, dtype=torch.float64, device=device)


def geometric_median(layout: ArenaLayout, grad_in: Addr, slot_stride: int, P: int, ws: GeoMedianWorkspace,
                     iters: int = 64, eps: float = 1e-6) -> torch.Tensor:
    """Per-tensor Weiszfeld geometric median of the P slots; result in ``ws.median`` (fp32 arena)."""
    lib = N.cuda()
    T = layout.ntensors
    dev = ws.median.device
    tv = layout.tile_view(dev)
    grid = stream_grid(layout)
    for it in range(iters + 1):
        pa = N.GeoMedPrepArgs(T, P, ws.dist2.data_ptr(), ws.move2.data_ptr(), ws.weights.data_ptr(), ws.done.data_ptr(), it, eps)
        N.check(lib.drc_geomed_prep(C.byref(pa), _stream()), "geomed_prep")
        if it == iters:
            break
        ga = N.GeoMedArgs(addr(grad_in), slot_stride, P, tv, ws.median.data_ptr(), ws.weights.data_ptr(), ws.done.data_ptr(),
                          ws.dist2.data_ptr(), ws.move2.data_ptr())
        N.check(lib.drc_geomed_iter(C.byref(ga), grid, _stream()), "geomed_iter")
    return ws.median


GEOMED_FAST_MAXP = 16


def geometric_median_weights(layout: ArenaLayout, grad_in: Addr, slot_stride: int, P: int, pair_d2: torch.Tensor,
                             weights: torch.Tensor, max_iter: int = 256, eps: float = 1e-10,
                             iters_out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Per-tensor geometric median as convex weights: ``median_t = sum_i weights[t, i] * slot_i`` (Weiszfeld run in weight
    space from the pairwise distances -- one pass over the slab; see csrc/cuda/robust.cu).  ``pair_d2``: zeroed fp64
    [T, P(P-1)/2] scratch (left zeroed); ``weights``: fp32 [T, P] out."""
    assert P <= GEOMED_FAST_MAXP
    lib = N.cuda()
    pa = N.PairDistArgs(addr(grad_in), slot_stride, P, layout.tile_view(weights.device), pair_d2.data_ptr())
    N.check(lib.drc_pair_dist(C.byref(pa), stream_grid(layout, 4), _stream()), "pair_dist")
    wa = N.GeoMedWeightsArgs(pair_d2.data_ptr(), layout.ntensors, P, max_iter, eps, weights.data_ptr(),
                             iters_out.data_ptr() if iters_out is not None else None)
    N.check(lib.drc_geomed_weights(C.byref(wa), _stream()), "geomed_weights")
    return weights


def krum_select(layout: ArenaLayout, grad_in: Addr, slot_stride: int, P: int, s: int, pair_d2: torch.Tensor,
                select: torch.Tensor, m: int = 1) -> None:
    """Krum (m = 1) or multi-Krum selection.  ``pair_d2``: zeroed fp64 [T, P*(P-1)/2] scratch (left zeroed); ``select``: int32
    [m, T] out, the m lowest-scoring slots of every tensor in ascending slot order ([T] is accepted for m = 1)."""
    assert 1 <= m <= P and select.numel() == m * layout.ntensors and select.dtype == torch.int32
    lib = N.cuda()
    pa = N.PairDistArgs(addr(grad_in), slot_stride, P, layout.tile_view(select.device), pair_d2.data_ptr())
    N.check(lib.drc_pair_dist(C.byref(pa), stream_grid(layout, 4), _stream()), "pair_dist")
    ka = N.KrumSelectArgs(pair_d2.data_ptr(), layout.ntensors, P, s, select.data_ptr(), m)
    N.check(lib.drc_krum_select(C.byref(ka), _stream()), "krum_select")


# ------------------------------------------------------------------------------------------------ GEMM (K10)
def gemm_bf16(A: torch.Tensor, B: torch.Tensor, *, a_mn: bool = False, b_mn: bool = False, out: Optional[torch.Tensor] = None,
              out_dtype: torch.dtype = torch.bfloat16, bias: Optional[torch.Tensor] = None, relu: bool = False,
              accumulate: bool = False, block_n: int = 0, cta_pair: Optional[bool] = None) -> torch.Tensor:
    """``C[M, N] = op(A) op(B)^T`` on tcgen05 tensor cores (``cta_pair``: force / forbid the cta_group::2 kernel; None = by size).

    K-major operands (default) are ``A[M, K]`` / ``B[N, K]``; with ``a_mn`` / ``b_mn`` the tensor passed is the
    transposed storage ``A[K, M]`` / ``B[K, N]`` (MN contiguous), so no transpose copy is ever needed.
    """
    assert A.dtype == torch.bfloat16 and B.dtype == torch.bfloat16 and A.is_cuda and B.is_cuda
    assert A.dim() == 2 and B.dim() == 2 and A.stride(1) == 1 and B.stride(1) == 1
    M, K = (A.shape[1], A.shape[0]) if a_mn else (A.shape[0], A.shape[1])
    Nn, Kb = (B.shape[1], B.shape[0]) if b_mn else (B.shape[0], B.shape[1])
    assert K == Kb, f"K mismatch {K} vs {Kb}"
    if out is None:
        out = torch.empty(M, Nn, dtype=out_dtype, device=A.device)
    assert out.shape == (M, Nn) and out.stride(1) == 1
    bias_f32 = bias.data_ptr() if bias is not None and bias.dtype == torch.float32 else None
    bias_b16 = bias.data_ptr() if bias is not None and bias.dtype == torch.bfloat16 else None
    # large K-major problems go to the CTA-pair kernel (tcgen05.mma.cta_group::2): measured 1.04x cuBLAS at 4096^3, 0.95x at
    # 16384 x 512 x 4608 vs 0.87x / 0.82x for the single-CTA kernel (profiles/gemm_bench_r2.json); small ones lose to it
    pair = os.environ.get("DRACO_GEMM_2CTA", "auto") if cta_pair is None else ("1" if cta_pair else "0")
    if (not a_mn and not b_mn and block_n in (0, 128, 256) and M >= 256 and Nn >= 128
            and (pair == "1" or (pair == "auto" and M >= 2048 and Nn >= 512 and K >= 1024))):
        return gemm2_bf16(A, B, out=out, bias=bias, relu=relu, accumulate=accumulate, block_n=block_n)
    code = N.cuda().drc_gemm_bf16(A.data_ptr(), A.stride(0), int(a_mn), B.data_ptr(), B.stride(0), int(b_mn), out.data_ptr(),
                                  out.stride(0), int(out.dtype == torch.float32), M, Nn, K, bias_f32, bias_b16, int(relu),
                                  int(accumulate), block_n, sm_count(A.device), A.device.index, _stream())
    N.check(code, "gemm_bf16")
    return out


def gemm2_bf16(A: torch.Tensor, B: torch.Tensor, *, out: Optional[torch.Tensor] = None, out_dtype: torch.dtype = torch.bfloat16,
               bias: Optional[torch.Tensor] = None, relu: bool = False, accumulate: bool = False, block_n: int = 0) -> torch.Tensor:
    """``C[M, N] = A[M, K] B[N, K]^T`` on CTA PAIRS (tcgen05.mma.cta_group::2, 256 x block_n tiles, csrc/cuda/gemm2_tcgen05.cu)."""
    assert A.dtype == torch.bfloat16 and B.dtype == torch.bfloat16 and A.is_cuda and A.dim() == 2 and B.dim() == 2
    assert A.stride(1) == 1 and B.stride(1) == 1 and A.shape[1] == B.shape[1]
    M, Kd, Nn = A.shape[0], A.shape[1], B.shape[0]
    if out is None:
        out = torch.empty(M, Nn, dtype=out_dtype, device=A.device)
    lib = N.cuda()
    if not getattr(lib, "_gemm2_ready", False):
        lib.drc_gemm2_bf16.argtypes = [N.ptr, N.i64, N.ptr, N.i64, N.ptr, N.i64] + [C.c_int] * 4 + [N.ptr, N.ptr] + [C.c_int] * 5 + [N.ptr]
        lib.drc_gemm2_bf16.restype = C.c_int
        lib._gemm2_ready = True
    bias_f32 = bias.data_ptr() if bias is not None and bias.dtype == torch.float32 else None
    bias_b16 = bias.data_ptr() if bias is not None and bias.dtype == torch.bfloat16 else None
    N.check(lib.drc_gemm2_bf16(A.data_ptr(), A.stride(0), B.data_ptr(), B.stride(0), out.data_ptr(), out.stride(0),
                               int(out.dtype == torch.float32), M, Nn, Kd, bias_f32, bias_b16, int(relu), int(accumulate), block_n,
                               sm_count(A.device), A.device.index, _stream()), "gemm2_bf16")
    return out


def gemm_supported(A: torch.Tensor, B: torch.Tensor) -> bool:
    """Shape/alignment gate of the TMA descriptors (16-byte rows and bases)."""
    return (A.is_cuda and A.dtype == torch.bfloat16 and B.dtype == torch.bfloat16 and A.stride(-1) == 1 and B.stride(-1) == 1
            and A.stride(0) % 8 == 0 and B.stride(0) % 8 == 0 and A.data_ptr() % 16 == 0 and B.data_ptr() % 16 == 0)
