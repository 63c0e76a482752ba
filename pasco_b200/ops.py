"""Tensor-level wrappers and autograd Functions over the C-ABI (include/pasco_sm100.h).

Everything here runs on CUDA through libpasco_sm100.so; torch supplies device memory, the
current stream and the autograd graph.  Row indices are int32, −1 = no row.
"""
from __future__ import annotations

import ctypes as C
import weakref
from typing import List, Optional, Sequence, Tuple

import torch

from . import _lib
from ._lib import call as _raw_call, ptr, int_array, load


def call(name, *args):
    global CALLS
    CALLS += 1
    _raw_call(name, *args)

_PRECISION = 3          # 3 = bf16x3 split ("fp32" parity mode), 1 = plain bf16 operands
_FORCE_SIMT = False     # validation switch: run every conv on the CUDA-core path
_SIMT_KINDS = None      # validation switch: subset of {'fwd','dgrad','wgrad'} forced onto the CUDA-core path
_SPLIT_K = True          # few-tile / many-offset convs (dense bottleneck) are split over the offsets
_FUSE_BN_STATS = True    # forward convs leave their output's column statistics for the BatchNorm that follows
_PENDING_STATS = None
_USE_PLANES = True      # gathered convs (K > 1) read pre-split bf16 planes with zero-fill cp.async copies (k_conv_pl /
                        # k_wgrad_pl); False = the round-1 register-gather kernels (kept for cross-checks)
PROFILE = None          # bench.py sets this to a list: (kind, start_event, end_event, meta) per conv launch
PAIR_COUNTS = {}        # nbr.data_ptr() → 0-dim device tensor with the number of valid pairs (profiling only)
CALLS = 0               # number of C-ABI compute calls (each launches >= 1 kernel of ours)


def set_precision(mode) -> None:
    """'fp32' (bf16x3 split operands, ~2^-16 relative) or 'bf16' (single bf16 MMA)."""
    global _PRECISION
    _PRECISION = {"fp32": 3, "bf16": 1, 3: 3, 1: 1}[mode]
    # library ops on the path (cuDNN dense bottleneck, cuBLAS 1x1 convs / projections) follow the same contract:
    # fp32 mode = no TF32 anywhere, bf16 mode = TF32 allowed for the library GEMMs/convs
    torch.backends.cudnn.allow_tf32 = _PRECISION == 1
    torch.backends.cuda.matmul.allow_tf32 = _PRECISION == 1


def get_precision() -> int:
    return _PRECISION


def force_simt(flag: bool, kinds=None) -> None:
    global _FORCE_SIMT, _SIMT_KINDS
    _FORCE_SIMT = bool(flag) and kinds is None
    _SIMT_KINDS = set(kinds) if (flag and kinds is not None) else None


_ERR = {}               # device → int32[1] error flag set by kernels (rows outside a dense volume); read at sync points


def _err_flag(dev) -> torch.Tensor:
    f = _ERR.get(dev)
    if f is None:
        f = _ERR[dev] = torch.zeros(1, dtype=torch.int32, device=dev)
    return f


def raise_pending_errors(dev=None) -> None:
    """Raise what MinkowskiEngine raises immediately (a coordinate outside the dense volume) — called where the host
    already synchronises (compact), and by tests."""
    for d, f in list(_ERR.items()):
        if dev is not None and d != dev:
            continue
        code = int(f.item())
        if code != 0:
            f.zero_()
            if code == 2:
                raise RuntimeError("pasco_b200: a coordinate or batch index lies outside [-32768, 32767] "
                                   "(coordinate keys pack 16 bits per component)")
            raise RuntimeError("pasco_b200: a coordinate lies outside the requested dense volume "
                               "(SparseTensor.dense / to_sparse: check min_coordinate and shape)")


def _i32(t: torch.Tensor) -> torch.Tensor:
    return t if t.dtype == torch.int32 else t.to(torch.int32)


# ----------------------------------------------------------------------------------------------
# hash tables / coordinate maps
# ----------------------------------------------------------------------------------------------
class HashTable:
    """Open-addressing table key(b,x,y,z) → row, resident in HBM."""

    def __init__(self, keys: torch.Tensor, vals: torch.Tensor):
        self.keys, self.vals = keys, vals
        self.capacity = keys.numel()


def _capacity(n: int) -> int:
    cap = 64
    while cap < 2 * n:
        cap <<= 1
    return cap


def hash_insert(coords: torch.Tensor) -> Tuple[HashTable, torch.Tensor]:
    """Insert int32 [N,4] rows.  Returns (table, first_row[N]) — first_row[i] == i iff row i wins."""
    n = coords.shape[0]
    cap = _capacity(n)
    dev = coords.device
    keys = torch.full((cap,), -1, dtype=torch.int64, device=dev)                 # 0xFF… = empty
    vals = torch.full((cap,), 0x7F7F7F7F, dtype=torch.int32, device=dev)
    first = torch.empty(n, dtype=torch.int32, device=dev)
    call("pasco_hash_insert", ptr(coords), n, ptr(keys), ptr(vals), cap, ptr(first), ptr(_err_flag(dev)))
    return HashTable(keys, vals), first


def hash_lookup(table: HashTable, query: torch.Tensor) -> torch.Tensor:
    out = torch.empty(query.shape[0], dtype=torch.int32, device=query.device)
    call("pasco_hash_lookup", ptr(query), query.shape[0], ptr(table.keys), ptr(table.vals), table.capacity, ptr(out))
    return out


def hash_remap(table: HashTable, new_row: torch.Tensor) -> None:
    call("pasco_hash_remap", ptr(table.vals), table.capacity, ptr(new_row))


def coords_floor(coords: torch.Tensor, stride: Sequence[int]) -> torch.Tensor:
    out = torch.empty_like(coords)
    call("pasco_coords_floor", ptr(coords), coords.shape[0], int(stride[0]), int(stride[1]), int(stride[2]), ptr(out))
    return out


def coords_generate_k2(coords: torch.Tensor, out_stride: Sequence[int]) -> torch.Tensor:
    out = torch.empty(coords.shape[0] * 8, 4, dtype=torch.int32, device=coords.device)
    call("pasco_coords_generate_k2", ptr(coords), coords.shape[0], int(out_stride[0]), int(out_stride[1]),
         int(out_stride[2]), ptr(out))
    return out


def kernel_map_probe(out_coords: torch.Tensor, table: HashTable, kernel_size: int, step: Sequence[int]) -> torch.Tensor:
    """nbr[K, N_out] for an odd kernel; step = tensor_stride·dilation per axis."""
    n = out_coords.shape[0]
    nbr = torch.empty(kernel_size ** 3, n, dtype=torch.int32, device=out_coords.device)
    call("pasco_kernel_map_probe", ptr(out_coords), n, ptr(table.keys), ptr(table.vals), table.capacity,
         kernel_size, int(step[0]), int(step[1]), int(step[2]), ptr(nbr))
    return nbr


def kernel_map_box(out_coords: torch.Tensor, table: HashTable, ksize: Sequence[int], step: Sequence[int]) -> torch.Tensor:
    """nbr[kx*ky*kz, N_out] for an anisotropic odd box kernel (offsets x fastest)."""
    n = out_coords.shape[0]
    K = int(ksize[0]) * int(ksize[1]) * int(ksize[2])
    nbr = torch.empty(K, n, dtype=torch.int32, device=out_coords.device)
    call("pasco_kernel_map_box", ptr(out_coords), n, ptr(table.keys), ptr(table.vals), table.capacity,
         int(ksize[0]), int(ksize[1]), int(ksize[2]), int(step[0]), int(step[1]), int(step[2]), ptr(nbr))
    return nbr


def kernel_map_down(child_coords: torch.Tensor, parent_table: HashTable, n_parent: int, ks: int,
                    child_stride: Sequence[int], want_nbr: bool = True):
    n = child_coords.shape[0]
    dev = child_coords.device
    parent_of = torch.empty(n, dtype=torch.int32, device=dev)
    slot_of = torch.empty(n, dtype=torch.int32, device=dev)
    nbr = torch.full((ks ** 3, n_parent), -1, dtype=torch.int32, device=dev) if want_nbr else None
    call("pasco_kernel_map_down", ptr(child_coords), n, ptr(parent_table.keys), ptr(parent_table.vals),
         parent_table.capacity, ks, int(child_stride[0]), int(child_stride[1]), int(child_stride[2]),
         ptr(parent_of), ptr(slot_of), ptr(nbr), n_parent)
    return parent_of, slot_of, nbr


# ----------------------------------------------------------------------------------------------
# order-preserving compaction
# ----------------------------------------------------------------------------------------------
def compact(mask: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor, int]:
    """mask bool/uint8 [N] → (kept_rows[int32 N'], new_row[int32 N], N').  One host sync (N')."""
    n = mask.shape[0]
    dev = mask.device
    m8 = mask.to(torch.uint8) if mask.dtype != torch.uint8 else mask
    m8 = m8.contiguous()
    if n == 0:
        z = torch.zeros(0, dtype=torch.int32, device=dev)
        return z, z, 0
    nb = (n + 1023) // 1024
    counts = torch.empty(nb, dtype=torch.int32, device=dev)
    call("pasco_mask_block_counts", ptr(m8), n, ptr(counts))
    incl = torch.cumsum(counts, 0, dtype=torch.int32)       # ≤ ~1k elements: plumbing
    offsets = (incl - counts).contiguous()
    total = int(incl[-1].item())
    if _ERR:
        raise_pending_errors(dev)
    new_row = torch.empty(n, dtype=torch.int32, device=dev)
    kept = torch.empty(total, dtype=torch.int32, device=dev)
    call("pasco_mask_compact", ptr(m8), n, ptr(offsets), ptr(new_row), ptr(kept))
    return kept, new_row, total


def gather_coords(coords: torch.Tensor, rows: torch.Tensor) -> torch.Tensor:
    out = torch.empty(rows.shape[0], 4, dtype=torch.int32, device=coords.device)
    call("pasco_gather_coords", ptr(coords), ptr(rows), rows.shape[0], ptr(out))
    return out


def _gather_rows(src: torch.Tensor, rows: torch.Tensor) -> torch.Tensor:
    out = torch.empty(rows.shape[0], src.shape[1], dtype=torch.float32, device=src.device)
    call("pasco_gather_rows", ptr(src), ptr(rows), rows.shape[0], src.shape[1], ptr(out))
    return out


def _scatter_rows(src: torch.Tensor, rows: torch.Tensor, dst: torch.Tensor, accumulate: bool) -> None:
    call("pasco_scatter_rows", ptr(src), ptr(rows), rows.shape[0], src.shape[1], ptr(dst), int(accumulate))


class GatherRows(torch.autograd.Function):
    """out[r] = src[rows[r]] (rows unique or −1).  Backward scatters into a zero tensor."""

    @staticmethod
    def forward(ctx, src, rows):
        ctx.save_for_backward(rows)
        ctx.n_src = src.shape[0]
        return _gather_rows(src.contiguous().float(), rows)

    @staticmethod
    def backward(ctx, g):
        (rows,) = ctx.saved_tensors
        gin = torch.zeros(ctx.n_src, g.shape[1], dtype=torch.float32, device=g.device)
        _scatter_rows(g.contiguous(), rows, gin, False)
        return gin, None


class UnionAdd(torch.autograd.Function):
    """out = zeros[N_out]; out[:N_a] = a; out[rows_b] += b   (coordinate-union add, decoder_v3.py:163)."""

    @staticmethod
    def forward(ctx, a, b, rows_b, n_out):
        ctx.save_for_backward(rows_b)
        ctx.na = a.shape[0]
        out = torch.zeros(n_out, a.shape[1], dtype=torch.float32, device=a.device)
        out[: a.shape[0]].copy_(a)
        _scatter_rows(b.contiguous(), rows_b, out, True)
        return out

    @staticmethod
    def backward(ctx, g):
        (rows_b,) = ctx.saved_tensors
        g = g.contiguous()
        return g[: ctx.na], _gather_rows(g, rows_b), None, None


# ----------------------------------------------------------------------------------------------
# dense <-> sparse
# ----------------------------------------------------------------------------------------------
def _geom(min_c, stride):
    return int_array(min_c), int_array(stride)


class ToDense(torch.autograd.Function):
    @staticmethod
    def forward(ctx, feats, coords, min_c, stride, shape):
        B, Cc, X, Y, Z = shape
        dense = torch.zeros(shape, dtype=torch.float32, device=feats.device)
        mc, st = _geom(min_c, stride)
        call("pasco_to_dense", ptr(feats.contiguous()), ptr(coords), feats.shape[0], Cc, mc, st, ptr(dense), B, X, Y, Z,
             ptr(_err_flag(feats.device)))
        ctx.save_for_backward(coords)
        ctx.meta = (tuple(min_c), tuple(stride), tuple(shape))
        return dense

    @staticmethod
    def backward(ctx, g):
        (coords,) = ctx.saved_tensors
        min_c, stride, shape = ctx.meta
        return from_dense_raw(g.contiguous(), coords, min_c, stride), None, None, None, None


def from_dense_raw(dense: torch.Tensor, coords: torch.Tensor, min_c, stride) -> torch.Tensor:
    B, Cc, X, Y, Z = dense.shape
    feats = torch.empty(coords.shape[0], Cc, dtype=torch.float32, device=dense.device)   # out-of-volume rows read as 0
    mc, st = _geom(min_c, stride)
    call("pasco_from_dense", ptr(dense), ptr(coords), coords.shape[0], Cc, mc, st, ptr(feats), B, X, Y, Z,
         ptr(_err_flag(dense.device)))
    return feats


class FromDense(torch.autograd.Function):
    @staticmethod
    def forward(ctx, dense, coords, min_c, stride):
        ctx.save_for_backward(coords)
        ctx.meta = (tuple(min_c), tuple(stride), tuple(dense.shape))
        return from_dense_raw(dense.contiguous().float(), coords, min_c, stride)

    @staticmethod
    def backward(ctx, g):
        (coords,) = ctx.saved_tensors
        min_c, stride, shape = ctx.meta
        B, Cc, X, Y, Z = shape
        dense = torch.zeros(shape, dtype=torch.float32, device=g.device)
        mc, st = _geom(min_c, stride)
        call("pasco_to_dense", ptr(g.contiguous()), ptr(coords), g.shape[0], Cc, mc, st, ptr(dense), B, X, Y, Z, None)
        return dense, None, None, None


def dense_occupancy(dense: torch.Tensor) -> torch.Tensor:
    B, Cc = dense.shape[:2]
    cells = dense[0, 0].numel()
    mask = torch.empty(B * cells, dtype=torch.uint8, device=dense.device)
    call("pasco_dense_occupancy", ptr(dense), B, Cc, cells, ptr(mask))
    return mask


# ----------------------------------------------------------------------------------------------
# sparse convolution
# ----------------------------------------------------------------------------------------------
class KernelMap:
    """Neighbour tables of one (in_map, out_map, kernel) triple, both directions.

    nbr   int32 [K, N_out]: input row feeding output row o through offset k (forward / wgrad)
    nbr_t int32 [K, N_in] : output row fed by input row i, table row k' using weight slice koff_t[k']
    """

    def __init__(self, nbr, n_in, n_out, nbr_t=None, koff_t=None, build_t=None):
        self.nbr, self.n_in, self.n_out = nbr, n_in, n_out
        if PROFILE is not None:
            PAIR_COUNTS[nbr.data_ptr()] = (nbr >= 0).sum()
        self._nbr_t, self._koff_t, self._build_t = nbr_t, koff_t, build_t
        self.K = nbr.shape[0]

    def transposed(self):
        if self._nbr_t is None:
            self._nbr_t, self._koff_t = self._build_t()
        return self._nbr_t, self._koff_t


class PackedWeights:
    """UMMA shared-memory images of one weight tensor (forward and transposed), owned by the module
    that owns the parameter and re-packed whenever the parameter changes (optimizer step, load_state_dict,
    device move).  Keyed by (data_ptr, version, shape) of that one parameter only."""

    def __init__(self):
        self._slots = {}

    def get(self, weight: torch.Tensor, transpose: bool) -> torch.Tensor:
        tag = (weight.data_ptr(), weight._version, tuple(weight.shape))
        hit = self._slots.get(transpose)
        if hit is not None and hit[0] == tag:
            return hit[1]
        K, Cin, Cout = weight.shape
        nbytes = _lib.load().pasco_conv_packed_bytes(K, Cin, Cout)
        buf = torch.empty(nbytes, dtype=torch.uint8, device=weight.device)
        call("pasco_conv_pack_weights", ptr(weight.detach().contiguous()), K, Cin, Cout, int(transpose), ptr(buf))
        self._slots[transpose] = (tag, buf)
        return buf


def use_planes(flag: bool) -> None:
    global _USE_PLANES
    _USE_PLANES = bool(flag)


def split_planes(x: torch.Tensor, scale=None, shift=None, act: int = 0):
    """x fp32 [N,C] → (hi, lo) bf16 planes [N,C] of act(x*scale+shift) with x ≈ hi + lo; lo is None in bf16 mode."""
    n, c = x.shape
    hi = torch.empty(n, c, dtype=torch.bfloat16, device=x.device)
    lo = torch.empty(n, c, dtype=torch.bfloat16, device=x.device) if _PRECISION == 3 else None
    call("pasco_split_planes", ptr(x), n, c, 0, ptr(scale), ptr(shift), act, ptr(hi), ptr(lo))
    return hi, lo


def _planes_ok(c_contract: int, kk: int, nbr) -> bool:
    return _USE_PLANES and nbr is not None and kk > 1 and c_contract % 64 == 0


def _tc_ok(c_contract: int, c_out: int, K: int, kind: str = "fwd") -> bool:
    if _SIMT_KINDS is not None and kind in _SIMT_KINDS:
        return False
    return (not _FORCE_SIMT) and c_contract % 64 == 0 and c_out % 16 == 0 and 16 <= c_out <= 256 and K <= 1024


def conv_apply(feats: torch.Tensor, weight: torch.Tensor, nbr: Optional[torch.Tensor], n_out: int,
               transpose_w: bool, koff: Optional[Sequence[int]], bias: Optional[torch.Tensor] = None,
               in_scale=None, in_shift=None, in_act: int = 0, packs: Optional[PackedWeights] = None,
               want_stats: bool = False, planes=None, planes_out: Optional[list] = None) -> torch.Tensor:
    """out[o] = Σ_k act(feats·scale+shift)[nbr[k,o]] @ Wk, Wk = W[koff[k]] (transposed when transpose_w).
    want_stats: the kernel's epilogue also accumulates the column sums / sums of squares of `out` (the training-mode
    BatchNorm statistics of the layer that follows) and leaves them for BatchNormAct (see take_pending_stats).
    planes: (hi, lo) bf16 planes of act(feats·scale+shift) if the caller already has them; planes_out: a list that
    receives the planes this call made (the backward pass reuses them for the weight gradient)."""
    K, Cin, Cout = weight.shape
    c_contract, c_out = (Cout, Cin) if transpose_w else (Cin, Cout)
    assert feats.shape[1] == c_contract
    feats = feats.contiguous()
    out = torch.empty(n_out, c_out, dtype=torch.float32, device=feats.device)
    kk = nbr.shape[0] if nbr is not None else 1
    koff_arr = int_array(koff) if koff is not None else None
    prof = PROFILE
    if prof is not None:
        ev0 = torch.cuda.Event(enable_timing=True)
        ev0.record()
    global _PENDING_STATS
    _PENDING_STATS = None            # statistics of an earlier launch never survive another convolution
    use_tc = _tc_ok(c_contract, c_out, kk, "dgrad" if transpose_w else "fwd")
    split_k = use_tc and _SPLIT_K and load().pasco_conv_splitk_workspace_bytes(kk, n_out, c_out) > 0
    path = "simt"
    if use_tc and not split_k and _planes_ok(c_contract, kk, nbr):
        path = "planes"
        hi, lo = planes if planes is not None else split_planes(feats, in_scale, in_shift, in_act)
        if planes_out is not None:
            planes_out.append((hi, lo))
        stats = None
        if want_stats and _FUSE_BN_STATS and n_out >= 4096:
            stats = torch.zeros(2, c_out, dtype=torch.float64, device=feats.device)
        call("pasco_conv_forward_planes", ptr(hi), ptr(lo), feats.shape[0], ptr(nbr), kk, n_out, c_contract, c_out,
             ptr((packs or PackedWeights()).get(weight, transpose_w)), koff_arr, ptr(bias), ptr(stats), ptr(out),
             _PRECISION, 0, 0)
        if stats is not None:
            _PENDING_STATS = (weakref.ref(out), out.data_ptr(), out._version, tuple(out.shape), stats)
    elif use_tc and _SPLIT_K and (ws_bytes := load().pasco_conv_splitk_workspace_bytes(kk, n_out, c_out)) > 0:
        path = "splitk"
        ws = torch.empty(ws_bytes // 4, dtype=torch.float32, device=feats.device)
        call("pasco_conv_forward_splitk", ptr(feats), feats.shape[0], ptr(nbr), kk, n_out, c_contract, c_out,
             ptr((packs or PackedWeights()).get(weight, transpose_w)), koff_arr, ptr(bias), ptr(in_scale), ptr(in_shift), in_act,
             ptr(out), _PRECISION, 0, 0, ptr(ws), ws_bytes)
    elif use_tc:
        path = "regs"
        stats = None
        if want_stats and _FUSE_BN_STATS and n_out >= 4096:
            stats = torch.zeros(2, c_out, dtype=torch.float64, device=feats.device)
        call("pasco_conv_forward_tc", ptr(feats), feats.shape[0], ptr(nbr), kk, n_out, c_contract, c_out,
             ptr((packs or PackedWeights()).get(weight, transpose_w)), koff_arr, ptr(bias), ptr(in_scale), ptr(in_shift), in_act,
             ptr(stats), ptr(out), _PRECISION, 0, 0)
        if stats is not None:
            _PENDING_STATS = (weakref.ref(out), out.data_ptr(), out._version, tuple(out.shape), stats)
    else:
        assert in_scale is None and in_act == 0, "fused prologue needs the tensor-core path"
        if nbr is None:
            nbr = torch.arange(n_out, dtype=torch.int32, device=feats.device).view(1, -1)
        call("pasco_conv_forward_simt", ptr(feats), ptr(nbr), kk, n_out, c_contract, c_out,
             ptr(weight.detach().contiguous()), int(transpose_w), koff_arr, ptr(bias), ptr(out))
    if prof is not None:
        ev1 = torch.cuda.Event(enable_timing=True)
        ev1.record()
        prof.append(("dgrad" if transpose_w else "fwd", ev0, ev1,
                     dict(n_in=feats.shape[0], n_out=n_out, K=kk, Cin=c_contract, Cout=c_out,
                          pairs=PAIR_COUNTS.get(nbr.data_ptr()) if nbr is not None else None,
                          tc=use_tc, precision=_PRECISION, path=path)))
    return out


def take_pending_stats(x: torch.Tensor) -> Optional[torch.Tensor]:
    """Column statistics a convolution epilogue produced for exactly this tensor (same storage, shape and version —
    any in-place change since bumps the version), or None.  Consumed once."""
    global _PENDING_STATS
    pend, _PENDING_STATS = _PENDING_STATS, None
    if pend is None:
        return None
    ref, dptr, ver, shape, stats = pend
    # the producing tensor must still be alive (a freed block re-used at the same address is another tensor) and x must
    # be that storage, unmodified
    if ref() is not None and dptr == x.data_ptr() and ver == x._version and shape == tuple(x.shape):
        return stats
    return None


def split_k(flag: bool) -> None:
    global _SPLIT_K
    _SPLIT_K = bool(flag)


def fuse_bn_stats(flag: bool) -> None:
    global _FUSE_BN_STATS
    _FUSE_BN_STATS = bool(flag)


def _workspace(nbytes: int, device) -> torch.Tensor:
    """Scratch memory for a library call, from the caching allocator (stream-ordered like the call itself)."""
    return torch.empty(max(nbytes // 4, 1), dtype=torch.float32, device=device)


def conv_wgrad(feats: torch.Tensor, gout: torch.Tensor, nbr: Optional[torch.Tensor], K: int, Cin: int, Cout: int,
               in_scale=None, in_shift=None, in_act: int = 0, in_planes=None, g_planes=None) -> torch.Tensor:
    """in_planes / g_planes: (hi, lo) bf16 planes of act(feats·scale+shift) and of gout when the caller has them
    (the forward pass made the former, the input-gradient launch of the same backward the latter)."""
    n_out = gout.shape[0]
    dW = torch.zeros(K, Cin, Cout, dtype=torch.float32, device=feats.device)
    feats, gout = feats.contiguous(), gout.contiguous()
    prof = PROFILE
    if prof is not None:
        ev0 = torch.cuda.Event(enable_timing=True)
        ev0.record()
    tc = _tc_ok(Cin, 64, 1, "wgrad") and Cin % 64 == 0 and Cout % 64 == 0 and Cout <= 256
    path = "planes" if tc and _planes_ok(Cin, K, nbr) else ("regs" if tc else "simt")
    if tc:
        # per-CTA partial dW, summed in a fixed order by the library (dW does not change from run to run)
        nbytes = _lib.load().pasco_conv_wgrad_workspace_bytes(K, n_out, Cin, Cout)
        ws = _workspace(nbytes, feats.device)
    if tc and _planes_ok(Cin, K, nbr):
        ih, il = in_planes if in_planes is not None else split_planes(feats, in_scale, in_shift, in_act)
        gh, gl = g_planes if g_planes is not None else split_planes(gout)
        call("pasco_conv_wgrad_planes", ptr(ih), ptr(il), feats.shape[0], ptr(nbr), K, n_out, Cin, Cout, ptr(gh), ptr(gl),
             ptr(dW), _PRECISION, 0, 0, ptr(ws), nbytes)
    elif tc:
        call("pasco_conv_wgrad_tc", ptr(feats), feats.shape[0], ptr(nbr), K, n_out, Cin, Cout, ptr(gout),
             ptr(in_scale), ptr(in_shift), in_act, ptr(dW), _PRECISION, 0, 0, ptr(ws), nbytes)
    else:
        assert in_scale is None and in_act == 0
        if nbr is None:
            nbr = torch.arange(n_out, dtype=torch.int32, device=feats.device).view(1, -1)
        nbytes = _lib.load().pasco_conv_wgrad_simt_workspace_bytes(K, n_out, Cin, Cout)
        ws = _workspace(nbytes, feats.device)
        call("pasco_conv_wgrad_simt", ptr(feats), ptr(nbr), K, n_out, Cin, Cout, ptr(gout), ptr(dW), ptr(ws), nbytes)
    if prof is not None:
        ev1 = torch.cuda.Event(enable_timing=True)
        ev1.record()
        prof.append(("wgrad", ev0, ev1, dict(n_in=feats.shape[0], n_out=n_out, K=K, Cin=Cin, Cout=Cout,
                                             pairs=PAIR_COUNTS.get(nbr.data_ptr()) if nbr is not None else None,
                                             tc=tc, precision=_PRECISION, path=path)))
    return dW


class SparseConv(torch.autograd.Function):
    """ME ConvolutionForward/Backward over a cached KernelMap."""

    @staticmethod
    def forward(ctx, feats, weight, bias, kmap: KernelMap, packs: Optional[PackedWeights] = None):
        ctx.kmap = kmap
        ctx.packs = packs
        ctx.has_bias = bias is not None
        made = []
        out = conv_apply(feats, weight, kmap.nbr, kmap.n_out, False, None,
                         bias.view(-1).contiguous() if bias is not None else None, packs=packs, want_stats=True,
                         planes_out=made)
        # the weight gradient gathers the same rows: keep the planes the forward made instead of splitting again
        ctx.n_planes = 0
        if made and weight.requires_grad:
            hi, lo = made[0]
            ctx.n_planes = 1 if lo is None else 2
            ctx.save_for_backward(feats, weight, *([hi] if lo is None else [hi, lo]))
        else:
            ctx.save_for_backward(feats, weight)
        return out

    @staticmethod
    def backward(ctx, g):
        feats, weight = ctx.saved_tensors[:2]
        in_planes = None
        if ctx.n_planes:
            in_planes = (ctx.saved_tensors[2], ctx.saved_tensors[3] if ctx.n_planes == 2 else None)
        kmap: KernelMap = ctx.kmap
        g = g.contiguous()
        gin = gw = gb = None
        K, Cin, Cout = weight.shape
        g_planes = None
        if _planes_ok(Cout, K, kmap.nbr) and _tc_ok(Cout, Cin, K, "dgrad") and \
                (ctx.needs_input_grad[0] and ctx.needs_input_grad[1]):
            g_planes = split_planes(g)          # one split of the output gradient serves dgrad (gather) and wgrad (B operand)
        if ctx.needs_input_grad[0]:
            nbr_t, koff_t = kmap.transposed()
            gin = conv_apply(g, weight, nbr_t, kmap.n_in, True, koff_t, packs=ctx.packs, planes=g_planes)
        if ctx.needs_input_grad[1]:
            gw = conv_wgrad(feats, g, kmap.nbr, K, Cin, Cout, in_planes=in_planes, g_planes=g_planes)
        if ctx.has_bias and ctx.needs_input_grad[2]:
            gb = g.sum(0, keepdim=True)
        return gin, gw, gb, None, None


# ----------------------------------------------------------------------------------------------
# pooling / reductions
# ----------------------------------------------------------------------------------------------
class MaxPoolRows(torch.autograd.Function):
    @staticmethod
    def forward(ctx, feats, parent_of, n_parent):
        feats = feats.contiguous()
        out = torch.full((n_parent, feats.shape[1]), float("-inf"), dtype=torch.float32, device=feats.device)
        call("pasco_maxpool_forward", ptr(feats), ptr(parent_of), feats.shape[0], feats.shape[1], ptr(out))
        ctx.save_for_backward(feats, parent_of, out)
        return out

    @staticmethod
    def backward(ctx, g):
        feats, parent_of, out = ctx.saved_tensors
        p = parent_of.long()
        hit = feats == out[p]
        return torch.where(hit, g[p], torch.zeros_like(feats)), None, None


class ScatterMax(torch.autograd.Function):
    @staticmethod
    def forward(ctx, src, index, n_seg):
        src = src.contiguous().float()
        index = index.contiguous().long()
        out = torch.full((n_seg, src.shape[1]), float("-inf"), dtype=torch.float32, device=src.device)
        arg = torch.full((n_seg, src.shape[1]), src.shape[0], dtype=torch.int64, device=src.device)
        call("pasco_scatter_max", ptr(src), ptr(index), src.shape[0], src.shape[1], ptr(out), n_seg, ptr(arg))
        ctx.save_for_backward(arg)
        ctx.n_src = src.shape[0]
        ctx.mark_non_differentiable(arg)
        return out, arg

    @staticmethod
    def backward(ctx, g, _):
        (arg,) = ctx.saved_tensors
        gsrc = torch.zeros(ctx.n_src + 1, g.shape[1], dtype=g.dtype, device=g.device)
        gsrc.scatter_(0, arg, g)            # arg == n_src for empty segments → dummy row
        return gsrc[: ctx.n_src], None, None


def scatter_max(src: torch.Tensor, index: torch.Tensor, dim: int = 0, out=None, dim_size: Optional[int] = None):
    """torch_scatter.scatter_max(src[P,C], index[P], dim=0) → (values, argmax); empty segments → 0
    (pasco/models/unet3d_sparse_v2.py:79)."""
    if dim != 0 or src.ndim != 2 or out is not None:
        raise NotImplementedError("pasco_b200.scatter_max: only src[P,C], dim=0 is on PaSCo's path")
    n_seg = int(index.max().item()) + 1 if dim_size is None else int(dim_size)
    return ScatterMax.apply(src, index, n_seg)


# ----------------------------------------------------------------------------------------------
# fused BatchNorm (+ activation) over rows
# ----------------------------------------------------------------------------------------------
def column_stats(x: torch.Tensor) -> torch.Tensor:
    """float64 [2, C]: column sums and sums of squares."""
    stats = torch.zeros(2, x.shape[1], dtype=torch.float64, device=x.device)
    call("pasco_bn_stats", ptr(x), x.shape[0], x.shape[1], ptr(stats))
    return stats


def affine_act(x, scale, shift, act: int = 0, residual=None):
    y = torch.empty_like(x)
    call("pasco_affine_act", ptr(x), x.shape[0], x.shape[1], ptr(scale), ptr(shift), act, ptr(residual), ptr(y))
    return y


def _bn_forward_coefs(x, gamma, beta, eps, group, running_mean, running_var, momentum):
    """Training-mode BatchNorm coefficients of x [N, C]: column statistics (left by the producing convolution's epilogue
    when available, else one reduction pass; summed over `group` for SyncBatchNorm) → one coefficient kernel that also
    updates the running statistics.  Returns scale, shift (y = x*scale + shift), mean, rstd, count_dev."""
    n, c = x.shape
    dev = x.device
    stats = take_pending_stats(x)
    if stats is None:
        stats = column_stats(x)
    count_dev = None
    if group is not None:
        packed = torch.cat([stats.view(-1), torch.full((1,), float(n), dtype=torch.float64, device=dev)])
        torch.distributed.all_reduce(packed, group=group)
        stats, count_dev = packed[:-1].contiguous(), packed[-1:].contiguous()
    scale, shift, mean, rstd = (torch.empty(c, dtype=torch.float32, device=dev) for _ in range(4))
    call("pasco_bn_finalize", ptr(stats), ptr(count_dev), C.c_double(float(n)), c, ptr(gamma), ptr(beta), C.c_float(eps),
         C.c_float(momentum if momentum is not None else 0.1), ptr(scale), ptr(shift), ptr(mean), ptr(rstd),
         ptr(running_mean), ptr(running_var))
    return scale, shift, mean, rstd, count_dev


def _bn_backward(gy, x, gamma, scale, shift, mean, rstd, count_dev, act, group, n):
    """Gradient of y = act(BN(x)) w.r.t. x, gamma, beta: one reduce pass → one coefficient kernel → one apply pass."""
    gy = gy.contiguous()
    c = x.shape[1]
    dev = x.device
    sums = torch.zeros(2, c, dtype=torch.float64, device=dev)
    call("pasco_bn_bwd_reduce", ptr(gy), ptr(x), x.shape[0], c, ptr(scale), ptr(shift), act, ptr(sums))
    div = 1.0
    if group is not None:
        # sums are global after the all-reduce; every rank then holds the global dgamma/dbeta, and the gradient
        # all-reduce (mean over ranks) of the data-parallel step leaves them unchanged only if divided here
        torch.distributed.all_reduce(sums, group=group)
        div = float(torch.distributed.get_world_size(group))
    ca, cb, cc, gg, gb = (torch.empty(c, dtype=torch.float32, device=dev) for _ in range(5))
    call("pasco_bn_bwd_coefs", ptr(sums), ptr(count_dev), C.c_double(float(n)), c, ptr(gamma), ptr(mean), ptr(rstd),
         C.c_float(div), ptr(ca), ptr(cb), ptr(cc), ptr(gg), ptr(gb))
    gx = torch.empty_like(x)
    call("pasco_bn_bwd_apply", ptr(gy), ptr(x), x.shape[0], c, ptr(scale), ptr(shift), act,
         ptr(ca), ptr(cb), ptr(cc), ptr(gx))
    return gx, gg, gb


class BatchNormAct(torch.autograd.Function):
    """y = act(BN(x)) with training-mode batch statistics over all rows (optionally summed over ranks =
    SyncBatchNorm).  Forward: column sums → one coefficient kernel (scale/shift, mean/rstd, running statistics) →
    one apply pass; backward: one reduce pass → one coefficient kernel → one apply pass."""

    @staticmethod
    def forward(ctx, x, gamma, beta, eps, act, group, running_mean=None, running_var=None, momentum=0.1):
        x = x.contiguous()
        scale, shift, mean, rstd, count_dev = _bn_forward_coefs(x, gamma, beta, eps, group, running_mean, running_var, momentum)
        y = affine_act(x, scale, shift, act)
        ctx.save_for_backward(x, gamma, scale, shift, mean, rstd, count_dev)
        ctx.act, ctx.group, ctx.n = act, group, x.shape[0]
        return y

    @staticmethod
    def backward(ctx, gy):
        x, gamma, scale, shift, mean, rstd, count_dev = ctx.saved_tensors
        gx, gg, gb = _bn_backward(gy, x, gamma, scale, shift, mean, rstd, count_dev, ctx.act, ctx.group, ctx.n)
        return gx, gg, gb, None, None, None, None, None, None


class BNActConv(torch.autograd.Function):
    """out = SparseConv(act(BN(x)))  as ONE autograd node on the plane-gather path: the BatchNorm apply pass writes the
    normalised activations directly as bf16 planes (hi [+ lo]) — the only form the convolution and its weight gradient
    read — so the fp32 copy of act(BN(x)) never exists: same HBM bytes as the plain apply pass, no separate split pass,
    and the planes double as the saved tensor of the backward pass (pre-activation residual blocks, mink.py:618-658:
    BN → ReLU → conv, twice per block)."""

    @staticmethod
    def forward(ctx, x, gamma, beta, weight, bias, eps, act, group, running_mean, running_var, momentum, kmap, packs):
        x = x.contiguous()
        scale, shift, mean, rstd, count_dev = _bn_forward_coefs(x, gamma, beta, eps, group, running_mean, running_var, momentum)
        hi, lo = split_planes(x, scale, shift, act)
        out = conv_apply(x, weight, kmap.nbr, kmap.n_out, False, None, bias.view(-1).contiguous() if bias is not None else None,
                         packs=packs, want_stats=True, planes=(hi, lo))
        ctx.kmap, ctx.packs, ctx.has_bias = kmap, packs, bias is not None
        ctx.act, ctx.group, ctx.n, ctx.has_lo = act, group, x.shape[0], lo is not None
        ctx.save_for_backward(x, gamma, scale, shift, mean, rstd, count_dev, weight, hi, *([lo] if lo is not None else []))
        return out

    @staticmethod
    def backward(ctx, g):
        x, gamma, scale, shift, mean, rstd, count_dev, weight, hi = ctx.saved_tensors[:9]
        lo = ctx.saved_tensors[9] if ctx.has_lo else None
        kmap = ctx.kmap
        g = g.contiguous()
        K, Cin, Cout = weight.shape
        g_planes = split_planes(g)
        nbr_t, koff_t = kmap.transposed()
        gy = conv_apply(g, weight, nbr_t, kmap.n_in, True, koff_t, packs=ctx.packs, planes=g_planes)
        gw = conv_wgrad(x, g, kmap.nbr, K, Cin, Cout, in_planes=(hi, lo), g_planes=g_planes) if ctx.needs_input_grad[3] else None
        gb = g.sum(0, keepdim=True) if ctx.has_bias and ctx.needs_input_grad[4] else None
        gx, gg, gbeta = _bn_backward(gy, x, gamma, scale, shift, mean, rstd, count_dev, ctx.act, ctx.group, ctx.n)
        return gx, gg, gbeta, gw, gb, None, None, None, None, None, None, None, None


def bn_act_conv(bn, x: torch.Tensor, act: int, group, weight, bias, kmap: "KernelMap", packs=None) -> torch.Tensor:
    """conv(act(BatchNorm(x))) — fused (BNActConv) when the layer runs on the plane-gather tensor-core path in training
    mode, the two separate nodes otherwise."""
    K, Cin, Cout = weight.shape
    fused = (bn.training and bn.running_mean is not None and x.is_cuda and _planes_ok(Cin, kmap.K, kmap.nbr)
             and _tc_ok(Cin, Cout, kmap.K, "fwd") and _tc_ok(Cout, Cin, kmap.K, "dgrad") and _tc_ok(Cin, 64, 1, "wgrad")
             and Cout % 64 == 0 and Cout <= 256
             and not (_SPLIT_K and load().pasco_conv_splitk_workspace_bytes(kmap.K, kmap.n_out, Cout) > 0)
             and not (_SPLIT_K and load().pasco_conv_splitk_workspace_bytes(kmap.K, kmap.n_in, Cin) > 0))
    if not fused:
        return SparseConv.apply(batchnorm_rows(bn, x, act, group), weight, bias, kmap, packs)
    with torch.no_grad():
        bn.num_batches_tracked += 1
    mom = bn.momentum if bn.momentum is not None else 1.0 / float(bn.num_batches_tracked)
    return BNActConv.apply(x, bn.weight, bn.bias, weight, bias, bn.eps, act, group, bn.running_mean, bn.running_var, mom,
                           kmap, packs)


ACT_NONE, ACT_RELU, ACT_LEAKY = 0, 1, 2


def _act_torch(z: torch.Tensor, act: int) -> torch.Tensor:
    if act == ACT_RELU:
        return torch.relu(z)
    if act == ACT_LEAKY:
        return torch.nn.functional.leaky_relu(z, 0.01)
    return z


def batchnorm_rows(bn, x: torch.Tensor, act: int = ACT_NONE, group=None) -> torch.Tensor:
    """act(BatchNorm(x)) over the rows of x [N, C] with the parameters / running statistics of a torch
    BatchNorm1d/3d/SyncBatchNorm module `bn`.  Training (or no running statistics): batch statistics through the fused
    kernels (ops.BatchNormAct).  Eval: a per-channel affine — through one fused kernel when no gradient is needed, through
    differentiable torch ops otherwise (frozen-BN fine-tuning keeps its graph)."""
    use_batch_stats = bn.training or bn.running_mean is None
    if use_batch_stats:
        if bn.training and bn.num_batches_tracked is not None:
            with torch.no_grad():
                bn.num_batches_tracked += 1
        gamma = bn.weight if bn.weight is not None else torch.ones(x.shape[1], device=x.device)
        beta = bn.bias if bn.bias is not None else torch.zeros(x.shape[1], device=x.device)
        mom = bn.momentum
        if mom is None and bn.num_batches_tracked is not None:          # cumulative moving average
            mom = 1.0 / float(bn.num_batches_tracked)
        rm, rv = (bn.running_mean, bn.running_var) if bn.training else (None, None)
        return BatchNormAct.apply(x, gamma, beta, bn.eps, act, group, rm, rv, mom)
    w = bn.weight if bn.weight is not None else 1.0
    scale = w * torch.rsqrt(bn.running_var + bn.eps)
    shift = (bn.bias if bn.bias is not None else 0.0) - bn.running_mean * scale
    if torch.is_grad_enabled() and (x.requires_grad or scale.requires_grad or shift.requires_grad):
        return _act_torch(x * scale + shift, act)
    return affine_act(x.contiguous(), scale.contiguous(), shift.contiguous(), act)


# ----------------------------------------------------------------------------------------------
# masked cross-attention of a few queries over all voxels (MaskPLS decoder)
# ----------------------------------------------------------------------------------------------
def pack_mask_bits(mask: torch.Tensor) -> torch.Tensor:
    """bool [Q,P] (True = masked) → int32 bit rows [Q, 2*ceil(P/64)], keys beyond P masked."""
    Q, P = mask.shape
    W = 2 * ((P + 63) // 64)
    pad = W * 32 - P
    m = torch.nn.functional.pad(mask, (0, pad), value=True) if pad else mask
    sh = torch.arange(32, device=mask.device, dtype=torch.int64)
    words = (m.view(Q, W, 32).to(torch.int64) << sh).sum(-1)
    return words.to(torch.int32).contiguous()


class MaskedCrossAttention(torch.autograd.Function):
    """out[q] = concat_h softmax_v(scale·q_h·k_h[v] | mask[q,v]) · v_h[v]  — blocks.py:73-92 with the mask of
    transformer_predictor_v2.py:220-289.  Forward: two streaming tcgen05 passes; backward: one streaming pass with
    five tcgen05 GEMM groups per 64-key tile that recomputes the probabilities from the saved log-sum-exp (xattn.cu)."""

    @staticmethod
    def forward(ctx, q, k, v, mask, heads: int):
        q, k, v = q.contiguous().float(), k.contiguous().float(), v.contiguous().float()
        Q, HD = q.shape
        P = k.shape[0]
        D = HD // heads
        scale = float(D) ** -0.5
        bits = pack_mask_bits(mask) if mask is not None else None
        out = torch.zeros(Q, HD, dtype=torch.float32, device=q.device)
        lse = torch.empty(heads, Q, dtype=torch.float32, device=q.device)
        nbytes = _lib.load().pasco_xattn_workspace_bytes(Q, P, heads, D)
        ws = torch.empty(max(nbytes // 4, 1), dtype=torch.float32, device=q.device)
        call("pasco_xattn_forward", ptr(q), ptr(k), ptr(v), ptr(bits), Q, P, heads, D, C.c_float(scale), ptr(out),
             ptr(lse), ptr(ws), nbytes)
        ctx.save_for_backward(q, k, v, bits, out, lse)
        ctx.heads, ctx.scale = heads, scale
        return out

    @staticmethod
    def backward(ctx, go):
        q, k, v, bits, out, lse = ctx.saved_tensors
        H, scale = ctx.heads, ctx.scale
        Q, HD = q.shape
        P = k.shape[0]
        go = go.contiguous().float()
        dq = torch.zeros_like(q)
        dk, dv = torch.empty_like(k), torch.empty_like(v)
        nbytes = _lib.load().pasco_xattn_workspace_bytes(Q, P, H, HD // H)
        ws = _workspace(nbytes, q.device)
        call("pasco_xattn_backward", ptr(q), ptr(k), ptr(v), ptr(bits), ptr(lse), ptr(out), ptr(go), Q, P, H, HD // H,
             C.c_float(scale), ptr(dq), ptr(dk), ptr(dv), ptr(ws), nbytes)
        return dq, dk, dv, None, None


# ----------------------------------------------------------------------------------------------
# dense Linear layers on the tensor-core conv kernel (K = 1, identity rows, column chunks <= 256)
# ----------------------------------------------------------------------------------------------
def _data_ptr_at(t: torch.Tensor, col: int) -> int:
    return t.data_ptr() + 4 * col


def _linear_tc_ok(n_rows: int, cin: int, cout: int) -> bool:
    return (not _FORCE_SIMT) and n_rows >= 4096 and cin % 64 == 0 and cout % 64 == 0


def _gemm_rows(x: torch.Tensor, w_nk: torch.Tensor, bias: Optional[torch.Tensor], out: torch.Tensor) -> None:
    """out[:, :] = x @ w_nkᵀ (+ bias) with w_nk [N, K] row-major (torch Linear layout), N in chunks of <= 256 columns."""
    global _PENDING_STATS
    _PENDING_STATS = None
    n_rows, kdim = x.shape
    N = w_nk.shape[0]
    assert x.is_contiguous() and out.is_contiguous() and kdim % 64 == 0 and N % 16 == 0
    for c0 in range(0, N, 256):
        cw = min(256, N - c0)
        wchunk = w_nk[c0:c0 + cw].contiguous()                       # [cw, K]  == ME layout [1, Cin'=cw, Cout'=K]
        packed = PackedWeights().get(wchunk.view(1, cw, kdim), True)  # B[n][k] = w[n][k]
        b = bias[c0:c0 + cw].contiguous() if bias is not None else None
        call("pasco_conv_forward_tc", ptr(x), n_rows, None, 1, n_rows, kdim, cw, ptr(packed), None, ptr(b), None, None, 0,
             None, C.c_void_p(_data_ptr_at(out, c0)), _PRECISION, 0, N)


class LinearTC(torch.autograd.Function):
    """y = x @ Wᵀ + b for tall x [N, Cin] on the tcgen05 conv kernel (bf16x3 / bf16 like the convolutions) instead of
    an fp32 CUDA-core library GEMM.  W is [Cout, Cin] (torch Linear layout)."""

    @staticmethod
    def forward(ctx, x, weight, bias):
        x = x.contiguous().float()
        y = torch.empty(x.shape[0], weight.shape[0], dtype=torch.float32, device=x.device)
        _gemm_rows(x, weight.detach(), bias.detach() if bias is not None else None, y)
        ctx.save_for_backward(x, weight)
        ctx.has_bias = bias is not None
        return y

    @staticmethod
    def backward(ctx, gy):
        x, weight = ctx.saved_tensors
        gy = gy.contiguous().float()
        gx = gw = gb = None
        if ctx.needs_input_grad[0]:
            gx = torch.empty_like(x)
            _gemm_rows(gy, weight.detach().t().contiguous(), None, gx)          # gx = gy @ W
        if ctx.needs_input_grad[1]:
            cout, cin = weight.shape
            gw = torch.empty(cout, cin, dtype=torch.float32, device=x.device)
            for c0 in range(0, cin, 256):                                        # dW[:, c0:c0+cw] = gyᵀ @ x[:, c0:c0+cw]
                cw = min(256, cin - c0)
                dw = torch.zeros(1, cout, cw, dtype=torch.float32, device=x.device)
                nbytes = _lib.load().pasco_conv_wgrad_workspace_bytes(1, gy.shape[0], cout, cw)
                ws = _workspace(nbytes, x.device)
                call("pasco_conv_wgrad_tc", ptr(gy), gy.shape[0], None, 1, gy.shape[0], cout, cw,
                     C.c_void_p(_data_ptr_at(x, c0)), None, None, 0, ptr(dw), _PRECISION, 0, cin, ptr(ws), nbytes)
                gw[:, c0:c0 + cw] = dw[0]
        if ctx.has_bias and ctx.needs_input_grad[2]:
            gb = gy.sum(0)
        return gx, gw, gb


def linear(x: torch.Tensor, weight: torch.Tensor, bias: Optional[torch.Tensor] = None) -> torch.Tensor:
    """F.linear for [N, Cin] inputs: tensor-core path when the shape allows (N >= 4096, Cin, Cout multiples of 64),
    the fp32 library GEMM otherwise (exactly what MinkowskiEngine does for 1x1 convolutions)."""
    if x.is_cuda and x.ndim == 2 and _linear_tc_ok(x.shape[0], weight.shape[1], weight.shape[0]):
        return LinearTC.apply(x, weight, bias)
    return torch.nn.functional.linear(x, weight, bias)


# ----------------------------------------------------------------------------------------------
# evaluation sweeps (pasco_b200/evaluation.py): outputs are accumulated into caller-zeroed tensors
# ----------------------------------------------------------------------------------------------
EVAL_ERR_ID = 3         # _err_flag code of the evaluation kernels: a label or segment id outside its table


def eval_ssc(prob: torch.Tensor, label: torch.Tensor, bounds: torch.Tensor, counts: torch.Tensor,
             sums: torch.Tensor) -> None:
    """prob float32 [K, cells], label uint8 [cells]; counts int64 [K*K + 4*(n_bins+1)], sums float64
    [2*(n_bins+1) + 2] (layouts: include/pasco_sm100.h)."""
    K, cells = prob.shape
    n_bins = bounds.numel() - 1
    nbytes = _lib.load().pasco_eval_ssc_workspace_bytes(cells, n_bins)
    ws = _workspace(nbytes, prob.device)
    call("pasco_eval_ssc", ptr(prob), ptr(label), cells, K, ptr(bounds), n_bins, ptr(counts), ptr(sums), ptr(ws), nbytes,
         ptr(_err_flag(prob.device)))


def eval_pairs(pred_id: torch.Tensor, row_cell: torch.Tensor, gt_id: torch.Tensor, label: torch.Tensor, n_gt: int,
               n_pred: int, table: torch.Tensor) -> None:
    """table int64 [(n_gt+1) * (n_pred+1)] += intersections of GT ids (gt_id int32 [cells]) and predicted ids
    (pred_id int32 [N] at cells row_cell int64 [N]) over known cells."""
    call("pasco_eval_pairs", ptr(pred_id), ptr(row_cell), pred_id.numel(), ptr(gt_id), ptr(label), gt_id.numel(),
         int(n_gt), int(n_pred), ptr(table), ptr(_err_flag(gt_id.device)))


def eval_calib(conf: torch.Tensor, pred_id: torch.Tensor, row_cell: torch.Tensor, gt_id: torch.Tensor,
               label: torch.Tensor, match: torch.Tensor, bounds: torch.Tensor, counts: torch.Tensor,
               sums: torch.Tensor) -> None:
    """Binned calibration of the rows' mask confidences; match int32 [n_pred+1] = GT id matched to each predicted id."""
    n_bins = bounds.numel() - 1
    nbytes = _lib.load().pasco_eval_calib_workspace_bytes(conf.numel(), n_bins)
    ws = _workspace(nbytes, conf.device)
    call("pasco_eval_calib", ptr(conf), ptr(pred_id), ptr(row_cell), conf.numel(), ptr(gt_id), ptr(label), gt_id.numel(),
         ptr(match), match.numel() - 1, ptr(bounds), n_bins, ptr(counts), ptr(sums), ptr(ws), nbytes,
         ptr(_err_flag(conf.device)))
