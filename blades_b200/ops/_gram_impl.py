"""ctypes launcher of the tcgen05 split-K Gram kernel (csrc/cuda/gram_tcgen05.cu)."""
from __future__ import annotations

import ctypes as C
from typing import List, Optional, Sequence, Tuple

import torch

from . import _loader


class GramBlockDesc(C.Structure):
    _fields_ = [("base", C.c_void_p), ("ld", C.c_longlong), ("rows", C.c_int)]


def _pad8(n: int) -> int:
    return (n + 7) // 8 * 8


def _num_sms(device) -> int:
    return torch.cuda.get_device_properties(device).multi_processor_count


def launch_gram(blocks: Sequence[Tuple[int, int, int]], d: int, col0: int, col1: int, out: torch.Tensor,
                split3: bool, device) -> List[int]:
    """blocks: (base_ptr, ld_floats, rows).  Accumulates into ``out`` ([tile_rows, ld] fp32, zeroed by the
    caller) over coordinates [col0, col1).  Returns, per block, the first padded row index."""
    lib = _loader.cuda_lib()
    arr = (GramBlockDesc * len(blocks))()
    starts, row = [], 0
    for i, (ptr, ld, rows) in enumerate(blocks):
        arr[i].base, arr[i].ld, arr[i].rows = ptr, ld, rows
        starts.append(row)
        row += _pad8(rows)
    lib.bl_gram_tcgen05.argtypes = [C.c_void_p, C.c_int, C.c_longlong, C.c_longlong, C.c_longlong, C.c_void_p,
                                    C.c_int, C.c_int, C.c_int, C.c_void_p]
    code = lib.bl_gram_tcgen05(C.cast(arr, C.c_void_p), len(blocks), d, col0, col1, out.data_ptr(),
                               out.stride(0), 1 if split3 else 0, _num_sms(device), _loader.stream_ptr(device))
    if code == -7:                       # 3xTF32 staging does not fit in shared memory for this row count
        return None
    _loader.check(code, "gram_tcgen05")
    _loader.count_launch()
    return starts


def split_blocks(ptr: int, ld: int, rows: int, max_rows: int = 256) -> List[Tuple[int, int, int]]:
    out, r = [], 0
    while r < rows:
        k = min(max_rows, rows - r)
        out.append((ptr + r * ld * 4, ld, k))
        r += k
    return out


#: one Gram pass reads at most this many rows (each block padded to 8) in at most this many blocks
MAX_PADDED_ROWS = 512
MAX_BLOCKS = 9


def padded_rows(row_counts: Sequence[int]) -> int:
    return sum(_pad8(r) for r in row_counts)


def gram_pass(blocks: Sequence[Tuple[int, int, int]], d: int, col0: int, col1: int, device,
              extra: Optional[torch.Tensor] = None, split3: bool = True, tf32_fallback: bool = False,
              scratch: Optional[torch.Tensor] = None):
    """One Gram pass over the row blocks ``(base_ptr, ld_floats, rows)`` (+ the rows of ``extra``, ``[e, d]``) and
    coordinates ``[col0, col1)``.  Returns (padded accumulators ``[tile_rows, ld]``, logical -> padded row list), or
    None when the kernel does not apply: unaligned blocks, more rows or blocks than one pass takes, or -- unless
    ``tf32_fallback``, which relaunches in plain tf32 -- 3xTF32 staging that does not fit.  The accumulators are a
    zeroed view of ``scratch`` when given, a new zeroed tensor otherwise."""
    if any(ptr % 16 or ld % 4 for ptr, ld, _ in blocks):
        return None
    blocks = [b for blk in blocks for b in split_blocks(*blk)]
    buf = None
    if extra is not None:
        extra = extra.reshape(-1, d)
        ld = blocks[0][1]
        buf = torch.zeros(extra.shape[0], ld, device=device, dtype=torch.float32)
        buf[:, :d] = extra
        blocks += split_blocks(buf.data_ptr(), ld, extra.shape[0])
    total_pad = padded_rows([b[2] for b in blocks])
    if total_pad > MAX_PADDED_ROWS or len(blocks) > MAX_BLOCKS:
        return None
    tile_rows = (total_pad + 127) // 128 * 128
    ldg = (total_pad + 31) // 32 * 32
    if scratch is None:
        out = torch.zeros(tile_rows, ldg, device=device, dtype=torch.float32)
    else:
        out = scratch[: tile_rows * ldg].view(tile_rows, ldg)
        out.zero_()
    starts = launch_gram(blocks, d, col0, col1, out, split3, device)
    if starts is None and tf32_fallback:
        starts = launch_gram(blocks, d, col0, col1, out, False, device)
    if starts is None:
        return None
    idx = []
    for (_, _, rows), s in zip(blocks, starts):
        idx += list(range(s, s + rows))
    return out, idx


def symmetrised(out: torch.Tensor, idx: Sequence[int]) -> torch.Tensor:
    """The logical ``[n, n]`` Gram ``out[idx][:, idx]`` of a pass's padded accumulators, symmetrised."""
    idx_t = torch.tensor(idx, device=out.device)
    G = out[idx_t][:, idx_t]
    return 0.5 * (G + G.T)
