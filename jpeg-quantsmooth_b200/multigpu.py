"""Geometry of an image sharded by MCU rows (SURVEY.md 8e), for callers that cut slabs
themselves: bench.py's multi-GPU arm, tools/run_configs.py and the tests.

The sharded run itself is the C slab engine (csrc/qs_cuda.cu run_slab / run_host_multi,
include/jpegqs_cuda.h "one image sharded by MCU rows").  Every rank owns a contiguous range of
MCU rows of every component; slabs are MCU aligned, so the luma, chroma and down-sampled luma
planes of a slab line up.  These functions state the same split as the engine's
jpegqs_cuda_run_host_multi, and the plane geometry its kernels use (include/jpegqs_cuda.h
jpegqs_cuda_plane_stride / _pad).
"""
from __future__ import annotations

from typing import List, Tuple

PLANE_PAD = 16


def plane_stride(wblk: int) -> int:
    return wblk * 8 + 2 * PLANE_PAD


def split_mcu_rows(total_mcu_rows: int, world: int) -> List[Tuple[int, int]]:
    """Contiguous [m0, m1) MCU-row ranges, sizes differing by at most one."""
    base, rem = divmod(total_mcu_rows, world)
    out, m = [], 0
    for r in range(world):
        n = base + (1 if r < rem else 0)
        out.append((m, m + n))
        m += n
    return out


def comp_block_rows(mcu_range: Tuple[int, int], v_samp: int, hblk: int) -> Tuple[int, int]:
    """Block rows of a component covered by an MCU-row range (libjpeg geometry: the last
    MCU row may be only partly present, image.blocks_for)."""
    return min(mcu_range[0] * v_samp, hblk), min(mcu_range[1] * v_samp, hblk)
