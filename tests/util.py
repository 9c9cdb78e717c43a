"""Shared helpers of the test-suite.

`apply_block` interprets a `pa_block_desc` (the strided-copy descriptor the
CUDA kernels execute) with NumPy, so the C++ planner can be checked against
the oracle on a CPU-only box.  It is a TEST interpreter of the descriptor
format, not a fallback of the product.
"""
from __future__ import annotations

import ctypes as C
import hashlib
import math
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import pencilarrays_b200 as pa  # noqa: E402
from oracle import pencil_oracle as O  # noqa: E402

DTYPES = {4: np.float32, 8: np.float64, 16: np.complex128, 2: np.uint16, 1: np.uint8}


def beq(a, b) -> bool:
    """Bit-exact comparison (NaN payloads and -0.0 included)."""
    a = np.ascontiguousarray(a)
    b = np.ascontiguousarray(b)
    return a.shape == b.shape and a.dtype.itemsize == b.dtype.itemsize and a.tobytes() == b.tobytes()


def golden_nbytes(z, k, r) -> int:
    """Length in bytes of the output of step k on rank r in a tests/golden fixture."""
    key = f"step{k}_rank{r}"
    return int(z[key + "_nbytes"]) if key + "_pos" in z.files else z[key].size


def matches_golden(z, k, r, got) -> bool:
    """`got` (the whole uint8 output of step k on rank r) against a tests/golden fixture:
    byte for byte where the fixture holds all of it; otherwise at the stored sample
    positions and through the SHA-256 of all bytes (see tests/golden/make_golden.py)."""
    key = f"step{k}_rank{r}"
    got = np.ascontiguousarray(got).view(np.uint8).reshape(-1)
    if key + "_pos" not in z.files:
        return got.tobytes() == z[key].tobytes()
    return (got.size == int(z[key + "_nbytes"]) and got[z[key + "_pos"]].tobytes() == z[key].tobytes()
            and hashlib.sha256(got.tobytes()).digest() == z[key + "_sha256"].tobytes())


def apply_block(desc, src_flat: np.ndarray, dst_flat: np.ndarray):
    """dst[off_d + sum k_i ds_i] = src[off_s + sum k_i ss_i] for k in the box."""
    nd = desc.nd
    ext = [desc.extent[i] for i in range(nd)]
    if any(e == 0 for e in ext):
        return
    it = src_flat.dtype.itemsize
    ss = [desc.src_stride[i] * it for i in range(nd)]
    ds = [desc.dst_stride[i] * it for i in range(nd)]
    s = np.lib.stride_tricks.as_strided(src_flat[desc.src_offset:], shape=ext, strides=ss,
                                        writeable=False)
    d = np.lib.stride_tricks.as_strided(dst_flat[desc.dst_offset:], shape=ext, strides=ds)
    d[...] = s


class EmuRank:
    """One emulated rank: Python-mirror objects + the oracle's view of the same rank."""

    def __init__(self, rank, nranks, pdims):
        self.comm = pa.Comm(rank, nranks)
        self.topo = pa.MPITopology(self.comm, pdims)


def make_ranks(pdims):
    n = math.prod(pdims)
    return [EmuRank(r, n, pdims) for r in range(n)]


def perm_of(p):
    return pa.NoPermutation() if p is None else pa.Permutation(*p)


def emulate_transpose_with_descriptors(plans, srcs, dsts, dtype):
    """Run pack -> exchange -> unpack for all emulated ranks using ONLY the C
    planner's descriptors/offsets.  `srcs`/`dsts`: flat NumPy arrays per rank.
    Returns (send_bufs, recv_bufs)."""
    n = len(plans)
    it = np.dtype(dtype).itemsize
    sends, recvs = [], []
    for r in range(n):
        info = plans[r].info
        sends.append(np.zeros(max(1, info.send_bytes // it), dtype=dtype))
        recvs.append(np.zeros(max(1, info.recv_bytes // it), dtype=dtype))
    if plans[0].info.dim == 0:
        for r in range(n):
            apply_block(plans[r].block(2), srcs[r], dsts[r])
        return sends, recvs
    nproc = plans[0].info.nproc
    for r in range(n):
        for p in range(1, nproc + 1):
            peer = plans[r].peer(p)
            apply_block(plans[r].block(0, p), srcs[r], recvs[r] if peer.is_self else sends[r])
    for r in range(n):
        for p in range(1, nproc + 1):
            peer = plans[r].peer(p)
            if peer.is_self:
                continue
            # the peer's receive slot for data coming from world rank r
            q = peer.world_rank
            for pp in range(1, nproc + 1):
                back = plans[q].peer(pp)
                if back.world_rank == plans[r].peer(plans[r].info.self_index).world_rank:
                    assert back.recv_count == peer.send_count
                    so, sc = peer.send_offset // it, peer.send_count // it
                    ro = back.recv_offset // it
                    recvs[q][ro:ro + sc] = sends[r][so:so + sc]
    for r in range(n):
        for p in range(1, nproc + 1):
            apply_block(plans[r].block(1, p), recvs[r], dsts[r])
    return sends, recvs


# (grid, size_global, [(decomp, perm), ...] chain, extra_dims, itemsize): the
# reference's own test cases (SURVEY.md §4) + the small BASELINE config
CASES = [
    # test/transpose.jl:24-60 -- x -> y -> z -> y -> x, uneven blocks
    dict(name="ref_transpose_2x2", grid=(2, 2), dims=(16, 21, 41), extra=(), it=8,
         chain=[((2, 3), None), ((1, 3), (2, 3, 1)), ((1, 2), (3, 2, 1)), ((1, 3), (2, 3, 1)),
                ((2, 3), None)]),
    dict(name="ref_transpose_3x2", grid=(3, 2), dims=(16, 21, 41), extra=(), it=8,
         chain=[((2, 3), None), ((1, 3), (2, 3, 1)), ((1, 2), (3, 2, 1)), ((1, 3), (2, 3, 1)),
                ((2, 3), None)]),
    dict(name="ref_transpose_4x2", grid=(4, 2), dims=(16, 21, 41), extra=(), it=8,
         chain=[((2, 3), None), ((1, 3), (2, 3, 1)), ((1, 2), (3, 2, 1))]),
    # test/transpose.jl:62-67 -- no permutation
    dict(name="ref_noperm", grid=(2, 2), dims=(16, 21, 41), extra=(), it=8,
         chain=[((2, 3), None), ((1, 3), None)]),
    # test/transpose.jl:69-74 -- unsorted decomp_dims (#57)
    dict(name="ref_unsorted", grid=(2, 3), dims=(16, 21, 41), extra=(), it=8,
         chain=[((2, 3), None), ((2, 1), None)]),
    # test/pencils.jl:460-480 -- extra dims (3,4), Float32
    dict(name="ref_extra_dims", grid=(2, 2), dims=(16, 21, 41), extra=(3, 4), it=4,
         chain=[((2, 3), None), ((1, 3), (2, 3, 1)), ((1, 2), (3, 2, 1))]),
    # test/pencils.jl:483-520 -- 1-D (slab) decomposition + local permute
    dict(name="ref_slab", grid=(4,), dims=(16, 21, 41), extra=(), it=4,
         chain=[((1,), None), ((2,), None), ((2,), (3, 2, 1))]),
    # test/pencils.jl:523-542 -- M = N, only the permutation changes, ComplexF32 (8 bytes)
    dict(name="ref_3d_decomp", grid=(2, 2, 1), dims=(16, 21, 41), extra=(), it=8,
         chain=[((1, 2, 3), None), ((1, 2, 3), (2, 3, 1))]),
    # test/array_types.jl:96-167 -- dims (20,16,4), slab, perm (2,3,1)
    dict(name="ref_array_types", grid=(3,), dims=(20, 16, 4), extra=(), it=8,
         chain=[((1,), None), ((2,), (2, 3, 1))]),
    # BASELINE.json configs[0]
    dict(name="baseline_cfg1", grid=(2, 1), dims=(64, 48, 32), extra=(), it=8,
         chain=[((2, 3), None), ((1, 3), (2, 1, 3))]),
    dict(name="baseline_cfg1_noperm", grid=(2, 1), dims=(64, 48, 32), extra=(), it=8,
         chain=[((2, 3), None), ((1, 3), None)]),
    # more processes than points along a dimension: empty blocks (Pencils.jl:193-218)
    dict(name="empty_blocks", grid=(5, 1), dims=(3, 7, 4), extra=(), it=8,
         chain=[((2, 3), None), ((1, 3), (2, 1, 3)), ((1, 2), (3, 2, 1))]),
    # ComplexF64 with PencilFFTs' usual permutations, 16-byte vectors
    dict(name="c128_fft_perms", grid=(2, 2), dims=(8, 12, 10), extra=(), it=16,
         chain=[((2, 3), None), ((1, 3), (2, 1, 3)), ((1, 2), (3, 2, 1))]),
    # 2-rank variants (what a 2-GPU box can run with real NCCL)
    dict(name="two_ranks_1x2", grid=(1, 2), dims=(16, 21, 41), extra=(), it=8,
         chain=[((2, 3), None), ((1, 3), (2, 3, 1)), ((1, 2), (3, 2, 1)), ((1, 3), (2, 3, 1)),
                ((2, 3), None)]),
    dict(name="two_ranks_2x1", grid=(2, 1), dims=(16, 21, 41), extra=(2,), it=16,
         chain=[((2, 3), None), ((1, 3), (2, 1, 3)), ((1, 2), (3, 2, 1)), ((1, 3), (2, 1, 3)),
                ((2, 3), None)]),
    dict(name="two_ranks_slab", grid=(2,), dims=(20, 16, 4), extra=(), it=4,
         chain=[((1,), None), ((2,), (2, 3, 1)), ((2,), (3, 2, 1)), ((3,), None)]),
    # BASELINE configs[4] in small: Float32, perms None -> (2,3,1) -> (3,1,2), grids (2,2) and (4,2)
    dict(name="cfg5_small_2x2", grid=(2, 2), dims=(32, 16, 24), extra=(), it=4,
         chain=[((2, 3), None), ((1, 3), (2, 3, 1)), ((1, 2), (3, 1, 2)), ((1, 3), (2, 3, 1)),
                ((2, 3), None)]),
    dict(name="cfg5_small_4x2", grid=(4, 2), dims=(32, 16, 24), extra=(), it=4,
         chain=[((2, 3), None), ((1, 3), (2, 3, 1)), ((1, 2), (3, 1, 2))]),
    # BASELINE configs[3] in small: ComplexF64 on the (4,2) grid, both schedules
    dict(name="cfg4_small_4x2", grid=(4, 2), dims=(16, 32, 16), extra=(), it=16,
         chain=[((2, 3), None), ((1, 3), (2, 1, 3)), ((1, 2), (3, 2, 1)), ((1, 3), (2, 1, 3)),
                ((2, 3), None)]),
    # ComplexF64, power-of-two local lines: the shapes the fused unpack+FFT kernel accepts
    dict(name="c128_pow2_2x2", grid=(2, 2), dims=(16, 32, 64), extra=(), it=16,
         chain=[((2, 3), None), ((1, 3), (2, 1, 3)), ((1, 2), (3, 2, 1))]),
    dict(name="c128_pow2_2x1", grid=(2, 1), dims=(32, 16, 8), extra=(3,), it=16,
         chain=[((2, 3), None), ((1, 3), (2, 1, 3)), ((1, 2), (3, 2, 1))]),
    # 2-byte elements, extra dim, 4-D data
    dict(name="u16_4d", grid=(2, 2), dims=(6, 5, 4, 7), extra=(2,), it=2,
         chain=[((3, 4), None), ((1, 4), (4, 3, 2, 1)), ((1, 2), (3, 4, 1, 2))]),
]


def build_chain(case):
    """Per chain step: list over ranks of (python Pencil, oracle OPencil)."""
    ranks = make_ranks(case["grid"])
    steps = []
    for (decomp, perm) in case["chain"]:
        pens = []
        for er in ranks:
            if not steps:
                p = pa.Pencil(er.topo, case["dims"], decomp, permute=perm_of(perm))
            else:
                base = steps[0][ranks.index(er)][0]
                p = pa.Pencil(base, decomp_dims=decomp, permute=perm_of(perm))
            op = O.OPencil(O.OTopology(case["grid"], er.comm.rank), case["dims"], decomp, perm)
            pens.append((p, op))
        steps.append(pens)
    return ranks, steps
