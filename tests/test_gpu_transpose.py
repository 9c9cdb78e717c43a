"""`transpose!` parity on the GPU, through the C ABI, against the oracle.

* every reference test case (tests/util.CASES) with all ranks emulated on one
  GPU: pa_pack / pa_unpack / pa_copy_self do the work, the harness only moves
  the packed blocks between the emulated ranks' buffers -- final arrays AND the
  send_buf / recv_buf wire layout must equal the oracle's, bit for bit;
* the public API (`Transposition`, `transpose_`, `ManyPencilArray`) on a
  1-rank grid: x -> y -> z -> y -> x, in place, local permutes, error cases;
* BASELINE full sizes via size-independent properties (round trip, gather
  equality evaluated on the device).
"""
import ctypes as C
import math

import numpy as np
import pytest
import torch

import pencilarrays_b200 as pa
from pencilarrays_b200._lib import lib, check
from pencilarrays_b200.transpositions import _Plan
from oracle import pencil_oracle as O
from util import CASES, DTYPES, beq, build_chain, golden_nbytes, matches_golden
from gpu_util import TORCH_OF, dev_bytes, host_bytes, emulate_transpose_gpu, ptr

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("case", CASES, ids=[c["name"] for c in CASES])
@pytest.mark.parametrize("fused_self", [False, True], ids=["staged_self", "fused_self"])
def test_reference_cases_emulated_ranks(case, fused_self):
    dtype = DTYPES[case["it"]]
    it = case["it"]
    extra = case["extra"]
    ranks, steps = build_chain(case)
    g = O.global_pattern(case["dims"], extra, it)
    cur_o = O.scatter(g, [po for (_, po) in steps[0]], extra, dtype)
    G = O.gather(cur_o)
    cur = [dev_bytes(a.data.reshape(-1, order="F")) for a in cur_o]
    for k in range(1, len(steps)):
        pin, pout = steps[k - 1], steps[k]
        nxt_o = [O.OArray.undef(dtype, po, *extra) for (_, po) in pout]
        states = O.transpose_all(nxt_o, cur_o, keep_states=True)
        assert beq(O.gather(nxt_o), G)
        plans = [_Plan(pin[r][0], pout[r][0], extra, it, pa.PointToPoint())
                 for r in range(len(ranks))]
        nxt = [torch.full((max(1, a.data.size * it),), 0xA5, dtype=torch.uint8, device="cuda")
               for a in nxt_o]
        sends, recvs = emulate_transpose_gpu(plans, cur, nxt, fused_self=fused_self)
        torch.cuda.synchronize()
        for r in range(len(ranks)):
            nb = nxt_o[r].data.size * it
            want = np.ascontiguousarray(nxt_o[r].data.reshape(-1, order="F")).view(np.uint8)
            assert host_bytes(nxt[r])[:nb].tobytes() == want.tobytes(), (k, r)
            if states is not None:
                st = states[r]
                ns, nr = plans[r].info.send_bytes, plans[r].info.recv_bytes
                assert host_bytes(sends[r])[:ns].tobytes() == st.send_buf.view(np.uint8)[:ns].tobytes()
                if not fused_self:
                    assert host_bytes(recvs[r])[:nr].tobytes() == st.recv_buf.view(np.uint8)[:nr].tobytes()
        cur_o = nxt_o
        cur = [t[:max(1, o.data.size * it)] for t, o in zip(nxt, nxt_o)]


@pytest.mark.parametrize("case", CASES, ids=[c["name"] for c in CASES])
def test_put_kernels_emulated_ranks(case):
    """K1-put (`pa_put`): each block stored directly into the destination rank's
    parent array -- here the emulated peers' arrays on the same GPU."""
    dtype, it, extra = DTYPES[case["it"]], case["it"], case["extra"]
    ranks, steps = build_chain(case)
    g = O.global_pattern(case["dims"], extra, it)
    cur_o = O.scatter(g, [po for (_, po) in steps[0]], extra, dtype)
    from gpu_util import stream_ptr
    for k in range(1, len(steps)):
        nxt_o = [O.OArray.undef(dtype, po, *extra) for (_, po) in steps[k]]
        O.transpose_all(nxt_o, cur_o)
        plans = [_Plan(steps[k - 1][r][0], steps[k][r][0], extra, it, pa.PeerPut())
                 for r in range(len(ranks))]
        if plans[0].info.dim != 0:
            cur = [dev_bytes(a.data.reshape(-1, order="F")) for a in cur_o]
            nxt = [torch.full((max(1, a.data.size * it),), 0xA5, dtype=torch.uint8, device="cuda")
                   for a in nxt_o]
            st = stream_ptr()
            for r, pl in enumerate(plans):
                check(lib.pa_copy_self(pl.h, ptr(cur[r]), ptr(nxt[r]), st))
                for p in range(1, pl.info.nproc + 1):
                    peer = pl.peer(p)
                    if not peer.is_self:
                        check(lib.pa_put(pl.h, p, ptr(cur[r]), ptr(nxt[peer.world_rank]), st))
            torch.cuda.synchronize()
            for r, a in enumerate(nxt_o):
                want = np.ascontiguousarray(a.data.reshape(-1, order="F")).view(np.uint8)
                assert host_bytes(nxt[r])[:want.size].tobytes() == want.tobytes(), (k, r)
            # K2-get (`pa_get`): pull each block out of the source rank's parent array
            for t in nxt:
                t.fill_(0x3C)
            for r, pl in enumerate(plans):
                check(lib.pa_copy_self(pl.h, ptr(cur[r]), ptr(nxt[r]), st))
                for p in range(1, pl.info.nproc + 1):
                    peer = pl.peer(p)
                    if not peer.is_self:
                        check(lib.pa_get(pl.h, p, ptr(cur[peer.world_rank]), ptr(nxt[r]), st))
            torch.cuda.synchronize()
            for r, a in enumerate(nxt_o):
                want = np.ascontiguousarray(a.data.reshape(-1, order="F")).view(np.uint8)
                assert host_bytes(nxt[r])[:want.size].tobytes() == want.tobytes(), ("get", k, r)
        cur_o = nxt_o


@pytest.mark.parametrize("itemsize", [24, 12, 48])
def test_non_power_of_two_element_sizes_gpu(itemsize):
    """24-byte (SVector{3,Float64}-like), 12-byte and 48-byte elements through the
    kernels: staged (pack/unpack), fused self block, put and get."""
    edt = np.dtype((np.void, itemsize))
    case = dict(name="odd_elsize", grid=(2, 2), dims=(6, 7, 5), extra=(2,), it=itemsize,
                chain=[((2, 3), None), ((1, 3), (2, 3, 1)), ((1, 2), (3, 2, 1)), ((1, 2), (1, 3, 2))])
    ranks, steps = build_chain(case)
    rng = np.random.default_rng(7)
    n_glob = math.prod(case["dims"]) * math.prod(case["extra"])
    gbytes = rng.integers(0, 256, size=(n_glob, itemsize), dtype=np.uint8)
    g = gbytes.reshape(case["dims"] + case["extra"] + (itemsize,), order="F")
    cur_o = O.scatter(g, [po for (_, po) in steps[0]], case["extra"], edt)
    from gpu_util import stream_ptr
    for k in range(1, len(steps)):
        nxt_o = [O.OArray.undef(edt, po, *case["extra"]) for (_, po) in steps[k]]
        O.transpose_all(nxt_o, cur_o)
        plans = [_Plan(steps[k - 1][r][0], steps[k][r][0], case["extra"], itemsize, pa.PeerPut())
                 for r in range(len(ranks))]
        cur = [dev_bytes(a.data.reshape(-1, order="F")) for a in cur_o]
        wants = [np.ascontiguousarray(a.data.reshape(-1, order="F")).view(np.uint8) for a in nxt_o]
        for mode in ("staged", "fused", "put", "get"):
            nxt = [torch.full((max(1, w.size),), 0x11, dtype=torch.uint8, device="cuda") for w in wants]
            if mode in ("staged", "fused") or plans[0].info.dim == 0:
                emulate_transpose_gpu(plans, cur, nxt, fused_self=(mode == "fused"))
            else:
                st = stream_ptr()
                for r, pl in enumerate(plans):
                    check(lib.pa_copy_self(pl.h, ptr(cur[r]), ptr(nxt[r]), st))
                    for p in range(1, pl.info.nproc + 1):
                        peer = pl.peer(p)
                        if peer.is_self:
                            continue
                        if mode == "put":
                            check(lib.pa_put(pl.h, p, ptr(cur[r]), ptr(nxt[peer.world_rank]), st))
                        else:
                            check(lib.pa_get(pl.h, p, ptr(cur[peer.world_rank]), ptr(nxt[r]), st))
            torch.cuda.synchronize()
            for r, w in enumerate(wants):
                assert host_bytes(nxt[r])[:w.size].tobytes() == w.tobytes(), (itemsize, k, r, mode)
        cur_o = nxt_o


# ---------------------------------------------------------------- public API, one rank
def _fill(u: pa.PencilArray, seed):
    raw = torch.randint(0, 256, (u.data.numel() * u.elsize,), dtype=torch.uint8, device="cuda",
                        generator=torch.Generator(device="cuda").manual_seed(seed))
    u.data.view(torch.uint8).reshape(-1).copy_(raw)


def _same_logical(u: pa.PencilArray, v: pa.PencilArray) -> bool:
    """gather(u) == gather(v) on one rank: compare the logical-order views bitwise."""
    a = torch.view_as_real(u.logical()) if u.dtype.is_complex else u.logical()
    b = torch.view_as_real(v.logical()) if v.dtype.is_complex else v.logical()
    a = a.contiguous().view(torch.uint8)
    b = b.contiguous().view(torch.uint8)
    return torch.equal(a, b)


@pytest.mark.parametrize("dtype", [torch.float64, torch.float32, torch.complex128])
@pytest.mark.parametrize("dims", [(16, 21, 41), (64, 48, 32)])
def test_api_round_trip_one_rank(dtype, dims):
    comm = pa.COMM_SELF
    topo = pa.MPITopology(comm, (1, 1))
    pen1 = pa.Pencil(topo, dims, (2, 3))
    pen2 = pa.Pencil(pen1, decomp_dims=(1, 3), permute=pa.Permutation(2, 3, 1))
    pen3 = pa.Pencil(pen2, decomp_dims=(1, 2), permute=pa.Permutation(3, 2, 1))
    u1 = pa.PencilArray.undef(dtype, pen1)
    u2 = pa.PencilArray.undef(dtype, pen2)
    u3 = pa.PencilArray.undef(dtype, pen3)
    _fill(u1, 1)
    u1_orig = u1.data.clone()
    with pytest.raises(pa.ArgumentError):       # direct x -> z is not possible (transpose.jl:44-45)
        pa.transpose_(u3, u1)
    for method in (pa.PointToPoint(), pa.Alltoallv()):
        for stage in (False, True):
            pa.transpose_(u2, u1, method=method, stage_self=stage)
            assert _same_logical(u1, u2)
            pa.transpose_(u3, u2, method=method, stage_self=stage)
            assert _same_logical(u2, u3)
            pa.transpose_(u2, u3, method=method, stage_self=stage)
            assert _same_logical(u2, u3)
            pa.transpose_(u1, u2, method=method, stage_self=stage)
            assert torch.equal(u1.data.view(torch.uint8), u1_orig.view(torch.uint8))
    # parent layout: parent(u2)[perm * I] == u1[I]  (arrays.jl:19-31)
    assert tuple(reversed(u2.data.shape)) == tuple(dims[i - 1] for i in (2, 3, 1))
    # no permutation + unsorted decomp_dims (transpose.jl:62-74)
    v = pa.PencilArray.undef(dtype, pa.Pencil(pen1, decomp_dims=(1, 3)))
    pa.transpose_(v, u1)
    assert _same_logical(u1, v)
    w = pa.PencilArray.undef(dtype, pa.Pencil(pen1, decomp_dims=(2, 1)))
    pa.transpose_(w, u1)
    assert _same_logical(u1, w)


def test_api_transposition_object_and_waitall():
    topo = pa.MPITopology(pa.COMM_SELF, (1,))
    px = pa.Pencil(topo, (20, 16, 4), (1,))
    py = pa.Pencil(px, decomp_dims=(2,), permute=pa.Permutation(2, 3, 1))
    assert px.buffers()[0] == py.buffers()[0]  # px.send_buf === py.send_buf (array_types.jl:134)
    ux = pa.PencilArray.undef(torch.float64, px)
    uy = pa.similar(ux, py)
    assert pa.pencil(uy) is py
    _fill(ux, 3)
    tr = pa.Transposition(uy, ux)
    assert tr.dim == 1
    pa.transpose_(tr, waitall=False)
    pa.Waitall(tr)
    assert _same_logical(ux, uy)
    assert pa.transpose_(uy, uy) is uy  # dest === src: no-op (Transpositions.jl:164)


def test_api_extra_dims_and_local_permute():
    topo = pa.MPITopology(pa.COMM_SELF, (1, 1))
    pen1 = pa.Pencil(topo, (16, 21, 41), (2, 3))
    pen2 = pa.Pencil(pen1, decomp_dims=(1, 3), permute=pa.Permutation(2, 3, 1))
    u1 = pa.PencilArray.undef(torch.float32, pen1, 3, 4)
    u2 = pa.PencilArray.undef(torch.float32, pen2, 3, 4)
    _fill(u1, 5)
    pa.transpose_(u2, u1)
    assert _same_logical(u1, u2)
    bad = pa.PencilArray.undef(torch.float32, pen2, 4, 3)
    with pytest.raises(pa.ArgumentError):  # extra dims differ (Transpositions.jl:99-103)
        pa.transpose_(bad, u1)
    # same decomposition, different permutation: permute_local! (pencils.jl:495-505)
    pen3 = pa.Pencil(pen2, permute=pa.Permutation(3, 2, 1))
    u3 = pa.PencilArray.undef(torch.float32, pen3, 3, 4)
    t = pa.Transposition(u3, u2)
    assert t.dim is None
    pa.transpose_(t)
    assert _same_logical(u1, u3)
    # identical configuration: plain copy (pencils.jl:512-516)
    v = pa.similar(u2)
    pa.transpose_(v, u2)
    assert torch.equal(v.data.view(torch.uint8), u2.data.view(torch.uint8))
    with pytest.raises(pa.DimensionMismatch):  # arrays.jl:108-114
        pa.PencilArray(pen2, torch.empty((41, 21, 16), device="cuda"))


@pytest.mark.parametrize("grid", [(1, 1), (1,)])
def test_api_in_place_many_pencil_array(grid):
    """ManyPencilArray: aliased src/dest (test/pencils.jl:224-239)."""
    topo = pa.MPITopology(pa.COMM_SELF, grid)
    dims = (16, 21, 41)
    if len(grid) == 2:
        pens = [pa.Pencil(topo, dims, (2, 3))]
        pens.append(pa.Pencil(pens[0], decomp_dims=(1, 3), permute=pa.Permutation(2, 3, 1)))
        pens.append(pa.Pencil(pens[1], decomp_dims=(1, 2), permute=pa.Permutation(3, 2, 1)))
    else:
        pens = [pa.Pencil(topo, dims, (1,))]
        pens.append(pa.Pencil(pens[0], decomp_dims=(2,)))
        pens.append(pa.Pencil(pens[1], permute=pa.Permutation(3, 2, 1)))  # local transpose
    A = pa.ManyPencilArray(torch.float64, *pens)
    u, v, w = A[1], A[2], A[3]
    assert u.data_ptr() == v.data_ptr() == w.data_ptr()
    _fill(u, 9)
    ref = pa.PencilArray(pens[0], u.data.clone())
    pa.transpose_(v, u)  # this also modifies `u`
    assert _same_logical(ref, v)
    pa.transpose_(w, v)
    assert _same_logical(ref, w)
    B = pa.ManyPencilArray(torch.float32, *pens, extra_dims=(3, 2))
    assert pa.extra_dims(B.first()) == pa.extra_dims(B.last()) == (3, 2)


def test_host_transpose_entry_point():
    """pa_transpose_host: host arrays in, host arrays out (H2D + transpose! + D2H)."""
    topo = pa.MPITopology(pa.COMM_SELF, (1, 1))
    dims = (24, 20, 12)
    pen1 = pa.Pencil(topo, dims, (2, 3))
    pen2 = pa.Pencil(pen1, decomp_dims=(1, 3), permute=pa.Permutation(2, 1, 3))
    plan = _Plan(pen1, pen2, (), 8, pa.PointToPoint())
    op1 = O.OPencil(O.OTopology((1, 1), 0), dims, (2, 3))
    op2 = O.OPencil(O.OTopology((1, 1), 0), dims, (1, 3), (2, 1, 3))
    g = O.global_pattern(dims, (), 8)
    (a,) = O.scatter(g, [op1], (), np.float64)
    b = O.OArray.undef(np.float64, op2)
    O.transpose_all([b], [a])
    hsrc = torch.from_numpy(a.data.reshape(-1, order="F").copy()).pin_memory()
    hdst = torch.empty(hsrc.numel(), dtype=torch.float64).pin_memory()
    check(lib.pa_transpose_host(plan.h, None, C.c_void_p(hsrc.data_ptr()),
                                C.c_void_p(hdst.data_ptr()), 1))
    assert hdst.numpy().tobytes() == b.data.reshape(-1, order="F").tobytes()


# ---------------------------------------------------------------- BASELINE sizes
@pytest.mark.parametrize("dims,dtype", [((256, 256, 256), torch.float64),
                                        ((512, 512, 512), torch.complex128)])
def test_full_size_properties(dims, dtype):
    """configs[1] (256^3 Float64, 1 GPU) and the 1-GPU shard of configs[3]:
    every permutation pair, gather equality on the device + exact round trip."""
    topo = pa.MPITopology(pa.COMM_SELF, (1, 1))
    pen1 = pa.Pencil(topo, dims, (2, 3))
    u1 = pa.PencilArray.undef(dtype, pen1)
    _fill(u1, 11)
    orig = u1.data.clone()
    perms2 = [pa.Permutation(2, 1, 3), pa.Permutation(2, 3, 1), pa.NoPermutation()]
    perms3 = [pa.Permutation(3, 2, 1), pa.Permutation(3, 1, 2), pa.Permutation(1, 3, 2)]
    for p2, p3 in zip(perms2, perms3):
        pen2 = pa.Pencil(pen1, decomp_dims=(1, 3), permute=p2)
        pen3 = pa.Pencil(pen2, decomp_dims=(1, 2), permute=p3)
        u2 = pa.PencilArray.undef(dtype, pen2)
        u3 = pa.PencilArray.undef(dtype, pen3)
        pa.transpose_(u2, u1)
        assert _same_logical(u1, u2)
        pa.transpose_(u3, u2)
        assert _same_logical(u1, u3)
        u2.data.zero_()
        pa.transpose_(u2, u3)
        u1.data.zero_()
        pa.transpose_(u1, u2)
        assert torch.equal(u1.data.view(torch.uint8), orig.view(torch.uint8))
        del u2, u3
    assert pa.launch_count() > 0


def test_gpu_path_against_committed_golden_fixtures():
    """The CUDA path against the COMMITTED fixtures tests/golden/*.npz (frozen oracle
    outputs, generator tests/golden/make_golden.py): the expected bytes come from the
    files, the live oracle only cuts the input pattern.  Emulated ranks, fused self
    block + pack/unpack of the remote blocks, through the C ABI."""
    import os
    gold = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
    files = sorted(f for f in os.listdir(gold) if f.endswith(".npz"))
    assert files
    for f in files:
        z = np.load(os.path.join(gold, f))
        case = dict(name=f, grid=tuple(int(v) for v in z["grid"]), dims=tuple(int(v) for v in z["dims"]),
                    extra=tuple(int(v) for v in z["extra"]), it=int(z["itemsize"]),
                    chain=[(tuple(int(v) for v in z[f"decomp{k}"]),
                            tuple(int(v) for v in z[f"perm{k}"]) or None) for k in range(int(z["nsteps"]))])
        dtype, it, extra = DTYPES[case["it"]], case["it"], case["extra"]
        ranks, steps = build_chain(case)
        g = O.global_pattern(case["dims"], extra, it)
        cur_o = O.scatter(g, [po for (_, po) in steps[0]], extra, dtype)
        cur = [dev_bytes(a.data.reshape(-1, order="F")) for a in cur_o]
        for k in range(1, len(steps)):
            plans = [_Plan(steps[k - 1][r][0], steps[k][r][0], extra, it, pa.PointToPoint())
                     for r in range(len(ranks))]
            sizes = [golden_nbytes(z, k, r) for r in range(len(ranks))]
            nxt = [torch.full((max(1, n),), 0xA5, dtype=torch.uint8, device="cuda") for n in sizes]
            emulate_transpose_gpu(plans, cur, nxt, fused_self=True)
            torch.cuda.synchronize()
            for r, n in enumerate(sizes):
                assert matches_golden(z, k, r, host_bytes(nxt[r])[:n]), (f, k, r)
            cur = [t[:max(1, n)] for t, n in zip(nxt, sizes)]
