"""Worker for the multi-process tests; launched with torch.distributed.run.

  mode "nccl": real path -- pa.transpose_ over NCCL, one GPU per rank;
  mode "ipc":  real path with the NCCL-free communicator (CUDA-IPC windows + flag
               words only): the ranks may SHARE one GPU, so a single-GPU box runs
               the whole multi-rank schedule -- one-sided puts/gets, the staged
               PointToPoint / Alltoallv schedules over the library's own copy
               kernels, waitall=false + Waitall, in-place fallback, empty blocks;
  mode "gloo": CPU box -- the C planner's descriptors are interpreted with
               NumPy (tests/util.apply_block) and the exchange follows the
               plan's peer table over gloo send/recv.  Checks the N>1 host
               logic (rank grid, peer table, counts, offsets) across real
               processes.
Every rank recomputes the whole oracle (sizes are small) and compares its own
part bit for bit.
"""
import os
import sys
import tempfile

import numpy as np
import torch
import torch.distributed as dist

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.dirname(HERE))

import pencilarrays_b200 as pa  # noqa: E402
from pencilarrays_b200.transpositions import _Plan  # noqa: E402
from oracle import pencil_oracle as O  # noqa: E402
from util import CASES, DTYPES, beq, perm_of, apply_block  # noqa: E402
import math  # noqa: E402


def gloo_transpose(plan, src, dtype, it, rank, nparts=1):
    """pack -> exchange -> unpack with the C planner's descriptors only; with nparts > 1
    every block travels as `nparts` separately packed, sent, received and unpacked
    pieces cut where `pa_plan_get_chunk` says (the chunked PointToPoint schedule)."""
    import ctypes as C
    from pencilarrays_b200._lib import lib, check, BlockDesc
    info = plan.info
    dst = np.zeros(max(1, info.length_out), dtype=dtype)
    if info.dim == 0:
        apply_block(plan.block(2), src, dst)
        return dst
    send = np.zeros(max(1, info.send_bytes // it), dtype=dtype)
    recv = np.zeros(max(1, info.recv_bytes // it), dtype=dtype)
    nproc, me = info.nproc, info.self_index

    def chunk(op, p, c):
        d, off, nb = BlockDesc(), C.c_int64(), C.c_int64()
        check(lib.pa_plan_get_chunk(plan.h, op, p, c, nparts, C.byref(d), C.byref(off), C.byref(nb)))
        return d, off.value, nb.value

    for p in range(1, nproc + 1):
        peer = plan.peer(p)
        if peer.is_self:
            apply_block(plan.block(0, p), src, recv)
        else:
            for c in range(nparts):
                apply_block(chunk(0, p, c)[0], src, send)
    reqs, keep = [], []
    for k in range(1, nproc):  # same rotation as the CUDA driver
        pt, pf = (me - 1 + k) % nproc + 1, (me - 1 - k) % nproc + 1
        to, fr = plan.peer(pt), plan.peer(pf)
        for c in range(nparts):
            _, so, sn = chunk(0, pt, c)
            _, ro, rn = chunk(1, pf, c)
            if sn:
                t = torch.from_numpy(send.view(np.uint8)[so:so + sn].copy())
                keep.append(t)
                reqs.append(dist.isend(t, to.world_rank, tag=c))
            if rn:
                t = torch.empty(rn, dtype=torch.uint8)
                keep.append((t, ro))
                reqs.append(dist.irecv(t, fr.world_rank, tag=c))
    for r in reqs:
        r.wait()
    for item in keep:
        if isinstance(item, tuple):
            t, ro = item
            recv.view(np.uint8)[ro:ro + t.numel()] = t.numpy()
    for p in range(1, nproc + 1):
        if plan.peer(p).is_self:
            apply_block(plan.block(1, p), recv, dst)
        else:
            for c in range(nparts):
                apply_block(chunk(1, p, c)[0], recv, dst)
    return dst


def main():
    mode = sys.argv[1]
    if mode == "nccl":
        comm = pa.comm_world(transport="nccl")
    elif mode == "ipc":
        comm = pa.comm_world(transport="ipc")
        assert comm.transport == "ipc" and comm.handle is not None
    else:
        dist.init_process_group("gloo")
        comm = pa.Comm(dist.get_rank(), dist.get_world_size())
    rank, world = comm.rank, comm.size
    # the directory every rank writes its PencilIO file to: the test's own, or (when the
    # worker is started by hand) one that rank 0 makes and tells the others about
    scratch = [os.environ.get("PA_TEST_SCRATCH") or (tempfile.mkdtemp(prefix="pa_mp_worker_")
                                                     if rank == 0 else None)]
    dist.broadcast_object_list(scratch, src=0)
    scratch = scratch[0]
    ran = 0
    extra_cases = []
    if mode != "gloo":
        # seeded random configurations (tests/test_random_configs.py) with this world size:
        # uneven / empty blocks, 2-d ... 4-d data, every permutation, 2 ... 16-byte elements
        from test_random_configs import RANDOM_CASES
        extra_cases = [dict(c, random=True) for c in RANDOM_CASES if math.prod(c["grid"]) == world][:6]
    for case in CASES + extra_cases:
        if math.prod(case["grid"]) != world:
            continue
        ran += 1
        dtype, it, extra = DTYPES[case["it"]], case["it"], case["extra"]
        topo = pa.MPITopology(comm, case["grid"])
        opens = [[O.OPencil(O.OTopology(case["grid"], r), case["dims"], d, p) for r in range(world)]
                 for (d, p) in case["chain"]]
        pens = []
        for i, (d, p) in enumerate(case["chain"]):
            pens.append(pa.Pencil(topo, case["dims"], d, permute=perm_of(p)) if i == 0 else
                        pa.Pencil(pens[0], decomp_dims=d, permute=perm_of(p)))
        g = O.global_pattern(case["dims"], extra, it)
        cur_o = O.scatter(g, opens[0], extra, dtype)
        # (method, overlap, waitall, tunables)
        variants = [(pa.PointToPoint(), True, True, {}), (pa.PointToPoint(), False, True, {}),
                    (pa.Alltoallv(), True, True, {}), (pa.PointToPoint(), True, False, {}),
                    (pa.PeerPut(), True, True, {}), (pa.PeerGet(), True, True, {}),
                    (pa.PeerGet(), True, False, {}),
                    (pa.PointToPoint(), True, True, {"p2p_chunks": 3}),
                    (pa.PointToPoint(), False, False, {"p2p_chunks": 2, "staged_ctas": 8}),
                    (pa.PeerPut(), True, True, {"multi_put": 0}),
                    (pa.PeerGet(), True, False, {"multi_put": 0}),
                    (pa.Alltoallv(), True, True, {"multi_put": 0})]
        if mode == "nccl":  # the own-kernel exchange beside NCCL on the same communicator
            variants += [(pa.PointToPoint(), True, True, {"ipc_exchange": 1}),
                         (pa.Alltoallv(), True, True, {"ipc_exchange": 1, "p2p_chunks": 2})]
        if case.get("random"):  # a shorter list: the point is the geometry, not the tunables
            variants = [(pa.PointToPoint(), True, True, {}), (pa.Alltoallv(), True, True, {}),
                        (pa.PeerPut(), True, True, {}), (pa.PeerGet(), True, False, {}),
                        (pa.PointToPoint(), True, False, {"p2p_chunks": 3})]
        defaults = {"p2p_chunks": 1, "staged_ctas": 0, "multi_put": 1, "ipc_exchange": 0}
        if mode == "gloo":
            cur = cur_o[rank].data.reshape(-1, order="F").copy()
        else:
            tdt = {4: torch.float32, 8: torch.float64, 16: torch.complex128, 2: torch.int16}[it]
            cur = pa.PencilArray.undef(tdt, pens[0], *extra)
            cur.data.view(torch.uint8).reshape(-1).copy_(torch.from_numpy(
                np.ascontiguousarray(cur_o[rank].data.reshape(-1, order="F")).view(np.uint8).copy()))
            torch.cuda.synchronize()
        for k in range(1, len(case["chain"])):
            cur_in = cur
            nxt_o = [O.OArray.undef(dtype, po, *extra) for po in opens[k]]
            O.transpose_all(nxt_o, cur_o)
            want = np.ascontiguousarray(nxt_o[rank].data.reshape(-1, order="F"))
            if mode == "gloo":
                plan = _Plan(pens[k - 1], pens[k], extra, it, pa.PointToPoint())
                got = gloo_transpose(plan, cur, dtype, it, rank)[:want.size]
                assert beq(got, want), (case["name"], k, rank)
                got3 = gloo_transpose(plan, cur, dtype, it, rank, nparts=3)[:want.size]
                assert beq(got3, want), (case["name"], k, rank, "chunks=3")
                cur = got
            else:
                nxt = None
                for (method, overlap, waitall, tun) in variants:
                    for name, v in {**defaults, **tun}.items():
                        pa.set_tunable(name, v)
                    nxt = pa.PencilArray.undef(tdt, pens[k], *extra)
                    nxt.data.view(torch.uint8).fill_(0x5A)
                    t = pa.Transposition(nxt, cur, method=method)
                    pa.transpose_(t, waitall=waitall, overlap=overlap)
                    if not waitall:
                        pa.Waitall(t)
                    torch.cuda.synchronize()
                    got = nxt.data.view(torch.uint8).reshape(-1).cpu().numpy()
                    assert got.tobytes() == want.view(np.uint8).tobytes(), \
                        (case["name"], k, rank, method, overlap, waitall, tun)
                for name, v in defaults.items():
                    pa.set_tunable(name, v)
                if case["name"].startswith("c128_"):
                    # fused unpack + FFT along the now-local contiguous dim (staged methods) on a
                    # NUMERIC field (the bit-pattern field holds NaNs and 1e300s): numpy.fft of
                    # the same global array cut for the destination pencil, FFT's own tolerance
                    rng = np.random.default_rng(5)
                    shape = tuple(case["dims"]) + tuple(extra)
                    G = (rng.standard_normal(shape) + 1j * rng.standard_normal(shape))
                    Gb = np.ascontiguousarray(G.reshape(-1, order="F")).view(np.uint8) \
                        .reshape(-1, 16).reshape(shape + (16,), order="F")
                    a_in = O.scatter(Gb, opens[k - 1], extra, dtype)[rank]
                    a_out = O.scatter(Gb, opens[k], extra, dtype)[rank]
                    src = pa.PencilArray.undef(tdt, pens[k - 1], *extra)
                    src.data.view(torch.uint8).reshape(-1).copy_(torch.from_numpy(
                        np.ascontiguousarray(a_in.data.reshape(-1, order="F")).view(np.uint8).copy()))
                    L = a_out.data.shape[0]
                    ok_shape = case["name"].startswith("c128_pow2")  # power-of-two lines, 8..1024
                    for method in (pa.PointToPoint(), pa.Alltoallv()):
                        for direction in ("forward", "backward"):
                            out = pa.PencilArray.undef(tdt, pens[k], *extra)
                            t = pa.Transposition(out, src, method=method)
                            if not ok_shape:
                                try:
                                    pa.transpose_(t, fft=direction)
                                    raise AssertionError("fused FFT accepted an unsupported shape")
                                except pa.ArgumentError:
                                    continue
                            pa.transpose_(t, fft=direction)
                            torch.cuda.synchronize()
                            ref = np.fft.fft(a_out.data, axis=0) if direction == "forward" else \
                                np.fft.ifft(a_out.data, axis=0) * L
                            got = np.ascontiguousarray(out.data.cpu().numpy()).reshape(-1)
                            want_f = np.ascontiguousarray(ref.reshape(-1, order="F"))
                            tol = 8 * np.finfo(np.float64).eps * np.log2(L) * np.abs(want_f).max()
                            assert np.abs(got - want_f).max() <= tol, \
                                ("fft", case["name"], k, rank, method, direction)
                    if ok_shape and k == 1 and len(case["chain"]) >= 3:
                        # a whole distributed 3-d FFT, PencilFFTs-style: fft along x in place, then
                        # x->y and y->z with the next transform fused into the unpack; every rank's
                        # z-pencil array must be its part of numpy.fft.fftn of the global array
                        ux = pa.PencilArray.undef(tdt, pens[0], *extra)
                        ux.data.copy_(src.data)
                        uy = pa.PencilArray.undef(tdt, pens[1], *extra)
                        uz = pa.PencilArray.undef(tdt, pens[2], *extra)
                        pa.fft_(ux, "forward")
                        pa.transpose_(pa.Transposition(uy, ux, method=pa.PointToPoint()), fft="forward")
                        pa.transpose_(pa.Transposition(uz, uy, method=pa.Alltoallv()), fft="forward")
                        torch.cuda.synchronize()
                        F = np.fft.fftn(G, axes=(0, 1, 2))
                        Fb = np.ascontiguousarray(F.reshape(-1, order="F")).view(np.uint8) \
                            .reshape(-1, 16).reshape(shape + (16,), order="F")
                        want3 = O.scatter(Fb, opens[2], extra, dtype)[rank].data.reshape(-1, order="F")
                        got3 = np.ascontiguousarray(uz.data.cpu().numpy()).reshape(-1)
                        n3 = math.prod(case["dims"])
                        tol3 = 8 * np.finfo(np.float64).eps * np.log2(n3) * np.abs(F).max()
                        assert np.abs(got3 - want3).max() <= tol3, ("fft3d", case["name"], rank)
                cur = nxt
            cur_o = nxt_o
        if mode != "gloo" and len(case["chain"]) >= 3 and not extra:
            # in place: ManyPencilArray over the first three pencils (test/pencils.jl:224-239)
            A = pa.ManyPencilArray(tdt, *pens[:3])
            o0 = O.scatter(g, opens[0], extra, dtype)
            A[1].data.view(torch.uint8).reshape(-1).copy_(torch.from_numpy(
                np.ascontiguousarray(o0[rank].data.reshape(-1, order="F")).view(np.uint8).copy()))
            o1 = [O.OArray.undef(dtype, po) for po in opens[1]]
            O.transpose_all(o1, o0)
            o2 = [O.OArray.undef(dtype, po) for po in opens[2]]
            O.transpose_all(o2, o1)
            src_bytes = A[1].data.view(torch.uint8).reshape(-1).clone()
            # one-sided methods must notice the aliasing and take the staged schedule
            for method in (pa.PointToPoint(), pa.PeerPut(), pa.PeerGet(), pa.Alltoallv()):
                A[1].data.view(torch.uint8).reshape(-1).copy_(src_bytes)
                pa.transpose_(A[2], A[1], method=method)
                pa.transpose_(A[3], A[2], method=method)
                torch.cuda.synchronize()
                got = A[3].data.view(torch.uint8).reshape(-1).cpu().numpy()
                want = np.ascontiguousarray(o2[rank].data.reshape(-1, order="F")).view(np.uint8)
                assert got.tobytes() == want.tobytes(), ("inplace", case["name"], rank, method)
    if mode != "gloo":
        # PencilIO with REAL ranks writing one file concurrently (mpi_io.jl layout): every rank
        # pwrite()s its sub-box, rank 0 checks the bytes against the gathered global array and
        # everybody reads its part back (test/io.jl:28-105)
        for case in [c for c in CASES if math.prod(c["grid"]) == world and c["it"] in (4, 8, 16)][:2]:
            dtype, it, extra = DTYPES[case["it"]], case["it"], case["extra"]
            tdt = {4: torch.float32, 8: torch.float64, 16: torch.complex128}[it]
            decomp, perm = case["chain"][1]
            topo = pa.MPITopology(comm, case["grid"])
            pen = pa.Pencil(topo, case["dims"], decomp, permute=perm_of(perm))
            open_ = [O.OPencil(O.OTopology(case["grid"], r), case["dims"], decomp, perm) for r in range(world)]
            g = O.global_pattern(case["dims"], extra, it)
            mine = O.scatter(g, open_, extra, dtype)[rank]
            u = pa.PencilArray.undef(tdt, pen, *extra)
            u.data.view(torch.uint8).reshape(-1).copy_(torch.from_numpy(
                np.ascontiguousarray(mine.data.reshape(-1, order="F")).view(np.uint8).copy()))
            fname = os.path.join(scratch, f"pa_io_{case['name']}.bin")
            with pa.open_(pa.MPIIODriver(), fname, comm, write=True, create=True) as ff:
                ff.write("u", u, chunks=False)
                ff.write("u_chunks", u, chunks=True)
            if rank == 0:
                nd = len(case["dims"])
                axes = tuple(range(nd)) if perm is None else tuple(q - 1 for q in perm)
                gl = np.transpose(g, axes + tuple(range(nd, g.ndim)))  # memory order + extra + bytes
                want = np.ascontiguousarray(gl.reshape(-1, it, order="F")).tobytes()
                raw = open(fname, "rb").read()
                assert raw[:len(want)] == want, ("pencilio layout", case["name"])
                assert len(raw) == 2 * len(want)
            for name in ("u", "u_chunks"):
                v = pa.PencilArray.undef(tdt, pen, *extra)
                v.data.view(torch.uint8).fill_(0x11)
                with pa.open_(pa.MPIIODriver(), fname, comm, read=True) as ff:
                    pa.read_(ff, v, name)
                assert torch.equal(v.data.view(torch.uint8), u.data.view(torch.uint8)), ("pencilio", name)
            dist.barrier()
            if rank == 0:
                os.remove(fname)
                os.remove(fname + ".json")
    dist.barrier()
    if rank == 0 and not os.environ.get("PA_TEST_SCRATCH"):
        os.rmdir(scratch)
    if rank == 0:
        print(f"MP_WORKER_OK mode={mode} world={world} cases={ran} launches={pa.launch_count()}")
    dist.destroy_process_group()


if __name__ == "__main__":
    try:
        main()
    except BaseException:
        import traceback
        tb = traceback.format_exc()
        sys.stderr.write("".join(f"WORKER-ERROR[{os.environ.get('RANK', '?')}] {l}\n"
                                 for l in tb.splitlines()))
        sys.stderr.flush()
        os._exit(1)
