#!/usr/bin/env python
"""bench.py -- `transpose!` throughput (GiB/s moved), the metric of BASELINE.json.

One STEP = the x -> y -> z -> y -> x chain of four `transpose!` calls
(x<->y and y<->z, both directions, PencilFFTs' usual permutations
None -> (2,1,3) -> (3,2,1)) over a synthetic ComplexF64 grid.  Weak scaling:
every GPU holds 2 GiB of the array (512^3 ComplexF64 per GPU), so that
N = 8 is exactly BASELINE configs[3] (1024^3 ComplexF64, process grid (4,2)).

  value     4 * global_bytes / 2^30 / step_time, whole job, inputs resident in HBM,
            CUDA events on the launching stream, max over ranks;
  e2e       the same step on HOST arrays through the library's host entry
            (pa_host_chain_*, the C ABI a PencilFFTs-style caller on `Array`s binds):
            every step uploads its input from pinned host memory and downloads its
            result; submits are asynchronous, two in flight;
  roofline  the slowest BASELINE-shape kernel (K1 pack / K2 unpack / K3 fused of
            configs[1], [3], [4]) timed live with CUDA events, against the measured
            HBM copy bandwidth;
  cpu_baseline / --impl reference   oracle/pa_oracle.c (the CPU port of the
            reference path) on the host cores, SAME grid as the GPU arm.

  python bench.py [--gpus N] [--steps K] [--warmup W]        # this framework
  python bench.py --impl reference ...                       # CPU port of the reference path
  python bench.py ... --dump-outputs bench_outputs   # also write what the last timed step computed

--dump-outputs DIR writes DIR/ux.npy, uy.npy, uz.npy (suffix _rank<r> when N > 1): the x-, y-
and z-pencil arrays as the last timed step left them, i.e. what the four transpose! calls hand
their caller, each a fixed sample when the whole would exceed 48 MiB in all.  The inputs are
seeded, so two builds run with the same arguments can be compared file by file.  Only uy and
uz carry computed data: the step is a round trip, so ux is the seeded input again (which the
round_trip_bit_exact check already confirms); a match in ux says nothing about the kernels.
"""
import argparse
import ctypes as C
import json
import math
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

GIB = float(1 << 30)
PER_GPU = (512, 512, 512)           # ComplexF64 shard per GPU: 2 GiB
CHAIN = [((2, 3), None), ((1, 3), (2, 1, 3)), ((1, 2), (3, 2, 1))]  # x, y, z pencils
LEGS = ["x->y", "y->z", "z->y", "y->x"]
# --workload: "cfg4" (default, above) or "cfg5" = BASELINE configs[4]: Float32,
# 1 GiB per GPU ((1024,512,512) per GPU -> 2048x1024x1024 at N = 8), perms None -> (2,3,1) -> (3,1,2)
WORKLOADS = {
    "cfg4": dict(per_gpu=PER_GPU, chain=CHAIN, dtype="complex128", itemsize=16, tname="ComplexF64",
                 perms="None->(2,1,3)->(3,2,1)", note="2 GiB per GPU; N=8 is BASELINE configs[3]"),
    "cfg5": dict(per_gpu=(1024, 512, 512),
                 chain=[((2, 3), None), ((1, 3), (2, 3, 1)), ((1, 2), (3, 1, 2))],
                 dtype="float32", itemsize=4, tname="Float32", perms="None->(2,3,1)->(3,1,2)",
                 note="1 GiB per GPU; N=8 is BASELINE configs[4]"),
}


def grid_and_dims(n, per_gpu=PER_GPU):
    grid = {1: (1, 1), 2: (2, 1), 4: (2, 2), 8: (4, 2)}[n]
    mult = {1: (1, 1, 1), 2: (2, 1, 1), 4: (2, 2, 1), 8: (2, 2, 2)}[n]
    return grid, tuple(a * b for a, b in zip(per_gpu, mult))


def measured_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region: the sampler
    runs from before the warm-up (nvidia-smi needs ~1 s to start) at 10 ms
    period; rows are time-stamped and only those inside [mark_start, mark_stop]
    (host clock, bracketing the timed steps) are reported.  If the region is
    shorter than the sampling allows, the rows within 250 ms of it are used and
    `window` says so."""
    Q = ("timestamp,clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.rows, self.proc, self.index = [], None, index
        self.t0 = self.t1 = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                 "--format=csv,noheader,nounits", "-lms", "10"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
            t = time.time()
            while not self.rows and time.time() - t < 3.0:  # wait for the first sample
                time.sleep(0.01)
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def mark_start(self):
        self.t0 = time.time()

    def mark_stop(self):
        self.t1 = time.time()

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.05)
        self.proc.terminate()  # exact PID we started
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

        def parse(rows):
            sm, mx, reasons = [], [], set()
            for _, r in rows:
                c = [x.strip() for x in r.split(",")]
                if len(c) < 7:
                    continue
                try:
                    sm.append(float(c[1]))
                    mx.append(float(c[2]))
                except ValueError:
                    continue
                for nme, v in zip(names, c[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(nme)
            return sm, mx, reasons

        t0, t1 = self.t0 or 0.0, self.t1 or float("inf")
        inside = [r for r in self.rows if t0 <= r[0] <= t1]
        window = "timed region"
        if len(inside) < 5:
            inside = [r for r in self.rows if t0 - 0.25 <= r[0] <= t1 + 0.25]
            window = "timed region +-250 ms (region shorter than the sampling period)"
        sm, mx, reasons = parse(inside)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "window": window, "region_ms": round((t1 - t0) * 1e3, 1),
                "reasons": sorted(reasons)}


DUMP_BYTES = 48 << 20  # all --dump-outputs files of one run together


def dump_outputs(outdir, arrays, rank, n, torch):
    """Saves each (name, PencilArray) as OUTDIR/<name>.npy: the parent (memory-order) array,
    flattened; complex as (count, 2) real.  An array above its share of DUMP_BYTES is reduced
    to a sample at sorted positions drawn from a fixed seed, the same in every run."""
    import numpy as np
    os.makedirs(outdir, exist_ok=True)
    for name, u in arrays:
        flat = u.data.reshape(-1)
        keep = DUMP_BYTES // (len(arrays) * n * flat.element_size())
        if flat.numel() > keep:
            idx = np.sort(np.random.default_rng(0).choice(flat.numel(), keep, replace=False))
            flat = flat[torch.from_numpy(idx).to(flat.device)]
        out = (torch.view_as_real(flat) if flat.is_complex() else flat).cpu().numpy()
        np.save(os.path.join(outdir, name + (f"_rank{rank}" if n > 1 else "") + ".npy"), out)


def workload_name(n, wl="cfg4"):
    W = WORKLOADS[wl]
    grid, dims = grid_and_dims(n, W["per_gpu"])
    return (f"x->y->z->y->x transpose! chain, {dims[0]}x{dims[1]}x{dims[2]} {W['tname']}, "
            f"process grid {grid}, perms {W['perms']} ({W['note']})")


# ------------------------------------------------------------------------- CPU port of the reference
def host_threads():
    return len(os.sched_getaffinity(0)) or 1, os.cpu_count() or 1


class CpuChain:
    """The x->y->z->y->x chain through oracle/pa_oracle.c: all N ranks emulated in
    one process (one worker per rank, spare threads split each rank's loops),
    exchange = memcpy standing in for MPI's shared-memory transport.  Staging
    buffers are shared by the four transposes (the reference shares them across
    the pencils of a family, Pencils.jl:265-270)."""

    def __init__(self, n, wl, per_gpu=None):
        import numpy as np
        from oracle import c_oracle
        W = WORKLOADS[wl]
        self.np = np
        self.dtype = np.dtype(W["dtype"])
        self.grid, self.dims = grid_and_dims(n, per_gpu or W["per_gpu"])
        self.nranks = math.prod(self.grid)
        cfg = W["chain"] + [W["chain"][1], W["chain"][0]]
        self.cts = [c_oracle.CTranspose(self.grid, self.dims, cfg[i][0], cfg[i][1], cfg[i + 1][0],
                                        cfg[i + 1][1], (), self.dtype) for i in range(4)]
        for ct in self.cts[1:]:  # one pair of staging arenas per rank, sized for the largest use
            for r in range(self.nranks):
                if ct.send[r].size > self.cts[0].send[r].size:
                    self.cts[0].send[r] = ct.send[r]
                if ct.recv[r].size > self.cts[0].recv[r].size:
                    self.cts[0].recv[r] = ct.recv[r]
        for ct in self.cts[1:]:
            ct.send, ct.recv = self.cts[0].send, self.cts[0].recv
        rng = np.random.default_rng(42)
        self.bufs = []
        for r in range(self.nranks):
            nmax = max(max(ct.sz[r][0], ct.sz[r][1]) for ct in self.cts)
            if self.dtype.kind == "c":
                a = rng.standard_normal(2 * nmax).view(self.dtype)
            else:
                a = rng.standard_normal(nmax).astype(self.dtype)
            self.bufs.append([a, np.zeros(nmax, dtype=self.dtype)])
        self.global_bytes = math.prod(self.dims) * self.dtype.itemsize

    def bytes_needed(n, wl):  # noqa: N805 -- static helper
        W = WORKLOADS[wl]
        _, dims = grid_and_dims(n, W["per_gpu"])
        return int(math.prod(dims) * W["itemsize"] * 4.2)  # 2 arrays + send + recv arenas (+ slack)

    def step(self, nthreads):
        ph = [0.0, 0.0, 0.0]
        for i, ct in enumerate(self.cts):
            p = ct.run([b[i % 2] for b in self.bufs], [b[(i + 1) % 2] for b in self.bufs],
                       nthreads=nthreads)
            ph = [x + y for x, y in zip(ph, p)]
        return ph

    def pick_threads(self, avail):
        """The CPU arm may use every host thread; on a big shared box more threads is
        not always faster (OpenMP barriers, memory channels), so the fastest of a few
        counts is kept."""
        cands = sorted({c for c in (self.nranks, 2 * self.nranks, 4 * self.nranks, 8, 16, 32, 64, avail)
                        if self.nranks <= c <= avail} or {min(avail, self.nranks)})
        best, best_t = cands[0], float("inf")
        for c in cands:
            t0 = time.perf_counter()
            self.step(c)
            dt = time.perf_counter() - t0
            if dt < best_t:
                best, best_t = c, dt
        return best, cands


def avail_host_bytes():
    try:
        import psutil
        return int(psutil.virtual_memory().available)
    except Exception:
        return 8 << 30


def cpu_config(n, wl):
    """The reference arm runs the GPU arm's own grid whenever host memory allows;
    otherwise every axis is halved (and the output says so)."""
    need = CpuChain.bytes_needed(n, wl)
    if need < 0.8 * avail_host_bytes():
        return None, need
    return tuple(s // 2 for s in WORKLOADS[wl]["per_gpu"]), need


def run_reference(args):
    """`--impl reference`: the CPU port of the reference path, on the GPU arm's config."""
    import numpy as np
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    n, wl = args.gpus, args.workload
    W = WORKLOADS[wl]
    per_gpu, need = cpu_config(n, wl)
    ch = CpuChain(n, wl, per_gpu)
    orig = [b[0].copy() for b in ch.bufs] if need < 0.5 * avail_host_bytes() else None
    avail, nproc = host_threads()
    ch.step(avail)  # first touch
    threads, cands = ch.pick_threads(avail)
    for _ in range(max(0, args.warmup - len(cands) - 1)):
        ch.step(threads)
    t0 = time.perf_counter()
    phases = [0.0, 0.0, 0.0]
    for _ in range(args.steps):
        phases = [x + y for x, y in zip(phases, ch.step(threads))]
    dt = (time.perf_counter() - t0) / args.steps
    ok = None
    if orig is not None:  # every step is a full round trip: the arrays are back where they started
        ok = all(np.array_equal(o.view(np.uint8), b[0].view(np.uint8)) for o, b in zip(orig, ch.bufs))
    val = 4 * ch.global_bytes / GIB / dt
    same = per_gpu is None
    sample_txt = (("the full workload: " if same else "EVERY AXIS HALVED (host memory short): ") +
                  f"x->y->z->y->x on a {ch.dims[0]}x{ch.dims[1]}x{ch.dims[2]} {W['tname']} grid, "
                  f"{ch.nranks} emulated rank(s), grid {ch.grid}; {threads} OpenMP threads "
                  f"(fastest of {cands}) of {avail} usable / {nproc} host threads")
    cfg = {"workload": workload_name(n, wl)}
    if not same:
        cfg["sample"] = sample_txt
    cfg["round_trip_bit_exact"] = ok
    print(json.dumps({
        "impl": "reference", "metric": "transpose_GiB_per_s", "value": round(val, 3), "unit": "GiB/s",
        "n_gpus": n, "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(dt * 1e3, 3),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": ("c128" if W["itemsize"] == 16 else "f32") + " (bytes; pure data movement)",
        "data": "synthetic", "config": cfg,
        "cpu_baseline": {"value": round(val, 3), "unit": "GiB/s", "cores": threads, "nproc": nproc,
                         "usable_threads": avail, "kind": "port", "sample": sample_txt,
                         "phase_s_per_step": [round(p / args.steps, 4) for p in phases]},
        "e2e": {"value": round(val, 3), "unit": "GiB/s", "h2d_bytes_per_step": 0,
                "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }))


def cpu_baseline(wl):
    """oracle/pa_oracle.c on the host cores, same grid as the N=1 GPU arm, bounded to ~10-20 s."""
    per_gpu, _ = cpu_config(1, wl)
    ch = CpuChain(1, wl, per_gpu)
    W = WORKLOADS[wl]
    avail, nproc = host_threads()
    ch.step(avail)
    threads, cands = ch.pick_threads(avail)
    t0 = time.perf_counter()
    reps = 0
    while True:
        ch.step(threads)
        reps += 1
        el = time.perf_counter() - t0
        if el > 10.0 or reps >= 200:
            break
    val = 4 * ch.global_bytes / GIB / (el / reps)
    return {"value": round(val, 3), "unit": "GiB/s", "cores": threads, "nproc": nproc,
            "usable_threads": avail, "kind": "port",
            "sample": ("the full N=1 workload: " if per_gpu is None else "every axis halved: ") +
                      f"x->y->z->y->x chain on a {ch.dims[0]}x{ch.dims[1]}x{ch.dims[2]} {W['tname']} "
                      f"grid, 1 emulated rank, {reps} repetitions in {el:.1f} s (oracle/pa_oracle.c, "
                      f"OpenMP over {threads} threads, fastest of {cands})"}


# ------------------------------------------------------------------------- B200 arm
def time_launches(fn, reps, torch):
    for _ in range(2):
        fn()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


def baseline_kernels(pa, torch, peak):
    """K1 pack / K2 unpack of BASELINE configs[3] and configs[4] as rank 0 of the
    (4,2) grid sees them (geometry only: `Comm(0, 8)` has no data plane), and
    r2c-shaped (odd leading extent) permutes, launched through the C ABI exactly as
    pa_transpose launches them; CUDA events around back-to-back launches, arrays of
    1-2 GiB (>> 126 MB L2)."""
    from pencilarrays_b200._lib import lib, check
    from pencilarrays_b200.transpositions import _Plan
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    out = {}
    cfgs = [("cfg4 1024^3 c128", (4, 2), (1024, 1024, 1024), WORKLOADS["cfg4"]["chain"], 16),
            ("cfg5 2048x1024x1024 f32", (4, 2), (2048, 1024, 1024), WORKLOADS["cfg5"]["chain"], 4)]
    for name, grid, dims, chain, es in cfgs:
        comm = pa.Comm(0, math.prod(grid))
        topo = pa.MPITopology(comm, grid)
        pens = []
        for i, (d, p) in enumerate(chain):
            perm = pa.NoPermutation() if p is None else pa.Permutation(*p)
            pens.append(pa.Pencil(topo, dims, d, permute=perm) if i == 0 else
                        pa.Pencil(pens[0], decomp_dims=d, permute=perm))
        for k, leg in ((1, "x->y"), (2, "y->z")):
            plan = _Plan(pens[k - 1], pens[k], (), es, pa.PointToPoint())
            info = plan.info
            src = torch.empty(info.length_in * es, dtype=torch.uint8, device="cuda")
            dst = torch.empty(info.length_out * es, dtype=torch.uint8, device="cuda")
            send = torch.empty(max(1, info.send_bytes), dtype=torch.uint8, device="cuda")
            recv = torch.empty(max(1, info.recv_bytes), dtype=torch.uint8, device="cuda")
            for t in (src, recv):
                t.random_()
            for op, label in ((0, "K1 pack"), (1, "K2 unpack")):
                def run():
                    for p in range(1, info.nproc + 1):
                        peer = plan.peer(p)
                        if op == 0:
                            check(lib.pa_pack(plan.h, p, C.c_void_p(src.data_ptr()), C.c_void_p(
                                recv.data_ptr() if peer.is_self else send.data_ptr()), st))
                        else:
                            check(lib.pa_unpack(plan.h, p, C.c_void_p(recv.data_ptr()),
                                                C.c_void_p(dst.data_ptr()), st))
                ms = time_launches(run, 5, torch)
                nb = 2 * (info.length_in if op == 0 else info.length_out) * es
                out[f"{label} {name} {leg} (rank 0 of (4,2): {info.nproc} blocks)"] = {
                    "ms": round(ms, 4), "alg_bytes": nb, "launches": info.nproc,
                    "GBps": round(nb / ms / 1e6, 1), "frac": round(nb / ms / 1e6 / peak, 4),
                    "baseline_shape": True}
            del src, dst, send, recv
            torch.cuda.empty_cache()
    # r2c-shaped grids: odd leading extents keep rows only element-aligned
    r2c = [("r2c (513,512,512) ComplexF32", (513, 512, 512), torch.complex64, 8),
           ("r2c (1025,512,256) Float32", (1025, 512, 256), torch.float32, 4),
           ("odd (1025,511,129) Float64", (1025, 511, 129), torch.float64, 8)]
    topo1 = pa.MPITopology(pa.COMM_SELF, (1, 1))
    for name, dims, dt, es in r2c:
        px = pa.Pencil(topo1, dims, (2, 3))
        py = pa.Pencil(px, decomp_dims=(1, 3), permute=pa.Permutation(2, 1, 3))
        pz = pa.Pencil(py, decomp_dims=(1, 2), permute=pa.Permutation(3, 2, 1))
        ux, uy, uz = (pa.PencilArray.undef(dt, p) for p in (px, py, pz))
        ux.data.view(torch.uint8).random_()
        for leg, (d, s) in (("x->y (2,1,3)", (uy, ux)), ("y->z (3,1,2)", (uz, uy)), ("y->x", (ux, uy))):
            t = pa.Transposition(d, s)
            ms = time_launches(lambda: pa.transpose_(t), 5, torch)
            nb = 2 * ux.data.numel() * es
            blk = t.plan.block(2)
            out[f"K3 fused {name} {leg}"] = {
                "ms": round(ms, 4), "alg_bytes": nb, "launches": 1, "GBps": round(nb / ms / 1e6, 1),
                "frac": round(nb / ms / 1e6 / peak, 4), "baseline_shape": False,
                "kernel_class": blk.kernel_class, "plan_align_bytes": blk.vec_bytes}
        del ux, uy, uz
        torch.cuda.empty_cache()
    return out


def fused_fft_rows(pa, torch, peak):
    """SURVEY 8(f2): transpose! with the 1-d FFT of the next step fused into its unpack
    (PA_FFT_FORWARD), against the unfused pair (this library's transpose! + cuFFT through
    torch.fft -- library code, the baseline).  512^3 ComplexF64, one GPU."""
    topo1 = pa.MPITopology(pa.COMM_SELF, (1, 1))
    dims = (512, 512, 512)
    px = pa.Pencil(topo1, dims, (2, 3))
    py = pa.Pencil(px, decomp_dims=(1, 3), permute=pa.Permutation(2, 1, 3))
    ux, uy = pa.PencilArray.undef(torch.complex128, px), pa.PencilArray.undef(torch.complex128, py)
    ux.data.view(torch.float64).normal_()
    t = pa.Transposition(uy, ux)
    tmp = torch.empty_like(uy.data)
    nb = 2 * ux.data.numel() * 16
    ms_tf = time_launches(lambda: (pa.transpose_(t), torch.fft.fft(uy.data, dim=-1, out=tmp)), 5, torch)
    pa.transpose_(t)
    torch.fft.fft(uy.data, dim=-1, out=tmp)
    ms_fused = time_launches(lambda: pa.transpose_(t, fft="forward"), 5, torch)
    err = float((uy.data - tmp).abs().max() / tmp.abs().max())
    return {"shape": "512^3 ComplexF64, x->y (2,1,3), 512-point lines",
            "fused_ms": round(ms_fused, 4), "unfused_ms": round(ms_tf, 4),
            "speedup": round(ms_tf / ms_fused, 3), "fused_alg_bytes": nb,
            "fused_GBps": round(nb / ms_fused / 1e6, 1), "fused_frac_of_hbm": round(nb / ms_fused / 1e6 / peak, 4),
            "max_rel_diff_vs_cufft": err}


def configs1_256cubed(pa, torch, peak):
    """BASELINE configs[1]: 256^3 Float64, 1 GPU, x->y for every permutation = one
    fused K3 launch per transpose!.  Two timings: `rotating` -- 24 back-to-back
    launches cycling over 6 source/destination pairs (1.5 GiB touched between two
    uses of the same array: nothing is served from the 126 MB L2, and launch gaps
    are hidden as they are in a real chain); `flushed` -- one launch at a time,
    each after a 256 MiB memset (cold L2 and an idle GPU: includes launch latency)."""
    res = {}
    topo1 = pa.MPITopology(pa.COMM_SELF, (1, 1))
    q1 = pa.Pencil(topo1, (256, 256, 256), (2, 3))
    NP = 6
    srcs = [pa.PencilArray.undef(torch.float64, q1) for _ in range(NP)]
    for a in srcs:
        a.data.normal_()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")  # > 126 MB L2
    nb = 2 * srcs[0].data.numel() * 8
    for perm in ((2, 1, 3), (2, 3, 1), (3, 2, 1), (3, 1, 2), (1, 3, 2), None):
        q2 = pa.Pencil(q1, decomp_dims=(1, 3),
                       permute=pa.NoPermutation() if perm is None else pa.Permutation(*perm))
        dsts = [pa.PencilArray.undef(torch.float64, q2) for _ in range(NP)]
        ts = [pa.Transposition(d, s) for d, s in zip(dsts, srcs)]

        def sweep():
            for t in ts:
                pa.transpose_(t)
        for _ in range(2):
            sweep()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(4):
            sweep()
        b.record()
        torch.cuda.synchronize()
        rot = a.elapsed_time(b) / (4 * NP)
        tot = 0.0
        for it in range(8):
            flush.zero_()  # evict src/dst from L2 between launches
            s_, e_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s_.record()
            pa.transpose_(ts[0])
            e_.record()
            torch.cuda.synchronize()
            if it >= 3:
                tot += s_.elapsed_time(e_) / 5
        res[f"x->y perm {perm}"] = {
            "rotating": {"ms": round(rot, 4), "GBps": round(nb / rot / 1e6, 1),
                         "frac_of_hbm_peak": round(nb / rot / 1e6 / peak, 3)},
            "flushed": {"ms": round(tot, 4), "GBps": round(nb / tot / 1e6, 1),
                        "frac_of_hbm_peak": round(nb / tot / 1e6 / peak, 3)}}
        del dsts, ts
    res["note"] = configs1_256cubed.__doc__.split("\n\n")[0].replace("\n    ", " ")
    return res


def pcie_peaks(torch, nbytes):
    """Plain pinned-memory copies of the shard size: the roofline of the e2e figure."""
    h1 = torch.empty(nbytes, dtype=torch.uint8).pin_memory()
    h2 = torch.empty(nbytes, dtype=torch.uint8).pin_memory()
    d1 = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
    d2 = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()

    def run(up, down):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(2):
            if up:
                with torch.cuda.stream(s1):
                    d1.copy_(h1, non_blocking=True)
            if down:
                with torch.cuda.stream(s2):
                    h2.copy_(d2, non_blocking=True)
        torch.cuda.synchronize()
        return 2 * nbytes / (time.perf_counter() - t0) / 1e9
    run(True, True)
    out = {"h2d_GBps": round(run(True, False), 1), "d2h_GBps": round(run(False, True), 1),
           "both_directions_GBps_each": round(run(True, True), 1)}
    del h1, h2, d1, d2
    return out


def run_b200(args):
    import torch
    import torch.distributed as dist
    import pencilarrays_b200 as pa
    from pencilarrays_b200._lib import lib, check

    n = args.gpus
    world = int(os.environ.get("WORLD_SIZE", "1"))
    assert world == n, f"--gpus {n} but WORLD_SIZE={world}: launch with torch.distributed.run"
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the transpose! path has no CPU fallback")
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local % torch.cuda.device_count())
    if args.nccl_ctas:
        pa.set_tunable("nccl_ctas", args.nccl_ctas)  # before the communicator exists
    comm = pa.comm_world() if n > 1 else pa.COMM_SELF
    rank = comm.rank
    W = WORKLOADS[args.workload]
    chain_cfg, isz = W["chain"], W["itemsize"]
    grid, dims = grid_and_dims(n, W["per_gpu"])
    topo = pa.MPITopology(comm, grid)
    px = pa.Pencil(topo, dims, chain_cfg[0][0])
    py = pa.Pencil(px, decomp_dims=chain_cfg[1][0], permute=pa.Permutation(*chain_cfg[1][1]))
    pz = pa.Pencil(py, decomp_dims=chain_cfg[2][0], permute=pa.Permutation(*chain_cfg[2][1]))
    dt = getattr(torch, W["dtype"])
    ux, uy, uz = (pa.PencilArray.undef(dt, p) for p in (px, py, pz))
    gen = torch.Generator(device="cuda").manual_seed(42 + rank)
    ux.data.view(torch.float64 if isz == 16 else dt).normal_(generator=gen)
    orig = ux.data.clone()
    if args.remote_ctas is not None:
        pa.set_tunable("remote_ctas", args.remote_ctas)
    if args.nccl_fences:
        pa.set_tunable("nccl_fences", 1)
    if args.no_nccl_register:
        pa.set_tunable("nccl_register", 0)
    if args.p2p_chunks is not None:
        pa.set_tunable("p2p_chunks", args.p2p_chunks)
    if args.staged_ctas is not None:
        pa.set_tunable("staged_ctas", args.staged_ctas)
    if args.ipc_exchange:
        pa.set_tunable("ipc_exchange", 1)
    if args.no_multi_put:
        pa.set_tunable("multi_put", 0)
    methods = {"alltoallv": pa.Alltoallv(), "pointtopoint": pa.PointToPoint(),
               "peerput": pa.PeerPut(), "peerget": pa.PeerGet()}
    pairs = [(uy, ux), (uz, uy), (uy, uz), (ux, uy)]

    def make_ts(name):
        """Transpositions of the chain for one method; a method that cannot be set up on
        ANY rank (e.g. CUDA IPC not permitted) is refused on all of them."""
        ok_here, ts_, msg = 1, None, ""
        try:
            ts_ = [pa.Transposition(d, s, method=methods[name]) for d, s in pairs]
        except pa.PencilError as e:
            ok_here, msg = 0, str(e)
            print(f"[rank {rank}] {name} unavailable: {e}", file=sys.stderr)
        if n > 1:
            flag = torch.tensor([ok_here], device="cuda")
            dist.all_reduce(flag, op=dist.ReduceOp.MIN)
            ok_here = int(flag.item())
        return (ts_ if ok_here else None), msg

    # auto: the one-sided put path over NVLink (fastest); if its windows cannot be set up,
    # every rank takes the NCCL PointToPoint path
    name = ("peerput" if n > 1 else "pointtopoint") if args.method == "auto" else args.method
    ts, _ = make_ts(name)
    if ts is None:
        if args.method != "auto" or name == "pointtopoint":
            raise SystemExit(f"method {name} could not be set up")
        name = "pointtopoint"
        ts, _ = make_ts(name)
        if ts is None:
            raise SystemExit("no transposition method could be set up")
    method = methods[name]
    overlap = not args.no_overlap

    def barrier():
        torch.cuda.synchronize()
        if n > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if n == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    ovl = [overlap]

    def chain(tl, evs=None):
        for i, t in enumerate(tl):
            pa.transpose_(t, waitall=True, overlap=ovl[0])
            if evs is not None:
                evs[i + 1].record()

    def timed_steps(tl, steps, warmup):
        for _ in range(warmup):
            chain(tl)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        legs = [[torch.cuda.Event(enable_timing=True) for _ in range(5)] for _ in range(steps)]
        e0.record()
        for k in range(steps):
            legs[k][0].record()
            chain(tl, legs[k])
        e1.record()
        barrier()
        ms_ = max_over_ranks(e0.elapsed_time(e1)) / steps
        leg = [0.0] * 4
        for k in range(steps):
            for i in range(4):
                leg[i] += legs[k][i].elapsed_time(legs[k][i + 1]) / steps
        return ms_, [max_over_ranks(x) for x in leg]

    # ---- device-resident timing -------------------------------------------------
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    for _ in range(args.warmup):
        chain(ts)
    barrier()
    sampler.mark_start()
    n0 = pa.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    legs = [[torch.cuda.Event(enable_timing=True) for _ in range(5)] for _ in range(args.steps)]
    e0.record()
    for k in range(args.steps):
        legs[k][0].record()
        chain(ts, legs[k])
    e1.record()
    barrier()
    sampler.mark_stop()
    launches = pa.launch_count() - n0
    clocks = sampler.stop() if rank == 0 else None
    ms = max_over_ranks(e0.elapsed_time(e1)) / args.steps
    leg_ms = [0.0] * 4
    for k in range(args.steps):
        for i in range(4):
            leg_ms[i] += legs[k][i].elapsed_time(legs[k][i + 1]) / args.steps
    leg_ms = [max_over_ranks(x) for x in leg_ms]
    ok = bool(torch.equal(ux.data.view(torch.uint8), orig.view(torch.uint8)))
    if args.dump_outputs:  # before the placement check below overwrites the arrays
        dump_outputs(args.dump_outputs, [("ux", ux), ("uy", uy), ("uz", uz)], rank, n, torch)
    gbytes = math.prod(dims) * isz
    value = 4 * gbytes / GIB / (ms * 1e-3)

    # ---- placement check at full size (not timed): a round trip alone would also pass for a
    # wrong-but-invertible shuffle, so every rank fills x with a function of the GLOBAL logical
    # index and checks that after x->y and y->z each element sits where the pencil geometry says:
    # parent(u)[perm * I] == global[I + offset]  (SURVEY 8c (ii); arrays.jl:327-337)
    def pattern(pen):
        rl = pa.range_local(pen)
        ax = [torch.arange(r.start - 1, r.stop - 1, device="cuda", dtype=torch.float64) for r in rl]
        lin = ax[0][:, None, None] + dims[0] * (ax[1][None, :, None] + dims[1] * ax[2][None, None, :])
        if isz == 16:
            return torch.complex(lin, -lin)
        return torch.remainder(lin, 16777216.0).to(dt)  # exact in Float32

    def placement(tl):
        good, perr = 0, None
        try:
            ux.logical().copy_(pattern(px))
            pa.transpose_(tl[0], waitall=True, overlap=overlap)
            pa.transpose_(tl[1], waitall=True, overlap=overlap)
            good = int(bool(torch.equal(uy.logical(), pattern(py))) and
                       bool(torch.equal(uz.logical(), pattern(pz))))
        except Exception as e:  # never lose the bench line over the checker
            perr = f"checker error: {type(e).__name__}: {e}"[:200]
        flag = torch.tensor([good], device="cuda")
        if n > 1:
            dist.all_reduce(flag, op=dist.ReduceOp.MIN)  # every rank takes part, whatever happened
        torch.cuda.empty_cache()
        return perr if perr else bool(flag.item())

    placed = placement(ts)
    ux.data.copy_(orig)

    # ---- the other methods beside it (N > 1): the schedules north_star names run over NCCL;
    # each gets warm-up, timed steps, round-trip and full-size placement checks in THIS run
    others = None
    if n > 1 and not args.only_default:
        others = {}
        variants = [("pointtopoint", {}), ("alltoallv", {}), ("peerget", {}),
                    ("pointtopoint", {"overlap": 0}), ("pointtopoint", {"self_first": 1}),
                    ("pointtopoint", {"p2p_chunks": 4}), ("pointtopoint", {"p2p_chunks": 8}),
                    ("pointtopoint", {"p2p_chunks": 4, "staged_ctas": -2}),
                    ("pointtopoint", {"p2p_chunks": 8, "staged_ctas": -1}),
                    ("pointtopoint", {"ipc_exchange": 1}),
                    ("pointtopoint", {"ipc_exchange": 1, "p2p_chunks": 4}),
                    ("alltoallv", {"ipc_exchange": 1}),
                    ("peerput", {"multi_put": 0}),
                    ("peerput", {"oneside_self_ctas": -1}), ("peerput", {"oneside_self_ctas": -2}),
                    ("peerput", {"remote_ctas": -8}), ("peerput", {"remote_ctas": -2}),
                    ("peerput", {"remote_ctas": -8, "oneside_self_ctas": -2})]
        if args.variants:
            variants = [v for i, v in enumerate(variants) if str(i) in args.variants.split(",")]
        elif not args.all_variants:
            # (chunked NCCL sends cost ~0.1 ms per operation: 2-3x slower at N=8, measured in
            #  profiles/r2_bench_n8.json -- kept out of the default run)
            variants = [v for v in variants if not (set(v[1]) & {"p2p_chunks", "self_first", "remote_ctas",
                                                                  "oneside_self_ctas"})]
        defaults = {"p2p_chunks": args.p2p_chunks or 1, "ipc_exchange": 1 if args.ipc_exchange else 0,
                    "multi_put": 0 if args.no_multi_put else 1, "staged_ctas": args.staged_ctas or 0,
                    "self_first": 0, "oneside_self_ctas": 0,
                    "remote_ctas": args.remote_ctas if args.remote_ctas is not None else -4}
        for mname, tun in variants:
            label = mname + "".join(f" {k}={v}" for k, v in tun.items())
            if mname == name and not tun:
                continue
            for k, v in {**defaults, **tun}.items():
                if k != "overlap":
                    pa.set_tunable(k, v)
            ovl[0] = bool(tun.get("overlap", overlap))
            tl, msg = make_ts(mname)
            if tl is None:
                others[label] = {"unavailable": msg[:160]}
            else:
                ux.data.copy_(orig)
                st_ = max(3, min(args.steps, 10))
                ms_m, leg_m = timed_steps(tl, st_, 3)
                rt = bool(torch.equal(ux.data.view(torch.uint8), orig.view(torch.uint8)))
                flag = torch.tensor([int(rt)], device="cuda")
                dist.all_reduce(flag, op=dist.ReduceOp.MIN)
                others[label] = {"value_GiBps": round(4 * gbytes / GIB / (ms_m * 1e-3), 2),
                                 "ms_per_step": round(ms_m, 4), "steps": st_,
                                 "leg_ms": dict(zip(LEGS, [round(x, 4) for x in leg_m])),
                                 "round_trip_bit_exact": bool(flag.item()),
                                 "placement_exact_full_size": placement(tl)}
            for k, v in defaults.items():
                pa.set_tunable(k, v)
            ovl[0] = overlap
        ux.data.copy_(orig)

    # ---- per-kernel roofline -----------------------------------------------------------
    peak, peak_src = measured_peak()
    shard = ux.data.numel() * isz
    kern = {}
    if n == 1:
        # each leg IS one launch of the fused permuting kernel (K3); live numbers from the timed steps
        for lname, m in zip(LEGS, leg_ms):
            kern[f"K3 fused permute {lname} (512^3 c128, the timed steps)"] = {
                "ms": round(m, 4), "alg_bytes": 2 * shard, "launches": 1,
                "GBps": round(2 * shard / m / 1e6, 1), "frac": round(2 * shard / m / 1e6 / peak, 4),
                "baseline_shape": True}
        if args.workload == "cfg4" and not args.quick:
            torch.cuda.empty_cache()
            kern.update(baseline_kernels(pa, torch, peak))
    else:
        st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
        for lname, t, src, dst in (("x->y", ts[0], ux, uy), ("y->z", ts[1], uy, uz)):
            info = t.plan.info
            if info.dim == 0:
                continue
            # (private arenas: the plan's own may be exposed to the peers' exchange kernels)
            send = torch.empty(max(1, info.send_bytes), dtype=torch.uint8, device="cuda")
            recv = torch.empty(max(1, info.recv_bytes), dtype=torch.uint8, device="cuda")
            scratch = torch.empty_like(dst.data)
            for op, label in ((0, "K1 pack"), (1, "K2 unpack")):
                def run():
                    for p in range(1, info.nproc + 1):
                        peer = t.plan.peer(p)
                        if op == 0:
                            check(lib.pa_pack(t.plan.h, p, C.c_void_p(src.data_ptr()), C.c_void_p(
                                recv.data_ptr() if peer.is_self else send.data_ptr()), st))
                        else:
                            check(lib.pa_unpack(t.plan.h, p, C.c_void_p(recv.data_ptr()),
                                                C.c_void_p(scratch.data_ptr()), st))
                m = time_launches(run, 5, torch)
                nb = 2 * (info.length_in if op == 0 else info.length_out) * isz
                kern[f"{label} {lname} (all {info.nproc} blocks)"] = {
                    "ms": round(m, 4), "alg_bytes": nb, "launches": info.nproc,
                    "GBps": round(nb / m / 1e6, 1), "frac": round(nb / m / 1e6 / peak, 4),
                    "baseline_shape": True}
            del send, recv, scratch
        torch.cuda.empty_cache()
    base = {k: v for k, v in kern.items() if v.get("baseline_shape")}
    dom = min(base.items(), key=lambda kv: kv[1]["GBps"]) if base else None
    rest = {k: v for k, v in kern.items() if not v.get("baseline_shape")}
    low = min(rest.items(), key=lambda kv: kv[1]["GBps"]) if rest else None
    def traffic_of(kernel_name):
        """DRAM bytes per launch of that kernel from the committed ncu capture
        (profiles/traffic.json, which names the file and the date); None when the selected
        kernel has no capture."""
        try:
            with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
                tj = json.load(f)
            for key, ent in tj.get("by_kernel", {}).items():
                if key in kernel_name:
                    return ent.get("bytes_per_launch"), {k: ent.get(k) for k in (
                        "kernel", "file", "date", "algorithmic_bytes_per_launch")}
        except Exception:
            pass
        return None, None

    # ---- BASELINE configs[1] beside it (N == 1): 256^3 Float64, 1 GPU, pack/unpack kernel only ----
    cfg1 = configs1_256cubed(pa, torch, peak) if (n == 1 and args.workload == "cfg4" and not args.quick) else None
    fused = None
    if n == 1 and args.workload == "cfg4" and not args.quick:
        torch.cuda.empty_cache()
        fused = fused_fft_rows(pa, torch, peak)
    if cfg1:
        for k, v in cfg1.items():
            if isinstance(v, dict):
                kern[f"K3 fused 256^3 Float64 {k} (configs[1], rotating buffers)"] = {
                    "ms": v["rotating"]["ms"], "alg_bytes": 2 * 256 ** 3 * 8, "launches": 1,
                    "GBps": v["rotating"]["GBps"], "frac": v["rotating"]["frac_of_hbm_peak"],
                    "baseline_shape": True}
        base = {k: v for k, v in kern.items() if v.get("baseline_shape")}
        dom = min(base.items(), key=lambda kv: kv[1]["GBps"])

    # ---- end to end: host arrays in, host arrays out, through the library's host entry ------
    torch.cuda.empty_cache()
    hin = torch.empty(ux.data.shape, dtype=dt).pin_memory()
    hin.copy_(orig)
    houts = [torch.empty(ux.data.shape, dtype=dt).pin_memory() for _ in range(2)]
    e2e_steps = max(4, min(args.steps, 8))
    ets, _ = make_ts(name)
    if args.host_slots:
        pa.set_tunable("host_slots", args.host_slots)
    if args.host_chunk_mib:
        pa.set_tunable("host_chunk_bytes", args.host_chunk_mib << 20)
    hc = pa.HostChain(ets)  # collective for the one-sided methods (windows on the chain's buffers)
    nfl = max(2, args.host_slots or 2)
    houts = houts + [torch.empty(ux.data.shape, dtype=dt).pin_memory() for _ in range(nfl - 2)]

    def e2e_run(steps):
        tk = []
        for i in range(steps):
            tk.append(hc.submit(hin, houts[i % nfl]))
            if i >= nfl - 1:
                hc.wait(tk[i - nfl + 1])  # `nfl` submits in flight: download(i-1) || upload(i)
        hc.wait()

    e2e_run(2)
    barrier()
    hc.time_begin()
    t_host = time.perf_counter()
    e2e_run(e2e_steps)
    e2e_dev_ms = hc.time_end()
    e2e_wall_ms = (time.perf_counter() - t_host) * 1e3
    barrier()
    e2e_ms = max_over_ranks(e2e_dev_ms) / e2e_steps
    e2e_ok = all(bool(torch.equal(h.view(torch.uint8), hin.view(torch.uint8))) for h in houts)
    e2e_val = 4 * gbytes / GIB / (e2e_ms * 1e-3)
    # one blocking transpose! on host arrays (pa_transpose_host): upload || kernel || download
    single = None
    if n == 1:
        t_xy = ts[0]
        hy = torch.empty(uy.data.shape, dtype=dt).pin_memory()
        pa.transpose_host_(t_xy, hin, hy)
        t0 = time.perf_counter()
        for _ in range(3):
            pa.transpose_host_(t_xy, hin, hy)
        single_ms = (time.perf_counter() - t0) / 3 * 1e3
        pa.transpose_(ts[0])  # (ux still holds `orig`)
        torch.cuda.synchronize()
        single = {"call": "pa_transpose_host, x->y, 2 GiB in + 2 GiB out, blocking",
                  "ms": round(single_ms, 2), "GiBps_moved": round(gbytes / GIB / (single_ms * 1e-3), 2),
                  "bit_exact_vs_device_path": bool(torch.equal(hy.view(torch.uint8).cuda(),
                                                               uy.data.view(torch.uint8)))}
        del hy
    del hc
    pcie = pcie_peaks(torch, min(shard, 1 << 30)) if rank == 0 else None

    # ---- exchange timing (N > 1): library CUDA-event sections, sequential phases ----
    sections = None
    if n > 1:
        sections = {"method": "PointToPoint, phases run strictly one after the other (PA_NO_OVERLAP)"}
        sts, _ = make_ts("pointtopoint")
        for lname, t in zip(LEGS[:2], sts or []):
            if t.dim is None:
                continue
            t.enable_timing(True)
            barrier()  # ranks enter together: otherwise the sections contain the skew
            pa.transpose_(t, waitall=True, overlap=False)
            tm = t.timings()
            t.enable_timing(False)
            info = t.plan.info
            sections[lname] = {"pack_ms": round(tm.pack_ms, 3), "exchange_ms": round(tm.exchange_ms, 3),
                               "unpack_ms": round(tm.unpack_ms, 3), "total_ms": round(tm.total_ms, 3),
                               "send_bytes": info.send_bytes,
                               "nvlink_GBps_out": round(info.send_bytes / max(tm.exchange_ms, 1e-6) / 1e6, 1),
                               "nvlink_frac_of_770": round(info.send_bytes / max(tm.exchange_ms, 1e-6) / 1e6 / 770, 3)}
        chain(ts)

    # ---- CPU baseline beside it (rank 0, N == 1 only) -------------------------------
    cpu = None
    if n == 1 and rank == 0 and not args.no_cpu:
        del hin, houts
        cpu = cpu_baseline(args.workload)

    if rank == 0:
        out = {
            "metric": "transpose_GiB_per_s", "value": round(value, 2), "unit": "GiB/s", "n_gpus": n,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(ms, 4),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": ("c128" if isz == 16 else "f32") + " (bytes; pure data movement)", "data": "synthetic",
            "config": {"workload": workload_name(n, args.workload), "method": repr(method), "overlap": overlap,
                       "transport": comm.transport,
                       "l2": "inputs (2 GiB per GPU) far larger than the 126 MB L2; no flush needed",
                       "round_trip_bit_exact": ok, "placement_exact_full_size": placed,
                       "leg_ms": dict(zip(LEGS, [round(x, 4) for x in leg_ms]))},
            "gpu_launches": int(launches),
            "clocks": clocks,
            "e2e": {"value": round(e2e_val, 2), "unit": "GiB/s", "ms_per_step": round(e2e_ms, 3),
                    "h2d_bytes_per_step": int(shard), "d2h_bytes_per_step": int(shard),
                    "steps": e2e_steps, "round_trip_bit_exact": e2e_ok,
                    "host_wall_ms_per_step": round(e2e_wall_ms / e2e_steps, 3),
                    "api": "pa_host_chain_submit / pa_host_chain_wait (C ABI, host pointers)",
                    "pcie": pcie, "single_call": single,
                    "note": "per step: the x-pencil array (bytes per GPU) is uploaded from pinned host "
                            "memory, the four transposes run on the device, the result is downloaded to "
                            "pinned host memory -- all inside the library's host chain; submits are "
                            "asynchronous with two in flight (download of step i || upload of step i+1: "
                            "PCIe is full duplex); timed with CUDA events from the first upload to the "
                            "last download, max over ranks"},
            "roofline": None if dom is None else {
                "bound": "hbm", "kernel": dom[0], "achieved": dom[1]["GBps"], "peak": peak,
                "unit": "GB/s", "frac": round(dom[1]["GBps"] / peak, 4), "traffic": traffic_of(dom[0])[0],
                "traffic_source": traffic_of(dom[0])[1], "peak_source": peak_src,
                "alg_bytes_per_launch": dom[1]["alg_bytes"] // max(1, dom[1].get("launches", 1)),
                "selection": "slowest of the BASELINE-shape kernels in `kernels` (K1 pack, K2 unpack, "
                             "K3 fused; configs[1], [3], [4])",
                "slowest_non_baseline_shape": None if low is None else
                {"kernel": low[0], "GBps": low[1]["GBps"], "frac": low[1]["frac"]},
                "timing": "CUDA events on the launching stream, back-to-back launches, this run"},
            "kernels": kern,
            "configs1_256cubed_f64": cfg1,
            "fused_fft": fused,
            "methods": others,
            "sections": sections,
            "cpu_baseline": cpu,
        }
        print(json.dumps(out))
    if n > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--method", default="auto",
                    choices=["auto", "pointtopoint", "alltoallv", "peerput", "peerget"])
    ap.add_argument("--no-overlap", action="store_true")
    ap.add_argument("--workload", default="cfg4", choices=sorted(WORKLOADS))
    ap.add_argument("--no-nccl-register", action="store_true",
                    help="staged methods: plain cudaMalloc arenas, no NCCL user-buffer registration")
    ap.add_argument("--nccl-fences", action="store_true",
                    help="one-sided methods: fence with NCCL groups instead of NVLink flags")
    ap.add_argument("--remote-ctas", type=int, default=None,
                    help="grid cap of the PeerPut/PeerGet kernels (tunable remote_ctas)")
    ap.add_argument("--p2p-chunks", type=int, default=None, help="tunable p2p_chunks")
    ap.add_argument("--nccl-ctas", type=int, default=None, help="ncclCommInitRankConfig min/maxCTAs")
    ap.add_argument("--staged-ctas", type=int, default=None, help="tunable staged_ctas")
    ap.add_argument("--ipc-exchange", action="store_true", help="staged methods over own copy kernels")
    ap.add_argument("--no-multi-put", action="store_true", help="one launch per peer block")
    ap.add_argument("--only-default", action="store_true", help="N>1: skip the other methods")
    ap.add_argument("--all-variants", action="store_true", help="N>1: also the chunked / reordered variants")
    ap.add_argument("--variants", default=None, help="N>1: comma-separated indices of the method variants to run")
    ap.add_argument("--host-slots", type=int, default=None, help="e2e: tunable host_slots (2..4)")
    ap.add_argument("--host-chunk-mib", type=int, default=None, help="e2e: tunable host_chunk_bytes")
    ap.add_argument("--quick", action="store_true", help="skip the side measurements (kernels, configs[1])")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the arrays the last timed step computed as DIR/<name>.npy")
    args = ap.parse_args()
    if args.gpus not in (1, 2, 4, 8):
        raise SystemExit("--gpus must be 1, 2, 4 or 8")
    if args.steps < 1:
        raise SystemExit("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        raise SystemExit("--dump-outputs writes the B200 arm's arrays: not with --impl reference")
    if args.warmup < 3:
        args.warmup = 3
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
