"""Generates tests/golden/*.npz from the oracle (the reference cannot run in
this image -- no Julia, no MPI -- so fixtures are oracle outputs frozen at
commit time; see oracle/pencil_oracle.py for the parity status).

An output above SAMPLE_OVER bytes is stored as a sample, so that every fixture stays
well under 1 MB: `<key>` holds the bytes at the sorted positions `<key>_pos` (drawn
from a fixed seed), `<key>_nbytes` the full length and `<key>_sha256` the digest of
all of it.  tests/util.matches_golden checks either form.
Run from the repo root:  python tests/golden/make_golden.py [CASE ...]   (default: all)"""
import hashlib
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
sys.path.insert(0, os.path.dirname(HERE))
from oracle import pencil_oracle as O  # noqa: E402
from util import CASES, DTYPES  # noqa: E402

PICK = ["ref_transpose_2x2", "ref_unsorted", "ref_extra_dims", "ref_slab", "baseline_cfg1",
        "two_ranks_2x1", "empty_blocks"]
SAMPLE_OVER = 1 << 16   # bytes of one rank's output above which only a sample is stored
SAMPLE = 2048           # positions in that sample


def store(out, key, b):
    if b.size <= SAMPLE_OVER:
        out[key] = b
        return
    pos = np.sort(np.random.default_rng(0).choice(b.size, SAMPLE, replace=False)).astype(np.uint32)
    out[key] = b[pos]
    out[key + "_pos"] = pos
    out[key + "_nbytes"] = np.array(b.size, dtype=np.int64)
    out[key + "_sha256"] = np.frombuffer(hashlib.sha256(b.tobytes()).digest(), dtype=np.uint8)


for case in CASES:
    if case["name"] not in (sys.argv[1:] or PICK):
        continue
    dtype, extra = DTYPES[case["it"]], case["extra"]
    out = dict(grid=np.array(case["grid"]), dims=np.array(case["dims"]),
               extra=np.array(extra, dtype=np.int64), itemsize=np.array(case["it"]),
               nsteps=np.array(len(case["chain"])))
    g = O.global_pattern(case["dims"], extra, case["it"])
    pens = [O.make_pencils(case["grid"], case["dims"], d, p) for (d, p) in case["chain"]]
    for k, (d, p) in enumerate(case["chain"]):
        out[f"decomp{k}"] = np.array(d)
        out[f"perm{k}"] = np.array(p if p else (), dtype=np.int64)
    cur = O.scatter(g, pens[0], extra, dtype)
    for k in range(1, len(pens)):
        nxt = [O.OArray.undef(dtype, p, *extra) for p in pens[k]]
        O.transpose_all(nxt, cur)
        for r, a in enumerate(nxt):
            store(out, f"step{k}_rank{r}", np.ascontiguousarray(a.data.reshape(-1, order="F")).view(np.uint8))
        cur = nxt
    np.savez_compressed(os.path.join(HERE, case["name"] + ".npz"), **out)
    print("wrote", case["name"])
