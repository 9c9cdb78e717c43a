"""Pins the oracle: (1) the reference's documented known answers, (2) the
properties its own test-suite checks (test/transpose.jl, test/pencils.jl),
(3) the committed golden fixtures, (4) C port == NumPy restatement."""
import os

import numpy as np
import pytest

from oracle import pencil_oracle as O
from oracle import c_oracle
from util import CASES, DTYPES, beq, matches_golden

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def test_known_answers_from_reference_docs():
    # docs/src/index.md:92-94: dims (42,31,29); a rank holds (1:42, 16:23, 20:29), size (42,8,10)
    pens = O.make_pencils((4, 3), (42, 31, 29), (2, 3))
    hit = [p for p in pens if p.axes_local == (range(1, 43), range(16, 24), range(20, 30))]
    assert len(hit) == 1 and hit[0].size_local() == (42, 8, 10)
    # docs/src/Pencils.md:40-50: (16,32,64) on 2x2 -> size_local (16,16,32)
    assert all(p.size_local() == (16, 16, 32) for p in O.make_pencils((2, 2), (16, 32, 64), (2, 3)))
    # src/arrays.jl:19-31: local (10,20,30), perm (2,3,1) -> parent dims (20,30,10), u[i,j,k] == parent[j,k,i]
    (p,) = O.make_pencils((1, 1), (10, 20, 30), (2, 3), (2, 3, 1))
    assert p.size_local(True) == (20, 30, 10)
    g = O.global_pattern((10, 20, 30), (), 8)
    (u,) = O.scatter(g, [p], (), np.float64)
    G = O.gather([u])
    assert G[4, 14, 24].tobytes() == u.data[14, 24, 4].tobytes()
    # data_ranges.jl:4-9 by hand; complete_dims examples of data_ranges.jl:11-14
    assert [tuple(O.local_data_range(p, 4, 21)) for p in (1, 2, 3, 4)] == [
        (1, 2, 3, 4, 5), (6, 7, 8, 9, 10), (11, 12, 13, 14, 15), (16, 17, 18, 19, 20, 21)]
    assert O.complete_dims(5, (2, 3), (42, 12)) == (1, 42, 12, 1, 1)
    assert O.complete_dims(5, (3, 2), (42, 12)) == (1, 12, 42, 1, 1)
    # MPI_Dims_create grids quoted in SURVEY.md section 8
    assert [O.dims_create(n, 2) for n in (2, 4, 6, 8, 12)] == [(2, 1), (2, 2), (3, 2), (4, 2), (4, 3)]
    # get_remote_indices docstring (Transpositions.jl:537-538): coords (2,3,5), R=1 -> (:,3,5)
    assert O.get_remote_indices(1, (2, 3, 5), 4) == [(1, 3, 5), (2, 3, 5), (3, 3, 5), (4, 3, 5)]


@pytest.mark.parametrize("grid", [(1, 1), (2, 1), (1, 2), (2, 2), (2, 3), (3, 2), (4, 2)])
def test_reference_transpose_testset(grid):
    """test/transpose.jl:24-77 restated."""
    dims = (16, 21, 41)
    g = O.global_pattern(dims, (), 8)
    p1 = O.make_pencils(grid, dims, (2, 3))
    p2 = O.make_pencils(grid, dims, (1, 3), (2, 3, 1))
    p3 = O.make_pencils(grid, dims, (1, 2), (3, 2, 1))
    u1 = O.scatter(g, p1, (), np.float64)
    G = O.gather(u1)
    new = lambda ps: [O.OArray.undef(np.float64, p) for p in ps]
    u2, u3 = new(p2), new(p3)
    with pytest.raises(ValueError):
        O.transpose_all(u3, u1)
    O.transpose_all(u2, u1)
    assert beq(O.gather(u2), G)
    O.transpose_all(u3, u2)
    assert beq(O.gather(u3), G)
    u2b = new(p2)
    O.transpose_all(u2b, u3)
    assert beq(O.gather(u2b), G)
    u1b = new(p1)
    O.transpose_all(u1b, u2b)
    assert all(beq(a.data, b.data) for a, b in zip(u1, u1b))
    for decomp in [(1, 3), (2, 1)]:  # no permutation; unsorted decomp_dims (#57)
        v = new(O.make_pencils(grid, dims, decomp))
        O.transpose_all(v, u1)
        assert beq(O.gather(v), G)


@pytest.mark.parametrize("case", CASES, ids=[c["name"] for c in CASES])
def test_c_port_equals_numpy_oracle(case):
    dtype = DTYPES[case["it"]]
    extra = case["extra"]
    g = O.global_pattern(case["dims"], extra, case["it"])
    pens = [O.make_pencils(case["grid"], case["dims"], d, p) for (d, p) in case["chain"]]
    cur = O.scatter(g, pens[0], extra, dtype)
    for k in range(1, len(pens)):
        nxt = [O.OArray.undef(dtype, p, *extra) for p in pens[k]]
        O.transpose_all(nxt, cur)
        (d0, p0), (d1, p1) = case["chain"][k - 1], case["chain"][k]
        ct = c_oracle.CTranspose(case["grid"], case["dims"], d0, p0, d1, p1, extra, dtype)
        srcs = [np.ascontiguousarray(a.data.reshape(-1, order="F")) for a in cur]
        for nth in (1, 3, 8):
            dsts = [np.zeros(max(1, a.data.size), dtype=dtype) for a in nxt]
            ct.run(srcs, dsts, nthreads=nth)
            for r, a in enumerate(nxt):
                assert beq(dsts[r][:a.data.size], a.data.reshape(-1, order="F")), (k, r, nth)
        cur = nxt


def test_golden_fixtures():
    """tests/golden/*.npz were produced by tests/golden/make_golden.py from this
    oracle at commit time; they freeze its behaviour (regression pin); the GPU path is
    compared against the same files in tests/test_gpu_transpose.py::
    test_gpu_path_against_committed_golden_fixtures."""
    files = sorted(f for f in os.listdir(GOLD) if f.endswith(".npz"))
    assert files, "golden fixtures missing"
    for f in files:
        z = np.load(os.path.join(GOLD, f))
        grid, dims = tuple(z["grid"]), tuple(z["dims"])
        extra, it = tuple(z["extra"]), int(z["itemsize"])
        dtype = DTYPES[it]
        chain = [(tuple(z[f"decomp{k}"]), tuple(z[f"perm{k}"]) or None) for k in range(int(z["nsteps"]))]
        g = O.global_pattern(dims, extra, it)
        pens = [O.make_pencils(grid, dims, d, p) for (d, p) in chain]
        cur = O.scatter(g, pens[0], extra, dtype)
        for k in range(1, len(pens)):
            nxt = [O.OArray.undef(dtype, p, *extra) for p in pens[k]]
            O.transpose_all(nxt, cur)
            for r, a in enumerate(nxt):
                assert matches_golden(z, k, r, a.data.reshape(-1, order="F").view(np.uint8)), (f, k, r)
            cur = nxt
