"""GPU (-m gpu), SURVEY.md 8f-1: the refinement kernels behind bmbs_refine (refine_warp: a warp per alignment for bands of up
to 32 cells; refine_dp: a thread per alignment for wider bands, and for every band with BMBS_REFINE_THREAD=1) against the CPU
refinement (host/postprocess.hpp banded_affine_align + fix_ends + recount_nm, pinned to the reference's
fast_recalculate_bs_Cigar by tests/test_refine_vs_reference.py): score, first / last window position, NM and every final
operation identical, on windows of both strands, reads with substitutions, insertions, deletions and N, k up to 31, read
lengths 30..640, windows that leave the strand, non-default scoring and phred64 qualities.  The whole-program SAM
comparisons of test_gpu_parity.py cover the host glue around it."""
import os
import numpy as np
import pytest

import bitmapperbs_b200 as B
from bitmapperbs_b200 import capi
from oracle_binding import OracleIndex, refine_final

pytestmark = pytest.mark.gpu


# small_grid: refine_warp's grid sized for one SM (16 blocks of 4 warps), so that each warp takes many alignments in turn
GRIDS = {"default": {}, "small_grid": {"BMBS_GRID_SMS": "1"}}


def load_index(golden, env):
    old = {k: os.environ.get(k) for k in env}
    os.environ.update(env)
    try:
        return B.Index(golden / "genome.fa.index")
    finally:
        for k, v in old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


@pytest.fixture(scope="module", params=list(GRIDS))
def gidx(golden, request):
    ix = load_index(golden, GRIDS[request.param])
    yield ix
    ix.close()


@pytest.fixture(scope="module")
def oidx(golden):
    return OracleIndex(golden / "genome.fa.index")


def make_items(oidx, rng, n, lengths, scoring):
    import ctypes as C
    from oracle_binding import lib
    N = oidx.N
    seqs, quals, items = bytearray(), bytearray(), np.zeros(n, dtype=capi.RefineItem)
    for i in range(n):
        L = int(rng.choice(lengths)); k = min(31, int(0.08 * L)) if i % 7 else int(rng.integers(0, 32))
        wlen = L + 2 * k
        strand = int(rng.integers(0, 2))
        kind = i % 23
        if kind == 0:
            site = strand * N + N - int(rng.integers(0, wlen))          # leaves the strand: all-N window
        elif kind == 1:
            site = strand * N + int(rng.integers(0, 3))
        else:
            site = strand * N + int(rng.integers(0, N - wlen))
        win = C.create_string_buffer(wlen + 8)
        lib().orc_window(oidx.h, site, wlen, win)
        w = np.frombuffer(win.raw[:wlen], dtype=np.uint8).copy()
        w[w == 0] = ord("A")
        src = list(w[k:k + L + 4])
        for _ in range(int(rng.integers(0, 3))):
            if len(src) > 12:
                del src[int(rng.integers(5, len(src) - 5))]
        for _ in range(int(rng.integers(0, 3))):
            if len(src) > 12:
                src.insert(int(rng.integers(5, len(src) - 5)), int(rng.choice(list(b"ACGT"))))
        read = np.array((src + list(rng.choice(list(b"ACGT"), size=L)))[:L], dtype=np.uint8)
        for _ in range(int(rng.integers(0, 5))):
            read[int(rng.integers(0, L))] = rng.choice(list(b"ACGTN"))
        conv = (read == ord("C")) & (rng.random(L) < 0.9)
        read[conv] = ord("T")
        q = (scoring[5] + rng.integers(0, 45, size=L)).astype(np.uint8)
        items[i] = (site, len(seqs), L, k, 0)
        seqs += read.tobytes(); quals += q.tobytes()
    return bytes(seqs), bytes(quals), items


@pytest.mark.parametrize("thread_kernel", [0, 1])
@pytest.mark.parametrize("seed,lengths,scoring", [(11, [100, 150], (6, 2, 1, 5, 3, 33)), (12, [30, 64, 250, 640], (6, 2, 1, 5, 3, 33)),
                                                  (13, [100, 151], (4, 1, 2, 3, 1, 33)), (14, [125], (6, 2, 1, 5, 3, 64))])
def test_refine_matches_cpu(gidx, oidx, seed, lengths, scoring, thread_kernel):
    rng = np.random.default_rng(seed)
    seqs, quals, items = make_items(oidx, rng, 1500, lengths, scoring)
    rf = B.Refiner(gidx)
    if thread_kernel:
        os.environ["BMBS_REFINE_THREAD"] = "1"
    try:
        res, ops = rf.refine(seqs, quals, items, scoring)
    finally:
        os.environ.pop("BMBS_REFINE_THREAD", None)
    assert int(res["n_ops"].sum()) == len(ops)
    assert (2 * items["k"].astype(int) + 1 <= 32).sum() > 300 and (2 * items["k"].astype(int) + 1 > 32).sum() > 50      # both kernels have work
    for i, it in enumerate(items):
        o, L = int(it["seq_off"]), int(it["len"])
        score, qb, qe, nm, cops = refine_final(oidx, it["site"], seqs[o:o + L], quals[o:o + L], int(it["k"]), scoring)
        r = res[i]
        assert (int(r["score"]), int(r["qb"]), int(r["qe"]), int(r["nm"])) == (score, qb, qe, nm), (i, it)
        assert np.array_equal(ops[int(r["ops_off"]): int(r["ops_off"]) + int(r["n_ops"])], cops), (i, it)
    rf.close()


def test_refine_empty_and_reuse(golden, oidx):
    for grid, env in GRIDS.items():
        ix = load_index(golden, env)
        rf = B.Refiner(ix)
        res, ops = rf.refine(b"", b"", np.zeros(0, dtype=capi.RefineItem))
        assert len(res) == 0 and len(ops) == 0
        rng = np.random.default_rng(5)
        for n in (3, 700, 40):                                     # buffers grow and are reused
            seqs, quals, items = make_items(oidx, rng, n, [100], (6, 2, 1, 5, 3, 33))
            res, ops = rf.refine(seqs, quals, items)
            s0, qb0, qe0, nm0, c0 = refine_final(oidx, items[0]["site"], seqs[:100], quals[:100], int(items[0]["k"]))
            assert (int(res[0]["score"]), int(res[0]["qb"]), int(res[0]["qe"]), int(res[0]["nm"])) == (s0, qb0, qe0, nm0), (grid, n)
        rf.close()
        ix.close()
