"""SURVEY.md 8f-1 (CIGAR + score): host/postprocess.hpp refine_alignment -- the CPU restatement the oracle CLI and the parity
tests use -- against the REFERENCE's own fast_recalculate_bs_Cigar (ksw.cpp:2578-3148, compiled into oracle/_ref/libref_ksw.so)
on seeded random alignments: substitutions only, insertions, deletions, N in read and window, bisulfite T/C pairs, both
strands, reversed qualities (mate 2), quality-dependent penalties, non-default scoring.  Bit-exact: start, end, NM, score, CIGAR.
Where the reference is not built, its results are compared through their stored digest (tests/reference_sha256.py)."""
import ctypes as C
from pathlib import Path

import numpy as np
import pytest

import reference_sha256
from oracle_binding import lib

ROOT = Path(__file__).resolve().parent.parent
REF = ROOT / "oracle/_ref/libref_ksw.so"


def make_case(rng, L, k, n_sub, n_ins, n_del, n_frac):
    """window of L + 2k bases and a read derived from window[k : k + L] with the given edits; returns what the verifier
    would report: (end_site, err) from a plain banded edit distance is not needed -- the refinement takes them as inputs,
    so they come from the true edit script (the DP must then find an alignment of its own)."""
    wlen = L + 2 * k
    win = rng.choice(list(b"ACGT"), size=wlen).astype(np.uint8)
    src = list(win[k:k + L + n_del])
    for _ in range(n_del):
        del src[int(rng.integers(5, len(src) - 5))]
    for _ in range(n_ins):
        src.insert(int(rng.integers(5, len(src) - 5)), int(rng.choice(list(b"ACGT"))))
    read = np.array(src[:L], dtype=np.uint8)
    if len(read) < L:
        read = np.concatenate([read, rng.choice(list(b"ACGT"), size=L - len(read)).astype(np.uint8)])
    for _ in range(n_sub):
        p = int(rng.integers(0, L)); read[p] = rng.choice([c for c in b"ACGT" if c != read[p]])
    conv = (read == ord("C")) & (rng.random(L) < 0.9)          # bisulfite: read T faces window C
    read[conv] = ord("T")
    if n_frac:
        read[rng.random(L) < n_frac] = ord("N")
        win[rng.random(wlen) < n_frac / 2] = ord("N")
    qual = (33 + rng.integers(2, 42, size=L)).astype(np.uint8)
    return win.tobytes(), read.tobytes(), qual.tobytes()


def edit_end(win, read, k):
    """plain bisulfite-aware banded DP: best (err, end) over the last row, as kernel 3 would report it"""
    L, W = len(read), len(win)
    INF = 10 ** 6
    prev = [0 if j <= 2 * k else INF for j in range(W + 1)]
    for i in range(1, L + 1):
        cur = [INF] * (W + 1)
        for j in range(max(1, i), min(W, i + 2 * k) + 1):
            t, p = read[i - 1], win[j - 1]
            m = 0 if (t == p or (t == ord("T") and p == ord("C"))) and t != ord("N") else 1
            cur[j] = min(prev[j - 1] + m, prev[j] + 1, cur[j - 1] + 1)
        prev = cur
    best = min(range(L, min(W, L + 2 * k) + 1), key=lambda j: (prev[j], abs(j - (L + k))))
    return prev[best], best - 1


@pytest.mark.parametrize("seed,L,k,scoring", [(1, 100, 8, (6, 2, 1, 5, 3, 33)), (2, 150, 12, (6, 2, 1, 5, 3, 33)), (3, 60, 4, (6, 2, 1, 5, 3, 33)),
                                              (4, 150, 12, (4, 1, 2, 3, 1, 33)), (5, 120, 9, (6, 2, 1, 5, 3, 64))])
def test_refine_matches_reference(seed, L, k, scoring):
    ref = C.CDLL(str(REF)) if REF.exists() else None
    orc = lib()
    rng = np.random.default_rng(seed)
    mp_max, mp_min, n_pen, go, ge, qb = scoring
    results = []
    for case in range(400):
        n_ins, n_del = int(rng.integers(0, 3)), int(rng.integers(0, 3))
        n_sub = int(rng.integers(0, 4))
        win, read, qual = make_case(rng, L, k, n_sub, n_ins, n_del, 0.01 if case % 5 == 0 else 0.0)
        if qb == 64:
            qual = bytes(q + 31 for q in qual)
        err, end = edit_end(win, read, k)
        if err > k:
            continue
        for forward in (1, 0):
            for rq in (0, 1):
                s2, e2, n2, sc2 = C.c_int(), C.c_uint64(), C.c_uint(), C.c_int(); c2 = C.create_string_buffer(4096)
                orc.orc_refine(win, len(win), read, L, k, end, err, forward, qual, rq, mp_max, mp_min, n_pen, go, ge, qb,
                               C.byref(s2), C.byref(e2), C.byref(n2), C.byref(sc2), c2, 4096)
                got = (s2.value, e2.value, n2.value, sc2.value, c2.value)
                if ref:
                    s1, e1, n1, sc1 = C.c_int(), C.c_uint64(), C.c_uint(), C.c_int(); c1 = C.create_string_buffer(4096)
                    ref.ref_cigar(win, len(win), read, L, k, end, err, forward, mp_max, mp_min, n_pen, go, ge, qual, rq, qb,
                                  C.byref(s1), C.byref(e1), C.byref(n1), C.byref(sc1), c1)
                    assert (s1.value, e1.value, n1.value, sc1.value, c1.value) == got, (case, forward, rq, read, win)
                results.append(got)
    assert len(results) > 800
    reference_sha256.check(f"refine:{seed}", repr(results).encode())
