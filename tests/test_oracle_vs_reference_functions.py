"""CPU: pins the restated hot-path functions against the reference's OWN code (oracle/_ref/libref_*.so, compiled
from /root/reference by oracle/build_ref.sh): banded bit-vector verification in all three lane widths and the
FM-index primitives.  Where the compiled reference is absent, the oracle's results are compared with the reference's
through their stored digest (tests/reference_sha256.py)."""
import ctypes as C
from pathlib import Path

import numpy as np
import reference_sha256
from oracle_binding import OracleIndex, lib as olib

ROOT = Path(__file__).resolve().parent.parent
BPM = ROOT / "oracle/_ref/libref_bpm.so"
FM = ROOT / "oracle/_ref/libref_fm.so"


def _cases(rng, n):
    for _ in range(n):
        L = int(rng.integers(18, 260))
        k = min(31, int(0.08 * L)) if rng.random() < 0.7 else int(rng.integers(0, 32))
        plen = L + 2 * k
        win = rng.choice(np.frombuffer(b"ACGT", dtype=np.uint8), size=plen)
        mode = rng.random()
        read = win[k:k + L].copy()
        if mode < 0.1:
            read = rng.choice(np.frombuffer(b"ACGT", dtype=np.uint8), size=L)          # decoy
        else:
            c = (read == ord("C")) & (rng.random(L) < 0.9); read[c] = ord("T")          # bisulfite
            for _e in range(int(rng.integers(0, k + 3))):
                p = int(rng.integers(0, len(read)))
                r = rng.random()
                if r < 0.6:
                    read[p] = rng.choice(np.frombuffer(b"ACGTN", dtype=np.uint8))
                elif r < 0.8 and len(read) > 20:
                    read = np.delete(read, p)
                else:
                    read = np.insert(read, p, rng.choice(np.frombuffer(b"ACGT", dtype=np.uint8)))
            if len(read) < L:
                read = np.concatenate([read, rng.choice(np.frombuffer(b"ACGT", dtype=np.uint8), size=L - len(read))])
            read = read[:L]
        if mode > 0.97:
            win = np.zeros(plen, dtype=np.uint8)                                            # out-of-genome window
        yield win.tobytes(), read.tobytes(), L, k


def test_bpm_matches_reference_all_lane_widths(built):
    R = C.CDLL(str(BPM)) if BPM.exists() else None
    O = olib()
    rng = np.random.default_rng(7)
    batch = []
    for win, read, L, k in _cases(rng, 6000):
        e_or = C.c_uint32(0)
        s_or = O.orc_bpm(win + b"\0" * 40, read + b"\0", L, k, C.byref(e_or))
        batch.append((win, read, L, k, s_or, e_or.value))
    assert sum(s >= 0 for *_, s, _e in batch) > 2000
    reference_sha256.check("bpm", repr([(s, e) for *_, s, e in batch]).encode())
    if R is None:
        return
    for win, read, L, k, s_or, e_or in batch:
        e_ref = C.c_uint(0)
        s_ref = R.ref_bpm_scalar(win + b"\0" * 40, L + 2 * k, read + b"\0", L, k, C.byref(e_ref))
        assert (s_ref, e_ref.value) == (s_or, e_or), (L, k)
    # SIMD variants: same read, 8 (or 4) windows
    for win, read, L, k, s_ref, e_ref in batch[:1500]:
        plen = L + 2 * k; stride = plen + 64
        buf = bytearray(stride * 8)
        wins = [win] + [bytes(rng.choice(np.frombuffer(b"ACGT", dtype=np.uint8), size=plen)) for _ in range(7)]
        for i, w in enumerate(wins):
            buf[i * stride:i * stride + plen] = w
        sites = (C.c_int * 8)(); errs = (C.c_uint * 8)()
        cb = (C.c_char * len(buf)).from_buffer(buf)
        if k <= 15:
            R.ref_bpm_8(cb, stride, plen, read + b"\0", L, k, sites, errs)
            assert (sites[0], errs[0]) == (s_ref, e_ref)
        R.ref_bpm_4(cb, stride, plen, read + b"\0", L, k, sites, errs)
        assert (sites[0], errs[0]) == (s_ref, e_ref)


def test_fm_primitives_match_reference(golden, built):
    R = None
    if FM.exists():
        R = C.CDLL(str(FM))
        R.ref_fm_lf.restype = C.c_uint64; R.ref_fm_lf.argtypes = [C.c_uint64, C.c_int]
        R.ref_fm_seed.restype = C.c_uint64; R.ref_fm_count.restype = C.c_uint64
        R.ref_fm_locate.argtypes = [C.c_uint64, C.POINTER(C.c_uint64)]
        assert R.ref_fm_load(str(golden / "genome.fa.index.bs").encode()) == 0
    ix = OracleIndex(golden / "genome.fa.index")
    O = olib()
    n_rows = 2 * ix.N + 1
    rng = np.random.default_rng(3)
    ours = []          # every oracle result below, in order: compared with the reference's through the stored digest
    for row in list(rng.integers(0, n_rows, size=20000)) + [0, 1, n_rows - 1, n_rows]:
        for c in range(3):
            ours.append(O.orc_lf(ix.h, int(row), c))
            if R:
                assert R.ref_fm_lf(int(row), c) == ours[-1]
    for row in list(rng.integers(0, n_rows, size=5000)) + [0, n_rows - 1]:
        b = C.c_uint64(0)
        assert O.orc_locate(ix.h, int(row), C.byref(b)) == 1
        ours.append(b.value)
        if R:
            a = C.c_uint64(0)
            assert R.ref_fm_locate(int(row), C.byref(a)) == 1 and a.value == b.value
    # seeds: patterns cut from the converted double-strand text (reversed reads) plus noise
    genome = b"".join(l.strip() for l in open(golden / "genome.fa", "rb") if not l.startswith(b">"))
    for _ in range(3000):
        L = int(rng.integers(16, 140)); p = int(rng.integers(0, len(genome) - 200))
        s = bytearray(genome[p:p + L].replace(b"C", b"T")[::-1])
        for _e in range(int(rng.integers(0, 3))):
            s[int(rng.integers(0, L))] = rng.choice(np.frombuffer(b"AGTN", dtype=np.uint8))
        s = bytes(s)
        u64 = C.c_uint64
        b = [u64(5), u64(9), u64(0)]
        h2 = O.orc_seed(ix.h, s + b"\0", L, *[C.byref(x) for x in b])
        ours += [h2, b[2].value] + ([b[0].value, b[1].value] if h2 else [])
        if R:
            a = [u64(5), u64(9), u64(0)]
            h1 = R.ref_fm_seed(s + b"\0", u64(L), *[C.byref(x) for x in a])
            assert (h1, a[2].value) == (h2, b[2].value)
            if h1:
                assert (a[0].value, a[1].value) == (b[0].value, b[1].value)
        b = [u64(5), u64(9)]
        h2 = O.orc_count(ix.h, s + b"\0", L, *[C.byref(x) for x in b])
        ours += [h2, b[0].value, b[1].value]
        if R:
            a = [u64(5), u64(9)]
            h1 = R.ref_fm_count(s + b"\0", u64(L), *[C.byref(x) for x in a])
            assert h1 == h2 and (a[0].value, a[1].value) == (b[0].value, b[1].value)
    reference_sha256.check("fm_primitives", repr(ours).encode())
