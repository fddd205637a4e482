#!/usr/bin/env python3
"""CIGAR refinement microbench (SURVEY.md 8f-1): n alignments of length L and error threshold k (default L = 150, k = 12) with
one indel each through bmbs_refine (H2D of reads + qualities, refine_warp<1> for k <= 15 or refine_warp<2> for k 16..31, D2H
of scores, NM and final operations), next to the same refinement on the host cores (host/postprocess.hpp through the oracle
library, one thread).  Cells = n * L * (2k + 1).

  python tools/bench_refine.py [--n 131072] [--L 150] [--k 12]          (run under `ncu -k regex:refine_` for the kernel alone)
"""
import argparse, gzip, json, shutil, subprocess, sys, tempfile, time
from pathlib import Path
import numpy as np
ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT)); sys.path.insert(0, str(ROOT / "tests"))
import bitmapperbs_b200 as B
from bitmapperbs_b200 import capi

ap = argparse.ArgumentParser(); ap.add_argument("--n", type=int, default=131072); ap.add_argument("--cpu-sample", type=int, default=2000)
ap.add_argument("--L", type=int, default=150); ap.add_argument("--k", type=int, default=12); a = ap.parse_args()
with tempfile.TemporaryDirectory() as td:
    td = Path(td)
    with gzip.open(ROOT / "tests/golden/genome.fa.gz", "rb") as f, open(td / "genome.fa", "wb") as o:
        shutil.copyfileobj(f, o)
    subprocess.run([str(ROOT / "bitmapperbs_b200/_build/bmbs-index"), str(td / "genome.fa")], check=True, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
    genome = np.frombuffer(b"".join(l.strip() for l in open(td / "genome.fa", "rb") if not l.startswith(b">")).upper(), dtype=np.uint8)
    L, k, n = a.L, a.k, a.n
    rng = np.random.default_rng(1)
    sites = rng.integers(1000, len(genome) - 1000, size=n)
    reads = np.empty((n, L), dtype=np.uint8)
    for i in range(n):                                           # window[k : k + L + 1] with one base deleted
        w = genome[sites[i] + k: sites[i] + k + L + 1]; d = 20 + i % 100
        reads[i, :d] = w[:d]; reads[i, d:] = w[d + 1:]
    items = np.zeros(n, dtype=capi.RefineItem); items["site"] = sites; items["seq_off"] = np.arange(n) * L; items["len"] = L; items["k"] = k
    seqs = reads.tobytes(); quals = bytes([ord("I")]) * (n * L)
    idx = B.Index(td / "genome.fa.index"); rf = B.Refiner(idx)
    rf.refine(seqs, quals, items)                                # warm-up: buffers grow
    best = 1e9; kbest = 1e9
    for _ in range(5):
        t = time.perf_counter(); res, ops = rf.refine(seqs, quals, items); best = min(best, time.perf_counter() - t); kbest = min(kbest, rf.kernel_ms())
    cells = n * L * (2 * k + 1)
    out = {"alignments": n, "L": L, "k": k, "call_ms": best * 1e3, "alignments_per_s": n / best, "gcups_call": cells / best / 1e9,
           "kernel_ms": kbest, "alignments_per_s_kernel": n / (kbest / 1e3), "gcups_kernel": cells / (kbest / 1e3) / 1e9,
           "ops_returned": int(len(ops)), "with_indel": int((res["n_ops"] > 1).sum())}
    from oracle_binding import OracleIndex, refine_final
    oi = OracleIndex(td / "genome.fa.index"); m = min(a.cpu_sample, n)
    t = time.perf_counter()
    for i in range(m):
        refine_final(oi, int(sites[i]), seqs[i * L:(i + 1) * L], quals[:L], k)
    dt = time.perf_counter() - t
    out["cpu_one_thread_alignments_per_s"] = m / dt
    print(json.dumps(out))
    rf.close(); idx.close()
