"""GPU (-m gpu): the device finishing (bmbs_batch_finish) against the oracle's restatement of the reference, record by record.
Single end: vote-ordered reduction in std::sort's order, ungapped CIGAR check, coordinates (orc_finish_se: std::sort + the
literal loop + try_cigar_without_path + place); the introsort replay on lists of every size class.  Paired end: hit compaction,
single-side filter, pair pick, the two chosen hits' records (orc_finish_pe), thread and warp kernels."""
import subprocess

import numpy as np
import pytest

import bitmapperbs_b200 as B
from bitmapperbs_b200 import capi, simulate as S
from conftest import read_fastq
from oracle_binding import OracleIndex, std_sort_order

pytestmark = pytest.mark.gpu


def device_finish(ix, reads, params=None):
    flat, offs = capi.flatten(reads)
    b = B.Batch(ix, 0, len(reads) + 1, len(flat) + 64, max(1 << 18, 64 * len(reads)))
    p = params or capi.default_params()
    b.upload(flat, offs); b.run(p); b.finish()
    res, cand, used = b.download()
    fin, mism, fb = b.download_final()
    c = b.finish_counters()
    b.close()
    return res, cand[:used], fin, mism, fb, c


def assert_same_final(gfin, gmism, ofin, omism, res, cand, allow_host=0):
    host = gfin["status"] == capi.FIN_HOST
    assert host.sum() <= allow_host, f"{host.sum()} reads handed back to the host"
    m = ~host
    for f in ("status", "flags", "sbd", "nm", "mapq_fixed", "k", "chrom_pos"):
        assert np.array_equal(gfin[f][m], ofin[f][m]), f
    # the window may differ among equally voted windows that end at the same place (same alignment): compare where it ends
    hit = m & np.isin(gfin["status"], [capi.FIN_UNIQUE, capi.FIN_DP])
    assert np.array_equal(gfin["site"][hit] + gfin["end_site"][hit].astype(np.uint64), ofin["site"][hit] + ofin["end_site"][hit].astype(np.uint64))
    dp = m & (gfin["status"] == capi.FIN_DP)
    assert np.array_equal(gfin["site"][dp], ofin["site"][dp]) and np.array_equal(gfin["end_site"][dp], ofin["end_site"][dp])
    uq = np.nonzero(m & (gfin["status"] == capi.FIN_UNIQUE))[0]
    assert np.array_equal(gfin["n_aux"][uq], ofin["n_aux"][uq])
    for r in uq:
        a, n = int(gfin["aux_first"][r]), int(gfin["n_aux"][r]); b = int(ofin["aux_first"][r])
        assert np.array_equal(gmism[a:a + n], omism[b:b + n]), r
    # handed-back reads carry their whole window list
    for r in np.nonzero(host)[0]:
        a, n = int(gfin["aux_first"][r]), int(gfin["n_aux"][r])
        assert n == res["n_cand"][r]


# index environments: the device's grid, and every persistent and grid-stride launch sized for one SM -- each warp or block of
# finish_long, finish_huge, finish_sorted and finish_pe_long then takes many reads in turn
GRIDS = {"default": {}, "small_grid": {"BMBS_GRID_SMS": "1"}}


def load_index(prefix, env):
    import os
    old = {k: os.environ.get(k) for k in env}
    os.environ.update(env)
    try:
        return B.Index(prefix)
    finally:
        for k, v in old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


@pytest.fixture(scope="module", params=list(GRIDS))
def idx_pair(golden, request):
    ix = load_index(golden / "genome.fa.index", GRIDS[request.param]); ox = OracleIndex(golden / "genome.fa.index")
    yield ix, ox
    ix.close()


@pytest.mark.parametrize("amb_out", [0, 1])
def test_finished_records_match_oracle_golden_reads(golden, idx_pair, amb_out):
    ix, ox = idx_pair
    reads = [r[1] for r in read_fastq(golden / "se100.fq")] + [r[1] for r in read_fastq(golden / "se250.fq")]
    genome = b"".join(l.strip() for l in open(golden / "genome.fa", "rb") if not l.startswith(b">"))
    N = len(genome)
    reads += [b"ACGT" * 4, b"N" * 100, genome[:100], genome[N - 100:], genome[119950:120050], genome[119900:120000], genome[120000:120100],
              genome[5000:5050] + b"N" + genome[5051:5100], genome[7000:7017] + b"R" + genome[7018:7100], b"T" * 60, b"TG" * 40, genome[9000:9999]]
    p = capi.default_params(ambiguous_out=amb_out)
    res, cand, fin, mism, fb, c = device_finish(ix, reads, p)
    ofin, omism = ox.finish_se(reads, res, cand, ambiguous_out=bool(amb_out))
    assert_same_final(fin, mism, ofin, omism, res, cand)
    st = fin["status"]
    assert (st == capi.FIN_UNIQUE).sum() > 1000 and (st == capi.FIN_DP).sum() > 20 and c["reads_dp"] == (st == capi.FIN_DP).sum()


@pytest.mark.parametrize("amb_out", [0, 1])
def test_finished_records_on_high_copy_repeats(built, tmp_path, amb_out):
    """window lists of every size: <= 16 (stable insertion sort), longer ones whose outcome does not depend on the order, and
    the ones finish_sorted replays std::sort for (the counters must show that each class occurred)"""
    chroms = S.random_genome([700000, 500000], seed=321, repeat_fraction=0.7, repeat_copies=(40, 1500), repeat_len=(200, 700), repeat_div=(0.005, 0.06))
    S.write_fasta(tmp_path / "g.fa", chroms)
    subprocess.run([str(built["indexer"]), "g.fa"], cwd=tmp_path, check=True, stderr=subprocess.DEVNULL)
    g, st = S.concat_genome(chroms)
    m1, _ = S.simulate_fast(g, st, 8000, 150, 17, paired=False, indel_reads=0.2)
    reads = [bytes(r) for r in m1]
    ox = OracleIndex(tmp_path / "g.fa.index")
    for grid, env in GRIDS.items():
        ix = load_index(tmp_path / "g.fa.index", env)
        try:
            res, cand, fin, mism, fb, c = device_finish(ix, reads, capi.default_params(ambiguous_out=amb_out))
            ofin, omism = ox.finish_se(reads, res, cand, ambiguous_out=bool(amb_out))
            n = res["n_cand"][res["state"] == B.VERIFY]
            assert (n > 16).sum() > 100 and (n > 256).any(), grid
            assert c["reads_sort_replayed"] > 10, (grid, c)
            assert_same_final(fin, mism, ofin, omism, res, cand, allow_host=(n > 2048).sum())
        finally:
            ix.close()


def test_device_sort_replay_equals_std_sort():
    """the warp routine that replays std::sort's partitions (finish_sorted) against std::sort itself: 6000 vote lists of 1..2048
    entries -- random, few distinct values, periodic, sparse, ramps, all equal"""
    rng = np.random.default_rng(5)
    lists = []
    for it in range(6000):
        n = int(rng.integers(1, 2049)) if it % 10 == 0 else int(rng.integers(1, 200))
        vr = int(rng.integers(1, 29))
        mode = it % 6
        if mode == 0:
            v = rng.integers(1, vr + 1, size=n)
        elif mode == 1:
            v = 1 + (np.arange(n) % vr)
        elif mode == 2:
            v = np.where(rng.random(n) < 0.1, rng.integers(1, vr + 1, size=n), 1)
        elif mode == 3:
            v = 1 + (vr * np.arange(n) // n)
        elif mode == 4:
            v = np.full(n, vr)
        else:
            v = 1 + ((vr * np.arange(n)[::-1]) // n)
        lists.append(v.astype(np.uint32))
    orders, ok = capi.debug_sort_order(lists)
    assert ok.all()
    for v, o in zip(lists, orders):
        assert np.array_equal(o.astype(np.uint32), std_sort_order(v)), len(v)


# ---- paired end: finish_pe / finish_pe_long against the oracle's restatement of the reference's pair logic (orc_finish_pe) ----
def device_finish_pe(ix, mates, params):
    flat, offs = capi.flatten(mates)
    b = B.Batch(ix, 0, len(mates) + 2, len(flat) + 64, max(1 << 18, 96 * len(mates)))
    b.upload(flat, offs, pe=True); b.run(params)
    res, cand, used = b.download()                     # the verified hit lists as the pair logic finds them
    res, cand = res.copy(), cand[:used].copy()
    b.finish()                                         # (compacts the lists in place on the device)
    fin, mism, fb = b.download_final()
    c = b.finish_counters()
    b.close()
    assert len(fb) == 0
    return res, cand, fin, mism, c


def assert_same_pairs(gfin, gmism, ofin, omism):
    for f in ("status", "flags", "sbd", "nm", "k", "chrom_pos", "site", "end_site", "n_aux"):
        assert np.array_equal(gfin[f], ofin[f]), f
    for r in np.nonzero(gfin["n_aux"])[0]:
        a, n, b = int(gfin["aux_first"][r]), int(gfin["n_aux"][r]), int(ofin["aux_first"][r])
        assert np.array_equal(gmism[a:a + n], omism[b:b + n]), r


def mates_of(golden, name):
    comp = bytes.maketrans(b"ACGT", b"TGCA")
    a = [r[1] for r in read_fastq(golden / f"{name}_1.fq")]; b = [r[1].translate(comp)[::-1] for r in read_fastq(golden / f"{name}_2.fq")]
    return [x for p in zip(a, b) for x in p]


@pytest.mark.parametrize("pe_short", [None, "0"])
@pytest.mark.parametrize("name,sensitive,amb_out,extra", [("pe150", 0, 0, {}), ("pe150", 1, 1, {}), ("pe100h", 0, 1, {}), ("pe100h", 1, 0, {}),
                                                          ("pe100h", 0, 0, {"e_rate": 0.05, "min_ins": 100, "max_ins": 350})])
def test_finished_pairs_match_oracle_golden_reads(golden, idx_pair, monkeypatch, name, sensitive, amb_out, extra, pe_short):
    ix, ox = idx_pair
    if pe_short is not None:
        monkeypatch.setenv("BMBS_PE_FIN_SHORT", pe_short)       # every pair through the warp kernel
    mates = mates_of(golden, name)
    p = capi.default_params(sensitive=sensitive, ambiguous_out=amb_out, **extra)
    res, cand, fin, mism, c = device_finish_pe(ix, mates, p)
    ofin, omism = ox.finish_pe(mates, res, cand, e_rate=p.e_rate, min_ins=p.min_ins, max_ins=p.max_ins, sensitive=bool(sensitive), ambiguous_out=bool(amb_out))
    assert_same_pairs(fin, mism, ofin, omism)
    st = fin["status"][0::2]
    assert (st == capi.FIN_UNIQUE).sum() + (st == capi.FIN_DP).sum() > len(st) // 5
    assert c["reads_dp"] == (fin["status"] == capi.FIN_DP).sum()


@pytest.mark.parametrize("sensitive", [0, 1])
def test_finished_pairs_on_high_copy_repeats(built, tmp_path, sensitive):
    """hit lists of hundreds of entries per mate: the staged lists and the warp-parallel pair pick of finish_pe_long, ties among
    equally good pairs (ambiguous pairs, second_best_diff 0) included"""
    chroms = S.random_genome([700000, 500000], seed=322, repeat_fraction=0.7, repeat_copies=(40, 1500), repeat_len=(400, 1500), repeat_div=(0.0, 0.05))
    S.write_fasta(tmp_path / "g.fa", chroms)
    subprocess.run([str(built["indexer"]), "g.fa"], cwd=tmp_path, check=True, stderr=subprocess.DEVNULL)
    g, st = S.concat_genome(chroms)
    m1, m2 = S.simulate_fast(g, st, 5000, 120, 23)
    comp = bytes.maketrans(b"ACGT", b"TGCA")
    mates = [x for a, b in zip(m1, m2) for x in (bytes(a), bytes(b).translate(comp)[::-1])]
    ox = OracleIndex(tmp_path / "g.fa.index")
    for grid, env in GRIDS.items():
        ix = load_index(tmp_path / "g.fa.index", env)
        try:
            for amb_out in (0, 1):
                p = capi.default_params(sensitive=sensitive, ambiguous_out=amb_out)
                res, cand, fin, mism, c = device_finish_pe(ix, mates, p)
                n = res["n_cand"][0::2] + res["n_cand"][1::2]
                assert (n > 48).sum() > 20 and (n > 100).any(), n.max()       # (fast mode: filter_pairs has already thinned the lists)
                ofin, omism = ox.finish_pe(mates, res, cand, sensitive=bool(sensitive), ambiguous_out=bool(amb_out))
                assert_same_pairs(fin, mism, ofin, omism)
                if not amb_out:
                    assert (fin["status"][0::2] == capi.FIN_AMBIGUOUS).sum() > 5, grid
                else:
                    assert (fin["flags"][0::2] & 2).astype(bool).sum() > 5, grid
        finally:
            ix.close()
