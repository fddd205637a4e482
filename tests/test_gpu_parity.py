"""GPU (-m gpu): the CUDA path, called through the C ABI, against the oracle restatement on the same seeded inputs,
against the committed golden SAM of the real reference, and -- at larger sizes -- through size-independent
properties.  Integer / index work: everything is compared bit-exactly."""
import subprocess
from pathlib import Path

import numpy as np
import pytest

import bitmapperbs_b200 as B
import reference_sha256
from bitmapperbs_b200 import capi, simulate as S
from conftest import read_fastq, revcomp, sam_body
from oracle_binding import OracleIndex

pytestmark = pytest.mark.gpu
ROOT_DIR = Path(__file__).resolve().parent.parent
ACGT = np.frombuffer(b"ACGT", dtype=np.uint8)


# index residency variants (DESIGN.md §3): what the loader picks for a genome this small (dense suffix array, 16-mer table
# only), the on-disk 1/8 suffix-array sampling with an 18-mer deep seed table, and the 20-mer table a 100 Mbp genome gets
# and the layout of texts beyond 2^32 rows (bits 32..39 of every suffix-array value in their own byte array) forced onto
# the small index together with the 20-mer table and the dense suffix array -- what a 3.1 Gbp genome gets; and the default
# index with every persistent and grid-stride launch sized for one SM, so that each lane, warp and block of those kernels
# takes many reads, windows and lists in turn (a batch of the suite is otherwise far smaller than one wave of their grids)
@pytest.fixture(scope="module", params=["default", "sampled_sa+18mer", "20mer", "wide_sa+20mer", "small_grid"])
def gidx(golden, request):
    import os
    env = {"default": {}, "sampled_sa+18mer": {"BMBS_SA": "sampled", "BMBS_KMER": "18"}, "20mer": {"BMBS_KMER": "20"},
           "wide_sa+20mer": {"BMBS_FORCE_WIDE": "1", "BMBS_KMER": "20", "BMBS_SA": "dense"}, "small_grid": {"BMBS_GRID_SMS": "1"}}[request.param]
    old = {k: os.environ.get(k) for k in ("BMBS_SA", "BMBS_KMER", "BMBS_FORCE_WIDE", "BMBS_GRID_SMS")}
    os.environ.update(env)
    try:
        ix = B.Index(golden / "genome.fa.index")
    finally:
        for k, v in old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v
    yield ix
    ix.close()


@pytest.fixture(scope="module")
def oidx(golden):
    return OracleIndex(golden / "genome.fa.index")


def assert_same_records(gres, gcand, ores, ocand, compare_vote=True):
    for f in ("state", "n_cand", "is_multiple_map"):
        assert np.array_equal(gres[f], ores[f]), f
    m = np.isin(gres["state"], [B.EXACT_UNIQUE, B.ONE_MISMATCH])
    assert np.array_equal(gres["site"][m], ores["site"][m])
    m3 = gres["state"] == B.ONE_MISMATCH
    assert np.array_equal(gres["one_mismatch_pos"][m3], ores["one_mismatch_pos"][m3])
    assert len(gcand) == len(ocand)
    assert np.array_equal(gres["first_cand"], ores["first_cand"])
    for f in ("site", "end_site", "err"):
        assert np.array_equal(gcand[f], ocand[f]), f
    if compare_vote:
        assert np.array_equal(gcand["vote"], ocand["vote"])


def test_single_end_records_match_oracle(golden, gidx, oidx):
    reads = [r[1] for r in read_fastq(golden / "se100.fq")] + [r[1] for r in read_fastq(golden / "se250.fq")]
    gres, gcand = gidx.map_batch_se(reads)
    ores, ocand = oidx.map_se(reads)
    assert_same_records(gres, gcand, ores, ocand)
    assert (gres["state"] == B.VERIFY).sum() > 100 and (gres["state"] == B.EXACT_UNIQUE).sum() > 100


def test_paired_end_records_match_oracle(golden, gidx, oidx):
    m1 = read_fastq(golden / "pe150_1.fq"); m2 = read_fastq(golden / "pe150_2.fq")
    mates = []
    for a, b in zip(m1, m2):
        mates += [a[1], revcomp(b[1])]
    gres, gcand = gidx.map_batch_pe(mates)
    ores, ocand = oidx.map_pe(mates)
    v = np.repeat(gres["state"] == B.VERIFY, gres["n_cand"])
    assert_same_records(gres, gcand, ores, ocand, compare_vote=False)
    assert np.array_equal(gcand["vote"][v], ocand["vote"][v])


def _slices(res, cand):
    """per-read slices of cand[] laid end to end (offsets differ between implementations, contents must not)"""
    idx = np.concatenate([np.arange(f, f + n) for f, n in zip(res["first_cand"].astype(np.int64), res["n_cand"].astype(np.int64))] or [np.zeros(0, np.int64)])
    return cand[idx]


@pytest.mark.parametrize("name", ["pe150", "pe100h"])
def test_sensitive_pairing_records_match_oracle(golden, gidx, oidx, name):
    """--pe --sensitive: final hit lists of both mates (primary hits, mate-filtered secondary hits, re-seeded secondaries)"""
    m1 = read_fastq(golden / f"{name}_1.fq"); m2 = read_fastq(golden / f"{name}_2.fq")
    mates = []
    for a, b in zip(m1, m2):
        mates += [a[1], revcomp(b[1])]
    gres, gcand = gidx.map_batch_pe(mates, params=capi.default_params(sensitive=1))
    ores, ocand, reseeded = oidx.map_pe_sensitive(mates)
    for f in ("state", "n_cand", "is_multiple_map"):
        assert np.array_equal(gres[f], ores[f]), f
    m = np.isin(gres["state"], [B.EXACT_UNIQUE, B.ONE_MISMATCH])
    assert np.array_equal(gres["site"][m], ores["site"][m])
    gs, os_ = _slices(gres, gcand), _slices(ores, ocand)
    for f in ("site", "end_site", "err"):
        assert np.array_equal(gs[f], os_[f]), f
    if name == "pe100h":
        assert reseeded.sum() > 100 and (ores["n_cand"][reseeded == 1] > 0).sum() > 3   # the re-seeding round is exercised and finds hits


@pytest.mark.parametrize("e_rate,seed_len,min_ins,max_ins", [(0.04, 20, 0, 500), (0.12, 40, 100, 1000), (0.2, 30, 0, 300)])
def test_non_default_parameters_match_oracle(golden, gidx, oidx, e_rate, seed_len, min_ins, max_ins):
    """-e / --seed / --min / --max other than the defaults, single end, pairs and sensitive pairs"""
    se = [r[1] for r in read_fastq(golden / "se100.fq")][:1500] + [r[1] for r in read_fastq(golden / "se250.fq")][:300]
    prm = capi.default_params(e_rate=e_rate, seed_len=seed_len, min_ins=min_ins, max_ins=max_ins)
    gres, gcand = gidx.map_batch_se(se, params=prm)
    ores, ocand = oidx.map_se(se, e_rate=e_rate, seed_len=seed_len)
    assert_same_records(gres, gcand, ores, ocand)
    m1 = read_fastq(golden / "pe100h_1.fq")[:1200]; m2 = read_fastq(golden / "pe100h_2.fq")[:1200]
    mates = []
    for a, b in zip(m1, m2):
        mates += [a[1], revcomp(b[1])]
    gres, gcand = gidx.map_batch_pe(mates, params=prm)
    ores, ocand = oidx.map_pe(mates, e_rate=e_rate, seed_len=seed_len, min_ins=min_ins, max_ins=max_ins)
    v = np.repeat(gres["state"] == B.VERIFY, gres["n_cand"])
    assert_same_records(gres, gcand, ores, ocand, compare_vote=False)
    assert np.array_equal(gcand["vote"][v], ocand["vote"][v])
    prm.sensitive = 1
    gres, gcand = gidx.map_batch_pe(mates, params=prm)
    ores, ocand, _ = oidx.map_pe_sensitive(mates, e_rate=e_rate, seed_len=seed_len, min_ins=min_ins, max_ins=max_ins)
    for f in ("state", "n_cand", "is_multiple_map"):
        assert np.array_equal(gres[f], ores[f]), f
    gs, os_ = _slices(gres, gcand), _slices(ores, ocand)
    for f in ("site", "end_site", "err"):
        assert np.array_equal(gs[f], os_[f]), f


def test_high_copy_repeats_every_candidate_sort_tier(built, tmp_path):
    """a genome of high-copy repeat families: candidate segments of every size class (registers <= 16, warp <= 32, warp with
    eight keys per lane <= 256, CTA <= 1024, CTA over shared / global memory above) and long seed chains with wide intervals;
    single-end and paired records against the oracle"""
    chroms = S.random_genome([700000, 500000], seed=321, repeat_fraction=0.7, repeat_copies=(40, 1500), repeat_len=(200, 700), repeat_div=(0.005, 0.06))
    S.write_fasta(tmp_path / "g.fa", chroms)
    subprocess.run([str(built["indexer"]), "g.fa"], cwd=tmp_path, check=True, stderr=subprocess.DEVNULL)
    g, st = S.concat_genome(chroms)
    m1, _ = S.simulate_fast(g, st, 6000, 150, 17, paired=False, indel_reads=0.2)
    a, b = S.simulate_fast(g, st, 2500, 120, 18)
    se = [bytes(r) for r in m1]
    mates = [x for pr in zip((bytes(r) for r in a), (revcomp(bytes(r)) for r in b)) for x in pr]
    ix = B.Index(tmp_path / "g.fa.index"); ox = OracleIndex(tmp_path / "g.fa.index")
    try:
        gres, gcand = ix.map_batch_se(se)
        ores, ocand = ox.map_se(se, cap=1 << 24)
        assert_same_records(gres, gcand, ores, ocand)
        n = gres["n_cand"][gres["state"] == B.VERIFY]
        assert (n > 16).any() and (n > 256).any(), "the data set no longer reaches the larger sort tiers"
        gres, gcand = ix.map_batch_pe(mates)
        ores, ocand = ox.map_pe(mates, cap=1 << 24)
        v = np.repeat(gres["state"] == B.VERIFY, gres["n_cand"])
        assert_same_records(gres, gcand, ores, ocand, compare_vote=False)
        assert np.array_equal(gcand["vote"][v], ocand["vote"][v])
    finally:
        ix.close()


def test_device_index_builder_writes_the_same_files(golden, built, tmp_path):
    """bmbs-index-gpu (suffix sort by library radix sorts + device BWT passes; data prep for the 3.1 Gbp bench genome) must
    write, byte for byte, the files of the CPU writer -- which are the reference's own (sha256 test in test_oracle_golden.py).
    Genomes: the golden one, and one of high-copy repeat families (groups of equal 32-symbol keys refined over many rounds)"""
    import filecmp, shutil
    gpu_tool = ROOT_DIR / "bitmapperbs_b200/_build/bmbs-index-gpu"
    if not gpu_tool.exists():
        pytest.skip("bmbs-index-gpu not built")
    chroms = S.random_genome([400000, 250000, 777], seed=4321, repeat_fraction=0.6, repeat_copies=(20, 800), repeat_len=(150, 3000), repeat_div=(0.0, 0.05))
    S.write_fasta(tmp_path / "rep.fa", chroms)
    shutil.copy(golden / "genome.fa", tmp_path / "gold.fa")
    for name in ("gold.fa", "rep.fa"):
        for tool, d in ((built["indexer"], "cpu"), (gpu_tool, "gpu")):
            (tmp_path / d).mkdir(exist_ok=True)
            shutil.copy(tmp_path / name, tmp_path / d / name)
            subprocess.run([str(tool), name], cwd=tmp_path / d, check=True, stderr=subprocess.DEVNULL)
        for ext in (".index", ".index.bs.pac", ".index.bs.index", ".index.bs.index.bwt", ".index.bs.index.sa", ".index.bs.index.occ"):
            assert filecmp.cmp(tmp_path / "cpu" / (name + ext), tmp_path / "gpu" / (name + ext), shallow=False), (name, ext)


def test_mixed_lengths_and_unequal_mates(golden, gidx, oidx):
    """reads of many lengths in one batch (ragged input); mates of different lengths in a pair"""
    rng = np.random.default_rng(11)
    se = []
    for r in read_fastq(golden / "se250.fq")[:400]:
        se.append(r[1][: int(rng.integers(18, 251))])
    se += [r[1][: int(rng.integers(30, 101))] for r in read_fastq(golden / "se100.fq")[:800]]
    gres, gcand = gidx.map_batch_se(se)
    ores, ocand = oidx.map_se(se)
    assert_same_records(gres, gcand, ores, ocand)
    m1 = read_fastq(golden / "pe150_1.fq")[:800]; m2 = read_fastq(golden / "pe150_2.fq")[:800]
    mates = []
    for a, b in zip(m1, m2):
        la, lb = int(rng.integers(40, 151)), int(rng.integers(40, 151))
        mates += [a[1][:la], revcomp(b[1][:lb])]
    for sens in (0, 1):
        gres, gcand = gidx.map_batch_pe(mates, params=capi.default_params(sensitive=sens))
        if sens:
            ores, ocand, _ = oidx.map_pe_sensitive(mates)
        else:
            ores, ocand = oidx.map_pe(mates)
        for f in ("state", "n_cand", "is_multiple_map"):
            assert np.array_equal(gres[f], ores[f]), (sens, f)
        gs, os_ = _slices(gres, gcand), _slices(ores, ocand)
        for f in ("site", "end_site", "err"):
            assert np.array_equal(gs[f], os_[f]), (sens, f)


def test_edge_case_reads(golden, gidx, oidx):
    genome = b"".join(l.strip() for l in open(golden / "genome.fa", "rb") if not l.startswith(b">"))
    N = len(genome)
    reads = [
        b"ACGT" * 4,                                  # 16 bp: never seeds (bwt.h:2089)
        b"A" * 9,                                     # L < 10: seed budget wraps to 25
        b"N" * 100,                                   # nothing but N
        genome[:100], genome[N - 100:],               # first / last bases of the concatenated genome
        revcomp(genome[:100]), revcomp(genome[N - 100:]),
        genome[119950:120050],                        # crosses the chr1 / chr2 boundary
        genome[5000:5100].replace(b"C", b"T"),        # fully converted
        genome[5000:5050] + b"N" + genome[5051:5100], # N in the middle
        genome[7000:7017] + b"R" + genome[7018:7100], # IUPAC base other than N
        b"ACGTTGCA" * 30,                             # junk, 240 bp
        genome[9000:9999],                            # 999 bp, k capped at 31
        genome[20000:20018],                          # 18 bp, shortest seedable read
        b"T" * 60, b"TG" * 40,                        # low complexity, no C
    ]
    gres, gcand = gidx.map_batch_se(reads)
    ores, ocand = oidx.map_se(reads)
    assert_same_records(gres, gcand, ores, ocand)
    # empty batch and the argument checks
    r0, c0 = gidx.map_batch_se([])
    assert len(r0) == 0 and len(c0) == 0
    with pytest.raises(B.BmbsError, match="1000"):
        gidx.map_batch_se([b"A" * 1001])


def _verify_cases(rng, oidx, n, L):
    N = oidx.N
    k = min(31, int(0.08 * L))
    reads, sites = [], []
    for _ in range(n):
        site = int(rng.integers(0, 2 * N))
        mode = rng.random()
        if mode < 0.02:
            edge = [N - L, N - 3, 2 * N - L - k, 2 * N - 2, 2 * N + 5, (1 << 64) - 7, 0, N]   # strand ends, wrapped coordinates
            site = edge[int(rng.integers(0, len(edge)))]
        win = oidx.window(site, L + 2 * k)
        base = np.frombuffer(win, dtype=np.uint8)[k:k + L].copy()
        if base[0] == 0 or mode < 0.05:
            base = ACGT[rng.integers(0, 4, size=L)]                  # decoy / out-of-genome window
        else:
            c = (base == ord("C")) & (rng.random(L) < 0.98); base[c] = ord("T")
            e = rng.choice([0, 0.01, 0.02, 0.04, 0.06, 0.08])
            for _e in range(rng.binomial(L, e)):
                p = int(rng.integers(0, len(base))); r = rng.random()
                if r < 2 / 3:
                    base[p] = rng.choice(np.frombuffer(b"ACGTN", dtype=np.uint8))
                elif r < 5 / 6 and len(base) > 20:
                    base = np.delete(base, p)
                else:
                    base = np.insert(base, p, ACGT[rng.integers(0, 4)])
            if len(base) < L:
                base = np.concatenate([base, ACGT[rng.integers(0, 4, size=L - len(base))]])
            base = base[:L]
        reads.append(base.tobytes()); sites.append(site)
    return reads, np.array(sites, dtype=np.uint64)


@pytest.mark.parametrize("L", [30, 100, 150, 200, 250, 640])
def test_verify_kernel_matches_oracle(gidx, oidx, L):
    rng = np.random.default_rng(1000 + L)
    reads, sites = _verify_cases(rng, oidx, 4000, L)
    idx = np.arange(len(reads), dtype=np.uint32)
    gend, gerr = gidx.verify(reads, idx, sites)
    oend, oerr = oidx.verify(reads, idx, sites)
    assert np.array_equal(gend, oend) and np.array_equal(gerr, oerr)
    assert (gend >= 0).sum() > 1500 and (gend < 0).sum() > 50


def test_verify_error_rate_other_than_default(gidx, oidx):
    rng = np.random.default_rng(77)
    reads, sites = _verify_cases(rng, oidx, 2000, 120)
    idx = np.arange(len(reads), dtype=np.uint32)
    for e in (0.0, 0.03, 0.2, 0.5):
        gend, gerr = gidx.verify(reads, idx, sites, e_rate=e)
        oend, oerr = oidx.verify(reads, idx, sites, e_rate=e)
        assert np.array_equal(gend, oend) and np.array_equal(gerr, oerr)


@pytest.mark.parametrize("name,args", [
    ("se100", ["--seq", "se100.fq"]),
    ("se250", ["--seq", "se250.fq"]),
    ("pe150", ["--seq1", "pe150_1.fq", "--seq2", "pe150_2.fq", "--pe"]),
    ("pe150s", ["--seq1", "pe150_1.fq", "--seq2", "pe150_2.fq", "--pe", "--sensitive"]),
    ("pe100h", ["--seq1", "pe100h_1.fq", "--seq2", "pe100h_2.fq", "--pe"]),
    ("pe100hs", ["--seq1", "pe100h_1.fq", "--seq2", "pe100h_2.fq", "--pe", "--sensitive"]),
])
@pytest.mark.parametrize("finish", ["device", "host", "device_warp_pairs", "device_small_grid"])
def test_mapper_sam_identical_to_reference_golden(golden, built, name, args, finish):
    """whole program: FASTQ -> GPU seed-and-verify through the C ABI -> finishing (device: reduction / pair pick, ungapped CIGAR,
    coordinates, banded DP per launch; host: the same from the window lists) -> MAPQ -> SAM, vs the reference's SAM"""
    import os
    # device_warp_pairs: every pair through the warp kernel of the pair finishing (staged lists, warp-parallel pair pick);
    # device_small_grid: every persistent and grid-stride launch sized for one SM, several batches in flight
    env = {**os.environ, **{"host": {"BMBS_HOST_FINISH": "1"}, "device_warp_pairs": {"BMBS_PE_FIN_SHORT": "0"},
                            "device_small_grid": {"BMBS_GRID_SMS": "1"}}.get(finish, {})}
    subprocess.run([str(built["bmbs"]), "--search", "genome.fa", *args, "-t", "4", "-o", "gpu.sam", "--mapstats", "gpu.stats", "--batch", "700"],
                   cwd=golden, check=True, stderr=subprocess.DEVNULL, env=env)
    assert sam_body(golden / "gpu.sam") == sam_body(golden / f"{name}.sam")
    assert (golden / "gpu.stats").read_text() == (golden / f"ref_{name}.stats").read_text()


def test_live_reference_binary_agrees_on_fresh_data(built, tmp_path):
    """fresh seeded data, larger than the golden set; compared with the reference's SAM and mapstats: their stored digests
    (tests/reference_sha256.py), and the reference itself where it is built"""
    chroms = S.random_genome([900000, 600000], seed=99, repeat_fraction=0.4, repeat_copies=(5, 60), repeat_len=(300, 4000))
    S.write_fasta(tmp_path / "g.fa", chroms)
    r, _ = S.simulate_reads(chroms, 12000, 125, seed=5, sub=0.025, indel=0.004, n_rate=0.002, random_qual=True, junk_fraction=0.03)
    S.write_fastq(tmp_path / "r.fq", r)
    a, b = S.simulate_reads(chroms, 6000, 100, seed=6, paired=True, sub=0.02, indel=0.003, random_qual=True, frag_range=(150, 420))
    S.write_fastq(tmp_path / "a.fq", a); S.write_fastq(tmp_path / "b.fq", b)
    c, d = S.simulate_reads(chroms, 8000, 120, seed=7, paired=True, sub=0.06, indel=0.008, n_rate=0.003, random_qual=True, frag_range=(150, 450), junk_fraction=0.03)
    S.write_fastq(tmp_path / "c.fq", c); S.write_fastq(tmp_path / "d.fq", d)
    # --pbat data: the reverse complements of directional reads (qualities reversed with them)
    comp = bytes.maketrans(b"ACGTacgt", b"TGCAtgca")
    with open(tmp_path / "r.fq", "rb") as f, open(tmp_path / "r_rc.fq", "wb") as o:
        ls = f.read().split(b"\n")
        for i in range(0, len(ls) - 1, 4):
            o.write(ls[i] + b"\n" + ls[i + 1].translate(comp)[::-1] + b"\n+\n" + ls[i + 3][::-1] + b"\n")
    subprocess.run([str(built["indexer"]), "g.fa"], cwd=tmp_path, check=True, stderr=subprocess.DEVNULL)
    for tag, args in (("se", ["--seq", "r.fq"]), ("pe", ["--seq1", "a.fq", "--seq2", "b.fq", "--pe"]),
                      ("pes", ["--seq1", "a.fq", "--seq2", "b.fq", "--pe", "--sensitive"]),
                      ("hard", ["--seq1", "c.fq", "--seq2", "d.fq", "--pe"]),
                      ("hards", ["--seq1", "c.fq", "--seq2", "d.fq", "--pe", "--sensitive"]),
                      ("se_e", ["--seq", "r.fq", "-e", "0.12", "--seed", "25"]),
                      ("hard_flags", ["--seq1", "c.fq", "--seq2", "d.fq", "--pe", "-e", "0.05", "--seed", "25", "--min", "50", "--max", "600"]),
                      ("hards_flags", ["--seq1", "c.fq", "--seq2", "d.fq", "--pe", "--sensitive", "-e", "0.1", "--min", "100", "--max", "450"]),
                      ("se_unmapped", ["--seq", "r.fq", "--unmapped_out"]),
                      ("hard_unmapped", ["--seq1", "c.fq", "--seq2", "d.fq", "--pe", "--unmapped_out"]),
                      ("hards_unmapped", ["--seq1", "c.fq", "--seq2", "d.fq", "--pe", "--sensitive", "--unmapped_out"]),
                      ("se_ambiguous", ["--seq", "r.fq", "--ambiguous_out"]),
                      ("se_both", ["--seq", "r.fq", "--ambiguous_out", "--unmapped_out"]),
                      ("hard_ambiguous", ["--seq1", "c.fq", "--seq2", "d.fq", "--pe", "--ambiguous_out", "--unmapped_out"]),
                      ("hards_ambiguous", ["--seq1", "c.fq", "--seq2", "d.fq", "--pe", "--sensitive", "--ambiguous_out"]),
                      ("se_pbat", ["--seq", "r_rc.fq", "--pbat", "--unmapped_out", "--ambiguous_out"]),
                      ("se_pbat_directional", ["--seq", "r.fq", "--pbat", "--unmapped_out"]),
                      ("pe_pbat", ["--seq1", "b.fq", "--seq2", "a.fq", "--pe", "--pbat"]),
                      ("hards_pbat", ["--seq1", "d.fq", "--seq2", "c.fq", "--pe", "--sensitive", "--pbat", "--unmapped_out"])):
        subprocess.run([str(built["bmbs"]), "--search", "g.fa", *args, "-t", "4", "-o", f"gpu_{tag}.sam", "--mapstats", f"gpu_{tag}.st"],
                       cwd=tmp_path, check=True, stderr=subprocess.DEVNULL)
        body, stats = sam_body(tmp_path / f"gpu_{tag}.sam"), (tmp_path / f"gpu_{tag}.st").read_text()
        reference_sha256.check(f"fresh_data:{tag}", b"".join(body) + stats.encode())
        if built["ref"].exists():
            subprocess.run([str(built["ref"]), "--search", "g.fa", *args, "-t", "1", "-o", f"cpu_{tag}.sam", "--mapstats", f"cpu_{tag}.st"],
                           cwd=tmp_path, check=True, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
            assert body == sam_body(tmp_path / f"cpu_{tag}.sam") and stats == (tmp_path / f"cpu_{tag}.st").read_text(), tag
        if "--pe" in args:      # the same pairs with every pair through the warp kernel of the pair finishing
            import os
            subprocess.run([str(built["bmbs"]), "--search", "g.fa", *args, "-t", "4", "-o", f"gpw_{tag}.sam", "--mapstats", f"gpw_{tag}.st"],
                           cwd=tmp_path, check=True, stderr=subprocess.DEVNULL, env={**os.environ, "BMBS_PE_FIN_SHORT": "0"})
            assert sam_body(tmp_path / f"gpw_{tag}.sam") == body, tag
            assert (tmp_path / f"gpw_{tag}.st").read_text() == stats, tag


def test_mapper_wide_suffix_array_gzip_input_and_two_gpus(golden, built, tmp_path):
    """whole program with (i) the > 2^32-row suffix-array layout forced on, (ii) gzip-compressed FASTQ input and (iii) the
    batches of one run spread over two GPUs (when the box has two): SAM and mapstats identical to the reference's golden files"""
    import gzip, os, shutil
    for f in ("se100.fq", "pe150_1.fq", "pe150_2.fq"):
        with open(golden / f, "rb") as i, gzip.open(golden / (f + ".gz"), "wb", compresslevel=1) as o:
            shutil.copyfileobj(i, o)
    import torch
    runs = [("wide", {"BMBS_FORCE_WIDE": "1", "BMBS_KMER": "20"}, []), ("gz", {}, [])]
    if torch.cuda.device_count() >= 2:
        runs.append(("gpus2", {}, ["--gpus", "2"]))
    for tag, env, extra in runs:
        gz = ".gz" if tag == "gz" else ""
        for name, args in (("se100", ["--seq", "se100.fq" + gz]), ("pe150s", ["--seq1", "pe150_1.fq" + gz, "--seq2", "pe150_2.fq" + gz, "--pe", "--sensitive"])):
            subprocess.run([str(built["bmbs"]), "--search", "genome.fa", *args, *extra, "-t", "4", "-o", f"{tag}.sam", "--mapstats", f"{tag}.stats", "--batch", "300"],
                           cwd=golden, check=True, stderr=subprocess.DEVNULL, env={**os.environ, **env})
            assert sam_body(golden / f"{tag}.sam") == sam_body(golden / f"{name}.sam"), (tag, name)
            assert (golden / f"{tag}.stats").read_text() == (golden / f"ref_{name}.stats").read_text(), (tag, name)


def test_one_call_cache_survives_index_reload(golden, oidx):
    """the one-call forms keep a batch context per (index, device); a new index that lands on a freed handle's address must
    not be served the old context (ADVICE r1): load / map / free / load / map, each result checked against the oracle"""
    reads = [r[1] for r in read_fastq(golden / "se100.fq")][:400]
    ores, ocand = oidx.map_se(reads)
    for _ in range(4):
        ix = B.Index(golden / "genome.fa.index")
        gres, gcand = ix.map_batch_se(reads)
        ix.close()
        assert_same_records(gres, gcand, ores, ocand)


def test_capacity_error_is_reported_with_needed_size(golden, gidx):
    reads = [r[1] for r in read_fastq(golden / "se100.fq")]
    flat, offs = capi.flatten(reads)
    import ctypes as C
    res = np.zeros(len(reads), dtype=capi.ReadResult); cand = np.zeros(4, dtype=capi.Cand); used = C.c_size_t(0)
    p = capi.default_params()
    L = capi.load_library()
    rc = L.bmbs_map_batch_se(gidx._h, 0, flat.ctypes.data, offs.ctypes.data, len(reads), C.byref(p), res.ctypes.data, cand.ctypes.data, 4, C.byref(used))
    assert rc == -4 and used.value > 4
    res2, cand2 = gidx.map_batch_se(reads)
    assert len(cand2) == used.value


def test_staged_batch_counters_and_idempotence(golden, gidx):
    reads = [r[1] for r in read_fastq(golden / "se100.fq")]
    flat, offs = capi.flatten(reads)
    b = B.Batch(gidx, 0, len(reads), len(flat) + 64, 1 << 18)
    p = capi.default_params()
    b.upload(flat, offs); b.run(p); r1, c1, u1 = b.download()
    c = b.counters(); t = b.timings()
    b.run(p); r2, c2, u2 = b.download()         # same inputs, same outputs
    assert u1 == u2 and np.array_equal(r1, r2) and np.array_equal(c1[:u1], c2[:u2])
    assert c["hash_queries"] >= len(reads) * 0.9 and c["occ_lookups"] > 0 and c["verified"] == (r1["n_cand"][r1["state"] == B.VERIFY]).sum()
    assert c["cells"] == sum(int(n) * len(rd) * (2 * min(31, int(0.08 * len(rd))) + 1) for n, rd, s in zip(r1["n_cand"], reads, r1["state"]) if s == B.VERIFY)
    assert t["total"] > 0 and b.launches() >= 12


@pytest.mark.parametrize("name,args", [("se100", ["--seq", "se100.fq"]), ("pe100hs", ["--seq1", "pe100h_1.fq", "--seq2", "pe100h_2.fq", "--pe", "--sensitive"])])
def test_mapper_bam_output_holds_the_same_records(golden, built, name, args):
    """--bam: the BGZF/BAM container written by the mapper decodes (gzip + struct only) to the records of the reference's SAM"""
    from test_host_bam import decode_bam
    subprocess.run([str(built["bmbs"]), "--search", "genome.fa", *args, "-t", "4", "--bam", "-o", "gpu.bam", "--batch", "700"],
                   cwd=golden, check=True, stderr=subprocess.DEVNULL)
    text, refs, recs, n_members = decode_bam(golden / "gpu.bam")
    assert text.startswith("@HD") and [r[0] for r in refs] == [l.split("\t")[1][3:] for l in text.splitlines() if l.startswith("@SQ")]
    lines = [l.decode().rstrip("\n").split("\t") for l in sam_body(golden / f"{name}.sam")]
    assert len(recs) == len(lines) and n_members > 3
    rid = {n: i for i, (n, _) in enumerate(refs)}
    for f, r in zip(lines, recs):
        assert (r["name"], r["flag"], r["rid"], r["pos"], r["mapq"], r["cigar"], r["seq"], r["qual"], r["tags"]) == \
               (f[0], int(f[1]), rid[f[2]], int(f[3]) - 1, int(f[4]), f[5], f[9], f[10], f[11:])
        assert r["npos"] == int(f[7]) - 1 and r["tlen"] == int(f[8])
    # and byte for byte what the reference's own writer (the stock reference linked with its vendored, patched htslib) puts out:
    # its stored digest, and the reference itself where it is built
    from test_host_bam import bam_payload
    gt, gd, gr = bam_payload(golden / "gpu.bam")
    reference_sha256.check(f"bmbs_bam:{name}", gd + gr)
    ref = ROOT_DIR / "oracle/_ref/bitmapperBS_bam"
    if ref.exists():
        subprocess.run([str(ref), "--search", "genome.fa", *args, "-t", "1", "--bam", "-o", "ref.bam"], cwd=golden, check=True, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
        rt, rd, rr = bam_payload(golden / "ref.bam")
        assert gd == rd and gr == rr
