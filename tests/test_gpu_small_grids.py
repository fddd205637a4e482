"""GPU (-m gpu): the persistent and grid-stride kernels beyond their first work item.  Their grids are sized for the device
(seed_reads: up to 148 x blocks-per-SM blocks of 128 lanes), so in a batch of a few thousand reads each lane, warp or block
takes one item and exits.  BMBS_GRID_SMS=n (read at index load) sizes every such launch for n SMs, BMBS_SEED_BLOCKS=1 leaves
one seed_reads block per SM: a lane then seeds many reads in turn -- the REFILL reset of its per-read state, the restaging of
its chunks, lanes of one warp in different reads' phases -- and every verify_windows thread, finishing warp and re-seeding
warp takes many items.  Against the oracle, bit-exactly, and against the same batches at other grid sizes."""
import subprocess

import numpy as np
import pytest

import bitmapperbs_b200 as B
from bitmapperbs_b200 import capi, simulate as S
from conftest import read_fastq, revcomp
from oracle_binding import OracleIndex
from test_gpu_finish import assert_same_final, assert_same_pairs, device_finish, device_finish_pe
from test_gpu_parity import _slices, _verify_cases, assert_same_records

pytestmark = pytest.mark.gpu
SEED_BLOCK = 128                                   # lanes of a seed_reads block
SMALL = {"BMBS_GRID_SMS": "1", "BMBS_SEED_BLOCKS": "1"}
GRID_KEYS = ("BMBS_GRID_SMS", "BMBS_SEED_BLOCKS")


def set_grid(m, env):
    """BMBS_GRID_SMS is read when an index loads, BMBS_SEED_BLOCKS when a batch first sizes its seed_reads grid: both stay set
    for the whole test"""
    for k in GRID_KEYS:
        m.delenv(k, raising=False)
    for k, v in env.items():
        m.setenv(k, v)


@pytest.fixture(scope="module")
def oidx(golden):
    return OracleIndex(golden / "genome.fa.index")


@pytest.fixture
def small_ix(golden, monkeypatch):
    set_grid(monkeypatch, SMALL)
    ix = B.Index(golden / "genome.fa.index")
    yield ix
    ix.close()


def golden_se(golden):
    return [r[1] for r in read_fastq(golden / "se100.fq")] + [r[1] for r in read_fastq(golden / "se250.fq")]


def pairs_of(golden, name, n=None):
    m1 = read_fastq(golden / f"{name}_1.fq")[:n]; m2 = read_fastq(golden / f"{name}_2.fq")[:n]
    return [x for a, b in zip(m1, m2) for x in (a[1], revcomp(b[1]))]


def run_staged(b, reads, params, pe=False):
    flat, offs = capi.flatten(reads)
    b.upload(flat, offs, pe=pe); b.run(params)
    res, cand, used = b.download()
    return res.copy(), cand[:used].copy()


def check_pe(gres, gcand, ores, ocand):
    v = np.repeat(gres["state"] == B.VERIFY, gres["n_cand"])
    assert_same_records(gres, gcand, ores, ocand, compare_vote=False)
    assert np.array_equal(gcand["vote"][v], ocand["vote"][v])


def check_pe_sensitive(gres, gcand, ores, ocand):
    for f in ("state", "n_cand", "is_multiple_map"):
        assert np.array_equal(gres[f], ores[f]), f
    m = np.isin(gres["state"], [B.EXACT_UNIQUE, B.ONE_MISMATCH])
    assert np.array_equal(gres["site"][m], ores["site"][m])
    gs, os_ = _slices(gres, gcand), _slices(ores, ocand)
    for f in ("site", "end_site", "err"):
        assert np.array_equal(gs[f], os_[f]), f


def test_small_grid_gives_each_lane_many_reads(golden, oidx, monkeypatch):
    """the hook does what the other tests rely on: at BMBS_GRID_SMS=1 / BMBS_SEED_BLOCKS=1 one seed_reads block of 128 lanes
    seeds the golden single-end set (about 28 reads a lane) and each verify_windows thread verifies several windows, with
    records identical to the oracle's; unset, the grids are sized for the device's SMs"""
    import torch
    reads = golden_se(golden)
    flat, offs = capi.flatten(reads)
    set_grid(monkeypatch, {})
    ix = B.Index(golden / "genome.fa.index")
    try:
        b = B.Batch(ix, 0, len(reads), len(flat) + 64, 1 << 18)
        run_staged(b, reads, capi.default_params())
        g = b.grid()
        b.close()
    finally:
        ix.close()
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    assert g[0] == sms and g[1] == (len(reads) + SEED_BLOCK - 1) // SEED_BLOCK and g[2] % sms == 0, g      # 29 blocks < one per SM
    set_grid(monkeypatch, SMALL)
    ix = B.Index(golden / "genome.fa.index")
    try:
        b = B.Batch(ix, 0, len(reads), len(flat) + 64, 1 << 18)
        gres, gcand = run_staged(b, reads, capi.default_params())
        g, c = b.grid(), b.counters()
        b.close()
    finally:
        ix.close()
    ores, ocand = oidx.map_se(reads)
    assert_same_records(gres, gcand, ores, ocand)
    print(f"small grid: grid() = {g}, {len(reads) / (SEED_BLOCK * g[1]):.1f} reads per seed_reads lane, "
          f"{c['verified']} windows = {c['verified'] / (g[2] * g[3]):.1f} per verify_windows thread")
    assert g[0] == 1 and g[1] == 1, g
    assert len(reads) >= 8 * SEED_BLOCK * g[1], g
    assert c["verified"] >= 2 * g[2] * g[3], (g, c)


# ---- lanes that switch between short and long reads: the 12-chunk staging cap of ReadPlanes (ns = L/32 + 2 capped at 12,
# reads of 352 bases and more read the rest from global memory) and the read-length limit, in both directions on one lane
LONG = [319, 320, 351, 352, 353, 383, 384, 416, 640, 1000]
LONG_MATES = [L for L in LONG if L <= 640]


def _genome(golden):
    return b"".join(l.strip() for l in open(golden / "genome.fa", "rb") if not l.startswith(b">"))


def _mutate(rng, s):
    """bisulfite conversion (C -> T at 98%), then substitutions, length-preserving indels and sometimes one N"""
    s = np.frombuffer(s, dtype=np.uint8).copy()
    L = len(s)
    c = (s == ord("C")) & (rng.random(L) < 0.98); s[c] = ord("T")
    for _ in range(rng.binomial(L, rng.choice([0.0, 0.005, 0.015, 0.03]))):
        s[int(rng.integers(0, L))] = ord(rng.choice(list("ACGT")))
    for _ in range(int(rng.integers(0, 3))):
        p = int(rng.integers(1, L - 1))
        if rng.random() < 0.5:
            s = np.concatenate([np.delete(s, p), np.frombuffer(bytes([rng.choice(list(b"ACGT"))]), dtype=np.uint8)])
        else:
            s = np.insert(s, p, ord(rng.choice(list("ACGT"))))[:L]
    if rng.random() < 0.2:
        s[int(rng.integers(0, L))] = ord("N")
    return s.tobytes()


def _slice(rng, genome, n):
    p = int(rng.integers(0, len(genome) - n))
    s = genome[p:p + n]
    return revcomp(s) if rng.random() < 0.5 else s


def mixed_se(golden, n=1200, seed=31):
    rng = np.random.default_rng(seed)
    genome = _genome(golden)
    out = []
    for i in range(n):
        L = int(rng.integers(18, 101)) if i % 2 == 0 else LONG[(i // 2) % len(LONG)]
        out.append(_mutate(rng, _slice(rng, genome, L)))
    return out


def mixed_pairs(golden, n=600, seed=32):
    """mates as stored (mate 2 already reverse-complemented): the two ends of one converted fragment of up to 1400 bases, in
    every fourth pair one mate with 10% more substitutions (no hit of its own: the --sensitive re-seeding round takes it);
    after each such pair two of the golden pe100h set, whose mates the re-seeding round does find hits for"""
    rng = np.random.default_rng(seed)
    genome = _genome(golden)
    hard = pairs_of(golden, "pe100h", 2 * n)
    out = []
    for i in range(n):
        if i % 2 == 0:
            l1, l2 = int(rng.integers(150, 201)), int(rng.integers(150, 201))
        else:
            l1, l2 = LONG_MATES[(i // 2) % len(LONG_MATES)], LONG_MATES[(i // 2 + 3) % len(LONG_MATES)]
        frag = _slice(rng, genome, int(rng.integers(max(l1, l2), 1401)))
        m1, m2 = _mutate(rng, frag[:l1]), _mutate(rng, frag[len(frag) - l2:])
        if i % 4 == 3:
            m2 = np.frombuffer(m2, dtype=np.uint8).copy()
            m2[rng.integers(0, l2, size=l2 // 10)] = np.frombuffer(b"ACGT", dtype=np.uint8)[rng.integers(0, 4, size=l2 // 10)]
            m2 = m2.tobytes()
        out += [m1, m2] + hard[4 * i:4 * i + 4]
    return out


def test_lanes_switch_between_short_and_long_reads(golden, oidx, small_ix):
    reads = mixed_se(golden)
    res, cand, fin, mism, fb, c = device_finish(small_ix, reads)
    ores, ocand = oidx.map_se(reads)
    assert_same_records(res, cand, ores, ocand)
    assert (res["state"] == B.VERIFY).sum() > 200 and (res["state"] == B.EXACT_UNIQUE).sum() > 50
    L = np.diff(capi.flatten(reads)[1]).astype(np.int64)
    assert ((L >= 352) & (res["n_cand"] > 0)).sum() > 100          # long reads found their windows, past the staging cap
    ofin, omism = oidx.finish_se(reads, res, cand)
    assert_same_final(fin, mism, ofin, omism, res, cand)
    assert (fin["status"] == capi.FIN_UNIQUE).sum() > 200 and (fin["status"] == capi.FIN_DP).sum() > 20


@pytest.mark.parametrize("sensitive", [0, 1])
def test_lanes_switch_between_short_and_long_mates(golden, oidx, small_ix, sensitive):
    mates = mixed_pairs(golden)
    p = capi.default_params(max_ins=1500, sensitive=sensitive)
    res, cand, fin, mism, c = device_finish_pe(small_ix, mates, p)
    if sensitive:
        ores, ocand, reseeded = oidx.map_pe_sensitive(mates, max_ins=1500)
        check_pe_sensitive(res, cand, ores, ocand)
        L = np.diff(capi.flatten(mates)[1]).astype(np.int64)
        assert (reseeded & (L >= 352)).sum() > 10 and (ores["n_cand"][reseeded == 1] > 0).sum() > 0   # long mates re-seeded; hits found
    else:
        ores, ocand = oidx.map_pe(mates, max_ins=1500)
        check_pe(res, cand, ores, ocand)
    ofin, omism = oidx.finish_pe(mates, res, cand, max_ins=1500, sensitive=bool(sensitive))
    assert_same_pairs(fin, mism, ofin, omism)
    st = fin["status"][0::2]
    assert (st == capi.FIN_UNIQUE).sum() + (st == capi.FIN_DP).sum() > len(st) // 3


# ---- results do not depend on the grid: the high-copy repeat genome (window lists of every size class, long seed chains)
@pytest.fixture(scope="module")
def repeat_genome(built, tmp_path_factory):
    d = tmp_path_factory.mktemp("repeats")
    chroms = S.random_genome([700000, 500000], seed=321, repeat_fraction=0.7, repeat_copies=(40, 1500), repeat_len=(200, 700), repeat_div=(0.005, 0.06))
    S.write_fasta(d / "g.fa", chroms)
    subprocess.run([str(built["indexer"]), "g.fa"], cwd=d, check=True, stderr=subprocess.DEVNULL)
    g, st = S.concat_genome(chroms)
    m1, _ = S.simulate_fast(g, st, 6000, 150, 17, paired=False, indel_reads=0.2)
    a, b = S.simulate_fast(g, st, 2500, 120, 18)
    se = [bytes(r) for r in m1]
    mates = [x for pr in zip((bytes(r) for r in a), (revcomp(bytes(r)) for r in b)) for x in pr]
    return d / "g.fa.index", se, mates


def _per_read(fin, aux, mism_or_cand):
    """each read's slice of the mismatch positions / handed-back windows (offsets follow completion order)"""
    return [mism_or_cand[int(a):int(a) + int(n)] for a, n in zip(fin["aux_first"], aux)]


def test_results_do_not_depend_on_the_grid(repeat_genome, monkeypatch):
    prefix, se, mates = repeat_genome
    grids = {"default": {}, "one_sm_one_seed_block": SMALL, "seven_sms": {"BMBS_GRID_SMS": "7"}}
    out = {}
    for name, env in grids.items():
        with monkeypatch.context() as m:
            set_grid(m, env)
            ix = B.Index(prefix)
            try:
                out[name] = (device_finish(ix, se, capi.default_params()),
                             device_finish_pe(ix, mates, capi.default_params(sensitive=1)))
            finally:
                ix.close()
    (res0, cand0, fin0, mism0, fb0, _), (pres0, pcand0, pfin0, pmism0, _) = out["default"]
    n = res0["n_cand"][res0["state"] == B.VERIFY]
    assert (n > 256).any() and (fin0["status"] == capi.FIN_DP).sum() > 20
    fields = [f for f in capi.Final.names if f != "aux_first"]
    for name in grids:
        if name == "default":
            continue
        (res, cand, fin, mism, fb, _), (pres, pcand, pfin, pmism, _) = out[name]
        for r0, c0, r1, c1 in ((res0, cand0, res, cand), (pres0, pcand0, pres, pcand)):
            assert np.array_equal(r0, r1), name
            assert np.array_equal(_slices(r0, c0), _slices(r1, c1)), name
        for f0, f1 in ((fin0, fin), (pfin0, pfin)):
            for f in fields:
                assert np.array_equal(f0[f], f1[f]), (name, f)
        uq = fin0["status"] == capi.FIN_UNIQUE
        for a, b in zip(_per_read(fin0[uq], fin0["n_aux"][uq], mism0), _per_read(fin[uq], fin["n_aux"][uq], mism)):
            assert np.array_equal(a, b), name
        host = fin0["status"] == capi.FIN_HOST
        for a, b in zip(_per_read(fin0[host], fin0["n_aux"][host], fb0), _per_read(fin[host], fin["n_aux"][host], fb)):
            assert np.array_equal(a, b), name
        pu = pfin0["n_aux"] > 0
        for a, b in zip(_per_read(pfin0[pu], pfin0["n_aux"][pu], pmism0), _per_read(pfin[pu], pfin["n_aux"][pu], pmism)):
            assert np.array_equal(a, b), name


def test_one_batch_context_runs_many_different_batches(golden, oidx, small_ix):
    """one staged context, batches of other sizes, modes and read lengths in turn, each against the oracle: counters, lists,
    cursors and the cached seed_reads sizing of an earlier batch must not leak into a later one"""
    se = golden_se(golden)
    short = [r[: 18 + i % 43] for i, r in enumerate(se[:40])]
    pe150 = pairs_of(golden, "pe150")
    pe100h = pairs_of(golden, "pe100h")
    genome = _genome(golden)
    amb = se[:1500] + [genome[9000:10000]] + se[1500:2000]
    rng = np.random.default_rng(640)
    vreads, vsites = _verify_cases(rng, oidx, 4000, 250)
    batches = [se, short, pe150, pe100h, amb, vreads]
    max_reads = max(len(x) for x in batches)
    max_bases = max(len(capi.flatten(x)[0]) for x in batches)
    b = B.Batch(small_ix, 0, max_reads + 2, max_bases + 64, 1 << 20)
    try:
        # 1. the golden single-end set, longest read 250
        g1, c1 = run_staged(b, se, capi.default_params())
        ores, ocand = oidx.map_se(se)
        assert_same_records(g1, c1, ores, ocand)
        # 2. 40 short reads: fewer staged chunks, a grid of one block
        gres, gcand = run_staged(b, short, capi.default_params())
        assert_same_records(gres, gcand, *oidx.map_se(short))
        # 3. pe150 --sensitive (re-seeding round)
        gres, gcand = run_staged(b, pe150, capi.default_params(sensitive=1), pe=True)
        check_pe_sensitive(gres, gcand, *oidx.map_pe_sensitive(pe150)[:2])
        # 4. pe100h fast, other -e / --min / --max
        p = capi.default_params(e_rate=0.05, min_ins=100, max_ins=350)
        gres, gcand = run_staged(b, pe100h, p, pe=True)
        check_pe(gres, gcand, *oidx.map_pe(pe100h, e_rate=0.05, min_ins=100, max_ins=350))
        # 5. single end with --ambiguous_out and one 1000-base read, finished on the device
        p = capi.default_params(ambiguous_out=1)
        res, cand = run_staged(b, amb, p)
        b.finish()
        fin, mism, fb = b.download_final()
        ofin, omism = oidx.finish_se(amb, res, cand, ambiguous_out=True)
        assert_same_final(fin, mism, ofin, omism, res, cand)
        # 6. verification alone over 4,000 windows
        flat, offs = capi.flatten(vreads)
        b.upload(flat, offs)
        idx = np.arange(len(vreads), dtype=np.uint32)
        b.verify(idx, vsites)
        gend, gerr = b.download_verify()
        oend, oerr = oidx.verify(vreads, idx, vsites)
        assert np.array_equal(gend, oend) and np.array_equal(gerr, oerr)
        # 7. the golden single-end set again
        g7, c7 = run_staged(b, se, capi.default_params())
        assert np.array_equal(g7, g1) and np.array_equal(c7, c1)
        assert b.grid()[:2] == [1, 1]
    finally:
        b.close()
