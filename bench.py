#!/usr/bin/env python3
"""bench.py -- throughput of the seed-and-verify hot path on B200, next to the reference CPU mapper.

Default workload = BASELINE.json configs[2] (SURVEY.md §8d cfg 3, the one the metric is quoted on): human-like synthetic genome
(24 chromosomes, half of it repeat families of 1-10 kbp elements copied 10-10^4 times at 1-15 % divergence, seed 1003),
150 bp single-end directional bisulfite reads (98 % C->T, 1 % substitutions, 14 % of the reads with one indel, seed 2003 +
rank), default -e 0.08.  `--scale` is the fraction of the 3.087 Gbp genome that is built (stated in config.workload); the
index is built once per box under --cache.  `--workload cfg2` (100 Mbp uniform, --pe) and `cfg4` (cfg3's genome, --pe
--sensitive) are kept for profiling.  A "step" is one pass of the whole device pipeline (pack -> seed -> locate -> votes ->
[pair filter] -> verify [-> sensitive pairing]) over one batch of `--reads` reads per GPU.

  value         reads/s, inputs already resident in HBM, CUDA-event time on the library's stream
  e2e           the same through the C ABI with pinned HOST buffers: H2D of the reads and D2H of the per-read records and
                verified candidate lists inside the timed region (what the host mapper calls per batch)
  roofline      dominant kernel group of the step against the measured HBM peak (MEASURED_PEAKS.json), algorithmic bytes in
                SURVEY.md §8d's units (10 B per table query, 40 B per occ lookup) and in this layout's own (8 B / 32 B)
  roofline_int  verify_windows against the measured integer-ALU peak: GCUPS and 14 word-ops per column per band word
  whole_program FASTQ -> SAM through the command line (bitmapperbs_b200/_build/bmbs) next to the reference's own `Total:`
                timers on the same file: the like-for-like number for the reference arm, whose timer covers its whole mapping
  cfg4          secondary: BASELINE.json configs[3] (the same genome, 150 bp pairs, --pe --sensitive) on the resident index,
                device reads/s and end to end through the C ABI, max over ranks like the headline (--no-cfg4 to skip)
  cpu_baseline  the REAL reference (oracle/_ref/bitmapperBS, compiled from /root/reference) with -t <host cores> on a
                bounded sample of the same reads, its own mapping timer (Bitmapper_main.cpp:262)

`--steps` timed steps are run in each timed loop (device-resident, end to end, cfg4).  `--dump-outputs DIR` writes what the
end-to-end loop's last step returned to the caller (see dump_outputs); the inputs are seeded, so two builds can be compared.
`--impl reference` times only that CPU run.  Multi-GPU (torchrun, one rank per GPU): read batches are sharded, the index is
replicated, no collective on the data path; per-GPU work is fixed ("weak").
"""
from __future__ import annotations

import argparse
import json
import os
import re
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

READ_LEN = 150
HUMAN_MBP = [250, 243, 198, 190, 181, 171, 159, 145, 138, 134, 135, 133, 114, 107, 102, 90, 83, 80, 59, 64, 47, 51, 156, 57]
REPEATS = dict(repeat_fraction=0.5, repeat_len=(1000, 10000), repeat_copies=(10, 10000), repeat_div=(0.01, 0.15))
DEFAULT_SCALE = {"cfg3": 1.0, "cfg4": 1.0, "cfg2": 1.0}     # BMBS_BENCH_SCALE=0.1 for quick runs


def log(*a):
    print(*a, file=sys.stderr, flush=True)


# ------------------------------------------------------------------------------------------------ workloads
class Workload:
    """what is mapped: genome recipe, read recipe, mapper flags"""

    def __init__(self, name: str, scale: float):
        self.name, self.scale = name, scale
        if name == "cfg2":
            self.chroms = [int(c * scale) for c in (40_000_000, 30_000_000, 20_000_000, 10_000_000)]
            self.genome_seed, self.repeat, self.dir = 1002, {}, f"cfg2_s1002_x{scale:g}"
            self.pe, self.sensitive, self.read_seed = True, False, 2002
        elif name in ("cfg3", "cfg4"):
            self.chroms = [int(x * 1_000_000 * scale) for x in HUMAN_MBP]
            self.genome_seed, self.repeat, self.dir = 1003, REPEATS, f"cfg3_s1003_x{scale:g}"
            self.pe, self.sensitive, self.read_seed = name == "cfg4", name == "cfg4", 2003 if name == "cfg3" else 2004
        else:
            raise SystemExit(f"unknown workload {name}")
        self.mbp = sum(self.chroms) / 1e6

    def describe(self, units: int) -> str:
        if self.name == "cfg2":
            return (f"cfg2: synthetic {self.mbp:g} Mbp genome (4 chr, uniform, seed 1002), {units} x 2 x {READ_LEN} bp paired-end directional "
                    f"bisulfite reads per GPU per step, --pe fast mode")
        g = (f"synthetic {self.mbp / 1000:.3f} Gbp genome = {self.scale:g} x BASELINE's 3.087 Gbp (24 chr, 50 % repeat families of 1-10 kbp "
             f"elements x 10-10^4 copies at 1-15 % divergence, seed 1003)")
        if self.name == "cfg3":
            return f"cfg3: {g}, {units} x {READ_LEN} bp single-end directional bisulfite reads per GPU per step (1 % substitutions, 14 % of reads with one indel), -e 0.08"
        return f"cfg4: {g}, {units} x 2 x {READ_LEN} bp paired-end reads per GPU per step, --pe --sensitive"

    def simulate(self, genome, starts, units, seed):
        """-> (mate1 [n, L], mate2 [n, L] in FASTQ orientation or None)"""
        from bitmapperbs_b200 import simulate as S
        if self.pe:
            return S.simulate_fast(genome, starts, units, READ_LEN, seed)
        return S.simulate_fast(genome, starts, units, READ_LEN, seed, paired=False, indel_reads=0.14 if self.name == "cfg3" else 0.0)

    def cli_flags(self):
        return (["--pe"] if self.pe else []) + (["--sensitive"] if self.sensitive else [])


def build_index(fa: Path):
    """index files next to `fa`: the device builder when this box has a GPU and the tool is built, else the CPU writer (data prep)"""
    from bitmapperbs_b200 import build as B
    idx, _ = B.build_tools()
    gpu_tool = ROOT / "bitmapperbs_b200/_build/bmbs-index-gpu"
    if gpu_tool.exists() and os.environ.get("BMBS_INDEXER", "gpu") != "cpu":
        r = subprocess.run([str(gpu_tool), str(fa)], stdout=subprocess.DEVNULL, stderr=subprocess.PIPE, text=True)
        if r.returncode == 0:
            return "gpu"
        log(f"[bench] device index builder failed ({r.stderr.strip()[-300:]}); using the CPU writer")
    subprocess.run([str(idx), str(fa)], check=True, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
    return "cpu"


def ensure_dataset(cache: Path, wl, build: bool = True):
    """genome + index under `cache`; built once per box (rank 0), reused by every later run.
    (tools/ call this as ensure_dataset(cache, scale, build) for the cfg2 genome.)"""
    if not isinstance(wl, Workload):
        wl = Workload("cfg2", float(wl))
    from bitmapperbs_b200 import simulate as S
    d = cache / wl.dir
    done = d / ".done"
    if build and not done.exists():
        d.mkdir(parents=True, exist_ok=True)
        t = time.time()
        chroms = S.random_genome(wl.chroms, seed=wl.genome_seed, **wl.repeat)
        S.write_fasta(d / "g.fa", chroms)
        g, st = S.concat_genome(chroms)
        np.save(d / "genome.npy", g); np.save(d / "starts.npy", st)
        del chroms, g
        t1 = time.time()
        how = build_index(d / "g.fa")
        done.write_text(how)
        log(f"[bench] genome written in {t1 - t:.1f}s, index built ({how}) in {time.time() - t1:.1f}s at {d}")
    while not done.exists():
        time.sleep(0.5)
    return d


def make_reads(d: Path, wl: Workload, units: int, seed: int):
    f = d / f"reads_{wl.name}_n{units}_s{seed}.npz"
    if f.exists():
        z = np.load(f)
        return z["m1"], (z["m2"] if "m2" in z.files else None)
    g = np.load(d / "genome.npy", mmap_mode="r"); st = np.load(d / "starts.npy")
    m1, m2 = wl.simulate(g, st, units, seed)
    tmp = d / f".tmp_{os.getpid()}_{seed}.npz"
    if m2 is None:
        np.savez(tmp, m1=m1)
    else:
        np.savez(tmp, m1=m1, m2=m2)
    os.replace(tmp, f)
    return m1, m2


def write_fastq_files(d: Path, wl: Workload, m1, m2, n: int, tag: str):
    from bitmapperbs_b200 import simulate as S
    n = min(n, len(m1))
    if wl.pe:
        fa, fb = d / f"{tag}_{wl.name}_{n}_1.fq", d / f"{tag}_{wl.name}_{n}_2.fq"
        if not fa.exists() or not fb.exists():
            S.write_fastq_matrix(fa, m1[:n], "/1"); S.write_fastq_matrix(fb, m2[:n], "/2")
        return n, ["--seq1", fa.name, "--seq2", fb.name]
    f = d / f"{tag}_{wl.name}_{n}.fq"
    if not f.exists():
        S.write_fastq_matrix(f, m1[:n], "")
    return n, ["--seq", f.name]


# ------------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    """SM clock and throttle reasons every 5 ms from a thread (NVML); `nvidia-smi -lms` as the fallback."""
    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu):
        self.rows = []; self.p = None; self.gpu = gpu; self.run = False; self.max_mhz = None; self.src = None

    def start(self):
        try:
            import pynvml as N
            N.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            idx = int(vis.split(",")[self.gpu]) if vis and all(x.strip().isdigit() for x in vis.split(",")) else self.gpu
            h = N.nvmlDeviceGetHandleByIndex(idx)
            self.max_mhz = float(N.nvmlDeviceGetMaxClockInfo(h, N.NVML_CLOCK_SM))
            reasons_fn = getattr(N, "nvmlDeviceGetCurrentClocksEventReasons", None) or N.nvmlDeviceGetCurrentClocksThrottleReasons
            bits = {"hw_slowdown": 0x8, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20, "sw_power_cap": 0x4}
            N.nvmlDeviceGetClockInfo(h, N.NVML_CLOCK_SM); reasons_fn(h)
            self.run = True; self.src = "nvml"

            def loop():
                while self.run:
                    try:
                        mhz = float(N.nvmlDeviceGetClockInfo(h, N.NVML_CLOCK_SM)); r = int(reasons_fn(h))
                        self.rows.append((time.time(), mhz, [k for k, b in bits.items() if r & b]))
                    except Exception:
                        pass
                    time.sleep(0.005)
            threading.Thread(target=loop, daemon=True).start()
            return
        except Exception:
            self.run = False
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "50"],
                                      stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.src = "nvidia-smi"
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.p = None

    def _read(self):
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.p.stdout:
            f = [x.strip() for x in line.split(",")]
            try:
                self.max_mhz = max(self.max_mhz or 0.0, float(f[1]))
                self.rows.append((time.time(), float(f[0]), [n for n, v in zip(names, f[2:6]) if v.lower().startswith("active")]))
            except Exception:
                continue

    def stop(self, t0=0.0, t1=1e30):
        """samples taken inside [t0, t1] (the timed region); if the region was shorter than a few sampling periods,
        every sample since start() -- the sampler is started before the warm-up, so those are under load too"""
        self.run = False
        if self.p:
            self.p.terminate()
        inside = [r for r in self.rows if t0 <= r[0] <= t1]
        rows = inside if len(inside) >= 3 else self.rows
        sm = [r[1] for r in rows]; reasons = sorted({x for r in rows for x in r[2]})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": self.max_mhz, "reasons": reasons, "samples": len(sm), "source": self.src,
                "window": "timed region" if len(inside) >= 3 else "warm-up + timed region"}


def bind_to_gpu_node(dev: int):
    """run on the cores of the NUMA node the GPU hangs off (page-locked buffers are then allocated there: the copies of an
    8-GPU run stay off the inter-socket link); returns the node or None when the box has one node / hides the topology"""
    try:
        import pynvml as N
        N.nvmlInit()
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        idx = int(vis.split(",")[dev]) if vis and all(x.strip().isdigit() for x in vis.split(",")) else dev
        bus = N.nvmlDeviceGetPciInfo(N.nvmlDeviceGetHandleByIndex(idx)).busId
        bus = (bus.decode() if isinstance(bus, bytes) else bus).lower()
        if len(bus.split(":")[0]) == 8:
            bus = bus[4:]
        node = int(Path(f"/sys/bus/pci/devices/{bus}/numa_node").read_text())
        if node < 0:
            return None
        cpus = set()
        for part in Path(f"/sys/devices/system/node/node{node}/cpulist").read_text().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            return node
    except Exception:
        pass
    return None


# ------------------------------------------------------------------------------------------------ command-line runs
def run_cli(exe: Path, d: Path, wl: Workload, seq_args, threads: int, out: str, extra=()):
    """`exe --search g.fa <reads> -t threads -o out`; returns (load_s, map_s, wall_s) from the program's own `Total:` line"""
    t = time.time()
    r = subprocess.run([str(exe), "--search", "g.fa", *seq_args, *wl.cli_flags(), "-t", str(threads), "-o", out, *extra],
                       cwd=d, stdout=subprocess.DEVNULL, stderr=subprocess.PIPE, text=True)
    wall = time.time() - t
    m = re.search(r"Total:\s+([0-9.]+)\s+([0-9.]+)", r.stderr)
    if r.returncode != 0 or not m:
        log(f"[bench] {exe.name} failed: {r.stderr[-500:]}")
        return None
    return float(m.group(1)), float(m.group(2)), wall

DUMP_BYTES = 64 << 20


def dump_outputs(out: Path, records, fields, lists):
    """--dump-outputs: the per-read records of the last timed step and the per-read lists they point into, as float64 .npy
    files (records: `<field>.npy`; lists: `<list>.npy` or `<list>_<field>.npy`, each read's entries in read order).  Offsets
    into the lists are left out: the device hands them out in completion order.  When everything would exceed DUMP_BYTES,
    a seeded sample of the reads (the same for the same outputs) is written; `read_index.npy` names the reads written.
    A list with no entries among the reads written (e.g. no read handed back to the host) writes no file.
    lists: name -> (array, first entry per read, entries per read, mask of the reads whose entries are in this array)"""
    n = len(records)
    m = n
    while True:
        idx = np.sort(np.random.default_rng(0).choice(n, m, replace=False)) if m < n else np.arange(n)
        take = {}
        for name, (arr, first, count, mask) in lists.items():
            f, c = first[idx][mask[idx]].astype(np.int64), count[idx][mask[idx]].astype(np.int64)
            take[name] = np.repeat(f - np.cumsum(c) + c, c) + np.arange(int(c.sum()))
        nbytes = 8 * m * (len(fields) + 1) + sum(8 * len(t) * max(1, len(lists[k][0].dtype.names or ())) for k, t in take.items())
        if nbytes <= DUMP_BYTES:
            break
        m //= 2
    out.mkdir(parents=True, exist_ok=True)
    np.save(out / "read_index.npy", idx.astype(np.float64))
    for f in fields:
        np.save(out / f"{f}.npy", records[f][idx].astype(np.float64))
    for name, t in take.items():
        if len(t) == 0:
            continue
        arr = lists[name][0][t]
        for f in arr.dtype.names or (None,):
            np.save(out / (f"{name}_{f}.npy" if f else f"{name}.npy"), (arr[f] if f else arr).astype(np.float64))
    return {"dir": str(out), "reads": int(m), "of_reads": int(n), "bytes": int(nbytes), "files": sorted(f.name for f in out.glob("*.npy"))}


def measure_cfg4(B, capi, torch, index, dev, d, scale, pairs, rank, steps, warmup, nb=4):
    """BASELINE.json configs[3] on the index that is already resident: cfg3's genome, 150 bp pairs, --pe --sensitive (the whole
    pair logic on the device: mate-range filter, hit compaction, one re-seeding round).  -> dict with the rank's device and
    end-to-end milliseconds for `steps` steps; the caller takes the maximum over ranks."""
    from bitmapperbs_b200.simulate import _revcomp_rows
    wl = Workload("cfg4", scale)
    m1, m2 = make_reads(d, wl, pairs, wl.read_seed + rank)
    n_reads = 2 * len(m1)
    mates = np.empty((n_reads, READ_LEN), dtype=np.uint8)
    mates[0::2] = m1; mates[1::2] = _revcomp_rows(m2)
    bases = mates.size
    h_flat = torch.empty(bases + 64, dtype=torch.uint8, pin_memory=True); h_flat.numpy()[:bases] = mates.ravel()
    h_offs = torch.empty(n_reads + 1, dtype=torch.int64, pin_memory=True); h_offs.numpy()[:] = np.arange(n_reads + 1, dtype=np.int64) * READ_LEN
    flat = h_flat.numpy()[:bases]; offs = h_offs.numpy().view(np.uint64)
    prm = capi.default_params(sensitive=1)
    cand_cap = 24 * n_reads
    while True:
        batches = [B.Batch(index, dev, n_reads, bases + 64, cand_cap) for _ in range(nb)]
        try:
            batches[0].upload(flat, offs, pe=True); batches[0].run(prm); batches[0].sync()
            hr = torch.empty(n_reads * capi.ReadResult.itemsize, dtype=torch.uint8, pin_memory=True)
            hc = torch.empty(cand_cap * capi.Cand.itemsize, dtype=torch.uint8, pin_memory=True)
            res, _, used = batches[0].download(hr.numpy().view(capi.ReadResult), hc.numpy().view(capi.Cand))
            states = np.bincount(res["state"], minlength=5)
            del hr, hc
            break
        except B.BmbsError as e:
            for x in batches:
                x.close()
            if e.code != -4:
                raise
            cand_cap *= 2
    # the pairs are finished on the device too (hit compaction, pair pick, ungapped CIGAR check, coordinates): two 32-byte records
    # per pair and the mismatch positions come back instead of the mates' hit lists
    bufs = []
    for _ in batches:
        hf = torch.empty(n_reads * capi.Final.itemsize, dtype=torch.uint8, pin_memory=True)
        hm = torch.empty((32 * n_reads + 64) * 2, dtype=torch.uint8, pin_memory=True)
        hb = torch.empty((1 << 16) * capi.Cand.itemsize, dtype=torch.uint8, pin_memory=True)
        bufs.append((hf, hm, hb, hf.numpy().view(capi.Final), hm.numpy().view(np.uint16), hb.numpy().view(capi.Cand)))

    def down(i):
        _, mm, fb = batches[i].download_final(bufs[i][3], bufs[i][4], bufs[i][5])
        return n_reads * capi.Final.itemsize + 2 * len(mm) + capi.Cand.itemsize * len(fb)
    for i in range(max(warmup, nb)):
        b = batches[i % nb]; b.upload(flat, offs, pe=True); b.run(prm); b.finish(); down(i % nb)
    torch.cuda.synchronize()
    stage, dev_ms = {}, 0.0
    for _ in range(steps):
        batches[0].run(prm); batches[0].finish()
        t = batches[0].timings()
        t["finish"] = batches[0].finish_counters()["device_us"] / 1000.0
        t["total"] += t["finish"]
        dev_ms += t["total"]
        for k, v in t.items():
            stage[k] = stage.get(k, 0.0) + v
    batches[0].sync()
    counters = batches[0].counters(); launches = batches[0].launches() * steps
    fin_status = np.bincount(bufs[0][3]["status"][0::2], minlength=5)
    torch.cuda.synchronize()
    e0 = time.perf_counter(); d2h = 0
    for i in range(steps):
        b = batches[i % nb]; b.upload(flat, offs, pe=True); b.run(prm); b.finish()
        if i >= nb - 1:
            d2h = down((i - (nb - 1)) % nb)
    for i in range(max(0, steps - (nb - 1)), steps):
        d2h = down(i % nb)
    e2e_ms = (time.perf_counter() - e0) * 1000
    for x in batches:
        x.close()
    return {"pair_status": {"no_pair": int(fin_status[0]), "reported": int(fin_status[1] + fin_status[3]), "ambiguous": int(fin_status[2])},"workload": wl.describe(len(m1)), "n_reads": n_reads, "steps": steps, "dev_ms": dev_ms, "e2e_ms": e2e_ms, "launches": launches,
            "stage_ms_per_step": {k: v / steps for k, v in stage.items()}, "work_per_step": counters, "h2d": int(bases + 8 * (n_reads + 1)), "d2h": int(d2h),
            "read_states": {"none": int(states[0]), "exact_unique": int(states[1]), "multi_exact": int(states[2]), "one_mismatch": int(states[3]), "verify": int(states[4])}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="cfg3", choices=["cfg3", "cfg2", "cfg4"])
    ap.add_argument("--reads", "--pairs", dest="units", type=int, default=1_000_000, help="reads (pairs) per GPU per step")
    ap.add_argument("--scale", type=float, default=None, help="fraction of the workload's full genome (cfg3/cfg4: of 3.087 Gbp)")
    ap.add_argument("--cache", default=os.environ.get("BMBS_BENCH_CACHE", "/tmp/bmbs_bench"))
    ap.add_argument("--ref-sample", type=int, default=500_000, help="reads (pairs) per reference-CPU run")
    ap.add_argument("--no-cpu-baseline", action="store_true", help="skip the reference runs and the whole-program comparison")
    ap.add_argument("--wp-reads", dest="wp_units", type=int, default=4_000_000, help="reads (pairs) of the whole-program comparison")
    ap.add_argument("--inflight", type=int, default=4, help="batches in flight in the end-to-end loop (measured: 2 -> 122, 3 -> 141, 4 -> 162, 6 -> 161 M reads/s)")
    ap.add_argument("--no-cfg4", action="store_true", help="skip the secondary cfg4 (--pe --sensitive) measurement on the same index")
    ap.add_argument("--cfg4-pairs", type=int, default=500_000, help="pairs per GPU per step of the cfg4 measurement")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step returned (rank 0) as .npy files under DIR")
    a = ap.parse_args()
    a.warmup = max(a.warmup, 3) if a.impl == "ours" else a.warmup
    scale = a.scale if a.scale is not None else float(os.environ.get("BMBS_BENCH_SCALE", DEFAULT_SCALE[a.workload]))
    wl = Workload(a.workload, scale)
    per_unit = 2 if wl.pe else 1

    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1")); local = int(os.environ.get("LOCAL_RANK", "0"))
    cache = Path(a.cache)
    cores = os.cpu_count() or 1
    workload = wl.describe(a.units)
    REF = ROOT / "oracle/_ref/bitmapperBS"

    # ---------------------------------------------------------------- reference arm
    if a.impl == "reference":
        if rank != 0:
            return 0
        if not REF.exists():
            print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref/bitmapperBS missing (built by oracle/build_ref.sh from /root/reference)"}))
            return 0
        d = ensure_dataset(cache, wl, True)
        m1, m2 = make_reads(d, wl, a.units, wl.read_seed)
        n, seq_args = write_fastq_files(d, wl, m1, m2, a.ref_sample, "ref")
        runs = []
        for _ in range(a.warmup + a.steps):
            r = run_cli(REF, d, wl, seq_args, cores, "/dev/null")
            if r is None:
                print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref/bitmapperBS failed on the workload"}))
                return 0
            runs.append(r)
        runs = runs[a.warmup:]
        map_s = sum(x[1] for x in runs)
        value = per_unit * n * len(runs) / map_s
        sample = (f"first {n} {'pairs' if wl.pe else 'reads'} of rank 0's batch per step, oracle/_ref/bitmapperBS {' '.join(wl.cli_flags())} -t {cores}, "
                  f"the reference's own mapping timer (index load excluded; covers seeding, verification, CIGAR, MAPQ and SAM text)")
        print(json.dumps({
            "impl": "reference", "metric": "mapped_reads_per_sec", "value": value, "unit": "reads/s", "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup,
            "ms_per_step": 1000 * map_s / len(runs), "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u64", "data": "synthetic",
            "config": {"workload": workload, "sample": sample, "reads_per_step": per_unit * n},
            "cpu_baseline": {"value": value, "unit": "reads/s", "cores": cores, "kind": "reference", "sample": sample},
            "e2e": {"value": value, "unit": "reads/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "load_s_per_step": sum(x[0] for x in runs) / len(runs), "wall_s_per_step": sum(x[2] for x in runs) / len(runs)}))
        return 0

    # ---------------------------------------------------------------- our arm
    # libraries (NCCL's version banner) may write to stdout: keep fd 1 for the one JSON line
    sys.stdout.flush()
    json_fd = os.dup(1); os.dup2(2, 1)
    import torch
    import bitmapperbs_b200 as B
    from bitmapperbs_b200 import capi
    dist = None
    if world > 1:
        import torch.distributed as dist
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = local
    torch.cuda.set_device(dev)
    full_affinity = os.sched_getaffinity(0)
    numa = bind_to_gpu_node(dev)         # pinned staging is first-touched by this process: keep it on the GPU's NUMA node
    d = ensure_dataset(cache, wl, rank == 0)
    if dist:
        dist.barrier()
    from bitmapperbs_b200 import shard
    m1, m2 = make_reads(d, wl, a.units, shard.rank_seed(wl.read_seed, rank))     # weak scaling: every rank maps its own reads
    n_units = len(m1); n_reads = per_unit * n_units
    if wl.pe:
        from bitmapperbs_b200.simulate import _revcomp_rows
        mates = np.empty((n_reads, READ_LEN), dtype=np.uint8)
        mates[0::2] = m1; mates[1::2] = _revcomp_rows(m2)
    else:
        mates = m1
    bases = mates.size
    # pinned host staging (torch is plumbing here: pinned memory, device selection, rendezvous)
    h_flat = torch.empty(bases + 64, dtype=torch.uint8, pin_memory=True); h_flat.numpy()[:bases] = mates.ravel()
    h_offs = torch.empty(n_reads + 1, dtype=torch.int64, pin_memory=True); h_offs.numpy()[:] = np.arange(n_reads + 1, dtype=np.int64) * READ_LEN
    flat = h_flat.numpy()[:bases]; offs = h_offs.numpy().view(np.uint64)

    t0 = time.time()
    index = B.Index(d / "g.fa.index", devices=(dev,))
    load_s = time.time() - t0
    log(f"[bench r{rank}] index resident: {index.device_bytes / 1e9:.2f} GB in {load_s:.1f}s")
    prm = capi.default_params(sensitive=1 if wl.sensitive else 0)
    cand_cap = 16 * n_reads
    while True:
        batch = B.Batch(index, dev, n_reads, bases + 64, cand_cap)
        batch.upload(flat, offs, pe=wl.pe); batch.run(prm)
        try:
            batch.sync()
            h_res = torch.empty(n_reads * capi.ReadResult.itemsize, dtype=torch.uint8, pin_memory=True)
            h_cand = torch.empty(cand_cap * capi.Cand.itemsize, dtype=torch.uint8, pin_memory=True)
            res = h_res.numpy().view(capi.ReadResult); cand = h_cand.numpy().view(capi.Cand)
            _, _, used = batch.download(res, cand)
            break
        except B.BmbsError as e:
            if e.code != -4:
                raise
            batch.close(); cand_cap *= 2
    states = np.bincount(res["state"], minlength=5)
    # single end: the device also finishes the reads (reduction in std::sort's order, ungapped CIGAR check, coordinates) and
    # 32-byte records come back instead of the window lists; pairs still return their lists (pair pick on the host)
    fin_mode = not wl.pe
    fin_cap = 32 * n_reads + 64; fb_cap = max(1 << 20, n_reads)

    def final_buffers():
        hf = torch.empty(n_reads * capi.Final.itemsize, dtype=torch.uint8, pin_memory=True)
        hm = torch.empty(fin_cap * 2, dtype=torch.uint8, pin_memory=True)
        hb = torch.empty(fb_cap * capi.Cand.itemsize, dtype=torch.uint8, pin_memory=True)
        keep.extend([hf, hm, hb])
        return hf.numpy().view(capi.Final), hm.numpy().view(np.uint16), hb.numpy().view(capi.Cand)
    # more in-flight batches for the end-to-end loop (each with its own stream and pinned result buffers): the H2D copy of
    # one batch overlaps the kernels of the previous one and the D2H copy of the one before
    keep = [h_res, h_cand]
    outs = [(batch, res, cand) + (final_buffers() if fin_mode else ())]
    for _ in range(a.inflight - 1):
        nb = B.Batch(index, dev, n_reads, bases + 64, cand_cap)
        if fin_mode:
            outs.append((nb, None, None) + final_buffers())
        else:
            hr = torch.empty(n_reads * capi.ReadResult.itemsize, dtype=torch.uint8, pin_memory=True)
            hc = torch.empty(cand_cap * capi.Cand.itemsize, dtype=torch.uint8, pin_memory=True)
            keep += [hr, hc]
            outs.append((nb, hr.numpy().view(capi.ReadResult), hc.numpy().view(capi.Cand)))
    NB = len(outs)

    def step_run(bb):
        bb.run(prm)
        if fin_mode:
            bb.finish()

    def step_download(o):
        """-> (bytes copied back, the arrays the call returned)"""
        if fin_mode:
            got = o[0].download_final(o[3], o[4], o[5])
            return n_reads * capi.Final.itemsize + 2 * len(got[1]) + capi.Cand.itemsize * len(got[2]), got
        r, c, u = o[0].download(o[1], o[2])
        return n_reads * capi.ReadResult.itemsize + u * capi.Cand.itemsize, (r, c[:u])
    clocks = ClockSampler(dev); clocks.start()
    for _ in range(max(0, a.warmup - 1)):
        step_run(batch)
    batch.sync()
    for i in range(max(a.warmup, NB)):
        o = outs[i % NB]
        o[0].upload(flat, offs, pe=wl.pe); step_run(o[0]); step_download(o)

    def barrier():
        torch.cuda.synchronize()
        if dist:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- timed: device-resident steps
    barrier()
    t_begin = time.time()
    stage = {}
    dev_ms = 0.0
    w0 = time.perf_counter()
    for _ in range(a.steps):
        step_run(batch)
        t = batch.timings()           # waits on the step's last event; CUDA-event times on the launching stream
        if fin_mode:
            t["finish"] = batch.finish_counters()["device_us"] / 1000.0
            t["total"] += t["finish"]
        dev_ms += t["total"]
        for k, v in t.items():
            stage[k] = stage.get(k, 0.0) + v
    batch.sync()
    wall_ms = (time.perf_counter() - w0) * 1000
    barrier()
    counters = batch.counters()
    launches = batch.launches() * a.steps
    fin_counters = batch.finish_counters() if fin_mode else None
    # ---- timed: end to end through the C ABI, host buffers in / out
    # (every step: H2D of the step's reads from pinned host memory, kernels, D2H of its records; NB batches in
    # flight on their own streams, as the host mapper drives them)
    barrier()
    e0 = time.perf_counter()
    d2h = 0
    for i in range(a.steps):
        o = outs[i % NB]
        o[0].upload(flat, offs, pe=wl.pe); step_run(o[0])
        if i >= NB - 1:
            d2h, last = step_download(outs[(i - (NB - 1)) % NB])
    for i in range(max(0, a.steps - (NB - 1)), a.steps):
        d2h, last = step_download(outs[i % NB])
    e2e_ms = (time.perf_counter() - e0) * 1000
    barrier()
    clk = clocks.stop(t_begin, time.time())
    if fin_mode:
        assert all(np.array_equal(outs[0][3]["status"], o[3]["status"]) and np.array_equal(outs[0][3]["chrom_pos"], o[3]["chrom_pos"]) for o in outs[1:])
        fin_status = np.bincount(outs[0][3]["status"], minlength=5)
    else:
        assert all(np.array_equal(outs[0][1]["state"], o[1]["state"]) for o in outs[1:])
    dumped = None
    if a.dump_outputs and rank == 0:
        if fin_mode:      # finished records; mismatch positions of the reads finished on the device, windows of those handed back
            fin, mm, fb = last
            host = fin["status"] == capi.FIN_HOST
            dumped = dump_outputs(Path(a.dump_outputs), fin, [f for f in capi.Final.names if f != "aux_first"],
                                  {"mismatch_pos": (mm, fin["aux_first"], fin["n_aux"], ~host), "handed_back": (fb, fin["aux_first"], fin["n_aux"], host)})
        else:             # per-read records and their verified windows
            res, cand = last
            dumped = dump_outputs(Path(a.dump_outputs), res, [f for f in capi.ReadResult.names if f not in ("first_cand", "reserved")],
                                  {"cand": (cand, res["first_cand"], res["n_cand"], np.ones(len(res), bool))})
    h2d = int(bases + 8 * (n_reads + 1)); d2h = int(d2h)
    os.sched_setaffinity(0, full_affinity)        # the command-line runs below use every core of the box

    # ---- secondary: BASELINE.json configs[3] (cfg4 = the same genome, --pe --sensitive) on the resident index
    c4 = None
    if wl.name == "cfg3" and not a.no_cfg4:
        for o in outs:
            o[0].close()
        try:
            c4 = measure_cfg4(B, capi, torch, index, dev, d, scale, a.cfg4_pairs, rank, a.steps, a.warmup, a.inflight)
        except Exception as e:      # the headline line must not depend on the secondary measurement
            log(f"[bench r{rank}] cfg4 measurement failed: {e}")
    c4_ms = [c4["dev_ms"], c4["e2e_ms"]] if c4 else [0.0, 0.0]
    # the slowest rank's times count (one MAX reduction outside the timed work)
    dev_ms, e2e_ms, wall_ms, c4_ms[0], c4_ms[1], c4_missing = shard.max_over_ranks(dist, [dev_ms, e2e_ms, wall_ms] + c4_ms + [0.0 if c4 else 1.0],
                                                                                   device=f"cuda:{dev}" if dist else None)
    if c4_missing:
        c4 = None
    if rank != 0:
        if dist:
            dist.destroy_process_group()
        return 0

    value = shard.whole_job_rate(n_reads, world, a.steps, dev_ms)
    e2e = shard.whole_job_rate(n_reads, world, a.steps, e2e_ms)
    # ---- roofline of the dominant kernel group (SURVEY.md §8d algorithmic bytes per unit)
    peaks = {}
    try:
        peaks = json.loads((ROOT / "MEASURED_PEAKS.json").read_text())
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0)); peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if peaks else "fallback 6.65 TB/s (B200_PROFILING.md)"
    per_step = {k: v / a.steps for k, v in stage.items()}
    c = counters
    dense = c["locate_lf_steps"] == 0
    # SURVEY §8d units (the reference's layout): 10 B per 16-mer query, 40 B per occ lookup, (80 B per LF step + 44 B) per located row;
    # this layout's own units (DESIGN.md §3): 8 B per table entry, 32 B per occ block, 4-5 B per located row of the dense suffix array
    survey = {"seed": 10 * c["hash_queries"] + 40 * c["occ_lookups"], "locate": 80 * c["locate_lf_steps"] + 44 * c["located_rows"], "verify": c["window_bytes"]}
    layout = {"seed": 8 * c["hash_queries"] + 32 * c["occ_lookups"],
              "locate": c["located_rows"] * (5 if index.genome_length * 2 >= (1 << 32) else 4) if dense else 80 * c["locate_lf_steps"] + 44 * c["located_rows"],
              "verify": c["window_bytes"]}
    names = {"seed": "seed_reads", "locate": "expand_locate", "verify": "verify_windows"}
    dom = max(names, key=lambda k: per_step[k])
    dms = per_step[dom]
    achieved = survey[dom] / (dms / 1000) / 1e9 if dms > 0 else 0.0
    # DRAM traffic of the same kernels from the committed `ncu --set full` capture (profiles/ncu_traffic.json), per launch
    traffic = None
    try:
        tj = json.loads((ROOT / "profiles/ncu_traffic.json").read_text())
        traffic = tj.get(wl.name, {}).get(names[dom], {}).get("dram_bytes_per_launch")
    except Exception:
        pass
    try:
        rs_peak = capi.random_sector_peak(dev)      # independent random 32-byte sector loads per second (measured live)
    except Exception:
        rs_peak = None
    accesses = {"seed": c["hash_queries"] + c["occ_lookups"], "locate": c["located_rows"] + c["locate_lf_steps"] * 2, "verify": None}
    # ---- integer roofline of verification: GCUPS and word-ops (14 per column per band word; 1 word for k <= 15, 2 above)
    try:
        int_peak = capi.int_pipe_peak(dev)
    except Exception:
        int_peak = None
    k_band = int(min(31, int(0.08 * READ_LEN)))
    words = 1 if k_band <= 15 else 2
    vms = per_step["verify"]
    gcups = c["cells"] / (vms / 1000) / 1e9 if vms > 0 else 0.0
    columns = c["cells"] / (2 * k_band + 1)
    int_ops = 14 * words * columns
    out = {
        "metric": "mapped_reads_per_sec", "value": value, "unit": "reads/s", "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
        "ms_per_step": dev_ms / a.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u64", "data": "synthetic",
        "config": {"workload": workload, "reads_per_step_per_gpu": n_reads,
                   "l2": f"inputs ({bases / 1e6:.0f} MB of reads, {index.device_bytes / 1e9:.1f} GB index) exceed the 126 MB L2; no flush needed",
                   "read_states": {"none": int(states[0]), "exact_unique": int(states[1]), "multi_exact": int(states[2]), "one_mismatch": int(states[3]), "verify": int(states[4])},
                   "index_hbm_bytes": index.device_bytes, "index_load_s": load_s, "genome_bases": index.genome_length},
        "e2e": {"value": e2e, "unit": "reads/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "ms_per_step": e2e_ms / a.steps, "batches_in_flight": NB,
                "numa_node": numa,
                "scope": ("C-ABI calls bmbs_batch_upload / _run / _finish / _download_final: H2D of the reads, kernels incl. the device finishing (reduction, ungapped CIGAR, "
                          "coordinates), D2H of one 32-byte record per read + mismatch positions (MAPQ table lookup and SAM text are in whole_program)") if fin_mode else
                         "C-ABI call: H2D of the reads, kernels, D2H of records + verified candidate lists (pair pick / CIGAR / SAM are in whole_program)"},
        "gpu_launches": launches,
        "clocks": clk,
        "stage_ms_per_step": per_step,
        "wall_ms_per_step": wall_ms / a.steps,
        "dumped_outputs": dumped,
        "verify_gcups": gcups,
        "work_per_step": counters,
        "finishing": ({"status": {"unmapped": int(fin_status[0]), "unique_ungapped": int(fin_status[1]), "ambiguous": int(fin_status[2]), "needs_dp": int(fin_status[3]),
                                  "handed_back_to_host": int(fin_status[4])}, **fin_counters} if fin_mode else None),
        "roofline": {"bound": "hbm", "kernel": names[dom], "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak if peak else None, "traffic": traffic,
                     "peak_source": peak_src, "kernel_ms": dms,
                     "algorithmic_bytes_per_launch": survey[dom], "units": "SURVEY 8d: 10 B per table query, 40 B per occ lookup, 80 B per locate LF step + 44 B per located row, window bytes",
                     "layout_bytes_per_launch": layout[dom], "layout_units": "this layout: 8 B per table entry, 32 B per occ block, 4-5 B per located row (dense suffix array)",
                     "layout_frac": layout[dom] / (dms / 1000) / 1e9 / peak if dms > 0 and peak else None,
                     # DRAM bytes the kernels really move (ncu, profiles/ncu_traffic.json) over the live kernel time: every random 8-byte
                     # table entry / 32-byte occ block costs a whole DRAM line, so this -- not the algorithmic figure -- is what loads HBM
                     "traffic_gbs": traffic / (dms / 1000) / 1e9 if traffic and dms > 0 else None,
                     "traffic_frac_of_peak": traffic / (dms / 1000) / 1e9 / peak if traffic and dms > 0 and peak else None,
                     "random_access_peak_per_s": rs_peak, "random_accesses_per_s": accesses[dom] / (dms / 1000) if accesses[dom] and dms > 0 else None,
                     "frac_of_random_access_peak": accesses[dom] / (dms / 1000) / rs_peak if accesses[dom] and dms > 0 and rs_peak else None,
                     "all_kernels": {names[k]: {"ms": per_step[k], "survey_bytes": survey[k], "layout_bytes": layout[k],
                                                "GBps": (survey[k] / (per_step[k] / 1000) / 1e9 if per_step[k] > 0 else 0.0)} for k in names}},
        "roofline_int": {"bound": "int-alu", "kernel": "verify_windows", "gcups": gcups, "cells_per_launch": c["cells"], "windows_per_launch": c["verified"],
                         "achieved": int_ops / (vms / 1000) / 1e12 if vms > 0 else 0.0, "peak": int_peak / 1e12 if int_peak else None, "unit": "T int32 ops/s",
                         "frac": int_ops / (vms / 1000) / int_peak if vms > 0 and int_peak else None, "kernel_ms": vms,
                         "units": f"14 word-ops per column per band word (SURVEY 8d), {words} word(s) for k = {k_band}; peak = measured LOP3+IADD3 rate (bmbs_ubench_int_pipe)"},
    }
    if c4:
        out["cfg4"] = {"workload": c4["workload"], "value": shard.whole_job_rate(c4["n_reads"], world, c4["steps"], c4_ms[0]), "unit": "reads/s", "steps": c4["steps"],
                       "ms_per_step": c4_ms[0] / c4["steps"], "reads_per_step_per_gpu": c4["n_reads"], "gpu_launches": c4["launches"],
                       "e2e": {"value": shard.whole_job_rate(c4["n_reads"], world, c4["steps"], c4_ms[1]), "unit": "reads/s", "h2d_bytes_per_step": c4["h2d"], "d2h_bytes_per_step": c4["d2h"],
                               "ms_per_step": c4_ms[1] / c4["steps"], "batches_in_flight": a.inflight},
                       "stage_ms_per_step": c4["stage_ms_per_step"], "work_per_step": c4["work_per_step"], "read_states": c4["read_states"], "pair_status": c4["pair_status"],
                       "scope": "secondary measurement on the same resident index (BASELINE.json configs[3]); device pipeline incl. the sensitive pair logic, the re-seeding round and the "
                                "pair finishing (hit compaction, pair pick, ungapped CIGAR check, coordinates); two 32-byte records per pair + mismatch positions back (banded DP of indel "
                                "mates, MAPQ, SAM text on the host); max over ranks like the headline"}
    # ---- the whole program and the reference on this box's host cores (rank 0, N == 1 only)
    if world == 1 and not a.no_cpu_baseline:
        BMBS = ROOT / "bitmapperbs_b200/_build/bmbs"
        # a file of --wp-reads reads (pairs) of its own: at 1 M reads the program's mapping phase is mostly its start-up
        wm1, wm2 = (m1, m2) if a.wp_units <= len(m1) else make_reads(d, wl, a.wp_units, wl.read_seed + 555)
        n, seq_args = write_fastq_files(d, wl, wm1, wm2, a.wp_units, "wp")
        wp = {"reads": per_unit * n, "host_cores": cores, "scope": "FASTQ file -> SAM file through the command line, index load and the program's mapping phase timed by its own `Total:` line; "
                                                                   "this build: the faster of two runs (the boxes are shared), both listed"}
        run_cli(BMBS, d, wl, seq_args, cores, "/dev/null")                               # page cache + driver warm-up
        gs = [x for x in (run_cli(BMBS, d, wl, seq_args, cores, "wp_gpu.sam") for _ in range(2)) if x]
        g = min(gs, key=lambda x: x[1]) if gs else None
        if g:
            wp["ours"] = {"load_s": g[0], "map_s": g[1], "wall_s": g[2], "reads_per_s_map": per_unit * n / g[1] if g[1] > 0 else None, "reads_per_s_wall": per_unit * n / g[2],
                          "map_s_all": [x[1] for x in gs]}
        if REF.exists():
            r = run_cli(REF, d, wl, seq_args, cores, "wp_ref.sam")
            if r:
                wp["reference"] = {"load_s": r[0], "map_s": r[1], "wall_s": r[2], "reads_per_s_map": per_unit * n / r[1] if r[1] > 0 else None, "reads_per_s_wall": per_unit * n / r[2]}
                if g:
                    wp["map_speedup"] = r[1] / g[1] if g[1] > 0 else None; wp["wall_speedup"] = r[2] / g[2]
                    try:      # same records?  (the reference's -t N order is not deterministic: compare sorted bodies)
                        import hashlib

                        def digest(p):      # multiset of the record lines: count + sum of their 128-bit digests (no sort of millions of lines)
                            k, acc = 0, 0
                            for line in open(p, "rb"):
                                if not line.startswith(b"@"):
                                    acc = (acc + int.from_bytes(hashlib.blake2b(line, digest_size=16).digest(), "little")) & ((1 << 128) - 1); k += 1
                            return k, acc
                        wp["sam_identical"] = digest(d / "wp_gpu.sam") == digest(d / "wp_ref.sam")
                    except Exception:
                        pass
            ns, sargs = write_fastq_files(d, wl, m1, m2, a.ref_sample, "ref")
            r2 = run_cli(REF, d, wl, sargs, cores, "/dev/null")
            if r2:
                out["cpu_baseline"] = {"value": per_unit * ns / r2[1], "unit": "reads/s", "cores": cores, "kind": "reference",
                                       "sample": f"first {ns} {'pairs' if wl.pe else 'reads'} of the step's batch, oracle/_ref/bitmapperBS {' '.join(wl.cli_flags())} -t {cores}, its own mapping timer (page cache warm)",
                                       "wall_s": r2[2]}
        for f in ("wp_gpu.sam", "wp_ref.sam"):
            try:
                (d / f).unlink()
            except OSError:
                pass
        out["whole_program"] = wp
        if "cpu_baseline" not in out:
            out["cpu_baseline"] = {"value": None, "unit": "reads/s", "cores": cores, "kind": "reference", "sample": "oracle/_ref/bitmapperBS unavailable"}
    elif world > 1:
        out["cpu_baseline"] = {"value": None, "unit": "reads/s", "cores": cores, "kind": "reference", "sample": "measured at N = 1 only (bench contract); see the N = 1 line and --impl reference"}
    sys.stdout.flush()
    os.write(json_fd, (json.dumps(out) + "\n").encode())
    if dist:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
