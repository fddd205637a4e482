"""Host finishing code of the product (bitmapperbs_b200/csrc/host/mapper.hpp: vote-ordered reduction, pair pick, CIGAR
refinement, MAPQ, SAM text; finish_single_final / finish_pair_final behind the finished records), on the CPU: fed with the ORACLE's per-read records -- the same arrays the GPU library returns
(tests/test_gpu_parity.py) -- its SAM must equal the golden SAM of the real reference, record for record, and the
--mapstats counters with it.  Covers single end, paired end fast and sensitive, and --unmapped_out, --ambiguous_out and --pbat
against the reference's output (tests/reference_sha256.py)."""
import subprocess
from pathlib import Path

import pytest

import reference_sha256
from conftest import sam_body

ROOT = Path(__file__).resolve().parent.parent


@pytest.fixture(scope="module")
def harness(built, tmp_path_factory):
    exe = tmp_path_factory.mktemp("hf") / "host_finish_harness"
    subprocess.run(["g++", "-O2", "-std=c++17", "-pthread", "-Wno-sign-compare", str(ROOT / "tests/host_finish_harness.cpp"), "-o", str(exe), "-lz"], check=True)
    return exe


CASES = [("se100", "se", ["se100.fq"]), ("se250", "se", ["se250.fq"]), ("se100", "sef", ["se100.fq"]), ("se250", "sef", ["se250.fq"]), ("pe150", "pe", ["pe150_1.fq", "pe150_2.fq"]),
         ("pe150s", "pes", ["pe150_1.fq", "pe150_2.fq"]), ("pe100h", "pe", ["pe100h_1.fq", "pe100h_2.fq"]), ("pe100hs", "pes", ["pe100h_1.fq", "pe100h_2.fq"]),
         # pairs through the finished records: orc_finish_pe (what the device's finish_pe is compared with) -> finish_pair_final
         ("pe150", "pef", ["pe150_1.fq", "pe150_2.fq"]), ("pe150s", "pesf", ["pe150_1.fq", "pe150_2.fq"]),
         ("pe100h", "pef", ["pe100h_1.fq", "pe100h_2.fq"]), ("pe100hs", "pesf", ["pe100h_1.fq", "pe100h_2.fq"])]


@pytest.mark.parametrize("name,mode,files", CASES)
def test_host_finish_matches_reference_golden(golden, harness, name, mode, files):
    out = golden / f"hf_{name}.sam"
    r = subprocess.run([str(harness), mode, "genome.fa", out.name, *files], cwd=golden, check=True, capture_output=True, text=True)
    assert sam_body(out) == sam_body(golden / f"{name}.sam")
    n, uq, am, rate = r.stdout.split()
    st = (golden / f"ref_{name}.stats").read_text().splitlines()
    assert int(st[0].split()[-1]) == int(n) and int(st[1].split(":")[1].split()[0]) == int(uq) and int(st[2].split(":")[1].split()[0]) == int(am)
    assert st[4].split()[-1] == f"{float(rate):.2f}%"


@pytest.mark.parametrize("mode,files", [("se", ["se100.fq"]), ("sef", ["se100.fq"]), ("pe", ["pe100h_1.fq", "pe100h_2.fq"]), ("pes", ["pe100h_1.fq", "pe100h_2.fq"]),
                                        ("pef", ["pe100h_1.fq", "pe100h_2.fq"]), ("pesf", ["pe100h_1.fq", "pe100h_2.fq"])])
def test_unmapped_out_matches_live_reference(golden, built, harness, mode, files):
    """against the reference's SAM: its stored digest, and the live reference where it is built"""
    subprocess.run([str(harness), mode, "genome.fa", f"hf_un_{mode}.sam", *files, "--unmapped_out"], cwd=golden, check=True, capture_output=True)
    ours = sam_body(golden / f"hf_un_{mode}.sam")
    reference_sha256.check(f"host_finish_unmapped_out:{mode}", b"".join(ours))
    if built["ref"].exists():
        args = ["--seq", files[0]] if mode in ("se", "sef") else ["--seq1", files[0], "--seq2", files[1], "--pe"] + (["--sensitive"] if mode in ("pes", "pesf") else [])
        subprocess.run([str(built["ref"]), "--search", "genome.fa", *args, "--unmapped_out", "-t", "1", "-o", f"ref_un_{mode}.sam"],
                       cwd=golden, check=True, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
        assert ours == sam_body(golden / f"ref_un_{mode}.sam")


@pytest.mark.parametrize("mode,files,flags", [("pe", ["pe100h_1.fq", "pe100h_2.fq"], ["--ambiguous_out"]), ("pes", ["pe100h_1.fq", "pe100h_2.fq"], ["--ambiguous_out", "--unmapped_out"]),
                                              ("pef", ["pe100h_1.fq", "pe100h_2.fq"], ["--ambiguous_out"]), ("pesf", ["pe100h_1.fq", "pe100h_2.fq"], ["--ambiguous_out", "--unmapped_out"]),
                                              ("pef", ["pe150_2.fq", "pe150_1.fq"], ["--pbat"]), ("pesf", ["pe100h_2.fq", "pe100h_1.fq"], ["--pbat", "--unmapped_out"]),
                                              ("pe", ["pe150_2.fq", "pe150_1.fq"], ["--pbat"]), ("pes", ["pe100h_2.fq", "pe100h_1.fq"], ["--pbat", "--unmapped_out"]),
                                              ("se", ["se100_rc.fq"], ["--pbat", "--unmapped_out"]), ("se", ["se100.fq"], ["--pbat", "--unmapped_out"]),
                                              ("sef", ["se100_rc.fq"], ["--pbat", "--unmapped_out"]), ("sef", ["se100.fq"], ["--pbat", "--unmapped_out"])])
def test_flag_rows_match_live_reference(golden, built, harness, mode, files, flags):
    """--ambiguous_out (paired end), --pbat (single end on reverse-complemented reads and on directional ones; paired end with
    the files swapped so that pairs still map) and --unmapped_out with them, against the reference's SAM (its stored digest, and the
    live reference where it is built)"""
    if not (golden / "se100_rc.fq").exists():
        comp = bytes.maketrans(b"ACGTacgt", b"TGCAtgca")
        ls = (golden / "se100.fq").read_bytes().split(b"\n")
        with open(golden / "se100_rc.fq", "wb") as o:
            for i in range(0, len(ls) - 1, 4):
                o.write(ls[i] + b"\n" + ls[i + 1].translate(comp)[::-1] + b"\n+\n" + ls[i + 3][::-1] + b"\n")
    tag = mode + "_" + "_".join(f.strip("-") for f in flags) + "_" + files[0].split(".")[0]
    args = ["--seq", files[0]] if mode in ("se", "sef") else ["--seq1", files[0], "--seq2", files[1], "--pe"] + (["--sensitive"] if mode in ("pes", "pesf") else [])
    subprocess.run([str(harness), mode, "genome.fa", f"hf_{tag}.sam", *files, *flags], cwd=golden, check=True, capture_output=True)
    ours = sam_body(golden / f"hf_{tag}.sam")
    assert len(ours) > 100
    reference_sha256.check(f"host_finish_flags:{tag}", b"".join(ours))
    if built["ref"].exists():
        subprocess.run([str(built["ref"]), "--search", "genome.fa", *args, *flags, "-t", "1", "-o", f"ref_{tag}.sam"],
                       cwd=golden, check=True, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
        assert ours == sam_body(golden / f"ref_{tag}.sam")
