"""Host BAM writer (bitmapperbs_b200/csrc/host/bam.hpp, behind `bmbs --bam`): the golden SAM files of the real reference are
turned into BAM by the same calls the mapper makes, decoded here with nothing but gzip + struct, and compared with the SAM
text field by field; and the record bytes are compared with what the reference's own writer produces (the stock reference linked
with its vendored, patched htslib: bam_prase.cpp:248-274 -> chhy_bam_write1_pure; oracle/_ref/bitmapperBS_bam)."""
import gzip
import struct
import subprocess
from pathlib import Path

import pytest

import reference_sha256

ROOT = Path(__file__).resolve().parent.parent
GOLDEN = ROOT / "tests/golden"


@pytest.fixture(scope="module")
def harness(tmp_path_factory):
    exe = tmp_path_factory.mktemp("bam") / "bam_harness"
    subprocess.run(["g++", "-O2", "-std=c++17", str(ROOT / "tests/host_bam_harness.cpp"), "-o", str(exe), "-lz"], check=True)
    return exe


def decode_bam(path):
    raw = open(path, "rb").read()
    # BGZF: every member carries the BC extra field with its own size, and the file ends with the 28-byte EOF member
    assert raw[-28:] == bytes.fromhex("1f8b08040000000000ff0600424302001b0003000000000000000000")
    at, n_members = 0, 0
    while at < len(raw):
        assert raw[at:at + 4] == b"\x1f\x8b\x08\x04" and raw[at + 12:at + 14] == b"BC"
        bsize = struct.unpack_from("<H", raw, at + 16)[0] + 1
        isize = struct.unpack_from("<I", raw, at + bsize - 4)[0]
        assert isize <= 65536
        at += bsize; n_members += 1
    assert at == len(raw)
    data = gzip.decompress(raw)
    assert data[:4] == b"BAM\x01"
    l_text = struct.unpack_from("<i", data, 4)[0]
    text = data[8:8 + l_text].decode()
    p = 8 + l_text
    n_ref = struct.unpack_from("<i", data, p)[0]; p += 4
    refs = []
    for _ in range(n_ref):
        l = struct.unpack_from("<i", data, p)[0]; p += 4
        name = data[p:p + l - 1].decode(); p += l
        refs.append((name, struct.unpack_from("<i", data, p)[0])); p += 4
    recs = []
    while p < len(data):
        bs = struct.unpack_from("<i", data, p)[0]; q = p + 4
        rid, pos, l_name, mapq, bin_, n_cig, flag, l_seq, nrid, npos, tlen = struct.unpack_from("<iiBBHHHiiii", data, q); q += 32
        name = data[q:q + l_name - 1].decode(); q += l_name
        cig = "".join(f"{c >> 4}{'MIDNSHP=X'[c & 15]}" for c in struct.unpack_from(f"<{n_cig}I", data, q)) or "*"; q += 4 * n_cig
        sq = data[q:q + (l_seq + 1) // 2]; q += (l_seq + 1) // 2
        seq = "".join("=ACMGRSVTWYHKDBN"[(sq[i // 2] >> (4 if i % 2 == 0 else 0)) & 15] for i in range(l_seq))
        qual = "".join(chr(c + 33) for c in data[q:q + l_seq]); q += l_seq
        aux = data[q:p + 4 + bs]
        tags = []
        a = 0
        while a < len(aux):
            tag, ty = aux[a:a + 2].decode(), chr(aux[a + 2]); a += 3
            size = {"C": 1, "c": 1, "S": 2, "s": 2, "I": 4, "i": 4}[ty]
            val = int.from_bytes(aux[a:a + size], "little", signed=ty.islower()); a += size
            tags.append(f"{tag}:i:{val}")
        recs.append(dict(name=name, flag=flag, rid=rid, pos=pos, mapq=mapq, bin=bin_, cigar=cig, nrid=nrid, npos=npos, tlen=tlen, seq=seq, qual=qual, tags=tags))
        p += 4 + bs
    return text, refs, recs, n_members


def reg2bin(beg, end):
    end -= 1
    for shift, off in ((14, 4681), (17, 585), (20, 73), (23, 9), (26, 1)):
        if beg >> shift == end >> shift:
            return off + (beg >> shift)
    return 0


@pytest.mark.parametrize("name", ["se100", "se250", "pe150", "pe100hs"])
def test_bam_matches_sam(harness, tmp_path, name):
    sam = tmp_path / f"{name}.sam"
    with gzip.open(GOLDEN / f"{name}.sam.gz", "rb") as f:
        body = f.read().decode()
    extra = "unmapped1\t4\t*\t0\t0\t*\t*\t0\t0\tACGTN\tIIII#\n" + "pairun\t77\t*\t0\t0\t*\t*\t0\t0\tAC\tII\npairun\t141\t*\t0\t0\t*\t*\t0\t0\tGT\tII\n"
    header = "".join(l + "\n" for l in body.splitlines() if l.startswith("@"))
    if "@SQ" not in header:     # the golden files hold records only: the header comes from the golden genome
        names, lens = [], []
        with gzip.open(GOLDEN / "genome.fa.gz", "rt") as g:
            for l in g:
                if l.startswith(">"):
                    names.append(l[1:].split()[0]); lens.append(0)
                else:
                    lens[-1] += len(l.strip())
        header = "@HD\tVN:1.4\tSO:unsorted\n" + "".join(f"@SQ\tSN:{n}\tLN:{k}\n" for n, k in zip(names, lens)) + "@PG\tID:BitMapperBS\tVN:1.0.2.3\tCL:test\n"
    lines = [l for l in body.splitlines() if l and not l.startswith("@")] + extra.splitlines()
    sam.write_text(header + "\n".join(lines) + "\n")
    out = tmp_path / f"{name}.bam"
    subprocess.run([str(harness), str(sam), str(out)], check=True)
    text, refs, recs, n_members = decode_bam(out)
    assert text == header
    sq = [(l.split("\t")[1][3:], int(l.split("\t")[2][3:])) for l in header.splitlines() if l.startswith("@SQ")]
    assert refs == sq
    rid = {n: i for i, (n, _) in enumerate(sq)}
    assert len(recs) == len(lines) and n_members >= 3
    for l, r in zip(lines, recs):
        f = l.split("\t")
        assert r["name"] == f[0] and r["flag"] == int(f[1]) and r["mapq"] == int(f[4]) and r["cigar"] == f[5]
        assert r["rid"] == (rid[f[2]] if f[2] != "*" else -1) and r["pos"] == int(f[3]) - 1
        assert r["nrid"] == (r["rid"] if f[6] == "=" else -1) and r["npos"] == int(f[7]) - 1 and r["tlen"] == int(f[8])
        assert r["seq"] == f[9] and r["qual"] == f[10] and r["tags"] == f[11:]
        import re
        ref_len = sum(int(n) for n, op in re.findall(r"(\d+)([MIDNSHP=X])", f[5]) if op in "MDN=X")
        assert r["bin"] == reg2bin(r["pos"], r["pos"] + (ref_len or 1))


# ---- against the reference's own BAM writer: oracle/_ref/bitmapperBS_bam is the stock reference linked with its vendored, patched
# htslib (chhy_bam_write1_pure, bam_prase.cpp:248-274; built by oracle/build_ref.sh from the reference's sources)
def bam_payload(path):
    """-> (header text, reference dictionary bytes, the records exactly as they stand in the decompressed stream)"""
    d = gzip.decompress(open(path, "rb").read())
    assert d[:4] == b"BAM\x01"
    l_text = struct.unpack_from("<i", d, 4)[0]
    p = 8 + l_text
    n_ref = struct.unpack_from("<i", d, p)[0]; q = p + 4
    for _ in range(n_ref):
        q += 4 + struct.unpack_from("<i", d, q)[0] + 4
    return d[8:8 + l_text].decode(), d[p:q], d[q:]


@pytest.fixture(scope="module")
def finish_harness(tmp_path_factory):
    exe = tmp_path_factory.mktemp("hf") / "host_finish_harness"
    subprocess.run(["g++", "-O2", "-std=c++17", "-pthread", "-Wno-sign-compare", str(ROOT / "tests/host_finish_harness.cpp"), "-o", str(exe), "-lz"], check=True)
    return exe


@pytest.mark.parametrize("name,args", [("se100", ["--seq", "se100.fq"]), ("se250", ["--seq", "se250.fq", "--unmapped_out"]),
                                       ("pe150", ["--seq1", "pe150_1.fq", "--seq2", "pe150_2.fq", "--pe"]),
                                       ("pe100hs", ["--seq1", "pe100h_1.fq", "--seq2", "pe100h_2.fq", "--pe", "--sensitive", "--unmapped_out"])])
def test_bam_records_identical_to_the_reference_writer(harness, finish_harness, golden, name, args):
    """the reference writes the same alignments once as SAM and once as BAM; the product's writer turns that SAM into a BAM whose
    reference dictionary and record bytes (every field, bin, packed sequence, tags) equal the reference's own.  Where the reference
    is not built, the SAM comes from the host finishing (held to the reference's SAM by test_host_finish.py) and the BAM bytes
    are compared with the reference's through their stored digest (tests/reference_sha256.py)."""
    ref = ROOT / "oracle/_ref/bitmapperBS_bam"
    if ref.exists():
        for out, fmt in ((f"refw_{name}.bam", ["--bam"]), (f"refw_{name}.sam", [])):
            subprocess.run([str(ref), "--search", "genome.fa", *args, *fmt, "-t", "1", "-o", out], cwd=golden, check=True, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
        sam = golden / f"refw_{name}.sam"
    else:
        mode = ("pes" if "--sensitive" in args else "pe") if "--pe" in args else "se"
        files = [a for a in args if a.endswith(".fq")]
        sam = golden / f"hfw_{name}.sam"
        subprocess.run([str(finish_harness), mode, "genome.fa", sam.name, *files, *(a for a in args if a == "--unmapped_out")],
                       cwd=golden, check=True, capture_output=True)
    subprocess.run([str(harness), str(sam), str(golden / f"ours_{name}.bam")], check=True)
    ot, od, orr = bam_payload(golden / f"ours_{name}.bam")
    assert len(orr) > 10000
    reference_sha256.check(f"bam_writer:{name}", od + orr)
    if ref.exists():
        rt, rd, rr = bam_payload(golden / f"refw_{name}.bam")
        assert od == rd and orr == rr
        strip = lambda t: [l for l in t.splitlines() if not l.startswith("@PG")]      # the @PG line carries each run's command line
        assert strip(ot) == strip(rt)
