"""include/lphash_b200_fastx.hpp (host ingest: FASTA/FASTQ text -> batch layout) against a direct
Python port of kseq_read (the reference's external/kseq.h:193-240), the parser of the reference's
drivers: record i of the batch must be the i-th `seq->seq.s`."""
import gzip
import json
import os
import subprocess

import numpy as np
import pytest

from conftest import GOLDEN_DIR, ROOT

SRC = os.path.join(ROOT, "tests", "cpp", "fastx_check.cpp")


def kseq_records(data: bytes) -> list[bytes]:
    """kseq_read in a loop until it returns < 0 (what `while (kseq_read(seq) >= 0)` processes)."""
    recs, p, n, last = [], 0, len(data), 0

    def getc():
        nonlocal p
        if p >= n:
            return -1
        c = data[p]
        p += 1
        return c

    def line(acc=2):
        """rest of the current line (KS_SEP_LINE) appended to a string that already holds `acc`
        characters: without the newline, and without a trailing CR if the string is then longer than
        one character (ks_getuntil2: `str->l > 1 && str->s[str->l-1] == '\\r'`); None at EOF"""
        nonlocal p
        if p >= n:
            return None
        e = data.find(b"\n", p)
        if e < 0:
            e = n
        s = data[p:e]
        p = min(e + 1, n)
        if acc + len(s) > 1 and (s.endswith(b"\r") if s else False):
            s = s[:-1]
        return s

    while True:
        if last == 0:
            c = getc()
            while c >= 0 and c not in (ord(">"), ord("@")):
                c = getc()
            if c < 0:
                break
            last = c
        if p >= n:  # ks_getuntil on an exhausted stream: -1
            break
        line()  # name + comment
        seq = bytearray()
        c = getc()
        while c >= 0 and c not in (ord(">"), ord("+"), ord("@")):
            if c != ord("\n"):
                seq.append(c)
                rest = line(len(seq))
                if rest is not None:
                    seq += rest
                    if not rest and len(seq) > 1 and seq.endswith(b"\r"):
                        del seq[-1]  # the line was only "\r" and the sequence is longer than it
            c = getc()
        if c in (ord(">"), ord("@")):
            last = c
        if c != ord("+"):
            recs.append(bytes(seq))
            if c < 0:
                break
            continue
        c = getc()  # skip the rest of the '+' line
        while c >= 0 and c != ord("\n"):
            c = getc()
        if c == -1:
            break  # -2: no quality string
        qual = 0
        while True:
            q = line(qual)
            if q is None:
                break
            qual += len(q)
            if qual >= len(seq):
                break
        last = 0
        if qual != len(seq):
            break  # -2
        recs.append(bytes(seq))
    return recs


CASES = {
    "fasta_multiline": b">a desc\nACGT\nACG\n\nAC\n>b\n>c\nNNNN\nacgu\n>d",
    "fasta_crlf": b">a\r\nACGT\r\nAC\r\n>b\r\nGG\r\n",
    # kseq keeps the CR of a lone "\r\n" line when it is the FIRST sequence line (accumulated length 1)
    "fasta_crlf_blank_first": b">a\r\n\r\nACGT\r\n\r\nAC\r\n>b\r\n\r\n>c\r\nG\r\n",
    "fastq_crlf_blank_first": b"@r1\r\n\r\nACG\r\n+\r\n\r\nIII\r\n@r2\r\nA\r\n+\r\nI\r\n",
    "fasta_leading_junk": b"junk\n\n>x\nAC\n",
    "fastq_4line": b"@r1\nACGTN\n+\nIIIII\n@r2 c\nAC\n+r2\nII\n",
    "fastq_multiline": b"@r1\nACGT\nAC\n+\nIII\nIII\n@r2\nGG\n+\n@@\n@r3\nT\n+\nI\n",
    "fastq_truncated_qual": b"@r1\nACGT\n+\nIIII\n@r2\nACGT\n+\nII\n",
    "fastq_no_qual": b"@r1\nACGT\n+\nIIII\n@r2\nACGT\n+",
    "mixed_markers_inside_lines": b">a\nAC>GT@A+C\nGG\n>b\nT\n",
    "empty": b"",
    "only_header_char": b">",
    "no_trailing_newline": b">a\nACGT",
}


@pytest.fixture(scope="module")
def exe(tmp_path_factory):
    d = tmp_path_factory.mktemp("fastx")
    out = str(d / "fastx_check")
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-Wall", "-Wextra", "-DLPHASH_B200_WITH_ZLIB",
                           "-I", os.path.join(ROOT, "include"), SRC, "-o", out, "-lz", "-pthread"])
    return out


def run(exe, path, tmp, chunk=None):
    outp = os.path.join(tmp, "out.bin")
    subprocess.check_call([exe, path, outp] + ([str(chunk)] if chunk else []))
    raw = open(outp, "rb").read()
    n = int(np.frombuffer(raw, dtype="<u8", count=1)[0])
    off = np.frombuffer(raw, dtype="<u8", count=n + 1, offset=8)
    bases = raw[8 * (n + 2):]
    return [bases[int(off[i]):int(off[i + 1])] for i in range(n)]


@pytest.mark.parametrize("name", sorted(CASES))
def test_matches_kseq_grammar(exe, tmp_path, name):
    data = CASES[name]
    path = str(tmp_path / (name + ".txt"))
    open(path, "wb").write(data)
    assert run(exe, path, str(tmp_path)) == kseq_records(data)


@pytest.mark.parametrize("chunk", [16, 23, 64, 4096])
@pytest.mark.parametrize("name", sorted(CASES))
def test_streaming_ingest_matches_kseq_grammar(exe, tmp_path, name, chunk):
    """stream_file: the text arrives in chunks (a record straddling a chunk end is held back and re-parsed with the
    next chunk; a FASTQ quality string cut by the chunk is not mistaken for a malformed one)."""
    data = CASES[name]
    path = str(tmp_path / (name + ".txt"))
    open(path, "wb").write(data)
    assert run(exe, path, str(tmp_path), chunk) == kseq_records(data)


def test_gzip_and_large_random(exe, tmp_path):
    rng = np.random.Generator(np.random.PCG64(5))
    parts = []
    for i in range(3000):
        ln = int(rng.integers(0, 400))
        seq = bytes(rng.choice(np.frombuffer(b"ACGTNacgt", dtype=np.uint8), size=ln))
        if i % 3 == 0:  # multi-line FASTA, width 60
            parts.append(b">s%d\n" % i + b"\n".join(seq[j:j + 60] for j in range(0, ln, 60)) + b"\n")
        elif i % 3 == 1:
            parts.append(b">s%d x\n" % i + seq + b"\n")
        else:
            parts.append(b"@q%d\n" % i + seq + b"\n+\n" + b"I" * ln + b"\n")
    data = b"".join(parts)
    path = str(tmp_path / "big.fx.gz")
    with gzip.open(path, "wb") as f:
        f.write(data)
    got = run(exe, path, str(tmp_path))
    want = kseq_records(data)
    assert len(got) == len(want) == 3000
    assert got == want
    for chunk in (97, 1000, 65536):  # the same through the streaming ingest (gz inflated chunk by chunk)
        assert run(exe, path, str(tmp_path), chunk) == want


@pytest.mark.parametrize("name", ["fasta_multiline", "fasta_crlf", "fastq_4line"])
def test_matches_python_reader_on_plain_files(exe, tmp_path, name):
    """lphash_b200/seqio.py (what the Python tests and tools read files with) agrees on ordinary files."""
    from lphash_b200 import seqio
    path = str(tmp_path / (name + ".txt"))
    open(path, "wb").write(CASES[name])
    assert run(exe, path, str(tmp_path)) == seqio.read_records(path)


KSEQ_DUMP = r"""
#include <zlib.h>
#include <stdio.h>
#include <stdint.h>
#include "kseq.h"
KSEQ_INIT(gzFile, gzread)
int main(int argc, char** argv) {
    gzFile fp = gzopen(argv[1], "r");
    if (!fp) return 2;
    kseq_t* seq = kseq_init(fp);
    uint64_t n = 0, total = 0, h = 0xcbf29ce484222325ULL;
    while (kseq_read(seq) >= 0) {
        ++n;
        total += seq->seq.l;
        for (size_t i = 0; i < seq->seq.l; ++i) h = (h ^ (unsigned char)seq->seq.s[i]) * 0x100000001b3ULL;
        h = (h ^ 0xff) * 0x100000001b3ULL;  /* record separator */
    }
    printf("%llu %llu %llx\n", (unsigned long long)n, (unsigned long long)total, (unsigned long long)h);
    kseq_destroy(seq);
    gzclose(fp);
    return 0;
}
"""

# the reference's source tree, where one is at hand: its own kseq.h is then compiled and compared too
REF_DIR = os.environ.get("LPHASH_REF_DIR")


def fnv_records(recs) -> int:
    """the fold kseq_dump prints: every byte of every record, 0xff after each record"""
    fold = 0xCBF29CE484222325
    for r in recs:
        for b in r:
            fold = ((fold ^ b) * 0x100000001B3) & 0xFFFFFFFFFFFFFFFF
        fold = ((fold ^ 0xFF) * 0x100000001B3) & 0xFFFFFFFFFFFFFFFF
    return fold


@pytest.mark.parametrize("rel", ["data/queries/salmonella_enterica.fasta.gz", "data/queries/ecoli1.fasta.gz",
                                 "data/queries/SRR5833294.10K.fastq.gz", "data/unitigs_stitched/se.ust.k31.fa.gz"])
def test_matches_the_reference_kseq_on_its_bundled_data(exe, tmp_path, rel):
    """The reference's bundled files (copies in tests/golden/config1): the records kseq_read yields (the port above),
    in the numbers of records and bases the reference's answers in expected.json were computed on; and, where
    LPHASH_REF_DIR names the reference's source tree, the same (records, bases, fold) as its own kseq.h."""
    path = os.path.join(GOLDEN_DIR, "config1", os.path.basename(rel))
    recs = run(exe, path, str(tmp_path))
    assert recs == kseq_records(gzip.open(path).read())
    exp = {q["file"]: q for q in json.load(open(os.path.join(GOLDEN_DIR, "config1", "expected.json")))["queries"].values()}
    assert (len(recs), sum(len(r) for r in recs)) == (exp[os.path.basename(rel)]["records"],
                                                      exp[os.path.basename(rel)]["bases"])
    if REF_DIR:
        src = tmp_path / "kseq_dump.c"
        src.write_text(KSEQ_DUMP)
        dump = str(tmp_path / "kseq_dump")
        subprocess.check_call(["gcc", "-O2", "-I", os.path.join(REF_DIR, "external"), str(src), "-o", dump, "-lz"])
        n, total, h = subprocess.check_output([dump, path], text=True).split()
        assert (len(recs), sum(len(r) for r in recs), fnv_records(recs)) == (int(n), int(total), int(h, 16))


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["k31_m20_u64", "k63_m24_u128"])
def test_example_query_driver_end_to_end(tmp_path, name):
    """examples/lphb_query.cpp: file -> fastx parser -> lphb_query_stream -> fold of all codes; the query
    batch of a golden written as multi-line FASTA (records with non-ACGT bytes that are not line
    structure characters included), gzip-compressed."""
    from conftest import fnv_fold, load_golden
    g = load_golden(name)
    exe = str(tmp_path / "lphb_query")
    libdir = os.path.join(ROOT, "lphash_b200")
    subprocess.check_call(["g++", "-std=c++17", "-O2", "-DLPHASH_B200_WITH_ZLIB", "-I", os.path.join(ROOT, "include"),
                           os.path.join(ROOT, "examples", "lphb_query.cpp"), "-o", exe, "-L", libdir,
                           "-llphash_b200", f"-Wl,-rpath,{libdir}", "-lz", "-pthread"])
    keep, parts = [], []
    for i, c in enumerate(g.contigs()):
        if any(b in c for b in (b"\n", b"\r", b">", b"@", b"+", b"\0")):
            continue  # cannot be expressed as a FASTA sequence line
        keep.append(i)
        parts.append(b">c%d\n" % i + b"\n".join(c[j:j + 70] for j in range(0, len(c), 70)) + b"\n")
    path = str(tmp_path / "q.fa.gz")
    with gzip.open(path, "wb") as f:
        f.write(b"".join(parts))
    off = g.q_code_offsets
    want = np.concatenate([g.q_codes[int(off[i]):int(off[i + 1])] for i in keep])
    fold = fnv_fold(want)
    out = subprocess.check_output([exe, g.lph, str(g.bits), path], text=True).strip().split(",")
    assert int(out[2]) == len(want)
    assert int(out[5], 16) == fold
    # tiny chunks (many batches, records held back across chunk ends) and the run-length output form
    for extra in (["0", "0"], ["0", "1", "runs"]):
        out = subprocess.check_output([exe, g.lph, str(g.bits), path] + extra, text=True).strip().split(",")
        assert int(out[2]) == len(want) and int(out[5], 16) == fold, extra
