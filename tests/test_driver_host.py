"""Host-side logic of the soap4 driver that needs no GPU: the zero-copy FASTQ fast path must see exactly the records the
kseq-style parser sees (the reference reads its input with kseq, soap4/kseq.h via QueryParser.cpp)."""
import gzip
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EXE = os.path.join(ROOT, "megapath_b200", "bin", "soap4_hosttest")      # the driver built with -DMP_TEST_HOOKS

pytestmark = pytest.mark.skipif(not os.path.exists(EXE), reason="driver binary not built (run __graft_entry__.build())")


def parse(path, generic):
    return subprocess.run([EXE, "__parse", path] + (["generic"] if generic else []), capture_output=True, check=True, timeout=120).stdout


CASES = {
    "plain": b"@r1/1\nACGT\n+\nIIII\n@r2/1 extra words\nGGCA\n+r2\nII#I\n",
    "crlf": b"@r1\r\nACGT\r\n+\r\nIIII\r\n@r2 c\r\nAC\r\n+\r\nII\r\n",
    "no_final_newline": b"@r1\nACGT\n+\nIIII\n@r2\nAC\n+\nII",
    "blank_lines": b"\n\n@r1\nACGT\n+\nIIII\n\n@r2\nAC\n+\nII\n\n",
    "multiline": b"@r1\nACGT\nACGT\n+\nIIII\nIIII\n@r2\nAC\n+\nII\n",
    "at_in_quality": b"@r1\nACGT\n+\n@III\n@r2\nACGA\n+\n@@@@\n@r3\nAC\n+\nI@\n",
    "qual_too_long": b"@r1\nACGT\n+\nIIIII\n@r2\nAC\n+\nII\n",
    "qual_short_continues": b"@r1\nACGT\n+\nII\nII\n@r2\nAC\n+\nII\n",
    "fasta": b">s1 desc\nACGTAC\nGT\n>s2\nAAA\n",
    "tabs": b"@r1\tSCORE:10;5,chr1;\nACGT\n+\nIIII\n@r2 \nAC\n+\nII\n",
    "empty": b"",
    "garbage_prefix": b"junk\n@r1\nAC\n+\nII\n",
}


@pytest.mark.parametrize("name", sorted(CASES))
def test_fast_path_equals_generic(tmp_path, name):
    p = tmp_path / (name + ".fq")
    p.write_bytes(CASES[name])
    assert parse(str(p), False) == parse(str(p), True)


def test_fast_path_large_and_gz(tmp_path):
    """records straddling the 4 MiB buffer boundary, plain and gzip"""
    rng = np.random.default_rng(5)
    recs = []
    for i in range(60000):
        L = int(rng.integers(30, 152))
        seq = bytes(rng.choice(np.frombuffer(b"ACGTN", dtype=np.uint8), L).tolist())
        qual = bytes(rng.integers(33, 74, L).astype(np.uint8).tolist())
        recs.append(b"@read%d/1%s\n%s\n+\n%s\n" % (i, b" c:%d" % i if i % 7 == 0 else b"", seq, qual))
    data = b"".join(recs)
    p = tmp_path / "big.fq"
    p.write_bytes(data)
    want = parse(str(p), True)
    assert want.count(b"\n") == 60000
    assert parse(str(p), False) == want
    g = tmp_path / "big.fq.gz"
    with gzip.open(g, "wb", compresslevel=1) as f:
        f.write(data)
    assert parse(str(g), False) == want


@pytest.mark.parametrize("size", [0, 5, 70000, 1 << 20])
def test_bgzf_chunks_concatenate_to_a_valid_stream(tmp_path, size):
    """BAM records are compressed into BGZF blocks by the formatting threads, chunk by chunk; the concatenation (after the
    buffered header bytes, before the EOF block) must decompress to the original bytes and every block must be a proper BGZF member"""
    rng = np.random.default_rng(size)
    data = bytes(rng.integers(0, 7, size).astype(np.uint8).tolist())
    src, dst = tmp_path / "in.bin", tmp_path / "out.bgzf"
    src.write_bytes(data)
    subprocess.run([EXE, "__bgzf", str(src), str(dst)], check=True, timeout=120)
    raw = dst.read_bytes()
    assert gzip.decompress(raw) == data
    # walk the members: gzip magic, FEXTRA with the BC subfield, BSIZE consistent, ISIZE <= 0xff00; the last one is the 28-byte EOF marker
    at, members = 0, 0
    while at < len(raw):
        assert raw[at:at + 4] == b"\x1f\x8b\x08\x04" and raw[at + 12:at + 16] == b"BC\x02\x00"
        bsize = int.from_bytes(raw[at + 16:at + 18], "little") + 1
        isize = int.from_bytes(raw[at + bsize - 4:at + bsize], "little")
        assert isize <= 0xff00
        at += bsize
        members += 1
    assert at == len(raw) and raw[-28:] == bytes.fromhex("1f8b08040000000000ff0600424302001b0003000000000000000000")
    assert members >= 2 if size else members == 1


@pytest.mark.parametrize("threads", [1, 3, 8])
def test_batch_loader_layout(tmp_path, threads):
    """The driver's batch loader (two parser threads writing mate-major storage, packer threads following them) must produce
    the buffers appendToQueryArrays would (QueryParser.cpp:184-203; megapath_b200.pack_queries is the host mirror the GPU
    tests feed the library with): read lengths truncated to maxReadLength-1, N -> 2, lower case, names without /1 /2,
    comments, qualities cut to the kept length, and a last partial group of 32."""
    import megapath_b200 as mp
    rng = np.random.default_rng(threads)
    npairs, maxlen = 1000 + 13, 101
    lut = np.zeros(256, np.uint8)
    for ch, v in zip(b"ACGTNacgtn", [0, 1, 2, 3, 2, 0, 1, 2, 3, 2]):
        lut[ch] = v
    recs = {1: [], 2: []}
    want_codes = np.zeros((2 * npairs, maxlen - 1), np.uint8)
    want_lens = np.zeros(2 * npairs, np.uint32)
    meta = []
    for p in range(npairs):
        for mate in (1, 2):
            L = int(rng.integers(20, 131))
            seq = bytes(rng.choice(np.frombuffer(b"ACGTNacgt", dtype=np.uint8), L).tolist())
            qual = bytes(rng.integers(33, 74, L).astype(np.uint8).tolist()).replace(b"@", b"A")
            comment = b"SCORE:7;3,chr1;" if p % 11 == 0 else b""
            recs[mate].append(b"@r%d/%d%s\n%s\n+\n%s\n" % (p, mate, (b" " + comment) if comment else b"", seq, qual))
            rid = 2 * p + mate - 1
            keep = min(L, maxlen - 1)
            want_codes[rid, :keep] = lut[np.frombuffer(seq[:keep], dtype=np.uint8)]
            want_lens[rid] = keep
            meta.append(b"r%d|%s|%s" % (p, comment, qual[:keep]))
    f1, f2, out = tmp_path / "a_1.fq", tmp_path / "a_2.fq", tmp_path / "pack.bin"
    f1.write_bytes(b"".join(recs[1])); f2.write_bytes(b"".join(recs[2]))
    subprocess.run([EXE, "__pack", str(f1), str(f2), str(maxlen), str(out), str(threads)], check=True, timeout=120)
    raw = out.read_bytes()
    n, wpq = np.frombuffer(raw[:8], dtype=np.uint32)
    assert n == 2 * npairs
    lens = np.frombuffer(raw[8:8 + 4 * n], dtype=np.uint32)
    assert (lens == want_lens).all()
    nwords = (n + 31) // 32 * 32 * wpq
    words = np.frombuffer(raw[8 + 4 * n:8 + 4 * n + 4 * nwords], dtype=np.uint32)
    want_words, want_wpq = mp.pack_queries(want_codes, want_lens, maxlen)
    assert wpq == want_wpq and (words == want_words).all()
    assert raw[8 + 4 * n + 4 * nwords:].split(b"\n")[:-1] == meta


LSAM_CASES = (b"@r1\tSCORE:50;50,seqA;48,seqB,seqC;\nACGT\n+\nIIII\n@r1\tIGNORE\nAC\n+\nII\n"
              b"@r2\tSCORE:0;\nA\n+\nI\n@r2\tSCORE:7;7,x;\nAA\n+\nII\n"
              b"@lone\tSCORE:31;31,only one;\nACG\n+\nIII\n"                      # a name that never pairs up
              b"@p/1\tSCORE:99;99,a;;95,b;\nACGT\n+\nIIII\n@p/2\tSCORE:99;99,a,,c;\nACGT\n+\nIIII\n"      # /1 /2 trimmed; empty fields
              b"@q\tSCORE:12;12,gi|1|ref|NC_1.1|;12,z\nAC\n+\nII\n@q\tSCORE:-3;5,w;\nAC\n+\nII\n"
              b"@tail\tSCORE:40;40,t;\nA\n+\nI\n")


@pytest.mark.parametrize("output_seq", ["1", "0"])
def test_lsam_mode_matches_reference_fastq2lsam(tmp_path, output_seq):
    """-lsam (the fused fastq2lsam step) prints what the reference's own cc/fastq2lsam prints for the same annotated FASTQ"""
    from conftest import run_ref_fastq2lsam
    f = tmp_path / "a.fq"
    f.write_bytes(LSAM_CASES)
    want = run_ref_fastq2lsam("cases", LSAM_CASES, output_seq, str(tmp_path))
    got = subprocess.run([EXE, "__lsam", str(f), output_seq], capture_output=True, check=True, timeout=60).stdout
    assert want.count(b"\n") == 10
    assert got == want


def _pack(f1, f2, maxlen, out, threads, env=None):
    subprocess.run([EXE, "__pack", str(f1), str(f2), str(maxlen), str(out), str(threads)], check=True, timeout=300,
                   env=dict(os.environ, **(env or {})))
    return open(out, "rb").read()


@pytest.mark.parametrize("kind", ["plain", "crlf", "multiline", "no_final_newline", "qual_mismatch_late"])
def test_parallel_mapped_parser_equals_sequential(tmp_path, kind):
    """Plain files are memory-mapped and a batch is parsed by several threads after its record boundaries have been located by
    counting newlines (parse_mapped); anything that is not strict four-line FASTQ makes the batch fall back to the sequential
    parser.  Either way the loader must hand over exactly what the sequential gz-style reader (MP_NO_MMAP=1) hands over."""
    rng = np.random.default_rng(len(kind))
    npairs = 9000
    nl = b"\r\n" if kind == "crlf" else b"\n"
    recs = {1: [], 2: []}
    for p in range(npairs):
        for mate in (1, 2):
            L = int(rng.integers(25, 140))
            seq = bytes(rng.choice(np.frombuffer(b"ACGTNacgt", dtype=np.uint8), L).tolist())
            qual = bytes(rng.integers(33, 74, L).astype(np.uint8).tolist())         # '@' and '+' appear at line starts
            comment = b" SCORE:9;4,chrZ;" if p % 5 == 0 else b""
            if kind == "multiline" and p % 1000 == 999:
                h = L // 2
                recs[mate].append(b"@q%d/%d%s" % (p, mate, comment) + nl + seq[:h] + nl + seq[h:] + nl + b"+" + nl + qual[:h] + nl + qual[h:] + nl)
            elif kind == "qual_mismatch_late" and p == npairs - 3 and mate == 2:
                recs[mate].append(b"@q%d/%d" % (p, mate) + nl + seq + nl + b"+" + nl + qual + b"I" + nl)    # refused by both readers the same way?
            else:
                recs[mate].append(b"@q%d/%d%s" % (p, mate, comment) + nl + seq + nl + b"+" + nl + qual + nl)
    d1, d2 = b"".join(recs[1]), b"".join(recs[2])
    if kind == "no_final_newline":
        d1, d2 = d1[:-1], d2[:-1]
    f1, f2 = tmp_path / "p_1.fq", tmp_path / "p_2.fq"
    f1.write_bytes(d1); f2.write_bytes(d2)
    if kind == "qual_mismatch_late":
        # a quality string longer than its sequence is an input error in either mode (kseq returns -2): both must fail, not diverge
        a = subprocess.run([EXE, "__pack", str(f1), str(f2), "131", str(tmp_path / "a.bin"), "6"], capture_output=True, timeout=300)
        b = subprocess.run([EXE, "__pack", str(f1), str(f2), "131", str(tmp_path / "b.bin"), "6"], capture_output=True, timeout=300, env=dict(os.environ, MP_NO_MMAP="1"))
        assert a.returncode == b.returncode
        if a.returncode == 0:
            assert open(tmp_path / "a.bin", "rb").read() == open(tmp_path / "b.bin", "rb").read()
        return
    got = _pack(f1, f2, 131, tmp_path / "a.bin", 6)
    want = _pack(f1, f2, 131, tmp_path / "b.bin", 6, {"MP_NO_MMAP": "1"})
    assert np.frombuffer(want[:4], dtype=np.uint32)[0] == 2 * npairs
    assert got == want


# ---- device ingest: the staging step that hands mp_fastq_upload the exact byte range of a batch.  The exact location and the fused
#      copy + count take the same block-wise newline index with different block counters; both must name the same bytes ----
def _stage(path, max_rec, threads, bpr=None):
    out = subprocess.run([EXE, "__stage", str(path), str(max_rec), str(threads)] + ([str(bpr)] if bpr else []), capture_output=True, check=True, timeout=120).stdout
    return [tuple(int(x) for x in l.split()) for l in out.decode().splitlines()]


@pytest.mark.parametrize("max_rec,threads", [(1000, 1), (1000, 5), (4096, 3), (100000, 4)])
def test_staging_names_the_byte_range_of_every_batch(tmp_path, max_rec, threads):
    """Variable-length records (names that grow, reads of 30 - 250 bases, comments): every batch is exactly max_rec records (the
    reference's batch size decides the order of stdout), located by block-wise newline counts with any number of threads; the fused
    copy + count pass finds the same range and copies it faithfully, or asks for the exact path (-2) when its estimate is too small."""
    rng = np.random.default_rng(max_rec + threads)
    n = 23456
    lens = rng.integers(30, 251, size=n)
    recs = [b"@read%d/1%s\n%s\n+\n%s\n" % (i, b" SCORE:5;5,x;" if i % 7 == 0 else b"", b"ACGT"[i % 4:i % 4 + 1] * int(lens[i]), b"I" * int(lens[i])) for i in range(n)]
    p = tmp_path / "v.fq"
    p.write_bytes(b"".join(recs))
    ends = np.cumsum([len(r) for r in recs])
    rows = _stage(p, max_rec, threads)
    pos, k = 0, 0
    for (nloc, newpos, nst, nbytes, same) in rows[:-1]:
        want = min(max_rec, n - k)
        assert nloc == want and newpos == ends[k + want - 1]
        assert nst == -2 or (nst == want and nbytes == newpos - pos and same == 1)
        pos, k = newpos, k + want
    assert k == n and rows[-1][0] == 0 and rows[-1][2] == 0
    assert sum(1 for r in rows[:-1] if r[2] > 0) >= len(rows) // 2          # the estimate holds for most batches


def test_staging_with_a_bad_estimate_asks_for_the_exact_path(tmp_path):
    recs = [b"@r%d\n%s\n+\n%s\n" % (i, b"A" * 200, b"I" * 200) for i in range(5000)]
    p = tmp_path / "w.fq"
    p.write_bytes(b"".join(recs))
    rows = _stage(p, 4000, 3, bpr=40.0)             # five times too small: the window cannot hold 4000 records within its capacity
    assert rows[0][0] == 4000 and rows[0][2] == -2


@pytest.mark.parametrize("name", ["no_final_newline", "multiline", "garbage_prefix", "fasta", "qual_short_continues"])
def test_staging_refuses_what_the_kernels_cannot_index(tmp_path, name):
    """Files that are not plain four-line FASTQ from their first record on never reach the device path (-1); CRLF files pass the
    newline count and are refused by k_fq_count on the device (tests/test_gpu_fastq_io.py)."""
    p = tmp_path / (name + ".fq")
    p.write_bytes(CASES[name])
    rows = _stage(p, 10, 2)
    assert rows[0][0] == -1 and rows[0][2] == -1


@pytest.mark.parametrize("output_seq,threads", [("1", 1), ("0", 1), ("1", 5), ("0", 5)], ids=["1", "0", "1-5threads", "0-5threads"])
def test_lsam_mode_randomized_against_reference_fastq2lsam(tmp_path, output_seq, threads):
    """20 000 records with generated comments -- IGNORE, zero / negative / signed scores, lists with several accessions per score, empty
    fields, long scores with dozens of one-letter accessions (the list outgrows twice the comment), names with and without /1 /2,
    unpaired names -- through -lsam and through the reference's own cc/fastq2lsam.  Records come two by two (a pair, or two unpaired
    names), so with several threads the text is cut every eighth line as the driver cuts a batch, and the pieces join to the same lines."""
    from conftest import run_ref_fastq2lsam
    rng = np.random.default_rng(int(output_seq) + 5)
    out = []
    for i in range(10000):
        paired = rng.random() < 0.9
        for m in (1, 2):
            kind = int(rng.integers(0, 8))
            sc = int(rng.integers(1, 400))
            if kind == 0:
                c = b"IGNORE"
            elif kind == 1:
                c = b"SCORE:0;"
            elif kind == 2:
                c = b"SCORE:-%d;7,x;" % sc
            elif kind == 3:
                c = b"SCORE: +%d;%d,acc%d;" % (sc, sc, i)
            elif kind == 4:
                c = b"SCORE:%d;%d,a%d,b%d,,c;;%d,z;" % (sc, sc, i, i, sc - 1)
            elif kind == 5:
                c = b"SCORE:%d;1234567890123,%s;" % (sc, b",".join(b"q" for _ in range(int(rng.integers(1, 60)))))
            elif kind == 6:
                c = b"SCORE:%d;%d,gi|%d|ref|NC_%d.1| some description, with a comma" % (sc, sc, i, i)
            else:
                c = b"SCORE:%d;" % sc
            name = b"r%d" % i if paired else b"r%d_%d" % (i, m)
            if rng.random() < 0.5:
                name += b"/%d" % m
            L = int(rng.integers(1, 120))
            out.append(b"@" + name + b"\t" + c + b"\n" + b"ACGT"[m:m + 1] * L + b"\n+\n" + b"I" * L + b"\n")
    f = tmp_path / "r.fq"
    f.write_bytes(b"".join(out))
    want = run_ref_fastq2lsam("randomized", b"".join(out), output_seq, str(tmp_path))
    got = subprocess.run([EXE, "__lsam", str(f), output_seq, str(threads)], capture_output=True, check=True, timeout=120).stdout
    assert want.count(b"\n") == 20000 and want.count(b"\t64\t") > 8000 and want.count(b"\t0\t") > 1000
    assert got == want
