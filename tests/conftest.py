import glob
import hashlib
import json
import os
import shutil
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
REF_DIR = os.path.join(ROOT, "oracle", "_ref")
BIN_DIR = os.path.join(ROOT, "megapath_b200", "bin")
REFERENCE_DIGESTS = os.path.join(ROOT, "tests", "golden", "reference_digests.json")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


def have_ref():
    return os.path.exists(os.path.join(REF_DIR, "soap4_dump")) and os.path.exists(os.path.join(REF_DIR, "2bwt-builder"))


# ---- the reference's outputs without the reference ----
# The reference binaries (oracle/_ref) are built from the original project's sources, which are not part of this repository.  Where
# they are not built, each call below runs the project's drop-in instead (bin/soap4, bin/2bwt-builder, soap4_hosttest __lsam) on the
# same arguments and checks what it produced against a SHA-256 digest stored in tests/golden/reference_digests.json.  Where they are
# built, the reference's own output is hashed the same way and checked against the same digest, so that a stored digest that is not
# the reference's fails there.  Outputs whose order depends on worker threads are hashed in an order-free form: pairs sorted by name,
# lines sorted, BAM records sorted.  MP_RECORD_REFERENCE_DIGESTS=<file> writes the digests to <file> instead of checking them; run
# with oracle/_ref built, that records the reference's.
_digest_cache = {}


def check_reference_digest(key, data):
    got = hashlib.sha256(data).hexdigest()
    record = os.environ.get("MP_RECORD_REFERENCE_DIGESTS")
    if record:
        d = json.load(open(record)) if os.path.exists(record) else {}
        assert d.setdefault(key, got) == got, "%s: two different outputs recorded under one key" % key
        with open(record, "w") as f:
            json.dump(d, f, indent=0, sort_keys=True)
        return
    if not _digest_cache:
        _digest_cache.update(json.load(open(REFERENCE_DIGESTS)))
    assert key in _digest_cache, "no stored digest of the reference's output for %r" % key
    assert got == _digest_cache[key], "%s: output differs from the reference's (sha256 %s, stored %s)" % (key, got, _digest_cache[key])


def _files_digest(paths):
    h = []
    for p in paths:
        s = hashlib.sha256()
        with open(p, "rb") as f:
            for blk in iter(lambda: f.read(1 << 24), b""):
                s.update(blk)
        h.append(s.hexdigest().encode())
    return b"\n".join(h)


def _canon_stdout(data):
    return canon_fastq(data) if data[:1] == b"@" else b"\n".join(sorted(data.split(b"\n")))


def _bam_outputs(out_prefix):
    return [p for p in [out_prefix + ".dpout.1", out_prefix + ".unpair"] + sorted(glob.glob(out_prefix + ".gout.*")) if os.path.isfile(p)]


def check_soap4_digest(stdout, index_prefix, fq1, out_prefix, ini, args):
    """a soap4 run (stdout and the BAM records written under out_prefix) against the stored digest of the reference's"""
    parts = [_canon_stdout(stdout)]
    if _bam_outputs(out_prefix):
        hdr, recs = canon_bam(_bam_outputs(out_prefix))
        # records with the same name and mate in any order; the RG tag holds the path of the first FASTQ file
        parts.append(repr((hdr, sorted(recs))).encode().replace(fq1.encode(), b"<fq1>"))
    # -T (worker threads) changes no output in these forms, and tests pick it from the machine's core count
    key = [a for i, a in enumerate(args) if a != "-T" and (i == 0 or args[i - 1] != "-T")]
    check_reference_digest(" ".join(["soap4", os.path.basename(out_prefix), os.path.basename(index_prefix), ini] + key), b"\0".join(parts))


def _soap4_stand_in(index_prefix, fq1, fq2, out_prefix, ini, args, cwd):
    """bin/soap4 with the reference's command line -> stdout bytes, pinned to the reference's output (stdout and BAM records)."""
    cmd = [os.path.join(BIN_DIR, "soap4"), "pair", index_prefix, fq1, fq2, "-o", out_prefix, "-C", os.path.join(ROOT, "megapath_b200", "ini", ini)] + args
    p = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.PIPE, cwd=cwd, timeout=1800)
    if p.returncode != 0:
        raise RuntimeError("soap4 driver failed: " + p.stderr.decode(errors="replace")[-1500:])
    check_soap4_digest(p.stdout, index_prefix, fq1, out_prefix, ini, args)
    return p.stdout


def build_index(fa, key, mask=False):
    """2bwt-builder <fa> [-U] -> fa + ".index": the reference's builder, or bin/2bwt-builder (GPU) with its files pinned to the
    reference builder's under `key`."""
    d = os.path.dirname(fa)
    if have_ref():
        shutil.copy(os.path.join(REF_DIR, "2bwt-builder.ini"), os.path.join(d, "2bwt-builder.ini"))
        subprocess.check_call([os.path.join(REF_DIR, "2bwt-builder"), fa] + (["-U"] if mask else []), cwd=d,
                              stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
    else:
        subprocess.check_call([os.path.join(BIN_DIR, "2bwt-builder"), fa] + (["-U"] if mask else []), cwd=d, stdout=subprocess.DEVNULL)
    check_reference_digest("2bwt-builder " + key, _files_digest([fa + ".index." + e for e in ("pac", "bwt", "fmv", "sa", "lkt", "tra", "amb")]))
    return fa + ".index"


def run_ref_fastq2lsam(key, fastq, output_seq, workdir, ordered=True):
    """The reference's cc/fastq2lsam <output_seq> on `fastq` -> stdout bytes, or the -lsam rewriting of soap4_hosttest pinned to it.
    ordered=False: `fastq` comes in worker-thread order, so the digest is over sorted lines."""
    if os.path.exists(os.path.join(REF_DIR, "fastq2lsam")):
        out = subprocess.run([os.path.join(REF_DIR, "fastq2lsam"), output_seq], input=fastq, capture_output=True, check=True, timeout=600).stdout
    else:
        path = os.path.join(workdir, key + ".lsam_in.fq")
        with open(path, "wb") as f:
            f.write(fastq)
        out = subprocess.run([os.path.join(BIN_DIR, "soap4_hosttest"), "__lsam", path, output_seq], capture_output=True, check=True, timeout=600).stdout
    check_reference_digest("fastq2lsam %s %s" % (key, output_seq), out if ordered else _canon_stdout(out))
    return out


def run_ref_soap4(workdir, index_prefix, fq1, fq2, out_name, max_len_opt, dump=True, ini="soap4.ini", threads=2, extra=()):
    """Runs the reference binary (instrumented variant) and returns (stdout_path, dump_dir).  Without the reference no seam dumps
    are written (dump_dir stays empty)."""
    dump_dir = os.path.join(workdir, out_name + ".dump")
    if os.path.isdir(dump_dir):
        shutil.rmtree(dump_dir)
    os.makedirs(dump_dir)
    env = dict(os.environ)
    if dump:
        env["MPH_DUMP_DIR"] = dump_dir
    out_fq = os.path.join(workdir, out_name + ".fq")
    args = ["-L", str(max_len_opt), "-T", str(threads), "-u", "750", "-F", "-nc"] + list(extra)
    if not have_ref():
        with open(out_fq, "wb") as fo:
            fo.write(_soap4_stand_in(index_prefix, fq1, fq2, os.path.join(workdir, out_name), ini, args, workdir))
        return out_fq, dump_dir
    cmd = [os.path.join(REF_DIR, "soap4_dump" if dump else "soap4"), "pair", index_prefix, fq1, fq2, "-o", os.path.join(workdir, out_name),
           "-C", os.path.join(REF_DIR, ini)] + args
    with open(out_fq, "wb") as fo, open(os.path.join(workdir, out_name + ".err"), "wb") as fe:
        subprocess.check_call(cmd, stdout=fo, stderr=fe, env=env, cwd=workdir)
    check_soap4_digest(open(out_fq, "rb").read(), index_prefix, fq1, os.path.join(workdir, out_name), ini, args)
    return out_fq, dump_dir


def need_index_builder():
    """Skips the calling test where no 2bwt-builder can run: bin/2bwt-builder builds on the GPU."""
    if not have_ref():
        import torch
        if not torch.cuda.is_available():
            pytest.skip("the test index needs a GPU (bin/2bwt-builder) or the reference's builder (oracle/_ref)")


@pytest.fixture(scope="session")
def workdir(tmp_path_factory):
    return str(tmp_path_factory.mktemp("mp"))


@pytest.fixture(scope="session")
def small_ref(workdir):
    """300 kbp, 6 sequences, with a few planted repeats; index written by 2bwt-builder (build_index)."""
    need_index_builder()
    from tools import synth
    fa = os.path.join(workdir, "ref.fa")
    seq, bounds = synth.make_ref(300000, 6, seed=42, repeat_frac=0.05)
    synth.write_fasta(fa, seq, bounds)
    return dict(fasta=fa, prefix=build_index(fa, "small_ref"), seq=seq, bounds=bounds)


@pytest.fixture(scope="session")
def second_ref(workdir, small_ref):
    """A second index for the NT-chunk chaining tests (runMegaPath.sh:184-226): three quarters of its sequences are diverged
    copies (1-3 % substitutions) of sequences of `small_ref`, the rest is unrelated, so that reads placed on `small_ref` hit it
    with scores above, equal to and below their first-chunk scores."""
    from tools import synth
    rng = np.random.default_rng(1234)
    seq, bounds = small_ref["seq"], small_ref["bounds"]
    parts = []
    for i in range(len(bounds) - 1):
        s = seq[bounds[i]:bounds[i + 1]].copy()
        if i % 4 == 3:
            s = synth.ALPHA[rng.integers(0, 4, size=len(s))]
        else:
            rate = (0.0, 0.01, 0.03)[i % 3]
            m = rng.random(len(s)) < rate
            s[m] = synth.ALPHA[rng.integers(0, 4, size=int(m.sum()))]
        parts.append(s)
    seq2 = np.concatenate(parts[::-1])
    b2 = np.concatenate([[0], np.cumsum([len(x) for x in parts[::-1]])]).astype(np.int64)
    d = os.path.join(workdir, "second")
    os.makedirs(d, exist_ok=True)
    fa = os.path.join(d, "ref2.fa")
    with open(fa, "wb") as f:
        for i in range(len(b2) - 1):
            f.write(b">chunk1_%d second index\n" % (i + 1) + seq2[b2[i]:b2[i + 1]].tobytes() + b"\n")
    return dict(fasta=fa, prefix=build_index(fa, "second_ref"), seq=seq2, bounds=b2)


def deinterleave(stdout_fastq, prefix, comment_edit=None):
    """cc/deinterleave.cpp in a few lines: the interleaved `soap4 -F` output -> <prefix>_1.fq / <prefix>_2.fq with the comment
    kept (kseq: name up to the first white space, comment after it; written back as "@name/<mate> comment").
    comment_edit(pair_index, mate, comment) may rewrite a comment (IGNORE / hand-made cases); pairs are taken in canonical order, so
    that the same pairs get the same edits whatever order the worker threads printed them in."""
    lines = canon_fastq(stdout_fastq).split(b"\n")
    recs = [lines[i:i + 4] for i in range(0, len(lines) - 3, 4)]
    out = [open(prefix + "_1.fq", "wb"), open(prefix + "_2.fq", "wb")]
    for k in range(0, len(recs) - 1, 2):
        for mate in (0, 1):
            hdr, sq, _, ql = recs[k + mate]
            parts = hdr[1:].split(None, 1)
            name, comm = parts[0], (parts[1] if len(parts) > 1 else b"")
            if name.endswith(b"/1") or name.endswith(b"/2"):
                name = name[:-2]
            if comment_edit:
                comm = comment_edit(k // 2, mate, comm)
            out[mate].write(b"@" + name + b"/%d" % (mate + 1) + (b" " + comm if comm else b"") + b"\n" + sq + b"\n+\n" + ql + b"\n")
    for f in out:
        f.close()
    return prefix + "_1.fq", prefix + "_2.fq"


def run_ref_raw(workdir, index_prefix, fq1, fq2, out_name, max_len_opt, ini, flags, threads=3, insert_high=750):
    """The reference binary with exactly `flags` (no implied -F / -nc) -> stdout bytes."""
    args = ["-L", str(max_len_opt), "-T", str(threads), "-u", str(insert_high)] + list(flags)
    if not have_ref():
        return _soap4_stand_in(index_prefix, fq1, fq2, os.path.join(workdir, out_name), ini, args, workdir)
    cmd = [os.path.join(REF_DIR, "soap4"), "pair", index_prefix, fq1, fq2, "-o", os.path.join(workdir, out_name),
           "-C", os.path.join(REF_DIR, ini)] + args
    p = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.PIPE, cwd=workdir, timeout=600)
    if p.returncode != 0:
        raise RuntimeError("reference soap4 failed: " + p.stderr.decode(errors="replace")[-1500:])
    check_soap4_digest(p.stdout, index_prefix, fq1, os.path.join(workdir, out_name), ini, args)
    return p.stdout


def make_reads(workdir, small_ref, name, pairs, rlen, seed, **kw):
    from tools import synth
    r1, r2 = synth.make_pairs(small_ref["seq"], small_ref["bounds"], pairs, rlen, seed, **kw)
    p = os.path.join(workdir, name)
    synth.write_fastq(p + "_1.fq", r1, 1)
    synth.write_fastq(p + "_2.fq", r2, 2)
    return p + "_1.fq", p + "_2.fq"


def load_pairs(fq1, fq2, trunc):
    from oracle import pyoracle as po
    a, la = po.read_fastq_codes(fq1, trunc=trunc)
    b, lb = po.read_fastq_codes(fq2, trunc=trunc)
    n = len(la)
    w = max(a.shape[1], b.shape[1])
    reads = np.zeros((2 * n, w), dtype=np.uint8)
    reads[0::2, :a.shape[1]] = a
    reads[1::2, :b.shape[1]] = b
    lens = np.zeros(2 * n, dtype=np.uint32)
    lens[0::2] = la
    lens[1::2] = lb
    return reads, lens


def canon_fastq(data):
    """Canonical form of the interleaved stdout FASTQ (SURVEY.md 0.8): pairs (mate 1 and mate 2 are written
    adjacently) sorted by read name; worker threads of the reference emit pairs in arbitrary order."""
    lines = data.split(b"\n")
    recs = [b"\n".join(lines[i:i + 4]) for i in range(0, len(lines) - 3, 4)]
    pairs = [(recs[i], recs[i + 1]) for i in range(0, len(recs) - 1, 2)]
    pairs.sort(key=lambda p: p[0].split(b"\t")[0])
    return b"\n".join(a + b"\n" + b for a, b in pairs) + b"\n"


def run_our_soap4(workdir, index_prefix, fq1, fq2, out_name, max_len_opt, ini="soap4.ini", extra=("-F", "-nc"), insert_high=750):
    """Runs the product's host driver (megapath_b200/bin/soap4) -> stdout bytes."""
    exe = os.path.join(ROOT, "megapath_b200", "bin", "soap4")
    ini_path = os.path.join(ROOT, "megapath_b200", "ini", ini)
    cmd = [exe, "pair", index_prefix, fq1, fq2, "-o", os.path.join(workdir, out_name), "-C", ini_path, "-L", str(max_len_opt),
           "-T", "2", "-u", str(insert_high)] + list(extra)
    p = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.PIPE, timeout=300)
    if p.returncode != 0:
        raise RuntimeError("soap4 driver failed: " + p.stderr.decode()[-2000:])
    return p.stdout


def read_bam(path):
    """Minimal BAM decoder (BGZF members are gzip members) -> (target names, target lengths, records).
    A record is a tuple of every field the reference writes: qname, flag, tid, pos, mapq, cigar, mtid, mpos, isize,
    seq, qual and the raw aux bytes."""
    import gzip
    import struct
    data = gzip.open(path, "rb").read()
    assert data[:4] == b"BAM\x01"
    l_text, = struct.unpack_from("<i", data, 4)
    o = 8 + l_text
    n_ref, = struct.unpack_from("<i", data, o)
    o += 4
    names, lens = [], []
    for _ in range(n_ref):
        ln, = struct.unpack_from("<i", data, o)
        names.append(data[o + 4:o + 4 + ln - 1].decode())
        lens.append(struct.unpack_from("<i", data, o + 4 + ln)[0])
        o += 8 + ln
    recs = []
    while o < len(data):
        bs, tid, pos, bmn, fnc, lseq, mtid, mpos, isize = struct.unpack_from("<iiiIIiiii", data, o)
        body = data[o + 36:o + 4 + bs]
        l_qname, mapq, nb = bmn & 0xff, (bmn >> 8) & 0xff, bmn >> 16
        flag, ncig = fnc >> 16, fnc & 0xffff
        qname = body[:l_qname - 1]
        p = l_qname
        cig = struct.unpack_from("<%dI" % ncig, body, p)
        p += 4 * ncig
        cigar = "".join("%d%s" % (c >> 4, "MIDNSHP=X"[c & 15]) for c in cig)
        seq = body[p:p + (lseq + 1) // 2]
        p += (lseq + 1) // 2
        qual = body[p:p + lseq]
        p += lseq
        recs.append((qname, flag, tid, pos, mapq, cigar, mtid, mpos, isize, nb, bytes(seq), bytes(qual), bytes(body[p:])))
        o += 4 + bs
    return names, lens, recs


def canon_bam(paths):
    out = []
    hdr = None
    for p in paths:
        names, lens, recs = read_bam(p)
        hdr = (names, lens)
        out.extend(recs)
    out.sort(key=lambda r: (r[0], r[1] & 0xC0))
    return hdr, out
