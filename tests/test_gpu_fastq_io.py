"""GPU suite: FASTQ ingest and annotated-FASTQ egress on the device (mp_fastq_upload / mp_format_fastq, csrc/mp_fastq.cu)
against the host loops they replace (the driver's kseq-style parser + appendToQueryArrays packing, QueryParser.cpp:160-260, and
its header_line / output_pair / output_unpaired formatter, BGS-IO.cpp:1348-1446, 1966-2091) and against the reference binary.
The device path is the default of bin/soap4 for plain FASTQ files with -F / -P; MP_HOST_IO=1 forces the host loops."""
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT, make_reads, canon_fastq, deinterleave, run_ref_raw, load_pairs

pytestmark = pytest.mark.gpu


def run_driver(workdir, prefix, fq1, fq2, name, lopt, ini, flags, env=None, threads=3):
    exe = os.path.join(ROOT, "megapath_b200", "bin", "soap4")
    cmd = [exe, "pair", prefix, fq1, fq2, "-o", os.path.join(workdir, name), "-C", os.path.join(ROOT, "megapath_b200", "ini", ini),
           "-L", str(lopt), "-T", str(threads), "-u", "750"] + list(flags)
    e = dict(os.environ)
    e.update(env or {})
    p = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.PIPE, timeout=300, env=e)
    assert p.returncode == 0, p.stderr.decode()[-2000:]
    return p.stdout, p.stderr.decode(errors="replace")


def first_diff(a, b):
    la, lb = a.split(b"\n"), b.split(b"\n")
    for i, (x, y) in enumerate(zip(la, lb)):
        if x != y:
            return i, x[:300], y[:300]
    return min(len(la), len(lb)), len(la), len(lb)


SETS = [
    ("clean", 150, 151, dict(model="clean"), "soap4.ini", ("-F", "-nc")),
    ("mixed", 100, 101, dict(model="divergent", one_random=0.10, unalignable=0.05), "soap4.ini", ("-F", "-nc")),
    ("var", 150, 151, dict(model="clean", varlen=True, n_rate=0.002, one_random=0.05), "soap4.ini", ("-F", "-nc")),
    ("nt2", 150, 151, dict(model="divergent", one_random=0.10, unalignable=0.02), "soap4-nt2.ini", ("-F", "-nc", "-top", "95")),
    ("pmode", 100, 101, dict(model="divergent", one_random=0.10, unalignable=0.05), "soap4.ini", ("-P", "-nc")),
    ("span", 150, 151, dict(model="clean", span_frac=0.05), "soap4.ini", ("-F", "-nc")),
    ("trunc", 150, 121, dict(model="clean", varlen=True), "soap4.ini", ("-F", "-nc")),       # reads longer than -L - 1 are cut
]


# every set as one batch; the sets with unplaced / rescued pairs and variable lengths also as several batches over the contexts
CASES = [(s, 0) for s in SETS] + [(s, 1024) for s in SETS if s[0] in ("mixed", "var", "nt2")]


@pytest.mark.parametrize("case", CASES, ids=["%s-%d" % (s[0], b) for s, b in CASES])
def test_device_io_is_byte_identical_to_host_io(workdir, small_ref, case):
    (name, rlen, lopt, kw, ini, flags), batch = case
    """Same process, same batches: stdout of the device loops == stdout of the host loops, byte for byte (single batch and
    several batches over two contexts; the stream order -- deep-DP pairs, rescued pairs, the rest -- included)."""
    fq1, fq2 = make_reads(workdir, small_ref, "dio_" + name, 3000, rlen, seed=91, **kw)
    env = {"MP_BATCH_READS": str(batch)} if batch else {}
    dev, err = run_driver(workdir, small_ref["prefix"], fq1, fq2, "dio_d_" + name, lopt, ini, flags, env)
    assert "formatting on the device" in err, err[-1500:]
    host, err2 = run_driver(workdir, small_ref["prefix"], fq1, fq2, "dio_h_" + name, lopt, ini, flags, dict(env, MP_HOST_IO="1"))
    assert "formatting on the host" in err2
    assert len(host) > 100000
    assert dev == host, first_diff(dev, host)


def _edit_comments(k, mate, comm, unsafe=False):
    if k % 19 == 3:
        return b"IGNORE"
    if k % 23 == 5 and mate == 1:
        return b"SCORE:0;"
    if k % 29 == 7:
        return b"SCORE:400;400,made_up_hit;"
    if k % 31 == 11 and mate == 0:
        return b""
    if k % 41 == 17:
        return b"SCORE:  +12;12,x y z;9,low;"          # blanks and a sign before the number, a name with blanks
    if k % 43 == 19:
        return b"SCORE:99999999999999999999;5,big;"    # strtol saturates, (int) of it is -1
    if unsafe and k % 37 == 13:
        return b"abc"                                  # shorter than "SCORE:": the reference reads past the string
    if unsafe and k % 47 == 23:
        return b"SCORE:30;30,a;9,low;junk"             # unterminated tail: the reference dereferences strchr's NULL
    return comm


@pytest.mark.parametrize("mode", ["-F", "-P"])
def test_device_io_chained_comments(workdir, small_ref, second_ref, mode):
    """Without -nc (every NT chunk after the first, runMegaPath.sh:199): previous SCORE: lists merged on the device ==
    host formatter == reference (canonical order), including IGNORE, signed, saturating and hand-made comments.  Comments the
    reference itself cannot read (it crashes on them) are compared between the device and the host formatter only."""
    fq1, fq2 = make_reads(workdir, small_ref, "dchain", 2500, 150, seed=78, model="divergent", one_random=0.10, unalignable=0.04)
    first = run_ref_raw(workdir, small_ref["prefix"], fq1, fq2, "dchain0", 151, "soap4-nt2.ini", ["-F", "-nc", "-top", "95"])
    flags = [mode, "-top", "95"]
    in1, in2 = deinterleave(first, os.path.join(workdir, "dchain_in"), _edit_comments)
    dev, err = run_driver(workdir, second_ref["prefix"], in1, in2, "dchain_d" + mode, 151, "soap4-nt2.ini", flags)
    assert "formatting on the device" in err
    host, _ = run_driver(workdir, second_ref["prefix"], in1, in2, "dchain_h" + mode, 151, "soap4-nt2.ini", flags, {"MP_HOST_IO": "1"})
    assert dev == host, first_diff(dev, host)
    want = canon_fastq(run_ref_raw(workdir, second_ref["prefix"], in1, in2, "dchain_r" + mode, 151, "soap4-nt2.ini", flags))
    assert want.count(b"IGNORE") > 100 and b"made_up_hit" in want
    got = canon_fastq(dev)
    assert got == want, first_diff(got, want)
    u1, u2 = deinterleave(first, os.path.join(workdir, "dchain_un"), lambda k, m, c: _edit_comments(k, m, c, unsafe=True))
    dev, _ = run_driver(workdir, second_ref["prefix"], u1, u2, "dchain_ud" + mode, 151, "soap4-nt2.ini", flags)
    host, _ = run_driver(workdir, second_ref["prefix"], u1, u2, "dchain_uh" + mode, 151, "soap4-nt2.ini", flags, {"MP_HOST_IO": "1"})
    assert dev == host, first_diff(dev, host)


def test_device_io_falls_back_on_anything_but_strict_fastq(workdir, small_ref):
    """CRLF line ends, multi-line records and a missing final newline are not for the kernels: the driver says so and the host
    parser takes the run -- same output as with MP_HOST_IO=1."""
    fq1, fq2 = make_reads(workdir, small_ref, "dfb", 600, 100, seed=5, model="clean")
    a, b = open(fq1, "rb").read(), open(fq2, "rb").read()
    want, _ = run_driver(workdir, small_ref["prefix"], fq1, fq2, "dfb_h", 101, "soap4.ini", ["-F", "-nc"], {"MP_HOST_IO": "1"})

    def wrapped(data):                                  # sequence and quality lines folded at 60 characters
        out = []
        lines = data.split(b"\n")
        for i in range(0, len(lines) - 3, 4):
            h, s, p, q = lines[i:i + 4]
            out += [h] + [s[k:k + 60] for k in range(0, len(s), 60)] + [p] + [q[k:k + 60] for k in range(0, len(q), 60)]
        return b"\n".join(out) + b"\n"
    variants = {"crlf": (a.replace(b"\n", b"\r\n"), b.replace(b"\n", b"\r\n")), "multi": (wrapped(a), wrapped(b)), "noeol": (a[:-1], b[:-1])}
    for tag, (x, y) in variants.items():
        p1, p2 = os.path.join(workdir, "dfb_%s_1.fq" % tag), os.path.join(workdir, "dfb_%s_2.fq" % tag)
        open(p1, "wb").write(x)
        open(p2, "wb").write(y)
        got, err = run_driver(workdir, small_ref["prefix"], p1, p2, "dfb_" + tag, 101, "soap4.ini", ["-F", "-nc"])
        assert "formatting on the host" in err, (tag, err[-800:])
        assert got == want, (tag, first_diff(got, want))


def test_fastq_upload_equals_batch_upload(workdir, small_ref):
    """Kernel seam: mp_fastq_upload leaves the batch exactly as the host packing + mp_batch_upload does -- same clamped lengths,
    same SeedPos arrays and candidates from the seeding stage -- for names with and without /1, comments, variable lengths,
    lower-case bases, N and reads longer than -L - 1."""
    import megapath_b200 as mp
    fq1, fq2 = make_reads(workdir, small_ref, "fqu", 1500, 150, seed=13, model="divergent", varlen=True, n_rate=0.004, one_random=0.05)

    def decorate(path, mate):
        lines = open(path, "rb").read().split(b"\n")
        for i in range(0, len(lines) - 3, 4):
            k = i // 4
            if k % 3 == 0:
                lines[i] = lines[i] + b" SCORE:12;12,abc;"
            elif k % 3 == 1:
                lines[i] = lines[i].split(b"/")[0]                      # no /<mate> suffix
            if k % 5 == 0:
                lines[i + 1] = lines[i + 1].lower()
        out = path.replace(".fq", "_d.fq")
        open(out, "wb").write(b"\n".join(lines))
        return out
    d1, d2 = decorate(fq1, 1), decorate(fq2, 2)
    for lopt in (151, 121):
        reads, lens = load_pairs(d1, d2, trunc=lopt - 1)
        P = mp.default_params(insert_low=1, insert_high=750, max_read_length=lopt)
        c = mp.Context(0)
        c.index_load(small_ref["prefix"])
        q, wpq = mp.pack_queries(reads, lens, lopt)
        c.batch_upload(q, lens, wpq)
        c.seed_pairs(P)
        rp, mpos = c.download_seedpos()
        cands = c.download_candidates()
        t1, t2 = open(d1, "rb").read(), open(d2, "rb").read()
        got_lens = c.fastq_upload(t1, t2, len(lens) // 2, lopt)
        assert np.array_equal(got_lens, lens)
        c.seed_pairs(P)
        rp2, mpos2 = c.download_seedpos()
        assert rp2.tobytes() == rp.tobytes() and mpos2.tobytes() == mpos.tobytes()
        assert c.download_candidates().tobytes() == cands.tobytes()
        # a record count other than the promised one, CR bytes and a broken record are refused, not guessed at
        with pytest.raises(mp.FastqFormatError):
            c.fastq_upload(t1, t2, len(lens) // 2 - 1, lopt)
        with pytest.raises(mp.FastqFormatError):
            c.fastq_upload(t1.replace(b"\n", b"\r\n", 1), t2, len(lens) // 2, lopt)
        with pytest.raises(mp.FastqFormatError):
            c.fastq_upload(t1.replace(b"\n+\n", b"\n-\n", 1), t2, len(lens) // 2, lopt)
        c.close()


def test_format_fastq_through_the_library(workdir, small_ref):
    """The C-ABI calls on their own (no driver): fastq_upload + align_pairs + format_fastq == bin/soap4 with the host loops."""
    import megapath_b200 as mp
    fq1, fq2 = make_reads(workdir, small_ref, "fql", 2000, 100, seed=21, model="divergent", one_random=0.10, unalignable=0.05)
    want, _ = run_driver(workdir, small_ref["prefix"], fq1, fq2, "fql_h", 101, "soap4.ini", ["-F", "-nc"], {"MP_HOST_IO": "1"})
    t1, t2 = open(fq1, "rb").read(), open(fq2, "rb").read()
    c = mp.Context(0)
    c.index_load(small_ref["prefix"])
    c.annotation_upload(small_ref["prefix"])
    lens = c.fastq_upload(t1, t2, 2000, 101)
    ilow = max(1, int(lens[0::2].max()), int(lens[1::2].max()))
    P = mp.default_params(insert_low=ilow, insert_high=750, max_read_length=101)
    c.align_pairs(P)
    got = c.format_fastq(top=0.95, mode=1, ignore_comments=True)
    assert got == want, first_diff(got, want)
    # a batch that came through mp_batch_upload has no text on the device: the call fails loudly
    reads, lens2 = load_pairs(fq1, fq2, trunc=100)
    q, wpq = mp.pack_queries(reads, lens2, 101)
    c.batch_upload(q, lens2, wpq)
    c.align_pairs(P)
    with pytest.raises(mp.MegapathError):
        c.format_fastq()
    c.close()


def test_device_io_on_two_gpus(workdir, small_ref):
    """-G 2: batches dealt to the contexts of two GPUs (staging buffers are page-locked once, for every device) print the stream
    one GPU prints."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    fq1, fq2 = make_reads(workdir, small_ref, "dio_g2", 4000, 100, seed=17, model="divergent", one_random=0.10, unalignable=0.05)
    env = {"MP_BATCH_READS": "1024"}
    one, _ = run_driver(workdir, small_ref["prefix"], fq1, fq2, "dio_g1", 101, "soap4.ini", ["-F", "-nc"], env)
    two, err = run_driver(workdir, small_ref["prefix"], fq1, fq2, "dio_g2", 101, "soap4.ini", ["-F", "-nc", "-G", "2"], env)
    assert "formatting on the device" in err
    assert two == one, first_diff(two, one)


def test_device_io_long_score_lists(workdir):
    """Eight near-identical sequences with long names: every read has a SCORE: list of several entries, far longer than the 64-byte
    slot k_fmt_measure composes header tails in, so k_fmt_write's in-place path (and the staging buffer's growth allowance) is what
    prints them.  Device == host formatter byte for byte, == reference after the canonical sort."""
    from conftest import build_index
    from tools import synth
    rng = np.random.default_rng(99)
    base = synth.ALPHA[rng.integers(0, 4, size=30000)]
    d = os.path.join(workdir, "copies")
    os.makedirs(d, exist_ok=True)
    fa = os.path.join(d, "copies.fa")
    seqs = []
    with open(fa, "wb") as f:
        for i in range(8):
            s = base.copy()
            m = rng.random(len(s)) < 0.004
            s[m] = synth.ALPHA[rng.integers(0, 4, size=int(m.sum()))]
            seqs.append(s)
            f.write(b">copy_%d_of_the_same_genome_with_a_long_description_line strain %d\n" % (i + 1, i) + s.tobytes() + b"\n")
    build_index(fa, "copies")
    seq = np.concatenate(seqs)
    bounds = np.arange(9, dtype=np.int64) * 30000
    r1, r2 = synth.make_pairs(seq, bounds, 1500, 100, 5, model="clean")
    p = os.path.join(d, "cp")
    synth.write_fastq(p + "_1.fq", r1, 1)
    synth.write_fastq(p + "_2.fq", r2, 2)
    flags = ["-F", "-nc", "-top", "95"]
    dev, err = run_driver(d, fa + ".index", p + "_1.fq", p + "_2.fq", "cp_d", 101, "soap4-nt2.ini", flags)
    assert "formatting on the device" in err
    host, _ = run_driver(d, fa + ".index", p + "_1.fq", p + "_2.fq", "cp_h", 101, "soap4-nt2.ini", flags, {"MP_HOST_IO": "1"})
    tails = [len(l.split(b"\t", 1)[1]) + 2 for l in host.split(b"\n")[0::4] if b"\t" in l]
    assert sum(t > 64 for t in tails) > 1000 and max(tails) > 300
    assert dev == host, first_diff(dev, host)
    want = canon_fastq(run_ref_raw(d, fa + ".index", p + "_1.fq", p + "_2.fq", "cp_r", 101, "soap4-nt2.ini", flags))
    got = canon_fastq(dev)
    assert got == want, first_diff(got, want)


@pytest.mark.parametrize("output_seq", ["0", "1"])
def test_device_io_lsam_mode(workdir, small_ref, output_seq):
    """-lsam: the device-made text, cut at pair boundaries and rewritten into fastq2lsam's lines by host threads, is byte-identical to
    the all-host path, over several batches and with more threads than pieces."""
    fq1, fq2 = make_reads(workdir, small_ref, "dio_lsam", 9000, 100, seed=8, model="divergent", one_random=0.10, unalignable=0.05)
    flags = ["-F", "-nc", "-top", "95", "-lsam", output_seq]
    for env in ({}, {"MP_BATCH_READS": "4096"}):
        dev, err = run_driver(workdir, small_ref["prefix"], fq1, fq2, "dio_ls_d", 101, "soap4-nt2.ini", flags, env, threads=5)
        assert "formatting on the device" in err
        host, _ = run_driver(workdir, small_ref["prefix"], fq1, fq2, "dio_ls_h", 101, "soap4-nt2.ini", flags, dict(env, MP_HOST_IO="1"), threads=5)
        assert dev.count(b"\n") == 18000 and dev.count(b"\t64\t") == 9000
        assert dev == host, first_diff(dev, host)


def test_device_io_mid_file_fallback(workdir, small_ref):
    """A file that stops being strict four-line FASTQ after the first batch: a CR inside a later batch sends that batch (only) through
    the host parser and formatter -- same stream as the all-host run; a folded record, which moves the batch boundaries the newline
    count promised, stops the run with a message instead of printing batches the reference would not have formed."""
    fq1, fq2 = make_reads(workdir, small_ref, "dio_mid", 3000, 100, seed=23, model="divergent", one_random=0.10, unalignable=0.05)
    env = {"MP_BATCH_READS": "1024"}
    a = open(fq1, "rb").read().split(b"\n")
    cr = list(a)
    cr[4 * 2000 + 1] += b"\r"                          # bases line of record 2000 (fourth batch of 512 pairs)
    cr[4 * 2000 + 3] += b"\r"
    p_cr = os.path.join(workdir, "dio_mid_cr_1.fq")
    open(p_cr, "wb").write(b"\n".join(cr))
    want, _ = run_driver(workdir, small_ref["prefix"], p_cr, fq2, "dio_mid_h", 101, "soap4.ini", ["-F", "-nc"], dict(env, MP_HOST_IO="1"))
    got, err = run_driver(workdir, small_ref["prefix"], p_cr, fq2, "dio_mid_d", 101, "soap4.ini", ["-F", "-nc"], env)
    assert "formatting on the device" in err
    assert got == want, first_diff(got, want)
    fold = list(a)
    s = fold[4 * 2000 + 1]
    fold[4 * 2000 + 1] = s[:50] + b"\n" + s[50:]       # one record of five lines: every later record boundary moves
    p_fold = os.path.join(workdir, "dio_mid_fold_1.fq")
    open(p_fold, "wb").write(b"\n".join(fold))
    exe = os.path.join(ROOT, "megapath_b200", "bin", "soap4")
    p = subprocess.run([exe, "pair", small_ref["prefix"], p_fold, fq2, "-o", os.path.join(workdir, "dio_mid_f"), "-C", os.path.join(ROOT, "megapath_b200", "ini", "soap4.ini"),
                        "-L", "101", "-T", "3", "-u", "750", "-F", "-nc"], stdout=subprocess.PIPE, stderr=subprocess.PIPE, timeout=300, env=dict(os.environ, **env))
    assert p.returncode != 0 and b"MP_HOST_IO=1" in p.stderr
