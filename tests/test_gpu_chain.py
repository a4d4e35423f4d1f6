"""GPU suite for soap4 -chain: one process runs a batch through every chunk index of an NT chunk chain (runMegaPath.sh:184-226) and
must print what the last step of `soap4 idx0 ... -nc | deinterleave | soap4 idx1 ... | deinterleave | soap4 idx2 ...` prints.  The
composition is our own binary run once per chunk, with the conftest deinterleave rule (order kept) between the runs; one step of it
is pinned to the reference in test_gpu_fastq_io.py / test_gpu_e2e.py.  Also the three library entry points behind it:
mp_index_bind, mp_fastq_chain and mp_index_load_budget."""
import gzip
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT, BIN_DIR, make_reads, read_bam, load_pairs
from test_chain_host import deinterleave_ordered

pytestmark = pytest.mark.gpu
INI = os.path.join(ROOT, "megapath_b200", "ini", "soap4-nt2.ini")
LOPT = 151


def soap4(index, fq1, fq2, out, flags, env=None, threads=3):
    cmd = [os.path.join(BIN_DIR, "soap4"), "pair", index, fq1, fq2, "-o", out, "-C", INI, "-L", str(LOPT), "-T", str(threads),
           "-u", "750", "-top", "95"] + list(flags)
    p = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.PIPE, timeout=600, env=dict(os.environ, **(env or {})))
    assert p.returncode == 0, p.stderr.decode(errors="replace")[-3000:]
    return p.stdout, p.stderr.decode(errors="replace")


def first_diff(a, b):
    la, lb = a.split(b"\n"), b.split(b"\n")
    for i, (x, y) in enumerate(zip(la, lb)):
        if x != y:
            return i, x[:300], y[:300]
    return min(len(la), len(lb)), len(la), len(lb)


@pytest.fixture(scope="session")
def third_ref(workdir, small_ref):
    """A third chunk index: every other sequence of small_ref with 2 % substitutions, under names of its own, plus an unrelated one."""
    from tools import synth
    rng = np.random.default_rng(77)
    seq, b = small_ref["seq"], small_ref["bounds"]
    parts = []
    for i in range(0, len(b) - 1, 2):
        s = seq[b[i]:b[i + 1]].copy()
        m = rng.random(len(s)) < 0.02
        s[m] = synth.ALPHA[rng.integers(0, 4, size=int(m.sum()))]
        parts.append(s)
    parts.append(synth.ALPHA[rng.integers(0, 4, size=40000)])
    d = os.path.join(workdir, "third")
    os.makedirs(d, exist_ok=True)
    fa = os.path.join(d, "ref3.fa")
    with open(fa, "wb") as f:
        for i, s in enumerate(parts):
            f.write(b">chunk2_%d third index\n" % (i + 1) + s.tobytes() + b"\n")
    subprocess.check_call([os.path.join(BIN_DIR, "2bwt-builder"), fa], cwd=d, stdout=subprocess.DEVNULL)
    return dict(prefix=fa + ".index")


@pytest.fixture(scope="session")
def chain_reads(workdir, small_ref):
    """3000 divergent pairs with random and unalignable mates; names of every kind the rewrite between chunks treats differently."""
    fq1, fq2 = make_reads(workdir, small_ref, "chain", 3000, 150, seed=57, model="divergent", one_random=0.10, unalignable=0.05)
    kinds = [b"p%d/1", b"p%d/2/1", b"p%d/3/1", b"p%d/1/2", b"/1", b"p%d", b""]
    outs = []
    for path, mate in ((fq1, 1), (fq2, 2)):
        lines = open(path, "rb").read().split(b"\n")
        for i in range(0, len(lines) - 3, 4):
            k = i // 4
            nm = kinds[k % len(kinds)]
            nm = nm % k if b"%d" in nm else nm
            if nm.endswith(b"/1") and mate == 2:
                nm = nm[:-1] + b"2"
            lines[i] = b"@" + nm
        out = path.replace(".fq", "_n.fq")
        open(out, "wb").write(b"\n".join(lines))
        outs.append(out)
    return outs


def compose(workdir, name, indexes, fq1, fq2, flags, env=None, last_flags=()):
    """The K-process pipeline: step 0 with flags (incl. -nc), every later step without -nc on the previous step's stdout after the
    deinterleave rewrite.  -> list of (stdout, output prefix) per step."""
    steps, a, b = [], fq1, fq2
    for k, idx in enumerate(indexes):
        out = os.path.join(workdir, "%s_c%d" % (name, k))
        fl = list(flags) if k == 0 else [x for x in flags if x != "-nc"]
        if k + 1 == len(indexes):
            fl += list(last_flags)
        so, _ = soap4(idx, a, b, out, fl, env)
        steps.append((so, out))
        if k + 1 < len(indexes):
            t1, t2 = deinterleave_ordered(so)
            a, b = out + "_in_1.fq", out + "_in_2.fq"
            open(a, "wb").write(t1)
            open(b, "wb").write(t2)
    return steps


def chain_flags(workdir, name, indexes):
    out = []
    for k, idx in enumerate(indexes[1:], 1):
        out += ["-chain", idx, os.path.join(workdir, "%s_c%d" % (name, k))]
    return out


@pytest.fixture(scope="session")
def indexes(small_ref, second_ref, third_ref):
    return [small_ref["prefix"], second_ref["prefix"], third_ref["prefix"]]


@pytest.mark.parametrize("mode", ["-F", "-P"])
@pytest.mark.parametrize("contexts", [1, 3])
def test_chain_equals_composition(workdir, indexes, chain_reads, mode, contexts):
    env = {"MP_BATCH_READS": "1024", "MP_CONTEXTS_PER_GPU": str(contexts)}
    fq1, fq2 = chain_reads
    want = compose(workdir, "cmp%s%d" % (mode, contexts), indexes, fq1, fq2, [mode, "-nc"], env)[-1][0]
    assert want.count(b"SCORE:") > 1000
    got, err = soap4(indexes[0], fq1, fq2, os.path.join(workdir, "ch%s%d_c0" % (mode, contexts)),
                     [mode, "-nc"] + chain_flags(workdir, "ch%s%d" % (mode, contexts), indexes), env)
    assert "formatting on the device" in err and "chunk 2: index " + indexes[2] in err
    assert got == want, first_diff(got, want)
    if contexts == 3:
        host, _ = soap4(indexes[0], fq1, fq2, os.path.join(workdir, "chh%s_c0" % mode),
                        [mode, "-nc"] + chain_flags(workdir, "chh%s" % mode, indexes), dict(env, MP_HOST_IO="1"))
        assert host == want, first_diff(host, want)


def _bam_records(prefix, fq1):
    out = []
    for ext in (".dpout.1", ".gout.1", ".unpair"):
        names, lens, recs = read_bam(prefix + ext)
        out.append((names, lens, repr(recs).encode().replace(fq1.encode(), b"<fq1>")))
    return out


def test_chain_bam_per_chunk(workdir, indexes, chain_reads):
    """-b -F: every chunk writes its own .dpout.1 / .gout.N / .unpair under its output prefix, with the records of that chunk's own run."""
    env = {"MP_BATCH_READS": "1024"}
    fq1, fq2 = chain_reads
    steps = compose(workdir, "bcmp", indexes, fq1, fq2, ["-F", "-nc", "-b"], env)
    got, _ = soap4(indexes[0], fq1, fq2, os.path.join(workdir, "bch_c0"), ["-F", "-nc", "-b"] + chain_flags(workdir, "bch", indexes), env)
    assert got == steps[-1][0], first_diff(got, steps[-1][0])
    step_in = [fq1] + [out + "_in_1.fq" for _, out in steps[:-1]]
    for k, (_, out) in enumerate(steps):
        assert _bam_records(os.path.join(workdir, "bch_c%d" % k), fq1) == _bam_records(out, step_in[k])
        assert os.path.exists(os.path.join(workdir, "bch_c%d.gout.3" % k))


@pytest.mark.parametrize("output_seq", ["0", "1"])
def test_chain_lsam(workdir, indexes, chain_reads, output_seq):
    env = {"MP_BATCH_READS": "1024"}
    fq1, fq2 = chain_reads
    want = compose(workdir, "lcmp" + output_seq, indexes, fq1, fq2, ["-F", "-nc"], env, last_flags=["-lsam", output_seq])[-1][0]
    for e in (env, dict(env, MP_HOST_IO="1")):
        got, _ = soap4(indexes[0], fq1, fq2, os.path.join(workdir, "lch%s_c0" % output_seq),
                       ["-F", "-nc", "-lsam", output_seq] + chain_flags(workdir, "lch" + output_seq, indexes), e)
        assert got == want, first_diff(got, want)


def test_chain_gzip_input(workdir, indexes, chain_reads):
    env = {"MP_BATCH_READS": "1024"}
    fq1, fq2 = chain_reads
    flags = ["-F", "-nc"] + chain_flags(workdir, "gch", indexes)
    plain, _ = soap4(indexes[0], fq1, fq2, os.path.join(workdir, "gch_c0"), flags, env)
    gz = []
    for p in (fq1, fq2):
        open(p + ".gz", "wb").write(gzip.compress(open(p, "rb").read(), 6))
        gz.append(p + ".gz")
    got, _ = soap4(indexes[0], gz[0], gz[1], os.path.join(workdir, "gch_c0"), flags, env)
    assert got == plain, first_diff(got, plain)


def test_chain_long_header_batch_on_the_host(workdir, indexes, chain_reads):
    """A later batch whose header is longer than the device record limit (a SCORE: comment of more than 60000 bytes) is refused by the
    device ingest and goes through every chunk on the host; the stream still equals the composition."""
    env = {"MP_BATCH_READS": "1024"}
    fq1, fq2 = chain_reads
    lines = open(fq1, "rb").read().split(b"\n")
    lines[4 * 1500] += b" SCORE:90;" + b"".join(b"90,chunk1_%d second index;" % (i % 6 + 1) for i in range(2800))
    assert len(lines[4 * 1500]) > 60000
    long1 = fq1.replace(".fq", "_long.fq")
    open(long1, "wb").write(b"\n".join(lines))
    want = compose(workdir, "hcmp", indexes, long1, fq2, ["-F", "-nc"], env)[-1][0]
    got, err = soap4(indexes[0], long1, fq2, os.path.join(workdir, "hch_c0"), ["-F", "-nc"] + chain_flags(workdir, "hch", indexes), env)
    assert "formatting on the device" in err and "host parser" in err
    assert got == want, first_diff(got, want)


def test_chain_on_two_gpus(workdir, indexes, chain_reads):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    env = {"MP_BATCH_READS": "1024"}
    fq1, fq2 = chain_reads
    flags = ["-F", "-nc"] + chain_flags(workdir, "g2ch", indexes)
    one, _ = soap4(indexes[0], fq1, fq2, os.path.join(workdir, "g2ch_c0"), flags, env)
    two, _ = soap4(indexes[0], fq1, fq2, os.path.join(workdir, "g2ch_c0"), flags + ["-G", "2"], env)
    assert two == one, first_diff(two, one)


# ---- library entry points ----
def _params(lens):
    import megapath_b200 as mp
    ilow = max(1, int(lens[0::2].max()), int(lens[1::2].max()))
    return mp.default_params(nt2=True, insert_low=ilow, insert_high=750, max_read_length=LOPT)


def _same_results(a, b):
    """Every result field the output is made of, CIGAR texts included (the arrays hold fields the output never reads)."""
    import megapath_b200 as mp
    pf = ("readID", "insertSize", "algnmt_1", "algnmt_2", "score_1", "score_2", "editdist_1", "editdist_2", "num_sameScore_1",
          "num_sameScore_2", "strand_1", "strand_2", "pad")
    sf = ("readID", "algnmt", "score", "editdist", "num_sameScore", "strand")
    for f, fields, cig in (("pairs", pf, ("cigar_1", "cigar_2")), ("rescued", pf, ("cigar_1", "cigar_2")), ("singles", sf, ("cigar",))):
        assert len(a[f]) == len(b[f]), f
        for x in fields:
            assert np.array_equal(a[f][x], b[f][x]), (f, x)
        for x in cig:
            assert [mp.cigar_at(a["cigars"], int(o)) for o in a[f][x]] == [mp.cigar_at(b["cigars"], int(o)) for o in b[f][x]], (f, x)


def test_index_bind(workdir, indexes, chain_reads):
    """A clone bound to owner B aligns and formats exactly as B's own context; bound back to A, exactly as A's."""
    import megapath_b200 as mp
    fq1, fq2 = chain_reads
    t1, t2 = open(fq1, "rb").read(), open(fq2, "rb").read()
    owners = []
    for idx in indexes[:2]:
        o = mp.Context(0)
        o.index_load(idx)
        o.annotation_upload(idx)
        owners.append(o)
    lens = owners[0].fastq_upload(t1, t2, 3000, LOPT)
    P = _params(lens)
    for o in owners:
        o.index_prepare(P)
    clone = owners[0].clone()
    with pytest.raises(mp.MegapathError):
        owners[0].index_bind(owners[1])                 # owners are not rebound
    with pytest.raises(mp.MegapathError):
        clone.index_bind(clone)                          # a clone owns no index
    for k in (1, 0):
        own = owners[k]
        own.fastq_upload(t1, t2, 3000, LOPT)
        want = own.align_pairs(P)
        want_txt = own.format_fastq(top=0.95, mode=1, ignore_comments=True)
        clone.fastq_upload(t1, t2, 3000, LOPT)
        clone.index_bind(own)
        got = clone.align_pairs(P)
        _same_results(got, want)
        assert clone.format_fastq(top=0.95, mode=1, ignore_comments=True) == want_txt
        assert clone.index_info()["hbmBytes"] == own.index_info()["hbmBytes"]
    clone.close()
    for o in owners:
        o.close()


def test_fastq_chain_equals_upload_of_the_rewritten_text(workdir, indexes, chain_reads):
    import megapath_b200 as mp
    fq1, fq2 = chain_reads
    t1, t2 = open(fq1, "rb").read(), open(fq2, "rb").read()
    c = mp.Context(0)
    c.index_load(indexes[0])
    c.annotation_upload(indexes[0])
    lens = c.fastq_upload(t1, t2, 3000, LOPT)
    with pytest.raises(mp.MegapathError, match="status -4"):
        c.fastq_chain(LOPT)                              # nothing formatted yet
    P = _params(lens)
    c.align_pairs(P)
    text = c.format_fastq(top=0.95, mode=1, ignore_comments=True)
    r1, r2 = deinterleave_ordered(text)
    got_lens = c.fastq_chain(LOPT)
    with pytest.raises(mp.MegapathError, match="status -4"):
        c.fastq_chain(LOPT)                              # the formatted text was consumed
    c.seed_pairs(P)
    gp, gm = c.download_seedpos()
    gc = c.download_candidates()
    d = mp.Context(0)
    d.index_load(indexes[0])
    want_lens = d.fastq_upload(r1, r2, 3000, LOPT)
    d.seed_pairs(P)
    wp, wm = d.download_seedpos()
    assert np.array_equal(got_lens, want_lens)
    assert gp.tobytes() == wp.tobytes() and gm.tobytes() == wm.tobytes()
    assert gc.tobytes() == d.download_candidates().tobytes()
    c.close()
    d.close()


def test_fastq_chain_refusal_keeps_the_formatted_text(workdir, indexes, chain_reads):
    """A record whose rewritten header reaches the device record limit: MP_ERR_FORMAT, and the formatted text is still fetchable."""
    import ctypes
    import megapath_b200 as mp
    fq1, fq2 = chain_reads
    a = open(fq1, "rb").read().split(b"\n")
    # a header of 59998 bytes without "/1": accepted by the ingest (below 60000), kept whole by the formatter (the previous score 400
    # keeps the list and no alignment reaches its cut), and 2 bytes longer once the rewrite adds "/1"
    hdr = b"@p0 SCORE:400;"
    while len(hdr) < 59998 - 12:
        hdr += b"400,x;"
    hdr += b"400," + b"x" * (59998 - len(hdr) - 5) + b";"
    assert len(hdr) == 59998
    a[0] = hdr
    t1, t2 = b"\n".join(a), open(fq2, "rb").read()
    c = mp.Context(0)
    c.index_load(indexes[0])
    c.annotation_upload(indexes[0])
    lens = c.fastq_upload(t1, t2, 3000, LOPT)
    c.align_pairs(_params(lens))
    f = mp.FormatParams(0.95, 1, 0)
    n = ctypes.c_uint64()
    c._check(c.L.mp_format_fastq(c.h, ctypes.byref(f), ctypes.byref(n)))
    with pytest.raises(mp.FastqFormatError):
        c.fastq_chain(LOPT)
    buf = ctypes.create_string_buffer(max(int(n.value), 1))
    c._check(c.L.mp_format_fetch(c.h, buf, n.value))
    text = buf.raw[:n.value]
    assert text.count(b"\n") == 4 * 6000 and max(len(x) for x in text.split(b"\n")) == 59998
    c.close()


def test_index_load_budget(workdir, indexes, chain_reads):
    """Budgets that leave the SA dense (u32), 40-bit or as the file's samples keep hbmBytes within the budget -- K-mer filter
    included -- and give the same results; a budget below the index without a dense SA is refused."""
    import megapath_b200 as mp
    fq1, fq2 = chain_reads
    reads, lens = load_pairs(fq1, fq2, trunc=LOPT - 1)
    q, wpq = mp.pack_queries(reads, lens, LOPT)
    P = _params(lens)
    os.environ["MP_DENSE_SA"] = "0"
    try:
        c = mp.Context(0)
        c.index_load(indexes[0])
        fixed = c.index_info()["hbmBytes"]             # BWT, LKT, text and the file's SA samples
        c.close()
    finally:
        del os.environ["MP_DENSE_SA"]
    ref = mp.Context(0)
    ref.index_load(indexes[0])
    n = ref.index_info()["textLength"]
    ref.batch_upload(q, lens, wpq)
    want = ref.align_pairs(P)
    ref.close()
    dense = (n + 1) * 4
    dense_cap = dense + dense // 8 + 256
    seen = []
    for budget in (fixed + dense_cap + (64 << 20), fixed + dense_cap - 1, fixed + 4096):
        c = mp.Context(0)
        c.index_load_budget(indexes[0], budget)
        c.index_prepare(P)
        hbm = c.index_info()["hbmBytes"]
        assert hbm <= budget
        seen.append(hbm)
        c.batch_upload(q, lens, wpq)
        _same_results(c.align_pairs(P), want)
        c.close()
    assert seen[0] >= fixed + dense and seen[0] > seen[1] > fixed >= seen[2] - 4096
    c = mp.Context(0)
    with pytest.raises(mp.MegapathError, match="status -5"):
        c.index_load_budget(indexes[0], fixed - 1)
    c.close()
