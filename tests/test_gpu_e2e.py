"""GPU suite, end to end: the product's soap4 driver (host C++ + libmegapath_b200.so) must print the same
annotated FASTQ as the reference binary on the same index and reads, after the canonical sort of pairs.
Covers all stages: deep DP (S1), single-end DP (S2), mate rescue (S3), unpaired output (S4)."""
import os

import numpy as np
import pytest

from conftest import make_reads, run_ref_soap4, run_our_soap4, canon_fastq, deinterleave, run_ref_raw

pytestmark = pytest.mark.gpu
G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")

E2E_SETS = [
    ("clean", 150, 151, dict(model="clean"), "soap4.ini", ("-F", "-nc")),
    ("mixed", 100, 101, dict(model="divergent", one_random=0.10, unalignable=0.05), "soap4.ini", ("-F", "-nc")),
    ("var", 150, 151, dict(model="clean", varlen=True, n_rate=0.002, one_random=0.05), "soap4.ini", ("-F", "-nc")),
    ("long", 250, 251, dict(model="divergent", one_random=0.05), "soap4.ini", ("-F", "-nc")),
    ("nt2", 150, 151, dict(model="divergent", one_random=0.10, unalignable=0.02), "soap4-nt2.ini", ("-F", "-nc", "-top", "95")),
    ("pmode", 100, 101, dict(model="divergent", one_random=0.10, unalignable=0.05), "soap4.ini", ("-P", "-nc")),
    ("span", 150, 151, dict(model="clean", span_frac=0.05), "soap4.ini", ("-F", "-nc")),
]


def first_diff(a, b):
    la, lb = a.split(b"\n"), b.split(b"\n")
    for i, (x, y) in enumerate(zip(la, lb)):
        if x != y:
            return i, x[:300], y[:300]
    return min(len(la), len(lb)), b"<end>", b"<end>"


@pytest.mark.parametrize("name,rlen,lopt,kw,ini,extra", E2E_SETS)
def test_e2e_stdout_matches_reference(workdir, small_ref, name, rlen, lopt, kw, ini, extra):
    npairs = 3000 if name != "long" else 800
    fq1, fq2 = make_reads(workdir, small_ref, "e2e_" + name, npairs, rlen, seed=31, **kw)
    ref_out, _ = run_ref_soap4(workdir, small_ref["prefix"], fq1, fq2, "e2eref_" + name, lopt, dump=False, ini=ini, threads=4,
                               extra=[x for x in extra if x not in ("-F", "-nc")] + (["-P"] if "-P" in extra else []))
    want = canon_fastq(open(ref_out, "rb").read())
    got = canon_fastq(run_our_soap4(workdir, small_ref["prefix"], fq1, fq2, "e2eour_" + name, lopt, ini=ini, extra=extra))
    assert len(want) > 1000
    assert got == want, first_diff(got, want)


@pytest.mark.parametrize("name", ["clean", "div", "nt2"])
def test_e2e_stdout_matches_golden(tmp_path, name):
    """Same check against the committed reference outputs (no oracle/_ref needed): index built by the GPU builder."""
    import megapath_b200 as mp
    z = np.load(os.path.join(G, name + ".npz"))
    lopt, nt2 = int(z["lopt"][0]), bool(z["nt2"][0])
    pac = np.fromfile(os.path.join(G, "idx.pac"), dtype=np.uint8)
    n = int(open(os.path.join(G, "idx.ann")).readline().split()[0])
    prefix = str(tmp_path / "g.index")
    c = mp.Context(0)
    c.index_build(pac[:(n + 3) // 4], n)
    c.index_save(prefix)
    c.close()
    for ext in ("ann", "amb", "tra"):
        open(prefix + "." + ext, "wb").write(open(os.path.join(G, "idx." + ext), "rb").read())
    got = canon_fastq(run_our_soap4(str(tmp_path), prefix, os.path.join(G, name + "_1.fq"), os.path.join(G, name + "_2.fq"), "g_" + name, lopt,
                                    ini="soap4-nt2.ini" if nt2 else "soap4.ini"))
    want = bytes(z["fastq"])
    assert got == want, first_diff(got, want)


BAM_SETS = [
    ("clean", 150, 151, dict(model="clean"), "soap4.ini", ("-b", "-F", "-nc")),
    ("mixed", 100, 101, dict(model="divergent", one_random=0.10, unalignable=0.05), "soap4.ini", ("-b", "-F", "-nc")),
    ("nofq", 100, 101, dict(model="divergent", one_random=0.10, unalignable=0.05), "soap4.ini", ("-b",)),
    ("span", 150, 151, dict(model="clean", span_frac=0.08), "soap4.ini", ("-b", "-F", "-nc")),
    ("nt2p", 150, 151, dict(model="divergent", one_random=0.10), "soap4-nt2.ini", ("-b", "-F", "-nc", "-top", "95", "-p")),
]


@pytest.mark.parametrize("name,rlen,lopt,kw,ini,extra", BAM_SETS)
def test_e2e_bam_matches_reference(workdir, small_ref, name, rlen, lopt, kw, ini, extra):
    """-b: decoded records of .dpout.1 + .gout.* + .unpair (flag, pos, MAPQ, CIGAR, mate fields, isize, seq, qual, every tag)
    equal the reference's after sorting by (read name, mate)."""
    import glob
    from conftest import canon_bam
    fq1, fq2 = make_reads(workdir, small_ref, "bam_" + name, 2500, rlen, seed=41, **kw)
    pre_r, pre_o = os.path.join(workdir, "bamref_" + name), os.path.join(workdir, "bamour_" + name)
    for f in glob.glob(pre_r + ".*") + glob.glob(pre_o + ".*"):
        if os.path.isfile(f):
            os.remove(f)
    ref_fq, _ = run_ref_soap4(workdir, small_ref["prefix"], fq1, fq2, "bamref_" + name, lopt, dump=False, ini=ini, threads=3,
                              extra=[x for x in extra if x not in ("-F", "-nc")])
    # run_ref_soap4 always passes -F -nc; the "nofq" set needs a run without them
    if "-F" not in extra:
        for f in glob.glob(pre_r + ".*"):
            if os.path.isfile(f) and not f.endswith(".fq"):
                os.remove(f)
        run_ref_raw(workdir, small_ref["prefix"], fq1, fq2, "bamref_" + name, lopt, ini, list(extra))
    got_fq = run_our_soap4(workdir, small_ref["prefix"], fq1, fq2, "bamour_" + name, lopt, ini=ini, extra=extra)
    if "-F" in extra:
        assert canon_fastq(got_fq) == canon_fastq(open(ref_fq, "rb").read())
    files = lambda pre: [pre + ".dpout.1", pre + ".unpair"] + sorted(glob.glob(pre + ".gout.*"))
    (hn_r, recs_r), (hn_o, recs_o) = canon_bam(files(pre_r)), canon_bam(files(pre_o))
    assert hn_r == hn_o
    assert len(recs_r) == len(recs_o) == 2 * 2500
    for a, b in zip(recs_o, recs_r):
        assert a == b, (a, b)


def _write_fq(path, recs, mate):
    with open(path, "wb") as f:
        for i, s in enumerate(recs):
            f.write(b"@e%d/%d\n" % (i, mate) + s + b"\n+\n" + b"I" * len(s) + b"\n")


def test_e2e_edge_cases_match_reference(workdir, small_ref):
    """Ragged and degenerate inputs: reads longer than -L (truncated to L-1, QueryParser.cpp:188), short reads, all-N reads
    (N -> G, IndexHandler.cpp:41-45), a read made of the last bases of the text, lower-case bases.
    Reads shorter than the DP cutoff max(0.2 L, 30) are outside the reference's defined behaviour: its SIMD kernel aborts the
    whole vector group (16 or 32 unrelated tasks, depending on the build) that contains such a task (CPU_DP.cpp:296-324), so
    its output for OTHER reads then depends on batch composition; lengths here start at 36."""
    rng = np.random.default_rng(5)
    seq = small_ref["seq"]
    comp = {65: 84, 67: 71, 71: 67, 84: 65}
    r1, r2 = [], []
    for k in range(400):
        st = int(rng.integers(0, len(seq) - 600))
        isz = int(rng.integers(260, 500))
        l1, l2 = int(rng.integers(36, 180)), int(rng.integers(36, 180))
        a = bytes(seq[st:st + l1])
        b = bytes(comp[c] for c in seq[st + isz - l2:st + isz][::-1])
        if k % 7 == 0:
            a = b"N" * l1
        if k % 11 == 0:
            b = b.lower()
        if k % 13 == 0:
            a = bytes(seq[len(seq) - l1:])                       # last bases of the text
        r1.append(a)
        r2.append(b)
    fq1, fq2 = os.path.join(workdir, "edge_1.fq"), os.path.join(workdir, "edge_2.fq")
    _write_fq(fq1, r1, 1)
    _write_fq(fq2, r2, 2)
    for lopt in (151, 101):
        ref_out, _ = run_ref_soap4(workdir, small_ref["prefix"], fq1, fq2, "edgeref%d" % lopt, lopt, dump=False, threads=2)
        want = canon_fastq(open(ref_out, "rb").read())
        got = canon_fastq(run_our_soap4(workdir, small_ref["prefix"], fq1, fq2, "edgeour%d" % lopt, lopt))
        assert got == want, first_diff(got, want)


def test_e2e_empty_input(workdir, small_ref):
    fq1, fq2 = os.path.join(workdir, "empty_1.fq"), os.path.join(workdir, "empty_2.fq")
    open(fq1, "wb").close()
    open(fq2, "wb").close()
    assert run_our_soap4(workdir, small_ref["prefix"], fq1, fq2, "emptyour", 151) == b""


# ---- header comment chaining: every NT chunk after the first runs WITHOUT -nc (runMegaPath.sh:184-226) and merges the
#      SCORE: list of the previous chunk into its own (BGS-IO.cpp:1348-1371, 1384-1446, 1966-2091) ----
def _edit_comments(k, mate, comm):
    if k % 19 == 3:
        return b"IGNORE"                         # passes through untouched (BGS-IO.cpp:1399-1401)
    if k % 23 == 5 and mate == 1:
        return b"SCORE:0;"                        # an unaligned read of the previous chunk
    if k % 29 == 7:
        return b"SCORE:400;400,made_up_hit;"      # better than anything this chunk can find: must survive, and cap -top
    if k % 31 == 11 and mate == 0:
        return b""                                # no comment at all
    return comm


@pytest.mark.parametrize("mode", ["F", "P", "Fb"])
def test_e2e_chained_comments_match_reference(workdir, small_ref, second_ref, mode):
    import glob
    from conftest import canon_bam
    fq1, fq2 = make_reads(workdir, small_ref, "chain", 2500, 150, seed=77, model="divergent", one_random=0.10, unalignable=0.04)
    # chunk 0: -nc; the reference's output (== ours, test_e2e_stdout_matches_reference) feeds chunk 1 of both programs
    first = run_ref_raw(workdir, small_ref["prefix"], fq1, fq2, "chain0", 151, "soap4-nt2.ini", ["-F", "-nc", "-top", "95"])
    assert first.count(b"SCORE:") > 4000
    in1, in2 = deinterleave(first, os.path.join(workdir, "chain_in"), _edit_comments)
    flags = {"F": ["-F", "-top", "95"], "P": ["-P", "-top", "95"], "Fb": ["-b", "-F", "-top", "95"]}[mode]
    pre_r, pre_o = os.path.join(workdir, "chain1ref_" + mode), os.path.join(workdir, "chain1our_" + mode)
    for f in glob.glob(pre_r + ".*") + glob.glob(pre_o + ".*"):
        if os.path.isfile(f):
            os.remove(f)
    want = canon_fastq(run_ref_raw(workdir, second_ref["prefix"], in1, in2, "chain1ref_" + mode, 151, "soap4-nt2.ini", flags))
    got = canon_fastq(run_our_soap4(workdir, second_ref["prefix"], in1, in2, "chain1our_" + mode, 151, ini="soap4-nt2.ini", extra=flags))
    assert want.count(b"chunk1_") > 1000 and want.count(b"seq") > 1000 and want.count(b"IGNORE") > 100 and b"made_up_hit" in want
    assert got == want, first_diff(got, want)
    if mode == "Fb":
        files = lambda pre: [pre + ".dpout.1", pre + ".unpair"] + sorted(glob.glob(pre + ".gout.*"))
        (hn_r, recs_r), (hn_o, recs_o) = canon_bam(files(pre_r)), canon_bam(files(pre_o))
        assert hn_r == hn_o and len(recs_r) == len(recs_o)
        for a, b in zip(recs_o, recs_r):
            assert a == b, (a, b)


@pytest.mark.parametrize("lopt", [76, 121, 201])
def test_e2e_max_read_length_sweep(workdir, small_ref, lopt):
    """-L sweep (BASELINE config 5): reads of exactly L-1 bases and mixed shorter ones, margins 25 / 30, K = 5 and 8 column strips"""
    rlen = lopt - 1
    fq1, fq2 = make_reads(workdir, small_ref, "sweep%d" % lopt, 1500 if lopt < 200 else 700, rlen, seed=lopt,
                          model="divergent", one_random=0.08, unalignable=0.03, varlen=(lopt == 121))
    ref_out, _ = run_ref_soap4(workdir, small_ref["prefix"], fq1, fq2, "sweepref%d" % lopt, lopt, dump=False, threads=4)
    want = canon_fastq(open(ref_out, "rb").read())
    got = canon_fastq(run_our_soap4(workdir, small_ref["prefix"], fq1, fq2, "sweepour%d" % lopt, lopt))
    assert len(want) > 1000
    assert got == want, first_diff(got, want)


def test_e2e_threads_and_contexts(workdir, small_ref, monkeypatch):
    """-T 7 and two contexts on one GPU (MP_CONTEXTS_PER_GPU=2) over several small batches (MP_BATCH_READS) give the single-context
    output: batches alternate between contexts that share the resident index (mp_clone)."""
    fq1, fq2 = make_reads(workdir, small_ref, "ctxs", 6000, 100, seed=91, model="divergent", one_random=0.08, unalignable=0.03)
    ref_out, _ = run_ref_soap4(workdir, small_ref["prefix"], fq1, fq2, "ctxsref", 101, dump=False, threads=4)
    want = canon_fastq(open(ref_out, "rb").read())
    monkeypatch.setenv("MP_BATCH_READS", "2048")
    for nctx in ("1", "2"):
        monkeypatch.setenv("MP_CONTEXTS_PER_GPU", nctx)
        got = canon_fastq(run_our_soap4(workdir, small_ref["prefix"], fq1, fq2, "ctxsour" + nctx, 101, extra=("-F", "-nc", "-T", "7")))
        assert got == want, (nctx, first_diff(got, want))


def test_e2e_cigar_text_fallback(workdir, small_ref, monkeypatch):
    """The traceback leaves each special CIGAR at the end of its pattern row and stage-S1 assembly copies it; when pattern and text
    would not both fit the row the assembly encodes from the pattern instead.  MP_CIG_TEXT=0 forces that path for every result:
    the decoded BAM records (CIGAR, NM / MD, positions, tags) must still equal the reference's."""
    monkeypatch.setenv("MP_CIG_TEXT", "0")
    name, rlen, lopt, kw, ini, extra = BAM_SETS[-1]
    test_e2e_bam_matches_reference(workdir, small_ref, "cigfb_" + name, rlen, lopt, kw, ini, extra)


def test_e2e_lsam_mode_matches_reference_pipe(workdir, small_ref):
    """`soap4 ... -F -lsam 1` == `reference soap4 ... -F | cc/fastq2lsam 1` (runMegaPath.sh:136), pair lines sorted by name"""
    from conftest import run_ref_fastq2lsam
    fq1, fq2 = make_reads(workdir, small_ref, "lsam", 2000, 150, seed=5, model="divergent", one_random=0.10, unalignable=0.05)
    first = run_ref_raw(workdir, small_ref["prefix"], fq1, fq2, "lsamref", 151, "soap4-nt2.ini", ["-F", "-nc", "-top", "95"])
    want = run_ref_fastq2lsam("e2e_lsam", first, "1", workdir, ordered=False)
    got = run_our_soap4(workdir, small_ref["prefix"], fq1, fq2, "lsamour", 151, ini="soap4-nt2.ini", extra=("-F", "-nc", "-top", "95", "-lsam", "1"))

    def canon(data):
        lines = data.split(b"\n")[:-1]
        pairs = [(lines[i], lines[i + 1]) for i in range(0, len(lines) - 1, 2)]
        return sorted(pairs)
    assert len(canon(want)) == 2000 and want.count(b"\t64\t") == 2000
    assert canon(got) == canon(want)


def test_e2e_builder_with_ambiguity_runs(workdir):
    """bin/2bwt-builder on a FASTA with short / long N runs, IUPAC codes and lower case: every index file equals the reference
    builder's (HSP.c:486-528 cut-outs + translate table), and soap4 on that index prints the reference's records (positions behind
    cut-out runs go through the translate table's corrections)."""
    import subprocess
    from conftest import ROOT, build_index
    from test_builder_fasta import fasta_with_ambiguity
    d = os.path.join(workdir, "amb")
    os.makedirs(d, exist_ok=True)
    raw = fasta_with_ambiguity(11, nseq=4, seqlen=60000)
    fa_ref, fa_our = os.path.join(d, "ref.fa"), os.path.join(d, "our.fa")
    for p in (fa_ref, fa_our):
        open(p, "wb").write(raw)
    build_index(fa_ref, "amb")
    subprocess.check_call([os.path.join(ROOT, "megapath_b200", "bin", "2bwt-builder"), fa_our], cwd=d, stdout=subprocess.DEVNULL)
    for ext in ("pac", "bwt", "fmv", "sa", "lkt", "tra", "amb"):
        assert open(fa_ref + ".index." + ext, "rb").read() == open(fa_our + ".index." + ext, "rb").read(), ext
    # FR pairs from the raw sequences (windows without ambiguity codes), a third of them right next to a run
    rng = np.random.default_rng(3)
    seqs = [b"".join(x.split(b"\n")[1:]).upper() for x in raw.split(b">")[1:]]
    comp = bytes.maketrans(b"ACGT", b"TGCA")
    r1, r2 = [], []
    while len(r1) < 1500:
        s = seqs[int(rng.integers(0, len(seqs)))]
        isz = int(rng.integers(260, 480))
        if len(r1) % 3 == 0:
            hits = [i for i in range(0, len(s) - 600, 50) if s[i] not in b"ACGT"]
            st = (hits[int(rng.integers(0, len(hits)))] + int(rng.integers(1, 40))) if hits else 0
        else:
            st = int(rng.integers(0, len(s) - 600))
        frag = s[st:st + isz]
        a, b = frag[:150], frag[-150:].translate(comp)[::-1]
        if len(frag) < isz or any(c not in b"ACGT" for c in a + b):
            continue
        r1.append(np.frombuffer(a, dtype=np.uint8))
        r2.append(np.frombuffer(b, dtype=np.uint8))
    from tools import synth
    fq1, fq2 = os.path.join(d, "amb_1.fq"), os.path.join(d, "amb_2.fq")
    synth.write_fastq(fq1, r1, 1)
    synth.write_fastq(fq2, r2, 2)
    ref_out, _ = run_ref_soap4(d, fa_ref + ".index", fq1, fq2, "ambref", 151, dump=False, threads=3)
    want = canon_fastq(open(ref_out, "rb").read())
    got = canon_fastq(run_our_soap4(d, fa_our + ".index", fq1, fq2, "ambour", 151))
    assert want.count(b"SCORE:") == 3000 and want.count(b"SCORE:0;") < 600
    assert got == want, first_diff(got, want)
    # and with BAM records (chromosome-relative positions, MD/NM) on the same index
    import glob
    from conftest import canon_bam
    for pre in ("ambrefb", "ambourb"):
        for f in glob.glob(os.path.join(d, pre) + ".*"):
            os.remove(f)
    run_ref_raw(d, fa_ref + ".index", fq1, fq2, "ambrefb", 151, "soap4.ini", ["-b", "-F", "-nc", "-p"])
    run_our_soap4(d, fa_our + ".index", fq1, fq2, "ambourb", 151, extra=("-b", "-F", "-nc", "-p"))
    files = lambda pre: [os.path.join(d, pre) + ".dpout.1", os.path.join(d, pre) + ".unpair"] + sorted(glob.glob(os.path.join(d, pre) + ".gout.*"))
    (hr, rr), (ho, ro) = canon_bam(files("ambrefb")), canon_bam(files("ambourb"))
    assert hr == ho and len(rr) == len(ro) == 3000
    for x, y in zip(ro, rr):
        assert x == y, (x, y)


def test_e2e_text_beyond_2_to_32(workdir):
    """BASELINE config 3 in small: a 4.4 Gbp synthetic reference (> 2^32 bases: 64-bit positions everywhere, bucketed index builder, sampled
    suffix array with LF walks, no dense 32-bit SA), soap4-nt2.ini -F -top 95, against the reference binary on the same index files.
    Needs ~60 GB of HBM, ~12 GB of /tmp and a few minutes; skipped when the box cannot hold it or MP_SKIP_HUGE is set."""
    import shutil
    import subprocess
    import torch
    import megapath_b200 as mp
    import bench
    if os.environ.get("MP_SKIP_HUGE"):
        pytest.skip("MP_SKIP_HUGE set")
    free, total = torch.cuda.mem_get_info(0)
    if free < 80e9 or shutil.disk_usage("/tmp").free < 20e9:
        pytest.skip("not enough HBM or /tmp space for the 4.4 Gbp index")
    d = "/tmp/mp_huge"
    os.makedirs(d, exist_ok=True)
    n, nseq = 4_400_000_000, 40
    dev = torch.device("cuda", 0)
    prefix = os.path.join(d, "huge.index")
    codes = bench.gen_ref_codes(n, 17, dev)
    bounds = bench.ref_bounds(n, nseq, 17)
    # near-duplicate "genomes": copies of 3 Mbp stretches with 1 % substitutions, so that -top 95 lists are not trivial
    g = torch.Generator(device=dev)
    g.manual_seed(5)
    for k in range(24):
        src, dst, ln = int(bounds[k % nseq]) + 1000, int(bounds[(k * 7 + 3) % nseq]) + 2_000_000 + 4_000_000 * (k // nseq), 3_000_000
        blk = codes[src:src + ln].clone()
        mut = torch.rand(ln, device=dev, generator=g) < 0.01
        blk[mut] = (blk[mut] + torch.randint(1, 4, (int(mut.sum()),), device=dev, generator=g, dtype=torch.uint8)) & 3
        codes[dst:dst + ln] = blk
    ctx = mp.Context(0)
    ctx.index_build_codes(codes, bounds, prefix)
    info = ctx.index_info()
    assert info["textLength"] == n > 2 ** 32
    bt = torch.from_numpy(bounds).to(dev)
    reads = bench.gen_batch(codes, bt, 100_000, 23, 150, "divergent", 0.02, 0.05).cpu().numpy()
    # a third of the pairs from the last 300 Mbp: positions above 2^32
    hi = bench.gen_batch(codes[-300_000_000:], torch.tensor([0, 300_000_000], device=dev), 30_000, 29, 150, "subs", 0.0, 0.0).cpu().numpy()
    reads[:60_000] = hi
    del codes
    ctx.close()
    torch.cuda.empty_cache()
    fqp = os.path.join(d, "huge")
    bench.write_fastq_sample(fqp, reads)
    ref = run_ref_raw(d, prefix, fqp + "_1.fq", fqp + "_2.fq", "hugeref", 151, "soap4-nt2.ini", ["-F", "-nc", "-top", "95"], threads=os.cpu_count() or 8)
    got = run_our_soap4(d, prefix, fqp + "_1.fq", fqp + "_2.fq", "hugeour", 151, ini="soap4-nt2.ini", extra=("-F", "-nc", "-top", "95"))
    want = canon_fastq(ref)
    assert want.count(b"SCORE:") == 200_000 and want.count(b"SCORE:0;") < 40_000
    assert canon_fastq(got) == want, first_diff(canon_fastq(got), want)
    shutil.rmtree(d, ignore_errors=True)
