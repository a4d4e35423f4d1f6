"""GPU suite: the CUDA path, called through the C-ABI (include/megapath_b200.h), against the
CPU oracle on the same seeded inputs.  Bit-exact: everything on this path is integer work."""
import numpy as np
import pytest

from conftest import make_reads, load_pairs
from oracle import pyoracle as po
from test_oracle_vs_ref import random_dp_tasks, exact_occurrence_tasks, DP_SHAPES, ref_detected_len

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx(small_ref):
    import megapath_b200 as mp
    c = mp.Context(0)
    c.index_load(small_ref["prefix"])
    yield c
    c.close()


def test_gpu_index_primitives(ctx, small_ref):
    ix = po.Index(small_ref["prefix"])
    info = ctx.index_info()
    assert info["textLength"] == ix.n and info["inverseSa0"] == ix.inverse_sa0
    rng = np.random.default_rng(3)
    idx = np.concatenate([rng.integers(0, ix.n + 2, size=50000), [0, 1, ix.inverse_sa0, ix.inverse_sa0 + 1, ix.n, ix.n + 1],
                          np.arange(0, 2000)]).astype(np.uint64)
    c = rng.integers(0, 4, size=len(idx)).astype(np.uint32)
    assert (ctx.occ(idx, c) == ix.occ(idx, c)).all()
    sidx = np.concatenate([rng.integers(0, ix.n + 1, size=20000), [0, ix.inverse_sa0, ix.n]]).astype(np.uint64)
    assert (ctx.sa(sidx) == ix.sa(sidx)).all()
    keys = np.concatenate([rng.integers(0, 4 ** 13, size=5000), [0, 1, 4 ** 13 - 1]]).astype(np.uint32)
    l, r = ctx.lkt(keys)
    for k, a, b in zip(keys[-400:], l[-400:], r[-400:]):
        assert ix.lkt(k) == (a, b)


@pytest.mark.parametrize("maxdna,maxread,fixed,clips", DP_SHAPES)
def test_gpu_dp_batch(ctx, maxdna, maxread, fixed, clips):
    import megapath_b200 as mp
    rng = np.random.default_rng(maxdna * 11 + maxread + clips[1])
    n = 300
    refs, dl, reads, rl = random_dp_tasks(rng, n, maxdna, maxread, fixed)
    cut = np.array([po.dp_cutoff(int(x)) for x in rl], dtype=np.int32)
    pd = mp.pack_dp_interleaved(refs, dl, maxdna)
    pr = mp.pack_dp_interleaved(reads, rl, maxread)
    sc, hl, mc, pats = ctx.dp_batch(pd, dl, maxdna, pr, rl, maxread, cut, clips[0], clips[1])
    nhit = 0
    for t in range(n):
        want = po.dp(refs[t, :dl[t]], reads[t, :rl[t]], clips[0], clips[1], -2, -3, int(cut[t]))
        got = (int(sc[t]), int(hl[t]), int(mc[t]), po.pattern_bytes(pats[t]) if sc[t] >= cut[t] else b"")
        assert got == want, (t, got, want)
        nhit += want[0] >= cut[t]
    assert nhit > n // 4


READ_SETS = [
    ("clean", 150, 151, dict(model="clean")),
    ("div", 100, 101, dict(model="divergent", one_random=0.05, unalignable=0.02)),
    ("var", 150, 151, dict(model="clean", varlen=True, n_rate=0.002)),
    ("long", 250, 251, dict(model="divergent")),
]


@pytest.mark.parametrize("name,rlen,lopt,kw", READ_SETS)
def test_gpu_seed_pair_and_deep_dp(ctx, workdir, small_ref, name, rlen, lopt, kw):
    import megapath_b200 as mp
    fq1, fq2 = make_reads(workdir, small_ref, "g_" + name, 1200 if name != "long" else 400, rlen, seed=21, **kw)
    reads, lens = load_pairs(fq1, fq2, trunc=lopt - 1)
    ix = po.Index(small_ref["prefix"])
    rp, mpos = ix.seed_pairs(reads, lens, po.mmp_params())
    insert_low = max(1, ref_detected_len(lens[0::2]), ref_detected_len(lens[1::2]))
    cands = po.pair_candidates(rp, mpos, lens, insert_low, 750)
    q, wpq = mp.pack_queries(reads, lens, lopt)
    ctx.batch_upload(q, lens, wpq)
    P = mp.default_params(insert_low=insert_low, insert_high=750, max_read_length=lopt)
    ctx.seed_pairs(P)
    grp, gmp = ctx.download_seedpos()
    assert grp.tobytes() == rp.tobytes() and gmp.tobytes() == mpos.tobytes()
    gc = ctx.download_candidates()
    assert gc.tobytes() == cands.tobytes()
    assert len(gc) > 100
    # stage S1 through the end-to-end call
    want, cells = po.deep_dp(ix, reads, lens, cands, insert_low, 750, lopt)
    res = ctx.align_pairs(P)
    got = res["pairs"]
    assert len(got) == len(want)
    for g, w in zip(got, want):
        for f in ("readID", "insertSize", "algnmt_1", "algnmt_2", "score_1", "score_2", "editdist_1", "editdist_2",
                  "num_sameScore_1", "num_sameScore_2", "strand_1", "strand_2", "startPos_1", "startPos_2",
                  "refDpLength_1", "refDpLength_2", "peLeftAnchor_1", "peLeftAnchor_2", "peRightAnchor_1", "peRightAnchor_2"):
            assert int(g[f]) == int(w[f]), (f, g, w)
        assert mp.cigar_at(res["cigars"], int(g["cigar_1"])) == w["cigar_1"]
        assert mp.cigar_at(res["cigars"], int(g["cigar_2"])) == w["cigar_2"]
    # best-hit choice on the device: exactly one result per pair is marked, the first with the maximal score sum
    i = 0
    while i < len(got):
        j = i
        while j < len(got) and got[j]["readID"] == got[i]["readID"]:
            j += 1
        sums = [int(got[k]["score_1"]) + int(got[k]["score_2"]) for k in range(i, j)]
        marks = [int(got[k]["pad"]) for k in range(i, j)]
        assert marks == [1 if k == sums.index(max(sums)) else 0 for k in range(j - i)], (i, sums, marks)
        i = j
    # dp_cells also counts the single-end / rescue tasks of pairs stage S1 left unaligned
    assert res["dp_cells"] >= cells and (len(res["singles"]) > 0 or res["dp_cells"] == cells)
    assert res["numDPAlignment"] == len(want)


def test_gpu_errors_are_loud(small_ref):
    import megapath_b200 as mp
    c = mp.Context(0)
    with pytest.raises(mp.MegapathError):
        c.index_load("/nonexistent/prefix")
    with pytest.raises(mp.MegapathError):
        c.seed_pairs(mp.default_params())
    c.close()


@pytest.mark.parametrize("large", [False, True])
@pytest.mark.parametrize("total,nseq,repeat_frac,seed", [(300000, 6, 0.05, 42), (70001, 1, 0.3, 5), (131072 + 255, 3, 0.0, 9), (65536 * 3, 2, 0.6, 11)])
def test_gpu_index_build_matches_reference_builder(workdir, total, nseq, repeat_frac, seed, large, monkeypatch):
    """mp_index_build + mp_index_save against the files 2bwt-builder writes for the same text
    (2BWT-Builder.c; BWTConstruct.c:994-1393; LTConstruct.c:46-96; HSP.c:560-699): byte-identical."""
    import os
    import megapath_b200 as mp
    from conftest import build_index
    from tools import synth
    if large:
        monkeypatch.setenv("MP_BUILD_LARGE", "1")       # the bucketed builder that texts >= 2^32 take (mp_build_large.cu)
    d = os.path.join(workdir, "b%d" % total)
    os.makedirs(d, exist_ok=True)
    seq, bounds = synth.make_ref(total, nseq, seed=seed, repeat_frac=repeat_frac)
    fa = os.path.join(d, "r.fa")
    synth.write_fasta(fa, seq, bounds)
    build_index(fa, "b%d" % total)
    codes = np.searchsorted(np.frombuffer(b"ACGT", dtype=np.uint8), seq).astype(np.uint8)
    c = mp.Context(0)
    c.index_build(mp.pack_text(codes), total)
    out = os.path.join(d, "mine.index")
    c.index_save(out)
    mp.save_annotation(out, total, ["seq%d" % (i + 1) for i in range(nseq)], bounds[:-1], np.diff(bounds))
    info = c.index_info()
    assert info["textLength"] == total
    for ext in (".pac", ".bwt", ".fmv", ".sa", ".lkt", ".tra", ".amb"):
        a = open(fa + ".index" + ext, "rb").read()
        b = open(out + ext, "rb").read()
        assert len(a) == len(b), ext
        assert a == b, ext
    # the built index answers like the loaded one
    ix = po.Index(fa + ".index")
    rng = np.random.default_rng(1)
    sidx = rng.integers(0, total + 1, size=4000).astype(np.uint64)
    assert (c.sa(sidx) == ix.sa(sidx)).all()
    c.close()


@pytest.mark.parametrize("stride", ["0", "1", "2", "3", "5", "8"])
def test_gpu_seeding_is_exact_for_every_filter_stride(workdir, small_ref, stride, monkeypatch):
    """The K-mer presence filter only skips starts that cannot produce a seed: SeedPos arrays must equal the oracle's with the
    filter off (MP_BLOOM=0) and with every probe stride (K = seedMinLength - (stride - 1)); the bench's 3.1 Gbp text uses
    stride 3, the small test texts would pick 8 on their own."""
    import megapath_b200 as mp
    if stride == "0":
        monkeypatch.setenv("MP_BLOOM", "0")
    else:
        monkeypatch.setenv("MP_BLOOM_STRIDE", stride)
    c = mp.Context(0)
    try:
        c.index_load(small_ref["prefix"])
        ix = po.Index(small_ref["prefix"])
        for name, rlen, lopt, kw in READ_SETS[:3]:
            fq1, fq2 = make_reads(workdir, small_ref, "s_" + name, 600, rlen, seed=33, **kw)
            reads, lens = load_pairs(fq1, fq2, trunc=lopt - 1)
            rp, mpos = ix.seed_pairs(reads, lens, po.mmp_params())
            q, wpq = mp.pack_queries(reads, lens, lopt)
            c.batch_upload(q, lens, wpq)
            P = mp.default_params(insert_low=max(1, int(lens.max())), insert_high=750, max_read_length=lopt)
            c.seed_pairs(P)
            grp, gmp = c.download_seedpos()
            assert grp.tobytes() == rp.tobytes() and gmp.tobytes() == mpos.tobytes(), (stride, name)
    finally:
        c.close()


@pytest.mark.parametrize("clips", [(130, 130), (10, 20), (0, 0)])
def test_gpu_dp_exact_occurrences(ctx, clips):
    """tasks the exact-occurrence test answers (occurrence at the window start / end, window == read, homopolymer and tandem
    windows with many occurrences, near-misses that must still go through the DP) == oracle, which
    test_dp_exact_occurrences_match_reference_callDP pins to the reference's callDP on the same tasks"""
    import megapath_b200 as mp
    rng = np.random.default_rng(977 + clips[0])
    n, maxdna, maxread = 192, 220, 152
    refs, dl, reads, rl = exact_occurrence_tasks(rng, n, maxdna, maxread)
    cut = np.array([po.dp_cutoff(int(x)) for x in rl], dtype=np.int32)
    sc, hl, mc, pats = ctx.dp_batch(mp.pack_dp_interleaved(refs, dl, maxdna), dl, maxdna, mp.pack_dp_interleaved(reads, rl, maxread), rl, maxread,
                                    cut, clips[0], clips[1])
    full = 0
    for t in range(n):
        want = po.dp(refs[t, :dl[t]], reads[t, :rl[t]], clips[0], clips[1], -2, -3, int(cut[t]))
        got = (int(sc[t]), int(hl[t]), int(mc[t]), po.pattern_bytes(pats[t]) if sc[t] >= cut[t] else b"")
        assert got == want, (t, got, want)
        full += want[0] == int(rl[t])
    assert full > n // 2


@pytest.mark.parametrize("hint", ["0", "17", "30", "95", "400"])
def test_gpu_dp_result_does_not_depend_on_the_diagonal_hint(ctx, hint, monkeypatch):
    """k_dp_fill only books cells that reach max(cutoff, lower bound from the task's hinted diagonal).  Whatever the hint says --
    the true diagonal, a wrong one, one outside the window -- score, tie count, hit offset and pattern must equal the oracle's."""
    import megapath_b200 as mp
    monkeypatch.setenv("MP_DP_TEST_HINT", hint)
    for maxdna, maxread, fixed, clips in (DP_SHAPES[0], DP_SHAPES[-1]):
        rng = np.random.default_rng(4242 + int(hint))
        n = 256
        refs, dl, reads, rl = random_dp_tasks(rng, n, maxdna, maxread, fixed)
        cut = np.array([po.dp_cutoff(int(x)) for x in rl], dtype=np.int32)
        sc, hl, mc, pats = ctx.dp_batch(mp.pack_dp_interleaved(refs, dl, maxdna), dl, maxdna, mp.pack_dp_interleaved(reads, rl, maxread), rl, maxread,
                                        cut, clips[0], clips[1])
        for t in range(n):
            want = po.dp(refs[t, :dl[t]], reads[t, :rl[t]], clips[0], clips[1], -2, -3, int(cut[t]))
            got = (int(sc[t]), int(hl[t]), int(mc[t]), po.pattern_bytes(pats[t]) if sc[t] >= cut[t] else b"")
            assert got == want, (hint, t, got, want)
    # exact repeats: many cells tie with the best score, every one of them has to be counted
    refs, dl, reads, rl = exact_occurrence_tasks(np.random.default_rng(7), 128, 220, 152)
    monkeypatch.setenv("MP_DP_EXACT", "0")          # read once per process: only effective if this test runs first; harmless otherwise
    cut = np.array([po.dp_cutoff(int(x)) for x in rl], dtype=np.int32)
    sc, hl, mc, pats = ctx.dp_batch(mp.pack_dp_interleaved(refs, dl, 220), dl, 220, mp.pack_dp_interleaved(reads, rl, 152), rl, 152, cut, 130, 130)
    for t in range(128):
        want = po.dp(refs[t, :dl[t]], reads[t, :rl[t]], 130, 130, -2, -3, int(cut[t]))
        got = (int(sc[t]), int(hl[t]), int(mc[t]), po.pattern_bytes(pats[t]) if sc[t] >= cut[t] else b"")
        assert got == want, (hint, t, got, want)


@pytest.mark.parametrize("mm,go", [(-3, -2), (-4, -6), (-2, -6), (-3, -3), (-4, -3)])
def test_gpu_dp_other_score_parameters(ctx, mm, go):
    """run-time score parameters (the generic kernel instantiation; CPU_DP.cpp:199-208 allows -4 <= mismatch, -6 <= open; mismatch = -1 divides by zero at :310)."""
    import megapath_b200 as mp
    rng = np.random.default_rng(100 - mm * 7 - go)
    n, maxdna, maxread = 160, 220, 152
    refs, dl, reads, rl = random_dp_tasks(rng, n, maxdna, maxread, False)
    cut = np.array([po.dp_cutoff(int(x)) for x in rl], dtype=np.int32)
    sc, hl, mc, pats = ctx.dp_batch(mp.pack_dp_interleaved(refs, dl, maxdna), dl, maxdna, mp.pack_dp_interleaved(reads, rl, maxread), rl, maxread,
                                    cut, 130, 130, mismatch=mm, gap_open=go)
    for t in range(n):
        want = po.dp(refs[t, :dl[t]], reads[t, :rl[t]], 130, 130, mm, go, int(cut[t]))
        got = (int(sc[t]), int(hl[t]), int(mc[t]), po.pattern_bytes(pats[t]) if sc[t] >= cut[t] else b"")
        assert got == want, (mm, go, t, got, want)


@pytest.mark.parametrize("env,val,walks", [("MP_DENSE_SA", "0", True), ("MP_SA40", "0", False), ("MP_SA40", "2", True), ("MP_SA40", "3", True)])
def test_gpu_sampled_sa_path(workdir, small_ref, monkeypatch, env, val, walks):
    """The SA representations of texts that do not fit a dense 32-bit array.  MP_DENSE_SA=0: only the file's 1/16 samples (u64) are
    resident and every SA lookup on the hot path is an LF walk.  MP_SA40=<shift>: the 40-bit sample arrays (u32 + u8) that texts of
    2^32 bases and more get, forced here on a small text -- every index (shift 0: no walks) or every 4th / 8th.  Seeds, candidates and
    stage-S1 results must not change."""
    import megapath_b200 as mp
    monkeypatch.setenv(env, val)
    c = mp.Context(0)
    try:
        c.index_load(small_ref["prefix"])
        ix = po.Index(small_ref["prefix"])
        rng = np.random.default_rng(5)
        sidx = np.concatenate([rng.integers(0, ix.n + 1, size=20000), [0, ix.inverse_sa0, ix.n]]).astype(np.uint64)
        assert (c.sa(sidx) == ix.sa(sidx)).all()
        for name, rlen, lopt, kw in READ_SETS[:3]:
            fq1, fq2 = make_reads(workdir, small_ref, "sa_" + name, 800, rlen, seed=77, **kw)
            reads, lens = load_pairs(fq1, fq2, trunc=lopt - 1)
            rp, mpos = ix.seed_pairs(reads, lens, po.mmp_params())
            insert_low = max(1, ref_detected_len(lens[0::2]), ref_detected_len(lens[1::2]))
            cands = po.pair_candidates(rp, mpos, lens, insert_low, 750)
            q, wpq = mp.pack_queries(reads, lens, lopt)
            c.batch_upload(q, lens, wpq)
            P = mp.default_params(insert_low=insert_low, insert_high=750, max_read_length=lopt)
            c.seed_pairs(P)
            grp, gmp = c.download_seedpos()
            assert grp.tobytes() == rp.tobytes() and gmp.tobytes() == mpos.tobytes(), name
            assert c.download_candidates().tobytes() == cands.tobytes(), name
            want, _ = po.deep_dp(ix, reads, lens, cands, insert_low, 750, lopt)
            res = c.align_pairs(P)
            assert len(res["pairs"]) == len(want)
            for g, w in zip(res["pairs"], want):
                for f in ("readID", "algnmt_1", "algnmt_2", "score_1", "score_2", "num_sameScore_1", "num_sameScore_2", "insertSize"):
                    assert int(g[f]) == int(w[f]), (name, f, g, w)
            assert (res["n_lf"] > 0) == walks     # the walks really happened (or, with a sample per index, did not)
    finally:
        c.close()


@pytest.mark.parametrize("lanes", ["4", "32"])
def test_gpu_hit_sort_group_sizes(workdir, small_ref, lanes, monkeypatch):
    """k_hit_sort orders a read's hits with 4 lanes per read on human-like data and with 32 on NT-like data (dozens of hits per
    read); forced either way here, both must give the oracle's SeedPos arrays."""
    import megapath_b200 as mp
    monkeypatch.setenv("MP_HIT_SORT_G", lanes)
    c = mp.Context(0)
    try:
        c.index_load(small_ref["prefix"])
        ix = po.Index(small_ref["prefix"])
        for name, rlen, lopt, kw in READ_SETS[:4]:
            fq1, fq2 = make_reads(workdir, small_ref, "hs_" + name, 700, rlen, seed=55, **kw)
            reads, lens = load_pairs(fq1, fq2, trunc=lopt - 1)
            rp, mpos = ix.seed_pairs(reads, lens, po.mmp_params())
            q, wpq = mp.pack_queries(reads, lens, lopt)
            c.batch_upload(q, lens, wpq)
            P = mp.default_params(insert_low=max(1, int(lens.max())), insert_high=750, max_read_length=lopt)
            c.seed_pairs(P)
            grp, gmp = c.download_seedpos()
            assert grp.tobytes() == rp.tobytes() and gmp.tobytes() == mpos.tobytes(), (lanes, name)
    finally:
        c.close()


def test_gpu_abi_rejects_overlong_reads(ctx):
    """A read that does not fit its 2-bit row, or is not shorter than maxReadLength, is refused at the C-ABI instead of corrupting
    neighbouring DP tasks (the reference truncates at parse time, QueryParser.cpp:188)."""
    import megapath_b200 as mp
    reads = np.zeros((2, 200), dtype=np.uint8)
    lens = np.array([200, 100], dtype=np.uint32)
    q, wpq = mp.pack_queries(reads, np.array([160, 100], dtype=np.uint32), 151)
    with pytest.raises(mp.MegapathError):
        ctx.batch_upload(q, lens, wpq)                       # 200 bases > 16 * wpq
    lens = np.array([155, 100], dtype=np.uint32)
    ctx.batch_upload(q, lens, wpq)
    with pytest.raises(mp.MegapathError):
        ctx.seed_pairs(mp.default_params(insert_low=150, insert_high=750, max_read_length=151))
