"""CPU suite: pins the oracle restatement (oracle/mp_oracle*.cpp) against the reference itself
(oracle/_ref: soap4_dump seam dumps, libref_dp.so = the reference's callDP, libref_bwt.so =
the reference's BWTOccValue / BWTSaValue / LT), and against digests of the reference's results (tests/conftest.py), which are all
that is checked where oracle/_ref is not built.  There the tests on the 300 kbp index need a GPU for bin/2bwt-builder and skip
without one."""
import numpy as np
import pytest

from conftest import make_reads, load_pairs, run_ref_soap4, have_ref, check_reference_digest
from oracle import pyoracle as po


def test_index_primitives_match_reference(small_ref):
    ix = po.Index(small_ref["prefix"])
    assert ix.n == 300000
    rng = np.random.default_rng(1)
    idx = np.concatenate([rng.integers(0, ix.n + 2, size=20000), [0, 1, ix.inverse_sa0, ix.inverse_sa0 + 1, ix.n, ix.n + 1]]).astype(np.uint64)
    c = rng.integers(0, 4, size=len(idx)).astype(np.uint32)
    sidx = np.concatenate([rng.integers(0, ix.n + 1, size=5000), [0, ix.inverse_sa0, ix.n]]).astype(np.uint64)
    keys = rng.integers(0, 4 ** 13, size=2000).astype(np.uint32)
    got_lkt = [ix.lkt(k) for k in keys[:300]]
    if have_ref():
        rx = po.RefIndex(small_ref["prefix"])
        assert rx.n == 300000
        assert (ix.occ(idx, c) == rx.occ(idx, c)).all()
        assert (ix.sa(sidx) == rx.sa(sidx)).all()
        l, r = rx.lkt(keys)
        for got, a, b in zip(got_lkt, l, r):
            assert got == (a, b)
    check_reference_digest("index primitives", ix.occ(idx, c).tobytes() + ix.sa(sidx).tobytes() + repr(got_lkt).encode())


def check_dp_against_reference(key, refs, dl, reads, rl, maxdna, maxread, clips, mm=-2, go=-3):
    """the restatement on every task against the reference's callDP (libref_dp.so), or against the digest of its results
    -> the reference's (score, hit offset, tie count, pattern) per task"""
    got = []
    for t in range(len(dl)):
        co = po.dp_cutoff(int(rl[t]))
        got.append(po.dp(refs[t, :dl[t]], reads[t, :rl[t]], clips[0], clips[1], mm, go, co))
    if have_ref():
        sc, hl, mc, pats = po.ref_dp(refs, dl, reads, rl, maxdna, maxread, clips[0], clips[1], mm, go)
        for t in range(len(dl)):
            want = (int(sc[t]), int(hl[t]), int(mc[t]), po.pattern_bytes(pats[t]) if sc[t] >= po.dp_cutoff(int(rl[t])) else b"")
            assert got[t] == want, (key, t, got[t], want)
    check_reference_digest("callDP " + key, repr(got).encode())
    return got


def random_dp_tasks(rng, n, maxdna, maxread, fixed=False):
    refs = np.zeros((n, maxdna), np.uint8)
    reads = np.zeros((n, maxread), np.uint8)
    dl = np.zeros(n, np.uint32)
    rl = np.zeros(n, np.uint32)
    for t in range(n):
        L = maxread - 2 if fixed else int(rng.integers(30, maxread + 1))
        alpha = 4 if rng.random() < 0.7 else 2          # low complexity -> many tied maxima
        rd = rng.integers(0, alpha, size=L).astype(np.uint8)
        body = list(rd)
        if rng.random() < 0.5:                           # forces soft clipping at one end
            k = int(rng.integers(1, 40))
            body = body[k:] if rng.random() < 0.5 else body[:-k]
        out = []
        for ch in body:
            r = rng.random()
            if r < 0.03:
                continue
            if r < 0.06:
                out.append(int(rng.integers(0, alpha)))
            if rng.random() < 0.06:
                ch = int(rng.integers(0, alpha))
            out.append(int(ch))
        w = list(rng.integers(0, alpha, size=int(rng.integers(0, 40)))) + out + list(rng.integers(0, alpha, size=int(rng.integers(0, 40))))
        if rng.random() < 0.1:
            w = list(rng.integers(0, 4, size=int(rng.integers(0, maxdna))))
        w = w[:maxdna]
        refs[t, :len(w)] = w
        dl[t] = len(w)
        reads[t, :L] = rd
        rl[t] = L
    return refs, dl, reads, rl


DP_SHAPES = [(220, 152, False, (130, 130)), (220, 152, True, (130, 130)), (160, 104, False, (130, 130)),
             (320, 252, False, (130, 130)), (752, 152, False, (130, 130)), (220, 152, False, (10, 20)), (220, 152, False, (0, 0))]


def exact_occurrence_tasks(rng, n, maxdna, maxread):
    """DP tasks whose read occurs WITHOUT any difference in the reference window: at offset 0, at the last offset, in the
    middle, several times (tandem / homopolymer windows), next to near-misses -- the cases the CUDA path answers without
    running the DP (k_dp_exact), so both the restatement and the CUDA path are pinned on them."""
    refs = np.zeros((n, maxdna), np.uint8)
    reads = np.zeros((n, maxread), np.uint8)
    dl = np.zeros(n, np.uint32)
    rl = np.zeros(n, np.uint32)
    for t in range(n):
        L = int(rng.integers(30, maxread + 1))
        kind = t % 8
        if kind == 5:                                    # homopolymer read in a homopolymer window: one occurrence per offset
            rd = np.full(L, int(rng.integers(0, 4)), np.uint8)
        elif kind == 6:                                  # short period: occurrences every `per` bases
            per = int(rng.integers(2, 6))
            rd = np.resize(rng.integers(0, 4, size=per).astype(np.uint8), L)
        else:
            rd = rng.integers(0, 4, size=L).astype(np.uint8)
        room = maxdna - L
        if kind == 0:
            left, right = 0, int(rng.integers(0, room + 1))                  # occurrence at the window start (row 0 reached)
        elif kind == 1:
            left, right = int(rng.integers(0, room + 1)), 0                  # ... at the window end
        elif kind == 2:
            left, right = 0, 0                                               # window == read
        else:
            left = int(rng.integers(0, room + 1)); right = int(rng.integers(0, room - left + 1))
        if kind in (5, 6):
            w = np.resize(rd[:per] if kind == 6 else rd[:1], left + L + right)
            if kind == 6:
                w = np.roll(w, left % per)               # keep an occurrence at `left`
        else:
            w = np.concatenate([rng.integers(0, 4, size=left), rd, rng.integers(0, 4, size=right)]).astype(np.uint8)
        if kind == 7 and left + L + right >= L + 1:      # a near-miss: one substitution, no exact occurrence (control)
            w = w.copy(); w[left + int(rng.integers(0, L))] ^= 1
        refs[t, :len(w)] = w
        dl[t] = len(w)
        reads[t, :L] = rd
        rl[t] = L
    return refs, dl, reads, rl


@pytest.mark.parametrize("clips", [(130, 130), (10, 20), (0, 0)])
def test_dp_exact_occurrences_match_reference_callDP(clips):
    rng = np.random.default_rng(977 + clips[0])
    n, maxdna, maxread = 192, 220, 152
    refs, dl, reads, rl = exact_occurrence_tasks(rng, n, maxdna, maxread)
    want = check_dp_against_reference("exact %d %d" % clips, refs, dl, reads, rl, maxdna, maxread, clips)
    assert sum(want[t][0] == int(rl[t]) for t in range(n)) > n // 2


@pytest.mark.parametrize("mm,go", [(-3, -2), (-4, -6), (-2, -6), (-3, -3), (-4, -3)])
def test_dp_other_score_parameters_match_reference_callDP(mm, go):
    """the restatement against the reference's own callDP for the score range it accepts (CPU_DP.cpp:199-208)"""
    rng = np.random.default_rng(100 - mm * 7 - go)
    n, maxdna, maxread = 160, 220, 152
    refs, dl, reads, rl = random_dp_tasks(rng, n, maxdna, maxread, False)
    check_dp_against_reference("scores %d %d" % (mm, go), refs, dl, reads, rl, maxdna, maxread, (130, 130), mm, go)


@pytest.mark.parametrize("maxdna,maxread,fixed,clips", DP_SHAPES)
def test_dp_matches_reference_callDP(maxdna, maxread, fixed, clips):
    rng = np.random.default_rng(maxdna * 7 + maxread + clips[0])
    n = 192
    refs, dl, reads, rl = random_dp_tasks(rng, n, maxdna, maxread, fixed)
    want = check_dp_against_reference("shape %d %d %d %d %d" % (maxdna, maxread, fixed, clips[0], clips[1]), refs, dl, reads, rl, maxdna, maxread, clips)
    assert sum(want[t][0] >= po.dp_cutoff(int(rl[t])) for t in range(n)) > n // 4


@pytest.mark.parametrize("name,rlen,lopt,kw", [
    ("clean", 150, 151, dict(model="clean")),
    ("div", 100, 101, dict(model="divergent", one_random=0.05, unalignable=0.02)),
    ("var", 150, 151, dict(model="clean", varlen=True, n_rate=0.002)),
])
def test_seeds_candidates_dp_match_reference_dumps(workdir, small_ref, name, rlen, lopt, kw):
    fq1, fq2 = make_reads(workdir, small_ref, name, 1500, rlen, seed=11, **kw)
    reads, lens = load_pairs(fq1, fq2, trunc=lopt - 1)
    ix = po.Index(small_ref["prefix"])
    rp, mp = ix.seed_pairs(reads, lens, po.mmp_params())
    # first-batch clamp of insert_low (SOAP4.cpp:465-474): default -v 1 -> max(1, detected lengths)
    insert_low = max(1, ref_detected_len(lens[0::2]), ref_detected_len(lens[1::2]))
    cands = po.pair_candidates(rp, mp, lens, insert_low, 750)
    assert len(cands) > 500
    # the reference's SeedPos arrays and CandidateInfo list, as a digest; its DP task dump is not stored here: DP tasks the
    # reference's pipeline dumped are checked against the restatement by test_golden.py (committed seam dumps of three read sets)
    check_reference_digest("seam dumps " + name, rp.tobytes() + mp.tobytes() + cands.tobytes())
    if not have_ref():
        return
    _, dump = run_ref_soap4(workdir, small_ref["prefix"], fq1, fq2, "ref_" + name, lopt)
    (drp, dmp), = po.read_seedpos_dump(dump + "/seedpos.bin")
    assert rp.tobytes() == drp.tobytes() and mp.tobytes() == dmp.tobytes()
    dc, = po.read_cand_dump(dump + "/cand.bin")
    assert cands.tobytes() == dc.tobytes()
    ntask = 0
    for rec in po.read_dp_dump(dump + "/dp.bin"):
        for (ref, rd, co, sc, hl, mc, pat) in rec["tasks"][:400]:
            got = po.dp(ref, rd, rec["clip_lt"], rec["clip_rt"], rec["mismatch"], rec["gap_open"], co)
            assert got == (sc, hl, mc, pat)
            ntask += 1
    assert ntask > 500


def ref_detected_len(lens):
    """GetReadLength (QueryParser.cpp:2253-2277): maximum over the first 999999 sampled reads."""
    return int(lens[:999999].max())


def closed_form_for_exact_occurrence(ref, read, cutoff):
    """What k_dp_exact writes (megapath_b200/csrc/mp_dp.cu) when `read` occurs unchanged in `ref`; None otherwise."""
    N, L = len(ref), len(read)
    if L == 0 or N < L or cutoff > L or cutoff <= 0:
        return None
    rb, qb = ref.tobytes(), read.tobytes()
    occ, first, at = 0, -1, rb.find(qb)
    while at >= 0:
        occ += 1
        if first < 0:
            first = at
        at = rb.find(qb, at + 1)
    if occ == 0:
        return None
    pat = b"M" * L + (b"SV\x00" if first == 0 else b"")
    return (L, first, min(occ, 255), pat)


def test_exact_occurrence_closed_form_equals_the_dp():
    """The theorem behind k_dp_exact, checked on thousands of tasks against the DP restatement (which the tests above pin to
    the reference's callDP): low-complexity alphabets give windows with many occurrences and near-occurrences."""
    rng = np.random.default_rng(20260)
    checked = multi = at_start = 0
    for trial in range(4000):
        alpha = int(rng.integers(1, 5))
        L = int(rng.integers(30, 153))
        N = int(rng.integers(L, 221))
        read = rng.integers(0, alpha, size=L).astype(np.uint8)
        ref = rng.integers(0, alpha, size=N).astype(np.uint8)
        if rng.random() < 0.8:                                    # plant one occurrence (others may exist by chance / periodicity)
            o = int(rng.integers(0, N - L + 1)) if rng.random() < 0.8 else 0
            ref[o:o + L] = read
        clips = [(130, 130), (0, 0), (10, 20), (5, 0), (0, 130)][trial % 5]
        cutoff = po.dp_cutoff(L)
        want = closed_form_for_exact_occurrence(ref, read, cutoff)
        if want is None:
            continue
        got = po.dp(ref, read, clips[0], clips[1], -2, -3, cutoff)
        got = (got[0], got[1], got[2], got[3])
        # pattern_bytes (the comparison form used by the other tests) ends at the first NUL: compare in that form
        assert got == (want[0], want[1], want[2], want[3].split(b"\x00")[0] if isinstance(got[3], bytes) and b"\x00" not in got[3] else want[3]), (trial, clips, got, want)
        checked += 1
        multi += want[2] > 1
        at_start += want[1] == 0
    assert checked > 2500 and multi > 300 and at_start > 300


# ---- the stdout contract's SCORE: header with comment chaining, pinned against the reference binary run here (CPU) ----
def _headers(stdout_fastq):
    """annotated FASTQ -> {(name, mate index within its pair): header line}"""
    lines = stdout_fastq.split(b"\n")
    recs = [lines[i] for i in range(0, len(lines) - 3, 4)]
    out = {}
    for k in range(0, len(recs) - 1, 2):
        for mate in (0, 1):
            out[(recs[k + mate][1:].split(b"\t")[0], mate)] = recs[k + mate]
    return out


@pytest.mark.parametrize("mode", ["-F", "-P"])
def test_fastq_header_restatement_matches_reference_chaining(workdir, small_ref, second_ref, mode):
    """oracle/pyoracle.fastq_header (getMappingFromHeader + the header composition of pairDeepDPOutputFastqAPI /
    unproperlypairDPOutputFastqAPI, BGS-IO.cpp:1348-1446, 1966-2091) against the reference itself: the reference's chunk-1 header
    WITHOUT -nc must be what the restatement makes of (its chunk-1 header WITH -nc = this run's own hits, the comment it was fed)."""
    import os
    from conftest import make_reads, run_ref_raw, deinterleave
    from oracle import pyoracle as po

    def edit(k, mate, comm):
        if k % 19 == 3:
            return b"IGNORE"
        if k % 23 == 5 and mate == 1:
            return b"SCORE:0;"
        if k % 29 == 7:
            return b"SCORE:400;400,made_up_hit;"
        if k % 31 == 11 and mate == 0:
            return b""
        if k % 41 == 17:
            return b"SCORE:  +12;12,x y z;9,low;"
        if k % 43 == 19:
            return b"SCORE:99999999999999999999;5,big;"
        return comm
    fq1, fq2 = make_reads(workdir, small_ref, "hdr", 2000, 150, seed=79, model="divergent", one_random=0.10, unalignable=0.04)
    first = run_ref_raw(workdir, small_ref["prefix"], fq1, fq2, "hdr0", 151, "soap4-nt2.ini", ["-F", "-nc", "-top", "95"])
    in1, in2 = deinterleave(first, os.path.join(workdir, "hdr_in"), edit)
    own = _headers(run_ref_raw(workdir, second_ref["prefix"], in1, in2, "hdr_own", 151, "soap4-nt2.ini", [mode, "-nc", "-top", "95"]))
    chained = _headers(run_ref_raw(workdir, second_ref["prefix"], in1, in2, "hdr_ch", 151, "soap4-nt2.ini", [mode, "-top", "95"]))
    comments = {}
    for mate, path in ((0, in1), (1, in2)):
        for line in open(path, "rb").read().split(b"\n")[0::4]:
            if line:
                parts = line[1:].split(None, 1)
                nm = parts[0][:-2] if parts[0][-2:] in (b"/1", b"/2") else parts[0]
                comments[(nm, mate)] = parts[1] if len(parts) > 1 else None
    assert len(own) == len(chained) == 4000
    n_merged = 0
    for key, hdr in own.items():
        name, tail = hdr[1:].split(b"\t", 1)
        assert tail.startswith(b"SCORE:")
        fields = tail[6:].split(b";")[:-1]
        own_best = int(fields[0])
        # this run's hits as the header lists them: one per sequence, ascending sequence order (names stand in for the ids)
        hits = [(i + 1, int(f.split(b",", 1)[0]), f.split(b",", 1)[1]) for i, f in enumerate(fields[1:])]
        want = chained[key]
        got = po.fastq_header(name, comments[key], own_best, hits, 0.95)
        assert got == want, (key, comments[key], hdr, got, want)
        n_merged += want != hdr
    assert n_merged > 500                  # the previous comment changed the header of many reads
