"""GPU suite: the DP path the alignment stages take (mp_dp_tasks -> k_dp_prepare -> k_dp_fill / k_dp_tb), which gathers each task's
window from the packed text and its read from the uploaded batch into packed rows of 16 bases per word, against the CPU oracle.
The cases sit where the packing can go wrong: window starts at every residue mod 16, the first and the last text base, reads
reverse-complemented across word boundaries, exact occurrences at both window ends and in repeats, differences only in the last
base of a word, rescue-sized windows, dropped tasks, and the exact-occurrence shortcut switched off."""
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
from oracle import pyoracle as po  # noqa: E402

pytestmark = pytest.mark.gpu

TEXT_LEN = 70013                 # not a multiple of 16: the last window word of a window ending at the last base is partial
HOMO, TANDEM = (10000, 400), (20000, 600)


def make_text():
    rng = np.random.default_rng(2024)
    t = rng.integers(0, 4, size=TEXT_LEN).astype(np.uint8)
    t[HOMO[0]:HOMO[0] + HOMO[1]] = 0
    t[TANDEM[0]:TANDEM[0] + TANDEM[1]] = np.resize(np.array([1, 2, 2, 3, 0], np.uint8), TANDEM[1])
    return t


def revcomp(x):
    return (3 - x[::-1]).astype(np.uint8)


def cutoff_for(L):
    return max(1, min(po.dp_cutoff(L), L))


class Cases:
    """tasks of one mp_dp_tasks call; the read of every task is its own batch read"""

    def __init__(self, text, rng):
        self.text, self.rng, self.tasks, self.reads, self.want = text, rng, [], [], []

    def add(self, ref_start, ref_len, oriented, strand, valid=1, drop=False, read_len=None):
        stored = oriented if strand == 1 else revcomp(oriented)
        L = len(oriented) if read_len is None else read_len
        cut = cutoff_for(max(L, 1))
        self.tasks.append((ref_start, ref_len, len(self.reads), L, strand, valid, cut, int(self.rng.integers(-1, 60)), 0))
        self.reads.append(stored)
        if drop or not valid:
            self.want.append((0, 0, 0, b""))
        else:
            self.want.append(po.dp(self.text[ref_start:ref_start + ref_len], oriented, 130, 130, -2, -3, cut))

    def mutated(self, seg, n_sub):
        r = seg.copy()
        for p in self.rng.choice(len(r), size=min(n_sub, len(r)), replace=False):
            r[p] = (r[p] + 1 + self.rng.integers(0, 3)) % 4
        return r

    def run(self, ctx, max_ref, max_read):
        import megapath_b200 as mp
        reads = list(self.reads) + ([np.zeros(1, np.uint8)] if len(self.reads) % 2 else [])
        width = max(len(r) for r in reads)
        codes = np.zeros((len(reads), width), np.uint8)
        lens = np.array([len(r) for r in reads], np.uint32)
        for i, r in enumerate(reads):
            codes[i, :len(r)] = r
        q, wpq = mp.pack_queries(codes, lens, 336)
        ctx.batch_upload(q, lens, wpq)
        tasks = np.array(self.tasks, dtype=mp.DP_TASK)
        sc, hl, mc, pats = ctx.dp_tasks(tasks, max_ref, max_read)
        bad = []
        for t, want in enumerate(self.want):
            got = (int(sc[t]), int(hl[t]), int(mc[t]), po.pattern_bytes(pats[t]) if sc[t] > 0 and sc[t] >= tasks[t]["cutoff"] else b"")
            if got != want:
                bad.append((t, self.tasks[t][:6], got, want))
        return bad


@pytest.fixture(scope="module")
def ctx():
    import megapath_b200 as mp
    text = make_text()
    c = mp.Context(0)
    c.index_build(mp.pack_text(text), TEXT_LEN)
    c.text = text
    yield c
    c.close()


def window_cases(text, rng):
    """window starts at every residue mod 16, at text position 0 and ending at the last text base; both strands"""
    cs = Cases(text, rng)
    N = 220
    starts = [int(rng.integers(100, TEXT_LEN // 16 - 100)) * 16 + r for r in range(16)] + [0, TEXT_LEN - N]
    for i, s in enumerate(starts):
        for strand in (1, 2):
            L = int(rng.integers(90, 153))
            off = int(rng.integers(0, N - L + 1))
            seg = text[s + off:s + off + L]
            cs.add(s, N, seg.copy() if i % 3 == 0 else cs.mutated(seg, 1 + i % 4), strand)
    # the read at both window ends exactly, and a window that ends at the last text base with the read at its end
    for s in (0, TEXT_LEN - N, 4099):
        for strand in (1, 2):
            cs.add(s, N, text[s:s + 150].copy(), strand)
            cs.add(s, N, text[s + N - 150:s + N].copy(), strand)
    return cs


def test_gpu_dp_packed_windows(ctx):
    cs = window_cases(ctx.text, np.random.default_rng(5))
    assert cs.run(ctx, 220, 152) == []


@pytest.mark.parametrize("max_read,lengths", [(160, (1, 15, 16, 17, 31, 32, 33, 150)), (256, (250, 161)), (320, (320, 300, 257))])
def test_gpu_dp_packed_read_lengths(ctx, max_read, lengths):
    """strand-2 reads (and strand 1 for contrast) at word-boundary lengths, for K = 5 / 8 / 10"""
    text, rng = ctx.text, np.random.default_rng(max_read)
    cs = Cases(text, rng)
    N = max_read + 80
    for L in lengths:
        for rep in range(6):
            s = int(rng.integers(30000, TEXT_LEN - N))
            off = int(rng.integers(0, N - L + 1))
            seg = text[s + off:s + off + L]
            cs.add(s, N, seg.copy() if rep < 2 else cs.mutated(seg, 1 + rep % 3), 2 if rep % 3 else 1)
    assert cs.run(ctx, N, max_read) == []


def occurrence_cases(text, rng):
    cs = Cases(text, rng)
    N = 220
    # homopolymer and tandem windows: dozens of occurrences
    for L in (40, 100, 150):
        cs.add(HOMO[0] + 50, N, np.zeros(L, np.uint8), 1)
        cs.add(HOMO[0] + 50, N, np.full(L, 3, np.uint8), 2)          # reverse complement of T...T is A...A
        seg = text[TANDEM[0] + 7:TANDEM[0] + 7 + L]
        cs.add(TANDEM[0] + 100, N, seg.copy(), 1)
        cs.add(TANDEM[0] + 100, N, seg.copy(), 2)
    # the read at window offset 0 and at N - L, in random text
    for strand in (1, 2):
        for L in (31, 64, 100, 152):
            s = int(rng.integers(30000, 60000))
            cs.add(s, N, text[s:s + L].copy(), strand)
            cs.add(s, N, text[s + N - L:s + N].copy(), strand)
    # near-misses: the only difference is the last base of a 16-base word of the read
    for strand in (1, 2):
        for L in (48, 100, 150):
            for last in range(15, L, 16):
                s = int(rng.integers(30000, 60000))
                off = int(rng.integers(0, N - L + 1))
                r = text[s + off:s + off + L].copy()
                r[last] = (r[last] + 1) % 4
                cs.add(s, N, r, strand)
    return cs


def test_gpu_dp_packed_exact_occurrences(ctx):
    cs = occurrence_cases(ctx.text, np.random.default_rng(11))
    assert cs.run(ctx, 220, 152) == []


def test_gpu_dp_packed_rescue_windows_and_dropped_tasks(ctx):
    """752-row windows of mate rescue; invalid tasks and tasks longer than the call's maxima are dropped, never read"""
    text, rng = ctx.text, np.random.default_rng(17)
    cs = Cases(text, rng)
    N = 752
    for i in range(24):
        s = int(rng.integers(0, TEXT_LEN - N)) if i else TEXT_LEN - N
        L = int(rng.integers(100, 153))
        off = int(rng.integers(0, N - L + 1))
        seg = text[s + off:s + off + L]
        cs.add(s, N, seg.copy() if i % 4 == 0 else cs.mutated(seg, 1 + i % 5), 1 + i % 2)
    s = 40000
    cs.add(s, N, text[s:s + 150].copy(), 1, valid=0)
    cs.add(s, N + 1, text[s:s + 150].copy(), 2, drop=True)                     # window longer than maxRefLen
    cs.add(s, N, text[s:s + 150].copy(), 1, drop=True, read_len=153)           # read longer than maxReadLen
    cs.add(s, N, text[s:s + 150].copy(), 2)
    assert cs.run(ctx, N, 152) == []


def _all_cases(ctx):
    bad = []
    bad += window_cases(ctx.text, np.random.default_rng(5)).run(ctx, 220, 152)
    bad += occurrence_cases(ctx.text, np.random.default_rng(11)).run(ctx, 220, 152)
    return bad


def test_gpu_dp_packed_without_exact_shortcut():
    """MP_DP_EXACT=0 sends every task through k_dp_fill / k_dp_tb; the library reads it once per process, hence a process of its own"""
    env = dict(os.environ, MP_DP_EXACT="0")
    r = subprocess.run([sys.executable, "-s", os.path.abspath(__file__)], env=env, cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-4000:] + r.stderr[-4000:]
    assert "ok" in r.stdout


if __name__ == "__main__":
    import megapath_b200 as mp
    text = make_text()
    c = mp.Context(0)
    c.index_build(mp.pack_text(text), TEXT_LEN)
    c.text = text
    bad = _all_cases(c)
    c.close()
    if bad:
        print(bad[:20])
        sys.exit(1)
    print("ok")
