"""CPU suite: the restatement of the device BGZF encoder (oracle/pybgzf.py) against zlib, against an independent DEFLATE parser
(pybgzf.parse_member), against Huffman builds that share no code with the kernel's, and against an independent bit count of the three
encodings; plus proof that the adversarial corpus below reaches every branch of mp_bgzf.cu it is meant to reach: length limiting of
the literal/length tree and of the code-length tree, all three block types, every length and distance code, the window edge.

tests/test_gpu_bgzf.py holds the device to this model byte for byte on the same corpus."""
import functools
import gzip
import heapq
import itertools
import zlib
from fractions import Fraction

import numpy as np
import pytest

from oracle import pybgzf

PIECE = pybgzf.PIECE


# ---- the adversarial corpus: seeded generators ----

def fib(k):
    f = [1, 1]
    while len(f) < k:
        f.append(f[-1] + f[-2])
    return f[:k]


def fibonacci_literals(seed=0):
    """byte counts F1..F22 in shuffled order (46 367 bytes, one piece): unrestricted depth 21 on the bytes alone.  The matches the
    dominant bytes make take the literal tree back to depth 13-14; fibonacci_tail reaches past 15."""
    rng = np.random.default_rng(seed)
    data = np.repeat(rng.permutation(256)[:22], fib(22))
    rng.shuffle(data)
    return data.astype(np.uint8).tobytes()


def without_repeats(seq, alphabet, rng, fixed=None):
    """seq (list of byte values) with a byte re-drawn from `alphabet` wherever a 3-byte string would repeat, so that the encoder finds
    no match in it; positions where `fixed` is set keep their byte"""
    seen = set()
    for i in range(2, len(seq)):
        g = (seq[i - 2], seq[i - 1], seq[i])
        while g in seen and (fixed is None or not fixed[i]):
            seq[i] = int(alphabet[rng.integers(0, len(alphabet))])
            g = (seq[i - 2], seq[i - 1], seq[i])
        seen.add(g)
    return seq


def background(rng, n=PIECE):
    return without_repeats(rng.integers(0, 256, n).tolist(), np.arange(256), rng)


def fibonacci_tail(k=12, seed=1):
    """one piece: bytes with counts F2..Fk over a background of the other bytes that has no repeated 3-byte string.  With the EOB as
    the second count of 1 the literal/length histogram is a Fibonacci chain below an even bulk: unrestricted depth 18, so the tree
    must be limited to 15.  (Counts F1, F1 beside the EOB would pair up level by level and stay at depth 14.)"""
    rng = np.random.default_rng(seed)
    perm = rng.permutation(256)
    tail, bulk = perm[:k - 1], perm[k - 1:]
    counts = fib(k)[1:]
    seq = bulk[rng.integers(0, len(bulk), PIECE)]
    pos = rng.choice(PIECE, sum(counts), replace=False)
    seq[pos] = np.repeat(tail, counts)
    fixed = np.zeros(PIECE, bool)
    fixed[pos] = True
    return bytes(without_repeats(seq.tolist(), bulk, np.random.default_rng(seed + 1000), fixed))


def code_length_fibonacci(seed):
    """one piece whose literal code lengths take eleven values with Fibonacci multiplicities (1, 1, 2, ... 89 symbols), the symbols
    of equal length scattered over the byte values so that they do not form 16-runs: the code-length code's histogram is then a
    Fibonacci-like chain too"""
    rng = np.random.default_rng(seed)
    mult = {4: 1, 5: 1, 6: 2, 7: 3, 8: 5, 9: 8, 10: 13, 11: 21, 12: 34, 13: 55, 14: 89}
    lens = np.concatenate([[l] * m for l, m in mult.items()])
    w = 2.0 ** -lens.astype(float)
    cnt = np.maximum(1, np.round(w / w.sum() * PIECE)).astype(int)
    data = np.repeat(rng.permutation(256)[:len(lens)], cnt)[:PIECE]
    rng.shuffle(data)
    return data.astype(np.uint8).tobytes()


@functools.lru_cache(None)
def deep_code_length_code():
    """deterministic seeded search with plan(): the first seed whose code-length code needs the 7-bit limit"""
    for seed in range(64):
        data = code_length_fibonacci(seed)
        if pybgzf.plan(data)["cl_depth"] > 7:
            return data
    raise AssertionError("no seed below 64 gives a code-length tree deeper than 7")


def _h3(b):
    b = np.frombuffer(bytes(b), np.uint8).astype(np.uint64)
    w3 = b[:-2] | b[1:-1] << 8 | b[2:] << 16
    return ((w3 * 2654435761) & 0xffffffff) >> (32 - pybgzf.HASH_BITS)


def _h4(b):
    b = np.frombuffer(bytes(b), np.uint8).astype(np.uint64)
    w4 = b[:-3] | b[1:-2] << 8 | b[2:-1] << 16 | b[3:] << 24
    return ((w4 * 2246822519) & 0xffffffff) >> (32 - pybgzf.HASH_BITS)


def _plant(buf, t, d, L):
    """copies buf[t-d : t-d+L] to t (byte by byte, so overlapping copies repeat) and makes the byte after the copy differ; True if
    the head tables will hold the source when t's tile is matched: no later position of an earlier tile shares its 3-byte (or its
    4-byte) hash, and the copy cannot start a byte earlier.  Otherwise buf is left as it was."""
    s, tile = t - d, t - t % pybgzf.TILE
    if d >= pybgzf.TILE and buf[t - 1] == buf[s - 1]:
        return False
    old = bytes(buf[t:t + L + 1])
    for k in range(L):
        buf[t + k] = buf[s + k]
    buf[t + L] = (buf[s + L] + 1 + buf[t + L] % 255) & 0xff
    h3, h4 = _h3(buf[s:tile + 2]), _h4(buf[s:tile + 3])
    fresh = buf.find(buf[t - 2:t + 1]) == t - 2 and buf.find(buf[t - 1:t + 2]) == t - 1     # no chance match across the start
    if fresh and (not (h3[1:tile - s] == h3[0]).any() or not (h4[1:tile - s] == h4[0]).any()):
        return True
    buf[t:t + L + 1] = old
    return False


@functools.lru_cache(None)
def every_length_and_distance_code(seed=3):
    """three pieces of background without repeated 3-byte strings; at the start of nearly every tile a copy, of every length 3..258
    in turn, from a distance that walks the 30 distance codes (rising with the tile, so that the far codes come where the piece is
    long enough), with a random extra-bits value"""
    rng = np.random.default_rng(seed)
    out = bytearray()
    lengths = iter(range(3, 259))
    for _ in range(3):
        buf = bytearray(background(rng))
        for k in range(1, 127):
            L = next(lengths, None)
            if L is None:
                break
            t = k * pybgzf.TILE
            c = (k - 1) * 30 // 126
            lo, hi = int(pybgzf.DIST_BASE[c]), int(pybgzf.DIST_BASE[c]) + (1 << int(pybgzf.DIST_EXTRA[c])) - 1
            for _ in range(64):
                if _plant(buf, t, int(rng.integers(lo, min(hi, t) + 1)), L):
                    break
        out += buf
    return bytes(out)


@functools.lru_cache(None)
def window_edge_copies(distance, seed=5):
    """one piece of background without repeated 3-byte strings with two 40-byte copies from exactly `distance` back: one whose source
    and target start a tile (position = 0 mod 512) and one whose source and target end a tile (= 511 mod 512); at 32769 the sources
    are on the same tile edges and the targets one byte further.  At 32768 (the DEFLATE window) both must be emitted as copies, at
    32769 neither."""
    rng = np.random.default_rng(seed)
    for _ in range(64):
        buf = bytearray(background(rng))
        t0 = 70 * pybgzf.TILE
        t1 = 110 * pybgzf.TILE + 511
        if _plant(buf, t0 + (distance - 32768), distance, 40) and _plant(buf, t1 + (distance - 32768), distance, 40):
            return bytes(buf)
    raise AssertionError("no seed plants both copies")


WINDOW_TARGETS = {32768: (70 * 512, 110 * 512 + 511), 32769: (70 * 512 + 1, 110 * 512 + 512)}


def hash_collisions(seed=7):
    """one piece built from 40 3-byte words that share one 3-byte hash and 40 4-byte words that share one 4-byte hash, in random
    order: most positions find a candidate in the head tables whose bytes differ"""
    rng = np.random.default_rng(seed)
    w = rng.integers(0, 1 << 32, 1 << 23, dtype=np.uint64)
    h3 = ((w & 0xffffff) * 2654435761 & 0xffffffff) >> 18
    h4 = (w * 2246822519 & 0xffffffff) >> 18
    words3 = np.unique(w[h3 == h3[0]] & 0xffffff)[:40]
    words4 = np.unique(w[h4 == h4[0]])[:40]
    out = bytearray()
    while len(out) < PIECE:
        if rng.random() < 0.5:
            out += int(words3[rng.integers(0, len(words3))]).to_bytes(3, "little")
        else:
            out += int(words4[rng.integers(0, len(words4))]).to_bytes(4, "little")
    return bytes(out[:PIECE])


def is_cost_edge(which, Q):
    dyn, fixed, stored = Q["dyn_bits"], Q["fixed_bits"], Q["stored_bits"]
    if which == "tie":                  # dynamic == fixed: the tie goes to dynamic
        return dyn == fixed and dyn < stored
    if which == "eob_dynamic":          # fixed wins by fewer bits than its EOB code (7)
        return fixed - 7 < dyn < fixed and dyn < stored
    return stored <= fixed < stored + 7 and dyn >= stored      # "eob_stored": stored wins by fewer bits than the EOB


@functools.lru_cache(None)
def cost_edge(which):
    """deterministic seeded search with plan() for a short piece whose block costs sit where a wrong tie rule or a cost without the
    EOB code changes the choice (is_cost_edge).  Letters from a small alphabet for the two dynamic/fixed edges; bytes >= 144 (9-bit
    fixed codes) for the fixed/stored edge."""
    for seed in range(100000):
        rng = np.random.default_rng(seed)
        if which == "eob_stored":
            data = rng.integers(144, 256, int(rng.integers(25, 41))).astype(np.uint8).tobytes()
        else:
            n, a = int(rng.integers(8, 200)), int(rng.integers(2, 40))
            data = (rng.integers(0, a, n) + 97).astype(np.uint8).tobytes()
        if is_cost_edge(which, pybgzf.plan(data)):
            return data
    raise AssertionError("no seed below 100000 gives a %s piece" % which)


EDGE_SIZES = [1, 2, 3, 4, 5, 511, 512, 513, 1023, 1024, 1025, PIECE - 512, PIECE - 511, PIECE - 1, PIECE]


def corpus_input(name):
    if name == "fibonacci_literals":
        return fibonacci_literals()
    if name == "fibonacci_tail":
        return fibonacci_tail()
    if name == "code_length_limit":
        return deep_code_length_code()
    if name == "every_code":
        return every_length_and_distance_code()
    if name.startswith("window_"):
        return window_edge_copies(int(name[7:]))
    if name == "hash_collisions":
        return hash_collisions()
    if name.startswith("cost_"):
        return cost_edge(name[5:])
    kind, size = name.split("_")
    from test_gpu_bgzf import contents
    return contents(kind, int(size))


CORPUS = (["fibonacci_literals", "fibonacci_tail", "code_length_limit", "every_code", "window_32768", "window_32769", "hash_collisions",
           "cost_tie", "cost_eob_dynamic", "cost_eob_stored"]
          + ["fastq_%d" % n for n in EDGE_SIZES] + ["random_%d" % n for n in (3, 4, 5, 512, 513)]
          + ["%s_%d" % (k, 2 * PIECE + 3) for k in ("zeros", "repeat", "random", "skewed", "all256", "bam", "fastq")])


@functools.lru_cache(None)
def model_of(name):
    """(input, model stream, [(piece, member bytes, plan, parse_member)])"""
    data = corpus_input(name)
    raw = pybgzf.compress(data)
    members = pybgzf.split_members(raw)
    rows = []
    for k, m in enumerate(members):
        piece = data[k * PIECE:(k + 1) * PIECE]
        rows.append((piece, m, pybgzf.plan(piece), pybgzf.parse_member(m)))
    return data, raw, rows


# ---- independent references: Huffman builds, the RFC 1951 code tables, a bit counter ----

def heap_huffman_cost(freq):
    """cost (sum of frequency x length) of a Huffman code built with a heap"""
    tick = itertools.count()
    h = [(f, next(tick)) for f in freq if f]
    heapq.heapify(h)
    cost = 0
    while len(h) > 1:
        a, _ = heapq.heappop(h)
        b, _ = heapq.heappop(h)
        cost += a + b
        heapq.heappush(h, (a + b, next(tick)))
    return cost


def package_merge_cost(freq, limit):
    """cost of an optimal code with lengths <= limit (Larmore & Hirschberg's package-merge)"""
    leaves = sorted(f for f in freq if f)
    n = len(leaves)
    level = [(f, np.eye(n, dtype=np.int64)[i]) for i, f in enumerate(leaves)]     # (weight, how often each leaf is in the item)
    merged = level
    for _ in range(limit - 1):
        pk = [(merged[i][0] + merged[i + 1][0], merged[i][1] + merged[i + 1][1]) for i in range(0, len(merged) - 1, 2)]
        merged = sorted(level + pk, key=lambda x: x[0])
    lens = sum(c for _, c in merged[:2 * n - 2])
    return int(np.dot(leaves, lens))


def padded(freq):
    """the histogram the kernel builds its tree from: at least two symbols, the lowest unused standing in at frequency 1"""
    f = [int(x) for x in freq]
    for s in range(len(f)):
        if sum(1 for x in f if x) >= 2:
            break
        if not f[s]:
            f[s] = 1
    return f


def _rfc_tables():
    """RFC 1951 3.2.5, written out from the table's rule: length codes 257..284 carry (code - 261) // 4 extra bits from code 265
    on, 285 is length 258; distance codes carry (code - 2) // 2 extra bits from code 4 on"""
    lsym, base = {}, 3
    for c in range(28):
        extra = max(0, (c - 4) // 4)
        for L in range(base, base + (1 << extra)):
            lsym[L] = (257 + c, extra)
        base += 1 << extra
    lsym[258] = (285, 0)
    dsym, base = [], 1
    for c in range(30):
        extra = max(0, (c - 2) // 2)
        dsym.append((base, c, extra))
        base += 1 << extra
    return lsym, dsym


LSYM, DSYM = _rfc_tables()


def dist_symbol(d):
    for base, c, extra in reversed(DSYM):
        if d >= base:
            return c, extra


def fixed_lit_len(s):
    return 8 if s < 144 else 9 if s < 256 else 7 if s < 280 else 8


def token_bits(tokens, lit_len, dist_len):
    bits = lit_len(256)
    for t in tokens:
        if isinstance(t, int):
            bits += lit_len(t)
        else:
            sym, lx = LSYM[t[0]]
            dc, dx = dist_symbol(t[1])
            bits += lit_len(sym) + lx + dist_len(dc) + dx
    return bits


def dynamic_header_bits(hclen, cl_lens, rle):
    return 3 + 5 + 5 + 4 + 3 * hclen + sum(cl_lens[s] + {16: 2, 17: 3, 18: 7}.get(s, 0) for s, _ in rle)


def kraft(lens):
    return sum(Fraction(1, 1 << l) for l in lens if l)


# ---- tests ----

@pytest.mark.parametrize("name", CORPUS)
def test_model_inflates_and_parses_to_the_input(name):
    data, raw, rows = model_of(name)
    assert gzip.decompress(raw) == data
    assert len(rows) == (len(data) + PIECE - 1) // PIECE
    for piece, m, _, P in rows:
        assert P["data"] == piece and P["isize"] == len(piece)
        assert P["crc"] == zlib.crc32(piece)
        assert len(m) <= 65536


@pytest.mark.parametrize("name", CORPUS)
def test_trees_are_complete_and_within_the_limits(name):
    for _, _, _, P in model_of(name)[2]:
        if P["btype"] != 2:
            continue
        for lens, limit in ((P["lit_lens"], 15), (P["dist_lens"], 15), (P["cl_lens"], 7)):
            used = [l for l in lens if l]
            assert max(used) <= limit, (lens, limit)
            assert kraft(used) == 1 or used == [1], ("Kraft sum %s" % kraft(used), lens)


@pytest.mark.parametrize("name", CORPUS)
def test_huffman_lengths_are_optimal(name):
    """without limiting: the cost of the heap-built Huffman code; with limiting: no better than package-merge's optimum"""
    for _, _, Q, _ in model_of(name)[2]:
        for freq, lens, depth, limit in ((Q["lit_freq"], Q["lit_lens"], Q["lit_depth"], 15), (Q["dist_freq"], Q["dist_lens"], Q["dist_depth"], 15),
                                         (Q["cl_freq"], Q["cl_lens"], Q["cl_depth"], 7)):
            f = padded(freq)
            cost = sum(a * int(b) for a, b in zip(f, lens))
            assert all(bool(a) == bool(b) for a, b in zip(f, lens))
            if depth <= limit:
                assert cost == heap_huffman_cost(f)
            else:
                best = package_merge_cost(f, limit)
                assert cost >= best
                print("%s: %d-bit limit from depth %d: cost %d, package-merge %d (gap %d bits)" % (name, limit, depth, cost, best, cost - best))


@pytest.mark.parametrize("name", CORPUS)
def test_chosen_block_is_the_smallest(name):
    """the decoded tokens re-encoded three ways and counted bit by bit: the emitted block is exactly as long as its count, and it is
    the smallest, dynamic winning a tie with fixed (dyn <= fixed && dyn < stored, else fixed < stored, else stored)"""
    for piece, _, Q, P in model_of(name)[2]:
        toks = P["tokens"]
        stored = 3 + 5 + 32 + 8 * len(piece)
        if P["btype"] == 0:                     # a stored block has no tokens: count the model's parse
            assert toks == list(piece)
            toks = [int(piece[p]) if not L else (int(L), int(D)) for p, L, D in zip(Q["starts"], Q["lengths"], Q["distances"])]
        fixed = 3 + token_bits(toks, fixed_lit_len, lambda c: 5)
        if P["btype"] == 2:
            lit, dist, cl, hclen, rle = P["lit_lens"], P["dist_lens"], P["cl_lens"], P["hclen"], P["rle"]
        else:
            lit, dist, cl, hclen, rle = Q["lit_lens"], Q["dist_lens"], Q["cl_lens"], Q["hclen"], Q["rle"]
        dyn = dynamic_header_bits(hclen, cl, rle) + token_bits(toks, lambda s: int(lit[s]), lambda c: int(dist[c]))
        assert P["block_bits"] == {0: stored, 1: fixed, 2: dyn}[P["btype"]]
        want = 2 if dyn <= fixed and dyn < stored else 1 if fixed < stored else 0
        assert P["btype"] == want, (name, dyn, fixed, stored)
        assert (Q["dyn_bits"], Q["fixed_bits"], Q["stored_bits"]) == (dyn, fixed, 8 * (5 + len(piece)))


def test_corpus_reaches_every_branch():
    """length limiting of the literal/length tree (pre-limit depth > 15) and of the code-length tree (> 7), all three block types,
    the tie and EOB cost edges, every length code 257..285 and distance code 0..29, distance 32768 and nothing further.

    The distance tree is not driven past 15 here (the corpus reaches 14).  That needs a Fibonacci chain of 17 distance codes,
    about 4 200 copies whose distances the head tables deliver exactly inside one piece; no generator for it is attempted, so the
    limiter is exercised on the literal/length and code-length trees only."""
    lit_depth = cl_depth = dist_depth = 0
    modes, len_syms, dist_codes, max_dist = set(), set(), set(), 0
    for name in CORPUS:
        for _, _, Q, P in model_of(name)[2]:
            lit_depth, dist_depth, cl_depth = max(lit_depth, Q["lit_depth"]), max(dist_depth, Q["dist_depth"]), max(cl_depth, Q["cl_depth"])
            modes.add(P["btype"])
            for t in P["tokens"]:
                if not isinstance(t, int):
                    len_syms.add(LSYM[t[0]][0])
                    dist_codes.add(dist_symbol(t[1])[0])
                    max_dist = max(max_dist, t[1])
    print("pre-limit depths: literal/length %d, distance %d, code-length %d" % (lit_depth, dist_depth, cl_depth))
    assert lit_depth > 15
    assert cl_depth > 7
    assert modes == {0, 1, 2}
    assert len_syms == set(range(257, 286))
    assert dist_codes == set(range(30))
    assert max_dist == 32768
    for which in ("tie", "eob_dynamic", "eob_stored"):
        assert is_cost_edge(which, model_of("cost_" + which)[2][0][2]), which


def test_every_length_is_emitted():
    """every length 3..258, so every extra-bits value of every length code"""
    lengths = set()
    for _, _, _, P in model_of("every_code")[2]:
        lengths |= {t[0] for t in P["tokens"] if not isinstance(t, int)}
    assert lengths >= set(range(3, 259))


@pytest.mark.parametrize("distance", [32768, 32769])
def test_window_edge(distance):
    """the copies at 32768 are emitted as copies from the tile edges; those at 32769 are not copies at all"""
    data, _, rows = model_of("window_%d" % distance)
    Q = rows[0][2]
    at = dict(zip(Q["starts"].tolist(), zip(Q["lengths"].tolist(), Q["distances"].tolist())))
    for t in WINDOW_TARGETS[distance]:
        assert data[t:t + 40] == data[t - distance:t - distance + 40]
        assert at.get(t) == ((40, 32768) if distance == 32768 else (0, 0)), (t, at.get(t))


def test_hash_collisions_are_common():
    """in the collision input, at a third of the positions the latest earlier position with the same 3-byte or 4-byte hash holds
    other bytes"""
    data = corpus_input("hash_collisions")
    collide = np.zeros(len(data), bool)
    for k, h in ((3, _h3(data)), (4, _h4(data))):
        last = {}
        for i, hv in enumerate(h.tolist()):
            if hv in last and data[last[hv]:last[hv] + k] != data[i:i + k]:
                collide[i] = True
            last[hv] = i
    assert collide.sum() > len(data) // 3, collide.sum()


def test_parser_rejects_broken_codes():
    """an over-subscribed and an incomplete literal/length code, and a second block, are refused"""
    data = corpus_input("fastq_%d" % PIECE)
    m = pybgzf.member(data)
    Q = pybgzf.plan(data)
    assert Q["mode"] == 2
    pybgzf.parse_member(m)
    # the first HCLEN entry (code-length symbol 16) widened from its length to 1: the code-length code is over-subscribed
    bits = int.from_bytes(m[18:22], "little")
    assert Q["cl_lens"][16] != 1
    broken = bytearray(m)
    broken[18:22] = (bits & ~(7 << 17) | 1 << 17).to_bytes(4, "little")
    with pytest.raises(pybgzf.DeflateError, match="code-length code is over-subscribed"):
        pybgzf.parse_member(bytes(broken))
    nonfinal = bytearray(m)
    nonfinal[18] &= 0xfe
    with pytest.raises(pybgzf.DeflateError, match="more than one block"):
        pybgzf.parse_member(bytes(nonfinal))
    with pytest.raises(pybgzf.DeflateError, match="over-subscribed"):
        pybgzf._Code([1, 1, 2], "literal/length", single_ok=True)
    with pytest.raises(pybgzf.DeflateError, match="incomplete"):
        pybgzf._Code([1, 2, 0], "literal/length", single_ok=True)
    pybgzf._Code([1, 0, 0], "distance", single_ok=True)
