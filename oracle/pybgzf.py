"""Plain restatement of the device BGZF encoder (megapath_b200/csrc/mp_bgzf.cu) and an independent DEFLATE parser.  TEST
INFRASTRUCTURE ONLY: importable from tests/.

compress(data) / member(piece) give the bytes k_bgzf_member + k_bgzf_gather give, member by member; plan(piece) exposes the
decisions behind them (tokens, trees, costs, the depth of every tree before length limiting).  Each step cites the kernel line it
restates and the RFC 1951 section it implements.

parse_member(raw) walks one BGZF member without zlib and returns what it holds: block type, HLIT / HDIST / HCLEN, the three
code-length arrays, the run-length symbols of the header, the tokens and the decoded bytes.  It shares no code with the encoder
model, so the tests can hold the two against each other.
"""
import zlib

import numpy as np
from numpy.lib.stride_tricks import sliding_window_view

PIECE = 0xff00                      # mp_bgzf.cu:30 BG_PIECE
TILE = 512                          # mp_bgzf.cu:29 BG_THREADS: one tile of positions per pass of the CTA
HASH_BITS = 14                      # mp_bgzf.cu:32
WINDOW = 32768                      # mp_bgzf.cu:33, RFC 1951 2.
MAX_MATCH = 258

# RFC 1951 3.2.5 (mp_bgzf.cu:35-40)
LEN_BASE = np.array([3, 4, 5, 6, 7, 8, 9, 10, 11, 13, 15, 17, 19, 23, 27, 31, 35, 43, 51, 59, 67, 83, 99, 115, 131, 163, 195, 227, 258])
LEN_EXTRA = np.array([0, 0, 0, 0, 0, 0, 0, 0, 1, 1, 1, 1, 2, 2, 2, 2, 3, 3, 3, 3, 4, 4, 4, 4, 5, 5, 5, 5, 0])
DIST_BASE = np.array([1, 2, 3, 4, 5, 7, 9, 13, 17, 25, 33, 49, 65, 97, 129, 193, 257, 385, 513, 769, 1025, 1537, 2049, 3073,
                      4097, 6145, 8193, 12289, 16385, 24577])
DIST_EXTRA = np.array([0, 0, 0, 0, 1, 1, 2, 2, 3, 3, 4, 4, 5, 5, 6, 6, 7, 7, 8, 8, 9, 9, 10, 10, 11, 11, 12, 12, 13, 13])
CL_ORDER = [16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15]
RLE_EXTRA = {16: 2, 17: 3, 18: 7}
# RFC 1951 3.2.6: the fixed literal/length code
FIXED_LIT = np.array([8] * 144 + [9] * 112 + [7] * 24 + [8] * 8)


def len_code(L):
    """match length 3..258 -> length code 0..28 (symbol 257 + code); mp_bgzf.cu:243 lenLut"""
    return np.searchsorted(LEN_BASE, L, side="right") - 1


def dist_code(d):
    """distance 1..32768 -> distance code 0..29; mp_bgzf.cu:247-248 distLut, 160 bg_dist_code"""
    return np.searchsorted(DIST_BASE, d, side="right") - 1


# ---- matching (mp_bgzf.cu:269-297) and the greedy parse (302-303) ----

def matches(piece):
    """-> (length, distance) per position, 0 where no match of 3+ bytes was found.

    Tile by tile (512 positions): every position i with i + 3 <= len looks up the head tables, which hold (position + 1) of the
    latest position of an *earlier* tile with the same 3-byte hash (w3 * 2654435761 >> 18) and the same 4-byte hash
    (w4 * 2246822519 >> 18; only where i + 4 <= len).  The 4-byte candidate is tried first, the 3-byte one is skipped when it is the
    same position, a candidate further than 32768 back is skipped, and a candidate replaces the best only if strictly longer.
    Lengths stop at 258 and at the end of the piece.  After the tile the heads take the tile's positions (atomicMax: the latest)."""
    n = len(piece)
    pad = np.zeros(n + MAX_MATCH + 8, np.uint8)
    pad[:n] = np.frombuffer(piece, np.uint8)
    b = pad.astype(np.uint64)
    w3 = b[0:n] | b[1:n + 1] << 8 | b[2:n + 2] << 16
    w4 = w3 | b[3:n + 3] << 24
    h3 = ((w3 * 2654435761) & 0xffffffff) >> (32 - HASH_BITS)
    h4 = ((w4 * 2246822519) & 0xffffffff) >> (32 - HASH_BITS)
    idx = np.arange(n, dtype=np.int64)
    ok3, ok4 = idx + 3 <= n, idx + 4 <= n
    win = sliding_window_view(pad, MAX_MATCH)
    head3 = np.zeros(1 << HASH_BITS, np.int64)
    head4 = np.zeros(1 << HASH_BITS, np.int64)
    outL = np.zeros(n, np.int64)
    outD = np.zeros(n, np.int64)
    for tile in range(0, n, TILE):
        i = idx[tile:tile + TILE]
        o3, o4 = ok3[i], ok4[i]
        c4 = np.where(o4, head4[h4[i]], 0)
        c3 = head3[h3[i]]
        c3 = np.where(c3 == c4, 0, c3)
        maxL = np.minimum(MAX_MATCH, n - i)
        bestL = np.zeros(len(i), np.int64)
        bestD = np.zeros(len(i), np.int64)
        for cand in (c4, c3):
            d = i - (cand - 1)
            valid = o3 & (cand > 0) & (d <= WINDOW)
            if not valid.any():
                continue
            vi, vc = i[valid], cand[valid] - 1
            eq = win[vc] == win[vi]
            L = np.where(eq.all(axis=1), MAX_MATCH, np.argmin(eq, axis=1))
            L = np.minimum(L, maxL[valid])
            better = L > bestL[valid]
            sel = np.flatnonzero(valid)[better]
            bestL[sel] = L[better]
            bestD[sel] = d[valid][better]
        keep = bestL >= 3
        outL[tile:tile + TILE] = np.where(keep, bestL, 0)
        outD[tile:tile + TILE] = np.where(keep, bestD, 0)
        np.maximum.at(head3, h3[i][o3], i[o3] + 1)
        np.maximum.at(head4, h4[i][o4], i[o4] + 1)
    return outL, outD


def parse(piece):
    """greedy parse -> token start positions: p += max(1, len[p]) (mp_bgzf.cu:303)"""
    L, D = matches(piece)
    Ll = L.tolist()
    starts, p, n = [], 0, len(piece)
    while p < n:
        starts.append(p)
        p += Ll[p] or 1
    starts = np.array(starts, np.int64)
    return starts, L[starts], D[starts]


# ---- Huffman code lengths (mp_bgzf.cu:102-146) ----

def build_lengths(freq, limit):
    """-> (lengths, depth before limiting).  Symbols sorted by (frequency, symbol); fewer than two used symbols are padded with the
    lowest-numbered unused ones at frequency 1 (trees.c keeps two codes per tree); Moffat-Katajainen in place (lines 117-132), depths
    clamped at 32 (135); miniz's limiting (136-143); lengths handed out shortest first to the most frequent symbols (144-145)."""
    n = len(freq)
    keys = [(int(f), s) for s, f in enumerate(freq) if f]
    for s in range(n):
        if len(keys) >= 2:
            break
        if not freq[s]:
            keys.append((1, s))
    keys.sort()
    used = len(keys)
    A = [f for f, _ in keys]
    root, leaf = 0, 2
    A[0] += A[1]
    for nxt in range(1, used - 1):
        if leaf >= used or A[root] < A[leaf]:
            A[nxt] = A[root]
            A[root] = nxt
            root += 1
        else:
            A[nxt] = A[leaf]
            leaf += 1
        if leaf >= used or (root < nxt and A[root] < A[leaf]):
            A[nxt] += A[root]
            A[root] = nxt
            root += 1
        else:
            A[nxt] += A[leaf]
            leaf += 1
    A[used - 2] = 0
    for nxt in range(used - 3, -1, -1):
        A[nxt] = A[A[nxt]] + 1
    avbl, u, dpth, root, nxt = 1, 0, 0, used - 2, used - 1
    while avbl > 0:
        while root >= 0 and A[root] == dpth:
            u += 1
            root -= 1
        while avbl > u:
            A[nxt] = dpth
            nxt -= 1
            avbl -= 1
        avbl, dpth, u = 2 * u, dpth + 1, 0
    depth = max(A)
    count = [0] * 33
    for a in A:
        count[min(a, 32)] += 1
    for i in range(limit + 1, 33):
        count[limit] += count[i]
        count[i] = 0
    total = sum(count[i] << (limit - i) for i in range(limit, 0, -1))
    while total != 1 << limit:
        count[limit] -= 1
        for i in range(limit - 1, 0, -1):
            if count[i]:
                count[i] -= 1
                count[i + 1] += 2
                break
        total -= 1
    lens = np.zeros(n, np.int64)
    j = used
    for i in range(1, limit + 1):
        for _ in range(count[i]):
            j -= 1
            lens[keys[j][1]] = i
    return lens, depth


def canonical_codes(lens):
    """RFC 1951 3.2.2 (mp_bgzf.cu:149-158), codes MSB-first"""
    lens = [int(x) for x in lens]
    cnt = [0] * 16
    for x in lens:
        cnt[x] += 1
    cnt[0] = 0
    nxt, code = [0] * 16, 0
    for b in range(1, 16):
        code = (code + cnt[b - 1]) << 1
        nxt[b] = code
    codes = []
    for x in lens:
        codes.append(nxt[x] if x else 0)
        if x:
            nxt[x] += 1
    return np.array(codes, np.int64)


def rle_lengths(all_lens):
    """run-length coding of the concatenated literal/length and distance code lengths (mp_bgzf.cu:184-197, RFC 1951 3.2.7):
    zeros as 18 (11..138) while 11 or more remain, then 17 (3..10); a non-zero length once, then 16 (3..6 repeats) while 3 or more
    remain; whatever is left as single symbols.  Runs may cross from the literal lengths into the distance lengths.
    -> list of (symbol, extra value)"""
    out, i, nl = [], 0, len(all_lens)
    while i < nl:
        v = int(all_lens[i])
        r = 1
        while i + r < nl and all_lens[i + r] == v:
            r += 1
        i += r
        if v == 0:
            while r >= 11:
                k = min(r, 138)
                out.append((18, k - 11))
                r -= k
            if r >= 3:
                out.append((17, r - 3))
                r = 0
        else:
            out.append((v, 0))
            r -= 1
            while r >= 3:
                k = min(r, 6)
                out.append((16, k - 3))
                r -= k
        out.extend([(v, 0)] * r)
    return out


def plan(piece):
    """the decisions bg_plan (mp_bgzf.cu:164-221) takes for one piece, as a dict:
    tokens (starts, lengths, distances), lit_freq / dist_freq / cl_freq, lit_lens / dist_lens / cl_lens, the pre-limit depths
    lit_depth / dist_depth / cl_depth, hlit / hdist / hclen, rle, the three costs in bits and mode (0 stored, 1 fixed, 2 dynamic)."""
    n = len(piece)
    arr = np.frombuffer(piece, np.uint8)
    starts, L, D = parse(piece)
    is_m = L > 0
    lc, dc = len_code(L[is_m]), dist_code(D[is_m])
    lit_freq = np.bincount(arr[starts[~is_m]], minlength=286)
    lit_freq += np.bincount(257 + lc, minlength=286)
    lit_freq[256] = 1                                                                 # EOB (line 324)
    dist_freq = np.bincount(dc, minlength=30)
    extra = int(LEN_EXTRA[lc].sum() + DIST_EXTRA[dc].sum())
    fixed_bits = 3 + extra + int((lit_freq * FIXED_LIT[:286]).sum()) + 5 * int(dist_freq.sum())      # lines 170-172
    lit_lens, lit_depth = build_lengths(lit_freq, 15)
    dist_lens, dist_depth = build_lengths(dist_freq, 15)
    hlit, hdist = 286, 30                                                              # lines 176-178
    while hlit > 257 and not lit_lens[hlit - 1]:
        hlit -= 1
    while hdist > 1 and not dist_lens[hdist - 1]:
        hdist -= 1
    rle = rle_lengths(np.concatenate([lit_lens[:hlit], dist_lens[:hdist]]))
    cl_freq = np.bincount([s for s, _ in rle], minlength=19)
    cl_lens, cl_depth = build_lengths(cl_freq, 7)
    hclen = 19                                                                         # line 200
    while hclen > 4 and not cl_lens[CL_ORDER[hclen - 1]]:
        hclen -= 1
    header_bits = 3 + 14 + 3 * hclen + sum(int(cl_lens[s]) + RLE_EXTRA.get(s, 0) for s, _ in rle)
    dyn_bits = header_bits + extra + int((lit_freq * lit_lens).sum()) + int((dist_freq * dist_lens).sum())
    stored_bits = (5 + n) * 8
    if dyn_bits <= fixed_bits and dyn_bits < stored_bits:                              # lines 207-220
        mode = 2
    elif fixed_bits < stored_bits:
        mode = 1
    else:
        mode = 0
    return dict(starts=starts, lengths=L, distances=D, n_literals=int((~is_m).sum()), n_matches=int(is_m.sum()),
                lit_freq=lit_freq, dist_freq=dist_freq, cl_freq=cl_freq, lit_lens=lit_lens, dist_lens=dist_lens, cl_lens=cl_lens,
                lit_depth=lit_depth, dist_depth=dist_depth, cl_depth=cl_depth, hlit=hlit, hdist=hdist, hclen=hclen, rle=rle,
                header_bits=header_bits, dyn_bits=dyn_bits, fixed_bits=fixed_bits, stored_bits=stored_bits, mode=mode)


# ---- emission (mp_bgzf.cu:326-383) ----

def _rev(code, length):
    """Huffman codes go out MSB first into the LSB-first bit stream (RFC 1951 3.1.1)"""
    out = np.zeros_like(code)
    for k in range(15):                                                                # code < 2^length: higher bits are 0
        out |= ((code >> k) & 1) << np.maximum(length - 1 - k, 0)
    return out


def pack_bits(values, lengths):
    """fields (value, bit count), LSB first, into bytes; the last byte is zero-padded"""
    values = np.asarray(values, np.uint64)
    lengths = np.asarray(lengths, np.int64)
    total = int(lengths.sum())
    starts = np.cumsum(lengths) - lengths
    off = np.arange(total, dtype=np.int64) - np.repeat(starts, lengths)
    bits = (np.repeat(values, lengths) >> off.astype(np.uint64)) & np.uint64(1)
    return np.packbits(bits.astype(np.uint8), bitorder="little").tobytes()


def member(piece):
    """one BGZF member (gzip header with the BC subfield and BSIZE, one final DEFLATE block, CRC-32, ISIZE) for 1..0xff00 bytes"""
    n = len(piece)
    assert 0 < n <= PIECE
    P = plan(piece)
    if P["mode"] == 0:                                                                 # RFC 1951 3.2.4 (lines 328-333)
        body = bytes([1, n & 0xff, n >> 8, ~n & 0xff, (~n >> 8) & 0xff]) + bytes(piece)
    else:
        if P["mode"] == 1:
            lit_lens, dist_lens = FIXED_LIT, np.full(30, 5)
            vals, lens = [1, 1], [1, 2]                                                # BFINAL, BTYPE 01
        else:
            lit_lens, dist_lens, cl_lens = P["lit_lens"], P["dist_lens"], P["cl_lens"]
            vals = [1, 2, P["hlit"] - 257, P["hdist"] - 1, P["hclen"] - 4] + [int(cl_lens[CL_ORDER[k]]) for k in range(P["hclen"])]
            lens = [1, 2, 5, 5, 4] + [3] * P["hclen"]
            cl_codes = _rev(canonical_codes(cl_lens), cl_lens)
            for s, x in P["rle"]:
                vals.append(int(cl_codes[s]))
                lens.append(int(cl_lens[s]))
                if s >= 16:
                    vals.append(x)
                    lens.append(RLE_EXTRA[s])
        lit_codes = _rev(canonical_codes(lit_lens), np.asarray(lit_lens))
        dist_codes = _rev(canonical_codes(dist_lens), np.asarray(dist_lens))
        arr = np.frombuffer(piece, np.uint8)
        L, D = P["lengths"], P["distances"]
        is_m = L > 0
        sym = np.where(is_m, 257 + len_code(np.maximum(L, 3)), arr[P["starts"]])
        lc = len_code(np.maximum(L, 3))
        dc = dist_code(np.maximum(D, 1))
        lit_lens = np.asarray(lit_lens)
        f = np.zeros((len(sym), 4, 2), np.int64)                                        # per token: symbol, length extra, distance, distance extra
        f[:, 0] = np.stack([lit_codes[sym], lit_lens[sym]], 1)
        f[:, 1] = np.where(is_m[:, None], np.stack([L - LEN_BASE[lc], LEN_EXTRA[lc]], 1), 0)
        f[:, 2] = np.where(is_m[:, None], np.stack([dist_codes[dc], np.asarray(dist_lens)[dc]], 1), 0)
        f[:, 3] = np.where(is_m[:, None], np.stack([D - DIST_BASE[dc], DIST_EXTRA[dc]], 1), 0)
        f = f.reshape(-1, 2)
        vals = np.concatenate([vals, f[:, 0], [lit_codes[256]]])
        lens = np.concatenate([lens, f[:, 1], [lit_lens[256]]])
        body = pack_bits(vals, lens)
    size = len(body) + 26
    hdr = bytes([31, 139, 8, 4, 0, 0, 0, 0, 0, 255, 6, 0, ord("B"), ord("C"), 2, 0, (size - 1) & 0xff, (size - 1) >> 8])
    return hdr + body + zlib.crc32(piece).to_bytes(4, "little") + n.to_bytes(4, "little")


def compress(data):
    """what mp_bgzf_compress returns: one member per 0xff00-byte piece, concatenated (no EOF marker)"""
    data = bytes(data)
    return b"".join(member(data[at:at + PIECE]) for at in range(0, len(data), PIECE))


def split_members(raw):
    """a run of BGZF members -> list of members, cut at their BSIZE fields"""
    out, at = [], 0
    while at < len(raw):
        if raw[at:at + 4] != b"\x1f\x8b\x08\x04" or raw[at + 12:at + 14] != b"BC":
            raise ValueError("no BGZF member at offset %d" % at)
        size = int.from_bytes(raw[at + 16:at + 18], "little") + 1
        out.append(raw[at:at + size])
        at += size
    return out


# ---- the parser: RFC 1952 framing with the BGZF extra field, RFC 1951 inflation; no zlib ----

class DeflateError(ValueError):
    pass


class _Bits:
    def __init__(self, data):
        self.data, self.pos, self.end = bytes(data) + b"\0" * 4, 0, 8 * len(data)

    def get(self, n):
        if self.pos + n > self.end:
            raise DeflateError("stream ends inside a field at bit %d" % self.pos)
        at = self.pos >> 3
        v = (int.from_bytes(self.data[at:at + 4], "little") >> (self.pos & 7)) & ((1 << n) - 1)
        self.pos += n
        return v


class _Code:
    """a prefix code from its code lengths: Kraft-checked, decoded through a full 2^maxlen table"""

    def __init__(self, lens, what, single_ok):
        self.lens = [int(x) for x in lens]
        counts = [0] * 16
        for x in self.lens:
            counts[x] += 1
        left = 1
        for b in range(1, 16):
            left = 2 * left - counts[b]
            if left < 0:
                raise DeflateError("%s code is over-subscribed (lengths %s)" % (what, self.lens))
        n_codes = sum(counts[1:])
        if left > 0 and not (n_codes == 0 and what == "distance") and not (single_ok and n_codes == 1 and counts[1] == 1):
            raise DeflateError("%s code is incomplete (lengths %s)" % (what, self.lens))
        self.what, self.maxlen = what, max(self.lens + [1])
        self.table = [None] * (1 << self.maxlen)
        code, nxt = 0, [0] * 16                                                        # RFC 1951 3.2.2
        for b in range(2, 16):
            code = (code + counts[b - 1]) << 1
            nxt[b] = code
        for s, x in enumerate(self.lens):
            if not x:
                continue
            c = nxt[x]
            nxt[x] += 1
            r = int(format(c, "0%db" % x)[::-1], 2)
            for k in range(1 << (self.maxlen - x)):
                self.table[r | k << x] = (s, x)

    def decode(self, bits):
        at = bits.pos >> 3
        peek = (int.from_bytes(bits.data[at:at + 4], "little") >> (bits.pos & 7)) & ((1 << self.maxlen) - 1)
        e = self.table[peek]
        if e is None:
            raise DeflateError("no %s code matches at bit %d" % (self.what, bits.pos))
        if bits.pos + e[1] > bits.end:
            raise DeflateError("stream ends inside a %s code" % self.what)
        bits.pos += e[1]
        return e[0]


def parse_member(raw):
    """one BGZF member -> dict(btype, bfinal, hlit, hdist, hclen, cl_lens, lit_lens, dist_lens, rle, tokens, data, block_bits,
    crc, isize).  tokens: an int for a literal byte, (length, distance) for a copy.  block_bits: bits from the block header to the
    end of the EOB code.  Raises DeflateError on anything a conforming inflater would refuse, and on more than one block."""
    raw = bytes(raw)
    if len(raw) < 26 or raw[:4] != b"\x1f\x8b\x08\x04" or raw[10:12] != b"\x06\x00" or raw[12:16] != b"BC\x02\x00":
        raise DeflateError("not a BGZF member header")
    if int.from_bytes(raw[16:18], "little") + 1 != len(raw):
        raise DeflateError("BSIZE %d does not match the member's %d bytes" % (int.from_bytes(raw[16:18], "little") + 1, len(raw)))
    bits = _Bits(raw[18:-8])
    out = dict(bfinal=bits.get(1), btype=bits.get(2), hlit=None, hdist=None, hclen=None, cl_lens=None, lit_lens=None, dist_lens=None,
               rle=None, tokens=[])
    if not out["bfinal"]:
        raise DeflateError("the member holds more than one block")
    data = bytearray()
    if out["btype"] == 0:                                                              # RFC 1951 3.2.4
        bits.pos = (bits.pos + 7) & ~7
        ln, nln = bits.get(16), bits.get(16)
        if ln != nln ^ 0xffff:
            raise DeflateError("stored block LEN/NLEN mismatch")
        at = bits.pos >> 3
        if at + ln > len(raw) - 26:
            raise DeflateError("stored block runs past the member")
        data += raw[18 + at:18 + at + ln]
        out["tokens"] = list(data)
        bits.pos += 8 * ln
    elif out["btype"] in (1, 2):
        if out["btype"] == 1:                                                          # RFC 1951 3.2.6: 288 and 32 symbols
            lit_lens, dist_lens = list(FIXED_LIT), [5] * 32
        else:                                                                          # RFC 1951 3.2.7
            hlit, hdist, hclen = bits.get(5) + 257, bits.get(5) + 1, bits.get(4) + 4
            if hlit > 286 or hdist > 30:
                raise DeflateError("HLIT %d / HDIST %d out of range" % (hlit, hdist))
            cl_lens = [0] * 19
            for k in range(hclen):
                cl_lens[CL_ORDER[k]] = bits.get(3)
            clc = _Code(cl_lens, "code-length", single_ok=False)
            lens, rle = [], []
            while len(lens) < hlit + hdist:
                s = clc.decode(bits)
                if s < 16:
                    rle.append((s, 0))
                    lens.append(s)
                    continue
                x = bits.get(RLE_EXTRA[s])
                rle.append((s, x))
                if s == 16:
                    if not lens:
                        raise DeflateError("repeat code 16 with no previous length")
                    lens += [lens[-1]] * (3 + x)
                else:
                    lens += [0] * ((3 if s == 17 else 11) + x)
            if len(lens) != hlit + hdist:
                raise DeflateError("code lengths run past HLIT + HDIST")
            lit_lens, dist_lens = lens[:hlit] + [0] * (286 - hlit), lens[hlit:] + [0] * (30 - hdist)
            if not lit_lens[256]:
                raise DeflateError("no code for end-of-block")
            out.update(hlit=hlit, hdist=hdist, hclen=hclen, cl_lens=cl_lens, rle=rle)
        out.update(lit_lens=lit_lens, dist_lens=dist_lens)
        litc = _Code(lit_lens, "literal/length", single_ok=True)
        distc = _Code(dist_lens, "distance", single_ok=True)
        toks = out["tokens"]
        while True:
            s = litc.decode(bits)
            if s < 256:
                data.append(s)
                toks.append(s)
                continue
            if s == 256:
                break
            if s > 285:
                raise DeflateError("literal/length symbol %d" % s)
            L = int(LEN_BASE[s - 257]) + bits.get(int(LEN_EXTRA[s - 257]))
            dc = distc.decode(bits)
            if dc > 29:
                raise DeflateError("distance symbol %d" % dc)
            d = int(DIST_BASE[dc]) + bits.get(int(DIST_EXTRA[dc]))
            if d > len(data):
                raise DeflateError("distance %d reaches before the start of the member (%d bytes out)" % (d, len(data)))
            for _ in range(L):
                data.append(data[-d])
            toks.append((L, d))
    else:
        raise DeflateError("block type 3")
    out["block_bits"] = bits.pos
    if (bits.pos + 7) >> 3 != len(raw) - 26:
        raise DeflateError("%d bytes of DEFLATE data, the block ends after %d" % (len(raw) - 26, (bits.pos + 7) >> 3))
    out["data"] = bytes(data)
    out["crc"] = int.from_bytes(raw[-8:-4], "little")
    out["isize"] = int.from_bytes(raw[-4:], "little")
    return out
