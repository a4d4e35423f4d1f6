"""CPU model of the device gzip inflater (megapath_b200/csrc/mp_gunzip.cu), written without zlib.

- `Decoder.run` restates `gz_run`: gzip framing (RFC 1952 2.3), stored / fixed / dynamic blocks (RFC 1951 3.2), and the stops the
  kernel makes -- at the first block header at or after a target bit, when `limit` symbols or the event list are full, when the input
  ends (every symbol whose bits are all present is delivered, as zlib's inflate delivers them) and at the first invalid symbol.
  Back-references before the chunk's first symbol become markers 256 + i (byte i of the 32 KiB before the chunk).
- `dyn_header_valid(data, bit)` is the block search's test (`k_gz_find` + `gz_dyn_header`): BFINAL = 0, BTYPE = 2, HLIT <= 286 and
  HDIST <= 30 codes (inflate.c TABLE), a complete code-length code (inftrees.c, CODES: incomplete refused), no repeat of a missing
  length or past HLIT + HDIST (inflate.c CODELENS), a nonzero end-of-block length, and lit/len and distance codes inflate_table
  accepts (over-subscribed refused; incomplete refused unless the only code has length 1; an all-zero distance code accepted).
- `inflate(data)` decodes a whole file and records every true block boundary; `plan(data)` replays `mp_gunzip_run` for one call with
  the whole file and `fin` set, and returns the counters the device reports in `mp_gunzip_stats`.
"""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import numpy as np  # noqa: E402

from megapath_b200 import GUNZIP_CHUNK as CHUNK, GUNZIP_SLOT as SLOT, GUNZIP_EVENTS as EVENTS  # noqa: E402

WIN = 32768
LEN_BASE = [3, 4, 5, 6, 7, 8, 9, 10, 11, 13, 15, 17, 19, 23, 27, 31, 35, 43, 51, 59, 67, 83, 99, 115, 131, 163, 195, 227, 258]
LEN_EXTRA = [0] * 8 + [1] * 4 + [2] * 4 + [3] * 4 + [4] * 4 + [5] * 4 + [0]
DIST_BASE = [1, 2, 3, 4, 5, 7, 9, 13, 17, 25, 33, 49, 65, 97, 129, 193, 257, 385, 513, 769, 1025, 1537, 2049, 3073, 4097, 6145, 8193,
             12289, 16385, 24577]
DIST_EXTRA = [0, 0, 0, 0, 1, 1, 2, 2, 3, 3, 4, 4, 5, 5, 6, 6, 7, 7, 8, 8, 9, 9, 10, 10, 11, 11, 12, 12, 13, 13]
CL_ORDER = [16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15]
FIXED = [8] * 144 + [9] * 112 + [7] * 24 + [8] * 8
FIXED_DIST = [5] * 32
# modes and results, as in mp_gunzip.cu
HEADER, BLOCK, DATA, TRAILER, END = range(5)
TARGET, FULL, NEED, S_END, ERROR = 1, 2, 3, 4, 5


class Bits:
    def __init__(self, data):
        self.d, self.nbits = data, len(data) * 8

    def peek(self, pos):
        """(up to 56 bits from pos, how many of them exist)"""
        b = pos >> 3
        v = int.from_bytes(self.d[b:b + 8], "little") >> (pos & 7)
        avail = max(0, min(56, self.nbits - pos))
        return v & ((1 << avail) - 1), avail


def check(lens, codes):
    """inftrees.c inflate_table's verdict: True = usable"""
    count = [0] * 16
    for x in lens:
        count[x] += 1
    mx = max((i for i in range(1, 16) if count[i]), default=0)
    if mx == 0:
        return not codes
    left = 1
    for ln in range(1, 16):
        left = 2 * left - count[ln]
        if left < 0:
            return False
    return not (left > 0 and (codes or mx != 1))


class Code:
    """canonical code (RFC 1951 3.2.2) as a table over its longest length: pattern -> (symbol, length)"""

    def __init__(self, lens):
        self.mx = max(lens) if any(lens) else 1
        self.lut = [None] * (1 << self.mx)
        count = [0] * 16
        for x in lens:
            count[x] += 1
        count[0] = 0
        code, first = 0, [0] * 16
        for ln in range(1, 16):
            code = (code + count[ln - 1]) << 1
            first[ln] = code
        for s, ln in enumerate(lens):
            if not ln:
                continue
            c = first[ln]
            first[ln] += 1
            r = int("{:0{}b}".format(c, ln)[::-1], 2)
            for k in range(r, 1 << self.mx, 1 << ln):
                self.lut[k] = (s, ln)

    def decode(self, v, avail):
        """symbol, its length; None = more input needed; -1 = no such code"""
        e = self.lut[v & ((1 << self.mx) - 1)]
        if e is not None and e[1] <= avail:
            return e
        if e is None and avail >= 15:
            return -1, 0
        return None


def dyn_header(br, pos):
    """gz_dyn_header from the bit after BTYPE: (0, pos, lens, nlen) valid; (1,) input ends inside; (-1,) invalid"""
    v, av = br.peek(pos)
    if av < 14:
        return (1,)
    nlen, ndist, ncode = (v & 31) + 257, ((v >> 5) & 31) + 1, ((v >> 10) & 15) + 4
    if nlen > 286 or ndist > 30:
        return (-1,)
    pos += 14
    cl = [0] * 19
    for i in range(ncode):
        v, av = br.peek(pos)
        if av < 3:
            return (1,)
        cl[CL_ORDER[i]] = v & 7
        pos += 3
    if not check(cl, True):
        return (-1,)
    cc = Code(cl)
    lens = []
    while len(lens) < nlen + ndist:
        v, av = br.peek(pos)
        r = cc.decode(v, min(av, 7) if av < 7 else av)
        if r is None:
            return (1,)
        s, used = r
        if s < 0:
            return (-1,)
        if s < 16:
            lens.append(s)
            pos += used
            continue
        xb = {16: 2, 17: 3, 18: 7}[s]
        if av < used + xb:
            return (1,)
        x = (v >> used) & ((1 << xb) - 1)
        if s == 16:
            if not lens:
                return (-1,)
            val, rep = lens[-1], 3 + x
        else:
            val, rep = 0, (3 if s == 17 else 11) + x
        if len(lens) + rep > nlen + ndist:
            return (-1,)
        pos += used + xb
        lens += [val] * rep
    if lens[256] == 0 or not check(lens[:nlen], False) or not check(lens[nlen:], False):
        return (-1,)
    return 0, pos, lens, nlen


def dyn_header_valid(data, bit, br=None):
    """the block search's test at one bit offset (k_gz_find)"""
    br = br or Bits(data)
    v, av = br.peek(bit)
    if av < 17 or (v & 7) != 4:
        return False
    return dyn_header(br, bit + 3)[0] == 0


def _crc_byte(c, b):
    c ^= b
    for _ in range(8):
        c = (c >> 1) ^ 0xEDB88320 if c & 1 else c >> 1
    return c


class State:
    def __init__(self, bit=0, mode=HEADER, first=True):
        self.bit, self.mode, self.first = bit, mode, first
        self.bfinal = self.btype = self.left = 0
        self.lens, self.nlen = None, 0
        self.hstage = self.hflags = self.hleft = self.hcrc = 0

    def copy(self):
        s = State()
        s.__dict__.update(self.__dict__)
        return s


def run(data, fin, st, target, limit, boundaries=None):
    """gz_run: -> (status, end state, symbols, events [(kind, out, crc, isize)]); boundaries collects (bit, out) of block headers"""
    st = st.copy()
    br, n = Bits(data), len(data)
    out, ev, member_at = [], [], None
    pos = st.bit
    lit = dist = None
    if st.mode == DATA and st.btype:
        lens = FIXED + FIXED_DIST if st.btype == 1 else st.lens
        nl = 288 if st.btype == 1 else st.nlen
        lit, dist = Code(lens[:nl]), Code(lens[nl:])

    def done(status):
        st.bit = pos
        if status == S_END:
            st.mode = END
        return status, st, out, ev
    while True:
        if st.mode == HEADER:
            if st.hstage == 0:
                if len(ev) >= EVENTS:                  # room for the start event before anything of the header is consumed
                    return done(FULL)
                at = pos >> 3
                rest = max(0, n - at)
                if not st.first:
                    if rest < 2:
                        return done(S_END if fin else NEED)
                    if data[at] != 0x1f or data[at + 1] != 0x8b:
                        return done(S_END)
                if rest < 10:
                    if st.first and rest >= 1 and (data[at] != 0x1f or (rest >= 2 and data[at + 1] != 0x8b)):
                        return done(ERROR)
                    return done(NEED)
                if data[at] != 0x1f or data[at + 1] != 0x8b or data[at + 2] != 8 or data[at + 3] & 0xe0:
                    return done(ERROR)
                c = 0xffffffff
                for i in range(10):
                    c = _crc_byte(c, data[at + i])
                st.hcrc, st.hflags, st.hstage = c, data[at + 3], 1
                pos = (at + 10) * 8
            at = pos >> 3
            if st.hstage == 1:
                if st.hflags & 4:
                    if at + 2 > n:
                        return done(NEED)
                    st.hleft = data[at] | data[at + 1] << 8
                    st.hcrc = _crc_byte(_crc_byte(st.hcrc, data[at]), data[at + 1])
                    at += 2
                    st.hstage = 2
                else:
                    st.hstage = 3
            if st.hstage == 2:
                while st.hleft and at < n:
                    st.hcrc = _crc_byte(st.hcrc, data[at])
                    at += 1
                    st.hleft -= 1
                if st.hleft:
                    pos = at * 8
                    return done(NEED)
                st.hstage = 3
            for f in (3, 4):
                if st.hstage != f:
                    continue
                if st.hflags & (8 if f == 3 else 16):
                    while True:
                        if at >= n:
                            pos = at * 8
                            return done(NEED)
                        b = data[at]
                        at += 1
                        st.hcrc = _crc_byte(st.hcrc, b)
                        if not b:
                            break
                st.hstage = f + 1
            if st.hstage == 5 and st.hflags & 2:
                if at + 2 > n:
                    pos = at * 8
                    return done(NEED)
                if (data[at] | data[at + 1] << 8) != (~st.hcrc & 0xffff):
                    return done(ERROR)
                at += 2
            pos = at * 8
            ev.append((0, len(out), 0, 0))
            member_at = len(out)
            st.mode, st.first, st.hstage = BLOCK, False, 0
            if boundaries is not None:
                boundaries.append((pos, len(out)))
            if pos >= target:
                return done(TARGET)
            continue
        if st.mode == BLOCK:
            v, av = br.peek(pos)
            if av < 3:
                return done(NEED)
            bf, bt = v & 1, (v >> 1) & 3
            if bt == 3:
                return done(ERROR)
            p = pos + 3
            if bt == 0:
                p = (p + 7) & ~7
                v, av = br.peek(p)
                if av < 32:
                    return done(NEED)
                ln, nln = v & 0xffff, (v >> 16) & 0xffff
                if ln != (~nln & 0xffff):
                    return done(ERROR)
                st.left = ln
                p += 32
            elif bt == 1:
                lit, dist = Code(FIXED), Code(FIXED_DIST)
            else:
                r = dyn_header(br, p)
                if r[0] == 1:
                    return done(NEED)
                if r[0] < 0:
                    return done(ERROR)
                _, p, st.lens, st.nlen = r
                lit, dist = Code(st.lens[:st.nlen]), Code(st.lens[st.nlen:])
            pos = p
            st.bfinal, st.btype, st.mode = bf, bt, DATA
            continue
        if st.mode == DATA:
            if st.btype == 0:
                at = pos >> 3
                k = min(st.left, n - at, limit - len(out))
                out += data[at:at + k]
                st.left -= k
                pos = (at + k) * 8
                if st.left:
                    return done(FULL if len(out) >= limit else NEED)
            else:
                while True:
                    v, av = br.peek(pos)
                    r = lit.decode(v, av)
                    if r is None:
                        return done(NEED)
                    s, used = r
                    if s < 0 or s > 285:
                        return done(ERROR)
                    if s < 256:
                        if len(out) >= limit:
                            return done(FULL)
                        out.append(s)
                        pos += used
                        continue
                    if s == 256:
                        pos += used
                        break
                    li = s - 257
                    lx = LEN_EXTRA[li]
                    if av < used + lx:
                        return done(NEED)
                    ln = LEN_BASE[li] + ((v >> used) & ((1 << lx) - 1))
                    r = dist.decode(v >> (used + lx), av - used - lx)
                    if r is None:
                        return done(NEED)
                    ds, used2 = r
                    if ds < 0 or ds > 29:
                        return done(ERROR)
                    dx = DIST_EXTRA[ds]
                    tot = used + lx + used2 + dx
                    if av < tot:
                        return done(NEED)
                    d = DIST_BASE[ds] + ((v >> (used + lx + used2)) & ((1 << dx) - 1))
                    o = len(out)
                    if member_at is not None and o - d < member_at:
                        return done(ERROR)
                    if o + ln > limit:
                        return done(FULL)
                    pos += tot
                    for k in range(ln):
                        f = o + k - d
                        out.append(out[f] if f >= 0 else 256 + WIN + f)
            if st.bfinal:
                st.mode = TRAILER
                continue
            st.mode = BLOCK
            if boundaries is not None:
                boundaries.append((pos, len(out)))
            if pos >= target:
                return done(TARGET)
            continue
        if st.mode == TRAILER:
            at = (pos + 7) >> 3
            if at + 8 > n:
                pos = at * 8
                return done(NEED)
            if len(ev) >= EVENTS:
                return done(FULL)
            ev.append((1, len(out), int.from_bytes(data[at:at + 4], "little"), int.from_bytes(data[at + 4:at + 8], "little")))
            pos = (at + 8) * 8
            st.mode, st.hstage = HEADER, 0
            continue
        return done(S_END)


def find(data):
    """k_gz_find: per chunk after the first, the first valid bit offset (None = merged) and the offsets examined"""
    n = len(data)
    nr = max(1, -(-n // CHUNK))
    bits = np.unpackbits(np.frombuffer(bytes(data) + bytes(8), np.uint8), bitorder="little").astype(np.uint32)
    br = Bits(data)
    cands, tested = [None] * nr, 0
    for r in range(1, nr):
        lo, hi = r * CHUNK * 8, min((r + 1) * CHUNK, n) * 8
        idx = np.arange(lo, hi)
        v = np.zeros(len(idx), np.uint32)
        for i in range(17):
            v |= bits[idx + i] << i
        ok = ((v & 7) == 4) & (((v >> 3) & 31) <= 29) & (((v >> 8) & 31) <= 29) & (idx + 17 <= n * 8)
        for b in idx[ok]:
            if dyn_header_valid(data, int(b), br):
                cands[r] = int(b)
                break
        tested += (cands[r] + 1 if cands[r] is not None else hi) - lo
    return cands, tested


def plan(data, fin=True):
    """mp_gunzip_run on the whole file in one call (dstCap large): the counters of mp_gunzip_stats, the output and the outcome"""
    data = bytes(data)
    cands, tested = find(data)
    stats = dict(chunks=len(cands), candidates_tested=tested, candidates=sum(c is not None for c in cands[1:]),
                 merged=sum(c is None for c in cands[1:]), false_candidates=0, overflows=0, rounds=0, members=0)
    starts = [State()] + [State(c, BLOCK, False) for c in cands[1:] if c is not None]
    m = len(starts)
    target = [starts[i + 1].bit if i + 1 < m else float("inf") for i in range(m)]
    res = [None] * m
    pending = list(range(m))
    cur, out, evs, status = 0, bytearray(), [], None
    while status is None:
        for c in pending:
            res[c] = run(data, fin, starts[c], target[c], SLOT)
        stats["rounds"] += 1
        pending = []
        while status is None and not pending:
            st, end, syms, ev = res[cur]
            P = len(out)
            for k, v in enumerate(syms):
                out.append(v if v < 256 else out[P - WIN + (v - 256)] if P - WIN + (v - 256) >= 0 else 0)
            evs += [(kind, P + o, crc, isz) for kind, o, crc, isz in ev]
            if st == TARGET:
                if cur + 1 < m and end.bit == starts[cur + 1].bit:
                    cur += 1
                    continue
                stats["false_candidates"] += 1
                cur += 1
                starts[cur] = end
                pending = [cur]
            elif st == FULL:
                stats["overflows"] += 1
                starts[cur] = end
                pending = [cur]
            else:
                status = st
    crc_ok = True
    mstart = 0
    import zlib as _z   # CRC-32 values only (the inflate itself does not use zlib)
    for kind, at, crc, isz in evs:
        if kind == 0:
            mstart = at
            continue
        seg = bytes(out[mstart:at])
        if _z.crc32(seg) != crc or len(seg) & 0xffffffff != isz:
            crc_ok = False
            break
        stats["members"] += 1
    stats["status"] = status
    stats["crc_ok"] = crc_ok
    stats["output"] = bytes(out)
    return stats


def gunzip(data):
    """What mp_gunzip_run delivers for the whole file with fin set: (bytes, None | "error" | "truncated").  One decoder from the start,
    then CRC-32 and ISIZE member by member; on an error, the bytes before it."""
    import zlib as _z   # CRC-32 values only
    data, state, out, ev = bytes(data), State(), bytearray(), []
    while True:
        st, state, syms, e = run(data, True, state, float("inf"), 1 << 62)
        P = len(out)
        for v in syms:                                  # a resumed run's markers: bytes of the 32 KiB before it
            out.append(v if v < 256 else out[P - WIN + (v - 256)])
        ev += [(kind, P + o, crc, isz) for kind, o, crc, isz in e]
        if st != FULL:                                  # the event list filled: resume, as the device does
            break
    out = bytes(out)
    mstart = 0
    for kind, at, crc, isz in ev:
        if kind == 0:
            mstart = at
        elif _z.crc32(out[mstart:at]) != crc or (at - mstart) & 0xffffffff != isz:
            return out[:at], "error"
    if st == ERROR:
        return out, "error"
    if st == NEED:
        return out, "truncated"
    return out, None


def inflate(data):
    """Whole-file decode from the start, one chunk: (output bytes, status, [(bit, output offset) of every true block header])"""
    bounds = []
    st, end, syms, ev = run(bytes(data), True, State(), float("inf"), 1 << 62, bounds)
    return bytes(syms), st, bounds
