"""Seeded gzip corpus for the device inflater (tests/test_gpu_gunzip.py) and its CPU model (tests/test_gunzip_model.py), and the
reference every output is held to: zlib, member by member, delivering exactly what zlib delivers before an error."""
import gzip
import struct
import zlib

import numpy as np


def fastq(n, seed, lmin=90, lmax=150):
    """Four-line FASTQ records in the style of the suite's read generator (random bases, Illumina-like qualities)."""
    rng = np.random.default_rng(seed)
    out = []
    for i in range(n):
        L = int(rng.integers(lmin, lmax + 1))
        s = np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, L)].tobytes()
        q = (rng.integers(2, 41, L) + 33).astype(np.uint8).tobytes()
        out.append(b"@r%d/1\n%s\n+\n%s\n" % (i, s, q))
    return b"".join(out)


def deflate(data, level=6, strategy=zlib.Z_DEFAULT_STRATEGY, flushes=()):
    """One gzip member; flushes: [(offset, zlib flush mode)] inserted into the stream."""
    co = zlib.compressobj(level, zlib.DEFLATED, 31, 8, strategy)
    out, at = [], 0
    for off, mode in flushes:
        out.append(co.compress(data[at:off]))
        out.append(co.flush(mode))
        at = off
    out.append(co.compress(data[at:]))
    out.append(co.flush())
    return b"".join(out)


def stored_member(payload):
    """A gzip member made only of stored blocks (at most 65535 bytes each)."""
    body = []
    for k in range(0, max(len(payload), 1), 65535):
        p = payload[k:k + 65535]
        final = k + 65535 >= len(payload)
        body.append(bytes([1 if final else 0]) + struct.pack("<HH", len(p), len(p) ^ 0xffff) + p)
    return (b"\x1f\x8b\x08\x00\x00\x00\x00\x00\x00\xff" + b"".join(body) + struct.pack("<II", zlib.crc32(payload), len(payload) & 0xffffffff))


def with_header_flags(data, level=6):
    """Every gzip header flag set: FTEXT, FHCRC, FEXTRA, FNAME, FCOMMENT."""
    raw = zlib.compressobj(level, zlib.DEFLATED, -15)
    body = raw.compress(data) + raw.flush()
    extra = b"ab\x04\x00xyzw" + b"Q" * 65000           # nearly one 64 KiB call
    hdr = b"\x1f\x8b\x08" + bytes([1 | 2 | 4 | 8 | 16]) + b"\x01\x02\x03\x04\x00\x03"
    hdr += struct.pack("<H", len(extra)) + extra + b"reads.fq\x00" + b"a comment\x00"
    hdr += struct.pack("<H", zlib.crc32(hdr) & 0xffff)
    return hdr + body + struct.pack("<II", zlib.crc32(data), len(data) & 0xffffffff)


def false_candidates(seed):
    """Stored blocks whose payload is itself deflate output: valid dynamic block headers sit at offsets that are no block start."""
    inner = zlib.compressobj(6, zlib.DEFLATED, -15)
    payload = inner.compress(fastq(3000, seed)) + inner.flush()
    return stored_member(payload * 3), payload * 3


def bgzf_model(data):
    """BGZF members as samtools writes them (0xff00-byte pieces, the BC extra subfield), from oracle/pybgzf.py's framing."""
    out = []
    for k in range(0, len(data), 0xff00):
        p = data[k:k + 0xff00]
        raw = zlib.compressobj(6, zlib.DEFLATED, -15)
        body = raw.compress(p) + raw.flush()
        bsize = 18 + len(body) + 8 - 1
        out.append(b"\x1f\x8b\x08\x04\x00\x00\x00\x00\x00\xff\x06\x00BC\x02\x00" + struct.pack("<H", bsize) + body +
                   struct.pack("<II", zlib.crc32(p), len(p)))
    return b"".join(out)


def far_back_member():
    """Two members where the second one's first match reaches into the first: zlib's "invalid distance too far back"."""
    a = gzip.compress(b"0123456789" * 100, 6)
    # a fixed block: literal 'x', then length 3 distance 5 (reaches 4 bytes before the member), then end of block
    bits = []

    def put(v, n, rev=False):
        if rev:
            v = int("{:0{}b}".format(v, n)[::-1], 2)
        for i in range(n):
            bits.append((v >> i) & 1)
    put(1, 1); put(1, 2)                        # BFINAL, BTYPE = fixed
    put(0x30 + ord("x"), 8, True)               # literal 'x'
    put(1, 7, True)                             # length code 257 = 3
    put(4, 5, True); put(0, 1)                  # distance code 4 (5..6), extra 0 -> 5
    put(0, 7, True)                             # end of block
    while len(bits) % 8:
        bits.append(0)
    body = bytes(int("".join(map(str, bits[i:i + 8][::-1])), 2) for i in range(0, len(bits), 8))
    b = b"\x1f\x8b\x08\x00\x00\x00\x00\x00\x00\xff" + body + struct.pack("<II", 0, 4)
    return a + b


def _bits_to_bytes(bits):
    while len(bits) % 8:
        bits.append(0)
    return bytes(int("".join(map(str, bits[i:i + 8][::-1])), 2) for i in range(0, len(bits), 8))


def distance_32768(seed, prefix=70000, copies=400):
    """Stored blocks of random bytes, then a fixed block of length-258 matches at distance 32768 (zlib's encoder never emits that
    distance): the references reach window byte 0, across a chunk edge and, fed in 64 KiB pieces, across call edges."""
    rng = np.random.default_rng(seed)
    head = rng.integers(0, 256, prefix, dtype=np.uint8).tobytes()
    body = b"".join(bytes([0]) + struct.pack("<HH", len(p), len(p) ^ 0xffff) + p for p in (head[k:k + 65535] for k in range(0, len(head), 65535)))
    bits = []

    def put(v, n, rev=False):
        if rev:
            v = int("{:0{}b}".format(v, n)[::-1], 2)
        for i in range(n):
            bits.append((v >> i) & 1)
    put(1, 1); put(1, 2)                                   # final fixed block
    for _ in range(copies):
        put(0xc5, 8, True)                                 # length code 285: 258
        put(29, 5, True); put(32768 - 24577, 13)           # distance code 29 + 13 extra bits: 32768
    put(0, 7, True)                                        # end of block
    out = bytearray(head)
    for _ in range(copies * 258):
        out.append(out[-32768])
    return (b"\x1f\x8b\x08\x00\x00\x00\x00\x00\x00\xff" + body + _bits_to_bytes(bits) +
            struct.pack("<II", zlib.crc32(bytes(out)), len(out) & 0xffffffff))


def far_back_across_chunks(seed):
    """A first member of 66000 stored random bytes, then a member whose dynamic blocks were deflated against the first member's tail
    as a preset dictionary: its references reach before its own start, from a block that lies in the second 64 KiB chunk, so the
    device meets them as markers of a chunk decoded from a block-search candidate, not inside the chunk that saw the header."""
    rng = np.random.default_rng(seed)
    a = rng.integers(0, 256, 66000, dtype=np.uint8).tobytes()
    text = a[-20000:] + fastq(200, seed)
    co = zlib.compressobj(6, zlib.DEFLATED, -15, 8, zlib.Z_DEFAULT_STRATEGY, a[-32768:])
    body = co.compress(text) + co.flush()
    return (gzip.compress(a, 0, mtime=0) + b"\x1f\x8b\x08\x00\x00\x00\x00\x00\x00\xff" + body +
            struct.pack("<II", zlib.crc32(text), len(text)))


def corpus(seed=0, big=True):
    """name -> gzip bytes.  big=False keeps every entry small enough for the pure-Python model."""
    n = 20000 if big else 2500
    fq = fastq(n, seed)
    c = {}
    for lv in (1, 6, 9):
        c["fastq_l%d" % lv] = gzip.compress(fq, lv, mtime=0)
    c["fixed"] = deflate(fq, 6, zlib.Z_FIXED)
    c["huffman_only"] = deflate(fq, 6, zlib.Z_HUFFMAN_ONLY)
    c["rle"] = deflate(fq, 6, zlib.Z_RLE)
    c["stored"] = deflate(fq, 0)
    c["sync_full_flush"] = deflate(fq, 6, flushes=[(len(fq) // 5, zlib.Z_SYNC_FLUSH), (len(fq) // 3, zlib.Z_FULL_FLUSH),
                                                   (len(fq) // 2, zlib.Z_SYNC_FLUSH)])
    c["false_candidates"] = false_candidates(seed)[0]
    rng = np.random.default_rng(seed + 1)
    noise = rng.integers(0, 256, 200000 if big else 70000, dtype=np.uint8).tobytes()
    # a long stored / fixed stretch (chunks without a candidate), then dynamic blocks again
    c["no_candidates"] = deflate(noise + fq[:50000], 6, zlib.Z_FIXED) if not big else gzip.compress(noise, 0) + gzip.compress(fq, 6)
    # back-references near the 32 KiB window edge across chunk and call edges: a random block repeated at distance 32000 (zlib's
    # encoder reaches at most 32506 back)
    blk = rng.integers(0, 256, 32000, dtype=np.uint8).tobytes()
    c["window_edge"] = gzip.compress(blk * (40 if big else 8), 9)
    c["zeros"] = gzip.compress(bytes((1 << 22) * (8 if big else 1)), 9)         # ~1000:1: slot overflows
    c["multi_member"] = gzip.compress(fq[:30000], 6) + gzip.compress(b"", 6) + gzip.compress(fq[30000:], 1)
    c["bgzf"] = bgzf_model(fq) + bgzf_model(b"")
    c["header_flags"] = with_header_flags(fq)
    c["trailing_bytes"] = gzip.compress(fq, 6) + b"\x00trailing garbage\n"
    c["distance_32768"] = distance_32768(seed)
    # empty members with FHCRC, more of them than one chunk's event list holds
    empty = b"\x1f\x8b\x08\x02\x00\x00\x00\x00\x00\xff"
    empty += struct.pack("<H", zlib.crc32(empty) & 0xffff) + b"\x03\x00" + struct.pack("<II", 0, 0)
    c["many_fhcrc_members"] = empty * 2100 + gzip.compress(fq[:5000], 6)
    return c


def _delivered(rest):
    """Bytes zlib's inflate delivers from one member before it reports an error (byte-by-byte feeding, exact)."""
    d = zlib.decompressobj(31)
    got = []
    for i in range(len(rest)):
        snap = d.copy()
        try:
            got.append(d.decompress(rest[i:i + 1]))
        except zlib.error:
            buf = rest[i:i + 1]
            while True:
                try:
                    o = snap.decompress(buf, 1)
                except zlib.error:
                    return b"".join(got)
                got.append(o)
                buf = snap.unconsumed_tail
                if not o and not buf:
                    return b"".join(got)
    return b"".join(got)


def zlib_reference(data):
    """(bytes zlib delivers, None | "error" | "truncated"), walking the members through unused_data; bytes after the last member
    that do not start with the gzip magic are ignored, as gzread ignores them."""
    out, pos, first = [], 0, True
    while True:
        rest = data[pos:]
        if not first and (len(rest) < 2 or rest[:2] != b"\x1f\x8b"):
            return b"".join(out), None
        d = zlib.decompressobj(31)
        try:
            o = d.decompress(rest)
        except zlib.error:
            return b"".join(out) + _delivered(rest), "error"
        out.append(o)
        if not d.eof:
            return b"".join(out), "truncated"
        pos = len(data) - len(d.unused_data)
        first = False
