"""GPU suite: BGZF compression on the device (mp_bgzf_compress, csrc/mp_bgzf.cu) checked with an independent inflater (Python's
zlib / gzip), member by member, against zlib's ratio on the same pieces, for determinism, and through the driver's -b output against
the zlib path that MP_HOST_IO=1 keeps; and byte for byte against the restatement oracle/pybgzf.py on the corpus of
tests/test_bgzf_model.py, across grids, contexts and reserve sizes."""
import ctypes
import gzip
import os
import struct
import subprocess
import zlib

import numpy as np
import pytest

from conftest import ROOT, make_reads
from test_bgzf_model import CORPUS, model_of

pytestmark = pytest.mark.gpu

PIECE = 0xff00
EOF_MEMBER = bytes.fromhex("1f8b08040000000000ff0600424302001b0003000000000000000000")


@pytest.fixture(scope="module")
def ctx():
    import megapath_b200 as mp
    c = mp.Context(0)
    yield c
    c.close()


def bam_like(n_records, seed):
    """Seeded BAM records as the driver writes them: 150 bp, Illumina-like qualities, RG/NM/X0/X1/XM/XO/XG/PH tags."""
    rng = np.random.default_rng(seed)
    out = bytearray()
    nt16 = np.array([1, 2, 4, 8], np.uint8)
    for i in range(n_records):
        name = b"read_%08d" % (i // 2)
        L = 150
        codes = rng.integers(0, 4, L)
        seq = (nt16[codes[0::2]] << 4 | nt16[codes[1::2]]).astype(np.uint8).tobytes()
        q = np.clip(np.round(36 - np.abs(rng.normal(0, 3, L)) - np.linspace(0, 8, L)), 2, 41).astype(np.uint8)
        q[rng.random(L) < 0.02] = 2
        mapped = rng.random() < 0.8
        ncig = 1 if mapped else 0
        cig = struct.pack("<I", L << 4) if mapped else b""
        aux = b"RGZsample_1.fq\0"
        if mapped:
            aux += b"NMi" + struct.pack("<i", int(rng.integers(0, 4))) + b"X0i" + struct.pack("<i", 1) + b"X1i" + struct.pack("<i", 0)
            aux += b"XMi" + struct.pack("<i", int(rng.integers(0, 4))) + b"XOi" + struct.pack("<i", 0) + b"XGi" + struct.pack("<i", 0)
            aux += b"PHi" + struct.pack("<i", 1)
        body = name + b"\0" + cig + seq + q.tobytes() + aux
        tid = int(rng.integers(0, 6)) if mapped else -1
        pos = int(rng.integers(0, 50000)) if mapped else -1
        flag = (0x1 | (0x40 if i % 2 == 0 else 0x80) | (0 if mapped else 0x4))
        hdr = struct.pack("<iiiIIiiii", 32 + len(body), tid, pos, (len(name) + 1) | (37 << 8), flag << 16 | ncig, L, tid, pos, 0)
        out += hdr + body
    return bytes(out)


def fastq_text(n_records, seed):
    rng = np.random.default_rng(seed)
    out = bytearray()
    for i in range(n_records):
        bases = np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, 150)].tobytes()
        q = (33 + np.clip(np.round(36 - np.abs(rng.normal(0, 3, 150))), 2, 41)).astype(np.uint8).tobytes()
        out += b"@read_%d/%d\tSCORE:%d;0,seq%d;\n" % (i // 2, i % 2 + 1, int(rng.integers(100, 151)), int(rng.integers(1, 7))) + bases + b"\n+\n" + q + b"\n"
    return bytes(out)


def window_edge(distance, n=70000, seed=5):
    """random bytes with one random 300-byte pattern repeated `distance` bytes later (32768 is the DEFLATE window, 32769 is just past it)"""
    rng = np.random.default_rng(seed)
    b = bytearray(rng.integers(0, 256, n, dtype=np.uint8).tobytes())
    b[1000 + distance:1300 + distance] = b[1000:1300]
    return bytes(b)


def contents(kind, n):
    rng = np.random.default_rng(n + 17)
    if kind == "zeros":
        return bytes(n)
    if kind == "repeat":
        return b"\x5a" * n
    if kind == "random":
        return rng.integers(0, 256, n, dtype=np.uint8).tobytes()
    if kind == "skewed":                     # a skewed histogram over all byte values, repeats only by chance
        return np.minimum(rng.geometric(0.02, n), 255).astype(np.uint8).tobytes()
    if kind == "all256":
        return (np.arange(n) % 256).astype(np.uint8).tobytes()
    if kind == "bam":
        return bam_like(n // 250 + 2, seed=n)[:n]
    if kind == "fastq":
        return fastq_text(n // 300 + 2, seed=n)[:n]
    raise ValueError(kind)


def walk_members(raw, data):
    """every member: gzip magic, FEXTRA with the BC subfield, BSIZE, ISIZE <= 0xff00, CRC-32 of the piece it decodes to"""
    at, pieces = 0, 0
    while at < len(raw):
        assert raw[at:at + 4] == b"\x1f\x8b\x08\x04" and raw[at + 10:at + 12] == b"\x06\x00" and raw[at + 12:at + 16] == b"BC\x02\x00"
        bsize = int.from_bytes(raw[at + 16:at + 18], "little") + 1
        assert bsize <= 65536
        crc, isize = struct.unpack_from("<II", raw, at + bsize - 8)
        assert 0 < isize <= PIECE
        piece = zlib.decompress(raw[at + 18:at + bsize - 8], -15)
        assert len(piece) == isize and piece == data[pieces * PIECE:pieces * PIECE + isize]
        assert zlib.crc32(piece) == crc
        at += bsize
        pieces += 1
    assert at == len(raw)
    assert pieces == (len(data) + PIECE - 1) // PIECE


SIZES = [0, 1, 2, PIECE - 1, PIECE, PIECE + 1, 1 << 20]
KINDS = ["zeros", "repeat", "random", "skewed", "all256", "bam", "fastq"]


@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("size", SIZES)
def test_round_trip(ctx, kind, size):
    data = contents(kind, size)
    raw = ctx.bgzf_compress(data)
    assert len(raw) <= (size + PIECE - 1) // PIECE * 65536
    assert gzip.decompress(raw) == data
    walk_members(raw, data)


@pytest.mark.parametrize("distance", [32768, 32769])
def test_window_edge(ctx, distance):
    data = window_edge(distance)
    raw = ctx.bgzf_compress(data)
    assert gzip.decompress(raw) == data
    walk_members(raw, data)


@pytest.mark.parametrize("kind", ["bam", "zeros", "random"])
def test_many_pieces(ctx, kind):
    """>= 64 MiB: about a thousand pieces, several per CTA"""
    if kind == "bam":
        one = bam_like(3000, seed=9)
        data = (one * ((64 << 20) // len(one) + 1))[:(64 << 20) + 12345]
    elif kind == "zeros":
        data = bytes((64 << 20) + 3)
    else:
        data = np.random.default_rng(4).integers(0, 256, (64 << 20) + 7, dtype=np.uint8).tobytes()
    raw = ctx.bgzf_compress(data)
    assert gzip.decompress(raw) == data
    walk_members(raw, data)


def zlib_pieces(data, level):
    total = 0
    for at in range(0, len(data), PIECE):
        c = zlib.compressobj(level, zlib.DEFLATED, -15, 8)
        total += len(c.compress(data[at:at + PIECE]) + c.flush()) + 26
    return total


@pytest.mark.parametrize("kind", ["bam", "fastq"])
def test_ratio_within_115_percent_of_zlib6(ctx, kind):
    data = contents(kind, 8 << 20)
    got = len(ctx.bgzf_compress(data))
    want = zlib_pieces(data, 6)
    assert got <= 1.15 * want, (got, want, got / want)


def test_deterministic_across_calls_and_contexts(ctx):
    import megapath_b200 as mp
    from tools import synth
    data = contents("bam", 3 << 20) + contents("fastq", 1 << 20) + contents("zeros", 100000)
    a = ctx.bgzf_compress(data)
    assert ctx.bgzf_compress(data) == a
    owner = mp.Context(0)
    seq, _ = synth.make_ref(20000, 1, seed=3, repeat_frac=0.0)
    codes = np.searchsorted(np.frombuffer(b"ACGT", dtype=np.uint8), seq).astype(np.uint8)
    owner.index_build(mp.pack_text(codes), len(codes))
    clone = owner.clone()
    assert clone.bgzf_compress(data) == a
    assert owner.bgzf_compress(data) == a
    clone.close()
    owner.close()


def test_argument_errors(ctx):
    import megapath_b200 as mp
    L = mp.lib()
    data = contents("bam", 100000)
    bound = mp.bgzf_bound(len(data))
    assert bound == 2 * 65536
    buf = ctypes.create_string_buffer(b"\xee" * (bound + 64), bound + 64)
    n = ctypes.c_uint64(12345)
    rc = L.mp_bgzf_compress(ctx.h, ctypes.c_char_p(data), len(data), buf, bound - 1, ctypes.byref(n))
    assert rc == -3 and n.value == 0
    assert buf.raw == b"\xee" * (bound + 64)
    rc = L.mp_bgzf_compress(ctx.h, ctypes.c_char_p(data), len(data), buf, bound, ctypes.byref(n))
    assert rc == 0 and 0 < n.value <= bound and buf.raw[n.value:] == b"\xee" * (bound + 64 - n.value)
    assert gzip.decompress(buf.raw[:n.value]) == data
    # n == 0 writes nothing, whatever the capacity
    empty = ctypes.create_string_buffer(b"\xee" * 64, 64)
    rc = L.mp_bgzf_compress(ctx.h, None, 0, empty, 0, ctypes.byref(n))
    assert rc == 0 and n.value == 0 and empty.raw == b"\xee" * 64
    assert ctx.bgzf_compress(b"") == b""
    assert L.mp_bgzf_compress(ctx.h, None, 10, buf, bound, ctypes.byref(n)) == -3
    assert L.mp_bgzf_reserve(ctx.h, 0) == -3
    ctx.bgzf_reserve(1 << 20)


# ---- byte for byte against the restatement (oracle/pybgzf.py; its own checks are in tests/test_bgzf_model.py) ----

def first_difference(got, want):
    """where two member runs part: the first differing member, with what parse_member makes of each side"""
    from oracle import pybgzf
    gm, wm = pybgzf.split_members(got), pybgzf.split_members(want)
    k = next((k for k, (g, w) in enumerate(zip(gm, wm)) if g != w), None)
    if k is None:
        return "%d members from the device, %d from the model" % (len(gm), len(wm))
    msg, tokens = "member %d differs" % k, []
    for side, m in (("device", gm[k]), ("model", wm[k])):
        try:
            P = pybgzf.parse_member(m)
        except pybgzf.DeflateError as e:
            msg += "\n  %s: undecodable: %s" % (side, e)
            continue
        tokens.append(P["tokens"])
        msg += "\n  %s: %d bytes, btype %d, HLIT %s HDIST %s HCLEN %s, %d tokens, lit lens %s, dist lens %s, cl lens %s" % (
            side, len(m), P["btype"], P["hlit"], P["hdist"], P["hclen"], len(P["tokens"]), P["lit_lens"], P["dist_lens"], P["cl_lens"])
    if len(tokens) == 2:
        a, b = tokens
        j = next((j for j, (x, y) in enumerate(zip(a, b)) if x != y), min(len(a), len(b)))
        msg += "\n  first differing token #%d: device %s, model %s" % (j, a[j] if j < len(a) else None, b[j] if j < len(b) else None)
    return msg


def assert_same_stream(got, want):
    assert got == want, first_difference(got, want)


@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("size", SIZES)
def test_device_equals_model(ctx, kind, size):
    from oracle import pybgzf
    data = contents(kind, size)
    assert_same_stream(ctx.bgzf_compress(data), pybgzf.compress(data))


@pytest.mark.parametrize("name", CORPUS)
def test_device_equals_model_on_the_corpus(ctx, name):
    """inputs that limit the literal/length and code-length trees, every length and distance code, the 32768 / 32769 window edge,
    hash collisions, piece lengths at the ok3 / ok4 and tile edges"""
    data, want, _ = model_of(name)
    assert_same_stream(ctx.bgzf_compress(data), want)


def sm_count():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def test_many_pieces_equal_the_model_at_sampled_pieces(ctx):
    """64 MiB (about a thousand pieces, several per CTA): the first and last pieces, pieces sms - 1, sms, sms + 1 and 2 sms (the
    second and third rounds of the persistent loop) and a seeded dozen, member bytes against the model"""
    from oracle import pybgzf
    one = bam_like(3000, seed=11) + fastq_text(2000, seed=12)
    data = (one * ((64 << 20) // len(one) + 1))[:(64 << 20) + 4321]
    members = pybgzf.split_members(ctx.bgzf_compress(data))
    n = len(members)
    assert n == (len(data) + PIECE - 1) // PIECE
    sms = sm_count()
    sample = {0, n - 1, sms - 1, sms, sms + 1, 2 * sms} | set(np.random.default_rng(8).choice(n, 12, replace=False).tolist())
    for k in sorted(sample):
        assert members[k] == pybgzf.member(data[k * PIECE:(k + 1) * PIECE]), "piece %d of %d (%d SMs)" % (k, n, sms)


def test_output_does_not_depend_on_the_grid(ctx):
    """one call over 3 sms + 5 pieces (sms CTAs, three or four pieces each) == calls on slices cut at piece boundaries (grids of 1,
    2, 7, sms - 1, sms, sms + 1 CTAs), concatenated"""
    sms = sm_count()
    data = contents("fastq", (3 * sms + 5) * PIECE - 77)
    whole = ctx.bgzf_compress(data)
    parts, at = [], 0
    for pieces in (1, 2, 7, sms - 1, sms, sms + 1, None):
        end = len(data) if pieces is None else at + pieces * PIECE
        parts.append(ctx.bgzf_compress(data[at:end]))
        at = end
    assert at == len(data)
    assert_same_stream(b"".join(parts), whole)


def test_two_contexts_at_once():
    """two clones of one index owner compress different inputs at the same time from two threads (one context per worker thread,
    as the driver runs them); each result equals the model's"""
    import threading
    import megapath_b200 as mp
    from oracle import pybgzf
    from tools import synth
    owner = mp.Context(0)
    seq, _ = synth.make_ref(20000, 1, seed=3, repeat_frac=0.0)
    owner.index_build(mp.pack_text(np.searchsorted(np.frombuffer(b"ACGT", dtype=np.uint8), seq).astype(np.uint8)), len(seq))
    clones = [owner.clone(), owner.clone()]
    inputs = [contents("bam", 20 * PIECE + 999), contents("fastq", 23 * PIECE - 5)]
    want = [pybgzf.compress(d) for d in inputs]
    got = [[], []]
    start = threading.Barrier(2)

    def work(k):
        start.wait()
        for _ in range(4):
            got[k].append(clones[k].bgzf_compress(inputs[k]))

    threads = [threading.Thread(target=work, args=(k,)) for k in range(2)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    for k in range(2):
        assert len(got[k]) == 4
        for g in got[k]:
            assert_same_stream(g, want[k])
    for c in clones:
        c.close()
    owner.close()


def test_reserve_sizes():
    """a call after reserving more than it needs, and a call larger than the last reserve, both equal the model"""
    import megapath_b200 as mp
    from oracle import pybgzf
    c = mp.Context(0)
    c.bgzf_reserve(16 << 20)
    small = contents("bam", 5 * PIECE + 17)
    assert_same_stream(c.bgzf_compress(small), pybgzf.compress(small))
    c.bgzf_reserve(PIECE)
    big = contents("fastq", 30 * PIECE + 1)
    assert_same_stream(c.bgzf_compress(big), pybgzf.compress(big))
    assert_same_stream(c.bgzf_compress(small), pybgzf.compress(small))
    c.close()


# ---- the driver's -b output: device compression (default) against zlib on the formatting threads (MP_HOST_IO=1) ----

def run_driver(workdir, prefix, fq1, fq2, name, lopt, ini, flags, env):
    exe = os.path.join(ROOT, "megapath_b200", "bin", "soap4")
    out = os.path.join(workdir, name)
    for suffix in (".dpout.1", ".gout.1", ".unpair"):
        if os.path.exists(out + suffix):
            os.remove(out + suffix)
    cmd = [exe, "pair", prefix, fq1, fq2, "-o", out, "-C", os.path.join(ROOT, "megapath_b200", "ini", ini),
           "-L", str(lopt), "-T", "3", "-u", "750"] + list(flags)
    e = dict(os.environ)
    e.update(env)
    p = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.PIPE, timeout=300, env=e)
    assert p.returncode == 0, p.stderr.decode()[-2000:]
    return p.stdout, {s: open(out + s, "rb").read() for s in (".dpout.1", ".gout.1", ".unpair")}


DRIVER_SETS = [("nt2", "soap4-nt2.ini", ("-b", "-F", "-top", "95")), ("plain", "soap4.ini", ("-b",))]
DRIVER_ENVS = [("batches", {"MP_BATCH_READS": "1024", "MP_CONTEXTS_PER_GPU": "2"}), ("defaults", {})]


@pytest.mark.parametrize("env", DRIVER_ENVS, ids=[e[0] for e in DRIVER_ENVS])
@pytest.mark.parametrize("setup", DRIVER_SETS, ids=[s[0] for s in DRIVER_SETS])
def test_driver_bam_matches_host_compression(workdir, small_ref, setup, env):
    name, ini, flags = setup
    ename, envd = env
    fq1, fq2 = make_reads(workdir, small_ref, "bgzf_" + name, 3000, 150, seed=77, model="divergent", one_random=0.10, unalignable=0.05)
    dev_out, dev = run_driver(workdir, small_ref["prefix"], fq1, fq2, "bgzf_d_%s_%s" % (name, ename), 151, ini, flags, envd)
    host_out, host = run_driver(workdir, small_ref["prefix"], fq1, fq2, "bgzf_h_%s_%s" % (name, ename), 151, ini, flags, dict(envd, MP_HOST_IO="1"))
    assert dev_out == host_out
    for suffix in dev:
        assert dev[suffix].endswith(EOF_MEMBER) and host[suffix].endswith(EOF_MEMBER), suffix
        d, h = gzip.decompress(dev[suffix]), gzip.decompress(host[suffix])
        assert d[:4] == b"BAM\x01"
        assert d == h, suffix
    assert len(gzip.decompress(dev[".unpair"])) > 100000
