"""Device gzip inflate (mp_gunzip_*): byte-for-byte equality with zlib on a seeded corpus, fed whole and in pieces, the same bytes
and MP_ERR_FORMAT where zlib refuses a truncated or corrupt stream, the block-search counters against the CPU model's plan, large
inputs over many chunks and calls, and concurrency with other work of the same context."""
import gzip
import threading
import zlib

import numpy as np
import pytest

import gz_corpus

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx():
    import megapath_b200 as mp
    c = mp.Context(0)
    yield c
    c.close()


@pytest.fixture(scope="module")
def corpus():
    return gz_corpus.corpus(0, big=True)


def _check_equal(got, want, name):
    if got != want:
        i = next((k for k in range(min(len(got), len(want))) if got[k] != want[k]), min(len(got), len(want)))
        raise AssertionError("%s: %d bytes vs zlib %d, first difference at %d" % (name, len(got), len(want), i))


def test_corpus_one_call(ctx, corpus):
    for name, data in corpus.items():
        want, err = gz_corpus.zlib_reference(data)
        assert err is None, name
        _check_equal(ctx.gunzip(data), want, name)


def test_corpus_in_pieces(ctx, corpus):
    rng = np.random.default_rng(5)
    import megapath_b200 as mp
    for name, data in corpus.items():
        want, _ = gz_corpus.zlib_reference(data)
        for _ in range(2):
            piece = int(rng.choice([mp.GUNZIP_MIN_DST, 65536 + int(rng.integers(1, 200000)), 1 << 20]))
            cap = int(rng.choice([mp.GUNZIP_MIN_DST, 65536 + int(rng.integers(1, 1 << 20)), 16 << 20]))
            _check_equal(ctx.gunzip(data, piece=piece, out_cap=cap), want, "%s piece %d cap %d" % (name, piece, cap))


def test_counters_match_model(ctx, corpus):
    """The device's block search and chain repair follow the CPU model's plan exactly, entry by entry."""
    from oracle import pygunzip
    small = gz_corpus.corpus(0, big=False)
    for name, data in small.items():
        with ctx.gunzip_stream(max(len(data), 65536)) as g:
            out, used, done = g.run(data, True, 64 << 20)
            st = g.stats()
        assert done, name
        plan = pygunzip.plan(data)
        for k in ("chunks", "candidates", "false_candidates", "merged", "overflows", "candidates_tested", "rounds", "members"):
            assert st[k] == plan[k], (name, k, st[k], plan[k])
    # the paths the corpus exists for really ran on the device
    with ctx.gunzip_stream(len(corpus["false_candidates"])) as g:
        g.run(corpus["false_candidates"], True, 64 << 20)
        assert g.stats()["false_candidates"] > 0
    with ctx.gunzip_stream(len(corpus["zeros"])) as g:
        g.run(corpus["zeros"], True, 64 << 20)
        assert g.stats()["overflows"] > 0


def test_large_fastq_many_chunks_and_calls(ctx):
    base = gz_corpus.fastq(100000, 11)            # ~13 MB of text
    rng = np.random.default_rng(3)
    parts, total = [], 0
    while total < (256 << 20):
        # reshuffle record order so that the stream does not repeat at the 32 KiB scale
        k = int(rng.integers(0, len(base) // 2))
        parts.append(base[k:] + base[:k])
        total += len(base)
    text = b"".join(parts)
    data = gzip.compress(text, 6)
    with ctx.gunzip_stream(32 << 20) as g:
        out = g.inflate(memoryview(data), 48 << 20)
        st = g.stats()
    assert out == text
    assert st["chunks"] > 100


def test_truncation_and_corruption(ctx):
    import megapath_b200 as mp
    rng = np.random.default_rng(9)
    text = gz_corpus.fastq(1500, 2)
    cases = [gzip.compress(text, 6), gz_corpus.deflate(text, 6, zlib.Z_FIXED), gz_corpus.deflate(text, 0), gz_corpus.far_back_member(),
             gz_corpus.far_back_across_chunks(4)]
    for data in cases:
        variants = [data[:int(rng.integers(1, len(data)))] for _ in range(6)] + [data[:len(data) - 4], data[:len(data) - 8], data[:5]]
        for _ in range(6):
            b = bytearray(data)
            b[int(rng.integers(10, len(b)))] ^= 1 << int(rng.integers(0, 8))
            variants.append(bytes(b))
        tail = bytearray(data); tail[-8] ^= 1; variants.append(bytes(tail))          # CRC-32
        tail = bytearray(data); tail[-1] ^= 1; variants.append(bytes(tail))          # ISIZE
        for v in variants:
            want, err = gz_corpus.zlib_reference(v)
            if err is None:
                assert ctx.gunzip(v) == want
                continue
            with pytest.raises(mp.GzipFormatError) as e:
                ctx.gunzip(v)
            _check_equal(e.value.partial, want, "damaged stream (%s)" % err)
    # the reference before its member's start is met as a marker of a chunk decoded from a candidate: refused by the marker check
    data = gz_corpus.far_back_across_chunks(4)
    with ctx.gunzip_stream(len(data)) as g:
        with pytest.raises(mp.GzipFormatError) as e:
            g.run(data, True, 64 << 20)
        assert g.stats()["chunks"] >= 2
    assert e.value.partial == gz_corpus.zlib_reference(data)[0] and "too far back" in str(e.value)


def test_two_clones_two_threads_and_batch_untouched(ctx, corpus):
    import megapath_b200 as mp
    a, b = corpus["fastq_l6"], corpus["bgzf"]
    wa, wb = gz_corpus.zlib_reference(a)[0], gz_corpus.zlib_reference(b)[0]
    from tools import synth
    owner = mp.Context(0)
    seq, bounds = synth.make_ref(20000, 1, seed=3, repeat_frac=0.0)
    owner.index_build(mp.pack_text(np.searchsorted(np.frombuffer(b"ACGT", dtype=np.uint8), seq).astype(np.uint8)), len(seq))
    c1, c2 = owner.clone(), owner.clone()
    res = {}

    def work(c, data, key):
        res[key] = [c.gunzip(data, piece=1 << 20, out_cap=4 << 20) for _ in range(3)]
    ts = [threading.Thread(target=work, args=(c1, a, "a")), threading.Thread(target=work, args=(c2, b, "b"))]
    [t.start() for t in ts]
    [t.join() for t in ts]
    assert all(x == wa for x in res["a"]) and all(x == wb for x in res["b"])
    # a gunzip call between the device FASTQ upload and the work on that batch leaves the resident batch as it was
    r1, r2 = synth.make_pairs(seq, bounds, 64, 100, seed=3, model="divergent", one_random=0.1)
    t1 = b"".join(b"@p%d/1\n" % i + x.tobytes() + b"\n+\n" + b"I" * len(x) + b"\n" for i, x in enumerate(r1))
    t2 = b"".join(b"@p%d/2\n" % i + x.tobytes() + b"\n+\n" + b"I" * len(x) + b"\n" for i, x in enumerate(r2))
    P = mp.default_params(insert_low=1, insert_high=750, max_read_length=101)
    c1.fastq_upload(t1, t2, len(r1), 101)
    c1.seed_pairs(P)
    before = [x.tobytes() for x in c1.download_seedpos()]
    c1.fastq_upload(t1, t2, len(r1), 101)
    assert c1.gunzip(a) == wa
    c1.seed_pairs(P)
    assert [x.tobytes() for x in c1.download_seedpos()] == before
    c1.close(); c2.close(); owner.close()


def test_argument_errors(ctx):
    import ctypes as C
    import megapath_b200 as mp
    L = mp.lib()
    h = C.c_void_p()
    assert L.mp_gunzip_open(None, 1 << 20, C.byref(h)) == -3
    assert L.mp_gunzip_open(ctx.h, 0, C.byref(h)) == -3
    with ctx.gunzip_stream(1 << 20) as g:
        data = gzip.compress(b"x" * 1000)
        dst = C.create_string_buffer(1 << 20)
        u, p, d = C.c_uint64(), C.c_uint64(), C.c_int()
        assert L.mp_gunzip_run(g.h, data, len(data), 1, dst, mp.GUNZIP_MIN_DST - 1, C.byref(u), C.byref(p), C.byref(d)) == -3
        assert L.mp_gunzip_run(g.h, data, (1 << 20) + 1, 1, dst, 1 << 20, C.byref(u), C.byref(p), C.byref(d)) == -3
        assert L.mp_gunzip_run(g.h, data, len(data), 1, None, 1 << 20, C.byref(u), C.byref(p), C.byref(d)) == -3
        assert L.mp_gunzip_stats(g.h, None) == -3
        assert L.mp_gunzip_run(g.h, data, len(data), 1, dst, 1 << 20, C.byref(u), C.byref(p), C.byref(d)) == 0
        assert d.value == 1 and p.value == 1000 and u.value == len(data)
    with pytest.raises(mp.GzipFormatError):
        ctx.gunzip(b"not a gzip file at all")
