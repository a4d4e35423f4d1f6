"""CPU suite: the model of the device gzip inflater (oracle/pygunzip.py) against zlib, on the seeded corpus of tests/gz_corpus.py and
on truncated and corrupted streams, and proof that the corpus reaches the paths it exists for."""
import os
import re
import struct
import zlib

import numpy as np

import gz_corpus
from oracle import pygunzip as pg

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_constants_match_header():
    import megapath_b200 as mp
    txt = open(os.path.join(ROOT, "include", "megapath_b200.h")).read()
    assert re.search(r"#define MP_GUNZIP_CHUNK (\d+)u", txt).group(1) == str(mp.GUNZIP_CHUNK)
    assert "#define MP_GUNZIP_SLOT (1u << %d)" % (mp.GUNZIP_SLOT.bit_length() - 1) in txt
    assert "#define MP_GUNZIP_EVENTS (MP_GUNZIP_CHUNK / 16u + 8u)" in txt and mp.GUNZIP_EVENTS == mp.GUNZIP_CHUNK // 16 + 8
    assert re.search(r"#define MP_GUNZIP_MIN_DST (\d+)u", txt).group(1) == str(mp.GUNZIP_MIN_DST)


def test_model_equals_zlib_on_corpus():
    for name, data in gz_corpus.corpus(0, big=False).items():
        want, err = gz_corpus.zlib_reference(data)
        assert err is None, name
        got, gerr = pg.gunzip(data)
        assert (got, gerr) == (want, None), name
        p = pg.plan(data)
        assert p["output"] == want and p["status"] == pg.S_END and p["crc_ok"], name


def test_true_boundaries_pass_the_search_test():
    """Every true dynamic block header (non-final) passes the block search's test: the search can only err towards false
    candidates, which the chain repairs, never towards missing a true start it reaches first."""
    data = gz_corpus.corpus(0, big=False)["fastq_l6"]
    out, st, bounds = pg.inflate(data)
    br = pg.Bits(data)
    dyn = [b for b, _ in bounds if (br.peek(b)[0] & 7) == 4]
    assert len(dyn) > 10
    assert all(pg.dyn_header_valid(data, b, br) for b in dyn)


def _damaged_cases():
    text = gz_corpus.fastq(300, 4)
    base = (gzip_member(text[:20000], 6) + gz_corpus.deflate(text[20000:40000], 6, zlib.Z_FIXED) + gz_corpus.deflate(text[40000:], 0) +
            gzip_member(text, 1))
    rng = np.random.default_rng(17)
    cases = [base[:int(k)] for k in rng.choice(np.arange(1, len(base)), 200, replace=False)]
    for _ in range(40):
        b = bytearray(base)
        b[int(rng.integers(0, len(b)))] ^= 1 << int(rng.integers(0, 8))
        cases.append(bytes(b))
    for off in (8, 7, 4, 1):                                   # CRC-32 and ISIZE of the last member
        b = bytearray(base); b[-off] ^= 0x10; cases.append(bytes(b))
    cases.append(gz_corpus.far_back_member())
    cases.append(gz_corpus.far_back_across_chunks(4))
    return cases


def gzip_member(data, level):
    import gzip
    return gzip.compress(data, level, mtime=0)


def test_model_equals_zlib_on_damaged_streams():
    for v in _damaged_cases():
        want, err = gz_corpus.zlib_reference(v)
        got, gerr = pg.gunzip(v)
        assert got == want, (len(v), len(got), len(want), err, gerr)
        assert (gerr is None) == (err is None)


def test_corpus_reaches_every_path():
    c = gz_corpus.corpus(0, big=False)
    p = pg.plan(c["false_candidates"])
    assert p["false_candidates"] > 0 and p["rounds"] == 1 + p["false_candidates"]
    _, payload = gz_corpus.false_candidates(0)
    cands, _ = pg.find(c["false_candidates"])
    out, _, bounds = pg.inflate(c["false_candidates"])
    true_bits = {b for b, _ in bounds}
    assert any(x is not None and x not in true_bits for x in cands)          # a valid header inside a stored payload
    assert pg.plan(c["zeros"])["overflows"] > 0                              # slot overflow and resume
    assert pg.plan(c["fixed"])["merged"] == pg.plan(c["fixed"])["chunks"] - 1  # no dynamic block: every chunk merged
    assert pg.plan(c["no_candidates"])["merged"] > 0
    assert pg.plan(c["multi_member"])["members"] == 3
    assert pg.plan(c["bgzf"])["members"] > 5
    assert pg.plan(c["many_fhcrc_members"])["overflows"] > 0                 # a full event list stops before a header, not inside it
    hf = c["header_flags"]
    assert hf[3] == 0x1f and len(hf) > 65000                                 # FTEXT FHCRC FEXTRA FNAME FCOMMENT, a long FEXTRA
    # the second member's first match reaches before the member: refused after its first literal
    got, err = pg.gunzip(gz_corpus.far_back_member())
    assert err == "error" and got.endswith(b"89x")
    # trailing bytes after the last member are ignored
    assert pg.gunzip(c["trailing_bytes"])[1] is None
    # a wrong header CRC is refused
    b = bytearray(hf)
    hlen = 10 + 2 + struct.unpack("<H", hf[10:12])[0] + len(b"reads.fq\x00a comment\x00")
    b[hlen] ^= 1
    assert pg.gunzip(bytes(b)) == (b"", "error")
