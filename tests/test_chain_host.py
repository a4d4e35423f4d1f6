"""CPU suite for soap4 -chain (the NT chunk chain in one process): the host rewrite of one chunk's stdout into the next chunk's two
read files (soap4_hosttest __deinterleave) against the rule tests/conftest.py's deinterleave applies, and the -chain argument checks."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT, BIN_DIR


def deinterleave_ordered(data):
    """conftest.deinterleave without its canonical sort: formatted soap4 -F text -> (mate 1 text, mate 2 text)."""
    lines = data.split(b"\n")
    recs = [lines[i:i + 4] for i in range(0, len(lines) - 3, 4)]
    out = [[], []]
    for k in range(0, len(recs) - 1, 2):
        for mate in (0, 1):
            hdr, sq, _, ql = recs[k + mate]
            parts = hdr[1:].split(None, 1)
            name, comm = parts[0], (parts[1] if len(parts) > 1 else b"")
            if name.endswith(b"/1") or name.endswith(b"/2"):
                name = name[:-2]
            out[mate].append(b"@" + name + b"/%d" % (mate + 1) + (b" " + comm if comm else b"") + b"\n" + sq + b"\n+\n" + ql + b"\n")
    return b"".join(out[0]), b"".join(out[1])


def _hosttest():
    exe = os.path.join(BIN_DIR, "soap4_hosttest")
    if not os.path.exists(exe):
        import megapath_b200 as mp
        mp.build()
    return exe


def random_formatted_text(rng, n_pairs):
    """Text of the form soap4 -F / -P prints: "@name\\tSCORE:...;" or "@name\\tIGNORE" headers, with names of every kind the rewrite
    treats differently."""
    names = [b"r%d", b"r%d/1", b"r%d/2", b"r%d/3", b"r%d/1/2", b"/1", b"/2", b"", b"r%d/", b"x/12", b"r%d/2/1"]
    seqnames = [b"chunk1_%d second index" % i for i in range(1, 8)] + [b"seq%d" % i for i in range(1, 5)]
    recs = []
    for p in range(n_pairs):
        for mate in (0, 1):
            nm = names[rng.integers(len(names))]
            nm = nm % p if b"%d" in nm else nm
            kind = rng.integers(6)
            if kind == 0:
                tail = b"\tIGNORE"
            elif kind == 1:
                tail = b"\tSCORE:0;"
            else:
                best = int(rng.integers(1, 300))
                entries = b"".join(b"%d,%s;" % (int(rng.integers(1, best + 1)), seqnames[rng.integers(len(seqnames))])
                                   for _ in range(int(rng.integers(0, 400 if kind == 5 else 4))))
                tail = b"\tSCORE:%d;" % best + entries
            L = int(rng.integers(1, 160))
            seq = bytes(rng.choice(list(b"ACGT"), size=L))
            qual = bytes(rng.integers(33, 74, size=L).astype(np.uint8))
            recs.append(b"@" + nm + tail + b"\n" + seq + b"\n+\n" + qual + b"\n")
    return b"".join(recs)


@pytest.mark.parametrize("seed", [1, 2, 3])
def test_host_deinterleave_equals_the_rule(tmp_path, seed):
    rng = np.random.default_rng(seed)
    data = random_formatted_text(rng, 3000 if seed == 1 else 300)
    path = str(tmp_path / "fmt.fq")
    open(path, "wb").write(data)
    subprocess.run([_hosttest(), "__deinterleave", path], check=True, timeout=120)
    want1, want2 = deinterleave_ordered(data)
    assert open(path + "_1.fq", "rb").read() == want1
    assert open(path + "_2.fq", "rb").read() == want2


def test_library_exports_the_chain_entry_points():
    import megapath_b200 as mp
    if not os.path.exists(mp.LIB_PATH):
        mp.build()
    lib = ctypes.CDLL(mp.LIB_PATH)
    for s in ("mp_index_bind", "mp_fastq_chain", "mp_index_load_budget"):
        assert hasattr(lib, s), s


@pytest.mark.parametrize("args,message", [
    (["-F", "-nc", "-chain", "idx1"], b"Please specify the index prefix and the output prefix after '-chain'"),
    (["-F", "-nc", "-chain"], b"Please specify the index prefix and the output prefix after '-chain'"),
    (["-nc", "-chain", "idx1", "out1"], b"-chain needs -F or -P"),
])
def test_chain_arguments_are_checked(tmp_path, args, message):
    _hosttest()
    exe = os.path.join(BIN_DIR, "soap4")
    cmd = [exe, "pair", str(tmp_path / "idx0"), str(tmp_path / "a.fq"), str(tmp_path / "b.fq"), "-o", str(tmp_path / "o"),
           "-C", os.path.join(ROOT, "megapath_b200", "ini", "soap4-nt2.ini")] + args
    p = subprocess.run(cmd, capture_output=True, timeout=60)
    assert p.returncode == 1
    assert message in p.stderr
