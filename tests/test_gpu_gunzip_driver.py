"""GPU suite: bin/soap4 on .fq.gz read files, inflated on the device (mp_gunzip_run on a context per mate file) and fed to the device
FASTQ loop, or to the host parser where that loop does not apply.  Every run is held to the plain .fq device run and to MP_HOST_IO=1,
which reads the same .gz files with gzread."""
import gzip
import os
import subprocess

import pytest

import gz_corpus
from conftest import ROOT, make_reads

pytestmark = pytest.mark.gpu


def run(workdir, prefix, fq1, fq2, name, lopt, ini, flags, env=None, threads=3):
    exe = os.path.join(ROOT, "megapath_b200", "bin", "soap4")
    cmd = [exe, "pair", prefix, fq1, fq2, "-o", os.path.join(workdir, name), "-C", os.path.join(ROOT, "megapath_b200", "ini", ini),
           "-L", str(lopt), "-T", str(threads), "-u", "750"] + list(flags)
    e = dict(os.environ)
    e.update(env or {})
    p = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.PIPE, timeout=300, env=e)
    return p.returncode, p.stdout, p.stderr.decode(errors="replace")


def run_ok(*a, **k):
    rc, out, err = run(*a, **k)
    assert rc == 0, err[-2000:]
    return out, err


def first_diff(a, b):
    la, lb = a.split(b"\n"), b.split(b"\n")
    for i, (x, y) in enumerate(zip(la, lb)):
        if x != y:
            return i, x[:300], y[:300]
    return min(len(la), len(lb)), len(la), len(lb)


def gz(path, data, level=6):
    with open(path, "wb") as f:
        f.write(gzip.compress(data, level))
    return path


# the sets of test_gpu_fastq_io.py (copied): name, read length, -L, read model, .ini, flags
SETS = [
    ("clean", 150, 151, dict(model="clean"), "soap4.ini", ("-F", "-nc")),
    ("mixed", 100, 101, dict(model="divergent", one_random=0.10, unalignable=0.05), "soap4.ini", ("-F", "-nc")),
    ("var", 150, 151, dict(model="clean", varlen=True, n_rate=0.002, one_random=0.05), "soap4.ini", ("-F", "-nc")),
    ("nt2", 150, 151, dict(model="divergent", one_random=0.10, unalignable=0.02), "soap4-nt2.ini", ("-F", "-nc", "-top", "95")),
    ("pmode", 100, 101, dict(model="divergent", one_random=0.10, unalignable=0.05), "soap4.ini", ("-P", "-nc")),
]
CASES = [(s, b) for s in SETS for b in (0, 1024)]


@pytest.mark.parametrize("case", CASES, ids=["%s-%d" % (s[0], b) for s, b in CASES])
def test_gz_equals_plain_and_host(workdir, small_ref, case):
    (name, rlen, lopt, kw, ini, flags), batch = case
    fq1, fq2 = make_reads(workdir, small_ref, "gzd_" + name, 3000, rlen, seed=91, **kw)
    g1, g2 = gz(fq1 + ".gz", open(fq1, "rb").read()), gz(fq2 + ".gz", open(fq2, "rb").read())
    env = {"MP_BATCH_READS": str(batch)} if batch else {}
    plain, _ = run_ok(workdir, small_ref["prefix"], fq1, fq2, "gzd_p_" + name, lopt, ini, flags, env)
    dev, err = run_ok(workdir, small_ref["prefix"], g1, g2, "gzd_d_" + name, lopt, ini, flags, env)
    assert "formatting on the device" in err, err[-1500:]
    host, err2 = run_ok(workdir, small_ref["prefix"], g1, g2, "gzd_h_" + name, lopt, ini, flags, dict(env, MP_HOST_IO="1"))
    assert "formatting on the host" in err2
    assert len(dev) > 100000
    assert dev == plain, first_diff(dev, plain)
    assert dev == host, first_diff(dev, host)


def test_gz_levels_bgzf_multi_member_and_mixed_mates(workdir, small_ref):
    fq1, fq2 = make_reads(workdir, small_ref, "gzm", 3000, 100, seed=5, model="divergent", one_random=0.10, unalignable=0.05)
    t1, t2 = open(fq1, "rb").read(), open(fq2, "rb").read()
    flags, env = ("-F", "-nc"), {"MP_BATCH_READS": "1024"}
    plain, _ = run_ok(workdir, small_ref["prefix"], fq1, fq2, "gzm_p", 101, "soap4.ini", flags, env)
    half = len(t1) // 2
    inputs = {
        "l1": (gz(fq1 + ".l1.gz", t1, 1), gz(fq2 + ".l1.gz", t2, 1)),
        "l6": (gz(fq1 + ".l6.gz", t1, 6), gz(fq2 + ".l6.gz", t2, 6)),
        "bgzf": (fq1 + ".bgzf.gz", fq2 + ".bgzf.gz"),
        "members": (fq1 + ".mm.gz", fq2 + ".mm.gz"),
        "one_mate": (gz(fq1 + ".om.gz", t1, 6), fq2),
    }
    open(inputs["bgzf"][0], "wb").write(gz_corpus.bgzf_model(t1) + gz_corpus.bgzf_model(b""))
    open(inputs["bgzf"][1], "wb").write(gz_corpus.bgzf_model(t2) + gz_corpus.bgzf_model(b""))
    open(inputs["members"][0], "wb").write(gzip.compress(t1[:half], 6) + gzip.compress(b"", 1) + gzip.compress(t1[half:], 9))
    open(inputs["members"][1], "wb").write(gzip.compress(t2[:1000], 1) + gzip.compress(t2[1000:], 6))
    for key, (a, b) in inputs.items():
        dev, err = run_ok(workdir, small_ref["prefix"], a, b, "gzm_" + key, 101, "soap4.ini", flags, env)
        assert "formatting on the device" in err, (key, err[-1500:])
        assert dev == plain, (key, first_diff(dev, plain))


def test_gz_bam_output(workdir, small_ref):
    """-b with .gz inputs (host parser, device inflate): the decoded BAM files equal the MP_HOST_IO=1 run's."""
    fq1, fq2 = make_reads(workdir, small_ref, "gzb", 3000, 150, seed=12, model="divergent", one_random=0.10, unalignable=0.02)
    g1, g2 = gz(fq1 + ".gz", open(fq1, "rb").read()), gz(fq2 + ".gz", open(fq2, "rb").read())
    outs = {}
    for tag, env in (("d", {}), ("h", {"MP_HOST_IO": "1"})):
        run_ok(workdir, small_ref["prefix"], g1, g2, "gzb_" + tag, 151, "soap4-nt2.ini", ("-b", "-F", "-top", "95"), env)
        outs[tag] = {s: gzip.decompress(open(os.path.join(workdir, "gzb_" + tag + s), "rb").read()) for s in (".dpout.1", ".gout.1", ".unpair")}
    assert outs["d"] == outs["h"]
    assert len(outs["d"][".unpair"]) > 10000


def test_gz_lsam(workdir, small_ref):
    fq1, fq2 = make_reads(workdir, small_ref, "gzl", 3000, 100, seed=8, model="divergent", one_random=0.10, unalignable=0.05)
    g1, g2 = gz(fq1 + ".gz", open(fq1, "rb").read()), gz(fq2 + ".gz", open(fq2, "rb").read())
    flags = ["-F", "-nc", "-top", "95", "-lsam", "0"]
    dev, err = run_ok(workdir, small_ref["prefix"], g1, g2, "gzl_d", 101, "soap4-nt2.ini", flags)
    assert "formatting on the device" in err
    host, _ = run_ok(workdir, small_ref["prefix"], g1, g2, "gzl_h", 101, "soap4-nt2.ini", flags, {"MP_HOST_IO": "1"})
    assert dev == host, first_diff(dev, host)


def test_gz_crlf_falls_back_to_host_parser(workdir, small_ref):
    fq1, fq2 = make_reads(workdir, small_ref, "gzc", 3000, 100, seed=23, model="divergent", one_random=0.10, unalignable=0.05)
    g1 = gz(fq1 + ".crlf.gz", open(fq1, "rb").read().replace(b"\n", b"\r\n"))
    g2 = gz(fq2 + ".gz", open(fq2, "rb").read())
    dev, err = run_ok(workdir, small_ref["prefix"], g1, g2, "gzc_d", 101, "soap4.ini", ("-F", "-nc"))
    assert "formatting on the host" in err
    host, _ = run_ok(workdir, small_ref["prefix"], g1, g2, "gzc_h", 101, "soap4.ini", ("-F", "-nc"), {"MP_HOST_IO": "1"})
    assert dev == host, first_diff(dev, host)


def test_gz_truncated_pair(workdir, small_ref):
    """A .gz pair cut inside the deflate data: the same stdout and exit status as reading the files with gzread."""
    fq1, fq2 = make_reads(workdir, small_ref, "gzt", 3000, 100, seed=31, model="divergent", one_random=0.10, unalignable=0.05)
    for frac in (0.5, 0.93):
        d1, d2 = gzip.compress(open(fq1, "rb").read(), 6), gzip.compress(open(fq2, "rb").read(), 6)
        g1, g2 = fq1 + ".t.gz", fq2 + ".t.gz"
        open(g1, "wb").write(d1[:int(len(d1) * frac)])
        open(g2, "wb").write(d2[:int(len(d2) * frac)])
        rc_d, dev, _ = run(workdir, small_ref["prefix"], g1, g2, "gzt_d", 101, "soap4.ini", ("-F", "-nc"))
        rc_h, host, _ = run(workdir, small_ref["prefix"], g1, g2, "gzt_h", 101, "soap4.ini", ("-F", "-nc"), {"MP_HOST_IO": "1"})
        assert rc_d == rc_h and dev == host, (frac, rc_d, rc_h, first_diff(dev, host))
