"""FASTA front end of the 2bwt-builder drop-in (megapath_b200/bin/2bwt-builder): .pac / .ann / .amb / .tra must be the bytes the
reference's HSPParseFASTAToPacked writes (2bwt-lib/HSP.c:354-699) for texts with ambiguity runs, IUPAC codes, lower case, stray
characters.  CPU only (--annotation-only); the GPU half (BWT, occ, SA, LKT of the same text) is tests/test_gpu_e2e.py."""
import os
import shutil
import subprocess

import numpy as np
import pytest

from conftest import REF_DIR, have_ref, check_reference_digest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EXE = os.path.join(ROOT, "megapath_b200", "bin", "2bwt-builder")
pytestmark = pytest.mark.skipif(not os.path.exists(EXE), reason="builder binary not built")


def fasta_with_ambiguity(seed, nseq=5, seqlen=30000, first_has_long_run=True):
    """Random sequences with short (<10) and long (>=10) runs of N and other IUPAC codes, lower-case stretches, runs at sequence
    starts and ends, runs broken across lines, digits and '*' inside the sequence."""
    rng = np.random.default_rng(seed)
    out = []
    for s in range(nseq):
        seq = bytearray(np.frombuffer(b"ACGT", dtype=np.uint8)[rng.integers(0, 4, size=seqlen)].tobytes())
        n_runs = int(rng.integers(3, 9)) if (s > 0 or first_has_long_run) else 0
        for r in range(n_runs):
            ln = int(rng.choice([1, 2, 5, 9, 10, 11, 40, 300]))
            if s == 0 and r == 0:
                ln = 57                                           # a cut-out run in the first sequence (see fasta_index.h)
            at = int(rng.integers(200, seqlen - 400))
            codes = b"NNNNNNRYKMSWBDHV"
            seq[at:at + ln] = bytes(codes[int(x)] for x in rng.integers(0, len(codes), size=ln))
        if s == 1:
            seq[0:25] = b"N" * 25                                 # run at the very start of a sequence
        if s == 2:
            seq[-31:] = b"n" * 31                                 # lower-case run at the very end
        if s == 3:
            seq[5000:5200] = bytes(seq[5000:5200]).lower()        # lower-case bases are bases (unless -U)
            seq[7000:7003] = b"12*"                               # not nucleotide codes: dropped
        name = b"seq%d some comment" % (s + 1) if s != 4 else b"gi|12345|ref|NC_000001.1| with gi"
        lines = [bytes(seq[i:i + 70]) for i in range(0, len(seq), 70)]
        out.append(b">" + name + b"\n" + b"\n".join(lines) + b"\n")
    return b"".join(out)


@pytest.mark.parametrize("seed,mask", [(1, False), (2, False), (3, True), (4, False)])
def test_annotation_and_pac_match_reference_builder(tmp_path, seed, mask):
    d = tmp_path
    fa = d / "r.fa"
    fa.write_bytes(fasta_with_ambiguity(seed, nseq=5 if seed != 4 else 2, seqlen=30000 if seed != 2 else 300000))
    def no_seed(ann):                        # RandomSeed=0 in 2bwt-builder.ini means "seed from the clock" (2BWT-Builder.c:462-465): the third
        first, rest = ann.split(b"\n", 1)    # number of the .ann header differs from run to run (nothing reads it back)
        return first.split()[:2], rest
    exts = ("ann", "amb", "tra", "pac")
    if have_ref():
        shutil.copy(os.path.join(REF_DIR, "2bwt-builder.ini"), d / "2bwt-builder.ini")
        subprocess.check_call([os.path.join(REF_DIR, "2bwt-builder"), str(fa)] + (["-U"] if mask else []), cwd=d,
                              stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
        want = {ext: open(str(fa) + ".index." + ext, "rb").read() for ext in exts}
        for ext in want:
            os.remove(str(fa) + ".index." + ext)
    subprocess.check_call([EXE, str(fa), "--annotation-only"] + (["-U"] if mask else []), cwd=d, stdout=subprocess.DEVNULL)
    got = {ext: open(str(fa) + ".index." + ext, "rb").read() for ext in exts}
    if have_ref():
        for ext in exts:
            if ext == "ann":
                assert no_seed(got[ext]) == no_seed(want[ext])
            else:
                assert got[ext] == want[ext], ext
    # the reference builder's files for this text, as a digest (tests/conftest.py)
    check_reference_digest("2bwt-builder --annotation-only %d %d" % (seed, mask),
                           repr(no_seed(got["ann"])).encode() + b"".join(got[ext] for ext in exts[1:]))
    assert int(got["tra"].split()[2]) >= 3                        # cut-out runs exist


def test_undefined_reference_input_is_refused(tmp_path):
    """a cut-out run in the third sequence with none before it: the reference indexes ambiguity[-1] (HSP.c:583-585)"""
    seqs = [b"ACGT" * 500, b"CAGT" * 500, b"ACGT" * 100 + b"N" * 50 + b"TTGA" * 100]
    fa = tmp_path / "u.fa"
    fa.write_bytes(b"".join(b">s%d\n%s\n" % (i, s) for i, s in enumerate(seqs)))
    p = subprocess.run([EXE, str(fa), "--annotation-only"], capture_output=True)
    assert p.returncode != 0 and b"out of bounds" in p.stderr
