#!/usr/bin/env python3
"""NT chunk chain on a B200: three synthetic chunk indexes of about 1 Gbp each and 4 Mi pairs of 150 bases, timed as
  1. the K-process composition through files on local disk: soap4 idx0 -nc > f0; deinterleave f0; soap4 idx1 > f1; ...; and
  2. one `soap4 ... -chain idx1 out1 -chain idx2 out2` run,
each with the last stdout to a file and discarded.  The two file outputs must have the same md5.  Prints one line per timing and a
JSON summary with the card name and power limit; `--out <file>` also writes the summary to that file."""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench
import megapath_b200 as mp

ap = argparse.ArgumentParser()
ap.add_argument("--out", help="write the JSON summary to this file as well")
ap.add_argument("--rounds", type=int, default=2, help="alternating rounds of the four timings")
args = ap.parse_args()
d = os.environ.get("MP_CHAIN_DIR", "/tmp/mp_chain")
os.makedirs(d, exist_ok=True)
n, npairs, K = int(os.environ.get("MP_CHAIN_GBP", "1")) * 1_000_000_000, 4 << 20, 3
dev = torch.device("cuda", 0)
exe = os.path.join(ROOT, "megapath_b200", "bin", "soap4")
deint = os.path.join(ROOT, "megapath_b200", "bin", "soap4_hosttest")
ini = os.path.join(ROOT, "megapath_b200", "ini", "soap4-nt2.ini")

prefixes, codes0 = [], None
for k in range(K):
    prefix = os.path.join(d, "chunk%d.index" % k)
    codes = bench.gen_ref_codes(n, 11 + k, dev)
    if k:                                  # later chunks share a diverged tenth of chunk 0, so that reads score on several chunks
        m = n // 10
        part = codes0[:m].clone()
        flip = torch.rand(m, device=dev) < 0.02
        part[flip] = torch.randint(0, 4, (int(flip.sum()),), device=dev, dtype=torch.uint8)
        codes[:m] = part
    if k == 0:
        codes0 = codes
    if not os.path.exists(prefix + ".sa"):
        c = mp.Context(0)
        c.index_build_codes(codes, bench.ref_bounds(n, 40, 11 + k), prefix)
        c.close()
    prefixes.append(prefix)
    if k:
        del codes
torch.cuda.empty_cache()
fq = [os.path.join(d, "r_%d.fq" % m) for m in (1, 2)]
if not os.path.exists(fq[1]):
    reads = bench.gen_batch(codes0, torch.from_numpy(bench.ref_bounds(n, 40, 11)).to(dev), npairs, 150, unalignable=0.02, one_random=0.05).cpu().numpy()
    lut = np.frombuffer(b"ACGT", dtype=np.uint8)
    for mate in (0, 1):
        rows = lut[reads[mate::2]]
        with open(fq[mate], "wb") as f:
            f.write(b"".join(b"@p%d/%d\n" % (i, mate + 1) + rows[i].tobytes() + b"\n+\n" + b"I" * rows.shape[1] + b"\n" for i in range(npairs)))
    del reads
del codes0
torch.cuda.empty_cache()
os.sync()


def soap4(index, a, b, out, flags, sink):
    t0 = time.time()
    with open(sink, "wb") as fo:
        p = subprocess.run([exe, "pair", index, a, b, "-o", out, "-C", ini, "-L", "151", "-T", "16", "-u", "750", "-F", "-top", "95"] + flags,
                           stdout=fo, stderr=subprocess.PIPE, timeout=3600)
    assert p.returncode == 0, p.stderr.decode()[-3000:]
    return time.time() - t0


def md5(path):
    h = hashlib.md5()
    with open(path, "rb") as f:
        for blk in iter(lambda: f.read(1 << 24), b""):
            h.update(blk)
    return h.hexdigest()


def composition(sink):
    t, a, b = 0.0, fq[0], fq[1]
    for k, idx in enumerate(prefixes):
        last = k + 1 == K
        out = os.path.join(d, "comp%d" % k)
        t += soap4(idx, a, b, out, ["-nc"] if k == 0 else [], sink if last else out + ".fq")
        if not last:
            t0 = time.time()
            subprocess.run([deint, "__deinterleave", out + ".fq"], check=True, timeout=3600)
            t += time.time() - t0
            a, b = out + ".fq_1.fq", out + ".fq_2.fq"
    return t


chain = sum((["-chain", prefixes[k], os.path.join(d, "chain%d" % k)] for k in range(1, K)), [])
res = {}
for rnd in range(args.rounds):             # the four timings alternate
    res.setdefault("composition_file_s", []).append(composition(os.path.join(d, "comp.out")))
    res.setdefault("chain_file_s", []).append(soap4(prefixes[0], fq[0], fq[1], os.path.join(d, "chain0"), ["-nc"] + chain, os.path.join(d, "chain.out")))
    res.setdefault("composition_null_s", []).append(composition("/dev/null"))
    res.setdefault("chain_null_s", []).append(soap4(prefixes[0], fq[0], fq[1], os.path.join(d, "chain0"), ["-nc"] + chain, "/dev/null"))
    print(rnd, {k: round(v[-1], 2) for k, v in res.items()}, flush=True)
same = md5(os.path.join(d, "comp.out")) == md5(os.path.join(d, "chain.out"))
smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True).stdout.strip()
summary = dict(gpu=smi, text_bp_per_chunk=n, chunks=K, pairs=npairs, read_length=150, md5_equal=same,
               output_bytes=os.path.getsize(os.path.join(d, "chain.out")), **{k: [round(x, 2) for x in v] for k, v in res.items()})
print(json.dumps(summary))
if args.out:
    json.dump(summary, open(args.out, "w"), indent=1)
assert same, "the chain and the composition printed different bytes"
