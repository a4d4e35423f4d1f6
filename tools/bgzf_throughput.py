#!/usr/bin/env python3
"""BGZF compression on the device (mp_bgzf_compress) against zlib, and the -b driver loop with it against MP_HOST_IO=1 (zlib on the
formatting threads), on a B200.

Workload: 20 Mbp GPU-built reference, 1.2 M synthetic pairs of 150 bases with Illumina-like qualities, written `rep` times
(default 2).  `bin/soap4 -C soap4-nt2.ini -b -F -top 95 -T 16` (the cfg3 command shape) runs alternately with MP_HOST_IO=1 and with
the defaults, twice each; the records of the first MP_HOST_IO=1 run, decompressed, are the library workload (about 0.9 GB per rep).
Output: the card's name and power limit, then one line per measurement; `--out FILE` also writes those lines to FILE.
Usage: bgzf_throughput.py [rep] [--out FILE]"""
import concurrent.futures as cf
import ctypes
import gzip
import os
import subprocess
import sys
import time
import zlib

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench
import megapath_b200 as mp

PIECE = 0xff00
lines_out = []


def say(s):
    print(s, flush=True)
    lines_out.append(s)


card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], stdout=subprocess.PIPE, text=True).stdout.strip()
say("card: %s" % card)
d = "/tmp/mp_bgzf_thr"
os.makedirs(d, exist_ok=True)
args = sys.argv[1:]
out_path = None
if "--out" in args:
    k = args.index("--out")
    out_path = args[k + 1]
    del args[k:k + 2]
n, npairs, rep = 20_000_000, 1_200_000, int(args[0]) if args else 2
dev = torch.device("cuda", 0)
codes = bench.gen_ref_codes(n, 5, dev)
bounds = bench.ref_bounds(n, 12, 5)
ctx = mp.Context(0)
prefix = os.path.join(d, "ref.index")
ctx.index_build_codes(codes, bounds, prefix)
ctx.close()
reads = bench.gen_batch(codes, torch.from_numpy(bounds).to(dev), npairs, 150, unalignable=0.02, one_random=0.03).cpu().numpy()
lut = np.frombuffer(b"ACGT", dtype=np.uint8)
rng = np.random.default_rng(1)
for mate in (0, 1):
    rows = lut[reads[mate::2]]
    L = rows.shape[1]
    qual = (33 + np.clip(np.round(37 - np.abs(rng.normal(0, 3, (npairs, L))) - np.linspace(0, 8, L)), 2, 41)).astype(np.uint8)
    names = np.char.add(np.char.add("@p", np.arange(npairs).astype(str)), "/%d" % (mate + 1)).astype("S")
    blob = b"".join(names[i] + b"\n" + rows[i].tobytes() + b"\n+\n" + qual[i].tobytes() + b"\n" for i in range(npairs))
    with open(os.path.join(d, "r_%d.fq" % (mate + 1)), "wb") as f:
        for _ in range(rep):
            f.write(blob)
fq1, fq2 = os.path.join(d, "r_1.fq"), os.path.join(d, "r_2.fq")
os.sync()
exe = os.path.join(ROOT, "megapath_b200", "bin", "soap4")
ini = os.path.join(ROOT, "megapath_b200", "ini", "soap4-nt2.ini")
total = npairs * rep
SUFFIXES = (".dpout.1", ".gout.1", ".unpair")

# ---- driver: cfg3 command shape, MP_HOST_IO=1 and the defaults alternated twice ----
for k, host in enumerate((1, 0, 1, 0)):
    out = os.path.join(d, "h%d" % k if host else "d%d" % k)
    with open("/dev/null", "wb") as fo:
        p = subprocess.run([exe, "pair", prefix, fq1, fq2, "-o", out, "-C", ini, "-L", "151", "-T", "16", "-u", "750", "-b", "-F", "-top", "95"],
                           stdout=fo, stderr=subprocess.PIPE, timeout=1800, env=dict(os.environ, MP_DRIVER_TIMING="1", **({"MP_HOST_IO": "1"} if host else {})))
    assert p.returncode == 0, p.stderr.decode()[-2000:]
    lines = p.stderr.decode().splitlines()
    loop = [float(l.split(":")[1].split()[0]) for l in lines if "Overall alignment time" in l][0]
    fmt = [(float(l.split(" format ")[1].split()[0]), float(l.split("bgzf compress ")[1].split(")")[0])) for l in lines if "[timing] batch" in l and " format " in l]
    sizes = {s: os.path.getsize(out + s) for s in SUFFIXES}
    say("driver %s: loop %.2f s = %.3f M pairs/s; BAM bytes %s (total %.1f MB); per batch format / bgzf compress (s): %s" % (
        "MP_HOST_IO=1" if host else "default (device BGZF)", loop, total / loop / 1e6, sizes, sum(sizes.values()) / 1e6,
        ", ".join("%.2f/%.2f" % f for f in fmt)))

# ---- library: the records of the first MP_HOST_IO=1 run ----
data = b"".join(gzip.open(os.path.join(d, "h0") + s, "rb").read() for s in SUFFIXES)
nbytes = len(data)
L = mp.lib()
ctx = mp.Context(0)
ctx.bgzf_reserve(nbytes)
src, dst = L.mp_host_alloc(nbytes), L.mp_host_alloc(mp.bgzf_bound(nbytes))
ctypes.memmove(src, data, nbytes)
ob = ctypes.c_uint64()
times = []
for it in range(4):                          # the first call is the warm-up (module load, first touch of the buffers)
    t0 = time.perf_counter()
    rc = L.mp_bgzf_compress(ctx.h, ctypes.c_void_p(src), nbytes, ctypes.c_void_p(dst), mp.bgzf_bound(nbytes), ctypes.byref(ob))
    times.append(time.perf_counter() - t0)
    assert rc == 0, L.mp_last_error()
dev_bytes = ob.value
assert gzip.decompress(ctypes.string_at(dst, dev_bytes)) == data
best, med = min(times[1:]), sorted(times[1:])[1]
say("library: %.3f GB of BAM records; mp_bgzf_compress (pinned host buffers, copies included) %.3f s median of 3 = %.2f GB/s (best %.2f GB/s); "
    "%d bytes = ratio %.4f" % (nbytes / 1e9, med, nbytes / med / 1e9, nbytes / best / 1e9, dev_bytes, dev_bytes / nbytes))


def zlib_piece(args):
    at, level = args
    c = zlib.compressobj(level, zlib.DEFLATED, -15, 8)
    return len(c.compress(data[at:at + PIECE]) + c.flush()) + 26


for level in (1, 6):
    with cf.ThreadPoolExecutor(16) as ex:
        t0 = time.perf_counter()
        zb = sum(ex.map(zlib_piece, [(at, level) for at in range(0, nbytes, PIECE)], chunksize=64))
        dt = time.perf_counter() - t0
    say("host zlib level %d, 16 threads, same 0xff00 pieces: %.3f s = %.3f GB/s; %d bytes = ratio %.4f; device / zlib size %.4f; device rate / this rate %.1fx" % (
        level, dt, nbytes / dt / 1e9, zb, zb / nbytes, dev_bytes / zb, (nbytes / med) / (nbytes / dt)))
L.mp_host_free(ctypes.c_void_p(src))
L.mp_host_free(ctypes.c_void_p(dst))
ctx.close()
if out_path:
    with open(out_path, "w") as f:
        f.write("\n".join(lines_out) + "\n")
