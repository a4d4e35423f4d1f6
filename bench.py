#!/usr/bin/env python3
"""bench.py -- read pairs aligned/sec of the soap4 alignment hot path on B200 (BASELINE.json metric).

One "step" = one pass of the whole hot path (MMP seeding -> SA resolution -> pairing -> deep DP with
traceback -> single-end DP -> mate rescue -> per-pair reduction) over one batch of synthetic read pairs,
through the C-ABI of libmegapath_b200.so (include/megapath_b200.h).

  value  : pairs/s with the batch already resident in HBM (mp_batch_upload outside the timed region),
           timed with CUDA events on the library's launching stream (mp_results.ms_total), max over ranks
  e2e    : pairs/s through the same C-ABI with HOST buffers: pinned-host -> HBM upload of the packed reads
           and the host-resident result arrays inside the timed region (wall clock between device syncs)
  roofline : the seeding kernel (k_mmp): algorithmic bytes = 64 B per occ evaluation + 16 B per LKT jump
           (SURVEY.md 8d) / its CUDA-event duration, against MEASURED_PEAKS.json hbm_gbs
  cpu_baseline : the reference's own soap4 (oracle/_ref/soap4, compiled from /root/reference by
           oracle/Makefile.ref) on a bounded sample of the same workload, all host cores

`--impl reference` times only that CPU arm.  Multi-GPU: one process per GPU (torchrun), index replicated,
disjoint read batches per rank, no collective on the data path ("weak" scaling).
"""
import argparse
import json
import os
import re
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

INSERT_LO, INSERT_HI = 250, 500
INSERT_HIGH_OPT = 750           # soap4 -u 750
DUMP_ROWS = 8192                # --dump-outputs: rows per result array (keeps a dump under 64 MB)

# BASELINE.json configs (SURVEY.md 8d).  `-L` is read length + 1: the reference truncates reads to L - 1 (QueryParser.cpp:188).
CONFIGS = {
    # cfg1: the reference's own CPU-runnable case
    "cfg1": dict(ref_mbp=50.0, nseq=12, read_len=150, model="subs", unalignable=0.0, one_random=0.0, ini="soap4.ini",
                 about="150bp pairs (substitutions per read from {0,0,0,1,1,2}) vs a 50 Mbp synthetic reference (12 seqs), soap4.ini -L 151 -u 750"),
    # cfg2: human-filtering stage; the configuration the metric is quoted on
    "cfg2": dict(ref_mbp=3100.0, nseq=24, read_len=150, model="subs", unalignable=0.01, one_random=0.01, ini="soap4.ini",
                 about="150bp pairs vs a 3.1 Gbp human-sized synthetic reference (24 seqs), soap4.ini -L 151 -u 750; 1% unalignable pairs, 1% one-mate-random"),
    # cfg3: NT classification stage at the largest size the box's disk and the reference arm's run time allow by default (the text is
    # beyond 2^32 bases: 64-bit positions, bucketed index builder, sampled SA); --ref-mbp raises it (DESIGN.md has the 60 Gbp HBM budget)
    "cfg3": dict(ref_mbp=8000.0, nseq=400, read_len=150, model="subs", unalignable=0.02, one_random=0.02, ini="soap4-nt2.ini", dups=200,
                 about="150bp pairs vs an 8 Gbp synthetic multi-genome reference (400 seqs, 200 planted 3 Mbp near-duplicates at 1% divergence), "
                       "soap4-nt2.ini -L 151 -u 750 -top 95; 2% unalignable pairs, 2% one-mate-random"),
    # cfg4: DP-heavy: most reads carry an indel, 5 % of the pairs have one random mate (single-end DP + mate rescue with 752-wide tables)
    "cfg4": dict(ref_mbp=3100.0, nseq=24, read_len=150, model="divergent", unalignable=0.0, one_random=0.05, ini="soap4.ini",
                 about="DP-heavy 150bp pairs (4% substitutions, 0.5% 1-3bp deletions, 0.5% 1-3bp insertions per base; 5% of the pairs with one random mate) "
                       "vs the 3.1 Gbp synthetic reference, soap4.ini -L 151 -u 750"),
    # cfg5: MegaPath-Amplicon-style read length
    "cfg5": dict(ref_mbp=100.0, nseq=50, read_len=250, model="subs", unalignable=0.01, one_random=0.01, ini="soap4.ini",
                 about="250bp pairs vs a 100 Mbp synthetic bacterial panel (50 seqs), soap4.ini -L 251 -u 750; 1% unalignable pairs, 1% one-mate-random"),
}


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=6)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default=os.environ.get("MP_BENCH_CONFIG", "cfg2"), choices=sorted(CONFIGS))
    ap.add_argument("--ref-mbp", type=float, default=float(os.environ.get("MP_BENCH_REF_MBP", "0")), help="override the config's reference size")
    ap.add_argument("--read-len", type=int, default=0, help="override the config's read length (-L sweep)")
    ap.add_argument("--pairs-per-step", type=int, default=int(os.environ.get("MP_BENCH_PAIRS", str(1 << 20))))
    ap.add_argument("--cpu-sample-pairs", type=int, default=int(os.environ.get("MP_BENCH_CPU_PAIRS", "200000")))
    ap.add_argument("--cli-pairs", type=int, default=int(os.environ.get("MP_BENCH_CLI_PAIRS", str(4 << 20))),
                    help="pairs in the FASTQ files of the e2e_cli leg (bin/soap4, FASTQ in -> annotated FASTQ out); 0 = skip")
    ap.add_argument("--no-cpu-baseline", action="store_true", help="skip the CPU legs (reference sample, parity at scale, e2e_cli)")
    ap.add_argument("--contexts", type=int, default=int(os.environ.get("MP_BENCH_CONTEXTS", "3")),
                    help="contexts (host thread + stream each) per GPU sharing one resident index; batches alternate between them")
    ap.add_argument("--workdir", default=os.environ.get("MP_BENCH_DIR", "/tmp/mpbench"))
    ap.add_argument("--prepare", action="store_true",
                    help="build what the CPU legs need and exit: the workload's index files (GPU builder, reference file formats) and the "
                         "FASTQ samples.  `--impl reference` runs this in a child process, so that the process which times the reference "
                         "never loads this repo's library")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the result arrays of the last timed step as DIR/<array>.<field>.npy (float64; "
                         "CIGARs as float32 byte rows), at most %d rows per array in a fixed, seeded sample" % DUMP_ROWS)
    ap.add_argument("--profile-step", action="store_true",
                    help="profiling aid (ncu --profile-from-start off): after the warm-up run ONE step on one context between "
                         "cudaProfilerStart/Stop and exit; prints no bench value")
    a = ap.parse_args()
    if a.dump_outputs and a.steps < 1:
        ap.error("--dump-outputs writes the results of the last timed step: it needs --steps 1 or more")
    a.cfg = dict(CONFIGS[a.config])
    if a.ref_mbp > 0:
        a.cfg["ref_mbp"] = a.ref_mbp
    if a.read_len > 0:
        a.cfg["read_len"] = a.read_len
    a.read_len, a.lopt = a.cfg["read_len"], a.cfg["read_len"] + 1
    return a


# ------------------------------------------------------------------------------------------------
# synthetic workload (SURVEY.md 8d cfg2 model: uniform i.i.d. ACGT reference in 24 sequences;
# FR pairs, insert U[250,500), substitutions per read from {0,0,0,1,1,2}, 1% unalignable pairs,
# 1% pairs with one random mate)
# ------------------------------------------------------------------------------------------------
def ref_bounds(n, nseq, seed):
    rng = np.random.default_rng(seed)
    cuts = np.sort(rng.choice(np.arange(1000, n - 1000), size=nseq - 1, replace=False))
    return np.concatenate([[0], cuts, [n]]).astype(np.int64)


def gen_ref_codes(n, seed, device):
    import torch
    g = torch.Generator(device=device)
    g.manual_seed(seed)
    out = torch.empty(n, dtype=torch.uint8, device=device)
    CH = 1 << 28
    for o in range(0, n, CH):
        m = min(CH, n - o)
        out[o:o + m] = torch.randint(0, 4, (m,), dtype=torch.uint8, device=device, generator=g)
    return out


def make_reference(args, device):
    """-> (codes on the device, sequence bounds): uniform i.i.d. ACGT; configs with "dups" get that many near-duplicate 3 Mbp blocks
    (1 % substitutions) copied between sequences, so that multi-hit / -top lists are not trivial (SURVEY.md 8d cfg3)."""
    import torch
    n = int(args.cfg["ref_mbp"] * 1e6)
    bounds = ref_bounds(n, args.cfg["nseq"], 42)
    codes = gen_ref_codes(n, 42, device)
    nd = int(args.cfg.get("dups", 0))
    if nd:
        g = torch.Generator(device=device)
        g.manual_seed(77)
        nseq, ln = args.cfg["nseq"], 3_000_000
        for k in range(nd):
            a, b = k % nseq, (k * 7 + 3) % nseq
            if bounds[a + 1] - bounds[a] < 2 * ln + 2000 or bounds[b + 1] - bounds[b] < 2 * ln + 2000:
                continue
            src, dst = int(bounds[a]) + 1000, int(bounds[b + 1]) - ln - 1000
            blk = codes[src:src + ln].clone()
            mut = torch.rand(ln, device=device, generator=g) < 0.01
            blk[mut] = (blk[mut] + torch.randint(1, 4, (int(mut.sum()),), device=device, generator=g, dtype=torch.uint8)) & 3
            codes[dst:dst + ln] = blk
    return codes, bounds


def gen_batch(ref_codes, bounds_t, npairs, seed, read_len=150, model="subs", unalignable=0.01, one_random=0.01):
    """-> (codes (2*npairs, read_len) uint8 on device, mate1 = even rows).
    model "subs": per-read substitutions drawn from {0,0,0,1,1,2}; "divergent": per base 4 % substitutions, 0.5 % deletions
    and 0.5 % insertions of 1-3 bases (SURVEY.md 8d cfg4)."""
    import torch
    dev = ref_codes.device
    g = torch.Generator(device=dev)
    g.manual_seed(seed)
    L = read_len
    W = L + 24 if model == "divergent" else L            # source window: room for deleted bases
    nseq = bounds_t.numel() - 1
    lo_i, hi_i = max(INSERT_LO, W + 10), max(INSERT_HI, W + 60)
    isz = torch.randint(lo_i, hi_i, (npairs,), device=dev, generator=g)
    sid = torch.randint(0, nseq, (npairs,), device=dev, generator=g)
    lo = bounds_t[sid]
    hi = torch.maximum(bounds_t[sid + 1] - isz, lo + 1)
    start = lo + (torch.rand(npairs, device=dev, generator=g, dtype=torch.float64) * (hi - lo).double()).long()
    start = torch.clamp(start, 0, ref_codes.numel() - hi_i - 1)
    ar = torch.arange(W, device=dev)
    src = torch.empty((2 * npairs, W), dtype=torch.uint8, device=dev)
    CH = 1 << 18
    for o in range(0, npairs, CH):
        s_ = start[o:o + CH]
        z = isz[o:o + CH]
        src[2 * o:2 * (o + len(s_)):2] = ref_codes[s_[:, None] + ar[None, :]]
        src[2 * o + 1:2 * (o + len(s_)):2] = 3 - ref_codes[(s_ + z)[:, None] - 1 - ar[None, :]]
    nreads = 2 * npairs
    if model == "divergent":
        out = torch.empty((nreads, L), dtype=torch.uint8, device=dev)
        for o in range(0, nreads, CH):
            blk = src[o:o + CH]
            n = blk.shape[0]
            u = torch.rand((n, W), device=dev, generator=g)
            sub = u < 0.04
            dele = (u >= 0.04) & (u < 0.045)
            ins = (u >= 0.045) & (u < 0.05)
            k = torch.randint(1, 4, (n, W), device=dev, generator=g)
            # a deletion event removes k source bases: mark the following k-1 as deleted too
            dmask = dele.clone()
            dmask[:, 1:] |= dele[:, :-1] & (k[:, :-1] >= 2)
            dmask[:, 2:] |= dele[:, :-2] & (k[:, :-2] >= 3)
            emit = (~dmask).long() + torch.where(ins & ~dmask, k, torch.zeros_like(k))      # bases written for this source base
            end = torch.cumsum(emit, dim=1)                                                     # kept base lands at end - 1
            delta = torch.randint(1, 4, (n, W), device=dev, generator=g).to(torch.uint8)
            base = torch.where(sub, (blk + delta) & 3, blk)
            o_blk = torch.randint(0, 4, (n, L), dtype=torch.uint8, device=dev, generator=g)    # inserted bases are random
            pos = end - 1
            ok = (~dmask) & (pos < L)
            rows = torch.arange(n, device=dev)[:, None].expand(n, W)
            o_blk[rows[ok], pos[ok]] = base[ok]
            out[o:o + n] = o_blk
        del src
    else:
        out = src
        nsub = torch.tensor([0, 0, 0, 1, 1, 2], device=dev)[torch.randint(0, 6, (nreads,), device=dev, generator=g)]
        rows = torch.arange(nreads, device=dev)
        for k in (1, 2):
            sel = rows[nsub >= k]
            cols = torch.randint(0, L, (sel.numel(),), device=dev, generator=g)
            delta = torch.randint(1, 4, (sel.numel(),), device=dev, generator=g).to(torch.uint8)
            out[sel, cols] = (out[sel, cols] + delta) & 3
    u = torch.rand(npairs, device=dev, generator=g)
    ua = torch.nonzero(u < unalignable).flatten()
    if ua.numel():
        out[2 * ua] = torch.randint(0, 4, (ua.numel(), L), dtype=torch.uint8, device=dev, generator=g)
        out[2 * ua + 1] = torch.randint(0, 4, (ua.numel(), L), dtype=torch.uint8, device=dev, generator=g)
    one = torch.nonzero((u >= unalignable) & (u < unalignable + one_random)).flatten()
    if one.numel():
        out[2 * one + 1] = torch.randint(0, 4, (one.numel(), L), dtype=torch.uint8, device=dev, generator=g)
    return out


def pack_queries_torch(codes, max_len_opt):
    """appendToQueryArrays layout (QueryParser.cpp:184-203) built with torch on the device:
    2-bit, 16 bases per word LSB-first, 32-read interleaved.  -> pinned host int32 tensor, wpq."""
    import torch
    n, L = codes.shape
    wpq = (max_len_opt + 15) // 16
    npad = (n + 31) // 32 * 32
    c = torch.zeros((npad, wpq * 16), dtype=torch.int64, device=codes.device)
    c[:n, :L] = codes
    sh = (2 * (torch.arange(wpq * 16, device=codes.device) % 16))
    w = (c << sh[None, :]).view(npad, wpq, 16).sum(dim=2)
    w = w.view(npad // 32, 32, wpq).permute(0, 2, 1).contiguous().view(-1)
    w32 = (w & 0xFFFFFFFF).to(torch.int64)
    w32 = torch.where(w32 >= (1 << 31), w32 - (1 << 32), w32).to(torch.int32)
    host = torch.empty(w32.shape, dtype=torch.int32, pin_memory=True)
    host.copy_(w32)
    return host, wpq


def write_fastq_sample(path_prefix, codes_np):
    """Interleaved rows (mate 1 = even) -> <prefix>_1.fq / _2.fq; fixed-width names so that the files are built with numpy."""
    lut = np.frombuffer(b"ACGT", dtype=np.uint8)
    n, L = codes_np.shape[0] // 2, codes_np.shape[1]
    ids = np.arange(n)
    digits = ((ids[:, None] // (10 ** np.arange(8, -1, -1))[None, :]) % 10 + 48).astype(np.uint8)       # 9 digits
    for mate in (0, 1):
        rec = np.empty((n, 2 + 9 + 3 + L + 3 + L + 1), dtype=np.uint8)
        rec[:, 0], rec[:, 1] = ord("@"), ord("p")
        rec[:, 2:11] = digits
        rec[:, 11], rec[:, 12], rec[:, 13] = ord("/"), ord("1") + mate, 10
        rec[:, 14:14 + L] = lut[codes_np[mate::2]]
        rec[:, 14 + L], rec[:, 15 + L], rec[:, 16 + L] = 10, ord("+"), 10
        rec[:, 17 + L:17 + 2 * L] = ord("I")
        rec[:, 17 + 2 * L] = 10
        with open("%s_%d.fq.tmp" % (path_prefix, mate + 1), "wb") as f:
            f.write(rec.tobytes())
        os.replace("%s_%d.fq.tmp" % (path_prefix, mate + 1), "%s_%d.fq" % (path_prefix, mate + 1))


def summary_keeping_results(c, P):
    """Context.align_pairs_summary for the step whose results --dump-outputs writes: the same mp_align_pairs call and counters, but
    the result set stays in the library's host arena (valid until c's next mp_align_pairs) -> (summary, mp_results)"""
    import ctypes as C
    import megapath_b200 as mp
    res = mp.Results()
    c._check(c.L.mp_align_pairs(c.h, C.byref(P), C.byref(res)))
    out = {name: getattr(res, name) for name, _ in mp.Results._fields_[8:]}
    out.update(c.last_stats())
    out["n_pairs"], out["n_singles"], out["n_rescued"] = res.n_pairs, res.n_singles, res.n_rescued
    out["result_bytes"] = (res.n_pairs + res.n_rescued) * mp.PAIR_RESULT.itemsize + res.n_singles * mp.SINGLE_RESULT.itemsize + res.cigar_bytes
    out["pairs_aligned"] = res.numDPAlignedPair + res.numRescuedPair
    return out, res


def copy_results(c, res):
    """numpy copies of the arrays of a result set summary_keeping_results left with context c; releases it"""
    import ctypes as C
    import megapath_b200 as mp

    def arr(p, n, dt):
        return np.frombuffer((C.c_char * (n * dt.itemsize)).from_address(p), dtype=dt).copy() if n else np.zeros(0, dtype=dt)
    out = dict(pairs=arr(res.pairs, res.n_pairs, mp.PAIR_RESULT), rescued=arr(res.rescued, res.n_rescued, mp.PAIR_RESULT),
               singles=arr(res.singles, res.n_singles, mp.SINGLE_RESULT),
               cigars=bytes((C.c_char * res.cigar_bytes).from_address(res.cigars)) if res.cigar_bytes else b"")
    c.L.mp_results_release(c.h, C.byref(res))
    return out


def dump_outputs(path, res):
    """The result set of mp_align_pairs (what a caller of the timed path receives) -> path/<array>.<field>.npy: the same seeded
    sample of rows for every field; CIGAR offsets replaced by the CIGAR text (one zero-padded byte row per result), so that two
    builds compare equal when they print the same alignments.  An array the step left empty (no rescued pairs, say) is not
    written; counts.npy holds the number of results of each array."""
    import megapath_b200 as mp
    os.makedirs(path, exist_ok=True)
    for seed, name in enumerate(("pairs", "rescued", "singles")):
        a = res[name]
        if not len(a):
            continue
        rng = np.random.default_rng(seed)
        rows = np.sort(rng.choice(len(a), size=DUMP_ROWS, replace=False)) if len(a) > DUMP_ROWS else np.arange(len(a))
        np.save(os.path.join(path, name + ".row.npy"), rows.astype(np.float64))
        for f in a.dtype.names:
            col = a[f][rows]
            if f.startswith("cigar"):
                text = [mp.cigar_at(res["cigars"], int(o)) for o in col]
                out = np.zeros((len(text), max([len(t) for t in text] + [1])), dtype=np.float32)
                for i, t in enumerate(text):
                    out[i, :len(t)] = np.frombuffer(t, dtype=np.uint8)
                np.save(os.path.join(path, "%s.%s.npy" % (name, f)), out)
            else:
                np.save(os.path.join(path, "%s.%s.npy" % (name, f)), col.astype(np.float64))
    np.save(os.path.join(path, "counts.npy"), np.array([len(res["pairs"]), len(res["rescued"]), len(res["singles"])], dtype=np.float64))


# ------------------------------------------------------------------------------------------------
# clocks sampling (B200_PROFILING.md)
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        if os.environ.get("MP_BENCH_NO_SAMPLER"):
            return
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                          "-lms", os.environ.get("MP_BENCH_SAMPLE_MS", "200")], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _pump(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for nm, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------
# workload cache: index files (reference format, so the reference binary runs on the same index) + FASTQ samples
# ------------------------------------------------------------------------------------------------
def workload_dir(args):
    n = int(args.cfg["ref_mbp"] * 1e6)
    return os.path.join(args.workdir, "ref%d_%d_%d" % (n, args.cfg["nseq"], int(args.cfg.get("dups", 0)))), n


def sample_prefix(args, tag, npairs):
    d, _ = workload_dir(args)
    return os.path.join(d, "sample_%s_%s_L%d_%d" % (tag, args.cfg["model"], args.read_len, npairs))


def ensure_index(args, ctx, device, rank, world):
    """Builds the synthetic reference + FM-index once per box (rank 0), in HBM, with the library's own GPU
    builder (mp_index_build), and saves it in the reference's on-disk format; other ranks load the files."""
    import torch
    d, n = workload_dir(args)
    prefix = os.path.join(d, "ref.index")
    ready = os.path.join(d, "READY")
    ref_codes, bounds = make_reference(args, device)
    t0 = time.time()
    if rank == 0 and not os.path.exists(ready):
        os.makedirs(d, exist_ok=True)
        ctx.index_build_codes(ref_codes, bounds, prefix)
        open(ready, "w").write("ok\n")
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
    if not ctx.has_index():
        ctx.index_load(prefix)
    return prefix, ref_codes, torch.from_numpy(bounds).to(device), time.time() - t0


def ensure_samples(args, ref_codes, bounds_t, which):
    """FASTQ files of the CPU legs, written once: "cpu" = the bounded sample the reference is timed on (and parity at scale is
    checked on), "cli" = the larger file pair of the e2e_cli leg."""
    for tag, npairs, seed in (("cpu", args.cpu_sample_pairs, 7_000_003), ("cli", args.cli_pairs, 9_000_011)):
        if tag not in which or npairs <= 0:
            continue
        fqp = sample_prefix(args, tag, npairs)
        if os.path.exists(fqp + "_2.fq"):
            continue
        CH = 1 << 19
        parts = [gen_batch(ref_codes, bounds_t, min(CH, npairs - o), seed + o, args.read_len, args.cfg["model"],
                           args.cfg["unalignable"], args.cfg["one_random"]).cpu().numpy() for o in range(0, npairs, CH)]
        write_fastq_sample(fqp, np.concatenate(parts) if len(parts) > 1 else parts[0])


def prepare(args):
    """`bench.py --prepare`: everything the CPU legs need, built by THIS process (which loads the library); the reference arm runs
    it as a child and then only executes oracle/_ref/soap4."""
    import torch
    import megapath_b200 as mp
    if not torch.cuda.is_available():
        raise SystemExit("bench.py --prepare needs a CUDA device (GPU index builder)")
    device = torch.device("cuda", 0)
    ctx = mp.Context(0)
    d, n = workload_dir(args)
    prefix = os.path.join(d, "ref.index")
    ref_codes, bounds = make_reference(args, device)
    if not os.path.exists(os.path.join(d, "READY")):
        os.makedirs(d, exist_ok=True)
        ctx.index_build_codes(ref_codes, bounds, prefix)
        open(os.path.join(d, "READY"), "w").write("ok\n")
    ctx.close()
    ensure_samples(args, ref_codes, torch.from_numpy(bounds).to(device), ("cpu",))
    return 0


def soap4_cmd(exe, ini_path, prefix, fq_prefix, out_prefix, lopt, threads):
    return [exe, "pair", prefix, fq_prefix + "_1.fq", fq_prefix + "_2.fq", "-o", out_prefix, "-C", ini_path,
            "-L", str(lopt), "-T", str(threads), "-u", str(INSERT_HIGH_OPT), "-F", "-nc"]


def parse_align_time(err):
    m = re.search(r"Overall alignment time \(excl\. read loading\)\s*:\s*([0-9.]+)", err)
    if not m:
        raise RuntimeError("could not parse the 'Overall alignment time' line")
    return float(m.group(1))


def run_reference_soap4(args, prefix, fq_prefix, out_prefix, threads, keep_stdout=False):
    """-> (align_seconds, wall_seconds, stdout path or None); align = the reference's own
    'Overall alignment time (excl. read loading)' (SOAP4.cpp:613)."""
    ref_dir = os.path.join(ROOT, "oracle", "_ref")
    exe = os.path.join(ref_dir, "soap4")
    if not os.path.exists(exe):
        raise RuntimeError("oracle/_ref/soap4 is not built (oracle/Makefile.ref)")
    cmd = soap4_cmd(exe, os.path.join(ref_dir, args.cfg["ini"]), prefix, fq_prefix, out_prefix, args.lopt, threads)
    t0 = time.time()
    with open(out_prefix + ".stdout.fq", "wb") as fo:
        p = subprocess.run(cmd, stdout=fo, stderr=subprocess.PIPE, cwd=os.path.dirname(out_prefix))
    wall = time.time() - t0
    err = p.stderr.decode(errors="replace")
    if p.returncode != 0:
        raise RuntimeError("reference soap4 failed (%d): %s" % (p.returncode, err[-400:]))
    if not keep_stdout:
        try:
            os.remove(out_prefix + ".stdout.fq")
        except OSError:
            pass
    return parse_align_time(err), wall, (out_prefix + ".stdout.fq" if keep_stdout else None)


def run_our_soap4(args, prefix, fq_prefix, out_prefix, threads, sink=None):
    """The product's drop-in binary (megapath_b200/bin/soap4): FASTQ files in, annotated FASTQ on stdout.
    -> (loop_seconds = its 'Overall alignment time' line, wall_seconds, stderr)"""
    exe = os.path.join(ROOT, "megapath_b200", "bin", "soap4")
    cmd = soap4_cmd(exe, os.path.join(ROOT, "megapath_b200", "ini", args.cfg["ini"]), prefix, fq_prefix, out_prefix, args.lopt, threads)
    t0 = time.time()
    with open(sink or (out_prefix + ".stdout.fq"), "wb") as fo:
        p = subprocess.run(cmd, stdout=fo, stderr=subprocess.PIPE,
                           env=dict(os.environ, MP_DRIVER_TIMING="1", **({"MP_TRACE": "2"} if os.environ.get("MP_BENCH_CLI_TRACE") else {})))
    wall = time.time() - t0
    err = p.stderr.decode(errors="replace")
    if p.returncode != 0:
        raise RuntimeError("bin/soap4 failed (%d): %s" % (p.returncode, err[-400:]))
    return parse_align_time(err), wall, err


def canonical_pairs(path):
    """annotated interleaved FASTQ -> sorted list of (mate-1 record, mate-2 record): the reference's worker threads print whole pairs
    in arbitrary order (SURVEY.md 0.8)"""
    with open(path, "rb") as f:
        lines = f.read().split(b"\n")
    recs = [b"\n".join(lines[i:i + 4]) for i in range(0, len(lines) - 3, 4)]
    pairs = [(recs[i], recs[i + 1]) for i in range(0, len(recs) - 1, 2)]
    pairs.sort()
    return pairs


def measured_peak():
    try:
        return float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"]), "measured"
    except Exception:
        return 6650.0, "fallback"


def ncu_traffic(kernel):
    """dram__bytes_read.sum + dram__bytes_write.sum of one launch of `kernel`, from the newest committed ncu --set full summary."""
    best = None
    for name in sorted(os.listdir(os.path.join(ROOT, "profiles"))) if os.path.isdir(os.path.join(ROOT, "profiles")) else []:
        if not (name.startswith("r") and "ncu_full" in name and name.endswith(".txt")):
            continue
        cur, rd, wr = None, None, None
        for ln in open(os.path.join(ROOT, "profiles", name)):
            if ln.startswith("== "):
                cur, rd, wr = ln, None, None
            elif cur and kernel in cur:
                f = ln.split()
                if ln.startswith("dram__bytes_read.sum") and len(f) >= 3:
                    rd = float(f[1]) * {"Gbyte": 1e9, "Mbyte": 1e6, "Kbyte": 1e3, "byte": 1.0}.get(f[2], 1.0)
                if ln.startswith("dram__bytes_write.sum") and len(f) >= 3:
                    wr = float(f[1]) * {"Gbyte": 1e9, "Mbyte": 1e6, "Kbyte": 1e3, "byte": 1.0}.get(f[2], 1.0)
                if rd is not None and wr is not None:
                    best = {"bytes_per_launch": rd + wr, "source": "profiles/" + name}
                    cur = None
    return best


def ncu_metric(kernel, metric):
    """one metric of `kernel` from the newest committed ncu --set full summary (profiles/rNN_ncu_full_*.txt) -> (value, source) or None"""
    best = None
    pdir = os.path.join(ROOT, "profiles")
    for name in sorted(os.listdir(pdir)) if os.path.isdir(pdir) else []:
        if not (name.startswith("r") and "ncu_full" in name and name.endswith(".txt")):
            continue
        cur = None
        for ln in open(os.path.join(pdir, name)):
            if ln.startswith("== "):
                cur = ln
            elif cur and kernel in cur and ln.startswith(metric):
                f = ln.split()
                try:
                    best = (float(f[1]), "profiles/" + name)
                except (IndexError, ValueError):
                    pass
    return best


def main():
    args = parse_args()
    # stdout carries exactly one JSON line: anything libraries print while we work (e.g. NCCL's version banner) goes to stderr
    sys.stdout.flush()
    saved_stdout = os.dup(1)
    os.dup2(2, 1)
    try:
        if args.prepare:
            return prepare(args)
        if args.impl == "reference":
            return run_reference_arm(args, saved_stdout)
        return run(args, saved_stdout)
    finally:
        sys.stdout.flush()
        os.dup2(saved_stdout, 1)


def emit(saved_stdout, obj):
    sys.stdout.flush()
    os.write(saved_stdout, (json.dumps(obj) + "\n").encode())


def base_config(args, pairs_per_step):
    return {"workload": "%s: %s; %d pairs per step" % (args.config, args.cfg["about"], pairs_per_step),
            "name": args.config, "pairs_per_step_per_gpu": pairs_per_step, "ref_mbp": args.cfg["ref_mbp"], "read_len": args.read_len,
            "l2": "", "parallelism": "replicated index, disjoint read batches per GPU, no data-path collective"}


def run_reference_arm(args, saved_stdout):
    """The reference's own CPU implementation (oracle/_ref/soap4 = /root/reference/soap4 compiled by oracle/Makefile.ref, AVX2 build),
    all host threads, on a bounded sample of the workload.  This process executes nothing of this repo's library: the index files and
    the FASTQ sample are produced by a child process (`bench.py --prepare`, untimed) when the box does not have them yet."""
    if int(os.environ.get("RANK", "0")) != 0:
        return 0
    ncores = os.cpu_count() or 1
    d, _ = workload_dir(args)
    prefix = os.path.join(d, "ref.index")
    npairs = args.cpu_sample_pairs
    fqp = sample_prefix(args, "cpu", npairs)
    if not (os.path.exists(os.path.join(d, "READY")) and os.path.exists(fqp + "_2.fq")):
        env = dict(os.environ)
        for k in ("RANK", "LOCAL_RANK", "WORLD_SIZE", "MASTER_ADDR", "MASTER_PORT"):
            env.pop(k, None)
        subprocess.check_call([sys.executable, os.path.abspath(__file__), "--prepare", "--config", args.config, "--workdir", args.workdir,
                               "--cpu-sample-pairs", str(npairs), "--ref-mbp", str(args.cfg["ref_mbp"]), "--read-len", str(args.read_len)],
                              env=env, stdout=sys.stderr)
    cfg = base_config(args, npairs)
    cfg["l2"] = "n/a (CPU run)"
    cfg["sample"] = "each step = the same bounded sample of %d pairs of the workload (the GPU arm runs %d pairs per step on the same index files)" % (
        npairs, args.pairs_per_step)
    vals = []
    for i in range(args.warmup + args.steps):
        a, w, _ = run_reference_soap4(args, prefix, fqp, os.path.join(d, "refout_ref"), ncores)
        if i >= args.warmup:
            vals.append(a)
    tot_align = sum(vals)
    value = npairs * len(vals) / tot_align
    cb = {"value": value, "unit": "pairs/s", "cores": ncores, "kind": "reference",
          "sample": "%d pairs per step of the same workload, oracle/_ref/soap4 -T %d (built -O3 -march=x86-64-v3: the AVX2 path, the widest the "
                    "reference has), its own 'Overall alignment time (excl. read loading)'" % (npairs, ncores)}
    emit(saved_stdout, {"impl": "reference", "metric": "read pairs aligned/sec", "value": value, "unit": "pairs/s", "n_gpus": args.gpus,
                      "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * tot_align / max(1, len(vals)),
                      "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8 (8-bit saturating SIMD DP, 2-bit FM-index)",
                      "data": "synthetic", "config": cfg, "cpu_baseline": cb,
                      "e2e": {"value": value, "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}})
    return 0


def run(args, saved_stdout):
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    ncores = os.cpu_count() or 1
    cfg = base_config(args, args.pairs_per_step)
    READ_LEN, MAX_READ_LEN_OPT = args.read_len, args.lopt

    import torch
    import megapath_b200 as mp
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: there is no CPU fallback for the product path")
    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=device)

    ctx = mp.Context(local)
    prefix, ref_codes, bounds_t, t_index = ensure_index(args, ctx, device, rank, world)
    info = ctx.index_info()
    cfg["l2"] = ("inputs larger than L2: %.1f GB HBM index gathered at random; every step also writes tens of GB of traceback tables, "
                 "which flushes the 126 MB L2 between steps" % (info["hbmBytes"] / 1e9))
    cfg["contexts_per_gpu"] = max(1, args.contexts)
    d, _ = workload_dir(args)
    cpu_legs = rank == 0 and world == 1 and not args.no_cpu_baseline
    if cpu_legs:
        ensure_samples(args, ref_codes, bounds_t, ("cpu", "cli"))

    # ---------------- our arm ----------------
    P = mp.default_params(nt2=args.cfg["ini"] == "soap4-nt2.ini", insert_low=READ_LEN, insert_high=INSERT_HIGH_OPT, max_read_length=MAX_READ_LEN_OPT)
    nb = min(args.warmup + args.steps, 6)
    batches = []
    lens = np.full(2 * args.pairs_per_step, READ_LEN, dtype=np.uint32)
    for b in range(nb):
        codes = gen_batch(ref_codes, bounds_t, args.pairs_per_step, 1000 + 97 * rank + b, READ_LEN, args.cfg["model"],
                          args.cfg["unalignable"], args.cfg["one_random"])
        host, wpq = pack_queries_torch(codes, MAX_READ_LEN_OPT)
        batches.append(host)
        del codes
    del ref_codes
    torch.cuda.empty_cache()
    h2d = batches[0].numel() * 4 + lens.nbytes
    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            import torch.distributed as dist
            dist.barrier()
        torch.cuda.synchronize()

    nctx = max(1, args.contexts)
    ctxs = [ctx]

    kept = []

    def run_steps(c, ids, upload, acc_out, keep_step=None):
        """steps `ids` on context c; upload=True: host buffers in (pinned -> HBM) every step; the result set of step `keep_step`
        stays with c and goes to `kept`"""
        for i in ids:
            if upload:
                c.batch_upload_ptr(batches[i % nb].data_ptr(), lens, wpq)
            t_call = time.perf_counter()
            if i == keep_step:
                s, res = summary_keeping_results(c, P)
                kept.append((c, res))
            else:
                s = c.align_pairs_summary(P)
            if os.environ.get("MP_BENCH_VERBOSE"):
                sys.stderr.write("  ctx %d step %d upload=%d: call %.1f ms (lib wall %.1f, seed %.1f, dp %.1f, fill %.1f, tb %.1f)\n" % (
                    ctxs.index(c) if c in ctxs else -1, i, int(upload), (time.perf_counter() - t_call) * 1e3, s["ms_wall"], s["ms_seed"], s["ms_dp"], s["ms_fill"], s["ms_tb"]))
            for k, v in s.items():
                acc_out[k] = acc_out.get(k, 0) + v

    # ---- warm-up (the K-mer filter is built once, before the other contexts borrow it) ----
    ctx.index_prepare(P)
    ctx.reserve(P, 2 * args.pairs_per_step)             # as the soap4 driver does before its batch loop (mp_reserve)
    run_steps(ctx, range(min(1, args.warmup)), True, {})
    for _ in range(nctx - 1):
        ctxs.append(ctx.clone())
        ctxs[-1].reserve(P, 2 * args.pairs_per_step)
    for ci, c in enumerate(ctxs):
        run_steps(c, range(ci, ci + max(args.warmup - (1 if ci == 0 else 0), 1)), True, {})
    if args.profile_step:
        torch.cuda.synchronize()
        torch.cuda.profiler.start()
        run_steps(ctx, [args.warmup], True, {})
        torch.cuda.synchronize()
        torch.cuda.profiler.stop()
        emit(saved_stdout, {"profile_step": True, "note": "one step under the profiler; not a bench value"})
        return 0
    sampler = ClockSampler(local)
    sampler.start()

    # ---- loop R: one context, steps back to back: per-kernel device times for the roofline (no overlap between kernels) ----
    barrier()
    l0 = mp.launch_count()
    acc = {}
    run_steps(ctx, range(args.warmup, args.warmup + args.steps), True, acc)
    barrier()
    launches = mp.launch_count() - l0
    acc["n_fill_launches"] = 0
    if os.environ.get("MP_BENCH_VERBOSE"):
        sys.stderr.write("rank %d loop R: %s\n" % (rank, json.dumps(dict({k: round(v / args.steps, 3) for k, v in acc.items() if k.startswith("ms_")}, exact=acc.get("dp_tasks_exact", 0) / max(1, acc.get("dp_tasks", 1))))))

    def pipelined(upload, keep_step=None):
        """K steps pulled from one queue by the contexts (one host thread each), so that a K that is not a multiple of the
        number of contexts leaves no context idle longer than one step; -> wall seconds between device syncs"""
        accs = [dict() for _ in ctxs]
        lock = threading.Lock()
        nxt = [args.warmup]

        def ids():
            while True:
                with lock:
                    i = nxt[0]
                    nxt[0] += 1
                if i >= args.warmup + args.steps:
                    return
                yield i
        ths = [threading.Thread(target=run_steps, args=(c, ids(), upload, accs[ci], keep_step)) for ci, c in enumerate(ctxs)]
        barrier()
        t0 = time.perf_counter()
        for t in ths:
            t.start()
        for t in ths:
            t.join()
        barrier()
        return time.perf_counter() - t0, accs

    # ---- loop A (value): every context's batch is resident in HBM before the clock starts; each step re-runs the whole
    #      hot path on it (the 10 GB of traceback tables a step writes flush L2 between steps) ----
    for ci, c in enumerate(ctxs):
        c.batch_upload_ptr(batches[(args.warmup + ci) % nb].data_ptr(), lens, wpq)
    dev_s, accsA = pipelined(False)
    dev_ms = dev_s * 1e3
    pairs_aligned_A = sum(a.get("pairs_aligned", 0) for a in accsA)
    # ---- loop B (e2e): the same through host buffers: pinned-host -> HBM upload of every batch, results in host memory ----
    last_step = args.warmup + args.steps - 1
    e2e_s, accsB = pipelined(True, last_step if args.dump_outputs else None)
    d2h = sum(a.get("result_bytes", 0) for a in accsB) / max(1, args.steps)
    clocks = sampler.stop()
    if args.dump_outputs:
        # loop B is the last timed pass; its last step aligned batch last_step % nb, the same batch on every run with these arguments
        dump_outputs(os.path.join(args.dump_outputs, "rank%d" % rank) if world > 1 else args.dump_outputs, copy_results(*kept[0]))

    from megapath_b200 import shard
    dev_ms_max, e2e_ms_max = shard.max_over_ranks([dev_ms, e2e_s * 1e3], device=device)     # slowest rank decides
    tot = shard.sum_counters({"pairs_aligned": pairs_aligned_A}, device=device)
    acc_pairs_all = tot["pairs_aligned"]
    total_pairs = args.pairs_per_step * args.steps * world
    value = total_pairs / (dev_ms_max / 1e3)
    e2e = total_pairs / (e2e_ms_max / 1e3)

    score40 = None
    if args.config == "cfg3":
        # the NT stage's downstream score cutoff (reassign / genKrakenReport, runMegaPath.sh:247-256) is applied to soap4's per-read best
        # score; report which fraction of the reads of one batch passes it (untimed)
        ctx.batch_upload_ptr(batches[0].data_ptr(), lens, wpq)
        full = ctx.align_pairs(P)
        best = full["pairs"][full["pairs"]["pad"] == 1]
        score40 = float(((best["score_1"] >= 40).sum() + (best["score_2"] >= 40).sum()) / (2.0 * args.pairs_per_step))
        del full, best
    hbm_peak, hbm_kind = measured_peak()
    # ---- roofline denominators MEASURED_PEAKS.json does not hold, measured now on this GPU (SURVEY.md 8d) ----
    try:
        gather32, gather64, dpx_peak = ctx.microbench(0), ctx.microbench(1), ctx.microbench(2)
    except Exception:
        gather32 = gather64 = dpx_peak = None
    steps = args.steps
    # dominant kernel: k_dp_fill (DP table fill).  cells the fill kernel really computed: tasks whose read occurs unchanged in its window are
    # answered by the exact-occurrence test (k_dp_exact, bit-identical results) and never reach it; dp_cells counts what the reference computes
    cells_filled = float(acc.get("dp_cells_filled") or acc["dp_cells"])
    gcups_fill = cells_filled / (acc["ms_fill"] / 1e3) / 1e9
    gcups_dp = acc["dp_cells"] / ((acc["ms_fill"] + acc["ms_tb"] + acc.get("ms_exact", 0.0)) / 1e3) / 1e9
    # DPX roofline (SURVEY.md 8d: the DP is bounded by the integer / DPX pipe).  The affine recurrence needs FOUR packed DPX
    # instructions per cell pair (D = add-max, I = add-max, H = max3, clip floor = max; two tasks share every 16x2 instruction), i.e. two
    # thread-instructions per cell; the kernel itself issues 6.4 per cell pair (two more add-max for the traceback flags, 0.4 for the
    # threshold test).  peak = the packed-16 DPX issue rate measured by mp_microbench(2) on this GPU (thread-instructions / s).
    DPX_RECURRENCE, DPX_KERNEL = 4.0, 6.4
    dpx_ach = gcups_fill * DPX_RECURRENCE / 2.0
    # seeding kernel: bytes it must gather = 8-byte filter probes + 16-byte LKT pairs + 64-byte occ blocks
    # (two per backward-search step that is not a text-compare step) + 4-byte SA values + 1 text byte per compare
    occ_steps = max(0.0, (acc["n_occ"] - 2.0 * acc["n_text"]) / 2.0)
    seed_bytes = 8.0 * acc["n_probe"] + 16.0 * acc["n_lkt"] + 128.0 * occ_steps + 4.0 * acc["n_sa"] + 1.0 * acc["n_text"]
    seed_ach = seed_bytes / (acc["ms_seed"] / 1e3) / 1e9
    traffic = ncu_traffic("k_dp_fill")
    roof = {"kernel": "k_dp_fill<%d,-2,-3> (packed 16-bit DPX table fill, the kernel with the largest share of the step)" % (5 if MAX_READ_LEN_OPT <= 160 else 8 if MAX_READ_LEN_OPT <= 256 else 10),
            "bound": "dpx", "achieved": dpx_ach, "peak": dpx_peak, "unit": "G DPX thread-instr/s", "frac": (dpx_ach / dpx_peak) if dpx_peak else None,
            "peak_kind": "measured now (mp_microbench kind 2: packed 16-bit DPX issue rate; MEASURED_PEAKS.json holds no integer-pipe figure)",
            "algorithmic": "%.0f packed DPX instructions per cell pair for the recurrence (D, I, H, clip floor) x cells the kernel fills / 2; cells = sum refLen*readLen "
                           "over the tasks it is given (SURVEY 8d)" % DPX_RECURRENCE,
            "frac_with_the_kernels_own_dpx_count": (gcups_fill * DPX_KERNEL / 2.0 / dpx_peak) if dpx_peak else None,
            "dpx_instr_per_cell_pair": {"recurrence": DPX_RECURRENCE, "kernel": DPX_KERNEL, "source": "static: SASS of the steady loop, profiles/r02_sass_k_dp_fill_steady_loop.txt"},
            # what actually limits the kernel: the integer ALU pipe as a whole (DPX min/max, PRMT, LOP3 share it; 9.8 instructions per
            # cell pair in the steady loop).  Busy fraction of that pipe from the newest committed ncu --set full capture (static, not live).
            "alu_pipe_busy_ncu": (lambda m: {"frac": m[0] / 100.0, "source": m[1], "metric": "sm__pipe_alu_cycles_active.avg.pct_of_peak_sustained_active"} if m else None)(
                ncu_metric("k_dp_fill", "sm__pipe_alu_cycles_active.avg.pct_of_peak_sustained_active")),
            # DRAM bytes (read + write) of ONE k_dp_fill launch from the newest committed ncu --set full capture
            "traffic": traffic["bytes_per_launch"] if traffic else None, "traffic_source": traffic["source"] if traffic else None,
            "ms_per_step": acc["ms_fill"] / steps,
            "hbm_note": {"achieved_gbs": gcups_fill, "peak_gbs": hbm_peak, "peak_kind": hbm_kind, "frac": gcups_fill / hbm_peak,
                         "algorithmic": "1 traceback byte written per DP cell the kernel computes"},
            "note": "per-kernel times come from a single-context pass (loop R), value/e2e from the pipelined passes",
            "compute": {"gcups_fill": gcups_fill, "gcups_reference_equivalent_all_dp_kernels": gcups_dp,
                        "exact_occurrence_test": {"tasks_per_step": acc.get("dp_tasks_exact", 0) / steps, "of_tasks_per_step": acc["dp_tasks"] / steps,
                                                  "ms_per_step": acc.get("ms_exact", 0.0) / steps,
                                                  "cells_filled_per_step": cells_filled / steps, "cells_reference_per_step": acc["dp_cells"] / steps}},
            "seeding": {"kernel": "k_mmp", "ms_per_step": acc["ms_seed"] / steps, "bytes_gathered_gbs": seed_ach,
                        "gather32_peak_gbs": gather32, "gather64_peak_gbs": gather64,
                        # every gather the kernel needs moves at least one 32-byte sector; occ blocks are 64-byte (two-sector) requests
                        "frac_of_gather_peak_on_bytes_needed": (seed_ach / gather32) if gather32 else None,
                        "counters_per_step": {k: acc[k] / steps for k in ("n_probe", "n_lkt", "n_occ", "n_sa", "n_text", "n_lf") if k in acc},
                        "note": "n_occ counts the occ evaluations the reference makes for the executed steps; starts rejected by the K-mer filter are not walked at all; "
                                "n_probe counts every filter probe issued, including re-probes that hit in L1"},
            "sa_lookup_gbs": (64.0 * acc["n_lf"] + 8.0 * acc["n_sa"]) / (acc["ms_sa"] / 1e3) / 1e9 if acc["ms_sa"] else None,
            "stage_ms_per_step": {k: acc[k] / steps for k in ("ms_seed", "ms_sa", "ms_pair", "ms_dp", "ms_fill", "ms_tb", "ms_exact", "ms_total", "ms_wall") if k in acc}}
    out = {"metric": "read pairs aligned/sec", "value": value, "unit": "pairs/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
           "ms_per_step": dev_ms_max / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int16/u8 (integer DP, 2-bit FM-index)",
           "data": "synthetic", "config": cfg, "clocks": clocks,
           "e2e": {"value": e2e, "unit": "pairs/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
           "gpu_launches": int(launches), "roofline": roof,
           "aligned_fraction": acc_pairs_all / (args.pairs_per_step * args.steps * world),
           "index_prepare_s": t_index}
    if score40 is not None:
        out["reads_with_score_ge_40_fraction"] = score40
    if cpu_legs:
        for c in ctxs[1:]:
            c.close()
        ctx.close()                       # the CLI legs load the index themselves: free this process's HBM first
        ctxs = [ctx]
        torch.cuda.empty_cache()
        npairs = args.cpu_sample_pairs
        fqp = sample_prefix(args, "cpu", npairs)
        try:
            a, w, ref_fq = run_reference_soap4(args, prefix, fqp, os.path.join(d, "refout_cpu"), ncores, keep_stdout=True)
            out["cpu_baseline"] = {"value": npairs / a, "unit": "pairs/s", "cores": ncores, "kind": "reference",
                                   "sample": "%d pairs of the same workload (same index files), oracle/_ref/soap4 -T %d, align loop %.1f s, wall %.1f s" % (
                                       npairs, ncores, a, w)}
            # parity where the numbers are made: the drop-in binary on the same index and sample must print the reference's records
            our_fq = os.path.join(d, "ourout_cpu.stdout.fq")
            run_our_soap4(args, prefix, fqp, os.path.join(d, "ourout_cpu"), ncores, sink=our_fq)
            want, got = canonical_pairs(ref_fq), canonical_pairs(our_fq)
            ndiff = sum(1 for x, y in zip(want, got) if x != y) + abs(len(want) - len(got))
            out["parity_at_scale"] = bool(ndiff == 0 and len(want) == npairs)
            out["parity_at_scale_detail"] = {"pairs_compared": len(want), "pairs_differing": ndiff,
                                             "what": "bin/soap4 vs oracle/_ref/soap4, annotated FASTQ of the CPU sample on the %.0f Mbp index, pairs sorted by name" % args.cfg["ref_mbp"]}
            for f in (ref_fq, our_fq):
                os.remove(f)
        except Exception as e:  # the baseline is reported, never the target: say why it is missing
            out.setdefault("cpu_baseline", {"value": None, "unit": "pairs/s", "cores": ncores, "kind": "reference", "sample": "unavailable: %s" % e})
            out.setdefault("parity_at_scale", None)
            out["parity_at_scale_error"] = str(e)[:300]
        if args.cli_pairs > 0:
            # e2e_cli: what the reference's own number means (SOAP4.cpp:613): FASTQ files in, annotated FASTQ out, the batch loop's wall time
            try:
                cli = sample_prefix(args, "cli", args.cli_pairs)
                os.sync()      # index and read files were written minutes ago at most: their write-back must not run beside the timed process
                loop_s, wall_s, cli_err = run_our_soap4(args, prefix, cli, os.path.join(d, "ourout_cli"), ncores, sink=os.path.join(d, "ourout_cli.stdout.fq"))
                sys.stderr.write("".join(l + "\n" for l in cli_err.splitlines() if "[timing]" in l or "Elapsed time on host" in l or "[mp_trace]" in l))
                out_bytes = os.path.getsize(os.path.join(d, "ourout_cli.stdout.fq"))
                os.remove(os.path.join(d, "ourout_cli.stdout.fq"))
                # the same run with stdout discarded: what the driver sustains when the consumer of its stdout is not the limit (a regular
                # file takes one thread's page-cache copy, about 4 - 5 GB/s on this box)
                loop0_s, _, cli_err0 = run_our_soap4(args, prefix, cli, os.path.join(d, "ourout_cli"), ncores, sink="/dev/null")
                out["e2e_cli"] = {"value": args.cli_pairs / loop_s, "unit": "pairs/s", "pairs": args.cli_pairs, "loop_s": loop_s, "process_wall_s": wall_s,
                                  "stdout_bytes": out_bytes, "value_stdout_discarded": args.cli_pairs / loop0_s, "loop_s_stdout_discarded": loop0_s,
                                  "io": "device" if "formatting on the device" in cli_err else "host",
                                  "what": "megapath_b200/bin/soap4 pair <index> r_1.fq r_2.fq -F -nc -T %d, stdout to a file; its 'Overall alignment time (excl. read "
                                          "loading)' line = wall time of the whole batch loop (parse + pack + upload + align + format + write; index load excluded, "
                                          "as in the reference)" % ncores}
            except Exception as e:
                out["e2e_cli"] = {"value": None, "unit": "pairs/s", "error": str(e)[:300]}
    if rank == 0:
        emit(saved_stdout, out)
    for c in ctxs[1:]:
        c.close()
    ctx.close()
    if world > 1:
        import torch.distributed as dist
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
