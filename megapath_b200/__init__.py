"""megapath_b200 -- B200-native soap4 alignment hot path (HKU-BAL/MegaPath), Python host mirror.

The product is libmegapath_b200.so (CUDA kernels + C-ABI, include/megapath_b200.h) and the
soap4-compatible C++ driver in csrc/.  This module only binds the C-ABI with ctypes so tests
and bench.py read like the reference's own call sequence (INDEXLoad -> load reads ->
soap3_dp_pair_align).  There is no CPU fallback: a missing library or GPU raises.
"""
import ctypes as C
import os
import subprocess
import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libmegapath_b200.so")


class MmpParams(C.Structure):
    _fields_ = [("seedSAsizeThreshold", C.c_int32), ("seedMinLength", C.c_int32),
                ("uniqThreshold", C.c_int32), ("indelFuzz", C.c_int32),
                ("goodSeedLen", C.c_int32), ("reseedLen", C.c_int32),
                ("reseedRLTratio", C.c_double), ("reseedAbsDiff", C.c_int32),
                ("shortSeedRatio", C.c_double)]


class AlignParams(C.Structure):
    _fields_ = [("mmp", MmpParams),
                ("matchScore", C.c_int32), ("mismatchScore", C.c_int32),
                ("openGapScore", C.c_int32), ("extendGapScore", C.c_int32),
                ("softClipLeft", C.c_int32), ("softClipRight", C.c_int32),
                ("insert_low", C.c_int32), ("insert_high", C.c_int32),
                ("peStrandLeftLeg", C.c_int32), ("peStrandRightLeg", C.c_int32),
                ("skipDefaultDP", C.c_int32), ("maxReadLength", C.c_int32)]


class Results(C.Structure):
    _fields_ = [("pairs", C.c_void_p), ("n_pairs", C.c_uint64),
                ("rescued", C.c_void_p), ("n_rescued", C.c_uint64),
                ("singles", C.c_void_p), ("n_singles", C.c_uint64),
                ("cigars", C.c_void_p), ("cigar_bytes", C.c_uint64),
                ("numDPAlignedPair", C.c_uint64), ("numDPAlignment", C.c_uint64),
                ("numSingleDPAligned", C.c_uint64), ("numSingleDPAlignment", C.c_uint64),
                ("numRescuedPair", C.c_uint64), ("numRescuedAlignment", C.c_uint64),
                ]


class Stats(C.Structure):
    _fields_ = [("n_occ", C.c_uint64), ("n_lf", C.c_uint64), ("n_sa", C.c_uint64), ("n_lkt", C.c_uint64),
                ("dp_cells", C.c_uint64), ("dp_tasks", C.c_uint64), ("n_probe", C.c_uint64), ("n_text", C.c_uint64),
                ("ms_seed", C.c_float), ("ms_sa", C.c_float), ("ms_pair", C.c_float),
                ("ms_dp", C.c_float), ("ms_total", C.c_float), ("ms_wall", C.c_float), ("ms_fill", C.c_float), ("ms_tb", C.c_float),
                ("dp_tasks_exact", C.c_uint64), ("dp_cells_filled", C.c_uint64), ("ms_exact", C.c_float), ("reserved_", C.c_float)]


SEEDPOS = np.dtype([("pos", "<u8"), ("strand_readID", "<u4"), ("paired_seedLength", "<u4")])
CAND = np.dtype([("readIDLeft", "<u4"), ("pad", "<u4"), ("pos0", "<u8"), ("pos1", "<u8")])
DP_TASK = np.dtype([("refStart", "<u8"), ("refLen", "<u4"), ("readID", "<u4"), ("readLen", "<u2"), ("strand", "u1"), ("valid", "u1"),
                    ("cutoff", "<i4"), ("diag", "<i2"), ("reserved_", "<u2")], align=True)      # mp_dp_task
PAIR_RESULT = np.dtype([
    ("readID", "<u4"), ("insertSize", "<i4"), ("algnmt_1", "<u8"), ("algnmt_2", "<u8"),
    ("score_1", "<i4"), ("score_2", "<i4"), ("editdist_1", "<i4"), ("editdist_2", "<i4"),
    ("num_sameScore_1", "<i4"), ("num_sameScore_2", "<i4"), ("strand_1", "u1"), ("strand_2", "u1"), ("pad", "<u2"),
    ("cigar_1", "<u4"), ("cigar_2", "<u4"), ("startPos_1", "<u8"), ("startPos_2", "<u8"),
    ("refDpLength_1", "<u4"), ("refDpLength_2", "<u4"), ("peLeftAnchor_1", "<u4"), ("peLeftAnchor_2", "<u4"),
    ("peRightAnchor_1", "<u4"), ("peRightAnchor_2", "<u4")], align=True)
SINGLE_RESULT = np.dtype([
    ("readID", "<u4"), ("cigar", "<u4"), ("algnmt", "<u8"), ("score", "<i4"), ("editdist", "<i4"),
    ("num_sameScore", "<i4"), ("strand", "u1"), ("pad", "u1", (3,)), ("seedAlignmentLength", "<u4"),
    ("startPos", "<u8"), ("refDpLength", "<u4"), ("peLeftAnchor", "<u4")], align=True)

_lib = None


class MegapathError(RuntimeError):
    pass


class FastqFormatError(MegapathError):
    """mp_fastq_upload: the text is not strict four-line FASTQ (MP_ERR_FORMAT)"""


MP_ERR_FORMAT = -6

# mp_gunzip constants (include/megapath_b200.h); the CPU model of the decoder (oracle/pygunzip.py) plans with them
GUNZIP_CHUNK = 65536
GUNZIP_SLOT = 1 << 20
GUNZIP_EVENTS = GUNZIP_CHUNK // 16 + 8
GUNZIP_MIN_DST = 65536


class GzipFormatError(MegapathError):
    """mp_gunzip_run refused the stream (MP_ERR_FORMAT); .partial holds the bytes zlib delivers before the error"""

    def __init__(self, msg, partial=b""):
        super().__init__(msg)
        self.partial = partial


class GunzipStats(C.Structure):         # mp_gunzip_stats_t
    _fields_ = [(f, C.c_uint64) for f in ("in_bytes", "out_bytes", "chunks", "candidates_tested", "candidates", "false_candidates",
                                          "merged", "overflows", "rounds", "members")] + [("ms_total", C.c_float), ("reserved_", C.c_float)]

    def as_dict(self):
        return {f: getattr(self, f) for f, _ in self._fields_ if f != "reserved_"}


class Annotation(C.Structure):          # mp_annotation
    _fields_ = [("dnaLength", C.c_uint64), ("numSeq", C.c_uint32), ("gridEntries", C.c_uint32), ("numTranslate", C.c_uint32), ("reserved_", C.c_uint32),
                ("grid", C.c_void_p), ("trStartPos", C.c_void_p), ("trChrID", C.c_void_p), ("names", C.c_void_p), ("nameOffsets", C.c_void_p)]


class FormatParams(C.Structure):        # mp_format_params
    _fields_ = [("top", C.c_double), ("megapathMode", C.c_int32), ("ignoreComments", C.c_int32)]


def build():
    """Compile the CUDA extension in-tree for sm_100a (nvcc cross-compiles without a GPU)."""
    subprocess.check_call(["make", "-s", "-C", os.path.join(HERE, "csrc")])


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise MegapathError("libmegapath_b200.so is not built (run __graft_entry__.build()); there is no CPU fallback")
        L = C.CDLL(LIB_PATH)
        L.mp_last_error.restype = C.c_char_p
        L.mp_init.argtypes = [C.c_int, C.POINTER(C.c_void_p)]
        L.mp_destroy.argtypes = [C.c_void_p]
        L.mp_clone.argtypes = [C.c_void_p, C.POINTER(C.c_void_p)]
        L.mp_index_bind.argtypes = [C.c_void_p, C.c_void_p]
        L.mp_index_load_budget.argtypes = [C.c_void_p, C.c_char_p, C.c_uint64]
        L.mp_fastq_chain.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p]
        L.mp_index_prepare.argtypes = [C.c_void_p, C.c_void_p]
        L.mp_reserve.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32]
        L.mp_index_load.argtypes = [C.c_void_p, C.c_char_p]
        L.mp_index_info.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.mp_index_build.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64]
        L.mp_index_save.argtypes = [C.c_void_p, C.c_char_p]
        L.mp_index_save_annotation.argtypes = [C.c_char_p, C.c_uint64, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p]
        L.mp_launch_count.restype = C.c_uint64
        L.mp_microbench.argtypes = [C.c_void_p, C.c_int, C.c_void_p]
        L.mp_occ.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64]
        L.mp_sa.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64]
        L.mp_lkt.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64]
        L.mp_batch_upload.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32]
        L.mp_seed_pairs.argtypes = [C.c_void_p, C.c_void_p]
        L.mp_download_seedpos.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.mp_download_candidates.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        L.mp_free.argtypes = [C.c_void_p]
        L.mp_dp_batch.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p, C.c_uint32,
                                  C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32,
                                  C.c_void_p, C.c_void_p, C.c_int32, C.c_int32]
        L.mp_dp_tasks.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32,
                                  C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.mp_align_pairs.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        L.mp_results_release.argtypes = [C.c_void_p, C.c_void_p]
        L.mp_last_stats.argtypes = [C.c_void_p, C.c_void_p]
        L.mp_default_params.argtypes = [C.c_void_p, C.c_int]
        L.mp_fastq_upload.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64, C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p]
        L.mp_annotation_upload.argtypes = [C.c_void_p, C.c_void_p]
        L.mp_format_fastq.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        L.mp_format_fetch.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64]
        L.mp_results_on_device.argtypes = [C.c_void_p, C.c_int]
        L.mp_fastq_reserve.argtypes = [C.c_void_p, C.c_uint64, C.c_uint32]
        L.mp_host_alloc.argtypes = [C.c_uint64]
        L.mp_host_alloc.restype = C.c_void_p
        L.mp_host_free.argtypes = [C.c_void_p]
        L.mp_bgzf_reserve.argtypes = [C.c_void_p, C.c_uint64]
        L.mp_bgzf_compress.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64, C.POINTER(C.c_uint64)]
        L.mp_gunzip_open.argtypes = [C.c_void_p, C.c_uint64, C.POINTER(C.c_void_p)]
        L.mp_gunzip_run.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_int, C.c_void_p, C.c_uint64,
                                    C.POINTER(C.c_uint64), C.POINTER(C.c_uint64), C.POINTER(C.c_int)]
        L.mp_gunzip_stats.argtypes = [C.c_void_p, C.c_void_p]
        L.mp_gunzip_close.argtypes = [C.c_void_p]
        _lib = L
    return _lib


def launch_count():
    """Kernels of libmegapath_b200.so launched so far in this process."""
    return int(lib().mp_launch_count())


def save_annotation(prefix, text_length, names, starts, lengths):
    """.ann/.amb/.tra for an ACGT-only multi-sequence text (HSP.c:569-699)."""
    arr = (C.c_char_p * len(names))(*[n.encode() for n in names])
    st = np.ascontiguousarray(starts, dtype=np.uint64)
    ln = np.ascontiguousarray(lengths, dtype=np.uint64)
    rc = lib().mp_index_save_annotation(prefix.encode(), int(text_length), len(names), arr, _ptr(st), _ptr(ln))
    if rc != 0:
        raise MegapathError("%s (status %d)" % (lib().mp_last_error().decode(), rc))


def pack_text(codes):
    """codes 0..3 (numpy uint8) -> .pac bytes: 4 bases per byte, first base in the top 2 bits."""
    n = len(codes)
    c = np.zeros((n + 3) // 4 * 4, dtype=np.uint8)
    c[:n] = codes
    c = c.reshape(-1, 4)
    return ((c[:, 0] << 6) | (c[:, 1] << 4) | (c[:, 2] << 2) | c[:, 3]).astype(np.uint8)


def bgzf_bound(n):
    """MP_BGZF_BOUND(n): output capacity mp_bgzf_compress needs for n input bytes."""
    return (n + 0xff00 - 1) // 0xff00 * 65536


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p)


def default_params(nt2=False, insert_low=1, insert_high=500, max_read_length=120):
    p = AlignParams()
    lib().mp_default_params(C.byref(p), int(nt2))
    p.insert_low, p.insert_high, p.maxReadLength = insert_low, insert_high, max_read_length
    return p


def words_per_query(max_read_length):
    """getWordPerQuery (dependencies.h:204-207)."""
    return (max_read_length + 15) // 16


def pack_queries(codes, lens, max_read_length):
    """Host mirror of appendToQueryArrays (QueryParser.cpp:184-203): 2-bit, 16 bases per word
    LSB-first, 32-read interleaved.  codes: (nReads, >=maxLen) uint8 in 0..3."""
    n = codes.shape[0]
    wpq = words_per_query(max_read_length)
    npad = (n + 31) // 32 * 32
    width = wpq * 16
    c = np.zeros((npad, width), dtype=np.uint32)
    w = min(width, codes.shape[1])
    c[:n, :w] = codes[:, :w]
    mask = np.arange(width)[None, :] < np.concatenate([lens, np.zeros(npad - n, dtype=lens.dtype)])[:, None]
    c *= mask
    shifts = (2 * (np.arange(width) % 16)).astype(np.uint32)
    words = (c << shifts[None, :]).reshape(npad, wpq, 16).sum(axis=2, dtype=np.uint64).astype(np.uint32)   # (npad, wpq)
    il = words.reshape(npad // 32, 32, wpq).transpose(0, 2, 1).reshape(-1)      # word j of read r at grp*32*wpq + 32*j + r%32
    return np.ascontiguousarray(il, dtype=np.uint32), wpq


def pack_dp_interleaved(seqs, lens, max_len):
    """Host mirror of packRead / repackDNA (DV-DPfunctions.cpp:3009-3073): 2-bit MSB-first,
    1-based, 32-task interleaved.  seqs: (n, max_len) uint8 codes."""
    n = seqs.shape[0]
    w = (max_len + 15) >> 4
    npad = (n + 31) // 32 * 32
    out = np.zeros(npad * w, dtype=np.uint32)
    for t in range(n):
        base = (t // 32) * 32 * w + (t % 32)
        for i in range(1, int(lens[t]) + 1):
            out[base + ((i >> 4) << 5)] |= np.uint32(int(seqs[t, i - 1]) & 3) << np.uint32((15 - (i & 15)) << 1)
    return out


class Context:
    """One GPU context (mp_context).  Method names follow include/megapath_b200.h."""

    def __init__(self, device=0, _clone_of=None):
        self.L = lib()
        self.h = C.c_void_p()
        if _clone_of is None:
            self._check(self.L.mp_init(device, C.byref(self.h)))
        else:
            self._check(self.L.mp_clone(_clone_of.h, C.byref(self.h)))
            self._has_index = True
            self._parent = _clone_of          # the index owner must outlive the clone

    def clone(self):
        """Second context on the same GPU sharing this context's resident index (mp_clone)."""
        return Context(_clone_of=self)

    def _check(self, rc):
        if rc != 0:
            raise MegapathError("%s (status %d)" % (self.L.mp_last_error().decode(), rc))

    def close(self):
        if self.h:
            self.L.mp_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- index ----
    def index_load(self, prefix):
        self._check(self.L.mp_index_load(self.h, prefix.encode()))
        self._has_index = True

    def index_load_budget(self, prefix, max_bytes):
        """mp_index_load with the resident index and its K-mer filter kept within max_bytes of HBM."""
        self._check(self.L.mp_index_load_budget(self.h, prefix.encode(), int(max_bytes)))
        self._has_index = True

    def index_bind(self, owner):
        """Points this clone at owner's resident index, K-mer filter and annotation (mp_index_bind)."""
        self._check(self.L.mp_index_bind(self.h, owner.h))
        self._bound = owner                   # the owner must outlive the binding

    def index_build(self, text2bit, n):
        """GPU FM-index construction from a .pac-packed text (replaces 2bwt-builder)."""
        text2bit = np.ascontiguousarray(text2bit, dtype=np.uint8)
        self._check(self.L.mp_index_build(self.h, _ptr(text2bit), n))
        self._has_index = True

    def index_build_codes(self, codes_t, bounds, prefix=None):
        """codes_t: torch uint8 tensor of codes 0..3 (any device); bounds: sequence boundaries (nseq+1).
        Builds the index in HBM and, if prefix is given, exports it in the reference's file formats."""
        import torch
        n = codes_t.numel()
        pad = (-n) % 4
        c = codes_t if pad == 0 else torch.cat([codes_t, torch.zeros(pad, dtype=torch.uint8, device=codes_t.device)])
        c = c.view(-1, 4)
        pac = ((c[:, 0] << 6) | (c[:, 1] << 4) | (c[:, 2] << 2) | c[:, 3]).to(torch.uint8).cpu().numpy()
        del c
        self.index_build(pac, n)
        if prefix is not None:
            self.index_save(prefix)
            b = np.asarray(bounds, dtype=np.uint64)
            save_annotation(prefix, n, ["seq%d" % (i + 1) for i in range(len(b) - 1)], b[:-1], b[1:] - b[:-1])

    def index_prepare(self, params):
        """Builds the K-mer presence filter for these parameters now (before clone())."""
        self._check(self.L.mp_index_prepare(self.h, C.byref(params)))

    def reserve(self, params, n_reads):
        """Pre-sizes the per-batch buffers for batches of up to n_reads reads (mp_reserve)."""
        self._check(self.L.mp_reserve(self.h, C.byref(params), int(n_reads)))

    def has_index(self):
        return getattr(self, "_has_index", False)

    def index_save(self, prefix):
        self._check(self.L.mp_index_save(self.h, prefix.encode()))

    def index_info(self):
        n, isa0, hbm = C.c_uint64(), C.c_uint64(), C.c_uint64()
        cum = (C.c_uint64 * 5)()
        self._check(self.L.mp_index_info(self.h, C.byref(n), C.byref(isa0), cum, C.byref(hbm)))
        return dict(textLength=n.value, inverseSa0=isa0.value, cumFreq=list(cum), hbmBytes=hbm.value)

    def occ(self, idx, c):
        idx = np.ascontiguousarray(idx, dtype=np.uint64)
        c = np.ascontiguousarray(c, dtype=np.uint32)
        out = np.empty(len(idx), dtype=np.uint64)
        self._check(self.L.mp_occ(self.h, _ptr(idx), _ptr(c), _ptr(out), len(idx)))
        return out

    def sa(self, idx):
        idx = np.ascontiguousarray(idx, dtype=np.uint64)
        out = np.empty(len(idx), dtype=np.uint64)
        self._check(self.L.mp_sa(self.h, _ptr(idx), _ptr(out), len(idx)))
        return out

    def lkt(self, keys):
        keys = np.ascontiguousarray(keys, dtype=np.uint32)
        l = np.empty(len(keys), dtype=np.uint64)
        r = np.empty(len(keys), dtype=np.uint64)
        self._check(self.L.mp_lkt(self.h, _ptr(keys), _ptr(l), _ptr(r), len(keys)))
        return l, r

    def microbench(self, kind):
        """0/1: random 32-/64-byte gather GB/s; 2: packed-16 DPX Ginstr/s (roofline denominators)."""
        out = C.c_double()
        self._check(self.L.mp_microbench(self.h, kind, C.byref(out)))
        return out.value

    # ---- batch ----
    def batch_upload(self, queries, read_lengths, wpq):
        queries = np.ascontiguousarray(queries, dtype=np.uint32)
        read_lengths = np.ascontiguousarray(read_lengths, dtype=np.uint32)
        self._keep = (queries, read_lengths)
        self._check(self.L.mp_batch_upload(self.h, _ptr(queries), _ptr(read_lengths), len(read_lengths), wpq))
        self._n_reads = len(read_lengths)

    def batch_upload_ptr(self, host_ptr, read_lengths, wpq):
        """Same call with a raw host pointer (e.g. a pinned torch tensor's data_ptr())."""
        read_lengths = np.ascontiguousarray(read_lengths, dtype=np.uint32)
        self._keep = (read_lengths,)
        self._check(self.L.mp_batch_upload(self.h, C.c_void_p(host_ptr), _ptr(read_lengths), len(read_lengths), wpq))

    def fastq_upload(self, text1, text2, n_pairs, max_read_length):
        """Device ingest (mp_fastq_upload): the raw four-line FASTQ text of n_pairs records per mate -> clamped read lengths.
        Raises FastqFormatError when the text is not strict four-line FASTQ (the caller's own parser takes the batch then)."""
        lens = C.POINTER(C.c_uint32)()
        self._keep = (text1, text2)
        rc = self.L.mp_fastq_upload(self.h, C.c_char_p(text1), len(text1), C.c_char_p(text2), len(text2), n_pairs,
                                    words_per_query(max_read_length), max_read_length, C.byref(lens))
        if rc == MP_ERR_FORMAT:
            raise FastqFormatError(self.L.mp_last_error().decode())
        self._check(rc)
        self._n_reads = 2 * n_pairs
        return np.ctypeslib.as_array(lens, shape=(2 * n_pairs,)).copy()

    def fastq_chain(self, max_read_length):
        """mp_fastq_chain: the batch's last formatted text, rewritten as the next chunk reads it, becomes the batch -> clamped read
        lengths.  Raises FastqFormatError when the ingest refuses the rewritten text (the formatted text is still fetchable then)."""
        lens = C.POINTER(C.c_uint32)()
        rc = self.L.mp_fastq_chain(self.h, words_per_query(max_read_length), max_read_length, C.byref(lens))
        if rc == MP_ERR_FORMAT:
            raise FastqFormatError(self.L.mp_last_error().decode())
        self._check(rc)
        return np.ctypeslib.as_array(lens, shape=(self._n_reads,)).copy()

    def annotation_upload(self, prefix):
        """mp_annotation_upload from <prefix>.ann / .tra (the tables getChrAndPos reads, BGS-IO.cpp:163-190)."""
        ann = open(prefix + ".ann").read().split("\n")
        n, ns = int(ann[0].split()[0]), int(ann[0].split()[1])
        names = [ann[1 + 2 * i].split(" ", 1)[1].encode() for i in range(ns)]
        tra = open(prefix + ".tra").read().split("\n")
        _, _, removed, grid_entries = (int(x) for x in tra[0].split())
        grid = np.array([int(x) for x in tra[1:1 + grid_entries]], dtype=np.uint32)
        rows = [tra[1 + grid_entries + j].split() for j in range(ns + removed)]
        tr_start = np.array([int(r[0]) for r in rows], dtype=np.uint64)
        tr_chr = np.array([int(r[1]) for r in rows], dtype=np.uint32)
        blob = b"".join(names)
        off = np.zeros(ns + 1, dtype=np.uint64)
        off[1:] = np.cumsum([len(x) for x in names])
        a = Annotation(n, ns, grid_entries, ns + removed, 0, _ptr(grid), _ptr(tr_start), _ptr(tr_chr), C.cast(C.c_char_p(blob), C.c_void_p), _ptr(off))
        self._check(self.L.mp_annotation_upload(self.h, C.byref(a)))

    def format_fastq(self, top=0.95, mode=1, ignore_comments=True):
        """Device egress (mp_format_fastq + mp_format_fetch): the annotated FASTQ text of the batch just aligned."""
        f = FormatParams(top, mode, 1 if ignore_comments else 0)
        n = C.c_uint64()
        self._check(self.L.mp_format_fastq(self.h, C.byref(f), C.byref(n)))
        buf = C.create_string_buffer(max(int(n.value), 1))
        self._check(self.L.mp_format_fetch(self.h, buf, n.value))
        return buf.raw[:n.value]

    def bgzf_reserve(self, max_bytes):
        """Pre-sizes the compression buffers for inputs of up to max_bytes (mp_bgzf_reserve)."""
        self._check(self.L.mp_bgzf_reserve(self.h, int(max_bytes)))

    def bgzf_compress(self, data):
        """Device BGZF compression (mp_bgzf_compress): any bytes -> a run of complete BGZF members (no EOF marker)."""
        data = bytes(data)
        cap = bgzf_bound(len(data))
        buf = C.create_string_buffer(max(cap, 1))
        n = C.c_uint64()
        self._check(self.L.mp_bgzf_compress(self.h, C.c_char_p(data), len(data), buf, cap, C.byref(n)))
        return buf.raw[:n.value]

    def gunzip_stream(self, max_in):
        """A Gunzip handle on this context for calls of up to max_in compressed bytes (mp_gunzip_open)."""
        return Gunzip(self, max_in)

    def gunzip(self, data, piece=None, out_cap=None):
        """Device gzip inflate of a whole file (mp_gunzip_run): fed piece bytes at a time (default: all at once), writing at most
        out_cap bytes per call (default: 64 MiB).  Raises GzipFormatError (with .partial) where zlib refuses the stream."""
        data = memoryview(bytes(data))
        piece = int(piece or max(len(data), GUNZIP_MIN_DST))
        with Gunzip(self, piece) as g:
            return g.inflate(data, out_cap)


    def seed_pairs(self, params):
        self._check(self.L.mp_seed_pairs(self.h, C.byref(params)))

    def download_seedpos(self):
        rp, mp = C.c_void_p(), C.c_void_p()
        nr, nm = C.c_uint64(), C.c_uint64()
        self._check(self.L.mp_download_seedpos(self.h, C.byref(rp), C.byref(nr), C.byref(mp), C.byref(nm)))
        a = np.frombuffer((C.c_char * (nr.value * 16)).from_address(rp.value), dtype=SEEDPOS).copy()
        b = np.frombuffer((C.c_char * (nm.value * 16)).from_address(mp.value), dtype=SEEDPOS).copy()
        self.L.mp_free(rp)
        self.L.mp_free(mp)
        return a, b

    def download_candidates(self):
        p, n = C.c_void_p(), C.c_uint64()
        self._check(self.L.mp_download_candidates(self.h, C.byref(p), C.byref(n)))
        out = np.frombuffer((C.c_char * (n.value * 24)).from_address(p.value), dtype=CAND).copy() if n.value else np.zeros(0, CAND)
        self.L.mp_free(p)
        return out

    # ---- DP seam ----
    def dp_batch(self, packed_dna, dna_lens, max_dna, packed_read, read_lens, max_read, cutoffs,
                 clip_lt=130, clip_rt=130, mismatch=-2, gap_open=-3):
        n = len(dna_lens)
        dna_lens = np.ascontiguousarray(dna_lens, dtype=np.uint32)
        read_lens = np.ascontiguousarray(read_lens, dtype=np.uint32)
        cutoffs = np.ascontiguousarray(cutoffs, dtype=np.int32)
        scores = np.zeros(n, dtype=np.int32)
        hits = np.zeros(n, dtype=np.uint32)
        cnts = np.zeros(n, dtype=np.uint32)
        pats = np.zeros((n, max_dna + max_read), dtype=np.uint8)
        cl = np.full(max(n, 1), clip_lt, dtype=np.uint32)
        cr = np.full(max(n, 1), clip_rt, dtype=np.uint32)
        self._check(self.L.mp_dp_batch(self.h, _ptr(packed_dna), _ptr(dna_lens), max_dna, _ptr(packed_read), _ptr(read_lens),
                                       max_read, _ptr(cutoffs), _ptr(scores), _ptr(hits), _ptr(cnts), _ptr(pats), n,
                                       _ptr(cl), _ptr(cr), mismatch, gap_open))
        return scores, hits, cnts, pats

    def dp_tasks(self, tasks, max_ref, max_read, clip_lt=130, clip_rt=130):
        """mp_dp_tasks: tasks (numpy array of DP_TASK) against the resident index and the uploaded batch -> scores, hits, counts, patterns."""
        tasks = np.ascontiguousarray(tasks, dtype=DP_TASK)
        n = len(tasks)
        scores = np.zeros(n, dtype=np.int32)
        hits = np.zeros(n, dtype=np.uint32)
        cnts = np.zeros(n, dtype=np.uint32)
        pats = np.zeros((n, max_ref + max_read), dtype=np.uint8)
        self._check(self.L.mp_dp_tasks(self.h, _ptr(tasks), n, max_ref, max_read, clip_lt, clip_rt, _ptr(scores), _ptr(hits), _ptr(cnts), _ptr(pats)))
        return scores, hits, cnts, pats

    # ---- whole stage sequence ----
    def align_pairs(self, params):
        """-> dict with numpy copies of the result arrays and the counters."""
        res = Results()
        self._check(self.L.mp_align_pairs(self.h, C.byref(params), C.byref(res)))

        def arr(p, n, dt):
            if not n:
                return np.zeros(0, dtype=dt)
            return np.frombuffer((C.c_char * (n * dt.itemsize)).from_address(p), dtype=dt).copy()
        out = dict(pairs=arr(res.pairs, res.n_pairs, PAIR_RESULT), rescued=arr(res.rescued, res.n_rescued, PAIR_RESULT),
                   singles=arr(res.singles, res.n_singles, SINGLE_RESULT),
                   cigars=bytes((C.c_char * res.cigar_bytes).from_address(res.cigars)) if res.cigar_bytes else b"")
        for name, _ in Results._fields_[8:]:
            out[name] = getattr(res, name)
        out.update(self.last_stats())
        self.L.mp_results_release(self.h, C.byref(res))
        return out

    def last_stats(self):
        """work counters and device timings of this context's last mp_align_pairs call (mp_last_stats)"""
        st = Stats()
        self._check(self.L.mp_last_stats(self.h, C.byref(st)))
        return {name: getattr(st, name) for name, _ in Stats._fields_ if name != "reserved_"}


def _summary(self, params):
    """mp_align_pairs without copying the result arrays out of the library's host arena:
    -> counters + sizes (bench.py)."""
    res = Results()
    self._check(self.L.mp_align_pairs(self.h, C.byref(params), C.byref(res)))
    out = {name: getattr(res, name) for name, _ in Results._fields_[8:]}
    out.update(self.last_stats())
    out["n_pairs"], out["n_singles"], out["n_rescued"] = res.n_pairs, res.n_singles, res.n_rescued
    out["result_bytes"] = (res.n_pairs + res.n_rescued) * PAIR_RESULT.itemsize + res.n_singles * SINGLE_RESULT.itemsize + res.cigar_bytes
    out["pairs_aligned"] = res.numDPAlignedPair + res.numRescuedPair
    self.L.mp_results_release(self.h, C.byref(res))
    return out


Context.align_pairs_summary = _summary


def cigar_at(cigars, off):
    end = cigars.index(b"\0", off)
    return cigars[off:end]


class Gunzip:
    """One gzip stream inflated on the device (mp_gunzip handle): run() one call at a time, or inflate() a whole buffer."""

    def __init__(self, ctx, max_in):
        self.ctx, self.L, self.max_in = ctx, ctx.L, int(max_in)
        self.h = C.c_void_p()
        ctx._check(self.L.mp_gunzip_open(ctx.h, self.max_in, C.byref(self.h)))

    def run(self, src, fin, out_cap=GUNZIP_MIN_DST):
        """One mp_gunzip_run call -> (output bytes, consumed, done).  src: the file's bytes from the previous call's consumed on."""
        src = bytes(src)
        dst = C.create_string_buffer(int(out_cap))
        consumed, produced, done = C.c_uint64(), C.c_uint64(), C.c_int()
        rc = self.L.mp_gunzip_run(self.h, C.c_char_p(src), len(src), int(bool(fin)), dst, int(out_cap), C.byref(consumed),
                                  C.byref(produced), C.byref(done))
        out = dst.raw[:produced.value]
        if rc == MP_ERR_FORMAT:
            raise GzipFormatError(self.L.mp_last_error().decode(), out)
        self.ctx._check(rc)
        return out, consumed.value, bool(done.value)

    def inflate(self, data, out_cap=None):
        data = memoryview(data)
        out_cap = int(out_cap or 64 << 20)
        parts, pos = [], 0
        while True:
            src = data[pos:pos + self.max_in]
            try:
                out, used, done = self.run(src, pos + len(src) == len(data), out_cap)
            except GzipFormatError as e:
                e.partial = b"".join(parts) + e.partial
                raise
            parts.append(out)
            pos += used
            if done:
                return b"".join(parts)
            if not out and not used:
                raise MegapathError("mp_gunzip_run made no progress")

    def stats(self):
        s = GunzipStats()
        self.ctx._check(self.L.mp_gunzip_stats(self.h, C.byref(s)))
        return s.as_dict()

    def close(self):
        if self.h:
            self.L.mp_gunzip_close(self.h)
            self.h = C.c_void_p()

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
