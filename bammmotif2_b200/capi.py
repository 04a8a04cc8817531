"""ctypes binding of the C ABI in include/bamm_b200.h (libbamm_b200.so, built in-tree by build.py).

This is plumbing for the tests and bench.py; the drop-in host side of the product is the C++ mirror of the
reference classes in bammmotif2_b200/host/. There is no fallback: if the library is missing the import fails,
and every compute call fails without a CUDA device.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("BAMM_LIB") or os.path.join(_HERE, "libbamm_b200.so")   # BAMM_LIB: kernel-variant experiments

_u8p, _u32p, _u64p, _f32p = (C.POINTER(t) for t in (C.c_uint8, C.c_uint32, C.c_uint64, C.c_float))
_vp = C.c_void_p

# name -> (restype, argtypes); every entry point declared in include/bamm_b200.h
SIGNATURES = {
    "bamm_version": (C.c_int, []),
    "bamm_last_error": (C.c_char_p, []),
    "bamm_device_count": (C.c_int, [C.POINTER(C.c_int)]),
    "bamm_set_device": (C.c_int, [C.c_int]),
    "bamm_plan_describe": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, C.c_uint64, C.POINTER(C.c_int32), C.c_uint64, _u64p]),
    "bamm_device_info": (C.c_int, [C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int), _u64p]),
    "bamm_seqset_create": (C.c_int, [_u8p, _u64p, C.c_uint64, C.c_int, _u64p, _u64p, C.c_uint64, C.POINTER(_vp)]),
    "bamm_seqset_index": (C.c_int, [_vp, C.c_int]),
    "bamm_seqset_get_index": (C.c_int, [_vp, C.c_int, _u32p]),
    "bamm_seqset_info": (C.c_int, [_vp, _u64p, _u64p, C.POINTER(C.c_int)]),
    "bamm_seqset_count_kmers": (C.c_int, [_vp, C.c_int, _u64p]),
    "bamm_seqset_destroy": (None, [_vp]),
    "bamm_seqset_get_codes": (C.c_int, [_vp, _u8p]),
    "bamm_seqset_get_offsets": (C.c_int, [_vp, _u64p]),
    "bamm_seqset_encode_text": (C.c_int, [C.c_char_p, C.c_uint64, _vp, C.c_uint64, _u64p, _u32p, C.c_uint64, C.c_int, C.c_int, _u8p, _u8p, _u64p, _u64p, C.POINTER(_vp)]),
    "bamm_seqset_forward_zeros": (C.c_int, [_vp, _u64p]),
    "bamm_seqset_code_windows": (C.c_int, [_vp, _u64p, _u64p, _u64p, C.c_uint64, _u8p]),
    "bamm_seqset_finish_patches": (C.c_int, [_vp, _u64p, _u64p, C.c_uint64]),
    "bamm_seqset_sample_negatives": (C.c_int, [_vp, _u64p, C.c_uint64, C.c_uint64, C.c_uint32, C.POINTER(_vp)]),
    "bamm_seqset_negative_kmer_counts": (C.c_int, [_vp, _u64p, C.c_uint64, _u64p]),
    "bamm_seqset_sample_negatives_shard": (C.c_int, [_vp, _u64p, C.c_uint64, C.c_uint64, C.c_uint32, C.c_uint64, _u64p, C.POINTER(_vp)]),
    "bamm_rand_stream": (C.c_int, [C.c_uint32, C.c_uint64, C.c_uint64, C.POINTER(C.c_int32)]),
    "bamm_em_create": (C.c_int, [_vp, _u64p, C.c_uint64, C.c_int, C.c_int, C.c_int, C.POINTER(_vp)]),
    "bamm_em_set_model": (C.c_int, [_vp, _f32p, _f32p, _f32p, C.c_float]),
    "bamm_em_estep": (C.c_int, [_vp, _f32p]),
    "bamm_em_mstep": (C.c_int, [_vp]),
    "bamm_em_optimize_q": (C.c_int, [_vp, _f32p]),
    "bamm_em_optimize": (C.c_int, [_vp, C.c_int, C.c_float, C.c_int, C.POINTER(C.c_int), _f32p, _f32p, _f32p]),
    "bamm_em_mask": (C.c_int, [_vp, C.c_float, C.c_float, C.c_int, C.POINTER(C.c_int), _f32p, _u64p, _f32p]),
    "bamm_em_iterate": (C.c_int, [_vp, C.c_int, _f32p, _f32p]),
    "bamm_em_get_model": (C.c_int, [_vp, _f32p]),
    "bamm_em_get_counts": (C.c_int, [_vp, _f32p]),
    "bamm_em_get_s": (C.c_int, [_vp, _f32p]),
    "bamm_em_get_q": (C.c_int, [_vp, _f32p]),
    "bamm_em_get_r": (C.c_int, [_vp, C.c_uint64, C.c_uint64, _f32p]),
    "bamm_em_r_size": (C.c_uint64, [_vp]),
    "bamm_em_last_timing": (C.c_int, [_vp, _f32p, _f32p]),
    "bamm_em_loop_timing": (C.c_int, [_vp, C.POINTER(C.c_int), _f32p, _f32p, _f32p, _f32p]),
    "bamm_bound_plan_describe": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_uint64, C.POINTER(C.c_int32), C.c_uint64, _u64p]),
    "bamm_set_device_group": (C.c_int, [C.POINTER(C.c_int), C.c_int]),
    "bamm_get_device_group": (C.c_int, [C.POINTER(C.c_int), C.c_int, C.POINTER(C.c_int)]),
    "bamm_em_loop_timing_estep": (C.c_int, [_vp, _f32p, _f32p, _f32p]),
    "bamm_em_set_exchange_buffer": (C.c_int, [_vp, _vp, C.c_uint64]),
    "bamm_em_launch_count": (C.c_int, [_vp, _u64p]),
    "bamm_em_estep_info": (C.c_int, [_vp, _u64p]),
    "bamm_em_bound_reuse_info": (C.c_int, [_vp, _u64p, C.POINTER(C.c_float)]),
    "bamm_em_destroy": (None, [_vp]),
    "bamm_em_exchange_buffer": (C.c_int, [_vp, C.POINTER(_vp), _u64p]),
    "bamm_em_set_global_nseq": (C.c_int, [_vp, C.c_uint64]),
    "bamm_em_estep_local": (C.c_int, [_vp]),
    "bamm_em_mstep_local": (C.c_int, [_vp]),
    "bamm_em_finish_iteration": (C.c_int, [_vp, C.c_int, _f32p, _f32p]),
    "bamm_em_stream": (C.c_int, [_vp, C.POINTER(_vp)]),
    "bamm_em_peer_alloc": (C.c_int, [_vp, C.c_int, C.c_int, _vp]),
    "bamm_em_peer_attach": (C.c_int, [_vp, _vp]),
    "bamm_em_peer_wait": (C.c_int, [_vp, C.c_int, C.POINTER(C.c_double), _u64p]),
    "bamm_score_last_timing": (C.c_int, [_f32p]),
    "bamm_seqset_sample_pwm_sites": (C.c_int, [_vp, _u64p, C.c_uint64, C.c_int, C.c_int, C.c_int, _f32p, C.c_float, C.POINTER(C.c_double), C.POINTER(C.c_int32), _u64p]),
    "bamm_sort_scores": (C.c_int, [_f32p, C.c_uint64, C.c_int]),
    "bamm_mops_pvalues": (C.c_int, [_f32p, C.c_uint64, _f32p, C.c_uint64, C.c_uint64, _f32p, _f32p]),
    "bamm_score_logodds": (C.c_int, [_vp, _u64p, C.c_uint64, C.c_int, C.c_int, C.c_int, _f32p, _f32p, _f32p, _u64p, _f32p]),
    "bamm_scan_create": (C.c_int, [_vp, _u64p, C.c_uint64, C.c_int, C.c_int, C.c_int, _f32p, _f32p, C.POINTER(_vp)]),
    "bamm_scan_hits": (C.c_int, [_vp, _vp, _u64p, C.c_uint64, C.c_uint64, C.c_float, _u64p, _vp, C.c_uint64, _u64p]),
    "bamm_scan_info": (C.c_int, [_vp, _u64p, _f32p, _f32p, _f32p]),
    "bamm_scan_destroy": (None, [_vp]),
}

# struct bamm_hit of include/bamm_b200.h
HIT_DTYPE = np.dtype([("seq", np.uint64), ("window", np.uint64), ("score", np.float32), ("p_value", np.float32),
                      ("e_value", np.float32), ("reserved", np.uint32)])

_lib = None


class BammError(RuntimeError):
    pass


def load():
    """Loads libbamm_b200.so and declares every prototype. Raises if the library has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise BammError("libbamm_b200.so is missing: run `python -m bammmotif2_b200.build` (there is no CPU fallback)")
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


def _check(rc):
    if rc != 0:
        raise BammError("bamm error %d: %s" % (rc, load().bamm_last_error().decode()))


def _ptr(a, ptype):
    return a.ctypes.data_as(ptype) if a is not None else None


def model_size(A, K, W):
    return sum(A ** (k + 1) * W for k in range(K + 1))


def bg_size(A, K):
    return sum(A ** (k + 1) for k in range(K + 1))


def bound_plan_describe(W, K, K_bg, budget=232448):
    """Bound plan of the pruned E-step as a dict (host arithmetic, no device): G, kd, fast, table_bytes, groups[...]; None without a plan."""
    buf = (C.c_int32 * 256)()
    n = C.c_uint64(0)
    _check(load().bamm_bound_plan_describe(W, K, K_bg, budget, buf, 256, C.byref(n)))
    if buf[0] == 0:
        return None
    G = buf[0]
    names = ("col0", "ncol", "lo", "shift", "shift2", "mask4", "base")
    groups = [dict(zip(names, [int(buf[4 + 7 * g + i]) & 0xffffffff if names[i] == "mask4" else int(buf[4 + 7 * g + i]) for i in range(7)])) for g in range(G)]
    return dict(G=G, kd=int(buf[1]), fast=bool(buf[2]), table_bytes=int(buf[3]), groups=groups)


def set_device_group(devices):
    """Devices one process drives together (bamm_set_device_group); [] or one device switches the group off."""
    arr = (C.c_int * max(len(devices), 1))(*devices)
    _check(load().bamm_set_device_group(arr, len(devices)))


def device_count():
    n = C.c_int(0)
    rc = load().bamm_device_count(C.byref(n))
    return n.value if rc == 0 else 0


def plan_describe(W, K, K_bg=0, reduced=True, budget=227 * 1024):
    """Column-group plan of the packed E-step as a list of passes (host arithmetic only, works without a GPU):
    [{G, kd, fast, table_bytes, ca, cb, first, last, groups: [{col0, ncol, lo, shift, shift2, mask4, base, colmask}]}];
    [] when no packed plan fits the budget."""
    out = np.zeros(1 + 32 * (8 + 8 * 16), np.int32)
    used = C.c_uint64(0)
    _check(load().bamm_plan_describe(int(W), int(K), int(K_bg), 1 if reduced else 0, int(budget),
                                     out.ctypes.data_as(C.POINTER(C.c_int32)), len(out), C.byref(used)))
    o = out[:used.value].astype(np.int64)
    passes, i = [], 1
    for _ in range(int(o[0])):
        G, kd, fast, tb, ca, cb, first, last = (int(x) for x in o[i:i + 8])
        i += 8
        groups = []
        for _g in range(G):
            c0, nc, lo, sh, sh2, m4, base, cm = (int(x) for x in o[i:i + 8])
            i += 8
            groups.append(dict(col0=c0, ncol=nc, lo=lo, shift=sh, shift2=sh2, mask4=m4 & 0xffffffff, base=base, colmask=cm & 0xffffffff))
        passes.append(dict(G=G, kd=kd, fast=bool(fast), table_bytes=tb, ca=ca, cb=cb, first=bool(first), last=bool(last), groups=groups))
    return passes


def rand_stream(seed, first, count):
    """rand() draws [first, first+count) after srand(seed), re-created on the device (glibc TYPE_3 generator)."""
    out = np.zeros(int(count), np.int32)
    _check(load().bamm_rand_stream(int(seed), int(first), int(count), out.ctypes.data_as(C.POINTER(C.c_int32))))
    return out


def sort_scores(scores, descending=False):
    a = np.ascontiguousarray(scores, np.float32).copy()
    _check(load().bamm_sort_scores(_ptr(a, _f32p), len(a), 1 if descending else 0))
    return a


def mops_pvalues(neg_scores, pos_scores, n_pos_sequences):
    neg = np.ascontiguousarray(neg_scores, np.float32)
    pos = np.ascontiguousarray(pos_scores, np.float32)
    p, e = np.empty(len(pos), np.float32), np.empty(len(pos), np.float32)
    _check(load().bamm_mops_pvalues(_ptr(neg, _f32p), len(neg), _ptr(pos, _f32p), len(pos), int(n_pos_sequences), _ptr(p, _f32p), _ptr(e, _f32p)))
    return p, e


def score_last_ms():
    t = C.c_float(0)
    _check(load().bamm_score_last_timing(C.byref(t)))
    return float(t.value)


def kmer_patches(codes, kmer):
    """Positions whose hash depends on rand() draws for a code-0 base (Sequence.cpp:38): every position within
    10 after a 0 code (k-mer hashes span 11 bases) — of the same sequence or not does not matter, a superset is
    fine because the patch carries the reference's own hash. Returns (positions, kmer values)."""
    zero = np.flatnonzero(codes == 0)
    if len(zero) == 0:
        return np.zeros(0, np.uint64), np.zeros(0, np.uint64)
    pos = (zero[:, None] + np.arange(11)[None, :]).ravel()
    pos = np.unique(pos[pos < len(codes)]).astype(np.uint64)
    return pos, np.ascontiguousarray(kmer[pos.astype(np.int64)], np.uint64)


class SeqSet:
    """Device-resident sequence set (bamm_seqset)."""

    def __init__(self, codes, offsets, A, patch_pos=None, patch_kmer=None):
        lib = load()
        self.codes = np.ascontiguousarray(codes, np.uint8)
        self.offsets = np.ascontiguousarray(offsets, np.uint64)
        self.A = int(A)
        pp = np.ascontiguousarray(patch_pos if patch_pos is not None else np.zeros(0), np.uint64)
        pk = np.ascontiguousarray(patch_kmer if patch_kmer is not None else np.zeros(0), np.uint64)
        h = _vp()
        _check(lib.bamm_seqset_create(_ptr(self.codes, _u8p), _ptr(self.offsets, _u64p), len(self.offsets) - 1, self.A,
                                      _ptr(pp, _u64p), _ptr(pk, _u64p), len(pp), C.byref(h)))
        self.h = h
        self.nseq = len(self.offsets) - 1
        self.npos = int(self.offsets[-1])

    @classmethod
    def _adopt(cls, h, A):
        """Wraps a set created by the library on the device (bamm_seqset_sample_negatives)."""
        self = cls.__new__(cls)
        self.h = h
        self.A = int(A)
        nseq, npos, a = C.c_uint64(0), C.c_uint64(0), C.c_int(0)
        _check(load().bamm_seqset_info(h, C.byref(nseq), C.byref(npos), C.byref(a)))
        self.nseq, self.npos = int(nseq.value), int(npos.value)
        self.offsets = np.zeros(self.nseq + 1, np.uint64)
        _check(load().bamm_seqset_get_offsets(h, _ptr(self.offsets, _u64p)))
        self.codes = None
        return self

    def sample_negatives(self, fold, seed=42, subset=None):
        """Device-side SeqGenerator::sample_bgseqset_by_fold (bit-identical to the reference's libc rand() stream);
        subset: template sequences (indices into this set, in sampling order), default all."""
        h = _vp()
        sub = np.ascontiguousarray(subset, np.uint64) if subset is not None else None
        _check(load().bamm_seqset_sample_negatives(self.h, _ptr(sub, _u64p), len(sub) if sub is not None else 0, int(fold), int(seed), C.byref(h)))
        return SeqSet._adopt(h, self.A)

    def negative_kmer_counts(self):
        """This shard's k-mer counters for the set-wide model of the negative sampler (orders 0..2 concatenated)."""
        out = np.zeros(self.A + self.A ** 2 + self.A ** 3, np.uint64)
        _check(load().bamm_seqset_negative_kmer_counts(self.h, None, 0, _ptr(out, _u64p)))
        return out

    def sample_negatives_shard(self, fold, draw_offset, global_counts, seed=42):
        """One shard of a negative set sampled over several devices (see include/bamm_b200.h)."""
        h = _vp()
        gc = np.ascontiguousarray(global_counts, np.uint64)
        _check(load().bamm_seqset_sample_negatives_shard(self.h, None, 0, int(fold), int(seed), int(draw_offset), _ptr(gc, _u64p), C.byref(h)))
        return SeqSet._adopt(h, self.A)

    def get_codes(self):
        out = np.zeros(self.npos, np.uint8)
        _check(load().bamm_seqset_get_codes(self.h, _ptr(out, _u8p)))
        return out

    def index(self, K):
        _check(load().bamm_seqset_index(self.h, K))

    def get_index(self, K):
        out = np.zeros(self.npos, np.uint32)
        _check(load().bamm_seqset_get_index(self.h, K, _ptr(out, _u32p)))
        return out

    def count_kmers(self, K):
        out = np.zeros(bg_size(self.A, K), np.uint64)
        _check(load().bamm_seqset_count_kmers(self.h, K, _ptr(out, _u64p)))
        return out

    def score(self, W, K, K_bg_model, v_all, vbg_all, subset=None, want_mops=True, out=None):
        """ScoreSeqSet::calcLogOdds. Returns (mops|None, zoops, z). out: optional (zoops float32[nsub], z uint64[nsub]) buffers
        to fill (e.g. pinned host memory) instead of fresh arrays."""
        sub = np.ascontiguousarray(subset, np.uint64) if subset is not None else None
        nsub = len(sub) if sub is not None else self.nseq
        if out is not None:
            zoops, z = out
            assert zoops.dtype == np.float32 and z.dtype == np.uint64 and len(zoops) == nsub and len(z) == nsub
        else:
            zoops = np.empty(nsub, np.float32)
            z = np.empty(nsub, np.uint64)
        mops = None
        if want_mops:
            ids = sub.astype(np.int64) if sub is not None else np.arange(self.nseq)
            L = (self.offsets[1:] - self.offsets[:-1]).astype(np.int64)[ids]
            mops = np.zeros(int((L - W + 1).sum()), np.float32)
        v = np.ascontiguousarray(v_all, np.float32)
        vb = np.ascontiguousarray(vbg_all, np.float32)
        _check(load().bamm_score_logodds(self.h, _ptr(sub, _u64p), nsub, W, K, K_bg_model, _ptr(v, _f32p), _ptr(vb, _f32p),
                                         _ptr(zoops, _f32p), _ptr(z, _u64p), _ptr(mops, _f32p)))
        return mops, zoops, z

    def close(self):
        if self.h:
            load().bamm_seqset_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class EM:
    """One EM problem on the device (bamm_em); mirrors the reference's EM class (src/refinement/EM.h:18-36)."""

    def __init__(self, seqset, W, K, K_bg_model, subset=None):
        self.seqset = seqset
        self.W, self.K, self.K_bg_model, self.A = W, K, K_bg_model, seqset.A
        sub = np.ascontiguousarray(subset, np.uint64) if subset is not None else None
        self.nsub = len(sub) if sub is not None else seqset.nseq
        h = _vp()
        _check(load().bamm_em_create(seqset.h, _ptr(sub, _u64p), self.nsub, W, K, K_bg_model, C.byref(h)))
        self.h = h
        self.msize = model_size(self.A, K, W)

    def set_model(self, v_all, vbg_all, alpha, q):
        v = np.ascontiguousarray(v_all, np.float32)
        vb = np.ascontiguousarray(vbg_all, np.float32)
        al = np.ascontiguousarray(alpha, np.float32).ravel()
        assert len(v) == self.msize and len(vb) == bg_size(self.A, self.K_bg_model) and len(al) == (self.K + 1) * self.W
        _check(load().bamm_em_set_model(self.h, _ptr(v, _f32p), _ptr(vb, _f32p), _ptr(al, _f32p), C.c_float(q)))

    def estep(self):
        llh = C.c_float(0)
        _check(load().bamm_em_estep(self.h, C.byref(llh)))
        return llh.value

    def mstep(self):
        _check(load().bamm_em_mstep(self.h))

    def optimize_q(self):
        q = C.c_float(0)
        _check(load().bamm_em_optimize_q(self.h, C.byref(q)))
        return q.value

    def optimize(self, optimize_q=False, epsilon=0.01, max_iter=1000):
        it = C.c_int(0)
        llh = np.zeros(max_iter, np.float32)
        vd = np.zeros(max_iter, np.float32)
        qt = np.zeros(max_iter, np.float32)
        _check(load().bamm_em_optimize(self.h, int(optimize_q), C.c_float(epsilon), max_iter, C.byref(it),
                                       _ptr(llh, _f32p), _ptr(vd, _f32p), _ptr(qt, _f32p)))
        n = it.value
        return dict(iterations=n, llh=llh[:n], vdiff=vd[:n], qtrace=qt[:n], v=self.model(), q=self.q())

    def mask(self, f=0.05, epsilon=0.01, max_iter=1000):
        """EM::mask (--advanceEM). Returns dict(iterations, llh, nkept, cutoff, v)."""
        it, llh, nk, cut = C.c_int(0), C.c_float(0), C.c_uint64(0), C.c_float(0)
        _check(load().bamm_em_mask(self.h, f, epsilon, max_iter, C.byref(it), C.byref(llh), C.byref(nk), C.byref(cut)))
        return dict(iterations=it.value, llh=llh.value, nkept=nk.value, cutoff=cut.value, v=self.model())

    def iterate(self, n_iter):
        llh, vd = C.c_float(0), C.c_float(0)
        _check(load().bamm_em_iterate(self.h, n_iter, C.byref(llh), C.byref(vd)))
        return llh.value, vd.value

    def model(self):
        out = np.zeros(self.msize, np.float32)
        _check(load().bamm_em_get_model(self.h, _ptr(out, _f32p)))
        return out

    def counts(self):
        out = np.zeros(self.msize, np.float32)
        _check(load().bamm_em_get_counts(self.h, _ptr(out, _f32p)))
        return out

    def s(self):
        out = np.zeros(self.A ** (self.K + 1) * self.W, np.float32)
        _check(load().bamm_em_get_s(self.h, _ptr(out, _f32p)))
        return out

    def q(self):
        q = C.c_float(0)
        _check(load().bamm_em_get_q(self.h, C.byref(q)))
        return q.value

    def r(self, first=0, count=None):
        count = self.nsub - first if count is None else count
        total = int(load().bamm_em_r_size(self.h))
        out = np.zeros(total, np.float32)
        _check(load().bamm_em_get_r(self.h, first, count, _ptr(out, _f32p)))
        return out

    def timing(self):
        e, m = C.c_float(0), C.c_float(0)
        _check(load().bamm_em_last_timing(self.h, C.byref(e), C.byref(m)))
        return e.value, m.value

    def loop_timing(self):
        """(iterations, estep_ms, maccum_ms, update_ms, total_ms) of the last iterate() call, CUDA events on the EM stream."""
        it = C.c_int(0)
        e, m, up, t = C.c_float(0), C.c_float(0), C.c_float(0), C.c_float(0)
        _check(load().bamm_em_loop_timing(self.h, C.byref(it), C.byref(e), C.byref(m), C.byref(up), C.byref(t)))
        return it.value, e.value, m.value, up.value, t.value

    def loop_timing_estep(self):
        """(masked_ms, bound_ms, exact_ms): the E-step share of loop_timing() by kernel of the pruned path."""
        a, b, c = C.c_float(0), C.c_float(0), C.c_float(0)
        _check(load().bamm_em_loop_timing_estep(self.h, C.byref(a), C.byref(b), C.byref(c)))
        return a.value, b.value, c.value

    def launch_count(self):
        n = C.c_uint64(0)
        _check(load().bamm_em_launch_count(self.h, C.byref(n)))
        return n.value

    def estep_info(self):
        """How the last E-step ran (bamm_em_estep_info): dict(pruned, G, G_bound, dense_ran, candidates, active, passes, plain_smem)."""
        a = (C.c_uint64 * 8)()
        _check(load().bamm_em_estep_info(self.h, a))
        return dict(pruned=bool(a[0]), G=int(a[1]), G_bound=int(a[2]), dense_ran=bool(a[3]), candidates=int(a[4]), active=int(a[5]),
                    passes=int(a[6]), plain_smem=bool(a[7]))

    def bound_reuse_info(self):
        """Bound reuse of the pruned E-step (bamm_em_bound_reuse_info): dict(enabled, full, watch, watched, last_watch, valid, log2_drift)."""
        a = (C.c_uint64 * 6)()
        d = C.c_float(0.0)
        _check(load().bamm_em_bound_reuse_info(self.h, a, C.byref(d)))
        return dict(enabled=bool(a[0]), full=int(a[1]), watch=int(a[2]), watched=int(a[3]), last_watch=bool(a[4]), valid=bool(a[5]),
                    log2_drift=float(d.value))

    def set_exchange_buffer(self, dev_ptr, words):
        _check(load().bamm_em_set_exchange_buffer(self.h, _vp(dev_ptr), words))

    # multi-GPU halves
    def exchange_buffer(self):
        p, w = _vp(), C.c_uint64(0)
        _check(load().bamm_em_exchange_buffer(self.h, C.byref(p), C.byref(w)))
        return p.value, w.value

    def stream(self):
        p = _vp()
        _check(load().bamm_em_stream(self.h, C.byref(p)))
        return p.value

    def peer_alloc(self, rank, world):
        """Allocates this rank's NVLink receive buffer; returns its 64-byte CUDA IPC handle."""
        buf = C.create_string_buffer(64)
        _check(load().bamm_em_peer_alloc(self.h, rank, world, C.cast(buf, _vp)))
        return buf.raw

    def peer_wait(self, reset=True):
        """(total_ms, waits): device time spent waiting for the slowest rank in the peer exchange since the last reset."""
        ms, n = C.c_double(0), C.c_uint64(0)
        _check(load().bamm_em_peer_wait(self.h, int(reset), C.byref(ms), C.byref(n)))
        return ms.value, n.value

    def peer_attach(self, handles):
        """handles: world x 64 bytes (rank order). Afterwards mstep_local pushes to every rank over NVLink."""
        buf = C.create_string_buffer(bytes(handles), len(handles))
        _check(load().bamm_em_peer_attach(self.h, C.cast(buf, _vp)))

    def set_global_nseq(self, n):
        _check(load().bamm_em_set_global_nseq(self.h, n))

    def estep_local(self):
        _check(load().bamm_em_estep_local(self.h))

    def mstep_local(self):
        _check(load().bamm_em_mstep_local(self.h))

    def finish_iteration(self, optimize_q=False, sync=True):
        if not sync and not optimize_q:
            _check(load().bamm_em_finish_iteration(self.h, 0, None, None))
            return None
        llh, vd = C.c_float(0), C.c_float(0)
        _check(load().bamm_em_finish_iteration(self.h, int(optimize_q), C.byref(llh), C.byref(vd)))
        return llh.value, vd.value

    def close(self):
        if self.h:
            load().bamm_em_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Scan:
    """Occurrence scan of one motif (bamm_scan): the negative windows of `negset[subset]` are scored and sorted on the device
    once; hits() then returns the windows of a positive set whose p-value is < p_cutoff."""

    def __init__(self, negset, W, K, K_bg_model, v_all, vbg_all, subset=None):
        sub = np.ascontiguousarray(subset, np.uint64) if subset is not None else None
        v = np.ascontiguousarray(v_all, np.float32)
        vb = np.ascontiguousarray(vbg_all, np.float32)
        h = _vp()
        _check(load().bamm_scan_create(negset.h if negset is not None else None, _ptr(sub, _u64p), len(sub) if sub is not None else 0,
                                       W, K, K_bg_model, _ptr(v, _f32p), _ptr(vb, _f32p), C.byref(h)))
        self.h = h

    def hits_page(self, posset, p_cutoff, n_pos_sequences, cursor=0, cap=1 << 20, subset=None):
        """One bamm_scan_hits call: (structured array of HIT_DTYPE, next cursor)."""
        sub = np.ascontiguousarray(subset, np.uint64) if subset is not None else None
        out = np.zeros(int(cap), HIT_DTYPE)
        cur, n = C.c_uint64(int(cursor)), C.c_uint64(0)
        _check(load().bamm_scan_hits(self.h, posset.h, _ptr(sub, _u64p), len(sub) if sub is not None else 0, int(n_pos_sequences),
                                     C.c_float(p_cutoff), C.byref(cur), out.ctypes.data_as(_vp), int(cap), C.byref(n)))
        return out[:n.value], cur.value

    def hits(self, posset, p_cutoff, n_pos_sequences=None, subset=None, cap=1 << 20):
        """Every hit of posset[subset] (default: all sequences), fetched in pages of `cap`: a page with fewer than `cap` hits
        is the last one. n_pos_sequences defaults to the number of scanned sequences."""
        n_pos = (len(subset) if subset is not None else posset.nseq) if n_pos_sequences is None else n_pos_sequences
        pages, cursor = [], 0
        while True:
            page, cursor = self.hits_page(posset, p_cutoff, n_pos, cursor, cap, subset)
            pages.append(page)
            if len(page) < cap:
                return np.concatenate(pages)

    def info(self):
        """dict(negative_windows, neg_score_ms, sort_ms, hits_ms): see bamm_scan_info."""
        n = C.c_uint64(0)
        a, b, c = C.c_float(0), C.c_float(0), C.c_float(0)
        _check(load().bamm_scan_info(self.h, C.byref(n), C.byref(a), C.byref(b), C.byref(c)))
        return dict(negative_windows=int(n.value), neg_score_ms=a.value, sort_ms=b.value, hits_ms=c.value)

    def close(self):
        if self.h:
            load().bamm_scan_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
