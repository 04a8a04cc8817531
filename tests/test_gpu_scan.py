"""Occurrence scan (-m gpu): bamm_scan_create / bamm_scan_hits (BaMMScan) against the existing route of `--scoreSeqset`,
bamm_score_logodds(mops) + bamm_mops_pvalues + the p < cutoff filter of ScoreSeqSet::write, compared bit for bit: the same
windows in the same order (subset order, then window ascending) with the same score, p and e.
"""
import os
import subprocess

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "bammmotif2_b200", "bin")


@pytest.fixture(scope="module")
def capi():
    from bammmotif2_b200 import capi
    capi.load()
    assert capi.device_count() >= 1, "no CUDA device: the product has no CPU fallback"
    return capi


def make_set(capi, oracle, A, W, seed, nseq, single_strand=False, Lmax=90, with_n=True):
    """Seeded ragged set encoded the reference's way; one record has stored length W (a single window)."""
    rng = np.random.default_rng(seed)
    enc = []
    for n in range(nseq):
        L = W if n == 7 else int(rng.integers(max(W, 20), max(W, 20) + Lmax))
        L0 = L if single_strand else max((L - 1) // 2, (W + 1) // 2)
        s = rng.integers(1, A + 1, size=L0, dtype=np.uint8)
        if with_n and n % 11 == 3:
            s[L0 // 3] = 0
        enc.append(s)
    oracle.srand(seed)
    codes, kmer, offsets = oracle.encode_sequences(enc, "EXTENDED" if A == 6 else "STANDARD", single_strand)
    pp, pk = capi.kmer_patches(codes, kmer)
    return capi.SeqSet(codes, offsets, A, pp, pk), kmer


def random_model(oracle, kmer, A, K, Kbg, W, seed):
    from bammmotif2_b200 import hostmodel
    _, vbg = oracle.bg_model(kmer, A, Kbg, hostmodel.default_bg_alpha(Kbg))
    alpha = hostmodel.default_motif_alpha(K, W)
    sites = np.random.default_rng(seed + 1).integers(1, A + 1, size=(200, W), dtype=np.uint8)
    return hostmodel.motif_from_sites(sites, A, K, alpha, vbg), vbg


def reference_hits(capi, pos, neg, W, K, Kbg, v, vbg, cutoff, subset=None, neg_subset=None, n_pos=None):
    """bamm_score_logodds(mops) on both sets, bamm_mops_pvalues, p < cutoff: (seq, window, score, p, e) in file order."""
    nmops, _, _ = neg.score(W, K, Kbg, v, vbg, subset=neg_subset)
    pmops, _, _ = pos.score(W, K, Kbg, v, vbg, subset=subset)
    ids = np.asarray(subset, np.int64) if subset is not None else np.arange(pos.nseq)
    n_pos = len(ids) if n_pos is None else n_pos
    p, e = capi.mops_pvalues(nmops, pmops, n_pos)
    LW1 = (pos.offsets[1:] - pos.offsets[:-1]).astype(np.int64)[ids] - W + 1
    seq = np.repeat(np.arange(len(ids)), LW1)
    window = np.arange(len(pmops)) - np.repeat(np.concatenate([[0], np.cumsum(LW1)[:-1]]), LW1)
    keep = p < np.float32(cutoff)
    return dict(seq=seq[keep], window=window[keep], score=pmops[keep], p=p[keep], e=e[keep]), nmops, pmops, p


def assert_same_hits(hits, ref):
    assert len(hits) == len(ref["seq"]), (len(hits), len(ref["seq"]))
    assert np.array_equal(hits["seq"].astype(np.int64), ref["seq"])
    assert np.array_equal(hits["window"].astype(np.int64), ref["window"])
    for f, g in (("score", "score"), ("p_value", "p"), ("e_value", "e")):
        assert np.array_equal(hits[f].view(np.uint32), np.asarray(ref[g], np.float32).view(np.uint32)), f
    assert not hits["reserved"].any()


SHAPES = [  # A, K, W, single strand, N bases
    (4, 2, 12, False, True),
    (4, 4, 20, False, True),
    (4, 2, 33, False, True),
    (4, 1, 63, True, False),
    (6, 5, 10, False, True),        # A^(K+1) W = 466560 floats: the table stays in L2
    (4, 8, 12, True, True),         # A^(K+1) = 262144: 32-bit k-mer indices
]


@pytest.mark.parametrize("A,K,W,single,with_n", SHAPES)
def test_hits_equal_the_existing_path(capi, oracle, A, K, W, single, with_n):
    Kbg = min(K, 2)
    pos, kmer = make_set(capi, oracle, A, W, 100 + W, 400, single, with_n=with_n)
    neg, _ = make_set(capi, oracle, A, W, 200 + W, 900, single, with_n=with_n)
    v, vbg = random_model(oracle, kmer, A, K, Kbg, W, 7)
    sc = capi.Scan(neg, W, K, Kbg, v, vbg)
    for cutoff in (0.01, 0.2):
        ref, _, _, _ = reference_hits(capi, pos, neg, W, K, Kbg, v, vbg, cutoff)
        assert len(ref["seq"]) > 0
        assert_same_hits(sc.hits(pos, cutoff), ref)
    # subsets out of order, on both sides; the one-window record (index 7) included
    rng = np.random.default_rng(W)
    sub = rng.permutation(pos.nseq)[:250]
    sub = np.concatenate([[7], sub[sub != 7]])
    nsub = rng.permutation(neg.nseq)[:600]
    sc2 = capi.Scan(neg, W, K, Kbg, v, vbg, subset=nsub)
    ref, _, _, _ = reference_hits(capi, pos, neg, W, K, Kbg, v, vbg, 0.05, subset=sub, neg_subset=nsub, n_pos=1234)
    assert_same_hits(sc2.hits(pos, 0.05, n_pos_sequences=1234, subset=sub), ref)


def test_cutoffs_and_paging(capi, oracle):
    A, K, Kbg, W = 4, 2, 2, 12
    pos, kmer = make_set(capi, oracle, A, W, 11, 300)
    neg, _ = make_set(capi, oracle, A, W, 12, 700)
    v, vbg = random_model(oracle, kmer, A, K, Kbg, W, 3)
    sc = capi.Scan(neg, W, K, Kbg, v, vbg)
    roff = np.concatenate([[0], np.cumsum((pos.offsets[1:] - pos.offsets[:-1]).astype(np.int64) - W + 1)])
    total = int(roff[-1])
    assert len(sc.hits(pos, 0.0)) == 0
    _, _, _, p = reference_hits(capi, pos, neg, W, K, Kbg, v, vbg, 0.0)
    # a cutoff equal to a window's p: that window is not a hit (strict <)
    c = np.float32(np.sort(p)[len(p) // 3])
    ref, _, _, _ = reference_hits(capi, pos, neg, W, K, Kbg, v, vbg, c)
    got = sc.hits(pos, float(c))
    assert_same_hits(got, ref)
    assert not (got["p_value"] == c).any() and (p == c).any()
    # every window (p <= 1 unless the interpolation overshoots), fetched in pages through the cursor
    for cutoff in (1.0, 2.0):
        ref, _, _, _ = reference_hits(capi, pos, neg, W, K, Kbg, v, vbg, cutoff)
        whole = sc.hits(pos, cutoff)
        assert_same_hits(whole, ref)
        paged = sc.hits(pos, cutoff, cap=997)
        assert_same_hits(paged, ref)
        page, cur = sc.hits_page(pos, cutoff, pos.nseq, cursor=0, cap=10)
        assert len(page) == 10 and cur == roff[ref["seq"][9]] + ref["window"][9] + 1
        rest, end = sc.hits_page(pos, cutoff, pos.nseq, cursor=cur, cap=10 ** 6)
        assert_same_hits(np.concatenate([page, rest]), ref)
        assert end == total
    page, cur = sc.hits_page(pos, 2.0, pos.nseq, cursor=total, cap=10)
    assert len(page) == 0 and cur == total
    page, cur = sc.hits_page(pos, 2.0, pos.nseq, cursor=5, cap=0)
    assert len(page) == 0 and cur == 5


def test_near_ties_in_the_interpolation_branch(capi, oracle):
    """One-column motif whose four scores sit 1.1e-5 and 0.9e-5 apart: the negatives hold many ties, positives tie with
    negatives, and for a tie below a gap just above eps = 1e-5 the interpolation gives p far below FPl / negN."""
    A, K, Kbg, W = 4, 0, 0, 1
    pos, kmer = make_set(capi, oracle, A, W, 21, 300, with_n=False)
    neg, _ = make_set(capi, oracle, A, W, 22, 800, with_n=False)
    vbg = np.full(4, 0.25, np.float32)
    target = np.array([0.0, 1.1e-5, 2.0e-5, 3.0], np.float64)
    v = (0.25 * np.exp(target) - 1e-5).astype(np.float32)
    sc = capi.Scan(neg, W, K, Kbg, v, vbg)
    ref, nmops, pmops, p = reference_hits(capi, pos, neg, W, K, Kbg, v, vbg, 2.0)
    vals = np.unique(nmops)
    assert len(vals) == 4
    gaps = np.diff(vals)[:2]
    assert 1e-5 < gaps[0] < 1.2e-5 and 0.8e-5 < gaps[1] < 1e-5, gaps
    negs = np.sort(nmops)
    FPl = len(negs) - np.searchsorted(negs, pmops, side="right")
    assert (p < (FPl - 5.0) / len(negs)).any()                 # the reversed-naming quirk, reproduced
    assert_same_hits(sc.hits(pos, 2.0), ref)
    for cutoff in np.unique(p)[:3]:                             # cutoffs on the tied p-values themselves
        r, _, _, _ = reference_hits(capi, pos, neg, W, K, Kbg, v, vbg, cutoff)
        assert_same_hits(sc.hits(pos, float(cutoff)), r)


def test_long_record_among_short_ones(capi, oracle):
    """A single-strand record of 7e7 bases (beyond 2^26) between short ones: the hits equal the reference computation, and a
    slice of window scores equals k_score's MOPS output (one warp per record)."""
    A, K, Kbg, W = 4, 2, 2, 16
    rng = np.random.default_rng(5)
    lens = [40, 7 * 10 ** 7, 17, 300, 16]
    codes = rng.integers(1, 5, size=sum(lens), dtype=np.uint8)
    offsets = np.concatenate([[0], np.cumsum(lens)]).astype(np.uint64)
    pos = capi.SeqSet(codes, offsets, A)
    nlens = rng.integers(16, 400, size=20000)
    neg = capi.SeqSet(rng.integers(1, 5, size=int(nlens.sum()), dtype=np.uint8),
                      np.concatenate([[0], np.cumsum(nlens)]).astype(np.uint64), A)
    vbg = np.concatenate([np.full(4 ** (k + 1), 0.25, np.float32) for k in range(Kbg + 1)])
    from bammmotif2_b200 import hostmodel
    sites = np.random.default_rng(9).integers(1, 5, size=(200, W), dtype=np.uint8)
    v = hostmodel.motif_from_sites(sites, A, K, hostmodel.default_motif_alpha(K, W), vbg)
    sc = capi.Scan(neg, W, K, Kbg, v, vbg)
    os.environ["BAMM_NO_PACKED"] = "1"                          # the reference scores through k_score
    try:
        ref, _, pmops, _ = reference_hits(capi, pos, neg, W, K, Kbg, v, vbg, 1e-3)
    finally:
        del os.environ["BAMM_NO_PACKED"]
    assert len(ref["seq"]) > 1000 and (ref["seq"] == 1).any()
    assert_same_hits(sc.hits(pos, 1e-3), ref)
    first = 40 - W + 1 + 6 * 10 ** 7                             # windows of record 1 from 6e7 on (beyond 2^26)
    page, cur = sc.hits_page(pos, float("inf"), 5, cursor=first, cap=200000)
    assert len(page) == 200000 and cur == first + 200000
    assert (page["seq"] == 1).all() and np.array_equal(page["window"].astype(np.int64), np.arange(6 * 10 ** 7, 6 * 10 ** 7 + 200000))
    assert np.array_equal(page["score"].view(np.uint32), pmops[first:first + 200000].view(np.uint32))


def test_errors(capi, oracle):
    from bammmotif2_b200.capi import BammError
    A, K, Kbg, W = 4, 2, 2, 12
    pos, kmer = make_set(capi, oracle, A, W, 31, 50)
    v, vbg = random_model(oracle, kmer, A, K, Kbg, W, 3)
    for w in (0, 64):
        with pytest.raises(BammError, match="motif width"):
            capi.Scan(pos, w, K, Kbg, np.zeros(len(v) // W * max(w, 1), np.float32), vbg)
    for k in (-1, 11):
        with pytest.raises(BammError, match="order K"):
            capi.Scan(pos, W, k, Kbg, v, vbg)
    with pytest.raises(BammError, match="empty negative set"):
        capi.Scan(pos, W, K, Kbg, v, vbg, subset=np.zeros(0, np.uint64))
    with pytest.raises(BammError, match="subset index out of range"):
        capi.Scan(pos, W, K, Kbg, v, vbg, subset=[0, pos.nseq])
    with pytest.raises(BammError, match="shorter than the motif"):
        capi.Scan(pos, 40, K, Kbg, np.resize(v, len(v) // W * 40), vbg)
    with pytest.raises(BammError, match="NULL"):
        capi.Scan(None, W, K, Kbg, v, vbg)
    sc = capi.Scan(pos, W, K, Kbg, v, vbg)
    with pytest.raises(BammError, match="subset index out of range"):
        sc.hits(pos, 0.1, subset=[3, pos.nseq + 2])
    short = capi.SeqSet(np.ones(30, np.uint8), np.array([0, 20, 30], np.uint64), A)
    with pytest.raises(BammError, match="shorter than the motif"):
        sc.hits(short, 0.1)
    with pytest.raises(BammError, match="cursor"):
        sc.hits_page(pos, 0.1, pos.nseq, cursor=10 ** 12)
    other, _ = make_set(capi, oracle, 6, W, 32, 20)
    with pytest.raises(BammError, match="alphabet"):
        sc.hits(other, 0.1)
    import ctypes as C
    lib = capi.load()
    n = C.c_uint64(0)
    assert lib.bamm_scan_hits(sc.h, pos.h, None, 0, 1, C.c_float(0.1), None, None, 0, C.byref(n)) == -1
    assert lib.bamm_scan_hits(None, pos.h, None, 0, 1, C.c_float(0.1), C.byref(C.c_uint64(0)), None, 0, C.byref(n)) == -1
    assert lib.bamm_scan_hits(sc.h, pos.h, None, 0, 1, C.c_float(0.1), C.byref(C.c_uint64(0)), None, 5, C.byref(n)) == -1
    assert lib.bamm_scan_create(pos.h, None, 0, W, K, Kbg, None, None, C.byref(C.c_void_p())) == -1
    assert lib.bamm_scan_info(None, None, None, None, None) == -1
    info = sc.info()
    assert info["negative_windows"] == int(((pos.offsets[1:] - pos.offsets[:-1]).astype(np.int64) - W + 1).sum())


# ----------------------------------------------------------------------------------------------- CLI
def run(cmd):
    p = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)
    assert p.returncode == 0, "%s\n%s\n%s" % (" ".join(cmd), p.stdout[-2000:], p.stderr[-2000:])
    return p


@pytest.fixture(scope="module")
def bins():
    from bammmotif2_b200 import build
    build.build_all()
    return BIN


def compare_runs(bins, tmp_path, fa, model_args, motifs, name):
    extra = ["--pvalCutoff", "0.01", "--saveLogOdds"]
    run([os.path.join(bins, "BaMMmotif"), str(tmp_path / "motif"), fa] + model_args + ["--scoreSeqset"] + extra)
    run([os.path.join(bins, "BaMMScan"), str(tmp_path / "scan"), fa] + model_args + extra)
    files = ["%s_motif_%d.occurrence" % (name, m) for m in motifs] + ["%s_motif_%d.logOddsZoops" % (name, m) for m in motifs]
    files.append(name + ".negSet.logOddsZoops")
    for f in files:
        a, b = open(tmp_path / "motif" / f, "rb").read(), open(tmp_path / "scan" / f, "rb").read()
        assert a == b, f
    assert open(tmp_path / "scan" / files[0]).read().count("\n") > 10


def test_cli_bamm_file_equals_score_seqset(bins, tmp_path):
    from bammmotif2_b200 import synth
    fwd, sites, _ = synth.planted_sequences(77, 1500, 150, 12)
    fwd = fwd.copy()
    fwd[::89, 30] = 0
    fa, bs = str(tmp_path / "syn.fasta"), str(tmp_path / "sites.block")
    synth.write_fasta(fa, fwd)
    synth.write_sites(bs, sites)
    run([os.path.join(bins, "BaMMmotif"), str(tmp_path / "train"), fa, "--bindingSiteFile", bs, "--EM", "-k", "3", "-K", "2"])
    model = ["--BaMMFile", str(tmp_path / "train" / "syn_motif_1.ihbcp"), "--bgModelFile", str(tmp_path / "train" / "syn.hbcp"),
             "-k", "3", "-K", "2"]
    compare_runs(bins, tmp_path, fa, model, [1], "syn")


def test_cli_two_pwms_equal_score_seqset(bins, tmp_path):
    from util import Golden
    fa = tmp_path / "JunD.fasta"
    open(fa, "wb").write(bytes(Golden("jund_k2")["fasta_text"]))
    meme = tmp_path / "pwm.meme"
    open(meme, "wb").write(bytes(Golden("jund_pwm_k1")["sites_text"]))
    compare_runs(bins, tmp_path, str(fa), ["--PWMFile", str(meme), "--maxPWM", "2", "-k", "1", "-K", "1"], [1, 2], "JunD")
