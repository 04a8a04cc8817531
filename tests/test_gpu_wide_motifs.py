"""Motifs wider than 32 columns (-m gpu): the index-array kernels walk the columns in blocks of 32 (DESIGN.md §4.6) up to
BAMM_MAX_MOTIF_WIDTH = 63; the packed 2-bit kernels keep W <= 32. Everything is compared with the CPU oracle, which has no
width limit, on seeded sequences encoded the reference's way (both strands with the rand()-drawn k-mer digits of the middle
N, ragged lengths down to L = W).
"""
import os
import subprocess

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

RTOL = 1e-5
FLT_MAX = float(np.finfo(np.float32).max)
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "bammmotif2_b200", "bin")


@pytest.fixture(scope="module")
def capi():
    from bammmotif2_b200 import capi
    capi.load()
    assert capi.device_count() >= 1, "no CUDA device: the product has no CPU fallback"
    return capi


def assert_rel(a, b, rtol, atol=0.0, what=""):
    a = np.asarray(a, np.float64)
    b = np.asarray(b, np.float64)
    err = np.abs(a - b)
    bad = err > rtol * np.abs(b) + atol
    assert not bad.any(), "%s: %d / %d outside tolerance, worst rel %.3g" % (
        what, int(bad.sum()), bad.size, float((err / np.maximum(np.abs(b), 1e-300)).max()))


def make_data(capi, oracle, A, W, seed, nseq=300, single_strand=False, Lmin=None, Lmax=90, with_n=True):
    """Seeded ragged set: stored lengths from W (one window, truncated columns) up; both strands unless single_strand.
    Returns (seqset, codes, kmer, offsets)."""
    rng = np.random.default_rng(seed)
    Lmin = Lmin or max(W, 20)
    enc = []
    for n in range(nseq):
        L = W if n == 7 else int(rng.integers(Lmin, Lmax + 1))
        L0 = L if single_strand else max((L - 1) // 2, W // 2)                  # stored L = 2 L0 + 1 >= W
        s = rng.integers(1, A + 1, size=L0, dtype=np.uint8)
        if with_n and n % 11 == 3:
            s[L0 // 3] = 0                                                      # an N inside the record
        enc.append(s)
    oracle.srand(seed)
    codes, kmer, offsets = oracle.encode_sequences(enc, "EXTENDED" if A == 6 else "STANDARD", single_strand)
    assert int(np.diff(offsets.astype(np.int64)).min()) <= W + 1
    pp, pk = capi.kmer_patches(codes, kmer)
    ss = capi.SeqSet(codes, offsets, A, pp, pk)
    return ss, codes, kmer, offsets


def initial_model(oracle, kmer, A, K, Kbg, W, seed):
    from bammmotif2_b200 import hostmodel
    nb, vbg = oracle.bg_model(kmer, A, Kbg, hostmodel.default_bg_alpha(Kbg))
    alpha = hostmodel.default_motif_alpha(K, W)
    sites = np.random.default_rng(seed + 1).integers(1, A + 1, size=(200, W), dtype=np.uint8)
    return hostmodel.motif_from_sites(sites, A, K, alpha, vbg), vbg, alpha, nb


def largest_window_product(kmer, offsets, A, K, W, s):
    """max over the windows of prod_j s[y(p+j)][j] and the LW1 of its sequence (float64)."""
    Yn = A ** (K + 1)
    logs = np.log(np.asarray(s, np.float64).reshape(Yn, W))
    y = (kmer % np.uint64(Yn)).astype(np.int64)
    best, best_lw1 = -np.inf, 1
    for n in range(len(offsets) - 1):
        a, b = int(offsets[n]), int(offsets[n + 1])
        LW1 = b - a - W + 1
        idx = np.arange(LW1)[:, None] + np.arange(W)[None, :]
        v = logs[y[a:b][idx], np.arange(W)[None, :]].sum(axis=1).max()
        if v - np.log(LW1) > best - np.log(best_lw1):
            best, best_lw1 = v, LW1
    return float(np.exp(best)), best_lw1


def em_against_oracle(capi, oracle, ss, kmer, offsets, A, K, W, v0, vbg, alpha, iters=2, subset=None, q=0.3):
    Kbg = min(K, 2)
    em = capi.EM(ss, W, K, Kbg, subset=subset)
    em.set_model(v0, vbg, alpha, q)
    nseq = len(offsets) - 1
    for it in range(iters):
        # the oracle starts every iteration from the model the device holds (a product of up to 63 table entries amplifies
        # last-bit differences of the previous iteration's model)
        v = em.model()
        s = oracle.linear_s(v, vbg, A, K, Kbg, W)
        big, lw1 = largest_window_product(kmer, offsets, A, K, W, s)
        assert big < 1e-6 * FLT_MAX / lw1, (big, lw1)               # the linear products cannot drift into inf / NaN
        r_ref, llh_ref = oracle.estep(kmer, offsets, A, K, W, s, q)
        n_ref = oracle.mstep(kmer, offsets, A, K, W, r_ref)
        v = oracle.update_v(n_ref, alpha.ravel(), vbg, A, K, W, v)
        llh = em.estep()
        assert abs(llh - llh_ref) <= RTOL * abs(llh_ref) + 1e-7 * nseq, (it, llh, llh_ref)
        assert_rel(em.r(), r_ref, RTOL, atol=1e-37, what="r it%d" % it)
        em.mstep()
        assert_rel(em.counts(), n_ref, RTOL, atol=1e-9, what="n it%d" % it)
        assert_rel(em.model(), v, RTOL, what="v it%d" % it)
    return em


@pytest.mark.parametrize("A,K,W", [(4, 0, 33), (4, 2, 40), (4, 3, 63), (4, 4, 48),      # table in shared memory
                                   (4, 4, 63), (4, 6, 36),                              # row-form E-step, k_mstep_cols
                                   (6, 2, 45), (6, 5, 36)])                             # EXTENDED alphabet
def test_em_per_iteration_against_oracle(capi, oracle, A, K, W):
    ss, _, kmer, offsets = make_data(capi, oracle, A, W, 100 * A + K + W)
    v0, vbg, alpha, _ = initial_model(oracle, kmer, A, K, min(K, 2), W, W)
    em_against_oracle(capi, oracle, ss, kmer, offsets, A, K, W, v0, vbg, alpha, iters=3)


def test_em_single_strand_against_oracle(capi, oracle):
    A, K, W = 4, 2, 40
    ss, _, kmer, offsets = make_data(capi, oracle, A, W, 5, single_strand=True, Lmax=150)
    v0, vbg, alpha, _ = initial_model(oracle, kmer, A, K, 2, W, 5)
    em_against_oracle(capi, oracle, ss, kmer, offsets, A, K, W, v0, vbg, alpha)


@pytest.mark.parametrize("K", [2, 4])
def test_em_fold_subset_against_oracle(capi, oracle, K):
    """A permuted fold subset (as FDR's cross-validation folds create them), smem tables (K = 2) and rows (K = 4)."""
    A, W = 4, 63
    ss, _, kmer, offsets = make_data(capi, oracle, A, W, 17 + K)
    sub = np.random.default_rng(3).permutation(len(offsets) - 1)[:170].astype(np.uint64)
    L = np.diff(offsets.astype(np.int64))
    sub_off = np.zeros(len(sub) + 1, np.uint64)
    sub_off[1:] = np.cumsum(L[sub.astype(np.int64)])
    sub_kmer = np.concatenate([kmer[int(offsets[i]):int(offsets[i + 1])] for i in sub])
    v0, vbg, alpha, _ = initial_model(oracle, kmer, A, K, 2, W, 9)
    em_against_oracle(capi, oracle, ss, sub_kmer, sub_off, A, K, W, v0, vbg, alpha, subset=sub)


def _with_env(env, fn):
    old = {k: os.environ.get(k) for k in env}
    os.environ.update(env)
    try:
        return fn()
    finally:
        for k, v in old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


def test_global_count_tables_give_the_same_bits(capi, oracle):
    """(4, 4, 63): the M-step with global count tables (BAMM_GEN_NO_COLS=1, k_mstep) and with column ranges in shared memory
    (k_mstep_cols) sum the same fixed-point integers."""
    A, K, W = 4, 4, 63
    ss, _, kmer, offsets = make_data(capi, oracle, A, W, 404)
    v0, vbg, alpha, _ = initial_model(oracle, kmer, A, K, 2, W, 404)

    def run():
        em = capi.EM(ss, W, K, 2)
        em.set_model(v0, vbg, alpha, 0.3)
        out = []
        for _ in range(2):
            llh = em.estep()
            r = em.r()
            em.mstep()
            out.append((llh, r, em.counts(), em.model()))
        return out

    a = run()
    b = _with_env({"BAMM_GEN_NO_COLS": "1"}, run)
    for (la, ra, na, va), (lb, rb, nb, vb) in zip(a, b):
        assert la == lb and np.array_equal(ra, rb) and np.array_equal(na, nb) and np.array_equal(va, vb)


def test_optimize_against_oracle(capi, oracle):
    """EM::optimize at (4, 2, 40): the reference's stop rule (v_diff < 0.01, or the llh falls after iteration 10) gives the same
    iteration count and the final model agrees. Seed 22: every llh change after iteration 10 of the oracle's run is at least
    1e-4 of the llh and every v_diff far from 0.01, so the count does not hinge on last-bit differences (asserted)."""
    A, K, W, seed = 4, 2, 40, 22
    ss, _, kmer, offsets = make_data(capi, oracle, A, W, seed, Lmax=120)
    v0, vbg, alpha, _ = initial_model(oracle, kmer, A, K, 2, W, seed)
    ref = oracle.em_optimize(kmer, offsets, A, K, W, 2, vbg, alpha.ravel(), v0, 0.3)
    llh = ref["llh"].astype(np.float64)
    assert np.all(np.abs(np.diff(llh)[9:]) > 1e-4 * np.abs(llh[10:])) and np.all(np.abs(ref["vdiff"] / 0.01 - 1.0) > 0.5)
    em = capi.EM(ss, W, K, 2)
    em.set_model(v0, vbg, alpha, 0.3)
    res = em.optimize()
    assert res["iterations"] == ref["iterations"]
    assert_rel(res["v"], ref["v"], 1e-4, what="v")


@pytest.mark.parametrize("W", [33, 47, 63])
def test_scoring_bit_exact(capi, oracle, W):
    """An all-regular ACGT set (at W <= 32 it would take the packed path): MOPS, ZOOPS and the arg-max are the oracle's bits,
    with and without MOPS. Sequence 0 is X X with the model's consensus planted in X: its best window and the copy 200
    positions later tie, and the first maximum must win."""
    A, K, Kbg = 4, 2, 2
    rng = np.random.default_rng(W)
    enc = [rng.integers(1, 5, size=int(rng.integers(W, 300)), dtype=np.uint8) for _ in range(400)]
    _, kmer, _ = oracle.encode_sequences(enc, "STANDARD", True)
    v0, vbg, alpha, _ = initial_model(oracle, kmer, A, K, Kbg, W, W)
    x = rng.integers(1, 5, size=200, dtype=np.uint8)
    x[50:50 + W] = 1 + np.asarray(v0[:4 * W], np.float32).reshape(4, W).argmax(axis=0)
    enc[0] = np.concatenate([x, x])
    codes, kmer, offsets = oracle.encode_sequences(enc, "STANDARD", True)
    omops, ozoops, oz = oracle.logodds(kmer, offsets, A, K, W, oracle.log_s(v0, vbg, A, K, Kbg, W))
    assert int(oz[0]) == 50 and omops[250] == ozoops[0], "the planted copy must tie the maximum"
    ss = capi.SeqSet(codes, offsets, A)
    mops, zoops, z = ss.score(W, K, Kbg, v0, vbg)
    assert np.array_equal(mops, omops) and np.array_equal(zoops, ozoops) and np.array_equal(z, oz)
    _, zoops2, z2 = ss.score(W, K, Kbg, v0, vbg, want_mops=False)
    assert np.array_equal(zoops2, ozoops) and np.array_equal(z2, oz)


def test_mask_against_oracle(capi, oracle):
    """EM::mask (--advanceEM) at W = 40: same kept windows and threshold, same iteration count, model / llh / counts within the
    tolerances of the fixture-based mask test. r is a product of W factors that each carry the final model's difference, so
    its tolerance, 2e-4 for the fixtures' W <= 10, grows with W / 10."""
    A, K, W = 4, 2, 40
    ss, _, kmer, offsets = make_data(capi, oracle, A, W, 40, Lmax=140)
    v0, vbg, alpha, _ = initial_model(oracle, kmer, A, K, 2, W, 40)
    em = capi.EM(ss, W, K, 2)
    em.set_model(v0, vbg, alpha, 0.3)
    res = em.mask(f=0.05)
    ref = oracle.em_mask(kmer, offsets, A, K, W, 2, vbg, alpha.ravel(), v0, 0.3, f=0.05)
    assert res["nkept"] == ref["nkept"] and np.float32(res["cutoff"]) == np.float32(ref["cutoff"])
    assert res["iterations"] == ref["iterations"]
    assert_rel(res["v"], ref["v"], 1e-4, what="v")
    assert abs(res["llh"] - ref["llh"]) <= 1e-4 * abs(ref["llh"])
    assert_rel(em.counts(), ref["n"], 1e-4, atol=1e-8, what="n")
    r = em.r()
    assert np.array_equal(r == 0, ref["r"] == 0)
    assert_rel(r, ref["r"], 2e-4 * W / 10, atol=1e-30, what="r")


def _sample_pwm(capi, ss, W, K=1):
    import ctypes as C
    nsub = ss.nseq
    score = np.full((4, W), 1.0, np.float32)
    u = np.random.default_rng(0).random(nsub)
    n_all = np.zeros(capi.model_size(ss.A, K, W), np.int32)
    z = np.zeros(nsub, np.uint64)
    capi._check(capi.load().bamm_seqset_sample_pwm_sites(ss.h, None, nsub, W, K, 4, score.ctypes.data_as(C.POINTER(C.c_float)),
                                                         C.c_float(0.3), u.ctypes.data_as(C.POINTER(C.c_double)),
                                                         n_all.ctypes.data_as(C.POINTER(C.c_int32)), z.ctypes.data_as(C.POINTER(C.c_uint64))))
    return n_all, z


def test_width_limits(capi, oracle):
    """W = 63 is accepted by EM, scoring and PWM sampling, W = 64 by none; the packed and bound plans stay at W <= 32."""
    ss, _, kmer, _ = make_data(capi, oracle, 4, 63, 1, nseq=40, Lmin=70)
    v0, vbg, alpha, _ = initial_model(oracle, kmer, 4, 1, 1, 63, 1)
    capi.EM(ss, 63, 1, 1).close()
    ss.score(63, 1, 1, v0, vbg)
    n_all, z = _sample_pwm(capi, ss, 63)
    assert n_all[:4 * 63].reshape(4, 63).sum(axis=0).max() <= ss.nseq and np.all(z <= 70)
    with pytest.raises(capi.BammError):
        capi.EM(ss, 64, 1, 1)
    v64 = np.full(capi.model_size(4, 1, 64), 0.25, np.float32)
    with pytest.raises(capi.BammError):
        ss.score(64, 1, 1, v64, vbg)
    with pytest.raises(capi.BammError):
        _sample_pwm(capi, ss, 64)
    with pytest.raises(capi.BammError):
        capi.bound_plan_describe(33, 2, 2)
    with pytest.raises(capi.BammError):
        capi.plan_describe(33, 2, 2)


# ------------------------------------------------------------------------------------------------------------- host side

@pytest.fixture(scope="module")
def bins():
    from bammmotif2_b200 import build
    build.build_all()
    return BIN


def run(cmd, **kw):
    p = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, **kw)
    assert p.returncode == 0, "%s\n%s\n%s" % (" ".join(cmd), p.stdout[-2000:], p.stderr[-2000:])
    return p


def test_pwm_initialisation_40_columns_host_equals_device(bins, oracle, tmp_path):
    """Motif::initFromPWM of a 40-column MEME motif: the device sampler (BAMM_DEVICE_PWMINIT=1) writes the host's initial model."""
    from bammmotif2_b200 import synth
    fwd, _, _ = synth.planted_sequences(40, 600, 150, 12)
    fa = str(tmp_path / "p.fasta")
    synth.write_fasta(fa, fwd)
    p = np.random.default_rng(40).dirichlet(np.full(4, 0.5), size=40)
    with open(tmp_path / "w.meme", "w") as f:
        f.write("MEME version 4\n\nALPHABET= ACGT\n\nBackground letter frequencies\nA 0.25 C 0.25 G 0.25 T 0.25\n\n")
        f.write("MOTIF WIDE40\nletter-probability matrix: alength= 4 w= 40 nsites= 100 E= 0\n")
        for row in p:
            f.write(" ".join("%.4f" % x for x in row) + "\n")
        f.write("\n")
    K, Kbg = 2, 1
    _, kmer, _ = oracle.encode_sequences([r for r in fwd], "STANDARD", False)
    from bammmotif2_b200 import hostmodel
    nb, _ = oracle.bg_model(kmer, 4, Kbg, hostmodel.default_bg_alpha(Kbg))
    np.asarray(nb, np.uint64).tofile(tmp_path / "bgn.u64")
    np.array([1.0, 10.0], np.float32).tofile(tmp_path / "abg.f32")
    outs = []
    for name, env in (("host", {}), ("dev", {"BAMM_DEVICE_PWMINIT": "1"})):
        d = tmp_path / name
        d.mkdir()
        run([os.path.join(bins, "host_check"), "pwminit", "STANDARD", fa, "0", str(K), str(Kbg), str(tmp_path / "bgn.u64"),
             str(tmp_path / "abg.f32"), str(tmp_path / "w.meme"), "1", "0.3", str(d)], env=dict(os.environ, **env))
        outs.append(open(d / "v_init_1.f32", "rb").read())
    assert len(outs[0]) == 4 * capi_model_size(4, K, 40) and outs[0] == outs[1]


def capi_model_size(A, K, W):
    return sum(A ** (k + 1) * W for k in range(K + 1))


def _blocks(path):
    """columns of a BaMM-format file: one blank-line-terminated block per position"""
    return sum(1 for line in open(path).read().split("\n")[:-1] if line == "")


def test_cli_extend_to_39_columns(bins, tmp_path):
    """--extend 14 13 on 12-column sites: W = 39 through EM, FDR and scoring; W = 64 is refused with the width message. With the
    reference binary built (oracle/_ref), both write the same background and agree on the model like the fresh-data CLI test."""
    from bammmotif2_b200 import synth
    fwd, sites, _ = synth.planted_sequences(3939, 2000, 120, 12)
    fa, bs = str(tmp_path / "syn.fasta"), str(tmp_path / "sites.block")
    synth.write_fasta(fa, fwd)
    synth.write_sites(bs, sites)
    args = ["--bindingSiteFile", bs, "--EM", "-k", "2", "-K", "2", "--FDR", "-n", "3", "-m", "2", "--scoreSeqset", "--saveBaMMs"]
    run([os.path.join(bins, "BaMMmotif"), str(tmp_path / "our"), fa] + args + ["--extend", "14", "13"])
    od = tmp_path / "our"
    assert _blocks(od / "syn_motif_1.ihbcp") == 39
    ref = os.path.join(ROOT, "oracle", "_ref", "BaMMmotif_ref")
    if os.path.exists(ref):
        run([ref, str(tmp_path / "ref"), fa] + args + ["--extend", "14", "13", "--threads", "1"], env=dict(os.environ, OMP_NUM_THREADS="1"))
        rd = tmp_path / "ref"
        for fn in ("syn.hbcp", "syn.hbp"):
            assert open(rd / fn, "rb").read() == open(od / fn, "rb").read(), fn
        for fn in ("syn_motif_1.ihbcp", "syn_motif_1.ihbp"):
            a = np.array(open(rd / fn).read().split(), np.float64)
            b = np.array(open(od / fn).read().split(), np.float64)
            assert a.shape == b.shape and np.all(np.abs(a - b) <= 1.2e-3 * np.abs(a) + 1e-30), fn
    p = subprocess.run([os.path.join(bins, "BaMMmotif"), str(tmp_path / "wide"), fa] + args + ["--extend", "26", "26"],
                       stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)
    assert p.returncode != 0 and "motif width 64" in p.stderr
