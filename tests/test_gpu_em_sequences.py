"""GPU suite: EM objects driven through the call sequences the C ABI allows (include/bamm_b200.h), not only set_model, then
(estep, [optimize_q], mstep) x n. The reference's EM (src/refinement/EM.h) allows more than that loop: estep again without an
mstep in between, optimize_q and mstep from any r (EM::MStep twice on one r gives the same model twice), and getR / getS
describe the last E-step, also after mask.

A small state machine over the CPU oracle (oracle/oracle.py) holds what the reference's EM holds after every call: v, q, the s
and r of the last E-step, n and the log likelihood. It is re-seeded from the device's model and q at every E-step (as
test_gpu_baseline_shapes.py does), so last-bit differences do not compound; the tolerances are that file's: rtol 1e-5, r atol
1e-37, counts atol 1e-7, v atol 1e-7 / alpha_K, llh 1e-5 |llh| + 1e-7 nseq.

Seeded random walks run the same calls on three EM objects in lockstep: bound reuse forced with a slack of 2 bits (small drifts
decide between the watch pass and the full pass), bound reuse off, and the dense E-step (no pruning). After every call the
model, counts, q and s of all three must be the same bits and match the state machine; r is read when the walk draws r()
(reading it materialises r, which would hide the path where r is not yet materialised). Directed cases name the sequences
where the device keeps state between calls: the drift bound of the bound reuse, the buffers of the last E-step, mask.
"""
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

RTOL = 1e-5
E_STATE = "bamm error -4:"
_KEYS = ("BAMM_BOUND_REUSE", "BAMM_BOUND_SLACK", "BAMM_NO_BOUND_REUSE", "BAMM_WATCH_FRAC", "BAMM_NO_SPARSE", "BAMM_CAND_FRAC")
SWITCHES = (("reuse", {"BAMM_BOUND_REUSE": "1", "BAMM_BOUND_SLACK": "2"}),
            ("no_reuse", {"BAMM_NO_BOUND_REUSE": "1"}),
            ("dense", {"BAMM_NO_SPARSE": "1"}))


@pytest.fixture(scope="module")
def capi():
    from bammmotif2_b200 import capi
    capi.load()
    assert capi.device_count() >= 1, "no CUDA device: the product has no CPU fallback"
    return capi


def make_em(capi, d, env, subset=None):
    """An EM object over data set d created under exactly the switches in env (they are read at creation)."""
    old = {k: os.environ.pop(k, None) for k in _KEYS}
    os.environ.update(env)
    try:
        return capi.EM(d["ss"], d["W"], d["K"], d["Kbg"], subset=subset)
    finally:
        for k in _KEYS:
            os.environ.pop(k, None)
        os.environ.update({k: v for k, v in old.items() if v is not None})


def assert_rel(a, b, rtol, atol, what):
    a = np.asarray(a, np.float64)
    b = np.asarray(b, np.float64)
    err = np.abs(a - b)
    bad = err > rtol * np.abs(b) + atol
    assert not bad.any(), "%s: %d / %d outside tolerance, first at %d (%.9g vs %.9g)" % (
        what, int(bad.sum()), bad.size, int(np.argmax(bad)), a.ravel()[int(np.argmax(bad))], b.ravel()[int(np.argmax(bad))])


# ---------------------------------------------------------------------------------------------------------------- data
def _hash(codes, A, single, mid, rng):
    """The reference's 11-mer hash of one stored sequence, an independent draw per (position, digit) of the N (Sequence.cpp:38)."""
    d = np.where(codes == 0, 0, codes.astype(np.int64) - 1)
    km = np.zeros(len(codes), np.uint64)
    for t in range(min(11, len(codes))):
        dig = d[:len(codes) - t].copy()
        if not single:
            isn = np.arange(len(codes) - t) == mid
            dig[isn] = rng.integers(0, A, size=int(isn.sum()))
        km[t:] += (dig * (A ** t)).astype(np.uint64)
    return km


def _ragged(seed, nseq, W, A):
    """Lengths from just above W to a few hundred bases, both strands (with the N) and some single-stranded records, a planted
    site in half of the sequences: windows over the N and truncated windows fill whole sequences, regions are ragged."""
    rng = np.random.default_rng(seed)
    pwm = rng.dirichlet(np.full(A, 0.3), size=W)
    sites = np.stack([rng.choice(A, size=200, p=pwm[j]) for j in range(W)], axis=1).astype(np.uint8) + 1
    comp = np.array([0, 4, 3, 2, 1, 3, 3], np.uint8)[:A + 1]            # ACGT(MH) -> TGCA(GG), Alphabet.cpp:12-27
    lens = np.concatenate([rng.integers(W // 2 + 1, 2 * W + 3, size=nseq // 2), rng.integers(2 * W, 300, size=nseq - nseq // 2)])
    rng.shuffle(lens)
    chunks, kmers, offs = [], [], [0]
    for n, L0 in enumerate(lens):
        fwd = rng.integers(1, A + 1, size=int(L0), dtype=np.uint8)
        if L0 >= W and n % 2 == 0:
            s0 = rng.integers(0, L0 - W + 1)
            fwd[s0:s0 + W] = sites[n % 200]
        single = (n % 7 == 3) and L0 >= W
        codes = fwd if single else np.concatenate([fwd, [0], comp[fwd][::-1]]).astype(np.uint8)
        chunks.append(codes); kmers.append(_hash(codes, A, single, int(L0), rng)); offs.append(offs[-1] + len(codes))
    codes, kmer, offsets = np.concatenate(chunks), np.concatenate(kmers), np.array(offs, np.uint64)
    assert np.diff(offsets.astype(np.int64)).min() >= W
    return codes, kmer, offsets, sites


_DATA = {}


def data(capi, oracle, name):
    """ragged: W=20, K=4 (pruned path); ragged_subset: the same set as a permuted index subset of 85 % of it (an FDR fold);
    a6: the EXTENDED alphabet at K=5, W=12 (generic index-array path)."""
    if name in _DATA:
        return _DATA[name]
    from bammmotif2_b200 import hostmodel
    if name == "ragged_subset":
        base = data(capi, oracle, "ragged")
        sub = np.random.default_rng(5).permutation(base["ss"].nseq)[:int(0.85 * base["ss"].nseq)].astype(np.uint64)
        o = base["offsets"].astype(np.int64)
        kmer = np.concatenate([base["kmer"][o[i]:o[i + 1]] for i in sub])
        offsets = np.concatenate([[0], np.cumsum(o[sub.astype(np.int64) + 1] - o[sub.astype(np.int64)])]).astype(np.uint64)
        _DATA[name] = dict(base, kmer=kmer, offsets=offsets, subset=sub)
        return _DATA[name]
    A, W, K, Kbg, nseq = {"ragged": (4, 20, 4, 2, 4000), "a6": (6, 12, 5, 2, 3000)}[name]
    codes, kmer, offsets, sites = _ragged({"ragged": 2020, "a6": 612}[name], nseq, W, A)
    pp, pk = capi.kmer_patches(codes, kmer)
    ss = capi.SeqSet(codes, offsets, A, pp, pk)
    _, vbg = oracle.bg_model(kmer, A, Kbg, hostmodel.default_bg_alpha(Kbg))
    alpha = hostmodel.default_motif_alpha(K, W)
    v0 = hostmodel.motif_from_sites(sites, A, K, alpha, vbg)
    _DATA[name] = dict(ss=ss, kmer=kmer, offsets=offsets, subset=None, A=A, W=W, K=K, Kbg=Kbg, vbg=vbg, alpha=alpha, v0=v0)
    return _DATA[name]


# ------------------------------------------------------------------------------------------------------- state machine
class RefEM:
    """What the reference's EM object holds after each call (EM.cpp:62-259, 505-519), on the oracle."""

    def __init__(self, orc, d):
        self.o, self.d = orc, d
        self.A, self.W, self.K, self.Kbg = d["A"], d["W"], d["K"], d["Kbg"]
        self.nseq = len(d["offsets"]) - 1
        self.alpha = d["alpha"]
        self.v = self.q = self.r = self.s_e = self.n = self.llh = None
        self.atol_v = 1e-7 / float(self.alpha[self.K].min())

    def linear_s(self, v):
        return self.o.linear_s(v, self.d["vbg"], self.A, self.K, min(self.K, self.Kbg), self.W)

    def set_model(self, v, q):
        self.v, self.q, self.r, self.s_e = np.array(v, np.float32), np.float32(q), None, None

    def estep(self, v_dev=None, q_dev=None):
        if v_dev is not None:                                   # re-seed from the device (checked against this state before)
            self.v, self.q = np.array(v_dev, np.float32), np.float32(q_dev)
        self.s_e = self.linear_s(self.v)
        self.r, _, self.llh = self.o.estep(self.d["kmer"], self.d["offsets"], self.A, self.K, self.W, self.s_e, float(self.q), want_double=True)
        return self.llh

    def mstep(self):
        self.n = self.o.mstep(self.d["kmer"], self.d["offsets"], self.A, self.K, self.W, self.r, accumulate_double=True)
        self.v = self.o.update_v(self.n, self.alpha.ravel(), self.d["vbg"], self.A, self.K, self.W, self.v.copy())

    def optimize_q(self):                                       # EM.cpp:515 with the exact sum of the posteriors
        n1 = float(np.sum(self.r, dtype=np.float64))
        self.q = np.float32((np.float32(self.nseq) - np.float32(n1) + np.float32(1)) / (np.float32(self.nseq) + np.float32(2)))
        return self.q

    def s(self):
        return self.s_e if self.r is not None else self.linear_s(self.v)

    # comparisons
    def check_llh(self, llh, what):
        assert abs(llh - self.llh) <= RTOL * abs(self.llh) + 1e-7 * self.nseq, (what, llh, self.llh)

    def check_r(self, r, what):
        assert_rel(r, self.r, RTOL, 1e-37, "r " + what)

    def check_state(self, model, counts, q, s, what):
        assert_rel(model, self.v, RTOL, self.atol_v, "v " + what)
        if self.n is not None:
            assert_rel(counts, self.n, RTOL, 1e-7, "n " + what)
        assert abs(q - self.q) <= RTOL * self.q, ("q " + what, q, self.q)
        assert_rel(s, self.s(), RTOL, self.atol_v / float(self.d["vbg"].min()), "s " + what)


# ------------------------------------------------------------------------------------------------------------- walks
CALLS = ("estep", "mstep", "optimize_q", "iterate", "set_model", "r", "s", "model", "counts", "q")
WEIGHTS = np.array([6, 5, 2, 2, 1, 2, 1, 1, 1, 1], np.float64)


def walk_calls(seed, n):
    rng = np.random.default_rng(seed)
    calls = []
    for _ in range(n):
        c = CALLS[rng.choice(len(CALLS), p=WEIGHTS / WEIGHTS.sum())]
        arg = None
        if c == "iterate":
            arg = int(rng.choice([0, 1, 3]))
        elif c == "set_model":
            arg = (bool(rng.integers(2)), float(rng.choice([0.1, 0.3, 0.6])))      # (initial model?, new q)
        calls.append((c, arg))
    return calls


def expect_state_error(capi, fn):
    with pytest.raises(capi.BammError, match=E_STATE):
        fn()


def same_lists(a, b, what):
    """The watch pass emits exactly the full pass's candidates: the candidate and active-list sizes of the last E-step agree."""
    ia, ib = a.estep_info(), b.estep_info()
    assert (ia["candidates"], ia["active"]) == (ib["candidates"], ib["active"]), (what, ia, ib, a.bound_reuse_info())


def same_bits(xs, what):
    for name, x in xs[1:]:
        assert np.array_equal(np.asarray(xs[0][1]), np.asarray(x)), "%s: %s and %s differ" % (what, xs[0][0], name)


@pytest.mark.parametrize("seed", [101, 202, 303])
@pytest.mark.parametrize("name", ["ragged", "ragged_subset", "a6"])
def test_random_call_walk(capi, oracle, name, seed):
    d = data(capi, oracle, name)
    ems = [(sw, make_em(capi, d, env, subset=d["subset"])) for sw, env in SWITCHES]
    ref = RefEM(oracle, d)
    dense_only = d["A"] != 4

    def each(fn):
        return [(sw, fn(em)) for sw, em in ems]

    def observe(what):
        outs = each(lambda em: (em.model(), em.counts(), em.q(), em.s()))
        for i, key in enumerate(("model", "counts", "q", "s")):
            if key != "counts" or ref.n is not None:            # (no M-step yet: the count buffers hold nothing)
                same_bits([(sw, o[i]) for sw, o in outs], "%s %s" % (key, what))
        m, n, q, s = outs[0][1]
        ref.check_state(m, n, q, s, what)

    def set_model(v, q):
        for _, em in ems:
            em.set_model(v, d["vbg"], d["alpha"], q)
        ref.set_model(v, q)

    def estep(what):
        llh = each(lambda em: em.estep())
        same_bits(llh, "llh " + what)
        if not dense_only:
            same_lists(ems[0][1], ems[1][1], what)
        ref.estep(ems[0][1].model(), ems[0][1].q())
        ref.check_llh(llh[0][1], what)

    # the prefix: forbidden calls after set_model, then two E-steps on unchanged tables (the second may take the watch pass)
    set_model(d["v0"], 0.3)
    for _, em in ems:
        expect_state_error(capi, em.mstep)
        expect_state_error(capi, em.optimize_q)
        expect_state_error(capi, em.r)
    observe("after set_model")
    estep("prefix estep 1")
    estep("prefix estep 2")
    if not dense_only:
        assert all(em.estep_info()["pruned"] == (sw != "dense") for sw, em in ems)
        info = ems[0][1].bound_reuse_info()
        assert info["enabled"] and info["watch"] >= 1 and np.isfinite(info["log2_drift"]), info
    observe("prefix")

    for step, (call, arg) in enumerate(walk_calls(seed, 32)):
        what = "%s seed %d step %d %s(%s)" % (name, seed, step, call, "" if arg is None else arg)
        if call == "estep":
            estep(what)
        elif call == "mstep":
            if ref.r is None:
                for _, em in ems:
                    expect_state_error(capi, em.mstep)
            else:
                for _, em in ems:
                    em.mstep()
                ref.mstep()
        elif call == "optimize_q":
            if ref.r is None:
                for _, em in ems:
                    expect_state_error(capi, em.optimize_q)
            else:
                qs = each(lambda em: em.optimize_q())
                same_bits(qs, what)
                ref.optimize_q()
                assert abs(qs[0][1] - ref.q) <= RTOL * ref.q, (what, qs[0][1], ref.q)
                ref.q = np.float32(qs[0][1])
        elif call == "iterate":
            v_start, q_start = ems[0][1].model(), ems[0][1].q()
            out = each(lambda em: em.iterate(arg))
            same_bits(out, what)
            if not dense_only:
                same_lists(ems[0][1], ems[1][1], what)
            if arg > 0:
                ref.estep(v_start, q_start)
                ref.mstep()
                for _ in range(arg - 1):
                    ref.estep()
                    ref.mstep()
            if ref.llh is not None:                     # iterate(0) returns the log likelihood of the last E-step
                ref.check_llh(out[0][1][0], what)
        elif call == "set_model":
            initial, q = arg
            set_model(d["v0"] if initial else ems[0][1].model(), q)
        elif call == "r":
            if ref.r is None:
                for _, em in ems:
                    expect_state_error(capi, em.r)
            else:
                rs = each(lambda em: em.r())
                same_bits(rs, what)
                ref.check_r(rs[0][1], what)
        # s, model, counts, q: read by observe() after every call
        observe(what)


def test_calls_out_of_order_are_state_errors(capi, oracle):
    """Every call that needs a model or an r returns BAMM_E_STATE without one, and leaves the object usable."""
    d = data(capi, oracle, "ragged")
    em = make_em(capi, d, {})
    for fn in (lambda: em.estep(), em.mstep, em.optimize_q, lambda: em.iterate(1), lambda: em.optimize(), lambda: em.mask(), em.r):
        expect_state_error(capi, fn)
    em.set_model(d["v0"], d["vbg"], d["alpha"], 0.3)
    em.estep()
    em.mstep()
    em.set_model(d["v0"], d["vbg"], d["alpha"], 0.3)           # a new model: the r of the last E-step is gone
    for fn in (em.mstep, em.optimize_q, em.r):
        expect_state_error(capi, fn)
    ref = RefEM(oracle, d)
    ref.set_model(d["v0"], 0.3)
    ref.estep()
    ref.check_llh(em.estep(), "estep after the errors")
    ref.check_r(em.r(), "after the errors")


# ---------------------------------------------------------------------------------------------------------- directed
@pytest.mark.parametrize("slack", [2, 6, 8])
def test_estep_optimize_q_estep(capi, oracle, slack):
    """estep -> optimize_q -> estep from a q far below its optimum: the candidate threshold falls by the q odds ratio while no
    table is built. The drift bound of the second E-step must carry that ratio (a watch pass needs it below 2^slack), and the
    result must be the bits of a run without bound reuse."""
    d = data(capi, oracle, "ragged")
    on = make_em(capi, d, {"BAMM_BOUND_REUSE": "1", "BAMM_BOUND_SLACK": str(slack)})
    off = make_em(capi, d, {"BAMM_NO_BOUND_REUSE": "1"})
    q0 = 0.05
    for em in (on, off):
        em.set_model(d["v0"], d["vbg"], d["alpha"], q0)
    assert on.estep() == off.estep()
    assert not on.bound_reuse_info()["last_watch"]
    q1 = on.optimize_q()
    assert q1 == off.optimize_q()
    qa, qb = float(np.float32(q0)), float(np.float32(q1))
    log2_ratio = float(np.log2(((1.0 - qa) / qa) / ((1.0 - qb) / qb)))
    assert log2_ratio > 2, (q0, q1)                     # the threshold fell by more than 2^2
    assert on.estep() == off.estep(), "log likelihood"
    same_lists(on, off, "second E-step")
    info = on.bound_reuse_info()
    if info["last_watch"]:
        assert np.isfinite(info["log2_drift"]) and info["log2_drift"] >= log2_ratio, (info, log2_ratio)
    print("slack %d: log2 q odds ratio %.3f," % (slack, log2_ratio), info)
    if log2_ratio < slack and 4 * info["watched"] <= d["ss"].npos:     # unchanged tables, a q ratio below 2^slack, a list that pays
        assert info["last_watch"], info
    assert np.array_equal(on.r(), off.r()), "r"
    on.mstep(); off.mstep()
    assert np.array_equal(on.counts(), off.counts()), "counts"
    assert np.array_equal(on.model(), off.model()), "model"
    assert on.estep() == off.estep(), "log likelihood of the next E-step"


def _planted(nseq, L0, W, seed=7):
    from bammmotif2_b200 import hostmodel, synth
    fwd, sites, _ = synth.planted_sequences(seed, nseq, L0, W)
    codes = synth.stored_both_strands(fwd)
    ppos, pkmer = synth.middle_n_patches(codes, seed)
    offsets = np.arange(nseq + 1, dtype=np.uint64) * np.uint64(codes.shape[1])
    return codes, offsets, ppos, pkmer, sites, hostmodel


def test_watch_overflow_dense_hold_then_moved_tables(capi):
    """A watch pass that overflows its candidate cap switches to the dense E-step and keeps the watch list valid. An mstep moves
    the tables during the hold, the hold's E-steps build none, and the E-step after the hold must bound the drift of the tables
    it runs with from those the list was built from. The candidate cap (BAMM_CAND_FRAC) is picked by bisection so that the full
    pass at the first q fits, the watch pass at the optimised q overflows, and the E-step after the hold fits again."""
    W, K, Kbg = 20, 4, 2
    codes, offsets, ppos, pkmer, sites, hostmodel = _planted(40000, 500, W)
    ss = capi.SeqSet(codes.ravel(), offsets, 4, ppos, pkmer)
    vbg = hostmodel.background_from_counts(ss.count_kmers(Kbg), 4, Kbg, hostmodel.default_bg_alpha(Kbg))
    alpha = hostmodel.default_motif_alpha(K, W)
    v0 = hostmodel.motif_from_sites(sites, 4, K, alpha, vbg)
    d = dict(ss=ss, W=W, K=K, Kbg=Kbg)
    q0 = 0.05

    def fits(frac, v, q):
        e = make_em(capi, d, {"BAMM_NO_BOUND_REUSE": "1", "BAMM_CAND_FRAC": repr(frac)})
        try:
            e.set_model(v, vbg, alpha, q)
            e.estep()
            return not e.estep_info()["dense_ran"]
        finally:
            e.close()

    def least_fitting(v, q):                    # (largest cap seen to overflow, smallest cap seen to fit), log bisection
        lo, hi = 0.002, 0.42
        if fits(lo, v, q):
            return 0.0, lo
        for _ in range(10):
            mid = float(np.sqrt(lo * hi))
            if fits(mid, v, q):
                hi = mid
            else:
                lo = mid
        return lo, hi

    def sequence_models(va):                    # q1 and the model after the M-step of the sequence below (same bits on every path)
        e = make_em(capi, d, {"BAMM_NO_BOUND_REUSE": "1"})
        e.set_model(va, vbg, alpha, q0)
        e.estep()
        q1 = e.optimize_q()
        e.estep()
        e.mstep()
        vb = e.model()
        e.close()
        return q1, vb

    # starting models: the planted one and the models after 1..3 iterations at q = 0.3 (the candidates shrink once EM is under way)
    em = make_em(capi, d, {"BAMM_NO_BOUND_REUSE": "1"})
    em.set_model(v0, vbg, alpha, 0.3)
    starts = [v0]
    for _ in range(3):
        em.estep()
        em.mstep()
        starts.append(em.model())
    em.close()
    found, tried = None, []
    for k, va in enumerate(starts):
        q1, vb = sequence_models(va)
        over1, _ = least_fitting(va, q1)        # the watch pass at (va, q1) must overflow: cap < over1
        _, fit2 = least_fitting(vb, q1)         # the E-step after the hold at (vb, q1) must fit: cap >= fit2
        tried.append("start %d: q1 %.4f, overflow below %.5g, fit from %.5g" % (k, q1, over1, fit2))
        if fit2 < over1:
            frac = float(np.sqrt(fit2 * over1))
            if fits(frac, va, q0):              # ... and the first full pass at (va, q0) must fit
                found = (va, q1, vb, frac)
                break
    print("; ".join(tried))
    if found is None:
        pytest.xfail("no candidate cap makes the watch pass overflow and the E-step after the hold fit: " + "; ".join(tried))
    v0, q1, v2, frac = found

    on = make_em(capi, d, {"BAMM_BOUND_REUSE": "1", "BAMM_CAND_FRAC": repr(frac)})
    off = make_em(capi, d, {"BAMM_NO_BOUND_REUSE": "1", "BAMM_CAND_FRAC": repr(frac)})

    def both(fn):
        a, b = fn(on), fn(off)
        return a, b

    for em in (on, off):
        em.set_model(v0, vbg, alpha, q0)
    a, b = both(lambda e: e.estep())
    assert a == b and not on.estep_info()["dense_ran"], on.estep_info()
    a, b = both(lambda e: e.optimize_q())
    assert a == b == q1
    a, b = both(lambda e: e.estep())
    assert a == b, "llh of the overflowing E-step"
    info, einfo = on.bound_reuse_info(), on.estep_info()
    if not (info["last_watch"] and einfo["dense_ran"] and info["valid"]):
        pytest.xfail("the E-step at the optimised q was not an overflowing watch pass: %s %s" % (info, einfo))
    both(lambda e: e.mstep())
    assert np.array_equal(on.model(), v2) and np.array_equal(off.model(), v2)
    for hold in range(2):                       # DENSE_HOLD_MIN E-steps on the dense path, no table built
        a, b = both(lambda e: e.estep())
        assert a == b, ("llh in the hold", hold)
        assert on.estep_info()["dense_ran"], (hold, on.estep_info())
    a, b = both(lambda e: e.estep())
    info, einfo = on.bound_reuse_info(), on.estep_info()
    print("E-step after the hold:", info, einfo)
    assert not einfo["dense_ran"], einfo
    assert a == b, "llh of the E-step after the hold"
    same_lists(on, off, "E-step after the hold")
    assert np.isfinite(info["log2_drift"]), info
    assert np.array_equal(on.r(0, 2000), off.r(0, 2000)), "r"
    both(lambda e: e.mstep())
    assert np.array_equal(on.counts(), off.counts()), "counts"
    assert np.array_equal(on.model(), off.model()), "model"


@pytest.mark.parametrize("env", [{}, {"BAMM_BOUND_REUSE": "1", "BAMM_BOUND_SLACK": "2"}, {"BAMM_NO_SPARSE": "1"}])
def test_mstep_twice_then_r_and_s(capi, oracle, env):
    """estep, mstep, mstep: the second update must not overwrite the tables the E-step read while r is still unmaterialised
    (pruned path); r() and s() describe the E-step, and the second M-step on the same r gives the same model."""
    d = data(capi, oracle, "ragged")
    em = make_em(capi, d, env)
    ref = RefEM(oracle, d)
    em.set_model(d["v0"], d["vbg"], d["alpha"], 0.3)
    ref.set_model(d["v0"], 0.3)
    ref.estep()
    ref.check_llh(em.estep(), "estep")
    assert em.estep_info()["pruned"] == ("BAMM_NO_SPARSE" not in env)
    em.mstep()
    v1 = em.model()
    em.mstep()
    ref.mstep()
    assert np.array_equal(em.model(), v1), "EM::MStep twice on one r gives the same model"
    ref.check_state(em.model(), em.counts(), em.q(), em.s(), "after two M-steps")
    ref.check_r(em.r(), "after two M-steps")
    ref.check_state(em.model(), em.counts(), em.q(), em.s(), "after r()")
    em.mstep()                                  # a third one, r materialised by now
    ref.check_state(em.model(), em.counts(), em.q(), em.s(), "after three M-steps")
    ref.estep(em.model(), em.q())
    ref.check_llh(em.estep(), "next estep")
    ref.check_r(em.r(), "next estep")


@pytest.mark.parametrize("estep_first", [True, False])
def test_mask_then_getters(capi, oracle, estep_first):
    """After mask, get_s / get_r / get_model / get_counts describe mask's final state: s and r of its last E-step, the model and
    counts of its last M-step. Stopped after 4 iterations, before it converges, so the s of the last E-step and the s of the
    final model differ (an even count: the double buffers then hold neither the E-step's table nor, after an earlier estep,
    the one that E-step left behind). Not re-seeded between mask's iterations: the tolerances are the mask parity test's (test_gpu_parity.py)."""
    d = data(capi, oracle, "ragged")
    em = make_em(capi, d, {})
    em.set_model(d["v0"], d["vbg"], d["alpha"], 0.3)
    if estep_first:
        em.estep()
    res = em.mask(f=0.05, max_iter=4)
    args = (d["kmer"], d["offsets"], d["A"], d["K"], d["W"], d["Kbg"], d["vbg"], d["alpha"], d["v0"], 0.3)
    ref = oracle.em_mask(*args, f=0.05, max_iter=4)
    # the s of the 4th E-step is the table of the model the first 3 iterations reach (mask is deterministic)
    ref3 = oracle.em_mask(*args, f=0.05, max_iter=3)
    assert ref3["iterations"] == 3
    lin_s = lambda v: oracle.linear_s(v, d["vbg"], d["A"], d["K"], min(d["K"], d["Kbg"]), d["W"])
    s_last, s_final = lin_s(ref3["v"]), lin_s(ref["v"])
    assert np.all(s_last > 0)
    assert np.max(np.abs(s_final.astype(np.float64) - s_last) / s_last) > 1e-2, "the case does not tell the two tables apart"
    assert res["nkept"] == ref["nkept"] and np.float32(res["cutoff"]) == np.float32(ref["cutoff"])
    assert res["iterations"] == ref["iterations"] == 4
    assert abs(res["llh"] - ref["llh"]) <= 1e-4 * abs(ref["llh"])
    assert_rel(em.s(), s_last, 1e-4, 0.0, "s")
    assert_rel(em.model(), ref["v"], 1e-4, 0.0, "v")
    assert_rel(em.counts(), ref["n"], 1e-4, 1e-8, "n")
    r = em.r()
    assert np.array_equal(r == 0, ref["r"] == 0)
    assert_rel(r, ref["r"], 2e-4, 1e-30, "r")


@pytest.mark.parametrize("env", [{}, {"BAMM_BOUND_REUSE": "1", "BAMM_BOUND_SLACK": "2"}])
def test_iterate_then_estep_and_r(capi, oracle, env):
    """iterate(n) leaves the buffers of its last E-step behind; an estep after it and r() must describe that new E-step."""
    d = data(capi, oracle, "ragged")
    em = make_em(capi, d, env)
    dense = make_em(capi, d, {"BAMM_NO_SPARSE": "1"})
    ref = RefEM(oracle, d)
    for e in (em, dense):
        e.set_model(d["v0"], d["vbg"], d["alpha"], 0.3)
    ref.set_model(d["v0"], 0.3)
    a, b = em.iterate(3), dense.iterate(3)
    assert a == b
    for _ in range(3):
        ref.estep()
        ref.mstep()
    ref.check_llh(a[0], "iterate(3)")
    ref.check_state(em.model(), em.counts(), em.q(), em.s(), "iterate(3)")
    llh = em.estep()
    assert llh == dense.estep()
    ref.estep(em.model(), em.q())
    ref.check_llh(llh, "estep after iterate(3)")
    r = em.r()
    assert np.array_equal(r, dense.r())
    ref.check_r(r, "estep after iterate(3)")
    ref.check_state(em.model(), em.counts(), em.q(), em.s(), "estep after iterate(3)")


def test_reuse_on_by_default(capi):
    """From 2^26 stored positions bound reuse is on without any switch. optimize(optimize_q=True) and the fused loop must give
    the bits of runs with BAMM_NO_BOUND_REUSE, and reuse must have taken the watch pass in each."""
    W, K, Kbg = 20, 4, 2
    codes, offsets, ppos, pkmer, sites, hostmodel = _planted(70000, 500, W, seed=11)
    assert int(offsets[-1]) >= 1 << 26
    ss = capi.SeqSet(codes.ravel(), offsets, 4, ppos, pkmer)
    del codes
    vbg = hostmodel.background_from_counts(ss.count_kmers(Kbg), 4, Kbg, hostmodel.default_bg_alpha(Kbg))
    alpha = hostmodel.default_motif_alpha(K, W)
    v0 = hostmodel.motif_from_sites(sites, 4, K, alpha, vbg)
    d = dict(ss=ss, W=W, K=K, Kbg=Kbg)
    on, off = make_em(capi, d, {}), make_em(capi, d, {"BAMM_NO_BOUND_REUSE": "1"})
    assert on.bound_reuse_info()["enabled"] and not off.bound_reuse_info()["enabled"]
    for em in (on, off):
        em.set_model(v0, vbg, alpha, 0.3)
    a, b = on.optimize(optimize_q=True), off.optimize(optimize_q=True)
    watch1 = on.bound_reuse_info()["watch"]
    print("optimize: %d iterations, %d watch passes" % (a["iterations"], watch1))
    assert watch1 >= 1
    for k in ("iterations", "llh", "vdiff", "qtrace", "v", "q"):
        assert np.array_equal(a[k], b[k]), k
    assert np.array_equal(on.counts(), off.counts())
    assert np.array_equal(on.r(0, 3000), off.r(0, 3000))
    for em in (on, off):
        em.set_model(v0, vbg, alpha, 0.3)
    assert on.iterate(12) == off.iterate(12)
    same_lists(on, off, "iterate(12)")
    print("iterate(12): %d watch passes" % (on.bound_reuse_info()["watch"] - watch1))
    assert on.bound_reuse_info()["watch"] > watch1
    assert np.array_equal(on.model(), off.model()) and np.array_equal(on.counts(), off.counts())
    assert np.array_equal(on.r(0, 3000), off.r(0, 3000))
