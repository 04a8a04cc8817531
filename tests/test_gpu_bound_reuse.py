"""GPU suite: bound reuse of the pruned E-step (DESIGN.md §4.1). With reuse on, an iteration whose bound tables moved little since
the last full bound pass re-bounds only the watch list of that pass; the candidate set is the full pass's by construction, so
model, counts, log likelihood and q must be BIT-identical to runs with BAMM_NO_BOUND_REUSE, iteration by iteration."""
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def capi():
    from bammmotif2_b200 import capi
    capi.load()
    assert capi.device_count() >= 1, "no CUDA device: the product has no CPU fallback"
    return capi


_DATA = {}


def data(name):
    """c3's plan at 40k sequences (W=20, K=4), order 5 (column passes of the exact product), W=8 (dense hold)."""
    if name not in _DATA:
        from bammmotif2_b200 import synth
        nseq, L0, W, K, Kbg = {"c3_40k": (40000, 500, 20, 4, 2), "k5_w20": (20000, 500, 20, 5, 2), "w8": (30000, 500, 8, 4, 2)}[name]
        fwd, sites, _ = synth.planted_sequences(7, nseq, L0, W)
        codes = synth.stored_both_strands(fwd)
        ppos, pkmer = synth.middle_n_patches(codes, 7)
        offsets = np.arange(nseq + 1, dtype=np.uint64) * np.uint64(codes.shape[1])
        _DATA[name] = dict(codes=codes, offsets=offsets, ppos=ppos, pkmer=pkmer, sites=sites, W=W, K=K, Kbg=Kbg)
    return _DATA[name]


def run(capi, name, env, iters=16, optimize_q=False, set_model_at=None, r_when=None):
    from bammmotif2_b200 import hostmodel
    d = data(name)
    keys = ("BAMM_NO_BOUND_REUSE", "BAMM_BOUND_REUSE", "BAMM_BOUND_SLACK", "BAMM_WATCH_FRAC")
    old = {k: os.environ.get(k) for k in keys}
    for k in keys:
        os.environ.pop(k, None)
    os.environ["BAMM_BOUND_REUSE"] = "1"             # these sets are below the size from which reuse is on by default
    os.environ.update(env)
    try:
        ss = capi.SeqSet(d["codes"].ravel(), d["offsets"], 4, d["ppos"], d["pkmer"])
        vbg = hostmodel.background_from_counts(ss.count_kmers(d["Kbg"]), 4, d["Kbg"], hostmodel.default_bg_alpha(d["Kbg"]))
        alpha = hostmodel.default_motif_alpha(d["K"], d["W"])
        v0 = hostmodel.motif_from_sites(d["sites"], 4, d["K"], alpha, vbg)
        em = capi.EM(ss, d["W"], d["K"], d["Kbg"])
        em.set_model(v0, vbg, alpha, 0.3)
        trace, r, r_it, watch_iters = [], None, None, 0
        for it in range(iters):
            if set_model_at == it:
                em.set_model(v0, vbg, alpha, 0.25)
            llh = em.estep()
            info = em.bound_reuse_info()
            watch_iters += int(info["last_watch"])
            if r_when is not None and r is None and r_when(it, info):
                r, r_it = em.r(), it
            q = em.optimize_q() if optimize_q else None
            em.mstep()
            trace.append((llh, q, em.model(), em.counts()))
        return dict(trace=trace, r=r, r_it=r_it, info=em.bound_reuse_info(), watch_iters=watch_iters, pruned=em.estep_info()["pruned"])
    finally:
        for k, v in old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


def assert_same(a, b):
    assert len(a["trace"]) == len(b["trace"])
    for it, (x, y) in enumerate(zip(a["trace"], b["trace"])):
        assert x[0] == y[0], ("llh", it)
        assert x[1] == y[1], ("q", it)
        assert np.array_equal(x[2], y[2]), ("model", it)
        assert np.array_equal(x[3], y[3]), ("counts", it)


@pytest.mark.parametrize("name,env", [("c3_40k", {}), ("k5_w20", {"BAMM_BOUND_SLACK": "6"})])      # (k5_w20 at slack 10: list > 1/4 of the windows)
def test_reuse_is_bit_identical(capi, name, env):
    off = run(capi, name, {"BAMM_NO_BOUND_REUSE": "1"})
    on = run(capi, name, env)
    assert off["pruned"] and not off["info"]["enabled"] and off["watch_iters"] == 0
    assert on["info"]["enabled"] and on["watch_iters"] >= 1, on["info"]
    assert_same(on, off)


@pytest.mark.parametrize("env,expect_watch", [({"BAMM_BOUND_SLACK": "0"}, False),                             # every pass a full one
                                              ({"BAMM_BOUND_SLACK": "30", "BAMM_WATCH_FRAC": "0.000001"}, False),  # the watch list overflows
                                              ({"BAMM_BOUND_SLACK": "5"}, True)])
def test_forced_branches(capi, env, expect_watch):
    off = run(capi, "c3_40k", {"BAMM_NO_BOUND_REUSE": "1"}, iters=10)
    on = run(capi, "c3_40k", env, iters=10)
    assert (on["watch_iters"] > 0) == expect_watch, on["info"]
    if not expect_watch:
        assert on["info"]["full"] >= 10
    assert_same(on, off)


def test_set_model_mid_run(capi):
    off = run(capi, "c3_40k", {"BAMM_NO_BOUND_REUSE": "1"}, iters=14, set_model_at=7)
    on = run(capi, "c3_40k", {}, iters=14, set_model_at=7)
    assert on["watch_iters"] >= 1
    assert_same(on, off)


def test_optimize_q(capi):
    off = run(capi, "c3_40k", {"BAMM_NO_BOUND_REUSE": "1"}, optimize_q=True)
    on = run(capi, "c3_40k", {}, optimize_q=True)
    assert len(set(t[1] for t in on["trace"])) > 1          # q moves, so the threshold moves
    assert_same(on, off)


def test_dense_hold_width_8(capi):
    off = run(capi, "w8", {"BAMM_NO_BOUND_REUSE": "1"}, iters=12)
    on = run(capi, "w8", {}, iters=12)
    assert_same(on, off)


def test_r_after_watch_pass(capi):
    on = run(capi, "c3_40k", {}, iters=10, r_when=lambda it, info: it >= 4 and info["last_watch"])
    assert on["r"] is not None, on["info"]
    off = run(capi, "c3_40k", {"BAMM_NO_BOUND_REUSE": "1"}, iters=10, r_when=lambda it, info: it == on["r_it"])
    assert np.array_equal(on["r"], off["r"])
    assert_same(on, off)
