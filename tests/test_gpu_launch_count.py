"""GPU suite: bamm_em_launch_count (bench.py reports it as gpu_launches) counts exactly the kernels an EM object runs. For every
call the count must move by the number of kernels torch.profiler's CUDA activity trace records during that call (copies and
memsets are not kernels). Plans: c3's pruned E-step with bound reuse (two bound kernels per E-step); order 5 at W=20, pruned
with column passes and dense with column passes (one launch per pass for the E-step kernels and the tables of every update);
the six-letter alphabet (single-stranded) on the index-array row path; order 8 (32-bit k-mer indices) on the row path with
global count tables."""
import json
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

_KEYS = ("BAMM_BOUND_REUSE", "BAMM_NO_BOUND_REUSE", "BAMM_BOUND_SLACK", "BAMM_WATCH_FRAC", "BAMM_NO_SPARSE", "BAMM_CAND_FRAC")
#        name: (A, nseq, L0, W, K, K_bg, env at bamm_em_create)
PLANS = {"c3_40k_reuse": (4, 40000, 500, 20, 4, 2, {"BAMM_BOUND_REUSE": "1"}),
         "k5_w20_pruned": (4, 20000, 500, 20, 5, 2, {}),
         "k5_w20_dense": (4, 20000, 500, 20, 5, 2, {"BAMM_NO_SPARSE": "1"}),
         "a6_rows": (6, 3000, 300, 12, 5, 2, {}),
         "k8_rows_u32": (4, 3000, 300, 12, 8, 2, {})}


@pytest.fixture(scope="module")
def capi():
    from bammmotif2_b200 import capi
    capi.load()
    assert capi.device_count() >= 1, "no CUDA device: the product has no CPU fallback"
    return capi


def kernels_during(fn, trace_path):
    """(kernels the device ran while fn() ran, fn's result), from the profiler's trace (fn synchronises the EM object's stream)."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        out = fn()
    prof.export_chrome_trace(str(trace_path))
    with open(trace_path) as f:
        events = json.load(f)["traceEvents"]
    return sum(1 for e in events if e.get("cat") == "kernel"), out


def make_em(capi, name):
    from bammmotif2_b200 import hostmodel, synth
    A, nseq, L0, W, K, Kbg, env = PLANS[name]
    fwd, sites, _ = synth.planted_sequences(7, nseq, L0, W, A=A)
    if A == 4:
        codes = synth.stored_both_strands(fwd)
        ppos, pkmer = synth.middle_n_patches(codes, 7)
    else:                                                            # single-stranded records without an N
        codes, ppos, pkmer = fwd, None, None
    offsets = np.arange(nseq + 1, dtype=np.uint64) * np.uint64(codes.shape[1])
    ss = capi.SeqSet(codes.ravel(), offsets, A, ppos, pkmer)
    vbg = hostmodel.background_from_counts(ss.count_kmers(Kbg), A, Kbg, hostmodel.default_bg_alpha(Kbg))
    alpha = hostmodel.default_motif_alpha(K, W)
    v0 = hostmodel.motif_from_sites(sites, A, K, alpha, vbg)
    old = {k: os.environ.pop(k, None) for k in _KEYS}
    os.environ.update(env)
    try:
        em = capi.EM(ss, W, K, Kbg)
    finally:
        for k in _KEYS:
            os.environ.pop(k, None)
        os.environ.update({k: v for k, v in old.items() if v is not None})
    em.set_model(v0, vbg, alpha, 0.3)
    return ss, em


@pytest.mark.parametrize("name", list(PLANS))
def test_launch_count_matches_the_kernels_run(capi, name, tmp_path):
    import torch
    torch.cuda.init()
    kernels_during(lambda: None, tmp_path / "warmup.json")          # the profiler's own start-up is not part of any call
    ss, em = make_em(capi, name)
    info, wrong = None, []
    for call, fn in (("estep", em.estep), ("r", em.r), ("mstep", em.mstep), ("estep", em.estep), ("mstep", em.mstep),
                     ("iterate(2)", lambda: em.iterate(2))):
        before = em.launch_count()
        ran, _ = kernels_during(fn, tmp_path / "trace.json")
        counted = em.launch_count() - before
        assert ran > 0 or call == "r", (name, call)          # (r of the row path is already normalised: nothing to launch)
        if counted != ran:
            wrong.append((call, counted, ran))
        if info is None:
            info = em.estep_info()
    assert not wrong, (name, "(call, counted, ran)", wrong)
    # the plans are the ones named
    reuse = em.bound_reuse_info()["enabled"]
    if name.startswith("c3"):
        assert info["pruned"] and info["passes"] == 1 and reuse
    elif name == "k5_w20_pruned":
        assert info["pruned"] and info["passes"] > 1
    elif name == "k5_w20_dense":
        assert not info["pruned"] and info["passes"] > 1
    else:
        assert info["passes"] == 0
