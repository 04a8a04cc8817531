"""EM iteration and ZOOPS scoring time of motifs wider than 32 columns (index-array kernels in column blocks, DESIGN.md §4.6)
next to W = 24 / 32 on the same kernels (BAMM_NO_PACKED=1), on one device.

    python tools/wide_bench.py [--nseq 300000] [--L0 500] [--steps 5] [--out FILE]

Data: seeded planted sequences, both strands with the middle N (stored length 2 L0 + 1). Per (W, K): ms per EM iteration
from the host clock around bamm_em_iterate and from its CUDA events (bamm_em_loop_timing), positions x iterations per
second and ns per window x column. Then ZOOPS-only scoring of --score-nseq sequences at W = 48. Prints one JSON line per
measurement, the first one naming the card, its power limit and its maximum SM clock.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True

from bammmotif2_b200 import capi, hostmodel, synth  # noqa: E402

CASES = [(24, True), (32, True), (40, False), (48, False), (63, False)]     # (W, BAMM_NO_PACKED)


def card():
    q = "name,power.limit,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=" + q, "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.TimeoutExpired):
        out = ""
    return dict(zip(q.split(","), [s.strip() for s in out.split(",")])) if out else {"nvidia-smi": "unavailable"}


def make_set(seed, nseq, L0):
    fwd, _, _ = synth.planted_sequences(seed, nseq, L0, 12)
    codes = synth.stored_both_strands(fwd)
    ppos, pkmer = synth.middle_n_patches(codes, seed)
    offsets = np.arange(nseq + 1, dtype=np.uint64) * np.uint64(codes.shape[1])
    return capi.SeqSet(codes.ravel(), offsets, 4, ppos, pkmer), codes.shape[1]


def emit(rec, out):
    line = json.dumps(rec)
    print(line, flush=True)
    if out:
        out.write(line + "\n")
        out.flush()


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--nseq", type=int, default=300000)
    ap.add_argument("--L0", type=int, default=500)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--orders", default="2,4")
    ap.add_argument("--score-nseq", type=int, default=1000000)
    ap.add_argument("--score-L0", type=int, default=100)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    capi.load()
    if capi.device_count() < 1:
        raise SystemExit("wide_bench needs a CUDA device")
    out = open(a.out, "w") if a.out else None
    emit(dict(card=card(), nseq=a.nseq, L0=a.L0, steps=a.steps, warmup=a.warmup), out)
    ss, L = make_set(1, a.nseq, a.L0)
    Kbg = 2
    vbg = hostmodel.background_from_counts(ss.count_kmers(Kbg), 4, Kbg, hostmodel.default_bg_alpha(Kbg))
    rng = np.random.default_rng(5)
    for K in [int(k) for k in a.orders.split(",")]:
        for W, no_packed in CASES:
            alpha = hostmodel.default_motif_alpha(K, W)
            v0 = hostmodel.motif_from_sites(rng.integers(1, 5, size=(500, W), dtype=np.uint8), 4, K, alpha, vbg)
            if no_packed:
                os.environ["BAMM_NO_PACKED"] = "1"
            try:
                em = capi.EM(ss, W, K, Kbg)
            finally:
                os.environ.pop("BAMM_NO_PACKED", None)
            em.set_model(v0, vbg, alpha, 0.3)
            em.iterate(a.warmup)
            t0 = time.perf_counter()
            em.iterate(a.steps)
            wall = (time.perf_counter() - t0) * 1e3 / a.steps
            it, e_ms, m_ms, u_ms, tot_ms = em.loop_timing()
            ev = tot_ms / max(it, 1)
            windows = a.nseq * (L - W + 1)
            emit(dict(W=W, K=K, no_packed=no_packed, ms_per_iter_host=round(wall, 4), ms_per_iter_events=round(ev, 4),
                      estep_ms=round(e_ms / max(it, 1), 4), mstep_ms=round(m_ms / max(it, 1), 4), update_ms=round(u_ms / max(it, 1), 4),
                      positions_iter_per_s=float("%.4g" % (ss.npos / (ev * 1e-3))),
                      ns_per_window_column=round(ev * 1e6 / (windows * W), 5), launches=em.launch_count()), out)
            em.close()
    ss.close()
    # ZOOPS-only scoring at W = 48
    W, K = 48, 2
    sc, L = make_set(2, a.score_nseq, a.score_L0)
    vbg = hostmodel.background_from_counts(sc.count_kmers(Kbg), 4, Kbg, hostmodel.default_bg_alpha(Kbg))
    alpha = hostmodel.default_motif_alpha(K, W)
    v0 = hostmodel.motif_from_sites(rng.integers(1, 5, size=(500, W), dtype=np.uint8), 4, K, alpha, vbg)
    sc.score(W, K, Kbg, v0, vbg, want_mops=False)                                    # warm-up: index, module load
    kern, wall = [], []
    for _ in range(3):
        t0 = time.perf_counter()
        sc.score(W, K, Kbg, v0, vbg, want_mops=False)
        wall.append((time.perf_counter() - t0) * 1e3)
        kern.append(capi.score_last_ms())
    emit(dict(score_W=W, K=K, nseq=a.score_nseq, stored_L=L, zoops_kernel_ms_median=float(np.median(kern)),
              zoops_call_ms_median=round(float(np.median(wall)), 3),
              ns_per_window_column=round(float(np.median(kern)) * 1e6 / (a.score_nseq * (L - W + 1) * W), 5)), out)


if __name__ == "__main__":
    main()
