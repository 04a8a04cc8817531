#!/usr/bin/env python
"""bench.py — throughput of the EM hot path (E-step + M-step + model update) on synthetic planted-motif data.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload c3|c2|tiny] [--impl reference] [--dump-outputs DIR]

A "step" is ONE EM iteration over the whole resident sequence set (E-step kernel, M-step accumulation kernel,
count reduction + Motif::updateV + next odds table). Metric: bp.iter/s = (sum of input bases L0) x iterations /
device time, order-K model on both strands (BASELINE.json). One process per GPU; under torchrun every rank holds
its own shard (weak scaling) and the per-iteration exchange is one NCCL all-reduce (SUM, int64) of the fixed-point
count table + 2 scalars, issued on the EM stream between the two halves of the iteration.

JSON keys follow the driver's contract; extra objects:
  roofline      dominant kernel vs the measured HBM copy bandwidth (MEASURED_PEAKS.json), algorithmic bytes 6 B/position/kernel
  cpu_baseline  the reference's own EStep/MStep (oracle/_ref/ref_time, all host threads) on a bounded sample, rank 0, N=1
  e2e           same metric through the C ABI from HOST buffers: upload + index build + K iterations + model read-back
`--impl reference` times only the CPU reference arm on the same workload definition (bounded sample per step).
`--dump-outputs DIR` writes what the last timed step returned as DIR/<name>.npy, so that two builds can be compared output for
output on the same seeded inputs. EM workloads: model (float32 v), counts (float32 n of the M-step), llh and vdiff (float32, one
value each), r_sample (float32 posteriors of a fixed, seeded sample of sequences, one row each) and r_sample_seqs (float64 indices
of those sequences). c4: zoops_pos / zoops_neg (float32 ZOOPS scores), argmax_pos / argmax_neg (float64 arg-max positions) and
rows_pos / rows_neg (float64 rows of the scored subsets they belong to; a seeded sample above one million rows per set).
"""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True      # no __pycache__ in the source tree, which may be read-only; outputs go to --dump-outputs DIR / temp dirs

from bammmotif2_b200 import synth  # noqa: E402
from bammmotif2_b200 import hostmodel  # noqa: E402
from bammmotif2_b200 import sharding  # noqa: E402

METRIC = "EM bp·iter/s (order-k, both strands)"
UNIT = "bp·iter/s"
Q = 0.3   # reference default prior (Global.cpp:52)


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None, help="timed steps (default 10); c5 and c4 --full time one whole CLI run instead")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--workload", default="c3", choices=sorted(synth.WORKLOADS))
    ap.add_argument("--nseq", type=int, default=0, help="override sequences per GPU (debug)")
    ap.add_argument("--K", type=int, default=-1, help="override the motif order (sweeps; the workload name gains a suffix)")
    ap.add_argument("--W", type=int, default=0, help="override the motif width (sweeps)")
    ap.add_argument("--L0", type=int, default=0, help="override the sequence length (sweeps)")
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--seed", type=int, default=1234)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--full", action="store_true", help="workload c4: the WHOLE --FDR run through the drop-in CLI (bin/BaMMmotif) instead of one fold's scoring")
    ap.add_argument("--no-strong", action="store_true", help="N > 1: skip the strong-scaling run (one set split over the ranks)")
    ap.add_argument("--cpu-sample", type=int, default=0, help="sequences in the CPU sample (default by workload)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step as DIR/<name>.npy (see the module docstring)")
    args = ap.parse_args()
    whole_run = args.workload == "c5" or (args.workload == "c4" and args.full)
    if whole_run and args.steps is not None:
        ap.error("--steps does not apply to --workload c5 or c4 --full: they time one whole command-line run")
    if args.steps is None:
        args.steps = 10
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "b200" or whole_run):
        ap.error("--dump-outputs writes the outputs of the timed device path (--workload c2, c3, tiny or c4 without --full)")
    return args


DUMP_SAMPLE_SEQS = 1024
DUMP_SAMPLE_BYTES = 32 << 20
DUMP_SCORES_PER_SET = 1_000_000


def dump_scores(out_dir, pos, neg):
    """c4: the ZOOPS scores (float32) and arg-max positions (float64) a caller of the timed step receives for the positive and
    the negative subset, each with the subset rows they belong to (float64); a set above DUMP_SCORES_PER_SET is a seeded sample."""
    os.makedirs(out_dir, exist_ok=True)
    for name, (zoops, z) in (("pos", pos), ("neg", neg)):
        rows = np.arange(len(zoops))
        if len(rows) > DUMP_SCORES_PER_SET:
            rows = np.sort(np.random.default_rng(0).choice(len(rows), size=DUMP_SCORES_PER_SET, replace=False))
        np.save(os.path.join(out_dir, "zoops_%s.npy" % name), zoops[rows].astype(np.float32))
        np.save(os.path.join(out_dir, "argmax_%s.npy" % name), z[rows].astype(np.float64))
        np.save(os.path.join(out_dir, "rows_%s.npy" % name), rows.astype(np.float64))


def dump_outputs(out_dir, em):
    """Writes the arrays a caller of the timed loop receives after its last iteration (bamm_em_iterate's llh / sum|dv|,
    bamm_em_get_model, bamm_em_get_counts, bamm_em_get_r) as float32 / float64 .npy files; r only for a seeded sample of
    sequences (every sequence of a bench set has the same length, so the sample is one row per sequence).
    Call it after the loop timings have been read: em.iterate(0) re-reads the last iteration's scalars and resets the timings."""
    from bammmotif2_b200 import capi
    os.makedirs(out_dir, exist_ok=True)
    llh, vdiff = em.iterate(0)
    nseq = em.nsub
    rsize = int(capi.load().bamm_em_r_size(em.h))
    assert rsize % nseq == 0, "sequences of unequal length"
    per_seq = rsize // nseq
    n = max(1, min(nseq, DUMP_SAMPLE_SEQS, DUMP_SAMPLE_BYTES // (4 * per_seq)))
    seqs = np.sort(np.random.default_rng(0).choice(nseq, size=n, replace=False))
    r = np.empty((n, per_seq), np.float32)
    for i, s in enumerate(seqs):
        capi._check(capi.load().bamm_em_get_r(em.h, int(s), 1, r[i].ctypes.data_as(capi._f32p)))
    arrays = {"model": em.model(), "counts": em.counts(), "llh": np.array([llh], np.float32), "vdiff": np.array([vdiff], np.float32),
              "r_sample": r, "r_sample_seqs": seqs.astype(np.float64)}
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def measured_traffic(workload, nseq, mstep_dominant):
    """DRAM bytes per iteration of the dominant phase (all its kernels) from the committed ncu --set full capture
    (profiles/traffic.json, written by tools/ncu_traffic.py); only valid for the workload and size that capture was taken on."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    try:
        t = json.load(open(p))
        if t.get("workload") == workload and int(t.get("nseq", -1)) == int(nseq):
            return t["mstep_bytes" if mstep_dominant else "estep_bytes"]
    except Exception:
        pass
    return None


class ClockSampler:
    """SM clock / throttle reasons while the timed region runs: NVML polled every 2 ms on a thread (plus one sample when the
    region starts and one when it ends, so that even a 4 ms region has two); nvidia-smi every 200 ms where NVML is missing."""

    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.index = index
        self.proc = None
        self.lines = []

    NVML_REASONS = ((0x8, "hw_slowdown"), (0x40, "hw_thermal_slowdown"), (0x20, "sw_thermal_slowdown"), (0x4, "sw_power_cap"))

    def _nvml_sample(self):
        n = self.nvml
        self.nv_sm.append(float(n.nvmlDeviceGetClockInfo(self.nv_h, n.NVML_CLOCK_SM)))
        bits = int(n.nvmlDeviceGetCurrentClocksThrottleReasons(self.nv_h))
        for bit, name in self.NVML_REASONS:
            if bits & bit:
                self.nv_reasons.add(name)

    def _nvml_loop(self):
        while not self.nv_stop.is_set():
            try:
                self._nvml_sample()
            except Exception:
                return
            self.nv_stop.wait(0.002)

    def _start_nvml(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nvml = pynvml
            self.nv_h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self.nv_max = float(pynvml.nvmlDeviceGetMaxClockInfo(self.nv_h, pynvml.NVML_CLOCK_SM))
            self.nv_sm, self.nv_reasons, self.nv_stop = [], set(), threading.Event()
            self._nvml_sample()
            self.nv_t = threading.Thread(target=self._nvml_loop, daemon=True)
            self.nv_t.start()
            return True
        except Exception:
            self.nvml = None
            return False

    def start(self):
        self.nvml = None
        if self._start_nvml():
            return
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.nvml is not None:
            self.nv_stop.set()
            self.nv_t.join(timeout=1)
            try:
                self._nvml_sample()
            except Exception:
                pass
            sm = sorted(self.nv_sm)
            return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": self.nv_max, "samples": len(sm),
                    "reasons": sorted(self.nv_reasons), "source": "nvml, 2 ms"}
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for l in self.lines:
            t = [x.strip() for x in l.split(",")]
            if len(t) < 7:
                continue
            try:
                sm.append(float(t[0])); mx = float(t[1])
            except ValueError:
                continue
            for nm, val in zip(names, t[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(nm)
        sm_sorted = sorted(sm)
        return {"sm_mhz": sm_sorted[len(sm_sorted) // 2] if sm else None, "sm_max_mhz": mx,
                "samples": len(sm), "reasons": sorted(reasons)}


def make_data(wl, nseq, seed, pinned=False, motif_seed=None):
    """Returns dict(codes [nseq, L] uint8 (optionally pinned), offsets, patches, sites, fwd)."""
    fwd, sites, _ = synth.planted_sequences(seed, nseq, wl["L0"], wl["W"], motif_seed=motif_seed)
    L = 2 * wl["L0"] + 1
    out = None
    if pinned:
        import torch
        out = torch.empty((nseq, L), dtype=torch.uint8, pin_memory=True).numpy()
    codes = synth.stored_both_strands(fwd, out=out)
    ppos, pkmer = synth.middle_n_patches(codes, seed)
    if pinned:                                   # every input of the end-to-end path starts in pinned host memory
        import torch
        pp = torch.empty(len(ppos), dtype=torch.int64, pin_memory=True).numpy().view(np.uint64)
        pk = torch.empty(len(pkmer), dtype=torch.int64, pin_memory=True).numpy().view(np.uint64)
        pp[:] = ppos; pk[:] = pkmer
        ppos, pkmer = pp, pk
    offsets = np.arange(nseq + 1, dtype=np.uint64) * np.uint64(L)
    return dict(codes=codes, offsets=offsets, ppos=ppos, pkmer=pkmer, sites=sites, fwd=fwd, L=L)


def initial_model(capi, ss, wl, sites, reduce_counts=None):
    """Background model from device k-mer counts (BackgroundModel.cpp:26-42, 441-472) + binding-site init.
    reduce_counts: sums the count vector over ranks, so that every shard starts from the same model."""
    A = 4
    n = ss.count_kmers(wl["K_bg"])
    if reduce_counts is not None:
        n = reduce_counts(n)
    vbg = hostmodel.background_from_counts(n, A, wl["K_bg"], hostmodel.default_bg_alpha(wl["K_bg"]))
    alpha = hostmodel.default_motif_alpha(wl["K"], wl["W"])
    v0 = hostmodel.motif_from_sites(sites, A, wl["K"], alpha, vbg)
    return v0, vbg, alpha


def cpu_reference_run(wl, sample_nseq, seed, steps, warmup, threads):
    """Runs the reference's own EStep/MStep (oracle/_ref/ref_time) on a bounded sample; falls back to the oracle
    port (same OpenMP structure) when the reference build is not there. Returns dict for the JSON line."""
    fwd, sites, _ = synth.planted_sequences(seed, sample_nseq, wl["L0"], wl["W"])
    bp = int(fwd.size)
    exe = os.path.join(ROOT, "oracle", "_ref", "ref_time")
    sample = "%d x %d bp sample of %s (same generator, seed %d), W=%d K=%d, %d timed iterations" % (
        sample_nseq, wl["L0"], wl["name"], seed, wl["W"], wl["K"], steps)
    if os.path.exists(exe):
        tmp = tempfile.mkdtemp(prefix="bamm_cpu_")
        fa, bs = os.path.join(tmp, "s.fasta"), os.path.join(tmp, "sites.block")
        synth.write_fasta(fa, fwd)
        synth.write_sites(bs, sites)
        env = dict(os.environ, BAMM_TIME_ITERS=str(steps), BAMM_TIME_WARMUP=str(warmup), OMP_NUM_THREADS=str(threads))
        cmd = [exe, tmp, fa, "--bindingSiteFile", bs, "--EM", "-k", str(wl["K"]), "-K", str(wl["K_bg"]), "--threads", str(threads)]
        out = subprocess.run(cmd, env=env, stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, check=True).stdout
        res = json.loads(out.strip().splitlines()[-1])
        per_iter = res["per_iter_s"]
        import shutil
        shutil.rmtree(tmp, ignore_errors=True)
        return dict(kind="reference", cores=threads, sample=sample, bp=bp, per_iter_s=per_iter,
                    estep_s=res["estep_s"], mstep_s=res["mstep_s"], value=bp * len(per_iter) / sum(per_iter))
    # port: oracle restatement with the reference's OpenMP structure
    from oracle import oracle as orc
    codes = synth.stored_both_strands(fwd)
    ppos, pkmer = synth.middle_n_patches(codes, seed)
    kmer = synth.full_kmers(codes, ppos, pkmer)
    offsets = np.arange(sample_nseq + 1, dtype=np.uint64) * np.uint64(codes.shape[1])
    A = 4
    nb, vbg = orc.bg_model(kmer, A, wl["K_bg"], hostmodel.default_bg_alpha(wl["K_bg"]))
    alpha = hostmodel.default_motif_alpha(wl["K"], wl["W"])
    v = hostmodel.motif_from_sites(sites, A, wl["K"], alpha, vbg)
    r = np.zeros(len(kmer), np.float32)
    n_all = np.zeros(orc.model_size(A, wl["K"], wl["W"]), np.float32)
    per_iter = []
    for it in range(warmup + steps):
        s = orc.linear_s(v, vbg, A, wl["K"], min(wl["K"], wl["K_bg"]), wl["W"])
        t0 = time.perf_counter()
        orc.em_iteration_omp(kmer, offsets, A, wl["K"], wl["W"], s, Q, r, n_all, threads)
        dt = time.perf_counter() - t0
        orc.update_v(n_all, alpha.ravel(), vbg, A, wl["K"], wl["W"], v)
        if it >= warmup:
            per_iter.append(dt)
    return dict(kind="port", cores=threads, sample=sample, bp=bp, per_iter_s=per_iter,
                value=bp * len(per_iter) / sum(per_iter))


def run_reference_arm(args, wl, rank):
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    sample = args.cpu_sample or wl["cpu_sample"]
    t0 = time.perf_counter()
    res = cpu_reference_run(wl, sample, args.seed, args.steps, max(args.warmup, 1), threads)
    wall = time.perf_counter() - t0
    ms = 1e3 * sum(res["per_iter_s"]) / len(res["per_iter_s"])
    line = {
        "impl": "reference", "metric": METRIC, "value": res["value"], "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": wl["desc"], "W": wl["W"], "K": wl["K"], "K_bg": wl["K_bg"], "step": "one EM iteration on the CPU sample",
                   "sample_nseq": sample, "seed": args.seed},
        "cpu_baseline": {"value": res["value"], "unit": UNIT, "cores": res["cores"], "kind": res["kind"], "sample": res["sample"]},
        "e2e": {"value": res["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "wall_s": wall,
    }
    print(json.dumps(line), flush=True)


# ---- config 4: the FDR data path (negative sampling + scoring) -------------------------------------------------------
C4_METRIC = "FDR scoring sequences/s (order-3, ZOOPS, one cross-validation fold)"
C4_UNIT = "sequences/s"


def c4_reference(wl, sample_nseq, seed, steps, warmup):
    """The reference's own negative sampling + ScoreSeqSet::calcLogOdds (serial in the reference, ScoreSeqSet.cpp:40) on a
    bounded sample of the positives with the same mFold (oracle/_ref/ref_time, BAMM_TIME_MODE=fdr)."""
    exe = os.path.join(ROOT, "oracle", "_ref", "ref_time")
    if not os.path.exists(exe):
        raise RuntimeError("oracle/_ref/ref_time is not built")
    fwd, sites, _ = synth.planted_sequences(seed, sample_nseq, wl["L0"], wl["W"])
    tmp = tempfile.mkdtemp(prefix="bamm_cpu_")
    fa, bs = os.path.join(tmp, "s.fasta"), os.path.join(tmp, "sites.block")
    synth.write_fasta(fa, fwd)
    synth.write_sites(bs, sites)
    env = dict(os.environ, BAMM_TIME_ITERS=str(steps), BAMM_TIME_WARMUP=str(warmup), BAMM_TIME_MODE="fdr", OMP_NUM_THREADS="1")
    cmd = [exe, tmp, fa, "--bindingSiteFile", bs, "--EM", "-k", str(wl["K"]), "-K", str(wl["K_bg"]), "-m", str(wl["mfold"]), "--threads", "1"]
    out = subprocess.run(cmd, env=env, stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, check=True).stdout
    import shutil
    shutil.rmtree(tmp, ignore_errors=True)
    res = json.loads(out.strip().splitlines()[-1])
    nseq_scored = res["npos_seq"] + res["nneg_seq"]
    per = res["per_iter_s"]
    return dict(kind="reference", cores=1, value=nseq_scored * len(per) / sum(per), per_iter_s=per,
                positions_per_s=res["positions_scored"] * len(per) / sum(per),
                neg_bases_per_s=(res["positions_scored"] - res["npos_seq"] * (2 * wl["L0"] + 1)) / res["sample_neg_s"],
                sample="%d x %d bp positives + %d sampled negatives (mFold %d; the reference raises mFold for sets below 5000 "
                       "sequences, mainBaMM.cpp:102-106), W=%d K=%d, calcLogOdds of all of them, %d timed passes, 1 thread "
                       "(the reference scores serially)" % (res["npos_seq"], wl["L0"], res["nneg_seq"], res["mfold"], wl["W"], wl["K"], len(per)))


C4F_METRIC = "FDR cross-validation sequences/s (whole --FDR run of the CLI: 5 folds of EM + scoring, 10x negatives, statistics, files)"


def run_c4_full(args, wl):
    """BASELINE.json configs[3] end to end through the drop-in command line (reference: mainBaMM.cpp:119-170 -> FDR::evaluateMotif,
    src/evaluation/FDR.cpp:28-145, calculatePR :147-276, write): FASTA in, .zoops.stats out. One process; --gpus N hands it N devices
    (BAMM_DEVICES: EM::optimize of every fold is split over them). value = (positives + sampled negatives scored) / wall seconds.
    --impl reference: the reference's own binary (oracle/_ref/BaMMmotif_ref, all host threads) on a bounded sample."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    ref = args.impl == "reference"
    nseq = args.nseq or (args.cpu_sample or 5_000 if ref else wl["nseq"])
    exe = os.path.join(ROOT, "oracle", "_ref", "BaMMmotif_ref") if ref else os.path.join(ROOT, "bammmotif2_b200", "bin", "BaMMmotif")
    if not os.path.exists(exe):
        raise SystemExit("%s is not built" % exe)
    tmp = tempfile.mkdtemp(prefix="bamm_c4_")
    t0 = time.perf_counter()
    fwd, sites, _ = synth.planted_sequences(args.seed, nseq, wl["L0"], wl["W"])
    fa, bs, out = os.path.join(tmp, "in.fasta"), os.path.join(tmp, "sites.block"), os.path.join(tmp, "out")
    synth.write_fasta(fa, fwd)
    synth.write_sites(bs, sites)
    os.makedirs(out)
    t_gen = time.perf_counter() - t0
    cmd = [exe, out, fa, "--bindingSiteFile", bs, "--EM", "-k", str(wl["K"]), "-K", str(wl["K_bg"]), "--FDR", "-m", str(wl["mfold"]), "-n", str(wl["cvfold"])]
    env = dict(os.environ)
    if ref:
        cmd += ["--threads", str(os.cpu_count() or 1)]
    else:
        env.update(BAMM_DEVICES=",".join(str(d) for d in range(max(args.gpus, 1))), BAMM_TRACE="1")
    t0 = time.perf_counter()
    p = subprocess.run(cmd, env=env, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)
    wall = time.perf_counter() - t0
    if p.returncode != 0:
        raise SystemExit("CLI failed: %s" % p.stderr[-500:])
    stages = {}
    for l in p.stderr.splitlines():
        if l.startswith("[bamm host] ") and l.rstrip().endswith(" ms"):
            t = l[len("[bamm host] "):].rsplit(" ", 2)
            stages[t[0]] = float(t[1])
    mfold = wl["mfold"]
    for l in p.stdout.splitlines():                 # the reference raises mFold for small sets (mainBaMM.cpp:102-106)
        if "mFold" in l and "=" in l:
            try: mfold = int(l.split("=")[-1].strip())
            except ValueError: pass
    stats = [f for f in os.listdir(out) if f.endswith(".zoops.stats")]
    head = open(os.path.join(out, stats[0])).readline().split() if stats else []
    scored = nseq // wl["cvfold"] * wl["cvfold"] + nseq * mfold // wl["cvfold"] * wl["cvfold"]
    import shutil
    shutil.rmtree(tmp, ignore_errors=True)
    value = scored / wall
    gpu_s = sum(v for k, v in stages.items() if k in ("negative set", "EM", "FDR folds")) * 1e-3
    line = {"metric": C4F_METRIC, "value": value, "unit": C4_UNIT, "n_gpus": args.gpus, "steps": 1, "warmup": 0, "ms_per_step": wall * 1e3,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": "synthetic %d x %d bp positives, --EM -k %d -K %d --FDR -m %d -n %d through the command line (FASTA in, files out)" % (
                           nseq, wl["L0"], wl["K"], wl["K_bg"], mfold, wl["cvfold"]),
                       "sequences_scored": scored, "wall_s": wall, "fasta_written_s": t_gen, "stages_ms": stages or None,
                       "device_path_s": gpu_s if stages else None, "occurrence_fraction": float(head[-1]) if head else None, "seed": args.seed,
                       "note": "wall clock of the whole process; the device path (negative sampling + EM + 5 folds of EM and scoring) is device_path_s, "
                               "the rest is FASTA parsing and the 11-million-line statistics file on the host"},
            "e2e": {"value": value, "unit": C4_UNIT, "h2d_bytes_per_step": int(nseq * (2 * wl["L0"] + 1)) if not ref else 0, "d2h_bytes_per_step": int(12 * scored) if not ref else 0,
                    "seconds": wall, "what": "the same run: this workload is end to end by construction"},
            "gpu_launches": None if ref else "not counted (separate process)"}
    if ref:
        line.update({"impl": "reference", "gpu_launches": 0,
                     "cpu_baseline": {"value": value, "unit": C4_UNIT, "cores": os.cpu_count(), "kind": "reference",
                                      "sample": "%d x %d bp positives, mFold %d (the reference raises it for sets below 5000 sequences), its own binary" % (nseq, wl["L0"], mfold)}})
    print(json.dumps(line), flush=True)
    return 0


def run_c5(args, wl):
    """BASELINE.json configs[4] through the drop-in command line: --PWMFile (the reference's shipped PWM_peng10.meme: six motifs,
    Motif::initFromPWM, src/init/Motif.cpp:192-333, incl. its alength quirk) --EM -k 5 --alphabet EXTENDED, one EM::optimize per
    motif (mainBaMM.cpp:119-170). The 6-letter alphabet runs on the index-array kernels (csrc/kernels.cuh). value = input bases x EM
    iterations of all motifs / seconds in EM::optimize; e2e = the same over the wall clock of the process."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    ref = args.impl == "reference"
    nseq = args.nseq or ((args.cpu_sample or 1_000) if ref else wl["nseq"])
    exe = os.path.join(ROOT, "oracle", "_ref", "BaMMmotif_ref") if ref else os.path.join(ROOT, "bammmotif2_b200", "bin", "BaMMmotif")
    if not os.path.exists(exe):
        raise SystemExit("%s is not built" % exe)
    tmp = tempfile.mkdtemp(prefix="bamm_c5_")
    fwd, _, _ = synth.planted_sequences(args.seed, nseq, wl["L0"], wl["W"])
    fa, meme, out = os.path.join(tmp, "in.fasta"), os.path.join(tmp, "pwm.meme"), os.path.join(tmp, "out")
    synth.write_fasta(fa, fwd)
    # the reference's example/PWM_peng10.meme travels inside a test fixture (tests/golden/jund_pwm_k1.npz, made by oracle/make_golden.py)
    open(meme, "wb").write(bytes(np.load(os.path.join(ROOT, "tests", "golden", "jund_pwm_k1.npz"))["sites_text"]))
    os.makedirs(out)
    nmotif = 6
    cmd = [exe, out, fa, "--PWMFile", meme, "--maxPWM", str(nmotif), "--EM", "-k", str(wl["K"]), "-K", str(wl["K_bg"]), "--alphabet", "EXTENDED", "--verbose"]
    env = dict(os.environ)
    if ref:
        cmd += ["--threads", str(os.cpu_count() or 1)]
    else:
        env.update(BAMM_DEVICES=",".join(str(d) for d in range(max(args.gpus, 1))), BAMM_TRACE="1")
    t0 = time.perf_counter()
    p = subprocess.run(cmd, env=env, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)
    wall = time.perf_counter() - t0
    if p.returncode != 0:
        raise SystemExit("CLI failed: %s" % p.stderr[-500:])
    stages = {}
    for l in p.stderr.splitlines():                 # BAMM_TRACE lines of the driver: wall time per stage (summed when a stage repeats)
        if l.startswith("[bamm host] ") and l.rstrip().endswith(" ms") and "FASTA reader" not in l:
            t = l[len("[bamm host] "):].rsplit(" ", 2)
            stages[t[0]] = stages.get(t[0], 0.0) + float(t[1])
    iters = sum(1 for l in p.stdout.splitlines() if " iter, llh=" in l)
    em_s = sum(float(l.split("Runtime for EM:")[1].split("seconds")[0]) for l in p.stdout.splitlines() if "Runtime for EM:" in l)
    import shutil
    shutil.rmtree(tmp, ignore_errors=True)
    bp = nseq * wl["L0"]
    value = bp * iters / em_s if em_s > 0 else 0.0
    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": iters, "warmup": 0, "ms_per_step": em_s / max(iters, 1) * 1e3,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": wl["desc"], "nseq": nseq, "L0": wl["L0"], "K": wl["K"], "K_bg": wl["K_bg"], "alphabet": "EXTENDED (A=6)", "motifs": nmotif,
                       "em_iterations_all_motifs": iters, "stages_ms": stages or None, "em_seconds": em_s, "wall_s": wall, "seed": args.seed,
                       "positions_iter_per_s": nseq * (2 * wl["L0"] + 1) * iters / em_s if em_s > 0 else 0.0,
                       "step": "one EM iteration of one motif (EM::optimize until the reference's stop rule, six motifs one after the other)"},
            "e2e": {"value": bp * iters / wall, "unit": UNIT, "h2d_bytes_per_step": int(nseq * (2 * wl["L0"] + 1) / max(iters, 1)) if not ref else 0,
                    "d2h_bytes_per_step": 20 if not ref else 0, "seconds": wall, "what": "FASTA in, six .ihbcp files out: wall clock of the whole process"},
            "gpu_launches": None if ref else "not counted (separate process)"}
    if ref:
        line.update({"impl": "reference", "gpu_launches": 0,
                     "cpu_baseline": {"value": value, "unit": UNIT, "cores": os.cpu_count(), "kind": "reference",
                                      "sample": "%d x %d bp, same command line, the reference's own binary" % (nseq, wl["L0"])}})
    print(json.dumps(line), flush=True)
    return 0


def run_c4(args, wl):
    if args.full:
        return run_c4_full(args, wl)
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    cpu_sample = args.cpu_sample or 2_000
    if args.impl == "reference":
        if rank != 0:
            return 0
        t0 = time.perf_counter()
        res = c4_reference(wl, cpu_sample, args.seed, args.steps, max(args.warmup, 1))
        print(json.dumps({
            "impl": "reference", "metric": C4_METRIC, "value": res["value"], "unit": C4_UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * sum(res["per_iter_s"]) / len(res["per_iter_s"]), "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": wl["desc"], "W": wl["W"], "K": wl["K"], "K_bg": wl["K_bg"], "positions_scored_per_s": res["positions_per_s"],
                       "negative_bases_sampled_per_s": res["neg_bases_per_s"]},
            "cpu_baseline": {"value": res["value"], "unit": C4_UNIT, "cores": 1, "kind": "reference", "sample": res["sample"]},
            "e2e": {"value": res["value"], "unit": C4_UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0, "wall_s": time.perf_counter() - t0}), flush=True)
        return 0
    import torch
    import torch.distributed as dist
    from bammmotif2_b200 import capi
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback)")
    torch.cuda.set_device(local_rank)
    capi._check(capi.load().bamm_set_device(local_rank))
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", local_rank))
    nseq = args.nseq or wl["nseq"]
    A, W, K, Kbg, mfold, cv = 4, wl["W"], wl["K"], wl["K_bg"], wl["mfold"], wl["cvfold"]
    data = make_data(wl, nseq, args.seed + 1000 * rank, pinned=True, motif_seed=args.seed if world > 1 else None)
    L = data["L"]
    ss = capi.SeqSet(data["codes"].reshape(-1), data["offsets"], A, data["ppos"], data["pkmer"])
    v0, vbg, alpha = initial_model(capi, ss, wl, data["sites"], None)
    em = capi.EM(ss, W, K, Kbg)
    em.set_model(v0, vbg, alpha, Q)
    em.iterate(3)                                       # a few EM iterations: the model a fold would score with
    v = em.model()
    em.close()
    # negative set on the device (bit-identical to the reference's host sampler)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    if world > 1:
        # shards of ONE negative set: set-wide k-mer counts summed over the ranks, every rank starts at its draw offset, so
        # the union of the shards is the set a single device (and the reference) samples for the union of the positives
        cnt = torch.from_numpy(ss.negative_kmer_counts().astype(np.int64)).cuda()
        dist.all_reduce(cnt, op=dist.ReduceOp.SUM)
        neg = ss.sample_negatives_shard(mfold, rank * nseq * L * mfold, cnt.cpu().numpy().astype(np.uint64))
    else:
        neg = ss.sample_negatives(mfold)
    torch.cuda.synchronize()
    t_neg = time.perf_counter() - t0
    # one fold: its share of the positives (FDR.cpp:49-57) and every cv-th negative (FDR.cpp:58-60)
    n_fold = nseq // cv
    def pinned(arr):
        t = torch.empty(arr.shape, dtype={np.dtype(np.uint64): torch.int64, np.dtype(np.float32): torch.float32}[arr.dtype], pin_memory=True)
        out = t.numpy().view(arr.dtype)
        out[...] = arr
        return out

    # inputs (subset ids) and results (ZOOPS score + arg-max per sequence) live in pinned host memory
    pos_sub = pinned(np.arange(0, n_fold, dtype=np.uint64))
    neg_sub = pinned(np.arange(0, neg.nseq, cv, dtype=np.uint64))
    out_pos = (pinned(np.zeros(len(pos_sub), np.float32)), pinned(np.zeros(len(pos_sub), np.uint64)))
    out_neg = (pinned(np.zeros(len(neg_sub), np.float32)), pinned(np.zeros(len(neg_sub), np.uint64)))
    nscored = len(pos_sub) + len(neg_sub)
    positions = nscored * L
    launches = 0

    def step():
        nonlocal launches
        _, zp, _ = ss.score(W, K, Kbg, v, vbg, subset=pos_sub, want_mops=False, out=out_pos)
        k1 = capi.score_last_ms()
        _, zn, _ = neg.score(W, K, Kbg, v, vbg, subset=neg_sub, want_mops=False, out=out_neg)
        launches += 4                                   # group-table + scoring kernel per call
        return k1 + capi.score_last_ms(), zp, zn

    for _ in range(args.warmup):
        step()
    sampler = ClockSampler(local_rank)
    sampler.start()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    kernel_ms, t0 = 0.0, time.perf_counter()
    for _ in range(args.steps):
        ms, zp, zn = step()
        kernel_ms += ms
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    clocks = sampler.stop()
    if args.dump_outputs and rank == 0:
        dump_scores(args.dump_outputs, out_pos, out_neg)
    if world > 1:
        t = torch.tensor([kernel_ms, wall], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        kernel_ms, wall = float(t[0].item()), float(t[1].item())
    peak, peak_src = peaks()
    value = nscored * world * args.steps / (kernel_ms * 1e-3)
    e2e_value = nscored * world * args.steps / wall
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        try:
            res = c4_reference(wl, cpu_sample, args.seed, 2, 1)
            cpu = {"value": res["value"], "unit": C4_UNIT, "cores": 1, "kind": "reference", "sample": res["sample"],
                   "positions_scored_per_s": res["positions_per_s"], "negative_bases_sampled_per_s": res["neg_bases_per_s"]}
        except Exception as ex:   # noqa: BLE001
            cpu = {"value": None, "unit": C4_UNIT, "cores": 1, "kind": "unavailable", "sample": str(ex)[:200]}
    if rank == 0:
        alg = 2.0 * positions                                  # SURVEY.md §8d: ZOOPS-only scoring reads the 2 B index per position
        ach = alg / (kernel_ms / args.steps * 1e-3) / 1e9
        print(json.dumps({
            "metric": C4_METRIC, "value": value, "unit": C4_UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": kernel_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic",
            "config": {"workload": wl["desc"], "positives_per_gpu": nseq, "negatives_per_gpu": neg.nseq, "L_stored": L, "W": W, "K": K, "K_bg": Kbg,
                       "mfold": mfold, "cvfold": cv, "sequences_scored_per_step": nscored, "positions_scored_per_s": positions * world * args.steps / (kernel_ms * 1e-3),
                       "negative_sampling": {"seconds": t_neg, "bases_per_s": neg.npos / t_neg,
                                             "what": "bamm_seqset_sample_negatives: k-mer counts, per-template models, rand() jump-ahead, sampling, classification + 2-bit packing"},
                       "l2": "inputs (%.1f GB packed bases per step) exceed the 126 MB L2" % (positions / 4 / 1e9), "seed": args.seed,
                       "step": "bamm_score_logodds of one fold's test positives + every %d-th negative (ZOOPS max + argmax per sequence)" % cv},
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": C4_UNIT, "h2d_bytes_per_step": int(8 * nscored + 4 * (len(v) + len(vbg))),
                    "d2h_bytes_per_step": int(12 * nscored), "seconds": wall,
                    "what": "the same calls timed on the host clock: subset ids + model H2D, table build, kernels, ZOOPS scores + argmax D2H"},
            "gpu_launches": launches,
            "roofline": {"bound": "hbm", "kernel": "k_score_zoops_packed", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                         "traffic": None, "peak_source": peak_src, "algorithmic_bytes_per_launch": alg,
                         "note": "issue-bound: column-group bound per window (G shared-memory lookups) + exact ascending-j re-scoring of the "
                                 "few windows near the maximum; the scores stay bit-identical to the reference"},
            "cpu_baseline": cpu}), flush=True)
    neg.close(); ss.close()
    if world > 1:
        dist.destroy_process_group()
    return 0


def bind_near_gpu(torch, local_rank):
    """N > 1: run this rank's host thread on the CPUs of the NUMA node its GPU hangs off, BEFORE the pinned input buffers are
    allocated (first touch puts their pages on that node), so that eight concurrent 1.2 GB uploads do not all cross the socket
    link. Returns the node, or None when the topology is not visible (single node, container without /sys, no permission)."""
    try:
        pr = torch.cuda.get_device_properties(local_rank)
        bus = "%04x:%02x:%02x.0" % (pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id)
        node = int(open("/sys/bus/pci/devices/%s/numa_node" % bus).read())
        if node < 0:
            return None
        cpus = set()
        for part in open("/sys/devices/system/node/node%d/cpulist" % node).read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        cpus &= os.sched_getaffinity(0)
        if not cpus:
            return None
        os.sched_setaffinity(0, cpus)
        return node
    except Exception:
        return None


def main():
    args = parse_args()
    wl = dict(synth.WORKLOADS[args.workload], name=args.workload)
    if args.workload == "c4":
        return run_c4(args, wl)
    if args.workload == "c5":
        return run_c5(args, wl)
    wl["cpu_sample"] = {"c3": 40_000, "c2": 50_000, "tiny": 2_000}[args.workload]
    if args.K >= 0 or args.W or args.L0:              # sweep variants are labelled as such: not a BASELINE.json config
        if args.K >= 0: wl["K"] = args.K; wl["K_bg"] = min(wl["K_bg"], args.K)
        if args.W: wl["W"] = args.W
        if args.L0: wl["L0"] = args.L0
        wl["desc"] += " [sweep variant: L0=%d W=%d K=%d]" % (wl["L0"], wl["W"], wl["K"])
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference_arm(args, wl, rank)
        return 0

    import torch
    import torch.distributed as dist
    from bammmotif2_b200 import capi

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback)")
    torch.cuda.set_device(local_rank)
    capi.load()
    capi._check(capi.load().bamm_set_device(local_rank))
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", local_rank))
    numa = bind_near_gpu(torch, local_rank) if world > 1 and not os.environ.get("BAMM_BENCH_NO_NUMA") else None

    nseq = args.nseq or wl["nseq"]
    A = 4
    # every rank holds a shard of ONE data set: same planted motif and binding sites, its own sequences
    data = make_data(wl, nseq, args.seed + 1000 * rank, pinned=True, motif_seed=args.seed)
    bp_local = nseq * wl["L0"]
    pos_local = nseq * data["L"]
    bp_total = bp_local * world

    # ---- resident run ---------------------------------------------------------------------------------------
    ss = capi.SeqSet(data["codes"].reshape(-1), data["offsets"], A, data["ppos"], data["pkmer"])
    def sum_over_ranks(counts):
        t = torch.from_numpy(counts.astype(np.int64)).cuda()
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return t.cpu().numpy().astype(np.uint64)

    v0, vbg, alpha = initial_model(capi, ss, wl, data["sites"], sum_over_ranks if world > 1 else None)
    em = capi.EM(ss, wl["W"], wl["K"], wl["K_bg"])
    em.set_model(v0, vbg, alpha, Q)
    stream = torch.cuda.ExternalStream(em.stream(), device=torch.device("cuda", local_rank))
    xt = None
    exchange = "none"

    def attach_peers(e):
        """NVLink peer exchange (fused into the M-step's reduction kernel); False if CUDA IPC is not available here."""
        try:
            mine = torch.frombuffer(bytearray(e.peer_alloc(rank, world)), dtype=torch.uint8).cuda()
            allh = torch.empty(world * 64, dtype=torch.uint8, device="cuda")
            dist.all_gather_into_tensor(allh, mine)
            e.peer_attach(allh.cpu().numpy().tobytes())
            ok = torch.ones(1, device="cuda")
        except Exception as ex:                       # noqa: BLE001 - any failure means: use the NCCL exchange
            sys.stderr.write("rank %d: peer exchange unavailable (%s)\n" % (rank, ex))
            ok = torch.zeros(1, device="cuda")
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
        return bool(ok.item() > 0)

    if world > 1:
        em.set_global_nseq(nseq * world)
        if os.environ.get("BAMM_EXCHANGE", "peer") == "peer" and attach_peers(em):
            exchange = "nvlink-peer (fused into the M-step reduce kernel)"
        else:
            words = em.exchange_buffer()[1]
            xt = torch.zeros(words, dtype=torch.int64, device="cuda")
            em.set_exchange_buffer(xt.data_ptr(), words)
            exchange = "nccl all-reduce (int64)"

    def run_iters(n):
        if world == 1 or xt is None:
            em.iterate(n)          # the loop runs inside the library (bamm_em_iterate); with peers attached the exchange is part of it
            return
        with torch.cuda.stream(stream):
            for _ in range(n):
                em.estep_local()
                em.mstep_local()
                if xt is not None:
                    sharding.allreduce_exchange(xt)
                em.finish_iteration(sync=False)
        stream.synchronize()

    run_iters(args.warmup)
    torch.cuda.synchronize()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()              # before the barrier: starting NVML takes milliseconds, which the other ranks would spend waiting
    if world > 1:
        if xt is None:
            em.peer_wait(reset=True)  # waits of the warm-up (ranks arrive at different times) do not count
        dist.barrier()
        torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    launches0 = em.launch_count()
    e0.record(stream)
    run_iters(args.steps)
    e1.record(stream)
    launches = em.launch_count() - launches0
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
        torch.cuda.synchronize()
    clocks = sampler.stop() if rank == 0 else None
    ms_total = e0.elapsed_time(e1)
    if world > 1:
        t = torch.tensor([ms_total], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_total = float(t.item())
    value = bp_total * args.steps / (ms_total * 1e-3)
    model_sha1 = hashlib.sha1(em.model().tobytes()).hexdigest()
    per_rank = None
    if world > 1:
        # every rank's own device times of the timed loop and its wait for the slowest rank inside the exchange
        it_r, e_r, m_r, u_r, tot_r = em.loop_timing() if xt is None else (args.steps, 0.0, 0.0, 0.0, e0.elapsed_time(e1))
        wait_ms, waits = em.peer_wait(reset=True) if xt is None else (0.0, 0)
        mine = torch.tensor([e_r / max(it_r, 1), m_r / max(it_r, 1), u_r / max(it_r, 1), tot_r / max(it_r, 1), wait_ms / max(waits, 1)], device="cuda", dtype=torch.float64)
        allr = [torch.zeros_like(mine) for _ in range(world)]
        dist.all_gather(allr, mine)
        cols = ["estep_ms", "mstep_accum_ms", "reduce_exchange_update_ms", "iteration_ms", "peer_wait_ms"]
        per_rank = {c: [round(float(t[i].item()), 4) for t in allr] for i, c in enumerate(cols)}
        per_rank["note"] = "peer_wait_ms: mean wait for the slowest rank per exchange of the timed loop (device clock, CTA 0 of k_peer_sum)"
        # identical models on every rank (integer exchange): all ranks must hold the same bits
        hs = [None] * world
        dist.all_gather_object(hs, model_sha1)
        per_rank["models_identical"] = len(set(hs)) == 1

    # per-kernel device times (CUDA events on the EM stream, recorded by the library inside the timed loop)
    roof = None
    if world == 1:
        iters, e_ms, m_ms, u_ms, _ = em.loop_timing()
        mk_ms, bd_ms, ex_ms = em.loop_timing_estep()
        info = em.estep_info()
        peak, peak_src = peaks()
        # SURVEY.md §8d: 12 B per position and iteration = E-step (2 B k-mer index + 4 B r) + M-step (2 B index + 4 B r). The E-step is
        # the dominant phase; on the pruned path it is three kernels (DESIGN.md §4.1), of which the bound pass touches every position.
        e_dom = e_ms >= m_ms
        bytes_phase = 6.0 * pos_local
        dom_ms = e_ms if e_dom else m_ms
        ach = bytes_phase / (dom_ms / iters * 1e-3) / 1e9
        if info["pruned"]:
            dom_name = "E-step = k_emasked + k_ebound + k_eexact (pruned path, G=%d exact / G1=%d bound groups)" % (info["G"], info["G_bound"])
        else:
            dom_name = "E-step = k_estep_packed (dense, G=%d groups, %d pass(es))" % (info["G"], info["passes"])
        if not e_dom:
            dom_name = "M-step accumulation (k_mstep_list_w / k_mstep_scan_w)"
        traffic = measured_traffic(args.workload, nseq, not e_dom)
        roof = {"bound": "hbm", "kernel": dom_name, "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                "traffic": traffic, "peak_source": peak_src, "algorithmic_bytes_per_launch": bytes_phase,
                "convention": "algorithmic bytes of the phase (6 B per stored position: 2 B k-mer index + 4 B posterior) / its mean device time per iteration",
                "estep_ms": e_ms / iters, "mstep_accum_ms": m_ms / iters, "reduce_update_ms": u_ms / iters,
                "estep_kernels_ms": {"k_emasked": mk_ms / iters, "k_ebound": bd_ms / iters, "k_eexact": ex_ms / iters},
                "k_ebound_index_GBps": (2.0 * pos_local / (bd_ms / iters * 1e-3) / 1e9) if bd_ms > 0 else None,
                "candidates_frac": info["candidates"] / float(pos_local), "active_frac": info["active"] / float(pos_local),
                "dense_fallback": bool(info["dense_ran"]) if info["pruned"] else None,
                "whole_iteration_frac_of_12B_roofline": (12.0 * pos_local / (ms_total / args.steps * 1e-3) / 1e9) / peak}
    llh_after = None
    if world == 1:
        llh_after = em.iterate(0)[0]
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, em)

    # ---- strong scaling: ONE set of wl["nseq"] sequences (rank 0's data) split into contiguous blocks over the ranks -----------
    strong = None
    if world > 1 and not args.no_strong:
        em.close(); ss.close()
        torch.cuda.synchronize()
        full = data if rank == 0 else make_data(wl, nseq, args.seed, pinned=False, motif_seed=args.seed)
        lo, hi = (rank * nseq) // world, ((rank + 1) * nseq) // world          # equal lengths: contiguous blocks of equal size
        L = full["L"]
        codes_s = np.ascontiguousarray(full["codes"][lo:hi])
        sel = (full["ppos"] >= np.uint64(lo * L)) & (full["ppos"] < np.uint64(hi * L))
        offs = np.arange(hi - lo + 1, dtype=np.uint64) * np.uint64(L)
        ss = capi.SeqSet(codes_s.reshape(-1), offs, A, full["ppos"][sel] - np.uint64(lo * L), full["pkmer"][sel])
        v0s, vbgs, alphas = initial_model(capi, ss, wl, full["sites"], sum_over_ranks)
        em = capi.EM(ss, wl["W"], wl["K"], wl["K_bg"])
        em.set_model(v0s, vbgs, alphas, Q)
        em.set_global_nseq(nseq)
        xt_keep, xt = xt, None
        if attach_peers(em):
            em.iterate(args.warmup)
            torch.cuda.synchronize(); dist.barrier(); torch.cuda.synchronize()
            st = torch.cuda.ExternalStream(em.stream(), device=torch.device("cuda", local_rank))
            s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s0.record(st)
            em.iterate(args.steps)
            s1.record(st)
            torch.cuda.synchronize(); dist.barrier(); torch.cuda.synchronize()
            t = torch.tensor([s0.elapsed_time(s1)], device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms_strong = float(t.item()) / args.steps
            hs = [None] * world
            dist.all_gather_object(hs, hashlib.sha1(em.model().tobytes()).hexdigest())
            strong = {"what": "the %d sequences of rank 0's set in %d contiguous blocks, same iterations from the same initial model" % (nseq, world),
                      "ms_per_step": ms_strong, "value": nseq * wl["L0"] / (ms_strong * 1e-3), "unit": UNIT,
                      "model_sha1": hs[0], "models_identical": len(set(hs)) == 1,
                      "compare": "model_sha1 equals the N=1 line's model_sha1 when the sharded model is bit-identical to the single-GPU one"}
        xt = xt_keep
        del full

    # ---- end-to-end through the C ABI from host buffers -------------------------------------------------------
    e2e = None
    if not args.no_e2e:
        em.close(); ss.close()
        del em, ss
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        t0 = time.perf_counter()
        ss2 = capi.SeqSet(data["codes"].reshape(-1), data["offsets"], A, data["ppos"], data["pkmer"])   # H2D from pinned host memory
        t1 = time.perf_counter()
        em2 = capi.EM(ss2, wl["W"], wl["K"], wl["K_bg"])                                                 # builds the index on the device
        em2.set_model(v0, vbg, alpha, Q)
        t2 = time.perf_counter()
        # every iteration ends with a device->host read of its result (log likelihood + sum|dv|), like EM::optimize's loop
        if world > 1:
            em2.set_global_nseq(nseq * world)
            peer2 = xt is None and attach_peers(em2)
            if not peer2:
                if xt is None:
                    xt = torch.zeros(em2.exchange_buffer()[1], dtype=torch.int64, device="cuda")
                em2.set_exchange_buffer(xt.data_ptr(), em2.exchange_buffer()[1])
            st2 = torch.cuda.ExternalStream(em2.stream(), device=torch.device("cuda", local_rank))
            for _ in range(args.steps):
                with torch.cuda.stream(st2):
                    em2.estep_local(); em2.mstep_local()
                    if not peer2:
                        sharding.allreduce_exchange(xt)
                e2e_llh, e2e_vdiff = em2.finish_iteration(sync=True)
        else:
            for _ in range(args.steps):
                em2.estep_local(); em2.mstep_local()
                e2e_llh, e2e_vdiff = em2.finish_iteration(sync=True)
        vfinal = em2.model()                                                                              # D2H
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        phases = {"seqset_create_s": t1 - t0, "em_create_set_model_s": t2 - t1, "iterations_s": time.perf_counter() - t2}
        if world > 1:
            t = torch.tensor([dt], device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dt = float(t.item())
        h2d = data["codes"].nbytes + data["offsets"].nbytes + data["ppos"].nbytes + data["pkmer"].nbytes + v0.nbytes + vbg.nbytes + alpha.nbytes
        d2h = vfinal.nbytes + 20 * args.steps
        e2e = {"value": bp_total * args.steps / dt, "unit": UNIT, "h2d_bytes_per_step": h2d / args.steps,
               "d2h_bytes_per_step": d2h / args.steps, "seconds": dt, "phases": phases,
               "what": "bamm_seqset_create (H2D of codes from pinned host memory) + index build + bamm_em_create/set_model + "
                       "%d iterations, each read back (llh, sum|dv|) + bamm_em_get_model (D2H); upload amortised over the %d iterations" % (args.steps, args.steps)}
        em2.close(); ss2.close()

    # ---- CPU baseline beside it (rank 0, N=1 only) --------------------------------------------------------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        try:
            threads = os.cpu_count() or 1
            res = cpu_reference_run(wl, args.cpu_sample or wl["cpu_sample"], args.seed, 3, 1, threads)
            cpu = {"value": res["value"], "unit": UNIT, "cores": res["cores"], "kind": res["kind"], "sample": res["sample"]}
        except Exception as ex:   # the baseline must never take the GPU number down with it
            cpu = {"value": None, "unit": UNIT, "cores": os.cpu_count(), "kind": "unavailable", "sample": str(ex)[:200]}

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": wl["desc"], "nseq_per_gpu": nseq, "L0": wl["L0"], "W": wl["W"], "K": wl["K"], "K_bg": wl["K_bg"],
                       "q": Q, "seed": args.seed, "step": "one EM iteration (E-step + M-step + updateV)",
                       "positions_per_gpu": pos_local, "positions_iter_per_s": pos_local * world * args.steps / (ms_total * 1e-3),
                       "l2": "inputs (%.1f GB index + r per GPU) exceed the 126 MB L2" % (6.0 * pos_local / 1e9) if 6.0 * pos_local > 2.0e8
                             else "inputs fit in L2; no flush between iterations (EM iterates over resident data)",
                       "parallelism": "sequence shards, dp%d" % world, "exchange": exchange,
                       **({"host_numa_node_rank0": numa} if world > 1 else {})},
            "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches),
        }
        if roof:
            line["roofline"] = roof
        if cpu:
            line["cpu_baseline"] = cpu
        if llh_after is not None:
            line["config"]["llh_after"] = llh_after
        line["model_sha1"] = model_sha1 if world == 1 else None
        if per_rank:
            line["per_rank"] = per_rank
        if strong:
            line["strong"] = strong
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
