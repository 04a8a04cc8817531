"""Occurrence scan (BaMMScan, DESIGN.md §4.7) on one device: the C ABI's phases, the command line against the existing
`BaMMmotif --scoreSeqset` route, and a genome-like set of chromosome-length records.

    python tools/scan_bench.py [--part abi cli genome] [--nseq 1000000] [--L0 500] [--orders 2 4] [--motifs 1 6] [--out FILE]

abi     seeded planted sequences (both strands, stored length 2 L0 + 1), negatives sampled on the device with fold 1 (-m 1),
        W = 20, cutoff 1e-4: device time of the negative scoring, of the sort and of the hit scan (CUDA events,
        bamm_scan_info), host wall time of each call, windows per second of the hit kernels; one motif and six.
cli     the same set as FASTA, a MEME file of six W = 20 PWMs, `--PWMFile F --maxPWM M -k K --pvalCutoff 1e-4` through
        bin/BaMMScan and through bin/BaMMmotif --scoreSeqset: wall time, peak host RSS (wait4), and whether the .occurrence
        files are byte-identical.
genome  24 single-strand records of seeded random lengths scaled to 1e9 bases in all: the time of sampling the negatives
        (fold 1), the scan's kernels, and ZOOPS scoring of the same set by k_score (one warp per record, BAMM_NO_PACKED=1).
Prints one JSON line per measurement; the first names the card, its power limit and its maximum SM clock.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True

from bammmotif2_b200 import capi, hostmodel, synth  # noqa: E402

BIN = os.path.join(ROOT, "bammmotif2_b200", "bin")
W = 20


def card():
    q = "name,power.limit,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=" + q, "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.TimeoutExpired):
        out = ""
    return dict(zip(q.split(","), [s.strip() for s in out.split(",")])) if out else {"nvidia-smi": "unavailable"}


def emit(rec, out):
    line = json.dumps(rec)
    print(line, flush=True)
    if out:
        out.write(line + "\n")
        out.flush()


def pwms(n, seed=5):
    rng = np.random.default_rng(seed)
    return [rng.dirichlet(np.full(4, 0.3), size=W) for _ in range(n)]


def models(K, n):
    """n order-K models of width W from the sites of seeded PWMs, against a uniform order-2 background."""
    vbg = np.concatenate([np.full(4 ** (k + 1), 0.25, np.float32) for k in range(3)])
    out = []
    for i, pwm in enumerate(pwms(n)):
        u = np.random.default_rng(100 + i).random((500, W))
        sites = np.minimum((u[:, :, None] > np.cumsum(pwm, axis=1)[None]).sum(axis=2), 3).astype(np.uint8) + 1
        out.append(hostmodel.motif_from_sites(sites, 4, K, hostmodel.default_motif_alpha(K, W), vbg))
    return out, vbg


def part_abi(args, out):
    fwd, _, _ = synth.planted_sequences(11, args.nseq, args.L0, W)
    codes = synth.stored_both_strands(fwd)
    ppos, pkmer = synth.middle_n_patches(codes, 11)
    offsets = np.arange(args.nseq + 1, dtype=np.uint64) * np.uint64(codes.shape[1])
    pos = capi.SeqSet(codes.ravel(), offsets, 4, ppos, pkmer)
    del codes, fwd
    t = time.perf_counter()
    neg = pos.sample_negatives(1)
    emit(dict(part="abi", what="negative sampling (fold 1)", seconds=time.perf_counter() - t, records=neg.nseq), out)
    windows = args.nseq * (2 * args.L0 + 1 - W + 1)
    for K in args.orders:
        vs, vbg = models(K, max(args.motifs))
        pos.index(K)
        neg.index(K)
        capi.Scan(neg, W, K, 2, vs[0], vbg).hits(pos, 1e-4)            # warm-up: modules, pools
        for nm in args.motifs:
            tot = dict(neg_score_ms=0.0, sort_ms=0.0, hits_ms=0.0, create_s=0.0, hits_s=0.0, hits=0)
            for v in vs[:nm]:
                t0 = time.perf_counter()
                sc = capi.Scan(neg, W, K, 2, v, vbg)
                t1 = time.perf_counter()
                h = sc.hits(pos, 1e-4)
                t2 = time.perf_counter()
                inf = sc.info()
                sc.close()
                for k in ("neg_score_ms", "sort_ms", "hits_ms"):
                    tot[k] += inf[k]
                tot["create_s"] += t1 - t0
                tot["hits_s"] += t2 - t1
                tot["hits"] += len(h)
            emit(dict(part="abi", K=K, W=W, motifs=nm, nseq=args.nseq, L0=args.L0, positive_windows=windows,
                      negative_windows=inf["negative_windows"], cutoff=1e-4, **tot,
                      hit_kernel_windows_per_s=windows * nm / (tot["hits_ms"] * 1e-3)), out)


def run_measured(cmd):
    t = time.perf_counter()
    p = subprocess.Popen(cmd, stdout=subprocess.DEVNULL, stderr=subprocess.PIPE)
    _, status, ru = os.wait4(p.pid, 0)
    wall = time.perf_counter() - t
    err = p.stderr.read().decode()[-500:]
    p.stderr.close()
    return wall, ru.ru_maxrss / 1024.0, os.waitstatus_to_exitcode(status), err


def part_cli(args, out):
    tmp = tempfile.mkdtemp(prefix="scan_bench_")
    fwd, _, _ = synth.planted_sequences(11, args.nseq, args.L0, W)
    fa = os.path.join(tmp, "pos.fasta")
    synth.write_fasta(fa, fwd)
    del fwd
    meme = os.path.join(tmp, "pwm.meme")
    with open(meme, "w") as f:
        f.write("MEME version 4\n\nALPHABET= ACGT\n\n")
        for i, pwm in enumerate(pwms(max(args.motifs))):
            f.write("MOTIF m%d\nletter-probability matrix: alength= 4 w= %d\n" % (i + 1, W))
            for row in pwm:
                f.write(" ".join("%.4f" % x for x in row) + "\n")
            f.write("\n")
    for K in args.orders:
        for nm in args.motifs:
            flags = ["--PWMFile", meme, "--maxPWM", str(nm), "-k", str(K), "-K", "2", "--pvalCutoff", "1e-4"]
            res = {}
            for name, exe, extra in (("BaMMScan", "BaMMScan", []), ("scoreSeqset", "BaMMmotif", ["--scoreSeqset"])):
                odir = os.path.join(tmp, "%s_k%d_m%d" % (name, K, nm))
                wall, rss, rc, err = run_measured([os.path.join(BIN, exe), odir, fa] + flags + extra)
                res[name] = dict(seconds=wall, peak_rss_mb=rss, exit=rc, **({"stderr": err} if rc else {}))
            same = all(open(os.path.join(tmp, "BaMMScan_k%d_m%d" % (K, nm), "pos_motif_%d.occurrence" % m), "rb").read() ==
                       open(os.path.join(tmp, "scoreSeqset_k%d_m%d" % (K, nm), "pos_motif_%d.occurrence" % m), "rb").read()
                       for m in range(1, nm + 1)) if all(r["exit"] == 0 for r in res.values()) else None
            lines = sum(1 for _ in open(os.path.join(tmp, "BaMMScan_k%d_m%d" % (K, nm), "pos_motif_1.occurrence"))) - 1 \
                if res["BaMMScan"]["exit"] == 0 else None
            emit(dict(part="cli", K=K, W=W, motifs=nm, nseq=args.nseq, L0=args.L0, mfold=1, cutoff=1e-4,
                      occurrence_files_identical=same, motif1_occurrences=lines, **res), out)
    subprocess.run(["rm", "-rf", tmp])


def part_genome(args, out):
    rng = np.random.default_rng(3)
    lens = rng.integers(10 ** 7, 15 * 10 ** 7 + 1, size=24)
    lens = (lens * (10 ** 9 / lens.sum())).astype(np.int64)
    offsets = np.concatenate([[0], np.cumsum(lens)]).astype(np.uint64)
    pos = capi.SeqSet(rng.integers(1, 5, size=int(offsets[-1]), dtype=np.uint8), offsets, 4)
    t = time.perf_counter()
    neg = pos.sample_negatives(1)
    emit(dict(part="genome", what="negative sampling (fold 1)", records=24, bases=int(offsets[-1]),
              min_record=int(lens.min()), max_record=int(lens.max()), seconds=time.perf_counter() - t), out)
    for K in args.orders:
        vs, vbg = models(K, 1)
        pos.index(K)
        neg.index(K)
        sc = capi.Scan(neg, W, K, 2, vs[0], vbg)
        sc.hits(pos, 1e-4)
        h = sc.hits(pos, 1e-4)
        inf = sc.info()
        sc.close()
        os.environ["BAMM_NO_PACKED"] = "1"
        pos.score(W, K, 2, vs[0], vbg, want_mops=False)
        pos.score(W, K, 2, vs[0], vbg, want_mops=False)
        kscore_ms = capi.score_last_ms()
        del os.environ["BAMM_NO_PACKED"]
        windows = int(offsets[-1]) - 24 * (W - 1)
        emit(dict(part="genome", K=K, W=W, windows=windows, hits=len(h), neg_score_ms=inf["neg_score_ms"], sort_ms=inf["sort_ms"],
                  scan_hits_ms=inf["hits_ms"], k_score_zoops_ms=kscore_ms,
                  scan_windows_per_s=windows / (inf["hits_ms"] * 1e-3), k_score_windows_per_s=windows / (kscore_ms * 1e-3)), out)


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--part", nargs="+", default=["abi", "cli", "genome"], choices=["abi", "cli", "genome"])
    ap.add_argument("--nseq", type=int, default=1_000_000)
    ap.add_argument("--L0", type=int, default=500)
    ap.add_argument("--orders", type=int, nargs="+", default=[2, 4])
    ap.add_argument("--motifs", type=int, nargs="+", default=[1, 6])
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    capi.load()
    if capi.device_count() < 1:
        raise SystemExit("scan_bench needs a CUDA device")
    out = open(args.out, "w") if args.out else None
    emit(dict(card=card()), out)
    for part in args.part:
        {"abi": part_abi, "cli": part_cli, "genome": part_genome}[part](args, out)


if __name__ == "__main__":
    main()
