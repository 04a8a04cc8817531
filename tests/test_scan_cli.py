"""bin/BaMMScan on the CPU: it builds, and it refuses a command line without an initial model or with an unknown option the
way bin/BaMMmotif does (same message, exit code 1) before any device work."""
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "bammmotif2_b200", "bin")


@pytest.fixture(scope="module")
def bins():
    from bammmotif2_b200 import build
    build.build_all()
    return BIN


def run(exe, args):
    return subprocess.run([exe] + args, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)


@pytest.mark.parametrize("args,message", [
    ([], "Error: No initial model is provided."),
    (["--PWMFile", "motifs.meme", "--noSuchOption", "3"], "Oops! Unknown option(s) remaining..."),
    (["--PWMFile", "motifs.meme", "--EM"], "--EM, --CGS, --advanceEM, --FDR and --scoreSeqset are options of BaMMmotif"),
])
def test_bammscan_rejects_bad_command_lines(bins, tmp_path, args, message):
    fa = tmp_path / "in.fasta"
    fa.write_text(">a\nACGTACGTACGTTTGACCA\n")
    scan = run(os.path.join(bins, "BaMMScan"), [str(tmp_path / "out"), str(fa)] + args)
    assert scan.returncode == 1 and message in scan.stderr, scan.stderr
    if "--EM" not in args:
        motif = run(os.path.join(bins, "BaMMmotif"), [str(tmp_path / "out2"), str(fa)] + args)
        assert motif.returncode == 1 and message in motif.stderr
