"""oracle/_ref (the copy of the reference's hot-path modules bench.py times as the CPU arm) is byte-identical to its source and
runs through the reference's stock code path. Skipped where neither the copy nor /root/reference exists."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import make_ref  # noqa: E402


def _ensure():
    if not make_ref.present():
        if not make_ref.source_available():
            pytest.skip("no reference sources and no oracle/_ref copy here")
        make_ref.make()


def test_copy_matches_manifest_and_source():
    _ensure()
    with open(os.path.join(make_ref.DEST, "MANIFEST.json")) as f:
        man = json.load(f)
    assert sorted(man["sha256"]) == sorted(make_ref.FILES)
    for rel, h in man["sha256"].items():
        assert make_ref.sha256(os.path.join(make_ref.DEST, rel)) == h
        src = os.path.join(make_ref.SRC_ROOT, rel)
        if os.path.isfile(src):
            assert make_ref.sha256(src) == h, "%s differs from the reference" % rel


def test_copy_is_not_tracked_by_git():
    with open(os.path.join(ROOT, ".gitignore")) as f:
        assert "oracle/_ref/" in f.read().split(), "oracle/_ref/ must stay git-ignored"
    r = subprocess.run(["git", "ls-files", "oracle/_ref"], cwd=ROOT, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)
    if r.returncode == 0:            # a git checkout: nothing under oracle/_ref is in the index either
        assert r.stdout.strip() == ""


def test_reference_loop_runs_from_the_copy():
    _ensure()
    out = subprocess.run([sys.executable, "-m", "oracle.ref_loop", "5", "0.3", "2"], cwd=ROOT, check=True, stdout=subprocess.PIPE,
                         text=True).stdout
    j = json.loads(out.strip().splitlines()[-1])
    assert j["kind"] == "reference" and j["value"] > 100 and "unmodified" in j["sample"]


def test_reference_loop_agrees_with_the_oracle_on_rates_order():
    """Sanity: the unmodified loop and the Python restatement play the same game (episode lengths of the same order)."""
    _ensure()
    code = ("import sys; sys.path.insert(0, %r)\n"
            "from oracle import ref_harness; ref_harness.use_copy(); m, A, B, S = ref_harness.load()\n"
            "import random; random.seed(3)\n"
            "env = S.selfplay_wrapper(B.HexEnv)(board_size=5); pol = S.BaseRandomPolicy(); obs, _ = env.reset(); n = eps = 0\n"
            "while eps < 200:\n"
            "    obs, r, d, _, _ = env.step(pol.choose_action(obs)); n += 1\n"
            "    if d: eps += 1; obs, _ = env.reset()\n"
            "print(n / eps)\n" % ROOT)
    mean_len = float(subprocess.run([sys.executable, "-c", code], check=True, stdout=subprocess.PIPE, text=True).stdout.split()[-1])
    assert 8.0 < mean_len < 14.0     # SURVEY section 8a: 10.9 env steps per episode at 5x5
