"""Driver contract checks that need no GPU: the reference arm of bench.py answers with one JSON
line and exit code 0 (with and without a torchrun-style environment), the argument defaults are
the documented ones, and __graft_entry__ exposes build() / smoke()."""
import json
import os
import subprocess
import sys

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(args, env=None):
    e = dict(os.environ)
    e.update(env or {})
    return subprocess.run([sys.executable, os.path.join(REPO, "bench.py")] + args, env=e,
                          stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=300)


def test_reference_arm_reports_unavailable_and_exits_zero():
    """Where no GPU is visible the reference arm says why in ONE JSON line, exit 0; on a GPU box
    it reports the measured number (tests/test_reference_arm.py covers the rest)."""
    r = _run(["--impl", "reference", "--gpus", "1", "--steps", "5", "--warmup", "3"],
             {"CUDA_VISIBLE_DEVICES": ""})
    assert r.returncode == 0, r.stderr
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and isinstance(d["unavailable"], str) and d["unavailable"]
    assert "\n" not in d["unavailable"]


def test_reference_arm_prints_on_rank_zero_only():
    # no GPU visible: the arm fails before the rendezvous, where this lone rank 1 would wait for
    # a rank 0 that never comes
    env = {"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1", "MASTER_ADDR": "127.0.0.1",
           "MASTER_PORT": "29999", "CUDA_VISIBLE_DEVICES": ""}
    r = _run(["--impl", "reference", "--gpus", "2"], env)
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_graft_entry_has_build_and_smoke():
    sys.path.insert(0, REPO)
    try:
        import __graft_entry__ as g
    finally:
        sys.path.pop(0)
    assert callable(g.build) and callable(g.smoke)
