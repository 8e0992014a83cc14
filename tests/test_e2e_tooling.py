"""The multi-replica end-to-end runner (tools/e2e/run_multi.py) in its orchestration dry run: mock
OpenAI backends instead of `vllm serve`, the UNMODIFIED reference router in front, the multi-round-QA
driver through it.  Keeps the round-2 runbook (DESIGN.md §9) executable; no GPU."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
# the unmodified reference router and harness, installed by `make -C oracle ref` (never part of the repository)
needs_reference = pytest.mark.skipif(not os.path.isdir(os.path.join(ROOT, "oracle", "_ref", "vllm_router")),
                                     reason="no reference install in oracle/_ref (make -C oracle ref)")
# what the unmodified harness sent, per (user, turn), made by tests/golden/make_harness_golden.py
HARNESS_GOLDEN = os.path.join(ROOT, "tests", "golden", "mrqa_harness_turns.json")
HARNESS_SHAPE = ["--num-users", "3", "--qps", "3", "--shared-system-prompt", "40",
                 "--user-history-prompt", "25", "--answer-len", "6", "--model", "m"]


def run(tmp_path, *extra):
    cmd = [sys.executable, os.path.join(ROOT, "tools", "e2e", "run_multi.py"), "--mock", "--num-users", "3",
           "--num-rounds", "2", "--qps", "8", "--shared-system-prompt", "20", "--user-history-prompt", "20",
           "--log-dir", str(tmp_path), *extra]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr[-2000:]
    return [json.loads(l) for l in out.stdout.splitlines() if l.startswith("{")]


@needs_reference
def test_round_robin_with_cache_server_mode(tmp_path):
    (r,) = run(tmp_path, "--routing", "roundrobin", "--modes", "remote")
    assert r["requests"] == 6 and r["failed"] == 0 and "vllm_router" in os.listdir(r["router"])
    assert "listening" in open(tmp_path / "cache_server_remote.log").read()


@needs_reference
def test_orchestrated_prefill_decode_routing(tmp_path):
    (r,) = run(tmp_path, "--routing", "pd", "--replicas", "4", "--modes", "private")
    assert r["requests"] == 6 and r["failed"] == 0
    log = open(tmp_path / "router_private.log").read()
    assert log.count("Prefill endpoint: http://127.0.0.1:810") == 8 + 6  # warm-up + run: every request went P then D
    assert "Decode endpoint: http://127.0.0.1:8102" in log and "Decode endpoint: http://127.0.0.1:8103" in log


def run_against_mock(cmd_of, cwd):
    """Run cmd_of(port) against a fresh recording mock backend; -> the requests it served that carry a user id."""
    import socket
    import time
    import urllib.request
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    mock = subprocess.Popen([sys.executable, os.path.join(ROOT, "tools", "mock_backend.py"), "--port", str(port), "--model", "m"],
                            stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL, start_new_session=True)
    try:
        for _ in range(100):
            try:
                urllib.request.urlopen(f"http://127.0.0.1:{port}/health", timeout=1)
                break
            except Exception:
                time.sleep(0.2)
        out = subprocess.run(cmd_of(port), capture_output=True, text=True, timeout=180, cwd=str(cwd))
        assert out.returncode == 0, out.stderr[-1500:]
        with urllib.request.urlopen(f"http://127.0.0.1:{port}/served") as r:
            return [r for r in json.loads(r.read().decode())["served"] if r["user"] is not None]
    finally:
        mock.terminate()              # exactly the process started above
        mock.wait(20)


def by_turn(rows):
    """{(user id, number of messages): (sha1 of the messages, max_tokens, stream)}"""
    return {(r["user"], r["n_messages"]): (r["sha1"], r["max_tokens"], r["stream"]) for r in rows}


def test_driver_sends_what_the_unmodified_harness_sends(tmp_path):
    """tools/e2e/mrqa_driver.py restates benchmarks/multi-round-qa/multi-round-qa.py.  The turns the unmodified
    harness sent to the recording mock backend are stored (HARNESS_GOLDEN); the driver, run against the same mock,
    must send, for every user id they have in common, byte-identical `messages` in every turn, the same
    max_tokens, stream=True and the x-user-id header."""
    with open(HARNESS_GOLDEN) as f:
        a = {(u, n): tuple(v) for u, n, *v in json.load(f)["turns"]}
    # the harness kept admitting new users while it ran (ids 2..12 in 7 s); give the driver the same id range —
    # what a turn contains depends on (user id, prompt shape, turn, previous answers) only
    mine_shape = ["--num-users", "12", "--qps", "24"] + HARNESS_SHAPE[4:]
    b = by_turn(run_against_mock(lambda port: [sys.executable, os.path.join(ROOT, "tools", "e2e", "mrqa_driver.py"),
                                               *mine_shape, "--num-rounds", "3", "--base-url", f"http://127.0.0.1:{port}/v1"],
                                 tmp_path))
    # The harness starts its first `num_users` sessions "mid-conversation" (set_internal_state,
    # multi-round-qa.py:302-318: their first request already asks question #k > 1); sessions admitted afterwards
    # start at question #1 like the driver's.  Compare those.
    common = sorted(k for k in set(a) & set(b) if int(k[0]) > 3)
    assert len(common) >= 12, (sorted(a), sorted(b))         # several users, all three turns of most of them
    for k in common:
        assert a[k] == b[k], k


@needs_reference
def test_run_e2e_can_drive_with_the_unmodified_harness(tmp_path):
    """`run_e2e.py --harness`: the engines are driven by the reference's own multi-round-qa.py (from
    oracle/_ref) and p50 TTFT is computed from its CSV."""
    import argparse
    import socket
    import time
    import urllib.request
    sys.path.insert(0, os.path.join(ROOT, "tools", "e2e"))
    import run_e2e
    if run_e2e.harness_path() is None:
        pytest.skip("reference harness not present on this machine")
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    mock = subprocess.Popen([sys.executable, os.path.join(ROOT, "tools", "mock_backend.py"), "--port", str(port), "--model", "m"],
                            stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL, start_new_session=True)
    try:
        for _ in range(100):
            try:
                urllib.request.urlopen(f"http://127.0.0.1:{port}/health", timeout=1)
                break
            except Exception:
                time.sleep(0.2)
        a = argparse.Namespace(num_users=3, num_rounds=2, qps=3.0, shared_system_prompt=20, user_history_prompt=20, answer_len=6)
        res = run_e2e.run_harness(f"http://127.0.0.1:{port}/v1", "m", a, str(tmp_path / "h.csv"), 6)
        assert res["harness_exit"] == 0 and res["requests"] >= 6, res
        assert res["ttft_p50_s"] is not None and res["ttft_p50_s"] < 1.0 and res["output_tokens_per_s"] > 0
        assert "multi-round-qa.py" in res["driver"]
    finally:
        mock.terminate()                  # exactly the process started above
        mock.wait(20)


@needs_reference
def test_run_scale_dry_run_with_the_unmodified_router_and_harness(tmp_path):
    """tools/e2e/run_scale.py (the 1/2/4/8-replica session of profiles/scale_8gpu_r02.json) in its orchestration dry
    run: mock engines started once, routers swapped per wave, the UNMODIFIED harness offering the load (CSV written
    under another cwd), kv-aware routing through the compat controller, N/2 + N/2 prefill/decode through the router."""
    cmd = [sys.executable, os.path.join(ROOT, "tools", "e2e", "run_scale.py"), "--gpus", "2", "--mock", "--seconds", "4",
           "--qps-per-replica", "3", "--users-per-replica", "3", "--num-rounds", "2", "--shared-system-prompt", "20",
           "--user-history-prompt", "20", "--pd-prompt-words", "40", "--pd-requests", "2", "--skip", "scale,sweep,cross",
           "--model-dir", str(tmp_path / "model"), "--log-dir", os.path.relpath(tmp_path / "logs")]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=os.getcwd())
    assert out.returncode == 0, out.stderr[-2000:]
    res = {d["experiment"]: d for d in (json.loads(l) for l in out.stdout.splitlines() if l.startswith('{"experiment"'))}
    assert {"n2_none_session", "n2_kv_session", "n2_kv_kvaware", "pd_direct", "pd_1p1d_router"} <= set(res)
    for name in ("n2_none_session", "n2_kv_session"):
        assert res[name]["requests"] > 0 and res[name]["harness_exit"] == 0 and res[name]["driver"].startswith("unmodified")
        assert os.path.exists(tmp_path / "logs" / f"harness_{name}.csv")            # a relative --log-dir works
    assert res["n2_kv_kvaware"]["failed"] == 0 and res["pd_1p1d_router"]["failed"] == 0 and res["pd_direct"]["requests"] == 2
    assert os.path.exists(tmp_path / "logs" / "scale_results.json")
