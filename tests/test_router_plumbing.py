"""BASELINE.json configs[0] and the router half of configs[3], with the UNMODIFIED reference router
(production-stack's src/vllm_router, installed into oracle/_ref by `make -C oracle ref`) — plumbing only, no GPU:

* round-robin across 2 mock OpenAI backends, 100 synthetic /v1/completions -> 100 x 200, 50/50,
  strictly alternating (the criterion of the reference's tests/e2e/test-routing.py:279-285);
* kv-aware routing: the router imports `lmcache.v1.cache_controller` from this repo's compat shim,
  workers register over ZMQ, and a prompt whose KV chunks sit in one instance's pool is routed to
  that instance (src/vllm_router/routers/routing_logic.py:332-428).

Skipped where oracle/_ref was not built: nothing of the reference is part of the repository.
"""
import json
import os
import signal
import socket
import subprocess
import sys
import time
import urllib.request

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF_SRC = os.path.join(ROOT, "oracle", "_ref")   # offline pip install of the reference, unmodified
pytestmark = pytest.mark.skipif(not os.path.isdir(os.path.join(REF_SRC, "vllm_router")),
                                reason="no reference install in oracle/_ref (make -C oracle ref)")


def free_port(host="127.0.0.1"):
    s = socket.socket()
    s.bind((host, 0))
    p = s.getsockname()[1]
    s.close()
    return p


def wait_http(url, timeout=60):
    t0 = time.time()
    while time.time() - t0 < timeout:
        try:
            with urllib.request.urlopen(url, timeout=2) as r:
                if r.status == 200:
                    return True
        except Exception:
            time.sleep(0.3)
    return False


def post(url, body, headers=None):
    req = urllib.request.Request(url, data=json.dumps(body).encode(),
                                 headers={"Content-Type": "application/json", **(headers or {})})
    with urllib.request.urlopen(req, timeout=30) as r:
        return r.status, json.loads(r.read().decode())


class Procs:
    def __init__(self):
        self.procs = []

    def start(self, cmd, env=None, log=None):
        p = subprocess.Popen(cmd, env=env, stdout=log or subprocess.DEVNULL, stderr=subprocess.STDOUT,
                             start_new_session=True)
        self.procs.append(p)
        return p

    def stop(self):
        for p in self.procs:
            try:
                os.killpg(p.pid, signal.SIGTERM)   # exactly the groups started here
            except Exception:
                pass
        for p in self.procs:
            try:
                p.wait(timeout=10)
            except Exception:
                try:
                    os.killpg(p.pid, signal.SIGKILL)
                except Exception:
                    pass


def router_env(extra_path=()):
    env = dict(os.environ)
    paths = [os.path.join(ROOT, "tests", "stubs"), REF_SRC, *extra_path]
    env["PYTHONPATH"] = os.pathsep.join(paths + [env.get("PYTHONPATH", "")])
    env["HF_HUB_OFFLINE"] = "1"
    return env


def test_config1_round_robin_two_mock_backends(tmp_path):
    ps = Procs()
    try:
        ports = [free_port(), free_port()]
        for p in ports:
            ps.start([sys.executable, os.path.join(ROOT, "tools", "mock_backend.py"), "--port", str(p), "--model", "m"])
        for p in ports:
            assert wait_http(f"http://127.0.0.1:{p}/health")
        rport = free_port()
        log = open(tmp_path / "router.log", "w")
        ps.start([sys.executable, "-m", "vllm_router.app", "--host", "127.0.0.1", "--port", str(rport),
                  "--service-discovery", "static",
                  "--static-backends", ",".join(f"http://127.0.0.1:{p}" for p in ports),
                  "--static-models", "m,m", "--routing-logic", "roundrobin"], env=router_env(), log=log)
        assert wait_http(f"http://127.0.0.1:{rport}/health", 90), open(tmp_path / "router.log").read()[-2000:]
        codes = []
        for i in range(100):
            st, body = post(f"http://127.0.0.1:{rport}/v1/completions",
                            {"model": "m", "prompt": f"req-{i}", "max_tokens": 10}, {"X-Request-Id": f"rid-{i}"})
            codes.append(st)
            assert body["choices"][0]["text"]
        assert codes == [200] * 100
        served = []
        for p in ports:
            with urllib.request.urlopen(f"http://127.0.0.1:{p}/served") as r:
                served.append(json.loads(r.read().decode())["served"])
        assert [len(s) for s in served] == [50, 50]
        order = sorted([(e["t"], i) for i, s in enumerate(served) for e in s])
        seq = [i for _, i in order]
        assert all(a != b for a, b in zip(seq, seq[1:])), "round robin must alternate"
    finally:
        ps.stop()


def test_config4_kvaware_routes_to_the_instance_holding_the_kv(tmp_path, shm_name):
    sys.path.insert(0, os.path.join(ROOT, "production-stack_b200"))
    from transformers import AutoTokenizer

    from b200kv import KVPool, _lib, chunk_keys
    from b200kv.controller_client import ControllerClient
    model_dir = str(tmp_path / "synth")
    subprocess.run([sys.executable, os.path.join(ROOT, "tools", "e2e", "make_model.py"), model_dir, "--layers", "2"],
                   check=True, stdout=subprocess.DEVNULL)
    ps = Procs()
    pools, clients = [], []
    try:
        hosts = ["127.0.0.1", "127.0.0.2"]          # two "pods": the router maps instance <- ip
        ports = [free_port(h) for h in hosts]
        for h, p in zip(hosts, ports):
            ps.start([sys.executable, os.path.join(ROOT, "tools", "mock_backend.py"), "--host", h, "--port", str(p),
                      "--model", model_dir, "--name", h])
        for h, p in zip(hosts, ports):
            assert wait_http(f"http://{h}:{p}/health")
        rport, cport = free_port(), free_port()
        log = open(tmp_path / "router.log", "w")
        env = router_env([os.path.join(ROOT, "production-stack_b200", "compat"), os.path.join(ROOT, "production-stack_b200")])
        ps.start([sys.executable, "-m", "vllm_router.app", "--host", "127.0.0.1", "--port", str(rport),
                  "--service-discovery", "static",
                  "--static-backends", ",".join(f"http://{h}:{p}" for h, p in zip(hosts, ports)),
                  "--static-models", f"{model_dir},{model_dir}", "--routing-logic", "kvaware",
                  "--session-key", "x-user-id", "--lmcache-controller-port", str(cport),
                  "--kv-aware-threshold", "64"], env=env, log=log)
        assert wait_http(f"http://127.0.0.1:{rport}/health", 120), open(tmp_path / "router.log").read()[-3000:]
        # the prompt whose KV "lives" on pod 2: tokenise exactly like the router will
        tok = AutoTokenizer.from_pretrained(model_dir)
        prompt = "Hi here some system prompt " + " ".join(["hi"] * 700)
        ids = np.asarray(tok.encode(prompt), dtype=np.int32)
        SLOT = 4096
        for i, h in enumerate(hosts):
            pool = KVPool(f"{shm_name}-{i}", 16 * SLOT, SLOT, _lib.POOL_CREATE)
            pools.append(pool)
            if i == 1:
                for j, k in enumerate(chunk_keys(ids, 256, 77)):
                    pool.reserve(int(k), min(256, len(ids) - j * 256), 0, 0)
                    pool.commit(int(k))
            clients.append(ControllerClient(f"127.0.0.1:{cport}", f"pod-{i}", f"{shm_name}-{i}", 77, 256,
                                            heartbeat_s=0.5, ip=h))
        # registrations travel over ZMQ to the in-router controller: wait until routing reflects them
        deadline = time.time() + 30
        while time.time() < deadline:
            st, body = post(f"http://127.0.0.1:{rport}/v1/completions",
                            {"model": model_dir, "prompt": prompt, "max_tokens": 1}, {"x-user-id": "probe"})
            if st == 200 and body.get("served_by") == "127.0.0.2":
                break
            time.sleep(0.5)
        hit_hosts = []
        for i in range(6):
            st, body = post(f"http://127.0.0.1:{rport}/v1/completions",
                            {"model": model_dir, "prompt": prompt, "max_tokens": 4}, {"x-user-id": f"u{i}"})
            assert st == 200
            hit_hosts.append(body["served_by"])
        assert hit_hosts == ["127.0.0.2"] * 6, (hit_hosts, open(tmp_path / "router.log").read()[-3000:])
        # a prompt nobody holds falls back to session hashing: sticky per user
        miss = [post(f"http://127.0.0.1:{rport}/v1/completions",
                     {"model": model_dir, "prompt": "hi " * 300 + str(n % 2), "max_tokens": 4},
                     {"x-user-id": "same-user"})[1]["served_by"] for n in range(4)]
        assert len(set(miss)) == 1
    finally:
        for c in clients:
            c.close()
        ps.stop()
        for i, p in enumerate(pools):
            p.close()
            KVPool.unlink(f"{shm_name}-{i}")


def test_reference_router_unit_tests_pass_on_top_of_the_stubs():
    """The stand-ins for the absent `uhashring` / `kubernetes` wheels (tests/stubs) must not bend the
    router's behaviour: the reference's OWN unit tests of session routing (stickiness, minimal movement on
    add/remove of an endpoint) and round-robin routing pass with them (`@pytest.mark.asyncio` tests run by
    tests/stubs/pytest_asyncio_shim.py; pytest-asyncio is absent too)."""
    env = dict(os.environ, PYTHONPATH=os.pathsep.join([os.path.join(ROOT, "tests", "stubs"), REF_SRC]))
    out = subprocess.run([sys.executable, "-m", "pytest", "-p", "pytest_asyncio_shim", "-p", "no:cacheprovider", "-q",
                          os.path.join(REF_SRC, "tests", "test_session_router.py"),
                          os.path.join(REF_SRC, "tests", "test_roundrobin_router.py")],
                         env=env, capture_output=True, text=True, timeout=300, cwd="/tmp")
    assert out.returncode == 0 and " passed" in out.stdout and "failed" not in out.stdout, out.stdout[-2000:]


def test_prefix_aware_router_concentrates_a_shared_system_prompt_on_one_backend(tmp_path):
    """Characterisation of the UNMODIFIED reference router (routing_logic.py:447-507, prefix/hashtrie.py:46-104) on
    the multi-round-QA harness's traffic shape: every conversation starts with the same system prompt, so the trie's
    deepest match always leads to the backend that served the first request — 'N replicas, prefix-aware' is one
    replica carrying everything.  This is what the N = 2 / 4 / 8 prefix-aware rows of profiles/scale_8gpu_r02.json
    show on real engines (1 376 of 1 394 requests on one replica); kept here so the finding stays reproducible
    without a GPU.  Nothing of this repository is on the routing path."""
    sys.path.insert(0, os.path.join(ROOT, "tools", "e2e"))
    import mrqa_driver
    ps = Procs()
    try:
        ports = [free_port() for _ in range(4)]
        for p in ports:
            ps.start([sys.executable, os.path.join(ROOT, "tools", "mock_backend.py"), "--port", str(p), "--model", "m"])
        for p in ports:
            assert wait_http(f"http://127.0.0.1:{p}/health")
        rport = free_port()
        log = open(tmp_path / "router.log", "w")
        ps.start([sys.executable, "-m", "vllm_router.app", "--host", "127.0.0.1", "--port", str(rport),
                  "--service-discovery", "static",
                  "--static-backends", ",".join(f"http://127.0.0.1:{p}" for p in ports),
                  "--static-models", ",".join(["m"] * 4), "--routing-logic", "prefixaware"], env=router_env(), log=log)
        assert wait_http(f"http://127.0.0.1:{rport}/health", 90), open(tmp_path / "router.log").read()[-2000:]
        n_users = 24
        for uid in range(1, n_users + 1):        # first turns of 24 different users, the harness's prompt (multi-round-qa.py:232-251)
            msgs = [{"role": "user", "content": mrqa_driver.system_prompt(uid, 300, 200) + mrqa_driver.question(1)}]
            st, _ = post(f"http://127.0.0.1:{rport}/v1/chat/completions",
                         {"model": "m", "messages": msgs, "max_tokens": 4, "temperature": 0}, {"x-user-id": str(uid)})
            assert st == 200
        counts = []
        for p in ports:
            with urllib.request.urlopen(f"http://127.0.0.1:{p}/served") as r:
                counts.append(len(json.loads(r.read().decode())["served"]))
        assert sum(counts) == n_users
        assert max(counts) >= n_users - 3, counts      # (almost) everything on ONE of the four backends
    finally:
        ps.stop()
