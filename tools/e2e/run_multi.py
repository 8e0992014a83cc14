"""Multi-replica multi-round-QA behind the UNMODIFIED reference router (BASELINE.json configs[2],
scaled to the GPUs given): N `vllm serve` replicas, one per GPU, every one with B200KVConnector and
— in the `shared` modes — ONE pinned host pool for the whole box (`B200KV_POOL_NAME`), fronted by
`python -m vllm_router.app --service-discovery static --routing-logic <roundrobin|session|prefixaware|kvaware>`
(pattern: /root/reference/tests/e2e/stress-test.sh:183-190), driven by tools/e2e/mrqa_driver.py.

The router is the reference's own code: imported from oracle/_ref (an offline `pip install --target` of a
production-stack checkout, made by `make -C oracle ref`, git-ignored) — never from this repo.

Modes:
  none       no connector            -> every turn re-prefills its whole context on whichever replica it lands
  private    connector, one pool per replica -> a turn hits only if it lands where its history was stored
  shared     connector, one pool per box     -> any replica retrieves what any other stored (one PCIe hop)
  shared8    shared, FP8 packed format
  tier       connector, one pool per replica + the device chunk tier (B200KV_DEVICE_TIER_GB=8): a turn that
             lands on the other replica is scattered straight from the owner's HBM over NVLink
  remote     connector, one pool per replica + the cache-server tier (`python -m b200kv.server`,
             LMCACHE_REMOTE_URL=lm://127.0.0.1:8095): a turn that lands on the other replica is fetched
             from the server into the local pinned pool, then loaded

    python tools/e2e/run_multi.py --replicas 2 --routing roundrobin --modes none,private,shared

`--routing kvaware` (BASELINE.json configs[3]): the router imports `lmcache.v1.cache_controller` from this
repo's compat tree, every replica registers with it (LMCACHE_ENABLE_CONTROLLER, LMCACHE_CONTROLLER_PULL_URL,
tutorials/assets/values-17-kv-aware.yaml:47-51), replica i listens on 127.0.0.(i+1) because the router
tells instances apart by IP (routing_logic.py:413-423), the model is served under its directory name so
the router can load the tokenizer, and the driver uses /v1/completions (SURVEY.md §8d config 4).

`--routing pd` (BASELINE.json configs[4]): `--routing-logic disaggregated_prefill_orchestrated`; the first
half of the replicas are prefillers (label p), the rest decoders (label d)
(examples/disaggregated_prefill_orchestrated/router-deploy.yaml:124-136); every turn is prefilled on a
p replica and its KV pulled by a d replica over NVLink (b200kv/pd.py).  Needs one GPU per replica.
"""
from __future__ import annotations

import argparse
import asyncio
import json
import os
import signal
import subprocess
import sys
import time
import urllib.request

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, HERE)
import mrqa_driver  # noqa: E402
from run_e2e import harness_path, run_harness, wait_ready  # noqa: E402

MODEL = "synth-llama3-8b"


def router_path() -> str:
    p = os.path.join(ROOT, "oracle", "_ref")
    if os.path.isdir(os.path.join(p, "vllm_router")):
        return p
    raise SystemExit("reference router not found: run `make -C oracle ref REFERENCE=<production-stack checkout>`")


def replica_env(mode: str, gpu: int, cpu_gb: float, pool_tag: str) -> tuple[dict, list[str]]:
    env = dict(os.environ)
    env["CUDA_VISIBLE_DEVICES"] = str(gpu)
    env["PYTHONPATH"] = os.path.join(ROOT, "production-stack_b200") + os.pathsep + env.get("PYTHONPATH", "")
    if mode == "none":
        return env, []
    env.update(LMCACHE_LOCAL_CPU="True", LMCACHE_MAX_LOCAL_CPU_SIZE=str(cpu_gb), LMCACHE_CHUNK_SIZE="256",
               B200KV_FORMAT="fp8" if mode.endswith("8") else "raw",
               LMCACHE_LMCACHE_INSTANCE_ID=f"replica-{gpu}")
    if mode.startswith("shared"):
        env["B200KV_POOL_NAME"] = f"/b200kv-box-{pool_tag}"
    if mode.startswith("remote"):
        env["LMCACHE_REMOTE_URL"] = "lm://127.0.0.1:8095"
    if mode.startswith("tier"):
        env["B200KV_DEVICE_TIER_GB"] = "8"
    cfg = {"kv_connector": "B200KVConnector", "kv_connector_module_path": "b200kv.connector", "kv_role": "kv_both",
               "kv_load_failure_policy": "recompute"}
    return env, ["--kv-transfer-config", json.dumps(cfg)]


def killpg(proc):
    try:
        os.killpg(proc.pid, signal.SIGTERM)    # exactly the process group started here
        proc.wait(timeout=60)
    except Exception:
        try:
            os.killpg(proc.pid, signal.SIGKILL)
        except Exception:
            pass


def scrape(port: int, needles=("external", "b200kv", "lmcache"), host: str = "127.0.0.1") -> dict:
    try:
        with urllib.request.urlopen(f"http://{host}:{port}/metrics", timeout=5) as r:
            txt = r.read().decode()
    except Exception:
        return {}
    return {ln.split(" ")[0]: float(ln.split(" ")[-1]) for ln in txt.splitlines()
            if ln and not ln.startswith("#") and any(n in ln for n in needles)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--replicas", type=int, default=2)
    ap.add_argument("--routing", default="roundrobin", choices=["roundrobin", "session", "prefixaware", "kvaware", "pd"])
    ap.add_argument("--modes", default="none,private,shared")
    ap.add_argument("--layers", type=int, default=32)
    ap.add_argument("--model-dir", default="/tmp/llama3-8b-synth")
    ap.add_argument("--max-model-len", type=int, default=4096)
    ap.add_argument("--gpu-mem-util", type=float, default=0.8)
    ap.add_argument("--cpu-gb", type=float, default=30.0, help="pool GB per replica (a shared pool gets replicas x this)")
    ap.add_argument("--startup-timeout", type=float, default=900)
    ap.add_argument("--log-dir", default=os.path.join(ROOT, "gpurun_out", "multi"))
    for a, d in (("--num-users", 32), ("--num-rounds", 4), ("--shared-system-prompt", 512),
                 ("--user-history-prompt", 1536), ("--answer-len", 64)):
        ap.add_argument(a, type=int, default=d)
    ap.add_argument("--qps", type=float, default=4.0)
    ap.add_argument("--same-gpu", action="store_true",
                    help="all replicas on GPU 0 (functional check of cross-replica reuse on one GPU: started one "
                         "after the other, --gpu-mem-util split between them; timings are not per-replica numbers)")
    ap.add_argument("--extra", default="", help="extra vllm serve args, e.g. --extra=--enforce-eager")
    ap.add_argument("--kv-aware-threshold", type=int, default=2000)
    ap.add_argument("--harness", action="store_true",
                    help="drive with the unmodified multi-round-qa harness (chat API; not for --routing kvaware / pd)")
    ap.add_argument("--harness-time", type=float, default=60.0)
    ap.add_argument("--mock", action="store_true", help="orchestration dry run: tools/mock_backend.py instead of vllm (no GPU)")
    args = ap.parse_args()
    args.log_dir = os.path.abspath(args.log_dir)     # the harness runs with another cwd
    os.makedirs(args.log_dir, exist_ok=True)
    if not args.mock:
        subprocess.run([sys.executable, os.path.join(HERE, "make_model.py"), args.model_dir, "--layers", str(args.layers),
                        "--max-len", str(max(args.max_model_len, 8192))], check=True, stdout=subprocess.DEVNULL)
    rpath = router_path()
    results = []
    kvaware = args.routing == "kvaware"
    model_name = args.model_dir if kvaware else MODEL       # the router's tokenizer is loaded from this name
    hosts = [f"127.0.0.{i + 1}" if kvaware else "127.0.0.1" for i in range(args.replicas)]
    for mode in args.modes.split(","):
        procs, logs = [], []
        t_mode = time.time()
        res = {"mode": mode, "same_gpu": args.same_gpu, "replicas": args.replicas, "routing": args.routing, "router": rpath}
        try:
            ports = [8100 + i for i in range(args.replicas)]
            if mode.startswith("remote"):
                senv = dict(os.environ, B200KV_SERVER_GB=str(args.cpu_gb * args.replicas),
                            PYTHONPATH=os.path.join(ROOT, "production-stack_b200") + os.pathsep + os.environ.get("PYTHONPATH", ""))
                slog = open(os.path.join(args.log_dir, f"cache_server_{mode}.log"), "w")
                logs.append(slog)
                procs.append(subprocess.Popen([sys.executable, "-m", "b200kv.server", "127.0.0.1", "8095"], env=senv,
                                              stdout=slog, stderr=subprocess.STDOUT, start_new_session=True))
            n_aux = len(procs)
            for i, port in enumerate(ports):
                gb = args.cpu_gb * (args.replicas if mode.startswith("shared") else 1)
                env, cargs = replica_env(mode, 0 if args.same_gpu else i, gb, f"{os.getpid()}-{mode}")
                env["LMCACHE_LMCACHE_INSTANCE_ID"] = f"replica-{i}"
                if kvaware and mode != "none":
                    env.update(LMCACHE_ENABLE_CONTROLLER="True", LMCACHE_CONTROLLER_PULL_URL="127.0.0.1:9000",
                               LMCACHE_LMCACHE_WORKER_HEARTBEAT_TIME="2", B200KV_ADVERTISE_IP=hosts[i])
                util = args.gpu_mem_util / args.replicas if args.same_gpu else args.gpu_mem_util
                cmd = [sys.executable, "-m", "vllm.entrypoints.openai.api_server", "--model", args.model_dir,
                       "--served-model-name", model_name, "--load-format", "dummy", "--dtype", "bfloat16",
                       "--max-model-len", str(args.max_model_len), "--no-enable-prefix-caching",
                       "--gpu-memory-utilization", str(util), "--port", str(port), "--seed", "0",
                       "--host", hosts[i]] + cargs + (args.extra.split() if args.extra else [])
                if args.mock:
                    cmd = [sys.executable, os.path.join(ROOT, "tools", "mock_backend.py"), "--host", hosts[i],
                           "--port", str(port), "--model", model_name]
                log = open(os.path.join(args.log_dir, f"vllm_{mode}_{i}.log"), "w")
                logs.append(log)
                procs.append(subprocess.Popen(cmd, env=env, stdout=log, stderr=subprocess.STDOUT, start_new_session=True))
                if args.same_gpu and not wait_ready(port, procs[-1], args.startup_timeout, hosts[i]):
                    break
            res["startup_s"] = time.time() - t_mode
            engines = procs[n_aux:]
            if len(engines) != len(ports) or not all(wait_ready(p, pr, args.startup_timeout, h) for p, pr, h in zip(ports, engines, hosts)):
                res["error"] = "replicas not ready"
                continue
            renv = dict(os.environ)
            extra_path = [os.path.join(ROOT, "production-stack_b200", "compat"),
                          os.path.join(ROOT, "production-stack_b200")] if kvaware else []
            renv["PYTHONPATH"] = os.pathsep.join([os.path.join(ROOT, "tests", "stubs"), rpath, *extra_path,
                                                  renv.get("PYTHONPATH", "")])
            renv["HF_HUB_OFFLINE"] = "1"
            rcmd = [sys.executable, "-m", "vllm_router.app", "--host", "127.0.0.1", "--port", "8090",
                    "--service-discovery", "static",
                    "--static-backends", ",".join(f"http://{h}:{p}" for h, p in zip(hosts, ports)),
                    "--static-models", ",".join([model_name] * len(ports)), "--routing-logic", args.routing]
            if args.routing == "session":
                rcmd += ["--session-key", "x-user-id"]
            if args.routing == "pd":
                n_p = max(1, args.replicas // 2)
                rcmd[rcmd.index("--routing-logic") + 1] = "disaggregated_prefill_orchestrated"
                rcmd += ["--static-model-labels", ",".join(["p"] * n_p + ["d"] * (args.replicas - n_p)),
                         "--prefill-model-labels", "p", "--decode-model-labels", "d"]
            if kvaware:
                rcmd += ["--session-key", "x-user-id", "--lmcache-controller-port", "9000",
                         "--kv-aware-threshold", str(args.kv_aware_threshold)]
            rlog = open(os.path.join(args.log_dir, f"router_{mode}.log"), "w")
            logs.append(rlog)
            router = subprocess.Popen(rcmd, env=renv, stdout=rlog, stderr=subprocess.STDOUT, start_new_session=True)
            procs.append(router)
            if not wait_ready(8090, router, 120):
                res["error"] = "router not ready"
                continue
            d = argparse.Namespace(base_url="http://127.0.0.1:8090/v1", model=model_name, api="completions" if kvaware else "chat",
                                   stream=args.routing != "pd",   # see mrqa_driver.one_request_blocking
                                   num_users=args.num_users,
                                   num_rounds=args.num_rounds, qps=args.qps,
                                   shared_system_prompt=args.shared_system_prompt,
                                   user_history_prompt=args.user_history_prompt, answer_len=args.answer_len,
                                   init_user_id=0, output=None)
            w = argparse.Namespace(**{**vars(d), "num_users": 2 * args.replicas, "num_rounds": 1,
                                      "shared_system_prompt": 50, "user_history_prompt": 50, "answer_len": 8,
                                      "qps": 8.0, "init_user_id": 9000})
            if args.harness and args.routing not in ("kvaware", "pd") and harness_path():
                res.update(run_harness("http://127.0.0.1:8090/v1", model_name, args,
                                       os.path.join(args.log_dir, f"harness_{mode}.csv"), args.harness_time))
            else:
                asyncio.run(mrqa_driver.run(w))
                rows, summary = asyncio.run(mrqa_driver.run(d))
                res.update(summary)
                with open(os.path.join(args.log_dir, f"mrqa_rows_{mode}.jsonl"), "w") as f:
                    for r in rows:
                        f.write(json.dumps(r) + "\n")
            res["replica_metrics"] = [scrape(p, host=h) for p, h in zip(ports, hosts)]
            res["router_requests_per_backend"] = scrape(8090, ("vllm:num_incoming_requests", "current_qps", "num_requests"))
        finally:
            for p in reversed(procs):
                killpg(p)
            for lg in logs:
                lg.close()
            if mode.startswith("shared"):     # the box-wide segment outlives its replicas: remove it
                import glob
                for f in glob.glob(f"/dev/shm/b200kv-box-{os.getpid()}-{mode}*"):   # name + "-<chunk bytes>"
                    os.unlink(f)
            print(json.dumps(res), flush=True)
            results.append(res)
            time.sleep(3)
    with open(os.path.join(args.log_dir, "multi_results.json"), "w") as f:
        json.dump(results, f, indent=1)


if __name__ == "__main__":
    main()
