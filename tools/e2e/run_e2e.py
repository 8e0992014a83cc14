"""End-to-end multi-round-QA on one B200 (BASELINE.json configs[1]): start `vllm serve` on a
synthetic Llama-3-8B (random-init weights, --load-format dummy) with a chosen KV connector, drive
it with tools/e2e/mrqa_driver.py, print one JSON line per mode.

Modes:
  none      no connector, prefix caching off   -> every turn re-prefills its whole context
  b200kv    this repo's connector, RAW (bit-exact) format
  b200kv8   this repo's connector, FP8 packed format
  b200kvq4  this repo's connector, Q4 group-wise 4-bit format (experimental)
  b200kv_cw / b200kv8_cw      chunk-wise loads (layer-wise overlap with the forward pass switched off)
  b200kv_async / b200kv_c64  variants: loads detached from the forward step / 64-token chunks
  offload   vLLM's in-tree CPU offload connector (same plugin slot; the runnable same-box stand-in
            for the absent lmcache wheel, SURVEY.md §8d "baseline 2a")

    python tools/e2e/run_e2e.py --modes none,b200kv --layers 32 --num-users 16 --num-rounds 4
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


def connector_args(mode: str, cpu_gb: float):
    env = {}
    if mode == "none":
        return [], env
    if mode.startswith("b200kv"):
        # b200kv | b200kv8 (fp8) | b200kv_async (detached loads) | b200kv_c64 (64-token chunks)
        env.update(LMCACHE_LOCAL_CPU="True", LMCACHE_MAX_LOCAL_CPU_SIZE=str(cpu_gb),
                   LMCACHE_CHUNK_SIZE="64" if "c64" in mode else "256",
                   B200KV_FORMAT="q4" if "q4" in mode else ("fp8" if "8" in mode.replace("c64", "") else "raw"),
                   B200KV_ASYNC_LOAD="1" if "async" in mode else "0",
                   B200KV_LAYERWISE="0" if "cw" in mode else "1")
        cfg = {"kv_connector": "B200KVConnector", "kv_connector_module_path": "b200kv.connector", "kv_role": "kv_both",
               "kv_load_failure_policy": "recompute"}
        return ["--kv-transfer-config", json.dumps(cfg)], env
    if mode == "offload":
        cfg = {"kv_connector": "OffloadingConnector", "kv_role": "kv_both",
               "kv_connector_extra_config": {"cpu_bytes_to_use": int(cpu_gb * (1 << 30))}}
        return ["--kv-transfer-config", json.dumps(cfg)], env
    raise ValueError(mode)


def harness_path() -> str | None:
    """The UNMODIFIED benchmarks/multi-round-qa/multi-round-qa.py: the byte-identical copy `make -C oracle ref`
    placed in the git-ignored oracle/_ref."""
    p = os.path.join(ROOT, "oracle", "_ref", "benchmarks", "multi-round-qa", "multi-round-qa.py")
    return p if os.path.exists(p) else None


def run_harness(base_url: str, model: str, a, out_csv: str, seconds: float) -> dict:
    """Drive the engine with the unmodified harness; p50 TTFT comes from the per-request CSV it writes
    (the harness itself prints the MEAN, multi-round-qa.py:497,526; SURVEY.md §8d)."""
    import csv
    import statistics
    hp = harness_path()
    cmd = [sys.executable, hp, "--num-users", str(a.num_users), "--num-rounds", str(a.num_rounds), "--qps", str(a.qps),
           "--shared-system-prompt", str(a.shared_system_prompt), "--user-history-prompt", str(a.user_history_prompt),
           "--answer-len", str(a.answer_len), "--model", model, "--base-url", base_url, "--time", str(int(seconds)),
           "--request-with-user-id", "--output", out_csv]
    t0 = time.time()
    out = subprocess.run(cmd, capture_output=True, text=True, cwd=os.path.dirname(out_csv) or ".")
    wall = time.time() - t0
    rows = list(csv.DictReader(open(out_csv))) if os.path.exists(out_csv) else []
    ttft = sorted(float(r["ttft"]) for r in rows)
    later = sorted(float(r["ttft"]) for r in rows if int(float(r["question_id"])) > 1)
    gen = sum(float(r["generation_tokens"]) for r in rows)
    span = (max(float(r["finish_time"]) for r in rows) - min(float(r["launch_time"]) for r in rows)) if rows else 0
    return {"driver": "unmodified harness " + hp, "harness_exit": out.returncode, "requests": len(rows), "wall_s": wall,
            "ttft_p50_s": statistics.median(ttft) if ttft else None,
            "ttft_mean_s": statistics.fmean(ttft) if ttft else None,
            "ttft_p50_later_turns_s": statistics.median(later) if later else None,
            "ttft_p90_s": ttft[int(0.9 * (len(ttft) - 1))] if ttft else None,
            "output_tokens_per_s": gen / span if span > 0 else None,
            "harness_tail": out.stdout[-600:] if out.returncode else ""}


def wait_ready(port: int, proc: subprocess.Popen, timeout: float, host: str = "127.0.0.1") -> bool:
    t0 = time.time()
    while time.time() - t0 < timeout:
        if proc.poll() is not None:
            return False
        try:
            with urllib.request.urlopen(f"http://{host}:{port}/health", timeout=2) as r:
                if r.status == 200:
                    return True
        except Exception:
            time.sleep(2)
    return False


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--modes", default="none,b200kv")
    ap.add_argument("--layers", type=int, default=32)
    ap.add_argument("--model-dir", default="/tmp/llama3-8b-synth")
    ap.add_argument("--port", type=int, default=8011)
    ap.add_argument("--max-model-len", type=int, default=4096)
    ap.add_argument("--gpu-mem-util", type=float, default=0.8)
    ap.add_argument("--cpu-gb", type=float, default=30.0)
    ap.add_argument("--startup-timeout", type=float, default=900)
    ap.add_argument("--extra", default="", help="extra vllm serve args (space separated)")
    ap.add_argument("--log-dir", default=os.path.join(ROOT, "gpurun_out"))
    for a, d in (("--num-users", 16), ("--num-rounds", 4), ("--shared-system-prompt", 512),
                 ("--user-history-prompt", 1536), ("--answer-len", 64)):
        ap.add_argument(a, type=int, default=d)
    ap.add_argument("--qps", type=float, default=2.0)
    ap.add_argument("--harness", action="store_true",
                    help="drive with the unmodified benchmarks/multi-round-qa harness for --harness-time seconds "
                         "instead of tools/e2e/mrqa_driver.py")
    ap.add_argument("--harness-time", type=float, default=60.0)
    args = ap.parse_args()
    if args.harness and harness_path() is None:
        raise SystemExit("--harness: the reference harness is not in oracle/_ref (make -C oracle ref)")
    args.log_dir = os.path.abspath(args.log_dir)     # the harness runs with another cwd
    os.makedirs(args.log_dir, exist_ok=True)
    subprocess.run([sys.executable, os.path.join(HERE, "make_model.py"), args.model_dir, "--layers", str(args.layers),
                    "--max-len", str(max(args.max_model_len, 8192))], check=True, stdout=subprocess.DEVNULL)
    results = []
    for mode in args.modes.split(","):
        cargs, cenv = connector_args(mode, args.cpu_gb)
        env = dict(os.environ)
        env.update(cenv)
        env["PYTHONPATH"] = os.path.join(ROOT, "production-stack_b200") + os.pathsep + env.get("PYTHONPATH", "")
        env.setdefault("VLLM_LOGGING_LEVEL", "INFO")
        cmd = [sys.executable, "-m", "vllm.entrypoints.openai.api_server", "--model", args.model_dir,
               "--served-model-name", "synth-llama3-8b", "--load-format", "dummy", "--dtype", "bfloat16",
               "--max-model-len", str(args.max_model_len), "--no-enable-prefix-caching",
               "--gpu-memory-utilization", str(args.gpu_mem_util), "--port", str(args.port), "--seed", "0",
               "--host", "127.0.0.1"] + cargs + (args.extra.split() if args.extra else [])
        log = open(os.path.join(args.log_dir, f"vllm_{mode}.log"), "w")
        t_start = time.time()
        proc = subprocess.Popen(cmd, env=env, stdout=log, stderr=subprocess.STDOUT, start_new_session=True)
        res = {"mode": mode, "layers": args.layers}
        try:
            if not wait_ready(args.port, proc, args.startup_timeout):
                res["error"] = f"server not ready (exit={proc.poll()}); see vllm_{mode}.log"
            else:
                res["startup_s"] = time.time() - t_start
                d = argparse.Namespace(base_url=f"http://127.0.0.1:{args.port}/v1", model="synth-llama3-8b",
                                       num_users=args.num_users, num_rounds=args.num_rounds, qps=args.qps,
                                       shared_system_prompt=args.shared_system_prompt,
                                       user_history_prompt=args.user_history_prompt, answer_len=args.answer_len,
                                       init_user_id=0, output=None)
                # warm-up like the harness (10 short requests, multi-round-qa.py:552-561)
                w = argparse.Namespace(**{**vars(d), "num_users": 4, "num_rounds": 1, "shared_system_prompt": 50,
                                          "user_history_prompt": 50, "answer_len": 8, "qps": 8.0, "init_user_id": 9000})
                if args.harness:      # the harness does its own warm-up (10 short requests, :552-561)
                    res.update(run_harness(f"http://127.0.0.1:{args.port}/v1", "synth-llama3-8b", args,
                                           os.path.join(args.log_dir, f"harness_{mode}.csv"), args.harness_time))
                else:
                    asyncio.run(mrqa_driver.run(w))
                    rows, summary = asyncio.run(mrqa_driver.run(d))
                    res.update(summary)
                    with open(os.path.join(args.log_dir, f"mrqa_rows_{mode}.jsonl"), "w") as f:
                        for r in rows:
                            f.write(json.dumps(r) + "\n")
                try:
                    with urllib.request.urlopen(f"http://127.0.0.1:{args.port}/metrics", timeout=5) as r:
                        txt = r.read().decode()
                    res["metrics"] = {ln.split(" ")[0]: float(ln.split(" ")[-1]) for ln in txt.splitlines()
                                      if ln and not ln.startswith("#") and ("prefix_cache" in ln or "external" in ln
                                                                             or "b200kv" in ln or "lmcache" in ln)}
                except Exception:
                    pass
        finally:
            try:
                os.killpg(proc.pid, signal.SIGTERM)  # exactly the process group started above
                proc.wait(timeout=60)
            except Exception:
                try:
                    os.killpg(proc.pid, signal.SIGKILL)
                except Exception:
                    pass
            log.close()
        print(json.dumps(res), flush=True)
        results.append(res)
        time.sleep(3)
    with open(os.path.join(args.log_dir, "e2e_results.json"), "w") as f:
        json.dump(results, f, indent=1)


if __name__ == "__main__":
    main()
