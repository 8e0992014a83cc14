"""Multi-round-QA workload driver — a restatement (not a copy) of the reference harness
benchmarks/multi-round-qa/multi-round-qa.py, for machines without a reference install.  What the
unmodified harness sent to a recording mock backend is stored under tests/golden/;
tests/test_e2e_tooling.py runs this driver against the same mock and requires byte-identical
`messages`, max_tokens, stream flag and x-user-id header for every (session, turn) they share (the
harness's first `num_users` sessions start mid-conversation, a ramp-up this driver does not imitate).
The traffic shape:

* first turn = "Hi, here's some system prompt: " + "hi "*S + "For user <id>, here are some other
  context: " + "hi "*U + question            (multi-round-qa.py:232-251)
* each later turn appends the previous answer and "Here's question #k: can you tell me a new long
  story with a happy ending?"                 (:246-251, :293-301)
* requests are /v1/chat/completions, stream=True, temperature 0, max_tokens = answer_len, header
  x-user-id: <id>                             (:126-140, :288)
* per-user gap = num_users / qps seconds; users join every gap*(rounds-1)/num_users s (:367-372)
* TTFT = time to the first non-empty streamed delta (:143-171); output = per-request rows
  (prompt_tokens, generation_tokens, ttft, generation_time, user_id, question_id, launch, finish)
  (:346-356) + the p50/mean TTFT and output tokens/s summary (:493-526).
"""
from __future__ import annotations

import argparse
import asyncio
import hashlib
import json
import statistics
import time

import aiohttp


def system_prompt(uid: int, S: int, U: int) -> str:
    return (f"Hi, here's some system prompt: {' '.join(['hi'] * S)}."
            f"For user {uid}, here are some other context: {' '.join(['hi'] * U)}.")


def question(k: int) -> str:
    return f"Here's question #{k}: can you tell me a new long story with a happy ending?"


def flatten(messages) -> str:
    """Completions mode (SURVEY.md §8d config 4): the conversation as ONE prompt string, so that the
    router's kv-aware lookup tokenises exactly what the engine will see (a chat request goes through
    the engine's chat template and would not match, src/vllm_router/routers/routing_logic.py:332-428)."""
    return "\n".join(m["content"] for m in messages)


async def one_request_blocking(session, base_url, model, messages, max_tokens, uid, api="chat"):
    """stream=False variant.  The reference router's orchestrated P/D path returns its StreamingResponse
    from inside the `async with` that owns the decode connection
    (src/vllm_router/services/request_service/request.py:846-872), so a streamed answer that has not fully
    arrived yet is cut off; through that path only non-streamed requests are reliable.  TTFT is then not
    observable at the client: `ttft` carries the total latency and the row says so."""
    t0 = time.time()
    body = {"model": model, "temperature": 0, "stream": False, "max_tokens": max_tokens}
    if api == "completions":
        body["prompt"] = flatten(messages)
    else:
        body["messages"] = messages
    path = "/completions" if api == "completions" else "/chat/completions"
    async with session.post(base_url + path, json=body, headers={"x-user-id": str(uid)}) as r:
        r.raise_for_status()
        obj = await r.json()
    t1 = time.time()
    ch = (obj.get("choices") or [{}])[0]
    text = ch.get("text") if api == "completions" else (ch.get("message") or {}).get("content")
    usage = obj.get("usage") or {}
    return {"body": text or "", "ttft": t1 - t0, "ttft_is_total_latency": True, "generation_time": 0.0,
            "prompt_tokens": usage.get("prompt_tokens", 0), "generation_tokens": usage.get("completion_tokens", 0),
            "launch_time": t0, "finish_time": t1}


async def one_request(session, base_url, model, messages, max_tokens, uid, api="chat"):
    t0 = time.time()
    first = None
    first_chunk = None
    text = []
    usage = {}
    body = {"model": model, "temperature": 0, "stream": True, "max_tokens": max_tokens,
            "stream_options": {"include_usage": True}}
    if api == "completions":
        body["prompt"] = flatten(messages)
    else:
        body["messages"] = messages
    path = "/completions" if api == "completions" else "/chat/completions"
    async with session.post(base_url + path, json=body, headers={"x-user-id": str(uid)}) as r:
        r.raise_for_status()
        async for raw in r.content:
            line = raw.decode().strip()
            if not line.startswith("data:"):
                continue
            data = line[5:].strip()
            if data == "[DONE]":
                break
            obj = json.loads(data)
            if obj.get("usage"):
                usage = obj["usage"]
            ch = obj.get("choices") or []
            if not ch:
                continue
            if first_chunk is None:
                first_chunk = time.time()
            delta = ch[0].get("delta", {})
            piece = delta.get("content") or delta.get("reasoning_content") or ch[0].get("text")
            if piece:
                if first is None:
                    first = time.time()
                text.append(piece)
    t1 = time.time()
    # the harness falls back to start_time (TTFT 0) when no text ever arrives
    # (multi-round-qa.py:160-166); with random-init weights an id may detokenise to "" — use the
    # first streamed chunk in that case so the number stays meaningful
    first = first if first is not None else (first_chunk if first_chunk is not None else t0)
    return {"body": "".join(text), "ttft": first - t0, "generation_time": t1 - first,
            "prompt_tokens": usage.get("prompt_tokens", 0), "generation_tokens": usage.get("completion_tokens", 0),
            "launch_time": t0, "finish_time": t1}


async def user_session(session, args, uid, start_delay, rows):
    await asyncio.sleep(start_delay)
    gap = args.num_users / args.qps
    history = []
    for k in range(1, args.num_rounds + 1):
        t_launch = time.time()
        prompt = question(k)
        if not history:
            prompt = system_prompt(uid, args.shared_system_prompt, args.user_history_prompt) + prompt
        history.append({"role": "user", "content": prompt})
        try:
            fn = one_request if getattr(args, "stream", True) else one_request_blocking
            res = await fn(session, args.base_url, args.model, history, args.answer_len, uid, getattr(args, "api", "chat"))
        except Exception as e:  # a failed request is recorded, not fatal (the harness logs and goes on)
            rows.append({"user_id": uid, "question_id": k, "error": repr(e)})
            return
        body = res.pop("body")
        history.append({"role": "assistant", "content": body})
        res.update(user_id=uid, question_id=k, body_sha1=hashlib.sha1(body.encode()).hexdigest()[:16])
        rows.append(res)
        wait = gap - (time.time() - t_launch)
        if wait > 0 and k < args.num_rounds:
            await asyncio.sleep(wait)


async def run(args):
    rows = []
    gap = args.num_users / args.qps
    join_gap = gap * (args.num_rounds - 1) / args.num_users if args.num_rounds > 1 else 0
    timeout = aiohttp.ClientTimeout(total=None)
    async with aiohttp.ClientSession(timeout=timeout) as session:
        t0 = time.time()
        await asyncio.gather(*[user_session(session, args, args.init_user_id + i + 1, i * join_gap, rows)
                               for i in range(args.num_users)])
        t1 = time.time()
    ok = [r for r in rows if "error" not in r]
    ttfts = sorted(r["ttft"] for r in ok)
    later = sorted(r["ttft"] for r in ok if r["question_id"] > 1)
    first = sorted(r["ttft"] for r in ok if r["question_id"] == 1)
    gen = sum(r["generation_tokens"] for r in ok)
    summary = {
        "requests": len(rows), "failed": len(rows) - len(ok), "wall_s": t1 - t0,
        "ttft_p50_s": statistics.median(ttfts) if ttfts else None,
        "ttft_mean_s": statistics.fmean(ttfts) if ttfts else None,
        "ttft_p50_first_turn_s": statistics.median(first) if first else None,
        "ttft_p50_later_turns_s": statistics.median(later) if later else None,
        "ttft_p90_s": ttfts[int(0.9 * (len(ttfts) - 1))] if ttfts else None,
        "output_tokens_per_s": gen / (t1 - t0) if t1 > t0 else None,
        "input_tokens_per_s": sum(r["prompt_tokens"] for r in ok) / (t1 - t0) if t1 > t0 else None,
        "mean_prompt_tokens": statistics.fmean(r["prompt_tokens"] for r in ok) if ok else None,
        "config": {k: getattr(args, k) for k in ("num_users", "num_rounds", "qps", "shared_system_prompt",
                                                 "user_history_prompt", "answer_len", "model")},
    }
    return rows, summary


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--base-url", default="http://127.0.0.1:8000/v1")
    ap.add_argument("--model", required=True)
    ap.add_argument("--num-users", type=int, default=16)
    ap.add_argument("--num-rounds", type=int, default=4)
    ap.add_argument("--qps", type=float, default=2.0)
    ap.add_argument("--shared-system-prompt", type=int, default=512)
    ap.add_argument("--user-history-prompt", type=int, default=1536)
    ap.add_argument("--answer-len", type=int, default=64)
    ap.add_argument("--init-user-id", type=int, default=0)
    ap.add_argument("--api", choices=["chat", "completions"], default="chat")
    ap.add_argument("--no-stream", dest="stream", action="store_false", help="stream=False; ttft = total latency")
    ap.add_argument("--output", default=None, help="per-request rows as JSON lines")
    args = ap.parse_args()
    rows, summary = asyncio.run(run(args))
    if args.output:
        with open(args.output, "w") as f:
            for r in rows:
                f.write(json.dumps(r) + "\n")
    print(json.dumps(summary))


if __name__ == "__main__":
    main()
