#!/usr/bin/env python
"""bench.py — KV offload hot path on B200 (driver contract: one JSON line on rank 0).

Workload (BASELINE.json configs[1], "Llama-3-8B, 1 replica on 1xB200, CPU-RAM offload,
multi-round-qa 4-turn 2K-ctx"): one step = the KV traffic of one scheduling wave of the
multi-round-QA harness — 16 user sessions x 2048-token context, Llama-3-8B KV geometry
(L=32, H_kv=8, D=128, bf16, block 16, chunk 256 => 128 KiB/token, 4 GiB per direction per step):

  e2e    (headline): every session is stored  (paged HBM -> fused gather -> pinned host pool) and
         then retrieved (pinned host pool -> staging -> scatter into *other* pages) through the
         reference-facing engine calls (KVEngine.store / .retrieve == lmcache_engine.store /
         .retrieve); D2H and H2D are inside the timed region; fresh token ids every step so every
         chunk is really written (LRU eviction included).
  value  : the same 32768 tokens gathered into / scattered from a DEVICE buffer (HBM only).
  roofline: dominant kernel = RAW gather (kv_bulk_copy_kernel<store>); algorithmic bytes =
         262144 B/token (SURVEY.md §8d) x tokens per launch / CUDA-event duration of that launch.

metric = KV payload GB/s (store+retrieve payload bytes / time).  `--impl reference` times the CPU
oracle port (oracle/liboracle.so; the lmcache wheel is absent from this image) on the host cores.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "production-stack_b200"))

L, H, D, BS, C = 32, 8, 128, 16, 256
NB = 8192                     # 16 GiB paged cache (BASELINE.md §3)
SESSIONS, CTX = 16, 2048      # one wave of the 2K-ctx multi-round-QA config
TOKEN_BYTES_ALL = 2 * L * H * D * 2   # 131072 B payload per token (bf16)
ALGO_BYTES_PER_TOKEN = 2 * TOKEN_BYTES_ALL  # HBM read + HBM write of the gather kernel
# --dump-outputs: a fixed, seeded sample of what each timed leg computed in its last step (~40 MiB in all)
DUMP_TOKENS = 32              # tokens of the wave whose K and V rows in every layer are written
DUMP_CHUNK_VALUES = 1 << 20   # values of the device leg's chunk buffer
DUMP_LIMIT_BYTES = 64 * 10**6


def peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))), "measured"
    except Exception:
        return {"hbm_gbs": 6650.0}, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md)."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.rows, self.proc = [], None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self) -> dict:
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 6:
                continue
            try:
                sm.append(float(f[0]))
                mx = float(f[1])
            except ValueError:
                continue
            for nme, v in zip(names, f[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(nme)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx,
                "reasons": sorted(reasons), "samples": len(sm)}


def slot_map(blocks: np.ndarray, n_tok: int) -> np.ndarray:
    """slot[i] = block_ids[i // 16] * 16 + i % 16 (vllm_v1_adapter.py:368-375) — input tables only."""
    i = np.arange(n_tok, dtype=np.int64)
    return np.asarray(blocks, dtype=np.int64)[i // BS] * BS + i % BS


def numa_nodes_of(addr: int) -> dict | None:
    """Pages per NUMA node of the mapping that contains `addr`, from /proc/self/numa_maps."""
    try:
        best = None
        for ln in open("/proc/self/numa_maps"):
            f = ln.split()
            a = int(f[0], 16)
            if a <= addr and (best is None or a > best[0]):
                best = (a, f)
        if best is None:
            return None
        out = {}
        for tok in best[1][1:]:
            if tok[0] == "N" and "=" in tok and tok[1:].split("=")[0].isdigit():
                out[tok.split("=")[0]] = int(tok.split("=")[1])
        return out or None
    except Exception:
        return None


def session_tokens(rank: int, step: int, s: int) -> np.ndarray:
    """Deterministic synthetic token ids, unique per (rank, step, session) so keys are fresh."""
    base = np.arange(CTX, dtype=np.int64)
    return ((base * 2654435761 + (rank * 1000003 + step * 10007 + s) * 97) % 128256).astype(np.int32)


# ------------------------------------------------------------------------------------------------
# reference arm / cpu_baseline: the oracle port on host cores
# ------------------------------------------------------------------------------------------------
def cpu_oracle_run(steps: int, warmup: int, sessions: int = SESSIONS, nb: int = NB, target_s: float = 0.0,
                   min_step_s: float = 0.0):
    """store+retrieve of `sessions` x 2K-ctx requests per step with oracle/liboracle.so (gather
    into a host chunk buffer = the CPU pool, scatter back into other pages) on the SAME configuration
    the GPU arm advertises: 16 sessions x 2048 tokens over an 8192-block (16 GiB) paged cache in host
    RAM.  Returns (GB/s payload, ms/step, threads, sample description).  target_s > 0: the number of
    steps is chosen so the timed sample is about that many seconds of CPU work.  min_step_s > 0: a
    step repeats the wave until it lasts that long (reference arm: K steps must add up to seconds,
    not milliseconds).  BENCH_REF_BLOCKS / BENCH_REF_SESSIONS shrink the case for CPU-only CI."""
    from tests import oracle_c
    sessions = int(os.environ.get("BENCH_REF_SESSIONS", sessions))
    nb = int(os.environ.get("BENCH_REF_BLOCKS", nb))
    nblk = CTX // BS
    nb = max(nb, sessions * nblk)
    pat = np.random.default_rng(0).integers(0, 2 ** 16, (BS, H, D), dtype=np.uint16)      # one 32 KiB tile
    layers = []
    for l in range(L):   # every page touched and distinct per (layer, plane, block); content is irrelevant to timing
        a = np.empty((2, nb, BS, H, D), dtype=np.uint16)
        a[:] = pat
        a[:, :, 0, 0, 0] = np.arange(2 * nb, dtype=np.uint16).reshape(2, nb) + l
        layers.append(a)
    perm = np.random.default_rng(1234).permutation(nb)
    dperm = np.random.default_rng(4321).permutation(nb)
    maps = [(slot_map(perm[s * nblk:(s + 1) * nblk], CTX), slot_map(dperm[s * nblk:(s + 1) * nblk], CTX))
            for s in range(sessions)]
    threads = oracle_c.lib().oracle_num_threads()
    keys_out = np.zeros(CTX // C, dtype=np.uint64)
    lib = oracle_c.lib()
    planes, stride = oracle_c.planes_of(layers)
    cb = 2 * L * C * H * D * 2
    pool = np.zeros(sessions * (CTX // C) * cb, dtype=np.uint8)   # the "CPU pool": reused every step

    def one_wave(step):
        for s, (sm, dm) in enumerate(maps):
            toks = session_tokens(0, step, s)
            lib.oracle_chunk_keys(toks.ctypes.data, CTX, C, 0, 1, keys_out.ctypes.data)
            slot = pool[s * (CTX // C) * cb:]
            lib.oracle_gather_raw(planes, 2 * L, stride, BS, H * D * 2, sm.ctypes.data, CTX, C, slot.ctypes.data, cb)
            lib.oracle_scatter_raw(planes, 2 * L, stride, BS, H * D * 2, dm.ctypes.data, CTX, C, slot.ctypes.data, cb)

    for w in range(warmup):
        one_wave(w)
    t0 = time.perf_counter()
    one_wave(warmup)
    wave_s = max(time.perf_counter() - t0, 1e-4)
    reps = max(1, int(np.ceil(min_step_s / wave_s))) if min_step_s > 0 else 1
    if target_s > 0:
        steps = int(min(4000, max(steps, target_s / (wave_s * reps))))
    t0 = time.perf_counter()
    for k in range(steps * reps):
        one_wave(warmup + 1 + k)
    dt = time.perf_counter() - t0
    payload = 2 * sessions * CTX * TOKEN_BYTES_ALL * steps * reps
    sample = (f"{steps} steps x {reps} wave(s) x {sessions} sessions x {CTX} tokens, {dt:.1f} s of CPU work, "
              f"paged cache {nb} blocks ({nb * 2 * L * BS * H * D * 2 / 2**30:.0f} GiB) in host RAM, RAW bf16, "
              f"{threads} threads")
    return payload / dt / 1e9, dt / steps * 1e3, threads, sample


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    # every step lasts >= 1.5 s of CPU work (the wave repeated), so K steps are seconds, not milliseconds
    gbps, ms, threads, sample = cpu_oracle_run(args.steps, max(args.warmup, 1), min_step_s=1.5)
    line = {
        "impl": "reference", "metric": "kv_offload_GBps", "value": gbps, "unit": "GB/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
        "data": "synthetic",
        "config": workload_config(args.gpus),
        "cpu_baseline": {"value": gbps, "unit": "GB/s", "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": gbps, "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "note": "reference path = third-party lmcache wheel, absent from this image; this is the oracle port "
                "(oracle/kv_oracle.c) of its store/retrieve on host cores",
    }
    print(json.dumps(line), flush=True)


def workload_config(n_gpus: int) -> dict:
    return {"workload": "multi-round-qa 2K-ctx wave: 16 sessions x 2048 tokens, Llama-3-8B KV "
                        "(L32 H8 D128 bf16, block 16, chunk 256), store+retrieve per step",
            "tokens_per_step_per_gpu": SESSIONS * CTX, "paged_blocks": NB,
            "l2_policy": "inputs (4 GiB/direction/step) larger than L2; no explicit flush",
            "parallelism": f"{n_gpus} independent replicas, one per GPU, no collective"}


# ------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------
def run_ours(args):
    import torch
    import torch.distributed as dist

    from b200kv import FMT_FP8, FMT_Q4, FMT_RAW, KVEngine, KVGeometry, KVPool

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a B200: the b200kv engine has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device(f"cuda:{local}")
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x: float) -> float:
        if world == 1:
            return x
        t = torch.tensor([x], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def gather_objects(obj):
        if world == 1:
            return [obj]
        out = [None] * world
        dist.all_gather_object(out, obj)
        return out

    geom = KVGeometry(L, H, D, NB, BS, C, 2, 0, FMT_RAW)
    g = torch.Generator(device=dev).manual_seed(rank)
    caches = [torch.randn((2, NB, BS, H, D), generator=g, device=dev, dtype=torch.float32).bfloat16()
              for _ in range(L)]
    n_chunks_step = SESSIONS * CTX // C
    pool = KVPool(None, (n_chunks_step + n_chunks_step // 2) * geom.chunk_bytes, geom.chunk_bytes, 1)
    # staging ring sized to absorb one whole wave per direction (store half + load half): a gather
    # never has to wait for the PCIe drain of an earlier session, so the compute stream is never
    # held back by store traffic (production default is 1 GiB, B200KV_STAGING_MB)
    eng = KVEngine(geom, pool, local, staging_bytes=2 * n_chunks_step * geom.chunk_bytes, owner=rank)
    eng.register_kv_caches(caches)
    # where the engine put this rank's pinned pool (it binds the pages to the GPU's own NUMA node when it
    # pins them, csrc/b200kv_engine.cu place_pool_pages) and where the kernel says they are
    placement = {"rank": rank, "policy": eng.numa_placement(),
                 "pages_per_node": numa_nodes_of(pool.slot_view(0).ctypes.data)}

    perm = torch.randperm(NB, generator=torch.Generator().manual_seed(1234)).numpy()
    dperm = torch.randperm(NB, generator=torch.Generator().manual_seed(4321)).numpy()
    nblk = CTX // BS
    src_maps = [slot_map(perm[s * nblk:(s + 1) * nblk], CTX) for s in range(SESSIONS)]
    dst_maps = [slot_map(dperm[s * nblk:(s + 1) * nblk], CTX) for s in range(SESSIONS)]
    all_src = np.concatenate(src_maps)
    all_dst = np.concatenate(dst_maps)
    stream = torch.cuda.current_stream()

    dumps = {}   # name -> array: what the timed legs computed in their last step (rank 0, --dump-outputs)
    dumping = bool(args.dump_outputs) and rank == 0
    if dumping:
        dump_slots = torch.as_tensor(np.sort(all_dst[np.random.default_rng(7).choice(len(all_dst), DUMP_TOKENS, replace=False)]),
                                     device=dev)
        dst_blocks = torch.as_tensor(dperm[:SESSIONS * nblk].copy(), device=dev)

    def dump_pages(leg, masks=None):
        """The pages the last step wrote into (every session's destination blocks): K and V of DUMP_TOKENS
        seeded tokens in every layer, a float64 sum per (layer, K|V, block) over all of them, and the
        retrieve masks the caller was given."""
        if masks is not None:
            dumps[f"{leg}_ret_mask"] = masks.astype(np.float32)
        dumps[f"{leg}_kv_rows"] = torch.stack([c.view(2, NB * BS, H, D)[:, dump_slots] for c in caches]).float().cpu().numpy()
        dumps[f"{leg}_block_sums"] = torch.stack([c.view(2, NB, -1)[:, dst_blocks].double().sum(-1)
                                                  for c in caches]).cpu().numpy()

    # ---- e2e leg: store + retrieve through the engine, host pool in the loop ------------------
    def e2e_step(step):
        # every session is stored, and retrieved as soon as ITS store has been committed to the
        # host index; retrieves of early sessions overlap the D2H of later ones (PCIe is full duplex)
        toks = [session_tokens(rank, step, s) for s in range(SESSIONS)]
        tickets = [eng.store(toks[s], None, src_maps[s], stream=stream) for s in range(SESSIONS)]
        masks = []
        for s in range(SESSIONS):
            eng.wait(tickets[s])
            masks.append(eng.retrieve(toks[s], None, dst_maps[s], stream=stream))
        return np.stack(masks)

    sampler = ClockSampler(local) if rank == 0 else None   # nvidia-smi needs ~1 s to start emitting
    for w in range(args.warmup):
        assert e2e_step(w).sum() == SESSIONS * CTX
    torch.cuda.synchronize()
    st0 = eng.stats()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    ev0.record(stream)
    for k in range(args.steps):
        got = e2e_step(args.warmup + k)
        assert got.sum() == SESSIONS * CTX, got.sum()
    eng.wait_all()
    ev1.record(stream)
    torch.cuda.synchronize()
    barrier()
    my_e2e_ms = ev0.elapsed_time(ev1) / args.steps
    if dumping:
        dump_pages("e2e", got)
    e2e_ms = max_over_ranks(my_e2e_ms)
    st1 = eng.stats()
    e2e_payload = 2 * SESSIONS * CTX * TOKEN_BYTES_ALL
    e2e_gbps = world * e2e_payload / (e2e_ms * 1e-3) / 1e9

    # ---- value leg: the same tokens, device-resident (HBM only) ---------------------------------
    dbuf = torch.empty(n_chunks_step * geom.chunk_bytes, dtype=torch.uint8, device=dev)

    def dev_step():
        eng.gather(all_src, dbuf.data_ptr(), stream)
        eng.scatter(all_dst, dbuf.data_ptr(), stream)

    for w in range(args.warmup):
        dev_step()
    torch.cuda.synchronize()
    st2 = eng.stats()
    gather_ms = []
    barrier()
    ev0.record(stream)
    for k in range(args.steps):
        dev_step()
        # kernel-only durations of this step's launches (CUDA events recorded by the library on
        # the launching stream); reading them synchronises the stream, which the next launch
        # would do anyway through the stream order.
        gather_ms.append((eng.last_kernel_ms(0), eng.last_kernel_ms(1)))
    ev1.record(stream)
    torch.cuda.synchronize()
    barrier()
    dev_ms = max_over_ranks(ev0.elapsed_time(ev1)) / args.steps
    st3 = eng.stats()
    if dumping:
        vals = dbuf.view(torch.bfloat16)
        pick = np.sort(np.random.default_rng(8).integers(0, vals.numel(), DUMP_CHUNK_VALUES))
        dumps["dev_chunks_sample"] = vals[torch.as_tensor(pick, device=dev)].float().cpu().numpy()
        dumps["dev_chunk_sums"] = np.array([float(x.double().sum()) for x in vals.view(n_chunks_step, -1)])
        dump_pages("dev")
    clocks = sampler.stop() if sampler else None
    value_gbps = world * e2e_payload / (dev_ms * 1e-3) / 1e9
    g_ms = float(np.mean([a for a, _ in gather_ms]))
    s_ms = float(np.mean([b for _, b in gather_ms]))

    # ---- decode-jitter leg (extra): a fixed compute kernel on the compute stream, alone and while a
    # 4 GiB store wave drains through the engine's low-priority streams (SURVEY §7 step 4) ----------
    jitter = None
    if rank == 0:
        try:
            xa = torch.randn((4096, 4096), device=dev, dtype=torch.bfloat16)
            xb = torch.randn((4096, 4096), device=dev, dtype=torch.bfloat16)
            big = torch.empty(1 << 28, device=dev, dtype=torch.bfloat16)     # 512 MiB: a decode step is HBM-bound

            def decode_like():           # weight-streaming (HBM) + a small GEMM, ~0.3 ms like one decode layer group
                big.mul_(1.0)
                torch.mm(xa, xb)

            def time_steps(n, with_store):
                evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(n)]
                tick = []
                if with_store:
                    toks = [session_tokens(rank, 5000 + with_store, s_) for s_ in range(SESSIONS)]
                    tick = [eng.store(toks[s_], None, src_maps[s_], stream=stream) for s_ in range(SESSIONS)]
                for e0, e1 in evs:
                    e0.record(stream)
                    decode_like()
                    e1.record(stream)
                torch.cuda.synchronize()
                for t_ in tick:
                    eng.wait(t_)
                return np.array([e0.elapsed_time(e1) for e0, e1 in evs])

            time_steps(20, 0)
            quiet = time_steps(200, 0)
            busy = np.concatenate([time_steps(200, k + 1) for k in range(3)])
            jitter = {"kernel": "512 MiB bf16 elementwise + 4096^3 bf16 GEMM per step, 200 steps",
                      "alone_ms_p50": float(np.median(quiet)), "alone_ms_p99": float(np.percentile(quiet, 99)),
                      "during_store_wave_ms_p50": float(np.median(busy)), "during_store_wave_ms_p99": float(np.percentile(busy, 99)),
                      "slowdown_p50": float(np.median(busy) / np.median(quiet)),
                      "note": "store wave = 16 x 2048-token requests (4 GiB gathered + D2H) issued right before the steps; "
                              "gather kernels run on a lowest-priority stream, D2H on the copy engine"}
            del xa, xb, big
        except Exception as e:
            jitter = {"error": repr(e)}

    # ---- peer-pull leg (N>1 only; extra): every rank pulls one wave out of its neighbour's HBM ----
    peer = None
    if world > 1:
        try:
            from b200kv.peers import connect_all_peers, exchange_kv_descriptors
            descs = exchange_kv_descriptors(eng)
            connect_all_peers(eng, descs, rank, device_of_rank=lambda r: r)
            nb_rank = (rank + 1) % world
            # destination pages disjoint from every rank's source pages, so what a neighbour reads is stable
            n_wave_blocks = SESSIONS * nblk
            pull_dst = slot_map(perm[n_wave_blocks:2 * n_wave_blocks], SESSIONS * CTX)
            src_blocks = torch.as_tensor(perm[:n_wave_blocks].copy(), device=dev)
            dst_blocks = torch.as_tensor(perm[n_wave_blocks:2 * n_wave_blocks].copy(), device=dev)
            wts = (torch.arange(BS * H * D, device=dev, dtype=torch.int64) % 65521 + 1)

            def block_sums(blocks):       # position-weighted checksum per (layer, K|V, block): [L, 2, n] int64
                out = torch.empty((L, 2, len(blocks)), dtype=torch.int64, device=dev)
                for l in range(L):
                    x = caches[l].view(torch.int16)[:, blocks].reshape(2, len(blocks), -1).to(torch.int64)
                    out[l] = (x * wts).sum(-1)
                return out

            mine = block_sums(src_blocks)
            all_sums = [torch.empty_like(mine) for _ in range(world)]
            dist.all_gather(all_sums, mine)
            for w in range(max(args.warmup, 1)):
                eng.wait(eng.peer_pull(nb_rank, all_src, pull_dst, stream=stream))
            barrier()
            ev0.record(stream)
            for k in range(args.steps):
                eng.peer_pull(nb_rank, all_src, pull_dst, stream=stream)
            ev1.record(stream)   # the compute stream waits for every pull
            torch.cuda.synchronize()
            barrier()
            pull_ms = max_over_ranks(ev0.elapsed_time(ev1)) / args.steps
            kern_ms = eng.last_kernel_ms(2)
            # every pulled page must equal the neighbour's source page (all layers, K and V, all blocks of the wave)
            bad = int((block_sums(dst_blocks) != all_sums[nb_rank]).sum().item())
            bad_total = sum(gather_objects(bad))
            per_gpu = SESSIONS * CTX * TOKEN_BYTES_ALL / (pull_ms * 1e-3) / 1e9
            peer = {"per_gpu_GBps": per_gpu, "aggregate_GBps": per_gpu * world, "ms_per_wave": pull_ms,
                    "kernel_ms": kern_ms, "kernel_GBps": SESSIONS * CTX * TOKEN_BYTES_ALL / (kern_ms * 1e-3) / 1e9,
                    "nvlink_peak_GBps": 770.0, "peak_kind": "B200_PROFILING.md measured peer copy per direction",
                    "frac_of_peak": SESSIONS * CTX * TOKEN_BYTES_ALL / (kern_ms * 1e-3) / 1e9 / 770.0,
                    "pattern": "rank r reads rank (r+1)%N: in-kernel P2P loads, no staging, no NCCL",
                    "verified": bad_total == 0, "mismatching_tiles": bad_total,
                    "checked_tiles_per_rank": int(mine.numel()),
                    "check": "position-weighted int64 checksum of every pulled (layer, K|V, block) tile vs the "
                             "checksum the owner computed of its source tile before the pulls"}
            if bad_total:
                raise SystemExit(f"peer pull moved wrong bytes: {bad_total} tiles differ from the owner's")
        except SystemExit:
            raise
        except Exception as e:  # never lose the headline line to the extra leg
            peer = {"error": repr(e)}

    eng.close()
    pool.close()

    # ---- compressed-format legs (extra, not the headline): the same wave in FP8 and Q4 ------------
    def format_leg(fmt, salt, leg):
        gq = KVGeometry(L, H, D, NB, BS, C, 2, 0, fmt)
        poolq = KVPool(None, (n_chunks_step + n_chunks_step // 2) * gq.chunk_bytes, gq.chunk_bytes, 1)
        eq = KVEngine(gq, poolq, local, staging_bytes=2 * n_chunks_step * gq.chunk_bytes, owner=rank)
        eq.register_kv_caches(caches)
        bq = torch.empty(n_chunks_step * gq.chunk_bytes, dtype=torch.uint8, device=dev)

        def q_e2e(step):
            toks = [session_tokens(rank, salt + step, s_) for s_ in range(SESSIONS)]
            tickets = [eq.store(toks[s_], None, src_maps[s_], stream=stream) for s_ in range(SESSIONS)]
            masks = []
            for s_ in range(SESSIONS):
                eq.wait(tickets[s_])
                masks.append(eq.retrieve(toks[s_], None, dst_maps[s_], stream=stream))
            return np.stack(masks)

        for w in range(max(args.warmup, 1)):
            q_e2e(w)
            eq.gather(all_src, bq.data_ptr(), stream)
            eq.scatter(all_dst, bq.data_ptr(), stream)
        barrier()
        ev0.record(stream)
        for k in range(args.steps):
            masks = q_e2e(args.warmup + k)
        eq.wait_all()
        ev1.record(stream)
        torch.cuda.synchronize()
        barrier()
        q_ms = max_over_ranks(ev0.elapsed_time(ev1)) / args.steps
        if dumping:
            dump_pages(leg, masks)
        km = []
        for k in range(args.steps):
            eq.gather(all_src, bq.data_ptr(), stream)
            eq.scatter(all_dst, bq.data_ptr(), stream)
            km.append((eq.last_kernel_ms(0), eq.last_kernel_ms(1)))
        torch.cuda.synchronize()
        pack, unpack = float(np.mean([a_ for a_, _ in km])), float(np.mean([b_ for _, b_ in km]))
        algo = SESSIONS * CTX * (TOKEN_BYTES_ALL + gq.payload_bytes_per_token)      # HBM read bf16 + write packed
        res = {"e2e_tokens_per_s": world * SESSIONS * CTX * 2 / (q_ms * 1e-3),
               "e2e_equiv_bf16_GBps": world * e2e_payload / (q_ms * 1e-3) / 1e9, "e2e_ms_per_step": q_ms,
               "host_link_bytes_per_token": gq.payload_bytes_per_token,
               "pack_kernel_ms": pack, "unpack_kernel_ms": unpack,
               "pack_kernel_algo_GBps": algo / (pack * 1e-3) / 1e9, "unpack_kernel_algo_GBps": algo / (unpack * 1e-3) / 1e9}
        eq.close()
        poolq.close()
        del bq
        return res

    fp8 = q4 = None
    if not args.no_fp8:
        fp8 = format_leg(FMT_FP8, 1000, "fp8")
        try:
            q4 = format_leg(FMT_Q4, 2000, "q4")
        except Exception as e:
            q4 = {"error": repr(e)}

    # ---- host-link ceiling for the e2e number: measured live at EVERY N, all ranks copying at once ---
    link = None
    try:
        nbytes = 1 << 30
        h_a = torch.empty(nbytes, dtype=torch.uint8).pin_memory()
        h_b = torch.empty(nbytes, dtype=torch.uint8).pin_memory()
        d_a = torch.empty(nbytes, dtype=torch.uint8, device=dev)
        d_b = torch.empty(nbytes, dtype=torch.uint8, device=dev)
        s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()

        def timed(fn, reps=4):
            fn()
            barrier()
            ev0.record(stream)
            for _ in range(reps):
                fn()
            ev1.record(stream)
            torch.cuda.synchronize()
            mine_ms = ev0.elapsed_time(ev1) / reps
            barrier()
            return max_over_ranks(mine_ms)

        def both():
            s1.wait_stream(stream)
            s2.wait_stream(stream)
            with torch.cuda.stream(s1):
                d_a.copy_(h_a, non_blocking=True)
            with torch.cuda.stream(s2):
                h_b.copy_(d_b, non_blocking=True)
            stream.wait_stream(s1)
            stream.wait_stream(s2)

        link = {"h2d_GBps": world * nbytes / timed(lambda: d_a.copy_(h_a, non_blocking=True)) / 1e6,
                "d2h_GBps": world * nbytes / timed(lambda: h_b.copy_(d_b, non_blocking=True)) / 1e6,
                "duplex_total_GBps": world * 2 * nbytes / timed(both) / 1e6,
                "how": f"cudaMemcpyAsync of 1 GiB pinned (cudaHostAlloc) buffers on all {world} GPU(s) at the same time, "
                       "CUDA events, max over ranks, this run (aggregate over the GPUs)"}
        del h_a, h_b, d_a, d_b
    except Exception as e:
        link = {"error": repr(e)}

    if dumping:
        total = sum(a.nbytes for a in dumps.values())
        assert total <= DUMP_LIMIT_BYTES, total
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, a in dumps.items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), a)

    per_rank = gather_objects({**placement, "e2e_ms_per_step": my_e2e_ms,
                               "e2e_GBps": e2e_payload / (my_e2e_ms * 1e-3) / 1e9})
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    pk, pk_kind = peaks()
    launch_tokens = SESSIONS * CTX
    achieved = launch_tokens * ALGO_BYTES_PER_TOKEN / (g_ms * 1e-3) / 1e9
    traffic, traffic_src = None, None
    tpath = os.path.join(ROOT, "profiles", "traffic_gather.json")
    if os.path.exists(tpath):
        try:
            tj = json.load(open(tpath))
            traffic = tj.get("dram_bytes_per_launch")
            traffic_src = "static: " + str(tj.get("source", "ncu --set full capture under profiles/")) + \
                          " (not re-measured in this run; a bench run is never profiled)"
        except Exception:
            traffic = None
    cpu_gbps, cpu_ms, cpu_threads, cpu_sample = cpu_oracle_run(3, 1, target_s=10.0)
    line = {
        "metric": "kv_offload_GBps", "value": value_gbps, "unit": "GB/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dev_ms,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
        "data": "synthetic", "config": workload_config(world),
        "e2e": {"value": e2e_gbps, "unit": "GB/s", "ms_per_step": e2e_ms,
                "h2d_bytes_per_step": (st1["h2d_bytes"] - st0["h2d_bytes"]) // args.steps,
                "d2h_bytes_per_step": (st1["d2h_bytes"] - st0["d2h_bytes"]) // args.steps,
                "kv_ttft_ms_per_2k_ctx_request": e2e_ms / (2 * SESSIONS)},
        "gpu_launches": (st1["n_kernel_launches"] - st0["n_kernel_launches"]) + (st3["n_kernel_launches"] - st2["n_kernel_launches"]),
        "roofline": {"bound": "hbm", "kernel": "kv_bulk_copy_kernel<store> (RAW gather, device-resident leg)",
                     "achieved": achieved, "peak": pk["hbm_gbs"], "unit": "GB/s", "frac": achieved / pk["hbm_gbs"],
                     "peak_kind": f"{pk_kind} MEASURED_PEAKS.json hbm_gbs (burst copy)",
                     "launch_ms": g_ms, "scatter_launch_ms": s_ms,
                     "scatter_achieved": launch_tokens * ALGO_BYTES_PER_TOKEN / (s_ms * 1e-3) / 1e9,
                     "algo_bytes_per_launch": launch_tokens * ALGO_BYTES_PER_TOKEN, "traffic": traffic,
                     "traffic_source": traffic_src},
        "roofline_e2e": None if not link or "error" in link else {
            "bound": "host link (PCIe + host memory system)", "achieved": e2e_gbps, "peak": link["duplex_total_GBps"],
            "unit": "GB/s", "frac": e2e_gbps / link["duplex_total_GBps"],
            "note": f"store D2H and retrieve H2D overlap (full duplex); peak = duplex pinned copy measured with all "
                    f"{world} GPU(s) copying at once, i.e. the ceiling this box gives {world} replica(s)", **link},
        "per_rank": per_rank,
        "cpu_baseline": {"value": cpu_gbps, "unit": "GB/s", "cores": cpu_threads, "kind": "port",
                         "sample": cpu_sample, "ms_per_step": cpu_ms},
        "clocks": clocks,
        "fp8": fp8,
        "q4": q4,
        "decode_jitter": jitter,
        "peer_pull": peer,
    }
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    sys.dont_write_bytecode = True   # the project modules imported below are in a tree bench.py leaves as it was
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-fp8", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write a seeded sample of what every timed leg computed in its last "
                         "step as DIR/<name>.npy (float32 / float64, ~40 MiB)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of the GPU arm (--impl ours)")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
