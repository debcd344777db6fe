#!/usr/bin/env python
"""bench.py -- secp256k1 verifies/sec of the go-ibft message-verification hot path on N B200s (one process per GPU).

A "step" is one pass of the hot path over one batch: the 10k-validator COMMIT round of SURVEY.md §8(d) config 3
(10,000 committed seals + 10,000 COMMIT sender signatures, 1 % adversarial, weighted voting power) replicated to
ITEMS_PER_GPU = 2^20 packed tuples per GPU (128 MiB of tuples: larger than the 126 MB L2, so no flush is needed between
iterations).  Every step runs: K1+K2 recover kernel over the rank's shard -> (N>1: one NCCL all-gather of the
pass/fail bitmap words) -> K3 quorum kernels over the complete bitmap.

  value   whole-job verifies/s with the tuples resident in HBM (CUDA events on the launching stream, max over ranks)
  e2e     the same metric through the host-buffer C-ABI call (ibft_verify_batch): H2D of the tuples and D2H of the
          bitmap + quorum results inside the timed region
  roofline  integer-issue roofline: verifies/s x 5.0e5 IMAD-class instructions (SURVEY.md §8d) / measured IMAD peak
  cpu_baseline / --impl reference   the C oracle (a port; the Go reference has no crypto and no toolchain here) on the
          box's host cores, on a bounded sample of the same workload.
  strong_scaling  ONE 10,000-seal round and ONE config-5 backlog (100k messages, 16 heights x 10k validators) split over the N
          ranks, every rank holding only its shard: device-timed latency (H2D .. D2H) p50/p95 per N (go-ibft_b200/sharding.py ShardedVerifier)
  ingress   64 threads of single-message IsValidValidator calls through the reference-facing verifier (the coalescer)
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

ITEMS_PER_GPU = 1 << 20
ALGO_IMAD_PER_VERIFY = 5.0e5      # SURVEY.md §8(d): 2.5e5 MAC32 = 5.0e5 mad.lo+mad.hi class instructions
ALGO_BYTES_PER_VERIFY = 128 + 133 / 2 + 1 / 8  # packed tuple + payload bytes (half the items hash a 133-byte payload) + 1 bit


def load_workload():
    d = np.load(os.path.join(ROOT, "tests", "golden", "config3.npz"))
    return d


def tile_items(items: np.ndarray, n: int) -> np.ndarray:
    reps = (n + len(items) - 1) // len(items)
    return np.ascontiguousarray(np.tile(items, reps)[:n])


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, gpu_index: int):
        super().__init__(daemon=True)
        self.gpu_index = gpu_index
        self.samples = []
        self.stop_flag = threading.Event()
        self.proc = None

    def run(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu_index), f"--query-gpu={q}", "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                if self.stop_flag.is_set():
                    break
                parts = [p.strip() for p in line.split(",")]
                if len(parts) >= 7:
                    self.samples.append(parts)
        except Exception:
            pass

    def stop(self):
        self.stop_flag.set()
        if self.proc:
            try:
                self.proc.terminate()
            except Exception:
                pass

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        sm = sorted(int(float(s[0])) for s in self.samples if s[0].replace(".", "").isdigit())
        mx = [int(float(s[1])) for s in self.samples if s[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [nm for k, nm in enumerate(names) if any(s[3 + k].lower().startswith("active") for s in self.samples)]
        pw = [float(s[2]) for s in self.samples if s[2].replace(".", "").isdigit()]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "power_w_max": max(pw) if pw else None, "samples": len(self.samples)}


def effective_cpus() -> int:
    """Host threads this process can actually run in parallel: the cgroup CPU quota (the GPU boxes expose 128 logical CPUs but
    cap the container at 16 CPUs' worth of time -- oversubscribing the quota makes the CPU baseline SLOWER), else affinity."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if quota != "max":
            n = min(n, max(1, int(int(quota) / int(period))))
    except Exception:
        try:
            q = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            p = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0:
                n = min(n, max(1, q // p))
        except Exception:
            pass
    return n


def cpu_arm(d, tuned: bool):
    """A CPU implementation of the path as fn(items, n_threads) -> bitmap: the plain C oracle (oracle/c/ibft_oracle.c), or the tuned
    arm (oracle/c/fast_recover.c: GLV + wNAF + lazily reduced field, binary inversions -- cross-checked against the plain port in
    tests/test_oracle_crypto.py and against the golden bitmap in every bench run that uses it)."""
    from oracle import coracle as co
    arena = d["arena"].tobytes()
    if tuned:
        co.fast_lib()
        return lambda items, n_threads: co.fast_verify_batch(items, arena, d["addrs"], n_threads)
    co.lib()
    gt = [0] * len(d["groups"])
    return lambda items, n_threads: co.verify_batch(items, arena, tables=[d["addrs"]], group_table=gt, n_threads=n_threads)


def tuned_arm_usable(d, items) -> bool:
    """the tuned arm is only ever timed after it reproduced the golden verdicts of the workload on this host"""
    try:
        probe = items[:2048]
        gold = np.unpackbits(d["bitmap"].view(np.uint8), bitorder="little")[: len(probe)]
        got = np.unpackbits(cpu_arm(d, True)(probe, 4).view(np.uint8), bitorder="little")[: len(probe)]
        return bool(np.array_equal(got, gold))
    except Exception:
        return False


def cpu_baseline(d, items, n_threads: int, target_seconds: float = 12.0, tuned: bool = False):
    """Times a CPU arm (kind "port") on a bounded sample of the same workload."""
    run = cpu_arm(d, tuned)
    probe = items[: max(64, 8 * n_threads)]
    t0 = time.perf_counter()
    run(probe, n_threads)
    rate = len(probe) / (time.perf_counter() - t0)
    n = int(min(1 << 18, max(len(probe), rate * target_seconds)))
    sample = tile_items(items, n)  # the config-3 batch, repeated as often as the time budget allows
    t0 = time.perf_counter()
    bm = run(sample, n_threads)
    dt = time.perf_counter() - t0
    return n / dt, n, bm


def cpu_baseline_legs(d, base_items, cores, scale: float = 1.0):
    """The cpu_baseline object of the JSON line: the fastest verified CPU arm as `value` (tuned arm when it reproduces the golden
    verdicts on this host, else the plain port), the plain port beside it, and the OpenSSL arm when libcrypto is there.
    scale < 1 shortens the samples (CPU-side self-test of this function)."""
    gold_bits = np.unpackbits(d["bitmap"].view(np.uint8), bitorder="little")[: len(base_items)]
    matches = lambda bm, n: bool(np.array_equal(np.unpackbits(bm.view(np.uint8), bitorder="little")[:n],  # noqa: E731
                                                np.tile(gold_bits, n // len(base_items) + 1)[:n]))
    vp, n_p, bm_p = cpu_baseline(d, base_items, cores, target_seconds=6.0 * scale)
    vp1, _, _ = cpu_baseline(d, base_items, 1, target_seconds=2.0 * scale)
    plain = {"value": vp, "unit": "verifies/s", "cores": cores, "single_thread": vp1, "matches_golden": matches(bm_p, n_p),
             "arm": "plain C oracle (oracle/c/ibft_oracle.c: fixed 4-bit windows, Fermat inversions, no endomorphism) -- the checker of the CUDA path"}
    threads_rule = "threads = the container's cgroup CPU quota (cpu.max), capped by affinity -- the same rule in BENCH and SCALE runs"
    if tuned_arm_usable(d, base_items):
        v, n_s, bm = cpu_baseline(d, base_items, cores, target_seconds=8.0 * scale, tuned=True)
        v1, _, _ = cpu_baseline(d, base_items, 1, target_seconds=2.0 * scale, tuned=True)
        out = {"value": v, "unit": "verifies/s", "cores": cores, "kind": "port",
               "arm": "tuned C arm (oracle/c/fast_recover.c: GLV + wNAF, 4x64-bit lazily reduced field, binary inversions)",
               "sample": f"{n_s} items (the config-3 batch repeated), {cores} threads, ~{8.0 * scale:g} s",
               "single_thread": v1, "matches_golden": matches(bm, n_s), "logical_cpus_visible": os.cpu_count(),
               "threads_rule": threads_rule, "plain_port": plain}
    else:
        out = dict(plain, kind="port", sample=f"{n_p} items (the config-3 batch repeated), {cores} threads, ~{6.0 * scale:g} s",
                   logical_cpus_visible=os.cpu_count(), threads_rule=threads_rule)
    # a third arm with a LIBRARY's point arithmetic (BASELINE.md §3 planned OpenSSL): OpenSSL 3's generic-curve code is slower
    # than the plain port on secp256k1; a libsecp256k1-class library (5x52 limbs, assembly: ~2x the tuned arm per core) is not
    # available offline
    from oracle import coracle as co
    if co.ossl_lib() is not None:
        sub = tile_items(base_items, max(256, int(4096 * max(1, cores // 4) * scale)))
        t0 = time.perf_counter()
        bm_o = co.ossl_verify_batch(sub, d["arena"].tobytes(), d["addrs"], cores)
        dt = time.perf_counter() - t0
        out["openssl_arm"] = {"value": len(sub) / dt, "unit": "verifies/s", "cores": cores, "kind": "openssl-3 EC_POINT_mul",
                              "matches_golden": matches(bm_o, len(sub))}
    return out


def run_reference(args):
    """--impl reference: the reference's CPU implementation of the path.  go-ibft verifies serially and delegates the
    arithmetic to the embedder (no crypto in the tree, no Go toolchain on the box), so this arm times the oracle port with
    all host threads -- the "goroutine-parallel CPU verify" the north star asks for."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    d = load_workload()
    items = np.ascontiguousarray(d["items"]).view(_item_dtype()).reshape(-1)
    cores = effective_cpus()
    # the fastest CPU arm this repo can field: the tuned one (GLV + wNAF) once it has reproduced the golden verdicts on this host,
    # else the plain port
    gold_all = np.unpackbits(d["bitmap"].view(np.uint8), bitorder="little")[: len(items)]
    v = None
    for tuned in ([True, False] if tuned_arm_usable(d, items) else [False]):
        run = cpu_arm(d, tuned)
        arm_name = ("tuned C arm (oracle/c/fast_recover.c: GLV + wNAF, 4x64-bit lazily reduced field)" if tuned
                    else "plain C oracle (oracle/c/ibft_oracle.c)")
        # bounded sample per step: ~2 s of work on all host threads (calibrated once), the config-3 batch repeated as needed
        t0 = time.perf_counter()
        run(items[: max(64, 4 * cores)], cores)
        rate = max(64, 4 * cores) / (time.perf_counter() - t0)
        sample_n = int(min(1 << 18, max(256, rate * 2.0)))
        sample = tile_items(items, sample_n)
        for _ in range(args.warmup):
            run(sample[: max(64, cores)], cores)
        t0 = time.perf_counter()
        for _ in range(args.steps):
            bm = run(sample, cores)
        dt = time.perf_counter() - t0
        if np.array_equal(np.unpackbits(bm.view(np.uint8), bitorder="little")[:sample_n], np.tile(gold_all, sample_n // len(items) + 1)[:sample_n]):
            v = sample_n * args.steps / dt
            break
    if v is None:
        raise SystemExit("bench --impl reference: the CPU arm's verdicts differ from the golden fixture")
    line = {"impl": "reference", "metric": "secp256k1_verifies_per_sec", "value": v, "unit": "verifies/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u32 (256-bit modular integer)", "data": "synthetic",
            "config": workload_config(args.gpus), "gpu_launches": 0,
            "cpu_baseline": {"value": v, "unit": "verifies/s", "cores": cores, "kind": "port", "arm": arm_name, "matches_golden": True,
                             "sample": f"{sample_n} items of the config-3 batch per step (bounded sample), {cores} threads"},
            "e2e": {"value": v, "unit": "verifies/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(line)


def _item_dtype():
    import ibft_b200 as ib
    return ib.ITEM_DTYPE


def workload_config(n_gpus):
    return {"workload": "config3: 10k-validator COMMIT round (10,000 committed seals + 10,000 COMMIT sender signatures, weighted "
                        "voting power, 1% adversarial) replicated to 2^20 packed tuples per GPU",
            "items_per_gpu": ITEMS_PER_GPU, "global_items": ITEMS_PER_GPU * n_gpus, "validators": 10000,
            "parallelism": f"shard{n_gpus} + one all-gather of (bitmap words | partial voted sets)" if n_gpus > 1 else "single",
            "l2": "inputs (128 MiB of tuples per GPU) exceed the 126 MB L2; no flush needed"}


DUMP_BYTES_MAX = 64 * 10**6


def dump_outputs(out_dir, bitmap_words, results, n_items, result_dtype):
    """Writes what a caller of the timed path receives from its last step, so that two builds can be compared output for
    output on identical inputs (the tiled config-3 fixture: nothing in the timed path's inputs is random):
      verdicts.npy       float32, the 0/1 verdict of every tuple; when that would exceed the 64 MB budget, a fixed seeded sample
                         of the tuples, whose indices are in verdicts_index.npy (float64)
      quorum_counts.npy  float64 (groups, 3): n_valid, n_distinct, has_quorum of every group
      quorum_power.npy   float64 (groups, 10): the 320-bit voted power of every group as little-endian 32-bit limbs (exact)"""
    os.makedirs(out_dir, exist_ok=True)
    bits = np.unpackbits(bitmap_words.cpu().numpy().view(np.uint8), bitorder="little")[:n_items]
    res = results.cpu().numpy().view(result_dtype)
    counts = np.stack([res["n_valid"], res["n_distinct"], res["has_quorum"]], axis=1).astype(np.float64)
    power = np.ascontiguousarray(res["power"]).view(np.uint32).astype(np.float64)
    budget = DUMP_BYTES_MAX - counts.nbytes - power.nbytes - 4 * 4096   # room for the .npy headers
    if 4 * n_items > budget:
        idx = np.sort(np.random.default_rng(0).choice(n_items, budget // 12, replace=False))  # 4 B verdict + 8 B index each
        bits = bits[idx]
        np.save(os.path.join(out_dir, "verdicts_index.npy"), idx.astype(np.float64))
    np.save(os.path.join(out_dir, "verdicts.npy"), bits.astype(np.float32))
    np.save(os.path.join(out_dir, "quorum_counts.npy"), counts)
    np.save(os.path.join(out_dir, "quorum_power.npy"), power)


def _pct(xs, q):
    xs = sorted(xs)
    return xs[min(len(xs) - 1, int(len(xs) * q))] if xs else None


def load_full_cache(name):
    """The full-size BASELINE configs 4 / 5 (tests/workloads.py config4_n10k / config5_full) as regenerated and cached by
    __graft_entry__.build() / the test suite under tests/golden/_cache/ (bench.py itself never runs the generator: it lives with
    the oracle).  Returns (workload, pin) or (None, reason)."""
    import hashlib
    import pickle
    cache = os.path.join(ROOT, "tests", "golden", "_cache", name + ".pkl")
    pin_path = os.path.join(ROOT, "tests", "golden", name + "_pin.npz")
    if not os.path.exists(cache) or not os.path.exists(pin_path):
        return None, f"{cache} absent (python -c 'import __graft_entry__ as g; g.build()' regenerates it)"
    pin = np.load(pin_path)
    with open(cache, "rb") as f:
        w = pickle.load(f)
    sha = lambda a: hashlib.sha256(a if isinstance(a, (bytes, bytearray)) else np.ascontiguousarray(a).tobytes()).digest()  # noqa: E731
    if sha(w["items"]) != bytes(pin["sha_items"]) or sha(w["arena"]) != bytes(pin["sha_arena"]):
        return None, "cached workload does not match the committed fingerprint"
    return w, pin


def strong_scaling_legs(args, ib, eng_weak, d, base_items, groups3, world, rank, local_rank, stream):
    """ONE 10,000-seal COMMIT round and ONE config-5 backlog split over the `world` ranks: each rank holds only its shard (tuples
    and payload bytes), verifies it, marks its votes, and ONE all-gather of (bitmap words | partial voted sets | counts) gives
    every rank the complete bitmap and the quorum results.  Timed host-to-host per repetition: barrier, then pinned host shard ->
    H2D -> kernels -> collective -> merge -> D2H of results + bitmap on every rank; the per-repetition time is the MAX over ranks.
    The bitmap of every repetition's configuration is checked against the golden fixture / the committed pin."""
    import importlib
    import torch
    import torch.distributed as dist
    sharding = importlib.import_module("go-ibft_b200.sharding")
    out = {"n_gpus": world, "timing": "CUDA events on the rank's stream around H2D of the shard .. kernels .. exchange .. D2H of results+bitmap, after a barrier; max over ranks per repetition",
           "collective": "one all_gather_into_tensor of (bitmap words | partial voted sets | valid counts) per round"}

    def timed(sv, reps):
        """per call: barrier, then H2D of the shard + kernels + exchange + D2H of the results, timed ON THE DEVICE (CUDA events on the
        stream everything is enqueued on), max over ranks per repetition.  A peer-memory exchange that times out on one rank is recorded
        and agreed on by all ranks after the loop (the barrier pattern stays intact), then raised everywhere."""
        ts, failed, res, bm = [], 0, None, None
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        for i in range(reps + 5):
            if world > 1:
                dist.barrier()
            torch.cuda.synchronize()
            ev0.record(sv.stream)
            sv.enqueue()
            ev1.record(sv.stream)
            try:
                res, bm = sv.finish()
            except RuntimeError:
                failed = 1
            ts.append(ev0.elapsed_time(ev1) * 1e3)
        t = torch.tensor(ts[5:] + [float(failed)], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        t = t.cpu()
        if float(t[-1]) != 0.0:
            raise RuntimeError("peer-memory exchange timed out on at least one rank")
        return [float(x) for x in t[:-1]], res, bm

    # ---- (a) one 10,000-seal round (config 3's committed seals)
    seal_group = list(d["groups"]).index("COMMIT_SEAL")
    sel = base_items["group"] == seal_group
    seals = np.ascontiguousarray(base_items[sel])
    gold = np.unpackbits(d["bitmap"].view(np.uint8), bitorder="little")[: len(base_items)][sel]
    n = len(seals)
    lo, hi = sharding.shard_bounds(n, world, rank)
    li, la = sharding.rebase_shard(seals, np.zeros(0, np.uint8), lo, hi)
    sv = sharding.ShardedVerifier(eng_weak, n, groups3, world, rank, li, la, stream)
    ts, res, bm = timed(sv, args.latency_reps)
    bits = np.unpackbits(bm.view(np.uint8), bitorder="little")[:n]
    if not np.array_equal(bits, gold):
        raise SystemExit("bench: sharded 10k round: bitmap differs from the golden fixture")
    out["round10k"] = {"workload": "ONE 10k-validator COMMIT round: 10,000 committed seals, weighted quorum", "items": n,
                       "items_per_gpu": int(hi - lo), "p50_us": _pct(ts, 0.5), "p95_us": _pct(ts, 0.95), "reps": len(ts),
                       "exchange": "nccl all_gather_into_tensor + merge kernel",
                       "has_quorum": bool(res[seal_group]["has_quorum"]), "bitmap_matches_golden": True}
    # the same round with the exchange done by ONE kernel over NVLink peer memory (no library collective)
    try:
        svp = sharding.ShardedVerifier(eng_weak, n, groups3, world, rank, li, la, stream, exchange="p2p")
        ts, resp, bmp = timed(svp, args.latency_reps)
        svp.close()
        if not np.array_equal(np.unpackbits(bmp.view(np.uint8), bitorder="little")[:n], gold) or resp.tobytes() != res.tobytes():
            raise SystemExit("bench: sharded 10k round (peer-memory exchange): results differ")
        out["round10k"]["peer_memory_exchange"] = {"p50_us": _pct(ts, 0.5), "p95_us": _pct(ts, 0.95), "reps": len(ts),
                                                   "exchange": "k_quorum_exchange: publish flag, wait for peers, merge out of peer memory (CUDA IPC over NVLink); "
                                                               "all-gather + merge in one launch", "results_equal_nccl_path": True}
    except (RuntimeError, AttributeError) as ex:
        out["round10k"]["peer_memory_exchange"] = {"unavailable": str(ex)[:200]}
    # ---- (b) config 5 at its stated size
    w, pin = load_full_cache("config5")
    if w is None:
        out["config5"] = {"skipped": pin}
    else:
        items, arena = w["items"], np.frombuffer(w["arena"], np.uint8)
        n = len(items)
        lo, hi = sharding.shard_bounds(n, world, rank)
        eng5 = ib.Engine(device=local_rank, max_items=max(32, hi - lo), max_payload_bytes=1 << 24, max_groups=w["n_groups"], max_table_slots=16,
                         max_validators=10_000)
        for k in range(16):
            eng5.set_validators(k, w["heights"][k], w["tables"][k], w["powers"])
        groups5 = eng5.groups(w["n_groups"], slot=w["group_table"])
        li, la = sharding.rebase_shard(items, arena, lo, hi)
        sv5 = sharding.ShardedVerifier(eng5, n, groups5, world, rank, li, la, stream)
        ts, res, bm = timed(sv5, max(20, args.latency_reps // 4))
        p2p5 = None
        try:
            sv5p = sharding.ShardedVerifier(eng5, n, groups5, world, rank, li, la, stream, exchange="p2p")
            tsp, resp, bmp = timed(sv5p, max(20, args.latency_reps // 4))
            sv5p.close()
            if not np.array_equal(bmp, pin["bitmap"]) or resp.tobytes() != res.tobytes():
                raise SystemExit("bench: sharded config 5 (peer-memory exchange): results differ")
            p2p5 = {"p50_us": _pct(tsp, 0.5), "p95_us": _pct(tsp, 0.95), "results_equal_nccl_path": True}
        except (RuntimeError, AttributeError) as ex:
            p2p5 = {"unavailable": str(ex)[:200]}
        if not np.array_equal(bm, pin["bitmap"]):
            raise SystemExit("bench: sharded config 5: bitmap differs from the committed oracle pin")
        want = pin["results"]
        for g in range(w["n_groups"]):
            if (int(res[g]["n_valid"]), int(res[g]["n_distinct"]), int(res[g]["has_quorum"])) != tuple(int(x) for x in want[g, :3]):
                raise SystemExit("bench: sharded config 5: quorum results differ from the committed oracle pin")
        p50 = _pct(ts, 0.5)
        out["config5"] = {"workload": "100,000 pending messages (144,953 signature tuples), 16 concurrent heights x 10,000-validator tables, "
                                      "45/45/9/1 PREPARE/COMMIT/ROUND_CHANGE/PREPREPARE, 1% adversarial; sharded by contiguous index range",
                          "items": n, "items_per_gpu": int(hi - lo), "payload_bytes_per_gpu": int(la.size), "groups": int(w["n_groups"]),
                          "p50_us": p50, "p95_us": _pct(ts, 0.95), "reps": len(ts), "verifies_per_s_at_p50": n / (p50 * 1e-6),
                          "bitmap_and_quorum_match_pin": True, "peer_memory_exchange": p2p5}
        eng5.close()
    return out


def wire_frames_from_payload_items(items, arena):
    """Gossip frames for the KIND_PAYLOAD tuples of a fixture: PayloadNoSig with the signature field (3) put back right after
    From (field 2) -- the canonical encoding of the signed message (messages/proto/messages.proto:24-44)."""
    frames = []
    a = np.ascontiguousarray(arena).tobytes()
    for it in items:
        p = a[int(it["payload_off"]): int(it["payload_off"]) + int(it["payload_len"])]
        assert p[0] == 0x0A and p[1] < 0x80 and p[2 + p[1]] == 0x12 and p[3 + p[1]] == 20
        cut = 2 + p[1] + 22
        sig = bytes(it["r"]) + bytes(it["s"]) + bytes([int(it["v"])])
        frames.append(p[:cut] + b"\x1a\x41" + sig + p[cut:])
    return frames


def ingress_leg(local_rank, n_threads=64):
    """n_threads threads of SINGLE-message IsValidValidator calls through the reference-facing verifier (the call pattern of
    core/ibft.go:1101-1128): the coalescer turns them into a few device batches.  Every message is asked once per verifier (the
    verdict cache would answer repeats); several verifiers in turn."""
    import importlib
    host = importlib.import_module("go-ibft_b200.host")
    # 64 callers: config 2's 2,000 sender messages; more callers: config 3's 10,000 COMMIT messages (each caller needs a few)
    d2 = np.load(os.path.join(ROOT, "tests", "golden", "config2.npz" if n_threads <= 64 else "config3.npz"))
    import ibft_b200 as ib
    items = np.ascontiguousarray(d2["items"]).view(ib.ITEM_DTYPE).reshape(-1)
    sel = items["kind"] == ib.KIND_PAYLOAD
    frames = wire_frames_from_payload_items(items[sel], d2["arena"])
    # what every frame's answer must be: the BULK path's verdict for the same message (tuple with signer = the frame's From)
    tuples = items[sel].copy()
    a = np.ascontiguousarray(d2["arena"]).tobytes()
    for k, it in enumerate(tuples):
        off = int(it["payload_off"])
        vlen = a[off + 1]
        tuples["signer"][k] = np.frombuffer(a[off + 4 + vlen: off + 24 + vlen], np.uint8)
    e0 = ib.Engine(device=local_rank, max_items=1 << 14, max_payload_bytes=1 << 22, max_groups=8, max_table_slots=2, max_validators=16384)
    e0.set_validators(0, int(d2["meta"][2]), d2["addrs"], d2["powers"])
    bulk, _, _ = e0.verify_batch(tuples, d2["arena"], e0.groups(len(d2["groups"])))
    e0.close()
    gold = np.unpackbits(bulk.view(np.uint8), bitorder="little")[: len(tuples)]
    addrs = [bytes(x) for x in d2["addrs"]]
    lat, elapsed, calls, asked, mismatches = [], 0.0, 0, 0, 0
    for _ in range(8 if n_threads <= 64 else 3):
        c = host.HostContext("gpu", {}, b"", host.EngineParams(local_rank, 1 << 14, 1 << 22, 32, 8, 16384, 0))
        c.set_validators(int(d2["meta"][2]), addrs, None)
        v, l, us = c.ingress_storm(frames, n_threads)
        mismatches += int((v != gold).sum())
        lat.extend(float(x) for x in l)
        elapsed += us
        calls += c.gpu_device_calls()
        asked += c.gpu_ingress_requests()
        c.close()
    if mismatches:
        raise SystemExit("bench: ingress leg: coalesced single-message answers differ from the bulk path's verdicts")
    return {"threads": n_threads, "single_message_calls": asked, "device_calls": calls, "calls_per_device_call": asked / max(1, calls),
            "msgs_per_s": asked / (elapsed * 1e-6), "p50_us": _pct(lat, 0.5), "p95_us": _pct(lat, 0.95),
            "answers_equal_bulk_path": True,
            "note": "IsValidValidator per inbound gossip message from 64 threads (core/ibft.go:1101-1128); a cache miss joins the "
                    "ingress queue, one leader flushes the queue in ONE device call (group commit, no timer)"}


def cpu_latency_legs(d, base_items, cores):
    """Metric 2's CPU side (BASELINE.md §3): the same 10,000 committed seals on the host cores -- all threads, and ONE thread in
    store order (the reference verifies one message at a time under its per-type mutex, messages/messages.go:174-176)."""
    from oracle import coracle as co
    seal_group = list(d["groups"]).index("COMMIT_SEAL")
    seals = np.ascontiguousarray(base_items[base_items["group"] == seal_group])
    gt = [0] * len(d["groups"])
    allc, serial = [], []
    for _ in range(7):
        t0 = time.perf_counter()
        co.verify_batch(seals, b"", tables=[d["addrs"]], group_table=gt, n_threads=cores)
        allc.append((time.perf_counter() - t0) * 1e6)
    for _ in range(3):
        t0 = time.perf_counter()
        co.verify_batch(seals, b"", tables=[d["addrs"]], group_table=gt, n_threads=1)
        serial.append((time.perf_counter() - t0) * 1e6)
    out = {"all_cores_p50": _pct(allc, 0.5), "all_cores_p95": _pct(allc, 0.95), "all_cores_threads": cores, "all_cores_reps": len(allc),
           "serial_reference_semantics_p50": _pct(serial, 0.5), "serial_reps": len(serial),
           "impl": "C oracle port (oracle/c/ibft_oracle.c)"}
    if co.ossl_lib() is not None:
        t0 = time.perf_counter()
        bm = co.ossl_verify_batch(seals, b"", d["addrs"], cores)
        out["openssl_all_cores_us"] = (time.perf_counter() - t0) * 1e6
    if tuned_arm_usable(d, base_items):
        tuned_all, tuned_serial = [], []
        for _ in range(7):
            t0 = time.perf_counter()
            co.fast_verify_batch(seals, b"", d["addrs"], cores)
            tuned_all.append((time.perf_counter() - t0) * 1e6)
        t0 = time.perf_counter()
        co.fast_verify_batch(seals, b"", d["addrs"], 1)
        tuned_serial.append((time.perf_counter() - t0) * 1e6)
        out["tuned_arm"] = {"all_cores_p50": _pct(tuned_all, 0.5), "serial_reference_semantics_p50": _pct(tuned_serial, 0.5),
                            "impl": "tuned C arm (oracle/c/fast_recover.c)"}
    return out


def hash_crossover_leg(eng):
    """IsValidProposalHash for ONE proposal (both sponges in one launch, host buffers in / 32 bytes out) against one CPU core, by
    proposal size; and the batch size from which the device wins at 1 KiB."""
    from oracle import coracle as co
    rng = np.random.default_rng(7)
    rows = []
    for size in (1 << 10, 1 << 16, 1 << 20):
        raw = rng.integers(0, 256, size, dtype=np.uint8).tobytes()
        g, c = [], []
        want = co.keccak256(co.keccak256(raw) + (3).to_bytes(8, "big"))
        for i in range(12):
            t0 = time.perf_counter()
            got = eng.proposal_hash_batch([raw], [3])[0]
            g.append((time.perf_counter() - t0) * 1e6)
            t0 = time.perf_counter()
            co.keccak256(co.keccak256(raw) + (3).to_bytes(8, "big"))
            c.append((time.perf_counter() - t0) * 1e6)
        rows.append({"proposal_bytes": size, "gpu_us_p50": _pct(g[2:], 0.5), "cpu_1core_us_p50": _pct(c[2:], 0.5), "match": got == want})
    batch = []
    raw1k = [rng.integers(0, 256, 1 << 10, dtype=np.uint8).tobytes() for _ in range(4096)]
    for nb in (1, 16, 256, 4096):
        t0 = time.perf_counter()
        eng.proposal_hash_batch(raw1k[:nb], [0] * nb)
        tg = (time.perf_counter() - t0) * 1e6
        t0 = time.perf_counter()
        for r in raw1k[:nb]:
            co.keccak256(co.keccak256(r) + bytes(8))
        batch.append({"proposals": nb, "gpu_us": tg, "cpu_1core_us": (time.perf_counter() - t0) * 1e6})
    return {"single_proposal": rows, "batch_of_1KiB_proposals": batch,
            "note": "a sponge is serial: for ONE proposal the device pays launch + copies and then runs one slow thread, so one CPU core "
                    "wins at every size; the device wins for batches.  The reference asks once per PREPARE and COMMIT (core/ibft.go:858, "
                    ":938); GpuVerifier hashes once per (proposal, round) and answers the other 19,999 calls from its cache."}


def config4_legs(ib, local_rank, stream):
    """BASELINE config 4 at 10k validators.  dedup mode: the 20,003 unique tuples of 10,000 ROUND_CHANGE messages with nested
    prepared certificates (10,000 of them IBFT_KIND_PAYLOAD2: a 1.1 KB head + a shared 909 KB certificate -- 9 GB of sponge input),
    host buffers in, bitmap + decision out.  raw mode: the nested PREPARE checks WITHOUT dedup, a 2^24-tuple slice, device resident."""
    import torch
    w, pin = load_full_cache("config4_n10k")
    if w is None:
        return {"skipped": pin}
    eng = ib.Engine(device=local_rank, max_items=1 << 15, max_payload_bytes=1 << 25, max_groups=4, max_table_slots=2, max_validators=10_000)
    eng.set_validators(0, w["height"], w["addrs"], None)
    g = eng.groups(1)
    ts = []
    for i in range(6):
        t0 = time.perf_counter()
        bm, res, _ = eng.verify_batch(w["items"], w["arena"], g)
        ts.append((time.perf_counter() - t0) * 1e3)
    if not np.array_equal(bm, pin["bitmap"]):
        raise SystemExit("bench: config 4 dedup mode: bitmap differs from the committed oracle pin")
    out = {"dedup_mode": {"tuples": int(len(w["items"])), "round_change_messages": int(w["n"]), "signed_bytes_hashed": int(sum(
        int(it["payload_len"]) + (int.from_bytes(bytes(it["digest"][8:12]), "little") if it["kind"] == 5 else 0) for it in w["items"])),
        "arena_bytes_uploaded": len(w["arena"]), "ms_p50": _pct(ts[1:], 0.5), "bitmap_matches_pin": True,
        "note": "host tuples -> bitmap + quorum on the host; dominated by the 10,000 sender digests (6,700 Keccak permutations each)"}}
    eng.close()
    # raw mode: 2^24 nested PREPARE checks (the 9,999 distinct PREPARE tuples tiled), one device-resident launch
    n_raw = 1 << 24
    prep = w["items"][w["n"] + 1: w["n"] + 1 + (w["n"] - 1)]
    free, _ = torch.cuda.mem_get_info()
    if free < 3 * n_raw * 128:
        out["raw_mode"] = {"skipped": "not enough free device memory for 2^24 tuples"}
        return out
    local, larena = __import__("importlib").import_module("go-ibft_b200.sharding").rebase_shard(prep, np.frombuffer(w["arena"], np.uint8), 0, len(prep))
    big = tile_items(local, n_raw)
    eng = ib.Engine(device=local_rank, max_items=1 << 12, max_payload_bytes=1 << 22, max_groups=4, max_table_slots=2, max_validators=10_000)
    eng.set_validators(0, w["height"], w["addrs"], None)
    eng.bind_groups(eng.groups(1))
    t_items = torch.from_numpy(big.view(np.uint8).reshape(-1, 128)).cuda()
    t_arena = torch.from_numpy(larena.copy()).cuda()
    t_bm = torch.zeros(n_raw // 32, dtype=torch.int32, device="cuda")
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    eng.verify_device(t_items.data_ptr(), n_raw, t_arena.data_ptr(), t_arena.numel(), 0, n_raw, t_bm.data_ptr(), 0, stream.cuda_stream)
    a.record(stream)
    for _ in range(2):
        eng.verify_device(t_items.data_ptr(), n_raw, t_arena.data_ptr(), t_arena.numel(), 0, n_raw, t_bm.data_ptr(), 0, stream.cuda_stream)
    b.record(stream)
    torch.cuda.synchronize()
    ms = a.elapsed_time(b) / 2
    ok = bool((t_bm == -1).all().item())
    out["raw_mode"] = {"tuples": n_raw, "ms_per_launch": ms, "verifies_per_s": n_raw / (ms * 1e-3), "all_valid": ok,
                       "note": "nested PREPARE checks of the certificates without dedup (~10k x 6,667 = 6.7e7 per round): 2^24-tuple slice, tuples resident"}
    del t_items, t_bm
    eng.close()
    return out


_REAL_STDOUT = None


def _claim_stdout():
    """rank 0 prints ONE JSON line on stdout.  Libraries write there too (NCCL's version banner when the box sets
    NCCL_DEBUG=VERSION); NCCL's logging environment is left alone -- instead file descriptor 1 is pointed at stderr for the
    duration of the run and the JSON line goes to the saved original descriptor."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)


def emit(line: dict):
    out = _REAL_STDOUT or sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def main():
    _claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--latency-reps", type=int, default=200)
    ap.add_argument("--no-key-cache-leg", action="store_true", help="skip the extra leg that times the key-registry path")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--skip-extras", action="store_true", help="headline + e2e + strong-scaling legs only (development: short multi-GPU runs)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the verdicts and quorum results of the last timed step to DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of the CUDA path (--impl ours)")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        run_reference(args)
        return

    import torch
    import torch.distributed as dist
    import ibft_b200 as ib

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (there is no CPU fallback)")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    n_gpus = world
    d = load_workload()
    base_items = np.ascontiguousarray(d["items"]).view(ib.ITEM_DTYPE).reshape(-1)
    n_local = ITEMS_PER_GPU
    n_global = n_local * n_gpus
    lo, hi = rank * n_local, (rank + 1) * n_local

    eng = ib.Engine(device=local_rank, max_items=n_local, max_payload_bytes=max(1 << 22, len(d["arena"])), max_groups=8,
                    max_table_slots=2, max_validators=16384)
    eng.set_validators(0, int(d["meta"][2]), d["addrs"], d["powers"])
    groups = eng.groups(len(d["groups"]))
    eng.bind_groups(groups)

    # ---- device-resident inputs: every rank holds ONLY ITS SHARD of the tuples (after the shard-local quorum change nothing reads
    # outside [lo, hi)); the kernels index tuples and bitmap words by GLOBAL item number, so they get rebased pointers
    reps_needed = (n_global + len(base_items) - 1) // len(base_items)
    host_local_np = np.ascontiguousarray(np.tile(base_items, reps_needed)[lo:hi]) if n_gpus > 1 else tile_items(base_items, n_global)
    t_items_local = torch.from_numpy(host_local_np.view(np.uint8).reshape(-1, 128)).cuda()

    class _ItemsView:                      # what the old code called t_items: a base pointer valid for indices [lo, hi)
        def data_ptr(self_inner):
            return t_items_local.data_ptr() - lo * 128
    t_items = _ItemsView()
    t_arena = torch.from_numpy(np.ascontiguousarray(d["arena"])).cuda()
    words_local = n_local // 32
    t_bitmap = torch.zeros(n_global // 32 if world == 1 else 1, dtype=torch.int32, device="cuda")
    t_results = torch.zeros(len(groups) * ib.RESULT_DTYPE.itemsize, dtype=torch.uint8, device="cuda")
    stream = torch.cuda.Stream()  # a real (non-default) stream: the C ABI launches on exactly this one
    torch.cuda.set_stream(stream)

    # N > 1: every rank resolves quorum only for ITS shard; the partial voted sets / counts ride in the same all-gather as the
    # bitmap words (one collective per step), then a tiny merge + reduce runs on every rank.
    if world > 1:
        W = eng.quorum_partial_words()
        t_local = torch.zeros(words_local + W, dtype=torch.int32, device="cuda")
        t_gather = torch.zeros(world * (words_local + W), dtype=torch.int32, device="cuda")
        bitmap_base = t_local.data_ptr() - (lo // 32) * 4   # the kernels index the bitmap by GLOBAL item number

    def step():
        if world == 1:
            eng.verify_device(t_items.data_ptr(), n_global, t_arena.data_ptr(), t_arena.numel(), lo, hi, t_bitmap.data_ptr(), 0,
                              stream.cuda_stream)
            eng.quorum_reduce_device(t_items.data_ptr(), n_global, t_bitmap.data_ptr(), len(groups), t_results.data_ptr(), stream.cuda_stream)
            return
        eng.verify_device(t_items.data_ptr(), n_global, t_arena.data_ptr(), t_arena.numel(), lo, hi, bitmap_base, 0, stream.cuda_stream)
        eng.quorum_mark_device(t_items.data_ptr(), n_global, lo, hi, bitmap_base, t_local.data_ptr() + words_local * 4, stream.cuda_stream)
        dist.all_gather_into_tensor(t_gather, t_local)
        eng.quorum_merge_device(t_gather.data_ptr() + words_local * 4, world, words_local + W, t_results.data_ptr(), stream.cuda_stream)

    def full_bitmap():
        if world == 1:
            return t_bitmap
        return t_gather.view(world, words_local + W)[:, :words_local].reshape(-1)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        step()
    barrier()
    # correctness of the timed configuration: bitmap must equal the replicated golden bitmap
    golden_bits = np.unpackbits(d["bitmap"].view(np.uint8), bitorder="little")[: len(base_items)]
    got_bits = np.unpackbits(full_bitmap().cpu().numpy().view(np.uint8), bitorder="little")[: n_global]
    reps = (n_global + len(base_items) - 1) // len(base_items)
    if not np.array_equal(got_bits, np.tile(golden_bits, reps)[:n_global]):
        raise SystemExit("bench: verdict bitmap differs from the golden bitmap -- refusing to report a number")

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
        time.sleep(0.3)
    barrier()
    launches0 = eng.launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev_k = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    ev0.record(stream)
    for i in range(args.steps):
        ev_k[i][0].record(stream)
        if world == 1:
            eng.verify_device(t_items.data_ptr(), n_global, t_arena.data_ptr(), t_arena.numel(), lo, hi, t_bitmap.data_ptr(), 0, stream.cuda_stream)
            ev_k[i][1].record(stream)
            eng.quorum_reduce_device(t_items.data_ptr(), n_global, t_bitmap.data_ptr(), len(groups), t_results.data_ptr(), stream.cuda_stream)
        else:
            eng.verify_device(t_items.data_ptr(), n_global, t_arena.data_ptr(), t_arena.numel(), lo, hi, bitmap_base, 0, stream.cuda_stream)
            ev_k[i][1].record(stream)
            eng.quorum_mark_device(t_items.data_ptr(), n_global, lo, hi, bitmap_base, t_local.data_ptr() + words_local * 4, stream.cuda_stream)
            dist.all_gather_into_tensor(t_gather, t_local)
            eng.quorum_merge_device(t_gather.data_ptr() + words_local * 4, world, words_local + W, t_results.data_ptr(), stream.cuda_stream)
    ev1.record(stream)
    barrier()
    launches = eng.launch_count() - launches0
    ms_total = ev0.elapsed_time(ev1)
    ms_kernel = sum(a.elapsed_time(b) for a, b in ev_k) / args.steps
    t = torch.tensor([ms_total, ms_kernel], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total, ms_kernel = float(t[0]), float(t[1])
    if rank == 0:
        time.sleep(0.2)
        sampler.stop()
    ms_per_step = ms_total / args.steps
    value = n_global / (ms_per_step * 1e-3)
    if args.dump_outputs and rank == 0:   # before any later leg writes t_results again
        dump_outputs(args.dump_outputs, full_bitmap(), t_results, n_global, ib.RESULT_DTYPE)

    # ---- e2e: host buffers through ibft_verify_batch (H2D + kernels + D2H inside the timed region)
    # the step's inputs live in PINNED host memory (torch pin_memory); the C ABI detects that and DMA-copies straight from it
    host_local = torch.from_numpy(host_local_np.view(np.uint8)).pin_memory().numpy().view(ib.ITEM_DTYPE).reshape(-1)
    arena_host = np.ascontiguousarray(d["arena"])
    e2e_steps = max(3, min(args.steps, 5))
    eng.verify_batch(host_local, arena_host, groups)
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        bm_local, res_local, _ = eng.verify_batch(host_local, arena_host, groups)
        if world > 1:
            tb = torch.from_numpy(bm_local.view(np.int32)).cuda()
            full = torch.empty(n_global // 32, dtype=torch.int32, device="cuda")
            dist.all_gather_into_tensor(full, tb)
            full.cpu()
    torch.cuda.synchronize()
    e2e_dt = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(e2e_dt, op=dist.ReduceOp.MAX)
    e2e_value = n_global * e2e_steps / float(e2e_dt[0])
    e2e_bits_ok = bool(np.array_equal(np.unpackbits(bm_local.view(np.uint8), bitorder="little")[: hi - lo], np.tile(golden_bits, reps)[lo:hi]))
    if not e2e_bits_ok:
        raise SystemExit("bench: e2e leg: verdict bitmap differs from the golden bitmap -- refusing to report a number")
    h2d = host_local.nbytes + arena_host.nbytes + groups.nbytes
    d2h = (n_local // 8) + n_local + len(groups) * ib.RESULT_DTYPE.itemsize  # bitmap + per-item status bytes + quorum results
    # the same call from PAGEABLE memory (what a cgo caller hands over: Go heap): the engine stages every chunk into its pinned
    # buffer on the calling thread before the DMA
    e2e_pageable = None
    if world == 1:
        eng.verify_batch(host_local_np, arena_host, groups)
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            bm_pg, _, _ = eng.verify_batch(host_local_np, arena_host, groups)
        e2e_pageable = n_global * e2e_steps / (time.perf_counter() - t0)
        if not np.array_equal(bm_pg, bm_local):
            raise SystemExit("bench: pageable e2e leg: bitmap differs")

    # ---- strong scaling: ONE round / ONE backlog split over the N ranks (all ranks take part)
    strong = strong_scaling_legs(args, ib, eng, d, base_items, groups, world, rank, local_rank, stream)

    if rank != 0:
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return

    if args.skip_extras:
        emit(({"metric": "secp256k1_verifies_per_sec", "value": value, "unit": "verifies/s", "n_gpus": n_gpus, "steps": args.steps,
                          "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                          "dtype": "u32 (256-bit modular integer)", "data": "synthetic", "config": workload_config(n_gpus),
                          "clocks": sampler.summary(), "gpu_launches": int(launches),
                          "e2e": {"value": e2e_value, "unit": "verifies/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h)},
                          "strong_scaling": strong, "note": "--skip-extras: development run without the latency / CPU / ingress legs"}))
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return

    # ---- quorum latency of ONE 10k-validator COMMIT round (10,000 committed seals), host buffers in / bitmap + quorum out
    seal_group = list(d["groups"]).index("COMMIT_SEAL")
    seals = np.ascontiguousarray(base_items[base_items["group"] == seal_group])
    # measured twice: tuples in pageable memory (what a cgo caller hands over: the engine stages them into its pinned buffer)
    # and in pinned memory (as the e2e leg above: DMA straight from the caller's buffer)
    seals_pinned = torch.from_numpy(seals.view(np.uint8)).pin_memory().numpy().view(ib.ITEM_DTYPE).reshape(-1)
    lat_pin = []
    for i in range(args.latency_reps + 5):
        t0 = time.perf_counter()
        eng.verify_batch(seals_pinned, b"", groups)
        if i >= 5:
            lat_pin.append((time.perf_counter() - t0) * 1e6)
    lat_pin.sort()
    lat = []
    for i in range(args.latency_reps + 5):
        t0 = time.perf_counter()
        _, res, _ = eng.verify_batch(seals, b"", groups)
        if i >= 5:
            lat.append((time.perf_counter() - t0) * 1e6)
    lat.sort()
    # device-only (no H2D): same round, tuples resident
    t_seals = torch.from_numpy(seals.view(np.uint8).reshape(-1, 128)).cuda()
    nb = (len(seals) + 31) // 32
    t_bm2 = torch.zeros(nb, dtype=torch.int32, device="cuda")
    lat_dev = []
    for i in range(args.latency_reps + 5):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream)
        eng.verify_device(t_seals.data_ptr(), len(seals), 0, 0, 0, len(seals), t_bm2.data_ptr(), 0, stream.cuda_stream)
        eng.quorum_reduce_device(t_seals.data_ptr(), len(seals), t_bm2.data_ptr(), len(groups), t_results.data_ptr(), stream.cuda_stream)
        b.record(stream)
        torch.cuda.synchronize()
        if i >= 5:
            lat_dev.append(a.elapsed_time(b) * 1e3)
    lat_dev.sort()
    # the same measurement for a 1,000-seal round (AUTO path selection: four-lane chain warps + helper warp, k_recover_qsplit)
    small = np.ascontiguousarray(seals[:1000])
    lat_small, lat_small_dev = [], []
    for i in range(args.latency_reps + 5):
        t0 = time.perf_counter()
        eng.verify_batch(small, b"", groups)
        if i >= 5:
            lat_small.append((time.perf_counter() - t0) * 1e6)
    for i in range(args.latency_reps + 5):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream)
        eng.verify_device(t_seals.data_ptr(), len(small), 0, 0, 0, len(small), t_bm2.data_ptr(), 0, stream.cuda_stream)
        eng.quorum_reduce_device(t_seals.data_ptr(), len(small), t_bm2.data_ptr(), len(groups), t_results.data_ptr(), stream.cuda_stream)
        b.record(stream)
        torch.cuda.synchronize()
        if i >= 5:
            lat_small_dev.append(a.elapsed_time(b) * 1e3)
    lat_small.sort()
    lat_small_dev.sort()

    # ---- the same workload with the key registry (engine flag key_cache): after a validator's first successful recovery its
    # signatures are VERIFIED against the learned key (two-pass: verify, then recover whatever was not accepted).  Reported
    # next to the headline, which never relies on learned state.  Same tuples, same bitmap check, same timing rules.
    known = None
    if world == 1 and not args.no_key_cache_leg:
        eng_k = ib.Engine(device=local_rank, max_items=n_global, max_payload_bytes=max(1 << 20, int(d["arena"].nbytes)), max_groups=8,
                          max_table_slots=2, max_validators=16384, key_cache=True)
        eng_k.set_validators(0, int(d["meta"][2]), d["addrs"], d["powers"])
        eng_k.bind_groups(groups)
        t_bm_k = torch.zeros(n_global // 32, dtype=torch.int32, device="cuda")

        def step_k():
            eng_k.verify_device(t_items.data_ptr(), n_global, t_arena.data_ptr(), t_arena.numel(), 0, n_global, t_bm_k.data_ptr(), 0, stream.cuda_stream)
            eng_k.quorum_reduce_device(t_items.data_ptr(), n_global, t_bm_k.data_ptr(), len(groups), t_results.data_ptr(), stream.cuda_stream)

        step_k()                      # cold pass: every signer is recovered, keys are learned
        torch.cuda.synchronize()
        keys_known = eng_k.refresh_key_tables()
        for _ in range(max(args.warmup, 3)):
            step_k()
        torch.cuda.synchronize()
        got_k = np.unpackbits(t_bm_k.cpu().numpy().view(np.uint8), bitorder="little")[: n_global]
        if not np.array_equal(got_k, np.tile(golden_bits, reps)[:n_global]):
            raise SystemExit("bench: key-registry path: verdict bitmap differs from the golden bitmap")
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        lk0 = eng_k.launch_count()
        a.record(stream)
        for _ in range(args.steps):
            step_k()
        b.record(stream)
        torch.cuda.synchronize()
        ms_k = a.elapsed_time(b) / args.steps
        eng_k.verify_batch(host_local, arena_host, groups)
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            bm_k, _, _ = eng_k.verify_batch(host_local, arena_host, groups)
        e2e_k = n_global * e2e_steps / (time.perf_counter() - t0)
        # the 10,000-seal round on the known-key LATENCY path (k_verify_known<32> + worklist k_recover_qsplit), host buffers in / out
        lat_known = []
        for i in range(args.latency_reps + 5):
            t0 = time.perf_counter()
            bm_s, _, _ = eng_k.verify_batch(seals, b"", groups)
            if i >= 5:
                lat_known.append((time.perf_counter() - t0) * 1e6)
        bm_plain, _, _ = eng.verify_batch(seals, b"", groups)
        if not np.array_equal(bm_s, bm_plain):
            raise SystemExit("bench: known-key latency path: bitmap differs from the recover path")
        # and an all-valid round (no worklist work at all): the 9,900 valid seals only
        seals_ok = np.ascontiguousarray(seals[np.unpackbits(bm_plain.view(np.uint8), bitorder="little")[: len(seals)] == 1])
        lat_known_ok = []
        for i in range(args.latency_reps + 5):
            t0 = time.perf_counter()
            eng_k.verify_batch(seals_ok, b"", groups)
            if i >= 5:
                lat_known_ok.append((time.perf_counter() - t0) * 1e6)
        known = {"value": n_global / (ms_k * 1e-3), "unit": "verifies/s", "ms_per_step": ms_k, "e2e": e2e_k, "keys_known": keys_known,
                 "gpu_launches": int(eng_k.launch_count() - lk0),
                 "round10k_p50_us": _pct(lat_known, 0.5), "round10k_p95_us": _pct(lat_known, 0.95),
                 "round10k_all_valid_p50_us": _pct(lat_known_ok, 0.5), "round10k_all_valid_items": int(len(seals_ok)),
                 "round10k_kernel": "k_verify_known<32> (one-warp CTAs, verification against the validator's comb table: 51 additions, no doubling) + k_recover_qsplit on the worklist",
                 "bitmap_matches_golden": bool(np.array_equal(np.unpackbits(bm_k.view(np.uint8), bitorder="little")[:n_global], np.tile(golden_bits, reps)[:n_global])),
                 "note": "engine flag IBFT_FLAG_KEY_CACHE: k_verify_known (ECDSA verification against the learned key through a per-validator comb table, 136 KiB each) + k_recover on the "
                         "worklist of everything not accepted; verdicts are the recover path's by construction; the first (cold) pass over "
                         "a validator set runs at the headline rate"}
        eng_k.close()

    imad_peak, wide_peak = eng.probe_int_peak()
    info = eng.device_info()
    kernel_rate = n_local / (ms_kernel * 1e-3)  # per GPU
    achieved = kernel_rate * ALGO_IMAD_PER_VERIFY
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    hbm_peak_gbs, hbm_src = 6650.0, "fallback 6.65 TB/s (B200_PROFILING.md)"
    if os.path.exists(peaks_path):
        try:
            pk = json.load(open(peaks_path))
            hbm_peak_gbs, hbm_src = float(pk.get("hbm_gbs", hbm_peak_gbs)), "MEASURED_PEAKS.json"
        except Exception:
            pass
    hbm_gbs = kernel_rate * ALGO_BYTES_PER_VERIFY / 1e9
    # DRAM traffic of the dominant kernel from the committed ncu --set full capture of this same configuration (per launch)
    traffic, traffic_src, executed = None, None, None
    tpath = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if os.path.exists(tpath):
        try:
            tj = json.load(open(tpath))
            if int(tj.get("items_per_launch", 0)) == n_local:
                traffic = float(tj["dram_bytes_read"]) + float(tj["dram_bytes_write"])
                traffic_src = tj.get("capture")
                executed = tj.get("executed")
        except Exception:
            pass
    line = {
        "metric": "secp256k1_verifies_per_sec", "value": value, "unit": "verifies/s", "n_gpus": n_gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u32 (256-bit modular integer)", "data": "synthetic", "config": workload_config(n_gpus),
        "clocks": sampler.summary(),
        "e2e": {"value": e2e_value, "unit": "verifies/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                "steps": e2e_steps, "api": "ibft_verify_batch (host buffers -> pinned staging -> H2D -> kernels -> D2H bitmap + quorum)",
                "input_memory": "caller-pinned (DMA straight from the caller's buffer)", "pageable_input_value": e2e_pageable,
                "pageable_note": "same call from pageable memory (a cgo caller's Go heap): + one host memcpy of every chunk into the engine's pinned staging"},
        "strong_scaling": strong,
        "gpu_launches": int(launches),
        "roofline": {"bound": "int32-imad-issue", "achieved": achieved / 1e12, "peak": imad_peak / 1e12, "unit": "T IMAD-class instr/s",
                     "frac": achieved / imad_peak, "traffic": traffic, "traffic_unit": "DRAM bytes per k_recover launch (ncu)",
                     "traffic_source": traffic_src, "algorithmic_bytes_per_launch": ALGO_BYTES_PER_VERIFY * n_local,
                     "executed_per_ncu": executed,
                     "issue_active_pct": (executed or {}).get("issue_active_pct"),
                     "fmaheavy_pipe_pct": (executed or {}).get("fmaheavy_pipe_cycles_active_pct"),
                     "binding_pipe_note": "from the committed ncu --set full capture of this kernel: the FMA-heavy pipe (IMAD / IMAD.WIDE; an IMAD.WIDE holds it 4 "
                                          "cycles per warp instruction) is the pipe that binds -- issue-active is low BECAUSE that pipe is busy",
                     "note": "frac uses SURVEY 8d's canonical-algorithm count (5.0e5 IMAD-class instr/verify); the kernel executes fewer "
                             "multiply instructions than that (GLV, combined generator table, safegcd, fused IMAD.WIDE), so frac can "
                             "exceed 1; executed_per_ncu gives the real instruction counts",
                     "kernel": "k_recover", "kernel_ms": ms_kernel, "kernel_verifies_per_s_per_gpu": kernel_rate,
                     "algorithmic_instr_per_verify": ALGO_IMAD_PER_VERIFY,
                     "peak_source": "dependent-free mad.lo.u32 probe on this GPU (ibft_probe_int_peak), measured live",
                     "wide_mac_peak_per_s": wide_peak, "wide_mac_frac_at_2.5e5_mac_per_verify": kernel_rate * 2.5e5 / wide_peak,
                     "hbm": {"achieved_gbs": hbm_gbs, "peak_gbs": hbm_peak_gbs, "frac": hbm_gbs / hbm_peak_gbs, "peak_source": hbm_src,
                             "note": "reported only to show HBM is not the bound"},
                     "kernel_regs": info["kernel_regs"], "kernel_smem_bytes": info["kernel_smem_bytes"]},
        "known_validator_path": known,
        "quorum_latency_us": {"config": "10k-validator COMMIT round, 10,000 committed seals, host tuples -> bitmap+quorum on host",
                              "reps": len(lat), "p50": lat[len(lat) // 2], "p95": lat[int(len(lat) * 0.95)],
                              "pinned_input_p50": lat_pin[len(lat_pin) // 2], "pinned_input_p95": lat_pin[int(len(lat_pin) * 0.95)],
                              "device_only_p50": lat_dev[len(lat_dev) // 2], "device_only_p95": lat_dev[int(len(lat_dev) * 0.95)],
                              "kernel": "k_recover_split (chain warps + helper warp; AUTO path for 7,105..14,208 signatures)",
                              "round_1000_seals": {"kernel": "k_recover_qsplit (four-lane chain warps + helper warp; AUTO path up to 7,104 signatures)", "p50": lat_small[len(lat_small) // 2],
                                                   "p95": lat_small[int(len(lat_small) * 0.95)],
                                                   "device_only_p50": lat_small_dev[len(lat_small_dev) // 2]}},
    }
    if not args.no_cpu_baseline and n_gpus == 1:
        cores = effective_cpus()
        line["cpu_baseline"] = cpu_baseline_legs(d, base_items, cores)
        line["quorum_latency_us"]["cpu"] = cpu_latency_legs(d, base_items, cores)
        line["proposal_hash"] = hash_crossover_leg(eng)
    if n_gpus == 1:
        line["ingress"] = ingress_leg(local_rank, 64)
        line["ingress"]["more_callers"] = ingress_leg(local_rank, 512)
        if "cpu_baseline" in line:
            line["ingress"]["cpu_oracle"] = {"single_call_us": 1e6 / line["cpu_baseline"]["single_thread"],
                                             "all_cores_msgs_per_s": line["cpu_baseline"]["value"], "cores": line["cpu_baseline"]["cores"]}
        line["config4"] = config4_legs(ib, local_rank, stream)
    emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
