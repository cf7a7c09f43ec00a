#!/usr/bin/env python
"""bench.py — the reference's headline metric on the reference's headline config.

metric   : configs explored/sec (BASELINE.json; time-to-verdict reported beside it)
workload : BASELINE config #3 exactly as SURVEY.md 8(d) writes it — 10k-op bank-transfer history, 32 clients,
           tau_op 10 ms, tau_think 0 (every client always has an op in flight: the hardest setting), linearizable by
           construction, seed 1; searched in the Knossos-exact space (7.1e9 configurations).
           One "step" = one complete linearizability check of that history through the C ABI.
           The CPU reference cannot finish this instance (it would need > 100 GB for its cache and ~1 h), so both
           arms also carry `verdict_to_verdict`: the same history shape at tau_think 5 ms (1.9e8 configurations),
           which both arms run to the verdict (round 1's headline instance).
           N > 1 : one such history per GPU as independent keys (ledgers), sharded by key, verdicts
           merged with one NCCL all_reduce(MAX)  -> weak scaling.

value    = configs / device time of the search kernels (CUDA events on the library's stream; inputs
           already in HBM)            e2e = configs / wall time of the C-ABI call with HOST buffers
           (flatten-prep, H2D, table clear, kernels, D2H verdict inside the timed region).

sharded  : beside the headline every line carries `"sharded"`: BASELINE configs #5 (50k-op cas-register, 30 %
           :info, K = 256 keys, one key poisoned) and #4 (100k-op set-full, K = 64 ledgers, one ledger
           poisoned) checked over the N GPUs — more shards than ranks, LPT partition, the merged verdict
           must flip to invalid with exactly one failure; STRONG scaling (total work fixed), time to the
           merged verdict as max over ranks plus every rank's own device time (imbalance is visible).

--impl reference : the CPU restatement of knossos.wgl (oracle/, kind "port" — the reference's own
           implementation is JVM-only and cannot run here) on the same history, each step a bounded
           sample (first --ref-configs configurations) on one thread per key like knossos.wgl (N keys ->
           N threads); it cannot reach the verdict of the headline instance (`time_to_verdict_s` null,
           `did_not_finish` says why), so ONE full run of the tau_think 5 ms instance is timed beside it
           (`verdict_to_verdict`, rank 0 only) — the same block the GPU arm prints: a verdict-to-verdict
           ratio on an instance both arms finish.  Its `sharded` object runs the same C5 / C4 histories
           over min(16 N, host cores) threads (independent/checker's fan-out).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

from jepsen_tigerbeetle_b200 import history as H  # noqa: E402
from jepsen_tigerbeetle_b200 import synth  # noqa: E402

METRIC = "configs explored/sec (time-to-verdict alongside) on 10k-op/32-client bank history"
UNIT = "configs/s"


def workload(seed, args, think_ms=None):
    spec = synth.SynthSpec("bank", args.ops, args.clients, seed,
                           tau_think_ns=(args.think_ms if think_ms is None else think_ms) * 1e6, stale_read=args.invalid)
    return synth.generate(spec)


def v2v_workload_name(args):
    return (f"C3 bank-transfer history: {args.ops} ops, {args.clients} clients, tau_op 10 ms, tau_think "
            f"{args.v2v_think_ms} ms, seed 1, {'one stale read (invalid)' if args.invalid else 'linearizable (valid)'}, "
            "Knossos-exact space")


def config_block(args, n_gpus):
    return {"workload": f"C3 bank-transfer history: {args.ops} ops, {args.clients} clients, 8 accounts, "
                        f"tau_op 10 ms, tau_think {args.think_ms} ms, seed 1+key, "
                        f"{'one stale read (invalid)' if args.invalid else 'linearizable (valid)'}",
            "keys": n_gpus, "sharding": "one key (ledger) per GPU" if n_gpus > 1 else "single key",
            "l2": "level windows up to 16 GiB and level arrays of 2 GB (45 M configurations per level) exceed the 126 MB L2",
            "model": "bank", "table": "16 B slots, linear probing, per-level window of 16 slots per configuration",
            "engine": "level-synchronous (csrc/jtb_level.cuh)",
            "search_space": "eager-read reduction (product default)" if args.eager_reads else
                            "Knossos-exact (JTB_OPT_NO_EAGER_READS): the same configurations the CPU reference visits"}


def sharded_workloads(args):
    """BASELINE configs #5 and #4 with ONE poisoned key each (the merged verdict must flip)."""
    c5 = synth.poison_c5(synth.config_c5(seed=1, n_ops=args.c5_ops), 7)
    c4 = synth.poison_c4(synth.config_c4(seed=1, n_keys=64, n_ops=args.c4_ops), 5)
    return c5, c4


def run_sharded_ours(args, ctx, rank, world, reduce_max, dist, dev):
    """Strong scaling over the N ranks: C5 through the WGL search, C4 through the set-full scan."""
    import torch
    from jepsen_tigerbeetle_b200 import distributed
    c5, c4 = sharded_workloads(args)
    mc = H.make_model(H.MODEL_CAS_REGISTER)
    out = {}
    for name, h in (("c5_K256_pinfo0.30_wgl_cas_register", c5), ("c4_K64_set_full", c4)):
        kern = [0.0]

        def check_fn(sub):
            if name.startswith("c5"):
                r = ctx.check_linearizable(sub, mc)
                kern[0] = r["seconds_kernel"]
                return r["shards"]
            r = ctx.check_set_full(sub, True)
            kern[0] = r["seconds_kernel"]
            return r["shards"]

        best = None
        for rep in range(3):
            if dist is not None:
                dist.barrier()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            res = distributed.check_sharded(h, check_fn, rank, world, reduce_max)
            torch.cuda.synchronize()
            wall = time.perf_counter() - t0
            t = torch.tensor([wall, kern[0]], dtype=torch.float64, device=dev)
            per_rank = [torch.zeros_like(t) for _ in range(world)]
            if dist is not None:
                dist.all_gather(per_rank, t)
            else:
                per_rank = [t]
            walls = [float(x[0]) for x in per_rank]
            kerns = [float(x[1]) for x in per_rank]
            rec = {"verdict": {0: "valid", 1: "unknown", 2: "invalid"}[res["valid"]],
                   "n_failures": int((res["shard_valid"] != 0).sum()), "keys": int(h.n_shards),
                   "events": int(h.n_events), "time_to_merged_verdict_s": max(walls),
                   "per_rank_wall_s": walls, "per_rank_kernel_s": kerns,
                   "shards_per_rank": [len(x) for x in distributed.assign_shards(distributed.shard_costs(h), world)]}
            if best is None or rec["time_to_merged_verdict_s"] < best["time_to_merged_verdict_s"]:
                best = rec
        out[name] = best
    out["scaling"] = "strong (fixed keys, LPT partition over the ranks; best of 3)"
    return out


def run_sharded_reference(args, world):
    import oracle
    c5, c4 = sharded_workloads(args)
    threads = max(1, min(16 * world, os.cpu_count() or 1))
    mc = H.make_model(H.MODEL_CAS_REGISTER)
    out = {"threads": threads}
    t = time.perf_counter()
    r = oracle.check_linearizable(c5, mc, oracle.ALGO_WGL_COMPACT, max_configs=50_000_000, n_threads=threads)
    out["c5_K256_pinfo0.30_wgl_cas_register"] = {
        "verdict": {0: "valid", 1: "unknown", 2: "invalid"}[r["valid"]], "n_failures": r["n_failures"],
        "keys": int(c5.n_shards), "time_to_merged_verdict_s": time.perf_counter() - t}
    t = time.perf_counter()
    r = oracle.check_set_full(c4, True)
    out["c4_K64_set_full"] = {"verdict": {0: "valid", 1: "unknown", 2: "invalid"}[r["valid"]],
                              "n_failures": r["n_failures"], "keys": int(c4.n_shards),
                              "time_to_merged_verdict_s": time.perf_counter() - t,
                              "note": "scan_oracle.cpp is single-threaded over the keys"}
    return out


class ClockSampler:
    """nvidia-smi clocks during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
            except (ValueError, IndexError):
                continue
            for nm, v in zip(names, r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def peak_hbm():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "of measured (MEASURED_PEAKS.json)"
        except Exception:  # noqa: BLE001
            pass
    return 6650.0, "of fallback (B200_PROFILING.md)"


def traffic_from_profile():
    p = os.path.join(ROOT, "profiles", "bench_traffic.json")
    if os.path.exists(p):
        try:
            return json.load(open(p))
        except Exception:  # noqa: BLE001
            pass
    return None


def reduced_search_check(h, m, args):
    """The headline instance's verdict from an independent CPU algorithm: the oracle's reduced bank decider
    (ALGO_LAZY_BANK: transfers linearized only when the frontier forces them or a read's balances require them — ~1e5
    configurations instead of ~7e9; NOT knossos.wgl, NOT the timed reference; equal to knossos.wgl in verdict and witness on
    every history both finish).  Both arms print it, so the record carries an identical verdict for the instance no
    exhaustive CPU search can finish."""
    import oracle
    t = time.perf_counter()
    try:
        r = oracle.check_linearizable(h, m, oracle.ALGO_LAZY_BANK, max_configs=50_000_000)
    except RuntimeError as e:   # histories outside the decider's scope
        return {"algo": "oracle ALGO_LAZY_BANK", "unavailable": str(e)}
    return {"algo": "oracle ALGO_LAZY_BANK (reduced search, CPU, 1 thread)", "verdict": {0: "valid", 1: "unknown", 2: "invalid"}[r["valid"]],
            "witness_index": r["shards"][0]["witness_index"], "configs": r["configs"], "seconds": time.perf_counter() - t}


def dump_outputs(path, out, shards, n_shards, rank, reduce_max):
    """Write what the last timed step returned as float64 .npy files under `path`: the merged verdict and, per key,
    what check_linearizable reports for it.  Timings are left out: they vary from run to run of the same build, so they
    would hide the differences a comparison of two builds looks for."""
    detail = np.full((4, n_shards), -1, np.int64)       # -1 = checked on another rank
    for s, r in zip(out["mine"], shards):
        detail[:, s] = (r["previous_ok_index"], r["cause"], r["configs"], r["probes"])
    if reduce_max is not None:
        detail = reduce_max(detail.ravel()).reshape(4, n_shards)
    if rank != 0:
        return
    os.makedirs(path, exist_ok=True)
    arrays = {"verdict": [out["valid"]], "shard_valid": out["shard_valid"], "shard_witness_index": out["shard_witness"],
              "shard_previous_ok_index": detail[0], "shard_cause": detail[1], "shard_configs": detail[2],
              "shard_probes": detail[3]}
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), np.asarray(a, dtype=np.float64))


def run_reference(args, rank, world):
    if rank != 0:
        return
    import oracle
    from concurrent.futures import ThreadPoolExecutor
    oracle.build()
    n_keys = max(1, world)
    parts = [workload(1 + k, args) for k in range(n_keys)]
    m = H.make_model(H.MODEL_BANK, accounts=range(1, 9))
    cores = n_keys  # knossos.wgl searches one history on one thread; independent/checker gives every key a thread

    def one(h):
        return oracle.check_linearizable(h, m, oracle.ALGO_WGL_COMPACT, max_configs=args.ref_configs)["configs"]

    pool = ThreadPoolExecutor(n_keys)      # the oracle releases the GIL inside ctypes calls
    for _ in range(args.warmup):
        list(pool.map(one, parts))
    configs, secs = 0, 0.0
    for _ in range(args.steps):
        t = time.perf_counter()
        configs += sum(pool.map(one, parts))
        secs += time.perf_counter() - t
    v = configs / secs
    sample = (f"first {args.ref_configs} configurations of every key's history per step, one thread per key "
              f"(knossos.wgl is single-threaded per history; {os.cpu_count()} host cores present)")
    line = {
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * secs / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int64",
        "data": "synthetic", "config": config_block(args, n_keys),
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "note": "CPU restatement of knossos.wgl (oracle/lin_oracle.cpp, -O3 -march=native); JVM Knossos cannot run here",
    }
    line["time_to_verdict_s"] = None
    line["verdict"] = "unknown"
    line["did_not_finish"] = ("the headline instance (tau_think 0) has 7.1e9 reachable configurations: knossos.wgl's cache would "
                              "need > 100 GB and ~1 h at the sampled rate; only the bounded sample above is timed")
    line["verdict_check"] = reduced_search_check(parts[0], m, args)
    if not args.no_full_run:
        hv = workload(1, args, think_ms=args.v2v_think_ms)
        t = time.perf_counter()
        r = oracle.check_linearizable(hv, m, oracle.ALGO_WGL_COMPACT, max_configs=args.ref_full_configs)
        dt = time.perf_counter() - t
        line["verdict_to_verdict"] = {
            "workload": v2v_workload_name(args), "time_to_verdict_s": dt,
            "verdict": {0: "valid", 1: "unknown", 2: "invalid"}[r["valid"]], "configs_to_verdict": r["configs"],
            "note": "ONE full run to the verdict, single thread (knossos.wgl is single-threaded), outside the timed steps"}
    if not args.no_sharded:
        line["sharded"] = run_sharded_reference(args, world)
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--ops", type=int, default=10000)
    ap.add_argument("--clients", type=int, default=32)
    ap.add_argument("--think-ms", type=float, default=0.0)
    ap.add_argument("--v2v-think-ms", type=float, default=5.0, help="tau_think of the instance both arms run to the verdict")
    ap.add_argument("--invalid", action="store_true", help="one stale read: exhaustive search, verdict invalid")
    ap.add_argument("--ref-configs", type=int, default=3_000_000)
    ap.add_argument("--cpu-baseline-configs", type=int, default=10_000_000)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-full-run", action="store_true", help="reference arm: skip the one full run to the verdict")
    ap.add_argument("--ref-full-configs", type=int, default=400_000_000, help="budget of that full run")
    ap.add_argument("--no-sharded", action="store_true", help="skip the C5 / C4 sharded workloads")
    ap.add_argument("--c5-ops", type=int, default=50000)
    ap.add_argument("--c4-ops", type=int, default=100000)
    ap.add_argument("--eager-reads", action="store_true",
                    help="time the product default (eager-read reduction: ~18x fewer configs, same verdict) instead of "
                         "the Knossos-exact search space the CPU reference explores")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the last step's verdict and per-key results to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the results of the GPU checker (--impl ours)")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    from jepsen_tigerbeetle_b200 import distributed, native
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the checker has no CPU fallback")
    dist = None
    if world > 1:
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    dev = torch.device("cuda", local_rank)
    n_keys = max(1, world)
    parts = [workload(1 + k, args) for k in range(n_keys)]
    h_all = H.concat_keys(parts) if n_keys > 1 else parts[0]
    m = H.make_model(H.MODEL_BANK, accounts=range(1, 9))
    ctx = native.Context(device=local_rank, eager_reads=args.eager_reads)
    reduce_max = distributed.torch_all_reduce_max(dev) if world > 1 else None
    last = {}

    def check_fn(sub):
        r = ctx.check_linearizable(sub, m)
        last.update(r)
        last["stats"] = ctx.stats()
        return r["shards"]

    def step():
        return distributed.check_sharded(h_all, check_fn, rank, world, reduce_max)

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(args.warmup, 3)):
        step()
    sampler = ClockSampler(local_rank)
    barrier()
    sampler.start()
    t0 = time.perf_counter()
    kern_s, configs, probes, algo_bytes, launches, h2d, d2h = 0.0, 0, 0, 0, 0, 0, 0
    verdict = None
    for _ in range(args.steps):
        out = step()
        verdict = out["valid"]
        kern_s += last["seconds_kernel"]
        configs += last["configs"]; probes += last["probes"]; algo_bytes += last["hbm_bytes_algorithmic"]
        launches += last["stats"]["kernel_launches"]; h2d += last["stats"]["h2d_bytes"]; d2h += last["stats"]["d2h_bytes"]
    barrier()
    wall = time.perf_counter() - t0
    clocks = sampler.stop()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, out, last["shards"], h_all.n_shards, rank, reduce_max)
    # max over ranks of the times, sum over ranks of the work
    agg = torch.tensor([kern_s, wall], dtype=torch.float64, device=dev)
    tot = torch.tensor([configs, probes, algo_bytes, launches, h2d, d2h], dtype=torch.float64, device=dev)
    if dist is not None:
        dist.all_reduce(agg, op=dist.ReduceOp.MAX)
        dist.all_reduce(tot, op=dist.ReduceOp.SUM)
    kern_max, wall_max = (float(x) for x in agg.cpu())
    mine_k = torch.tensor([kern_s], dtype=torch.float64, device=dev)
    gathered = [torch.zeros_like(mine_k) for _ in range(world)]
    if dist is not None:
        dist.all_gather(gathered, mine_k)
    else:
        gathered = [mine_k]
    per_rank_kern = [float(x[0]) for x in gathered]
    sharded = None
    if not args.no_sharded:
        with native.Context(device=local_rank) as sctx:      # product defaults (eager reads, scouts)
            sharded = run_sharded_ours(args, sctx, rank, world, reduce_max, dist, dev)
    configs_t, probes_t, bytes_t, launches_t, h2d_t, d2h_t = (float(x) for x in tot.cpu())
    if rank == 0:
        peak, peak_src = peak_hbm()
        achieved = bytes_t / world / kern_max / 1e9  # per GPU, GB/s (algorithmic bytes / launch time)
        tr = traffic_from_profile()
        if tr and not (args.think_ms == tr.get("think_ms", 0.0) and args.ops == 10000 and args.clients == 32
                       and not args.eager_reads and not args.invalid):
            tr = None   # the capture is of the default workload only
        line = {
            "metric": METRIC, "value": configs_t / kern_max, "unit": UNIT, "n_gpus": world,
            "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": 1e3 * wall_max / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int64",
            "data": "synthetic", "config": config_block(args, n_keys),
            "verdict": {0: "valid", 1: "unknown", 2: "invalid"}[verdict],
            "time_to_verdict_s": wall_max / args.steps, "time_to_verdict_kernel_s": kern_max / args.steps,
            "configs_per_step": configs_t / args.steps, "probes_per_step": probes_t / args.steps,
            "probes_per_s": probes_t / kern_max,
            "e2e": {"value": configs_t / wall_max, "unit": UNIT,
                    "h2d_bytes_per_step": h2d_t / args.steps, "d2h_bytes_per_step": d2h_t / args.steps},
            "gpu_launches": int(launches_t),
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak, "traffic": tr["dram_bytes_per_launch"] if tr else None,
                         "traffic_source": tr.get("source") if tr else None,
                         "peak_source": peak_src, "kernel": last["stats"].get("engine_level") and "level_search_kernel<bank,KW=2,exact>"
                         or "wgl_search_kernel<bank,KW=2>",
                         "algorithmic_bytes": "16 B x (probes + inserts) per launch (SURVEY 8(d))",
                         "random_probe_ceiling_GBps": tr.get("table_probe_algo_GBps") if tr else None},
            "clocks": clocks,
        }
        line["per_rank_kernel_s_per_step"] = [x / args.steps for x in per_rank_kern]
        if sharded is not None:
            line["sharded"] = sharded
        if world == 1 and not args.no_full_run:
            hv = workload(1, args, think_ms=args.v2v_think_ms)
            with native.Context(device=local_rank, eager_reads=args.eager_reads) as vctx:
                vr = min((vctx.check_linearizable(hv, m) for _ in range(3)), key=lambda r: r["seconds_total"])
            line["verdict_to_verdict"] = {
                "workload": v2v_workload_name(args), "time_to_verdict_s": vr["seconds_total"], "kernel_s": vr["seconds_kernel"],
                "verdict": {0: "valid", 1: "unknown", 2: "invalid"}[vr["valid"]], "configs_to_verdict": vr["configs"],
                "note": "C-ABI call with host buffers, best of 3"}
        if world == 1 and not args.eager_reads:
            with native.Context(device=local_rank, eager_reads=True) as ectx:
                for _ in range(2):
                    er = ectx.check_linearizable(parts[0], m)
                line["product_default_eager_reads"] = {
                    "time_to_verdict_s": er["seconds_total"], "kernel_s": er["seconds_kernel"], "configs": er["configs"],
                    "verdict": {0: "valid", 1: "unknown", 2: "invalid"}[er["valid"]],
                    "note": "same verdict from ~20x fewer configurations; not used for `value`/`e2e`"}
        if world == 1 and not args.no_cpu_baseline:
            import oracle
            oracle.build()
            t = time.perf_counter()
            r = oracle.check_linearizable(parts[0], m, oracle.ALGO_WGL_COMPACT, max_configs=args.cpu_baseline_configs)
            dt = time.perf_counter() - t
            vc = reduced_search_check(parts[0], m, args)
            vc["identical_to_gpu_verdict"] = vc.get("verdict") == line["verdict"]
            line["verdict_check"] = vc
            line["cpu_baseline"] = {
                "value": r["configs"] / dt, "unit": UNIT, "cores": 1, "kind": "port",
                "sample": f"first {r['configs']} configurations of the same history, single thread "
                          f"(knossos.wgl is single-threaded per history); {os.cpu_count()} host cores present",
                "seconds": dt}
        print(json.dumps(line))
    ctx.close()
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
