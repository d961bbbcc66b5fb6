#!/usr/bin/env python3
"""bench.py — job-placements/sec per scheduling round (BASELINE.json metric).

A "step" is one scheduling CYCLE: `--pools` (default 8) independent pools of the configuration the
metric is quoted on — C3 = 100k nodes × 1M queued jobs × 64 queues each — one full
PreemptingQueueScheduler.Schedule round per pool (evict → schedule → oversubscribed evict →
re-schedule → unbind), like FairSchedulingAlgo.Schedule walks the pools of a cluster
(scheduling_algo.go:129-160).  The cycle is FIXED: with N GPUs rank r owns pools r, r+N, …
(strong scaling); a rank runs its pools concurrently (a round is one persistent CTA on one SM).

  value  : placements of the whole cycle per second with the inputs already resident in HBM
           (armada_round_run only; every round timed with CUDA events on its stream; the cycle lasts
           as long as its longest round; max over ranks).  ms_per_round = latency of ONE round.
  e2e    : the same through the reference-facing C ABI with HOST buffers on both sides
           (armada_round_upload / run / download per pool, copies inside the timed region; with N > 1
           the cycle's claims are all-gathered over NCCL inside it too)
  roofline: dominant kernel k_schedule_pass; achieved = probes × N × (8·D+4) algorithmic bytes
           (SURVEY.md §8d) ÷ its CUDA-event duration, against the measured HBM copy bandwidth
  cpu_baseline: the C++ restatement of the reference round (oracle "port") on pool 0, 1 host core
  parity : the device result of pool 0 diffed bit-for-bit against that oracle run
  extra_workloads: C2 / C4 / C5 on the device with their own parity checks (N = 1 only)

`--impl reference` times the oracle port on the same cycle (the same pools one after the other, the
way the reference schedules them) on the host cores; rank 0 only.

`--dump-outputs DIR` writes what the last timed device-resident cycle computed (see dump_outputs) so
that two builds can be compared output for output on identical seeded inputs.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

# The tree may be read-only where the benchmark runs, and it must be left as build() left it.
sys.dont_write_bytecode = True

# Before anything creates the CUDA context: one hardware work queue per concurrent round (the pools
# of a cycle run on one stream each; with the default of 8 queues two of them can share one).
os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")
# NCCL prints its version banner (and, with NCCL_DEBUG set, more) to STDOUT, in front of the one JSON line the
# contract allows there: everything any library writes to file descriptor 1 goes to stderr, and the JSON line is
# written to the real stdout at the end (emit()).
_REAL_STDOUT = os.dup(1)
os.dup2(2, 1)


def emit(line: dict) -> None:
    sys.stdout.flush()
    os.write(_REAL_STDOUT, (json.dumps(line) + "\n").encode())

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

METRIC = "job-placements/sec per scheduling round; 100k nodes x 1M jobs"
UNIT = "placements/s"


def make_workload(name: str, seed_offset: int = 0):
    from armada_b200 import synth
    if name == "C3":
        return synth.config_c3(seed=synth.SEED + seed_offset)
    if name == "C2":
        return synth.config_c2()
    if name == "C4":
        return synth.config_c4(seed=synth.SEED + seed_offset)
    if name == "C5":
        return synth.config_c5(seed=synth.SEED + seed_offset)
    if "@" in name:  # scaled instance (bounded CPU sample / parity scale)
        return synth.scaled(name.split("@")[0], float(name.split("@")[1]))
    if name == "C1":
        return synth.config_c1()
    raise SystemExit(f"unknown workload {name}")


def workload_config(name, inp, n_gpus, pools):
    return {
        "workload": name, "step": f"one scheduling cycle = {pools} pools, one full round each",
        "nodes": int(inp.num_nodes), "queues": int(inp.num_queues), "jobs": int(inp.num_jobs),
        "resources": int(inp.num_resources), "priority_levels": int(inp.num_priorities),
        "pools": pools, "parallelism": f"{pools} pools round-robin over {n_gpus} GPU(s), a rank's pools concurrently (one CTA each)",
        "l2": "flushed between timed steps (256 MiB write)",
    }


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200",
                                          "-i", str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_traffic():
    p = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(p):
        try:
            return json.load(open(p)).get("k_schedule_pass_dram_bytes_per_launch")
        except Exception:
            return None
    return None


def host_cores():
    return os.cpu_count() or 1


def cpu_baseline(name: str, budget_s: float = 12.0, keep_result: bool = False):
    """Oracle port timed on ONE host core (the reference round is single-goroutine) on a bounded
    sample: pool 0 of the cycle (one full round of the named configuration), best of ≤ 5 runs."""
    import oracle_lib
    t0 = time.perf_counter()
    r = make_workload(name)
    inp = r.to_input()
    res = oracle_lib.round_schedule(inp)  # warm (page-in, allocator)
    t = time.perf_counter()
    res = oracle_lib.round_schedule(inp)
    dt = time.perf_counter() - t
    placed = int(res.stats.placements)
    reps = 1
    while time.perf_counter() - t0 < budget_s and reps < 5:
        t = time.perf_counter()
        res = oracle_lib.round_schedule(inp)
        dt = min(dt, time.perf_counter() - t)
        reps += 1
    out = {"value": placed / dt, "unit": UNIT, "cores": 1, "host_cores": host_cores(), "kind": "port",
           "sample": f"pool 0 of the cycle: {name} full round ({inp.num_nodes} nodes x {inp.num_jobs} jobs), best of {reps} runs, "
                     f"{dt:.3f} s/round, C++ restatement of the reference (Go toolchain unavailable; the reference round is "
                     f"single-goroutine, so 1 of the box's {host_cores()} cores)", "placements": placed, "seconds": dt}
    return (out, res) if keep_result else out


def run_reference(args):
    """The reference arm: the same cycle (the same `--pools` pools of the named configuration, one
    round each, one after the other like scheduling_algo.go:129-160) on the host cores, through the
    oracle port.  Runs exactly `--warmup` untimed and `--steps` timed cycles."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    name = args.workload
    import oracle_lib
    inputs = []
    keep = []
    for p in range(args.pools):
        r = make_workload(name, seed_offset=p)
        keep.append(r)
        inputs.append(r.to_input())
    for _ in range(args.warmup):
        for inp in inputs:
            oracle_lib.round_schedule(inp)
    t = time.perf_counter()
    placed = 0
    for _ in range(args.steps):
        for inp in inputs:
            res = oracle_lib.round_schedule(inp)
            placed += int(res.stats.placements)
    dt = time.perf_counter() - t
    val = placed / dt
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "int64+f64", "data": "synthetic",
        "config": workload_config(name, inputs[0], args.gpus, args.pools),
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": 1, "host_cores": host_cores(), "kind": "port",
                         "sample": f"{args.pools} pools x {name} full round, {args.steps} cycles after {args.warmup} warm-up cycles; "
                                   f"C++ restatement of the reference scheduler (single-goroutine algorithm, pools one after the "
                                   f"other => 1 of {host_cores()} host cores; Go toolchain unavailable here)"},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    emit(line)
    return 0


def extra_workload(dev, name, parity_name=None, steps=2):
    """One more BASELINE configuration on the device (resident inputs, best of `steps` runs after a
    warm-up; steps == 0: the first run is the measurement) with a bit-exact diff against the oracle on
    `parity_name` (default: the same input)."""
    import oracle_lib
    r = make_workload(name)
    inp = r.to_input()
    dev.upload(inp)
    best = dev.run()  # (warm-up; the only run when steps == 0)
    for _ in range(steps):
        st = dev.run()
        if st.device_ms < best.device_ms or best is None:
            best = st
    got = dev.download()
    out = {"value": best.placements / (best.device_ms / 1e3), "unit": UNIT, "ms_per_round": best.device_ms,
           "placements": int(best.placements), "scheduled": int(got.out.num_result_scheduled),
           "preempted": int(got.out.num_result_preempted), "nodes": int(inp.num_nodes), "jobs": int(inp.num_jobs)}
    if parity_name is None or parity_name == name:
        t = time.perf_counter()
        want = oracle_lib.round_schedule(inp)
        out["cpu_port_ms_per_round"] = (time.perf_counter() - t) * 1e3
        bad = got.diff(want)
        out["parity"] = {"checked": True, "against": f"oracle, {name} full size", "diffs": len(bad), "detail": bad[:3]}
    else:
        r2 = make_workload(parity_name)
        inp2 = r2.to_input()
        got2 = dev.schedule(inp2)
        t = time.perf_counter()
        want2 = oracle_lib.round_schedule(inp2)
        out["cpu_port_ms_per_round_at_parity_scale"] = (time.perf_counter() - t) * 1e3
        bad = got2.diff(want2)
        out["parity"] = {"checked": True, "against": f"oracle, {parity_name} (the reference's fair-preemption walk is quadratic; "
                                                     f"full size is covered by conservation properties)", "diffs": len(bad), "detail": bad[:3]}
        # size-independent properties at full size
        a = got
        ok = bool((a.node_alloc[0] >= 0).all())
        out["full_size_properties"] = {"no_oversubscription_at_evicted_priority": ok}
    return out


DUMP_LIMIT_BYTES = 64 * 10**6


def dump_outputs(out_dir, pools, results, inputs, job_sample=1 << 16, node_sample=1 << 13):
    """Write the output arrays a caller receives from armada_round_download for each pool in `pools`
    (results[i] belongs to pools[i]) as DIR/<name>.npy in float64, with the pool as the leading axis.
    Each pool's job and node axes are cut to a fixed sample (seed 0, sorted, the same in every run;
    job_sample.npy / node_sample.npy hold the indices); the sample is halved until the whole dump
    fits in DUMP_LIMIT_BYTES.  Integers are exact below 2**53; larger resource totals are rounded to
    float64.  The scalar results go to num_*.npy / termination_reason.npy with shape (pools,)."""
    from armada_b200.model import RoundResult
    inp0 = inputs[pools[0]]
    names = [n for n in RoundResult.ARRAYS if n != "job_excluded_nodes" or inp0.collect_excluded_nodes]
    if results[0].first_pass:
        names += ["job_seq_first_pass", "job_reason_first_pass"]
    while True:
        out = {"pool": np.asarray(pools, np.float64)}
        kj = min([job_sample] + [int(inputs[p].num_jobs) for p in pools])
        kn = min([node_sample] + [int(inputs[p].num_nodes) for p in pools])
        jidx = [np.sort(np.random.default_rng(0).choice(int(inputs[p].num_jobs), kj, replace=False)) for p in pools]
        nidx = [np.sort(np.random.default_rng(0).choice(int(inputs[p].num_nodes), kn, replace=False)) for p in pools]
        out["job_sample"] = np.stack(jidx).astype(np.float64)
        out["node_sample"] = np.stack(nidx).astype(np.float64)
        for n in names:
            rows = []
            for res, ji, ni in zip(results, jidx, nidx):
                a = getattr(res, n)
                if n.startswith("job_"):
                    a = a[ji]
                elif n == "node_alloc":
                    a = a[..., ni]
                rows.append(a.astype(np.float64))
            out[n] = np.stack(rows)
        for n in RoundResult.SCALARS:
            out[n] = np.asarray([getattr(res.out, n) for res in results], np.float64)
        total = sum(a.nbytes for a in out.values())
        if total <= DUMP_LIMIT_BYTES:
            break
        if job_sample <= 1 and node_sample <= 1:
            raise SystemExit(f"--dump-outputs: {total} bytes even with one job and one node per pool")
        job_sample, node_sample = max(1, job_sample // 2), max(1, node_sample // 2)
    os.makedirs(out_dir, exist_ok=True)
    for n, a in out.items():
        np.save(os.path.join(out_dir, f"{n}.npy"), a)
    return total


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="C3")
    ap.add_argument("--pools", type=int, default=8, help="pools per scheduling cycle (fixed: strong scaling over GPUs)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed cycle as DIR/<name>.npy (float64)")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "ours" or args.steps < 1):
        ap.error("--dump-outputs needs --impl ours and at least one timed step")
    if args.impl == "reference":
        return run_reference(args)
    args.warmup = max(args.warmup, 3)

    import torch
    import torch.distributed as dist
    from armada_b200 import pools as poolmod
    from armada_b200.model import RoundResult
    from armada_b200.scheduler import DeviceRound

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback)")
    torch.cuda.set_device(local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    P = args.pools
    mine = poolmod.pools_of_rank(P, rank, world)
    rt = torch.cuda.cudart()

    def pin(a):
        # page-granular: only large buffers are registered (small ones share pages)
        if a.nbytes >= (1 << 20):
            try:
                rt.cudaHostRegister(a.ctypes.data, a.nbytes, 0)
            except Exception:
                pass

    raws, inputs = {}, [None] * P
    for p in range(P):
        if p in mine or p == 0:
            raws[p] = make_workload(args.workload, seed_offset=p)
            inputs[p] = raws[p].to_input()
    for p in mine:
        for a in raws[p]._keep:
            pin(a)
    h2d = sum(raws[p].h2d_bytes() for p in mine)
    cyc = poolmod.PoolCycle(inputs, rank, world, lambda: DeviceRound(local))
    results = {p: RoundResult(inputs[p]) for p in mine}
    d2h_names = ("job_state", "job_node", "job_scheduled_at_priority", "job_preempted_at_priority", "job_method", "job_reason",
                 "node_alloc", "queue_allocated", "queue_allocated_by_pc", "queue_fair_share")
    for res in results.values():
        for nm in RoundResult.ARRAYS:
            pin(getattr(res, nm))
    d2h = sum(getattr(res, n).nbytes for res in results.values() for n in d2h_names)
    flush = torch.empty(256 * 2**20, dtype=torch.uint8, device="cuda")
    max_jobs = int(inputs[0].num_jobs)

    # ---- resident inputs: every owned pool keeps its own device context ---------------------------
    cyc.upload_resident()
    for _ in range(args.warmup):
        flush.zero_()
        stats_list = cyc.run_resident()
    sampler = ClockSampler(local)
    sampler.start()
    barrier()
    # The owned pools of a cycle run concurrently (one persistent CTA each).  Every round is timed on the
    # device with CUDA events on its own stream; the cycle lasts as long as its longest round (all rounds
    # are launched together), cross-checked against the wall clock of the bracketed call.
    dev_ms, pass_ms, round_ms, wall_ms, placements, probes, launches = 0.0, 0.0, 0.0, 0.0, 0, 0, 0
    for _ in range(args.steps):
        flush.zero_()
        torch.cuda.synchronize()
        tw = time.perf_counter()
        stats_list = cyc.run_resident()
        torch.cuda.synchronize()
        wall_ms += (time.perf_counter() - tw) * 1e3
        dev_ms += max((st.device_ms for st in stats_list), default=0.0)
        for st in stats_list:
            round_ms += st.device_ms
            pass_ms += st.schedule_pass_ms
            placements += int(st.placements)
            probes += int(st.probes)
            launches += int(st.gpu_launches)
    barrier()
    stats = stats_list[0] if stats_list else None
    # ---- end to end: host buffers in, host buffers out, every pool of every cycle; with more than
    # one rank the cycle's claims are gathered on all ranks (one all_gather over NCCL)
    for _ in range(1):
        out = cyc.schedule_cycle(results)  # untimed: the second pair of device contexts allocates its buffers
        if world > 1:  # … and the claims exchange its slabs and its NCCL connections
            poolmod.gather_claims(out, P, max_jobs, rank, world, dist)
    barrier()
    e2e_s = 0.0
    e2e_placed = 0
    for i in range(args.steps):
        flush.zero_()
        barrier()
        t = time.perf_counter()
        out = cyc.schedule_cycle(results)
        if world > 1:
            poolmod.gather_claims(out, P, max_jobs, rank, world, dist)
        torch.cuda.synchronize()
        e2e_s += time.perf_counter() - t
        e2e_placed += sum(int(out[p].stats.placements) for p in mine)
    barrier()
    clocks = sampler.stop()
    if args.dump_outputs and rank == 0:
        # the resident contexts still hold the last timed resident cycle (the end-to-end leg uses its own)
        dump_outputs(args.dump_outputs, mine, [cyc.download_resident(i) for i in range(len(mine))], inputs)

    tm = torch.tensor([dev_ms, e2e_s * 1e3, pass_ms], dtype=torch.float64, device="cuda")
    cnt = torch.tensor([placements, e2e_placed, probes, launches], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(tm, op=dist.ReduceOp.MAX)
        dist.all_reduce(cnt, op=dist.ReduceOp.SUM)
    tm, cnt = tm.cpu().numpy(), cnt.cpu().numpy()
    rc = 0
    if rank == 0:
        inp = inputs[0]
        value = cnt[0] / (tm[0] / 1e3)
        e2e_value = cnt[1] / (tm[1] / 1e3)
        N, Dn = int(inp.num_nodes), int(inp.num_resources)
        probe_bytes = N * (8 * Dn + 4)
        peak, peak_src = measured_peak()
        n_launch = args.steps * len(mine)
        achieved = (probes * probe_bytes) / (pass_ms / 1e3) / 1e9 if pass_ms > 0 else 0.0
        iters = max(1, int(stats.phase_cycles[4]))
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": tm[0] / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "int64+f64", "data": "synthetic", "config": workload_config(args.workload, inp, world, P),
            "ms_per_round": round_ms / max(1, n_launch),
            "cycle": {"pools_in_flight_per_gpu": len(mine), "ms_per_cycle_device": tm[0] / args.steps, "ms_per_cycle_wall": wall_ms / args.steps,
                      "round_ms_by_pool_last_step": [round(st.device_ms, 2) for st in stats_list],
                      "note": "a round is one persistent CTA on one SM; the pools of a cycle a rank owns run concurrently (up to 8 per GPU). "
                              "ms_per_round is the latency of ONE round (CUDA events on its stream) while the others run"},
            "placements_per_round": int(placements / max(1, n_launch)),
            "loop_iterations_per_round": int(stats.loop_iterations),
            "batch_mode": {"iterations": int(stats.phase_cycles[4]), "batches": int(stats.batch_cycles[6]),
                           "cycles_per_batched_iteration": {n: round(int(stats.batch_cycles[i]) / iters, 1) for i, n in enumerate(
                               ("item_build", "horizon", "merge_rank", "node_assign", "commit_repeek", "control"))}},
            "gpu_launches": int(cnt[3]),
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                    "ms_per_step": tm[1] / args.steps,
                    "note": "armada_round_upload/run/download with host buffers for every pool of the cycle, one device context and one "
                            "host thread per owned pool, all in flight together; wall clock from the first upload to the last download"},
            "roofline": {"bound": "hbm", "kernel": "k_schedule_pass", "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak, "traffic": ncu_traffic(), "peak_source": peak_src,
                         "algorithmic_bytes_per_probe": probe_bytes, "probes_per_launch": int(probes / max(1, n_launch)),
                         "kernel_ms_per_launch": pass_ms / max(1, n_launch),
                         "kernel_share_of_step": pass_ms / round_ms if round_ms else None,
                         "sm_cycles_per_placement": (pass_ms / 1e3) * (clocks.get("sm_mhz") or 1965.0) * 1e6 / max(1, placements),
                         "note": "scan-equivalent convention of SURVEY.md 8(d): the sorted index answers a probe without re-reading "
                                 "every node row, so frac > 1 is possible; the kernel is a latency-bound dependency chain and the honest "
                                 "gauge of head-room is sm_cycles_per_placement (DESIGN.md 5.4)"},
        }
        if not args.no_cpu_baseline:
            base, want = cpu_baseline(args.workload, keep_result=True)
            line["cpu_baseline"] = base
            got = results[0]
            bad = got.diff(want)
            line["parity"] = {"checked": True, "against": f"oracle, pool 0 of the cycle ({args.workload} full size), the result of the "
                                                          f"last timed end-to-end cycle", "diffs": len(bad), "detail": bad[:3],
                              "arrays": list(RoundResult.ARRAYS) + list(RoundResult.SCALARS)}
            if bad:
                rc = 3
        if not args.no_extras and world == 1 and args.workload == "C3":
            extras = {}
            with DeviceRound(local) as dev:
                # (C5 at full size is one run each side: about a minute on the device — every iteration of that
                # round goes through the general loop and its one-SM level scans — and 15 s for the oracle, whose
                # fair-preemption walk is replaced by its exact indexed form above 4096 evicted jobs)
                for nm, par, steps in (("C2", None, 2), ("C4", None, 2), ("C5", None, 0)):
                    try:
                        extras[nm] = extra_workload(dev, nm, par, steps)
                        if extras[nm]["parity"]["diffs"]:
                            rc = 3
                    except Exception as e:  # an extra workload must not take the headline down
                        extras[nm] = {"error": str(e)[:300]}
            line["extra_workloads"] = extras
        emit(line)
    cyc.close()
    if world > 1:
        dist.destroy_process_group()
    return rc


if __name__ == "__main__":
    sys.exit(main())
