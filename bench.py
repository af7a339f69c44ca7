#!/usr/bin/env python3
"""bench.py — headline benchmark of blance_b200 (contract: see the task statement).

Metric (BASELINE.json): partition-assignments/sec on the 1 048 576-partition x
1 024-node synthetic cluster (configs[3]: heterogeneous node + partition weights,
stickiness, 16 nodes removed / 16 added), i.e. partitions planned per second by ONE
complete PlanNextMapEx (all convergence iterations, plan.go:23-58).

  step        one complete plan of that cluster
  value       partitions/s with the tables resident in HBM (blance_plan_run), device
              time from CUDA events on the library's stream, max over ranks
  e2e         the same through blance_plan_next_map with HOST buffers: staging, H2D,
              all kernels, D2H inside the timed region
  roofline    of the dominant kernel k_assign_pass_spec: algorithmic bytes per findBestNodes
              step (SURVEY.md section 8d: 16*N + (N/8)(1+R*k) + 8*slots + 12) x steps /
              its device time, against the measured HBM copy bandwidth
  cpu_baseline  the literal C++ restatement of the Go planner (oracle/literal.cpp: string
              hash maps + comparison sort, the reference's asymptotics) on a bounded
              sample of the same cluster shape, 1 core (the reference planner is
              single-goroutine).  Go itself cannot run here (no toolchain).

  parity      sha256 of the result next to the oracle's (profiles/parity_cfg4.json); e2e_string_api: the same
              plan through the string API (maps of strings in and out); batch_cfg5: BASELINE config 5
              (1 024 instances in one blance_plan_next_map_batch call) on this GPU

--gpus N: the greedy chain of one plan is sequential (each step reads the counts the
previous step wrote), so one plan does not shard; N ranks plan the SAME cluster, one plan
per GPU — "replicas only", weak scaling, no collective in the data path;
torch.distributed(nccl) is used for the barrier and the max over ranks.  What shards is the
batch: tools/bench_cfg5.py runs config 5 over 1/2/4/8 GPUs through blance_ctx_create_multi.

--impl reference: the CPU arm — slices of the real workload's first inner plan through the
literal oracle on the box's host cores (rank 0 only).

--dump-outputs DIR: after the timed steps, rank 0 writes what the last timed plan returned to its caller
(blance_plan_fetch) as DIR/<name>.npy, so that two builds can be compared output for output on the same
seeded cluster.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

CFG = 4
METRIC = "partition-assignments/sec, 1M parts x 1024 nodes (partitions planned per second by one complete PlanNextMapEx)"
UNIT = "partitions/s"


def b_alg(n_nodes, n_rules, k, slots):
    return 16 * n_nodes + (n_nodes // 8) * (1 + n_rules * k) + 8 * slots + 12


def measured_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except Exception:
                pass
        sm = [float(r[0]) for r in self.rows if len(r) >= 7 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) >= 7 and r[1].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            if len(r) >= 7:
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


WORKLOAD = "cfg4: PlanNextMapEx 1048576 partitions x 1024 nodes, k=(1,2), node+partition weights, stickiness, -16/+16 nodes"
# Every partition takes exactly one findBestNodes step per state pass (plan.go:268) and the cluster does not converge
# (tests/test_gpu_parity.py::test_cfg4_full_size_bit_exact pins iters_run == MaxIterationsPerPlan == 10 on the GPU and on
# the oracle), so a complete plan is 2 passes x 10 iterations = 20 steps per partition.
STEPS_PER_PARTITION = 2 * 10


def literal_slices(parts, n_slices, slice_steps):
    """The reference-equivalent CPU path (oracle/literal.cpp: string hash maps + comparison sort, statement for
    statement plan.go) on the REAL maps of the workload: the cfg-4 PartitionMap of `parts` partitions is built once,
    one inner plan (plan.go:60) starts on it, and the greedy chain of its two state passes is timed in slices of
    `slice_steps` consecutive findBestNodes steps.  Returns the per-slice seconds."""
    from oracle_loader import literal
    from blance_b200 import synth                      # table builder only: loads no native product code
    L = literal()
    t = synth.make_rebalance(CFG, P=parts)
    kw = synth.to_dicts(t, CFG)
    kw["partitions_to_assign"] = None                  # the same map object twice, as blance's callers do
    kw["max_iterations"] = 1
    per_pass = ((n_slices + 1) // 2) * slice_steps
    r = L.plan_next_map_ex(**kw, max_steps_per_pass=per_pass, slice_steps=slice_steps, memoize_partition_scores=True)
    return list(r["slice_seconds"])[:n_slices]


def cpu_literal_sample(parts, seed_offset=0):
    """The literal oracle on a cfg-4-shaped cluster with `parts` partitions x 1024 nodes, one inner plan.
    Returns (findBestNodes steps, seconds)."""
    from oracle_loader import literal
    from blance_b200 import synth
    L = literal()
    t = synth.make_rebalance(CFG, P=parts, seed_offset=seed_offset)
    kw = synth.to_dicts(t, CFG)
    kw["max_iterations"] = 1
    r = L.plan_next_map_ex(**kw)
    return r["steps"], r["seconds"]


def cpu_fast_sample(parts):
    import ctypes
    from oracle_loader import fast_lib_path
    from blance_b200 import synth, tables
    fast = ctypes.CDLL(fast_lib_path())
    fast.oracle_fast_plan_next_map.argtypes = [ctypes.c_void_p, ctypes.c_void_p]
    t = synth.make_rebalance(CFG, P=parts)
    t.max_iters = 1
    r = tables.PlanResult(t)
    s = t.struct()
    t0 = time.perf_counter()
    fast.oracle_fast_plan_next_map(ctypes.byref(s), ctypes.byref(r.out))
    return r.steps, time.perf_counter() - t0


def ncu_traffic(steps_per_launch):
    """DRAM bytes per k_assign_pass launch from the committed ncu --set full capture
    (profiles/ncu_traffic.json: dram read+write bytes per step of one captured launch), scaled to
    the bench's steps per launch; None when no capture is committed."""
    try:
        with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as f:
            return float(json.load(f)["dram_bytes_per_step"]) * steps_per_launch
    except Exception:
        return None


DUMP_LIMIT = 64 << 20


def dump_outputs(out_dir, res):
    """next_rows / next_shape / warn of a PlanResult as float32 (node ids, shapes and warning flags are small
    integers, exact in float32) and its counters (iters_run, converged, steps) as float64.  Above DUMP_LIMIT bytes
    a fixed seeded sample of partitions is written, their indices in partition_index.npy."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"next_rows": res.next_rows, "next_shape": res.next_shape, "warn": res.warn}
    n_parts = res.next_rows.shape[0]
    row_bytes = 4 * sum(a.shape[1] for a in arrays.values())
    if n_parts * row_bytes > DUMP_LIMIT:
        n_keep = (DUMP_LIMIT - 4096) // (row_bytes + 8)          # 4 KiB for the .npy headers and the counters
        idx = np.sort(np.random.default_rng(0).choice(n_parts, n_keep, replace=False))
        arrays = {k: a[idx] for k, a in arrays.items()}
        np.save(os.path.join(out_dir, "partition_index.npy"), idx.astype(np.float64))
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a.astype(np.float32))
    np.save(os.path.join(out_dir, "counters.npy"), np.array([res.iters_run, res.converged, res.steps], np.float64))


def shared_config(n_parts, n_nodes):
    """The part of `config` both arms print identically."""
    return {"workload": WORKLOAD if (n_parts, n_nodes) == (1048576, 1024) else
            "cfg4 shape at %d partitions x %d nodes (debug size, not the headline)" % (n_parts, n_nodes),
            "n_parts": n_parts, "n_nodes": n_nodes, "steps_per_partition": float(STEPS_PER_PARTITION)}


def run_reference(args, rank, world):
    """--impl reference: the reference's own algorithm on the host cores.  One bench step = one slice of
    `--cpu-slice-steps` consecutive findBestNodes steps of the real workload's first inner plan."""
    if rank != 0:
        return
    parts = args.parts or 1048576
    n = args.warmup + args.steps
    secs = literal_slices(parts, n, args.cpu_slice_steps)
    timed = secs[args.warmup:]
    total = sum(timed)
    steps_per_s = args.cpu_slice_steps * len(timed) / total
    value = steps_per_s / STEPS_PER_PARTITION
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * total / max(1, len(timed)), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64 score / int32 tables", "data": "synthetic",
        "config": shared_config(parts, 1024),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": 1, "kind": "port",
                         "findBestNodes_steps_per_s": steps_per_s,
                         "sample": "oracle/literal.cpp (C++ restatement of plan.go with the reference's string maps and "
                                   "comparison sort; Go itself cannot be built in this image) on the real %d x 1024 cfg-4 maps: "
                                   "%d slices of %d consecutive findBestNodes steps of the first inner plan (both state passes), "
                                   "timed inside the pass loop; partitions/s = steps/s / %d steps per partition; 1 core because "
                                   "the reference planner is single-goroutine" % (parts, len(timed), args.cpu_slice_steps, STEPS_PER_PARTITION)},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="blance_b200")
    ap.add_argument("--parts", type=int, default=None, help="override the partition count (debug only; invalidates the headline)")
    ap.add_argument("--cpu-sample-parts", type=int, default=1024)
    ap.add_argument("--cpu-slice-steps", type=int, default=256, help="findBestNodes steps per reference-arm bench step")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-string-api", action="store_true")
    ap.add_argument("--no-batch", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the last timed plan's result arrays to DIR/<name>.npy (float32 / float64)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs needs the GPU implementation: the reference arm times slices of a plan and returns no map")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import numpy as np
    import torch
    from blance_b200 import synth, tables

    dist = None
    if world > 1:
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    # every rank plans the SAME cluster (replicas): the chain's length depends on the data, so different seeds per rank
    # would make the max over ranks a property of the slowest seed rather than of the machine
    t = synth.make_rebalance(CFG, P=args.parts)
    ctx = tables.Context(local_rank)
    plan = ctx.upload(t)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)     # > L2 (126 MB)

    for _ in range(max(args.warmup, 3)):
        ctx.run(plan)
    res = ctx.fetch(plan, tables.PlanResult(t))
    steps_per_plan, iters, sticky = int(res.steps), int(res.iters_run), int(res.sticky_steps)

    sampler = ClockSampler(local_rank) if rank == 0 else None
    barrier()
    if sampler:
        sampler.start()
    launches0 = ctx.kernel_launches()
    kernel_ms, pass_ms, pass_launches = [], [], 0
    for _ in range(args.steps):
        flush.zero_()                       # L2 flush between timed iterations (not timed)
        torch.cuda.synchronize()
        ctx.run(plan)
        k, p, n = ctx.timing(plan)
        kernel_ms.append(k)
        pass_ms.append(p)
        pass_launches += n
    barrier()
    launches = ctx.kernel_launches() - launches0
    clocks = sampler.stop() if sampler else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, ctx.fetch(plan, tables.PlanResult(t)))
    total_ms = sum(kernel_ms)
    tt = torch.tensor([total_ms, sum(pass_ms)], dtype=torch.float64, device=dev)
    if dist is not None:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    total_ms_max, pass_ms_max = float(tt[0]), float(tt[1])
    per_rank = [total_ms / args.steps]
    if dist is not None:
        g = [torch.zeros(1, dtype=torch.float64, device=dev) for _ in range(world)]
        dist.all_gather(g, torch.tensor([total_ms / args.steps], dtype=torch.float64, device=dev))
        per_rank = [float(x[0]) for x in g]

    # ---- end to end through the C ABI with host buffers -----------------------------------
    h2d = sum(np.asarray(getattr(t, f)).nbytes for f in
              ("prev_rows", "cur_rows", "prev_shape", "cur_shape", "part_in_prev", "part_in_assign", "part_weight",
               "part_has_weight", "part_name_rank", "node_removed", "node_added", "node_weight", "node_has_weight",
               "extra_tot_first", "extra_tot_rest", "ie_mask"))
    out = tables.PlanResult(t)
    d2h = out.next_rows.nbytes + out.next_shape.nbytes + out.warn.nbytes
    ctx.plan_next_map(t, out)               # warm-up of the e2e path
    barrier()
    e2e_s = []
    e2e_steps = args.steps
    for _ in range(e2e_steps):
        t0 = time.perf_counter()
        ctx.plan_next_map(t, out)
        e2e_s.append(time.perf_counter() - t0)
    barrier()
    te = torch.tensor([sum(e2e_s)], dtype=torch.float64, device=dev)
    if dist is not None:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_total = float(te[0])
    same = bool(np.array_equal(out.next_rows, res.next_rows))

    # ---- CalcPartitionMoves over the whole map (prev -> next), through the C ABI with host buffers -----
    ctx.calc_partition_moves(t.state_slot_off, t.prev_rows, out.next_rows, False)
    t0 = time.perf_counter()
    mv = ctx.calc_partition_moves(t.state_slot_off, t.prev_rows, out.next_rows, False)
    moves_s = time.perf_counter() - t0
    moves_ops = int(mv[3].sum())

    # ---- outside every timed region: the result's digest next to the oracle's (profiles/parity_cfg4.json, written by
    # tools/make_parity_digest.py; the full arrays are compared in tests/test_gpu_parity.py::test_cfg4_full_size_bit_exact)
    import hashlib
    parity = {"sha256_gpu": hashlib.sha256(np.ascontiguousarray(res.next_rows).tobytes()).hexdigest(), "sha256_oracle": None,
              "iters_run": iters, "steps": steps_per_plan}
    try:
        with open(os.path.join(ROOT, "profiles", "parity_cfg4.json")) as f:
            pj = json.load(f)
        if args.parts is None and pj.get("n_parts") == t.n_parts:
            parity["sha256_oracle"] = pj["sha256_next_rows"]
            parity["equal"] = (parity["sha256_gpu"] == pj["sha256_next_rows"] and iters == pj["iters_run"] and steps_per_plan == pj["steps"])
    except Exception:
        pass

    # ---- the string API end to end (PartitionMap of strings in and out: InternPlan + C ABI + UninternPlan + the caller-map
    # mutation of plan.go:49-52), on the same cluster, rank 0 only; the map is built natively (no Python dicts in the timing)
    string_api = None
    if rank == 0 and not args.no_string_api:
        import blance_b200
        removed = np.nonzero(t.node_removed)[0].tolist()
        added = np.nonzero(t.node_added)[0].tolist()
        reps = []
        for _ in range(2):       # the first call pays the page faults of its fresh allocations
            d = blance_b200._host.bench_string_api(t.prev_rows, t.n_nodes, [int(x) for x in t.state_constraints], removed, added,
                                                   t.node_weight, t.part_weight, t.part_has_weight, [int(x) for x in t.state_stickiness], 10)
            reps.append(d)
        d = reps[-1]
        string_api = {"value": t.n_parts / (d["total_ms"] / 1e3), "unit": UNIT, "ms": d["total_ms"], "first_call_ms": reps[0]["total_ms"],
                      "intern_ms": d["intern_ms"], "c_abi_call_ms": d["call_ms"], "unintern_ms": d["unintern_ms"],
                      "caller_map_mutation_ms": d["mutate_ms"], "host_threads": d["host_threads"],
                      "result_equals_resident_run": bool(np.array_equal(d["next_rows"], res.next_rows)),
                      "note": "blance.PlanNextMapEx of the C++ host twin (host_api.cpp) on %d string partitions; what a Go host "
                              "pays when it does not keep its maps interned" % t.n_parts}

    # ---- BASELINE config 5 on this GPU: 1 024 independent instances (multi-tenant fan-out) in one batch call; the struct
    # arrays are built once, the timed call is blance_plan_next_map_batch alone (H2D, all kernels, D2H inside)
    batch = None
    if rank == 0 and not args.no_batch:
        n_inst = 1024
        fresh = [synth.make_fresh(5, seed_offset=i) for i in range(n_inst)]
        prep = ctx.prepare_batch(fresh)
        got = ctx.run_batch(prep)
        rebs = [synth.make_rebalance(5, g.next_rows, seed_offset=i) for i, g in enumerate(got)]
        prep2 = ctx.prepare_batch(rebs)
        ctx.run_batch(prep2)                                  # warm-up
        ts_ = []
        for _ in range(3):
            t0 = time.perf_counter()
            r5 = ctx.run_batch(prep2)
            ts_.append(time.perf_counter() - t0)
        best = min(ts_)
        parts5 = sum(x.n_parts for x in rebs)
        batch = {"workload": "cfg5: %d independent PlanNextMapEx instances (1024 partitions x 64 nodes, rack rules), rebalance stage" % n_inst,
                 "value": parts5 / best, "unit": UNIT, "ms": 1e3 * best, "instances_per_s": n_inst / best,
                 "device_ms": float(r5[0].device_ms), "n_gpus": 1,
                 "note": "wall time of the C call with host buffers; multi-GPU sharding of the batch: tools/bench_cfg5.py, profiles/"}

    if rank == 0:
        P, N = t.n_parts, t.n_nodes
        value = world * P * args.steps / (total_ms_max / 1e3)
        e2e_value = world * P * args.steps / e2e_total
        bytes_per_step = b_alg(N, 0, 2, t.n_slots)
        peak, peak_src = measured_peak()
        pass_s = pass_ms_max / 1e3
        achieved = steps_per_plan * args.steps * bytes_per_step / pass_s / 1e9 if pass_s > 0 else None
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": total_ms_max / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64 score / int32 tables", "data": "synthetic",
            "config": shared_config(P, N),
            "run": {"step": "one complete plan (%d convergence iterations, %d findBestNodes steps)" % (iters, steps_per_plan),
                    "steps_per_partition_measured": steps_per_plan / P,
                    "findBestNodes_steps_per_s": world * steps_per_plan * args.steps / (total_ms_max / 1e3),
                    "accepted_fraction": sticky / max(1, steps_per_plan),
                    "parallelism": "replicas only: %d rank(s) plan the same cluster, one plan per GPU; no data-path collective" % world,
                    "ms_per_step_per_rank": per_rank,
                    "l2": "256 MiB device buffer rewritten between timed iterations (L2 flush)",
                    "timing": "CUDA events on the library stream, max over ranks"},
            "parity": parity,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                    "ms_per_step": 1e3 * e2e_total / args.steps, "result_equals_resident_run": same},
            "calc_partition_moves": {"partitions_per_s": P / moves_s, "ms": 1e3 * moves_s, "ops": moves_ops,
                                     "note": "moves.go:41-119 for all partitions in one launch, prevMap -> nextMap, host buffers "
                                             "(H2D of both maps and D2H of the op lists inside the timed call)"},
            "e2e_string_api": string_api,
            "batch_cfg5": batch,
            "gpu_launches": int(launches),
            "clocks": clocks,
            "roofline": {"bound": "hbm", "kernel": "k_assign_pass_spec (the speculative assign pass; k_assign_pass runs the passes that do not qualify)", "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": (achieved / peak) if achieved else None, "traffic": ncu_traffic(steps_per_plan * args.steps / max(1, pass_launches)),
                         "peak_source": peak_src, "bytes_per_findBestNodes_step": bytes_per_step,
                         "steps_per_launch": steps_per_plan * args.steps / max(1, pass_launches),
                         "t_step_ns": 1e9 * pass_s / (steps_per_plan * args.steps),
                         "note": "the pass is a loop-carried dependency chain (latency bound), not a streaming kernel; "
                                 "see DESIGN.md"},
        }
        if world == 1 and not args.no_cpu_baseline:
            st, sec = cpu_literal_sample(args.cpu_sample_parts)
            spp = steps_per_plan / P
            fst, fsec = cpu_fast_sample(32768)
            line["cpu_baseline"] = {
                "value": st / sec / spp, "unit": UNIT, "cores": 1, "kind": "port",
                "findBestNodes_steps_per_s": st / sec,
                "sample": "literal C++ restatement of the Go planner (oracle/literal.cpp) on one inner plan of a %d-partition x "
                          "%d-node cluster of the same shape (%d findBestNodes steps, %.1f s); partitions/s = steps/s / %.1f steps "
                          "per partition of the full workload" % (args.cpu_sample_parts, N, st, sec, spp),
                "best_cpu_array_oracle": {"value": fst / fsec / spp, "unit": UNIT, "findBestNodes_steps_per_s": fst / fsec,
                                          "sample": "oracle/fast.c, 32768 x %d, one inner plan" % N}}
            line["cpu_array_oracle"] = dict(line["cpu_baseline"]["best_cpu_array_oracle"], cores=1, kind="port",
                                            note="the best CPU restatement we have (array form, O(N) arg-min per pick): the ratio "
                                                 "to THIS says what the GPU kernel buys; the literal restatement above is the reference's cost")
        print(json.dumps(line), flush=True)
    ctx.free(plan)
    ctx.close()
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
