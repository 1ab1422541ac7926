#!/usr/bin/env python3
"""bench.py — pods scheduled/sec of Scheduler.Solve on a synthetic cluster (BASELINE.json metric).

  python bench.py --gpus N --steps K --warmup W            our arm (CUDA path through the C-ABI)
  python bench.py --impl reference --gpus N --steps K ...   the reference's algorithm on the host CPU (oracle port)
  ... --dump-outputs DIR                                    also write the last timed Solve's Result as DIR/<name>.npy

A "step" is one Solve over one batch of synthetic pods. Workload at N=1: BASELINE.json configs[3], the configuration the
metric's target is quoted on (C4: 100 000 pods with pod anti-affinity + zone / hostname topology spread x 1 000 instance
types) — it fits one GPU. `--config 2|3` select the smaller configurations; the default line carries them as secondary
blocks (`config_c2`, `config_c3`).
  value     pods/s with the encoded problem already resident in HBM (sort + feasibility + pack kernels), L2 flushed
            before every step, timed with CUDA events on the library's stream, max over ranks.
  e2e       the same metric through the reference-facing call with HOST data: the string-level model (what NewScheduler
            receives) -> host encoder -> ksched_solve (pod / topology upload, kernels, result download) -> decode to the
            ([]*Node, []*ExistingNode) shape. The instance-type catalog stays resident, as across reconciles.
            `e2e.solve_only` is ksched_solve alone (flat structs in, flat structs out).
  roofline  the dominant kernel (pack_kernel); roofline_feasibility the kernel BASELINE.json's 40 % target names.
N>1: one Solve is a sequential first-fit chain and does not shard (DESIGN.md section 8: "replicas only"): every rank
runs its own independent Solve of the same shape (seed 42 + rank), no collective on the data path; value = pods all ranks
scheduled / slowest rank's time, scaling "weak".
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))

CONFIGS = {
    1: dict(pods=100, types=10, nodes=0, name="C1: 100 pods x 10 instance types (reference benchmark shape)"),
    2: dict(pods=10_000, types=500, nodes=0, name="C2: 10k pods x 500 instance types, cpu/mem requests only, 1 provisioner"),
    3: dict(pods=50_000, types=1000, nodes=0, name="C3: 50k pods nodeSelector+taints x 1k instance types, 3 provisioners"),
    4: dict(pods=100_000, types=1000, nodes=0, name="C4: 100k pods anti-affinity+topology-spread (zone,hostname) x 1k instance types"),
}
CPU_SAMPLE = {1: 100, 2: 10_000, 3: 3_000, 4: 2_000}  # pods the literal oracle solves in ~10-20 s on one core


def measured_peak():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            return float(json.loads(p.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def ncu_traffic(kernel):
    p = ROOT / "profiles" / "traffic.json"
    if p.exists():
        try:
            return json.loads(p.read_text()).get(kernel)
        except Exception:
            return None
    return None


def golden(config, pods, types, seed):
    """the committed full-size oracle result of this exact workload (tests/golden/fullsize), or None"""
    p = ROOT / "tests" / "golden" / "fullsize" / f"c{config}.json"
    if p.exists():
        g = json.loads(p.read_text())
        if g.get("pods") == pods and g.get("types") == types and g.get("seed") == seed:
            return g
    return None


DUMP_LIMIT = 64 << 20
DUMP_OPTION_BYTES = 16 << 20  # C4's full option matrix (20 000 nodes x 1 000 types) is 80 MB: a fixed sample of its rows


def dump_outputs(problem, res, out_dir):
    """Write the Result of the last timed Solve as .npy files, so that two builds can be compared output for output:
      assign                   [pods] node each pod was placed on, -1 if unschedulable
      relax_level              [pods] preference relaxation level of each pod
      new_node_info            [new nodes, 3] provisioner (weight order), pod count, instance-type option count
      new_node_requests_<res>  [new nodes] summed requests of resource <res>
      new_node_launch          [new nodes, 2] launched instance type and its price, -1 where the result has no launch choice
      new_node_options         [rows, instance types] 1 where the type is an option of the node (float32)
      new_node_options_rows    [rows] which new nodes those rows are: all of them, or a sample fixed by seed 0 when the
                               full matrix exceeds DUMP_OPTION_BYTES
    Every other file is float64, which holds these integers and the memory requests (~1e13 milli-bytes) exactly."""
    nodes = res.to_dict(brief=True)["newNodes"]
    out = {"assign": res.assign, "relax_level": res.relax_level, "new_node_info": res.new_node_info()}
    for name in sorted({k for n in nodes for k in n["requests"]}):
        out[f"new_node_requests_{name}"] = [n["requests"].get(name, 0) for n in nodes]
    out["new_node_launch"] = np.array([[n["launch"]["type"], n["launch"]["price"]] if "launch" in n else [-1, -1] for n in nodes]).reshape(-1, 2)
    out = {k: np.asarray(v, dtype=np.float64) for k, v in out.items()}
    n_types = problem.counts()["instance_types"]
    rows = min(len(nodes), DUMP_OPTION_BYTES // (4 * n_types))
    pick = np.sort(np.random.default_rng(0).choice(len(nodes), rows, replace=False))
    options = np.zeros((rows, n_types), dtype=np.float32)
    for r, i in enumerate(pick):
        options[r, res.new_node_options(int(i))] = 1
    out["new_node_options"] = options
    out["new_node_options_rows"] = pick.astype(np.float64)
    total = sum(a.nbytes for a in out.values())
    if total > DUMP_LIMIT:
        raise RuntimeError(f"--dump-outputs: {total} bytes exceed the {DUMP_LIMIT}-byte limit; use a smaller workload")
    out_dir.mkdir(parents=True, exist_ok=True)
    for name, a in out.items():
        np.save(out_dir / f"{name}.npy", a)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""

    def __init__(self, index):
        self.index = index
        self.samples = []
        self.proc = None

    def start(self):
        q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
            "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.samples.append(line.strip())

    def mark(self):
        """the timed region starts here: earlier samples (nvidia-smi needs a few hundred ms to start) are dropped"""
        self.samples = []

    def stop(self):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()
        sm, mx, reasons = [], 0, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for s in self.samples:
            f = [x.strip() for x in s.split(",")]
            if len(f) < 6:
                continue
            try:
                sm.append(float(f[0]))
                mx = max(mx, float(f[1]))
            except ValueError:
                continue
            for n, v in zip(names, f[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx or None, "reasons": sorted(reasons), "samples": len(sm)}


def workload_config(args):
    cfg = CONFIGS[args.config]
    return cfg, args.pods or cfg["pods"], args.types or cfg["types"]


def public_config(cfg, pods, types):
    """identical keys in both arms (the driver compares them)"""
    return {"workload": cfg["name"], "pods": pods, "instance_types": types}


def run_reference(args, rank, world):
    """The reference's algorithm on the host CPU: the literal C++ oracle port, one thread (Scheduler.Solve is a single
    goroutine; the Go toolchain is absent so the reference itself cannot run). Each step solves a bounded sample of the
    workload: the reference's cost per pod grows with the number of nodes it has opened, so the rate on the sample is an
    UPPER bound of its rate on the full workload."""
    if rank != 0:
        return
    from __graft_entry__ import load_pkg
    import oracle_lib
    pkg, oracle = load_pkg(), oracle_lib.load()
    cfg, pods, types = workload_config(args)
    budget_s = 200.0
    sample = min(pods, CPU_SAMPLE[args.config])
    res = pkg.Result()
    while True:
        problem = pkg.Problem.synth(args.config, sample, types, 42, cfg["nodes"])
        t0 = time.perf_counter()
        oracle.solve(problem, res)
        first = time.perf_counter() - t0
        if first * (args.steps + args.warmup) <= budget_s or sample <= 250:
            break
        sample = max(250, sample // 2)
    for _ in range(max(0, args.warmup - 1)):
        oracle.solve(problem, res)
    total, scheduled = 0.0, 0
    for _ in range(args.steps):
        t0 = time.perf_counter()
        oracle.solve(problem, res)
        total += time.perf_counter() - t0
        scheduled = int((res.assign >= 0).sum())
    value = scheduled * args.steps / total
    sample_desc = f"first-fit Solve of a {sample}-pod batch of the same generator ({types} instance types), {args.steps} runs of {total / args.steps:.2f} s; " \
                  f"literal port, 1 thread of {os.cpu_count()}; the per-pod cost grows with the batch, so this over-states the reference at {pods} pods"
    line = {
        "impl": "reference", "metric": "pods scheduled/sec (Scheduler.Solve)", "value": value, "unit": "pods/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1000 * total / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "int64", "data": "synthetic",
        "config": public_config(cfg, pods, types),
        "cpu_baseline": {"value": value, "unit": "pods/s", "cores": 1, "kind": "port", "sample": sample_desc},
        "e2e": {"value": value, "unit": "pods/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    if args.dump_outputs:
        dump_outputs(problem, res, args.dump_outputs)
    print(json.dumps(line), flush=True)


def secondary(pkg, config, steps=3):
    """one resident + one end-to-end measurement of a smaller BASELINE configuration (rank 0, N=1)"""
    cfg = CONFIGS[config]
    problem = pkg.Problem.synth(config, cfg["pods"], cfg["types"], 42, 0)
    rs = pkg.ResidentSolve(problem)
    rs.set_count_visited(False)
    rs.load()
    rs.run(flush_l2=True)
    ph = {"sort_us": 0.0, "feasibility_us": 0.0, "pack_us": 0.0, "total_us": 0.0}
    for _ in range(steps):
        rs.run(flush_l2=True)
        t = rs.timings()
        for k in ph:
            ph[k] += t[k]
    res = rs.download()
    sched = int((res.assign >= 0).sum())
    pkg.solve_timed(problem)
    tot = 0.0
    for _ in range(steps):
        _, t = pkg.solve_timed(problem)
        tot += t["total_us"]
    g = golden(config, cfg["pods"], cfg["types"], 42)
    out = {"workload": cfg["name"], "pods": cfg["pods"], "instance_types": cfg["types"], "scheduled": sched, "new_nodes": int(res.num_new_nodes),
           "value": sched * steps / (ph["total_us"] * 1e-6), "unit": "pods/s", "ms_per_step": ph["total_us"] / steps / 1000,
           "phases_ms_per_step": {k[:-3]: v / steps / 1000 for k, v in ph.items()},
           "e2e_value": sched * steps / (tot * 1e-6), "e2e_ms_per_step": tot / steps / 1000, "steps": steps, "warmup": 1}
    if g:
        out["parity_vs_oracle"] = bool(int(res.digest()) == g["digest"])
    return out


C5 = dict(nodes=5000, pods=50_000, types=1000, name="C5: multi-node consolidation, 5k existing nodes / 50k bound pods x 1k instance types")
OPT_CAP = 1024  # instance-type options exchanged per verdict


def c5_block(pkg, torch, dist, rank, world, steps):
    """BASELINE config 5 as one consolidation pass per step: candidates ranked on the device, the cluster resident on every
    rank's GPU (ksched_load_cluster), the multi-node binary search with its probes one per GPU (speculative frontier, SURVEY
    8e) and single-node consolidation's worst case - every candidate simulated - sharded by position. The only exchange is ONE ncclAllGather of
    the verdicts per round on the scheduler handle's communicator. value = pods re-packed per second over every simulation
    run; parity = command + probe trace equal to the committed oracle run (tests/golden/fullsize/c5.json)."""
    problem = pkg.Problem.synth(5, C5["pods"], C5["types"], 42, C5["nodes"])
    if world > 1:
        import ctypes as C
        uid = torch.zeros(128, dtype=torch.uint8, device="cuda")
        if rank == 0:
            buf = (C.c_ubyte * 128)()
            assert pkg.lib().ksched_nccl_unique_id(buf) == 0
            uid.copy_(torch.tensor(list(buf), dtype=torch.uint8))
        dist.broadcast(uid, 0)
        raw = bytes(uid.cpu().tolist())
        pkg._check(pkg.lib().kh_nccl_init(raw, rank, world))

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def gather(mine, per_rank):
        """{key: (action, options)} of every rank through one ncclAllGather of fixed-size int records"""
        if world == 1:
            return dict(mine)
        rec = 3 + OPT_CAP
        flat = []
        for key, (action, options) in list(mine.items())[:per_rank]:
            flat += [key, action, len(options)] + list(options[:OPT_CAP]) + [0] * (OPT_CAP - min(len(options), OPT_CAP))
        flat += [-1] * (per_rank * rec - len(flat))
        out = {}
        for part in pkg.nccl_allgather_i32(flat, world):
            for q in range(per_rank):
                r = part[q * rec:(q + 1) * rec]
                if r[0] >= 0:
                    out[r[0]] = (r[1], r[3:3 + r[2]])
        return out

    stats = {"multi_s": 0.0, "single_s": 0.0, "rank_s": 0.0, "open_s": 0.0, "repacked": 0, "simulations": 0}
    last = {}
    for step in range(steps + 1):  # the first pass is the warm-up
        barrier()
        t0 = time.perf_counter()
        order, cost = pkg.rank_candidates(problem)
        t1 = time.perf_counter()
        sess = pkg.ClusterSession(problem)
        barrier()
        t2 = time.perf_counter()
        n = sess.n_candidates
        evaluated = []

        def probe_many(counts):
            mine = {}
            for i, c in enumerate(counts):
                if i % world == rank:
                    mine[c] = sess.probe_sets([list(range(c))], True)[0]
            evaluated.extend(counts)
            return gather(mine, (len(counts) + world - 1) // world)

        action, removed, options, rounds, path = pkg.speculative_binary_search(n, probe_many, world)
        barrier()
        t3 = time.perf_counter()
        # single-node consolidation, worst case: every candidate is simulated (singlenodeconsolidation.go:54-77 walks the whole list
        # when no command validates). The simulations are independent: positions split over the ranks, 64 per device call.
        per = (n + world - 1) // world
        lo, hi = min(n, rank * per), min(n, (rank + 1) * per)
        hit = None
        for b in range(lo, hi, 64):
            res = sess.probe_sets([[i] for i in range(b, min(hi, b + 64))], False)
            for q, (a, o) in enumerate(res):
                if a and hit is None:
                    hit = (b + q, a, o)
        hits = gather({hit[0]: (hit[1], hit[2])} if hit else {}, 1)
        barrier()
        t4 = time.perf_counter()
        sess.close()
        single = min(hits.items())[0:1] + min(hits.items())[1] if hits else None
        if step == 0:
            continue
        stats["rank_s"] += t1 - t0; stats["open_s"] += t2 - t1; stats["multi_s"] += t3 - t2; stats["single_s"] += t4 - t3
        stats["repacked"] += 10 * sum(evaluated)
        stats["simulations"] += len(evaluated)
        last = {"action": action, "nodes_removed": removed, "n_options": len(options), "rounds": rounds, "probes_on_path": path,
                "single_node": {"position": single[0], "action": single[1], "n_options": len(single[2])} if single else None,
                "candidates": n, "first_candidates": order[:4]}
    out = {"workload": C5["name"], "nodes": C5["nodes"], "bound_pods": C5["pods"], "instance_types": C5["types"], "steps": steps, "warmup": 1,
           "value": stats["repacked"] / stats["multi_s"], "unit": "pods re-packed/s (multi-node search, every simulation run)",
           "multi_node_search_ms": 1000 * stats["multi_s"] / steps, "simulations_per_search": stats["simulations"] / steps,
           "single_node_all_candidates_ms": 1000 * stats["single_s"] / steps,
           "single_node_simulations_per_s": C5["nodes"] * steps / stats["single_s"], "rank_candidates_ms": 1000 * stats["rank_s"] / steps,
           "load_cluster_ms": 1000 * stats["open_s"] / steps, "sharding": f"probes one per GPU over {world} GPU(s), one ncclAllGather of verdicts per round",
           "result": last}
    g = ROOT / "tests" / "golden" / "fullsize" / "c5.json"
    if g.exists():
        gold = json.loads(g.read_text())
        m = gold["multi_node"]
        seq = [c for c in m["probes"]]
        out["parity_vs_oracle"] = bool(last["action"] == m["action"] and last["nodes_removed"] == m["nodes_removed"] and last["n_options"] == len(m["options"]) and
                                       last["probes_on_path"] == seq)
        out["oracle_seconds_same_search_1_core"] = gold["oracle_seconds_multi_node"]
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", type=int, default=4, choices=sorted(CONFIGS))
    ap.add_argument("--pods", type=int, default=0)
    ap.add_argument("--types", type=int, default=0)
    ap.add_argument("--no-cpu-baseline", action="store_true", help="skip the CPU legs and the secondary configurations (profiling runs)")
    ap.add_argument("--no-c5", action="store_true", help="skip the consolidation block (config_c5)")
    ap.add_argument("--dump-outputs", metavar="DIR", type=Path,
                    help="write the Result of the last timed Solve (rank 0) as DIR/<name>.npy (see dump_outputs)")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1 and "KSCHED_HOST_THREADS" not in os.environ:
        # the host encoder / decoder split their per-pod and per-node passes over the cores: N replicas share the box
        os.environ["KSCHED_HOST_THREADS"] = str(max(2, min(16, (os.cpu_count() or 16) // world)))

    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    from __graft_entry__ import load_pkg
    pkg = load_pkg()
    if not torch.cuda.is_available() or pkg.device_count() < 1:
        raise RuntimeError("bench.py needs a CUDA device: the solver has no CPU path")
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    L = pkg.lib()
    L.kh_set_device(local_rank)

    cfg, pods, types = workload_config(args)
    seed = 42 + rank  # replicas: every rank solves its own batch of the same shape
    problem = pkg.Problem.synth(args.config, pods, types, seed, cfg["nodes"])
    t0 = time.perf_counter()
    rs = pkg.ResidentSolve(problem)
    encode_s = time.perf_counter() - t0
    t0 = time.perf_counter()
    rs.load_catalog()
    catalog_s = time.perf_counter() - t0
    rs.set_count_visited(False)
    rs.load()

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if dist is None:
            return x
        tt = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        return float(tt.item())

    def sum_over_ranks(x):
        if dist is None:
            return x
        tt = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(tt, op=dist.ReduceOp.SUM)
        return float(tt.item())

    # ---- value: resident problem, kernels only
    sampler = ClockSampler(local_rank)
    sampler.start()  # nvidia-smi is up and sampling by the time the warm-ups are done
    for _ in range(args.warmup):
        rs.run(flush_l2=True)
    barrier()
    sampler.mark()
    phase = {"sort_us": 0.0, "feasibility_us": 0.0, "pack_us": 0.0, "allreduce_us": 0.0, "total_us": 0.0}
    wall0 = time.perf_counter()
    for _ in range(args.steps):
        rs.run(flush_l2=True)
        t = rs.timings()
        for k in phase:
            phase[k] += t[k]
    barrier()
    wall = time.perf_counter() - wall0
    clocks = sampler.stop()
    dev_s = max_over_ranks(phase["total_us"] * 1e-6)
    res = rs.download()
    scheduled = int((res.assign >= 0).sum())
    tm = rs.timings()
    all_scheduled = sum_over_ranks(float(scheduled))
    value = all_scheduled * args.steps / dev_s

    # ---- e2e: string-level model -> encode -> ksched_solve (upload, kernels, download) -> decode
    for _ in range(2):
        pkg.solve_timed(problem)
    barrier()
    e2e_ph = {"encode_us": 0.0, "catalog_us": 0.0, "solve_us": 0.0, "decode_us": 0.0, "total_us": 0.0}
    for _ in range(args.steps):
        r2, t = pkg.solve_timed(problem)
        for k in e2e_ph:
            e2e_ph[k] += t[k]
    barrier()
    tm_e2e = rs.timings()  # the handle's counters of the last ksched_solve
    e2e_s = max_over_ranks(e2e_ph["total_us"] * 1e-6)
    e2e_value = all_scheduled * args.steps / e2e_s
    e2e_same = bool(int(r2.digest()) == int(res.digest()))
    # ksched_solve alone (flat structs in and out)
    rs.solve_e2e()
    so_us = 0.0
    for _ in range(args.steps):
        us, _ = rs.solve_e2e()
        so_us += us
    barrier()
    so_s = max_over_ranks(so_us * 1e-6)

    # ---- feasibility kernel alone, cold L2, CUDA events on the launching stream
    rs.load()
    rs.run(flush_l2=False)
    k1_us = sorted(rs.run_feasibility(flush_l2=True) for _ in range(max(8, args.steps)))
    k1_avg = sum(k1_us) / len(k1_us)
    peak, peak_src = measured_peak()
    k1_bytes = tm["feasibility_bytes"]
    k1_gbs = k1_bytes / (k1_avg * 1e-6) / 1e9
    d = rs.dims
    gold = golden(args.config, pods, types, seed)
    if gold:
        nodes_visited = int(gold["nodes_visited"])  # the oracle emits the same statistic (SURVEY 8d K2)
    else:
        rs.set_count_visited(True)
        rs.load()
        rs.run()
        nodes_visited = int(rs.download().nodes_visited)
        rs.set_count_visited(False)
        rs.load()
    pack_avg_us = phase["pack_us"] / args.steps
    pack_bytes = nodes_visited * 128 + d["pods"] * 256
    pack_gbs = pack_bytes / (pack_avg_us * 1e-6) / 1e9

    details = {"scheduled": scheduled, "new_nodes": int(res.num_new_nodes), "seed": seed,
               "l2": "flushed before every timed step (256 MiB write)",
               "parallelism": "1 Solve per GPU" + (f", {world} independent replicas (seed 42 + rank), no data-path collective" if world > 1 else ""),
               "phases_ms_per_step": {k[:-3]: v / args.steps / 1000 for k, v in phase.items()},
               "encode_host_ms": 1000 * encode_s, "catalog_load_ms": 1000 * catalog_s, "wall_ms_per_step": 1000 * wall / args.steps,
               "library_kernels_per_step": "1x cub::DeviceRadixSort::SortPairs over the packed key's significant bits (3 cub kernels, not counted in gpu_launches)",
               "host_threads": os.environ.get("KSCHED_HOST_THREADS", "default (up to 16)"),
               "limiter": "pack_kernel: one CTA, a sequential first-fit chain over the pods; closed-form steps (level / fill / bulk fresh nodes / "
                          "rounds of the mask run) place several pods per iteration (DESIGN.md section 4)"}
    line = {
        "metric": "pods scheduled/sec (Scheduler.Solve)", "value": value, "unit": "pods/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1000 * dev_s / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "int64", "data": "synthetic",
        "config": public_config(cfg, pods, types),
        "details": details,
        "e2e": {"value": e2e_value, "unit": "pods/s", "h2d_bytes_per_step": int(tm_e2e["h2d_bytes"]), "d2h_bytes_per_step": int(tm_e2e["d2h_bytes"]),
                "ms_per_step": 1000 * e2e_s / args.steps,
                "path": "kh_scheduler_solve_timed: string-level model -> khost::encode -> ksched_solve(handle, problem*, result*) with host buffers -> decode",
                "phases_ms_per_step": {k[:-3]: v / args.steps / 1000 for k, v in e2e_ph.items()},
                "same_result_as_resident_run": e2e_same,
                "solve_only": {"value": all_scheduled * args.steps / so_s, "unit": "pods/s", "ms_per_step": 1000 * so_s / args.steps,
                               "path": "ksched_solve(handle, problem*, result*) with host buffers (flat structs in and out)"}},
        # own kernels per resident Solve: reset_kernel, sort_key1, gather_rows, class_feasibility, feasibility, pack, finalize_options
        # (profiles/r02b_launch_shares.txt)
        "gpu_launches": 7 * args.steps,
        "roofline": {"kernel": "pack_kernel", "bound": "hbm", "achieved": pack_gbs, "peak": peak, "unit": "GB/s", "frac": pack_gbs / peak,
                     "traffic": ncu_traffic(f"pack_kernel_c{args.config}"), "peak_source": peak_src, "algorithmic_bytes": int(pack_bytes),
                     "us_per_launch": pack_avg_us,
                     "note": "latency-bound sequential first-fit chain; bytes = nodes_visited*128 + P*256 (SURVEY 8d K2) with the reference's "
                             "nodes_visited (it also walks full nodes; the kernel keeps them out of its active set)"},
        "roofline_feasibility": {"kernel": "feasibility_kernel", "bound": "hbm", "achieved": k1_gbs, "peak": peak, "unit": "GB/s", "frac": k1_gbs / peak,
                                 "traffic": ncu_traffic(f"feasibility_kernel_c{args.config}"), "peak_source": peak_src, "algorithmic_bytes": int(k1_bytes),
                                 "us_per_launch": k1_avg, "us_min": k1_us[0],
                                 "physical_bytes": int(d["pods"] * 32 + d["pods"] * d["templates"] * d["type_words"] * 8 + d["pods"] * 8),
                                 "class_pass_us": rs.timings()["class_feasibility_us"],
                                 "note": "bytes = P*256 + C*256 + P*C/8 (SURVEY 8d K1), cold L2, this workload's shape. Pods of one class share "
                                         "their row: class_feasibility_kernel evaluates the n_classes distinct rows, this kernel streams the dense "
                                         "matrix (physical: one 32-byte sector of every pod row + the matrix + the best vector)"},
        "clocks": clocks,
    }
    if not args.no_c5:
        rs = None  # the handle now serves the consolidation pass
        line["config_c5"] = c5_block(pkg, torch, dist, rank, world, 2)
    if rank == 0:
        if gold:
            details["parity_vs_oracle"] = bool(int(res.digest()) == gold["digest"])
            details["parity_source"] = "whole-result digest of the committed full-size oracle run (tests/golden/fullsize); the oracle is the C++ " \
                                       "restatement of the Go algorithm under canonical rules R1-R6 (DESIGN.md section 6), the Go reference itself cannot run here"
        if world == 1 and not args.no_cpu_baseline:
            import oracle_lib
            oracle = oracle_lib.load()
            sample = min(pods, CPU_SAMPLE[args.config])
            sp = problem if sample == pods else pkg.Problem.synth(args.config, sample, types, 42, cfg["nodes"])
            want = pkg.Result()
            t0 = time.perf_counter()
            oracle.solve(sp, want)
            cpu_s = time.perf_counter() - t0
            cpu_sched = int((want.assign >= 0).sum())
            line["cpu_baseline"] = {"value": cpu_sched / cpu_s, "unit": "pods/s", "cores": 1, "kind": "port",
                                    "sample": f"literal oracle Solve of a {sample}-pod batch of the same generator x {types} instance types, 1 run, "
                                              f"{cpu_s:.2f} s, 1 thread of {os.cpu_count()} (over-states the reference at {pods} pods: its per-pod cost grows with the batch)"}
            if sample == pods and not gold:
                details["parity_vs_oracle"] = bool((want.assign == res.assign).all() and want.num_new_nodes == res.num_new_nodes)
            for c in (2, 3):
                if c != args.config:
                    line[f"config_c{c}"] = secondary(pkg, c)
        if args.dump_outputs:
            dump_outputs(problem, res, args.dump_outputs)
        print(json.dumps(line), flush=True)
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
