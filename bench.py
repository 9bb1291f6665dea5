#!/usr/bin/env python
"""bench.py -- FK + end-effector Jacobian throughput of the Kuka iiwa 7-DoF (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

One *step* = one pass of the hot path (one `drmb200_fk_jacobian` launch: pos, quat, J_lin, J_ang
of `iiwa_link_ee`) over one batch of 65 536 synthetic joint configurations (BASELINE.json
configs[1]).  Inputs are resident in HBM before the timed region; the step cycles through ROTATE
distinct buffer sets (> the 126 MB L2) so no launch finds its data in L2.

Launch pattern of the headline number: the K launches are replayed from a CUDA graph (the per-launch
Python/ctypes overhead would otherwise exceed the ~3 us kernel) as four independent chains (graph
branches; the batches are independent), each chain stream-ordered with programmatic dependent launch
enabled in the library (`fk_pdl` = 2, include/drm_b200.h): a launch may start its loads and arithmetic
while its predecessor is still storing and waits for it before its own first global write.
`launch_modes` reports, per launch: ONE stream with PDL, one stream without any overlap (what a single
isolated call costs on the device), four branches without PDL (round 1), four branches with PDL.

Timing: the timed region of K steps is repeated REPS times; every repetition is bracketed by a barrier
+ synchronize on both sides and timed with CUDA events on the launching stream, with a GPU-side delay
queued ahead of the first event so that the graph launch is already enqueued when the clock starts
(the region measures the device, not the host's launch latency).  Each rank reports the MEDIAN of its
repetitions, the job reports the MAX over ranks.

Extra keys on the JSON line (see DESIGN.md "Measurement"):
  roofline            dominant kernel vs the measured HBM copy bandwidth (MEASURED_PEAKS.json)
  roofline_large_batch  the same kernel on 2^22 configurations per launch (the asymptotic figure)
  launch_modes        us per launch: one stream + PDL, one stream, 4 graph branches, 4 branches + PDL (the headline)
  e2e                 same metric through the host-buffer C-ABI call (H2D + kernel + D2H per step)
  cpu_baseline        the UNMODIFIED reference (baseline/_ref) on the host cores, bounded sample
  cpu_baseline_port   the vectorised torch CPU port of the same algorithm (oracle/drm_oracle.py)
  clocks              nvidia-smi SM clocks / throttle reasons sampled during the timed regions

`--dump-outputs DIR` writes what the last timed step computed on rank 0 -- pos, quat, J_lin, J_ang of its 65 536
configurations -- as DIR/<name>.npy (float32, 12.8 MB).  The inputs are seeded, so two builds run with the same
arguments can be compared output for output.

`--impl reference` times the reference's own CPU implementation through its public API
(`DifferentiableRobotModel.compute_endeffector_jacobian`, unmodified, installed into baseline/_ref by
`__graft_entry__.build()`; its third-party XML-parser dependency is replaced by oracle/refshim) --
rank 0 only.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np
import torch

REPO = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, REPO)

BATCH = 65536                 # BASELINE.json configs[1]
EE_LINK = "iiwa_link_ee"
N_DOF = 7
BYTES_PER_CONFIG = 28 * N_DOF + 28      # 4n (q) + 12 (pos) + 16 (quat) + 24n (J_lin, J_ang) = 224
ROTATE = 16                   # 16 x 14.7 MB = 235 MB of distinct buffers > 126 MB L2
GRAPH_NODES = 512
REPS = 11
METRIC = "FK+Jacobian configs/sec (Kuka iiwa 7-DoF)"
UNIT = "configs/s"
REF_DIR = os.path.join(REPO, "baseline", "_ref")
REF_SHIM = os.path.join(REPO, "oracle", "refshim")     # stand-in for the reference's urdf_parser_py dependency


def bench_config(n_gpus):
    """Identical for both arms: what is computed, not how it is launched."""
    return {"workload": "Kuka iiwa 7-DoF FK + end-effector Jacobian, batch 65536 per step per GPU "
                        "(BASELINE.json configs[1])",
            "urdf": "kuka_iiwa/urdf/iiwa7.urdf", "ee_link": EE_LINK, "batch_per_step_per_gpu": BATCH,
            "global_batch_per_step": BATCH * n_gpus,
            "parallelism": f"batch-sharded x{n_gpus}, no data-path collective",
            "inputs": "q ~ U(joint limits), seeded per rank",
            "l2_policy": f"GPU arm: inputs / outputs rotate over {ROTATE} distinct buffer sets "
                         f"({ROTATE * BATCH * BYTES_PER_CONFIG / 1e6:.0f} MB) > the 126 MB L2, no launch finds its data in L2"}


def measured_peak_gbs():
    path = os.path.join(REPO, "MEASURED_PEAKS.json")
    try:
        with open(path) as fh:
            return float(json.load(fh)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def sample_q(limits, batch, seed):
    """q ~ U(lower, upper) per joint; `limits` = model.get_joint_limits()."""
    gen = torch.Generator().manual_seed(seed)
    lo = torch.tensor([float(l["lower"]) for l in limits], dtype=torch.float64)
    hi = torch.tensor([float(l["upper"]) for l in limits], dtype=torch.float64)
    return (lo + (hi - lo) * torch.rand(batch, len(limits), generator=gen, dtype=torch.float64)).to(torch.float32)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons every 100 ms while the timed regions run."""
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.rows, self.proc, self.thread, self.t0, self.t1 = [], None, None, None, None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={gpu_index}", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits",
                 "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def mark_start(self):
        self.t0 = time.time()

    def mark_end(self):
        self.t1 = time.time()

    def summary(self):
        if self.proc is not None:
            time.sleep(0.15)
            self.proc.terminate()
        parsed = []
        for ts, line in self.rows:
            parts = [p.strip() for p in line.split(",")]
            if len(parts) < 7:
                continue
            try:
                parsed.append((ts, float(parts[0]), float(parts[1]), parts[3:7]))
            except ValueError:
                continue
        if not parsed:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0, "note": "nvidia-smi unavailable"}
        inside = [p for p in parsed if self.t0 is not None and self.t0 <= p[0] <= (self.t1 or 1e30) + 0.1]
        use = inside if inside else parsed
        clocks = sorted(p[1] for p in use)
        names = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")
        reasons = sorted({names[i] for p in use for i in range(4) if p[3][i].lower().startswith("active")})
        return {"sm_mhz": clocks[len(clocks) // 2], "sm_max_mhz": max(p[2] for p in use), "reasons": reasons,
                "samples": len(use), "window": "timed regions" if inside else "whole run (timed regions < sampling period)"}


# ------------------------------------------------------------------------------------------------
# CPU arms: the unmodified reference (baseline/_ref) and the vectorised port (oracle/)
# ------------------------------------------------------------------------------------------------
_REF_MODEL = None


def reference_model():
    """The reference's own DifferentiableKUKAiiwa on the CPU, imported from baseline/_ref (None if not installed)."""
    global _REF_MODEL
    if _REF_MODEL is None:
        if not os.path.isdir(os.path.join(REF_DIR, "differentiable_robot_model")):
            _REF_MODEL = False
        else:
            for p in (REF_SHIM, REF_DIR):
                if p not in sys.path:
                    sys.path.insert(0, p)
            from differentiable_robot_model.robot_model import DifferentiableKUKAiiwa as RefKuka
            _REF_MODEL = RefKuka()
    return _REF_MODEL or None


def _reference_call(model, q):
    with torch.no_grad():
        return model.compute_endeffector_jacobian(q, EE_LINK)     # computes pos / quat on the way (robot_model.py:641)


def _port_call(robot, q):
    from oracle import drm_oracle as O
    with torch.no_grad():
        R, p, _, _, _ = O.kinematic_state(robot, q)
        e = robot.index(EE_LINK)
        quat = O.quaternion(R[e])
        lin, ang = O.jacobian(robot, q, EE_LINK)
    return p[e], quat, lin, ang


def pick_threads(call, q):
    """Both CPU arms issue thousands of small torch ops; one intra-op thread per core is rarely the fastest
    setting on a many-core host.  Probe a few thread counts once and keep the fastest ('all the host threads it
    can use')."""
    cores = os.cpu_count() or 1
    best = (torch.get_num_threads(), float("inf"))
    for nt in sorted({1, 4, 8, 16, 32, cores}):
        if nt > cores:
            continue
        torch.set_num_threads(nt)
        call(q)
        t0 = time.perf_counter()
        call(q)
        dt = time.perf_counter() - t0
        if dt < best[1]:
            best = (nt, dt)
    torch.set_num_threads(best[0])
    return best[0]


def cpu_arm(kind):
    """(call, limits, description) of a CPU implementation: 'reference' = baseline/_ref, 'port' = oracle/drm_oracle.py."""
    import differentiable_robot_model_b200 as drm
    ours = drm.DifferentiableKUKAiiwa(device="cpu")          # host-side model only: joint limits + URDF path
    limits = ours.get_joint_limits()
    if kind == "reference":
        model = reference_model()
        if model is None:
            return None, limits, None
        return (lambda q: _reference_call(model, q)), limits, \
            "the UNMODIFIED reference (baseline/_ref, DifferentiableKUKAiiwa.compute_endeffector_jacobian, torch CPU fp32, " \
            "per-element Python quaternion loop as shipped)"
    from oracle import drm_oracle as O
    robot = O.load_robot(ours.urdf_path, torch.float32)
    return (lambda q: _port_call(robot, q)), limits, \
        "oracle/drm_oracle.py (torch CPU port of the reference's per-link algorithm, fp32, vectorised quaternion)"


def time_cpu(call, q, n_calls, warmup=1):
    for _ in range(warmup):
        call(q)
    times = []
    for _ in range(n_calls):
        t0 = time.perf_counter()
        call(q)
        times.append(time.perf_counter() - t0)
    return times


def bounded_sample(call, limits, budget_s, n_calls, max_batch=BATCH):
    """Batch per call such that n_calls calls cost about budget_s: one call costs t0 + c * batch (fit from two probes)."""
    lo = min(time_cpu(call, sample_q(limits, 64, 1), 2, warmup=1))
    hi = min(time_cpu(call, sample_q(limits, 1024, 2), 2, warmup=0))
    c = max((hi - lo) / (1024 - 64), 1e-9)
    t0 = max(lo - 64 * c, 0.0)
    per_call = budget_s / max(1, n_calls)
    return int(max(64, min(max_batch, (per_call - t0) / c)))


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    if args.steps is None:
        args.steps = 20
    kind = "reference"
    call, limits, what = cpu_arm("reference")
    if call is None:                                         # baseline/_ref missing: the port is the stand-in, and says so
        kind = "port"
        call, limits, what = cpu_arm("port")
    cores = pick_threads(call, sample_q(limits, 512, 3))
    warm = max(1, min(args.warmup, 3))
    batch = bounded_sample(call, limits, 90.0, args.steps + warm)
    q = sample_q(limits, batch, 0)
    times = time_cpu(call, q, args.steps, warmup=warm)
    total = sum(times)
    value = batch * len(times) / total
    sample = (f"{len(times)} steps x {batch} Kuka FK+Jacobian configurations (a bounded sample of the 65536-configuration "
              f"step) through {what}; {cores} intra-op threads (fastest of the probed counts on this {os.cpu_count()}-core host)")
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": len(times), "warmup": args.warmup, "ms_per_step": 1e3 * total / len(times),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": bench_config(args.gpus),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }))


# ------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None, help="default 20000 (GPU arm) / 20 (--impl reference)")
    ap.add_argument("--warmup", type=int, default=2000)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--reps", type=int, default=REPS, help="repetitions of the timed K-step region (median reported)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-large", action="store_true")
    ap.add_argument("--no-modes", action="store_true")
    ap.add_argument("--no-sharded", action="store_true", help="skip the sharded BASELINE configs 4 and 5 (scripts/bench_sharded.py)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the last timed step's outputs (rank 0) as DIR/{pos,quat,jac_lin,jac_ang}.npy, float32")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3)
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the GPU arm's outputs; it does not apply to --impl reference")

    if args.impl == "reference":
        run_reference_arm(args)
        return
    if args.steps is None:
        args.steps = 20000
    args.steps = max(args.steps, 1)
    args.reps = max(args.reps, 1)

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    assert world == args.gpus or world == 1, f"--gpus {args.gpus} but WORLD_SIZE={world}"

    # one process per GPU: run this rank's host thread (graph launches, event records) and its page-locked buffers on
    # the NUMA node of its GPU -- before CUDA is initialised and before anything is timed
    numa_bound = False
    if world > 1 and os.environ.get("DRMB200_BENCH_NUMA_BIND", "1") != "0":
        from differentiable_robot_model_b200.parallel import bind_to_device_numa_node
        visible = os.environ.get("CUDA_VISIBLE_DEVICES")
        phys = int(visible.split(",")[local_rank]) if visible and visible.split(",")[local_rank].isdigit() else local_rank
        numa_bound = bind_to_device_numa_node(phys)

    import torch.distributed as dist
    import differentiable_robot_model_b200 as drm
    from differentiable_robot_model_b200 import engine, parallel

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    model = drm.DifferentiableKUKAiiwa(device=dev)
    table = model._link_table()
    if world > 1:
        table = parallel.broadcast_link_table(model)        # the single NCCL broadcast of the data path
    topo, ee = model._topology, model._name_to_idx_map[EE_LINK]
    limits = model.get_joint_limits()

    # ---- synthetic inputs, per-rank seed, resident in HBM ------------------------------------------
    qs, outs = [], []
    for r in range(ROTATE):
        qs.append(sample_q(limits, BATCH, seed=1000 * rank + r).to(dev))
        outs.append((torch.empty(BATCH, 3, device=dev), torch.empty(BATCH, 4, device=dev),
                     torch.empty(BATCH, 3, N_DOF, device=dev), torch.empty(BATCH, 3, N_DOF, device=dev)))

    def step(i):
        engine.fk_jacobian_raw(topo, ee, table, qs[i % ROTATE], out=outs[i % ROTATE])

    stream = torch.cuda.Stream(device=dev)
    sampler = ClockSampler(local_rank) if rank == 0 else None
    side = [torch.cuda.Stream(device=dev) for _ in range(3)]
    spin_cycles = 600_000                                     # ~0.3 ms GPU-side delay ahead of the first event

    def barrier():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def capture(n_nodes, first, branches):
        """n_nodes kernel nodes; branches == 1: one stream-ordered chain, else `branches` parallel chains."""
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=stream):
            if branches > 1:
                fork = torch.cuda.Event()
                fork.record(stream)
                for s in side[:branches - 1]:
                    s.wait_event(fork)
            for i in range(first, first + n_nodes):
                lane = i % branches
                if lane == 0:
                    step(i)
                else:
                    with torch.cuda.stream(side[lane - 1]):
                        step(i)
            if branches > 1:
                for s in side[:branches - 1]:
                    join = torch.cuda.Event()
                    join.record(s)
                    stream.wait_event(join)
        return g

    def timed_regions(steps, reps, pdl, branches, warm_replays):
        """[ms per K-step region] * reps on this rank, and the launch description."""
        engine.set_option("fk_pdl", pdl)
        nodes = max(1, min(GRAPH_NODES, steps))
        graph = capture(nodes, 0, branches)
        replays, rest = divmod(steps, nodes)
        tail_graph = capture(rest, replays * nodes, branches) if rest else None      # the remainder is graph-launched too
        for _ in range(warm_replays):
            graph.replay()
        if tail_graph is not None:
            tail_graph.replay()
        stream.synchronize()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        out = []
        host_launches = engine.launch_count()
        for _ in range(reps):
            barrier()
            torch.cuda._sleep(spin_cycles)                   # on `stream`: the launches below queue up behind it
            ev0.record(stream)
            for _ in range(replays):
                graph.replay()
            if tail_graph is not None:
                tail_graph.replay()
            ev1.record(stream)
            stream.synchronize()
            barrier()
            out.append(ev0.elapsed_time(ev1))
        assert engine.launch_count() == host_launches, "timed launches must all be graph replays"
        desc = (f"CUDA graph of {nodes} kernel nodes, " +
                ("one stream-ordered chain" if branches == 1 else f"{branches} parallel branches (independent batches in flight)") +
                (" with programmatic dependent launch (fk_pdl 2: a launch overlaps its predecessor up to its first global write)"
                 if pdl == 2 else "") + f", replayed {replays}x + one {rest}-node tail graph")
        del graph, tail_graph
        return out, desc

    def job_ms(per_rank_ms):
        """median over this rank's repetitions, MAX over ranks"""
        t = torch.tensor([statistics.median(per_rank_ms)], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    with torch.cuda.stream(stream):
        engine.set_option("fk_pdl", 2)
        for i in range(min(args.warmup, 64)):
            step(i)
        stream.synchronize()
        warm_replays = max(1, (args.warmup - 64) // max(1, min(GRAPH_NODES, args.steps)))
        if sampler:
            sampler.mark_start()
        # headline pattern: 4 independent chains of launches (graph branches), each chain stream-ordered with programmatic
        # dependent launch -- the batches are independent, and a 20-step region amortises the first launch's latency best
        # that way (63 us against 65.5 us for one chain); one chain alone is reported in `launch_modes`
        head_branches = max(1, min(4, int(os.environ.get("DRMB200_BENCH_BRANCHES", "4"))))
        region_ms, launch_desc = timed_regions(args.steps, args.reps, pdl=2, branches=head_branches, warm_replays=warm_replays)
        if sampler:
            sampler.mark_end()
        elapsed_ms = job_ms(region_ms)
        dumped = None
        if args.dump_outputs and rank == 0:                  # copied now: the sections below reuse these buffers
            dumped = {name: t.cpu().numpy() for name, t in
                      zip(("pos", "quat", "jac_lin", "jac_ang"), outs[(args.steps - 1) % ROTATE])}

        modes = None
        if not args.no_modes:
            k = 2048                                        # enough launches that the ramp of the first one is amortised
            r = min(args.reps, 7)
            modes = {"steps_per_region": k, "reps": r,
                     "stream_ordered_pdl_us": job_ms(timed_regions(k, r, 2, 1, 1)[0]) * 1e3 / k,
                     "stream_ordered_us": job_ms(timed_regions(k, r, 0, 1, 1)[0]) * 1e3 / k,
                     "branches4_us": job_ms(timed_regions(k, r, 0, 4, 1)[0]) * 1e3 / k,
                     "branches4_pdl_us": job_ms(timed_regions(k, r, 2, 4, 1)[0]) * 1e3 / k,
                     "note": "us per 65536-configuration launch (median of reps, max over ranks): ONE stream with programmatic "
                             "dependent launch (fk_pdl 2) / one stream, nothing overlapping = what a single isolated call costs "
                             "on the device / four graph branches (round 1's pattern) / four branches with PDL (the headline)"}
        engine.set_option("fk_pdl", 2)

    gpu_launches = args.steps                                    # fk_jacobian_kernel launches inside ONE timed region
    value = world * args.steps * BATCH / (elapsed_ms * 1e-3)
    peak, peak_src = measured_peak_gbs()
    us_per_launch = elapsed_ms * 1e3 / args.steps
    achieved = BATCH * BYTES_PER_CONFIG / (us_per_launch * 1e-6) / 1e9

    result = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": elapsed_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": bench_config(world),
        "launch": launch_desc,
        "l2_policy": f"rotating {ROTATE} distinct buffer sets ({ROTATE * BATCH * BYTES_PER_CONFIG / 1e6:.0f} MB) > L2",
        "timing": {"reps": args.reps, "region_ms_this_rank": [round(x, 5) for x in region_ms],
                   "statistic": "median over repetitions per rank, max over ranks; CUDA events on the launching stream, "
                                "GPU-side delay queued ahead of the first event, barrier + synchronize around every repetition",
                   "numa_bound": numa_bound},
        "gpu_launches": gpu_launches,
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": None, "peak_source": peak_src, "kernel": "fk_jacobian_kernel<7, 64, WITH_JAC, packed> (TMA bulk staging)",
                     "algorithmic_bytes_per_launch": BATCH * BYTES_PER_CONFIG, "us_per_launch": us_per_launch},
    }
    if modes is not None:
        result["launch_modes"] = modes

    if rank == 0:
        prof = os.path.join(REPO, "profiles", "fk_jacobian_traffic.json")
        if os.path.exists(prof):
            try:
                result["roofline"]["traffic"] = json.load(open(prof)).get("dram_bytes_per_launch_batch65536")
            except Exception:
                pass

    # ---- asymptotic figure: 2^22 configurations per launch -----------------------------------------
    if not args.no_large and rank == 0:
        big = 1 << 22
        del outs
        torch.cuda.empty_cache()
        q_big = torch.cat([qs[i % ROTATE] for i in range(big // BATCH)])
        out_big = (torch.empty(big, 3, device=dev), torch.empty(big, 4, device=dev),
                   torch.empty(big, 3, N_DOF, device=dev), torch.empty(big, 3, N_DOF, device=dev))
        engine.set_option("fk_pdl", 0)
        with torch.cuda.stream(stream):
            for _ in range(3):
                engine.fk_jacobian_raw(topo, ee, table, q_big, out=out_big)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            stream.synchronize()
            reps = 20
            e0.record(stream)
            for _ in range(reps):
                engine.fk_jacobian_raw(topo, ee, table, q_big, out=out_big)
            e1.record(stream)
            stream.synchronize()
        ms = e0.elapsed_time(e1) / reps
        ach = big * BYTES_PER_CONFIG / (ms * 1e-3) / 1e9
        result["roofline_large_batch"] = {"batch_per_launch": big, "bytes_per_launch": big * BYTES_PER_CONFIG,
                                          "ms_per_launch": ms, "configs_per_s": big / (ms * 1e-3), "achieved": ach,
                                          "peak": peak, "unit": "GB/s", "frac": ach / peak,
                                          "l2_policy": "0.94 GB per launch >> L2", "launch": "plain stream-ordered launches, no PDL"}
        del q_big, out_big
        torch.cuda.empty_cache()
        engine.set_option("fk_pdl", 2)

    # ---- the sharded BASELINE configs (4: Allegro fingertips, 5: Kuka training step) on this rank's shard --------
    if not args.no_sharded:
        try:
            sys.path.insert(0, os.path.join(REPO, "scripts"))
            import bench_sharded
            peak_gbs = peak
            c4 = bench_sharded.config4(dev, rank, barrier)
            c5 = bench_sharded.config5(dev, rank, world, dist if world > 1 else None, barrier)
            t4f, t4p, t5 = (job_ms([c4["fused_ms_per_step"]]), job_ms([c4["per_tip_ms_per_step"]]), job_ms([c5["ms_per_step"]]))
            b4, b5 = c4["per_gpu_batch"], c5["per_gpu_batch"]
            result["sharded_configs"] = {
                "config4_allegro_fk_jac_4_fingertips": {
                    "global_batch": b4 * world, "per_gpu_batch": b4, "fused_launch_ms_per_step": t4f,
                    "fused_configs_per_s": world * b4 / (t4f * 1e-3),
                    "fused_hbm_frac_per_gpu": b4 * c4["algorithmic_bytes_per_config"] / (t4f * 1e-3) / 1e9 / peak_gbs,
                    "four_single_tip_launches_ms_per_step": t4p, "four_single_tip_configs_per_s": world * b4 / (t4p * 1e-3),
                    "collective": "none (batch-sharded)"},
                "config5_kuka_fk_jac_rnea_backward_adam": {
                    "global_batch": b5 * world, "per_gpu_batch": b5, "ms_per_step": t5, "configs_per_s": world * b5 / (t5 * 1e-3),
                    "allreduce_scalars_per_step": c5["allreduce_scalars"], "step": c5["step"], "final_loss_rank0": c5["final_loss"],
                    "ms_per_step_with_nccl_allreduce_and_torch_adam_this_rank": c5["ms_per_step_nccl_allreduce_torch_adam"]},
                "timing": "median over repetitions per rank, max over ranks; weak scaling (fixed per-GPU shard)"}
            if world == 1:                                   # BASELINE config 3 is a single-GPU config
                c3 = bench_sharded.config3(dev, barrier)
                result["sharded_configs"]["config3_panda_inverse_dynamics_single_gpu"] = c3
        except Exception as exc:                              # report, do not hide
            result["sharded_configs"] = {"error": f"{type(exc).__name__}: {exc}"}

    # ---- end to end through the host-buffer C-ABI call ---------------------------------------------
    if not args.no_e2e:
        e2e_steps = max(3, min(args.steps, 200))
        q_host = [qs[i].cpu().pin_memory() for i in range(2)]
        host_out = [(torch.empty(BATCH, 3).pin_memory(), torch.empty(BATCH, 4).pin_memory(),
                     torch.empty(BATCH, 3, N_DOF).pin_memory(), torch.empty(BATCH, 3, N_DOF).pin_memory())
                    for _ in range(2)]
        torch.cuda.synchronize(dev)
        for i in range(3):
            engine.fk_jacobian_host(topo, ee, local_rank, table, q_host[i % 2], *host_out[i % 2])
        e2e_ms = []
        for _ in range(min(args.reps, 5)):
            if world > 1:
                dist.barrier()
            torch.cuda.synchronize(dev)
            t0 = time.perf_counter()
            for i in range(e2e_steps):
                engine.fk_jacobian_host(topo, ee, local_rank, table, q_host[i % 2], *host_out[i % 2])
            torch.cuda.synchronize(dev)
            e2e_ms.append((time.perf_counter() - t0) * 1e3)
        dt = job_ms(e2e_ms) * 1e-3
        result["e2e"] = {"value": world * e2e_steps * BATCH / dt, "unit": UNIT,
                         "h2d_bytes_per_step": BATCH * 4 * N_DOF, "d2h_bytes_per_step": BATCH * (28 + 24 * N_DOF),
                         "steps": e2e_steps, "reps": len(e2e_ms),
                         "api": "drmb200_fk_jacobian_host (pinned host buffers in and out)",
                         "numa_bound": numa_bound,
                         "transfer": "fused: one launch per step, the kernel's TMA bulk copies read q from and write all "
                                     "outputs to the pinned HOST buffers over PCIe (no staging copies); the bytes below "
                                     "cross PCIe inside the timed region every step",
                         "timing": "host wall clock around the blocking calls (they return after the last D2H); median over "
                                   "repetitions per rank, max over ranks"}

    if rank == 0:
        result["clocks"] = sampler.summary()
        if not args.no_cpu_baseline and world == 1:         # reported at N = 1 only
            for kind, key, budget in (("reference", "cpu_baseline", 15.0), ("port", "cpu_baseline_port", 8.0)):
                try:
                    call, lim, what = cpu_arm(kind)
                    if call is None:
                        continue
                    cores = pick_threads(call, sample_q(lim, 512 if kind == "reference" else 8192, 3))
                    n_calls = 5
                    b = bounded_sample(call, lim, budget, n_calls)
                    times = time_cpu(call, sample_q(lim, b, 0), n_calls)
                    result[key] = {"value": b * len(times) / sum(times), "unit": UNIT, "cores": cores, "kind": kind,
                                   "sample": f"{len(times)} calls x {b} configurations of the same workload through {what}; "
                                             f"{cores} intra-op threads (fastest probed on this {os.cpu_count()}-core host), "
                                             f"{sum(times):.1f} s"}
                except Exception as exc:
                    result[key] = {"error": f"{type(exc).__name__}: {exc}"}
            if "cpu_baseline" not in result and "cpu_baseline_port" in result:
                result["cpu_baseline"] = result["cpu_baseline_port"]
            # context: the scalar C restatement of the same algorithm on all cores (oracle/drm_oracle.c)
            try:
                from oracle.c_oracle import CRobot
                from oracle import drm_oracle as O2
                rb = O2.load_robot(model.urdf_path, torch.float32)
                cq = sample_q(limits, 1 << 20, 0)
                cr = CRobot(rb)
                cr.fk_jacobian(rb.index(EE_LINK), cq.numpy())
                t0 = time.perf_counter()
                cr.fk_jacobian(rb.index(EE_LINK), cq.numpy())
                result["cpu_baseline_c_port"] = {
                    "value": (1 << 20) / (time.perf_counter() - t0), "unit": UNIT, "cores": os.cpu_count(),
                    "kind": "port", "sample": "2^20 configurations through oracle/drm_oracle.c (scalar C, one pthread per core)"}
            except Exception as exc:      # the C oracle is optional context
                result["cpu_baseline_c_port"] = {"error": str(exc)}
        if dumped is not None:
            os.makedirs(args.dump_outputs, exist_ok=True)
            for name, arr in dumped.items():
                np.save(os.path.join(args.dump_outputs, name + ".npy"), arr)
        print(json.dumps(result))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
