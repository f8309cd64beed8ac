#!/usr/bin/env python
"""bench.py — (pod,node) predicate-cells/sec of the fused scheduling pass on N B200s (BASELINE.json metric).

One "step" = one pass of the hot path over one batch of synthetic pods: feasible mask (resource_fits +
nodeSelector) + feasible count + argmax-score binding for every pod of the batch against the resident node
snapshot (SURVEY.md §8d generator).

  N = 1   workload c3 = BASELINE.json configs[2]: 1M pods x 50k nodes (5e10 cells), the configuration the roofline is
          quoted on.  The same line carries a secondary object "c2" (configs[1], 100k x 10k) measured the same way.
  N > 1   workload c3 sharded on the pods dimension = BASELINE.json configs[3] ("C4"): rank r takes pods
          [r*1M/N, (r+1)*1M/N) against the replicated node table -> STRONG scaling.  The step ends when every rank
          holds every rank's bindings: the all-gather is fused into the argmax kernels (direct NVLink stores into the
          peers' CUDA-IPC gather buffers + one release flag per pair, include/ksched.h ks_exchange); `--exchange nccl`
          runs the round-1 formulation instead (one ncclAllGather on a side stream).
          `--workload c2` keeps round 1's weak-scaling run (100k pods per rank).

  value     : cells/s with the pod batch already resident in HBM (device-space ks_select), CUDA events,
              max over ranks; L2 is flushed between timed iterations.
  e2e       : the same pass through the C ABI with HOST buffers (pinned): H2D of the pod batch and D2H of the
              bindings inside the timed region (the feasible mask is produced but stays in HBM).
  e2e_objects : Pod/Node OBJECTS (quantity strings, label maps) in, bindings out, through ksh_select_nodes (host
              packer on all host threads + the same device pass) - examples/pack_bench.cpp.
  roofline  : dominant kernel's algorithmic bytes / its CUDA-event duration vs MEASURED_PEAKS.json hbm_gbs; traffic and
              pipe fractions come from the committed ncu --set full capture of the same kernel (profiles/traffic.json).
  cpu_baseline / --impl reference : the CPU restatement of the reference's per-cell path (oracle/, string
              parsing + per-cell re-summation of bound pods) on the host cores.  The Rust reference itself
              cannot be built in this image (no rustc/cargo), so kind = "port".

  --dump-outputs DIR : after the timed resident steps of each workload, rank 0 writes what the last of them returned,
              as DIR/<workload>_<name>.npy: node_idx (float32) and score (float64) of every pod of the batch (all ranks'
              shards in pod order), feasible_count (float32) of rank 0's shard and, unless --no-mask, the feasible mask of
              DUMP_MASK_ROWS pods of that shard (mask_rows: [rows, N] float32 0/1; mask_row_ids: their pod indices,
              float64), rows drawn with the workload's seed.  Inputs are generated from fixed seeds, so two builds run
              with the same arguments can be compared file by file.  About 48 MB for the default c3 + c2 run.
"""
import argparse
import importlib.util
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

METRIC = "pod_node_predicate_cells_per_sec"
UNIT = "cells/s"
FALLBACK_HBM_GBS = 6650.0
PKG_DIR = os.path.join(ROOT, "kube-scheduler-rs-reference_b200")
DUMP_MASK_ROWS = 128  # c3: 128 x 50k nodes x 4 B = 25.6 MB of the 6.25 GB mask


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c3", choices=["c2", "c3"])
    ap.add_argument("--path", default="auto", choices=["auto", "direct", "bitpar"])
    ap.add_argument("--policy", default="leftover", choices=["leftover", "least_allocated"])
    ap.add_argument("--exchange", default="p2p", choices=["p2p", "nccl"], help="N>1: how the bindings are all-gathered")
    ap.add_argument("--no-mask", action="store_true", help="do not emit the feasible mask (bindings only)")
    ap.add_argument("--mask-pitch", default="aligned", choices=["aligned", "minimal"],
                    help="row pitch of the mask buffer: ks_mask_row_bytes_aligned (256-byte blocks) or the smallest legal one")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-secondary", action="store_true", help="N=1: skip the secondary c2 object")
    ap.add_argument("--no-objects", action="store_true", help="N=1: skip the object-level end-to-end figure")
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="CPU work budget of the baseline sample")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step as DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    return args


def hbm_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return FALLBACK_HBM_GBS, "fallback (B200_PROFILING.md 6.65 TB/s)"


def usable_cores():
    """Host threads this process may really use: CPU affinity mask, capped by the cgroup CPU quota."""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    quota = None
    try:
        with open("/sys/fs/cgroup/cpu.max") as f:  # cgroup v2
            q, per = f.read().split()
            if q != "max":
                quota = float(q) / float(per)
    except Exception:
        try:
            with open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us") as f:
                q = float(f.read())
            with open("/sys/fs/cgroup/cpu/cpu.cfs_period_us") as f:
                per = float(f.read())
            if q > 0:
                quota = q / per
        except Exception:
            pass
    if quota is not None:
        n = max(1, min(n, int(quota)))
    return n, {"affinity": len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else None,
               "cgroup_quota": quota, "os_cpu_count": os.cpu_count()}


def load_standalone(name):
    """synth / objects are pure Python: the reference arm loads them by path so that it never maps libksched.so."""
    spec = importlib.util.spec_from_file_location(f"ks_ref_{name}", os.path.join(PKG_DIR, f"{name}.py"))
    mod = importlib.util.module_from_spec(spec)
    sys.modules[spec.name] = mod
    spec.loader.exec_module(mod)
    return mod


class ClockSampler:
    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
             "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.path = tempfile.mktemp(prefix="ks_clocks_", suffix=".csv")
        self.proc = None
        try:
            # `timeout`: if this process dies the sampler must not outlive it for long (a profiler wrapping the bench
            # waits for every child)
            self.proc = subprocess.Popen(
                ["timeout", "300", "nvidia-smi", "-i", str(gpu_index), f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits",
                 "-lms", "20"], stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.proc is None:
            out["reasons"] = ["nvidia-smi unavailable"]
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, smax, reasons = [], [], set()
        try:
            for line in open(self.path):
                f = [x.strip() for x in line.split(",")]
                if len(f) < 9:
                    continue
                try:
                    sm.append(float(f[1]))
                    smax.append(float(f[2]))
                except ValueError:
                    continue
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            os.unlink(self.path)
        except Exception:
            pass
        if sm:
            out.update(sm_mhz=statistics.median(sm), sm_max_mhz=max(smax), samples=len(sm))
        out["reasons"] = sorted(reasons)
        return out


def algorithmic_bytes(P, N, W, B, mask):
    """SURVEY.md §8d: every input read once, every output written once."""
    pods = P * (16 + 8 * W)
    nodes = N * (32 + 8 * W)
    bound = B * 20
    outs = P * 16
    m = P * ((N + 7) // 8) if mask else 0
    return {"pods": pods, "nodes": nodes, "bound": bound, "bindings": outs, "mask": m,
            "step_total": pods + nodes + bound + outs + m,
            "dominant_kernel": pods + nodes + m + P * 4}  # mask kernel: pods + node index in, mask + counts out


def spread(xs):
    xs = sorted(xs)
    return {"min": xs[0], "median": statistics.median(xs), "max": xs[-1]}


# ------------------------------------------------------------------------------------------------ CPU arm
def cpu_reference_arm(cl, objects, seconds, policy, cores):
    """Time the oracle's faithful per-cell path (string parse + bound re-sum per cell, like
    src/predicates.rs:20-77) on a bounded pod sample of the SAME workload.  Returns (cells/s, n, seconds)."""
    from oracle import orc
    nodes_s, bound_s, _ = objects.cluster_specs(cl, pod_slice=slice(0, 0))
    arena = objects.ObjectArena()
    nodes, bound = arena.nodes(nodes_s), arena.pods(bound_s)
    oc = orc.Cluster(nodes, cl.N, bound, cl.B)
    probe_n = max(4 * cores, 16)

    def run(first, count):
        _, _, pods_s = objects.cluster_specs(cl, pod_slice=slice(first, first + count))
        pods = arena.pods(pods_s)
        t0 = time.perf_counter()
        oc.run(pods, count, policy=policy, want_mask=True, nthreads=cores)
        return time.perf_counter() - t0

    t_probe = run(0, probe_n)
    per_pod = t_probe / probe_n
    n = int(max(probe_n, min(cl.P - probe_n, seconds / max(per_pod, 1e-9))))
    t = run(probe_n, n)
    return n * cl.N / t, n, t


def reference_main(args):
    """--impl reference: the CPU restatement of the reference's own per-cell path on the host cores.
    Under torchrun only rank 0 works.  Nothing of the product is loaded here: synth/objects are pure Python and are
    imported by path, the arithmetic is oracle/."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    synth, objects = load_standalone("synth"), load_standalone("objects")
    from oracle import orc
    cl = synth.config(args.workload)
    policy = 0 if args.policy == "leftover" else 1
    cores, core_info = usable_cores()
    nodes_s, bound_s, _ = objects.cluster_specs(cl, pod_slice=slice(0, 0))
    arena = objects.ObjectArena()
    nodes, bound = arena.nodes(nodes_s), arena.pods(bound_s)
    oc = orc.Cluster(nodes, cl.N, bound, cl.B)
    # size one step to ~4 s of wall time with all cores
    probe = max(cores, 4)
    _, _, ps = objects.cluster_specs(cl, pod_slice=slice(0, probe))
    pp = arena.pods(ps)
    t0 = time.perf_counter()
    oc.run(pp, probe, policy=policy, nthreads=cores)
    per_pod = (time.perf_counter() - t0) / probe
    budget = min(4.0, 150.0 / max(1, args.steps + args.warmup))
    n = int(max(probe, min(2000, budget / max(per_pod, 1e-9))))
    times = []
    for it in range(args.warmup + args.steps):
        first = (probe + it * n) % max(1, cl.P - n)
        _, _, ps = objects.cluster_specs(cl, pod_slice=slice(first, first + n))
        pods = arena.pods(ps)
        t0 = time.perf_counter()
        oc.run(pods, n, policy=policy, want_mask=True, nthreads=cores)
        dt = time.perf_counter() - t0
        if it >= args.warmup:
            times.append(dt)
    ms = 1e3 * sum(times) / len(times)
    value = n * cl.N / (ms * 1e-3)
    sample = f"{n} pods x {cl.N} nodes per step ({n * cl.N} cells) of workload {args.workload}, {cores} host threads"
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "strong" if args.workload == "c3" else "weak",
        "vs_baseline": None, "dtype": "int64", "data": "synthetic",
        "config": {"workload": f"{args.workload}: {cl.P} pods x {cl.N} nodes, resource_fits + nodeSelector, policy {args.policy}",
                   "note": "CPU restatement (oracle/) of the reference per-cell path; the Rust reference cannot be "
                           "built here (no rustc/cargo); each step is a bounded pod sample",
                   "step_ms": spread([1e3 * t for t in times]), "host_cores": core_info},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)
    return 0


# ------------------------------------------------------------------------------------------------ GPU arm
def run_workload(ks, torch, dist, args, workload, world, rank, local, steps, warmup, sampler_cb=None):
    """Measure one workload; returns a dict (the same on every rank for the reduced figures)."""
    dev = torch.device("cuda", local)
    policy = ks.KS_SCORE_LEFTOVER if args.policy == "leftover" else ks.KS_SCORE_LEAST_ALLOCATED
    flags = {"auto": ks.KS_SELECT_AUTO, "direct": ks.KS_SELECT_FORCE_DIRECT, "bitpar": ks.KS_SELECT_FORCE_BITPAR}[args.path]
    emit_mask = not args.no_mask

    # ---- workload: node snapshot replicated, pods sharded ----
    P_all, N = ks.synth.SHAPES[workload]
    seed = ks.synth.SEEDS[workload]
    strong = workload == "c3"
    if strong:  # C4: the one 1M-pod batch is cut into `world` shards
        cl_all = ks.synth.make(P_all, N, seed)
        lo, hi = ks.multigpu.shard_bounds(P_all, world, rank)
        cl = cl_all.take_pods(lo, hi - lo)
        cap = ks.multigpu.shard_capacity(P_all, world)
        total_pods = P_all
    else:  # round-1 weak scaling: every rank its own 100k-pod shard of a world*100k batch
        cl_all = ks.synth.make(P_all * world, N, seed)
        cl = cl_all.take_pods(rank * P_all, P_all)
        cap = P_all
        total_pods = P_all * world
    ac, am, lab, bn, bc, bm, rc, rm, sel = cl.packed()
    W = cl.label_words
    snap = ks.Snapshot(local)
    snap.set_nodes(ac, am, lab)
    snap.set_bound(bn, bc, bm)
    P = cl.P

    stream = torch.cuda.Stream()
    row = ks.mask_row_bytes_aligned(N) if args.mask_pitch == "aligned" else ks.mask_row_bytes(N)
    d_rc = torch.from_numpy(rc).to(dev)
    d_rm = torch.from_numpy(rm).to(dev)
    d_sel = torch.from_numpy(np.ascontiguousarray(sel).view(np.int64)).to(dev)
    d_cnt = torch.empty(max(P, 1), dtype=torch.int32, device=dev)
    d_mask = torch.empty((P, row), dtype=torch.uint8, device=dev) if emit_mask else None
    xch, exchange_note = None, None
    use_nccl = False
    if world > 1:
        if args.exchange == "p2p":
            try:
                xch = ks.multigpu.PeerExchange(local, world, rank, cap)
                exchange_note = "fused into the argmax kernels: direct NVLink stores into CUDA-IPC gather buffers + release flags"
            except Exception as e:  # IPC not permitted on this box: say so and use the collective
                exchange_note = f"NCCL all-gather (CUDA IPC unavailable: {e})"
                use_nccl = True
            ok = torch.tensor([0 if use_nccl else 1], dtype=torch.int32, device=dev)
            dist.all_reduce(ok, op=dist.ReduceOp.MIN)
            if int(ok.item()) == 0 and not use_nccl:
                xch.close()
                xch, use_nccl = None, True
                exchange_note = "NCCL all-gather (CUDA IPC unavailable on another rank)"
        else:
            use_nccl = True
            exchange_note = "1 NCCL all-gather of bindings/step (side stream, under the mask kernel)"
    if xch is not None:
        p_idx, p_score = xch.node_idx_ptr, xch.score_ptr
        d_bind = None
    else:
        # bindings of one shard packed in one buffer: [score i64 | node_idx i32] = 12 B per pod (capacity `cap`)
        d_bind = torch.zeros(cap * 12, dtype=torch.uint8, device=dev)
        p_score = d_bind.data_ptr()
        p_idx = p_score + 8 * cap
    d_all = torch.empty(world * cap * 12, dtype=torch.uint8, device=dev) if use_nccl else None
    side = torch.cuda.Stream() if use_nccl else None
    ev_ready = torch.cuda.Event() if use_nccl else None
    ev_gathered = torch.cuda.Event() if use_nccl else None
    if use_nccl:
        ev_ready.record(stream)  # materialise the underlying cudaEvent handles
        ev_gathered.record(stream)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2
    h_rc = torch.from_numpy(rc).pin_memory()
    h_rm = torch.from_numpy(rm).pin_memory()
    h_sel = torch.from_numpy(np.ascontiguousarray(sel).view(np.int64)).pin_memory()
    h_bind = torch.empty(max(P, 1) * 16, dtype=torch.uint8).pin_memory()

    def step_resident(timing):
        snap.select_raw(P, d_rc, d_rm, d_sel, ks.KS_MEM_DEVICE, p_idx, p_score, d_cnt, ks.KS_MEM_DEVICE,
                        mask=d_mask, mask_row_bytes=row if emit_mask else 0, mask_space=ks.KS_MEM_DEVICE,
                        policy=policy, flags=flags | (ks.KS_SELECT_TIMING if timing else 0), stream=stream.cuda_stream,
                        ready_event=ev_ready.cuda_event if use_nccl else None, exchange=xch)
        if use_nccl:
            # the ONE collective of the step runs on a side stream as soon as the library signals that node_idx and
            # score are final, i.e. under the mask kernel; the step ends when both the select and the gather are done
            side.wait_event(ev_ready)
            with torch.cuda.stream(side):
                ks.multigpu.all_gather_bindings(d_bind, d_all)
                ev_gathered.record(side)
            stream.wait_event(ev_gathered)

    def step_e2e():
        hp = h_bind.data_ptr()
        snap.select_raw(P, h_rc, h_rm, h_sel, ks.KS_MEM_HOST, hp + 8 * P, hp, hp + 12 * P, ks.KS_MEM_HOST,
                        mask=d_mask, mask_row_bytes=row if emit_mask else 0, mask_space=ks.KS_MEM_DEVICE,
                        policy=policy, flags=flags, stream=stream.cuda_stream)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def gathered_bindings():
        """node_idx [world, cap] int32 and score [world, cap] int64 as this rank holds them after a step."""
        if xch is not None:
            return xch.read()
        g = (d_all if use_nccl else d_bind).cpu().numpy().reshape(-1, cap * 12)
        return g[:, 8 * cap:12 * cap].copy().view(np.int32), g[:, :8 * cap].copy().view(np.int64)

    def shard_len(r):
        lo_r, hi_r = ks.multigpu.shard_bounds(P_all, world, r) if strong else (0, P_all)
        return hi_r - lo_r

    def last_step_outputs():
        """--dump-outputs: the arrays a caller of step_resident holds after it (module docstring)."""
        g_idx, g_score = gathered_bindings()
        out = {"node_idx": np.concatenate([g_idx[r, :shard_len(r)] for r in range(world)]),
               "score": np.concatenate([g_score[r, :shard_len(r)] for r in range(world)]),
               "feasible_count": d_cnt[:P].cpu().numpy().view(np.uint32)}
        if emit_mask:
            rows = np.sort(np.random.default_rng(seed).choice(P, size=min(P, DUMP_MASK_ROWS), replace=False))
            picked = d_mask.index_select(0, torch.from_numpy(rows).to(dev)).cpu().numpy()
            out["mask_rows"] = np.unpackbits(picked, axis=1, bitorder="little")[:, :N]
            out["mask_row_ids"] = rows
        dtypes = {"score": np.float64, "mask_row_ids": np.float64}
        for name, a in out.items():
            f = a.astype(dtypes.get(name, np.float32))
            assert np.array_equal(f.astype(a.dtype), a), f"{name} is not exactly representable as {f.dtype}"
            out[name] = f
        return out

    # ---- warm-up ----
    for _ in range(max(warmup, 3)):
        step_resident(False)
        stream.synchronize()
        step_e2e()
        barrier()  # p2p: nobody starts the next exchange step before everybody has finished this one
    # The timed region lasts only a few ms, shorter than nvidia-smi's sampling period, so the same step is kept
    # running (untimed) for ~0.4 s right before it: the clock / throttle samples are taken under exactly this load.
    # (the iteration count is fixed by rank 0 and broadcast: every rank must issue the same number of exchange steps)
    t_soak = time.perf_counter()
    for _ in range(5):
        step_resident(False)
    stream.synchronize()
    n_soak = torch.tensor([max(5, min(20000, int(0.4 / max((time.perf_counter() - t_soak) / 5, 1e-6))))],
                          dtype=torch.int64, device=dev)
    if world > 1:
        dist.broadcast(n_soak, src=0)
    for _ in range(int(n_soak.item())):
        step_resident(False)
    stream.synchronize()
    barrier()

    # ---- timed: K resident steps (CUDA events on the launching stream, L2 flushed between iterations) ----
    launches0 = ks.launch_count()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    kern_ms, scan_ms, call_ms = [], [], []
    barrier()
    t_wall0 = time.perf_counter()
    for k in range(steps):
        with torch.cuda.stream(stream):
            flush.fill_(k & 0xFF)
            ev[k][0].record(stream)
        step_resident(False)  # all-device call: the library replays its cached CUDA graph
        with torch.cuda.stream(stream):
            ev[k][1].record(stream)
    barrier()
    t_wall = time.perf_counter() - t_wall0
    launches = ks.launch_count() - launches0
    dumped = last_step_outputs() if args.dump_outputs and rank == 0 else None
    # device-clock stamps of the last timed step (us from the first kernel of the step seen by the stamps)
    xtrace = None
    if xch is not None or os.environ.get("KS_TRACE") == "1":
        marks = {}
        if os.environ.get("KS_TRACE") == "1":
            tr = snap.last_trace()
            t0 = tr.pop("t0_ns")
            for name, v in tr.items():
                if isinstance(v, tuple):
                    marks[name + "_start"], marks[name + "_end"] = t0 + 1e3 * v[0], t0 + 1e3 * v[1]
                else:
                    marks[name] = t0 + 1e3 * v
        if xch is not None:
            marks.update({"exchange_" + k: v for k, v in xch.trace_ns().items() if v})
        if marks:
            t0 = min(marks.values())
            xtrace = {k: round((v - t0) / 1e3, 2) for k, v in sorted(marks.items(), key=lambda kv: kv[1])}
    # same K steps again with per-kernel CUDA events inside the library (dominant-kernel duration for the roofline;
    # in this mode the library runs the argmax scan after the mask kernel instead of beside it, so the event pair
    # times the mask kernel alone - the measured HBM peak it is compared with is also a kernel timed alone)
    for k in range(steps):
        with torch.cuda.stream(stream):
            flush.fill_(k & 0xFF)
        step_resident(True)
        stream.synchronize()
        t = snap.last_timings()
        kern_ms.append(t[0])
        scan_ms.append(t[1])
        call_ms.append(t[2])
    barrier()
    step_ms = [a.elapsed_time(b) for a, b in ev]
    total_ms = torch.tensor([sum(step_ms)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(total_ms, op=dist.ReduceOp.MAX)
    ms_per_step = float(total_ms.item()) / steps
    cells_per_step = total_pods * N
    value = cells_per_step / (ms_per_step * 1e-3)

    # ---- timed: K end-to-end steps (host buffers, copies inside; wall clock around the blocking call) ----
    barrier()
    e2e_t = []
    for k in range(steps):
        with torch.cuda.stream(stream):
            flush.fill_(k & 0xFF)
        stream.synchronize()
        t0 = time.perf_counter()
        step_e2e()
        e2e_t.append(time.perf_counter() - t0)
    barrier()
    e2e_ms = torch.tensor([1e3 * sum(e2e_t)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(e2e_ms, op=dist.ReduceOp.MAX)
    e2e_value = cells_per_step / (float(e2e_ms.item()) / steps * 1e-3)
    if sampler_cb:
        sampler_cb()

    # ---- sanity: the resident and e2e passes produced the same bindings; the gather delivered every shard ----
    step_resident(False)
    stream.synchronize()
    if xch is not None:
        snap.exchange_check()
    barrier()
    hb = h_bind.numpy()
    e_score, e_idx, e_cnt = hb[:8 * P].view(np.int64), hb[8 * P:12 * P].view(np.int32), hb[12 * P:16 * P].view(np.uint32)
    g_idx, g_score = gathered_bindings()
    assert np.array_equal(g_idx[rank, :P], e_idx) and np.array_equal(g_score[rank, :P], e_score), "resident and e2e bindings differ"
    assert np.array_equal(d_cnt.cpu().numpy()[:P].view(np.uint32), e_cnt), "resident and e2e feasible counts differ"
    assert np.array_equal(e_idx < 0, e_cnt == 0)
    if world > 1:  # every shard arrived everywhere: compare with what each rank computed itself (checksums via all-gather)
        mine = torch.tensor([int(e_idx.astype(np.int64).sum()), int((e_score & 0xFFFFFFFF).sum())], dtype=torch.int64, device=dev)
        sums = [torch.zeros_like(mine) for _ in range(world)]
        dist.all_gather(sums, mine)
        for r in range(world):
            n_r = shard_len(r)
            got = (int(g_idx[r, :n_r].astype(np.int64).sum()), int((g_score[r, :n_r] & 0xFFFFFFFF).sum()))
            assert got == (int(sums[r][0].item()), int(sums[r][1].item())), f"rank {rank}: shard {r} of the gather is wrong"
            assert g_idx[r, :n_r].min() >= -1 and g_idx[r, :n_r].max() < N
    barrier()

    # store-only ceiling of this device, measured on the mask buffer itself (a plain 256-bit-store fill): the copy-based
    # HBM peak counts read + write bytes, a kernel that only writes cannot reach it (DESIGN.md section 7)
    write_peak = None
    if emit_mask and d_mask is not None and d_mask.numel() >= (1 << 20):
        try:
            write_peak = ks.capi.measure_write_bandwidth(local, d_mask.data_ptr(), d_mask.numel() // 32 * 32, 4)
        except Exception:
            write_peak = None
    ab = algorithmic_bytes(P, N, W, cl.B, emit_mask)
    peak, peak_src = hbm_peak()
    k_ms = sum(kern_ms) / len(kern_ms)
    achieved = ab["dominant_kernel"] / (k_ms * 1e-3) / 1e9
    path = snap.last_path()
    cap_info = {}
    try:  # figures of the committed ncu --set full capture of this kernel on this workload (per launch)
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            cap_info = json.load(f).get(f"{workload}_{path}", {}) if world == 1 else {}
            if not isinstance(cap_info, dict):
                cap_info = {"dram_bytes": cap_info}
    except Exception:
        pass
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": cap_info.get("dram_bytes"), "kernel": "k_mask_rows" if path == "bitpar" else "k_select_direct",
                "kernel_ms": k_ms, "kernel_ms_spread": spread(kern_ms),
                "rest_of_step_ms": sum(scan_ms) / len(scan_ms), "algorithmic_bytes": ab["dominant_kernel"],
                "step_algorithmic_bytes": ab["step_total"], "step_frac": ab["step_total"] / (ms_per_step * 1e-3) / 1e9 / peak,
                "peak_source": peak_src, "write_peak": write_peak,
                "frac_of_write_peak": (achieved / write_peak) if write_peak else None,
                "write_peak_source": "ks_measure_write_bandwidth: store-only fill of the mask buffer in this run (GB/s)",
                "ncu": {k: v for k, v in cap_info.items() if k != "dram_bytes"} or None}
    res = {
        "workload": workload, "P": P, "N": N, "W": W, "B": cl.B, "seed": seed, "path": path, "value": value,
        "ms_per_step": ms_per_step, "step_ms": spread(step_ms), "e2e_value": e2e_value, "e2e_ms": spread([1e3 * t for t in e2e_t]),
        "launches": int(launches), "roofline": roofline, "t_wall": t_wall, "call_ms": sum(call_ms) / len(call_ms),
        "total_pods": total_pods, "strong": strong, "exchange": exchange_note, "emit_mask": emit_mask,
        "xtrace": xtrace,
        "h2d": P * (16 + 8 * W), "d2h": P * 16, "row": row,
    }
    if world == 1:
        # for information: the reference's own policy (<=5 seeded draws per pod, src/main.rs:49-71) on the same batch,
        # host buffers in and out; it evaluates <=5 cells per pod, so it is quoted in pods/s, not cells/s
        snap.select_sampling(rc[:1024], rm[:1024], sel[:1024], seed=seed)
        t0 = time.perf_counter()
        s_idx, s_used, _, _ = snap.select_sampling(rc, rm, sel, seed=seed)
        t_s = time.perf_counter() - t0
        res["reference_policy"] = {"pods_per_s": P / t_s, "cells_evaluated": int(s_used.sum()),
                                   "bound_frac": float((s_idx >= 0).mean()), "argmax_bound_frac": float((e_idx >= 0).mean()),
                                   "note": "ks_select_sampling, ATTEMPTS=5, seeded; not part of value/e2e"}
    res["_cl"] = cl
    res["_packed"] = (ac, am, lab, rc, rm, sel)
    if xch is not None:
        xch.close()
    snap.close()
    del d_mask, flush
    torch.cuda.empty_cache()
    if dumped is not None:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, a in dumped.items():
            np.save(os.path.join(args.dump_outputs, f"{workload}_{name}.npy"), a)
    return res


def main():
    args = parse_args()
    if args.impl == "reference":
        return reference_main(args)

    import torch
    import torch.distributed as dist
    import ksched_pkg
    ks = ksched_pkg.load()

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available() or ks.device_count() == 0:
        print(json.dumps({"error": "no CUDA device: bench.py has no CPU fallback for the product arm"}), flush=True)
        return 2
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    # clocks are sampled over warm-up + both timed loops of the headline workload
    sampler = ClockSampler(local) if rank == 0 else None
    clocks = {}

    def stop_sampler():
        nonlocal sampler
        if sampler:
            clocks.update(sampler.stop())
            sampler = None

    try:
        r = run_workload(ks, torch, dist, args, args.workload, world, rank, local, args.steps, args.warmup, stop_sampler)
    finally:  # a failed run must not leave nvidia-smi running
        stop_sampler()
    sec = None
    if world == 1 and args.workload == "c3" and not args.no_secondary:
        sec = run_workload(ks, torch, dist, args, "c2", 1, 0, local, args.steps, args.warmup)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return 0

    P, N, W = r["P"], r["N"], r["W"]
    wl = args.workload
    if wl == "c3" and world > 1:
        wl_text = (f"c4 = c3 sharded on pods: {r['total_pods']} pods / {world} GPUs = {P} pods/GPU x {N} nodes "
                   f"({r['total_pods'] * N:.3g} cells per step in total)")
    else:
        wl_text = f"{wl}: {P} pods/GPU x {N} nodes ({P * N:.3g} cells/GPU)"
    line = {
        "metric": METRIC, "value": r["value"], "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": r["ms_per_step"], "higher_is_better": True, "scaling": "strong" if r["strong"] else "weak",
        "vs_baseline": None, "dtype": "int64", "data": "synthetic",
        "config": {
            "workload": f"{wl_text}, resource_fits + nodeSelector + argmax score ({args.policy}), "
                        f"mask {'emitted' if r['emit_mask'] else 'not emitted'}",
            "label_words": W, "bound_pods": r["B"], "seed": hex(r["seed"]), "path": r["path"],
            "mask_row_pitch_bytes": r["row"], "mask_row_min_bytes": ks.mask_row_bytes(N),
            "trace": os.environ.get("KS_TRACE") == "1",
            "parallelism": f"pods sharded x{world}, node table replicated" + (f"; bindings exchange: {r['exchange']}" if world > 1 else ""),
            "l2": "256 MiB flush write between timed iterations", "wall_s_timed_region": r["t_wall"],
            "clocks_window": "0.4 s untimed soak of the same step + both timed loops (timed region alone is a few ms)",
            "call_ms_inside_library": r["call_ms"], "step_ms": r["step_ms"], "e2e_ms": r["e2e_ms"],
            **({"trace_us_rank0_last_timed_step": r["xtrace"]} if r.get("xtrace") else {}),
        },
        "clocks": clocks or None,
        "e2e": {"value": r["e2e_value"], "unit": UNIT, "h2d_bytes_per_step": r["h2d"], "d2h_bytes_per_step": r["d2h"],
                "note": "host pinned pods in, bindings out; feasible mask written to HBM, not copied to host"},
        "gpu_launches": r["launches"],
        "roofline": r["roofline"],
    }
    if "reference_policy" in r:
        line["reference_policy"] = r["reference_policy"]
    if sec is not None:
        line["c2"] = {"workload": f"c2: {sec['P']} pods x {sec['N']} nodes (BASELINE.json configs[1]), same measurement",
                      "value": sec["value"], "ms_per_step": sec["ms_per_step"], "step_ms": sec["step_ms"],
                      "e2e": {"value": sec["e2e_value"], "h2d_bytes_per_step": sec["h2d"], "d2h_bytes_per_step": sec["d2h"]},
                      "gpu_launches": sec["launches"], "roofline": sec["roofline"]}
    if world == 1 and not args.no_objects:
        # Pod/Node objects in -> bindings out (ksh_select_nodes: host packer on all host threads + the device pass);
        # objects are built natively by examples/pack_bench.cpp, the way a Rust/C host would hold them
        try:
            import bench_pack
            t0 = time.perf_counter()
            pk = bench_pack.native(wl, local)
            line["e2e_objects"] = {"value": pk["select_nodes_objects_cells_per_s"], "unit": UNIT,
                                   "ms_per_call": pk["select_nodes_objects_ms"], "host_threads": pk["threads"],
                                   "hardware_concurrency": pk["hardware_concurrency"], "pack_pods_per_s": pk["pods_per_s"],
                                   "reconcile_batch_10k_ms": pk["reconcile_batch_10k_ms"],
                                   "note": f"ksh_select_nodes over {pk['pods']} Pod objects x {pk['nodes']} Node objects "
                                           f"(strings parsed on the host inside the call); {time.perf_counter() - t0:.1f} s incl. object generation"}
        except Exception as e:
            line["e2e_objects"] = {"error": str(e)[:300]}
    if world == 1 and not args.no_cpu_baseline:
        # second CPU figure (BASELINE.md §3 "CPU-packed"): the same SoA int64 + bitmask algorithm the GPU runs, C,
        # all usable host threads, on a pod sample — what a well-written CPU scheduler core could do with packed inputs
        from oracle import orc
        cores, core_info = usable_cores()
        cl = r["_cl"]
        ac, am, lab, rc, rm, sel = r["_packed"]
        n_pk = min(P, 20000)
        fc_h, fm_h = cl.free()
        t0 = time.perf_counter()
        orc.run_packed(fc_h, fm_h, ac, am, lab, rc[:n_pk], rm[:n_pk], sel[:n_pk], policy=0 if args.policy == "leftover" else 1,
                       want_mask=True, nthreads=cores)
        t_pk = time.perf_counter() - t0
        cps, n, t = cpu_reference_arm(cl, ks.objects, args.cpu_seconds, 0 if args.policy == "leftover" else 1, cores)
        line["cpu_baseline"] = {"value": cps, "unit": UNIT, "cores": cores, "kind": "port", "host_cores": core_info,
                                "sample": f"first {n} pods x {N} nodes ({n * N} cells, {t:.1f} s) of the same workload, "
                                          f"faithful per-cell path (quantity parse + bound-pod re-sum per cell)",
                                "packed_soa": {"value": n_pk * N / t_pk, "unit": UNIT, "cores": cores,
                                               "sample": f"first {n_pk} pods x {N} nodes, same SoA/bitmask algorithm in C "
                                                         f"(oracle packed flavour), mask + argmax, {t_pk:.2f} s"}}
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
