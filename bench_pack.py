"""Host packer throughput (SURVEY.md §8f #1): Pod/Node OBJECTS (quantity strings, label maps) -> the SoA int64 /
label-bitmask arrays the device consumes, through a packing-only context (KSH_DEVICE_NONE).  Pure host work: runs
without a GPU.  Compiles and runs examples/pack_bench.cpp (objects built natively, the way a Rust/C host holds them)
and prints its JSON line; `--python-objects` adds the same calls over the ctypes objects of the test-suite generator
(scattered Python allocations: a lower bound, dominated by cache misses in the caller's objects).
KSH_THREADS sets the host thread count."""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
SHAPES = {"c2": (10_000, 100_000, 100_000), "c3": (50_000, 1_000_000, 500_000)}  # nodes, pods, bound pods


def native(workload, device=-1):
    """The executable is built in a temporary directory: the source tree may be read-only."""
    libdir = os.path.join(ROOT, "kube-scheduler-rs-reference_b200")
    n, p, b = SHAPES[workload]
    with tempfile.TemporaryDirectory(prefix="ks_pack_bench_") as tmp:
        exe = os.path.join(tmp, "pack_bench")
        subprocess.run(["g++", "-O2", "-std=c++17", "-I" + os.path.join(ROOT, "include"), os.path.join(ROOT, "examples", "pack_bench.cpp"),
                        "-L" + libdir, "-lksched", "-Wl,-rpath," + libdir, "-pthread", "-o", exe], check=True)
        out = subprocess.run([exe, str(n), str(p), str(b), str(device)], check=True, capture_output=True, text=True).stdout
    return json.loads(out)


def python_objects(workload):
    import ksched_pkg
    ks = ksched_pkg.load()
    cl = ks.synth.config(workload)
    nodes_s, bound_s, pods_s = ks.objects.cluster_specs(cl)
    arena = ks.objects.ObjectArena()
    nodes, bound, pods = arena.nodes(nodes_s), arena.pods(bound_s), arena.pods(pods_s)
    best = {}
    with ks.host.Context(ks.host.KSH_DEVICE_NONE) as ctx:
        for _ in range(3):
            for name, call in (("set_nodes", lambda: ctx.set_nodes(nodes, cl.N)),
                               ("set_cluster_pods", lambda: ctx.set_cluster_pods(bound, cl.B)),
                               ("pack_pods", lambda: ctx.pack_pods(pods, cl.P))):
                t0 = time.perf_counter()
                call()
                best[name] = min(best.get(name, 1e9), 1e3 * (time.perf_counter() - t0))
    return {"nodes": cl.N, "bound_pods": cl.B, "pods": cl.P, "ms": best, "pods_per_s": cl.P / best["pack_pods"] * 1e3}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="c2", choices=list(SHAPES))
    ap.add_argument("--python-objects", action="store_true")
    ap.add_argument("--device", type=int, default=-1, help="B200 ordinal: also time the object-level ksh_select_nodes / ksh_reconcile_batch")
    args = ap.parse_args()
    line = native(args.workload, args.device)
    line["workload"] = args.workload
    if args.python_objects:
        line["python_objects"] = python_objects(args.workload)
    print(json.dumps(line))
    return 0


if __name__ == "__main__":
    sys.exit(main())
