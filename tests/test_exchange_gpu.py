"""Fused all-gather of the bindings (include/ksched.h ks_exchange; SURVEY.md §8e) on real hardware.

Two processes = two ranks.  With one visible GPU both ranks share cuda:0 (a CUDA-IPC mapping of another process's
allocation on the same device is still a peer mapping, so the kernels, flags and the wait are the real ones); with
two or more GPUs each rank takes its own device and the stores cross NVLink.  torch.distributed (gloo) only carries
the 64-byte IPC handles.  Every rank must end up with every rank's bindings, bit-exact against the CPU oracle of the
unsharded batch, on both kernel paths, over several steps (sequence numbers) and with an empty shard."""
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
pytestmark = pytest.mark.gpu


def _worker(rank, world, port, P, N, flags, steps, policy, q):
    try:
        sys.path.insert(0, ROOT)
        import torch
        import torch.distributed as dist
        import ksched_pkg
        ks = ksched_pkg.load()
        from oracle import orc
        os.environ["MASTER_ADDR"] = "127.0.0.1"
        os.environ["MASTER_PORT"] = str(port)
        dist.init_process_group("gloo", rank=rank, world_size=world)
        device = rank % max(1, torch.cuda.device_count())
        torch.cuda.set_device(device)
        dev = torch.device("cuda", device)
        cl = ks.synth.make(P, N, seed=9090 + N, bound_per_node=4)
        ac, am, lab, bn, bc, bm, rc, rm, sel = cl.packed()
        lo, hi = ks.multigpu.shard_bounds(P, world, rank)
        cap = ks.multigpu.shard_capacity(P, world)
        n = hi - lo
        snap = ks.Snapshot(device)
        snap.set_nodes(ac, am, lab)
        snap.set_bound(bn, bc, bm)
        xch = ks.multigpu.PeerExchange(device, world, rank, max(cap, 1))
        t = [torch.from_numpy(np.ascontiguousarray(x[lo:hi]).view(np.int64).copy()).to(dev) for x in (rc, rm, sel)]
        cnt = torch.zeros(max(n, 1), dtype=torch.int32, device=dev)
        row = ks.mask_row_bytes(N)
        mask = torch.zeros((max(n, 1), row), dtype=torch.uint8, device=dev)
        st = torch.cuda.Stream()
        fc, fm = orc.free_reduce(ac, am, bn, bc, bm)
        ok = True
        for step in range(steps):
            rc_it = rc + 50 * step  # new requests every step: stale data in a gather buffer would be detected
            t[0].copy_(torch.from_numpy(np.ascontiguousarray(rc_it[lo:hi])))
            torch.cuda.synchronize()
            dist.barrier()  # nobody overwrites a gather buffer that a peer is still reading
            snap.select_raw(n, t[0], t[1], t[2], ks.KS_MEM_DEVICE, xch.node_idx_ptr, xch.score_ptr, cnt, ks.KS_MEM_DEVICE,
                            mask=mask, mask_row_bytes=row, mask_space=ks.KS_MEM_DEVICE, policy=policy, flags=flags,
                            stream=st.cuda_stream, exchange=xch)
            st.synchronize()
            snap.exchange_check()
            g_idx, g_score = xch.read()
            fi, fs, fcn, fmask, _ = orc.run_packed(fc, fm, ac, am, lab, rc_it, rm, sel, policy=policy, want_mask=True, nthreads=2 if P * N < 10**9 else 16)
            for r in range(world):
                l, h = ks.multigpu.shard_bounds(P, world, r)
                ok &= np.array_equal(g_idx[r, :h - l], fi[l:h]) and np.array_equal(g_score[r, :h - l], fs[l:h])
            ok &= np.array_equal(cnt.cpu().numpy()[:n].view(np.uint32), fcn[lo:hi])
            ok &= np.array_equal(mask.cpu().numpy()[:n], fmask[lo:hi])
            dist.barrier()
        xch.close()
        snap.close()
        q.put((rank, bool(ok), n, ""))
        dist.destroy_process_group()
    except Exception as e:  # report instead of hanging the parent
        import traceback
        q.put((rank, False, -1, traceback.format_exc()[-1500:] + str(e)))


@pytest.mark.parametrize("P,N,flags,steps,policy", [
    (40000, 3000, 2, 3, 0), (3001, 2500, 1, 3, 0), (1, 5000, 2, 3, 0), (90000, 50000, 2, 1, 0), (40000, 3000, 2, 3, 1)],
    ids=["40000-3000-2-3", "3001-2500-1-3", "1-5000-2-3", "90000-50000-2-1", "40000-3000-2-3-least_allocated"])
def test_fused_exchange_two_ranks(P, N, flags, steps, policy):
    """flags 2 = bit-parallel path (stores fused into the argmax kernels), 1 = per-cell path (push kernel);
    policy 1 = KS_SCORE_LEAST_ALLOCATED, whose bit-parallel argmax kernel (k_least_alloc) stores to the peers itself;
    P = 1 leaves rank 1 with an empty shard; 90000 x 50000 is a long mask pass (282 MB per rank): 896-thread mask CTAs with
    128-thread argmax CTAs beside them, where the small cases run the argmax kernels on SMs the mask kernel leaves free."""
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 32000 + (os.getpid() % 2000) + flags
    procs = [ctx.Process(target=_worker, args=(r, 2, port, P, N, flags, steps, policy, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = [q.get(timeout=600) for _ in procs]
    for p in procs:
        p.join(timeout=60)
    assert sorted(r[0] for r in res) == [0, 1], res
    assert all(r[1] for r in res), res
    assert sum(r[2] for r in res) == P
