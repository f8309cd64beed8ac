"""The two-chunk host pipeline of ks_select: host-space pods and outputs on the bit-parallel path from 262144 pods up
(no host-space mask, no timing).  The second pod chunk is copied in while the first computes and the bindings of each
chunk travel back on their own; the results must be those of the oracle, bit for bit, with and without a cached graph."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

P, N = 300_001, 2_500  # odd P: the two chunks differ in size (150000 + 150001 pods)


@pytest.fixture(scope="module")
def cluster(ks, orc):
    cl = ks.synth.make(P, N, seed=0x91BE)
    ac, am, lab, bn, bc, bm, rc, rm, sel = cl.packed()
    assert lab.shape[1] == 1
    fc, fm = orc.free_reduce(ac, am, bn, bc, bm)
    return cl, fc, fm


def _snapshot(ks, cl):
    ac, am, lab, bn, bc, bm = cl.packed()[:6]
    snap = ks.Snapshot(0)
    snap.set_nodes(ac, am, lab)
    snap.set_bound(bn, bc, bm)
    return snap


def test_pipeline_pageable_numpy(ks, orc, cluster):
    """Pageable buffers: the pipeline runs without a graph."""
    cl, fc, fm = cluster
    ac, am, lab, bn, bc, bm, rc, rm, sel = cl.packed()
    o_idx, o_score, o_cnt = orc.run_packed(fc, fm, ac, am, lab, rc, rm, sel, want_mask=False)[:3]
    with _snapshot(ks, cl) as snap:
        r = snap.select(rc, rm, sel, want_mask=False)
    assert r.path == "bitpar"
    assert np.array_equal(r.node_idx, o_idx)
    assert np.array_equal(r.score, o_score)
    assert np.array_equal(r.feasible_cnt, o_cnt)


def test_pipeline_pinned_graph_replay(ks, orc, cluster):
    """Pinned pods and outputs with a device-space mask: captured, replayed, then replayed over new request values
    written into the same pinned buffers."""
    import torch
    cl, fc, fm = cluster
    ac, am, lab, bn, bc, bm, rc, rm, sel = cl.packed()
    dev = torch.device("cuda:0")
    row_min, row = ks.mask_row_bytes(N), ks.mask_row_bytes_aligned(N)
    h_rc = torch.from_numpy(rc.copy()).pin_memory()
    h_rm = torch.from_numpy(rm.copy()).pin_memory()
    h_sel = torch.from_numpy(np.ascontiguousarray(sel).view(np.int64)).pin_memory()
    idx = torch.empty(P, dtype=torch.int32).pin_memory()
    score = torch.empty(P, dtype=torch.int64).pin_memory()
    cnt = torch.empty(P, dtype=torch.int32).pin_memory()
    mask = torch.empty((P, row), dtype=torch.uint8, device=dev)
    rc2 = rc.copy()
    rc2[1::3] += 700  # pods in both chunks change
    with _snapshot(ks, cl) as snap:
        for rep, req in enumerate((rc, rc, rc2)):
            h_rc.copy_(torch.from_numpy(req))
            idx.fill_(-7)
            score.fill_(-7)
            cnt.fill_(-7)
            mask.fill_(0xA5)
            torch.cuda.synchronize()
            snap.select_raw(P, h_rc, h_rm, h_sel, ks.KS_MEM_HOST, idx, score, cnt, ks.KS_MEM_HOST, mask=mask,
                            mask_row_bytes=row, mask_space=ks.KS_MEM_DEVICE)
            assert snap.last_path() == "bitpar", rep
            o_idx, o_score, o_cnt, o_mask, _ = orc.run_packed(fc, fm, ac, am, lab, req, rm, sel, want_mask=True)
            assert np.array_equal(idx.numpy(), o_idx), f"node_idx, call {rep}"
            assert np.array_equal(score.numpy(), o_score), f"score, call {rep}"
            assert np.array_equal(cnt.numpy().view(np.uint32), o_cnt), f"feasible_cnt, call {rep}"
            m = mask.cpu().numpy()
            assert np.array_equal(m[:, :row_min], o_mask), f"mask, call {rep}"
            assert (m[:, row_min:] == 0).all(), f"mask padding, call {rep}"
