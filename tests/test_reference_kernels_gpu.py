"""Three-way parity on the GPU: the reference's OWN CUDA kernels vs the CPU oracle vs this repo's kernels.  The reference
kernels' outputs are the golden vectors under tests/golden/, written on B200 by tests/golden/make_golden.py from
oracle/_ref (the reference's kernels compiled unmodified for sm_100a), so no reference build is needed here."""
import os

import numpy as np
import pytest
import torch

from oracle import oracle
from tests.golden import cases
from tests.util import assert_hough_rows_equal, to_np

pytestmark = pytest.mark.gpu

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def load(name):
    return np.load(os.path.join(GOLD, name + ".npz"))


def T(a, dev):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev)


def rows(g):
    return g["box"], g["pose"], g["target"], g["weight"], g["domain"]


@pytest.mark.parametrize("name", ["h_test_a", "h_train_b", "h_thr_c", "h_skip1_d"])
def test_hough_reference_vs_oracle_vs_ours(cuda, name):
    from posecnn_b200.hough_voting_gpu_layer import hough_voting_gpu_op as op
    g = load(name)
    r_votes = g["votes"].astype(np.float32)
    sc, is_train, vt, pt, skip = cases.hough_inputs(name)
    d = [T(sc[k], cuda) for k in ("label", "vertex", "extents", "meta")]
    gt = T(sc["gt"], cuda) if len(sc["gt"]) else None
    o_outs, dbg = oracle.hough_voting_gpu(sc["label"], sc["vertex"], sc["extents"], sc["meta"], sc["gt"], is_train, vt, pt,
                                          skip, debug=True)
    # reference kernels vs CPU restatement: votes within the ambiguity bound, rows equal
    dv = np.abs(r_votes - dbg["votes"])
    assert (dv <= dbg["ambig"]).all(), f"oracle differs from the reference kernel on {int((dv > dbg['ambig']).sum())} cells"
    assert int(g["num_rois"]) == dbg["num_rois"]
    assert_hough_rows_equal(rows(g), o_outs, is_train)
    # this repo's kernels vs the reference kernels, directly
    planes = op.hough_vote_planes(*d, skip)
    dv2 = np.abs(to_np(planes) - r_votes)
    assert (dv2 <= dbg["ambig"]).all(), f"{int((dv2 > dbg['ambig']).sum())} cells differ from the reference kernel"
    got = op.hough_voting_gpu(*d, gt, is_train, vt, pt, skip)
    assert_hough_rows_equal(got, rows(g), is_train)


def test_hough_reference_launcher_as_shipped(cuda):
    """The reference launcher exactly as shipped (atomicAdd list order).  With skip_pixels = 1 every
    pixel votes, so the vote set is order independent and the op output must match ours as a set."""
    from posecnn_b200.hough_voting_gpu_layer import hough_voting_gpu_op as op
    g = load("h_skip1_d_shipped")
    sc, is_train, vt, pt, skip = cases.hough_inputs("h_skip1_d")
    d = [T(sc[k], cuda) for k in ("label", "vertex", "extents", "meta")]
    gt = T(sc["gt"], cuda)
    got = op.hough_voting_gpu(*d, gt, 0, vt, pt, 1)
    assert int(g["num_rois"]) == got[0].shape[0]
    assert_hough_rows_equal(got, rows(g), 0, as_set=True)


def test_pixel_ops_reference_vs_ours(cuda):
    from posecnn_b200.average_distance_loss import average_distance_loss_op as aop
    from posecnn_b200.backprojecting_layer import backprojecting_op as bop
    from posecnn_b200.hard_label_layer import hard_label_op as hop
    from posecnn_b200.projecting_layer import projecting_op as pop
    from posecnn_b200.roi_pooling_layer import roi_pooling_op as rop
    dev = cuda
    data, rois, grad = cases.roi_inputs()
    g = load("roi_pool")
    for pc, (rt, ra) in ((0, (g["top"], g["argmax"])), (1, (g["top_cls"], g["argmax_cls"]))):
        ot, oa = rop.roi_pool(T(data, dev), T(rois, dev), 7, 7, 1.0 / 16.0, pc)
        np.testing.assert_array_equal(to_np(oa), ra)
        np.testing.assert_array_equal(to_np(ot), rt)
        wt_, wa_ = oracle.roi_pool(data, rois, 7, 7, 1.0 / 16.0, pc)
        np.testing.assert_array_equal(wa_, ra)
    og = rop.roi_pool_grad(T(data, dev), T(rois, dev), T(g["argmax"], dev), T(grad, dev), 7, 7, 1.0 / 16.0, 0)
    np.testing.assert_allclose(to_np(og), g["grad_in"], rtol=1e-5, atol=1e-6)
    g = load("hard_label")
    prob, gtl = cases.hard_label_inputs()
    for thr in (1.0, 0.5):
        np.testing.assert_array_equal(to_np(hop.hard_label(T(prob, dev), T(gtl, dev), thr)), g[f"thr_{thr}"].astype(np.float32))
    g = load("projection")
    c = cases.projection_inputs()
    d = {k: T(v, dev) for k, v in c.items()}
    otd, otl, otf = bop.backproject(d["data"], d["label"], d["depth"], d["meta"], d["label_3d"], 16, 3, 0.02)
    # same fp32 expressions, same contraction -> identical on the same device
    np.testing.assert_array_equal(to_np(otf), g["top_flag"].astype(np.float32))
    np.testing.assert_allclose(to_np(otd), g["top_data"], rtol=1e-6, atol=1e-6)
    np.testing.assert_allclose(to_np(otl), g["top_label"], rtol=1e-6, atol=1e-6)
    np.testing.assert_array_equal(to_np(pop.project(d["vox"], d["depth"], d["meta"], 3, 0.02)), g["project"])
    np.testing.assert_array_equal(to_np(bop.backproject_grad(d["data"], d["depth"], d["meta"], d["g3"], 16)), g["backproject_grad"])
    np.testing.assert_allclose(to_np(pop.project_grad(d["vox"], d["depth"], d["meta"], d["g2"], 3, 0.02)), g["project_grad"],
                               rtol=1e-6, atol=1e-6)
    g = load("average_distance")
    pred, targ, wt, pts, sym = cases.avgdist_inputs()
    a = [T(x, dev) for x in (pred, targ, wt, pts, sym)]
    ol, od = aop.average_distance_loss(*a, 0.01)
    np.testing.assert_allclose(to_np(ol), g["loss"], rtol=1e-4)
    np.testing.assert_allclose(to_np(od), g["diff"], rtol=1e-3, atol=1e-4 * float(np.abs(g["diff"]).max()))
