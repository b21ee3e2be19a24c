"""CPU-only tests (-m "not gpu"): the oracle's own properties, the host-side op modules and
the C ABI surface (library loads, every symbol declared in include/posecnn_b200.h is exported).
No compute call is made without a GPU."""
import ctypes
import os
import re

import numpy as np
import pytest

from oracle import oracle
from posecnn_b200 import synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_abi_exports_every_declared_symbol(native_lib):
    hdr = open(os.path.join(ROOT, "include", "posecnn_b200.h")).read()
    names = sorted(set(re.findall(r"\b(pcnn_[a-z0-9_]+)\s*\(", hdr)))
    assert len(names) >= 15
    for n in names:
        assert hasattr(native_lib, n), f"{n} declared in include/posecnn_b200.h but not exported"
    assert native_lib.pcnn_version() >= 100


def test_abi_argument_validation_without_gpu(native_lib):
    # validation happens before any CUDA call, so these are safe on a CPU-only box
    nbytes = ctypes.c_size_t(0)
    assert native_lib.pcnn_hough_vote_workspace_bytes(1, 480, 640, 22, 10, ctypes.c_float(-1.0), ctypes.byref(nbytes)) == 0
    assert nbytes.value > 0
    small = nbytes.value
    assert native_lib.pcnn_hough_vote_workspace_bytes(32, 480, 640, 22, 10, ctypes.c_float(-1.0), ctypes.byref(nbytes)) == 0
    assert nbytes.value > small
    assert native_lib.pcnn_hough_vote_workspace_bytes(1, 480, 640, 1, 10, ctypes.c_float(-1.0), ctypes.byref(nbytes)) == -1
    native_lib.pcnn_last_error.restype = ctypes.c_char_p
    assert b"C >= 2" in native_lib.pcnn_last_error()
    assert native_lib.pcnn_hough_vote_workspace_bytes(1, 480, 640, 22, 0, ctypes.c_float(-1.0), ctypes.byref(nbytes)) == -1
    assert native_lib.pcnn_roi_pool_fwd(None, None, 1, 5, 1, 4, 4, 4, 7, 7, ctypes.c_float(1.0), 0, None, None, None) == -1


def test_host_planning_without_gpu(native_lib):
    """Host-side planning of the round-2 kernels (no CUDA call): Hough band height by batch size, weight-gradient work split incl. the
    paired Cout = Cin = 64 case and the single-split (direct-epilogue) fully connected case, NULL / shape validation of the new entries."""
    nbytes = ctypes.c_size_t(0)
    ws = {}
    for B in (1, 2, 4, 8, 16, 32, 64):
        assert native_lib.pcnn_hough_vote_workspace_bytes(B, 480, 640, 22, 10, ctypes.c_float(-1.0), ctypes.byref(nbytes)) == 0
        ws[B] = nbytes.value
    assert all(ws[a] < ws[b] for a, b in zip((1, 2, 4, 8, 16, 32), (2, 4, 8, 16, 32, 64)))      # monotone in the batch size
    # 8-row bands below ~16 items per resident CTA (B <= 8 at C = 22, H = 480), 16 rows above: the per-image band table doubles
    assert ws[8] / 8 > ws[16] / 16
    for (B, H, W, Cin, Cout, k) in [(16, 480, 640, 64, 64, 3), (2, 20, 36, 64, 64, 3), (16, 60, 80, 512, 512, 3), (1, 1, 117, 25088, 4096, 1),
                                    (1, 1, 37, 1024, 256, 1), (4, 30, 40, 512, 64, 1)]:
        assert native_lib.pcnn_conv_wgrad_workspace_bytes(B, H, W, Cin, Cout, k, ctypes.byref(nbytes)) == 0
        per_split = 4 * k * k * Cin * Cout
        assert nbytes.value >= per_split and nbytes.value % 256 == 0
        splits = nbytes.value // per_split
        assert 1 <= splits <= 2 * 148                                                              # at most two waves of work items
    assert native_lib.pcnn_conv_wgrad_workspace_bytes(1, 8, 8, 48, 64, 3, ctypes.byref(nbytes)) == -1  # Cin % 64
    f1 = ctypes.c_float(1.0)
    assert native_lib.pcnn_up8_heads_bwd_ex(None, None, None, None, f1, f1, None, None, None, None, None, f1, f1, f1, 1, 8, 8, 22, 64, 128,
                                            None, None, None, None, ctypes.c_size_t(0), None) == -1
    assert native_lib.pcnn_vertex_loss_fused_lowres_fwd(None, None, None, None, 1, 64, 96, 22, ctypes.c_float(1.0), ctypes.c_float(1.0), None,
                                                        None, ctypes.c_size_t(0), None) == -1


def test_ops_refuse_cpu_tensors(native_lib):
    import torch
    from posecnn_b200.hard_label_layer import hard_label_op
    from posecnn_b200.roi_pooling_layer import roi_pooling_op
    with pytest.raises(RuntimeError, match="CUDA tensor"):
        hard_label_op.hard_label(torch.zeros(1, 2, 2, 3), torch.zeros(1, 2, 2, dtype=torch.int32), 1.0)
    with pytest.raises(RuntimeError, match="CUDA tensor"):
        roi_pooling_op.roi_pool(torch.zeros(1, 4, 4, 4), torch.zeros(1, 7), 7, 7, 1.0, 0)


def test_reference_style_imports():
    """lib/networks/network.py:6-26 imports `<layer>.<layer>_op`; with posecnn_b200/ on sys.path
    the same statements resolve to this package."""
    import subprocess, sys
    code = ("import sys; sys.path.insert(0, %r); sys.path.insert(0, %r);"
            "import hough_voting_gpu_layer.hough_voting_gpu_op as h, roi_pooling_layer.roi_pooling_op as r,"
            "hard_label_layer.hard_label_op as hl, backprojecting_layer.backprojecting_op as b,"
            "projecting_layer.projecting_op as p, average_distance_loss.average_distance_loss_op as a;"
            "assert all(hasattr(m, n) for m, n in [(h,'hough_voting_gpu'),(h,'hough_voting_gpu_grad'),(r,'roi_pool'),"
            "(r,'roi_pool_grad'),(hl,'hard_label'),(hl,'hard_label_grad'),(b,'backproject'),(b,'backproject_grad'),"
            "(p,'project'),(p,'project_grad'),(a,'average_distance_loss'),(a,'average_distance_loss_grad')])"
            % (ROOT, os.path.join(ROOT, "posecnn_b200")))
    subprocess.check_call([sys.executable, "-c", code])


def test_oracle_hough_recovers_planted_centres():
    sc = synth.make_scene(batch=2, height=120, width=160, num_classes=5, objects_per_image=2, seed=11,
                          dir_noise=0.0, min_pixels=520)
    outs, dbg = oracle.hough_voting_gpu(sc["label"], sc["vertex"], sc["extents"], sc["meta"], sc["gt"], 0, -1.0, 0.02, 10,
                                        debug=True)
    box, pose = outs[0], outs[1]
    found = {(int(r[0]), int(r[1])): r for r in box}
    assert dbg["num_rois"] == len(found) >= 2
    K = synth.intrinsics(120, 160)
    for (b, cls, cx, cy, z) in sc["centers"]:
        if (sc["label"][b] == cls).sum() <= 500:
            continue
        r = found[(b, cls)]
        x, y = 0.5 * (r[2] + r[4]), 0.5 * (r[3] + r[5])
        assert abs(x - cx) <= 3 and abs(y - cy) <= 3        # SURVEY App. A.1: >= 3 px tolerance for the cone vote
        row = [i for i in range(box.shape[0]) if int(box[i, 0]) == b and int(box[i, 1]) == cls][0]
        assert abs(pose[row, 6] - z) < 0.02 * z
        assert abs(pose[row, 4] - z * (x - K[0, 2]) / K[0, 0]) < 1e-3


def test_oracle_hough_dummy_row_and_cap():
    sc = synth.make_scene(batch=1, height=60, width=80, num_classes=3, objects_per_image=1, seed=2, min_pixels=100)
    # every object is below the 500-pixel label threshold -> dummy zero row (hough_voting_gpu_op.cc:379-383)
    outs = oracle.hough_voting_gpu(sc["label"], sc["vertex"], sc["extents"], sc["meta"], sc["gt"], 0, -1.0, 0.02, 10)
    assert outs[0].shape == (1, 7) and not outs[0].any()
    # batch 64 -> cap = 128 / 64 = 2 maxima per image (SURVEY finding 3)
    sc = synth.make_scene(batch=1, height=120, width=160, num_classes=6, objects_per_image=4, seed=5, min_pixels=520)
    lab = np.repeat(sc["label"], 64, 0)[:64]
    cnt = sum((sc["label"][0] == c).sum() > 500 for c in range(1, 6))
    assert cnt >= 3
    outs, dbg = oracle.hough_voting_gpu(lab[:64], np.repeat(sc["vertex"], 64, 0), sc["extents"], np.repeat(sc["meta"], 64, 0),
                                        sc["gt"], 0, -1.0, 0.02, 10, debug=False), None
    box = outs[0]
    assert box.shape[0] == 64 * 2
    assert np.bincount(box[:, 0].astype(int)).tolist() == [2] * 64


def test_oracle_hough_train_rows():
    sc = synth.make_scene(batch=1, height=120, width=160, num_classes=4, objects_per_image=2, seed=3, min_pixels=520)
    outs = oracle.hough_voting_gpu(sc["label"], sc["vertex"], sc["extents"], sc["meta"], sc["gt"], 1, -1.0, 0.02, 10)
    box, pose, target, weight, domain = outs
    assert box.shape[0] % 9 == 0 and box.shape[0] >= 9
    for g in range(box.shape[0] // 9):
        base = box[9 * g]
        ww, hh = base[4] - base[2], base[5] - base[3]
        for j in range(1, 9):
            r = box[9 * g + j]
            assert r[0] == base[0] and r[1] == base[1] and r[6] == base[6]
            np.testing.assert_allclose([r[4] - r[2], r[5] - r[3]], [ww, hh], rtol=1e-5)
            assert abs(abs(r[2] - base[2]) / ww - 0.05) < 1e-4 or r[2] == base[2]
        np.testing.assert_array_equal(pose[9 * g:9 * g + 9], np.repeat(pose[9 * g:9 * g + 1], 9, 0))
        cls = int(base[1])
        # the synthetic gt pose projects onto the planted ellipse -> IoU > 0.2 -> target = gt quaternion
        gt_row = [r for r in sc["gt"] if int(r[1]) == cls][0]
        np.testing.assert_allclose(target[9 * g, 4 * cls:4 * cls + 4], gt_row[6:10])
        assert weight[9 * g:9 * g + 9, 4 * cls:4 * cls + 4].all() and weight.sum() <= box.shape[0] * 4
    assert not domain.any()
    outs0 = oracle.hough_voting_gpu(sc["label"], sc["vertex"], sc["extents"], sc["meta"], None, 1, -1.0, 0.02, 10)
    assert outs0[4].all() and not outs0[3].any()      # num_gt == 0 -> domain flag 1 (.cu.cc:433-436)


def test_oracle_roi_pool_properties():
    rng = np.random.default_rng(0)
    data = rng.standard_normal((2, 12, 16, 8)).astype(np.float32)
    rois = synth.make_rois(6, 2, height=96, width=128, num_classes=5, seed=1)
    top, arg = oracle.roi_pool(data, rois, 7, 7, 1.0 / 8.0)
    assert top.shape == (6, 7, 7, 8) and arg.dtype == np.int32
    flat = data.reshape(2, -1)
    for n in range(6):
        b = int(rois[n, 0])
        m = arg[n] >= 0
        np.testing.assert_array_equal(top[n][m], flat[b][arg[n][m]])     # value at argmax
        assert (top[n][~m] == 0).all()                                   # empty bins -> 0, argmax -1
        assert ((arg[n][m] % 8) == np.broadcast_to(np.arange(8), arg[n].shape)[m]).all()  # channel preserved
    g = rng.standard_normal(top.shape).astype(np.float32)
    gin = oracle.roi_pool_grad(data, rois, arg, g, 7, 7, 1.0 / 8.0)
    np.testing.assert_allclose(gin.sum(), g[arg >= 0].sum(), rtol=1e-4)  # every pooled gradient lands somewhere


def test_oracle_hard_label():
    rng = np.random.default_rng(1)
    prob = rng.random((1, 5, 7, 4)).astype(np.float32)
    gt = rng.integers(-1, 4, (1, 5, 7)).astype(np.int32)
    out = oracle.hard_label(prob, gt, 0.5)
    assert set(np.unique(out)) <= {0.0, 1.0} and (out.sum(-1) <= 1).all()
    exp = np.zeros_like(prob)
    for idx in np.ndindex(1, 5, 7):
        g = gt[idx]
        if g != -1 and (g > 0 or prob[idx][g] < 0.5):
            exp[idx][g] = 1
    np.testing.assert_array_equal(out, exp)
    assert (oracle.hard_label(prob, gt, 1.0)[gt == 0][:, 0] == 1).all()   # threshold 1.0 (lov_color_2d.yml:26)


def test_oracle_project_backproject_consistency():
    case = synth.make_projection_case(1, 24, 32, 4, 3, 16, seed=4)
    out, amb = oracle.project(case["vox"], case["depth"], case["meta"], return_ambig=True)
    assert out.shape == (1, 24, 32, 4)
    # every non-zero output pixel equals some voxel of the grid (gather), zeros where the ray leaves the grid
    voxset = {tuple(np.round(v, 6)) for v in case["vox"].reshape(-1, 4)}
    nz = out.reshape(-1, 4)[np.abs(out.reshape(-1, 4)).sum(1) > 0]
    assert len(nz) > 100 and all(tuple(np.round(v, 6)) in voxset for v in nz[:200])
    td, tl, tf = oracle.backproject(case["data"], case["label"], case["depth"], case["meta"], case["label_3d"], 16, 3, 0.02)
    assert td.shape == (1, 16, 16, 16, 4) and tl.shape == (1, 16, 16, 16, 3) and tf.shape == td.shape
    assert set(np.unique(tf)) <= {0.0, 1.0}
    empty = tf[..., 0] == 0
    np.testing.assert_array_equal(tl[empty], case["label_3d"][empty])      # fallback to label_3d
    assert (td[empty] == 0).all()


def test_oracle_average_distance_properties():
    pts = synth.make_model_points(22, 200)
    sym = synth.LOV_SYMMETRY
    pred, targ, wt = synth.make_pose_batch(8, 22, seed=3)
    loss, diff = oracle.average_distance_loss(pred, targ, wt, pts, sym, 0.01)
    assert loss.shape == (1,) and diff.shape == pred.shape and loss[0] >= 0
    assert (diff[wt == 0] == 0).all()
    # identical prediction and target -> zero distance -> below the margin -> zero loss and gradient
    loss0, diff0 = oracle.average_distance_loss(targ, targ, wt, pts, sym, 0.01)
    assert loss0[0] == 0 and not diff0.any()
    # finite-difference check of d loss / d q on a non-symmetric class with margin 0
    n = [i for i in range(8) if wt[i].any() and sym[int(np.argmax(wt[i]) // 4)] == 0][0]
    c = int(np.argmax(wt[n]) // 4)
    l0, d0 = oracle.average_distance_loss(pred, targ, wt, pts, sym, 0.0)
    for k in range(4):
        p2 = pred.copy(); p2[n, 4 * c + k] += 1e-3
        l1, _ = oracle.average_distance_loss(p2, targ, wt, pts, sym, 0.0)
        fd = (l1[0] - l0[0]) / 1e-3
        assert abs(fd - d0[n, 4 * c + k]) < 5e-3 * max(1.0, abs(fd)), (k, fd, d0[n, 4 * c + k])


def test_cpu_hough_ransac_config0():
    """BASELINE configs[0]: the reference's CPU hough_voting_layer (RANSAC, restated in oracle/cpu_hough_ransac.cpp) on
    one synthetic 640x480 frame with 2 classes: planted centre within 2 px, t_z (mean LOG depth, the reference's own
    quirk: ransac.h:105-116 has no exp) within 2 %, bit-identical across runs at 1 thread (mt19937 seed 1305)."""
    from oracle import cpu_hough
    sc = synth.make_scene(batch=1, height=480, width=640, num_classes=2, seed=1234 + 1000 * 0, dir_noise=0.02)
    (b, cls, cx, cy, z), = sc["centers"]
    box, pose = cpu_hough.hough_voting(sc["label"], sc["vertex"], sc["extents"], sc["meta"], is_train=0, threads=1)
    assert box.shape == (1, 6) and int(box[0, 0]) == 0 and int(box[0, 1]) == 1
    x, y = 0.5 * (box[0, 2] + box[0, 4]), 0.5 * (box[0, 3] + box[0, 5])
    assert abs(x - cx) <= 2.0 and abs(y - cy) <= 2.0
    assert abs(pose[0, 6] - np.log(z)) <= 0.02 * abs(np.log(z)) + 1e-3
    np.testing.assert_allclose(pose[0, :4], [1, 0, 0, 0])
    box2, pose2 = cpu_hough.hough_voting(sc["label"], sc["vertex"], sc["extents"], sc["meta"], is_train=0, threads=1)
    np.testing.assert_array_equal(box, box2); np.testing.assert_array_equal(pose, pose2)
    # nothing above minArea -> the CPU op's dummy row has cls = -1 (hough_voting_op.cc:208-222)
    empty = np.zeros_like(sc["label"])
    b0, p0 = cpu_hough.hough_voting(empty, sc["vertex"], sc["extents"], sc["meta"])
    assert b0.shape == (1, 6) and b0[0, 1] == -1
    # train mode: 9 jittered rows per detection (hough_voting_op.cc:790-855)
    bt, pt = cpu_hough.hough_voting(sc["label"], sc["vertex"], sc["extents"], sc["meta"], is_train=1, threads=1)
    assert bt.shape[0] % 9 == 0 and bt.shape[0] >= 9   # train mode keeps all surviving hypotheses (refSteps < 4 rule)
    ww, hh = bt[0, 4] - bt[0, 2], bt[0, 5] - bt[0, 3]
    np.testing.assert_allclose(bt[1:9, 4] - bt[1:9, 2], ww, rtol=1e-5); np.testing.assert_allclose(bt[1:9, 5] - bt[1:9, 3], hh, rtol=1e-5)


def test_result_records_roundtrip(tmp_path):
    """Record layout handed to ICP / the .mat writer (lib/fcn/test.py:1327-1351,1415-1423, lov.py:431-438)."""
    import scipy.io
    from posecnn_b200.utils import results
    rec = np.zeros((8, 15), np.float32)
    rec[0] = [1, 5, 10, 20, 110, 220, 900, 1, 0, 0, 0, 0.1, 0.2, 0.9, 1]
    rec[1] = [0, 3, 30, 40, 90, 100, 700, 0.5, 0.5, 0.5, 0.5, -0.1, 0.0, 1.1, 1]
    rec[2] = [1, 7, 50, 60, 70, 80, 500, 0, 1, 0, 0, 0.0, 0.3, 0.7, 1]
    per_image = results.split_detections(rec, batch=2)
    assert [r.shape[0] for r, _ in per_image] == [1, 2]
    rois, poses = per_image[1]
    assert rois[:, 1].tolist() == [5.0, 7.0] and poses[1].tolist() == rec[2, 7:14].tolist()
    seg = results.segmentation_record(np.zeros((480, 640), np.int32), rois, poses)
    assert sorted(seg) == ["labels", "poses", "poses_icp", "poses_refined", "rois"] and seg["poses_icp"].shape == (2, 7)
    p = results.icp_parameters([[1066.778, 0, 312.9869], [0, 1067.487, 241.3109], [0, 0, 1]], 10000.0)
    np.testing.assert_allclose(p, [1066.778, 1067.487, 312.9869, 241.3109, 0.25, 6.0, 10000.0], rtol=1e-6)
    f = str(tmp_path / "000001.mat")
    results.save_mat(f, seg)
    back = scipy.io.loadmat(f)
    np.testing.assert_array_equal(back["rois"], rois)
    np.testing.assert_array_equal(back["poses"], poses)
    assert back["labels"].shape == (480, 640)


def test_bench_reference_arm_prints_one_json_line():
    """bench.py --impl reference (the CPU arm the driver launches next to ours): exactly one JSON line on stdout with
    the contract's keys, nothing from /root/reference needed at run time."""
    import json
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    p = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1"],
                       capture_output=True, text=True, timeout=600, cwd=root)
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [l for l in p.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, lines
    d = json.loads(lines[0])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "config", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["impl"] == "reference" and d["value"] > 0 and d["cpu_baseline"]["cores"] >= 1 and d["e2e"]["value"] == d["value"]


# lib/networks/network.py:6-26, verbatim
NETWORK_PY_IMPORTS = """\
import backprojecting_layer.backprojecting_op as backproject_op
import backprojecting_layer.backprojecting_op_grad
import projecting_layer.projecting_op as project_op
import projecting_layer.projecting_op_grad
import computing_label_layer.computing_label_op as compute_label_op
import computing_flow_layer.computing_flow_op as compute_flow_op
import computing_flow_layer.computing_flow_op_grad
import triplet_loss.triplet_loss_op as triplet_loss_op
import triplet_loss.triplet_loss_op_grad
import average_distance_loss.average_distance_loss_op as average_distance_loss_op
import average_distance_loss.average_distance_loss_op_grad
import hough_voting_layer.hough_voting_op as hough_voting_op
import hough_voting_layer.hough_voting_op_grad
import hough_voting_gpu_layer.hough_voting_gpu_op as hough_voting_gpu_op
import hough_voting_gpu_layer.hough_voting_gpu_op_grad
import roi_pooling_layer.roi_pooling_op as roi_pool_op
import roi_pooling_layer.roi_pooling_op_grad
import gradient_reversal_layer.gradient_reversal_op as gradient_reversal_op
import gradient_reversal_layer.gradient_reversal_op_grad
import hard_label_layer.hard_label_op as hard_label_op
import hard_label_layer.hard_label_op_grad
"""
# sha256 of lines 6-26 of the reference's lib/networks/network.py (newline-terminated), taken from the file itself
NETWORK_PY_IMPORTS_SHA256 = "c9cf9ad65096914c4b85d5c10480df5f85f7a3050d33cd36294d9d8b6a0bd79a"

# the op symbols lib/networks/network.py calls on those modules (network.py:226-340)
NETWORK_PY_SYMBOLS = {
    "backproject_op": ["backproject", "backproject_grad"], "project_op": ["project", "project_grad"],
    "compute_label_op": ["compute_label"], "compute_flow_op": ["compute_flow", "compute_flow_grad"],
    "triplet_loss_op": ["triplet_loss", "triplet_loss_grad"],
    "average_distance_loss_op": ["average_distance_loss", "average_distance_loss_grad"],
    "hough_voting_op": ["hough_voting", "hough_voting_grad"],
    "hough_voting_gpu_op": ["hough_voting_gpu", "hough_voting_gpu_grad"], "roi_pool_op": ["roi_pool", "roi_pool_grad"],
    "gradient_reversal_op": ["gradient_reversal", "gradient_reversal_grad"], "hard_label_op": ["hard_label", "hard_label_grad"],
}


def test_reference_import_paths_resolve():
    """Replays EVERY op import statement of lib/networks/network.py:6-26 verbatim with posecnn_b200/ on sys.path (the
    way the reference puts lib/ on it, tools/_init_paths.py): all 21 must resolve, every symbol network.py uses must be
    callable, and the out-of-scope ops (SURVEY.md §8(b) stubs) must fail loudly when called instead of falling back."""
    import hashlib
    import subprocess
    import sys
    assert hashlib.sha256(NETWORK_PY_IMPORTS.encode()).hexdigest() == NETWORK_PY_IMPORTS_SHA256
    prog = (
        "import sys; sys.path.insert(0, %r); sys.path.insert(0, %r)\n" % (ROOT, os.path.join(ROOT, "posecnn_b200"))
        + NETWORK_PY_IMPORTS
        + "syms = %r\n" % NETWORK_PY_SYMBOLS
        + "for m, names in syms.items():\n"
        + "    for n in names:\n"
        + "        assert callable(getattr(globals()[m], n)), (m, n)\n"
        + "for m, n in (('compute_label_op', 'compute_label'), ('compute_flow_op', 'compute_flow'), ('triplet_loss_op', 'triplet_loss'),\n"
        + "             ('gradient_reversal_op', 'gradient_reversal'), ('hough_voting_op', 'hough_voting')):\n"
        + "    try:\n"
        + "        getattr(globals()[m], n)(None, None, None, None, None, 0)\n"
        + "    except NotImplementedError:\n"
        + "        continue\n"
        + "    raise SystemExit('stub %s.%s did not raise' % (m, n))\n"
        + "print('IMPORTS_OK')\n")
    out = subprocess.run([sys.executable, "-c", prog], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0 and "IMPORTS_OK" in out.stdout, out.stderr[-2000:]


def test_dgrad_weight_transform_matches_autograd():
    """Host logic for the backward-data pass (DESIGN.md plan item 3): the forward kernel on tap-flipped, channel-transposed
    weights computes d x.  Checked on CPU: F.conv2d with the transformed weights == torch.autograd of the forward conv."""
    import torch
    import torch.nn.functional as F
    from posecnn_b200 import conv
    g = torch.Generator().manual_seed(0)
    for k, ci, co in ((3, 8, 16), (1, 16, 8)):
        w = torch.randn((k, k, ci, co), generator=g)                       # HWIO, network.py:166-170
        x = torch.randn((2, ci, 9, 11), generator=g, requires_grad=True)
        y = F.conv2d(x, w.permute(3, 2, 0, 1), padding=k // 2)
        dy = torch.randn(y.shape, generator=g)
        y.backward(dy)
        wt = conv.hwio_to_tc_dgrad(w).float()                               # [Cin][k*k*Cout], K order (tap, cout)
        assert wt.shape == (ci, k * k * co)
        w_d = wt.reshape(ci, k, k, co).permute(0, 3, 1, 2)                   # OIHW of the dgrad convolution
        dx = F.conv2d(dy.to(torch.bfloat16).float(), w_d, padding=k // 2)    # what conv_bf16(dy, wt, 0, k, relu=False) computes
        assert torch.allclose(dx, x.grad, rtol=2e-2, atol=2e-2 * x.grad.abs().max().item())
        exact = F.conv2d(dy, torch.flip(w, (0, 1)).permute(2, 3, 0, 1), padding=k // 2)   # same transform in fp32: exact
        assert torch.allclose(exact, x.grad, rtol=1e-4, atol=1e-4)


def test_blob_helpers():
    """Host halves of the input pre-processing (lib/utils/blob.py:48-71, lib/fcn/test.py:72-76)."""
    from posecnn_b200.utils import blob
    rng = np.random.default_rng(0)
    im = rng.integers(0, 256, (37, 53, 3), dtype=np.uint8)
    p = blob.pad_im(im, 16)
    assert p.shape == (48, 64, 3) and (p[:37, :53] == im).all() and not p[37:].any() and not p[:, 53:].any()
    want = np.pad(im, ((0, 11), (0, 11), (0, 0)), "constant", constant_values=0)          # what np.lib.pad does in the reference
    np.testing.assert_array_equal(p, want)
    assert blob.pad_im(im[:, :, 0], 16, value=7).shape == (48, 64) and blob.pad_im(p, 16).shape == p.shape
    assert blob.unpad_im(p, 16).shape == p.shape                                             # the reference's unpad: no-op on padded sizes
    cb = blob.color_blob([im, im[:20, :30]])
    assert cb.shape == (2, 48, 64, 3) and cb.dtype == np.uint8 and (cb[1, :20, :30] == im[:20, :30]).all()
    assert np.abs(cb[0, 40, 60].astype(np.float32) - blob.PIXEL_MEANS).max() <= 0.5          # padded pixels ~ zero after mean subtraction
    d = rng.integers(0, 6000, (37, 53)).astype(np.uint16)
    db = blob.depth_blob([d])
    ref = np.clip(d.astype(np.float32) / 2000.0, 0, 1) * 255
    ref = np.tile(ref[:, :, np.newaxis], (1, 1, 3)) - blob.PIXEL_MEANS                       # test.py:72-76
    np.testing.assert_array_equal(db[0, :37, :53], ref.astype(np.float32))
    assert db.shape == (1, 48, 64, 3) and not db[0, 37:].any()
