"""Generate tests/golden/*.npz by running the REFERENCE'S OWN CUDA kernels
(oracle/_ref/libposecnn_ref.so = /root/reference/lib/*/*_gpu.cu.cc compiled unmodified for
sm_100a behind oracle/ref_shim) on the GPU box.

    gpurun -- 'python tests/golden/make_golden.py gpurun_out/golden'
    cp gpurun_out/golden/*.npz tests/golden/

The Hough vectors use the canonical list order (oracle/ref_driver.cu: ref_hough_canonical);
vote planes are stored as int16 (full planes for the small cases, row/column marginals +
arg-max for the 640x480 case)."""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import ref  # noqa: E402
from tests.golden import cases  # noqa: E402


def main(out_dir):
    os.makedirs(out_dir, exist_ok=True)
    dev = torch.device("cuda:0")
    T = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    N = lambda t: t.detach().cpu().numpy()
    for name in cases.HOUGH_CASES:
        sc, is_train, vt, pt, skip = cases.hough_inputs(name)
        gt = T(sc["gt"]) if len(sc["gt"]) else None
        outs, nr, votes = ref.hough_canonical(T(sc["label"]), T(sc["vertex"]), T(sc["extents"]), T(sc["meta"]), gt,
                                              is_train, vt, pt, skip)
        v = N(votes)
        d = dict(box=N(outs[0]), pose=N(outs[1]), target=N(outs[2]), weight=N(outs[3]), domain=N(outs[4]),
                 num_rois=np.int32(nr), row_sum=v.sum(3).astype(np.int32), col_sum=v.sum(2).astype(np.int32),
                 plane_max=v.reshape(v.shape[0], v.shape[1], -1).max(2).astype(np.int32),
                 plane_argmax=v.reshape(v.shape[0], v.shape[1], -1).argmax(2).astype(np.int32))
        if v.shape[2] * v.shape[3] <= 160 * 120:
            d["votes"] = v.astype(np.int16)
        np.savez_compressed(os.path.join(out_dir, name + ".npz"), **d)
        print(name, "rows", nr, "max votes", v.max())
    # the reference launcher as shipped (atomicAdd list order): with skip_pixels = 1 every pixel votes, so its rows
    # are order independent as a set
    sc, _, vt, pt, _ = cases.hough_inputs("h_skip1_d")
    outs, nr = ref.hough_full(T(sc["label"]), T(sc["vertex"]), T(sc["extents"]), T(sc["meta"]), T(sc["gt"]), 0, vt, pt, 1)
    np.savez_compressed(os.path.join(out_dir, "h_skip1_d_shipped.npz"), box=N(outs[0]), pose=N(outs[1]), target=N(outs[2]),
                        weight=N(outs[3]), domain=N(outs[4]), num_rois=np.int32(nr))
    print("h_skip1_d_shipped rows", nr)
    data, rois, grad = cases.roi_inputs()
    top, arg = ref.roi_pool(T(data), T(rois), 7, 7, 1.0 / 16.0, 0)
    gin = ref.roi_pool_grad(T(data), T(rois), arg, T(grad), 7, 7, 1.0 / 16.0, 0)
    topc, argc = ref.roi_pool(T(data), T(rois), 7, 7, 1.0 / 16.0, 1)
    np.savez_compressed(os.path.join(out_dir, "roi_pool.npz"), top=N(top), argmax=N(arg), grad_in=N(gin), top_cls=N(topc),
                        argmax_cls=N(argc))
    prob, gtl = cases.hard_label_inputs()
    np.savez_compressed(os.path.join(out_dir, "hard_label.npz"),
                        **{f"thr_{t}": N(ref.hard_label(T(prob), T(gtl), t)).astype(np.uint8) for t in (1.0, 0.5)})
    c = cases.projection_inputs()
    td, tl, tf = ref.backproject(T(c["data"]), T(c["label"]), T(c["depth"]), T(c["meta"]), T(c["label_3d"]), 16, 3, 0.02)
    pj = ref.project(T(c["vox"]), T(c["depth"]), T(c["meta"]))
    bg = ref.backproject_grad(T(c["g3"]), T(c["depth"]), T(c["meta"]), 48, 64)
    pg = ref.project_grad(T(c["g2"]), T(c["depth"]), T(c["meta"]), 16, 3, 0.02)
    np.savez_compressed(os.path.join(out_dir, "projection.npz"), top_data=N(td), top_label=N(tl), top_flag=N(tf).astype(np.uint8),
                        project=N(pj), backproject_grad=N(bg), project_grad=N(pg))
    pred, targ, wt, pts, sym = cases.avgdist_inputs()
    loss, diff = ref.average_distance_loss(T(pred), T(targ), T(wt), T(pts), T(sym), 0.01)
    np.savez_compressed(os.path.join(out_dir, "average_distance.npz"), loss=N(loss), diff=N(diff))
    print("golden vectors written to", out_dir)


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "gpurun_out", "golden"))
