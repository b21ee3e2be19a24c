#!/usr/bin/env python
"""bench.py — frames/s of the PoseCNN hot path on synthetic 640x480 batches (BASELINE.json).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload full|hough|rgbd|project|train] [--batch B]
                    [--dump-outputs DIR]
    python bench.py --impl reference ...      # the same path restated on the host cores (oracle/cpu_pipeline.py)

One JSON line on stdout (rank 0).  A "step" is one pass of the hot path over ONE GLOBAL batch of `--batch` synthetic
frames: with N GPUs the batch is cut into contiguous image shards (strong scaling, SURVEY.md §8(e): index_size =
128 / B_global, global batch indices, one NCCL all-gather of the pose-hypothesis records per step); the weak-scaling
figure (a full batch per GPU) is reported beside it in `weak`.  Device time is measured with CUDA events on the
launching stream; clocks are sampled with nvidia-smi during the timed region.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

H, W, C = 480, 640, 22
HOUGH_BYTES_PER_FRAME = H * W * 4 * (1 + 3 * C) + 48 * 4 + C * 12  # SURVEY §8(d): label + vertex_pred + meta + extents
VGG_FLOP_PER_FRAME = 187.918e9  # sum of 2*M*K*N over conv1_1..conv5_3 (SURVEY §8(d))
METRIC_FULL = "frames/sec on 640x480 RGB, 21 classes, batch 32 (VGG16 + Hough + ROI pose head)"
# kernels of one step's CUDA graph: trunk 14 (conv1 fused, 12 conv of which 3 with fused pool, pool4) + 1x1 heads 4 +
# lowres_heads + up8_heads + hough 7 + roi_pool_pair + 3 x (fc_tc + fc_finish) + nms_pose
LAUNCHES_FULL = 14 + 4 + 2 + 7 + 1 + 6 + 1
TRAIN_OWN_LAUNCHES_PER_STEP = 209   # own kernels of one training step (ncu launch list); the run counts them live with CUPTI when it can


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm_gbs=d["hbm_gbs"], bf16_tflops=d["bf16_tflops"], bf16_tflops_sustained=d.get("bf16_tflops_sustained"),
                    source="measured (MEASURED_PEAKS.json)")
    return dict(hbm_gbs=6650.0, bf16_tflops=1590.0, bf16_tflops_sustained=1400.0, source="fallback (B200_PROFILING.md)")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx, self.rows, self.proc = gpu_index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.idx)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc is None:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["nvidia-smi unavailable"])
        time.sleep(0.15)
        self.proc.terminate()
        sm = [float(r[1]) for r in self.rows if len(r) >= 9 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) >= 9 and r[2].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            if len(r) >= 9:
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
        return dict(sm_mhz=float(np.median(sm)) if sm else None, sm_max_mhz=max(mx) if mx else None,
                    reasons=sorted(reasons), samples=len(sm))


def dist_setup(n_gpus):
    import torch
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")   # NCCL prints its version line on stdout otherwise
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    else:
        torch.cuda.set_device(0)
    return rank, world, local


def barrier(world):
    if world > 1:
        import torch.distributed as dist
        dist.barrier()


def max_over_ranks(x, world):
    if world > 1:
        import torch
        import torch.distributed as dist
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())
    return float(x)


def count_own_launches(fn):
    """Kernels of THIS repo launched by one call of fn(), counted with CUPTI through torch.profiler (every kernel on the device is
    seen, also those launched through the C ABI); ATen / NCCL / memcpy / memset activities are not counted.  None if the profiler
    is unavailable."""
    try:
        import torch
        from torch.profiler import ProfilerActivity, profile
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            fn()
            torch.cuda.synchronize()
        own = other = 0
        per = {}
        for ev in prof.events():
            if ev.device_type != torch.autograd.DeviceType.CUDA:
                continue
            n = ev.name
            if n.startswith(("Memcpy", "Memset")) or "nccl" in n.lower():
                continue
            if "at::" in n or "cub::" in n or n.startswith(("void at", "nvjet", "cutlass", "sm90", "sm100")):
                other += 1
                key = "library (ATen)"
            else:
                own += 1
                key = n.split("(")[0].replace("void ", "")[:48]
            a = per.setdefault(key, [0.0, 0])
            a[0] += float(getattr(ev, "device_time", 0.0) or getattr(ev, "cuda_time", 0.0)) / 1e3
            a[1] += 1
        top = sorted(per.items(), key=lambda kv: -kv[1][0])[:16]
        return dict(own=own, library=other, kernel_ms_top={k: [round(v[0], 3), v[1]] for k, v in top},
                    kernel_ms_total=round(sum(v[0] for v in per.values()), 3)) if own + other > 0 else None
    except Exception as e:  # pragma: no cover
        print("launch count via torch.profiler failed: %s" % e, file=sys.stderr)
        return None


def profile_json(name):
    try:
        return json.load(open(os.path.join(ROOT, "profiles", name)))
    except Exception:
        return None


DUMP_BYTES = 60 * 1000 * 1000     # array data of --dump-outputs; with the .npy headers it stays under 64 MB
_OUTPUTS = None     # host copies of what the timed path returned in its last step (--dump-outputs)


def keep_outputs(named):
    """Copy the tensors of `named` (nested dicts flattened as `outer.inner`) to the host for --dump-outputs: float64 stays
    float64, everything else becomes float32.  Each array gets an equal share of DUMP_BYTES; a larger one is replaced
    by its elements at a fixed sample of flat indices (numpy default_rng(0).choice(numel, share, replace=False), sorted),
    so that two runs or two builds sample the same elements."""
    import torch
    flat = {}

    def walk(d, pre):
        for k, v in d.items():
            if isinstance(v, dict):
                walk(v, pre + k + ".")
            elif torch.is_tensor(v):
                flat[(pre + k).replace("/", "_")] = v.detach()
    walk(named, "")
    share = DUMP_BYTES // max(1, len(flat))
    global _OUTPUTS
    _OUTPUTS = {}
    for name, t in flat.items():
        dt = torch.float64 if t.dtype == torch.float64 else torch.float32
        k = share // dt.itemsize
        if t.numel() > k:
            idx = np.sort(np.random.default_rng(0).choice(t.numel(), k, replace=False))
            t = t.reshape(-1)[torch.from_numpy(idx).to(t.device)]
            name += ".sample"
        _OUTPUTS[name] = t.to(dt).cpu().numpy()
    return _OUTPUTS


def write_outputs(out_dir):
    os.makedirs(out_dir, exist_ok=True)
    for name, a in _OUTPUTS.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


# ------------------------------------------------------------------------------------------
# Hough workload: batch of synthetic label / vertex maps (SURVEY §8(d) scenes; configs[1] scaled to batch B)
# ------------------------------------------------------------------------------------------
HOUGH_UNIQUE_FRAMES = 8
_SCENES = {}


def hough_scenes(rank=0):
    """The 8 distinct §8(d) scenes every Hough figure of a run is measured on (GPU batches tile them; the CPU op runs
    the very same frames): seed 1234 + 1000 * config_id(1) + image index."""
    if rank not in _SCENES:
        from posecnn_b200 import synth
        _SCENES[rank] = synth.make_scene(batch=HOUGH_UNIQUE_FRAMES, height=H, width=W, num_classes=C, seed=1234 + 1000 * 1 + 100 * rank)
    return _SCENES[rank]


def hough_inputs(batch, rank):
    sc = hough_scenes(rank)
    reps = (batch + HOUGH_UNIQUE_FRAMES - 1) // HOUGH_UNIQUE_FRAMES
    tile = lambda a: np.concatenate([a] * reps, 0)[:batch]
    return dict(label=tile(sc["label"]), vertex=tile(sc["vertex"]), meta=tile(sc["meta"]), extents=sc["extents"])


def measure_hough(B, rank, world, local, steps, warmup, use_graph=True, e2e_batch=32, want_e2e=True, dump=False):
    """Device time of the Houghvotinggpu op alone (dense vertex_pred input, the registered op signature) on the §8(d)
    scenes: CUDA-graph replay of the one C call (7 launches + 1 memset node), L2 flushed between timed iterations."""
    import torch
    from posecnn_b200.hough_voting_gpu_layer import hough_voting_gpu_op as hop
    dev = torch.device("cuda", local)
    inp = hough_inputs(B, rank)
    label = torch.from_numpy(inp["label"]).to(dev)
    vertex = torch.from_numpy(inp["vertex"]).to(dev)
    meta = torch.from_numpy(inp["meta"]).to(dev)
    ext = torch.from_numpy(inp["extents"]).to(dev)
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)  # > 126 MB L2

    def step():
        return hop.hough_voting_gpu_capacity(label, vertex, ext, meta, None, 0, -1.0, 0.02, 10)

    for _ in range(max(warmup, 3)):
        out = step()
    torch.cuda.synchronize()
    graph = None
    if use_graph:
        try:
            side = torch.cuda.Stream(device=dev)
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                step()
            torch.cuda.current_stream().wait_stream(side)
            torch.cuda.synchronize()
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                out = step()
            graph.replay()
            torch.cuda.synchronize()
        except Exception as e:  # pragma: no cover - fall back to eager launches
            print("hough workload: CUDA graph capture failed (%s); timing eager launches" % e, file=sys.stderr)
            graph = None
    barrier(world)
    evs = []
    for _ in range(steps):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        if graph is not None:
            graph.replay()
        else:
            out = step()
        e1.record()
        evs.append((e0, e1))
    torch.cuda.synchronize()
    barrier(world)
    if dump:
        keep_outputs(dict(zip(("rois", "poses", "poses_target", "poses_weight", "domain", "num_rois", "status"), out)))
    ms = [a.elapsed_time(b) for a, b in evs]
    total_ms = max_over_ranks(float(np.sum(ms)), world)
    ms_step = total_ms / steps
    nrois = int(out[5].item())
    n_fg = int((label > 0).sum().item())
    res = dict(batch=B, device_ms=ms_step, frames_per_s=B * world / (ms_step * 1e-3), rois=nrois, cuda_graph=graph is not None,
               footprint_gbs=HOUGH_BYTES_PER_FRAME * B / (ms_step * 1e-3) / 1e9,
               compulsory_bytes_per_frame=4 * H * W + 12 * n_fg // B, foreground_fraction=n_fg / float(B * H * W))

    # end to end through the public op with HOST buffers: pinned H2D of label + vertex + meta, D2H of the rows
    if want_e2e:
        eb = min(B, e2e_batch)
        h_label = torch.from_numpy(inp["label"][:eb]).pin_memory()
        h_vertex = torch.from_numpy(inp["vertex"][:eb]).pin_memory()
        h_meta = torch.from_numpy(inp["meta"][:eb]).pin_memory()
        d_label, d_vertex, d_meta = torch.empty_like(label[:eb]), torch.empty_like(vertex[:eb]), torch.empty_like(meta[:eb])
        h_box = torch.empty((1152, 7), dtype=torch.float32).pin_memory()
        h_pose = torch.empty((1152, 7), dtype=torch.float32).pin_memory()
        h_n = torch.empty((1,), dtype=torch.int32).pin_memory()

        def e2e_step():
            d_label.copy_(h_label, non_blocking=True)
            d_vertex.copy_(h_vertex, non_blocking=True)
            d_meta.copy_(h_meta, non_blocking=True)
            o = hop.hough_voting_gpu_capacity(d_label, d_vertex, ext, d_meta, None, 0, -1.0, 0.02, 10)
            h_box.copy_(o[0], non_blocking=True)
            h_pose.copy_(o[1], non_blocking=True)
            h_n.copy_(o[5], non_blocking=True)
            torch.cuda.current_stream().synchronize()

        e2e_step()
        torch.cuda.synchronize()
        k = steps
        t0 = time.perf_counter()
        for _ in range(k):
            e2e_step()
        dt = max_over_ranks((time.perf_counter() - t0) / k, world)
        res["e2e"] = dict(value=eb * world / dt, unit="frames/s", batch_per_gpu=eb,
                          h2d_bytes_per_step=int(h_label.numel() * 4 + h_vertex.numel() * 4 + h_meta.numel() * 4),
                          d2h_bytes_per_step=int(h_box.numel() * 4 + h_pose.numel() * 4 + 4),
                          note="the op's registered inputs are the dense fp32 label / vertex_pred maps (82 MB/frame): e2e is the PCIe "
                               "upload of those maps")
    return res


def cpu_hough_same_frames():
    """The reference's CPU hough_voting_layer (RANSAC, oracle/cpu_hough_ransac.cpp) on the SAME 8 scenes."""
    try:
        from oracle import cpu_hough
    except Exception as e:  # pragma: no cover
        return dict(value=None, unit="frames/s", cores=0, kind="port", sample="unavailable: %s" % e)
    return cpu_hough.timed_on_scenes(hough_scenes(0))


def run_hough(args, rank, world, local):
    B = args.batch
    sampler = ClockSampler(local)
    sampler.start()
    rec = measure_hough(B, rank, world, local, args.steps, args.warmup, not args.no_graph, args.e2e_batch, not args.no_e2e,
                        args.dump_outputs and rank == 0)
    clocks = sampler.stop()
    peaks = measured_peaks()
    traffic = profile_json("r02_hough_traffic.json")
    res = dict(
        metric="frames/sec on 640x480, 21 classes (Hough voting op)", value=rec["frames_per_s"], unit="frames/s",
        n_gpus=world, steps=args.steps, warmup=max(args.warmup, 3), ms_per_step=rec["device_ms"], higher_is_better=True,
        scaling="weak", vs_baseline=None, dtype="f32/int32", data="synthetic",
        config=dict(workload="hough_voting_gpu batch %d x 640x480 x 22 classes (configs[1] at batch %d)" % (B, B),
                    global_batch=B * world, l2="flushed between timed iterations (256 MB write)", rois=rec["rois"],
                    cuda_graph=rec["cuda_graph"]),
        clocks=clocks, gpu_launches=7 * args.steps,
        roofline=dict(bound="hbm", achieved=rec["footprint_gbs"], peak=peaks["hbm_gbs"], unit="GB/s",
                      frac=rec["footprint_gbs"] / peaks["hbm_gbs"], traffic=(traffic or {}).get("dram_bytes_per_step_b%d" % B),
                      peak_source=peaks["source"],
                      note="achieved = op-boundary footprint 82.33 MB/frame (label + full vertex_pred) / whole-op device "
                           "time; the kernels read only the sampled pixels' 12 B, so >1.0 is possible (SURVEY §8(d))"),
    )
    if "e2e" in rec:
        res["e2e"] = rec["e2e"]
    return res


# ------------------------------------------------------------------------------------------
# Full workload (BASELINE configs[2]): VGG16 + heads + Hough + ROI pool + pose head + NMS, ONE global batch of B frames of
# 640x480, 22 classes, seeded random-init weights (Kaiming; the reference's sigma = 0.001 init yields all-background
# labels, SURVEY finding 10), synthetic uint8 images.
# ------------------------------------------------------------------------------------------
def make_network(dev, input_format="COLOR"):
    from posecnn_b200.networks.vgg16_convs import vgg16_convs
    return vgg16_convs(input_format=input_format, num_classes=C, device=dev).init_random(seed=0)


def rotating_inputs(h_img_np, dev, min_bytes=140 * 1024 * 1024, max_bufs=48):
    """Device-resident input batches that together exceed the 126 MB L2 (the timing rule's "inputs larger than L2"):
    the same frames rolled along the batch axis, so every buffer is a distinct tensor with identical statistics."""
    import torch
    nb = int(min(max_bufs, max(2, -(-min_bytes // h_img_np.nbytes))))
    return [torch.from_numpy(np.roll(h_img_np, k, axis=0).copy()).to(dev) for k in range(nb)]


def measure_pipeline(net, imgs_np, meta, ext, rank, world, dev, steps, warmup, batch_global, batch_offset, use_graph, want_e2e,
                     extra_inputs=None, dump=False):
    """K timed steps of the sharded pipeline: graph replay on the compute stream, records all-gathered on the
    communication stream (double-buffered), one event pair around the whole region, max over ranks."""
    import torch
    from posecnn_b200 import parallel
    from posecnn_b200.networks.vgg16_convs import GraphedForward
    B = imgs_np.shape[0]
    bufs = rotating_inputs(imgs_np, dev)
    kw = dict(dense_vertex=False, batch_global=batch_global, batch_offset=batch_offset)
    if extra_inputs:
        kw.update(extra_inputs)
    if use_graph:
        fwd = GraphedForward(net, bufs[0], meta, ext, pack_records=True, **kw)
        run = lambda x: fwd(x)
    else:
        def run(x):
            L = dict(net.forward(x, meta, ext, sync_rois=False, **kw))
            L["records"] = parallel.pack_detections(L)
            return L
    L = run(bufs[0])
    pipe = parallel.GatherPipeline(world, L["records"])

    def step(x):
        pipe.before_step()
        L = run(x)
        return pipe.submit(L["records"]), L

    for i in range(max(warmup, 3)):
        step(bufs[i % len(bufs)])
    pipe.drain()
    torch.cuda.synchronize()
    barrier(world)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(steps):
        last, L = step(bufs[i % len(bufs)])
    pipe.drain()
    e1.record()
    torch.cuda.synchronize()
    barrier(world)
    ms_step = max_over_ranks(e0.elapsed_time(e1) / steps, world)
    in_step_gather_ms = float(np.mean([pipe.last_gather_ms(last), pipe.last_gather_ms(last - 1)])) if steps >= 2 else None
    gathered = pipe.results(last)
    if dump:    # before anything below runs the step again and overwrites the graph's output buffers
        keep_outputs(dict(L, records_gathered=gathered))
    ndet = int((gathered[:, -1] > 0).sum().item())
    out = dict(ms_step=ms_step, layers=L, detections=ndet, nbufs=len(bufs), pipe=pipe, in_step_gather_ms=in_step_gather_ms, step=step,
               bufs=bufs)

    if want_e2e:
        # end to end through the public API with HOST buffers: every step uploads its own pinned uint8 batch (H2D) and
        # reads the gathered pose records back (D2H), all inside the timed region.  The upload of step i+1 runs on a copy
        # stream while step i computes (double-buffered device input), as a serving loop would do.
        h_img = torch.from_numpy(imgs_np).pin_memory()
        h_rec = [torch.empty(tuple(gathered.shape), dtype=torch.float32).pin_memory() for _ in range(2)]
        d_in = [torch.empty_like(bufs[0]) for _ in range(2)]
        copy_stream = torch.cuda.Stream(device=dev)
        up_done = [torch.cuda.Event() for _ in range(2)]
        consumed = [torch.cuda.Event() for _ in range(2)]
        main = torch.cuda.current_stream()

        def upload(i):
            b = i & 1
            with torch.cuda.stream(copy_stream):
                copy_stream.wait_event(consumed[b])       # the step that last read this buffer has finished with it
                d_in[b].copy_(h_img, non_blocking=True)
                up_done[b].record(copy_stream)

        def run_e2e(k):
            for b in range(2):
                consumed[b].record(main)
            upload(0)
            for i in range(k):
                b = i & 1
                if i + 1 < k:
                    upload(i + 1)
                main.wait_event(up_done[b])
                idx, _ = step(d_in[b])
                consumed[b].record(main)
                h_rec[b].copy_(pipe.results(idx), non_blocking=True)
            main.synchronize()

        run_e2e(2)
        barrier(world)
        k = steps               # wall clock over the timed steps; the first upload of the window cannot overlap anything
        t0 = time.perf_counter()
        run_e2e(k)
        dt = max_over_ranks((time.perf_counter() - t0) / k, world)
        out["e2e"] = dict(value=batch_global_frames(batch_global, B, world) / dt, unit="frames/s", h2d_bytes_per_step=int(h_img.numel()),
                          d2h_bytes_per_step=int(h_rec[0].numel() * 4),
                          note="pinned host uint8 images -> gathered pose records on the host, per rank; upload of step i+1 "
                               "overlapped with the compute of step i on a copy stream; wall clock over %d steps, max over ranks" % k)
    return out


def batch_global_frames(batch_global, local, world):
    """Frames one step processes across all ranks: the global batch when the ranks hold shards of it (strong), else
    world x local (independent full batches per rank, weak)."""
    return batch_global if batch_global != local or world == 1 else local * world


def run_full(args, rank, world, local, input_format="COLOR"):
    import torch
    from posecnn_b200 import parallel, synth
    dev = torch.device("cuda", local)
    Bg = args.batch
    off, Bl = parallel.shard_range(Bg, rank, world)
    if Bl < 1:
        raise SystemExit("--batch %d cannot be sharded over %d GPUs" % (Bg, world))
    net = make_network(dev, input_format)
    rgb_all, depth_all = synth.make_images(Bg, H, W, seed=21)                 # the ONE global batch, identical on every rank
    K = synth.intrinsics(H, W)
    meta_all = torch.from_numpy(np.stack([synth.make_meta(K)] * Bg)).to(dev)
    ext = torch.from_numpy(synth.extents_for(C)).to(dev)
    extra_probe, extra_shard, extra_weak = None, None, None
    if input_format == "RGBD":
        dm = torch.from_numpy((depth_all * 1000.0).astype(np.float32)).to(dev)        # depth image in millimetres (lib/fcn/test.py:70)
        extra_probe, extra_shard, extra_weak = dict(depth=dm[:8]), dict(depth=dm[off:off + Bl]), dict(depth=dm)
    probe = torch.from_numpy(rgb_all[:8]).to(dev)
    bg_shift = net.calibrate_background(probe, meta_all[:8], ext, 0.75, **(extra_probe or {}))  # identical on every rank
    del probe
    sampler = ClockSampler(local)
    sampler.start()  # nvidia-smi needs ~100 ms to produce its first sample: start before the warm-up steps
    m = measure_pipeline(net, rgb_all[off:off + Bl], meta_all[off:off + Bl], ext, rank, world, dev, args.steps, args.warmup, Bg, off,
                         not args.no_graph, not args.no_e2e, extra_shard, args.dump_outputs and rank == 0)
    clocks = sampler.stop()
    ms_step, L, e2e = m["ms_step"], m["layers"], m.get("e2e")
    nlabels = int((L["label_2d"] > 0).sum().item())

    # communication: one all-gather of [cap_rows, 15] f32 per rank and step, on the comm stream
    comm = None
    if world > 1:
        import torch.distributed as dist
        pipe = m["pipe"]
        rec = L["records"]
        torch.cuda.synchronize(); barrier(world)
        outb = torch.empty((world * rec.shape[0], rec.shape[1]), dtype=rec.dtype, device=dev)
        evs = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        for _ in range(5):
            dist.all_gather_into_tensor(outb, rec)
        evs[0].record()
        for _ in range(20):
            dist.all_gather_into_tensor(outb, rec)
        evs[1].record()
        torch.cuda.synchronize()
        ag_us = 1e3 * evs[0].elapsed_time(evs[1]) / 20
        evp = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        evp[0].record()
        for _ in range(10):
            parallel.pack_detections(L)
        evp[1].record()
        torch.cuda.synchronize()
        in_step = 1e3 * (m["in_step_gather_ms"] or 0.0)
        comm = dict(allgather_us=max_over_ranks(ag_us, world), allgather_in_step_us=max_over_ranks(in_step, world),
                    skew_us=max_over_ranks(max(0.0, in_step - ag_us), world), pack_us=1e2 * evp[0].elapsed_time(evp[1]),
                    payload_bytes_per_rank=int(rec.numel() * 4), stream="side stream, double-buffered against the next step's graph",
                    note="allgather_us: back-to-back collectives with the ranks in lockstep; allgather_in_step_us: the collective "
                         "inside the timed steps (waits for the slowest rank) — it runs under the NEXT step's compute, so "
                         "skew_us is hidden unless it exceeds a step; pack_us: eager launch of the packing ops (captured in "
                         "the step's graph in the timed path)")

    # dominant kernel class: the tensor-core conv stack of this rank's shard, timed alone with events
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)
    d_img = m["bufs"][0]
    tr = []
    for _ in range(args.steps):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); net._trunk(d_img); e1.record()
        torch.cuda.synchronize()
        tr.append(e0.elapsed_time(e1))
    trunk_ms = float(np.median(tr))
    ntrunks = 2 if input_format == "RGBD" else 1
    # Houghvotinggpu alone as the pipeline runs it (vertex head sampled from `lowres`) on the network's own label maps
    from posecnn_b200.hough_voting_gpu_layer import hough_voting_gpu_op as hop
    hs = []
    for _ in range(args.steps):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        hop.hough_voting_gpu_capacity(L["label_2d"], None, ext, meta_all[off:off + Bl], None, 0, -1.0, 0.02, 10, lowres=net._last_lowres,
                                      bias_vertex=net.params["vertex_pred/biases"], batch_global=Bg, batch_offset=off)
        e1.record()
        torch.cuda.synchronize()
        hs.append(e0.elapsed_time(e1))
    hough_net_ms = float(np.median(hs))
    del flush

    # weak scaling beside it: every rank runs a FULL batch of Bg frames (its own ROI budget of a batch of Bg), records gathered
    weak = None
    if world > 1 and not args.no_weak:
        del m
        torch.cuda.empty_cache()
        rgb_w, _ = synth.make_images(Bg, H, W, seed=21 + rank)
        mw = measure_pipeline(net, rgb_w, meta_all, ext, rank, world, dev, args.steps, args.warmup, Bg, 0, not args.no_graph, False,
                              extra_weak)
        weak = dict(scaling="weak", per_gpu_batch=Bg, global_batch=Bg * world, ms_per_step=mw["ms_step"],
                    value=Bg * world / (mw["ms_step"] * 1e-3), unit="frames/s",
                    note="every rank treats its %d frames as one reference batch (ROI budget 128 // %d per image); a GLOBAL batch of "
                         "%d frames would leave 128 // %d = %d ROIs per image under the reference's rule" % (Bg, Bg, Bg * world, Bg * world, 128 // (Bg * world)))
        del mw

    peaks = measured_peaks()
    tf = VGG_FLOP_PER_FRAME * Bl / (trunk_ms * 1e-3) / 1e12
    burst, sust = peaks["bf16_tflops"], peaks["bf16_tflops_sustained"] or peaks["bf16_tflops"]
    traffic = profile_json("r02_full_b32_trunk_traffic.json") or profile_json("r01_full_b32_trunk_traffic.json")
    res = dict(
        metric=METRIC_FULL if input_format == "COLOR" else "frames/sec on 640x480 RGB-D, 21 classes, batch 32 (two-trunk VGG16 + Hough + ROI pose head)",
        value=Bg / (ms_step * 1e-3),
        unit="frames/s", n_gpus=world, steps=args.steps, warmup=max(args.warmup, 3), ms_per_step=ms_step, higher_is_better=True,
        scaling="strong", vs_baseline=None,
        dtype="bf16 operands / fp32 accumulate (conv stack, 1x1 heads), fp16 operands / fp32 accumulate (fc6-fc8), fp32 / int32 elsewhere",
        data="synthetic",
        config=dict(workload=("configs[2]: full VGG16+Hough+ROI inference" if input_format == "COLOR" else
                              "configs[3] network: RGB-D two-trunk VGG16+Hough+ROI inference") +
                             ", random-init (Kaiming, seed 0) weights, ONE global batch of %d 640x480 uint8 BGR frames" % Bg,
                    global_batch=Bg, per_gpu_batch=Bl,
                    parallelism="contiguous image shards x%d of the global batch (index_size = 128 // %d, global batch indices), NCCL "
                                "all-gather of post-NMS pose records on a side stream" % (world, Bg),
                    l2="no flush: %d rotating device-resident input batches (%.0f MB > 126 MB L2) and %.1f GB of activations per step"
                       % (m_nbufs(Bl), m_nbufs(Bl) * Bl * H * W * 3 / 1e6, 0.172 * Bl * ntrunks),
                    detections_last_step=int(L["num_detections"].item()), cuda_graph=not args.no_graph,
                    dense_vertex_pred=False,
                    foreground_fraction=nlabels / float(Bl * H * W),
                    background_calibration="score/biases[0] += %.4g so that ~75%% of pixels are background (YCB-like fill); "
                                           "un-calibrated random init labels ~100%% of pixels foreground" % bg_shift),
        clocks=clocks, gpu_launches=(LAUNCHES_FULL + (14 if input_format == "RGBD" else 0)) * args.steps,
        roofline=dict(bound="tensor", achieved=tf, peak=burst, unit="TFLOP/s", frac=tf / burst, frac_sustained=tf / sust,
                      peak_sustained=sust, traffic=(traffic or {}).get("trunk_dram_bytes_per_launch_group") if (traffic or {}).get("batch") == Bl else None,
                      peak_source=peaks["source"] + ": burst cuBLAS bf16 (kernel group timed alone); frac_sustained = vs the sustained figure",
                      kernel="conv trunk: k_conv1_tc, k_conv_row2 x3, k_conv_tc<256> x9, 1 max-pool (3 pools fused)",
                      ms_per_launch_group=trunk_ms * ntrunks, frames_per_launch_group=Bl,
                      note="achieved = 187.918 GFLOP/frame x this rank's frames / device time of the conv trunk (13 tcgen05 launches, im2col "
                           "and three of the four max-pools fused into them), CUDA events, L2 flushed; BF16 operands, FP32 accumulation"),
        breakdown_ms=dict(step=ms_step, conv_trunk=trunk_ms * ntrunks, hough_on_network_maps=hough_net_ms),
        hough_on_network_maps=dict(ms=hough_net_ms, frames=Bl, footprint_gbs=HOUGH_BYTES_PER_FRAME * Bl / (hough_net_ms * 1e-3) / 1e9,
                                   frac=HOUGH_BYTES_PER_FRAME * Bl / (hough_net_ms * 1e-3) / 1e9 / peaks["hbm_gbs"],
                                   note="eager launches of the op as the pipeline runs it (vertex sampled from the 1/8-resolution head "
                                        "tensor, no dense vertex_pred) on the random-init network's own label maps, which are noise-like "
                                        "(fragmented classes, every class present): an upper bound on the op's cost; the SURVEY 8(d) "
                                        "scene figure is `hough` / `roofline_hough`"),
    )
    if e2e:
        res["e2e"] = e2e
    if comm:
        res["comm"] = comm
    if weak:
        res["weak"] = weak
    return res, net


def m_nbufs(Bl):
    return int(min(48, max(2, -(-140 * 1024 * 1024 // (Bl * H * W * 3)))))


# ------------------------------------------------------------------------------------------
# RGB-D geometry path (BASELINE configs[3]): Backproject + Project, ONE global batch of B frames sharded over the GPUs
# (per-image ops, no exchange at all), G = 128, Cf = 64, kernel_size 3, threshold 0.02 (SURVEY §8(d))
# ------------------------------------------------------------------------------------------
def run_project(args, rank, world, local):
    import torch
    from posecnn_b200 import parallel, synth
    from posecnn_b200.backprojecting_layer import backprojecting_op as bop
    from posecnn_b200.projecting_layer import projecting_op as pop
    dev = torch.device("cuda", local)
    Bg, G, Cf, ks, thr = args.batch, args.grid, 64, 3, 0.02
    off, Bl = parallel.shard_range(Bg, rank, world)
    case = synth.make_projection_case(min(Bl, 4), H, W, 4, 3, 8, seed=5 + rank)
    reps = -(-Bl // case["depth"].shape[0])
    depth = torch.from_numpy(np.concatenate([case["depth"]] * reps, 0)[:Bl]).to(dev)
    meta = torch.from_numpy(np.stack([synth.make_meta(synth.intrinsics(H, W), G)] * Bl)).to(dev)
    g = torch.Generator(device=dev).manual_seed(7 + rank)
    data = torch.randn((Bl, H, W, Cf), device=dev, generator=g)
    lab = torch.rand((Bl, H, W, C), device=dev, generator=g)
    l3 = torch.rand((Bl, G, G, G, C), device=dev, generator=g)

    def step():
        top_data, top_label, top_flag = bop.backproject(data, lab, depth, meta, l3, G, ks, thr)
        return pop.project(top_data, depth, meta, ks, thr)

    sampler = ClockSampler(local)
    sampler.start()
    for _ in range(max(args.warmup, 3)):
        out = step()
    torch.cuda.synchronize()
    barrier(world)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    tb0, tb1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        out = step()
    e1.record()
    torch.cuda.synchronize()
    barrier(world)
    clocks = sampler.stop()
    ms_step = max_over_ranks(e0.elapsed_time(e1) / args.steps, world)
    if args.dump_outputs and rank == 0:
        keep_outputs(dict(project=out))
    # the dominant kernel alone
    tb0.record()
    for _ in range(args.steps):
        td = bop.backproject(data, lab, depth, meta, l3, G, ks, thr)
    tb1.record()
    torch.cuda.synchronize()
    bp_ms = tb0.elapsed_time(tb1) / args.steps
    peaks = measured_peaks()
    bp_bytes = Bl * G ** 3 * (2 * Cf + C) * 4 + Bl * H * W * (Cf + C + 1) * 4
    pj_bytes = Bl * H * W * (4 + 8 * Cf)
    gbs = bp_bytes / (bp_ms * 1e-3) / 1e9
    e2e = None
    if not args.no_e2e:
        eb = min(Bl, 4)      # host staging of the 2-D inputs of 4 frames; the 3-D label grid stays resident (it is the op's state)
        h_data, h_lab, h_depth = data[:eb].cpu().pin_memory(), lab[:eb].cpu().pin_memory(), depth[:eb].cpu().pin_memory()
        d_data, d_lab, d_depth = torch.empty_like(data[:eb]), torch.empty_like(lab[:eb]), torch.empty_like(depth[:eb])
        h_out = torch.empty((eb, H, W, Cf), dtype=torch.float32).pin_memory()

        def e2e_step():
            d_data.copy_(h_data, non_blocking=True); d_lab.copy_(h_lab, non_blocking=True); d_depth.copy_(h_depth, non_blocking=True)
            td_, tl_, tf_ = bop.backproject(d_data, d_lab, d_depth, meta[:eb], l3[:eb], G, ks, thr)
            h_out.copy_(pop.project(td_, d_depth, meta[:eb], ks, thr), non_blocking=True)
            torch.cuda.current_stream().synchronize()

        e2e_step()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            e2e_step()
        dt = max_over_ranks((time.perf_counter() - t0) / args.steps, world)
        e2e = dict(value=eb * world / dt, unit="frames/s", batch_per_gpu=eb, h2d_bytes_per_step=int((h_data.numel() + h_lab.numel() + h_depth.numel()) * 4),
                   d2h_bytes_per_step=int(h_out.numel() * 4), note="pinned host feature / label / depth maps in, projected features out")
    res = dict(
        metric="frames/sec on 640x480 RGB-D (Backproject + Project, grid %d^3, 64 channels)" % G, value=Bg / (ms_step * 1e-3), unit="frames/s",
        n_gpus=world, steps=args.steps, warmup=max(args.warmup, 3), ms_per_step=ms_step, higher_is_better=True, scaling="strong",
        vs_baseline=None, dtype="f32", data="synthetic",
        config=dict(workload="configs[3]: backprojecting_layer + projecting_layer, ONE global batch of %d frames image-sharded x%d "
                             "(per-image ops: no collective), G = %d, Cf = 64, C = 22, kernel_size 3, threshold 0.02" % (Bg, world, G),
                    global_batch=Bg, per_gpu_batch=Bl,
                    l2="no flush: %.1f GB written and %.1f GB read per step on this rank (>> 126 MB L2)" % (bp_bytes / 1e9, (bp_bytes + pj_bytes) / 1e9)),
        clocks=clocks, gpu_launches=2 * args.steps,
        roofline=dict(bound="hbm", achieved=gbs, peak=peaks["hbm_gbs"], unit="GB/s", frac=gbs / peaks["hbm_gbs"], traffic=None,
                      peak_source=peaks["source"], kernel="k_backproject (dominant: %.2f of %.2f ms per step)" % (bp_ms, ms_step),
                      note="achieved = B*G^3*(2Cf+C)*4 written + B*H*W*(Cf+C+1)*4 read (SURVEY 8(d)) / kernel time"),
        breakdown_ms=dict(step=ms_step, backproject=bp_ms, project=ms_step - bp_ms),
    )
    if e2e:
        res["e2e"] = e2e
    return res


# ------------------------------------------------------------------------------------------
# Training step (BASELINE configs[4]): forward + backward + SGD-momentum update of the whole network with hard_label cross entropy,
# vertex smooth-L1 and average_distance_loss, ONE global batch of B frames sharded over the GPUs, gradients all-reduced over NCCL
# ------------------------------------------------------------------------------------------
def run_train(args, rank, world, local):
    import torch
    from posecnn_b200 import parallel, synth
    from posecnn_b200.networks.vgg16_convs import vgg16_convs
    from posecnn_b200.train import Trainer
    dev = torch.device("cuda", local)
    Bg = args.batch
    off, Bl = parallel.shard_range(Bg, rank, world)
    net = vgg16_convs(num_classes=C, device=dev, is_train=True, fold_vertex_head=False).init_random(seed=0)
    # O(1) logits / pre-activations, as a trained network has (a Kaiming-initialised output layer saturates softmax and tanh)
    net.params["score/weights"] *= 0.02; net.params["vertex_pred/weights"] *= 0.02; net.params["fc8/weights"] *= 0.01
    net.prepare()
    tr = Trainer(net, lr=1e-4, momentum=0.9, weight_decay=1e-4, vertex_w=1.0, vertex_w_inside=10.0, margin=0.01, world=world)
    nu = min(Bg, 8)
    sc = synth.make_scene(batch=nu, height=H, width=W, num_classes=C, seed=4234, other_channel_noise=False)
    reps = -(-Bg // nu)
    label_all = np.concatenate([sc["label"]] * reps, 0)[:Bg]
    centers = np.zeros((nu, C, 3), np.float32)
    for (b, cls, cx, cy, z) in sc["centers"]:
        centers[b, cls] = (cx, cy, z)
    centers_all = np.concatenate([centers] * reps, 0)[:Bg]
    gts = []
    for r_ in range(reps):
        g = sc["gt"].copy(); g[:, 0] += r_ * nu; gts.append(g)
    gt_all = np.concatenate(gts, 0); gt_all = gt_all[gt_all[:, 0] < Bg]
    rgb, _ = synth.make_images(Bg, H, W, seed=21)
    T = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    data, gtl, cen = T(rgb[off:off + Bl]), T(label_all[off:off + Bl]), T(centers_all[off:off + Bl])
    meta = T(np.stack([synth.make_meta(synth.intrinsics(H, W))] * Bl)); ext = T(synth.extents_for(C)); gtp = T(gt_all)
    pts = T(synth.make_model_points(C, 2620)); sym = T(synth.LOV_SYMMETRY)
    h_img = torch.from_numpy(rgb[off:off + Bl]).pin_memory(); h_lab = torch.from_numpy(label_all[off:off + Bl]).pin_memory()

    def step(d, l):
        return tr.step(d, l, cen, meta, ext, gtp, pts, sym, batch_global=Bg, batch_offset=off)

    sampler = ClockSampler(local)
    sampler.start()
    for _ in range(max(args.warmup, 3)):
        out = step(data, gtl)
    torch.cuda.synchronize(); barrier(world)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        out = step(data, gtl)
    e1.record()
    torch.cuda.synchronize(); barrier(world)
    clocks = sampler.stop()
    ms_step = max_over_ranks(e0.elapsed_time(e1) / args.steps, world)
    if args.dump_outputs and rank == 0:
        keep_outputs(out)
    # end to end: pinned host images + label maps in, the loss scalar out, every step; the upload of step i + 1 runs on a copy stream
    # while step i computes (double-buffered device inputs), as a training loop with a prefetching loader does
    d_in = [torch.empty_like(data) for _ in range(2)]
    l_in = [torch.empty_like(gtl) for _ in range(2)]
    h_loss = torch.empty((1,), dtype=torch.float32).pin_memory()
    copy_stream = torch.cuda.Stream(device=dev)
    up_done = [torch.cuda.Event() for _ in range(2)]
    consumed = [torch.cuda.Event() for _ in range(2)]
    main = torch.cuda.current_stream()

    def upload(i):
        b = i & 1
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(consumed[b])
            d_in[b].copy_(h_img, non_blocking=True); l_in[b].copy_(h_lab, non_blocking=True)
            up_done[b].record(copy_stream)

    def run_e2e(k):
        for b in range(2):
            consumed[b].record(main)
        upload(0)
        for i in range(k):
            b = i & 1
            if i + 1 < k:
                upload(i + 1)
            main.wait_event(up_done[b])
            o = step(d_in[b], l_in[b])
            consumed[b].record(main)
            h_loss.copy_(o["loss"], non_blocking=True)
        main.synchronize()

    run_e2e(2)                                    # first touch of the staging buffers, allocator growth
    barrier(world)
    k = args.steps
    t0 = time.perf_counter()
    run_e2e(k)
    dt = max_over_ranks((time.perf_counter() - t0) / k, world)
    launches = count_own_launches(lambda: step(data, gtl))
    peaks = measured_peaks()
    flop = 3.0 * VGG_FLOP_PER_FRAME * Bl                      # forward + input-gradient + weight-gradient GEMMs of the trunk
    tf = flop / (ms_step * 1e-3) / 1e12
    sust = peaks["bf16_tflops_sustained"] or peaks["bf16_tflops"]
    return dict(
        metric="frames/sec, training step (VGG16 + heads + Hough + ROI pose head, hard_label + vertex + average_distance losses, SGD momentum)",
        value=Bg / (ms_step * 1e-3), unit="frames/s", n_gpus=world, steps=args.steps, warmup=max(args.warmup, 3), ms_per_step=ms_step,
        higher_is_better=True, scaling="strong", vs_baseline=None,
        dtype="bf16 operands / fp32 accumulate (convolutions fwd + dgrad + wgrad), fp16 operands (fc6-fc8), fp32 master weights / losses", data="synthetic",
        config=dict(workload="configs[4]: training step, ONE global batch of %d 640x480 frames, synthetic YCB-shaped labels / poses, 22 classes, "
                             "keep_prob 1.0" % Bg, global_batch=Bg, per_gpu_batch=Bl,
                    parallelism="image shards x%d, global loss normalisers, per-tensor NCCL all-reduce (SUM) of the gradients on a side stream" % world,
                    l2="no flush: %.1f GB of saved activations per step (>> 126 MB L2)" % (0.31 * Bl), rois_rows=int(out["num_rois"].item()),
                    losses=dict(cls=float(out["loss_cls"].item()), vertex=float(out["loss_vertex"].item()), pose=float(out["loss_pose"].item()))),
        clocks=clocks, gpu_launches=(launches["own"] if launches else TRAIN_OWN_LAUNCHES_PER_STEP) * args.steps,
        launches_per_step=launches or dict(own=TRAIN_OWN_LAUNCHES_PER_STEP, source="ncu launch list profiles/r02_train_b16_launches.csv"),
        roofline=dict(bound="tensor", achieved=tf, peak=sust, unit="TFLOP/s", frac=tf / sust, traffic=None, peak_source=peaks["source"] + " (sustained: a kernel "
                      "group inside a long step)", kernel="trunk GEMMs: 13 forward convolutions + 12 dgrad (k_conv_tc / k_conv_row2) + 12 wgrad (k_wgrad_tc)",
                      note="achieved = 3 x 187.918 GFLOP/frame x this rank's frames / WHOLE step time (heads, losses, pose head, update included)"),
        e2e=dict(value=Bg / dt, unit="frames/s", h2d_bytes_per_step=int(h_img.numel() + h_lab.numel() * 4), d2h_bytes_per_step=4,
                 note="pinned host uint8 images + int32 label maps in (upload of step i + 1 overlapped with step i on a copy stream), loss scalar out; "
                      "wall clock over %d steps" % k))


# ------------------------------------------------------------------------------------------
# CPU arm: the same path restated on the host cores (oracle/cpu_pipeline.py)
# ------------------------------------------------------------------------------------------
def cpu_pipeline_sample(frames_per_step, steps, warmup, threads=None):
    from oracle import cpu_pipeline as cp
    from posecnn_b200 import synth
    import torch
    host = cp.host_cores()
    params = cp.init_random(C, 0)
    rgb, _ = synth.make_images(32, H, W, seed=21)            # the GPU arm's global batch
    K = synth.intrinsics(H, W)
    meta = np.stack([synth.make_meta(K)] * frames_per_step)
    ext = synth.extents_for(C)
    # "all the host threads it can use" is decided by measurement: on a 128-thread host the all-cores run of the fp32
    # conv stack is ~10x SLOWER than 8-16 threads (oversubscription / cgroup quota); time the conv trunk of one frame at
    # 4, 8, ... host cores and keep the fastest.
    x = (torch.from_numpy(rgb[:1]).float() - torch.tensor(cp.PIXEL_MEANS)).permute(0, 3, 1, 2).contiguous()
    sweep = {}
    for c in sorted({c for c in (4, 8, 16, 32, 64, host) if c <= host}):
        torch.set_num_threads(c)
        with torch.no_grad():
            cp.R.trunk(params, x)                               # warm the thread pool
            t0 = time.perf_counter()
            cp.R.trunk(params, x)
        sweep[c] = time.perf_counter() - t0
        if sweep[c] > 2.0 * min(sweep.values()):
            break
    cores = min(sweep, key=sweep.get)
    torch.set_num_threads(cores)
    cp.calibrate_background(params, rgb[:2], C, 0.75)
    hthreads = threads or min(16, cores)
    tm = []
    for i in range(warmup):
        cp.forward(params, rgb[(i * frames_per_step) % 32:][:frames_per_step], meta, ext, C, hthreads)
    t0 = time.perf_counter()
    for i in range(steps):
        cp.forward(params, rgb[((i + warmup) * frames_per_step) % 32:][:frames_per_step], meta, ext, C, hthreads, tm)
    dt = (time.perf_counter() - t0) / steps
    parts = np.mean(np.stack([np.pad(t, (0, 4 - len(t))) for t in tm]), 0) if tm else np.zeros(4)
    return dict(value=frames_per_step / dt, unit="frames/s", cores=cores, kind="port", ms_per_step=1e3 * dt,
                sample="%d frame(s) of the GPU arm's batch per step x %d steps: BGR - means, VGG16 trunk + dense-deconv heads (torch fp32, "
                       "%d threads = fastest of a measured sweep), CPU hough_voting_layer (RANSAC port, %d OpenMP threads), RoiPool x2 (C oracle), fc6-fc8 (torch fp32), "
                       "NMS + pose assembly" % (frames_per_step, steps, cores, hthreads),
                breakdown_ms=dict(trunk=1e3 * parts[0], heads=1e3 * parts[1], hough=1e3 * parts[2], pose_head_nms=1e3 * parts[3]),
                host_cores=host, thread_sweep_trunk_s={str(k): round(v, 3) for k, v in sweep.items()})


def reference_arm(args):
    fps = 1
    r = cpu_pipeline_sample(fps, args.steps, max(1, min(args.warmup, 2)))
    return dict(impl="reference", metric=METRIC_FULL, value=r["value"], unit="frames/s", n_gpus=0, steps=args.steps, warmup=args.warmup,
                ms_per_step=r["ms_per_step"], higher_is_better=True, scaling="strong", vs_baseline=None, dtype="fp32 (torch CPU) / f64 (RANSAC)",
                data="synthetic",
                config=dict(workload="configs[2]: full VGG16+Hough+ROI inference, random-init (Kaiming, seed 0) weights, 640x480 uint8 BGR "
                                     "frames of the same global batch; bounded sample of %d frame(s) per step on the host cores" % fps,
                            global_batch=32, frames_per_step=fps),
                cpu_baseline=dict(value=r["value"], unit="frames/s", cores=r["cores"], kind="port", sample=r["sample"],
                                  breakdown_ms=r["breakdown_ms"]),
                e2e=dict(value=r["value"], unit="frames/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0))


_JSON_OUT = None


def claim_stdout():
    """stdout carries exactly ONE line, the result JSON: keep a private handle on the real stdout and point fd 1 at
    stderr so that anything a library prints (NCCL's version banner, torchrun notices) cannot end up next to it."""
    global _JSON_OUT
    if _JSON_OUT is None:
        sys.stdout.flush()
        _JSON_OUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)
    return _JSON_OUT


def emit(result):
    out = claim_stdout()
    out.write(json.dumps(result) + "\n")
    out.flush()


def main():
    claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10, help="timed steps of every timed loop of the workload")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="full", choices=["hough", "full", "rgbd", "project", "train"])
    ap.add_argument("--batch", type=int, default=32, help="frames of the GLOBAL batch per step (sharded over the GPUs)")
    ap.add_argument("--grid", type=int, default=128, help="voxel grid size of --workload project")
    ap.add_argument("--e2e-batch", type=int, default=32)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-graph", action="store_true", help="eager launches instead of one CUDA graph per step")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-weak", action="store_true", help="skip the weak-scaling record of multi-GPU runs")
    ap.add_argument("--no-hough-record", action="store_true", help="skip the Hough-op sub-records of the default line")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the timed path computed in its last timed step as DIR/<name>.npy "
                                                          "(float32 / float64, sampled to at most 64 MB in all)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")

    if args.impl == "reference":
        rank = int(os.environ.get("RANK", "0"))
        if rank != 0:
            return
        emit(reference_arm(args))
        return

    rank, world, local = dist_setup(args.gpus)
    if args.workload == "hough":
        res = run_hough(args, rank, world, local)
    elif args.workload == "project":
        res = run_project(args, rank, world, local)
    elif args.workload == "train":
        if args.batch == 32:
            args.batch = 64                                   # configs[4] names batch 64
        res = run_train(args, rank, world, local)
    else:
        res, net = run_full(args, rank, world, local, "RGBD" if args.workload == "rgbd" else "COLOR")
        if rank == 0 and world == 1 and args.workload == "full" and not args.no_hough_record:
            del net
            import torch
            torch.cuda.empty_cache()
            peaks = measured_peaks()
            hb = {}
            for B in (32, 1):
                r = measure_hough(B, 0, 1, 0, args.steps, args.warmup, True, 32, True)
                r["frac"] = r["footprint_gbs"] / peaks["hbm_gbs"]
                hb["b%d" % B] = r
            traffic = profile_json("r02_hough_traffic.json")
            if traffic:
                hb["physical_dram_bytes_per_step"] = traffic
            if not args.no_cpu_baseline:
                cpu = cpu_hough_same_frames()
                hb["cpu_same_frames"] = cpu
                if cpu.get("value"):
                    hb["gpu_over_cpu"] = dict(device_b32=hb["b32"]["frames_per_s"] / cpu["value"], e2e_b32=hb["b32"]["e2e"]["value"] / cpu["value"],
                                              device_b1=hb["b1"]["frames_per_s"] / cpu["value"])
            hb["note"] = ("Houghvotinggpu op alone on the SURVEY 8(d) synthetic scenes (8 distinct frames tiled to the batch; the CPU op runs "
                          "the same 8 frames): footprint = 82.33 MB/frame (label + dense vertex_pred) / device time of the whole op "
                          "(CUDA-graph replay, L2 flushed); peak = measured HBM copy bandwidth; the kernels read only ~2 MB/frame "
                          "(compulsory_bytes_per_frame), so the footprint fraction is a throughput-per-input-byte figure, not DRAM traffic")
            res["hough"] = hb
            res["roofline_hough"] = dict(bound="hbm", achieved=hb["b32"]["footprint_gbs"], peak=peaks["hbm_gbs"], unit="GB/s",
                                         frac=hb["b32"]["frac"], ms=hb["b32"]["device_ms"], scenes="SURVEY 8(d) synthetic scenes, batch 32")
    if rank == 0:
        if args.dump_outputs:
            write_outputs(args.dump_outputs)
        if not args.no_cpu_baseline and world == 1 and args.workload in ("full",):
            try:
                res["cpu_baseline"] = cpu_pipeline_sample(1, 4, 1)
            except Exception as e:  # pragma: no cover
                res["cpu_baseline"] = dict(value=None, unit="frames/s", cores=0, kind="port", sample="unavailable: %s" % e)
        emit(res)
    if world > 1:
        import torch.distributed as dist
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
