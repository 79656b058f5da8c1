#!/usr/bin/env python
"""bench.py -- frames/sec of the MeMOTR per-frame hot path on B200 (contract: see DESIGN.md "Measurement").

  python bench.py [--gpus N] [--steps K] [--warmup W] [--mode bf16|fp32] [--impl reference] [--dump-outputs DIR]
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...

The hot path of one frame: level flattening + position maps -> 6-layer deformable encoder -> 6-layer decoder (300 detect +
100 track queries) -> class/box heads -> RuntimeTracker glue -> QueryUpdater.update_tracks_embedding, on a synthetic
1333x800 4-scale pyramid (S = 22323 tokens), DanceTrack hyper-parameters (BASELINE.json configs[1] minus the ResNet-50
backbone, which SURVEY.md section 8 marks out of scope), weights drawn from the reference's own initialisation
(memotr_b200/synthetic.py:reference_init_state_dict -- the configuration tests/test_engine_gpu.py holds to the north star's
parity bars against the reference modules).

A "step" is ONE CLIP of --clip-frames (64) chained frames -- BASELINE.json configs[3]: the frames of the clip are sharded
over the N GPUs in contiguous sub-clips (memotr_b200/clip.py:shard_frames, 64/N frames per GPU), every rank runs its
sub-clip with its own track state, and the ranks exchange their complete track memory (every TrackInstances field) with ONE
NCCL all-gather per clip.  Total work per step is fixed, so N > 1 is STRONG scaling.

  value   frames/s (whole job: K clips x 64 frames / time) with the frame inputs already resident in HBM (CUDA-graph replay
          of the whole per-frame step; 6 distinct frames rotate through the input buffers, device-to-device, inside the
          timed region).
  e2e     the same metric through the public API (memotr_b200.engine.ClipRunner) with HOST buffers: every frame copies the
          4 feature maps + 4 masks from pinned host memory -- on a copy stream, double buffered -- runs the step and reads the
          frame's result rows back to pinned host memory.
  roofline   MSDA forward (encoder-shaped launch, the dominant memory-bound kernel): algorithmic bytes / duration, duration
          from CUDA events recorded inside the captured graph around that launch.
  cpu_baseline / --impl reference   the reference's CPU path (oracle/frame.py, the torch restatement pinned against the
          reference modules) on the host cores; one step of the reference arm = one frame of the clip (bounded sample).
  extras  exact_two_phase (the bit-exact sharded clip: frame-parallel encoder phase + hand-off chain), msda_sweep
          (BASELINE.json configs[4]), msda_backward, fp32 mode, gpu_reference (the reference's CUDA op + PyTorch eager).
"""
import argparse
import json
import os
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)


def _metric_name():
    """BASELINE.json's metric string, verbatim (the file is part of the repo snapshot)."""
    try:
        return json.load(open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "BASELINE.json")))["metric"]
    except Exception:                                                    # noqa: BLE001
        return "frames/sec at 1333x800, 300 det+100 track queries"


METRIC = _metric_name()
N_TRACKS = 100
N_ROT = 6            # resident frames rotating through the input buffers: 6 x 22.9 MB > L2 together with the workspace
WORKLOAD = "DanceTrack hot path: transformer(6 enc + 6 dec, d256, ffn2048, 4 levels S=22323) + heads + tracker glue + " \
           "QueryUpdater, 300 det + 100 track queries, batch 1, synthetic 1333x800 pyramid, backbone excluded"


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d, "measured (MEASURED_PEAKS.json)"
    return {"hbm_gbs": 6650.0, "bf16_tflops_sustained": 1430.2}, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """SM clock / throttle reasons sampled IN-PROCESS through NVML every 5 ms while the timed region runs (a 100 ms
    nvidia-smi poll cannot see a region of a few hundred ms).  Started before the warm-up, marked at the timed region."""
    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, index):
        self.rows, self.t_mark, self.stop_flag, self.ok = [], None, False, False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv, self.h = pynvml, pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception as e:                                              # noqa: BLE001
            self.err = repr(e)

    def _run(self):
        nv = self.nv
        while not self.stop_flag:
            try:
                self.rows.append((time.perf_counter(), nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM),
                                  nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)))
            except Exception:                                               # noqa: BLE001
                pass
            time.sleep(0.005)

    def start(self):
        if self.ok:
            self.thread = threading.Thread(target=self._run, daemon=True)
            self.thread.start()

    def mark(self):
        self.t_mark = time.perf_counter()

    def stop(self):
        if not self.ok:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvml unavailable: " + getattr(self, "err", "?")], "samples": 0}
        t_end = time.perf_counter()
        self.stop_flag = True
        self.thread.join(timeout=2)
        rows = [r for r in self.rows if self.t_mark is None or self.t_mark <= r[0] <= t_end] or self.rows
        sm = sorted(r[1] for r in rows)
        mask = 0
        for r in rows:
            mask |= int(r[2])
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(n for b, n in self.REASONS.items() if mask & b), "samples": len(rows),
                "how": "NVML in-process, 5 ms period, samples inside the timed region"}


def _pick_cpu_threads(sd, x, cfg):
    """torch intra-op thread count that runs the reference CPU path fastest on this host.  "All the host threads" is
    not automatically the fastest setting: on the 128-core GPU hosts the default (one thread per core) ran a frame in
    52 s against a few seconds with fewer threads (oversubscription on many small ops).  Probe = one encoder layer."""
    from oracle import frame as oframe
    src, mask, pos, shapes, lsi, vr = oframe.flatten_levels(sd, "transformer", x["srcs"], x["masks"], x["pos"])
    ref = oframe.encoder_reference_points(shapes, vr, "cpu")
    n_cpu = os.cpu_count() or 1
    best, best_t = None, float("inf")
    for t in sorted({min(c, n_cpu) for c in (8, 16, 32, 64, n_cpu)}):
        torch.set_num_threads(t)
        with torch.no_grad():
            for rep in range(2):
                t0 = time.perf_counter()
                oframe.encoder_layer(sd, "transformer.encoder.layers.0", src, pos, ref, shapes, lsi, mask, cfg)
                dt = time.perf_counter() - t0
        if dt < best_t:
            best, best_t = t, dt
        if dt > 4 * best_t:
            break
    torch.set_num_threads(best)
    return best


def _weights(cfg):
    from memotr_b200 import synthetic as synth
    return synth.reference_init_state_dict(cfg, seed=0)


def cpu_reference_fps(steps, warmup):
    """The reference's CPU path (torch fp32 on the host cores) through the functional oracle.  One step = one frame."""
    from oracle import frame as oframe
    from oracle import synth
    cfg = oframe.dancetrack_cfg()
    sd = _weights(cfg)
    x = synth.frame_inputs(cfg, synth.DANCETRACK_SHAPES, N_TRACKS, seed=1)
    threads = _pick_cpu_threads(sd, x, cfg)
    tracks = dict(x["tracks"])
    times = []
    with torch.no_grad():
        for i in range(warmup + steps):
            t0 = time.perf_counter()
            res = oframe.frame_forward(sd, x["srcs"], x["masks"], x["pos"], tracks["ref_pts"], tracks["query_embed"], cfg)
            nd = cfg["n_det_queries"]
            tracks.update(boxes=res["pred_bboxes"][0, nd:], logits=res["pred_logits"][0, nd:],
                          output_embed=res["outputs"][0, nd:])
            tracks.update({k: v for k, v in oframe.update_tracks(sd, tracks, cfg).items() if k != "is_pos"})
            if i >= warmup:
                times.append(time.perf_counter() - t0)
    return len(times) / sum(times), threads


def fp32_modes_fps(dev, sd, cfg, tracker, frames, n_frames=12):
    """The engine's fp32-accurate modes on the same workload (frame after frame, one CUDA graph per frame): "fp32tc" (large GEMMs on
    the tensor cores at fp32 accuracy, parity <= 1e-4) and "fp32" (everything on CUDA cores).  Extras: the headline is the bf16 mode."""
    from memotr_b200 import synthetic as synth
    from memotr_b200.engine import FrameEngine
    out = {}
    for mode in ("fp32tc", "fp32"):
        eng = FrameEngine(sd, cfg, synth.DANCETRACK_SHAPES, N_TRACKS, dev, mode=mode, tracker=tracker, ori_size=(1920, 1080),
                          pos_embed=dict(temperature=20))
        x0 = frames[0]
        eng.load_frame(x0["srcs"], x0["masks"], None, x0["tracks"]["ref_pts"], x0["tracks"]["query_embed"])
        eng.load_tracks(x0["tracks"])
        if eng.trk is not None:
            eng.trk.reset(x0["tracks"])
        eng.capture()
        for _ in range(3):
            eng.replay()
        torch.cuda.synchronize(dev)
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        for _ in range(n_frames):
            eng.replay()
        e.record()
        torch.cuda.synchronize(dev)
        out[mode] = round(n_frames / (s.elapsed_time(e) * 1e-3), 1)
        del eng
        torch.cuda.empty_cache()
    return out


def gpu_reference_fps(dev, steps, warmup):
    """The reference GPU path restated: stock PyTorch fp32 ops (TF32 off, main.py:96-97) + the reference's own CUDA op
    compiled into oracle/_ref.  Reported beside our numbers; None when the .so did not travel."""
    ref_dir = os.path.join(ROOT, "oracle", "_ref")
    if not os.path.exists(os.path.join(ref_dir, "MultiScaleDeformableAttention.so")):
        return None
    sys.path.insert(0, ref_dir)
    import MultiScaleDeformableAttention as MSDA
    from oracle import frame as oframe
    from oracle import synth
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    cfg = oframe.dancetrack_cfg()
    sd = {k: v.to(dev) for k, v in _weights(cfg).items()}
    x = synth.frame_inputs(cfg, synth.DANCETRACK_SHAPES, N_TRACKS, seed=1)
    srcs, masks, pos = ([t.to(dev) for t in x[k]] for k in ("srcs", "masks", "pos"))
    tracks = {k: v.to(dev) for k, v in x["tracks"].items()}

    def core(value, shapes_t, lsi, loc, attn):
        return MSDA.ms_deform_attn_forward(value.contiguous(), shapes_t, lsi, loc.contiguous(), attn.contiguous(), 64)

    def step():
        res = oframe.frame_forward(sd, srcs, masks, pos, tracks["ref_pts"], tracks["query_embed"], cfg, core=core)
        nd = cfg["n_det_queries"]
        tracks.update(boxes=res["pred_bboxes"][0, nd:], logits=res["pred_logits"][0, nd:],
                      output_embed=res["outputs"][0, nd:])
        tracks.update({k: v for k, v in oframe.update_tracks(sd, tracks, cfg).items() if k != "is_pos"})

    with torch.no_grad():
        for _ in range(warmup):
            step()
        torch.cuda.synchronize(dev)
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        for _ in range(steps):
            step()
        e.record()
        torch.cuda.synchronize(dev)
    return steps / (s.elapsed_time(e) * 1e-3)


def dump_outputs(eng, out_dir):
    """The arrays a caller receives for the frame the engine ran last: the reference's output dict (FrameEngine.results),
    the live rows of the track table and the frame's result rows (tracker on the device), or the track state the caller
    keeps (--no-tracker).  fp32, integer fields as float64 (exact); about 26 MB at the DanceTrack size."""
    import numpy as np
    arrays = dict(eng.results())
    if eng.trk is not None:
        arrays.update({"track_" + k: v for k, v in eng.table.active().items()})
        ids, boxes, scores, keep = eng.trk.split_results(eng.trk.res_flat)
        arrays.update(result_ids=ids, result_boxes=boxes, result_scores=scores, result_keep=keep)
    else:
        arrays.update({"track_" + k: v for k, v in eng.st.items()})
    os.makedirs(out_dir, exist_ok=True)
    for k, v in arrays.items():
        v = v.detach().cpu()
        np.save(os.path.join(out_dir, k + ".npy"), (v.float() if v.is_floating_point() else v.double()).numpy())


def _timeit_us(fn, iters, warmup, flush):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(iters):
        flush.add_(1.0)
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        fn()
        e.record()
        torch.cuda.synchronize()
        ts.append(s.elapsed_time(e) * 1e3)
    ts.sort()
    return ts[len(ts) // 2]


def msda_extras(dev, hbm_peak):
    """BASELINE.json configs[4]: MSDA forward HBM GB/s, 1280x720 pyramid, K in {4,8,16} x L in {4,5}, encoder-shaped launch
    (the windowed kernel on encoder-like sampling patterns) and the decoder-shaped launch (Lq = 800, global-memory kernel);
    plus the backward op on the DanceTrack encoder shape (fp32, the MSDeformAttnFunction path).  L2 flushed between iterations."""
    from memotr_b200 import kernels, synthetic as synth
    import memotr_b200
    flush = torch.empty(256 * 1024 * 1024 // 4, device=dev)
    sweep = []
    for L, shapes in ((4, synth.BDD_SHAPES), (5, synth.BDD_SHAPES_L5)):
        shp = torch.as_tensor(shapes, dtype=torch.long)
        lsi = torch.cat((shp.new_zeros(1), shp.prod(1).cumsum(0)[:-1])).to(dev)
        shp = shp.to(dev)
        for K in (4, 8, 16):
            value, vr, loc, attn, shift = synth.encoder_msda_inputs(shapes, H=8, K=K, seed=7, noise_px=0.15)
            value, vr, loc, attn = value.half().to(dev), vr.to(dev), loc.to(dev), attn.to(dev)
            S = value.shape[0]
            radius = min((K - 1) / 2 + 0.9, 6.0)
            nbytes = S * 256 * 2 + S * 8 * L * K * 12 + S * 256 * 2
            t_enc = _timeit_us(lambda: kernels.msda_forward_window(value, shapes, vr, n_heads=8, n_points=K, loc=loc, attn=attn,
                                                                   shift=shift, radius=radius), 10, 3, flush)
            Lq = 800                                                          # 300 det + 500 track queries (BDD100K config)
            dl, da = loc[:Lq].contiguous(), attn[:Lq].contiguous()
            dbytes = S * 256 * 2 + Lq * 8 * L * K * 12 + Lq * 256 * 2
            t_dec = _timeit_us(lambda: kernels.msda_forward_strided(value, shp, lsi, n_heads=8, n_levels=L, n_points=K, loc=dl,
                                                                    attn=da), 10, 3, flush)
            sweep.append({"L": L, "K": K, "S": S, "encoder_us": round(t_enc, 2), "encoder_gbs": round(nbytes / t_enc / 1e3, 1),
                          "encoder_frac": round(nbytes / t_enc / 1e3 / hbm_peak, 4), "decoder_Lq": Lq, "decoder_us": round(t_dec, 2),
                          "decoder_gbs": round(dbytes / t_dec / 1e3, 1), "decoder_frac": round(dbytes / t_dec / 1e3 / hbm_peak, 4)})
    # backward, DanceTrack encoder shape, fp32
    value, shp, lsi, loc, attn = (t.to(dev) for t in synth.msda_inputs(synth.DANCETRACK_SHAPES, Lq=22323, K=4, seed=1))
    go = torch.randn(1, 22323, 256, device=dev)
    t_bwd = _timeit_us(lambda: memotr_b200.ms_deform_attn_backward(value, shp, lsi, loc, attn, go, 64), 10, 3, flush)
    bbytes = (22323 * 256 * 3 + 22323 * 8 * 16 * 3 * 2 + 22323 * 256) * 4      # SURVEY.md 8d: ~160 MB
    bwd = {"shape": "DanceTrack encoder call, fp32", "us": round(t_bwd, 1), "algorithmic_bytes": bbytes,
           "gbs": round(bbytes / t_bwd / 1e3, 1), "frac": round(bbytes / t_bwd / 1e3 / hbm_peak, 4)}
    return sweep, bwd


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=8)      # clips; 8 x 64 frames ~ 1 s timed at N = 1
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--mode", default="bf16", choices=["bf16", "fp32", "fp32tc"],
                    help="fp32: CUDA-core fp32 GEMMs; fp32tc: the fp32 engine with its large GEMMs on the tensor cores at fp32 accuracy")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--clip-frames", type=int, default=64)
    ap.add_argument("--no-baselines", action="store_true", help="skip the cpu_baseline / gpu_reference / extras legs")
    ap.add_argument("--no-pipeline", action="store_true",
                    help="A/B: frame after frame on one stream (default: the recurrent tail of frame k overlaps the encoder of frame k+1)")
    ap.add_argument("--upload-pos", action="store_true",
                    help="upload the position maps with every frame (A/B; default: rebuilt on the device from the masks)")
    ap.add_argument("--no-tracker", action="store_true",
                    help="leave the RuntimeTracker glue out of the step (A/B; default: on the device, inside the graph)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed frame returned (frame outputs, track table, result rows) to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    W, K, CLIP = max(args.warmup, 3), args.steps, args.clip_frames

    if args.impl == "reference":
        # the reference's own CPU implementation of the path, host threads, rank 0 only; one step = one frame of the clip
        if rank != 0:
            return
        fps, threads = cpu_reference_fps(K, W)
        print(json.dumps({
            "impl": "reference", "metric": METRIC, "value": fps, "unit": "frames/s", "n_gpus": args.gpus, "steps": K,
            "warmup": W, "ms_per_step": 1e3 / fps, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "note": "reference CPU path = PyTorch fp32 ops on the host cores with "
                       "ms_deform_attn_core_pytorch as the sampling core (oracle/frame.py, pinned to the reference modules); "
                       "a step of this arm is ONE frame of the clip (bounded sample of the 64-frame step of our arm)"},
            "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": os.cpu_count(), "threads": threads, "kind": "port",
                             "sample": f"{K} frames after {W} warm-up frames; torch intra-op threads = fastest of "
                                       f"8/16/32/64/{os.cpu_count()} on a one-encoder-layer probe"},
            "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        }))
        return

    assert torch.cuda.is_available(), "bench.py needs a GPU (there is no CPU fallback for the product path)"
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)     # (NCCL_DEBUG is left to the caller: its banner goes to stderr)

    from memotr_b200 import clip as clip_mod
    from memotr_b200 import synthetic as synth
    from memotr_b200.engine import ClipRunner, FrameEngine
    cfg = synth.dancetrack_cfg()
    sd = _weights(cfg)
    my_frames = clip_mod.shard_frames(CLIP, world, rank)
    frames = [synth.frame_inputs(cfg, synth.DANCETRACK_SHAPES, N_TRACKS, seed=1 + i, padded=True) for i in range(N_ROT)]
    # Tracker glue on the device (memotr_b200/tracker.py).  The weights are untrained, so the thresholds are pinned such that
    # the 100 loaded tracks stay live and nothing is born: the step keeps BASELINE.json's 300 det + 100 track queries.
    tracker = None if args.no_tracker else dict(det_score_thresh=2.0, track_score_thresh=0.0, miss_tolerance=30,
                                                result_score_thresh=0.5)
    # Position maps: a function of the padding masks alone (PositionEmbeddingSine), rebuilt on the device every frame
    # instead of crossing PCIe (the box's pinned H2D rate, ~26 GB/s, would cap e2e at 564 frames/s with them).
    pos_embed = None if args.upload_pos else dict(temperature=20)
    eng = FrameEngine(sd, cfg, synth.DANCETRACK_SHAPES, N_TRACKS, dev, mode=args.mode, tracker=tracker,
                      ori_size=(1920, 1080), pos_embed=pos_embed)
    L, C = eng.L, eng.C

    # resident copies of the rotating frames + pinned host copies for the e2e leg
    res_src = [[f["srcs"][l].reshape(C, -1).to(dev) for l in range(L)] for f in frames]
    res_mask = [[f["masks"][l].reshape(-1).to(torch.uint8).to(dev) for l in range(L)] for f in frames]
    res_pos = [[f["pos"][l].reshape(C, -1).to(dev) for l in range(L)] for f in frames] if args.upload_pos else None
    pin = lambda t: t.contiguous().pin_memory()                                      # noqa: E731
    host = [{"srcs": [pin(t) for t in f["srcs"]], "pos": [pin(t) for t in f["pos"]],
             "masks": [pin(t.to(torch.uint8)) for t in f["masks"]]} for f in frames]
    x0 = frames[0]
    eng.load_frame(x0["srcs"], x0["masks"], x0["pos"] if args.upload_pos else None, x0["tracks"]["ref_pts"],
                   x0["tracks"]["query_embed"])
    eng.load_tracks(x0["tracks"])
    if eng.trk is not None:
        eng.trk.reset(x0["tracks"])
    # Two captured graphs of the same step(): forward + tracker + updater + feedback.  The plain one is what a user replays.
    # The instrumented one carries 17 event-record nodes (gather launches, section marks); every such node breaks a
    # programmatic-dependent-launch edge, so it is replayed for the LAST frame of every clip only: those frames are inside the
    # timed region and are where `roofline` and `sections_us` are sampled (since the pipelined clip: the last frame of the LAST
    # clip of the timed region only).
    eng.capture()
    g_plain, plain_launches = eng.graph, eng.graph_launches
    eng.enable_msda_timer()
    eng.capture()
    g_instr = eng.graph
    eng.graph, eng.graph_launches = g_plain, plain_launches
    pipelined = (not args.no_pipeline) and args.mode == "bf16" and eng.dec_cluster and len(my_frames) >= 3
    if pipelined:
        eng.capture_pipeline()

    def feed_resident(i):
        for l in range(L):
            eng.in_src[l].copy_(res_src[i % N_ROT][l], non_blocking=True)
            eng.in_mask[l].copy_(res_mask[i % N_ROT][l], non_blocking=True)
            if res_pos is not None:
                eng.in_pos[l].copy_(res_pos[i % N_ROT][l], non_blocking=True)

    tracks0 = {k: (v.to(dev) if torch.is_tensor(v) else v) for k, v in x0["tracks"].items()}   # resident: D2D copies below

    def reset_clip():
        """Start of a (sub-)clip: the clip's initial tracks (device-to-device, nothing pageable inside the timed region)."""
        eng.in_track_ref.copy_(tracks0["ref_pts"], non_blocking=True)
        eng.in_track_embed.copy_(tracks0["query_embed"], non_blocking=True)
        eng.load_tracks(tracks0, non_blocking=True)
        if eng.trk is not None:
            eng.trk.reset_async(tracks0, max_obj_id=N_TRACKS)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    align = torch.zeros(1, device=dev)

    def device_align():
        """Start of a timed region, N > 1: dist.barrier() aligns the HOSTS to within their scheduling jitter (milliseconds, measured
        3.3 ms at N = 4 -- 3.6 % of a 4-clip region, paid by every rank at the first all-gather); one tiny all-reduce enqueued right
        before the start event aligns the DEVICES: every rank's timed region begins when the collective completes."""
        if world > 1:
            dist.all_reduce(align)

    gathered = {}
    xev = []          # MEMOTR_BENCH_TIME_EXCHANGE=1: (before, after) event pairs around the per-clip exchange (diagnostic)
    time_x = os.environ.get("MEMOTR_BENCH_TIME_EXCHANGE", "0") == "1"

    def clip_exchange():
        """One NCCL all-gather of the complete track memory per clip (SURVEY.md 8e, memotr_b200/clip.py)."""
        if world > 1 and time_x:
            ev = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
            ev[0].record()
            _clip_exchange()
            ev[1].record()
            xev.append(ev)
        else:
            _clip_exchange()

    def _clip_exchange():
        if world > 1:
            if eng.trk is not None:
                gathered["last"] = clip_mod.gather_track_memory({k: eng.table[k] for k in clip_mod.FLOAT_FIELDS + clip_mod.INT_FIELDS},
                                                                eng.table.n_active, eng.trk.max_obj_id)
            else:
                gathered["last"] = clip_mod.gather_track_memory(eng.st)

    def run_clip_resident(instr):
        """One clip.  instr: the clip's last frame runs sequentially through the instrumented graph (the LAST clip of the timed
        region and of the warm-up: where `roofline` / `sections_us` are sampled; one frame per timed region, not per clip, so
        that short sub-clips at large N do not pay for it every time)."""
        reset_clip()
        idx = list(my_frames)
        if pipelined:
            n_pipe = len(idx) - 1 if instr else len(idx)
            eng.run_clip_pipelined(n_pipe, lambda j: feed_resident(idx[j]))
            if instr:
                feed_resident(idx[-1])
                g_instr.replay()
        else:
            for j, i in enumerate(idx):
                feed_resident(i)
                (g_instr if instr and j == len(idx) - 1 else g_plain).replay()
        clip_exchange()

    def run_clips_resident(n_clips):
        """n_clips clips back to back.  Pipelined: ONE stream of clips (FrameEngine.run_clips_pipelined) -- the tail of a clip's last
        frame overlaps the encoder of the next clip's first frame, the all-gather and the track reset sit between the two in stream
        order; the last frame of the last clip runs sequentially through the instrumented graph."""
        if n_clips <= 0:
            return
        if not pipelined:
            for k in range(n_clips):
                run_clip_resident(k == n_clips - 1)
            return
        idx = list(my_frames)
        lens = [len(idx)] * (n_clips - 1) + [len(idx) - 1]

        def between(c):
            if c == n_clips - 1:
                feed_resident(idx[-1])
                g_instr.replay()
                clip_exchange()
            else:
                clip_exchange()
                reset_clip()
        reset_clip()
        eng.run_clips_pipelined(lens, lambda c, j: feed_resident(idx[j]), between)

    # ---- resident-input throughput ("value") -----------------------------------------------------------------
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    run_clips_resident(W)
    barrier()
    sampler.mark()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    device_align()
    t0.record()
    host_t0 = time.perf_counter()
    run_clips_resident(K)
    host_enqueue_ms = (time.perf_counter() - host_t0) * 1e3 / (K * max(len(my_frames), 1))
    t1.record()
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(eng, args.dump_outputs)
    ms = torch.tensor([t0.elapsed_time(t1)], device=dev)
    ms_all = None
    if world > 1:
        ms_all = [torch.zeros_like(ms) for _ in range(world)]
        dist.all_gather(ms_all, ms)
        ms_all = [float(t.item()) for t in ms_all]
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms_total = float(ms.item())
    tracks_live = int(eng.table.n_active.item()) if eng.trk is not None else N_TRACKS
    if eng.trk is not None:
        eng.trk.check_overflow()
        assert tracks_live == N_TRACKS, f"the bench workload drifted: {tracks_live} live tracks instead of {N_TRACKS}"
    if world > 1:      # the gathered memory really holds every rank's tracks (ids of the pinned workload: 0 .. 99 on every rank)
        m = clip_mod.unpack_track_state(gathered["last"][world - 1], eng.nt, eng.C, eng.ncls)
        assert int(m["n_active"].item()) == tracks_live and m["ids"][:tracks_live].tolist() == list(range(tracks_live))
    # CPU cost of launching one step with an empty queue (the in-loop figure above includes back-pressure from the GPU)
    torch.cuda.synchronize(dev)
    h0 = time.perf_counter()
    for _ in range(4):
        eng.replay()
    host_launch_ms = (time.perf_counter() - h0) * 1e3 / 4
    torch.cuda.synchronize(dev)
    msda_us = eng.msda_times_us()                       # the 6 encoder MSDA launches of the last replayed step
    sections = eng.section_times_us()
    # the fused encoder FFN (largest kernel by time, tensor-bound) timed on its own after the run: event nodes around it
    # inside the graph would cost the programmatic-launch overlap with its neighbours (measured: -4 % step throughput)
    ffn_us = None
    if eng.fused_mlp and args.mode == "bf16" and rank == 0:
        ly = eng.enc[0]
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(12)]
        for i in range(8):
            if i >= 2:
                ev[2 * (i - 2)].record()
            eng.mlp2(eng.src1, eng.C, ly["lin1"], ly["lin2"], eng.pre, eng.C, eng.S, eng.hid, c_dtype=0)
            if i >= 2:
                ev[2 * (i - 2) + 1].record()
        torch.cuda.synchronize(dev)
        ffn_us = [ev[2 * i].elapsed_time(ev[2 * i + 1]) * 1e3 for i in range(6)]

    # ---- end to end through the public API with host buffers ("e2e") ----------------------------------------------
    runner = ClipRunner(eng)
    h2d, d2h = runner.h2d_bytes, runner.d2h_bytes
    hf = [(h["srcs"], h["pos"] if args.upload_pos else None, h["masks"]) for h in host]

    def e2e_clip():
        reset_clip()
        idx = list(my_frames)
        if pipelined:        # the public pipelined clip call: H2D of frame k+2, encoder of frame k+1 and tail of frame k overlap
            runner.run_clip_pipelined([hf[i % N_ROT] for i in idx], sync=False)
            clip_exchange()
            return
        if idx:
            runner.prefetch(0, *hf[idx[0] % N_ROT])
        for j, i in enumerate(idx):
            if j + 1 < len(idx):
                runner.prefetch((j + 1) % 2, *hf[idx[j + 1] % N_ROT])
            runner.run(j % 2)
        clip_exchange()

    e2e_clip()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    device_align()
    e0.record()
    for _ in range(K):
        e2e_clip()
    e1.record()
    barrier()
    runner.check()                                      # overflow of the device track table would have been silent otherwise
    ems = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if world > 1:
        dist.all_reduce(ems, op=dist.ReduceOp.MAX)
    e2e_fps = K * CLIP / (float(ems.item()) * 1e-3)

    # ---- the exact sharded clip (bit-identical to one GPU running the whole clip): frame-parallel phase + hand-off chain ----
    exact = None
    if not args.no_baselines:
        def run_exact():
            reset_clip()
            eng.run_clip_two_phase(CLIP, lambda i: feed_resident(i))
        for _ in range(2):
            run_exact()
        barrier()
        x0e, x1e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        x0e.record()
        n_exact = max(2, K // 2)
        for _ in range(n_exact):
            run_exact()
        x1e.record()
        barrier()
        xms = torch.tensor([x0e.elapsed_time(x1e)], device=dev)
        if world > 1:
            dist.all_reduce(xms, op=dist.ReduceOp.MAX)
        exact = {"value": n_exact * CLIP / (float(xms.item()) * 1e-3), "unit": "frames/s", "clips": n_exact,
                 "what": "memotr_b200/clip.py:run_clip_two_phase -- phase 1 (flattening, encoder, decoder value projection) "
                         "frame-parallel over the ranks, phase 2 (decoder, heads, tracker, updater) as a hand-off chain of the "
                         "packed track memory (NCCL send/recv); results bit-identical to the sequential clip"}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant memory-bound kernel (MSDA forward, encoder-shaped launch) ---------------------------------
    S, H, LK = eng.S, eng.H, eng.L * cfg["n_enc_points"]
    esz = 2 if args.mode == "bf16" else 4
    # value read once + output written once (activation dtype) + sampling locations and weights (fp32): BASELINE.md sec. 3
    alg_bytes = S * H * 32 * esz + S * H * 32 * esz + S * H * LK * 3 * 4
    pk, peak_src = peaks()
    peak = pk["hbm_gbs"]
    traffic, traffic_src = None, None
    tpath = os.path.join(ROOT, "profiles", "r02_msda_window_traffic.json")
    if eng.msda_window and os.path.exists(tpath):        # dram bytes of this kernel from the committed ncu --set full capture
        tj = json.load(open(tpath))
        traffic = tj["dram_bytes_read"] + tj["dram_bytes_write"]
        traffic_src = "STATIC: profiles/r02_msda_window_traffic.json (ncu --set full capture of the same launch, committed; not re-measured by this run)"
    dur = sum(msda_us) / len(msda_us)
    achieved = alg_bytes / dur / 1e3
    fps = K * CLIP / (ms_total * 1e-3)
    kname = ("msda_window_kernel (TMA-staged fp16 value-map windows in shared memory)" if eng.msda_window else
             "msda_fwd_h16 (fp16 value map, global-memory gather)" if eng.value_f16 else "msda_fwd_vec (fp32)")
    out = {
        "metric": METRIC, "value": fps, "unit": "frames/s", "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": ms_total / K, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "bf16" if args.mode == "bf16" else "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD,
                   "step": f"one clip of {CLIP} chained frames sharded over the GPUs in contiguous sub-clips ({len(my_frames)} frames on rank 0), "
                           "one NCCL all-gather of the complete track memory (all TrackInstances fields) per clip",
                   "frame_pipelining": ("on: the recurrent tail of frame k (decoder + heads, tracker glue, query updater -- a latency chain "
                                        "on ~100 SMs) runs concurrently with the encoder of frame k+1 on a second stream, one forked CUDA "
                                        "graph per frame (FrameEngine.run_clip_pipelined; results identical to the sequential clip, "
                                        "tests/test_tracker_gpu.py); the K clips of the timed region are one stream (the last tail of a "
                                        "clip overlaps the first encoder of the next; all-gather and track reset in between); the last "
                                        "frame of the last timed clip runs sequentially through the instrumented graph" if pipelined else "off (--no-pipeline / fp32 / sub-clip shorter than 3 frames)"),
                   "weights": "reference initialisation distributions (synthetic.reference_init_state_dict), random-init, no checkpoint",
                   "l2": f"inputs larger than L2: {N_ROT} resident frames x {h2d / 1e6:.1f} MB rotate through the input buffers and a "
                         "step touches ~0.5 GB of workspace (L2 = 126 MB)",
                   "position_maps": "uploaded with every frame (--upload-pos)" if args.upload_pos else
                   "PositionEmbeddingSine rebuilt on the device from the padding masks inside the captured step",
                   "tracker": ("RuntimeTracker.update + select_active_tracks + result filter on the device inside the "
                               f"captured step; thresholds pinned so that {tracks_live} tracks stay live and none is born")
                   if eng.trk is not None else "off (--no-tracker)",
                   "arithmetic": "bf16 GEMM operands + fp16 value maps + fp32 accumulate/residual/LayerNorm/geometry; parity vs the "
                                 "reference modules <= 1e-2 on every output (tests/test_engine_gpu.py, frame_full_refinit)"
                   if args.mode == "bf16" else
                   ("fp32 everywhere (TF32 off, as the reference); the large-M GEMMs on the tensor cores at fp32 accuracy: two-term "
                    "fp16 operand splits, three products, fp32 accumulation (memotr_linear_f32x3); parity <= 1e-4 (measured 1.3e-5) on "
                    "frame_full_refinit" if args.mode == "fp32tc" else "fp32 everywhere on CUDA cores (TF32 off, as the reference)")},
        "clocks": clocks,
        "e2e": {"value": e2e_fps, "unit": "frames/s", "h2d_bytes_per_step": h2d * CLIP, "d2h_bytes_per_step": d2h * CLIP,
                "h2d_bytes_per_frame": h2d, "d2h_bytes_per_frame": d2h},
        "gpu_launches": eng.graph_launches * K * len(my_frames) * world,
        "frames_per_step": CLIP, "ms_per_frame": ms_total / (K * max(len(my_frames), 1)), "rank_ms": ms_all,
        **({"exchange_us": [round(a.elapsed_time(b) * 1e3, 1) for a, b in xev[-8:]]} if xev else {}),
        "sections_us": {k: round(v, 1) for k, v in sections.items()},
        "host_enqueue_ms_per_frame": round(host_enqueue_ms, 3),
        "host_graph_launch_ms": round(host_launch_ms, 3),
        "roofline": {"kernel": kname + " -- encoder-shaped launch, Lq = S = 22323", "bound": "hbm",
                     "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                     "traffic_source": traffic_src,
                     "peak_source": peak_src, "algorithmic_bytes": alg_bytes, "duration_us": dur,
                     "samples": f"{len(msda_us)} launches (the encoder layers of the last frame of the last timed clip), CUDA "
                                "events recorded inside the captured graph; all other frames replay the same step without "
                                "event nodes",
                     "on_chip_floor_us": 19.6,
                     "ceiling_note": "the gather reads S*H*L*K*4 corners*64 B = 731 MB of taps per launch through the SMs' shared-memory "
                                     "pipes (128 B/clk/SM): 19.6 us, i.e. at most 0.44 of the HBM roofline by on-chip bandwidth alone; see DESIGN.md"},
    }
    if ffn_us:      # second roofline object: the largest kernel by time is tensor-bound (fused encoder FFN)
        fdur = sum(ffn_us) / len(ffn_us)
        flops = 2.0 * 2.0 * eng.S * eng.C * eng.Fd
        tpeak = float(pk.get("bf16_tflops_sustained", 1430.2))
        tburst = float(pk.get("bf16_tflops", 1671.8))
        out["roofline_tensor"] = {"kernel": "mlp2_tc_kernel -- fused encoder FFN (22323 x 256 -> 2048 -> 256), main launch + tail-split launch",
                                  "bound": "tensor", "achieved": flops / fdur / 1e6, "peak": tburst, "unit": "TFLOP/s",
                                  "frac": flops / fdur / 1e6 / tburst, "frac_of_sustained_peak": flops / fdur / 1e6 / tpeak,
                                  "flop": flops, "duration_us": fdur,
                                  "peak_source": "MEASURED_PEAKS.json bf16 dense: burst (this timing is the kernel alone, back to back)",
                                  "samples": "6 back-to-back launches after the timed region (CUDA events; operands L2-warm)",
                                  "note": "shared-memory-bandwidth-bound in its cta_group::1 form, see profiles/r01_mlp2_ncu.md"}
    if exact:
        out["exact_two_phase"] = exact
    if not args.no_baselines and world == 1:      # the CPU / reference-GPU legs and the op-level extras are timed at N = 1 only
        cpu_fps, threads = cpu_reference_fps(3, 1)
        out["cpu_baseline"] = {"value": cpu_fps, "unit": "frames/s", "cores": os.cpu_count(), "threads": threads, "kind": "port",
                               "sample": "3 frames of the clip after 1 warm-up (oracle/frame.py on the host cores, torch fp32; "
                                         f"intra-op threads = fastest of 8/16/32/64/{os.cpu_count()} on a one-layer probe)"}
        g = gpu_reference_fps(dev, 10, 3)
        out["gpu_reference"] = {"value": g, "unit": "frames/s",
                                "what": "reference models/ops CUDA op (oracle/_ref, compiled from /root/reference) + stock "
                                        "PyTorch fp32 eager modules (TF32 off) on the same GPU and inputs"} if g else None
        try:
            fm = fp32_modes_fps(dev, sd, cfg, tracker, frames)
            out["fp32_modes"] = {"unit": "frames/s", **fm,
                                 "what": "the engine's fp32-accurate modes on the same frames, sequential CUDA-graph replays: fp32tc = "
                                         "every nn.Linear on the tensor cores at fp32 accuracy (two-term fp16 operand splits, three "
                                         "products, fp32 accumulation: memotr_linear_f32x3; parity <= 1e-4 on frame_full_refinit, "
                                         "measured 1.3e-5), fp32 = every GEMM on CUDA cores"}
        except Exception as e:                                              # noqa: BLE001
            out["fp32_modes"] = {"error": repr(e)}
        try:
            sweep, bwd = msda_extras(dev, peak)
            out["msda_sweep"] = {"what": "BASELINE.json configs[4]: 1280x720 pyramid, 8 heads, encoder-shaped (windowed kernel, ring + "
                                         "0.15 px offsets) and decoder-shaped Lq=800 (global-memory kernel) launches, L2 flushed",
                                 "rows": sweep}
            out["msda_backward"] = bwd
        except Exception as e:                                              # noqa: BLE001 -- extras must not lose the headline
            out["msda_sweep"] = {"error": repr(e)}
    print(json.dumps(out))
    sys.stdout.flush()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
