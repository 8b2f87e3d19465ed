#!/usr/bin/env python
"""bench.py — frames/s of the WVN hot path (BASELINE.json metric) on N B200s of one node.

    python bench.py --gpus 1 --steps 10 --warmup 3
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
        --master-port P bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference ...        (the reference algorithm on the host CPU cores)
    python bench.py --config c5 ...             (BASELINE.json config 5: ViT-B/8, 64x64 tokens, B = 128 per GPU)

One "step" = ``HotPathStep.step`` (wild_visual_navigation_b200/hot_path.py — the object tests/test_bench_path_gpu.py
holds to the oracle) over one batch of synthetic frames per GPU:
  DINO ViT forward -> STEGO head -> per-image k-means of the code (run_clustering=True, the reference's default) ->
  per-pixel cluster argmax -> relabel -> per-segment feature pooling + centroids + adjacency -> per-pixel
  traversability MLP (trav + confidence maps) -> one online train step (fwd + loss + bwd + Adam) on the pooled rows,
with the MLP statistics / gradient all-reduced by the library's NCCL communicator when N > 1 (weak scaling).
STEGO's flip-TTA (a second backbone pass) is OFF in the headline and in both arms; ``variants.flip_tta`` in the JSON
line is the same step with it ON, measured in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

METRIC = "frames/sec end-to-end (DINO feat + seg + MLP train-step) at 448x448"
PATCH = 8
CONFIGS = {
    # BASELINE.json configs[2] (+ configs[1]'s per-pixel maps): the configuration the metric is quoted on
    "c3": dict(backbone="vit_small", img=448, batch=32, dim=384, heads=6, depth=12,
               label="C3+C2: ViT-S/8@448"),
    # BASELINE.json configs[4]: ViT-B/8 "at 518x518" -> the stride-8 conv floors 518 to a 64x64 token grid (512 px);
    # frames here are 512x512 (the 6 border pixels of a 518 crop never reach the conv), B = 128 per GPU
    "c5": dict(backbone="vit_base", img=512, batch=128, dim=768, heads=12, depth=12,
               label="C5: ViT-B/8, 64x64 tokens (518 floors to 512)"),
}
IMG, BATCH = CONFIGS["c3"]["img"], CONFIGS["c3"]["batch"]   # the headline workload (tests import these)
K_IMAGE_CLUSTERS, KMEANS_ITERS = 20, 10


def read_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("bf16_tflops_sustained", 1400.0), d.get("hbm_gbs", 6650.0), "measured"
    return 1400.0, 6650.0, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region (B200_PROFILING.md)."""

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm = sorted(float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit())
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            for i, n in enumerate(names):
                if len(r) > 3 + i and r[3 + i].lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def make_weights(config="c3"):
    from oracle.dino_vit import ViTConfig, synthetic_state_dict
    from oracle.stego_head import synthetic_head

    c = CONFIGS[config]
    cfg = ViTConfig.from_name(c["backbone"], PATCH, c["img"])
    # ViT-B: the qkv std is scaled so that the attention logits keep the spread they have at D = 384 (see
    # tests/test_path_gpu.py::test_vit_base_tokens_parity_512 for both settings)
    attn_std = 0.09 if c["dim"] == 384 else 0.09 / 2 ** 0.5
    return cfg, synthetic_state_dict(cfg, seed=1, attn_std=attn_std), synthetic_head(cfg.dim, 90, 32, 27, seed=3)


def synthetic_images(n_sets, batch, seed, img=IMG):
    g = torch.Generator().manual_seed(seed)
    return [torch.rand(batch, 3, img, img, generator=g) for _ in range(n_sets)]


DUMP_MAX_ELEMENTS = 1 << 20   # per output array of --dump-outputs
DUMP_MAX_BYTES = 64 << 20     # all arrays of --dump-outputs together


def dump_outputs(out_dir, outputs):
    """Writes every tensor of ``outputs`` as ``out_dir/<name>.npy``: floating tensors as float32, integer and bool ones as
    float64 (exact).  A tensor of more than DUMP_MAX_ELEMENTS elements is written flattened, as the elements at
    DUMP_MAX_ELEMENTS sorted flat indices drawn from a generator seeded with 0: the same shape gives the same sample, so
    the files of two builds compare element for element.  More than DUMP_MAX_BYTES in all raises before anything is
    written."""
    import numpy as np

    arrays = {}
    for name, t in outputs.items():
        if t is None:
            continue
        t = t.detach()
        if t.numel() > DUMP_MAX_ELEMENTS:
            g = torch.Generator().manual_seed(0)
            idx = torch.randint(t.numel(), (DUMP_MAX_ELEMENTS,), generator=g).sort().values
            t = t.reshape(-1)[idx.to(t.device)]
        arrays[name] = (t.float() if t.is_floating_point() else t.double()).cpu().numpy()
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_MAX_BYTES:
        raise RuntimeError(f"--dump-outputs: {total} bytes of outputs, more than {DUMP_MAX_BYTES}")
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


# ------------------------------------------------------------------------------------------------
# reference arm / cpu baseline / gpu-eager baseline: the oracle (a port of the pure-Python reference path)
# ------------------------------------------------------------------------------------------------
def oracle_frames_per_s(config, frames_per_step, steps, warmup, device, cores=None, sdpa=False):
    """The reference's own order of operations (eager fp32 PyTorch, frame by frame, oracle/pipeline.py) on ``device``:
    ViT -> STEGO head + k-means + argmax -> relabel / adjacency / centers / pooling -> per-pixel MLP -> one train step."""
    import oracle.dino_vit as dv
    from oracle.pipeline import cpu_step
    from oracle.wvn_path import mlp_init

    if cores:
        torch.set_num_threads(cores)
    cfg, sd, hd = make_weights(config)
    sd = {k: v.to(device) for k, v in sd.items()}
    hd = {k: v.to(device) for k, v in hd.items()}
    mlp_sd = {k: v.to(device) for k, v in mlp_init(cfg.dim, (256, 32), seed=42).items()}
    opt = None
    mean, std = torch.tensor([0.3], device=device), torch.tensor([0.1], device=device)
    imgs = synthetic_images(1, frames_per_step, seed=0, img=CONFIGS[config]["img"])[0].to(device)
    dv.USE_SDPA = sdpa
    try:
        times = []
        for i in range(warmup + steps):
            if device != "cpu":
                torch.cuda.synchronize()
            t0 = time.perf_counter()
            _, _, mlp_sd, opt, _ = cpu_step(imgs, sd, cfg, hd, mlp_sd, opt, mean, std, supervision_seed=2 + i,
                                            n_image_clusters=K_IMAGE_CLUSTERS, kmeans_iters=KMEANS_ITERS)
            if device != "cpu":
                torch.cuda.synchronize()
            times.append(time.perf_counter() - t0)
    finally:
        dv.USE_SDPA = False
    t = sum(times[warmup:])
    return frames_per_step * steps / t, 1000.0 * t / steps


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = min(os.cpu_count() or 1, args.cpu_threads) if args.cpu_threads > 0 else (os.cpu_count() or 1)
    fps, ms = oracle_frames_per_s(args.config, args.cpu_frames, args.steps, args.warmup, "cpu", cores)
    sample = (f"{args.cpu_frames} frame(s) per step, {args.warmup} warm-up + {args.steps} timed steps, oracle port of the "
              f"reference path (eager fp32 torch, {cores} threads)")
    line = {
        "impl": "reference", "metric": METRIC, "value": fps, "unit": "frames/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, frames_per_step=args.cpu_frames),
        "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


def workload_config(args, frames_per_step):
    c = CONFIGS[args.config]
    return {"workload": f"{c['label']} -> STEGO head + per-image k-means (K={K_IMAGE_CLUSTERS}, {KMEANS_ITERS} iterations) + "
                        "per-pixel argmax -> relabel -> segment pooling/centroids/adjacency -> per-pixel MLP trav+confidence "
                        "-> online train step (fwd+loss+bwd+Adam)",
            "frames_per_gpu_per_step": frames_per_step, "image": f"{c['img']}x{c['img']}",
            "backbone": f"DINO {c['backbone']}/8 (random-init, seeded)", "stego_flip_tta": False, "run_clustering": True,
            "parallelism": f"dp{args.gpus} (independent frames; in-library NCCL all-reduce of MLP stats + grads)",
            "l2": "inputs rotate over 3 image batches (3 x 77 MB > 126 MB L2); activations >> L2"}


# ------------------------------------------------------------------------------------------------
# B200 arm
# ------------------------------------------------------------------------------------------------
def run_b200(args):
    import ctypes

    import torch.distributed as dist

    from wild_visual_navigation_b200 import HotPathStep, _C

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = f"cuda:{local}"
    pg = None
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device(dev))
        pg = dist.group.WORLD
    _C.require_device()
    lib = _C.lib()

    c = CONFIGS[args.config]
    S = c["img"]
    cfg, sd, hd = make_weights(args.config)
    B = args.batch if args.batch > 0 else c["batch"]
    chunk = args.chunk if args.chunk > 0 else 32
    hp = HotPathStep(dev, sd, hd, batch=B, input_size=S, backbone_type=c["backbone"], patch_size=PATCH, chunk=chunk,
                     flip_tta=False, run_clustering=True, n_image_clusters=K_IMAGE_CLUSTERS, process_group=pg)
    smax = hp.smax
    # synthetic supervision for up to B*smax pooled rows (SURVEY.md §8d), indexed by the compacted row number
    g = torch.Generator().manual_seed(2 + rank)
    yv_all = (torch.rand(B * smax, generator=g) < 0.16).to(dev)
    y_all = torch.where(yv_all, torch.rand(B * smax, generator=g).clamp(min=0.001).to(dev), torch.zeros(B * smax, device=dev))

    frames = synthetic_images(3, B, seed=100 + rank, img=S)
    if args.ingest == "u8":
        frames = [(t * 255).round().to(torch.uint8).permute(0, 2, 3, 1).contiguous() for t in frames]
    host_imgs = [t.pin_memory() for t in frames]
    dev_imgs = [t.to(dev) for t in host_imgs]

    def step(img):
        return hp.step(img, y_all, yv_all)

    # ---- end-to-end leg: every step copies its frames host->device (pinned) and EVERYTHING the feature node publishes
    # or logs device->host — trav / conf maps, the int32 segment image, pooled features, centers, edge list (+ counts)
    # and the loss metrics (wvn_feature_extractor_node.py:373-393, wvn_learning_node.py train log) — on copy streams so
    # that step k's transfers overlap step k-1 / k+1's compute (double-buffered, as a camera loop around the API would).
    def host_like(t, dtype=None):
        return torch.empty(t.shape, dtype=dtype or t.dtype).pin_memory()

    r0 = step(dev_imgs[0])
    torch.cuda.synchronize()
    out_keys = ["trav", "conf", "seg", "feat", "centers", "edges", "n_edges", "n_segments"]
    host_out = {k: host_like(r0[k], torch.int32 if k == "seg" else None) for k in out_keys}
    host_out["metrics"] = torch.empty(6).pin_memory()
    d2h_bytes = sum(t.numel() * t.element_size() for t in host_out.values())
    s_in, s_out = torch.cuda.Stream(), torch.cuda.Stream()
    img_buf = [torch.empty_like(host_imgs[0], device=dev) for _ in range(2)]
    out_buf = [{k: torch.empty(v.shape, dtype=v.dtype, device=dev) for k, v in host_out.items()} for _ in range(2)]
    ev_in = [torch.cuda.Event() for _ in range(2)]
    ev_used = [torch.cuda.Event() for _ in range(2)]
    ev_done = [torch.cuda.Event() for _ in range(2)]
    ev_out = [torch.cuda.Event() for _ in range(2)]
    state = {"primed": False}

    def h2d(k):
        with torch.cuda.stream(s_in):
            s_in.wait_event(ev_used[k % 2])                        # compute no longer reads this buffer
            img_buf[k % 2].copy_(host_imgs[k % 3], non_blocking=True)
            ev_in[k % 2].record(s_in)

    def step_e2e(k):
        cur = torch.cuda.current_stream()
        if not state["primed"]:
            h2d(k)
            state["primed"] = True
        cur.wait_event(ev_in[k % 2])
        h2d(k + 1)                                                 # prefetch the next step's frames
        r = step(img_buf[k % 2])
        ev_used[k % 2].record(cur)
        cur.wait_event(ev_out[k % 2])                              # previous D2H out of this slot finished
        ob = out_buf[k % 2]
        for key in out_keys:
            ob[key].copy_(r[key])                                  # (seg: int64 -> the int32 image the node publishes)
        ob["metrics"].copy_(hp.te._trainer.metrics)
        ev_done[k % 2].record(cur)
        with torch.cuda.stream(s_out):
            s_out.wait_event(ev_done[k % 2])
            for key, h in host_out.items():
                h.copy_(ob[key], non_blocking=True)
            ev_out[k % 2].record(s_out)

    def drain_e2e():
        torch.cuda.current_stream().wait_stream(s_out)
        torch.cuda.current_stream().wait_stream(s_in)
        state["primed"] = False

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, finish=None):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for k in range(steps):
            fn(k)
        if finish is not None:
            finish()                                               # the last D2H is inside the timed region
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return ms.item()

    for k in range(args.warmup):
        step(dev_imgs[k % 3])
    if args.profile_only:  # short, launch-list friendly run for ncu (no CPU leg, no e2e leg)
        for k in range(args.steps):
            step(dev_imgs[k % 3])
        torch.cuda.synchronize()
        print(json.dumps({"profile_only": True, "launches": int(lib.wvn_launch_count())}))
        return
    for k in range(min(2, args.warmup)):
        step_e2e(k)
    drain_e2e()

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    lib.wvn_profile_enable(3 if args.profile_gemm else 1)   # CUDA events around the roofline kernel's launches
    l0 = lib.wvn_launch_count()
    last = {}

    def timed_step(k):
        r = step(dev_imgs[k % 3])
        if k == args.steps - 1:   # only the last result: earlier steps' outputs are freed as without the dump
            last["r"] = r

    total_ms = timed(timed_step, args.steps)
    launches = lib.wvn_launch_count() - l0
    prof_ms = (ctypes.c_float * 2)()
    prof_n = (ctypes.c_longlong * 2)()
    _C.check(lib.wvn_profile_collect(prof_ms, prof_n))
    lib.wvn_profile_enable(0)
    if args.dump_outputs and rank == 0:
        # the step's result dict (maps, segmentation, pooled rows, graph, tokens) and the train step's loss metrics
        dump_outputs(args.dump_outputs, last["r"] | {"metrics": hp.te._trainer.metrics})
    e2e_ms = timed(step_e2e, args.steps, finish=drain_e2e)
    clocks = sampler.stop() if rank == 0 else None

    ms_per_step = total_ms / args.steps
    value = world * B * args.steps / (total_ms / 1000.0)
    e2e_value = world * B * args.steps / (e2e_ms / 1000.0)

    # ---- extra legs (N = 1 only; outside the timed regions above): flip-TTA variant, B = 1 latency, GPU-eager baseline
    variants, latency, gpu_eager = None, None, None
    if world == 1 and not args.no_extras:
        # per-frame latency of the deployment case (one camera frame at a time, B = 1): median over 30 frames after
        # 5 warm-ups, maps + pooled rows left on the device
        from wild_visual_navigation_b200 import HotPathStep as _HP

        hp1 = _HP(dev, sd, hd, batch=1, input_size=S, backbone_type=c["backbone"], patch_size=PATCH, chunk=1,
                  flip_tta=False, run_clustering=True, n_image_clusters=K_IMAGE_CLUSTERS)
        one = dev_imgs[0][:1].contiguous()
        lat = []
        for i in range(35):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            hp1.step(one, y_all, yv_all)
            e1.record()
            torch.cuda.synchronize()
            if i >= 5:
                lat.append(e0.elapsed_time(e1))
        lat.sort()
        latency = {"batch": 1, "ms_median": lat[len(lat) // 2], "ms_p90": lat[int(len(lat) * 0.9)],
                   "note": "HotPathStep.step on one frame (feature extraction + per-pixel maps + train step), device-timed"}
        try:  # the same step replayed as one CUDA graph (launch latency removed)
            hp1.capture(one, y_all, yv_all)
            glat = []
            for i in range(35):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                hp1.replay(one)
                e1.record()
                torch.cuda.synchronize()
                if i >= 5:
                    glat.append(e0.elapsed_time(e1))
            glat.sort()
            latency["graph_ms_median"], latency["graph_ms_p90"] = glat[len(glat) // 2], glat[int(len(glat) * 0.9)]
        except Exception as e:  # noqa: BLE001 — the eager figure stands; say why the graph one is missing
            latency["graph_error"] = str(e)[:200]
        del hp1
        hpt = _HP(dev, sd, hd, batch=B, input_size=S, backbone_type=c["backbone"], patch_size=PATCH, chunk=chunk,
                  flip_tta=True, run_clustering=True, n_image_clusters=K_IMAGE_CLUSTERS)
        fimgs = [t if t.dtype != torch.uint8 else t.permute(0, 3, 1, 2).float().div(255) for t in dev_imgs]
        for k in range(2):
            hpt.step(fimgs[k % 3], y_all, yv_all)
        ns = max(3, args.steps // 2)
        tta_ms = timed(lambda k: hpt.step(fimgs[k % 3], y_all, yv_all), ns)
        variants = {"flip_tta": {"value": B * ns / (tta_ms / 1000.0), "unit": "frames/s", "steps": ns,
                                 "note": "same step with STEGO's flip test-time augmentation (two backbone passes)"}}
        del hpt
        torch.cuda.empty_cache()
        if args.gpu_eager_frames > 0:
            ef, _ = oracle_frames_per_s(args.config, args.gpu_eager_frames, 2, 1, dev)
            es, _ = oracle_frames_per_s(args.config, args.gpu_eager_frames, 2, 1, dev, sdpa=True)
            gpu_eager = {"value": ef, "sdpa_value": es, "unit": "frames/s", "kind": "port",
                         "sample": f"{args.gpu_eager_frames} frame(s) per step, 1 warm-up + 2 timed steps, the oracle port of the "
                                   "reference path as eager fp32 PyTorch on this same GPU (tf32 off); sdpa_value = the same with "
                                   "F.scaled_dot_product_attention instead of the materialised attention",
                         "speedup_e2e": e2e_value / ef if ef > 0 else None}
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peak_tf, peak_gbs, peak_src = read_peaks()
    n_tok = (S // PATCH) ** 2 + 1
    attn_flop_per_frame_head = 4.0 * n_tok * n_tok * 64
    attn_launches = max(1, prof_n[0])
    frames_per_launch = B * c["depth"] * args.steps / attn_launches
    attn_avg_ms = prof_ms[0] / attn_launches
    flops_per_launch = attn_flop_per_frame_head * c["heads"] * frames_per_launch
    achieved_tf = flops_per_launch / (attn_avg_ms * 1e-3) / 1e12 if attn_avg_ms > 0 else 0.0
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "attention_traffic.json")
    if os.path.exists(tpath) and args.config == "c3":
        traffic = json.load(open(tpath)).get("dram_bytes_per_launch")

    cores = min(os.cpu_count() or 1, args.cpu_threads) if args.cpu_threads > 0 else (os.cpu_count() or 1)
    cpu_fps = None
    if args.cpu_frames > 0 and world == 1:
        cpu_fps = oracle_frames_per_s(args.config, args.cpu_frames, 2, 1, "cpu", cores)[0]

    vit_gflop = 315.1 if args.config == "c3" else 1316.0
    line = {
        "metric": METRIC, "value": value, "unit": "frames/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "bf16 operands / fp32 accumulate (ViT, STEGO head, per-pixel MLP); fp32 (k-means, train step)",
        "data": "synthetic",
        "config": workload_config(args, B) | {"vit_chunk_frames": chunk, "ingest": args.ingest, "bench_config": args.config},
        "e2e": {"value": e2e_value, "unit": "frames/s", "h2d_bytes_per_step": host_imgs[0].numel() * host_imgs[0].element_size(),
                "d2h_bytes_per_step": d2h_bytes, "ms_per_step": e2e_ms / args.steps,
                "d2h": "trav + conf maps, int32 segment image, pooled features, centers, edges (+ counts), loss metrics"},
        "gpu_launches": int(launches), "gpu_launches_per_step": launches / args.steps,
        "clocks": clocks,
        "roofline": {"kernel": {"1": "attention_kernel", "2": "attention2_kernel", "3": "attention3_kernel", "5": "attention5_kernel"}.get(os.environ.get("WVN_ATTN_IMPL", "5"), "?") + " (fused QK^T-softmax-PV, tcgen05)", "bound": "tensor",
                     "achieved": achieved_tf, "peak": peak_tf, "unit": "TFLOP/s", "frac": achieved_tf / peak_tf,
                     "peak_source": f"{peak_src} bf16_tflops_sustained (kernel timed inside the step)",
                     "traffic": traffic, "avg_launch_ms": attn_avg_ms, "launches": int(prof_n[0]),
                     "share_of_step": prof_ms[0] / total_ms if total_ms > 0 else None,
                     "gemm_share_of_step": prof_ms[1] / total_ms if (total_ms > 0 and prof_n[1] > 0) else None,
                     "gemm_launches": int(prof_n[1]) if prof_n[1] > 0 else None},
        "cpu_baseline": {"value": cpu_fps, "unit": "frames/s", "cores": cores, "kind": "port",
                         "sample": f"{args.cpu_frames} frame(s) per step, 1 warm-up + 2 timed steps of the oracle port "
                                   f"(eager fp32 torch, {cores} host threads)"},
        "gpu_eager_baseline": gpu_eager, "latency": latency, "variants": variants,
        "whole_path_tflops": value * (vit_gflop + 1.36 + 47.69 * (S / 448.0) ** 2) / 1000.0,
    }
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="c3", choices=sorted(CONFIGS), help="c3 = the metric's configuration (ViT-S/8@448, "
                    "B=32 per GPU); c5 = BASELINE.json config 5 (ViT-B/8, 64x64 tokens, B=128 per GPU)")
    ap.add_argument("--batch", type=int, default=0, help="frames per GPU per step (0 = the config's)")
    ap.add_argument("--chunk", type=int, default=32, help="frames per ViT activation chunk")
    ap.add_argument("--cpu-frames", type=int, default=1, help="frames per step of the bounded CPU sample (~3-6 s per frame)")
    ap.add_argument("--cpu-threads", type=int, default=32,
                    help="torch CPU threads for the CPU legs (0 = all host cores).  Measured on the 128-thread B200 host: the "
                         "eager oracle runs 1 frame in ~3 s on 32 threads and in 42 s on 128 (thread sync on its many small "
                         "ops), so 32 is what 'all the threads it can use' means for this code")
    ap.add_argument("--gpu-eager-frames", type=int, default=2, help="frames per step of the GPU-eager oracle leg (0 = skip)")
    ap.add_argument("--no-extras", action="store_true", help="skip the latency / flip-TTA / GPU-eager legs")
    ap.add_argument("--profile-only", action="store_true", help="setup + warmup + steps only (for ncu)")
    ap.add_argument("--profile-gemm", action="store_true",
                    help="also time every GEMM launch with CUDA events (gemm_share_of_step; ~280 extra event pairs per step)")
    ap.add_argument("--ingest", default="f32", choices=["f32", "u8"],
                    help="frame format at the boundary: f32 = (B,3,H,W) float in [0,1] (the reference's boundary, "
                         "BASELINE.json); u8 = camera frames (B,H,W,3) uint8, ingest fused into the patch loader (SURVEY.md §8f)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the outputs of the last one as DIR/<name>.npy (float32 / float64; "
                         "arrays above 2^20 elements as a fixed, seeded sample of them) to compare two builds")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and (args.impl != "b200" or args.profile_only):
        ap.error("--dump-outputs writes the timed steps of --impl b200 (not with --profile-only)")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
