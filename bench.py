#!/usr/bin/env python
"""bench.py - images/sec of the MonoFlex per-image hot path on B200 (BASELINE.json), synthetic 384x1280 KITTI-shaped batches,
random-init weights of the reference architecture.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--batch 8] [--precision strict|fast] [--impl ours|reference|torch_gpu]
    python bench.py --train [--gpus N] [--graph 1|0] ...                       # BASELINE configs[2] / configs[4]
    python bench.py ... --dump-outputs DIR     # also write what the last timed step returned to DIR/<name>.npy

Inference (configs[1]; --batch 32 = configs[3]): a "step" = one pass of DLA-34 + IDA-up + DCNv2 + predictor + NMS / top-k / 3D
decode over one batch. ONE JSON line (rank 0):
  value        images/s, inputs resident in HBM, CUDA events on the launching stream, max over ranks - in the HEADLINE precision:
               "strict" (fp16 hi/lo pair arithmetic, the mode that meets the 1e-3 parity contract with the fp32 reference)
  e2e          images/s through the public module API from pinned HOST buffers (H2D of the images and D2H of the detections
               inside the timed region)
  modes        the same two numbers for both precisions ("fast" = single fp16 tensor-core pass, 2-4e-3 end to end)
  roofline     the kernel GROUP with the largest share of the step's device time (per-launch CUDA events): algorithmic FLOPs /
               its time vs the measured bf16 peak; `blocks` lists every group (stem, base convs, DCN, offset convs, head, ...)
               with its time share, TFLOP/s and - where an ncu capture is committed - the tensor-pipe % from profiles/
  decode_roofline  the two decode kernels vs the measured HBM peak
  cpu_baseline the CPU oracle (port of the reference's torch path) timed on this box's host cores on a bounded sample
--train: one step = train-mode forward + 11-term loss + whole-network backward + gradient exchange + AdamW (see bench_train).
--impl reference: the reference's CPU path (oracle port; its native extension cannot be built on torch >= 1.11, DESIGN.md) with
every useful host thread, each step one bounded sample (a batch-1 forward / train step); prints the steps it actually ran.
--impl torch_gpu: the same restated reference graph executed by stock PyTorch on the GPU (cuDNN convs + torchvision
deform_conv2d), TF32 off and on - the "practical bar" of SURVEY 8d, stated as context, never the product path.
"""
import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

H, W = 384, 1280
METRIC = "images/sec @ 384x1280 batch 8 (DLA-34+DCNv2+heads+decode inference)"
FWD_GF_PER_IMG = 178.6               # SURVEY 8d: conv FLOPs / image, forward
TRAIN_GF_PER_IMG = 3 * FWD_GF_PER_IMG   # dgrad + wgrad = 2x forward (DCN backward counted as 2x its forward contraction)
TRAIN_METRIC = "images/sec @ 384x1280 batch 8/GPU (full train step: fwd+bwd+AdamW, DLA-34+DCNv2+heads+losses)"


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("hbm_gbs", 6650.0), d.get("bf16_tflops_sustained", 1400.0), d.get("bf16_tflops", 1590.0), "measured"
    return 6650.0, 1400.0, 1590.0, "fallback"


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.stop_flag = index, [], False

    def run(self):
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                f = [v.strip() for v in out.strip().split(",")]
                if len(f) >= 6:
                    self.samples.append(f)
            except Exception:
                pass
            time.sleep(0.1)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unsampled"]}
        sm = sorted(float(s[0]) for s in self.samples)
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(s[2 + i].lower().startswith("active") for s in self.samples)]
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": float(self.samples[0][1]), "reasons": reasons,
                "samples": len(sm)}


def cpu_threads():
    """torch-CPU convolutions stop scaling (and the gather-heavy DCN restatement regresses) beyond ~32 threads:
    measured 91 s/img with 128 threads vs 19 s/img with fewer on the round-1 box. Use at most 32."""
    return min(os.cpu_count() or 1, 32)


def dump_outputs(out_dir, arrays):
    """{name: array} -> out_dir/<name>.npy, float32 arrays as they are and everything else as float64. The inputs are
    seeded, so two builds run with the same arguments can be compared output for output."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        a = np.asarray(a)
        np.save(os.path.join(out_dir, name + ".npy"), a if a.dtype == np.float32 else a.astype(np.float64))


# ------------------------------------------------------------------------------------------------ CPU reference path
def cpu_eval_steps(max_steps, warmup, threads, budget_s):
    """The reference's CPU inference path (oracle port): batch-1 full-resolution eval forwards, at most `max_steps` timed ones
    within `budget_s` seconds. Returns (seconds per image, timed steps)."""
    import torch
    from monoflex_b200 import synthetic as syn
    from oracle import monoflex_oracle as mo
    torch.set_num_threads(threads)
    sd = syn.make_state_dict(0)
    x = syn.make_images(1, H, W)
    tg = syn.make_targets(1, W // 4, H // 4)
    ts, t_start = [], time.perf_counter()
    with torch.no_grad():
        for i in range(warmup + max_steps):
            t0 = time.perf_counter()
            mo.detector_eval(sd, x, tg['edge_indices'], tg['edge_len'], tg['calib_P'], tg['pad_size'], tg['size'], 0.2)
            dt = time.perf_counter() - t0
            if i >= warmup:
                ts.append(dt)
            if time.perf_counter() - t_start + dt > budget_s and len(ts) >= 1:
                break
    return sum(ts) / len(ts), len(ts)


def cpu_train_steps(max_steps, warmup, threads, budget_s):
    """The reference's CPU training path (oracle port + torch autograd + torch.optim.AdamW with the reference's param groups):
    batch-1 full-resolution train steps. Returns (seconds per image, timed steps)."""
    import torch
    from monoflex_b200 import synthetic as syn
    from oracle import monoflex_oracle as mo
    torch.set_num_threads(threads)
    sd = {k: (v.clone().requires_grad_(True) if v.is_floating_point() and "running_" not in k else v)
          for k, v in syn.make_state_dict(seed=0).items()}
    params = [{"params": [v], "lr": 3e-4 * (2.0 if "bias" in k else 1.0)} for k, v in sd.items() if v.requires_grad]
    opt = torch.optim.AdamW(params, lr=3e-4, weight_decay=1e-5, betas=(0.9, 0.99))
    fields = syn.make_train_targets(1, empty_image=1)
    images = syn.make_images(1, H, W, seed=1)
    idx, n, _ = syn.edge_indices()
    ts, t_start = [], time.perf_counter()
    for i in range(warmup + max_steps):
        t0 = time.perf_counter()
        loss, _ = mo.detector_train_losses(sd, images, fields, idx.unsqueeze(0), torch.tensor([n]), [syn.KITTI_P2])
        opt.zero_grad()
        sum(loss.values()).backward()
        opt.step()
        dt = time.perf_counter() - t0
        if i >= warmup:
            ts.append(dt)
        if time.perf_counter() - t_start + dt > budget_s and len(ts) >= 1:
            break
    return sum(ts) / len(ts), len(ts)


def reference_arm(args, config, cores):
    """`--impl reference`: CPU path only, rank 0, bounded samples, prints the steps it actually ran."""
    budget = float(os.environ.get("MF_REF_BUDGET_S", "150"))
    warm = 1 if args.warmup > 0 else 0
    if args.train:
        sec, n = cpu_train_steps(args.steps, warm, cores, budget)
        sample = "%d batch-1 full-resolution train steps (fwd + bwd + AdamW) of the CPU oracle port, %.0f s budget" % (n, budget)
        metric = TRAIN_METRIC
    else:
        sec, n = cpu_eval_steps(args.steps, warm, cores, budget)
        sample = "%d batch-1 full-resolution eval forwards (incl. NMS / top-k / 3D decode) of the CPU oracle port, %.0f s budget" % (n, budget)
        metric = METRIC
    v = 1.0 / sec
    print(json.dumps({"impl": "reference", "metric": metric, "value": v, "unit": "images/s", "n_gpus": args.gpus,
                      "steps": n, "steps_requested": args.steps, "warmup": warm, "ms_per_step": sec * 1e3,
                      "step_definition": "one bounded sample = ONE image (the reference's PostProcessor is batch-1 only, SURVEY H8)",
                      "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                      "config": config,
                      "cpu_baseline": {"value": v, "unit": "images/s", "cores": cores, "kind": "port", "sample": sample +
                                       " (the reference's torch path restated; its _ext cannot be built on torch 2.11)"},
                      "e2e": {"value": v, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))


# ------------------------------------------------------------------------------------------------ stock-PyTorch GPU arm
def torch_gpu_arm(args, config):
    """SURVEY 8d "practical bar": the restated reference graph on the GPU through stock PyTorch (cuDNN fp32 convs,
    torchvision.ops.deform_conv2d for DCNv2), TF32 off and on. Context only."""
    import torch
    import torchvision
    from monoflex_b200 import synthetic as syn
    from oracle import monoflex_oracle as mo
    dev = torch.device("cuda", 0)
    B = args.batch
    sd = {k: v.to(dev) for k, v in syn.make_state_dict(0).items()}
    x = syn.make_images(B, H, W).to(dev)
    tg = syn.make_targets(B, W // 4, H // 4)
    ei, el = tg['edge_indices'].to(dev), tg['edge_len'].to(dev)
    orig = mo.dcn_v2_forward
    mo.dcn_v2_forward = lambda xx, w, b, off, m: torchvision.ops.deform_conv2d(xx, off, w, b, padding=1, mask=m)
    out = {}
    try:
        for tf32 in (False, True):
            torch.backends.cudnn.allow_tf32 = tf32
            torch.backends.cuda.matmul.allow_tf32 = tf32
            with torch.no_grad():
                for _ in range(2):
                    feats = mo.backbone(sd, x)
                    mo.predictor(sd, feats, ei, el)
                torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(args.steps):
                    feats = mo.backbone(sd, x)
                    mo.predictor(sd, feats, ei, el)
                e1.record()
                torch.cuda.synchronize()
            out["tf32_on" if tf32 else "tf32_off"] = B * args.steps / (e0.elapsed_time(e1) * 1e-3)
    finally:
        mo.dcn_v2_forward = orig
    print(json.dumps({"impl": "torch_gpu", "metric": METRIC, "value": out["tf32_off"], "unit": "images/s", "n_gpus": 1,
                      "steps": args.steps, "higher_is_better": True, "dtype": "f32 (cuDNN) / tf32", "data": "synthetic",
                      "config": config, "images_per_s": out,
                      "note": "backbone + predictor only (no decode), eager PyTorch kernels: context for the product numbers"}))


# ------------------------------------------------------------------------------------------------ per-launch roofline
def launch_flops(name, a):
    """ALGORITHMIC FLOPs (2 x MACs of the reference's layer) of one C-ABI launch - strict-precision launches issue 3x as many
    tensor-core products, that is an implementation cost and not counted."""
    if name == "mf_conv2d_nhwc_f16":
        _, _, b_, h_, w_, cin, _, _, _, kh, kw, stride, pad, cout = a[:14]
        ho, wo = (h_ + 2 * pad - kh) // stride + 1, (w_ + 2 * pad - kw) // stride + 1
        return 2.0 * b_ * ho * wo * cout * kh * kw * cin
    if name == "mf_dcn_nhwc_f16":
        _, _, b_, h_, w_, cin = a[:6]
        return 2.0 * b_ * h_ * w_ * a[11] * 9 * cin
    if name == "mf_head_fused":          # nbranch x (3x3 Cin->256) + the 1x1 heads (53 real output channels)
        _, _, b_, h_, w_, cin = a[:6]
        return 2.0 * b_ * h_ * w_ * (a[11] * 256 * 9 * cin + 53 * 256)
    if name == "mf_conv2d_rows_f16":
        _, b_, h_, w_, cin, _, _, _, _, kh, kw, stride, pad, cout = a[:14]
        ho, wo = (h_ + 2 * pad - kh) // stride + 1, (w_ + 2 * pad - kw) // stride + 1
        return 2.0 * b_ * ho * wo * cout * kh * kw * (3 if cin == 8 else cin)
    if name == "mf_conv2d_rows_f16x2":
        _, b_, h_, w_, cin, _, _, _, _, _, kh, kw, stride, pad, cout = a[:15]
        ho, wo = (h_ + 2 * pad - kh) // stride + 1, (w_ + 2 * pad - kw) // stride + 1
        return 2.0 * b_ * ho * wo * cout * kh * kw * (3 if cin == 8 else cin)
    if name == "mf_conv2d_nhwc_f16x2":
        _, _, _, b_, h_, w_, cin, _, _, _, kh, kw, stride, pad, cout = a[:15]
        ho, wo = (h_ + 2 * pad - kh) // stride + 1, (w_ + 2 * pad - kw) // stride + 1
        return 2.0 * b_ * ho * wo * cout * kh * kw * (3 if (cin == 16 and kh == 7) else cin)
    if name == "mf_dcn_nhwc_f16x2":
        _, _, _, b_, h_, w_, cin = a[:7]
        return 2.0 * b_ * h_ * w_ * a[12] * 9 * cin
    if name == "mf_head_conv_f16x2":     # strict: nbranch x (3x3 Cin->256) with the 1x1 heads (ntot outputs) in the epilogue
        _, _, _, b_, h_, w_, cin = a[:7]
        return 2.0 * b_ * h_ * w_ * (a[10] * 256 * 9 * cin + a[16] * 256)
    return 0.0


def launch_group(name, a, plan_kind):
    """role of a launch in the step (the groups of SURVEY 8d / VERDICT item 7)"""
    if name in ("mf_conv2d_rows_f16", "mf_conv2d_rows_f16x2"):
        return "stem"
    if name in ("mf_dcn_nhwc_f16", "mf_dcn_nhwc_f16x2"):
        return "dcn"
    if name in ("mf_head_fused", "mf_head_conv_f16x2"):
        return "head"
    if name == "mf_head2_reduce":
        return "head_1x1"
    if name in ("mf_conv2d_nhwc_f16", "mf_conv2d_nhwc_f16x2"):
        x2 = name.endswith("x2")
        cin, kh, cout = (a[6], a[10], a[14]) if x2 else (a[5], a[9], a[13])
        hh = a[4] if x2 else a[3]
        if plan_kind == "head":
            return "head" if kh == 3 else ("head_1x1" if hh > 1 else "edge_fusion")
        if cout == 27:
            return "offset_convs"
        if hh >= 192 or cin <= 16:
            return "stem"
        return "base_convs"
    if name.startswith("mf_upsample") or name.startswith("mf_maxpool"):
        return "upsample_pool"
    if name.startswith("mf_edge") or name == "mf_sigmoid_clamp":
        return "edge_fusion"
    return "other"


KERNEL_OF_GROUP = {
    "stem": "rows_conv_kernel (csrc/mf_rows.cu) + igemm2_kernel<.., MODE_CONV> for the stride-2 layer",
    "base_convs": "igemm2_kernel<BLOCK_N, MODE_CONV_TMA> (csrc/mf_igemm2.cu): DLA-34 levels 2-5, roots, projects",
    "dcn": "igemm2_kernel<BLOCK_N, MODE_DCN, 16> (csrc/mf_igemm2.cu): fused DCNv2 gather + contraction, 16 layers",
    "offset_convs": "igemm2_kernel<32, MODE_CONV_TMA>: the 16 conv_offset_mask 3x3 convs (27 channels)",
    "head": "predictor 9 x (3x3 64->256 + IABN) + 1x1 heads: head_fused_kernel (fast) / igemm2_kernel<256, MODE_CONV_TMA, 4, HEAD2> "
            "N=2304 pair GEMM with the 1x1 heads contracted in the epilogue (strict)",
    "head_1x1": "head2_reduce_kernel: fixed-order sum of the eight partial planes + bias -> cls / reg maps (strict only)",
    "upsample_pool": "upsample_add / maxpool2 (HBM-bound layout kernels)",
    "edge_fusion": "edge gather + Conv1d GEMM + indexed add + sigmoid",
}


def group_table(rows_b, rows_h, tf_peak):
    table, groups = [], {}
    for kind, rows in (("backbone", rows_b), ("head", rows_h)):
        for name, a, ms in rows:
            gf = launch_flops(name, a) / 1e9
            g = launch_group(name, a, kind)
            table.append({"kernel": name, "group": g, "ms": ms, "gflop": gf})
            e = groups.setdefault(g, {"ms": 0.0, "gflop": 0.0, "launches": 0})
            e["ms"] += ms
            e["gflop"] += gf
            e["launches"] += 1
    total = sum(e["ms"] for e in groups.values())
    for g, e in groups.items():
        e["share_of_step"] = e["ms"] / total
        e["tflops"] = e["gflop"] / e["ms"] if e["ms"] > 0 else 0.0
        e["frac_of_peak"] = e["tflops"] / tf_peak
    return table, groups, total


def ncu_facts(precision):
    """tensor-pipe % / DRAM bytes per launch from the committed ncu captures (profiles/ncu_facts_r02.json), keyed by group"""
    p = os.path.join(ROOT, "profiles", "ncu_facts_r02.json")
    if not os.path.exists(p):
        return {}
    return json.load(open(p)).get(precision, {})


# ------------------------------------------------------------------------------------------------ training bench
def bench_train(args, rank, world, local_rank, config):
    """BASELINE configs[2] (1 GPU) / configs[4] (N GPUs, 8 images each, NCCL gradient all-reduce): one step = train-mode
    forward (batch-statistics BN) + 11-term loss + whole-network backward + gradient exchange + AdamW, through the module API
    the reference trainer calls (engine/trainer.py:103-126 == monoflex_b200.train.Trainer.step)."""
    import torch
    import torch.distributed as dist
    from monoflex_b200 import parallel
    from monoflex_b200 import synthetic as syn
    from monoflex_b200.config import default_cfg
    from monoflex_b200.model.detector import KeypointDetector
    from monoflex_b200.train import Trainer
    assert torch.cuda.is_available(), "bench.py needs a GPU (no CPU fallback)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    parallel.init("nccl", dev)
    B = args.batch
    cfg = default_cfg(width=W, height=H)
    model = KeypointDetector(cfg)
    model.load_state_dict(syn.make_state_dict(0))
    model = model.to(dev)
    sync_bn = bool(args.sync_bn) and world > 1
    if sync_bn:                                   # the reference's own conversion call (tools/plain_train_net.py:131-132)
        model = torch.nn.SyncBatchNorm.convert_sync_batchnorm(model)
    use_graph = args.graph != 0
    tr = Trainer(model, cfg, use_cuda_graph=use_graph, graph_warmup=2)
    n_in = 3
    fields = [syn.make_train_targets(B, seed=5 + rank * n_in + i, empty_image=B) for i in range(n_in)]
    host_tg = [[t.pin_memory() for t in syn.make_train_param_lists(f)] for f in fields]     # as a pin_memory data loader hands them over
    dev_tg = [[t.to(dev) for t in tl] for tl in host_tg]
    host_imgs = [syn.make_images(B, H, W, seed=100 + rank * n_in + i).pin_memory() for i in range(n_in)]
    dev_imgs = [h.to(dev) for h in host_imgs]
    label_bytes = sum(v.numel() * v.element_size() for t in host_tg[0] for v in t.extra_fields.values() if torch.is_tensor(v))

    graph_err = None
    try:
        for i in range(max(3, args.warmup)):
            tr.step(dev_imgs[i % n_in], dev_tg[i % n_in], sync_log=False)
        torch.cuda.synchronize()
    except Exception as e:                       # capture failed: report it and measure the eager step instead
        if not use_graph:
            raise
        graph_err = "%s: %s" % (type(e).__name__, str(e)[:300])
        torch.cuda.synchronize()
        tr.use_cuda_graph, tr._graph = False, None
        model.heads.predictor._targets_preloaded = False
        for i in range(3):
            tr.step(dev_imgs[i % n_in], dev_tg[i % n_in], sync_log=False)
        torch.cuda.synchronize()

    def barrier():
        parallel.barrier()
        torch.cuda.synchronize()

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(args.steps):
        loss_dict, log = tr.step(dev_imgs[i % n_in], dev_tg[i % n_in], sync_log=False)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    if args.dump_outputs and rank == 0:          # the captured step re-uses its loss buffers: read them before the next step
        dump_outputs(args.dump_outputs, dict([("loss_" + k, v.float().cpu().numpy()) for k, v in loss_dict.items()] +
                                             [("log_" + k, v) for k, v in log.resolve().items()]))
    barrier()
    # exposed gradient-exchange time: the NCCL all-reduce of the arena alone, same buckets (N > 1)
    ms_ar = 0.0
    if world > 1:
        from monoflex_b200 import solver
        a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        solver.allreduce_grads(tr.optimizer.arena, tr.bucket_bytes, tr.group)
        barrier()
        a0.record()
        for _ in range(5):
            solver.allreduce_grads(tr.optimizer.arena, tr.bucket_bytes, tr.group)
        a1.record()
        torch.cuda.synchronize()
        ms_ar = a0.elapsed_time(a1) / 5
        barrier()
    # end to end: images + labels from (pinned) host memory every step, the logged losses of EVERY step read back on the host
    # (the reference's trainer logs them per iteration) - one step late: step i's scalars are copied out asynchronously
    # (DeferredLog.snapshot) and read after step i+1 has been enqueued, so the host-side target handling of the next batch
    # overlaps the running step instead of serialising with it
    # The image batch of step i+1 travels host -> device on a copy stream into the other of two staging buffers while step i
    # computes (the usual pinned-memory prefetcher of a training input pipeline); all of it inside the timed region.
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    xbufs = [torch.empty_like(dev_imgs[0]) for _ in range(2)]
    copied = [torch.cuda.Event() for _ in range(2)]
    consumed = [torch.cuda.Event() for _ in range(2)]
    copy_stream, main = torch.cuda.Stream(), torch.cuda.current_stream()

    def prefetch(i):
        with torch.cuda.stream(copy_stream):
            xbufs[i % 2].copy_(host_imgs[i % n_in], non_blocking=True)
            copied[i % 2].record(copy_stream)

    def e2e_loop(n):
        prev_log, last = None, None
        prefetch(0)
        for i in range(n):
            main.wait_event(copied[i % 2])
            tg = [t.to(dev) for t in host_tg[i % n_in]]
            loss_dict, log = tr.step(xbufs[i % 2], tg, sync_log=False)
            consumed[i % 2].record(main)               # the step's copy-in of this staging buffer is enqueued before this point
            if i + 1 < n:
                if i >= 1:
                    copy_stream.wait_event(consumed[(i + 1) % 2])
                prefetch(i + 1)
            if prev_log is not None:
                last = prev_log.resolve()
            prev_log = log
        return prev_log.resolve()

    e2e_loop(2)                                        # untimed: first use of the copy stream and of the pinned log staging
    torch.cuda.synchronize()
    copy_stream.synchronize()
    t0.record()
    last_log = e2e_loop(args.steps)
    t1.record()
    torch.cuda.synchronize()
    assert all(math.isfinite(v) for v in last_log.values())
    ms_e2e = t0.elapsed_time(t1)
    barrier()
    if rank == 0:
        sampler.stop_flag = True
    ms, ms_e2e, ms_ar = parallel.max_over_ranks([ms, ms_e2e, ms_ar], device=dev)
    value = world * B * args.steps / (ms * 1e-3)
    e2e = world * B * args.steps / (ms_e2e * 1e-3)
    if rank == 0:
        hbm, tf_sus, tf_burst, which = peaks()
        ach = value * TRAIN_GF_PER_IMG / 1e3 / world                   # TFLOP/s per GPU, algorithmic
        total = float(sum(v.item() for v in loss_dict.values()))
        n_launch = None
        lp = os.path.join(ROOT, "profiles", "train_step_launches_r02.json")
        if os.path.exists(lp):
            n_launch = json.load(open(lp)).get("launches_per_step")
        line = {"metric": TRAIN_METRIC, "value": value, "unit": "images/s", "n_gpus": world, "steps": args.steps,
                "warmup": max(3, args.warmup), "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "mode": "train",
                "dtype": "f16 operands / activations / activation gradients (loss scale %g), f32 accumulate, f32 master weights, "
                         "moments and weight gradients" % model.loss_scale,
                "data": "synthetic", "config": config, "clocks": sampler.summary(),
                "e2e": {"value": e2e, "unit": "images/s", "h2d_bytes_per_step": B * 3 * H * W * 4 + label_bytes,
                        "d2h_bytes_per_step": 22 * 4, "ms_per_step": ms_e2e / args.steps,
                        "pipeline": "every step's logged losses are read on the host, one step late (async pinned copy): "
                                    "host-side target handling of batch i+1 overlaps step i; the image batch of step i+1 is copied host -> device on "
                                    "a second stream (double-buffered) while step i computes"},
                "gpu_launches": (n_launch * args.steps) if n_launch else None,
                "gpu_launches_note": "kernels of one step counted from the ncu launch list of tools/profile_train_step.py "
                                     "(profiles/train_step_launches_r02.json); with --graph 1 they replay from ONE cudaGraphLaunch",
                "cuda_graph": bool(tr.use_cuda_graph and tr._graph is not None), "cuda_graph_error": graph_err,
                "skipped_steps": tr.optimizer.skipped_steps(), "final_loss": total,
                "roofline": {"bound": "tensor", "kernel": "whole train step (conv fwd + dgrad + wgrad stack)",
                             "achieved": ach, "peak": tf_sus, "unit": "TFLOP/s", "frac": ach / tf_sus, "traffic": None,
                             "algorithmic_gflop_per_image": TRAIN_GF_PER_IMG,
                             "peak_source": "%s bf16 sustained" % which},
                "gradient_exchange": ("none (1 GPU)" if world == 1 else
                                      {"what": "bucketed NCCL all-reduce of the 83.8 MB fp32 gradient arena (3 x 32 MB), 1/world "
                                               "folded into the AdamW kernel; after backward, not overlapped",
                                       "ms_per_step_alone": ms_ar, "share_of_step": ms_ar / (ms / args.steps)}),
                "batchnorm": ("SyncBatchNorm: statistics over the global batch (reference runs/monoflex.yaml USE_SYNC_BN True), 2C doubles "
                              "all-reduced per layer and direction" if sync_bn else
                              "per-GPU batch statistics (USE_SYNC_BN False)")}
        print(json.dumps(line))
    if world > 1:
        # NCCL collectives were captured inside the step's CUDA graph (SyncBatchNorm): tearing the communicator down while the
        # graph still references it hung destroy_process_group on the 2-GPU run of round 2 - drop the graph, drain, then leave
        # without the teardown (a benchmark process; the driver only needs the JSON line and exit code 0)
        sys.stdout.flush()
        tr._graph = None
        torch.cuda.synchronize()
        parallel.barrier()
        os._exit(0)


# ------------------------------------------------------------------------------------------------ inference bench
def time_inference(model, targets, host_imgs, dev_imgs, steps, B, dev, barrier, keep_last=False):
    """-> (ms device-resident, ms end-to-end, d2h bytes, last) for `steps` forwards of `model` in its current precision;
    `last` is what `forward_async(...).result()` returned for the last device-resident step if `keep_last`, else None"""
    import torch
    n_in = len(dev_imgs)
    with torch.no_grad():
        for i in range(3):
            model(dev_imgs[i % n_in], targets)
    torch.cuda.synchronize()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    with torch.no_grad():
        for i in range(steps):
            pending = model.forward_async(dev_imgs[i % n_in], targets)    # no host sync inside the device-resident loop
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    last = pending.result() if keep_last else None     # before the next forward re-uses the decode workspace
    barrier()
    # end to end: pinned host -> H2D (copy stream, one batch ahead) -> model -> D2H of the detections
    copy_stream = torch.cuda.Stream(device=dev)
    bufs = [torch.empty_like(dev_imgs[0]) for _ in range(2)]
    ready = [torch.cuda.Event() for _ in range(2)]
    done = [torch.cuda.Event() for _ in range(2)]

    def prefetch(i):
        j = i % 2
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(done[j])
            bufs[j].copy_(host_imgs[i % n_in], non_blocking=True)
            ready[j].record(copy_stream)

    def e2e_loop(n):
        prefetch(0)
        prev = None
        with torch.no_grad():
            for i in range(n):
                j = i % 2
                if i + 1 < n:
                    prefetch(i + 1)
                torch.cuda.current_stream().wait_event(ready[j])
                cur = model.forward_async(bufs[j], targets).stage()       # H2D done -> forward -> async D2H of the detections
                done[j].record()
                if prev is not None:                                       # read step i-1 on the host while step i runs
                    prev.result()
                prev = cur
            prev.result()

    for j in range(2):
        done[j].record()
    e2e_loop(3)                  # untimed: first use of the copy stream, the pinned result staging, the staging buffers
    torch.cuda.synchronize()
    barrier()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    e2e_loop(steps)
    t1.record()
    torch.cuda.synchronize()
    ms_e2e = t0.elapsed_time(t1)
    barrier()
    return ms, ms_e2e, B * 50 * 14 * 4 + 4 * B, last


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--batch", type=int, default=8)
    ap.add_argument("--impl", default="ours", choices=("ours", "reference", "torch_gpu"))
    ap.add_argument("--precision", default="strict", choices=("strict", "fast"),
                    help="HEADLINE precision. strict (default): hi/lo fp16 pair arithmetic, meets the 1e-3 parity contract; "
                         "fast: one fp16 pass. Both are measured and reported under `modes`")
    ap.add_argument("--train", action="store_true", help="BASELINE configs[2] / configs[4]: full train step instead of inference")
    ap.add_argument("--graph", type=int, default=1, help="--train: capture the whole step in a CUDA graph (1) or run it eagerly (0)")
    ap.add_argument("--sync-bn", type=int, default=1, help="--train, N > 1: SyncBatchNorm like the reference's yaml (1, default) or per-GPU statistics (0)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-launches", default=None, help="write the per-launch timing table (json) to this path")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="after the timed steps, write what the last one returned (rank 0) as DIR/<name>.npy: the detections "
                         "and per-image counts, or with --train the loss terms and logged scalars")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of the project's own path (--impl ours)")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    cores = cpu_threads()
    cfg_name = "configs[3]" if args.batch == 32 else "configs[1]"
    config = {"workload": "DLA-34+DCNv2+heads+decode inference, batch %d/GPU, 384x1280 synthetic, %dxB200 (BASELINE %s)"
              % (args.batch, args.gpus, cfg_name), "batch_per_gpu": args.batch, "height": H, "width": W,
              "parallelism": "replicas x%d (images shard across GPUs, no data-path collective)" % args.gpus,
              "l2": "4 rotating input batches (189 MB at B=8) + >= 1.8 GB activation working set >> 126 MB L2"}
    if args.train:
        config["workload"] = ("full train step (fwd+bwd+AdamW), batch %d/GPU, 384x1280 synthetic KITTI labels, %dxB200 (BASELINE %s)"
                              % (args.batch, args.gpus, "configs[2]" if args.gpus == 1 else "configs[4]: DDP, NCCL grad all-reduce"))
        config["parallelism"] = "dp%d (batch dim sharded, gradient all-reduce)" % args.gpus
        config["l2"] = "3 rotating batches; ~10 GB activation + gradient working set >> 126 MB L2"

    if args.impl == "reference":
        if rank == 0:
            reference_arm(args, config, cores)
        return
    if args.impl == "torch_gpu":
        if rank == 0:
            torch_gpu_arm(args, config)
        return
    if args.train:
        return bench_train(args, rank, world, local_rank, config)

    import torch
    import torch.distributed as dist
    from monoflex_b200 import parallel
    from monoflex_b200 import synthetic as syn
    from monoflex_b200.config import default_cfg
    from monoflex_b200.model.detector import KeypointDetector
    assert torch.cuda.is_available(), "bench.py needs a GPU (no CPU fallback)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    parallel.init("nccl", dev)
    B = args.batch
    model = KeypointDetector(default_cfg(width=W, height=H))
    model.load_state_dict(syn.make_state_dict(0))
    model = model.to(dev).eval()
    tg = syn.make_targets(B, W // 4, H // 4)
    targets = [t.to(dev) for t in syn.make_param_lists(tg)]
    n_in = 4
    host_imgs = [syn.make_images(B, H, W, seed=100 + rank * n_in + i).pin_memory() for i in range(n_in)]
    dev_imgs = [h.to(dev) for h in host_imgs]

    def barrier():
        parallel.barrier()
        torch.cuda.synchronize()

    other = "fast" if args.precision == "strict" else "strict"
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    model.set_precision(args.precision)
    with torch.no_grad():
        for i in range(max(3, args.warmup)):
            model(dev_imgs[i % n_in], targets)
    ms, ms_e2e, d2h, last = time_inference(model, targets, host_imgs, dev_imgs, args.steps, B, dev, barrier,
                                           keep_last=bool(args.dump_outputs) and rank == 0)
    if last is not None:
        rows, counts = last
        dump_outputs(args.dump_outputs, {"detections": rows.numpy(), "detections_per_image": counts})
    launches_per_step = model.backbone.last_plan.n_launch + model.heads.predictor.last_plan.n_launch + 1 + 2
    if rank == 0:
        sampler.stop_flag = True
    ms, ms_e2e = parallel.max_over_ranks([ms, ms_e2e], device=dev)
    value = world * B * args.steps / (ms * 1e-3)
    e2e = world * B * args.steps / (ms_e2e * 1e-3)
    modes = {args.precision: {"value": value, "e2e": e2e, "ms_per_step": ms / args.steps}}

    roofline = decode = cpu = blocks = None
    if rank == 0:
        hbm, tf_sus, tf_burst, which = peaks()
        # ------------------------------------------------------------ per-launch timing of the headline precision
        with torch.no_grad():
            model.backbone(dev_imgs[0])
            for rep in range(3):
                rows_b = model.backbone.last_plan.run_timed()
                rows_h = model.heads.predictor.last_plan.run_timed()
        table, groups, total = group_table(rows_b, rows_h, tf_sus)
        facts = ncu_facts(args.precision)
        for g, e in groups.items():
            e["kernel"] = KERNEL_OF_GROUP.get(g, g)
            if g in facts:
                e["ncu"] = facts[g]
        top = max((g for g in groups if groups[g]["gflop"] > 0), key=lambda g: groups[g]["ms"])
        conv_gf = sum(e["gflop"] for e in groups.values())
        tg_ = groups[top]
        step_tf = B * FWD_GF_PER_IMG / (ms / args.steps)                # GFLOP / ms == TFLOP/s, one GPU's step
        roofline = {"bound": "tensor", "kernel": "%s: %s" % (top, tg_["kernel"]),
                    "selection": "the kernel group with the largest share of the step's device time (per-launch CUDA events)",
                    "achieved": tg_["tflops"], "peak": tf_sus, "unit": "TFLOP/s", "frac": tg_["frac_of_peak"],
                    "traffic": (facts.get(top) or {}).get("dram_bytes_per_launch"),
                    "tensor_pipe_pct_ncu": (facts.get(top) or {}).get("tensor_pipe_pct"),
                    "peak_source": "%s bf16 sustained (kernel timed inside the step; fp16 operands run at the bf16 rate)" % which,
                    "flops_convention": "algorithmic 2 x MACs of the reference's layers%s" % (
                        "; strict precision issues 3 tensor-core products per MAC, so the tensor pipe is ~3x busier than "
                        "`frac` says" if args.precision == "strict" else ""),
                    "share_of_step": tg_["share_of_step"], "launch_time_sum_ms": total,
                    "conv_stack_tflops": conv_gf / total, "conv_stack_frac": conv_gf / total / tf_sus,
                    "whole_step_tflops": step_tf, "whole_step_frac": step_tf / tf_sus}
        blocks = groups
        if args.dump_launches:
            os.makedirs(os.path.dirname(os.path.abspath(args.dump_launches)), exist_ok=True)
            json.dump({"precision": args.precision, "total_ms": total, "groups": groups, "launches": table},
                      open(args.dump_launches, "w"), indent=1)
        # ------------------------------------------------------------ decode kernels (BASELINE metric: "decode HBM GB/s")
        post = model.heads.post_processor
        hp = model.heads.predictor.last_plan
        meta = post.prepare_targets(targets, True, dev)
        flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
        post.launch(hp.cls, hp.reg, meta)
        torch.cuda.synchronize()
        dgraph = torch.cuda.CUDAGraph()                    # the two kernels as they run in the product (inside a CUDA graph):
        with torch.cuda.graph(dgraph):                     # eager ctypes launches would add ~10 us of host gap between them
            post.launch(hp.cls, hp.reg, meta)
        dts = []
        for rep in range(7):
            flush.zero_()                                  # evict cls/reg from L2: the decode is their first reader
            d0, d1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            d0.record()
            dgraph.replay()
            d1.record()
            torch.cuda.synchronize()
            dts.append(d0.elapsed_time(d1))
        dec_ms = sorted(dts)[len(dts) // 2]
        dec_bytes = B * (3 * 96 * 320 * 4 + 50 * 50 * 4 + 50 * 14 * 4 + 1400)       # SURVEY 8d: 382.8 KB / image
        decode = {"bound": "hbm", "kernel": "nms_topk_stage1 + topk_decode_stage2", "achieved": dec_bytes / dec_ms / 1e6,
                  "peak": hbm, "unit": "GB/s", "frac": dec_bytes / dec_ms / 1e6 / hbm, "ms": dec_ms,
                  "algorithmic_bytes": dec_bytes,
                  "note": "latency-bound by construction (SURVEY H7): %.1f us of pure DRAM time at peak" % (dec_bytes / hbm / 1e3)}
    # ---------------------------------------------------------------- the other precision (fewer steps: context number)
    model.set_precision(other)
    steps2 = max(5, args.steps // 2)
    ms2, ms2_e2e, _, _ = time_inference(model, targets, host_imgs, dev_imgs, steps2, B, dev, barrier)
    ms2, ms2_e2e = parallel.max_over_ranks([ms2, ms2_e2e], device=dev)
    modes[other] = {"value": world * B * steps2 / (ms2 * 1e-3), "e2e": world * B * steps2 / (ms2_e2e * 1e-3),
                    "ms_per_step": ms2 / steps2, "steps": steps2}
    model.set_precision(args.precision)

    if rank == 0:
        if world == 1 and not args.no_cpu_baseline:
            sec, n = cpu_eval_steps(6, 1, cores, 30.0)          # ~15-20 s of CPU work: a bounded sample, not the target
            cpu = {"value": 1.0 / sec, "unit": "images/s", "cores": cores, "kind": "port",
                   "sample": "%d full-resolution batch-1 eval forward(s) of the CPU oracle (%.1f s of CPU work each)" % (n, sec)}
        modes["strict"]["parity"] = "<= 1e-3 of the fp32 reference end to end (tests/test_gpu_model.py: 1.7e-4 .. 4.5e-4 measured)"
        modes["fast"]["parity"] = "2-7e-3 end to end (fp16 operand / activation rounding of ~50 stacked layers)"
        line = {"metric": METRIC if B == 8 else METRIC.replace("batch 8", "batch %d" % B), "value": value, "unit": "images/s",
                "n_gpus": world, "steps": args.steps,
                "warmup": max(3, args.warmup), "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "precision": args.precision,
                "dtype": ("f16 hi/lo pair operands (3 products per K step), f32 accumulate (tcgen05 kind::f16): fp32-grade"
                          if args.precision == "strict" else "f16 operands, f32 accumulate (tcgen05 kind::f16)"),
                "data": "synthetic", "config": config, "clocks": sampler.summary(),
                "e2e": {"value": e2e, "unit": "images/s", "h2d_bytes_per_step": B * 3 * H * W * 4,
                        "d2h_bytes_per_step": d2h, "ms_per_step": ms_e2e / args.steps},
                "modes": modes, "gpu_launches": launches_per_step * args.steps, "roofline": roofline, "blocks": blocks,
                "decode_roofline": decode, "cpu_baseline": cpu}
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
