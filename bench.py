#!/usr/bin/env python
"""Benchmark of the depth-guided texture-diffusion hot path (BASELINE.json metric: RGB-D images/s
at 384^2).

    python bench.py [--gpus N --steps K --warmup W]            # our arm (N>1: under torchrun)
    python bench.py --impl reference [...]                      # CPU arm: the unmodified reference module (oracle/_ref)
    python bench.py [...] --dump-outputs DIR                    # also write the last timed step's outputs as DIR/*.npy

One "step" = one pass of the hot path (prompt_encoder + 16 ShapePropDecoders + injection layout,
cod.py:1467-1505 minus the PVT blocks) over one batch of synthetic RGB-D input.  Workload =
BASELINE.json configs[1]: COD inference, batch 64 per GPU, 384x384, bf16.  The path shards by
image, so N GPUs run N independent replicas on different images (weak scaling, no collective).
Rank 0 prints ONE JSON line.
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
for p in (ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

import torch  # noqa: E402

METRIC = "rgbd_images_per_sec_384"
UNIT = "images/s"
# algorithmic FLOPs (2*MAC) of the tensor-core GEMMs per 384^2 image: 36 ConvNeXt blocks x 2
# pointwise GEMMs + 3 down-sample convs, as executed (DESIGN.md "Work per unit")
GEMM_FLOP_PER_IMAGE = 36 * 2 * 2 * 9216 * 128 * 512 + 2 * (2304 * 512 * 256 + 576 * 1024 * 512 + 144 * 2048 * 1024)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=64, help="images per GPU per step")
    ap.add_argument("--size", type=int, default=384)
    ap.add_argument("--precision", default="bf16", choices=["bf16", "fp32"])
    ap.add_argument("--train-eager", action="store_true", help="training leg without CUDA graph capture (DDP when N > 1)")
    ap.add_argument("--cpu-sample", type=int, default=8, help="images per CPU-baseline step")
    ap.add_argument("--no-eager-reference", action="store_true", help="skip the reference-eager-on-GPU baseline leg")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-diffusion", action="store_true")
    ap.add_argument("--no-train", action="store_true")
    ap.add_argument("--no-highres", action="store_true")
    ap.add_argument("--no-backbone", action="store_true")
    ap.add_argument("--train-batch", type=int, default=16, help="images per GPU per training step (configs[2])")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step returned (rank 0) as DIR/<name>.npy, float32; tensors above "
                         "the per-tensor share of 48 MiB are reduced to a fixed, seeded sample of their elements")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


# ------------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.stop, self.th = index, [], threading.Event(), None

    def _run(self):
        # NVML in-process (a sample every ~5 ms, so that a 10-step timed region of ~140 ms yields a real median);
        # the nvidia-smi subprocess (~100 ms per query) is the fallback when the binding is unavailable
        try:
            import pynvml
            pynvml.nvmlInit()
            h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            mx = pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM)
            get_reasons = getattr(pynvml, "nvmlDeviceGetCurrentClocksEventReasons", None) or \
                pynvml.nvmlDeviceGetCurrentClocksThrottleReasons
            bits = [0x8, 0x40, 0x20, 0x4]   # HwSlowdown, HwThermalSlowdown, SwThermalSlowdown, SwPowerCap
            while not self.stop.is_set():
                sm = pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)
                r = int(get_reasons(h))
                self.rows.append([str(sm), str(mx)] + ["Active" if r & b else "Not Active" for b in bits])
                self.stop.wait(0.005)
            return
        except Exception:
            pass
        while not self.stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                      "-i", str(self.index)], capture_output=True, text=True, timeout=5).stdout
                self.rows.append([c.strip() for c in out.strip().split(",")])
            except Exception:
                pass
            self.stop.wait(0.1)

    def __enter__(self):
        self.th = threading.Thread(target=self._run, daemon=True)
        self.th.start()
        return self

    def __exit__(self, *a):
        self.stop.set()
        self.th.join(timeout=6)

    def summary(self):
        sm = sorted(int(r[0]) for r in self.rows if len(r) >= 6 and r[0].isdigit())
        mx = [int(r[1]) for r in self.rows if len(r) >= 6 and r[1].isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) >= 6 and r[2 + i].lower().startswith("active")
                                                          for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


def diffusion_microbench(OP, dev, peaks, C=256, S=1024, steps=(1, 2, 4, 8, 16)):
    """MessagePassing core (cod.py:1190-1205), shared weights, NHWC, 1024^2 x 256 (BASELINE configs[3]), T sweep, both
    storage dtypes.  One launch per step (DESIGN.md section 9: at C = 256 the per-step tensor / FMA time is at or
    above the per-step HBM time, so fusing steps only adds halo recomputation).  Reported per T: time, the GB/s the
    kernel achieves per step, and the fraction of the T-fused roofline of SURVEY.md 8(d) (algorithmic bytes
    T-independent)."""
    g = torch.Generator("cpu").manual_seed(0)
    x = torch.randn(1, S, S, C, generator=g).to(dev)
    wgt = torch.rand(1, 49, S, S, generator=g).to(dev)
    hbm = float(peaks.get("hbm_gbs", 6650.0))
    fma_roof = 148 * 128 * 2 * 1.965e9

    def timed(xx, T, reps=3):
        for _ in range(2):
            OP.message_passing_tiled(xx, wgt, T)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        a.record()
        for _ in range(reps):
            OP.message_passing_tiled(xx, wgt, T)
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / reps

    step_bytes = (2 * C + 49) * S * S * 4
    out = {"shape": [1, C, S, S], "k": 7, "layout": "NHWC", "weights": "shared (wc=1)", "hbm_peak_gbs": hbm,
           "alg_bytes_per_step_f32": step_bytes, "sweep": []}
    for T in steps:
        ms = timed(x, T)
        flops = 2.0 * 49 * C * S * S * T
        bound_ms = max(step_bytes / (hbm * 1e9), flops / fma_roof) * 1e3     # fused-T roofline (SURVEY 8d)
        out["sweep"].append({"T": T, "ms": ms, "gbs_per_step": step_bytes * T / (ms * 1e-3) / 1e9,
                             "tflops": flops / (ms * 1e-3) / 1e12, "frac_of_fused_roofline": bound_ms / ms})
    out["hbm_frac_T1"] = out["sweep"][0]["gbs_per_step"] / hbm
    out["kernel_f32"] = ("mp_tc_f32_kernel: banded GEMM on tcgen05 as three bf16 products (A_hi X_hi + A_hi X_lo + A_lo X_hi, "
                         "16-bit split operands, fp32 accumulate), <= 1e-5 of the float64 oracle")
    # the CUDA-core kernel of round 1 (fp32 weights broadcast from shared memory) for comparison, T = 1
    for _ in range(2):
        OP.message_passing_tiled(x, wgt, 1, impl="simt")
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    for _ in range(3):
        OP.message_passing_tiled(x, wgt, 1, impl="simt")
    b.record()
    torch.cuda.synchronize()
    out["simt_f32_T1_ms"] = a.elapsed_time(b) / 3
    # bf16 storage / fp32 accumulate (configs[3] second dtype): banded GEMM on tcgen05 (mp_tc.cu)
    xb = x.to(torch.bfloat16)
    del x
    bb = (2 * C * 2 + 49 * 4) * S * S
    exec_flops = 2.0 * 336 * C * S * S
    out["alg_bytes_per_step_bf16"] = bb
    out["bf16_storage"] = []
    for T in (1, 4, 16):
        ms = timed(xb, T)
        out["bf16_storage"].append({"T": T, "ms": ms, "gbs_per_step": bb * T / (ms * 1e-3) / 1e9,
                                    "hbm_frac_per_step": bb * T / (ms * 1e-3) / 1e9 / hbm,
                                    "executed_mma_tflops": exec_flops * T / (ms * 1e-3) / 1e12})
    b1 = out["bf16_storage"][0]
    out["bf16_storage_T1"] = {"ms": b1["ms"], "alg_bytes": bb, "gbs": b1["gbs_per_step"], "hbm_frac": b1["hbm_frac_per_step"]}
    out["kernel"] = ("bf16 storage: mp_tc_kernel = banded GEMM Y[128 px,C] = A[128,336].X[336,C] on tcgen05 (TMA halo boxes as "
                     "MN-major operand, weights operand rebuilt per tile); fp32 storage: mp_tc_f32_kernel (same GEMM as three "
                     "bf16 products of split operands)")
    del wgt
    out["w2_fused_regressor"] = diffusion_microbench_w2(OP, dev, xb, hbm, fma_roof, C, S)
    out["cpu_port"] = diffusion_microbench_cpu()
    return out


def diffusion_microbench_cpu(C=256, S=256, T=1):
    """The same operator through the oracle port on the host cores at a REDUCED size (the reference's
    unfold formulation needs 49x the state; 1024^2 would be 49 GiB): element-iterations per second so that it
    can be set beside the GPU sweep (1024^2 x 256 x T elements per call there)."""
    from oracle import texture_diffuser_ref as O
    g = torch.Generator("cpu").manual_seed(0)
    x = torch.randn(1, C, S, S, generator=g)
    wgt = torch.rand(1, 49, S, S, generator=g)
    torch.set_num_threads(os.cpu_count() or 1)
    with torch.no_grad():
        O.message_passing_core(x, wgt, 7, T)
        t0 = time.perf_counter()
        O.message_passing_core(x, wgt, 7, T)
        dt = time.perf_counter() - t0
    return {"shape": [1, C, S, S], "T": T, "seconds": dt, "elements_per_s": C * S * S * T / dt,
            "cores": os.cpu_count() or 1, "kind": "port (oracle.message_passing_core, fp32 torch CPU)"}


def backbone_bench(TD, dev, world, rank, args, common, sharding, steps=5):
    """SURVEY.md 8f-1 (next row): the whole `pvt_v2_b2.forward_features` (cod.py:1455-1509) -- the hot path plus
    the 16 PVT-v2 blocks that consume the prompts -- batch `--batch` per GPU, images/s of the job."""
    from dgtd_b200.twig.model import pvt
    net = pvt.pvt_v2_b2().eval()
    common.fill_params_(net, seed=0)
    net = net.to(dev)
    TD.set_precision(net, args.precision)
    B, S = args.batch, args.size
    image, depth = common.synthetic_inputs(B, S, seed=300 + rank)
    image, depth = image.to(dev), depth.to(dev)
    for _ in range(2):
        net.forward_features(image, depth)
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(steps):
        net.forward_features(image, depth)
    b.record()
    torch.cuda.synchronize()
    t = sharding.max_over_ranks(a.elapsed_time(b) / 1e3, dev)
    del net
    torch.cuda.empty_cache()
    return {"value": world * B * steps / t, "unit": "images/s", "batch_per_gpu": B, "size": S, "ms_per_step": t / steps * 1e3,
            "precision": args.precision,
            "what": "pvt_v2_b2.forward_features = texture-diffusion hot path + 4 patch embeds + 16 PVT-v2 blocks "
                    "(spatial-reduction attention on mma.sync, Mix-FFN on tcgen05 GEMMs)"}


def full_model_bench(TD, dev, world, rank, args, common, sharding, steps=5):
    """SURVEY.md 8f-2 / 8f-4 (next rows): the whole `cod` model in predict mode (cod.py:147-217 without the PNG side
    effects) -- backbone with the texture prompts, Hitnet iterative decoder (exact fp32 kernels), sigmoid -- and
    the MAE / S-measure evaluation of the batch (twig/metric), batch `--batch` per GPU, images/s of the job."""
    from dgtd_b200.twig.metric import sod_metrics
    from dgtd_b200.twig.model import hitnet
    from dgtd_b200.twig.ops import capi
    net = hitnet.cod(win_size=22, filter_ratio=0.9, using_sam=True, using_depth=True, finetune=True,
                     binary_thresh=0.2, pretrain_sam=None, head=None).eval()
    common.hitnet_fixture_params_(net.hitnet, seed=0)
    net = net.to(dev)
    TD.set_precision(net, args.precision)
    B, S = args.batch, args.size
    image, depth = common.synthetic_inputs(B, S, seed=400 + rank)
    image, depth = image.to(dev), depth.to(dev)
    label = (torch.rand(B, 1, S, S, generator=torch.Generator("cpu").manual_seed(5)) > 0.5).float().to(dev)

    def timed(fn, n):
        for _ in range(2):
            fn()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0 = capi.launch_count()
        a.record()
        for _ in range(n):
            fn()
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / n, (capi.launch_count() - l0) // n
    ms, launches = timed(lambda: net(None, image, label, depth, mode="predict"), steps)
    t = sharding.max_over_ranks(ms / 1e3, dev)
    _, feats = net.hitnet.backbone._forward_features_nhwc(image, depth)
    dec_ms, dec_launches = timed(lambda: net.hitnet.decode(feats, want_stage_preds=False), steps)
    prob, _ = net(None, image, label, depth, mode="predict")
    met_ms, _ = timed(lambda: sod_metrics(prob, label), 10)
    met4_ms, _ = timed(lambda: sod_metrics(prob, label, curves=True), 10)
    vals = sod_metrics(prob, label).mean(0).tolist()
    # BASELINE configs[4] for the whole model: 8 images of 768^2 sharded by image, no collective
    hi = None
    try:
        hb = max(1, 8 // world)
        hi_img, hi_dep = common.synthetic_inputs(hb, 768, seed=500 + rank)
        hi_img, hi_dep = hi_img.to(dev), hi_dep.to(dev)
        hms, _ = timed(lambda: net.hitnet.predict_logits(hi_img, hi_dep, (768, 768)), 3)
        ht = sharding.max_over_ranks(hms / 1e3, dev)
        hi = {"value": world * hb / ht, "unit": "images/s", "size": 768, "batch_per_gpu": hb, "ms_per_step": ht * 1e3}
        del hi_img, hi_dep
    except Exception as e:  # noqa: BLE001
        hi = {"error": f"{type(e).__name__}: {e}"[:300]}
    # end to end through the host-facing pipeline: pinned image + depth + label in, per-image (MAE, S-measure) out
    e2e = None
    try:
        from dgtd_b200.twig.pipeline import HostPipeline
        nb = steps + 2
        host = [tuple(t.cpu().pin_memory() for t in (image, depth, label)) for _ in range(2)]
        outs = [torch.empty(B, 2 + 2 * 256, dtype=torch.float64).pin_memory() for _ in range(2)]

        def fwd(im, dp, lb):      # all four evaluators of cod.yml:123-128: (MAE, S) + the F / E curves per image
            prob_, _ = net(None, im, lb, dp, mode="predict")
            vals_, cur_ = sod_metrics(prob_, lb, curves=True)
            return (torch.cat([vals_, cur_.reshape(B, -1)], dim=1),)
        pipe = HostPipeline(None, None, device=dev, forward=fwd)
        for _ in pipe.run((host[i & 1] for i in range(2)), lambda m: m, outs):
            pass
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        last = None
        for _, _, done in pipe.run((host[i & 1] for i in range(nb)), lambda m: m, outs):
            last = done
        last.synchronize()
        dt = sharding.max_over_ranks(time.perf_counter() - t0, dev)
        e2e = {"value": world * B * nb / dt, "unit": "images/s",
               "h2d_bytes_per_step": int(sum(t.numel() * t.element_size() for t in host[0])),
               "d2h_bytes_per_step": int(outs[0].numel() * 8),
               "what": "pinned host image + depth + label -> predict -> MAE / S-measure / F- and E-measure curves -> 4 KB per image back"}
    except Exception as e:  # noqa: BLE001
        e2e = {"error": f"{type(e).__name__}: {e}"[:300]}
    # small-batch serving latency: eager (Python-issued launches) against the captured predict step
    latency = None
    if rank == 0:
        try:
            from dgtd_b200.twig import graphs
            li, ld = image[:1].contiguous(), depth[:1].contiguous()
            eager_ms, _ = timed(lambda: net.hitnet.predict_logits(li, ld, (S, S)), 10)
            run = graphs.GraphedPredict(net, li, ld)
            graph_ms, _ = timed(lambda: run(), 20)
            latency = {"batch": 1, "eager_ms": eager_ms, "graph_replay_ms": graph_ms,
                       "note": "cod.forward(mode='tensor') at batch 1: the eager path is bound by issuing ~630 launches"}
            del run
        except Exception as e:  # noqa: BLE001
            latency = {"error": f"{type(e).__name__}: {e}"[:300]}
    cpu_port = None
    if rank == 0 and not args.no_cpu_baseline:
        # the reference's CPU path for the same model: oracle port (pinned to the unmodified Hitnet), fp32, all host
        # threads, a bounded sample of 2 images of the same size
        from oracle import hitnet_ref as HR
        cores = os.cpu_count() or 1
        torch.set_num_threads(cores)
        p32 = {k: v.detach().float().cpu() for k, v in net.hitnet.state_dict().items() if v.dtype.is_floating_point}
        ci, cd = common.synthetic_inputs(2, S, seed=400)
        with torch.no_grad():
            HR.hitnet_forward(ci[:1], cd[:1], p32)
            t0 = time.perf_counter()
            _, cp1, cp2 = HR.hitnet_forward(ci, cd, p32)
            HR.predict_logits(cp1, cp2, (S, S))
            dt = time.perf_counter() - t0
        cpu_port = {"value": 2 / dt, "unit": "images/s", "cores": cores, "kind": "port",
                    "sample": f"2 images {S}x{S}, fp32 torch CPU, {cpu_model()}"}
    del net
    torch.cuda.empty_cache()
    # decoder FLOPs per image on the stride-8 grid g = S/8 (cod.py:752-805): 2 CABs x 2 conv3 at 64 ch on (2g)^2,
    # per iteration 2x2 conv3 at 32 ch on (g/4)^2, 64 ch on (g/2)^2, 96 ch on g^2, conv4 96->32, compress 8x8
    g = S // 8
    per_iter = 4 * 2 * 9 * (32 * 32 * (g // 4) ** 2 + 64 * 64 * (g // 2) ** 2 + 96 * 96 * g * g) + 2 * 9 * 96 * 32 * g * g
    flops = 4 * 2 * 9 * 64 * 64 * (2 * g) ** 2 + 4 * per_iter + 3 * 2 * 64 * 64 * 32 * (g // 4) ** 2
    return {"value": world * B / t, "unit": "images/s", "batch_per_gpu": B, "size": S, "ms_per_step": t * 1e3,
            "precision": (f"{args.precision} (decoder: bf16 im2col + tcgen05 GEMM, fp32 accumulate / activations)"
                          if args.precision == "bf16" else "fp32 (exact CUDA-core implicit GEMMs)"),
            "launches_per_step": int(launches),
            "decoder_ms": dec_ms, "decoder_launches": int(dec_launches),
            "decoder_gflop_per_image": flops / 1e9, "decoder_tflops": flops * B / (dec_ms * 1e-3) / 1e12,
            "metrics_ms": met_ms, "metrics_all_four_ms": met4_ms, "metrics_gbs": B * S * S * (8 + 2 + 2) / (met_ms * 1e-3) / 1e9,
            "metrics_note": "MAE + S-measure of the batch: 8 B/pixel read + 2 B/pixel written in pass 1, 2 B/pixel read in pass 2",
            "mae_smeasure_vs_random_label": vals, "cpu_baseline": cpu_port, "latency_batch1": latency, "e2e": e2e, "highres_768": hi,
            "what": "cod.forward(mode='predict'): pvt_v2_b2 backbone with the texture prompts + Hitnet decoder "
                    "(4 feedback iterations) + sigmoid"}


def loss_bench(dev, peaks, common, B=16, S=384, steps=10):
    """SURVEY.md 8f-3 (next row): structure loss + deep supervision (cod.py:75-84, 135-141) forward + backward on
    five B x 1 x S x S logit maps.  Pure bandwidth: the weight map is computed once (8 B/pixel), each of the
    four weighted maps reads 12 B/pixel forward and moves 16 B/pixel backward."""
    from dgtd_b200.twig.model import losses as M
    preds, gts = common.loss_inputs(B, S, S, seed=1)
    g = torch.Generator("cpu").manual_seed(2)
    P1 = [(2.0 * torch.randn(B, 1, S, S, generator=g)).to(dev).requires_grad_(True) for _ in range(4)]
    P2 = preds.to(dev).requires_grad_(True)
    label = gts.to(dev)

    def one():
        loss = M.deep_supervision_loss(P1, P2, label)
        loss.backward()
        for t in P1 + [P2]:
            t.grad = None
    for _ in range(3):
        one()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(steps):
        one()
    b.record()
    torch.cuda.synchronize()
    ms = a.elapsed_time(b) / steps
    nbytes = B * S * S * (8 + 4 * (12 + 16))
    hbm = float(peaks.get("hbm_gbs", 6650.0))
    return {"ms": ms, "images_per_s": B / (ms * 1e-3), "alg_bytes": nbytes, "gbs": nbytes / (ms * 1e-3) / 1e9,
            "hbm_frac": nbytes / (ms * 1e-3) / 1e9 / hbm, "batch": B, "size": S,
            "note": "5 supervised maps, fwd + bwd, 12 launches; latency-bound at this size (labels and logits fit in L2)"}


def highres_bench(TD, enc, dec, dev, world, rank, args, common, sharding, S=768, total=8, steps=5):
    """BASELINE configs[4]: high-resolution inference, 8 images of 768^2 sharded by image over the GPUs
    (8 / N per GPU, no collective); images/s of the whole job, device time, max over ranks."""
    B = max(1, total // world)
    image, depth = common.synthetic_inputs(B, S, seed=200 + rank)
    image, depth = image.to(dev), depth.to(dev)
    for _ in range(2):
        TD.texture_prompts(enc, dec, image, depth, precision=args.precision, want_embedding3=False)
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(steps):
        TD.texture_prompts(enc, dec, image, depth, precision=args.precision, want_embedding3=False)
    b.record()
    torch.cuda.synchronize()
    t = sharding.max_over_ranks(a.elapsed_time(b) / 1e3, dev)
    return {"value": world * B * steps / t, "unit": "images/s", "size": S, "batch_per_gpu": B, "ms_per_step": t / steps * 1e3,
            "sharding": "by image, no collective"}


def diffusion_microbench_w2(OP, dev, xb, hbm, fma_roof, C, S):
    """Weight mode W2 (SURVEY.md 8d config 4): the model's per-channel weights sigmoid(Wr g + br) are
    generated on chip from the 3-channel guide (49 GiB if materialised).  Algorithmic bytes per iteration
    (2*C*s + 3*4)*H*W; algorithmic FLOPs 2*49*C*H*W (stencil) + C*49*14*H*W (regressor + sigmoid).  One
    pass per iteration, weights regenerated every pass; the bound is the MUFU/FMA issue rate, not HBM."""
    g = torch.Generator("cpu").manual_seed(1)
    guide = torch.randn(1, 3, S, S, generator=g).to(dev)
    reg_w = (torch.randn(C * 49, 3, generator=g) * 0.5).to(dev)
    reg_b = torch.randn(C * 49, generator=g).to(dev)
    mufu_roof = 148 * 16 * 1.965e9            # MUFU lane-ops/s (16 per SM per clock)
    res = {"weights": "per-channel, generated on chip (wc=C)", "sweep": []}
    x32 = xb.float()
    cases = [("f32", x32, False, 1), ("f32", x32, False, 4), ("f32", x32, True, 1), ("bf16", xb, True, 1)]
    for name, x, fast, T in cases:
        es = 4 if name == "f32" else 2
        for _ in range(2):
            OP.message_passing_regress(x, guide, reg_w, reg_b, T, fast_sigmoid=fast)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        a.record()
        for _ in range(2):
            OP.message_passing_regress(x, guide, reg_w, reg_b, T, fast_sigmoid=fast)
        b.record()
        torch.cuda.synchronize()
        ms = a.elapsed_time(b) / 2
        nbytes = (2 * C * es + 12) * S * S
        flops = (2.0 * 49 + 49 * 14) * C * S * S * T
        mufu = (1 if fast else 2) * 49.0 * C * S * S * T
        bound_ms = max(nbytes / (hbm * 1e9), flops / fma_roof, mufu / mufu_roof) * 1e3
        res["sweep"].append({"storage": name, "sigmoid": "tanh.approx" if fast else "ex2+rcp", "T": T, "ms": ms,
                             "alg_bytes_per_iter": nbytes, "gbs_per_iter": nbytes * T / (ms * 1e-3) / 1e9,
                             "tflops": flops / (ms * 1e-3) / 1e12, "mufu_ms": mufu / mufu_roof * 1e3,
                             "fma_ms": flops / fma_roof * 1e3, "hbm_ms": nbytes / (hbm * 1e9) * 1e3 * T,
                             "roofline_ms": bound_ms, "frac_of_roofline": bound_ms / ms})
    return res


def train_bench(TD, enc, dec, dev, world, rank, local, args, common, sharding, steps=5, warmup=2, precision="bf16",
                measure_reduce=True):
    """Forward + backward of the hot path (block-level autograd Functions; `precision` selects the exact
    fp32 CUDA-core path or the bf16 tcgen05 path) on `train-batch` images per GPU.  Default: the step is
    captured in a CUDA graph and replayed (twig/graphs.py); with N > 1 the flat gradient buffer is
    all-reduced over NCCL after every replay.  --train-eager: Python-issued launches, gradients reduced by
    DistributedDataParallel (bucketed all-reduce overlapped with backward -- the reference's mechanism,
    cod.py:8,238)."""
    import torch.distributed as dist
    import torch.nn as nn
    from dgtd_b200.twig import graphs

    B, S = args.train_batch, args.size
    image, depth = common.synthetic_inputs(B, S, seed=100 + rank)
    image, depth = image.to(dev), depth.to(dev)
    enc.train(); dec.train()
    n_grad = sum(p.numel() for p in list(enc.parameters()) + list(dec.parameters()) if p.requires_grad)

    # the optimizer of config/sod.yml:56-76 (AdamW lr 5e-4, wd 0.1, custom_keys lr multipliers) as one fused launch
    # over flat parameter / gradient / moment buffers; parameter values are saved and restored around the leg
    from dgtd_b200.twig.optim import SOD_CUSTOM_KEYS, FusedAdamW
    named = [("hitnet.backbone.prompt_encoder." + n, p) for n, p in enc.named_parameters() if p.requires_grad] + \
            [("hitnet.backbone.prompt_decoder." + n, p) for n, p in dec.named_parameters() if p.requires_grad]
    saved = [p.detach().clone() for _, p in named]
    opt = FusedAdamW(named, lr=5e-4, weight_decay=0.1, custom_keys=SOD_CUSTOM_KEYS)

    if args.train_eager:
        class HotPath(nn.Module):
            def __init__(self, enc, dec):
                super().__init__()
                self.prompt_encoder, self.prompt_decoder = enc, dec

            def forward(self, image, depth):
                return graphs.default_loss(*TD.texture_prompts_train(self.prompt_encoder, self.prompt_decoder, image,
                                                                     depth, precision=precision))

        model = HotPath(enc, dec).train()
        if world > 1:
            model = nn.parallel.DistributedDataParallel(model, device_ids=[local], find_unused_parameters=True)

        def one():
            opt.zero_grad()
            model(image, depth).backward()
            opt.step()
        launch = "eager (Python-issued launches)"
        reduce = "DistributedDataParallel bucketed NCCL all-reduce" if world > 1 else "none (1 GPU)"
    else:
        step = graphs.GraphedTrainStep(enc, dec, image, depth, precision=precision, flat_grad=opt.flat_grad)

        def one():
            step()
            opt.step()
        launch = "CUDA graph replay of fwd+bwd + one fused AdamW launch"
        reduce = (step.bucketer.describe() + " inside the captured step (overlaps backward)") if world > 1 else "none (1 GPU)"

    def timed_loop(fn, n):
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(n):
            fn()
        b.record()
        torch.cuda.synchronize()
        return sharding.max_over_ranks(a.elapsed_time(b) / 1e3, dev)

    for _ in range(warmup):
        one()
    t = timed_loop(one, steps)
    allreduce_ms = in_situ_ms = after_ms = None
    if world > 1 and not args.train_eager and measure_reduce:
        # exposed time of the gradient reduction, IN SITU: the same captured step with the reduction left out
        # (reduce="none": gradients stay local), timed the same way; and the round-1 scheme (one all-reduce of the whole
        # flat buffer after the replay) for comparison
        step.close()
        local = graphs.GraphedTrainStep(enc, dec, image, depth, precision=precision, flat_grad=opt.flat_grad, reduce="none")

        def one_local():
            local()
            opt.step()
        for _ in range(warmup):
            one_local()
        t_local = timed_loop(one_local, steps)
        in_situ_ms = (t - t_local) / steps * 1e3
        del local
        after = graphs.GraphedTrainStep(enc, dec, image, depth, precision=precision, flat_grad=opt.flat_grad, reduce="after")

        def one_after():
            after()
            opt.step()
        for _ in range(warmup):
            one_after()
        after_ms = (timed_loop(one_after, steps) - t_local) / steps * 1e3
        del after
        for _ in range(3):                                   # NCCL sets its channels up lazily per op / size
            dist.all_reduce(opt.flat_grad, op=dist.ReduceOp.AVG)
        allreduce_ms = timed_loop(lambda: dist.all_reduce(opt.flat_grad, op=dist.ReduceOp.AVG), steps) / steps * 1e3
    e, f = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e.record()
    for _ in range(5):
        opt.step()
    f.record()
    torch.cuda.synchronize()
    opt_ms = e.elapsed_time(f) / 5
    with torch.no_grad():
        for (_, p), v in zip(named, saved):
            p.copy_(v)
    for p in list(enc.parameters()) + list(dec.parameters()):
        p.grad = None
    enc.eval(); dec.eval()
    return {"value": world * B * steps / t, "unit": UNIT, "batch_per_gpu": B, "steps": steps, "ms_per_step": t / steps * 1e3,
            "precision": precision, "launch": launch,
            "optimizer": f"fused AdamW (config/sod.yml:56-76: lr 5e-4, wd 0.1, custom_keys lr multipliers), 1 launch, "
                         f"{n_grad} parameters, 28 B/parameter",
            "optimizer_ms": opt_ms, "optimizer_gbs": n_grad * 28 / (opt_ms * 1e-3) / 1e9,
            "grad_allreduce": f"{reduce}, {n_grad} fp32 grads" if world > 1 else reduce,
            "allreduce_in_situ_ms": in_situ_ms, "allreduce_after_replay_exposed_ms": after_ms,
            "allreduce_standalone_ms": allreduce_ms, "allreduce_exposed_ms": in_situ_ms}


def full_model_train_bench(dev, world, rank, args, common, sharding, steps=5, warmup=2, precision="bf16"):
    """BASELINE configs[2] on the WHOLE model: `cod.forward(mode='loss')` (cod.py:118-146: pvt_v2_b2 backbone with the
    texture prompts, Hitnet decoder with train-mode BatchNorm, deep supervision) + backward + the fused AdamW of
    config/sod.yml:56-76 over all 114 M parameters, `train-batch` images per GPU; the step is one CUDA-graph replay
    (twig/graphs.py::GraphedModelTrainStep), gradients reduced in buckets over NCCL inside it when N > 1."""
    import torch.distributed as dist
    from dgtd_b200.twig import graphs
    from dgtd_b200.twig.model import hitnet
    from dgtd_b200.twig.optim import SOD_CUSTOM_KEYS, FusedAdamW
    B, S = args.train_batch, args.size
    torch.manual_seed(0)
    net = hitnet.cod(win_size=22, filter_ratio=0.9, using_sam=True, using_depth=True, finetune=True, binary_thresh=0.2)
    common.hitnet_fixture_params_(net.hitnet, seed=0)
    net = net.to(dev).train()
    image, depth = common.synthetic_inputs(B, S, seed=200 + rank)
    _, label = common.loss_inputs(B, S, S, seed=300 + rank)
    image, depth, label = image.to(dev), depth.to(dev), label.to(dev)
    named = [(n, p) for n, p in net.named_parameters() if p.requires_grad]
    n_grad = sum(p.numel() for _, p in named)
    opt = FusedAdamW(named, lr=5e-4, weight_decay=0.1, custom_keys=SOD_CUSTOM_KEYS)
    n0 = capi_launches()
    step = graphs.GraphedModelTrainStep(net, image, depth, label, precision=precision, flat_grad=opt.flat_grad)
    launches_per_step = (capi_launches() - n0) // 4         # 3 warm-up passes + the capture

    def one():
        step()
        opt.step()

    def timed_loop(fn, n):
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(n):
            fn()
        b.record()
        torch.cuda.synchronize()
        return sharding.max_over_ranks(a.elapsed_time(b) / 1e3, dev)

    for _ in range(warmup):
        one()
    t = timed_loop(one, steps)
    loss = float(step.loss)
    grad_less = [n for n, p in named if p.grad is None or float(p.grad.abs().max()) == 0.0]
    exposed = None
    if world > 1:
        step.close()
        local = graphs.GraphedModelTrainStep(net, image, depth, label, precision=precision, flat_grad=opt.flat_grad,
                                             reduce="none")

        def one_local():
            local()
            opt.step()
        for _ in range(warmup):
            one_local()
        exposed = (t - timed_loop(one_local, steps)) / steps * 1e3
    return {"value": world * B * steps / t, "unit": UNIT, "batch_per_gpu": B, "steps": steps, "ms_per_step": t / steps * 1e3,
            "precision": precision, "parameters": n_grad, "launches_per_step": int(launches_per_step),
            "loss_after": loss, "loss_finite": bool(loss == loss and abs(loss) < 1e30), "grad_less_parameters": len(grad_less),
            "what": "cod.forward(mode='loss') + backward + fused AdamW, all parameters, train-mode BatchNorm (per-GPU "
                    "statistics), DropPath on; one CUDA-graph replay per step",
            "grad_allreduce": (step.bucketer.describe() if step.bucketer is not None else "none (1 GPU)"),
            "allreduce_exposed_ms": exposed}


DUMP_BYTES = 48 << 20


def dump_outputs(outdir: str, e1, toks) -> None:
    """Write embedding1 and the prompt tokens of one hot-path step as `<name>.npy` (names of
    `common.flatten_outputs`), float32, so that two builds can be compared output for output.  A tensor
    with more elements than its share of DUMP_BYTES keeps at most that many, at distinct flat indices drawn
    from a generator seeded by the tensor's name: the same arguments select the same elements in every run."""
    import zlib
    import numpy as np
    import common
    named = {k: v for k, v in common.flatten_outputs(e1, None, toks).items() if v is not None}
    cap = DUMP_BYTES // (4 * len(named))
    os.makedirs(outdir, exist_ok=True)
    for name, t in named.items():
        flat = t.detach().reshape(-1)
        if flat.numel() > cap:
            g = torch.Generator("cpu").manual_seed(zlib.crc32(name.encode()))
            idx = torch.randint(flat.numel(), (cap,), generator=g).unique()
            flat = flat[idx.to(flat.device)]
        np.save(os.path.join(outdir, name + ".npy"), flat.float().cpu().numpy())


def capi_launches() -> int:
    from dgtd_b200.twig.ops import capi
    return capi.launch_count()


def cpu_model() -> str:
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                return line.split(":", 1)[1].strip()
    except Exception:
        pass
    return "unknown"


def cpu_reference_rate(size: int, images: int, steps: int, warmup: int):
    """The reference's own CPU implementation of the hot path on the host cores, fp32, all threads: the
    UNMODIFIED module staged by oracle/make_ref.py (`kind: "reference"`; cod.py:1467-1505 minus the PVT
    blocks, eval mode, no_grad); the oracle port only when the staged file is missing (`kind: "port"`).
    Returns (images/s, seconds per step, cores, kind)."""
    import common
    from oracle import ref_loader as R
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    image, depth = common.synthetic_inputs(images, size)
    grids = common.pvt_token_grids((size, size))
    if R.reference_available():
        m = R.load_reference()
        pe, pd = R.build_reference_hot_path(m, seed=0, img_size=size)
        pe, pd = pe.eval(), pd.eval()
        kind = "reference"

        def one():
            with R.on_cpu():
                R.reference_hot_path(pe, pd, image, depth, grids)
    else:
        from oracle import texture_diffuser_ref as O
        TD = common.package()
        enc, dec = TD.build_texture_diffuser(seed=0)
        pe = {k: v.detach().float() for k, v in enc.state_dict().items()}
        pd = {k: v.detach().float() for k, v in dec.state_dict().items()}
        kind = "port"

        def one():
            O.texture_prompts(image, depth, pe, pd)
    times = []
    with torch.no_grad():
        for i in range(warmup + steps):
            t0 = time.perf_counter()
            one()
            if i >= warmup:
                times.append(time.perf_counter() - t0)
    dt = sum(times) / len(times)
    return images / dt, dt, cores, kind


def _gpu_time(fn, steps, warmup=2):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(steps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / steps


def gpu_eager_reference(dev, args, common, ours):
    """The bar of SURVEY.md 8(d) config 2 (iii) / BASELINE.md 4: the UNMODIFIED reference module (staged copy,
    oracle/make_ref.py) in eager PyTorch on the SAME B200 -- fp32 and `torch.autocast(bfloat16)` -- on the same
    batch: hot path (cod.py:1467-1505 minus the PVT blocks), the whole model in predict semantics (cod.py:179-180
    without the PNG side effects), and eager `MessagePassing` (cod.py:1201-1205) at configs[3] size run
    channel-chunked (its `unfold` is 49x the state: 49 GiB un-chunked).  `ours` = this library's numbers for the
    same legs, so that every ratio is stated against stock PyTorch on the same GPU, not against a CPU."""
    import torch.nn.functional as F
    from oracle import ref_loader as R
    if not R.reference_available():
        return {"unavailable": "oracle/_ref/twig/model/cod.py not staged (run oracle/make_ref.py where /root/reference exists)"}
    m = R.load_reference()
    B, S = args.batch, args.size
    out = {"what": "unmodified reference module, eager PyTorch %s on the same GPU, batch %d, %dx%d" % (torch.__version__, B, S, S),
           "tf32": bool(torch.backends.cuda.matmul.allow_tf32), "cudnn_tf32": bool(torch.backends.cudnn.allow_tf32)}
    image, depth = common.synthetic_inputs(B, S, seed=0)
    image, depth = image.to(dev), depth.to(dev)
    grids = common.pvt_token_grids((S, S))
    pe, pd = R.build_reference_hot_path(m, seed=0, img_size=S)
    pe, pd = pe.to(dev).eval(), pd.to(dev).eval()
    with torch.no_grad():
        ms32 = _gpu_time(lambda: R.reference_hot_path(pe, pd, image, depth, grids), 3, 1)
        with torch.autocast("cuda", dtype=torch.bfloat16):
            ms16 = _gpu_time(lambda: R.reference_hot_path(pe, pd, image, depth, grids), 5, 2)
    out["hot_path"] = {"fp32_ms": ms32, "fp32_images_per_s": B / ms32 * 1e3, "bf16_autocast_ms": ms16,
                       "bf16_autocast_images_per_s": B / ms16 * 1e3, "ours_bf16_ms": ours.get("hot_ms"),
                       "speedup_vs_bf16_autocast": (ms16 / ours["hot_ms"]) if ours.get("hot_ms") else None}
    del pe, pd
    torch.cuda.empty_cache()
    try:
        net = m.cod(win_size=22, filter_ratio=0.9, using_sam=True, using_depth=True, finetune=True,
                    binary_thresh=0.2, pretrain_sam=None, head=None).to(dev).eval()

        def predict():
            _, P1, P2 = net.hitnet(image, depth)
            return F.interpolate(P1[-1] + P2, size=(S, S), mode="bilinear", align_corners=False).sigmoid()
        with torch.no_grad():
            f32 = _gpu_time(predict, 2, 1)
            with torch.autocast("cuda", dtype=torch.bfloat16):
                f16 = _gpu_time(predict, 3, 1)
        out["full_model_predict"] = {"fp32_ms": f32, "fp32_images_per_s": B / f32 * 1e3, "bf16_autocast_ms": f16,
                                     "bf16_autocast_images_per_s": B / f16 * 1e3, "ours_bf16_ms": ours.get("full_ms"),
                                     "speedup_vs_bf16_autocast": (f16 / ours["full_ms"]) if ours.get("full_ms") else None}
        del net
    except Exception as e:  # noqa: BLE001
        out["full_model_predict"] = {"error": f"{type(e).__name__}: {e}"[:300]}
    torch.cuda.empty_cache()
    # eager MessagePassing core at configs[3] size, shared weights, T = 1, 16 channels per chunk (3.3 GB unfold)
    try:
        C, HW, CH = 256, 1024, 16
        g = torch.Generator("cpu").manual_seed(0)
        x = torch.randn(1, C, HW, HW, generator=g).to(dev)
        wgt = torch.rand(1, 49, HW, HW, generator=g).to(dev)

        def mp_step():
            w_ = wgt.view(1, 1, 49, HW * HW)
            nw = w_ / (torch.sum(w_, dim=2).unsqueeze(2) + 1e-5)                    # cod.py:1201
            ys = []
            for c0 in range(0, C, CH):
                u = F.unfold(x[:, c0:c0 + CH], kernel_size=7, padding=3).view(1, CH, 49, HW * HW)   # cod.py:1204
                ys.append((u * nw).sum(2).view(1, CH, HW, HW))                      # cod.py:1205
            return torch.cat(ys, 1)
        with torch.no_grad():
            mp_ms = _gpu_time(mp_step, 2, 1)
        out["message_passing_1024x256_T1"] = {"ms": mp_ms, "chunk_channels": CH, "ours_fp32_ms": ours.get("mp_ms"),
                                              "speedup": (mp_ms / ours["mp_ms"]) if ours.get("mp_ms") else None}
        del x, wgt
    except Exception as e:  # noqa: BLE001
        out["message_passing_1024x256_T1"] = {"error": f"{type(e).__name__}: {e}"[:300]}
    torch.cuda.empty_cache()
    return out


# ------------------------------------------------------------------------------------------------
def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    steps, warmup = max(1, args.steps), max(0, args.warmup)
    n = args.cpu_sample if args.cpu_sample > 0 else 8
    rate, dt, cores, kind = cpu_reference_rate(args.size, n, steps, warmup)
    sample = (f"{n} images of the batch-{args.batch} workload per step ({steps} timed + {warmup} warm-up steps), fp32, "
              f"eval/no_grad, torch {torch.__version__} CPU, {cores} threads, {cpu_model()}")
    what = ("the UNMODIFIED reference module (oracle/_ref copy of twig/model/cod.py: prompt_encoder + 4 prompt_decoders + "
            "injection, cod.py:1467-1505 minus the PVT blocks)" if kind == "reference" else "oracle port of the reference modules")
    line = {
        "impl": "reference", "metric": METRIC, "value": rate, "unit": UNIT, "n_gpus": args.gpus,
        "steps": steps, "warmup": warmup, "ms_per_step": dt * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"COD inference hot path, batch {args.batch}/GPU, {args.size}x{args.size} RGB-D "
                               f"(BASELINE configs[1]); CPU arm = {what}"},
        "cpu_baseline": {"value": rate, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": rate, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def run_ours(args):
    import torch.distributed as dist
    import common
    TD = common.package()
    from dgtd_b200.twig.ops import capi
    from dgtd_b200.twig.ops.functions import texture_diffusion_func as OP

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a GPU (no CPU fallback on the product path)"
    torch.cuda.set_device(local)
    if world > 1:
        os.environ.setdefault("NCCL_DEBUG", "WARN")   # keep NCCL's version banner off stdout (one JSON line)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)
    B, S = args.batch, args.size

    enc, dec = TD.build_texture_diffuser(seed=0)
    common.perturb_regressor_(enc)
    enc, dec = enc.to(dev).eval(), dec.to(dev).eval()
    # every rank gets different images (seed = rank): the path shards by image
    image_h, depth_h = common.synthetic_inputs(B, S, seed=rank)
    image_h, depth_h = image_h.pin_memory(), depth_h.pin_memory()
    image, depth = image_h.to(dev), depth_h.to(dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)   # > 126 MB L2

    def step(img, dep):
        return TD.texture_prompts(enc, dec, img, dep, precision=args.precision, want_embedding3=False)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(args.warmup, 3)):
        step(image, depth)
    barrier()

    # ---- timed region: inputs resident in HBM --------------------------------------------------
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    n0 = capi.launch_count()
    with ClockSampler(local) as clocks:
        for a, b in ev:
            outs = None                         # the previous step's outputs are freed before the next step runs
            flush.zero_()                       # L2 flush between timed iterations (not timed)
            a.record()
            outs = step(image, depth)
            b.record()
        barrier()
    launches = capi.launch_count() - n0
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, outs[0], outs[2])
    outs = None
    from dgtd_b200.twig import sharding
    t_dev = sum(a.elapsed_time(b) for a, b in ev) / 1e3
    t_max = sharding.max_over_ranks(t_dev, dev)                     # device time, max over ranks
    value = world * B * args.steps / t_max

    # ---- end to end: pinned host inputs -> H2D -> path -> D2H of the result ---------------------
    # (twig/pipeline.py: copy of batch i+1 and read-back of result i-1 overlap the compute of batch i;
    #  every step's inputs cross PCIe inside the timed region)
    from dgtd_b200.twig.pipeline import HostPipeline
    res_h = [torch.empty(B, (S // 32) ** 2, 512, dtype=torch.float32).pin_memory() for _ in range(2)]   # last-stage prompt tokens
    pipe = HostPipeline(enc, dec, precision=args.precision, want_embedding3=False, device=dev)
    select = lambda e1, e3, toks: toks[3][2].float()
    e2e_steps = args.steps   # the same K as the device-timed loop; the un-overlapped first copy (pipeline fill) is inside
    for _ in pipe.run([(image_h, depth_h)] * 2, select, res_h):   # warm the pipeline's buffers
        pass
    barrier()
    t0 = torch.cuda.Event(enable_timing=True)
    t1 = torch.cuda.Event(enable_timing=True)
    t0.record()
    last = None
    for _, _, done in pipe.run([(image_h, depth_h)] * e2e_steps, select, res_h):
        last = done
    last.synchronize()
    torch.cuda.current_stream().wait_event(last)
    t1.record()
    barrier()
    e2e = world * B * e2e_steps / sharding.max_over_ranks(t0.elapsed_time(t1) / 1e3, dev)
    h2d = image_h.numel() * 4 + depth_h.numel() * 4
    d2h = res_h[0].numel() * 4

    # ---- roofline of the dominant kernel family (tcgen05 GEMM), measured live with CUDA events ---
    roof = None
    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        prof = OP.enable_gemm_profile(True) if hasattr(OP, "enable_gemm_profile") else None
        if prof is not None and args.precision == "bf16":
            for _ in range(2):
                step(image, depth)
            torch.cuda.synchronize()
            # dominant kernel instance: tc_gemm2_kernel on the large pointwise GEMMs (N, K >= 512: stages 2-3,
            # 62 of the 75 trunk GEMMs and ~80% of the step's tensor FLOPs); the short-K stage-0/1 GEMMs are
            # bound by their 600 MB of hidden-activation traffic / the GELU epilogue, not by the tensor pipe
            flops, ms, n = OP.collect_gemm_profile(min_n=512, min_k=512)
            fa, msa, na = OP.collect_gemm_profile(min_n=128, min_k=128)
            OP.enable_gemm_profile(False)
            peak = float(peaks.get("bf16_tflops_sustained", 1400.0))
            ach = flops / (ms * 1e-3) / 1e12 if ms > 0 else 0.0
            roof = {"bound": "tensor", "achieved": ach, "peak": peak, "unit": "TFLOP/s", "frac": ach / peak,
                    "traffic": 270.0e6, "traffic_note": "DRAM bytes of one stage-2 pwconv2 launch (M=36864,N=512,K=2048) "
                    "from profiles/r2_ncu_stage2_gemms.md (229.2 MB read + 40.8 MB written; 271.1 MB in "
                    "profiles/r1_ncu_full_stage2.md); algorithmic bytes of that launch 302 MB",
                    "kernel": "tc_gemm2_kernel (tcgen05 cta_group::2) on the stage-2/3 pointwise GEMMs (N, K >= 512)",
                    "launches_timed": n, "avg_launch_ms": ms / max(n, 1),
                    "all_trunk_gemms": {"achieved": fa / (msa * 1e-3) / 1e12 if msa > 0 else 0.0, "launches": na,
                                        "note": "incl. the memory/epilogue-bound stage-0/1 shapes (K = 128, 256)"},
                    "peak_source": "MEASURED_PEAKS.json bf16_tflops_sustained" if peaks else "fallback"}

    # ---- fwd+bwd (BASELINE configs[2]: SOD training, batch 16/GPU, 384^2, data parallel) ----------
    train = None
    if not args.no_train:
        # auxiliary legs never take the headline line down with them: a failure is reported in place
        try:
            train = train_bench(TD, enc, dec, dev, world, rank, local, args, common, sharding, precision="bf16")
            train["fp32_exact"] = train_bench(TD, enc, dec, dev, world, rank, local, args, common, sharding, steps=2,
                                              precision="fp32", measure_reduce=False)
        except Exception as e:   # noqa: BLE001
            train = dict(train or {}, error=f"{type(e).__name__}: {e}"[:300])

    full_train = None
    if not args.no_train and not args.no_backbone:
        try:
            full_train = full_model_train_bench(dev, world, rank, args, common, sharding)
        except Exception as e:   # noqa: BLE001
            full_train = {"error": f"{type(e).__name__}: {e}"[:300]}
        torch.cuda.empty_cache()

    # ---- high-resolution inference (BASELINE configs[4]: B = 8 at 768^2, sharded by image) --------
    highres = None
    if not args.no_highres:
        try:
            highres = highres_bench(TD, enc, dec, dev, world, rank, args, common, sharding)
        except Exception as e:   # noqa: BLE001
            highres = {"error": f"{type(e).__name__}: {e}"[:300]}

    # ---- next row 8f-1: the full backbone that consumes the prompts ----------------------------------
    backbone = None
    if not args.no_backbone:
        try:
            backbone = backbone_bench(TD, dev, world, rank, args, common, sharding)
        except Exception as e:   # noqa: BLE001
            backbone = {"error": f"{type(e).__name__}: {e}"[:300]}

    full_model = None
    if not args.no_backbone:
        try:
            full_model = full_model_bench(TD, dev, world, rank, args, common, sharding)
        except Exception as e:  # noqa: BLE001
            full_model = {"error": f"{type(e).__name__}: {e}"[:300]}
    loss_leg = None
    if rank == 0 and not args.no_backbone:
        try:
            loss_leg = loss_bench(dev, peaks if rank == 0 else {}, common)
        except Exception as e:   # noqa: BLE001
            loss_leg = {"error": f"{type(e).__name__}: {e}"[:300]}

    # ---- diffusion microbench (BASELINE configs[3]): MessagePassing core, 1024^2 x 256, shared weights
    diff = None
    if rank == 0 and not args.no_diffusion:
        try:
            diff = diffusion_microbench(OP, dev, peaks if rank == 0 else {})
        except Exception as e:   # noqa: BLE001
            diff = {"error": f"{type(e).__name__}: {e}"[:300]}

    cpu = None
    if rank == 0 and not args.no_cpu_baseline:
        n_cpu = min(args.cpu_sample, 8)
        rate, dt, cores, kind = cpu_reference_rate(S, n_cpu, 2, 1)
        cpu = {"value": rate, "unit": UNIT, "cores": cores, "kind": kind,
               "sample": f"{n_cpu} images of the same workload per step, 2 timed + 1 warm-up steps, fp32 torch CPU, {cpu_model()}"}

    eager = None
    if rank == 0 and not args.no_eager_reference:
        ours = {"hot_ms": t_max / args.steps * 1e3,
                "full_ms": (full_model or {}).get("ms_per_step"),
                "mp_ms": ((diff or {}).get("sweep") or [{}])[0].get("ms")}
        try:
            eager = gpu_eager_reference(dev, args, common, ours)
        except Exception as e:   # noqa: BLE001
            eager = {"error": f"{type(e).__name__}: {e}"[:300]}

    if rank == 0:
        def pick(d, *keys):
            return {k: d.get(k) for k in keys if isinstance(d, dict) and k in d} if isinstance(d, dict) else d
        # the driver keeps the TAIL of this line: the compact `summary` object goes last, bulky per-sweep detail first
        summary = {
            "hot_path": {"images_per_s": value, "ms_per_step": t_max / args.steps * 1e3, "e2e_images_per_s": e2e},
            "train_fwd_bwd": pick(train, "value", "ms_per_step", "batch_per_gpu", "precision", "allreduce_exposed_ms",
                                  "allreduce_in_situ_ms", "grad_allreduce", "error"),
            "train_fp32_exact": pick((train or {}).get("fp32_exact"), "value", "ms_per_step"),
            "full_model_train": pick(full_train, "value", "ms_per_step", "batch_per_gpu", "precision", "parameters",
                                     "launches_per_step", "loss_finite", "grad_less_parameters", "allreduce_exposed_ms",
                                     "error"),
            "highres_768": pick(highres, "value", "ms_per_step", "batch_per_gpu", "error"),
            "full_model_predict": pick(full_model, "value", "ms_per_step", "error"),
            "full_model_predict_e2e": pick((full_model or {}).get("e2e"), "value", "h2d_bytes_per_step", "d2h_bytes_per_step", "error"),
            "diffusion_W1": ({"fp32_ms_by_T": {str(r["T"]): round(r["ms"], 4) for r in diff.get("sweep", [])},
                              "hbm_frac_T1": diff.get("hbm_frac_T1"),
                              "bf16_storage_T1_ms": (diff.get("bf16_storage_T1") or {}).get("ms"),
                              "bf16_storage_hbm_frac": (diff.get("bf16_storage_T1") or {}).get("hbm_frac"),
                              "simt_f32_T1_ms": diff.get("simt_f32_T1_ms"),
                              "kernel": diff.get("kernel")} if isinstance(diff, dict) and "sweep" in diff else diff),
            "gpu_eager_reference": eager,
        }
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": t_max / args.steps * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": args.precision, "data": "synthetic",
            "config": {"workload": f"COD inference hot path (prompt_encoder + 16 ShapePropDecoders + token layout), "
                                   f"batch {B}/GPU, {S}x{S} RGB-D, random-init weights (BASELINE configs[1])",
                       "l2": "256 MiB buffer written between timed iterations", "sharding": "by image, no collective"},
            "e2e": {"value": e2e, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "result": "stage-4 prompt tokens of the last block (B,144,512) fp32"},
            "gpu_launches": int(launches), "clocks": clocks.summary(),
            "roofline": roof, "cpu_baseline": cpu,
            "diffusion_microbench": diff, "structure_loss": loss_leg, "backbone_forward_features": backbone,
            "full_model_predict": full_model, "train_fwd_bwd": train, "full_model_train": full_train,
            "highres_768": highres,
            "summary": summary,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    args = parse()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
