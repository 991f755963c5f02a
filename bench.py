#!/usr/bin/env python
"""Benchmark of the denoising-loop hot path (BASELINE.json): images/sec for SD-v1 512x512, 50-step PLMS, CFG 7.5.

  python bench.py --gpus N --steps K --warmup W            # B200 engine (torchrun launches one rank per GPU)
  python bench.py --impl reference --steps K --warmup W    # CPU baseline arm (oracle port of the reference, host cores)
  python bench.py ... --dump-outputs DIR                   # also write the last timed step's images (DIR/images.npy)

The inputs are the same on every run. The outputs are not bit-identical from run to run: graph mode times its GEMM
tile / split-K candidates per process and GroupNorm partial sums meet in fp64 atomics, so two runs of one build differ
by 1 (of 255) in a few percent of the pixels (5 % on a B200); compare dumps of two builds with that tolerance.

A "step" is one pass of the hot path over one batch: CLIP text encode of [uncond; prompts] -> 51 guided UNet
evaluations (PLMS-50) -> AutoencoderKL decode -> uint8 images. Weights are seeded random-init of the SD-v1
architecture (no checkpoint offline), data is synthetic (seeded token ids and start noise).
Prints ONE JSON line (rank 0).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "images_per_sec_sdv1_512x512_plms50_cfg7.5"
UNET_GF_PER_SAMPLE = 803.27     # SURVEY.md §8(d): algorithmic GFLOP per UNet evaluation per sample @ 64x64 latent
VAE_DEC_GF = 2514.5             # per image @ 512x512
CLIP_GF_PER_PROMPT = 13.0
DUMP_BYTES = 64 * 10**6         # --dump-outputs writes at most this much in all


def dump_outputs(out_dir, arrays):
    """Write each array as out_dir/<name>.npy in float32. An array over its share of DUMP_BYTES is replaced by a fixed,
    seeded sample of its elements (the same indices for the same shape), so runs of two builds compare element for
    element."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    budget = DUMP_BYTES // len(arrays) // 4 - 32    # float32 elements per array; 128 bytes left for the .npy header
    for name, a in arrays.items():
        a = a.detach().float().cpu()
        if a.numel() > budget:
            idx = torch.randperm(a.numel(), generator=torch.Generator().manual_seed(0))[:budget].sort().values
            a = a.flatten()[idx]
        np.save(os.path.join(out_dir, name + ".npy"), a.numpy())


def gemm_dram_traffic():
    """DRAM bytes per gemm_tc launch from the committed ncu capture of one UNet evaluation (dram__bytes_read.sum +
    dram__bytes_write.sum per launch, `ncu --metrics ... -k regex:gemm_tc python scripts/profile_unet.py`): newest round
    first. Returns (bytes per launch or None, source file, launches in the capture)."""
    import csv
    for name in ("r02_gemm_dram.csv", "r01_gemm_dram.csv"):
        path = os.path.join(ROOT, "profiles", name)
        if not os.path.exists(path):
            continue
        try:
            rows = [r for r in csv.reader(l for l in open(path) if l.startswith('"'))]
            hdr = rows[0]
            i_id, i_name, i_unit, i_val = hdr.index("ID"), hdr.index("Metric Name"), hdr.index("Metric Unit"), hdr.index("Metric Value")
            scale = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
            tot, ids = 0.0, set()
            for r in rows[1:]:
                if r[i_name].startswith("dram__bytes_"):
                    tot += float(r[i_val].replace(",", "")) * scale.get(r[i_unit], 1.0)
                    ids.add(r[i_id])
            if ids:
                return tot / len(ids), "profiles/" + name, len(ids)
        except Exception:
            continue
    return None, None, 0


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(tensor_burst=d["bf16_tflops"], tensor_sustained=d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                    hbm=d["hbm_gbs"], source="measured (MEASURED_PEAKS.json)")
    return dict(tensor_burst=1590.0, tensor_sustained=1400.0, hbm=6650.0, source="fallback (B200_PROFILING.md)")


class ClockSampler:
    """nvidia-smi clocks/throttle reasons sampled DURING the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.rows, self.proc, self.idx = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.idx), "-lms", "200"], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return None
        self.proc.terminate()
        sm = sorted(int(float(r[1])) for r in self.rows if len(r) >= 9 and r[1].replace(".", "").isdigit())
        if not sm:
            return None
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            if len(r) >= 9:
                for n, v in zip(names, r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
        mx = max(int(float(r[2])) for r in self.rows if len(r) >= 9)
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------ CPU arm
def cpu_unet_eval_seconds(threads, reps=1):
    """Time the oracle's UNet evaluation (N_s = 2, 64x64 latent, fp32) on the host cores."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import ldm_oracle as O
    import sdb200  # noqa: F401
    from sdb200 import arch
    torch.set_num_threads(threads)
    sd = arch.random_state_dict(arch.unet_param_shapes(arch.SD_V1_UNET), 11)
    g = torch.Generator().manual_seed(0)
    x = torch.randn(2, 4, 64, 64, generator=g)
    ctx = torch.randn(2, 77, 768, generator=g)
    t = torch.tensor([981, 981])
    times = []
    with torch.no_grad():
        for _ in range(reps):
            t0 = time.perf_counter()
            O.unet_forward(sd, x, t, ctx)
            times.append(time.perf_counter() - t0)
    return times


def run_reference(args):
    """`--impl reference`: the reference's CPU implementation of the path (oracle port; /root/reference cannot travel
    to the GPU box) on all host threads. Each step = a bounded sample: ONE guided UNet evaluation (N_s=2, 64x64);
    images/sec is extrapolated as 1 / (51 * t_eval + t_decode) with the VAE decode timed once."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = min(os.cpu_count() or 1, 32)   # more threads than this slow the fp32 einsum/conv path down
    times = cpu_unet_eval_seconds(threads, reps=args.warmup + args.steps)[args.warmup:]
    t_eval = sum(times) / len(times)
    import ldm_oracle as O
    from sdb200 import arch
    # the rest of an image, timed for real once: AutoencoderKL decode of a 64x64 latent (512x512 image) and the CLIP text
    # encode of [uncond; prompt]
    vsd = arch.random_state_dict(arch.vae_param_shapes(arch.SD_V1_VAE), 12)
    z = torch.randn(1, 4, 64, 64, generator=torch.Generator().manual_seed(1))
    with torch.no_grad():
        t0 = time.perf_counter()
        O.decode_first_stage(vsd, z)
        t_dec = time.perf_counter() - t0
    t_clip = 0.0
    try:
        csd = arch.random_state_dict(arch.clip_param_shapes(arch.SD_V1_CLIP), 13)
        ids = torch.randint(0, 49406, (2, 77), generator=torch.Generator().manual_seed(2))
        with torch.no_grad():
            t0 = time.perf_counter()
            O.clip_text(csd, ids, arch.SD_V1_CLIP["num_attention_heads"])
            t_clip = time.perf_counter() - t0
    except Exception as ex:   # the CLIP port is optional for the CPU arm; the decode and the UNet evaluations dominate
        t_clip = 0.0
        print(f"bench.py: CLIP leg of the CPU arm skipped ({ex!r})", file=sys.stderr)
    value = 1.0 / (51 * t_eval + t_dec + t_clip)
    sample = (f"per step: 1 guided UNet eval N_s=2 @64x64 fp32 ({t_eval:.2f} s, bounded sample of the 51 per image); once: "
              f"AutoencoderKL decode 64x64 -> 512x512 ({t_dec:.1f} s) and CLIP encode of 2x77 tokens ({t_clip:.2f} s); "
              "image time = 51*eval + decode + clip")
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": value, "unit": "images/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1000.0 * t_eval, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"txt2img SD-v1-4 random-init, 512x512, 50 PLMS steps (51 UNet evals), CFG 7.5, "
                               f"batch {args.batch} per GPU", "parallelism": f"dp{args.gpus}",
                   "device": f"host CPU, {threads} threads (one image stream; the CPU arm does not scale with --gpus)"},
        "cpu_baseline": {"value": value, "unit": "images/s", "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))


# ------------------------------------------------------------------------------------------------ GPU arm
def run_gpu(args):
    import torch.distributed as dist
    import sdb200
    from sdb200 import ops, pipeline

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the sdb200 engine has no CPU fallback; use --impl reference)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    B = args.batch

    model = pipeline.build_model()
    pipeline.load_random_weights(model, dev, gen_device=dev)   # same seeds on every rank -> identical weights
    if world > 1:
        # NCCL broadcast of the packed weights from rank 0 over NVLink (SURVEY §8e) instead of N host loads
        sdb200.dist.broadcast_weights(model.model.diffusion_model.W, model.first_stage_model.W,
                                      model.cond_stage_model.W, src=0)
    pipe = pipeline.Txt2Img(model, sampler="plms", steps=50, scale=7.5, height=512, width=512, cuda_graph=True)

    # synthetic inputs: seeded token ids (BOS + tokens + EOS padding) and start noise, per global sample index
    g = torch.Generator().manual_seed(1234 + rank)
    ids_h = torch.randint(0, 49406, (B, 77), generator=g)
    ids_h[:, 0] = 49406
    ids_h[:, 20:] = 49407
    un_h = torch.full((B, 77), 49407, dtype=torch.long)
    un_h[:, 0] = 49406
    lo, hi = sdb200.dist.shard_range(B * world, rank, world)
    xT_h = sdb200.dist.batch_noise(lo, hi, (4, 64, 64), seed=42)   # per GLOBAL sample index: world-size independent
    ids_p, un_p, xT_p = ids_h.pin_memory(), un_h.pin_memory(), xT_h.pin_memory()
    out_h = torch.empty((B, 512, 512, 3), dtype=torch.uint8).pin_memory()
    ids_d, un_d, xT_d = ids_h.to(dev), un_h.to(dev), xT_h.to(dev)
    gathered = [torch.empty((B, 512, 512, 3), dtype=torch.uint8, device=dev) for _ in range(world)] if rank == 0 else None

    def step_resident():
        img = pipe(ids_d, un_d, x_T=xT_d)
        if world > 1:   # gather of decoded uint8 images to rank 0 over NVLink
            dist.gather(img, gathered, dst=0)
        return img

    def step_e2e():
        i = ids_p.to(dev, non_blocking=True)
        u = un_p.to(dev, non_blocking=True)
        x = xT_p.to(dev, non_blocking=True)
        img = pipe(i, u, x_T=x)
        if world > 1:
            dist.gather(img, gathered, dst=0)
        out_h.copy_(img, non_blocking=True)
        return img

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        """Runs `steps` steps between two events; returns (ms, what the last step returned)."""
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            out = fn()
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms), out

    for _ in range(max(args.warmup, 3)):
        step_resident()
    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
    n0 = ops.launch_count()
    if os.environ.get("SDB_PROFILE_RANGE"):   # ncu --profile-from-start off: only the timed steps are captured
        torch.cuda.profiler.start()
    ms_total, last_img = timed(step_resident, args.steps)
    if os.environ.get("SDB_PROFILE_RANGE"):
        torch.cuda.profiler.stop()
    launches = (ops.launch_count() - n0) // args.steps
    clk = clocks.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        # the images the last timed step handed its caller (all ranks' on rank 0), before later steps reuse `gathered`
        dump_outputs(args.dump_outputs, {"images": torch.cat(gathered) if world > 1 else last_img})
    step_e2e()
    ms_e2e, _ = timed(step_e2e, args.steps)
    # sanity of what was timed (outside the timed region): the latent the 51 evaluations produce is finite and the
    # decoded image is not constant — a NaN anywhere in the UNet would show here
    lat = pipe(ids_d, un_d, x_T=xT_d, return_latent=True)
    img_chk = out_h.float()
    output_ok = bool(torch.isfinite(lat).all()) and float(lat.std()) > 0 and float(img_chk.std()) > 0

    # UNet step time (graph replay of one guided evaluation, N_s = 2B), L2 flushed between repetitions
    unet = model.model.diffusion_model
    gk = next(iter(unet._graphs.values()))
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)
    ts = []
    for _ in range(10):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        gk["graph"].replay()
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    unet_ms = sorted(ts)[len(ts) // 2]

    # roofline of the dominant kernel family (tcgen05 GEMM / implicit conv): record every sdb_gemm descriptor of one
    # UNet evaluation, then replay exactly those launches back to back through the C ABI between two CUDA events on the
    # launching stream (no Python op overhead in between), L2 flushed before each replay
    roof = None
    if rank == 0:
        import ctypes as C
        unet.use_cuda_graph = False
        x2 = gk["x"].clone()
        t2 = torch.full((x2.shape[0],), 981.0, device=dev)
        unet._forward_impl(x2, t2, gk["kvs"])
        ops.RECORD = []
        keep_out = unet._forward_impl(x2, t2, gk["kvs"])
        recs, ops.RECORD = ops.RECORD, None
        unet.use_cuda_graph = True
        lib = sdb200.lib.load()
        stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
        n0 = ops.launch_count()
        reps = []
        for _ in range(5):
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda._sleep(int(2e7))   # ~10 ms head start so the host is ahead of the GPU for the whole replay
            e0.record()
            for d, _, _ in recs:
                lib.sdb_gemm(C.byref(d), stream)
            e1.record()
            torch.cuda.synchronize()
            reps.append(e0.elapsed_time(e1))
        gemm_kernels = (ops.launch_count() - n0) // 5
        ms = sorted(reps)[len(reps) // 2]
        fl = sum(r[1] for r in recs)
        n = len(recs)
        pk = peaks()
        ach = fl / (ms * 1e-3) / 1e12
        traffic, traffic_src, traffic_n = gemm_dram_traffic()
        roof = {"kernel": "gemm_tc_kernel (tcgen05 GEMM / implicit 3x3 conv, all tile shapes) + its split-K epilogue",
                "bound": "tensor", "achieved": ach, "peak": pk["tensor_sustained"], "unit": "TFLOP/s",
                "frac": ach / pk["tensor_sustained"], "traffic": traffic,
                "traffic_note": f"ncu dram__bytes_read+write summed over the {traffic_n} gemm_tc launches of one UNet evaluation "
                                f"/ {traffic_n}, read at run time from {traffic_src}; algorithmic bytes per launch ~9.1 MB "
                                "(weights 1.72 GB + operands)",
                "peak_source": pk["source"] + ", sustained bf16", "launches_per_unet_eval": n,
                "kernels_per_unet_eval": int(gemm_kernels),
                "algorithmic_gflop_per_launch": fl / n / 1e9, "avg_launch_us": 1000.0 * ms / n,
                "gemm_ms_per_unet_eval": ms, "gemm_share_of_unet_eval": ms / unet_ms,
                "unet_eval": {"ms": unet_ms, "algorithmic_tflop": UNET_GF_PER_SAMPLE * 2 * B / 1e3,
                              "achieved_tflops": UNET_GF_PER_SAMPLE * 2 * B / 1e3 / (unet_ms * 1e-3),
                              "frac_of_peak": UNET_GF_PER_SAMPLE * 2 * B / 1e3 / (unet_ms * 1e-3) / pk["tensor_sustained"]}}
        del keep_out

    # supplementary: the same pipeline at a larger per-GPU batch (BASELINE metric quotes batch 1/8/32); not the headline
    extra = None
    if rank == 0 and world == 1 and args.extra_batch > 1:
        Bx = args.extra_batch
        gx = torch.Generator().manual_seed(99)
        idx = torch.randint(0, 49406, (Bx, 77), generator=gx)
        idx[:, 0] = 49406
        idx[:, 20:] = 49407
        unx = torch.full((Bx, 77), 49407, dtype=torch.long)
        unx[:, 0] = 49406
        idx, unx = idx.to(dev), unx.to(dev)
        xTx = sdb200.dist.batch_noise(0, Bx, (4, 64, 64), seed=43).to(dev)
        for _ in range(2):
            pipe(idx, unx, x_T=xTx)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        pipe(idx, unx, x_T=xTx)
        e1.record()
        torch.cuda.synchronize()
        msx = e0.elapsed_time(e1)
        extra = {"batch": Bx, "images_per_s": Bx / (msx * 1e-3), "ms_per_batch": msx,
                 "achieved_tflops": Bx * (51 * 2 * UNET_GF_PER_SAMPLE + VAE_DEC_GF) / 1e3 / (msx * 1e-3)}

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        threads = min(os.cpu_count() or 1, 32)
        t_eval = min(cpu_unet_eval_seconds(threads, reps=2))
        cpu = {"value": 1.0 / (51 * t_eval), "unit": "images/s", "cores": threads, "kind": "port",
               "sample": f"2 oracle UNet evals (N_s=2, 64x64 latent, fp32), best {t_eval:.2f} s; image = 51 evals, "
                         "VAE/CLIP excluded (favours the CPU)"}

    if rank == 0:
        images = B * world
        value = images * args.steps / (ms_total * 1e-3)
        e2e = images * args.steps / (ms_e2e * 1e-3)
        line = {
            "metric": METRIC, "value": value, "unit": "images/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms_total / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "fp16", "data": "synthetic",
            "config": {"workload": f"txt2img SD-v1-4 random-init, 512x512, 50 PLMS steps (51 UNet evals), CFG 7.5, "
                                   f"batch {B} per GPU", "parallelism": f"dp{world}", "l2": "weights 2.1 GB > 126 MB L2; "
                                   "no explicit flush inside a step (UNet-only timing flushes L2)",
                       "arithmetic": "fp16 tensor-core operands, fp32 accumulate / residual stream / norms / softmax",
                       "algorithmic_tflop_per_image": (51 * 2 * UNET_GF_PER_SAMPLE + VAE_DEC_GF + 2 * CLIP_GF_PER_PROMPT) / 1e3},
            "unet_step_ms": unet_ms, "gpu_launches": int(launches), "output_finite": output_ok,
            "e2e": {"value": e2e, "unit": "images/s", "h2d_bytes_per_step": int(ids_p.nbytes + un_p.nbytes + xT_p.nbytes),
                    "d2h_bytes_per_step": int(out_h.nbytes)},
            "roofline": roof, "cpu_baseline": cpu, "clocks": clk, "larger_batch": extra,
        }
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--batch", type=int, default=1, help="images per GPU per step")
    ap.add_argument("--impl", default="sdb200", choices=["sdb200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--extra-batch", type=int, default=8, help="also time one step at this per-GPU batch (0: skip)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the uint8 images of the last one as float32 to DIR/images.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "sdb200":
        ap.error("--dump-outputs writes the images of the sdb200 pipeline; --impl reference times UNet evaluations only")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
