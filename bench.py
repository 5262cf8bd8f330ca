#!/usr/bin/env python3
"""bench.py — 256-px images/sec with 35-step CFG sampling (BASELINE.json metric, configs[1]) + every other BASELINE config.

One "step" = one full pass of the hot path over one batch: `DiffusionGenerator.generate` semantics for B images
(35 model calls on the 2B-sample CFG batch through the CUDA-graph sampler) + the VAE decode of the B latents.

    python bench.py --gpus 1 --steps 5 --warmup 3                 # this repo (libtld_b200, sm_100a)
    python -m torch.distributed.run --nnodes=1 --nproc-per-node 8 --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus 8 --steps 5 --warmup 3                     # one process per GPU
    python bench.py --impl reference --steps 2 --warmup 1         # reference algorithm on the host cores
    python bench.py --steps 5 --warmup 3 --dump-outputs DIR       # + the last timed step's images / latents as DIR/*.npy

The inputs (weights, labels, noise) are seeded, so two builds run with the same arguments can be compared output for output
on what `--dump-outputs` writes.  The latents repeat bit for bit from run to run; the decoded images do not, because the
VAE's GroupNorm statistics are summed with shared-memory atomics in no fixed order (two runs on a B200 differed by 4e-3
relative Frobenius), so compare images with a tolerance.

Prints ONE JSON line (rank 0).  Headline keys (the contract): `value` = whole-job images/s with inputs resident in HBM;
`e2e` = the same metric through the public API with pinned HOST inputs (H2D of labels+noise, D2H of the decoded images inside
the timed region); `roofline` = the kernel with the largest share of the step, timed alone with CUDA events; `cpu_baseline`
= the oracle port (oracle/tld_oracle.py, the reference algorithm in torch fp32) on the box's host cores over a bounded sample.

`configs` (same run, same N GPUs) covers the other BASELINE.json configurations:
  px512_b16          configs[2]: 4x64x64 latent, 35-step CFG, batch 16 per GPU (+ VAE decode)
  px1024_sweep       configs[4]: 4x128x128 latent, 50-step CFG, batch 1..32 per GPU: ms/step, images/s, model TFLOP/s
  train_step         configs[3]: train.main's step (forward, MSE, backward, gradient all-reduce over NCCL overlapped with the
                     backward, fused Adam+EMA), 32 samples per GPU (= 256 global at 8 GPUs): ms, samples/s, and the exposed
                     all-reduce time (same step with the all-reduce switched off)
  train_step_b256    (N = 1 only) the whole 256-sample batch on one GPU
Context numbers: `roofline.cublas_same_shape` (torch.matmul = cuBLAS on the dominant GEMM's shape) and `stock_torch_b200`
(the oracle port run on the GPU with stock PyTorch kernels, fp32 and bf16 autocast) — the "honest bar" of SURVEY.md §8d.
Weights are random-init (no checkpoint offline), data synthetic.
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

IMG, D, L, N_ITER, GUIDANCE = 32, 768, 12, 35, 6.0  # BASELINE configs[1]: 100M denoiser, 4x32x32 latent


def fwd_flops_per_sample(img=IMG, d=D, layers=L) -> float:
    """SURVEY.md §8d: F_fwd(N) = L * F_blk + F_eh"""
    n = (img // 2) ** 2
    blk = 24 * n * d * d + 4 * n * n * d + 80 * n * d + 8 * d * d
    eh = 2 * n * 16 * 16 + 4 * n * 16 * d + 2 * (256 * d + d * d) + 2 * 768 * d
    return float(layers * blk + eh)


# ------------------------------------------------------------------------------------------ clocks sampler
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx = float(r[1])
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "samples": len(sm),
                "reasons": sorted(reasons)}


def host_cores() -> int:
    """CPU threads this process may really use: min(affinity mask, cgroup cpu quota) — os.cpu_count() alone
    over-subscribes badly inside a CPU-limited container."""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    try:
        with open("/sys/fs/cgroup/cpu.max") as f:
            quota, period = f.read().split()
        if quota != "max":
            n = min(n, max(1, int(float(quota) / float(period))))
    except Exception:
        try:  # cgroup v1
            q = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0 and per > 0:
                n = min(n, max(1, q // per))
        except Exception:
            pass
    return max(1, n)


def cpu_threads() -> int:
    """torch threads of the CPU arm: more than ~32 only adds synchronisation overhead to the oracle's fp32 GEMMs (on the
    96-thread scaling host round 1's in-line baseline got SLOWER with all threads)."""
    return min(host_cores(), 32)


# ------------------------------------------------------------------------------------------ reference / cpu arm
def cpu_generation(num_imgs: int, n_iter: int, threads: int) -> float:
    """One bounded pass of the reference algorithm on the host: oracle sampler + oracle VAE decode. Returns seconds."""
    from oracle import tld_oracle as O
    from oracle import vae_oracle as V
    from transformer_latent_diffusion_b200.vae import AutoencoderKLDecoder

    torch.set_num_threads(threads)
    cfg = O.OracleCfg(image_size=IMG, embed_dim=D, n_layers=L)
    if not hasattr(cpu_generation, "_state"):
        torch.manual_seed(0)
        vae_sd = {k: v.detach() for k, v in AutoencoderKLDecoder().state_dict().items()}
        cpu_generation._state = (O.synth_state_dict(cfg, 0), vae_sd)
    sd, vae_sd = cpu_generation._state
    g = torch.Generator().manual_seed(1)
    labels = torch.randn(num_imgs, 768, generator=g)
    seeds = torch.randn(num_imgs, 4, IMG, IMG, generator=g)
    t0 = time.perf_counter()
    with torch.no_grad():
        lat = O.generate_latents(sd, cfg, labels, seeds, n_iter=n_iter, class_guidance=GUIDANCE, exponent=1,
                                 sharp_f=0, bright_f=0, use_ddpm_plus=True)
        V.decode(vae_sd, lat * 8)
    return time.perf_counter() - t0


def run_reference(args) -> None:
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return  # the CPU arm runs on rank 0 only
    threads = cpu_threads()
    sample_imgs = args.cpu_images
    for _ in range(args.warmup):
        cpu_generation(sample_imgs, N_ITER, threads)
    t = 0.0
    for _ in range(args.steps):
        t += cpu_generation(sample_imgs, N_ITER, threads)
    value = sample_imgs * args.steps / t
    sample = (f"{sample_imgs} image(s) (CFG batch {2 * sample_imgs}) x {N_ITER} CFG steps + VAE decode per step, fp32, "
              f"{threads} torch threads of {host_cores()} usable cores; kind=port: /root/reference does not exist on the GPU box "
              "and its imports (clip, diffusers, accelerate) are absent, so the pinned oracle port is timed")
    print(json.dumps({
        "impl": "reference", "metric": "images_per_sec_256px_35step_cfg", "value": value, "unit": "images/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "100M denoiser 256px sampling: 4x32x32 latent, 35-step CFG (oracle port on host CPU)",
                   "images_per_step": sample_imgs, "n_iter": N_ITER, "class_guidance": GUIDANCE},
        "cpu_baseline": {"value": value, "unit": "images/s", "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }))


# ------------------------------------------------------------------------------------------ B200 arm helpers
def _events():
    return torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)


def _time_rotating(fn, nbuf: int, reps: int = 20, warm: int = 3) -> float:
    """ms per call; fn(i) works on operand set i % nbuf (the sets together exceed L2)"""
    for i in range(warm):
        fn(i % nbuf)
    e0, e1 = _events()
    torch.cuda.synchronize()
    e0.record()
    for i in range(reps):
        fn(i % nbuf)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def _profile_traffic(name: str):
    """dram bytes per launch of `name` from the committed ncu capture (profiles/r02_kernel_traffic.json), or None"""
    try:
        with open(os.path.join(ROOT, "profiles", "r02_kernel_traffic.json")) as f:
            t = json.load(f)
        e = t.get(name)
        return (e["dram_bytes"], e.get("source")) if e else (None, None)
    except Exception:
        return None, None


def time_dominant_kernels(lib, peaks) -> dict:
    """The kernel with the largest share of the 256-px step is the fused MLP front half (mlp.0 up-projection on the tensor
    cores + depthwise 3x3 + GELU on the CUDA cores, T = 32768 tokens): timed alone, CUDA events on the launch stream, operands
    rotated through sets larger than L2.  Next to it: the plain tcgen05 GEMM of the same shape and torch.matmul (cuBLAS)."""
    import math

    M, N, K = 128 * (IMG // 2) ** 2, 4 * D, D
    nbuf = 3  # 3 x (50 MB A + 200 MB out) > 126 MB L2
    A = [torch.randn(M, K, device="cuda").bfloat16() for _ in range(nbuf)]
    W = (torch.randn(N, K, device="cuda") / math.sqrt(K)).bfloat16()
    bias = torch.randn(N, device="cuda")
    w9 = torch.randn(9, N, device="cuda") / 3
    dwb = torch.randn(N, device="cuda") * 0.1
    C = [torch.empty(M, N, device="cuda", dtype=torch.bfloat16) for _ in range(nbuf)]
    st = torch.cuda.current_stream().cuda_stream
    L_ = lib.load()

    def fused(i):
        lib.check(L_.tld_op_gemm_up_dwconv_gelu(lib.ptr(A[i]), lib.ptr(W), lib.ptr(bias), None, None, lib.ptr(w9), lib.ptr(dwb),
                                                lib.ptr(C[i]), M // 256, K, N, st), "fused")

    def gemm(i):
        lib.check(L_.tld_op_gemm(1, lib.ptr(A[i]), lib.ptr(W), M, N, K, lib.ptr(C[i]), lib.ptr(bias), st), "gemm")

    Wt = W.t()

    def cublas(i):
        torch.matmul(A[i], Wt, out=C[i])

    ms_fused, ms_gemm, ms_cublas = _time_rotating(fused, nbuf), _time_rotating(gemm, nbuf), _time_rotating(cublas, nbuf)
    gemm_flops = 2.0 * M * N * K
    flops = gemm_flops + 2.0 * 9 * M * N          # + the depthwise taps (SURVEY.md §8d: 72 N D per sample per block)
    peak = peaks.get("bf16_tflops")
    src = "measured (MEASURED_PEAKS.json bf16_tflops, burst)"
    if not peak:
        peak, src = 1590.0, "fallback (B200_PROFILING.md)"
    traffic, tsrc = _profile_traffic("gemm_up_dwconv_gelu_kernel")
    achieved = flops / (ms_fused * 1e-3) / 1e12
    del A, C
    return {"bound": "tensor",
            "kernel": "gemm_up_dwconv_gelu_kernel (mlp.0 up-projection M=32768 N=3072 K=768 on tcgen05 CTA-pair tiles + depthwise 3x3 + GELU "
                      "on the CUDA cores in the epilogue; the largest share of the 256-px step)",
            "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak, "peak_source": src,
            "ms_per_launch": ms_fused, "flops_per_launch": flops, "traffic": traffic, "traffic_source": tsrc,
            "algorithmic_bytes_per_launch": 2.0 * (M * K + N * K + M * N),
            "method": "CUDA events around 20 back-to-back launches on the launch stream, 3 rotating operand sets (>L2)",
            "plain_gemm_same_shape": {"kernel": "gemm_bf16_tn_kernel<BN=256,EPI_BIAS_BF16,CTAS=2>", "ms_per_launch": ms_gemm,
                                      "tflops": gemm_flops / (ms_gemm * 1e-3) / 1e12, "frac": gemm_flops / (ms_gemm * 1e-3) / 1e12 / peak},
            "cublas_same_shape": {"kernel": "torch.matmul bf16 (cuBLAS), no bias", "ms_per_launch": ms_cublas,
                                  "tflops": gemm_flops / (ms_cublas * 1e-3) / 1e12}}


def stock_torch_b200(dev) -> dict:
    """Context, not the product: the oracle port (plain torch ops, the reference's algorithm) run ON the B200 with stock PyTorch
    kernels (cuBLAS / cuDNN / ATen) in fp32 and under bf16 autocast — SURVEY.md §8d's "honest bar".  Bounded sample."""
    from oracle import tld_oracle as O

    cfg = O.OracleCfg(image_size=IMG, embed_dim=D, n_layers=L)
    sd = {k: v.to(dev) for k, v in O.synth_state_dict(cfg, 0).items()}
    B = 16
    g = torch.Generator().manual_seed(1)
    labels = torch.randn(B, 768, generator=g).to(dev)
    seeds = torch.randn(B, 4, IMG, IMG, generator=g).to(dev)
    out = {"images_per_step": B, "n_iter": N_ITER, "note": "denoiser loop only (no VAE), eager stock PyTorch on the same GPU"}
    for name, ctx in (("fp32", torch.autocast("cuda", enabled=False)), ("bf16_autocast", torch.autocast("cuda", dtype=torch.bfloat16))):
        try:
            with torch.no_grad(), ctx:
                O.generate_latents(sd, cfg, labels, seeds, n_iter=4, class_guidance=GUIDANCE, exponent=1, sharp_f=0, bright_f=0)
                torch.cuda.synchronize()
                e0, e1 = _events()
                e0.record()
                O.generate_latents(sd, cfg, labels, seeds, n_iter=N_ITER, class_guidance=GUIDANCE, exponent=1, sharp_f=0, bright_f=0)
                e1.record()
                torch.cuda.synchronize()
            ms = e0.elapsed_time(e1)
            out[name] = {"ms_per_model_call": ms / N_ITER, "images_per_s_denoiser_only": B / (ms * 1e-3)}
        except Exception as e:  # noqa: BLE001
            out[name] = {"error": f"{type(e).__name__}: {e}"[:200]}
    return out


DUMP_BYTES = 64 * 10**6  # --dump-outputs writes at most this much in all


def dump_outputs(path: str, outputs: dict) -> None:
    """Each output as `path/<name>.npy` in float32.  Above DUMP_BYTES in all, every output keeps the same rows of the batch,
    a sample fixed by seed 0 and the batch size, so two runs with the same arguments write the same samples."""
    import numpy as np

    arrays = {k: v.detach().float().cpu() for k, v in outputs.items()}
    n = next(iter(arrays.values())).shape[0]
    row_bytes = sum(4 * v[0].numel() for v in arrays.values())
    keep = min(n, DUMP_BYTES // row_bytes)
    if keep < n:
        rows = torch.randperm(n, generator=torch.Generator().manual_seed(0))[:keep].sort().values
        arrays = {k: v[rows] for k, v in arrays.items()}
    os.makedirs(path, exist_ok=True)
    for k, v in arrays.items():
        np.save(os.path.join(path, k + ".npy"), v.numpy())
    print(f"bench.py: wrote {', '.join(f'{k}{tuple(v.shape)}' for k, v in arrays.items())} (float32, {keep} of {n} "
          f"images) to {path}", file=sys.stderr)


def run_b200(args) -> None:
    from transformer_latent_diffusion_b200 import _lib
    from transformer_latent_diffusion_b200.denoiser import Denoiser
    from transformer_latent_diffusion_b200.diffusion import DiffusionGenerator
    from transformer_latent_diffusion_b200.vae import AutoencoderKLDecoder

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}: launch with torch.distributed.run --nproc-per-node {args.gpus}")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback in the product path)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist = None
    if world > 1:
        import torch.distributed as dist_mod

        dist = dist_mod
        # stdout carries exactly one JSON line: NCCL prints its "NCCL version ..." banner to stdout when the first
        # communicator is created, so file descriptor 1 points at stderr while that happens
        sys.stdout.flush()
        saved_stdout = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=dev)
            dist.barrier()
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved_stdout, 1)
            os.close(saved_stdout)

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, k):
        """device ms of k calls, barrier + synchronize on both sides, max over ranks"""
        e0, e1 = _events()
        barrier()
        e0.record()
        for _ in range(k):
            fn()
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if dist is not None:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms)

    peaks = {}
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            peaks = json.load(f)
    except Exception:
        pass
    sustained = peaks.get("bf16_tflops_sustained") or 1400.0

    B = args.batch  # images per GPU per step (weak scaling: fixed per-GPU work)
    torch.manual_seed(0)
    model = Denoiser(IMG, 256, 2, D, 0, L).to(dev).eval()
    vae = AutoencoderKLDecoder().to(device=dev, dtype=torch.bfloat16).eval()
    gen = DiffusionGenerator(model, vae, dev, torch.float32)
    g = torch.Generator().manual_seed(1 + rank)
    labels_h = torch.randn(B, 768, generator=g).pin_memory()
    seeds_h = torch.randn(B, 4, IMG, IMG, generator=torch.Generator().manual_seed(11 + rank)).pin_memory()
    labels_d, seeds_d = labels_h.to(dev), seeds_h.to(dev)
    out_h = torch.empty(B, 3, 8 * IMG, 8 * IMG).pin_memory()
    last = {}  # what the latest resident step returned, as DiffusionGenerator.generate returns it

    def step_resident():
        lat = gen.generate_latents(labels_d, n_iter=N_ITER, num_imgs=B, class_guidance=GUIDANCE, img_size=IMG,
                                   sharp_f=0, bright_f=0, exponent=1, seeds=seeds_d)
        last["images"] = vae.decode(lat * 8)[0]
        last["latents"] = lat
        return last["images"]

    def step_e2e():  # public API call with host tensors; the image comes back to (pinned) host memory
        lab = labels_h.to(dev, non_blocking=True)
        sd = seeds_h.to(dev, non_blocking=True)
        lat = gen.generate_latents(lab, n_iter=N_ITER, num_imgs=B, class_guidance=GUIDANCE, img_size=IMG,
                                   sharp_f=0, bright_f=0, exponent=1, seeds=sd)
        out_h.copy_(vae.decode(lat * 8)[0], non_blocking=True)

    for _ in range(max(args.warmup, 3)):
        step_resident()
    # denoiser-only loop time of one step (device events inside the library)
    step_resident()
    torch.cuda.synchronize()
    loop_ms, launches = gen.last_stats()

    sampler = ClockSampler(local)
    sampler.start()
    vae_launches0 = vae.own_launches
    ms_total = timed(step_resident, args.steps)
    vae_launches = vae.own_launches - vae_launches0
    clocks = sampler.stop()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last)
    step_e2e()
    ms_e2e = timed(step_e2e, args.steps)

    value = world * B * args.steps / (ms_total * 1e-3)
    e2e_val = world * B * args.steps / (ms_e2e * 1e-3)

    configs = {}
    if not args.headline_only:
        configs = other_configs(args, dev, dist, world, rank, timed, vae, sustained)

    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return
    roof = time_dominant_kernels(_lib, peaks)
    flops_img = 2 * N_ITER * fwd_flops_per_sample() + AutoencoderKLDecoder.flops_per_image(IMG)
    step_flops = 2 * B * fwd_flops_per_sample()
    line = {
        "metric": "images_per_sec_256px_35step_cfg", "value": value, "unit": "images/s", "n_gpus": world,
        "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_total / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": {"workload": "100M denoiser 256px sampling: 4x32x32 latent, 35-step CFG, batch=64 per GPU + VAE decode",
                   "images_per_gpu_per_step": B, "n_iter": N_ITER, "class_guidance": GUIDANCE, "cfg_batch": 2 * B,
                   "parallelism": f"batch-sharded x{world}, no collective", "weights": "random-init",
                   "l2": "inputs larger than L2: 202 MB bf16 weights + >1 GB activations per step vs 126 MB L2",
                   "denoiser": "libtld_b200 (hand-written sm_100a, CUDA-graph step, 5 kernels per block: norm1, fused qkv projection + "
                               "attention, norm2 + folded 2-token cross-attention + norm3, fused up-projection + depthwise conv + "
                               "GELU, down-projection + residual)",
                   "vae_decode": "libtld_b200 tcgen05 implicit-GEMM conv3x3 + fused GroupNorm/SiLU/upsample kernels (bf16); parity "
                                 "UNPINNED to diffusers (third-party, absent): checked against oracle/vae_oracle.py, which is cross-checked against torchtitan's LDM AutoEncoder (same architecture) on random weights"},
        "denoiser_step_ms": loop_ms / N_ITER, "denoiser_only_images_per_s_per_gpu": B / (loop_ms * 1e-3),
        "denoiser_step_frac_of_sustained_bf16_peak": step_flops / (loop_ms / N_ITER * 1e-3) / 1e12 / sustained,
        "flops_accounting": "SURVEY.md 8d model FLOPs of the reference's formulation (24 n d^2 + ... per block); the folded "
                            "cross-attention does not execute the 2 n d^2 q-projection of each block, so executed_step_tflop is lower",
        "model_step_tflop": step_flops / 1e12,
        "executed_step_tflop": (step_flops - 2 * B * L * 2 * (IMG // 2) ** 2 * D * D) / 1e12,
        "flops_per_image": flops_img,
        "model_tflops_whole_step": flops_img * value / 1e12,
        "frac_of_sustained_bf16_peak_whole_step": flops_img * value / 1e12 / (sustained * world),
        "e2e": {"value": e2e_val, "unit": "images/s", "ms_per_step": ms_e2e / args.steps,
                "h2d_bytes_per_step": labels_h.numel() * 4 + seeds_h.numel() * 4, "d2h_bytes_per_step": out_h.numel() * 4},
        "gpu_launches": int(launches) * args.steps + int(vae_launches),
        "clocks": clocks,
        "roofline": roof,
        "configs": configs,
    }
    if world == 1 and not args.no_cpu_baseline:
        try:
            line["stock_torch_b200"] = stock_torch_b200(dev)
        except Exception as e:  # noqa: BLE001
            line["stock_torch_b200"] = {"error": f"{type(e).__name__}: {e}"[:200]}
        # the oracle port on the host cores, in a child process with a hard time limit (bounded sample)
        threads = cpu_threads()
        n = args.cpu_images
        try:
            r = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference", "--steps", "1",
                                "--warmup", "0", "--cpu-images", str(n)], capture_output=True, text=True, timeout=300)
            ref = json.loads(r.stdout.strip().splitlines()[-1])
            line["cpu_baseline"] = ref["cpu_baseline"]
        except Exception as e:  # noqa: BLE001
            line["cpu_baseline"] = {"value": None, "unit": "images/s", "cores": threads, "kind": "port",
                                    "sample": f"{n} image(s) x {N_ITER} CFG steps + VAE decode did not finish: {type(e).__name__}"}
    print(json.dumps(line))
    if dist is not None:
        dist.destroy_process_group()


def other_configs(args, dev, dist, world, rank, timed, vae, sustained) -> dict:
    """BASELINE.json configs[2], [3], [4] measured in the same run on the same N GPUs (every rank does the same per-GPU
    work; times are max over ranks, throughputs whole-job)."""
    from transformer_latent_diffusion_b200.denoiser import Denoiser
    from transformer_latent_diffusion_b200.diffusion import DiffusionGenerator
    from transformer_latent_diffusion_b200.optim import FusedAdamEMA
    from transformer_latent_diffusion_b200.train import train_step

    res = {}

    def sampling(img, batches, n_iter, reps, with_vae):
        torch.manual_seed(0)
        m = Denoiser(img, 256, 2, D, 0, L).to(dev).eval()
        gen = DiffusionGenerator(m, vae, dev, torch.float32)
        rows = []
        for b in batches:
            labels = torch.randn(b, 768, device=dev)
            seeds = torch.randn(b, 4, img, img, device=dev)

            def lat():
                return gen.generate_latents(labels, n_iter=n_iter, num_imgs=b, class_guidance=GUIDANCE, img_size=img, sharp_f=0,
                                            bright_f=0, exponent=1, seeds=seeds)

            def full():
                vae.decode(lat() * 8)

            lat()
            lat()
            ms = timed(lat, reps) / reps
            row = {"images_per_gpu": b, "cfg_batch": 2 * b, "ms_per_model_call": ms / n_iter,
                   "images_per_s_denoiser_only": world * b / (ms * 1e-3),
                   "model_tflops_per_gpu": 2 * b * n_iter * fwd_flops_per_sample(img) / (ms * 1e-3) / 1e12,
                   "frac_of_sustained_bf16_peak": 2 * b * n_iter * fwd_flops_per_sample(img) / (ms * 1e-3) / 1e12 / sustained}
            if with_vae:
                full()
                msf = timed(full, reps) / reps
                row["images_per_s_with_vae_decode"] = world * b / (msf * 1e-3)
                row["ms_per_generation_with_vae_decode"] = msf
            rows.append(row)
        del m, gen
        torch.cuda.empty_cache()
        return rows

    try:
        res["px512_b16"] = dict(sampling(64, [16], N_ITER, 3, True)[0], workload="configs[2]: 4x64x64 latent, 35-step CFG, batch 16 "
                                "per GPU, batch-sharded (no collective)", n_iter=N_ITER)
    except Exception as e:  # noqa: BLE001
        res["px512_b16"] = {"error": f"{type(e).__name__}: {e}"[:300]}
    try:
        res["px1024_sweep"] = {"workload": "configs[4]: 4x128x128 latent (4096 tokens/sample), 50-step CFG, batch per GPU swept",
                               "n_iter": 50, "rows": sampling(128, [1, 2, 4, 8, 16, 32], 50, 1, False)}
    except Exception as e:  # noqa: BLE001
        res["px1024_sweep"] = {"error": f"{type(e).__name__}: {e}"[:300]}

    def training(batch, steps, label):
        torch.manual_seed(0)
        m = Denoiser(IMG, 256, 2, D, 0, L).to(dev).train()
        if dist is not None:
            for p in m.parameters():
                dist.broadcast(p.data, src=0)
        ema = None
        if rank == 0:
            import copy

            ema = copy.deepcopy(m)
        opt = FusedAdamEMA(m, lr=3e-4, ema_model=ema, alpha=0.999)
        m.grad_views = True
        x = torch.randn(batch, 4, IMG, IMG, device=dev)
        eps = torch.randn(batch, 4, IMG, IMG, device=dev)
        sig = torch.rand(batch, 1, device=dev)
        lab = torch.randn(batch, 768, device=dev)
        xn = sig.view(-1, 1, 1, 1) * eps + (1 - sig.view(-1, 1, 1, 1)) * x

        def one():
            train_step(m, opt, x, xn, sig, lab)

        for _ in range(3):
            one()
        ms = timed(one, steps) / steps
        out = {"workload": label, "samples_per_gpu": batch, "global_batch": batch * world, "ms_per_step": ms,
               "samples_per_s": world * batch / (ms * 1e-3),
               "model_tflops_per_gpu": 3 * batch * fwd_flops_per_sample() / (ms * 1e-3) / 1e12,
               "frac_of_sustained_bf16_peak": 3 * batch * fwd_flops_per_sample() / (ms * 1e-3) / 1e12 / sustained,
               "optimizer": "FusedAdamEMA (tld_adam_ema_step), EMA on rank 0",
               "allreduce_bytes_per_step": 4 * sum(p.numel() for p in m.parameters()) if world > 1 else 0}
        if world > 1:
            # the same step without any gradient exchange: the difference is the all-reduce time the backward could not hide
            m.overlap_grad_allreduce = False
            import transformer_latent_diffusion_b200.train as T

            saved = T.allreduce_gradients
            T.allreduce_gradients = lambda model: None
            try:
                for _ in range(2):
                    one()
                ms0 = timed(one, steps) / steps
            finally:
                T.allreduce_gradients = saved
                m.overlap_grad_allreduce = True
            out["ms_per_step_without_allreduce"] = ms0
            out["allreduce_exposed_ms"] = ms - ms0
            out["collective"] = "NCCL all-reduce (AVG, fp32) of per-block gradient ranges on a side stream, overlapped with the backward"
        del m, opt, ema
        torch.cuda.empty_cache()
        return out

    try:
        res["train_step"] = training(32, 10, "configs[3]: train.main step, 100M model, bf16 operands, 32 samples per GPU (256 global "
                                     "at 8 GPUs), synthetic latents + embeddings")
    except Exception as e:  # noqa: BLE001
        res["train_step"] = {"error": f"{type(e).__name__}: {e}"[:300]}
    if world == 1:
        try:
            res["train_step_b256"] = training(256, 5, "configs[3] on ONE GPU: the whole 256-sample batch")
        except Exception as e:  # noqa: BLE001
            res["train_step_b256"] = {"error": f"{type(e).__name__}: {e}"[:300]}
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=64, help="images per GPU per step")
    ap.add_argument("--cpu-images", type=int, default=4, help="images per CPU step (bounded sample; BASELINE.md asks for B=4)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--headline-only", action="store_true", help="skip the other BASELINE configs (512 px, 1024 px sweep, training)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the images and latents of the last timed step (rank 0) as "
                                                          "DIR/<name>.npy, float32, at most 64 MB in all")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes what the b200 arm computed")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
