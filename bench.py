#!/usr/bin/env python
"""Benchmark of the UNet denoise hot path (see DESIGN.md "Measurement").

    python bench.py --gpus N --steps K --warmup W            # B200-native arm
    python bench.py --impl reference --gpus N ...            # reference CPU path (oracle port)

One "step" = one UNet forward over this rank's batch of synthetic latents (default: the CFG
pair, B = 2, of SD-1.5 at 512x512 -> 4x64x64 latents, fp16, CUDA graph on = BASELINE.json
configs[1]).  `value` = latents pushed through one UNet forward per second, whole job
(N GPUs x B x K / max-over-ranks device time).  Prints ONE JSON line on rank 0.

Extra keys in the same line (the headline numbers stay the ones above):
  gpu_library_baseline  the SAME UNet run by the GPU libraries the reference dispatches to
                        (cuDNN NHWC convs, cuBLASLt linears, SDPA flash attention; fp16, captured in
                        a torch.cuda.CUDAGraph, same inputs / steps) -- a same-box GPU comparator,
                        method of /root/reference/examples/optimize_stable_diffusion_pipeline.py:127-151
  config4               BASELINE configs[4] per-rank shard: 8 latents per GPU at 4x64x64 and 4x128x128
  config2_sdxl          BASELINE configs[2] (N = 1 only): SDXL-base, 8 latents 4x128x128, bf16
  first_call_s          weight packing + plan build + warm-up + graph capture of the headline config
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "stable-fast_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

import torch  # noqa: E402

METRIC = "unet_latent_steps_per_s"
UNIT = "latents through one UNet forward per second (SD-1.5 20-step ms/img = 2*20*1000/value)"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--model", default="sd15", choices=["sd15", "sdxl", "tiny"])
    ap.add_argument("--batch", type=int, default=2, help="latents per GPU per step")
    ap.add_argument("--global-batch", type=int, default=0,
                    help="strong scaling: total latents sharded over the GPUs (BASELINE configs[4])")
    ap.add_argument("--size", type=int, default=64, help="latent height = width")
    ap.add_argument("--dtype", default="fp16", choices=["fp16", "bf16"])
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-roofline", action="store_true")
    ap.add_argument("--dump-ops", default="", help="write per-op CUDA-event timings (JSON lines)")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="write the UNet output of the last timed step as DIR/sample.npy (float32; "
                         "sample_rank<r>.npy per rank when --gpus > 1)")
    ap.add_argument("--no-extras", action="store_true",
                    help="skip gpu_library_baseline / config4 / config2_sdxl (profiling runs)")
    return ap.parse_args()


# ------------------------------------------------------------------------------------------------
class ClockSampler:
    """Samples SM clocks / throttle reasons with nvidia-smi while the timed region runs."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                 "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:  # noqa: BLE001
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        rows = [r for r in self.rows if len(r) >= 6 and r[0].isdigit()]
        if not rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        sm = sorted(int(r[0]) for r in rows)
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(r[2 + i] == "Active" for r in rows)]
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": int(rows[0][1]), "reasons": reasons,
                "samples": len(rows)}


def load_peaks():
    """(burst TFLOP/s, sustained TFLOP/s, HBM GB/s, source).  A kernel family timed alone as a short
    CUDA graph at full clocks is compared with the BURST figure; `frac_sustained` is kept beside it."""
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        burst = d.get("bf16_tflops", d.get("bf16_tflops_sustained"))
        return burst, d.get("bf16_tflops_sustained", burst), d.get("hbm_gbs"), "measured (MEASURED_PEAKS.json)"
    return 1590.0, 1400.0, 6650.0, "fallback (B200_PROFILING.md)"


def usable_cores():
    """Host threads this process may really use: affinity mask, capped by a cgroup CPU quota."""
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            txt = open(path).read().split()
            if path.endswith("cpu.max"):
                quota, period = txt[0], float(txt[1])
            else:
                quota, period = txt[0], float(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if quota not in ("max", "-1"):
                n = max(1, min(n, int(float(quota) / period)))
            break
        except (OSError, ValueError, IndexError):
            continue
    return n


def workload_name(args, batch, ctx_dim):
    return (f"{args.model} UNet2DConditionModel forward, {batch} latent(s) 4x{args.size}x{args.size} "
            f"per step per GPU (B=2 = the CFG pair of one {args.size * 8}^2 image), text 77x{ctx_dim}, "
            "random-init weights")


def job_config(args, batch, world, total_latents, ctx_dim, weight_gb):
    """Identical for the B200 arm and the reference arm (the driver compares the two dicts)."""
    return {"workload": workload_name(args, batch, ctx_dim),
            "cuda_graph": not args.no_graph,
            "global_batch": total_latents, "parallelism": f"dp{world}",
            "l2": f"inputs larger than L2: the {weight_gb:.2f} GB 16-bit weight set streams from HBM every step"}


def weight_gigabytes(model):
    from sfast_b200.synthetic import CONFIGS
    from sfast_b200.unet_spec import param_shapes, spec_from_config
    spec = spec_from_config(CONFIGS[model])
    return sum(int(torch.Size(sh).numel()) for sh in param_shapes(spec).values()) * 2 / 1e9


def cross_dim(args):
    from sfast_b200.synthetic import CONFIGS
    return CONFIGS[args.model]["cross_attention_dim"]


# ------------------------------------------------------------------------------------------------
def cpu_reference_run(args, steps, warmup):
    """The reference's CPU path for this workload = plain eager PyTorch fp32 (every sfast op falls
    back to aten on CPU: /root/reference/src/sfast/csrc/operators/cublas/cublas_gemm.cpp:705-710,
    /root/reference/src/sfast/triton/torch_ops.py:116-126), run on the oracle restatement of the
    UNet because diffusers is not installable here.  One step = the same batch as the GPU arm."""
    from oracle import unet_oracle as uo
    cores = usable_cores()
    torch.set_num_threads(cores)
    cfg = {"sd15": uo.sd15_config, "sdxl": uo.sdxl_config, "tiny": uo.tiny_config}[args.model]()
    m = uo.build_unet(cfg, seed=0)
    g = torch.Generator().manual_seed(0)
    nb = args.batch
    s = torch.randn(nb, 4, args.size, args.size, generator=g)
    e = torch.randn(nb, 77, cfg.cross_attention_dim, generator=g)
    kw = {}
    if cfg.addition_embed_type == "text_time":
        kw["added_cond_kwargs"] = {"text_embeds": torch.randn(nb, 1280, generator=g),
                                   "time_ids": torch.tensor([[1024., 1024, 0, 0, 1024, 1024]] * nb)}
    times = []
    with torch.no_grad():
        for _ in range(warmup):
            m(s, torch.tensor(999.0), e, **kw)
        for i in range(steps):
            t0 = time.perf_counter()
            out = m(s, torch.tensor(999.0 - 50 * i), e, **kw)
            times.append(time.perf_counter() - t0)
    times.sort()
    med = times[len(times) // 2]
    return {"value": nb / med, "ms_per_step": med * 1e3, "steps": steps, "warmup": warmup, "cores": cores,
            "sample_out": out.sample,
            "sample": f"{steps} timed fp32 eager forward(s) of {nb} {args.model} latent(s) "
                      f"4x{args.size}x{args.size} (the same batch as one GPU rank) after {warmup} warm-up(s), "
                      f"{cores} threads, median"}


def run_reference(args, rank):
    """Reference arm: the reference's CPU path on the box's host cores.  It is ONE host whatever
    --gpus says: the value is the host's latents/s and does not grow with N (a per-N ratio against
    it compares N GPUs with the same one host)."""
    if rank != 0:
        return
    world = args.gpus
    r = cpu_reference_run(args, args.steps, args.warmup)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"sample": r["sample_out"]})
    total = args.global_batch if args.global_batch else args.batch * world
    line = {
        "impl": "reference", "metric": METRIC, "value": r["value"], "unit": UNIT,
        "n_gpus": args.gpus, "steps": r["steps"], "warmup": r["warmup"], "ms_per_step": r["ms_per_step"],
        "higher_is_better": True, "scaling": "strong" if args.global_batch else "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": job_config(args, args.batch, world, total, cross_dim(args), weight_gigabytes(args.model)),
        "arm": "fp32 CPU eager (the reference's CPU path = aten fallbacks) on the oracle port; one host "
               "process, independent of --gpus",
        "cpu_baseline": {"value": r["value"], "unit": UNIT, "cores": r["cores"], "kind": "port",
                         "sample": r["sample"]},
        "e2e": {"value": r["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
def run_b200(args, rank, world, local):
    from sfast.compilers.diffusion_pipeline_compiler import CompilationConfig, compile_unet
    from sfast_b200 import _lib, dist as sdist
    from sfast_b200.synthetic import CONFIGS, SyntheticUNet
    from sfast_b200.unet_spec import param_shapes, random_state_dict, spec_from_config

    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    dtype = torch.float16 if args.dtype == "fp16" else torch.bfloat16
    cfg = CONFIGS[args.model]
    spec = spec_from_config(cfg)
    if args.global_batch:
        lo, hi = sdist.shard_batch(args.global_batch, rank, world)
        batch, scaling = hi - lo, "strong"
    else:
        batch, scaling = args.batch, "weak"
    # weights: rank 0 draws them, ONE broadcast over NCCL/NVLink, zero collectives afterwards
    sd0 = random_state_dict(spec, seed=0, dtype=dtype, device=dev) if rank == 0 else None
    sd = sdist.broadcast_state_dict(param_shapes(spec), sd0, dtype, dev) if world > 1 else sd0
    unet = SyntheticUNet(cfg, state_dict=sd, dtype=dtype, device=dev)
    cc = CompilationConfig.Default()
    cc.enable_cuda_graph = not args.no_graph
    unet = compile_unet(unet, cc)
    compiled = unet.forward._compiled

    ctx_dim = spec.cross_attention_dim
    g = torch.Generator().manual_seed(1234 + rank)
    n_var = 4  # a few distinct host inputs so steps are not identical
    host_s = [torch.randn(batch, 4, args.size, args.size, generator=g).to(dtype).pin_memory()
              for _ in range(n_var)]
    host_e = [torch.randn(batch, 77, ctx_dim, generator=g).to(dtype).pin_memory()
              for _ in range(n_var)]
    host_out = torch.empty(batch, 4, args.size, args.size, dtype=dtype).pin_memory()
    kw = {}
    if spec.addition_embed_type == "text_time":
        kw["added_cond_kwargs"] = {
            "text_embeds": torch.randn(batch, 1280, generator=g).to(dev, dtype),
            "time_ids": torch.tensor([[1024., 1024, 0, 0, 1024, 1024]] * batch, device=dev)}
    dev_s = [t.to(dev) for t in host_s]
    dev_e = [t.to(dev) for t in host_e]
    tsteps = [torch.tensor(float(999 - 50 * (i % 20)), device=dev) for i in range(20)]

    lib = _lib.lib()
    n0 = lib.sfb_launch_count()
    unet(dev_s[0], tsteps[0], dev_e[0], **kw)  # builds plan (+ graph): eager warm-up + capture
    torch.cuda.synchronize()
    gp = next(iter(compiled._cached.values()))
    plan = gp.plan
    # first call = eager warm-up pass + (graph capture | eager step): two passes over the plan
    launches_per_step = (lib.sfb_launch_count() - n0) // 2

    def barrier():
        if world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, warmup):
        for i in range(warmup):
            fn(i)
        barrier()
        sampler = ClockSampler(local)
        if rank == 0:
            sampler.start()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(steps):
            fn(i)
        e1.record()
        barrier()
        clocks = sampler.stop() if rank == 0 else None
        ms = sdist.max_over_ranks(e0.elapsed_time(e1), dev)
        return ms, clocks

    # --- device-resident arm: inputs already in HBM; per step = static-buffer copies + graph replay
    last = {}

    def step_dev(i):
        last["sample"] = unet(dev_s[i % n_var], tsteps[i % 20], dev_e[i % n_var], **kw).sample

    ms_dev, clocks = timed(step_dev, args.steps, max(args.warmup, 3))
    if args.dump_outputs:
        # copied before the next arm reuses the graph's static output buffer
        outputs = {"sample" if world == 1 else f"sample_rank{rank}": last["sample"].float().cpu()}

    # --- end-to-end arm: pinned host inputs -> H2D -> public API call -> D2H of the result
    def step_e2e(i):
        s = host_s[i % n_var].to(dev, non_blocking=True)
        e = host_e[i % n_var].to(dev, non_blocking=True)
        out = unet(s, tsteps[i % 20], e, **kw).sample
        host_out.copy_(out, non_blocking=True)

    ms_e2e, _ = timed(step_e2e, args.steps, max(args.warmup, 3))
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, outputs, budget=(64 << 20) // world)

    weight_gb = sum(int(torch.Size(sh).numel()) for sh in param_shapes(spec).values()) * 2 / 1e9
    flops_per_step = plan.flops()
    total_latents = batch * world if not args.global_batch else args.global_batch
    value = total_latents * args.steps / (ms_dev / 1e3)
    e2e_value = total_latents * args.steps / (ms_e2e / 1e3)
    h2d = host_s[0].numel() * 2 + host_e[0].numel() * 2
    d2h = host_out.numel() * 2

    roofline = None
    if not args.no_roofline:
        roofline = measure_roofline(plan, lib, args.dump_ops, f"{args.model}-b{batch}-s{args.size}")
    first_call_s = compiled.first_call_s
    # ---- extra measurements (every rank runs them so that ranks stay in step; rank 0 reports)
    extras = {}
    if not args.no_extras and args.model == "sd15" and args.size == 64 and not args.global_batch:
        extras["config4"] = {
            "what": "BASELINE configs[4] per-rank shard: 8 latents per GPU (bs 64 over 8 GPUs), SD-1.5 fp16, "
                    f"CUDA graph, at this N = {world}",
            "latent_64": shard_bench(unet, compiled, 8, 64, dtype, dev, world, sdist),
            "latent_128": shard_bench(unet, compiled, 8, 128, dtype, dev, world, sdist),
        }
        if world == 1:
            extras["gpu_library_baseline"] = gpu_library_baseline(args, sd, batch, dtype, dev, dev_s, dev_e, tsteps)
    del unet, compiled, plan, gp
    if not args.no_extras and args.model == "sd15" and world == 1 and not args.global_batch:
        extras["config2_sdxl"] = sdxl_bench(dev)
        extras["config3_svd"] = svd_bench(dev)
        extras["vae_decode"] = vae_bench(dev)
        extras["text_encoder"] = text_encoder_bench(dev)
    cpu_base = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        r = cpu_reference_run(args, steps=2, warmup=1)
        cpu_base = {"value": r["value"], "unit": UNIT, "cores": r["cores"], "kind": "port",
                    "sample": r["sample"]}
    if rank != 0:
        return
    ms_step = ms_dev / args.steps
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": ms_step, "higher_is_better": True,
        "scaling": scaling, "vs_baseline": None, "dtype": args.dtype, "data": "synthetic",
        "config": job_config(args, batch, world, total_latents, ctx_dim, weight_gb),
        "sd15_20step_unet_ms_per_img": 20 * ms_step if (args.model == "sd15" and batch == 2) else None,
        "algorithmic_tflop_per_step": flops_per_step / 1e12,
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d,
                "d2h_bytes_per_step": d2h, "ms_per_step": ms_e2e / args.steps},
        "gpu_launches": int(launches_per_step * args.steps),
        "kernel_launches_per_step": int(launches_per_step),
        "first_call_s": first_call_s,
        "clocks": clocks,
        "roofline": roofline,
        "cpu_baseline": cpu_base,
        **extras,
    }
    print(json.dumps(line), flush=True)


def dump_outputs(dirname, arrays, budget=64 << 20):
    """Write each tensor as DIR/<name>.npy in float32, all together within `budget` bytes.  A tensor
    over its share is replaced by a fixed seeded sample: its flat elements at the indices stored
    beside it as DIR/<name>_index.npy (float64), so that two builds still compare element for element."""
    import numpy as np
    os.makedirs(dirname, exist_ok=True)
    share = budget // len(arrays)
    for name, t in arrays.items():
        a = t.numpy().astype(np.float32)
        if a.nbytes > share:
            n = (share - 4096) // 12  # a float32 value and a float64 index per kept element, headers
            idx = np.sort(np.random.default_rng(0).choice(a.size, n, replace=False))
            np.save(os.path.join(dirname, f"{name}_index.npy"), idx.astype(np.float64))
            a = a.reshape(-1)[idx]
        np.save(os.path.join(dirname, f"{name}.npy"), a)


def family_rates(plan):
    """Steady-state rate of each kernel family of a plan: the family's launches (same buffers, same
    order) captured alone in a CUDA graph and replayed -- CUDA events, launch gaps included."""
    def time_graph(ops, iters=5):
        st = torch.cuda.current_stream()
        for op in ops:
            op.launch(st.cuda_stream)
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            cs = torch.cuda.current_stream().cuda_stream
            for op in ops:
                op.launch(cs)
        for _ in range(2):
            g.replay()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(iters):
            g.replay()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / iters

    burst, sustained, hbm, src = load_peaks()
    fams = {}
    for op in plan.all_ops():
        fams.setdefault(getattr(op.fn, "__name__", "other"), []).append(op)
    out = {"peak_source": src}
    for name, key in (("sfb_gemm", "gemm"), ("sfb_attention", "attention")):
        ops_ = fams.get(name)
        if ops_:
            ms = time_graph(ops_)
            tf = sum(o.flops for o in ops_) / (ms / 1e3) / 1e12
            out[key] = {"launches": len(ops_), "ms": ms, "tflops": tf, "frac_of_burst_peak": tf / burst,
                        "frac_of_sustained_peak": tf / sustained}
    gn = [o for n, l in fams.items() if n.startswith("sfb_group_norm") for o in l]
    if gn:
        ms = time_graph(gn)
        gbs = sum(o.bytes for o in gn) / (ms / 1e3) / 1e9
        out["group_norm"] = {"launches": len(gn), "ms": ms, "gbs": gbs, "frac_of_hbm_peak": gbs / hbm}
    return out


def shard_bench(unet, compiled, batch, size, dtype, dev, world, sdist, steps=10, warmup=3):
    """`batch` latents of 4 x size x size per GPU through the already compiled SD-1.5 UNet (new plan +
    CUDA graph for the new shape, same packed weights): whole-job latents/s + per-family rates."""
    g = torch.Generator().manual_seed(77)
    s = torch.randn(batch, 4, size, size, generator=g).to(dev, dtype)
    e = torch.randn(batch, 77, compiled.spec.cross_attention_dim, generator=g).to(dev, dtype)
    ts = [torch.tensor(float(999 - 50 * i), device=dev) for i in range(steps)]
    for i in range(warmup):
        unet(s, ts[i % steps], e)
    if world > 1:
        torch.distributed.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(steps):
        unet(s, ts[i], e)
    e1.record()
    if world > 1:
        torch.distributed.barrier()
    torch.cuda.synchronize()
    ms = sdist.max_over_ranks(e0.elapsed_time(e1), dev) / steps
    key = next(k for k in compiled._cached if k[0] == batch and k[1] == size)
    plan = compiled._cached[key].plan
    out = {"latents_per_gpu": batch, "latent": f"4x{size}x{size}", "ms_per_step": ms,
           "latents_per_s": batch * world / (ms / 1e3), "steps": steps, "warmup": warmup,
           "algorithmic_tflop_per_step_per_gpu": plan.flops() / 1e12,
           "step_tflops_per_gpu": plan.flops() / (ms / 1e3) / 1e12, **family_rates(plan)}
    del compiled._cached[key]
    torch.cuda.empty_cache()
    return out


def sdxl_bench(dev, steps=5, warmup=3):
    """BASELINE configs[2]: SDXL-base UNet, 8 latents (bs 4 x CFG) of 4x128x128, bf16, CUDA graph."""
    from sfast.compilers.diffusion_pipeline_compiler import CompilationConfig, compile_unet
    from sfast_b200.synthetic import CONFIGS, SyntheticUNet
    torch.cuda.empty_cache()
    dtype, B = torch.bfloat16, 8
    unet = SyntheticUNet(CONFIGS["sdxl"], seed=0, dtype=dtype, device=dev)
    cc = CompilationConfig.Default()
    cc.enable_cuda_graph = True
    unet = compile_unet(unet, cc)
    g = torch.Generator().manual_seed(5)
    s = torch.randn(B, 4, 128, 128, generator=g).to(dev, dtype)
    e = torch.randn(B, 77, 2048, generator=g).to(dev, dtype)
    kw = {"added_cond_kwargs": {"text_embeds": torch.randn(B, 1280, generator=g).to(dev, dtype),
                                "time_ids": torch.tensor([[1024., 1024, 0, 0, 1024, 1024]] * B, device=dev)}}
    ts = [torch.tensor(float(999 - 30 * i), device=dev) for i in range(steps)]
    for i in range(warmup):
        unet(s, ts[i % steps], e, **kw)
    torch.cuda.synchronize()
    sampler = ClockSampler(dev.index or 0)
    sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(steps):
        unet(s, ts[i], e, **kw)
    e1.record()
    torch.cuda.synchronize()
    clocks = sampler.stop()
    ms = e0.elapsed_time(e1) / steps
    compiled = unet.forward._compiled
    plan = next(iter(compiled._cached.values())).plan
    out = {"what": "BASELINE configs[2]: SDXL-base UNet forward, 8 latents 4x128x128 (bs 4 x CFG), bf16, "
                   "CUDA graph, 1 GPU, random-init weights",
           "ms_per_step": ms, "latents_per_s": B / (ms / 1e3), "sdxl_30step_unet_s_per_batch4": 30 * ms / 1e3,
           "steps": steps, "warmup": warmup, "first_call_s": compiled.first_call_s,
           "algorithmic_tflop_per_step": plan.flops() / 1e12,
           "step_tflops": plan.flops() / (ms / 1e3) / 1e12, "clocks": clocks, **family_rates(plan)}
    del unet, compiled, plan
    torch.cuda.empty_cache()
    return out


def svd_bench(dev, steps=3, warmup=2):
    """BASELINE configs[3]: StableVideoDiffusion-XT UNet (UNetSpatioTemporalConditionModel), 576 x 1024,
    25 frames, CFG pair of videos (B = 2), fp16, CUDA graph; s/clip = 25 denoising steps of the UNet."""
    from sfast.compilers.diffusion_pipeline_compiler import CompilationConfig, compile_unet
    from sfast_b200.synthetic import CONFIGS, SyntheticUNet
    try:
        torch.cuda.empty_cache()
        dtype, B, F_ = torch.float16, 2, 25
        unet = SyntheticUNet(CONFIGS["svd"], seed=0, dtype=dtype, device=dev)
        cc = CompilationConfig.Default()
        cc.enable_cuda_graph = True
        unet = compile_unet(unet, cc)
        g = torch.Generator().manual_seed(6)
        s = torch.randn(B, F_, 8, 72, 128, generator=g).to(dev, dtype)
        e = torch.randn(B, 1, 1024, generator=g).to(dev, dtype)
        tid = torch.tensor([[6.0, 127.0, 0.02]] * B, device=dev, dtype=dtype)
        ts = [torch.tensor(1.6 - 0.06 * i, device=dev) for i in range(max(steps, warmup))]
        for i in range(warmup):
            unet(s, ts[i], e, tid)
        torch.cuda.synchronize()
        sampler = ClockSampler(dev.index or 0)
        sampler.start()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(steps):
            unet(s, ts[i], e, tid)
        e1.record()
        torch.cuda.synchronize()
        clocks = sampler.stop()
        ms = e0.elapsed_time(e1) / steps
        compiled = unet.forward._compiled
        plan = next(iter(compiled._cached.values())).plan
        out = {"what": "BASELINE configs[3]: SVD-XT UNet forward, 2 videos (CFG pair) x 25 frames of 8x72x128 "
                       "latents (576x1024), fp16, CUDA graph, 1 GPU, random-init weights",
               "ms_per_step": ms, "svd_xt_25step_unet_s_per_clip": 25 * ms / 1e3, "steps": steps, "warmup": warmup,
               "first_call_s": compiled.first_call_s, "kernel_launches_per_step": len(plan.all_ops()),
               "algorithmic_tflop_per_step": plan.flops() / 1e12, "step_tflops": plan.flops() / (ms / 1e3) / 1e12,
               "clocks": clocks, **family_rates(plan)}
        del unet, compiled, plan
        torch.cuda.empty_cache()
        return out
    except Exception as exc:  # noqa: BLE001
        torch.cuda.empty_cache()
        return {"unavailable": repr(exc)[:300]}


def vae_bench(dev, steps=10, warmup=3):
    """SD VAE decode (compile_vae): 4x64x64 latent -> 3x512x512 image, fp16, CUDA graph."""
    from sfast.compilers.diffusion_pipeline_compiler import CompilationConfig, compile_vae
    from sfast_b200.synthetic import SyntheticVAE
    try:
        vae = SyntheticVAE(seed=0, dtype=torch.float16, device=dev)
        cc = CompilationConfig.Default()
        cc.enable_cuda_graph = True
        vae = compile_vae(vae, cc)
        z = torch.randn(1, 4, 64, 64, generator=torch.Generator().manual_seed(2)).to(dev, torch.float16)
        for _ in range(warmup):
            vae.decode(z)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            vae.decode(z)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / steps
        plan = next(iter(vae.decode._compiled._cached.values())).plan
        out = {"what": "SD-1.5 VAE decode, 1 latent 4x64x64 -> 3x512x512, fp16, CUDA graph", "ms_per_image": ms,
               "algorithmic_tflop": plan.flops() / 1e12, "tflops": plan.flops() / (ms / 1e3) / 1e12,
               "steps": steps, "warmup": warmup}
        del vae, plan
        torch.cuda.empty_cache()
        return out
    except Exception as exc:  # noqa: BLE001
        torch.cuda.empty_cache()
        return {"unavailable": repr(exc)[:300]}


def text_encoder_bench(dev, steps=20, warmup=3):
    """CLIP ViT-L/14 text encoder (the SD-1.5 / SDXL `text_encoder`): 2 prompts x 77 tokens, fp16, through
    `compile_text_encoder` on transformers' own CLIPTextModel (random init) -- and the same module run
    eagerly (library kernels) on the same GPU beside it.  Host ids -> device copy inside the timed call."""
    try:
        import copy
        import transformers
        from sfast.compilers.diffusion_pipeline_compiler import CompilationConfig, compile_text_encoder
        cfg = transformers.CLIPTextConfig(vocab_size=49408, hidden_size=768, intermediate_size=3072,
                                          num_hidden_layers=12, num_attention_heads=12, max_position_embeddings=77,
                                          hidden_act="quick_gelu", eos_token_id=2, projection_dim=768)
        torch.manual_seed(0)
        eager = transformers.CLIPTextModel(cfg).eval().to(dev, torch.float16)
        fast = copy.deepcopy(eager)
        cc = CompilationConfig.Default()
        cc.enable_cuda_graph = True
        fast = compile_text_encoder(fast, cc)
        ids = torch.randint(0, 49407, (2, 77), generator=torch.Generator().manual_seed(1)).pin_memory()

        def timed(m):
            with torch.no_grad():
                for _ in range(warmup):
                    m(ids.to(dev, non_blocking=True))
                torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(steps):
                    out = m(ids.to(dev, non_blocking=True))[0]
                e1.record()
                torch.cuda.synchronize()
            return e0.elapsed_time(e1) / steps, out

        ms_fast, o_fast = timed(fast)
        ms_eager, o_eager = timed(eager)
        plan = next(iter(fast.forward._cached.values())).plan
        out = {"what": "CLIP ViT-L/14 text encoder, 2 x 77 tokens, fp16, CUDA graph (transformers CLIPTextModel, random init)",
               "ms_per_call": ms_fast, "eager_library_ms_per_call": ms_eager, "speedup_vs_eager": ms_eager / ms_fast,
               "kernel_launches": len(plan.all_ops()), "algorithmic_gflop": plan.flops() / 1e9,
               "max_abs_diff_vs_eager_fp16": float((o_fast.float() - o_eager.float()).abs().max()),
               "steps": steps, "warmup": warmup}
        del fast, eager, plan
        torch.cuda.empty_cache()
        return out
    except Exception as exc:  # noqa: BLE001
        torch.cuda.empty_cache()
        return {"unavailable": repr(exc)[:300]}


def gpu_library_baseline(args, sd, batch, dtype, dev, dev_s, dev_e, tsteps):
    """Same-box GPU comparator: the SAME UNet (same random weights, same synthetic inputs) executed
    by the GPU libraries the reference's fused operators dispatch to -- cuDNN NHWC convolutions
    (/root/reference/src/sfast/csrc/operators/cudnn/cudnn_convolution_impl.cc), cuBLASLt linears
    (csrc/operators/cublas/CUDABlas.cc) and a flash SDPA kernel (the reference leaves
    aten::scaled_dot_product_attention untouched when xformers is off) -- fp16, channels_last,
    cudnn.benchmark, whole step captured in a torch.cuda.CUDAGraph; timing method of
    /root/reference/examples/optimize_stable_diffusion_pipeline.py:127-151.  The module tree is the
    oracle restatement of diffusers' UNet (diffusers itself is not installable offline); NOT the
    reference's own Triton / CUTLASS fusions, which do not build against this torch."""
    from oracle import unet_oracle as uo
    try:
        cfg = {"sd15": uo.sd15_config, "sdxl": uo.sdxl_config, "tiny": uo.tiny_config}[args.model]()
        with torch.device("meta"):
            m = uo.UNet2DConditionModel(cfg)
        m = m.to_empty(device=dev).to(dtype)
        m.load_state_dict({k: v.to(dtype) for k, v in sd.items()})
        m = m.eval().to(memory_format=torch.channels_last)
        torch.backends.cudnn.benchmark = True
        s0 = dev_s[0].clone().contiguous(memory_format=torch.channels_last)
        e0_, t0 = dev_e[0].clone(), tsteps[0].clone()
        with torch.no_grad():
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                for _ in range(3):
                    m(s0, t0, e0_)
            torch.cuda.current_stream().wait_stream(side)
            torch.cuda.synchronize()
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                out = m(s0, t0, e0_).sample

            def step(i):
                s0.copy_(dev_s[i % len(dev_s)])
                e0_.copy_(dev_e[i % len(dev_e)])
                t0.copy_(tsteps[i % 20])
                graph.replay()
                return out.clone()

            for i in range(max(args.warmup, 3)):
                step(i)
            torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for i in range(args.steps):
                step(i)
            b.record()
            torch.cuda.synchronize()
        ms = a.elapsed_time(b) / args.steps
        res = {"value": batch / (ms / 1e3), "unit": UNIT, "ms_per_step": ms, "steps": args.steps,
               "warmup": max(args.warmup, 3),
               "what": "oracle restatement of the UNet in fp16 channels_last on this GPU: cuDNN convs, "
                       "cuBLASLt linears, SDPA attention, aten GroupNorm/LayerNorm, torch.cuda.CUDAGraph, "
                       f"cudnn.benchmark on; torch {torch.__version__}"}
        del m, graph, out
        torch.cuda.empty_cache()
        return res
    except Exception as exc:  # noqa: BLE001 -- a comparator must never take the bench line down
        torch.cuda.empty_cache()
        return {"unavailable": repr(exc)[:300]}


def ncu_traffic(prefix, workload=None):
    """DRAM bytes per launch of the kernel family, from the committed ncu launch list of this same
    command (profiles/rNN_ncu_launch_summary.json, made by tests/summarize_ncu.py; ncu flushes the
    caches before every kernel, so this is cold-cache traffic)."""
    import glob
    files = sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_ncu_launch_summary*.json")))
    if not files:
        return {"traffic": None}
    # the newest committed launch list of THIS workload (one file per workload: ..._summary[_b8].json)
    d, src = None, None
    for f in reversed(files):
        cand = json.load(open(f))
        if workload is None or cand.get("workload") == workload:
            d, src = cand, f
            break
    if d is None:
        return {"traffic": None, "traffic_note": f"no ncu launch list committed for {workload}"}
    files = [src]
    n = b = 0
    for name, f in d.get("families", {}).items():
        if name.startswith(prefix) and "dram_bytes_per_launch" in f:
            n += f["launches"]
            b += f["dram_bytes_per_launch"] * f["launches"]
    if not n:
        return {"traffic": None}
    return {"traffic": b / n, "traffic_unit": "DRAM bytes per launch (read + write, ncu, cold caches)",
            "traffic_source": os.path.relpath(files[-1], ROOT)}


def measure_roofline(plan, lib, dump_path="", workload=None):
    """Per-op CUDA-event timing of one eager pass over the plan (after the timed region).  The
    dominant kernel is the tcgen05 GEMM / implicit-GEMM conv; its roofline is the tensor pipe."""
    stream = torch.cuda.current_stream()
    for _ in range(2):
        plan.run()
    torch.cuda.synchronize()
    evs = []
    for op in plan.all_ops():
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream)
        op.launch(stream.cuda_stream)
        b.record(stream)
        evs.append((op, a, b))
    torch.cuda.synchronize()
    if dump_path:
        with open(dump_path, "w") as f:
            for op, a, b in evs:
                extra = {}
                if getattr(op.fn, "__name__", "") == "sfb_gemm":
                    p = op.keep[0]
                    extra = {"M": p.M, "N": p.N, "K": p.K, "splits": p.splits, "conv": p.a_mode,
                             "epi": p.epi}
                f.write(json.dumps({"op": op.name, "fn": getattr(op.fn, "__name__", "?"),
                                    "us": a.elapsed_time(b) * 1e3, "flops": op.flops,
                                    "bytes": op.bytes, **extra}) + "\n")
    # steady-state cost of the dominant kernel family: all of the step's sfb_gemm launches (same
    # buffers, same order) captured in a CUDA graph and replayed, timed with CUDA events
    gemm_ops = [op for op, _, _ in evs if getattr(op.fn, "__name__", "") == "sfb_gemm"]
    gg = torch.cuda.CUDAGraph()
    with torch.cuda.graph(gg):
        cs = torch.cuda.current_stream().cuda_stream
        for op in gemm_ops:
            op.launch(cs)
    for _ in range(3):
        gg.replay()
    torch.cuda.synchronize()
    g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    g0.record()
    for _ in range(10):
        gg.replay()
    g1.record()
    torch.cuda.synchronize()
    gemm_graph_ms = g0.elapsed_time(g1) / 10
    fam = {}
    for op, a, b in evs:
        key = getattr(op.fn, "__name__", None) or str(op.name)
        d = fam.setdefault(key, {"ms": 0.0, "flops": 0, "bytes": 0, "n": 0})
        d["ms"] += a.elapsed_time(b)
        d["flops"] += op.flops
        d["bytes"] += op.bytes
        d["n"] += 1
    total_ms = sum(d["ms"] for d in fam.values())
    peak_tf, peak_sust, peak_bw, src = load_peaks()
    g = fam.get("sfb_gemm", {"ms": 1e-9, "flops": 0, "n": 1, "bytes": 0})
    achieved = g["flops"] / (gemm_graph_ms / 1e3) / 1e12
    shares = {k: round(v["ms"] / total_ms, 4) for k, v in sorted(fam.items(), key=lambda kv: -kv[1]["ms"])}
    # every GEMM launch against ITS OWN roofline: max(FLOPs / tensor peak, operand bytes / HBM peak) --
    # the family mixes tensor-bound convolutions with projections whose arithmetic intensity is below
    # the ridge (K <= 640: ~100 FLOP/B) and weight-bandwidth-bound low-resolution layers
    by = {"tensor": [0, 0.0, 0.0], "hbm": [0, 0.0, 0.0]}
    for op, a, b in evs:
        if getattr(op.fn, "__name__", "") != "sfb_gemm":
            continue
        t_t, t_m = op.flops / (peak_tf * 1e12) * 1e6, op.bytes / (peak_bw * 1e9) * 1e6
        k = "tensor" if t_t >= t_m else "hbm"
        by[k][0] += 1
        by[k][1] += max(t_t, t_m)
        by[k][2] += a.elapsed_time(b) * 1e3
    by_launch = {k: {"launches": v[0], "roofline_us": round(v[1], 1), "measured_us_eager_events": round(v[2], 1),
                     "frac": round(v[1] / v[2], 4) if v[2] else None} for k, v in by.items()}
    tot_b, tot_m = sum(v[1] for v in by.values()), sum(v[2] for v in by.values())
    by_launch["all"] = {"roofline_us": round(tot_b, 1), "measured_us_eager_events": round(tot_m, 1),
                        "frac": round(tot_b / tot_m, 4) if tot_m else None}
    att = fam.get("sfb_attention")
    extra = {"by_launch_own_roofline": by_launch}
    if att:
        extra["attention_tflops"] = att["flops"] / (att["ms"] / 1e3) / 1e12
    gn = fam.get("sfb_group_norm_apply")
    if gn:
        extra["group_norm_apply_gbs"] = gn["bytes"] / (gn["ms"] / 1e3) / 1e9
    return {"bound": "tensor", "kernel": "gemm_tc_kernel (tcgen05 GEMM / implicit-GEMM 3x3 conv, all instances)",
            "achieved": achieved, "peak": peak_tf, "unit": "TFLOP/s", "frac": achieved / peak_tf,
            "frac_of_sustained_peak": achieved / peak_sust,
            "peak_source": f"{src}: bf16_tflops (burst -- the family is timed alone as a short CUDA graph)",
            "launches_per_step": g["n"], "avg_launch_us": gemm_graph_ms * 1e3 / max(g["n"], 1),
            "timing": "all sfb_gemm launches of one step replayed as a CUDA graph, CUDA events, 10 replays",
            "avg_launch_us_eager_events": g["ms"] * 1e3 / max(g["n"], 1),
            "flop_per_step": g["flops"], **ncu_traffic("gemm_tc_kernel", workload),
            "eager_step_ms": total_ms, "time_share_by_entry_point": shares, **extra}


def main():
    args = parse()
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank)
        return
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: the B200 arm needs a CUDA device (no CPU fallback); "
                         "use --impl reference for the CPU baseline")
    if world > 1:
        from sfast_b200 import dist as sdist
        sdist.init_from_env("nccl")
    run_b200(args, rank, world, local)
    if world > 1:
        torch.distributed.barrier()
        torch.distributed.destroy_process_group()


if __name__ == "__main__":
    main()
