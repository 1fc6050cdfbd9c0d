"""bench.py -- images/sec of the Amodal-DAv2 forward pass (BASELINE.json metric) on N B200s, one process per GPU.

  python bench.py --gpus 1 --steps K --warmup W              # this repo's CUDA path
  torchrun ... bench.py --gpus N --steps K --warmup W        # N ranks, images sharded, no data-path collective
  python bench.py --impl reference --steps K --warmup W      # the reference algorithm on the host CPU cores (oracle port)

A step = one forward pass over one synthetic batch. Default workload = BASELINE.json configs[2]: ViT-L, 518x518, guide =
mask+observation, 32 images per GPU (weak scaling; with N > 1 the same JSON line also carries `strong` = the configuration
as BASELINE words it, global batch 32 sharded over the N GPUs). `value` is device-timed (CUDA events on the launch stream,
inputs resident in HBM); `e2e` goes through the public model API with pinned host buffers, H2D and D2H inside the timed
region. Outside the timed regions the same run also: checks one image of the timed output against the CPU oracle
(`parity`), times the reference algorithm with stock torch kernels on the same GPU (`gpu_eager_baseline`: fp32 without
TF32, and bf16 autocast -- the "kernel to beat" on this box) and on the host cores (`cpu_baseline`), and measures the other
BASELINE configurations (`other_configs`). Prints ONE JSON line on rank 0.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

# Algorithmic FLOPs per image (2*MAC over every GEMM / conv / QK^T / PV; SURVEY.md section 6 and 8d)
GFLOP_PER_IMAGE = {("vits", 518): 119.4, ("vitb", 518): 396.3, ("vitl", 518): 1389.6, ("vitl", 1036): 7764.3,
                   ("vitg", 518): 5771.4}
PROF_CLASSES = ["gemm_tcgen05_linear", "gemm_tcgen05_conv3x3", "attention_tcgen05", "layernorm", "channel_ln_relu",
                "upsample_bilinear", "gather", "tail_gather"]
# BASELINE.json `configs`, by (encoder, size, per-GPU batch)
BASELINE_CONFIGS = {("vits", 518, 1): "configs[0]", ("vitb", 518, 8): "configs[1]", ("vitl", 518, 32): "configs[2]",
                    ("vitl", 1036, 4): "configs[3]", ("vitg", 518, 8): "configs[4] (per-GPU share of batch 64 over 8 GPUs)"}
GT = "mask+observation"


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d["hbm_gbs"], tf_burst=d["bf16_tflops"], tf_sustained=d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                    src="measured (MEASURED_PEAKS.json)")
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sustained=1400.0, src="fallback (B200_PROFILING.md)")


class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons every 100 ms. It is started BEFORE the warm-up (NVML start-up takes up to
    a second and must not land inside the timed region) and only the samples that arrive between mark_begin() and
    mark_end() -- the timed region -- are reported."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, uuid):
        self.rows, self.proc, self.uuid = [], None, uuid
        self.t_begin, self.t_end = None, None

    def mark_begin(self):
        self.t_begin = time.time()

    def mark_end(self):
        self.t_end = time.time()

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", self.uuid, f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:  # noqa: BLE001
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:  # noqa: BLE001
            self.proc.kill()
        sm, smax, power, reasons = [], None, [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        t0 = self.t_begin or 0.0
        t1 = (self.t_end or time.time()) + 0.05
        for ts, r in self.rows:
            if ts < t0 or ts > t1:
                continue
            f = [x.strip() for x in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                smax = float(f[1])
                power.append(float(f[2]))
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": smax,
                "power_w_max": max(power) if power else None, "samples": len(sm), "reasons": sorted(reasons)}


class NvmlSampler:
    """Same report as ClockSampler, sampled in-process through NVML (pynvml) from a thread every 100 ms: three light
    queries (SM clock, power, clocks-event reasons) instead of an nvidia-smi process that re-queries the device in a
    loop."""

    def __init__(self, uuid):
        self.uuid, self.rows, self.ok = uuid, [], False
        self.t_begin, self.t_end, self._stop = None, None, threading.Event()

    def mark_begin(self):
        self.t_begin = time.time()

    def mark_end(self):
        self.t_end = time.time()

    def start(self):
        try:
            import pynvml as N
            N.nvmlInit()
            self.N = N
            self.h = N.nvmlDeviceGetHandleByUUID(self.uuid.encode() if isinstance(self.uuid, str) else self.uuid)
            self.smax = float(N.nvmlDeviceGetMaxClockInfo(self.h, N.NVML_CLOCK_SM))
            self.ok = True
            self.t = threading.Thread(target=self._run, daemon=True)
            self.t.start()
        except Exception:  # noqa: BLE001
            self.ok = False

    def _run(self):
        N = self.N
        while not self._stop.is_set():
            try:
                self.rows.append((time.time(), float(N.nvmlDeviceGetClockInfo(self.h, N.NVML_CLOCK_SM)),
                                  N.nvmlDeviceGetPowerUsage(self.h) / 1e3,
                                  int(N.nvmlDeviceGetCurrentClocksEventReasons(self.h))))
            except Exception:  # noqa: BLE001
                pass
            self._stop.wait(0.1)

    def stop(self):
        if not self.ok:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["NVML unavailable"]}
        self._stop.set()
        self.t.join(timeout=2)
        N = self.N
        bits = {"hw_slowdown": N.nvmlClocksThrottleReasonHwSlowdown,
                "hw_thermal_slowdown": N.nvmlClocksThrottleReasonHwThermalSlowdown,
                "sw_thermal_slowdown": N.nvmlClocksThrottleReasonSwThermalSlowdown,
                "sw_power_cap": N.nvmlClocksThrottleReasonSwPowerCap,
                "hw_power_brake_slowdown": getattr(N, "nvmlClocksThrottleReasonHwPowerBrakeSlowdown", 0x80),
                "sync_boost": getattr(N, "nvmlClocksThrottleReasonSyncBoost", 0x10)}
        t0 = self.t_begin or 0.0
        t1 = (self.t_end or time.time()) + 0.05
        rows = [r for r in self.rows if t0 <= r[0] <= t1]
        reasons = sorted(n for n, b in bits.items() if any(r[3] & b for r in rows))
        return {"sm_mhz": statistics.median([r[1] for r in rows]) if rows else None, "sm_max_mhz": self.smax,
                "power_w_max": max([r[2] for r in rows]) if rows else None, "samples": len(rows), "reasons": reasons,
                "how": "in-process NVML, 100 ms"}


# ------------------------------------------------------------------------------------------------ CPU / reference legs
def cpu_reference_rate(encoder, size, steps, warmup):
    """Times the oracle (CPU restatement of the reference forward) on all host cores: `steps` images, ONE image per step.
    Returns (images/s, s/image, threads, output of the last step)."""
    import torch
    from oracle import amodal_oracle as O
    from oracle import synth
    torch.set_num_threads(os.cpu_count() or 1)
    sd = synth.make_state_dict(encoder, GT, 0)
    inp = synth.make_inputs(1, size, size, 0)
    times = []
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        out = O.forward(sd, encoder, GT, inp["x"], None, inp["guide_mask"], inp["observation"])
        if i >= warmup:
            times.append(time.perf_counter() - t0)
    sec = sum(times) / len(times)
    return 1.0 / sec, sec, torch.get_num_threads(), out


def cpu_context():
    """SURVEY.md section 8d asks for the CPU model and the ViT-S 518x518 single-image time next to the baseline."""
    model = ""
    try:
        for ln in open("/proc/cpuinfo"):
            if ln.startswith("model name"):
                model = ln.split(":", 1)[1].strip()
                break
    except OSError:
        pass
    _, sec_s, _, _ = cpu_reference_rate("vits", 518, 5, 1)
    return {"cpu_model": model, "os_cpu_count": os.cpu_count(), "vits_518_b1_s_per_image": sec_s}


def run_reference(a):
    """Reference arm: the reference algorithm (oracle port; the reference is pure Python and /root/reference does not exist
    on the GPU box) on the host CPU cores. A step here is ONE image of the named architecture and resolution -- a bounded
    sample of the workload (a 32-image CPU step would take ~30 s); images/s is batch-size independent on the CPU."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    rate, sec, cores, out = cpu_reference_rate(a.encoder, a.size, a.steps, a.warmup)
    dumped = None
    if a.dump_outputs:
        import torch
        os.makedirs(a.dump_outputs, exist_ok=True)
        dumped = dump_outputs(torch, out, os.path.join(a.dump_outputs, "depth.npy"), DUMP_BYTES)
    sample = (f"{a.steps} steps x 1 image per step ({a.encoder} {a.size}x{a.size}, fp32, torch CPU, {cores} threads) after "
              f"{a.warmup} warm-up; NOT the {a.batch}-image step of the GPU arm")
    cfg = workload_config(a, a.gpus)
    cfg["reference_step"] = "1 image per step (bounded CPU sample of the same architecture and resolution)"
    line = {
        "impl": "reference", "metric": "images/sec", "value": rate, "unit": "images/s", "n_gpus": a.gpus,
        "steps": a.steps, "warmup": a.warmup, "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": cfg,
        "cpu_baseline": {"value": rate, "unit": "images/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": rate, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "dump_outputs": dumped,
    }
    print(json.dumps(line), flush=True)


def workload_config(a, world, per_gpu=None, encoder=None, size=None):
    encoder, size = encoder or a.encoder, size or a.size
    if per_gpu is None:
        per_gpu = a.batch if a.scaling == "weak" else max(a.batch // world, 1)
    in_mb = per_gpu * 5 * size * size * 4 / 1e6
    d = {"vits": 384, "vitb": 768, "vitl": 1024, "vitg": 1536}[encoder]
    x_mb = per_gpu * ((size // 14) ** 2 + 1) * d * 4 / 1e6  # fp32 residual stream alone, rewritten every block
    l2 = (f"per step {in_mb:.0f} MB of inputs and a {x_mb:.0f} MB fp32 token stream (plus GBs of bf16 activations) stream through "
          f"the 126 MB L2" if in_mb + x_mb > 126 else
          f"small-batch configuration: inputs ({in_mb:.0f} MB) and token stream ({x_mb:.0f} MB) fit the 126 MB L2 and are NOT "
          f"flushed between steps -- latency figure, not the headline metric")
    tag = BASELINE_CONFIGS.get((encoder, size, per_gpu))
    return {"workload": f"AmodalDAv2 {encoder} {size}x{size} guide=mask+observation forward, batch {per_gpu}/GPU"
                        + (f" (BASELINE.json {tag})" if tag else " (not a BASELINE.json configuration)"),
            "encoder": encoder, "height": size, "width": size, "per_gpu_batch": per_gpu,
            "global_batch": per_gpu * world, "parallelism": f"image-sharded x{world}, weights replicated, no collective",
            "cuda_graph": bool(getattr(a, "graph", False)), "l2": l2}


# ------------------------------------------------------------------------------------------------ GPU helpers
def make_model(pkg, torch, encoder, dev):
    """Random-init weights of the named architecture (no checkpoints offline). The guidance conv is zero-initialised by the
    reference (dav2.py:55-61) -- randomise it so the guide path does real work."""
    torch.manual_seed(0)
    model = pkg.AmodalDAv2(guide_type=GT, encoder=encoder, pretrained=False)
    with torch.no_grad():
        model.encoder.pretrained.patch_embed_guidance.proj.weight.normal_(std=0.02)
        model.encoder.pretrained.patch_embed_guidance.proj.bias.uniform_(-0.05, 0.05)
    return model.to(dev).eval()


def make_inputs(torch, B, H, W, dev, seed):
    g = torch.Generator(device=dev).manual_seed(seed)
    x = torch.rand(B, 3, H, W, device=dev, generator=g)
    low = torch.rand(B, 1, max(H // 37, 2), max(W // 37, 2), device=dev, generator=g)
    mask = (torch.nn.functional.interpolate(low, size=(H, W), mode="bilinear") > 0.5).float() * 2 - 1
    obs = torch.rand(B, 1, H, W, device=dev, generator=g) * 2 - 1
    return x, mask, obs


def timed_loop(torch, fn, steps, warmup, barrier, per_step=None):
    """W untimed calls, then K calls between two CUDA events on the current stream, barrier + synchronize on both sides.
    The reported time is (last event - first event) / K; `per_step` (a list) additionally receives the K step durations
    from events recorded between the steps, so that an outlier step is visible in the JSON line."""
    out = None
    for _ in range(warmup):
        out = fn()
    barrier()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(steps + 1)]
    ev[0].record()
    for i in range(steps):
        out = fn()
        ev[i + 1].record()
    barrier()
    if per_step is not None:
        per_step.extend(round(ev[i].elapsed_time(ev[i + 1]), 3) for i in range(steps))
    return ev[0].elapsed_time(ev[steps]) / steps, out


def parity_check(torch, model, x, mask, obs, out, idx=0):
    """One image of the timed output against the CPU oracle on the same weights / inputs (outside every timed region)."""
    from oracle import amodal_oracle as O
    world = int(os.environ.get("WORLD_SIZE", "1"))
    torch.set_num_threads(max(1, (os.cpu_count() or 1) // world))  # torchrun pins OMP_NUM_THREADS=1
    sd = {k: v.detach().float().cpu() for k, v in model.state_dict().items()}
    xi, mi, oi = x[idx:idx + 1].cpu(), mask[idx:idx + 1].cpu(), obs[idx:idx + 1].cpu()
    t0 = time.perf_counter()
    ref = O.forward(sd, model.encoder_name, GT, xi, None, mi, oi)
    sec = time.perf_counter() - t0
    got = out[idx:idx + 1].detach().float().cpu()
    rel = ((got - ref).abs() / ref.abs().clamp_min(1e-6)).max().item()
    absrel = O.abs_relative_difference(got.clone(), ref, mi > 0).item()
    return {"image": idx, "rel": rel, "absrel": absrel, "rel_tol": 1e-2, "absrel_tol": 1e-3,
            "ok": bool(rel <= 1e-2 and absrel <= 1e-3), "oracle_s": sec,
            "how": "max per-pixel |out-ref|/ref and AbsRel over the mask of one image of the timed batch vs oracle/amodal_oracle.py "
                   "(fp32, CPU) on the same weights and inputs"}


def gpu_eager_baseline(torch, model, x, mask, obs, steps=3, warmup=2):
    """The reference algorithm with stock torch kernels (cuBLAS / cuDNN / ATen eager, materialised softmax(QK^T)V as in
    attention.py:49-62) on the SAME GPU and the same batch: fp32 with TF32 off (the precision the reference runs in) and
    torch.autocast(bfloat16). This is the same-box 'kernel to beat' (SURVEY.md section 8d); none of this repo's kernels run here."""
    from oracle import amodal_oracle as O
    res = {"native": "torch eager: cuBLAS / cuBLASLt GEMMs, cuDNN convolutions, ATen softmax / layer_norm / interpolate",
           "torch": torch.__version__, "batch": int(x.shape[0]), "steps": steps, "warmup": warmup}
    sd = {k: v.detach().float() for k, v in model.state_dict().items()}
    tf32 = (torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32)
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    try:
        def run():
            return O.forward(sd, model.encoder_name, GT, x, None, mask, obs)
        for name, ctx in (("fp32_no_tf32", None), ("bf16_autocast", torch.autocast("cuda", dtype=torch.bfloat16))):
            try:
                def fn():
                    if ctx is None:
                        return run()
                    with ctx:
                        return run()
                ms, _ = timed_loop(torch, fn, steps, warmup, torch.cuda.synchronize)
                res[name] = {"ms_per_step": ms, "images_per_s": x.shape[0] / (ms / 1e3)}
            except Exception as e:  # noqa: BLE001  (e.g. out of memory at an unusual --batch)
                res[name] = {"error": repr(e)[:200]}
            torch.cuda.empty_cache()
    finally:
        torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = tf32
    return res


def measure_config(torch, pkg, dev, encoder, size, batch, steps, warmup, peaks, model=None, graph=True):
    """Device-timed images/s of one more BASELINE configuration (same kernels, same timing rules)."""
    own = model is None
    if own:
        model = make_model(pkg, torch, encoder, dev)
    x, mask, obs = make_inputs(torch, batch, size, size, dev, 4321)
    was = bool(getattr(model, "_graph", False))
    model.set_graph(graph)
    ms, out = timed_loop(torch, lambda: model(x, guide_rgb=None, guide_mask=mask, observation=obs), steps, max(warmup, 4),
                         torch.cuda.synchronize)
    model.set_graph(was)
    ok = bool(torch.isfinite(out).all().item())
    rate = batch / (ms / 1e3)
    gf = GFLOP_PER_IMAGE.get((encoder, size))
    r = {"workload": f"{encoder} {size}x{size} batch {batch}", "baseline_config": BASELINE_CONFIGS.get((encoder, size, batch)),
         "value": rate, "unit": "images/s", "ms_per_step": ms, "steps": steps, "warmup": warmup, "finite": ok,
         "gpu_launches_per_step": model.launch_count(), "cuda_graph": bool(graph),
         "model_tflops": rate * gf / 1e3 if gf else None,
         "frac_of_sustained_peak": rate * gf / 1e3 / peaks["tf_sustained"] if gf else None,
         "frac_of_burst_peak": rate * gf / 1e3 / peaks["tf_burst"] if gf else None}
    del x, mask, obs, out
    if own:
        del model
    torch.cuda.empty_cache()
    return r


DUMP_BYTES = 64 * 2 ** 20


def dump_outputs(torch, out, path, max_bytes):
    """Writes the depth map a caller of the timed path receives to `path` (.npy, float32) for output-by-output comparison
    of two builds. An output larger than `max_bytes` is replaced by a fixed, seeded sample of its elements (flat, in
    index order), so two runs with the same arguments write the same elements."""
    import numpy as np
    a = out.detach().float().cpu().flatten()
    cap = max_bytes // 4
    if a.numel() > cap:
        idx = torch.randperm(a.numel(), generator=torch.Generator().manual_seed(0))[:cap].sort().values
        a = a[idx]
    else:
        a = a.view(out.shape)
    np.save(path, a.numpy())
    return {"file": os.path.basename(path), "shape": list(out.shape), "dtype": "float32", "elements": a.numel(),
            "sampled": a.numel() < out.numel()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--encoder", default="vitl")
    ap.add_argument("--size", type=int, default=518)
    ap.add_argument("--batch", type=int, default=32, help="images per GPU (weak) / total (strong)")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true",
                    help="skip parity / gpu_eager_baseline / other_configs / strong (profiling runs under ncu)")
    ap.add_argument("--graph", action="store_true", help="(default) replay the forward as a CUDA graph: ada_set_graph")
    ap.add_argument("--no-graph", action="store_true",
                    help="launch the ~214 kernels of a forward one by one instead (same kernels, same results; measured "
                         "0.7 ms per step slower at batch 32 and exposed to host-side launch stalls)")
    ap.add_argument("--profile-steps", type=int, default=2)
    ap.add_argument("--detail", default="", help="write per-launch-signature timings of the profile pass to this JSON file")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="after the timed steps, write the output of the last timed step to DIR/depth.npy (float32; "
                         "depth_rank<r>.npy per rank with several GPUs; a fixed seeded sample above 64 MB in all)")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    a.warmup = max(a.warmup, 3) if a.impl == "b200" else a.warmup
    a.graph = not a.no_graph
    if a.impl == "reference":
        return run_reference(a)

    import torch
    import torch.distributed as dist
    import amodal_depth_anything_b200 as pkg
    from amodal_depth_anything_b200.shard import max_over_ranks

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl b200 needs a CUDA device; there is no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    cfg = workload_config(a, world)
    B, H, W = cfg["per_gpu_batch"], a.size, a.size
    peaks = load_peaks()

    model = make_model(pkg, torch, a.encoder, dev)
    if a.graph:
        model.set_graph(True)
    x, mask, obs = make_inputs(torch, B, H, W, dev, 1234 + rank)

    def step():
        return model(x, guide_rgb=None, guide_mask=mask, observation=obs)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    sampler = None
    if rank == 0:  # in-process NVML; the nvidia-smi loop only where pynvml is missing
        uuid = "GPU-" + str(torch.cuda.get_device_properties(dev).uuid)
        sampler = NvmlSampler(uuid)
        sampler.start()
        if not sampler.ok:
            sampler = ClockSampler(uuid)
            sampler.start()
    for _ in range(a.warmup):
        out = step()
    barrier()
    # more untimed steps until the device has been under load for ~1.5 s: on some boxes of the pool the first second of a
    # process showed single steps stalling by 20-40 ms (power management settling; `ms_steps_rank0` makes such a step visible)
    t_w = time.time()
    while time.time() - t_w < 1.5:
        out = step()
        torch.cuda.synchronize()
    barrier()
    if sampler:
        sampler.mark_begin()
    step_ms = []
    ms, out = timed_loop(torch, step, a.steps, 0, barrier, step_ms)
    if sampler:
        sampler.mark_end()
    clocks = sampler.stop() if sampler else None
    ms = max_over_ranks(ms, dev)
    launches = model.launch_count()
    assert torch.isfinite(out).all()
    dumped = None
    if a.dump_outputs:
        os.makedirs(a.dump_outputs, exist_ok=True)
        name = "depth.npy" if world == 1 else f"depth_rank{rank}.npy"
        dumped = dump_outputs(torch, out, os.path.join(a.dump_outputs, name), DUMP_BYTES // world)

    # ---- end to end through the public API: pinned host inputs -> H2D -> forward -> D2H, every step
    hx, hm, ho = x.cpu().pin_memory(), mask.cpu().pin_memory(), obs.cpu().pin_memory()
    hout = torch.empty(B, 1, H, W).pin_memory()

    from amodal_depth_anything_b200.pipeline import StreamedInference
    runner = StreamedInference(model, dev)
    houts = [hout, torch.empty_like(hout).pin_memory()]

    def e2e_run(n):
        # every step: H2D of that step's pinned inputs, forward through the public model call, D2H of its result;
        # copies of neighbouring steps overlap the kernels (copy streams), all inside the timed region
        runner.run(((hx, hm, ho) for _ in range(n)), [houts[i & 1] for i in range(n)])

    e2e_run(2)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    e2e_run(a.steps)
    e1.record()
    barrier()
    e2e_ms = max_over_ranks(e0.elapsed_time(e1) / a.steps, dev)
    h2d = (hx.numel() + hm.numel() + ho.numel()) * 4
    d2h = hout.numel() * 4
    e2e_same = bool(torch.equal(houts[(a.steps - 1) & 1], out.cpu()))  # the streamed path returns the same numbers

    # ---- strong scaling as BASELINE words configs[2]: the GLOBAL batch (default 32) sharded over the N GPUs
    strong = None
    if world > 1 and a.scaling == "weak" and not a.no_extras:
        per = max(a.batch // world, 1)
        sx, sm_, so = make_inputs(torch, per, H, W, dev, 99 + rank)
        use_graph = a.graph  # CUDA-graph replay like the headline loop (PDL is automatic below 12000 tokens)
        model.set_graph(use_graph)
        s_ms, s_out = timed_loop(torch, lambda: model(sx, guide_rgb=None, guide_mask=sm_, observation=so), a.steps,
                                 max(a.warmup, 4), barrier)
        s_ms = max_over_ranks(s_ms, dev)
        model.set_graph(a.graph)
        strong = {"scaling": "strong", "global_batch": per * world, "per_gpu_batch": per, "ms_per_step": s_ms,
                  "value": per * world / (s_ms / 1e3), "unit": "images/s", "cuda_graph": use_graph,
                  "finite": bool(torch.isfinite(s_out).all().item()),
                  "note": "BASELINE.json configs[2] as worded: batch 32 sharded at N GPUs; device-timed, max over ranks"}
        del sx, sm_, so, s_out

    # ---- per-kernel-class CUDA-event breakdown (separate pass: the events add gaps, so it is not the headline number)
    import ctypes
    from amodal_depth_anything_b200 import _lib as L
    lib = L.load()
    breakdown, roof = {}, None
    if a.profile_steps > 0:
        lib.ada_set_profile(model._handle, 1)
        for _ in range(a.profile_steps):
            step()
        if a.detail and rank == 0:
            cap = 4096
            meta, rms = (ctypes.c_int32 * (5 * cap))(), (ctypes.c_double * cap)()
            nrec = lib.ada_profile_records(model._handle, cap, meta, rms)
            agg = {}
            for i in range(max(nrec, 0)):
                c, m_, n_, k_, tag = meta[5 * i:5 * i + 5]
                key = f"{PROF_CLASSES[c]} M={m_} N={n_} K={k_} epi={tag & 15} act={(tag >> 4) & 15} bn={(tag >> 8) & 0xfff} cg={tag >> 20}"
                e = agg.setdefault(key, {"ms": 0.0, "n": 0, "flops": 2.0 * m_ * n_ * k_})
                e["ms"] += rms[i]
                e["n"] += 1
            rows = []
            for key, e in agg.items():
                avg = e["ms"] / e["n"]
                rows.append({"sig": key, "launches": e["n"] // a.profile_steps, "avg_ms": avg,
                             "ms_per_step": e["ms"] / a.profile_steps,
                             "tflops": e["flops"] / avg / 1e9 if e["flops"] else None})
            rows.sort(key=lambda r: -r["ms_per_step"])
            json.dump(rows, open(a.detail, "w"), indent=1)
        n = len(PROF_CLASSES)
        msv, fl, by = (ctypes.c_double * n)(), (ctypes.c_double * n)(), (ctypes.c_double * n)()
        ln = (ctypes.c_int32 * n)()
        L.check(lib.ada_profile_read(model._handle, n, msv, fl, by, ln))
        lib.ada_set_profile(model._handle, 0)
        tot = sum(msv) or 1.0
        for i, name in enumerate(PROF_CLASSES):
            if ln[i]:
                e = {"ms_per_step": msv[i] / a.profile_steps, "share": msv[i] / tot,
                     "launches_per_step": ln[i] // a.profile_steps}
                if fl[i]:   # tensor-bound classes: algorithmic FLOP rate against the measured bf16 peaks
                    e["tflops"] = fl[i] / msv[i] / 1e9
                    e["frac_of_sustained_peak"] = e["tflops"] / peaks["tf_sustained"]
                    e["frac_of_burst_peak"] = e["tflops"] / peaks["tf_burst"]
                else:       # HBM-bound classes: algorithmic bytes against the measured copy bandwidth
                    e["gbs"] = by[i] / msv[i] / 1e6
                    e["frac_of_hbm_peak"] = e["gbs"] / peaks["hbm"]
                breakdown[name] = e
        # dominant kernel = gemm_tcgen05_kernel (linear + implicit-conv launches of the same kernel)
        g_ms, g_fl, g_n = msv[0] + msv[1], fl[0] + fl[1], ln[0] + ln[1]
        ach = g_fl / g_ms / 1e9
        traffic, traffic_note = None, None
        try:  # DRAM bytes per launch: STATIC, from the committed `ncu --set full` capture of this command (ncu cannot run inside bench.py)
            for tf in ("r02_ncu_traffic.json", "r01_ncu_traffic.json"):
                tp = os.path.join(ROOT, "profiles", tf)
                if os.path.exists(tp) and (a.encoder, a.size, a.batch) == ("vitl", 518, 32):
                    tj = json.load(open(tp))
                    traffic = tj["mean_dram_bytes_per_launch"]
                    traffic_note = (f"STATIC value read from profiles/{tf} (ncu --set full capture of this workload, not measured in "
                                    f"this run): mean over the 4 linear GEMMs of one encoder block, algorithmic "
                                    f"{tj['mean_algorithmic_bytes_per_launch']} B/launch; {tj['source']}")
                    break
        except Exception:  # noqa: BLE001
            pass
        roof = {"kernel": "gemm_tcgen05_kernel", "bound": "tensor", "achieved": ach, "peak": peaks["tf_sustained"],
                "unit": "TFLOP/s", "frac": ach / peaks["tf_sustained"], "frac_of_burst": ach / peaks["tf_burst"],
                "peak_burst": peaks["tf_burst"], "traffic": traffic, "traffic_note": traffic_note,
                "peak_source": peaks["src"] + ": `peak`/`frac` use the sustained bf16 figure (kernel timed inside a long step); "
                                              "`frac_of_burst` uses the burst figure",
                "flops_per_launch": g_fl / g_n, "avg_launch_ms": g_ms / g_n, "launches_per_step": g_n // a.profile_steps,
                "share_of_step": g_ms / tot}

    extras = rank == 0 and world == 1 and not a.no_extras
    parity = eager = None
    other = []
    if rank == 0 and not a.no_extras:
        parity = parity_check(torch, model, x, mask, obs, out)
    if extras:
        eager = gpu_eager_baseline(torch, model, x, mask, obs)
        if (a.encoder, a.size, a.batch) == ("vitl", 518, 32):
            # the other BASELINE.json configurations, same kernels and timing rules (ViT-L 1036^2 reuses the loaded weights)
            other.append(measure_config(torch, pkg, dev, "vitl", 1036, 4, 5, 3, peaks, model=model))
    cpu_base = None
    if rank == 0 and world == 1 and not a.no_cpu_baseline:
        rate, sec, cores, _ = cpu_reference_rate(a.encoder, a.size, 3, 1)
        cpu_base = {"context": cpu_context(), "value": rate, "unit": "images/s", "cores": cores, "kind": "port",
                    "sample": f"3 images of the same workload ({a.encoder} {a.size}x{a.size}, ONE image per step, fp32 torch CPU "
                              f"oracle) after 1 warm-up, {sec:.2f} s/image"}
    workspace_gb = model.workspace_bytes() / 2 ** 30
    if extras and (a.encoder, a.size, a.batch) == ("vitl", 518, 32):
        del model, runner
        torch.cuda.empty_cache()
        other.append(measure_config(torch, pkg, dev, "vitb", 518, 8, 10, 3, peaks))
        other.append(measure_config(torch, pkg, dev, "vitg", 518, 8, 5, 3, peaks))

    if rank == 0:
        gb = cfg["global_batch"]
        value = gb / (ms / 1e3)
        gf = GFLOP_PER_IMAGE.get((a.encoder, a.size))
        line = {
            "metric": "images/sec", "value": value, "unit": "images/s", "n_gpus": world, "steps": a.steps,
            "warmup": a.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": a.scaling, "vs_baseline": None,
            "dtype": "bf16", "data": "synthetic", "config": cfg, "ms_steps_rank0": step_ms,
            "e2e": {"value": gb / (e2e_ms / 1e3), "unit": "images/s", "h2d_bytes_per_step": h2d * world,
                    "d2h_bytes_per_step": d2h * world, "ms_per_step": e2e_ms, "same_result_as_device_timed_call": e2e_same,
                    "how": "StreamedInference: pinned host -> H2D -> AmodalDAv2.forward -> D2H per step, copies on side streams"},
            "gpu_launches": launches * a.steps,
            "clocks": clocks,
            "roofline": roof,
            "parity": parity,
            "model_tflops_per_gpu": value * gf / 1e3 / world if gf else None,
            "model_frac_of_peak": (value * gf / 1e3 / world) / peaks["tf_sustained"] if gf else None,
            "model_frac_of_burst_peak": (value * gf / 1e3 / world) / peaks["tf_burst"] if gf else None,
            "breakdown": breakdown,
            "strong": strong,
            "gpu_eager_baseline": eager,
            "other_configs": other or None,
            "cpu_baseline": cpu_base,
            "workspace_gb": workspace_gb,
            "dump_outputs": dumped,
        }
        if eager:
            for k in ("fp32_no_tf32", "bf16_autocast"):
                if eager.get(k, {}).get("images_per_s"):
                    eager[k]["speedup_of_this_repo"] = value / eager[k]["images_per_s"]
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
