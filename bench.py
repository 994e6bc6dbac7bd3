#!/usr/bin/env python
"""bench.py -- frames/s of the AdaNeRF hot path (BASELINE.json metric: frames/sec at 800x800 and rays/sec).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload NAME] [--single-process]
                    [--dump-outputs DIR]

A "step" is one pass of the whole hot path (rays -> sampling MLP -> threshold / compaction -> posenc -> shading MLP ->
composite) over one frame of synthetic input: procedurally generated pinhole rays from the view-cell centre, random-init
networks (seed 0, the reference's own initialisers) or the reference's shipped trained Pavillon networks (no datasets /
checkpoints offline).

  value : frames/s with every input already resident in HBM (camera pose only; rays generated on the device), timed with
          CUDA events on the launching stream, max over ranks.
  e2e   : the same metric from HOST buffers to HOST buffers: ray directions start in (page-locked) host memory, the RGB
          frame ends there; at N > 1 the NCCL gather of the tiles and the D2H copy of the gathered frame are inside.
  N > 1 : default workload: weak scaling -- rank r renders rows [800 r, 800 (r+1)) of an 800 x 800N frame (640 000 rays per
          GPU), one NCCL gather of the RGB tiles to rank 0 per frame, left in flight under the next frame (two frames in flight);
          value = 800x800-frame equivalents per second over all ranks.  `--workload 1600x1600_thr0.2_K8` (BASELINE config
          4): STRONG scaling -- the 1600 x 1600 frame is fixed, rank r renders rows [1600 r / N, 1600 (r+1) / N).
  --single-process : N GPUs driven by ONE process through the multi-GPU C ABI (include/adanerf_b200_multi.h:
          ncclCommInitAll, grouped send / recv gather) instead of one torchrun rank per GPU.
  --impl reference : the reference's CPU path (the oracle port of TrainConfig.inference, torch CPU, all host threads); every
          step is a bounded ray sample of the same frame.
  --dump-outputs DIR : after the timed steps, the RGB frame of the last timed step -- what the caller of the timed path
          receives: the frame at N = 1, the gathered frame on the first GPU at N > 1 -- as DIR/rgb.npy, float32 [rays, 3].
          The inputs are a function of the arguments only, so two builds can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True      # the benchmark only reads the tree, which may be read-only

WORKLOADS = {
    # BASELINE.json configs[1]: 800x800, thr 0.2, K = 8 (~8 samples/ray with random-init nets: every ray saturates at K)
    "800x800_thr0.2_K8": dict(W=800, H=800, thr=0.2, K=8, weights="rand", scaling="weak"),
    # configs[2]: 800x800, dense 128 samples/ray
    "800x800_dense_K128": dict(W=800, H=800, thr=0.0, K=128, weights="rand", scaling="weak"),
    # ragged synthetic variant (shaped sampling net: 1..8 samples per ray)
    "800x800_thr0.2_K8_shaped": dict(W=800, H=800, thr=0.2, K=8, weights="shaped", scaling="weak"),
    # configs[3]: one 1600x1600 frame row-tiled over the GPUs (strong scaling)
    "1600x1600_thr0.2_K8": dict(W=1600, H=1600, thr=0.2, K=8, weights="rand", scaling="strong"),
}
# NDC / LLFF variant (configs/fine_training_ndc.ini: 30-feature sampling net, linear depths, ndc_rays in stage 3), K = 16
WORKLOADS["800x800_ndc_thr0.15_K16"] = dict(W=800, H=800, thr=0.15, K=16, weights="ndc", scaling="weak")
# configs[4]: threshold sweep on the reference's shipped trained Pavillon networks (ragged at every threshold)
for _k in (8, 16):
    for _t in (0.05, 0.1, 0.2, 0.3, 0.5):
        WORKLOADS[f"800x800_pav_thr{_t}_K{_k}"] = dict(W=800, H=800, thr=_t, K=_k, weights="pavillon", scaling="weak")
FLOP_PER_SAMPLE_MLP1 = 1186816.0   # SURVEY.md 8(d): 2 * 593 408 MAC, unpadded
FLOP_PER_RAY_MLP0 = 898048.0
SHADING_KERNEL = "mlp_sh_kernel"
DUMP_BYTES = 64 << 20
PAVILLON_NPZ = os.path.join(ROOT, "tests", "golden", "weights_pavillon.npz")


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm_gbs=d.get("hbm_gbs", 6650.0), tflops=d.get("bf16_tflops", 1590.0), tflops_sustained=d.get("bf16_tflops_sustained", 1400.0),
                    source="MEASURED_PEAKS.json (bf16_tflops: burst -- the kernel sits in a ~7 ms step inside a <0.5 s run; "
                           "bf16_tflops_sustained for reference)")
    return dict(hbm_gbs=6650.0, tflops=1590.0, tflops_sustained=1400.0, source="fallback (B200_PROFILING.md)")


def ncu_summary():
    for tag in ("r2", "r1"):
        p = os.path.join(ROOT, "profiles", f"ncu_{tag}_summary.json")
        if os.path.exists(p):
            try:
                return json.load(open(p)), tag
            except Exception:
                pass
    return {}, None


def ncu_traffic(kernel):
    """DRAM bytes per launch of `kernel` from the committed ncu --set full summary (None when absent)."""
    table, tag = ncu_summary()
    try:
        key = kernel if kernel in table else next(k for k in table if k.startswith(kernel))
        return int(table[key]["dram_rd"] + table[key]["dram_wr"]), tag
    except Exception:
        return None, tag


def stage_rooflines(stage_ms, rays, samples, thr, peaks, n_feat0=90):
    """Per stage: algorithmic work (SURVEY.md 8d) / measured stage time of the profiled chunk, against the measured peak.
    `impl` = the bytes this implementation moves by construction (packed bf16 hi / lo tiles instead of fp32 rows), where it
    differs from the 8(d) figure."""
    r, m = float(rays), float(samples)
    hbm = peaks["hbm_gbs"]
    out = {}

    def add(name, ms, work, unit, peak, bound, impl=None):
        if ms > 0:
            ach = work / (ms * 1e-3) / (1e9 if unit == "GB/s" else 1e12)
            out[name] = dict(bound=bound, achieved=ach, peak=peak, unit=unit, frac=ach / peak)
            if impl is not None:
                out[name]["impl_bytes_frac"] = impl / (ms * 1e-3) / 1e9 / peak
    add("stage0_features", stage_ms[0], r * (12 + 4 * n_feat0 + 24), "GB/s", hbm, "hbm", impl=r * (12 + 512 + 24))   # 8(d): dirs in, [N,F0] fp32 + ray o/d out
    add("mlp0", stage_ms[1], r * (FLOP_PER_RAY_MLP0 - 2.0 * 256 * (90 - n_feat0)), "TFLOP/s", peaks["tflops"], "tensor")   # algorithmic flops (x3 MMAs issued for the split)
    if thr > 0:
        add("stage2_sample", stage_ms[2], r * (512 + 8) + m * 16, "GB/s", hbm, "hbm")
    add("stage3_posenc", stage_ms[3], m * (8 + 192) + r * 24, "GB/s", hbm, "hbm", impl=m * (8 + 256) + r * 24)   # 8(d) bf16 figure: 96 x 2 B
    add("mlp1", stage_ms[4], m * FLOP_PER_SAMPLE_MLP1, "TFLOP/s", peaks["tflops"], "tensor")
    add("stage5_composite", stage_ms[5], m * 20 + r * 20, "GB/s", hbm, "hbm")
    return out


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index=0):
        self.samples, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.samples.append(line.strip())

    def stop(self):
        if not self.proc:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["nvidia-smi unavailable"])
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for s in self.samples:
            f = [x.strip() for x in s.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        sm.sort()
        return dict(sm_mhz=sm[len(sm) // 2] if sm else None, sm_max_mhz=max(mx) if mx else None,
                    samples=len(sm), reasons=sorted(reasons))


def workload_config(name, cfg, n_gpus):
    """The `config` object: a function of (workload, number of GPUs) only, so that both arms print the same one."""
    W, H = cfg["W"], cfg["H"]
    strong = cfg["scaling"] == "strong"
    Hn = H if strong else H * n_gpus
    par = "single GPU" if n_gpus == 1 else f"row-bands x{n_gpus} + 1 NCCL gather of RGB tiles to the first GPU per frame (two frames in flight)"
    return dict(workload=name, frame=f"{W}x{Hn}", rays_per_gpu_per_step=int(W * Hn // n_gpus), thr=cfg["thr"], K=cfg["K"], weights=cfg["weights"],
                scaling=cfg["scaling"], parallelism=par,
                l2="per-frame working set (packed features + activations I/O, >1 GB) exceeds the 126 MB L2; no explicit flush",
                mlp0="bf16x3 split precision (fp32-class)", mlp1="bf16 operands, fp32 accumulate")


def dump_outputs(out_dir, arrays):
    """name -> array as <out_dir>/<name>.npy in float32.  An array larger than its share of DUMP_BYTES keeps every s-th
    row only (the smallest s that fits), the same rows on every run."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        a = np.asarray(a, dtype=np.float32)
        stride = -(-a.nbytes // (DUMP_BYTES // len(arrays)))
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a[::stride]))


# ------------------------------------------------------------------------------------------------- CPU reference arm
class CpuReference:
    """Oracle port of the reference CPU path, set up ONCE: weights, the frame's ray directions, the thread count that is
    fastest for these 256-wide GEMMs on this host.  sample(budget_s) renders consecutive chunks of 8192 rays
    (inferenceChunkSize, configs/*.ini:31) of the frame, continuing where the previous call stopped, until ~budget_s passed."""

    def __init__(self, cfg, threads=None):
        import torch
        from oracle import adanerf_oracle as orc
        self.torch, self.orc, self.cfg = torch, orc, cfg
        W, H = cfg["W"], cfg["H"]
        self.n_frame = W * H
        if cfg["weights"] == "pavillon":
            from adanerf_b200 import synthetic
            self.scene = orc.SCENE_PAVILLON
            self.sd0, self.sd1 = synthetic.load_weights_npz(PAVILLON_NPZ)
        elif cfg["weights"] == "ndc":
            self.scene = orc.SCENE_PAVILLON_NDC
            self.sd0, self.sd1 = orc.make_weights("ndc", seed=0)
        else:
            self.scene = orc.SCENE_BARBERSHOP
            self.sd0, self.sd1 = orc.make_weights(cfg["weights"], seed=0)
        self.dirs = torch.from_numpy(orc.generate_ray_directions(W, H, self.scene["fov"]).reshape(-1, 3)).float()
        self.pose = torch.tensor(self.scene["view_cell_center"], dtype=torch.float32)
        self.rot = torch.eye(3)
        self.chunk = 8192 if cfg["K"] <= 16 else 1024
        # consecutive chunks walk the frame in ray order and wrap around: the timed steps together render whole frames
        self.starts = list(range(0, self.n_frame - self.chunk + 1, self.chunk))
        if self.starts[-1] + self.chunk < self.n_frame:
            self.starts.append(self.n_frame - self.chunk)
        self.cursor = -1
        if threads is None:
            # oneMKL on many-core hosts is fastest well below the core count for these 256-wide GEMMs: probe a few thread
            # counts on a quarter chunk once and keep the best ("all the host threads it can use")
            ncpu = os.cpu_count() or 8
            best, threads = None, None
            q = max(256, self.chunk // 4)
            for c in sorted({c for c in (8, 16, 32, 64, ncpu) if c <= ncpu}):
                torch.set_num_threads(c)
                self._render(0, q)
                t = time.perf_counter()
                self._render(q, q)
                t = time.perf_counter() - t
                if best is None or t < best:
                    best, threads = t, c
        torch.set_num_threads(threads)
        self.threads = torch.get_num_threads()
        self._render(self.starts[0], self.chunk)   # warm-up chunk (the first call is ~10x slower)

    def _render(self, start, n):
        return self.orc.render_rays(self.pose, self.rot, self.dirs[start:start + n], self.sd0, self.sd1, self.scene, self.cfg["thr"], self.cfg["K"])

    def sample(self, budget_s):
        rays, t0 = 0, time.perf_counter()
        while True:
            self.cursor = (self.cursor + 1) % len(self.starts)
            self._render(self.starts[self.cursor], self.chunk)
            rays += self.chunk
            el = time.perf_counter() - t0
            if el >= budget_s:
                break
        return dict(rays=rays, seconds=el, rays_per_s=rays / el, frames_per_s=rays / el / self.n_frame, cores=self.threads,
                    sample=f"{rays} rays ({rays // self.chunk} consecutive chunks of {self.chunk} of the {self.cfg['W']}x{self.cfg['H']} frame) "
                           f"in {el:.1f} s, torch {self.torch.__version__} CPU fp32, {self.threads} threads")


def run_reference(args, cfg, name):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    ref = CpuReference(cfg)
    n_frame = cfg["W"] * cfg["H"]
    # every step is a bounded sample of the frame, sized so that the whole run takes ~2.5 minutes
    per_step = max(2.0, min(30.0, 150.0 / max(1, args.steps + args.warmup)))
    for _ in range(args.warmup):
        ref.sample(per_step)
    rays, secs, last = 0, 0.0, None
    for _ in range(args.steps):
        last = ref.sample(per_step)
        rays += last["rays"]
        secs += last["seconds"]
    fps = rays / secs / n_frame
    sample = (f"{args.steps} steps of ~{per_step:.1f} s walking the frame in ray order: {rays} rays in {secs:.1f} s = {rays / n_frame:.2f} full frames; per step: "
              + last["sample"])
    line = dict(impl="reference", metric=f"frames_per_sec_{cfg['W']}x{cfg['H']}", value=fps, unit="frames/s", n_gpus=args.gpus,
                steps=args.steps, warmup=args.warmup, ms_per_step=1000.0 * secs / args.steps, higher_is_better=True, scaling=cfg["scaling"],
                vs_baseline=None, dtype="f32", data="synthetic",
                config=workload_config(name, cfg, args.gpus),
                rays_per_sec=rays / secs, frames_rendered=rays / n_frame, step_is="a bounded ray sample of the frame (value = rays/s of the sample / rays per frame)",
                cpu_baseline=dict(value=fps, unit="frames/s", cores=last["cores"], kind="port", sample=sample),
                e2e=dict(value=fps, unit="frames/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0))
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------------------ our arm
def make_renderer_inputs(cfg, torch, Renderer, synthetic, device, W, H):
    if cfg["weights"] == "pavillon":
        scene = synthetic.SCENE_PAVILLON
        sd0, sd1 = synthetic.load_weights_npz(PAVILLON_NPZ)
        r = Renderer(scene, device=device, sampling_net=sd0, shading_net=sd1)
    elif cfg["weights"] == "ndc":
        scene = synthetic.SCENE_PAVILLON_NDC
        sd0, sd1 = synthetic.make_weights("ndc", seed=0)
        r = Renderer(scene, device=device, sampling_net=sd0, shading_net=sd1)
    else:
        scene = synthetic.SCENE_BARBERSHOP
        r = Renderer(scene, device=device)
        pose = torch.tensor(scene["view_cell_center"], dtype=torch.float32)

        def probe_logits(sd0):   # W-shaped recipe: raw sampling-net outputs on every 157th ray of an 800x800 grid
            r.set_weights(0, sd0)
            x0, _, _ = r.stage0(pose, torch.eye(3), r.generate_ray_directions(800, 800)[::157].contiguous())
            return r.mlp0(x0)

        sd0, sd1 = synthetic.make_weights(cfg["weights"], seed=0, logits_fn=probe_logits)
        r.set_weights(0, sd0)
        r.set_weights(1, sd1)
    return r, scene, sd0, sd1


def run_ours(args, cfg, name):
    import numpy as np
    import torch
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world == 1 and args.gpus > 1:
        raise SystemExit("launch with torchrun for --gpus > 1 (one process per GPU), or pass --single-process")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    import __graft_entry__ as ge
    ge.build()
    from adanerf_b200 import Renderer, synthetic
    from adanerf_b200.tiling import row_bands
    W, H, thr, K = cfg["W"], cfg["H"], cfg["thr"], cfg["K"]
    strong = cfg["scaling"] == "strong"
    r, scene, _, _ = make_renderer_inputs(cfg, torch, Renderer, synthetic, local, W, H)
    pose = torch.tensor(scene["view_cell_center"], dtype=torch.float32)
    rot = torch.eye(3)
    if strong:      # the frame is fixed: this rank's row band of it
        Hn = H
        row0, rows = row_bands(H, world)[rank]
        if any(b[1] != rows for b in row_bands(H, world)):
            raise SystemExit("strong-scaling workload needs H divisible by the number of GPUs")
    else:           # weak: an H x N-high frame, one H-row band per rank
        Hn, row0, rows = H * world, H * rank, H
    n_rays = rows * W
    bands = [torch.empty((n_rays, 3), dtype=torch.float32, device="cuda") for _ in range(2)]
    frames = [torch.empty((world * n_rays, 3), dtype=torch.float32, device="cuda") for _ in range(2)] if world > 1 else None
    pending = [None, None]
    # the gathered frame as per-rank tile views (dist.gather's gather_list); A/B modes: profiles/r2/gather_ab/ (8 GPUs, weak
    # scaling: no collective 6.62 ms, gather to rank 0 6.70, all-gather 6.80 whether left in flight or not -- NCCL's kernel and the
    # persistent MLP kernels do not share SMs)
    tiles = [list(f.view(world, n_rays, 3).unbind(0)) for f in frames] if world > 1 else None
    gather_mode = os.environ.get("ADN_BENCH_GATHER", "root")

    def step(f):
        """One frame: render this rank's band, then ONE NCCL gather of the RGB tiles to rank 0, left in flight while the next
        frame's band is rendered into the other buffer."""
        k = f & 1
        if pending[k] is not None:
            pending[k].wait()            # the buffers of frame f - 2
            pending[k] = None
        r.render_camera(pose, rot, W, Hn, thr, K, row0=row0, rows=rows, out=bands[k])
        if world > 1:
            if gather_mode == "root":        # default: ONE NCCL gather of the tiles to rank 0 (grouped send / recv), left in flight
                pending[k] = dist.gather(bands[k], tiles[k] if rank == 0 else None, dst=0, async_op=True)
            elif gather_mode == "overlap":   # A/B: all-gather (every rank receives the frame), left in flight
                pending[k] = dist.all_gather_into_tensor(frames[k], bands[k], async_op=True)
            elif gather_mode == "sync":      # A/B: all-gather serialised behind the composite (round 1)
                dist.all_gather_into_tensor(frames[k], bands[k])
            # "none": no collective at all (the spread between the GPUs of the box)

    def drain():
        for k in range(2):
            if pending[k] is not None:
                pending[k].wait()
                pending[k] = None

    for f in range(max(args.warmup, 3)):
        step(f)
    drain()
    torch.cuda.synchronize()
    l0 = r.stats()["kernel_launches"]
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for f in range(args.steps):
        step(f)
    drain()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    last = (args.steps - 1) & 1          # buffers of the last timed frame, overwritten by the e2e and profiled renders below
    last_rgb = None
    if args.dump_outputs and rank == 0:
        last_rgb = (frames[last] if world > 1 and gather_mode != "none" else bands[last]).cpu().numpy()
    ms_by_rank = [ms / args.steps]
    if world > 1:
        t = torch.tensor([ms], device="cuda")
        every = torch.empty(world, device="cuda")
        dist.all_gather_into_tensor(every, t)
        ms_by_rank = [float(x) / args.steps for x in every.tolist()]   # the spread between the GPUs of the box (power caps differ)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
        dist.barrier()
    clocks = sampler.stop() if rank == 0 else None
    st = r.stats()
    launches = st["kernel_launches"] - l0
    m_samples = st["n_samples"]
    ms_per_step = ms / args.steps
    frames_per_step = 1.0 if strong else float(world)       # strong: one fixed frame per step; weak: `world` 800x800 frames
    value = frames_per_step * 1000.0 / ms_per_step
    rays_per_sec = world * n_rays * 1000.0 / ms_per_step

    # ---- end to end: host ray directions -> host RGB frame (H2D, render, NCCL gather, D2H inside the timed region)
    dirs_host = np.ascontiguousarray(r.generate_ray_directions(W, Hn, row0=row0, rows=rows).cpu().numpy())   # this rank's band
    if world == 1:
        rgb_host = np.empty((n_rays, 3), dtype=np.float32)
        r.register_host_buffer(dirs_host)       # caller-owned, reused every frame: DMA in place
        r.register_host_buffer(rgb_host)

        def e2e_step():
            r.render_rays_host(pose, rot, dirs_host, thr, K, want_nsamples=False, out=rgb_host)
        result = rgb_host
        h2d, d2h, api = dirs_host.nbytes + 48, n_rays * 12, "adn_render_rays_host"
    else:
        dirs_pin = torch.from_numpy(dirs_host).pin_memory()
        dirs_dev = torch.empty((n_rays, 3), dtype=torch.float32, device="cuda")
        frame_pin = torch.empty((world * n_rays, 3), dtype=torch.float32).pin_memory() if rank == 0 else None

        def e2e_step():
            dirs_dev.copy_(dirs_pin, non_blocking=True)
            r.render_rays(pose, rot, dirs_dev, thr, K, want_nsamples=False, out=bands[0])
            dist.gather(bands[0], tiles[0] if rank == 0 else None, dst=0)
            if rank == 0:
                frame_pin.copy_(frames[0], non_blocking=True)
            torch.cuda.synchronize()
        result = frame_pin.numpy() if rank == 0 else None
        h2d, d2h, api = dirs_host.nbytes + 48, (world * n_rays * 12 if rank == 0 else 0), \
            "render_rays (H2D of the band's dirs) + NCCL gather to rank 0 + D2H of the gathered frame"
    for _ in range(3):
        e2e_step()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        e2e_step()
    e2e_s = time.perf_counter() - t0
    if world > 1:
        t = torch.tensor([e2e_s], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_s = float(t.item())
    e2e_value = frames_per_step * args.steps / e2e_s
    finite = bool(np.isfinite(result).all()) if result is not None else True

    # ---- per-stage device times (CUDA events around each stage inside the context) for the roofline.  The context profiles the
    # FIRST chunk of a call (~8 Mi samples of scratch per chunk, whole rows): render exactly that chunk so that the sample count
    # the statistics report is the profiled one.
    chunk_rays = max(8192, (8 << 20) // K)
    chunk_rays = ((chunk_rays + 127) // 128) * 128
    if chunk_rays % W:
        chunk_rays = (chunk_rays // W + 1) * W
    prof_rows = min(rows, chunk_rays // W)
    r.set_option("profile", 1)
    stage_ms = np.zeros(6)
    n_prof = 5
    for _ in range(n_prof):
        r.render_camera(pose, rot, W, Hn, thr, K, row0=row0, rows=prof_rows, out=bands[0][:prof_rows * W])
        pst = r.stats()
        stage_ms += np.array(pst["ms_stage"])
    stage_ms /= n_prof
    prof_rays, prof_samples = prof_rows * W, int(pst["n_samples"])
    r.set_option("profile", 0)

    if rank == 0:
        peaks = measured_peaks()
        mlp1_flop = FLOP_PER_SAMPLE_MLP1 * prof_samples
        achieved = mlp1_flop / (stage_ms[4] * 1e-3) / 1e12 if stage_ms[4] > 0 else 0.0
        traffic, tag = ncu_traffic(SHADING_KERNEL)
        if args.cpu_seconds > 0:
            cpu = CpuReference(cfg).sample(args.cpu_seconds)
        else:
            cpu = dict(frames_per_s=None, cores=0, sample="skipped (--cpu-seconds 0)")
        line = dict(
            metric=f"frames_per_sec_{W}x{H}", value=value, unit="frames/s", n_gpus=world, steps=args.steps,
            warmup=max(args.warmup, 3), ms_per_step=ms_per_step, higher_is_better=True, scaling=cfg["scaling"], vs_baseline=None,
            dtype="bf16", data="synthetic",
            config=workload_config(name, cfg, world), samples_profiled_chunk=int(prof_samples), gather_mode=gather_mode if world > 1 else None,
            rays_per_sec=rays_per_sec, samples_per_ray=float(prof_samples) / prof_rays,
            e2e=dict(value=e2e_value, unit="frames/s", h2d_bytes_per_step=int(h2d), d2h_bytes_per_step=int(d2h), api=api, finite=finite),
            gpu_launches=int(launches),
            ms_per_step_by_rank=[round(x, 3) for x in ms_by_rank],
            clocks=clocks,
            stage_ms=dict(zip(["stage0_features", "mlp0", "stage2_sample", "stage3_posenc", "mlp1", "stage5_composite"],
                              [round(float(x), 4) for x in stage_ms])),
            roofline=dict(kernel=f"{SHADING_KERNEL} (shading MLP, first chunk of the frame: {prof_rays} rays, {prof_samples} samples)", bound="tensor", achieved=achieved,
                          peak=peaks["tflops"], unit="TFLOP/s", frac=achieved / peaks["tflops"],
                          frac_of_sustained=achieved / peaks["tflops_sustained"], traffic=traffic,
                          traffic_unit=f"bytes of DRAM read+write per launch (profiles/ncu_{tag}_summary.json, ncu --set full)",
                          peak_source=peaks["source"]),
            roofline_stages=stage_rooflines(stage_ms, prof_rays, prof_samples, thr, peaks, n_feat0=30 if cfg["weights"] == "ndc" else 90),
            cpu_baseline=dict(value=cpu["frames_per_s"], unit="frames/s", cores=cpu["cores"], kind="port", sample=cpu["sample"]),
        )
        print(json.dumps(line))
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, dict(rgb=last_rgb))
    r.close()
    if world > 1:
        dist.destroy_process_group()


def run_single_process(args, cfg, name):
    """N GPUs, ONE process: the multi-GPU C ABI (row bands, ncclCommInitAll, grouped send / recv gather on device 0, two
    frames in flight).  value: device-resident; e2e: the gathered frame copied to host memory every frame."""
    import numpy as np
    import torch
    import __graft_entry__ as ge
    ge.build()
    from adanerf_b200 import synthetic
    from adanerf_b200.multi import MultiRenderer
    W, H, thr, K = cfg["W"], cfg["H"], cfg["thr"], cfg["K"]
    G = args.gpus
    strong = cfg["scaling"] == "strong"
    Hn = H if strong else H * G
    if cfg["weights"] == "pavillon":
        scene = synthetic.SCENE_PAVILLON
        sd0, sd1 = synthetic.load_weights_npz(PAVILLON_NPZ)
    elif cfg["weights"] == "ndc":
        scene = synthetic.SCENE_PAVILLON_NDC
        sd0, sd1 = synthetic.make_weights("ndc", seed=0)
    elif cfg["weights"] == "rand":
        scene = synthetic.SCENE_BARBERSHOP
        sd0, sd1 = synthetic.make_weights("rand", seed=0)
    else:
        raise SystemExit("--single-process supports the rand / pavillon workloads")
    m = MultiRenderer(scene, list(range(G)), sd0, sd1)
    pose, rot = torch.tensor(scene["view_cell_center"], dtype=torch.float32), torch.eye(3)
    for _ in range(max(args.warmup, 3)):
        m.render_camera(pose, rot, W, Hn, thr, K)
        m.wait_frame()
    sampler = ClockSampler(0)
    sampler.start()
    for d in range(G):
        torch.cuda.synchronize(d)
    t0 = time.perf_counter()
    m.render_camera(pose, rot, W, Hn, thr, K)
    for _ in range(args.steps - 1):
        m.render_camera(pose, rot, W, Hn, thr, K)     # frame f + 1 enqueued before frame f is read
        m.wait_frame()
    frame = m.wait_frame()
    secs = time.perf_counter() - t0
    last_rgb = frame.cpu().numpy() if args.dump_outputs else None    # the library reuses the frame's buffer
    clocks = sampler.stop()
    render_ms, gather_ms = m.last_times()
    host = torch.empty((W * Hn, 3), dtype=torch.float32).pin_memory().numpy()   # caller-owned page-locked frame buffer
    t0 = time.perf_counter()
    for _ in range(args.steps):
        m.render_camera(pose, rot, W, Hn, thr, K)
        m.wait_frame(host_out=host)
    e2e_s = time.perf_counter() - t0
    frames_per_step = 1.0 if strong else float(G)
    rays = W * Hn
    line = dict(metric=f"frames_per_sec_{W}x{H}", value=frames_per_step * args.steps / secs, unit="frames/s", n_gpus=G, steps=args.steps,
                warmup=max(args.warmup, 3), ms_per_step=1000.0 * secs / args.steps, higher_is_better=True, scaling=cfg["scaling"],
                vs_baseline=None, dtype="bf16", data="synthetic",
                config=workload_config(name, cfg, G), driver="one process, all devices through include/adanerf_b200_multi.h (grouped ncclSend / ncclRecv gather)",
                rays_per_sec=rays * args.steps / secs, timing="host clock around the pipelined loop (device work of all GPUs inside)",
                band_ms_last_frame=[round(x, 3) for x in render_ms], gather_ms_last_frame=[round(x, 3) for x in gather_ms],
                e2e=dict(value=frames_per_step * args.steps / e2e_s, unit="frames/s", h2d_bytes_per_step=48, d2h_bytes_per_step=rays * 12,
                         api="adn_multi_render_camera + adn_multi_wait_frame(host)", finite=bool(np.isfinite(host).all())),
                clocks=clocks)
    print(json.dumps(line))
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, dict(rgb=last_rgb))
    m.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="800x800_thr0.2_K8", choices=sorted(WORKLOADS))
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="CPU baseline sample budget")
    ap.add_argument("--single-process", action="store_true", help="drive --gpus devices from one process (multi-GPU C ABI)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the output of the last timed step to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs: the reference arm's steps are time-bounded ray samples, not fixed outputs")
    cfg = WORKLOADS[args.workload]
    if args.impl == "reference":
        run_reference(args, cfg, args.workload)
    elif args.single_process:
        run_single_process(args, cfg, args.workload)
    else:
        run_ours(args, cfg, args.workload)


if __name__ == "__main__":
    main()
