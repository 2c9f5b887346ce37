#!/usr/bin/env python
"""bench.py -- rendered faces/sec of the FENeRF volumetric render hot path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--model A|B]
                    [--precision guard|fast|exact] [--no-graph] [--quick] [--dump-outputs DIR]

A "step" is one pass of the hot path over one batch of synthetic latents: BASELINE.json configs[1]
-- 128x128 image, 24 (+24 hierarchical) samples per ray, batch 4 per GPU, forward-only -- through
the reference-facing generator API (``generator(z, **metadata)`` under no_grad), then the frame
all-gather when N > 1.  Weights are the reference's random init under manual_seed(0); latents are
N(0,1); camera poses gaussian (h_stddev 0.3, v_stddev 0.155); nerf_noise 0.  Every timed arm (resident,
end to end, per model and precision mode) starts from the same device state: queue drained, SETTLE_S
of idle, W warm-up steps, then exactly K timed steps (StepRunner.settle says why).  One JSON line on
stdout (rank 0).  Nothing here reads /root/reference.

--dump-outputs DIR writes what the headline arm's last timed step returned to its caller: DIR/pixels.npy
(every rank's frames, as read on the host) and DIR/poses.npy, float32.  The latents, the weights and the
seed of the device RNG are fixed, so the same arguments give the same inputs on every run and two builds can
be compared output for output.
"""
import argparse
import json
import math
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402
import torch  # noqa: E402

FLOP_PER_POINT = {"A": 1053696, "B": 1341440}   # SURVEY.md section 8d (B: label chain pre-multiplied)
MODEL_NAME = {"A": "ImplicitGenerator3d+TALLSIREN", "B": "DoubleImplicitGenerator3d+TextureEmbeddingPiGAN256SEMANTICDISENTANGLE_DIM_96"}
IMG, STEPS_PER_RAY, BATCH_PER_GPU = 128, 24, 4
SETTLE_S = 1.0      # idle time in front of every timed arm (StepRunner.settle)
DUMP_BYTES = 63 << 20   # --dump-outputs stays under 64 MB in all


def metadata(img_size=IMG):
    return dict(img_size=img_size, fov=12, ray_start=0.88, ray_end=1.12, num_steps=STEPS_PER_RAY, h_stddev=0.3,
                v_stddev=0.155, h_mean=math.pi * 0.5, v_mean=math.pi * 0.5, hierarchical_sample=True,
                sample_dist='gaussian', clamp_mode='relu', nerf_noise=0.0, last_back=False)


def build_generator(model, device):
    from fenerf_b200.generators import generators as g
    from fenerf_b200.siren import siren as s
    torch.manual_seed(0)
    if model == "A":
        gen = g.ImplicitGenerator3d(s.TALLSIREN, 256, 4)
    else:
        gen = g.DoubleImplicitGenerator3d(s.TextureEmbeddingPiGAN256SEMANTICDISENTANGLE_DIM_96, 256, 256, 22)
    gen.eval()
    gen.to(device)
    gen.device = device
    gen.siren.device = device
    return gen


def make_latents(model, n_batches, batch, seed0=1000):
    out = []
    for i in range(n_batches):
        torch.manual_seed(seed0 + i)
        out.append(tuple(torch.randn(batch, 256) for _ in range(1 if model == "A" else 2)))
    return out


# ------------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms while the timed regions run."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.path = tempfile.mktemp(suffix=".csv")
        self.proc = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(gpu_index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in open(self.path).read().splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(names, f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        try:
            os.remove(self.path)
        except OSError:
            pass
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        sm.sort()
        # the busy samples are the upper half (idle gaps between regions clock down)
        busy = sm[len(sm) // 2:]
        return {"sm_mhz": busy[len(busy) // 2], "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm)}


def dist_setup(n_gpus):
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        # stdout carries exactly one JSON line: NCCL prints its version banner there at NCCL_DEBUG=VERSION and
        # =WARN, so drop those levels and send whatever NCCL logs at other levels to stderr
        if os.environ.get("NCCL_DEBUG", "").upper() in ("VERSION", "WARN"):
            del os.environ["NCCL_DEBUG"]
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    return world, rank, local


def max_over_ranks(ms, device, world):
    if world == 1:
        return ms
    import torch.distributed as dist
    t = torch.tensor([ms], dtype=torch.float64, device=device)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def barrier(world):
    if world > 1:
        import torch.distributed as dist
        dist.barrier()


# ------------------------------------------------------------------------------------------------
def cpu_faces_per_sec(model, steps, warmup, budget_s=200.0):
    """The reference's CPU path (the oracle port: same ATen ops in the same order, all host
    threads) on a bounded sample of the cfg2 workload.  Returns (faces/s, description, cores)."""
    from oracle import render_oracle as oracle
    avail = os.cpu_count() or 1
    gen = build_generator(model, "cpu")
    lat = make_latents(model, 1, 1)[0]
    film = oracle.film_from_latents(gen.siren, lat)
    # Give the reference the thread count it runs best with: torch defaults to one thread per core,
    # which on a 100+-core host is slower than a smaller pool for these (P, 256) tensors.  Probe at
    # 32 px (per-ray cost is resolution independent), keep the fastest.
    probe, cores = None, avail
    for n in sorted({avail, 64, 32, 16, 8}, reverse=True):
        if n > avail:
            continue
        torch.set_num_threads(n)
        oracle.render(gen.siren, film, metadata(16))
        t0 = time.perf_counter()
        oracle.render(gen.siren, film, metadata(32))
        dt = time.perf_counter() - t0
        if probe is None or dt < probe:
            probe, cores = dt, n
    torch.set_num_threads(cores)
    per_face = probe * (IMG / 32) ** 2
    r = IMG
    while r > 32 and per_face * (r / IMG) ** 2 * (steps + warmup) > budget_s:
        r //= 2
    md = metadata(r)
    for _ in range(warmup):
        oracle.render(gen.siren, film, md)
    t0 = time.perf_counter()
    for _ in range(steps):
        oracle.render(gen.siren, film, md)
    dt = (time.perf_counter() - t0) / steps
    frac = (r / IMG) ** 2
    sample = ("%d step(s) of %dx%d rays (%.3g of one cfg2 face, B=1, %d+%d samples/ray), oracle port, fp32, %d threads (best of a "
              "thread-count probe on %d host cores); the port takes 0.93-1.16x the live reference's time on the build container "
              "(profiles/r02_port_vs_reference.txt)" % (steps, r, r, frac, STEPS_PER_RAY, STEPS_PER_RAY, cores, avail))
    return frac / dt, sample, cores


def run_reference_arm(args, world, rank):
    if rank != 0:
        return
    value, sample, cores = cpu_faces_per_sec(args.model, args.steps, max(args.warmup, 1))
    line = {
        "impl": "reference", "metric": "rendered faces/sec at 128px x 24 samples/ray", "value": value,
        "unit": "faces/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 / value, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, world),
        "cpu_baseline": {"value": value, "unit": "faces/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "faces/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


def workload_config(args, world):
    return {"workload": "cfg2: %s, %dx%d, %d+%d samples/ray hierarchical, batch %d/GPU, forward-only render" % (
                MODEL_NAME[args.model], IMG, IMG, STEPS_PER_RAY, STEPS_PER_RAY, BATCH_PER_GPU),
            "global_batch": BATCH_PER_GPU * world, "parallelism": "dp%d (images sharded, one frame all-gather)" % world,
            "precision_mode": args.precision,
            "l2_policy": "inputs_larger_than_l2 (per-step working set ~140 MB of RNG draws, sample points and raw outputs vs "
                         "126 MB L2; fresh latents and RNG draws every step, also under graph replay)"}


# ------------------------------------------------------------------------------------------------
class StepRunner:
    """One model's render step in both arms (inputs resident / end to end), eager or as a captured CUDA graph."""

    def __init__(self, args, model, world, rank, device, n_batches, precision=None, use_graph=True):
        from fenerf_b200.dist import FrameGatherer
        from fenerf_b200.graphs import GraphedRender
        self.args, self.model, self.world, self.rank, self.device = args, model, world, rank, device
        self.precision = precision or args.precision
        self.gen = build_generator(model, device)
        self.md = dict(metadata(), precision=self.precision)
        B = BATCH_PER_GPU
        self.B = B
        self.C_img = self.gen.output_dim - 1
        self.lat_host = [tuple(z.pin_memory() for z in zs) for zs in make_latents(model, n_batches, B, 1000 + 97 * rank)]
        self.lat_dev = [tuple(z.to(device) for z in zs) for zs in self.lat_host]
        self.gatherer = FrameGatherer(B, self.C_img, IMG, device)
        self.out_host = [torch.empty((world * B, self.C_img, IMG, IMG), dtype=torch.float32).pin_memory() for _ in range(2)]
        # device-side staging, double-buffered: the render / gather output buffer is rewritten every step (it is the
        # captured graph's static output), so the step's frames are moved aside (a ~2 us D2D copy) and the D2H runs from
        # there on the copy stream -- the next step never waits for a D2H
        self.stage = [torch.empty((world * B, self.C_img, IMG, IMG), dtype=torch.float32, device=device) for _ in range(2)]
        self.out_done = [torch.cuda.Event() for _ in range(2)]
        self.frames_ready = [torch.cuda.Event() for _ in range(2)]
        self.copy_stream = torch.cuda.Stream(device=device)
        self.host_sink = 0.0
        self.first_e2e = 0
        self.last_out = None
        self.graph = None
        if use_graph:
            with torch.no_grad():
                self.graph = GraphedRender(self.gen, self.lat_dev[0], self.md)

    def render(self, latents):
        if self.graph is not None:
            return self.graph(*latents)[0]
        with torch.no_grad():
            return self.gen(*latents, **self.md)[0]

    def step_resident(self, i):
        return self.gatherer.gather(self.render(self.lat_dev[i % len(self.lat_dev)]))

    def step_e2e(self, i):
        k = i % len(self.lat_host)
        if i > self.first_e2e + 1:
            # stage[i & 1] was last read by the D2H of step i-2: long finished, but keep the order explicit
            torch.cuda.current_stream().wait_event(self.out_done[i & 1])
        if self.graph is not None:
            out = self.graph(*self.lat_host[k])                    # H2D straight into the captured input buffers
        else:
            zs = tuple(z.to(self.device, non_blocking=True) for z in self.lat_host[k])
            with torch.no_grad():
                out = self.gen(*zs, **self.md)
        self.last_out = out                                        # (frames, poses), as the generator returns them
        allf = self.gatherer.gather(out[0])
        self.stage[i & 1].copy_(allf)
        self.frames_ready[i & 1].record()
        self.copy_stream.wait_event(self.frames_ready[i & 1])
        with torch.cuda.stream(self.copy_stream):   # D2H on its own stream: the next step's kernels do not queue behind it
            self.out_host[i & 1].copy_(self.stage[i & 1], non_blocking=True)
            self.out_done[i & 1].record()
        # double-buffered serving loop: the host reads step i-1's frames while step i is queued; every step's
        # frames reach the host and are read inside the timed region
        if i > self.first_e2e:
            self.read_frames(i - 1)

    def read_frames(self, i):
        self.out_done[i & 1].synchronize()
        self.host_sink += float(self.out_host[i & 1][0, 0, 0, 0]) + float(self.out_host[i & 1][-1, -1, -1, -1])

    def settle(self):
        """Both arms start from the same device state: queue drained, then SETTLE_S of idle, then their warm-up steps.  On
        this part the power limiter pulls the SM clock down within ~0.1-0.2 s of full load (profiles/r02_diag_e2e.txt:
        the same graph replay takes 3.13-3.18 ms per step in a 20-step burst from idle and 3.48-3.56 ms once capped, with or
        without the host copies), so an arm timed right behind another one measured the limiter, not its pipeline."""
        torch.cuda.synchronize()
        time.sleep(SETTLE_S)

    def time_resident(self, steps, warmup):
        from fenerf_b200 import _lib
        self.settle()
        for i in range(warmup):
            self.step_resident(i)
        barrier(self.world); torch.cuda.synchronize()
        l0 = _lib.launch_count()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        for i in range(steps):
            self.step_resident(warmup + i)
        ev1.record()
        torch.cuda.synchronize(); barrier(self.world)
        ms = max_over_ranks(ev0.elapsed_time(ev1), self.device, self.world) / steps
        return ms, _lib.launch_count() - l0

    def time_e2e(self, steps, warmup):
        n_pre = warmup
        self.first_e2e = 0
        self.settle()
        for i in range(n_pre):
            self.step_e2e(i)
        if n_pre:
            self.read_frames(n_pre - 1)
        barrier(self.world); torch.cuda.synchronize()
        self.first_e2e = warmup
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        for i in range(steps):
            self.step_e2e(warmup + i)
        self.read_frames(warmup + steps - 1)            # the last step's frames, inside the timed region
        ev1.record()
        torch.cuda.synchronize(); barrier(self.world)
        return max_over_ranks(ev0.elapsed_time(ev1), self.device, self.world) / steps

    def launches_per_step(self):
        """Kernels of libfenerf_b200 in one step (a replayed graph launches them without passing through the
        library's host counter, so count them on an eager step)."""
        from fenerf_b200 import _lib
        l0 = _lib.launch_count()
        with torch.no_grad():
            self.gen(*self.lat_dev[0], **self.md)
        torch.cuda.synchronize()
        return int(_lib.launch_count() - l0)

    def bytes_per_step(self):
        return sum(z.numel() * 4 for z in self.lat_host[0]), self.out_host[0].numel() * 4


def measure_model(args, model, world, rank, local, steps, warmup, precision=None, sustained_s=0.0, roofline=True,
                  keep_outputs=False):
    device = torch.device("cuda", local)
    n_batches = min(steps + warmup, 64)
    r = StepRunner(args, model, world, rank, device, n_batches, precision=precision, use_graph=not args.no_graph)
    ms_step, _ = r.time_resident(steps, warmup)
    ms_e2e = r.time_e2e(steps, warmup)
    outputs = None
    if keep_outputs:
        # the last timed step: its frames as the host read them, its poses from every rank
        from fenerf_b200.dist import gather_frames
        outputs = {"pixels": r.out_host[(warmup + steps - 1) & 1].float().numpy().copy(),
                   "poses": gather_frames(r.last_out[1]).float().cpu().numpy()}
    B = BATCH_PER_GPU
    h2d, d2h = r.bytes_per_step()
    lps = r.launches_per_step()
    out = {"model": MODEL_NAME[model], "precision_mode": r.precision, "value": world * B / (ms_step / 1e3), "unit": "faces/s",
           "ms_per_step": ms_step, "cuda_graph": r.graph is not None,
           "e2e": {"value": world * B / (ms_e2e / 1e3), "unit": "faces/s", "ms_per_step": ms_e2e, "h2d_bytes_per_step": h2d,
                   "d2h_bytes_per_step": d2h,
                   "pipeline": "pinned latents -> H2D -> render (one CUDA graph launch) -> frame all-gather -> D2D into a double-buffered "
                               "staging tensor -> D2H on a copy stream into double-buffered pinned memory; step i-1's frames are read on "
                               "the host while step i runs"},
           "gpu_launches_per_step": lps, "gpu_launches": lps * steps}
    if sustained_s > 0:
        # a >= 3 s run: long enough to leave the boost clock / reach the power limit (VERDICT r1, weak #8)
        n = max(steps, int(sustained_s * 1e3 / ms_step) + 1)
        sampler = ClockSampler(local) if rank == 0 else None
        ms_long, _ = r.time_resident(n, 3)
        clocks = sampler.stop() if sampler else None
        out["sustained"] = {"steps": n, "seconds": ms_long * n / 1e3, "value": world * B / (ms_long / 1e3), "unit": "faces/s",
                            "ms_per_step": ms_long, "clocks": clocks}
    if roofline:
        out["roofline"] = field_roofline(r.gen, args, model, r.precision, r.lat_dev[0], metadata(), device)
    if outputs is not None:
        out["outputs"] = outputs
    return out


def dump_outputs(out_dir, outputs):
    """DIR/<name>.npy per array.  Past DUMP_BYTES a fixed, seeded subset of the images is kept (sorted; DIR/image_index.npy
    holds their indices)."""
    os.makedirs(out_dir, exist_ok=True)
    pixels, poses = outputs["pixels"], outputs["poses"]
    n = pixels.shape[0]
    keep = max(1, min(n, DUMP_BYTES // (pixels[0].nbytes + poses[0].nbytes)))
    if keep < n:
        idx = np.sort(np.random.default_rng(0).choice(n, keep, replace=False))
        pixels, poses = pixels[idx], poses[idx]
        np.save(os.path.join(out_dir, "image_index.npy"), idx.astype(np.float64))
    np.save(os.path.join(out_dir, "pixels.npy"), pixels)
    np.save(os.path.join(out_dir, "poses.npy"), poses)


def measure_train_step(args, world, rank, local):
    """BASELINE configs[2]-shaped generator work of one training iteration of
    CelebA_double_semantic_texture_embedding_256_dim_96 (curriculums.py:132-177) on one GPU: batch 32 as batch_split 4 x 8
    (train_double_latent_semantic.py:279-292, 334-347, 405-446): per split two no_grad renders (the fakes of the two
    discriminator steps) and one differentiable render + backward; then Adam on the generator.  The discriminators are
    outside the hot path: the loss is a fixed random projection of the frames."""
    device = torch.device("cuda", local)
    gen = build_generator("B", device)
    gen.train()
    R, S, BATCH, SPLIT = 64, 24, 32, 4
    md = dict(metadata(R), precision=args.precision)
    opt = torch.optim.Adam(gen.parameters(), lr=6e-5, betas=(0.0, 0.9))
    scaler = torch.amp.GradScaler("cuda")
    w = torch.randn((BATCH // SPLIT, gen.output_dim - 1, R, R), device=device) / (R * R)

    def iteration():
        for _ in range(2):
            with torch.no_grad():
                for _ in range(SPLIT):
                    gen(torch.randn(BATCH // SPLIT, 256, device=device), torch.randn(BATCH // SPLIT, 256, device=device), **md)
        opt.zero_grad(set_to_none=True)
        for _ in range(SPLIT):
            with torch.autocast("cuda", dtype=torch.float16):
                px, _ = gen(torch.randn(BATCH // SPLIT, 256, device=device), torch.randn(BATCH // SPLIT, 256, device=device), **md)
                loss = (px * w).sum()
            scaler.scale(loss).backward()
        scaler.unscale_(opt)
        torch.nn.utils.clip_grad_norm_(gen.parameters(), 10)
        scaler.step(opt)
        scaler.update()

    for _ in range(2):
        iteration()
    torch.cuda.synchronize()
    n = 5
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(n):
        iteration()
    ev1.record()
    torch.cuda.synchronize()
    ms = ev0.elapsed_time(ev1) / n
    return {"workload": "cfg3-shaped: %s, %dx%d, %d+%d samples/ray, batch %d as %d x %d, per iteration 2 no_grad renders + "
                        "1 differentiable render + backward per split, Adam step; synthetic loss (fixed projection of the frames)"
                        % (MODEL_NAME["B"], R, R, S, S, BATCH, SPLIT, BATCH // SPLIT),
            "ms_per_iteration": ms, "faces_rendered_per_iteration": 3 * BATCH, "rendered_faces_per_s": 3 * BATCH / (ms / 1e3),
            "iterations_per_s": 1e3 / ms, "backward": "fenerf_b200/backward.py (CUDA kernels + the library's tcgen05 GEMMs, csrc/gemm5.cu), fp16 streams"}


def run_ours(args, world, rank, local):
    from fenerf_b200 import _lib, ops
    device = torch.device("cuda", local)
    torch.cuda.set_device(device)
    _lib.lib()
    ops.set_default_precision(args.precision)
    torch.manual_seed(4242 + rank)
    sampler = ClockSampler(local) if rank == 0 else None
    main = measure_model(args, args.model, world, rank, local, args.steps, args.warmup, sustained_s=0.0,
                         keep_outputs=args.dump_outputs is not None)
    clocks = sampler.stop() if sampler else None
    outputs = main.pop("outputs", None)
    extras = {}
    if not args.quick:
        other = "B" if args.model == "A" else "A"
        short = max(5, min(args.steps, 10))
        # the >= 3 s run of the headline workload, the other field (the curriculum BASELINE configs[2..4] name), the
        # three precision modes, and the training-step shape
        extras["sustained"] = measure_model(args, args.model, world, rank, local, args.steps, 3, sustained_s=3.0,
                                            roofline=False)["sustained"]
        extras["model_" + other.lower()] = measure_model(args, other, world, rank, local, short, 3)
        modes = {}
        for mode in ("exact", "fast", "guard"):
            if mode == args.precision:
                modes[mode] = main["value"]
            else:
                modes[mode] = measure_model(args, args.model, world, rank, local, 3 if mode == "exact" else short, 3,
                                            precision=mode, roofline=False)["value"]
        extras["modes"] = {"unit": "faces/s", **modes}
        if world == 1:
            try:
                extras["train_step"] = measure_train_step(args, world, rank, local)
            except Exception as e:   # never lose the headline line to the extra
                extras["train_step"] = {"error": repr(e)[:300]}
    if rank != 0:
        return
    if outputs is not None:
        dump_outputs(args.dump_outputs, outputs)
    line = {
        "metric": "rendered faces/sec at 128px x 24 samples/ray", "value": main["value"], "unit": "faces/s",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": main["ms_per_step"],
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f16 operands / f32 accumulate (tcgen05) + f32 refinement" if args.precision != "exact" else "f32",
        "data": "synthetic", "config": workload_config(args, world), "clocks": clocks,
        "e2e": main["e2e"], "gpu_launches": main["gpu_launches"], "gpu_launches_per_step": main["gpu_launches_per_step"],
        "cuda_graph": main["cuda_graph"], "roofline": main.get("roofline"),
    }
    line.update(extras)
    if world == 1 and not args.no_cpu_baseline:
        v, sample, cores = cpu_faces_per_sec(args.model, 1, 0, budget_s=40.0)
        line["cpu_baseline"] = {"value": v, "unit": "faces/s", "cores": cores, "kind": "port", "sample": sample}
    emit(line)


def field_roofline(gen, args, model, precision, latents, md, device):
    """Times the point-network launches of one step with CUDA events on the launching stream
    (same sizes and inputs as inside the step: ray_setup -> field -> resample -> field).  The launches are
    timed alone behind a GPU-side spin, i.e. in the burst-clock regime: `frac` is against the BURST bf16 peak of
    MEASURED_PEAKS.json (`frac_of_sustained_peak` is given beside it)."""
    from fenerf_b200 import ops
    from fenerf_b200.generators import volumetric_rendering as vr
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = peaks.get("bf16_tflops") or 1700.0
    peak_src = "MEASURED_PEAKS.json bf16_tflops (burst: the kernel is timed alone, ~1.5 ms launches)" if peaks else "fallback (B200_PROFILING.md ~1.7 PF burst)"
    B, S, R = latents[0].shape[0], md["num_steps"], md["img_size"]
    N = R * R
    with torch.no_grad():
        if model == "A":
            film = gen.siren.film_table(*gen.siren.mapping_network(latents[0]))
        else:
            fg, pg = gen.siren.geo_mapping_network(latents[0]); fa, pa = gen.siren.app_mapping_network(latents[1])
            film = gen.siren.film_table(fg, fa, pg, pa)
        rd = ops.make_render_desc(batch=B, img_size=R, num_steps=S, hierarchical=True, clamp_mode='relu', nerf_noise=0.0,
                                  fov=md["fov"], precision=precision)
        x_lin, y_lin, z_lin = vr.ray_tables(R, S, md["ray_start"], md["ray_end"], device)
        c2w, _, _ = ops.camera_poses(B, 'gaussian', 0.3, 0.155, md["h_mean"], md["v_mean"], vr.DeviceRng(device), device)
        durations = []
        for it in range(6):
            pts, z, dirs, org = ops.ray_setup(rd, x_lin, y_lin, z_lin, c2w, torch.rand(B, N, S, 1, device=device))
            e = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
            # keep the GPU busy (~2 ms spin) while the host queues the launches below, so the events
            # bracket kernel execution and not Python launch latency on an idle GPU
            torch.cuda._sleep(4_000_000)
            e[0].record()
            raw_c = ops.siren_points(gen.siren, pts.reshape(B, N * S, 3), film, dirs, precision=rd.precision)
            e[1].record()
            z_f, pts_f, _ = ops.resample(rd, raw_c.reshape(B, N, S, -1), z, dirs, org, None, torch.rand(B * N, S, device=device))
            e[2].record()
            ops.siren_points(gen.siren, pts_f.reshape(B, N * S, 3), film, dirs, precision=rd.precision)
            e[3].record()
            torch.cuda.synchronize()
            if it > 0:
                durations += [e[0].elapsed_time(e[1]), e[2].elapsed_time(e[3])]
    durations.sort()
    ms = durations[len(durations) // 2] if len(durations) % 2 else 0.5 * (durations[len(durations) // 2 - 1] + durations[len(durations) // 2])
    flops = B * N * S * FLOP_PER_POINT[model]
    achieved = flops / (ms * 1e-3) / 1e12
    traffic = None
    try:
        traffic = json.load(open(os.path.join(ROOT, "profiles", "traffic.json"))).get("%s_%s" % (model, precision))
    except Exception:
        pass
    return {"bound": "tensor", "kernel": "siren point network (%s, model %s)" % (precision, model), "achieved": achieved, "peak": peak,
            "unit": "TFLOP/s", "frac": achieved / peak, "traffic": traffic, "ms_per_launch": ms,
            "flop_per_launch": flops, "peak_source": peak_src,
            "frac_of_sustained_peak": achieved / peaks["bf16_tflops_sustained"] if peaks.get("bf16_tflops_sustained") else None}


_RESULT_FD = None


def claim_stdout():
    """stdout carries exactly one JSON line.  Libraries underneath write there too (NCCL's version banner,
    whatever the box's NCCL_DEBUG is), so the real stdout is kept aside and fd 1 points at stderr until
    `emit` writes the line."""
    global _RESULT_FD
    sys.stdout.flush()
    _RESULT_FD = os.dup(1)
    os.dup2(2, 1)


def emit(line):
    data = (json.dumps(line) + "\n").encode()
    if _RESULT_FD is None:
        sys.stdout.write(data.decode()); sys.stdout.flush()
    else:
        os.write(_RESULT_FD, data)


def main():
    claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--model", default="A", choices=["A", "B"])
    ap.add_argument("--precision", default=os.environ.get("FENERF_B200_PRECISION", "guard"), choices=["guard", "fast", "exact"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-graph", action="store_true", help="run the step eagerly instead of as a captured CUDA graph")
    ap.add_argument("--quick", action="store_true", help="headline numbers only (no sustained run / other model / modes / train step)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's frames and poses as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs is not None and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        world, rank = int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("RANK", "0"))
        run_reference_arm(args, world, rank)
        return
    world, rank, local = dist_setup(args.gpus)
    try:
        run_ours(args, world, rank, local)
    finally:
        if world > 1:
            import torch.distributed as dist
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
