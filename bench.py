#!/usr/bin/env python
"""Benchmark contract of the B200-native NeRF hot path.

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--dump-outputs DIR]

One "step" = one full NeRF training iteration (BASELINE.json configs[1]: 800x800 synthetic Lego-shaped views,
4096-ray batch per GPU, 64 coarse + 128 fine samples, fp16 tensor-core MLP with fp32 accumulate, Adam step
included).  Rank 0 prints ONE JSON line.  See DESIGN.md "Measurement" for what every field means.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

N_RAYS, N_COARSE, N_FINE = 4096, 64, 128
WIDTH = HEIGHT = 800
N_TRAIN_VIEWS = 16          # synthetic views resident in HBM (16 x 640k rays x 64 B = 0.66 GB)
METRIC, UNIT = 'nerf_train_rays_per_s', 'rays/s'
# algorithmic work (SURVEY.md 8d): MACs per MLP evaluation
FLOP_FWD, FLOP_DGRAD, FLOP_WGRAD = 2 * 593408, 2 * 557696, 2 * 593408
WGRAD_KB_PER_TILE = 1424    # K4b algorithmic bytes: both stashes read once per (layer, operand) job (DESIGN.md section 4)
KERNELS_PER_STEP = 18       # OUR launches per step (ncu launch list, profiles/): pack x2, K1, K2, K3 x2, K5 x2, K8 loss, K6 x2, K4a x2, K4b x2, K7 Adam update x2 + tick (+ ~9 torch RNG / memset / copy nodes; the bench loop adds the K0 gather when it assembles a batch)
N_TEST_VIEWS = 200          # config C: the test set that is sharded across ranks by view
RENDER_VIEWS_PER_RANK = 8   # bounded sample of this rank's shard that is actually rendered and timed (config C)
SUSTAINED_SECONDS = 5.0     # extra clock-sampled run of the training step (long enough for the power governor to settle)
# dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed `ncu --set full` capture
# (profiles/r01_ncu_mlp_summary.md), keyed like the live table
NCU_TRAFFIC_BYTES = {'K4b_mlp_wgrad_fine': 8.944e9 + 0.004e9, 'K3_mlp_fwd_fine': 0.0255e9 + 4.209e9, 'K4a_mlp_dgrad_fine': 0.254e9 + 3.888e9}


def workload_config(n_gpus: int) -> dict:
    return {'workload': f'vanilla NeRF (nerf_lego model) training step, {WIDTH}x{HEIGHT} synthetic Lego-shaped views, '
                        f'{N_RAYS}-ray batch per GPU, {N_COARSE} coarse + {N_FINE} fine samples/ray',
            'rays_per_step_per_gpu': N_RAYS, 'n_coarse': N_COARSE, 'n_fine': N_FINE,
            'global_rays_per_step': N_RAYS * n_gpus,
            'parallelism': 'single GPU' if n_gpus == 1 else f'data parallel x{n_gpus}: per-rank ray batches, NCCL all-reduce of the flat MLP gradient',
            'l2': 'working set per step (9.5 GB of activation/gradient stash) exceeds the 126 MB L2; no explicit flush needed'}


# ------------------------------------------------------------------------------------------------
# clocks sampling (nvidia-smi during the timed region)
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    FIELDS = ('clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
              'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

    def __init__(self, index: int) -> None:
        self.index, self.samples, self.proc = index, [], None

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', f'--id={self.index}', f'--query-gpu={self.FIELDS}', '--format=csv,noheader,nounits',
                                          '-lms', '100'], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            parts = [p.strip() for p in line.split(',')]
            if len(parts) >= 7:
                self.samples.append(parts)

    def __exit__(self, *_):
        if self.proc is not None:
            self.proc.terminate()

    def summary(self) -> dict:
        if not self.samples:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['unavailable']}
        sm = sorted(int(float(s[0])) for s in self.samples)
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        reasons = [n for i, n in enumerate(names) if any(s[3 + i].lower().startswith('active') for s in self.samples)]
        return {'sm_mhz': sm[len(sm) // 2], 'sm_max_mhz': int(float(self.samples[0][1])), 'reasons': reasons,
                'power_w_max': max(float(s[2]) for s in self.samples), 'samples': len(sm)}


# ------------------------------------------------------------------------------------------------
# CPU arm: the reference's algorithm on the host cores (oracle port; /root/reference is absent on the GPU box)
# ------------------------------------------------------------------------------------------------
def cpu_train_step_factory(n_rays: int):
    from oracle import nerf_oracle as O
    sd = {k: v.clone().requires_grad_('frequency' not in k) for k, v in O.init_state_dict(0).items()}
    opt = torch.optim.Adam([v for v in sd.values() if v.requires_grad], lr=5e-4)
    g = torch.Generator().manual_seed(0)
    o = torch.randn(n_rays, 3, generator=g) * 0.1 + torch.tensor([0.0, -4.0, 0.5])
    d = torch.nn.functional.normalize(torch.randn(n_rays, 3, generator=g) * 0.2 + torch.tensor([0.0, 1.0, -0.1]), dim=-1) * 1.05
    v = torch.nn.functional.normalize(d, dim=-1)
    rgb, alpha, bg = torch.rand(n_rays, 3, generator=g), torch.ones(n_rays, 1), torch.ones(3)

    def step():
        out = O.render_rays(sd, o, d, v, 2.0, 6.0, bg, N_COARSE, N_FINE, torch.rand(n_rays, N_COARSE), torch.rand(n_rays, N_FINE))
        loss = O.nerf_loss(out, rgb, alpha, bg)
        opt.zero_grad()
        loss.backward()
        opt.step()
        return float(loss.detach())
    return step


def time_cpu(n_rays: int, steps: int, warmup: int) -> float:
    step = cpu_train_step_factory(n_rays)
    for _ in range(warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    return n_rays * steps / (time.perf_counter() - t0)


def use_all_host_threads() -> int:
    """torchrun exports OMP_NUM_THREADS=1 to every rank; the CPU legs are meant to use all the host threads they can."""
    torch.set_num_threads(max(torch.get_num_threads(), os.cpu_count() or 1))
    return torch.get_num_threads()


def reference_train_step_factory(n_rays: int):
    """The UNMODIFIED reference's own training-iteration body (src/Methods/NeRF/Trainer.py:51-63: render_rays -> NeRFLoss ->
    backward -> Adam step) when its tree is present (/root/reference in the build container, or baseline/_ref); None otherwise
    (the GPU box: a Python reference cannot travel, the oracle port is timed instead and labelled so)."""
    try:
        from oracle import ref_loader
        if ref_loader.reference_root() is None:
            return None
        ref = ref_loader.load_reference(n_samples=N_COARSE + N_FINE, coarse_ratio=N_COARSE / (N_COARSE + N_FINE) + 1e-7)
        from Methods.NeRF.Loss import NeRFLoss  # noqa: the reference's module
    except Exception as e:  # noqa: BLE001
        print(f'reference tree unusable ({type(e).__name__}: {e}); timing the oracle port', file=sys.stderr)
        return None
    method, DS = ref['method'], ref['ds_utils']
    model = method.MODEL('bench').build()
    renderer = method.RENDERER(model)
    opt = torch.optim.Adam(model.parameters(), lr=5e-4)
    loss_fn = NeRFLoss(1.0, 0.0, True)
    g = torch.Generator().manual_seed(0)
    o = torch.randn(n_rays, 3, generator=g) * 0.1 + torch.tensor([0.0, -4.0, 0.5])
    d = torch.nn.functional.normalize(torch.randn(n_rays, 3, generator=g) * 0.2 + torch.tensor([0.0, 1.0, -0.1]), dim=-1) * 1.05
    bg = torch.ones(3)
    rays = DS.RayBatch(origin=o, direction=d, view_direction=torch.nn.functional.normalize(d, dim=-1), rgb=torch.rand(n_rays, 3, generator=g),
                       alpha=torch.ones(n_rays, 1))
    cam = ref['PerspectiveCamera'](shared_settings=ref['SharedCameraSettings'](bg, 2.0, 6.0), width=WIDTH, height=HEIGHT, focal_x=1111.11, focal_y=1111.11)

    def step():
        out = renderer.render_rays(rays, cam, randomize_samples=True)
        loss = loss_fn(out, rays, bg)
        loss.backward()
        opt.step()
        opt.zero_grad()
        return float(loss)
    return step


def run_reference_arm(args) -> None:
    """`--impl reference`: the reference's own CPU implementation of the path on the host cores -- the unmodified reference
    when its tree is present, else its algorithm restated in oracle/nerf_oracle.py (pinned to the reference by tests/golden);
    all host threads, bounded sample per step."""
    rank = int(os.environ.get('RANK', 0))
    if rank != 0:
        return
    threads = use_all_host_threads()
    probe = 128
    kind = 'reference' if reference_train_step_factory(probe) is not None else 'port'
    factory = reference_train_step_factory if kind == 'reference' else cpu_train_step_factory
    step = factory(probe)
    step()
    t0 = time.perf_counter()
    step()
    per_ray = (time.perf_counter() - t0) / probe
    budget = 100.0 / max(args.steps + args.warmup, 1)           # seconds per step so the whole run stays within minutes
    n_rays = int(min(N_RAYS, max(64, budget / per_ray)))
    step = factory(n_rays)
    for _ in range(args.warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()
    value = n_rays * args.steps / (time.perf_counter() - t0)
    what = "the unmodified reference's render_rays + NeRFLoss + Adam" if kind == 'reference' else 'fp32 PyTorch oracle port, autograd + Adam'
    sample = f'{n_rays}-ray training steps ({N_COARSE}+{N_FINE} samples, {what}) of the {N_RAYS}-ray workload'
    print(json.dumps({
        'impl': 'reference', 'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': args.gpus, 'steps': args.steps, 'warmup': args.warmup,
        'ms_per_step': 1e3 * n_rays / value, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'fp32',
        'data': 'synthetic', 'config': workload_config(args.gpus),
        'cpu_baseline': {'value': value, 'unit': UNIT, 'cores': threads, 'kind': kind, 'sample': sample},
        'e2e': {'value': value, 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}, 'gpu_launches': 0}), flush=True)


# ------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------
def measured_peaks() -> tuple[dict, str]:
    path = ROOT / 'MEASURED_PEAKS.json'
    if path.exists():
        return json.loads(path.read_text()), 'measured (MEASURED_PEAKS.json)'
    return {'hbm_gbs': 6650.0, 'bf16_tflops': 1590.0, 'bf16_tflops_sustained': 1400.0}, 'fallback (B200_PROFILING.md)'


def instrumented_kernel_times(trainer, step_obj, reps: int = 3) -> dict:
    """Per-kernel device time of one training iteration: the same call sequence as the captured step, run eagerly
    with a CUDA event pair around every C-ABI launch on the launching (current) stream."""
    from nerficg_b200 import ops
    s = step_obj
    n, dev = s.n, s.dev
    flats = [b.flat_params for b in s.blocks]
    times: dict[str, list[float]] = {}

    def timed(name, fn):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        out = fn()
        b.record()
        times.setdefault(name, []).append((a, b))
        return out

    for _ in range(reps):
        for flat, packed in zip(flats, s.packed):
            timed('pack', lambda: ops.mlp_pack(flat, packed, True))
        u_c = torch.rand((n, s.nc), device=dev)
        z_c = timed('K1_stratified', lambda: ops.sample_stratified(n, s.nc, s.near, s.far, u_c, dev))
        rs_c = timed('K3_mlp_fwd_coarse', lambda: ops.mlp_forward(s.packed[0], flats[0], s.origin, s.direction, s.view_direction, z_c, None, s.stash[0]))
        rgb_c, _, _, w_c = timed('K5_composite_fwd_coarse', lambda: ops.composite_forward(z_c, rs_c, s.direction, s.bg, True))
        u_f = torch.rand(n, s.nf, device=dev)
        z = timed('K2_importance', lambda: ops.sample_importance(z_c, w_c, s.nf, u_f))
        rs_f = timed('K3_mlp_fwd_fine', lambda: ops.mlp_forward(s.packed[1], flats[1], s.origin, s.direction, s.view_direction, z, None, s.stash[1]))
        rgb, _, _, _ = timed('K5_composite_fwd_fine', lambda: ops.composite_forward(z, rs_f, s.direction, s.bg))
        g = (rgb - s.rgb_gt) * (2.0 / rgb.numel())
        grads = [torch.zeros_like(f) for f in flats]
        d_rs = timed('K6_composite_bwd_fine', lambda: ops.composite_backward(z, rs_f, s.direction, s.bg, g, None, None, True, s.scale))
        timed('K4a_mlp_dgrad_fine', lambda: ops.mlp_backward_dgrad(d_rs, rs_f, s.stash[1], s.ws, s.packed[1], flats[1], n, z.shape[1]))
        timed('K4b_mlp_wgrad_fine', lambda: ops.mlp_backward_wgrad(grads[1], s.stash[1], s.ws, n, z.shape[1], s.scale))
        g_c = (rgb_c - s.rgb_gt) * (2.0 / rgb_c.numel())
        d_rs_c = timed('K6_composite_bwd_coarse', lambda: ops.composite_backward(z_c, rs_c, s.direction, s.bg, g_c, None, None, True, s.scale))
        timed('K4a_mlp_dgrad_coarse', lambda: ops.mlp_backward_dgrad(d_rs_c, rs_c, s.stash[0], s.ws, s.packed[0], flats[0], n, s.nc))
        timed('K4b_mlp_wgrad_coarse', lambda: ops.mlp_backward_wgrad(grads[0], s.stash[0], s.ws, n, s.nc, s.scale))
    torch.cuda.synchronize()
    return {k: sum(a.elapsed_time(b) for a, b in v[1:]) / max(len(v) - 1, 1) * (2 if k == 'pack' else 1) for k, v in times.items()}


def run_gpu_arm(args) -> None:
    rank = int(os.environ.get('RANK', 0))
    local_rank = int(os.environ.get('LOCAL_RANK', 0))
    world = int(os.environ.get('WORLD_SIZE', 1))
    if world != args.gpus and world > 1:
        raise SystemExit(f'--gpus {args.gpus} but WORLD_SIZE={world}')
    from nerficg_b200 import Framework
    Framework.setup(None, {'RENDERER.N_SAMPLES': N_COARSE + N_FINE, 'RENDERER.COARSE_RATIO': N_COARSE / (N_COARSE + N_FINE) + 1e-7,
                           'TRAINING.BATCH_SIZE': N_RAYS, 'TRAINING.NUM_ITERATIONS': 500000, 'GLOBAL.LOG_LEVEL': 0}, device_index=local_rank)
    dev = Framework.config.GLOBAL.DEFAULT_DEVICE
    if world > 1:
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        import datetime
        # a mismatched collective must abort the run in two minutes, not in NCCL's default ten
        torch.distributed.init_process_group('nccl', device_id=dev, timeout=datetime.timedelta(seconds=120))
    from nerficg_b200.Datasets import RayBatch
    from nerficg_b200.Datasets.Synthetic import SyntheticLegoDataset
    from nerficg_b200.Implementations import Methods

    torch.manual_seed(0)                         # identical initial weights on every rank
    trainer = Methods.get_training_instance('NeRF')
    model, renderer = trainer.model, trainer.renderer
    assert (renderer.n_samples_coarse_nerf, renderer.n_samples_nerf) == (N_COARSE, N_FINE)
    torch.manual_seed(1000 + rank)               # per-rank ray batches and sampling noise
    dataset = SyntheticLegoDataset(WIDTH, HEIGHT, N_TRAIN_VIEWS, RENDER_VIEWS_PER_RANK, seed=rank, device=dev)
    dataset.precompute_rays(['train'])
    pool = dataset.ray_collection['train'].all_rays
    camera = dataset.default_camera
    n_pool = len(pool)

    def device_batch() -> RayBatch:
        return pool[torch.randint(0, n_pool, (N_RAYS,), device=dev)]

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            torch.distributed.barrier()
            torch.cuda.synchronize()

    # ---- warm-up (>= 3; the first two fused steps run eagerly, the third captures the CUDA graph) ----
    warmup = max(args.warmup, 3)
    for _ in range(warmup):
        trainer.fused_step(device_batch(), camera)
    sync_all()
    if args.profile_steps > 0:   # ncu --profile-from-start off: only these graph replays are captured (never a bench value)
        torch.cuda.profiler.start()
        for _ in range(args.profile_steps):
            trainer.fused_step(device_batch(), camera)
        torch.cuda.synchronize()
        torch.cuda.profiler.stop()
        _leave(world)
        return

    # ---- timed region A: inputs resident in HBM, device-timed, max over ranks ----
    batches = [device_batch() for _ in range(min(args.steps, 64))]
    sync_all()
    with ClockSampler(local_rank) as clocks:
        start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        start.record()
        for i in range(args.steps):
            loss = trainer.fused_step(batches[i % len(batches)], camera)
        end.record()
        sync_all()
        elapsed_ms = start.elapsed_time(end)
        # the regions below keep training, so what the last timed step returned (the loss in the step's static buffer)
        # and left in the model (its parameters) is copied now
        dumped = {'loss': loss.clone(), **{k: p.detach().clone() for k, p in model.named_parameters()}} if args.dump_outputs else None
        # ---- timed region B (end to end): pinned host buffers -> H2D copy every step, loss read back every step ----
        host = []
        for b in batches[:8]:
            host.append({k: getattr(b, k).cpu().pin_memory() for k in ('origin', 'direction', 'view_direction', 'rgb', 'alpha')})
        h2d = sum(t.numel() * 4 for t in host[0].values())
        sync_all()
        e_start, e_end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e_start.record()
        losses = []
        for i in range(args.steps):
            # the public call with HOST buffers: the step copies the pinned fields straight into its static device buffers
            # (five H2D copies on the step's stream), replays the captured iteration, and the loss is read back
            rb = RayBatch(**host[i % len(host)], _skip_post_init=True)
            losses.append(trainer.fused_step(rb, camera).item())    # D2H read of the step's loss
        e_end.record()
        sync_all()
        e2e_sync_ms = e_start.elapsed_time(e_end)
        # the same loop as a training script writes it: every step's loss still crosses to the host inside the timed region,
        # but through a two-deep pinned ring read one step late, so the host enqueues step i+1 while step i runs
        ring = [torch.empty((), dtype=torch.float32).pin_memory() for _ in range(2)]
        landed = [torch.cuda.Event(), torch.cuda.Event()]
        sync_all()
        p_start, p_end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        p_start.record()
        losses_p = []
        for i in range(args.steps):
            rb = RayBatch(**host[i % len(host)], _skip_post_init=True)
            ring[i & 1].copy_(trainer.fused_step(rb, camera), non_blocking=True)
            landed[i & 1].record()
            if i > 0:
                landed[(i - 1) & 1].synchronize()
                losses_p.append(float(ring[(i - 1) & 1]))
        landed[(args.steps - 1) & 1].synchronize()
        losses_p.append(float(ring[(args.steps - 1) & 1]))
        p_end.record()
        sync_all()
        e2e_ms = p_start.elapsed_time(p_end)
        assert len(losses_p) == args.steps and all(x == x for x in losses_p)
    if world > 1:
        t = torch.tensor([elapsed_ms, e2e_ms, e2e_sync_ms], device=dev, dtype=torch.float64)
        torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
        elapsed_ms, e2e_ms, e2e_sync_ms = t.tolist()
    value = N_RAYS * world * args.steps / (elapsed_ms * 1e-3)
    e2e_value = N_RAYS * world * args.steps / (e2e_ms * 1e-3)

    # ---- sustained clocks: the same step for >= SUSTAINED_SECONDS with nvidia-smi sampling (the K-step region above is too
    # short for the power governor to settle; this is the number a long training run sees) ----
    n_sus = max(int(SUSTAINED_SECONDS * 1e3 / (elapsed_ms / args.steps)), args.steps)
    sync_all()
    with ClockSampler(local_rank) as sus_clocks:
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s0.record()
        for i in range(n_sus):
            trainer.fused_step(batches[i % len(batches)], camera)
        s1.record()
        sync_all()
        sus_ms = s0.elapsed_time(s1)
    if world > 1:
        t = torch.tensor([sus_ms], device=dev, dtype=torch.float64)
        torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
        sus_ms = t.item()
    sustained = {'steps': n_sus, 'seconds': sus_ms * 1e-3, 'ms_per_step': sus_ms / n_sus, 'value': N_RAYS * world * n_sus / (sus_ms * 1e-3),
                 'unit': UNIT, 'clocks': sus_clocks.summary()}

    # ---- config C, rendering throughput (second half of the metric): the 200 test views are sharded across ranks by view
    # (dist.shard_range, no collective); every rank renders a bounded sample of ITS shard through the public call
    # NeRFRenderer.render_image(view) -- K0 ray generation inside the timed region, one full-size warm-up view outside ----
    from nerficg_b200 import dist
    shard = dist.shard_range(N_TEST_VIEWS, rank, world)
    test_views = dataset.test()
    my_views = [test_views[i % len(test_views)] for i in list(shard)[:RENDER_VIEWS_PER_RANK]]
    dataset.train()
    del batches, host
    trainer._fused.clear()           # the training stashes (9.5 GB) are not needed any more
    view_ms = []
    with torch.no_grad():
        renderer.RAY_BATCH_SIZE = 65536
        model.eval()
        renderer.render_image(my_views[0])               # full-size warm-up view (allocator, lazy module loads)
        sync_all()
        with ClockSampler(local_rank) as render_clocks:
            marks = [torch.cuda.Event(enable_timing=True) for _ in range(len(my_views) + 1)]
            marks[0].record()
            n_render_rays = 0
            for i, v in enumerate(my_views):
                out = renderer.render_image(v)
                n_render_rays += out['rgb'].shape[0] * out['rgb'].shape[1]
                marks[i + 1].record()
            sync_all()
        render_ms = marks[0].elapsed_time(marks[-1])
        view_ms = [round(marks[i].elapsed_time(marks[i + 1]), 2) for i in range(len(my_views))]
    if world > 1:
        t = torch.tensor([render_ms], device=dev, dtype=torch.float64)
        torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
        render_ms = t.item()
    render_mrays = n_render_rays * world / (render_ms * 1e-3) / 1e6
    render_tflops = FLOP_FWD * (N_COARSE + N_COARSE + N_FINE) * n_render_rays * world / render_ms / 1e9

    if rank != 0:
        _leave(world)   # the remaining work (per-kernel table, CPU baseline) is rank 0's alone and uses no collective

    # ---- per-kernel roofline (rank 0): live CUDA-event timing of every launch of one iteration ----
    peaks, peak_source = measured_peaks()
    # (rank 0 alone from here on: nothing below may issue a collective -- the step object is built without running its body)
    from nerficg_b200.Methods.NeRF.Trainer import _FusedStep
    probe_step = _FusedStep(trainer, N_RAYS, camera, False)
    pb = device_batch()
    probe_step.origin.copy_(pb.origin); probe_step.direction.copy_(pb.direction); probe_step.view_direction.copy_(pb.view_direction)
    probe_step.rgb_gt.copy_(pb.rgb); probe_step.alpha_gt.copy_(pb.alpha)
    kt = instrumented_kernel_times(trainer, probe_step)
    evals = {'coarse': N_RAYS * N_COARSE, 'fine': N_RAYS * (N_COARSE + N_FINE)}
    n_tiles = {k: (v + 127) // 128 for k, v in evals.items()}
    table = {}
    for name, ms in kt.items():
        which = 'coarse' if name.endswith('coarse') else 'fine'
        row = {'ms': round(ms, 4)}
        if name.startswith('K3'):
            row.update(bound='tensor', achieved=FLOP_FWD * evals[which] / ms / 1e9, peak=peaks['bf16_tflops_sustained'], unit='TFLOP/s')
        elif name.startswith('K4a'):
            row.update(bound='tensor', achieved=FLOP_DGRAD * evals[which] / ms / 1e9, peak=peaks['bf16_tflops_sustained'], unit='TFLOP/s')
        elif name.startswith('K4b'):   # operands re-read from the stashes: 1424 KB per 128-sample tile (DESIGN.md)
            row.update(bound='hbm', achieved=WGRAD_KB_PER_TILE * 1024 * n_tiles[which] / ms / 1e6, peak=peaks['hbm_gbs'], unit='GB/s',
                       tensor_tflops=FLOP_WGRAD * evals[which] / ms / 1e9)
        elif name.startswith('K5'):
            s = N_COARSE if which == 'coarse' else N_COARSE + N_FINE
            row.update(bound='hbm', achieved=N_RAYS * ((24 if which == 'coarse' else 20) * s + 32) / ms / 1e6, peak=peaks['hbm_gbs'], unit='GB/s')
        elif name.startswith('K6'):
            s = N_COARSE if which == 'coarse' else N_COARSE + N_FINE
            row.update(bound='hbm', achieved=N_RAYS * (36 * s + 48) / ms / 1e6, peak=peaks['hbm_gbs'], unit='GB/s')
        if 'achieved' in row:
            row['frac'] = row['achieved'] / row['peak']
        table[name] = row
    total_kernel_ms = sum(r['ms'] for r in table.values())
    for r in table.values():
        r['share'] = round(r['ms'] / total_kernel_ms, 4)
    dom_name = max((k for k in table if 'achieved' in table[k]), key=lambda k: table[k]['ms'])
    dom = table[dom_name]
    roofline = {'kernel': dom_name, 'bound': dom['bound'], 'achieved': dom['achieved'], 'peak': dom['peak'], 'unit': dom['unit'],
                'frac': dom['frac'], 'traffic': NCU_TRAFFIC_BYTES.get(dom_name), 'traffic_unit': 'bytes per launch (ncu --set full, profiles/)', 'peak_source': peak_source + ('; sustained figure: the kernel is timed inside a long step' if dom['bound'] == 'tensor' else ''),
                'ms_per_launch': dom['ms'], 'share_of_step': dom['share'],
                'mlp_tensor_tflops_whole_step': (FLOP_FWD + FLOP_DGRAD + FLOP_WGRAD) * (evals['coarse'] + evals['fine']) / (elapsed_ms / args.steps) / 1e9}

    # ---- config E: HBM-bound stages at 65,536 rays (L2 flushed before every timed launch) ----
    sys.path.insert(0, str(ROOT / 'tools'))
    import stress_sweep
    stress = {'workload': 'config E: 65,536-ray batch, sampling + compositing only, L2 flush (512 MB fill + 512 MB read) before every launch',
              'peak_gbs': peaks['hbm_gbs'], 'rows': stress_sweep.run(65536, iters=5, device=str(dev))}
    for row in stress['rows']:
        for k in row['kernels'].values():
            k['frac'] = round(k['gbs'] / peaks['hbm_gbs'], 3)

    # ---- CPU baseline: the oracle port on this box's host cores, bounded sample ----
    threads = use_all_host_threads()     # (torchrun exports OMP_NUM_THREADS=1)
    cpu_rays = 1024
    cpu_value = time_cpu(cpu_rays, steps=3, warmup=1)
    cpu_baseline = {'value': cpu_value, 'unit': UNIT, 'cores': threads, 'kind': 'port',
                    'sample': f'3 training steps of {cpu_rays} rays ({N_COARSE}+{N_FINE} samples) of the same workload, fp32 PyTorch oracle, {os.cpu_count()} logical CPUs'}

    print(json.dumps({
        'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': world, 'steps': args.steps, 'warmup': warmup,
        'ms_per_step': elapsed_ms / args.steps, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
        'dtype': 'fp16 operands, fp32 accumulate (fp32 sampling/compositing/optimizer)', 'data': 'synthetic', 'config': workload_config(world),
        'e2e': {'value': e2e_value, 'unit': UNIT, 'h2d_bytes_per_step': h2d, 'd2h_bytes_per_step': 4, 'ms_per_step': e2e_ms / args.steps,
                'last_loss': losses_p[-1],
                'how': 'pinned host RayBatch -> H2D into the step buffers -> captured iteration -> loss D2H into a two-deep pinned ring, read by the host one step late',
                'blocking_read_ms_per_step': e2e_sync_ms / args.steps},
        'gpu_launches': KERNELS_PER_STEP * args.steps, 'clocks': clocks.summary(),
        'roofline': roofline, 'kernels': table, 'cpu_baseline': cpu_baseline,
        'sustained': sustained,
        'render': {'metric': 'nerf_render_mrays_per_s', 'value': render_mrays, 'unit': 'Mrays/s', 'n_gpus': world,
                   'workload': f'config C: {N_TEST_VIEWS} test views {WIDTH}x{HEIGHT} sharded by view over {world} rank(s), no collective; '
                               f'{len(my_views)} views of each rank\'s shard timed through NeRFRenderer.render_image (K0 ray generation inside), {N_COARSE}+{N_FINE} samples',
                   'rays_per_gpu': n_render_rays, 'views_per_gpu_timed': len(my_views), 'views_in_shard': len(shard), 'ms': render_ms,
                   'ms_per_view_rank0': view_ms, 'per_gpu_mrays': render_mrays / world, 'tensor_tflops': render_tflops,
                   'tensor_frac_of_burst_peak_per_gpu': render_tflops / world / peaks['bf16_tflops'], 'clocks': render_clocks.summary()},
        'stress': stress,
    }), flush=True)
    if dumped is not None:
        dump_outputs(Path(args.dump_outputs), dumped)
    _leave(world)


def dump_outputs(out_dir: Path, arrays: dict[str, torch.Tensor]) -> None:
    """Writes every array as out_dir/<name>.npy in float32, so that two builds run with the same arguments (hence the
    same seeded inputs) can be compared output for output."""
    import numpy as np
    host = {k: v.detach().float().cpu().numpy() for k, v in arrays.items()}
    total = sum(a.nbytes for a in host.values())
    assert total <= 64 << 20, f'{total} bytes of outputs exceed the 64 MB dump budget'
    out_dir.mkdir(parents=True, exist_ok=True)
    for name, a in host.items():
        np.save(out_dir / f'{name}.npy', a)


def _leave(world: int) -> None:
    """Ends a rank.  Under torchrun the process exits without tearing the NCCL communicator down: destroying a process
    group whose collectives live inside a captured CUDA graph hung at exit (measured: the 2-GPU run printed its line and
    then sat in destroy_process_group until the timeout), and the OS reclaims everything anyway."""
    sys.stdout.flush()
    sys.stderr.flush()
    if world > 1:
        torch.cuda.synchronize()
        os._exit(0)


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=30)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--profile-steps', type=int, default=0, help='run N steps between cudaProfilerStart/Stop and exit (for ncu)')
    ap.add_argument('--deadline', type=float, default=900.0,
                    help='seconds after which a run that is still going dumps every thread\'s stack to stderr and exits 1 '
                         '(a rank stuck in a collective must not hold a multi-GPU box until the caller\'s own limit)')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='after the timed steps, write what the last one computed (its loss and the updated model parameters) '
                         'as DIR/<name>.npy (float32; rank 0)')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and args.impl != 'ours':
        ap.error('--dump-outputs writes the outputs of the CUDA training step (--impl ours)')
    if args.deadline > 0:
        import faulthandler
        faulthandler.dump_traceback_later(args.deadline, exit=True)
    if args.impl == 'reference':
        run_reference_arm(args)
    else:
        run_gpu_arm(args)


if __name__ == '__main__':
    main()
