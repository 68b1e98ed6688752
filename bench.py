#!/usr/bin/env python
"""bench.py -- rendered frames/sec at 64^2 neural x 96 samples -> 512^2 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    (N > 1: python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...)

A "step" is one pass of the hot path over one batch: G.synthesis(ws, c) for 8 latents of the random-init
ide3d-ffhq-64-512 generator (tri-plane backbone -> fused ray-march at 64^2 x 96 -> super-resolution to 512^2), yaw
sweep -- BASELINE.json configs[1].  Weak scaling: every rank renders its own 8-frame batch.

value : whole-job frames/s with ws / cameras already resident in HBM (CUDA events, max over ranks, L2 flushed
        between timed iterations).
e2e   : the same metric through the public call a user makes (stream_frames_sharded: host ws / cameras -> H2D from
        pinned memory -> synthesis -> uint8 frames -> all_gather over NCCL when N > 1 -> D2H), copies inside the
        timed region.
roofline : the fused ray-march kernel (dominant kernel of the renderer), timed live with CUDA events on its stream
        inside the synthesis steps; algorithmic bytes = 51.20 MB per frame (both tri-planes once + outputs).
cpu_baseline : the oracle port (stock torch-CPU ops chained like the reference's free functions) on the host cores,
        bounded sample = 1 frame of the same workload.
--impl reference : that CPU path as the timed arm (rank 0 only).
--dump-outputs DIR : after the timed steps, rank 0 writes the images its last timed step returned to DIR/image.npy (float32
        [8, 3, 512, 512], 25 MB).  Inputs and the ray jitter seed of that step are fixed, so two builds can be compared output
        for output.
"""

import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

sys.dont_write_bytecode = True           # the source tree may be read-only: no __pycache__ next to the sources
ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

BATCH = 8
NUM_STEPS = 96
RENDER = 64
PLANE = 256
FRAME_ALGO_BYTES = 2 * 96 * PLANE * PLANE * 4 + RENDER * RENDER * (32 + 19 + 1 + 1) * 4   # 51.20 MB (SURVEY §8d)
METRIC = 'rendered frames/sec at 64^2 neural x 96 samples -> 512^2'
TRAFFIC_JSON = os.path.join(ROOT, 'profiles', 'raymarch_traffic.json')      # dram bytes of the ray-march launch, written from an ncu --set full capture


def raymarch_traffic():
    """(bytes per launch | None, source).  The number is a citation of a committed ncu capture of THIS kernel version, not a constant in
    the bench: profiles/raymarch_traffic.json = {"kernel": ..., "dram_bytes_read": ..., "dram_bytes_write": ..., "capture": "profiles/..."}."""
    try:
        t = json.load(open(TRAFFIC_JSON))
        return int(t['dram_bytes_read']) + int(t['dram_bytes_write']), f"{t.get('capture', TRAFFIC_JSON)} ({t.get('kernel', '?')})"
    except Exception:
        return None, 'no ncu capture committed for this kernel version'


def make_labels(n):
    """Host labels: cam2world from the product's own pose helpers (training/volumetric_rendering.py:147-213)."""
    from ide3d_b200.training.volumetric_rendering import create_cam2world_matrix, sample_camera_positions
    yaws = math.pi / 2 + torch.linspace(-0.5, 0.5, n)
    intr = torch.tensor([4.2647, 0, 0.5, 0, 4.2647, 0.5, 0, 0, 1], dtype=torch.float32)
    cs = []
    for y in yaws:
        o, _, _ = sample_camera_positions('cpu', n=1, r=2.7, horizontal_mean=float(y), vertical_mean=math.pi / 2, mode=None)
        m = create_cam2world_matrix(-o, o, device='cpu')
        cs.append(torch.cat([m.reshape(1, 16), intr.reshape(1, 9)], 1))
    return torch.cat(cs)


def make_latents(n, z_dim, offset=0):
    return torch.from_numpy(np.stack([np.random.RandomState(offset + i).randn(z_dim) for i in range(n)])).float()


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms while the timed region runs."""
    Q = ('clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
         'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', f'--id={self.index}', f'--query-gpu={self.Q}', '--format=csv,noheader,nounits',
                                          '-lms', '200'], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([v.strip() for v in line.split(',')])

    def __exit__(self, *exc):
        if self.proc is not None:
            time.sleep(0.25)
            self.proc.terminate()
            self.thread.join(timeout=2)

    def summary(self):
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
            except (ValueError, IndexError):
                continue
            for name, v in zip(('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'), r[3:7]):
                if v.lower().startswith('active'):
                    reasons.add(name)
        if not sm:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable'], 'samples': 0}
        return {'sm_mhz': float(np.median(sm)), 'sm_max_mhz': float(max(mx)), 'reasons': sorted(reasons), 'samples': len(sm)}


def measured_peak_gbs():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        try:
            return float(json.load(open(p))['hbm_gbs']), 'measured (MEASURED_PEAKS.json hbm_gbs)'
        except Exception:
            pass
    return 6650.0, 'fallback (B200_PROFILING.md 6.65 TB/s)'


def pick_cpu_threads():
    """Use the host cores the way that is FASTEST for this path: torch-CPU's small-op chain slows down badly when it is
    spread over every hardware thread of a 128-core host (51 s/frame at 128 threads vs ~3 s at 8), so time one render-only
    frame at a few thread counts and keep the best.  Reported as `cores`."""
    from oracle import renderer as orr
    ncpu = os.cpu_count() or 1
    cands = sorted({c for c in (8, 16, 32, 64, ncpu) if c <= ncpu})
    g = torch.Generator().manual_seed(0)
    tex = torch.randn(1, 96, 128, 128, generator=g)
    dec = orr.Decoder.random(hidden=64, seed=1)
    cam = torch.eye(4)[None].clone()
    cam[0, 2, 3] = 2.7
    best = None
    for c in cands:
        torch.set_num_threads(c)
        orr.render_frames(tex, tex, dec, cam, num_steps=24, resolution=(32, 32))
        t0 = time.perf_counter()
        orr.render_frames(tex, tex, dec, cam, num_steps=24, resolution=(32, 32))
        dt = time.perf_counter() - t0
        if best is None or dt < best[1]:
            best = (c, dt)
    torch.set_num_threads(best[0])
    return best[0]


def cpu_reference_fps(G_cpu, ws1, c1, reps):
    """Oracle port on the host cores: full synthesis of ONE frame of the same workload.  Also returns that frame (the live parity check)."""
    from oracle.backend import cpu_reference_ops
    times = []
    with torch.no_grad(), cpu_reference_ops():
        G_cpu.synthesis(ws1, c=c1, render_params=dict(num_steps=NUM_STEPS), noise_mode='const', perturb='hash', seed=1)   # warm-up
        for _ in range(reps):
            t0 = time.perf_counter()
            img = G_cpu.synthesis(ws1, c=c1, render_params=dict(num_steps=NUM_STEPS), noise_mode='const', perturb='hash', seed=1)
            times.append(time.perf_counter() - t0)
    return 1.0 / float(np.mean(times)), float(np.mean(times)), img


def gpu_reference_chain_ms(G, img_v, seg_v, cam, reps=3):
    """The REFERENCE renderer's op chain on the same GPU, same planes, same decoder (north-star comparison: fused kernel >= 20x this):
    a1 rays, a2 jitter, a3 cam2world bmm, a5 F.grid_sample x 6, decoder matmuls + softplus, a7 compositing -- the oracle's restatement of
    volumetric_rendering.py:34-136 / dnnlib/util.py:580-617 executed on CUDA tensors, every stage materialised in HBM as the reference
    does (tests/test_gpu_speedup.py is the same measurement as a test).  NCHW planes, as the reference's fp32 path keeps them."""
    from oracle import renderer as R
    from oracle.backend import _decoder_from_renderer
    dec = _decoder_from_renderer(G.synthesis.renderer)
    for k in ('w1', 'b1', 'w2', 'b2'):
        setattr(dec, k, getattr(dec, k).to(img_v.device))
    tex, seg = img_v.contiguous(), seg_v.contiguous()
    n, S = tex.shape[0], NUM_STEPS
    box = G.synthesis.renderer.box_scale

    def chain():
        with torch.device(img_v.device):
            u = torch.rand(n, RENDER * RENDER, S, 1)
            pts, zv, d = R.initial_rays(n, S, 18.0, (RENDER, RENDER), 2.25, 3.3)
            pts, zv = R.perturb(pts, zv, d, u)
            pw, _, _ = R.to_world(pts, d, cam)
            coords = pw.reshape(n, -1, 3) * box
            out = dec(R.sample_triplane_torch(coords, tex), R.sample_triplane_torch(coords, seg)).reshape(n, RENDER * RENDER, S, R.N_OUT)
            return R.composite(out, d, zv, clamp_mode='softplus')

    chain()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        chain()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


def build_generator(device):
    from ide3d_b200.compat import random_init_generator
    from ide3d_b200.torch_utils import custom_ops
    custom_ops.verbosity = 'none'
    return random_init_generator(device=device, seed=0)


def run_reference(args, rank):
    """--impl reference: the CPU path is the timed arm.  Rank 0 only; other ranks exit 0 without work."""
    if rank != 0:
        return
    pick_cpu_threads()
    G = build_generator('cpu')
    z = make_latents(1, G.z_dim)
    c = make_labels(BATCH)[BATCH // 2:BATCH // 2 + 1]
    from oracle.backend import cpu_reference_ops
    with torch.no_grad(), cpu_reference_ops():
        ws = G.mapping(z, c)
    kw = dict(render_params=dict(num_steps=NUM_STEPS), noise_mode='const', perturb='hash', seed=1)
    with torch.no_grad(), cpu_reference_ops():
        G.synthesis(ws, c=c, **kw)                      # one untimed warm-up (each step is ~10 s of CPU work)
        t0 = time.perf_counter()
        for _ in range(args.steps):
            G.synthesis(ws, c=c, **kw)
        dt = time.perf_counter() - t0
    fps = args.steps / dt
    cores = torch.get_num_threads()
    sample = '1 frame per step (of the 8-frame batch): full synthesis backbone -> 64^2x96 render -> 512^2 SR, torch-CPU ops'
    line = {'impl': 'reference', 'metric': METRIC, 'value': fps, 'unit': 'frames/s', 'n_gpus': args.gpus, 'steps': args.steps,
            'warmup': args.warmup, 'ms_per_step': 1e3 * dt / args.steps, 'higher_is_better': True, 'scaling': 'weak',
            'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
            'config': {'workload': 'configs[1]: 64^2 x 96 -> 512^2, random-init ide3d-ffhq-64-512, yaw sweep', 'frames_per_step': 1,
                       'arm': 'oracle port of the reference PyTorch path on host cores'},
            'cpu_baseline': {'value': fps, 'unit': 'frames/s', 'cores': cores, 'kind': 'port', 'sample': sample},
            'e2e': {'value': fps, 'unit': 'frames/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
            'gpu_launches': 0}
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=10)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--cpu-reps', type=int, default=2, help='timed repetitions of the 1-frame CPU baseline')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--dump-outputs', metavar='DIR', help='write the images of the last timed step to DIR/image.npy')
    args = ap.parse_args()

    if args.impl == 'reference':
        run_reference(args, int(os.environ.get('RANK', '0')))
        return

    from ide3d_b200 import _lib, dist as idist, render
    from ide3d_b200.torch_utils import custom_ops
    custom_ops.verbosity = 'none'            # keep stdout to the one JSON line
    rank, world, device = idist.init_from_env()
    assert device.type == 'cuda', 'bench.py needs a CUDA device (the product has no CPU path)'
    assert world == args.gpus or world == 1, f'--gpus {args.gpus} but WORLD_SIZE={world}'
    import torch.distributed as tdist
    torch.backends.cudnn.benchmark = True

    G = build_generator(device)
    z_host = make_latents(BATCH, G.z_dim, offset=rank * BATCH)
    c_host = make_labels(BATCH)
    with torch.no_grad():
        ws = G.mapping(z_host.to(device), c_host.to(device))
    c = c_host.to(device)
    kw = dict(render_params=dict(num_steps=NUM_STEPS), noise_mode='const')
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=device)      # 256 MB > 126 MB L2

    def barrier():
        if world > 1:
            tdist.barrier()
        torch.cuda.synchronize()

    def step():
        return G.synthesis(ws, c=c, **kw)

    # e2e leg: ONE public call renders steps x world x 8 frames from pinned host ws / c; every batch's inputs are uploaded and
    # its uint8 frames gathered over the ranks and downloaded to pinned host memory inside the timed region (the download of
    # batch i overlaps the rendering of batch i+1 -- the frame loop of gen_videos.py as a pipeline).
    def e2e_inputs(steps):
        reps = steps * world
        return ws.cpu().repeat(reps, 1, 1).pin_memory(), c_host.repeat(reps, 1).pin_memory()

    def run_e2e(ws_pin, c_pin):
        return idist.stream_frames_sharded(G, ws_pin, c_pin, rank, world, batch=BATCH, **kw)

    with torch.no_grad():
        for _ in range(max(args.warmup, 3)):
            step()
        run_e2e(*e2e_inputs(2))
        barrier()

        # ---------------- value: device-resident inputs, per-iteration events, L2 flushed between iterations
        render.kernel_events = []
        launches0 = _lib.launch_count()
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
        with ClockSampler(device.index or 0) as clocks:
            barrier()
            torch.cuda.profiler.start()           # no-op unless run under `ncu --profile-from-start off`
            for i, (a, b) in enumerate(ev):
                if i == len(ev) - 1:
                    torch.manual_seed(0)          # the step's ray jitter seed is drawn from torch's generator: fix it for --dump-outputs
                flush.zero_()
                a.record()
                out = step()
                b.record()
            barrier()
            torch.cuda.profiler.stop()
        launches = _lib.launch_count() - launches0
        dev_ms = sum(a.elapsed_time(b) for a, b in ev)
        kern = render.kernel_events
        render.kernel_events = None
        kern_ms = float(np.mean([a.elapsed_time(b) for a, b, _ in kern]))

        # ---------------- e2e: host inputs, copies inside the timed region
        ws_pin, c_pin = e2e_inputs(args.steps)
        run_e2e(ws_pin, c_pin)                      # allocates the pinned result buffer of this size once
        barrier()
        t0 = time.perf_counter()
        frames_host = run_e2e(ws_pin, c_pin)        # returns after the last frame is in host memory
        barrier()
        e2e_wall = time.perf_counter() - t0
        assert rank != 0 or (frames_host.shape[0] == args.steps * world * BATCH and frames_host.device.type == 'cpu')

        # ---------------- renderer only (planes resident, channels-last): the kernel's own throughput per frame
        voxel_ws, _ = G.synthesis.split_ws(ws)
        img_v, seg_v = G.synthesis.backbone(voxel_ws, noise_mode='const')
        cam = c[:, :16].reshape(-1, 4, 4)
        ev3 = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
        for a, b in ev3:
            flush.zero_()
            a.record()
            G.synthesis.renderer(img_v, seg_v, cam, img_size=RENDER, num_steps=NUM_STEPS)   # planes as the backbone delivers them (NHWC: no layout pass; NCHW with IDE3D_CHANNELS_LAST=0: + 2 passes)
            b.record()
        torch.cuda.synchronize()
        renderer_ms = float(np.mean([a.elapsed_time(b) for a, b in ev3]))
        chain_ms = gpu_reference_chain_ms(G, img_v, seg_v, cam.reshape(-1, 4, 4)) if rank == 0 else None
        # one frame for the live parity check (same ws / camera / jitter seed as the CPU baseline's frame)
        img_parity = G.synthesis(ws[:1], c=c[:1], render_params=dict(num_steps=NUM_STEPS), noise_mode='const', perturb='hash', seed=1) if rank == 0 else None

    t = torch.tensor([dev_ms, e2e_wall * 1e3], dtype=torch.float64, device=device)
    if world > 1:
        tdist.all_reduce(t, op=tdist.ReduceOp.MAX)
    dev_ms, e2e_ms = float(t[0]), float(t[1])

    if rank == 0 and args.dump_outputs:
        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, 'image.npy'), out.float().cpu().numpy())

    if rank == 0:
        peak, peak_src = measured_peak_gbs()
        frames_total = BATCH * args.steps * world
        value = frames_total / (dev_ms * 1e-3)
        e2e_value = frames_total / (e2e_ms * 1e-3)
        achieved = BATCH * FRAME_ALGO_BYTES / (kern_ms * 1e-3) / 1e9
        traffic, traffic_src = raymarch_traffic()
        line = {
            'metric': METRIC, 'value': value, 'unit': 'frames/s', 'n_gpus': world, 'steps': args.steps, 'warmup': max(args.warmup, 3),
            'ms_per_step': dev_ms / args.steps, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
            'dtype': 'f32', 'data': 'synthetic',
            'config': {'workload': 'configs[1]: batch=8 latents, 64^2 neural render x 96 samples -> 512^2 SR, yaw sweep, '
                                   'random-init ide3d-ffhq-64-512 (TriPlaneGenerator seed 0)',
                       'frames_per_step_per_gpu': BATCH, 'plane': [96, PLANE, PLANE], 'l2': 'flushed (256 MB write) between timed iterations',
                       'timing': 'CUDA events per iteration on the launching stream, max over ranks', 'parallelism': f'frames sharded x{world}, no data-path collective'},
            'e2e': {'value': e2e_value, 'unit': 'frames/s', 'h2d_bytes_per_step': int((ws_pin.numel() * 4 + c_pin.numel() * 4) // args.steps),
                    'd2h_bytes_per_step': int(BATCH * world * 3 * 512 * 512), 'call': 'ide3d_b200.dist.stream_frames_sharded (pinned host ws/c -> uint8 frames in pinned host memory; D2H of batch i overlaps batch i+1)'},
            'gpu_launches': int(launches),
            'roofline': {'kernel': 'tc3::raymarch_tc3_kernel (fused gather + tcgen05 decoder MLP, compositing folded into the layer-2 operand)', 'bound': 'hbm', 'achieved': achieved, 'peak': peak, 'unit': 'GB/s',
                         'frac': achieved / peak, 'traffic': traffic, 'traffic_source': traffic_src, 'peak_source': peak_src, 'kernel_ms': kern_ms,
                         'algorithmic_bytes_per_launch': BATCH * FRAME_ALGO_BYTES,
                         'kernel_only_fps': BATCH / (kern_ms * 1e-3), 'renderer_fps_incl_layout_pass': BATCH / (renderer_ms * 1e-3),
                         'reference_gpu_chain_ms': chain_ms, 'vs_reference_gpu_chain': chain_ms / kern_ms,
                         'vs_reference_gpu_chain_note': 'reference renderer op chain (rays, jitter, bmm, 6x grid_sample, decoder matmuls, compositing; every stage in HBM) on this GPU, same planes and decoder, / kernel_ms; north-star target >= 20',
                         'note': 'HBM is not the limiter of this kernel: 24 texel lines per sample are served by L1/L2 and the kernel is gather-latency bound (profiles/r02k_ncu_raymarch_tc3.txt); frac is reported as the contract asks'},
            'clocks': clocks.summary(),
        }
        if not args.no_cpu_baseline and world == 1:
            pick_cpu_threads()
            Gc = build_generator('cpu')
            fps, sec, img_cpu = cpu_reference_fps(Gc, ws[:1].cpu(), c_host[:1], args.cpu_reps)
            diff = (img_parity.float().cpu() - img_cpu.float()).abs()
            q = lambda t: (t * 127.5 + 128).clamp(0, 255).to(torch.uint8).to(torch.int16)
            lv = (q(img_parity.float().cpu()) - q(img_cpu.float())).abs()
            line['parity'] = {'what': 'frame 0 of the batch, full synthesis (backbone -> 64^2x96 render -> 512^2), GPU (as benched: cuDNN TF32 convolutions) vs the CPU oracle (fp32)',
                              'image_max_abs_diff': float(diff.max()), 'image_max_abs_ref': float(img_cpu.abs().max()), 'uint8_max_levels': int(lv.max()),
                              'uint8_mean_levels': float(lv.float().mean()), 'tolerance': 'tests/test_gpu_fullsize.py: image 1e-2 x max|ref| under TF32 (1e-4 with fp32 convolutions)'}
            line['cpu_baseline'] = {'value': fps, 'unit': 'frames/s', 'cores': torch.get_num_threads(), 'kind': 'port',
                                    'sample': f'1 frame of the batch (full synthesis, {sec:.1f} s each, {args.cpu_reps} reps + 1 warm-up), oracle port on torch-CPU ops'}
        print(json.dumps(line))
    if world > 1:
        tdist.barrier()
        tdist.destroy_process_group()


if __name__ == '__main__':
    main()
