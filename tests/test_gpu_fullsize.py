"""Parity AT THE TIMED CONFIGURATION (BASELINE configs[1]; VERDICT r1 "what's weak" #1, #3).

bench.py times the full-size random-init ide3d-ffhq-64-512 generator (256^2 x 96-channel tri-planes, 64^2 rays x 96 samples,
512^2 output) with cuDNN's default TF32 convolutions.  The whole-path test in test_gpu_generator.py runs a reduced generator
with TF32 off, so it does not describe the benched arithmetic.  Here the SAME generator object bench.py builds
(compat.random_init_generator(seed=0)) renders two frames of the bench's yaw sweep on the GPU and on the CPU oracle
(oracle.backend.cpu_reference_ops: reference NCHW layout, reference op chain, fp32), stage by stage:

    planes   : backbone output img_v / seg_v                                    (cuDNN convs + this package's FIR / epilogues)
    render   : fused ray-march on IDENTICAL planes (the oracle's) -> feat / depth / weights   (sigma enters through weights)
    image    : final 512^2 image and the uint8 frame

twice: cudnn.allow_tf32 = False (fp32 convolutions; tight tolerances) and the bench's default TF32 (stated tolerances).
Tolerances are relative to max|reference tensor| and were set from the errors measured on B200 (printed by the test,
pytest -s; bench.py repeats the one-frame comparison live and reports it as `parity`).

Also here: the 256^3 sigma grid of extract_shapes.py (config 4) as a TEST (it was a builder-run script in round 1): the
in-kernel point generator reproduces create_samples' float-division quirk bit for bit at full size, slabs concatenate to
the whole grid bit for bit; and one config-5-sized op tensor (512 ch x 512^2) through parity asserts."""

import json
import math
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

# relative tolerances (x max|ref|): (fp32 convolutions, TF32 convolutions)
# measured on B200 (profiles/r02a_parity_fullsize_and_determinism.txt): fp32 planes 2.6e-6, feat 6.3e-6, depth 9.1e-7, weights 3.6e-6,
# image 1.1e-5, uint8 <= 1 level;  TF32 (the benched arithmetic) planes 8.6e-4, image 2.1e-3, uint8 <= 2 levels (mean 0.08)
TOL = {
    'planes': (3e-5, 5e-3),
    'feat': (1e-4, 1e-4),        # renderer on identical planes: independent of the convolution precision
    'depth': (1e-5, 1e-5),
    'weights': (5e-5, 5e-5),
    'image': (1e-4, 1e-2),
}


def _labels(n):
    from bench import make_labels
    return make_labels(8)[[0, 7][:n]]


@pytest.fixture(scope='module')
def fullsize():
    from bench import NUM_STEPS, make_latents
    from ide3d_b200.compat import random_init_generator
    from oracle.backend import cpu_reference_ops
    torch.set_num_threads(min(32, os.cpu_count() or 8))
    G = random_init_generator(device='cpu', seed=0)
    n = 2
    z, c = make_latents(n, G.z_dim), _labels(n)
    kw = dict(noise_mode='const')
    with torch.no_grad(), cpu_reference_ops():
        ws = G.mapping(z, c)
        voxel_ws, block_ws = G.synthesis.split_ws(ws)
        img_v, seg_v = G.synthesis.backbone(voxel_ws, **kw)
        cam = c[:, :16].reshape(-1, 4, 4)
        feat, depth, weights = G.synthesis.renderer(img_v, seg_v, cam, img_size=64, num_steps=NUM_STEPS, perturb='hash', seed=7,
                                                    return_weights=True)
        out = G.synthesis(ws, c=c, render_params=dict(num_steps=NUM_STEPS), perturb='hash', seed=7, return_dict=True, **kw)
    ref = dict(img_v=img_v, seg_v=seg_v, feat=feat, depth=depth, weights=weights, image=out['image'], image_depth=out['image_depth'])
    return G, ws, c, ref, NUM_STEPS


def _rel(a, b):
    a, b = a.detach().float().cpu(), b.detach().float().cpu()
    return (a - b).abs().max().item() / max(1e-12, b.abs().max().item())


@pytest.mark.parametrize('tf32', [False, True])
def test_fullsize_synthesis_matches_cpu_oracle(fullsize, tf32):
    G, ws, c, ref, S = fullsize
    col = 1 if tf32 else 0
    saved = torch.backends.cudnn.allow_tf32
    Gd = G.cuda()
    rep = {}
    try:
        torch.backends.cudnn.allow_tf32 = tf32
        with torch.no_grad():
            wsd, cd = ws.cuda(), c.cuda()
            voxel_ws, _ = Gd.synthesis.split_ws(wsd)
            img_v, seg_v = Gd.synthesis.backbone(voxel_ws, noise_mode='const')
            rep['planes'] = max(_rel(img_v, ref['img_v']), _rel(seg_v, ref['seg_v']))
            cam = cd[:, :16].reshape(-1, 4, 4)
            # renderer on the oracle's own planes: isolates the fused kernel from the convolution precision
            feat, depth, weights = Gd.synthesis.renderer(ref['img_v'].cuda(), ref['seg_v'].cuda(), cam, img_size=64, num_steps=S,
                                                         perturb='hash', seed=7, return_weights=True)
            rep['feat'], rep['depth'], rep['weights'] = _rel(feat, ref['feat']), _rel(depth, ref['depth']), _rel(weights, ref['weights'])
            out = Gd.synthesis(wsd, c=cd, render_params=dict(num_steps=S), perturb='hash', seed=7, return_dict=True, noise_mode='const')
            rep['image'] = _rel(out['image'], ref['image'])
            to8 = lambda t: (t.float().cpu() * 127.5 + 128).clamp(0, 255).to(torch.uint8).int()
            d8 = (to8(out['image']) - to8(ref['image'])).abs()
            rep['uint8_max_levels'], rep['uint8_mean_levels'] = int(d8.max()), float(d8.float().mean())
    finally:
        torch.backends.cudnn.allow_tf32 = saved
        G.cpu()
    print('full-size parity', 'tf32' if tf32 else 'fp32', json.dumps(rep))
    for k, tol in TOL.items():
        assert rep[k] <= tol[col], (k, rep, tol[col])
    assert rep['uint8_max_levels'] <= (1 if not tf32 else 6), rep


def test_sigma_grid_256_is_bit_identical_to_create_samples_path(fullsize):
    """config 4: ide3d_sigma_grid generates 0.9 * create_samples(256, [0,0,0], 1.0) in the kernel (extract_shapes.py:84-86,
    :102-103, the fractional y/x voxel indices included); the explicit-points path through sample_voxel must give the SAME
    bits, and z-slabs (dist.sigma_grid_sharded's partition) must concatenate to the whole grid bit for bit."""
    from ide3d_b200 import dist as idist
    from oracle import renderer as orr
    G, ws, c, ref, S = fullsize
    Gd = G.cuda()
    try:
        with torch.no_grad():
            R = Gd.synthesis.renderer
            tex, seg = R.as_planes(ref['img_v'][:1].cuda()), R.as_planes(ref['seg_v'][:1].cuda())
            N = 256
            whole = R.sigma_grid(tex, seg, grid_n=N, cube_length=1.0)
            pts, _, _ = orr.create_samples(N, [0, 0, 0], 1.0)
            pts = (0.9 * pts).cuda()
            explicit = torch.empty(1, N ** 3, device='cuda')
            step = 1 << 22
            for h in range(0, N ** 3, step):
                explicit[:, h:h + step] = R.sample_voxel(tex, seg, pts[:, h:h + step], sigma_only=True)[..., 0]
            assert torch.equal(whole, explicit)
            parts = []
            for r in range(8):
                first, count = idist.slab_range(N ** 3, r, 8)
                parts.append(R.sigma_grid(tex, seg, grid_n=N, cube_length=1.0, first=first, count=count))
            assert torch.equal(torch.cat(parts, dim=-1), whole)
            # and against the CPU oracle on a strided sample of the grid (the full 16.7 M-point oracle pass takes minutes)
            sel = torch.arange(0, N ** 3, 4099)
            cpu = orr.sample_voxel(ref['img_v'][:1], ref['seg_v'][:1], __import__('oracle.backend', fromlist=['x'])._decoder_from_renderer(G.cpu().synthesis.renderer),
                                   pts[:, sel].cpu(), 2.0)[..., -1]
            assert (whole[:, sel].cpu() - cpu).abs().max().item() <= 3e-5 * max(1.0, cpu.abs().max().item())
    finally:
        G.cpu()


@pytest.mark.parametrize('layout', ['contiguous', 'channels_last'])
def test_config5_sized_ops_parity(layout):
    """One 512-channel x 512^2 tensor (config 5) through upfirdn2d (up / down / filter) and bias_act against the oracle on a
    channel subset (the oracle ops are per-channel independent: checking 8 of the 512 channels of the full-size call pins the
    full-size launch configuration -- grid sizes, tile maps, 32-bit index math -- at a CPU cost of seconds)."""
    from ide3d_b200.torch_utils.ops import bias_act, upfirdn2d
    from oracle import ops as oops
    g = torch.Generator().manual_seed(0)
    x = torch.randn(1, 512, 512, 512, generator=g)
    b = torch.randn(512, generator=g)
    xd = x.cuda()
    if layout == 'channels_last':
        xd = xd.contiguous(memory_format=torch.channels_last)
    f = oops.setup_filter([1, 3, 3, 1])
    fd = f.cuda()
    ch = torch.tensor([0, 1, 63, 64, 255, 256, 510, 511])
    xs = x[:, ch]
    cases = {
        'upsample2d': (lambda: upfirdn2d.upsample2d(xd, fd), lambda: oops.upsample2d(xs, f)),
        'downsample2d': (lambda: upfirdn2d.downsample2d(xd, fd), lambda: oops.downsample2d(xs, f)),
        'filter2d': (lambda: upfirdn2d.filter2d(xd, fd), lambda: oops.filter2d(xs, f)),
        'bias_act': (lambda: bias_act.bias_act(xd, b.cuda(), act='lrelu', clamp=256), lambda: oops.bias_act(xs, b[ch], 1, 'lrelu', None, None, 256)),
    }
    for name, (ours, orc) in cases.items():
        y = ours()[:, ch.cuda()].float().cpu()
        r = orc()
        assert y.shape == r.shape, name
        err = (y - r).abs().max().item()
        assert err <= 2e-5 * max(1.0, r.abs().max().item()), (name, layout, err)
        del y
        torch.cuda.empty_cache()
