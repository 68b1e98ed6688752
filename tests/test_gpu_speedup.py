"""North-star target (BASELINE.json): the fused ray-march >= 20x the reference renderer's single-GPU frames/s at
64^2 x 96 samples.  The "reference renderer on the GPU" is the reference's own op chain -- a1 rays, a2 jitter,
a3 cam2world bmm, a5 F.grid_sample x 6, decoder matmuls, a7 compositing -- executed by the oracle on CUDA tensors
(every stage materialised in HBM, as volumetric_rendering.py does).  The measured ratio is printed (pytest -s).
Round-1 status: 11.0x measured on B200 (composed chain 16.6 ms, fused 1.51 ms per 8 frames) -- the 20x target is NOT met yet; the assertion below only guards the measured level against regressions."""

import json

import pytest
import torch

pytestmark = pytest.mark.gpu


def _composed_on_device(R, planes_tex, planes_seg, dec, cam, S, u):
    with torch.device('cuda'):                       # the oracle's factory calls (linspace/ones/zeros) land on the GPU
        pts, zv, d = R.initial_rays(planes_tex.shape[0], S, 18.0, (64, 64), 2.25, 3.3)
        pts, zv = R.perturb(pts, zv, d, u)
        pw, dw, ow = R.to_world(pts, d, cam)
        coords = pw.reshape(planes_tex.shape[0], -1, 3) * 2.0
        f_tex = R.sample_triplane_torch(coords, planes_tex)
        f_seg = R.sample_triplane_torch(coords, planes_seg)
        out = dec(f_tex, f_seg).reshape(planes_tex.shape[0], 64 * 64, S, R.N_OUT)
        return R.composite(out, d, zv, clamp_mode='softplus')


def test_fused_renderer_vs_composed_reference_chain_on_gpu():
    from oracle import renderer as R
    from ide3d_b200 import render
    from test_gpu_renderer import _random_case, three_head_from_dense

    N, S = 8, 96
    dev = torch.device('cuda')
    tex, seg, dec, cam = _random_case(N, 256, seed=21)              # band-limited 256^2 planes, three-head decoder, yaw sweep
    pdec = render.PackedDecoder(three_head_from_dense(dec.w1, dec.b1, dec.w2, dec.b2), dev)
    tex, seg, cam = tex.to(dev), seg.to(dev), cam.to(dev)
    for k in ('w1', 'b1', 'w2', 'b2'):
        setattr(dec, k, getattr(dec, k).to(dev))
    u = torch.rand(N, 4096, S, 1, device=dev)
    tex_cl, seg_cl = render.as_planes(tex), render.as_planes(seg)

    def fused():
        return render.raymarch(tex_cl, seg_cl, pdec, cam, resolution=(64, 64), num_steps=S, jitter_u=u.reshape(N, 4096, S),
                               clamp_mode='softplus', convert_layout=False)

    def timed(fn, reps, warm):
        for _ in range(warm):
            fn()
        torch.cuda.synchronize()
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0.record()
        for _ in range(reps):
            r = fn()
        t1.record()
        torch.cuda.synchronize()
        return t0.elapsed_time(t1) / reps, r

    ms_ref, (rgb_ref, depth_ref, _) = timed(lambda: _composed_on_device(R, tex, seg, dec, cam, S, u), 3, 1)
    ms_fused, (feat, depth, _) = timed(fused, 20, 3)
    err = (feat - rgb_ref).abs().max().item()
    ratio = ms_ref / ms_fused
    rec = dict(frames=N, num_steps=S, composed_reference_chain_ms=ms_ref, fused_ms=ms_fused, speedup=ratio,
               composed_fps=N / ms_ref * 1e3, fused_fps=N / ms_fused * 1e3, max_abs_feature_diff=err)
    print(json.dumps(rec))
    assert err < 3e-4
    assert (depth.reshape(N, -1) - depth_ref.reshape(N, -1)).abs().max().item() < 1e-4
    assert ratio >= 8.0, rec          # north-star target is 20; see the module docstring
