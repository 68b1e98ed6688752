#!/usr/bin/env python
"""Generate tests/golden/*.npz by running the REFERENCE's own Python functions (imported read-only
from /root/reference) on small seeded inputs, and assert on the spot that oracle/ reproduces them.

Run in the build container only (the GPU box has no /root/reference):

    PYTHONDONTWRITEBYTECODE=1 python tests/golden/make_golden.py

The committed .npz files are the contract that tests/test_oracle_golden.py (CPU) and the -m gpu parity
tests replay.  The reference ships no tests or golden vectors of its own (SURVEY.md §4), so these
recorded reference outputs are what pins the oracle.
"""

import ast
import math
import os
import sys

import numpy as np
import torch

REF = '/root/reference'
HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.dont_write_bytecode = True
sys.path.insert(0, REF)
sys.path.insert(1, ROOT)

from training import volumetric_rendering as ref_vr            # noqa: E402  (reference)
from dnnlib.util import sample_from_triplane as ref_triplane    # noqa: E402
from torch_utils.ops import upfirdn2d as ref_up                 # noqa: E402
from torch_utils.ops import bias_act as ref_ba                  # noqa: E402
from torch_utils.ops import filtered_lrelu as ref_fl            # noqa: E402
from torch_utils.ops import conv2d_resample as ref_cr           # noqa: E402

import oracle                                                    # noqa: E402
from oracle import renderer as orr, ops as oops, camera as ocam  # noqa: E402

DEV = torch.device('cpu')


def t2n(d):
    return {k: (v.detach().numpy() if isinstance(v, torch.Tensor) else np.asarray(v)) for k, v in d.items()}


def save(name, **arrs):
    path = os.path.join(HERE, name + '.npz')
    np.savez_compressed(path, **t2n(arrs))
    print(f'{name:24s} {os.path.getsize(path) / 1024:8.1f} KB')


def close(a, b, tol=2e-6, what=''):
    a = torch.as_tensor(a).double()
    b = torch.as_tensor(b).double()
    err = (a - b).abs().max().item() if a.numel() else 0.0
    assert a.shape == b.shape and err <= tol, f'{what}: shape {tuple(a.shape)} vs {tuple(b.shape)} err {err:g}'
    return err


# ------------------------------------------------------------------ a1 rays
def g_rays():
    for tag, (n, S, fov, res, rs, re) in {'a': (2, 6, 18.0, (8, 8), 2.25, 3.3), 'b': (1, 5, 30.0, (6, 4), 0.5, 1.5)}.items():
        p, z, d = ref_vr.get_initial_rays_trig(n, S, DEV, fov, res, rs, re)
        po, zo, do = orr.initial_rays(n, S, fov, res, rs, re)
        close(p, po, what='rays.points'); close(z, zo, what='rays.z'); close(d, do, what='rays.d')
        save(f'rays_{tag}', n=n, num_steps=S, fov=fov, resolution=np.array(res), ray_start=rs, ray_end=re,
             points=p, z_vals=z, rays_d_cam=d)


# ------------------------------------------------------------------ a2+a3 jitter + world transform
def g_transform():
    n, S, res = 2, 6, (8, 8)
    p, z, d = ref_vr.get_initial_rays_trig(n, S, DEV, 18.0, res, 2.25, 3.3)
    cam = torch.from_numpy(ocam.look_at_pose(np.array([[1.2], [1.9]], np.float32), np.array([[1.4], [1.7]], np.float32),
                                             [0, 0, 0.2], radius=2.7, batch_size=2))
    torch.manual_seed(123)
    u = torch.rand(z.shape)                      # what perturb_points will draw first (:101)
    torch.manual_seed(123)
    pw, zj, dw, ow, _pitch, _yaw = ref_vr.transform_sampled_points(p, z, d, DEV, camera=cam)
    pj, zo = orr.perturb(p, z, d, u)
    pwo, dwo, owo = orr.to_world(pj, d, cam)
    close(zj, zo, what='xf.z'); close(pw, pwo, what='xf.pw'); close(dw, dwo, what='xf.dw'); close(ow, owo, what='xf.ow')
    save('transform', points=p, z_vals=z, rays_d_cam=d, camera=cam, u=u, points_world=pw, z_jit=zj,
         dirs_world=dw, origins_world=ow)


# ------------------------------------------------------------------ a4 cameras
def g_camera():
    hs = np.array([math.pi / 2, 1.1, 2.0], np.float32)
    vs = np.array([math.pi / 2, 1.3, 1.9], np.float32)
    out = {}
    for i, (h, v) in enumerate(zip(hs, vs)):
        o, phi, th = ref_vr.sample_camera_positions(DEV, n=1, r=2.7, horizontal_mean=float(h), vertical_mean=float(v), mode=None)
        oo, _, _ = ocam.sample_camera_positions(n=1, r=2.7, horizontal_mean=float(h), vertical_mean=float(v), mode=None)
        close(o, oo, what='cam.origin')
        m = ref_vr.create_cam2world_matrix(-o, o, device=DEV)
        close(m, ocam.create_cam2world_matrix(-oo, oo), what='cam.c2w')
        la = ref_vr.LookAtPoseSampler.sample(float(h), float(v), torch.tensor([0, 0, 0.2]), radius=2.7)
        close(la, ocam.look_at_pose(float(h), float(v), [0, 0, 0.2], radius=2.7), what='cam.lookat')
        out[f'origin{i}'] = o; out[f'c2w{i}'] = m; out[f'lookat{i}'] = la
    save('camera', h=hs, v=vs, radius=2.7, lookat=np.array([0, 0, 0.2], np.float32), **out)


# ------------------------------------------------------------------ a5 tri-plane gather
def g_triplane():
    g = torch.Generator().manual_seed(7)
    grid = torch.randn(2, 96, 12, 12, generator=g)
    coords = (torch.rand(2, 300, 3, generator=g) * 2.6 - 1.3)      # includes out-of-range taps
    coords[0, :4] = torch.tensor([[-1., -1., -1.], [1., 1., 1.], [0., 0., 0.], [0.999, -0.999, 0.5]])
    f = ref_triplane(coords, grid)
    close(f, orr.sample_triplane(coords, grid), tol=3e-6, what='triplane')
    close(f, orr.sample_triplane_torch(coords, grid), tol=1e-6, what='triplane_torch')
    save('triplane', grid=grid, coords=coords, feat=f)


# ------------------------------------------------------------------ a7 compositing
def g_integration():
    g = torch.Generator().manual_seed(11)
    n, R, S, C = 2, 10, 12, 52
    rgb_sigma = torch.randn(n, R, S, C, generator=g)
    rgb_sigma[..., -1] *= 4
    z = torch.sort(torch.rand(n, R, S, 1, generator=g) * 1.05 + 2.25, dim=2)[0]
    d = torch.randn(n, R, 3, generator=g)
    cases = {
        'softplus': dict(clamp_mode='softplus'),
        'relu': dict(clamp_mode='relu'),
        'lastback': dict(clamp_mode='softplus', last_back=True),
        'white': dict(clamp_mode='softplus', white_back=True, max_depth=3.5),
        'fillw': dict(clamp_mode='relu', fill_mode='weight'),
    }
    out = {}
    for k, kw in cases.items():
        rgb, dep, w = ref_vr.fancy_integration(rgb_sigma.clone(), d, z, DEV, noise_std=0, **kw)
        ro, do_, wo = orr.composite(rgb_sigma.clone(), d, z, **kw)
        close(rgb, ro, tol=5e-6, what=k + '.rgb'); close(dep, do_, tol=5e-6, what=k + '.depth'); close(w, wo, what=k + '.w')
        out[k + '_rgb'] = rgb; out[k + '_depth'] = dep; out[k + '_weights'] = w
    save('integration', rgb_sigma=rgb_sigma, z_vals=z, rays_d_cam=d, **out)


# ------------------------------------------------------------------ a8 importance sampling
def g_pdf():
    g = torch.Generator().manual_seed(5)
    R, S = 9, 12
    z = torch.sort(torch.rand(R, S, generator=g) + 2, dim=1)[0]
    bins = 0.5 * (z[:, :-1] + z[:, 1:])            # [R, S-1]
    w = torch.rand(R, S - 2, generator=g)
    w[3] = 0                                        # a ray with zero weights
    det = ref_vr.sample_pdf(bins, w, 8, det=True)
    close(det, orr.sample_pdf(bins, w, 8, det=True), what='pdf.det')
    torch.manual_seed(77)
    u = torch.rand(R, 8)
    torch.manual_seed(77)
    rnd = ref_vr.sample_pdf(bins, w, 8, det=False)
    close(rnd, orr.sample_pdf(bins, w, 8, det=False, u=u), what='pdf.rand')
    save('sample_pdf', bins=bins, weights=w, det=det, u=u, rnd=rnd)


# ------------------------------------------------------------------ composed chain (reference functions + decoder)
def g_chain():
    g = torch.Generator().manual_seed(3)
    n, S, res = 2, 12, (8, 8)
    tex = torch.randn(n, 96, 16, 16, generator=g)
    seg = torch.randn(n, 96, 16, 16, generator=g)
    dec = orr.Decoder.random(hidden=64, seed=4, three_head=True)      # the fused kernel's three-head shape
    cam = torch.from_numpy(ocam.look_at_pose(np.array([[1.3], [1.8]], np.float32), np.array([[1.5], [1.65]], np.float32),
                                             [0, 0, 0.2], radius=2.7, batch_size=2))
    box_scale = 2.0
    p, z, d = ref_vr.get_initial_rays_trig(n, S, DEV, 18.0, res, 2.25, 3.3)
    torch.manual_seed(9)
    u = torch.rand(z.shape)
    torch.manual_seed(9)
    pw, zj, dw, ow, _, _ = ref_vr.transform_sampled_points(p, z, d, DEV, camera=cam)
    coords = pw.reshape(n, -1, 3) * box_scale
    ft = ref_triplane(coords, tex)
    fs = ref_triplane(coords, seg)
    raw = dec(ft, fs).reshape(n, res[0] * res[1], S, 52)
    rgb, dep, w = ref_vr.fancy_integration(raw, d, zj, DEV, noise_std=0, clamp_mode='softplus')
    ro, do_, wo = orr.render_frames(tex, seg, dec, cam, fov=18.0, num_steps=S, ray_start=2.25, ray_end=3.3,
                                    resolution=res, box_scale=box_scale, jitter_u=u)
    close(rgb, ro, tol=1e-5, what='chain.rgb'); close(dep, do_, tol=1e-5, what='chain.depth'); close(w, wo, tol=1e-5, what='chain.w')
    save('chain', planes_tex=tex, planes_seg=seg, w1=dec.w1, b1=dec.b1, w2=dec.w2, b2=dec.b2, camera=cam, u=u,
         box_scale=box_scale, num_steps=S, resolution=np.array(res), rgb=rgb, depth=dep, weights=w,
         raw=raw, points_world=pw)
    # same inputs through a dense 64 -> 64 -> 52 decoder (the fused kernel's single-head shape)
    dd = orr.Decoder.random(hidden=64, seed=6, three_head=False)
    rawd = dd(ft, fs).reshape(n, res[0] * res[1], S, 52)
    rgbd, depd, wd = ref_vr.fancy_integration(rawd, d, zj, DEV, noise_std=0, clamp_mode='relu', last_back=True)
    rod, dod, wod = orr.render_frames(tex, seg, dd, cam, fov=18.0, num_steps=S, ray_start=2.25, ray_end=3.3,
                                      resolution=res, box_scale=box_scale, jitter_u=u, clamp_mode='relu', last_back=True)
    close(rgbd, rod, tol=1e-5, what='chain_dense.rgb'); close(depd, dod, tol=1e-5, what='chain_dense.depth'); close(wd, wod, tol=1e-5, what='chain_dense.w')
    save('chain_dense', w1=dd.w1, b1=dd.b1, w2=dd.w2, b2=dd.b2, rgb=rgbd, depth=depd, weights=wd)
    # sigma-only voxel query on the same planes (sample_voxel contract, extract_shapes.py:146)
    pts = torch.rand(n, 50, 3, generator=g) - 0.5
    sv = dec(ref_triplane(pts * box_scale, tex), ref_triplane(pts * box_scale, seg)).reshape(n, 50, 52)
    close(sv, orr.sample_voxel(tex, seg, dec, pts, box_scale), tol=1e-5, what='voxel')
    save('voxel', points=pts, out=sv)


# ------------------------------------------------------------------ two-pass chain: every stage a reference function
def g_chain_hier():
    """The reference tree has sample_pdf (volumetric_rendering.py:224-265) but no caller, so the ORDER below is ours
    (the one its docstring prescribes); every stage in it -- rays, jitter, world transform, tri-plane gather, compositing,
    sample_pdf -- is the reference's own function run here."""
    g = torch.Generator().manual_seed(21)
    n, S, NI, res = 2, 12, 12, (8, 8)
    R = res[0] * res[1]
    # band-limited planes (generator planes are smooth): the fine depths are a function of the coarse weights, and white noise would
    # turn their 1e-6-level differences into feature differences that measure the input's slope, not the implementation
    smooth = lambda: torch.nn.functional.interpolate(torch.randn(n, 96, 6, 6, generator=g), size=(16, 16), mode='bicubic',
                                                     align_corners=True).contiguous()
    tex, seg = smooth(), smooth()
    dec = orr.Decoder.random(hidden=64, seed=8, three_head=True)
    cam = torch.from_numpy(ocam.look_at_pose(np.array([[1.45], [1.7]], np.float32), np.array([[1.55], [1.6]], np.float32),
                                             [0, 0, 0.2], radius=2.7, batch_size=2))
    box_scale = 2.0
    p, z, d = ref_vr.get_initial_rays_trig(n, S, DEV, 18.0, res, 2.25, 3.3)
    torch.manual_seed(31)
    u = torch.rand(z.shape)
    torch.manual_seed(31)
    pw, zj, dw, ow, _, _ = ref_vr.transform_sampled_points(p, z, d, DEV, camera=cam)
    coords = pw.reshape(n, -1, 3) * box_scale
    raw = dec(ref_triplane(coords, tex), ref_triplane(coords, seg)).reshape(n, R, S, 52)
    _, _, w = ref_vr.fancy_integration(raw, d, zj, DEV, noise_std=0, clamp_mode='softplus')
    zf = zj.reshape(n * R, S)
    mid = 0.5 * (zf[:, :-1] + zf[:, 1:])
    torch.manual_seed(41)
    ui = torch.rand(n * R, NI)
    torch.manual_seed(41)
    fine = ref_vr.sample_pdf(mid, w.reshape(n * R, S)[:, 1:-1] + 1e-5, NI, det=False).detach().reshape(n, R, NI, 1)
    fine_pts = ow.unsqueeze(2) + dw.unsqueeze(2) * fine
    cf = fine_pts.reshape(n, -1, 3) * box_scale
    raw_f = dec(ref_triplane(cf, tex), ref_triplane(cf, seg)).reshape(n, R, NI, 52)
    all_z, idx = torch.sort(torch.cat([zj, fine], -2), dim=-2)
    all_raw = torch.gather(torch.cat([raw, raw_f], -2), -2, idx.expand(-1, -1, -1, 52))
    rgb, dep, wa = ref_vr.fancy_integration(all_raw, d, all_z, DEV, noise_std=0, clamp_mode='softplus')
    ro, do_, wo, zo = orr.render_frames_hierarchical(tex, seg, dec, cam, fov=18.0, num_steps=S, n_importance=NI, ray_start=2.25,
                                                     ray_end=3.3, resolution=res, box_scale=box_scale, jitter_u=u, importance_u=ui)
    close(all_z, zo, tol=2e-6, what='hier.z'); close(rgb, ro, tol=1e-5, what='hier.rgb')
    close(dep, do_, tol=1e-5, what='hier.depth'); close(wa, wo, tol=1e-5, what='hier.w')
    save('chain_hier', planes_tex=tex, planes_seg=seg, w1=dec.w1, b1=dec.b1, w2=dec.w2, b2=dec.b2, camera=cam, u=u, importance_u=ui,
         box_scale=box_scale, num_steps=S, n_importance=NI, resolution=np.array(res), fine=fine, z_all=all_z, rgb=rgb, depth=dep,
         weights=wa)


# ------------------------------------------------------------------ create_samples quirk
def g_create_samples():
    src = open(os.path.join(REF, 'extract_shapes.py')).read()
    fn = [n for n in ast.parse(src).body if isinstance(n, ast.FunctionDef) and n.name == 'create_samples'][0]
    ns = {'np': np, 'torch': torch}
    exec(compile(ast.Module([fn], []), 'extract_shapes.py', 'exec'), ns)     # run the reference's own function
    s, origin, vs = ns['create_samples'](N=8, voxel_origin=[0, 0, 0], cube_length=1.0)
    so, oo, vo = orr.create_samples(8, [0, 0, 0], 1.0)
    close(s, so, what='create_samples')
    save('create_samples', N=8, cube_length=1.0, samples=s, origin=origin, voxel_size=vs)


# ------------------------------------------------------------------ ops
def g_bias_act():
    g = torch.Generator().manual_seed(21)
    x = torch.randn(3, 5, 4, 6, generator=g) * 3
    b = torch.randn(5, generator=g)
    out = {}
    for act in ref_ba.activation_funcs:
        for tag, kw in {'d': {}, 'c': dict(alpha=0.3, gain=1.7, clamp=0.9)}.items():
            y = ref_ba.bias_act(x, b, dim=1, act=act, impl='ref', **kw)
            close(y, oops.bias_act(x, b, 1, act, **kw), what=f'bias_act.{act}.{tag}')
            out[f'{act}_{tag}'] = y
    xl = torch.randn(7, 5, generator=g)
    out['dim1_2d'] = ref_ba.bias_act(xl, b, dim=1, act='lrelu', impl='ref')
    out['nobias'] = ref_ba.bias_act(x, None, act='swish', impl='ref')
    save('bias_act', x=x, b=b, x2d=xl, **out)


UPFIR_CASES = {
    # name: (filter taps or 2-D, up, down, padding, flip, gain)
    'up2_4x4': ([1, 3, 3, 1], 2, 1, [2, 1, 2, 1], False, 4.0),
    'down2_4x4': ([1, 3, 3, 1], 1, 2, [1, 1, 1, 1], False, 1.0),
    'filt_4x4': ([1, 3, 3, 1], 1, 1, [1, 1, 1, 1], False, 4.0),     # the conv-up post filter
    'filt_flip': ([1, 2, 4, 3], 1, 1, [2, 1, 2, 1], True, 1.0),
    'asym': ([[1, 2, 0], [0, 3, 1]], (2, 1), (1, 2), [3, 0, -1, 2], False, 0.5),
    'sep8': ([1, 2, 3, 4, 4, 3, 2, 1], 2, 2, [3, 4, 4, 3], False, 1.0),
    'up4_down1': ([1, 4, 6, 4, 1], (4, 4), (1, 1), [2, 2, 2, 2], False, 16.0),
    'crop': ([1, 1], 1, 1, [-1, -2, 0, -1], False, 1.0),
    'ident': (None, 1, 1, 0, False, 1.0),
}


def g_upfirdn2d():
    g = torch.Generator().manual_seed(31)
    x = torch.randn(2, 3, 9, 7, generator=g)
    out = {}
    for name, (taps, up, down, pad, flip, gain) in UPFIR_CASES.items():
        f = None if taps is None else ref_up.setup_filter(taps)
        if f is not None:
            close(f, oops.setup_filter(taps), what='setup_filter.' + name)
        y = ref_up.upfirdn2d(x, f, up=up, down=down, padding=pad, flip_filter=flip, gain=gain, impl='ref')
        close(y, oops.upfirdn2d(x, f, up=up, down=down, padding=pad, flip_filter=flip, gain=gain), tol=3e-6, what='upfirdn2d.' + name)
        if f is not None and f.ndim == 2:
            upp = (up, up) if isinstance(up, int) else up
            dnn = (down, down) if isinstance(down, int) else down
            close(y, oops.upfirdn2d_direct(x, f, upp, dnn, oops._pad4(pad), flip, gain), tol=3e-6, what='direct.' + name)
        out[name] = y
        if f is not None:
            out[name + '_f'] = f
    f = ref_up.setup_filter([1, 3, 3, 1])
    out['upsample2d'] = ref_up.upsample2d(x, f, impl='ref'); close(out['upsample2d'], oops.upsample2d(x, f), tol=3e-6, what='upsample2d')
    out['downsample2d'] = ref_up.downsample2d(x, f, impl='ref'); close(out['downsample2d'], oops.downsample2d(x, f), tol=3e-6, what='downsample2d')
    out['filter2d'] = ref_up.filter2d(x, f, impl='ref'); close(out['filter2d'], oops.filter2d(x, f), tol=3e-6, what='filter2d')
    save('upfirdn2d', x=x, **out)


def g_filtered_lrelu():
    import scipy.signal
    g = torch.Generator().manual_seed(41)
    x = torch.randn(2, 3, 16, 16, generator=g) * 2
    b = torch.randn(3, generator=g)
    f12 = torch.as_tensor(scipy.signal.firwin(numtaps=12, cutoff=0.25, width=0.5), dtype=torch.float32)
    f2d = torch.outer(f12[:8], f12[:8]); f2d = f2d / f2d.sum()
    cases = {
        'su2_sd2': dict(fu=f12 * 2 ** 0, fd=f12, up=2, down=2, padding=[5, 6, 5, 6], clamp=1.5),
        'su2_sd1': dict(fu=f12, fd=None, up=2, down=1, padding=[5, 6, 5, 6], clamp=None),
        'su1_sd2': dict(fu=None, fd=f12, up=1, down=2, padding=[5, 6, 5, 6], clamp=2.0, slope=0.1, gain=1.3),
        'fu2_fd2': dict(fu=f2d, fd=f2d, up=2, down=2, padding=[7, 8, 7, 8], clamp=1.0, flip_filter=True),
        'su4_sd2': dict(fu=torch.cat([f12, f12]) / 2, fd=f12, up=4, down=2, padding=[17, 18, 17, 18], clamp=0.8),
        'plain': dict(fu=None, fd=None, up=1, down=1, padding=0, clamp=0.7),
    }
    out = {}
    for k, kw in cases.items():
        y = ref_fl.filtered_lrelu(x, b=b, impl='ref', **kw)
        close(y, oops.filtered_lrelu(x, b=b, **kw), tol=5e-6, what='flrelu.' + k)
        out[k] = y
        for a in ('fu', 'fd'):
            if kw[a] is not None:
                out[f'{k}_{a}'] = kw[a]
    save('filtered_lrelu', x=x, b=b, **out)


def g_conv2d_resample():
    g = torch.Generator().manual_seed(51)
    x = torch.randn(2, 4, 8, 8, generator=g)
    w3 = torch.randn(6, 4, 3, 3, generator=g)
    w1 = torch.randn(6, 4, 1, 1, generator=g)
    wg = torch.randn(6, 2, 3, 3, generator=g)
    f = ref_up.setup_filter([1, 3, 3, 1])
    cases = {
        'up2_k3': dict(w=w3, f=f, up=2, padding=1, flip_weight=False),
        'up2_k3_g2': dict(w=wg, f=f, up=2, padding=1, groups=2, flip_weight=False),
        'same_k3': dict(w=w3, padding=1),
        'down2_k3': dict(w=w3, f=f, down=2, padding=1),
        'up2_k1': dict(w=w1, f=f, up=2),
        'down2_k1': dict(w=w1, f=f, down=2),
    }
    out = {}
    for k, kw in cases.items():
        y = ref_cr.conv2d_resample(x, **kw)
        close(y, oops.conv2d_resample(x, **kw), tol=3e-5, what='conv2d_resample.' + k)
        out[k] = y
    save('conv2d_resample', x=x, w3=w3, w1=w1, wg=wg, f=f, **out)


def g_networks():
    """a13: the reference's own layer classes (inversion/networks.py: MappingNetwork :246, SynthesisBlock :718, SegSynthesisBlock
    :966, with SynthesisLayer :330 / ToRGBLayer :670 / modulated_conv2d :55 inside) run on CPU with seeded parameters; the product's
    restatement (ide3d_b200.training.networks) must LOAD THE SAME state_dict and reproduce the outputs.  inversion/networks.py needs two
    dead numpy-1.x imports stubbed (SURVEY.md §8c) -- no source edit."""
    import types
    for name, attr in (('numpy.lib.arraysetops', 'isin'), ('numpy.lib.function_base', 'angle')):
        m = types.ModuleType(name)
        setattr(m, attr, getattr(np, attr))
        sys.modules.setdefault(name, m)
    import inversion.networks as rn
    from ide3d_b200.training import networks as mine
    from oracle.backend import cpu_reference_ops
    layer = dict(layer_name='inversion.networks.SynthesisLayer')
    out = {}

    def randomise(mod, gen):
        for p in mod.parameters():                       # StyleGAN init leaves biases / noise strengths at 0: make every term count
            if p.ndim == 0:
                p.data.fill_(0.3)
            elif p.ndim == 1:
                p.data.copy_(torch.randn(p.shape, generator=gen) * 0.5)

    def put(prefix, sd):
        for k, v in sd.items():
            out[f'{prefix}/{k}'] = v.detach().clone()

    g = torch.Generator().manual_seed(11)
    torch.manual_seed(11)
    # ---- mapping
    rm = rn.MappingNetwork(z_dim=16, c_dim=25, w_dim=12, num_ws=5, num_layers=2).eval()
    rm.w_avg.copy_(torch.randn(12, generator=g) * 0.1)
    z, c = torch.randn(3, 16, generator=g), torch.randn(3, 25, generator=g)
    with torch.no_grad():
        w_ref = rm(z, c, truncation_psi=0.7, truncation_cutoff=3)
    mm = mine.MappingNetwork(z_dim=16, c_dim=25, w_dim=12, num_ws=5, num_layers=2).eval()
    mm.load_state_dict(rm.state_dict())
    with torch.no_grad(), cpu_reference_ops():
        close(mm(z, c, truncation_psi=0.7, truncation_cutoff=3), w_ref, 2e-6, 'mapping')
    put('map', rm.state_dict())
    out.update(map_z=z, map_c=c, map_ws=w_ref)

    # ---- SynthesisBlock: first block (const input) and an upsampling block, eval (grouped weight-modulated conv) and train
    #      (activation-scaled conv) forms of modulated_conv2d
    for tag, in_ch in (('b0', 0), ('b1', 16)):
        rb = rn.SynthesisBlock(in_ch, 8, w_dim=12, resolution=16, img_channels=6, is_last=False, architecture='skip', **layer)
        randomise(rb, g)
        mb = mine.SynthesisBlock(in_ch, 8, w_dim=12, resolution=16, img_channels=6, is_last=False)
        mb.load_state_dict(rb.state_dict())
        x = torch.randn(2, 16, 8, 8, generator=g) if in_ch else None
        img = torch.randn(2, 6, 8, 8, generator=g) if in_ch else None
        ws = torch.randn(2, 3 if in_ch else 2, 12, generator=g)
        put(tag, rb.state_dict())
        out[f'{tag}_ws'] = ws
        if in_ch:
            out[f'{tag}_x'], out[f'{tag}_img'] = x, img
        for mode in ('eval', 'train'):
            getattr(rb, mode)(); getattr(mb, mode)()
            with torch.no_grad():
                xo, io = rb(x, None if img is None else img.clone(), ws, noise_mode='const')
                with cpu_reference_ops():
                    xm, im = mb(x, None if img is None else img.clone(), ws, noise_mode='const')
            close(xm, xo, 1e-5, f'{tag} {mode} x'); close(im, io, 1e-5, f'{tag} {mode} img')
            out[f'{tag}_{mode}_x'], out[f'{tag}_{mode}_img'] = xo, io

    # ---- SegSynthesisBlock (dual path).  The reference class has separate torgb / toseg layers; the product evaluates both heads
    #      as one 1x1 modulated convolution with ONE affine (the real generator's block has three children, DESIGN.md §3), which is
    #      the same function exactly when the two affines coincide -- so the golden case ties toseg.affine to torgb.affine.
    rs = rn.SegSynthesisBlock(16, 8, w_dim=12, resolution=16, img_channels=6, seg_channels=4, is_last=False, architecture='skip', **layer)
    randomise(rs, g)
    rs.toseg.affine.load_state_dict(rs.torgb.affine.state_dict())
    ms = mine.SegSynthesisBlock(16, 8, w_dim=12, resolution=16, img_channels=6, seg_channels=4, is_last=False)
    sd = {k: v for k, v in rs.state_dict().items() if not k.startswith(('torgb.', 'toseg.'))}
    sd['torgb.weight'] = torch.cat([rs.torgb.weight, rs.toseg.weight], 0)
    sd['torgb.bias'] = torch.cat([rs.torgb.bias, rs.toseg.bias], 0)
    sd['torgb.affine.weight'], sd['torgb.affine.bias'] = rs.torgb.affine.weight, rs.torgb.affine.bias
    ms.load_state_dict(sd)
    x, img, seg = torch.randn(2, 16, 8, 8, generator=g), torch.randn(2, 6, 8, 8, generator=g), torch.randn(2, 4, 8, 8, generator=g)
    ws = torch.randn(2, 3, 12, generator=g)
    rs.eval(); ms.eval()
    with torch.no_grad():
        xo, io, so = rs(x, img.clone(), seg.clone(), ws, noise_mode='const')
        with cpu_reference_ops():
            xm, im, sm = ms(x, img.clone(), ws, condition_img=seg.clone(), noise_mode='const')
    close(xm, xo, 1e-5, 'seg x'); close(im, io, 1e-5, 'seg img'); close(sm, so, 1e-5, 'seg seg')
    put('seg', sd)
    out.update(seg_x=x, seg_img=img, seg_seg=seg, seg_ws=ws, seg_out_x=xo, seg_out_img=io, seg_out_seg=so)
    save('networks', **out)


# ------------------------------------------------------------------ gen_videos.py frame loop (config 3)
def g_video_loop():
    """The (w, camera) pair the reference's gen_interp_video hands to G.synthesis for every (frame, grid cell), recorded from the
    unmodified frame loop (gen_videos.py:112-129) with seeds [3, 1, 4, 1, 5, 9, 2, 6], w_frames=3, a 2x1 grid, psi 0.7, cutoff 4;
    the keyframe mapping call (its z, c and the ws it returned, from a small random-init generator); and layout_grid
    (gen_videos.py:24-38) applied to seeded uint8 frames."""
    import types
    from oracle.backend import cpu_reference_ops
    from ide3d_b200.training.triplane import TriPlaneGenerator
    for name in ('imageio', 'mrcfile'):                  # output writers the recorded path never reaches
        sys.modules.setdefault(name, types.ModuleType(name))
    gv = __import__('gen_videos')
    torch.manual_seed(0)
    G = TriPlaneGenerator(z_dim=32, w_dim=32, img_resolution=64, plane_resolution=32, render_size=16, channel_base=512,
                          channel_max=16, sr_channels=(8, 8), mapping_kwargs=dict(num_layers=2)).eval().requires_grad_(False)
    calls, mapped = [], {}

    def record_mapping(z, c, **kw):
        assert kw == dict(truncation_psi=0.7, truncation_cutoff=4)
        mapped.update(map_z=z, map_c=c, map_ws=G.mapping(z, c, **kw))
        return mapped['map_ws']

    class Recorder:
        z_dim = G.z_dim

        def parameters(self):
            return G.parameters()

        @staticmethod
        def mapping(z, c, **kw):
            return record_mapping(z, c, **kw)

        @staticmethod
        def synthesis(ws, c, **kw):
            calls.append((ws.detach().clone(), c.detach().clone()))
            n = ws.shape[0]
            return torch.zeros(n, 3, 4, 4), torch.zeros(n, 19, 4, 4)

    class Writer:
        def append_data(self, a):
            pass

        def close(self):
            pass

    sys.modules['imageio'].get_writer = lambda *a, **k: Writer()
    with torch.no_grad(), cpu_reference_ops():
        gv.gen_interp_video(Recorder(), 'unused.mp4', image_mode='image_seg', device=torch.device('cpu'), seeds=[3, 1, 4, 1, 5, 9, 2, 6],
                            w_frames=3, grid_dims=(2, 1), psi=0.7, truncation_cutoff=4)
    calls = calls[1:]                                    # the warm-up call (:89)
    F, gh, gw = 12, 1, 2
    assert len(calls) == F * gh * gw
    frames = torch.randint(0, 255, (F * gh * gw, 3, 5, 7), dtype=torch.uint8, generator=torch.Generator().manual_seed(0))
    grids = np.stack([gv.layout_grid(frames[f * gh * gw:(f + 1) * gh * gw], grid_w=gw, grid_h=gh, float_to_uint8=False) for f in range(F)])
    save('video_loop', ws=torch.cat([w for w, _ in calls]), c=torch.cat([c for _, c in calls]), frames=frames, grids=grids, **mapped)


if __name__ == '__main__':
    torch.set_num_threads(4)
    fns = dict(rays=g_rays, transform=g_transform, camera=g_camera, triplane=g_triplane, integration=g_integration, pdf=g_pdf,
               chain=g_chain, chain_hier=g_chain_hier, create_samples=g_create_samples, bias_act=g_bias_act, upfirdn2d=g_upfirdn2d,
               filtered_lrelu=g_filtered_lrelu, conv2d_resample=g_conv2d_resample, networks=g_networks, video_loop=g_video_loop)
    for name in (sys.argv[1:] or list(fns)):              # `make_golden.py networks` regenerates one fixture only
        fns[name]()
    print('all reference outputs reproduced by oracle/ within tolerance')
