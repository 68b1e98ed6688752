"""CPU: the reference's OWN caller scripts (gen_images.py, gen_videos.py, extract_shapes.py, viz/renderer.py -- imported
unmodified, as the bytecode __graft_entry__.build() compiles from the original IDE-3D project into oracle/_ref/ by
oracle/build_ref.py) run against this package through `compat.install()`.

What is stubbed, and why it does not touch the contract under test:
  * `legacy.load_network_pkl`  -> returns a small random-init TriPlaneGenerator (no checkpoint pickle exists offline)
  * `dnnlib.util.open_url`     -> dummy context manager (the "pickle path" is never read)
  * imageio / plyfile / skimage -> absent output-writer dependencies of the scripts (SURVEY.md §8c); `mrcfile` is supplied by
    compat.install() (ide3d_b200.mrc, a numpy MRC2014 writer)
  * torch.device('cuda') inside the scripts -> 'cpu', and the CUDA entry points -> oracle (no GPU in this container)
  * torchvision's save_image   -> recorder (the scripts call it with the removed `range=` keyword)
Those tests skip when oracle/_ref/ was not built.  The batched video driver is compared with the reference's frame loop through
a recording of that loop stored in tests/golden/video_loop.npz (tests/golden/make_golden.py), so it runs everywhere."""

import contextlib
import importlib
import os
import sys
import types

import numpy as np
import pytest
import torch

from conftest import ROOT, T, load_golden

REF = os.path.join(ROOT, 'oracle', '_ref')
needs_reference = pytest.mark.skipif(not os.path.isfile(os.path.join(REF, 'gen_images.pyc')),
                                     reason='oracle/_ref not built: no checkout of the original project at build time')


@pytest.fixture()
def ref_env(monkeypatch):
    from oracle.backend import cpu_reference_ops
    import ide3d_b200.compat as compat
    from ide3d_b200.training.triplane import TriPlaneGenerator

    saved = dict(sys.modules)
    monkeypatch.syspath_prepend(REF)
    monkeypatch.setattr(sys, 'dont_write_bytecode', True)
    for name in ('imageio', 'plyfile', 'skimage', 'skimage.measure'):      # mrcfile: compat.install() supplies ide3d_b200.mrc
        monkeypatch.setitem(sys.modules, name, types.ModuleType(name))
    sys.modules['skimage'].measure = sys.modules['skimage.measure']
    compat.install()                                     # training.*, torch_utils.* -> this package

    torch.manual_seed(0)
    G = TriPlaneGenerator(z_dim=32, w_dim=32, img_resolution=64, plane_resolution=32, render_size=16, channel_base=512,
                          channel_max=16, sr_channels=(8, 8), mapping_kwargs=dict(num_layers=2)).eval().requires_grad_(False)
    legacy = types.ModuleType('legacy')
    legacy.load_network_pkl = lambda f: {'G_ema': G}
    monkeypatch.setitem(sys.modules, 'legacy', legacy)
    import dnnlib                                        # the reference's own dnnlib (EasyDict, seg_tools, util.open_url)
    monkeypatch.setattr(dnnlib.util, 'open_url', lambda *a, **k: contextlib.nullcontext(None))

    real_device = torch.device

    class _Dev:                                          # scripts hard-code torch.device('cuda')
        def __call__(self, *a, **k):
            return real_device('cpu')

    with cpu_reference_ops():
        yield G, _Dev()
    ours = {'training', 'torch_utils', 'dnnlib', 'legacy', 'gen_images', 'gen_videos', 'extract_shapes', 'camera_utils', 'mrcfile', 'viz'}
    for k in list(sys.modules):                          # drop only what this fixture introduced (cv2 & co. cannot re-import)
        if k not in saved and k.split('.')[0] in ours:
            del sys.modules[k]
    for k in ours:
        if k in saved:
            sys.modules[k] = saved[k]


@needs_reference
def test_gen_images_runs_unchanged(ref_env, tmp_path, monkeypatch):
    G, dev = ref_env
    gen_images = importlib.import_module('gen_images')
    saved_imgs = {}
    monkeypatch.setattr(gen_images, 'save_image', lambda t, path, **kw: saved_imgs.__setitem__(os.path.basename(path), t.clone()))
    monkeypatch.setattr(gen_images.torch, 'device', dev)
    try:
        gen_images.generate_images.callback(network_pkl='unused.pkl', seeds=[3], truncation_psi=0.7, noise_mode='const', outdir=str(tmp_path))
    finally:
        monkeypatch.undo()
    assert set(saved_imgs) == {'seed0003.png', 'seed0003_seg.png'}
    img, seg = saved_imgs['seed0003.png'], saved_imgs['seed0003_seg.png']
    assert img.shape == (3, 3, 64, 64) and seg.shape == (3, 3, 64, 64)          # 3 yaws; mask2color gives RGB maps
    assert torch.isfinite(img).all() and not torch.allclose(img[0], img[2])     # different yaws, different views


@needs_reference
def test_extract_shapes_block_walk_runs_unchanged(ref_env, monkeypatch):
    G, dev = ref_env
    es = importlib.import_module('extract_shapes')
    z = torch.from_numpy(np.random.RandomState(0).randn(1, G.z_dim))
    label = torch.tensor([1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1, 2.7, 0, 0, 0, 1, 4.2647, 0, 0.5, 0, 4.2647, 0.5, 0, 0, 1])[None].float()
    vox = es.sample_generator_ide3d(G, None, z.float(), label, cube_length=1.0, voxel_resolution=12, psi=0.7, max_batch=500,
                                    h_stddev=0., v_stddev=0., num_steps=96)
    assert vox.shape == (12, 12, 12) and np.isfinite(vox).all() and vox.std() > 0


@needs_reference
def test_gen_videos_frame_loop_runs_unchanged(ref_env, monkeypatch):
    G, dev = ref_env
    frames = []

    class _Writer:
        def append_data(self, a):
            frames.append(np.asarray(a))

        def close(self):
            pass

    sys.modules['imageio'].get_writer = lambda *a, **k: _Writer()
    gv = importlib.import_module('gen_videos')
    gv.gen_interp_video(G, 'unused.mp4', seeds=[0, 1], w_frames=2, grid_dims=(1, 1), psi=0.7, truncation_cutoff=4,
                        image_mode='image_seg', device=torch.device('cpu'))
    assert len(frames) == 4                                                      # 2 keyframes x 2 frames
    assert frames[0].dtype == np.uint8 and frames[0].shape == (64, 128, 3)       # image | colourised mask, side by side


@needs_reference
def test_extract_shapes_main_writes_mrc_through_the_shim(ref_env, tmp_path, monkeypatch):
    """The script's __main__ block end to end on CPU: argparse -> load (stubbed pickle) -> block walk -> sample_voxel chunks ->
    `mrcfile.new_mmap(...)` (ide3d_b200.mrc via compat.install) + np.save; the .mrc holds the same grid as the .npy."""
    import runpy
    from ide3d_b200 import mrc
    out = tmp_path / 'shapes'
    monkeypatch.setattr(sys, 'argv', ['extract_shapes.py', '--network', 'unused.pkl', '--seeds', '0', '--voxel_resolution', '10',
                                      '--cube_size', '1.0', '--outdir', str(out)])
    runpy.run_path(os.path.join(REF, 'extract_shapes.pyc'), run_name='__main__')
    grid = np.load(out / '0.npy')
    vol, hdr = mrc.read_mrc(str(out / '0.mrc'))
    assert grid.shape == (10, 10, 10) and np.array_equal(vol, grid.astype(np.float32)) and hdr['mode'] == 2


def test_batched_video_inputs_equal_the_reference_frame_loop():
    """ide3d_b200.video.interp_video_inputs computes, up front, exactly the (w, camera) pair the reference's frame loop hands to
    G.synthesis for every (frame, grid cell) (gen_videos.py:112-129) -- as recorded from the unmodified gen_interp_video in
    tests/golden/video_loop.npz -- and layout_frames is layout_grid (gen_videos.py:24-38) applied per frame.  The mapping network
    replays the keyframe ws of the recording, so the comparison pins the spline and camera arithmetic, not the host's float32 matmuls."""
    from ide3d_b200 import video
    g = load_golden('video_loop')

    class Recorded:
        z_dim = 32

        @staticmethod
        def mapping(z, c, truncation_psi, truncation_cutoff):
            assert (truncation_psi, truncation_cutoff) == (0.7, 4)
            assert torch.equal(z, T(g['map_z'])) and (c - T(g['map_c'])).abs().max() < 1e-6
            return T(g['map_ws'])

    ws, c, (F, gh, gw) = video.interp_video_inputs(Recorded(), seeds=[3, 1, 4, 1, 5, 9, 2, 6], w_frames=3, grid_dims=(2, 1), psi=0.7,
                                                   truncation_cutoff=4, device=torch.device('cpu'))
    ref_ws, ref_c = T(g['ws']), T(g['c'])
    assert (F, gh, gw) == (12, 1, 2) and F * gh * gw == ref_ws.shape[0] == ws.shape[0] == c.shape[0]
    assert ws.dtype == ref_ws.dtype == torch.float64
    assert (ws - ref_ws).abs().max() < 1e-9 and (c - ref_c).abs().max() < 1e-6

    mine = video.layout_frames(T(g['frames']), F, gh, gw)
    for f in range(F):
        assert np.array_equal(mine[f].numpy(), g['grids'][f])


@needs_reference
def test_viz_renderer_render_impl_runs_unchanged(ref_env, monkeypatch):
    """viz/renderer.py (the interactive visualizer's backend, imported unmodified): Renderer._render_impl walks the generator contract
    -- get_network (deepcopy + .to), G.img_resolution / G.synthesis.num_ws / named_buffers / G.mapping.w_avg / G.backbone.num_ws,
    positional G.synthesis(w, c, noise_mode=, force_fp32=), forward hooks on every sub-module -- on CPU, with CUDA-only plumbing
    (events, pinned buffers, the literal 'cuda' device) neutralised and matplotlib (absent) stubbed."""
    G, dev = ref_env

    class _Event:
        def __init__(self, *a, **k):
            pass

        def record(self, *a):
            pass

        def synchronize(self):
            pass

        def elapsed_time(self, other):
            return 0.0

    for name in ('matplotlib', 'matplotlib.cm'):
        monkeypatch.setitem(sys.modules, name, types.ModuleType(name))
    sys.modules['matplotlib'].cm = sys.modules['matplotlib.cm']
    monkeypatch.setattr(torch.cuda, 'Event', _Event)
    monkeypatch.setattr(torch.Tensor, 'pin_memory', lambda self, *a, **k: self)
    real_to = torch.nn.Module.to

    def to_cpu_when_cuda(self, *args, **kwargs):
        args = tuple('cpu' if (isinstance(a, str) and a.startswith('cuda')) or (isinstance(a, torch.device) and a.type == 'cuda') else a for a in args)
        return real_to(self, *args, **kwargs)

    monkeypatch.setattr(torch.nn.Module, 'to', to_cpu_when_cuda)
    vr = importlib.import_module('viz.renderer')
    import dnnlib
    R = vr.Renderer()
    R._device = torch.device('cpu')
    res = dnnlib.EasyDict()
    R._render_impl(res, pkl='unused.pkl', w0_seeds=[[0, 0.75], [1, 0.25]], stylemix_idx=[1, 2], stylemix_seed=2, trunc_psi=0.7, trunc_cutoff=4,
                   yaw=0.2, pitch=0.1)
    assert 'error' not in res
    assert res.img_resolution == 64 and res.num_ws == G.synthesis.num_ws and res.has_noise and not res.has_input_transform
    assert res.image.dtype == torch.uint8 and tuple(res.image.shape) == (64, 64, 3)
    names = [l.name for l in res.layers]
    assert 'synthesis' in names and any(n.startswith('synthesis.vb32') for n in names) and any(n.startswith('synthesis.b64') for n in names)
    assert res.stats.shape == (6,) and torch.isfinite(res.stats).all()
