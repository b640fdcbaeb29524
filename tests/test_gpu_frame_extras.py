"""ABI 3 frame extras on the GPU — lens distortion (iterative OpenCV / f-theta), distortion map, depth of field, glow modes, environment map,
the Distortion render mode: nsb_render against the CPU oracle AND against the reference's own CUDA path (oracle/_ref's nvcc build of
init_rays_with_payload_kernel_nerf / pixel_to_ray / composite_kernel_nerf / render_nerf). Newton iterations and sincosf: these frames are
held to the 1e-3 frame tolerance (DESIGN.md section 3); what is measured is printed."""
import ctypes as C

import numpy as np
import pytest

from nerfshop_b200 import abi
from nerfshop_b200 import synthetic as syn
from ref_golden import Recorded
from test_frame_extras_cpu import CASES, H, W, _dof

ref = Recorded("gpu_frame_extras")  # outputs of oracle/_ref's CUDA build stored under tests/golden/ref/ (ref_golden.py)

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def maps():
    import torch

    env, dist = syn.make_envmap(), syn.make_distortion_map()
    return {"env": env, "dist": dist, "env_dev": torch.from_numpy(env).cuda(), "dist_dev": torch.from_numpy(dist).cuda()}


class _DevPtr:  # quacks like the numpy array CASES expects (.ctypes.data, .shape) but points at device memory
    def __init__(self, t):
        self.shape = tuple(t.shape)
        self.ctypes = type("p", (), {"data": t.data_ptr()})()


def _frames(model, case, maps, cam=17, w=W, h=H):
    host = CASES[case](syn.make_frame(model, syn.orbit_cameras(120)[cam], w, h), {"env": maps["env"], "dist": maps["dist"]})
    dev = CASES[case](syn.make_frame(model, syn.orbit_cameras(120)[cam], w, h), {"env": _DevPtr(maps["env_dev"]), "dist": _DevPtr(maps["dist_dev"])})
    return host, dev


def _rel(a, b):
    return (np.abs(a - b) / np.maximum(1.0, np.abs(b))).max(-1)


@pytest.mark.parametrize("case", list(CASES))
def test_native_vs_oracle(scene, oracle, renderer, maps, case):
    model, _ = scene
    f_host, f_dev = _frames(model, case, maps)
    fb_o, d_o, st_o, margin = oracle.render(f_host, want_margin=True)
    fb, depth = renderer.render(f_dev)
    fb, depth = fb.cpu().numpy(), depth.cpu().numpy()
    err = _rel(fb, fb_o)
    ok = margin > 2e-5
    print(f"\n{case}: native vs oracle L-inf {err[ok].max():.3e} ({(~ok).sum()} threshold pixels excluded), > 1e-4: {(err > 1e-4).sum()} of {err.size}; samples {renderer.stats().n_samples} vs {st_o.n_samples}")
    if case.startswith("glow") or case == "everything":
        assert (err[ok] > 1e-3).sum() <= 3 and err[ok].max() < 3e-3
    else:
        assert err[ok].max() <= 1e-3
    assert (err > 1e-4).mean() < 0.02
    hit = (fb_o[..., 3] > 0.2) & ok
    assert np.abs(depth - d_o)[hit].max() < 0.25


@pytest.mark.parametrize("case", list(CASES))
def test_native_vs_reference_cuda(scene, renderer, maps, case):
    import torch

    model, occ = scene
    rc = ref.RefCuda(occ)
    try:
        _, f_dev = _frames(model, case, maps, cam=63, w=320, h=180)
        fb, depth = renderer.render(f_dev)
        # the reference's frame is stored at a seeded sample of 12,000 of the 57,600 pixels
        sel = torch.from_numpy(np.sort(np.random.default_rng(11).choice(320 * 180, 12_000, replace=False))).cuda()
        fb_r, depth_r, info = rc.render(f_dev, renderer, shrink=lambda o: (o[0].reshape(-1, 4)[sel], None, o[2]), also=(maps["env"], maps["dist"]))
        torch.cuda.synchronize()
        fb = fb.reshape(-1, 4)[sel]
        err = ((fb - fb_r).abs() / fb_r.abs().clamp(min=1.0)).amax(-1)
        n_bad = int((err > 1e-3).sum())
        print(f"\n{case}: native vs the reference's CUDA path L-inf {float(err.max()):.3e}; pixels > 1e-4: {int((err > 1e-4).sum())} of {err.numel()}; identical: {bool(torch.equal(fb, fb_r))}")
        assert (fb_r[..., 3] > 0).float().mean().item() > 0.2
        # termination flips are not masked here (no margin from the reference): allow a handful of pixels, 6 in the whole frame,
        # at that rate over the sample
        assert n_bad <= int(np.ceil(6 * sel.numel() / (320 * 180))) and float(err.max()) < 5e-2
        assert float((err > 1e-4).float().mean()) < 0.02
    finally:
        rc.close()


@pytest.mark.parametrize("with_map", [False, True])
def test_distortion_render_mode(scene, oracle, renderer, maps, with_map):
    model, _ = scene
    f_host = syn.make_frame(model, syn.orbit_cameras(120)[17], W, H)
    f_dev = syn.make_frame(model, syn.orbit_cameras(120)[17], W, H)
    f_host.render_mode = f_dev.render_mode = abi.NSB_RENDER_DISTORTION
    if with_map:
        syn.set_maps(f_host, distortion_ptr=maps["dist"].ctypes.data, distortion_shape=maps["dist"].shape)
        syn.set_maps(f_dev, distortion_ptr=maps["dist_dev"].data_ptr(), distortion_shape=maps["dist"].shape)
    fb_o, d_o, _, _ = oracle.render(f_host)
    fb, depth = renderer.render(f_dev)
    assert np.abs(fb.cpu().numpy() - fb_o).max() <= 1e-5 and np.array_equal(depth.cpu().numpy(), d_o)
    assert renderer.stats().n_samples == 0


def test_general_camera_sample_stream_and_partition(scene, oracle, renderer, maps):
    """Lens-distorted, defocused frame: the sample stream against the oracle; and the image-plane partition (the rays travel to the persistent
    renderer in a side buffer indexed by queue slot) reproduces the single-GPU frame bit for bit, at 1080p too."""
    import torch

    model, _ = scene
    f = _dof(syn.set_camera_distortion(syn.make_frame(model, syn.orbit_cameras(120)[40], 96, 54), abi.NSB_CAMERA_DISTORTION_ITERATIVE, [0.08, -0.02, 0.003, -0.002]))
    pix = np.arange(0, 96 * 54, 7, dtype=np.uint32)
    rec, idx, cnt = renderer.march_trace(f, pix, 48)
    rec_o, idx_o, cnt_o = oracle.march_trace(f, pix, 48)
    same = np.minimum(cnt, 48) == np.minimum(cnt_o, 48)
    both = (cnt > 0) & (cnt_o > 0)
    d = np.abs(rec[both, 0, 0] - rec_o[both, 0, 0])
    print(f"\ngeneral-camera sample stream: counts equal on {same.mean() * 100:.2f} % of {pix.size} rays; first-sample t median diff {np.median(d):.2e}, max {d.max():.2e}")
    assert same.mean() > 0.97 and np.median(d) < 1e-6 and (d > 1e-4).mean() < 0.02
    for (w, h) in ((176, 99), (1920, 1080)):
        g = _dof(syn.set_camera_distortion(syn.make_frame(model, syn.orbit_cameras(120)[60], w, h), abi.NSB_CAMERA_DISTORTION_ITERATIVE, [0.08, -0.02, 0.003, -0.002]))
        full, dfull = renderer.render(g)
        full, dfull = full.clone(), dfull.clone()
        again, _ = renderer.render(g)
        assert torch.equal(full, again)
        world = 3
        acc, dacc = torch.zeros_like(full), torch.zeros_like(dfull)
        for rank in range(world):
            g.tile_rank, g.tile_world = rank, world
            fb, depth = renderer.render(g)
            n_tiles = renderer.tiles_for_rank(w, h, rank, world)
            packed = torch.zeros((n_tiles * 128, 4), dtype=torch.float32, device="cuda")
            pdepth = torch.zeros(n_tiles * 128, dtype=torch.float32, device="cuda")
            renderer.pack_tiles(fb, depth, rank, world, packed, pdepth)
            renderer.unpack_tiles(packed, pdepth, rank, world, acc, dacc)
        torch.cuda.synchronize()
        assert torch.equal(acc, full) and torch.equal(dacc, dfull)


def test_frame_extras_validation(scene, renderer):
    import torch

    model, _ = scene
    fb = torch.zeros((H, W, 4), device="cuda")
    dp = torch.zeros((H, W), device="cuda")

    def status(mut):
        f = syn.make_frame(model, syn.orbit_cameras(120)[17], W, H)
        mut(f)
        return renderer.lib.nsb_render(renderer.ctx, C.byref(f), fb.data_ptr(), dp.data_ptr(), None)

    assert status(lambda f: setattr(f, "focus_z", -1.0)) == abi.NSB_ERR_UNSUPPORTED          # the reference's Slice side path
    assert status(lambda f: setattr(f, "dof", 0.01)) == abi.NSB_ERR_INVALID                   # depth of field without a focus distance
    assert status(lambda f: setattr(f, "camera_distortion_mode", 3)) == abi.NSB_ERR_INVALID
    assert status(lambda f: setattr(f, "render_mode", 9)) == abi.NSB_ERR_UNSUPPORTED         # Slice
    assert status(lambda f: setattr(f, "render_mode", 2)) == abi.NSB_ERR_UNSUPPORTED         # Normals
    assert status(lambda f: None) == abi.NSB_OK
