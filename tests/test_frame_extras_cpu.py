"""ABI 3 frame extras — lens distortion (iterative OpenCV / f-theta), distortion map, depth of field, glow modes, environment map, the Distortion
render mode — CPU side: the oracle against oracle/_ref = the reference's own init_rays_with_payload_kernel_nerf / pixel_to_ray /
composite_kernel_nerf / render_nerf compiled for the CPU. These paths run Newton iterations and sincosf: they are held to the 1e-3 frame
tolerance (DESIGN.md section 3), not to bit-exact ray generation."""
import numpy as np
import pytest

from nerfshop_b200 import abi
from nerfshop_b200 import synthetic as syn
from ref_golden import Recorded

ref = Recorded("frame_extras_cpu")  # outputs of oracle/_ref stored under tests/golden/ref/ (ref_golden.py)

W, H = 112, 63
CASES = {
    "iterative": lambda f, k: syn.set_camera_distortion(f, abi.NSB_CAMERA_DISTORTION_ITERATIVE, [0.08, -0.02, 0.003, -0.002]),
    "ftheta": lambda f, k: syn.set_camera_distortion(f, abi.NSB_CAMERA_DISTORTION_FTHETA, [0.0, 1.0 / (1.05 * H), 0.0, 2e-8, 0.0, W, H]),
    "dof": lambda f, k: _dof(f),
    "distortion_map": lambda f, k: syn.set_maps(f, distortion_ptr=k["dist"].ctypes.data, distortion_shape=k["dist"].shape),
    "envmap": lambda f, k: syn.set_maps(f, envmap_ptr=k["env"].ctypes.data, envmap_shape=k["env"].shape),
    "glow_grid_cutline": lambda f, k: _glow(f, 3, 0.62),
    "glow_mask_to_alpha": lambda f, k: _glow(f, 5, 0.58),
    "glow_radial": lambda f, k: _glow(f, 9, 1.3),
    "glow_grid_mode": lambda f, k: _glow(f, 16, 0.0),
    "everything": lambda f, k: _glow(_dof(syn.set_maps(syn.set_camera_distortion(f, abi.NSB_CAMERA_DISTORTION_ITERATIVE, [0.05, 0.01, -0.002, 0.001]),
                                                      envmap_ptr=k["env"].ctypes.data, envmap_shape=k["env"].shape,
                                                      distortion_ptr=k["dist"].ctypes.data, distortion_shape=k["dist"].shape)), 7, 0.6),
}


def _dof(f):
    f.dof, f.focus_z, f.spp_index = 0.012, 1.25, 3
    return f


def _glow(f, mode, cutoff):
    f.glow_mode, f.glow_y_cutoff = mode, cutoff
    return f


def _first_t(out):
    """What the ray-stream tests read of the reference's march_trace: payload.t after the first step (rec[:, 0, 7]) and the sample counts."""
    rec, _, cnt, _ = out
    first = np.zeros((rec.shape[0], 1, 8), np.float32)
    first[:, 0, 7] = rec[:, 0, 7]
    return first, None, cnt, None


def frame_for(model, case, keep):
    f = syn.make_frame(model, syn.orbit_cameras(120)[17], W, H)
    return CASES[case](f, keep)


@pytest.mark.parametrize("case", list(CASES))
def test_oracle_vs_reference_render_nerf(scene, oracle, case):
    model, occ = scene
    keep = {"env": syn.make_envmap(), "dist": syn.make_distortion_map()}
    f = frame_for(model, case, keep)
    plain = syn.make_frame(model, syn.orbit_cameras(120)[17], W, H)
    fb_o, d_o, st, margin = oracle.render(f, want_margin=True)
    fb_r, d_r, info = ref.render(f, occ, lambda c: oracle.inference(c), also=keep)
    fb_p = oracle.render(plain)[0]
    # glow colours are HDR (the cut line reaches ~100) and come from cos(800 x): the 1e-3 contract is applied relative to the value there
    err = (np.abs(fb_o - fb_r) / np.maximum(1.0, np.abs(fb_o))).max(-1)
    ok = margin > 2e-5
    print(f"\n{case}: L-inf {err[ok].max():.3e} ({(~ok).sum()} threshold pixels excluded); > 1e-4: {(err > 1e-4).sum()} of {err.size}; differs from the plain frame by {np.abs(fb_o - fb_p).max():.3f}")
    assert np.abs(fb_o - fb_p).max() > 0.02, "the feature must be visible"
    if case.startswith("glow") or case == "everything":  # a 1-ulp position difference is amplified by y * 80 and cos(x * 16 pi * 16): a handful of cut-line pixels reach 1.2e-3
        assert (err[ok] > 1e-3).sum() <= 3 and err[ok].max() < 3e-3
    else:
        assert err[ok].max() <= 1e-3
    assert (err > 1e-4).mean() < 0.02
    hit = (fb_r[..., 3] > 0.2) & ok
    if "env" not in case and case != "everything":
        assert np.array_equal(fb_o[..., 3] > 0, fb_r[..., 3] > 0)
    assert np.abs(d_o - d_r)[hit].max() < 0.25


@pytest.mark.parametrize("with_map", [False, True])
def test_distortion_render_mode(scene, oracle, with_map):
    """ERenderMode::Distortion (init_rays :2596-2607): the map itself x 50 + 0.5 in (r, g), (0.5, 1) in (b, a), depth 1, for the rays that enter the AABB."""
    model, occ = scene
    dist = syn.make_distortion_map()
    f = syn.make_frame(model, syn.orbit_cameras(120)[17], W, H)
    f.render_mode = abi.NSB_RENDER_DISTORTION
    if with_map:
        syn.set_maps(f, distortion_ptr=dist.ctypes.data, distortion_shape=dist.shape)
    fb_o, d_o, st, _ = oracle.render(f)
    fb_r, d_r, _ = ref.render(f, occ, lambda c: oracle.inference(c), also=dist if with_map else None)
    assert np.abs(fb_o - fb_r).max() <= 1e-5 and np.array_equal(d_o, d_r)
    inside = fb_o[..., 3] == 1.0
    assert inside.mean() > 0.3 and np.all(d_o[inside] == 1.0) and np.all(fb_o[inside][:, 2] == 0.5)
    if not with_map:
        assert np.all(fb_o[inside][:, :2] == 0.5)
    else:
        assert np.abs(fb_o[inside][:, :2] - 0.5).max() > 0.2


def test_ray_stream_with_lens_distortion(scene, oracle):
    """The sample stream of a lens-distorted, depth-of-field frame: oracle vs the reference kernels (init_rays_with_payload_kernel_nerf + advance_pos_nerf +
    generate_next_nerf_network_inputs). Rays agree to float rounding; where the first samples fall in the same cells the streams have the same length."""
    model, occ = scene
    f = _dof(syn.set_camera_distortion(syn.make_frame(model, syn.orbit_cameras(120)[40], 96, 54), abi.NSB_CAMERA_DISTORTION_ITERATIVE, [0.08, -0.02, 0.003, -0.002]))
    pix = np.arange(0, 96 * 54, 7, dtype=np.uint32)
    MS = 48
    rec_o, idx_o, cnt_o = oracle.march_trace(f, pix, MS)
    rec_r, ray_r, cnt_r, alive_r = ref.march_trace(f, occ, pix, MS, shrink=_first_t)
    cnt_o = np.minimum(cnt_o, MS)
    assert (cnt_o > 0).mean() > 0.3
    # Newton undistortion + sincosf: rays agree to float rounding, so a handful of rays may gain or lose a sample at a cell face
    assert (cnt_o == cnt_r).mean() > 0.97, (cnt_o == cnt_r).mean()
    both = (cnt_o > 0) & (cnt_r > 0)
    first_o = (rec_o[both, 0, 0] + rec_o[both, 0, 1]).astype(np.float32)  # t + dt of the first sample = payload.t after the first step (rec[..., 7])
    d = np.abs(first_o - rec_r[both, 0, 7])
    print(f"\nlens-distorted, defocused ray stream: {both.sum()} rays; sample counts equal on {(cnt_o == cnt_r).mean() * 100:.2f} %; first-sample t: median diff {np.median(d):.2e}, max {d.max():.2e}")
    assert np.median(d) < 1e-6 and (d > 1e-4).mean() < 0.02


@pytest.mark.parametrize("seed", range(6))
def test_random_general_cameras_ray_stream(scene, oracle, seed):
    """Random lens distortion (both models), distortion-map amplitude, aperture, focus distance, sample index and rolling shutter: the oracle's
    rays and first samples against the reference kernels' (init_rays_with_payload_kernel_nerf + advance_pos_nerf), pixel for pixel."""
    model, occ = scene
    rng = np.random.default_rng(1000 + seed)
    w, h = 80, 45
    f = syn.make_frame(model, syn.orbit_cameras(120)[int(rng.integers(0, 120))], w, h, spp=int(rng.integers(0, 64)))
    if rng.random() < 0.5:
        syn.set_camera_distortion(f, abi.NSB_CAMERA_DISTORTION_ITERATIVE, list(rng.uniform(-1, 1, 4) * np.array([0.15, 0.05, 0.01, 0.01])))
    else:
        syn.set_camera_distortion(f, abi.NSB_CAMERA_DISTORTION_FTHETA, [0.0, rng.uniform(0.8, 1.2) / h, 0.0, rng.uniform(-3e-8, 3e-8), 0.0, w, h])
    dist = syn.make_distortion_map(amplitude=float(rng.uniform(0.0, 0.02)), seed=seed)
    if rng.random() < 0.7:
        syn.set_maps(f, distortion_ptr=dist.ctypes.data, distortion_shape=dist.shape)
    if rng.random() < 0.7:
        f.dof, f.focus_z = float(rng.uniform(0.002, 0.03)), float(rng.uniform(0.6, 2.0))
    f.rolling_shutter[1] = float(rng.uniform(0.0, 0.3))
    f.rolling_shutter[3] = float(rng.uniform(0.0, 0.2))
    cam1 = np.array(list(f.camera1), np.float32)
    cam1[9:12] += rng.uniform(-0.02, 0.02, 3).astype(np.float32)  # camera0 != camera1: the rolling shutter interpolates them
    for i in range(12):
        f.camera0[i] = float(cam1[i])
    pix = np.arange(w * h, dtype=np.uint32)
    MS = 8
    rec_o, idx_o, cnt_o = oracle.march_trace(f, pix, MS)
    rec_r, ray_r, cnt_r, alive_r = ref.march_trace(f, occ, pix, MS, shrink=_first_t)
    cnt_o = np.minimum(cnt_o, MS)
    both = (cnt_o > 0) & (cnt_r > 0)
    d = np.abs((rec_o[both, 0, 0] + rec_o[both, 0, 1]).astype(np.float32) - rec_r[both, 0, 7])
    print(f"\nseed {seed}: {both.sum()} rays with samples; counts equal on {(cnt_o == cnt_r).mean() * 100:.2f} %; first-sample t identical on {(d == 0).mean() * 100:.2f} %, max diff {d.max():.2e}")
    assert both.sum() > 300
    assert (cnt_o == cnt_r).mean() > 0.98
    assert (d == 0).mean() > 0.95 and (d > 1e-4).mean() < 0.02
