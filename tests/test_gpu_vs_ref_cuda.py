"""The CUDA path of this repository against the reference's OWN CUDA path, on the GPU.

oracle/_ref/libnerfshop_ref_cuda.so is the nvcc (sm_100a) build of the reference's sources — Testbed::render_nerf, NerfTracer::trace /
init_rays_from_camera and every kernel they launch, interpolate_tet, translate_in_box, compute_residual_poisson_kernel (oracle/ref_build.py,
oracle/ref_driver_cuda.cu) — with one substitution: tiny-cuda-nn's network (absent submodule) is this repository's nsb_inference. So what
these tests pin, against code the reference's authors wrote and the same compiler's FMA contraction, is everything AROUND the network:
ray generation, jitter, occupancy stepping, compaction/termination semantics, deformation, membrane blend, composite, shade.

  * ray / sample stream (t, dt, warped position): bit for bit;
  * frames without operators, including the 1920x1080 north-star configuration: bit for bit (L-inf = 0);
  * frames with operators: <= 1e-3 (measured 3e-5): interpolate_tet's barycentrics agree to 1 ulp only — ptxas fuses the mul/sub pairs of the
    reference kernel's cross products inconsistently (shared sub-expressions across the four same_side tests), which is not a contract.
The reference's outputs are replayed from tests/golden/ref/gpu_vs_ref_cuda/ (ref_golden.py): bit-exact frames as SHA-256 digests of their
bytes, sample streams for a seeded sample of the rays, toleranced frames at a seeded sample of the pixels.
"""

import numpy as np
import pytest

from edit_fixtures import e1, e3
from nerfshop_b200 import abi, editing
from nerfshop_b200 import synthetic as syn
from ref_golden import Recorded, frame_digests, sha

ref = Recorded("gpu_vs_ref_cuda")
pytestmark = pytest.mark.gpu

_a = 0.4
ROT = np.array([[np.cos(_a), -np.sin(_a), 0], [np.sin(_a), np.cos(_a), 0], [0, 0, 1]], np.float32)


def _affine():
    return editing.AffineDuplication((0.5, 0.5, 0.5), (0.12, 0.12, 0.12), (0.03, 0.0, -0.1), rotation=ROT, hide_original=True, correct_dir=True)


@pytest.fixture(scope="module")
def ref_cuda(scene):
    model, occ = scene
    rc = ref.RefCuda(occ)
    yield rc
    rc.close()


@pytest.mark.parametrize("cam_index,spp", [(17, 0), (63, 0), (99, 5)])
def test_sample_stream_bit_exact_vs_reference_kernels(scene, renderer, ref_cuda, cam_index, spp):
    model, occ = scene
    W, H, MS = 192, 108, 64
    f = syn.make_frame(model, syn.orbit_cameras(120)[cam_index], W, H, spp=spp)
    pix = np.random.default_rng(cam_index).choice(W * H, 6000, replace=False).astype(np.uint32)
    rec, idx, cnt = renderer.march_trace(f, pix, MS)
    # the reference's sample counts are stored for every ray, its stream for a seeded sample of 600 of the rays that have samples
    sub, rec_r, cnt_r = ref_cuda.march_trace(f, pix, MS, shrink=lambda o: _stream_sample(o[0], o[2], 600, 100 + cam_index))
    assert np.array_equal(np.minimum(cnt, MS), cnt_r)
    assert cnt_r.sum() > 100_000
    rec, cnt_r = rec[sub], cnt_r[sub]
    amin, amax = np.array(list(f.train_aabb_min), np.float32), np.array(list(f.train_aabb_max), np.float32)
    valid = np.arange(MS)[None, :] < cnt_r[:, None]
    t_after = (rec[..., 0] + rec[..., 1]).astype(np.float32)  # payload.t after `t += dt` (generate_next_nerf_network_inputs)
    assert np.array_equal(t_after[valid], rec_r[..., 7][valid])
    wp = ((rec[..., 2:5] - amin) / (amax - amin)).astype(np.float32)  # warp_position(pos, train_aabb): one sub, one div per component
    assert np.array_equal(wp[valid], rec_r[..., 0:3][valid])
    min_step = np.float32(np.float32(1.73205080757) / np.float32(1024.0))
    wdt = ((rec[..., 1] - min_step) / (min_step * np.float32(16.0) - min_step)).astype(np.float32)  # warp_dt
    assert np.array_equal(wdt[valid], rec_r[..., 3][valid])


def _stream_sample(rec, cnt, k, seed):
    """shrink of march_trace: (rays drawn, their records, every ray's count). k rays are drawn among those with samples; of their records
    only the channels the test reads (warped position, warped dt, payload.t) are kept, zero past each ray's count."""
    sub = np.sort(np.random.default_rng(seed).choice(np.nonzero(cnt)[0], k, replace=False))
    out = np.zeros((k,) + rec.shape[1:2] + (8,), np.float32)
    valid = np.arange(rec.shape[1])[None, :] < cnt[sub, None]
    out[..., [0, 1, 2, 3, 7]] = np.where(valid[..., None], rec[sub][..., [0, 1, 2, 3, 7]], 0)
    return sub, out, cnt


@pytest.mark.parametrize("cam_index,mode", [(17, abi.NSB_RENDER_SHADE), (63, abi.NSB_RENDER_SHADE), (5, abi.NSB_RENDER_DEPTH), (40, abi.NSB_RENDER_COST), (77, abi.NSB_RENDER_POSITIONS)])
def test_frame_identical_to_reference_render_nerf(scene, renderer, ref_cuda, cam_index, mode):
    import torch

    model, occ = scene
    f = syn.make_frame(model, syn.orbit_cameras(120)[cam_index], 320, 180)
    f.render_mode = mode
    fb, depth = renderer.render(f)
    st = renderer.stats()
    fb_r, depth_r, info = ref_cuda.render(f, renderer, shrink=frame_digests)
    torch.cuda.synchronize()
    assert st.n_samples > 100_000 and info["n_calls"] % 2 == 0 and info["n_inferred"] >= 2 * st.n_samples  # the reference infers every batch twice
    assert sha(fb) == fb_r
    assert sha(depth) == depth_r


def test_north_star_1080p_frames_identical_to_reference_render_nerf(scene, renderer, ref_cuda):
    """configs[0]/[1]: nerf/fox camera C0 and orbit cameras at 1920x1080, no edits: RGBA and depth equal the reference's CUDA path bit for bit."""
    import torch

    model, occ = scene
    cams = [syn.fox_camera0()] + [syn.orbit_cameras(120)[i] for i in (0, 45, 90)]
    for cam in cams:
        f = syn.make_frame(model, cam, 1920, 1080)
        fb, depth = renderer.render(f)
        fb_r, depth_r, info = ref_cuda.render(f, renderer, shrink=frame_digests)
        torch.cuda.synchronize()
        assert (fb[..., 3] > 0).float().mean().item() > 0.2
        assert sha(fb) == fb_r, "RGBA differs from the reference's"
        assert sha(depth) == depth_r


def _edit_sample(fb_ref, fb_unedited, k_region, k_rest, seed):
    """shrink of an edited frame: (pixels drawn, the reference's RGBA there, size of the edit region). k_region pixels are drawn among those
    the edit changes (the reference's frame differs from the unedited one by > 1e-3), k_rest among the others."""
    import torch

    region = ((fb_ref - fb_unedited).abs().amax(-1) > 1e-3).reshape(-1).cpu().numpy()
    rng = np.random.default_rng(seed)
    inside, outside = np.nonzero(region)[0], np.nonzero(~region)[0]
    sel = np.sort(np.concatenate([rng.choice(inside, min(k_region, inside.size), replace=False), rng.choice(outside, k_rest, replace=False)]))
    sel = torch.from_numpy(sel).cuda()
    return sel, fb_ref.reshape(-1, 4)[sel], int(inside.size)


def _edit_scenes(model):
    yield "E1 (configs[2]: one cage)", [c.to_op() for c in e1(model)], 1
    ops = [c.to_op() for c in e3(model)] + [_affine().to_op()]
    yield "E3 + affine, poisson_target on (configs[3])", ops, 1
    yield "E3 + affine, poisson_target off", ops, 0


def test_edit_operator_kernels_vs_reference(scene, renderer):
    model, occ = scene
    ops = [c.to_op() for c in e3(model)] + [_affine().to_op()]
    renderer.set_edit_operators(ops)
    rc = ref.RefCuda(occ, ops)
    try:
        rng = np.random.default_rng(3)
        n = 400_000
        c = np.zeros((n, 7), np.float32)
        c[:, :3] = rng.uniform(0.38, 0.64, (n, 3))
        d = rng.standard_normal((n, 3)).astype(np.float32)
        c[:, 4:] = (d / np.linalg.norm(d, axis=1, keepdims=True) + 1) * 0.5
        c = c[np.sort(np.random.default_rng(30).choice(n, 25_000, replace=False))]  # the reference's outputs are stored for this seeded sample
        k = c.shape[0] / n
        cn, mn = renderer.map_rays(c)
        cr, mr = rc.map_rays(c)
        moved = (cr[:, :3] != c[:, :3]).any(axis=1)
        assert moved.sum() > 20_000 * k and mr.sum() > 10_000 * k
        assert np.array_equal(mn, mr)                                   # empty mask: identical
        assert np.array_equal((cn[:, :3] != c[:, :3]).any(axis=1), moved)  # same samples found a tet / a box
        assert np.array_equal(cn[:, 3:], cr[:, 3:])                     # dt and mapped direction: identical
        assert np.abs(cn[:, :3] - cr[:, :3]).max() <= 2.0 ** -23        # mapped position: 1 ulp (see module docstring)
        sh, od, rd = renderer.poisson_residuals(c)
        sh_r, od_r, rd_r = rc.poisson_residuals(c)
        assert (od_r != 0).sum() > 5000 * k and np.array_equal(od != 0, od_r != 0)
        assert np.allclose(od, od_r, rtol=1e-6, atol=1e-5) and np.allclose(rd, rd_r, rtol=1e-6, atol=1e-5) and np.allclose(sh, sh_r, rtol=1e-6, atol=1e-6)
    finally:
        rc.close()
        renderer.set_edit_operators([])


def test_edited_1080p_frames_vs_reference_render_nerf(scene, renderer):
    """configs[2] and configs[3] at 1920x1080 against the reference's CUDA path (map_rays / compute_poisson_full_residuals / membrane composite)."""
    import torch

    model, occ = scene
    cam = syn.orbit_cameras(120)[17]
    for name, ops, target in _edit_scenes(model):
        renderer.set_edit_operators(ops)
        rc = ref.RefCuda(occ, ops)
        try:
            f = syn.make_frame(model, cam, 1920, 1080)
            f.apply_operators, f.poisson_target = 1, target
            f0 = syn.make_frame(model, cam, 1920, 1080)
            fb0, _ = renderer.render(f0)
            fb0 = fb0.clone()
            fb, depth = renderer.render(f)
            st = renderer.stats()
            sel, fb_r, n_region = rc.render(f, renderer, shrink=lambda o: _edit_sample(o[0], fb0, 15_000, 5_000, 7))
            torch.cuda.synchronize()
            err = (fb.reshape(-1, 4)[sel] - fb_r).abs().amax(-1)
            print(f"\n{name}: L-inf {err.max().item():.3e}, pixels > 1e-4: {(err > 1e-4).sum().item()} of {sel.numel()} sampled ({n_region} in the edit region), "
                  f"edit changed {((fb - fb0).abs().amax(-1) > 1e-3).sum().item()} pixels, old-density samples {st.n_old_samples}")
            assert ((fb - fb0).abs().amax(-1) > 1e-3).sum().item() > 5000
            assert err.max().item() <= 1e-3
            # <= 50 such pixels in the frame: at that rate, were they all in the edit region, the sample would hold 50 * 15,000 / n_region + 50 * 5,000 / (W * H)
            assert (err > 1e-4).sum().item() <= int(np.ceil(50 * (min(15_000, n_region) / n_region + 5_000 / (1920 * 1080))))
        finally:
            rc.close()
            renderer.set_edit_operators([])
