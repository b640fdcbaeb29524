"""Pins oracle/ (and the product's host geometry) to oracle/_ref = the reference's OWN sources compiled for the CPU.

oracle/_ref/libnerfshop_ref.so is built by oracle/ref_build.py from /root/reference (unmodified headers, src/common_nerf.cu, and the
functions listed in ref_build.EXTRACTS — Testbed::render_nerf, NerfTracer::trace, init_rays_from_camera, every kernel they launch,
interpolate_tet, translate_in_box, compute_residual_poisson_kernel, Cage::compute_mvc over mvc.h, TetMesh::update_local_rotations
over svd3.h, TetMesh::build_tet_grid) behind stand-ins for the absent submodules (oracle/ref_shim/). Only tiny-cuda-nn's network is
missing: where a frame is rendered, the reference's NerfNetwork::inference_mixed_precision is a call-back into the oracle's.

Comparison rules: integer / index / bit work must be identical. fp32 values that depend on how a compiler contracts a*b+c
into FMAs (the reference sets no -fmad flag: the bits of a real build are nvcc's choice; the GPU tests settle those against
the nvcc build of the same sources, tests/test_gpu_vs_ref_cuda.py) are compared in ulps and every mismatch count is printed.
"""
import ctypes as C

import numpy as np
import pytest

from edit_fixtures import e1, e3, make_cage
from nerfshop_b200 import abi, editing
from nerfshop_b200 import synthetic as syn
from oracle import oracle as orc
from ref_golden import Recorded, sha

ref = Recorded("oracle_vs_ref")  # outputs of oracle/_ref stored under tests/golden/ref/ (ref_golden.py)


_a = 0.4
ROT = np.array([[np.cos(_a), -np.sin(_a), 0], [np.sin(_a), np.cos(_a), 0], [0, 0, 1]], np.float32)


def ulps(a, b):
    a, b = np.ascontiguousarray(a, np.float32), np.ascontiguousarray(b, np.float32)
    return np.abs(a.view(np.int32).astype(np.int64) - b.view(np.int32).astype(np.int64))


# ---- integer / bit-exact functions (random_val.cuh:159-322, common_nerf.cu:117-177, tcnn morton/pcg32) --------------------------
def test_sobol_morton_mip_pcg32_bit_exact():
    L = orc.lib()
    rng = np.random.default_rng(0)
    n = 100_000
    index, seed = rng.integers(0, 2 ** 32, n, dtype=np.uint64).astype(np.uint32), rng.integers(0, 2 ** 32, n, dtype=np.uint64).astype(np.uint32)
    index[:64] = np.arange(64)
    got = ref.ld_random_val(index[:20000], seed[:20000])
    want = np.array([L.orc_ld_random_val(int(i), int(s)) for i, s in zip(index[:20000], seed[:20000])], np.float32)
    assert np.array_equal(got[:20000], want)
    for spp in (0, 1, 2, 5, 17, 1000):
        off = np.zeros(2, np.float32)
        L.orc_pixel_offset(spp, off.ctypes.data)
        assert np.array_equal(off, ref.ld_random_pixel_offset(spp)), spp
    xyz = rng.integers(0, 1024, (20000, 3)).astype(np.uint32)
    assert np.array_equal(ref.morton3D(xyz), np.array([L.orc_morton3D(int(a), int(b), int(c)) for a, b, c in xyz], np.uint32))
    # mip_from_pos / cascaded_grid_idx_at, including the AABB centre (frexpf(0)) and cell boundaries
    pos = rng.uniform(-1.5, 2.5, (20000, 3)).astype(np.float32)
    pos[:8] = 0.5
    pos[8:16] = np.float32(0.5) + np.float32(2.0) ** -np.arange(1, 9, dtype=np.float32)[:, None]
    dt = rng.uniform(0.0015, 0.25, 20000).astype(np.float32)
    mp, md, cell = ref.mip(pos, dt)
    want_mp = np.array([L.orc_mip_from_pos(float(x), float(y), float(z)) for x, y, z in pos], np.int32)
    assert np.array_equal(mp, want_mp)
    want_cell = np.array([L.orc_cascaded_grid_idx_at(float(x), float(y), float(z), int(m)) for (x, y, z), m in zip(pos, md)], np.uint32)
    assert np.array_equal(cell, want_cell)
    # pcg32 with skip-ahead (generate_grid_samples_nerf_nonuniform: rng.advance(i*4))
    for adv in (0, 4, 123456789, 2 ** 40 + 12):
        u, _ = ref.pcg32(1337, 1, adv, 64)
        st = orc.pcg32_seed(1337, 1)
        if adv:
            orc.pcg32_advance(st, adv)
        assert np.array_equal(u, orc.pcg32_next(st, 64)), adv


def test_srgb_sh9_activations():
    rng = np.random.default_rng(1)
    x = rng.uniform(-12, 12, 50000).astype(np.float32)[:10000]  # the reference's outputs are stored for the first 10,000
    # the oracle's composite uses the same formulas; here the numpy restatement of each is the reference function itself
    s = rng.uniform(0, 1.2, 50000).astype(np.float32)[:10000]
    lin = ref.srgb_to_linear(s)
    want = np.where(s <= 0.04045, s / np.float32(12.92), np.power((s + np.float32(0.055)) / np.float32(1.055), np.float32(2.4)))
    assert np.abs(lin - want).max() < 2e-6
    rgb, dens = ref.activations(x, abi.NSB_ACT_LOGISTIC)
    assert np.abs(rgb - 1.0 / (1.0 + np.exp(-x.astype(np.float64)))).max() < 1e-6
    _, dens = ref.activations(x, abi.NSB_ACT_EXPONENTIAL)
    assert np.allclose(dens, np.exp(x.astype(np.float64)), rtol=2e-6)
    rgb, _ = ref.activations(x, abi.NSB_ACT_EXPONENTIAL)
    assert np.allclose(rgb, np.exp(np.clip(x.astype(np.float64), -10, 10)), rtol=2e-6)


# ---- ray generation + occupancy stepping: init_rays_with_payload_kernel_nerf, advance_pos_nerf, generate_next_nerf_network_inputs --
@pytest.mark.parametrize("cam_index,spp", [(17, 0), (63, 0), (99, 5)])
def test_march_vs_reference_kernels(scene, oracle, cam_index, spp):
    model, occ = scene
    W, H, MS = 192, 108, 64
    f = syn.make_frame(model, syn.orbit_cameras(120)[cam_index], W, H, spp=spp)
    pix = np.random.default_rng(cam_index).choice(W * H, 4000, replace=False).astype(np.uint32)
    rec_o, idx_o, cnt_o = oracle.march_trace(f, pix, MS)
    # the reference's sample counts are stored for every ray, its sample stream for a seeded sample of 400 of the rays that have samples
    sub, rec_r, cnt_r = ref.march_trace(f, occ, pix, MS, shrink=lambda o: _stream_sample(o[0], o[2], 400, 100 + cam_index))
    # same rays enter, same number of occupied samples on every ray
    assert np.array_equal(np.minimum(cnt_o, MS), cnt_r)
    assert cnt_r.sum() > 50_000
    rec_o, cnt_r = rec_o[sub], cnt_r[sub]
    amin, amax = np.array(list(f.train_aabb_min), np.float32), np.array(list(f.train_aabb_max), np.float32)
    total = bad_t = bad_p = bad_dt = 0
    max_ulp = 0
    for k in range(sub.size):
        c = int(cnt_r[k])
        if c == 0:
            continue
        t, dt, pos = rec_o[k, :c, 0], rec_o[k, :c, 1], rec_o[k, :c, 2:5]
        total += c
        bad_t += int(((t + dt).astype(np.float32) != rec_r[k, :c, 7]).sum())          # payload.t after `t += dt`
        d = np.abs(((pos - amin) / (amax - amin)).astype(np.float32) - rec_r[k, :c, 0:3])  # warp_position(pos, train_aabb), values in [0, 1]
        bad_p += int((d > 0).any(axis=1).sum())
        max_ulp = max(max_ulp, float(d.max()) / 2.0 ** -24)
    print(f"\ncam {cam_index} spp {spp}: {total} samples; t-stream mismatches {bad_t}; warped positions differing {bad_p} ({100.0 * bad_p / total:.1f} %, max {max_ulp:.1f} ulp of 1.0)")
    # the dt lattice (t, dt, and with them the occupancy cell sequence) is bit-identical to the reference's kernels
    assert bad_t == 0
    # positions: identical up to the FMA contraction of the camera matrix product / normalisation (compiler's choice), i.e. a few ulps
    assert max_ulp <= 8


def _stream_sample(rec, cnt, k, seed):
    """shrink of march_trace: (rays drawn, their records, every ray's count). k rays are drawn among those with samples; of their
    records only the channels the test reads (warped position, payload.t) are kept, zero past each ray's count."""
    sub = np.sort(np.random.default_rng(seed).choice(np.nonzero(cnt)[0], k, replace=False))
    out = np.zeros((k,) + rec.shape[1:2] + (8,), np.float32)
    valid = np.arange(rec.shape[1])[None, :] < cnt[sub, None]
    out[..., [0, 1, 2, 7]] = np.where(valid[..., None], rec[sub][..., [0, 1, 2, 7]], 0)
    return sub, out, cnt


# ---- Testbed::render_nerf of the reference (its own host loop, compaction, composite, shade) with the oracle's network plugged in --
@pytest.mark.parametrize("mode", [abi.NSB_RENDER_SHADE, abi.NSB_RENDER_DEPTH, abi.NSB_RENDER_COST])
def test_frame_vs_reference_render_nerf(scene, oracle, mode):
    model, occ = scene
    f = syn.make_frame(model, syn.orbit_cameras(120)[17], 128, 72)
    f.render_mode = mode
    fb_o, d_o, st, margin = oracle.render(f, want_margin=True)
    fb_r, d_r, info = ref.render(f, occ, lambda c: oracle.inference(c))
    # Depth / Cost colours are not in [0, 1] (z * depth_scale reaches ~10): the 1e-3 contract is applied relative to the value there.
    # A ray whose accumulated alpha lands within 2e-5 of the termination threshold may take the other branch (DESIGN.md section 3).
    err = (np.abs(fb_o - fb_r) / np.maximum(1.0, np.abs(fb_o))).max(-1)
    ok = (margin > 2e-5) | (fb_o[..., 3] == 0)
    print(f"\nmode {mode}: L-inf {err[ok].max():.3e} ({(~ok).sum()} threshold pixels excluded, worst of them {err[~ok].max() if (~ok).any() else 0:.3e}); pixels > 1e-4: {(err > 1e-4).sum()} of {err.size}; "
          f"reference inferred {info['n_inferred']} rows in {info['n_calls']} calls, oracle {st.n_samples} samples")
    assert (fb_r[..., 3] > 0).mean() > 0.3 and (~ok).mean() < 0.02
    # same hit set (compact_kernel_nerf's A > 0.001 filter), same background pixels
    assert np.array_equal(fb_o[..., 3] > 0, fb_r[..., 3] > 0)
    if mode == abi.NSB_RENDER_SHADE:
        assert err[ok].max() <= 1e-3
    else:  # a 1-ulp position difference can move one sample across an occupancy cell face: the debug colours (not in [0,1]) show it
        assert (err[ok] > 1e-3).sum() <= 2 and err[ok].max() < 1e-2  # Cost: one step = 1/128
    assert (err > 1e-4).mean() < 0.01
    hit = fb_r[..., 3] > 0.2
    assert np.abs(d_o - d_r)[hit & (margin > 2e-5)].max() < 0.25  # depth of the max-weight sample: may flip between neighbouring samples
    # the reference infers every round's whole batch twice (testbed_nerf.cu:2892, :2913)
    assert info["n_calls"] % 2 == 0 and info["n_inferred"] >= 2 * st.n_samples


def test_edited_frame_vs_reference_render_nerf(scene):
    """configs[3]-style: three cages (one with membrane arrays, poisson_target on, one copy) + an affine duplication."""
    model, occ = scene
    cages = e3(model)
    ops = [c.to_op() for c in cages]
    aff = editing.AffineDuplication((0.5, 0.5, 0.5), (0.12, 0.12, 0.12), (0.03, 0.0, -0.1), rotation=ROT, hide_original=True, correct_dir=True)
    ops.append(aff.to_op())
    o = orc.Oracle(model.desc, model.params, occ, ops)
    for target in (1, 0):
        f = syn.make_frame(model, syn.orbit_cameras(120)[17], 112, 63)
        f.apply_operators, f.poisson_target = 1, target
        fb_o, d_o, st, margin = o.render(f, want_margin=True)
        plain = orc.Oracle(model.desc, model.params, occ)
        fb_r, d_r, info = ref.render(f, occ, lambda c: plain.inference(c), ops=ops)
        err = np.abs(fb_o - fb_r).max(-1)
        print(f"\nE3+affine poisson_target={target}: L-inf {err.max():.3e}; > 1e-4: {(err > 1e-4).sum()} of {err.size}")
        assert np.abs(fb_o - syn_unedited(model, occ, f)).max() > 0.05  # the edit is visible
        assert err.max() <= 1e-3
        assert (err > 1e-4).mean() < 0.02


def syn_unedited(model, occ, f):
    g = abi.NsbFrame.from_buffer_copy(f)
    g.apply_operators = 0
    return orc.Oracle(model.desc, model.params, occ).render(g)[0]


# ---- EditOperator::map_rays / compute_poisson_full_residuals: interpolate_tet, translate_in_box, compute_residual_poisson_kernel ----
def test_map_rays_and_poisson_vs_reference_kernels(scene):
    model, occ = scene
    cages = e3(model)
    ops = [c.to_op() for c in cages]
    ops.append(editing.AffineDuplication((0.5, 0.5, 0.5), (0.12, 0.12, 0.12), (0.03, 0.0, -0.1), rotation=ROT, hide_original=True, correct_dir=True).to_op())
    o = orc.Oracle(model.desc, model.params, occ, ops)
    rng = np.random.default_rng(3)
    n = 120_000
    c = np.zeros((n, 7), np.float32)
    c[:, :3] = rng.uniform(0.38, 0.64, (n, 3))  # around the cages (warped units)
    d = rng.standard_normal((n, 3)).astype(np.float32)
    c[:, 4:] = (d / np.linalg.norm(d, axis=1, keepdims=True) + 1) * 0.5
    co, mo = o.map_rays(c)
    moved = (co[:, :3] != c[:, :3]).any(axis=1)
    assert moved.sum() > 5000 and mo.sum() > 300
    # the reference's outputs are stored for a seeded sample of 20,000 of the coordinates
    sub = np.sort(np.random.default_rng(30).choice(n, 20_000, replace=False))
    c, co, mo, moved = c[sub], co[sub], mo[sub], moved[sub]
    bound = lambda m: int(np.ceil(m * sub.size / n))  # a count allowed over all n coordinates, at the same rate over the sample
    cr, mr = ref.map_rays(ops, c)
    flips = int((mo != mr).sum()) + int(((cr[:, :3] != c[:, :3]).any(axis=1) != moved).sum())
    dpos, ddir = np.abs(co[:, :3] - cr[:, :3]) / 2.0 ** -24, np.abs(co[:, 4:] - cr[:, 4:]) / 2.0 ** -24  # warped values live in [0, 1]: in ulps of 1.0
    big = (dpos > 64).any(axis=1)  # a sample that landed in a different tet on a shared face would show as a large jump
    print(f"\nmap_rays: {moved.sum()} moved, {mo.sum()} masked; mask/moved flips {flips}; position max {dpos.max():.1f} ulp ({(dpos > 0).any(axis=1).sum()} differ), direction max {ddir.max():.1f} ulp; {big.sum()} large jumps")
    assert flips <= bound(2) and big.sum() <= bound(2)
    assert np.percentile(dpos.max(axis=1), 99.9) <= 8 and np.percentile(ddir.max(axis=1), 99.9) <= 8
    sh_o, od_o, rd_o = o.poisson_residuals(c)
    sh_r, od_r, rd_r = ref.poisson_residuals(ops, c)
    inside = od_o != 0
    assert inside.sum() > 2000 * sub.size / n and np.array_equal(inside, od_r != 0) or abs(int(inside.sum()) - int((od_r != 0).sum())) <= 2
    both = inside & (od_r != 0)
    assert np.allclose(od_o[both], od_r[both], rtol=2e-5, atol=1e-5) and np.allclose(rd_o[both], rd_r[both], rtol=2e-5, atol=1e-5)
    assert np.allclose(sh_o[both], sh_r[both], rtol=2e-5, atol=2e-5)


# ---- per-edit geometry of the PRODUCT's host code vs mvc.h / svd3.h / tet_mesh.cu --------------------------------------------------
def test_mvc_vs_reference_mvc_h(scene):
    model, _ = scene
    cage = make_cage(model, (0.5, 0.62, 0.78), (0.17, 0.17, 0.17), n_lattice=4)
    pts = cage.original_vertices.copy()
    rng = np.random.default_rng(0)
    extra = rng.uniform(0.2, 1.0, (500, 3)).astype(np.float32)          # inside and outside the cage
    on_vertex = cage.cage_original[:3].copy()                            # special case: on a cage vertex -> one-hot
    on_face = (cage.cage_original[cage.cage_triangles[0]] * np.array([[0.2], [0.3], [0.5]], np.float32)).sum(0, keepdims=True)  # 2-D barycentric
    pts = np.concatenate([pts, extra, on_vertex, on_face]).astype(np.float32)
    for gamma in (0.0, 2.0):
        w_ref = ref.compute_mvc(cage.cage_original, cage.cage_triangles, pts, gamma=gamma if gamma else 1.0, original=gamma == 0.0)
        w = np.zeros_like(w_ref)
        assert cage.lib.nsb_compute_mvc(cage.cage_original.ctypes.data, cage.cage_original.shape[0], cage.cage_triangles.ctypes.data, cage.cage_triangles.shape[0],
                                        pts.ctypes.data, pts.shape[0], gamma, w.ctypes.data) == 0
        n_in = cage.original_vertices.shape[0]
        e = np.abs(w - w_ref).max(axis=1)
        print(f"\nMVC gamma={gamma}: max |w - w_ref| = {e[:n_in].max():.3e} over the {n_in} tet-mesh vertices (inside the cage: what the operator uses), "
              f"{e[n_in:].max():.3e} over {e.size - n_in} arbitrary points (mvc.h stores its intermediates in float; outside the cage the weights exceed 1 and its rounding noise shows)")
        assert e[:n_in].max() < 5e-6
        assert e[n_in:].max() < 5e-3
        assert np.array_equal(w[-4:-1], w_ref[-4:-1])  # on a cage vertex: one-hot in both
        assert np.abs(w_ref.sum(1) - 1).max() < 1e-5


def test_local_rotations_vs_reference_svd3(scene):
    """TetMesh::update_local_rotations: R = U V^T from svd3.h, no reflection fix — including a mirrored and a flattened tet."""
    model, _ = scene
    cage = make_cage(model, (0.5, 0.62, 0.78), (0.17, 0.17, 0.17), n_lattice=3)
    ov, tets = cage.original_vertices.copy(), cage.tets.copy()
    dv = cage.vertices.copy()
    t_mirror, t_flat = 5, 9
    vm = tets[t_mirror]
    used_elsewhere = lambda v: (tets == v).sum() > 1
    dv2 = dv.copy()
    # deform every vertex of a mirrored / flattened tet (shared vertices drag their neighbours along: all rotations are compared)
    dv2[vm] = dv[vm] * np.array([-1, 1, 1], np.float32) + np.array([2 * 0.5, 0, 0], np.float32)  # mirror in x about x = 0.5
    vf = tets[t_flat]
    dv2[vf, 2] = dv[vf, 2].mean()                                                              # flatten in z
    rot_ref, off_ref, idx_ref, bbox_ref, obits_ref = ref.tet_mesh_build(ov, dv2, tets, model.aabb_min, model.aabb_max)
    rot = np.zeros((tets.shape[0], 9), np.float32)
    assert cage.lib.nsb_local_rotations(dv2.ctypes.data, ov.ctypes.data, tets.ctypes.data, tets.shape[0], rot.ctypes.data) == 0
    err = np.abs(rot - rot_ref).max(axis=1)
    dets = np.array([np.linalg.det(r.reshape(3, 3)) for r in rot_ref])
    print(f"\nrotations: max err {err.max():.3e}; reference det range [{dets.min():.3f}, {dets.max():.3f}]; worst tets {np.argsort(err)[-3:]}")
    # svd3.h keeps U and V proper rotations (the smallest singular value carries the sign): R is a rotation even for the mirrored tets
    assert np.abs(dets - 1).max() < 1e-3
    flat = np.array([np.linalg.matrix_rank((dv2[t[1:]] - dv2[t[0]]).astype(np.float64), tol=1e-6) < 3 for t in tets])
    print(f"  {flat.sum()} flattened tets: max err {err[flat].max():.3e} (svd3.h's 4 approximate Jacobi sweeps on a rank-2 matrix); others {err[~flat].max():.3e}")
    # svd3.h is the approximate side (4 fixed Jacobi sweeps, rsqrt-based Givens): against numpy's SVD in float64 the product is within
    # 1e-7 and svd3.h within 1.1e-3 on the strongly sheared neighbours of the mirrored tet; ordinary tets agree to float rounding
    assert np.percentile(err, 90) < 1e-5
    assert err.max() < 3e-3


def test_tet_grid_vs_reference_build_tet_grid(scene):
    """TetMesh::build_tet_grid (tet_mesh.cu:368-673) and build_original_tet_grid (:76-235), the reference's own code on a deformed lattice cage:
    the product's host rebuild (nsb_host_geometry.cpp, what the GPU rebuild kernels are pinned to) yields the same per-cell tet SETS (the
    reference appends in tet order per thread chunk; the interpolate_tet walk takes the first containing tet, so order is compared too where
    the reference's is deterministic: it is, its 32 std::threads write disjoint cell ranges), the same CSR offsets, and the same canonical bitfield."""
    model, _ = scene
    cage = make_cage(model, (0.5, 0.62, 0.78), (0.17, 0.17, 0.17), n_lattice=4)
    rot_ref, off_ref, idx_ref, bbox_ref, obits_ref = ref.tet_mesh_build(cage.original_vertices, cage.vertices, cage.tets, model.aabb_min, model.aabb_max)
    off, idx = cage.lut_offsets, np.asarray(cage.lut_idx)
    assert off_ref[-1] == idx_ref.size and off[-1] == idx.size
    print(f"\ntet LUT: {idx.size} entries here, {idx_ref.size} in the reference build; occupied cells {np.count_nonzero(np.diff(off))} / {np.count_nonzero(np.diff(off_ref))}")
    same_offsets = np.array_equal(off, off_ref)
    if same_offsets:
        same_order = np.array_equal(idx, idx_ref)
        if not same_order:  # same sets per cell?
            cells = np.nonzero(np.diff(off))[0]
            bad = [c for c in cells if sorted(idx[off[c]:off[c + 1]]) != sorted(idx_ref[off[c]:off[c + 1]])]
            assert not bad, f"{len(bad)} cells hold different tet sets, e.g. cell {bad[0]}"
        print(f"  offsets identical; lists identical in order: {same_order}")
    else:
        # conservative rasterisation may differ on cells a tet only touches: every reference entry must be present here or vice versa — report both
        n_cells = off.size - 1
        cnt, cnt_ref = np.diff(off).astype(np.int64), np.diff(off_ref).astype(np.int64)
        diff = np.nonzero(cnt != cnt_ref)[0]
        print(f"  {diff.size} of {n_cells} cells differ in list length (here-minus-reference: min {int((cnt - cnt_ref)[diff].min())}, max {int((cnt - cnt_ref)[diff].max())})")
        missing = 0
        for c in diff[:20000]:
            a, b = set(idx[off[c]:off[c + 1]].tolist()), set(idx_ref[off_ref[c]:off_ref[c + 1]].tolist())
            missing += len(b - a)
        assert missing == 0, f"{missing} reference (cell, tet) pairs are absent from the product's LUT"
    assert np.array_equal(cage.original_bitfield, obits_ref), f"{np.count_nonzero(cage.original_bitfield != obits_ref)} canonical-bitfield bytes differ"
    bb = np.stack([cage.vertices.min(0), cage.vertices.max(0)])
    assert np.array_equal(bb, bbox_ref[:2]) or np.allclose(bb, bbox_ref[:2], atol=0), (bb, bbox_ref)


def test_occupancy_update_sample_draw_vs_reference_kernel(scene, oracle):
    """Row (f)-2: generate_grid_samples_nerf_nonuniform (common_nerf.cu:179-208), the reference's own kernel, against the sample draw inside the
    oracle's update_density_grid — both launches (uniform, then non-uniform on m_rng advanced by 2^32), warped positions bit for bit."""
    from nerfshop_b200.rng import Pcg32

    rng0 = Pcg32(4242)
    grid0 = np.zeros(abi.NSB_GRID_CELLS, np.float32)
    grid0[::3] = 0.02      # cells above the non-uniform threshold 0.01
    grid0[5::7] = -1.0     # untrained cells both passes must step over
    n_uni, n_non, step, n_casc = 20_000, 12_000, 7, 3
    u = abi.NsbGridUpdate()
    u.n_uniform_samples, u.n_nonuniform_samples, u.reset_grid, u.n_cascades = n_uni, n_non, 0, n_casc
    u.decay, u.ema_step, u.rng_state, u.rng_inc = 0.95, step, rng0.state, rng0.inc
    u.train_aabb_min[:] = (-1.5, -1.5, -1.5)
    u.train_aabb_max[:] = (2.5, 2.5, 2.5)
    u.density_activation, u.apply_operators = abi.NSB_ACT_EXPONENTIAL, 0
    _, _, _, samples = oracle.update_density_grid(u, grid0, want_samples=True)
    amin, amax = np.array(list(u.train_aabb_min), np.float32), np.array(list(u.train_aabb_max), np.float32)
    pos1, idx1 = ref.grid_samples(n_uni, rng0.state, rng0.inc, step, amin, amax, grid0, n_casc, -0.01)
    r2 = rng0.copy()
    r2.advance(1 << 32)  # m_rng.advance() between the two launches (testbed_nerf.cu:3576)
    pos2, idx2 = ref.grid_samples(n_non, r2.state, r2.inc, step, amin, amax, grid0, n_casc, 0.01)
    # both are warp_position(pos, aabb): what NerfNetwork::density is fed
    got = samples[:, :3]
    want = np.concatenate([pos1, pos2])
    same = (got == want).all(axis=1)
    print(f"\noccupancy-update sample draw: {same.sum()} of {same.size} warped positions identical; max |diff| {np.abs(got - want).max():.2e}")
    assert same.mean() > 0.999 and np.abs(got - want).max() < 1e-6
    G = 128 ** 3
    assert (idx1 < n_casc * G).all() and (idx2 < n_casc * G).all() and (grid0[idx2] > 0.01).mean() > 0.9  # ten tries at one cell in three


@pytest.mark.parametrize("fill", ["sparse", "dense_low"])
def test_bitfield_from_density_grid_vs_reference_kernels(fill):
    """Row (f)-2 / snapshot load: grid_to_bitfield + bitfield_max_pool (testbed_nerf.cu:514-555), launched as update_density_grid_mean_and_bitfield
    does (:3642-3658), against the oracle's density-grid -> bitfield conversion (to which nsb_upload_density_grid / nsb_update_density_grid are
    pinned). The threshold is min(NERF_MIN_OPTICAL_THICKNESS, mean): one case on each side of it."""
    rng = np.random.default_rng(3)
    G = 128 ** 3
    grid = np.zeros(abi.NSB_GRID_CELLS, np.float32)
    if fill == "sparse":   # mean < 0.01: the mean is the threshold
        idx = rng.choice(3 * G, 200_000, replace=False)
        grid[idx] = rng.uniform(0.0, 0.5, idx.size).astype(np.float32)
        grid[rng.choice(3 * G, 5000, replace=False)] = -1.0
    else:                  # mean > 0.01: NERF_MIN_OPTICAL_THICKNESS is
        grid[: 3 * G] = rng.uniform(0.0, 0.06, 3 * G).astype(np.float32)
    bits_o, mean_o = orc.density_grid_to_bitfield(grid)
    bits_r = ref.grid_to_bitfield(grid, mean_o, shrink=sha)  # compared bit for bit: its digest is stored
    exact_mean = float(np.maximum(grid[:G].astype(np.float64), 0).sum() / G)  # the reference reduces the first cascade only (n_elements = 128^3)
    print(f"\n{fill}: mean {mean_o:.6g} (float64 sum {exact_mean:.6g}); bitfield identical {sha(bits_o) == bits_r}; set bits {np.unpackbits(bits_o).sum()}")
    assert abs(mean_o - exact_mean) <= 1e-6 * max(exact_mean, 1e-6) + 1e-9
    assert (mean_o < 0.01) == (fill == "sparse")
    assert sha(bits_o) == bits_r
    assert np.unpackbits(bits_o).sum() > 100_000


@pytest.mark.parametrize("edited", [False, True])
def test_occupancy_update_vs_reference_update_density_grid_nerf_operator(scene, oracle, edited):
    """Row (f)-2 end to end: the reference's OWN Testbed::update_density_grid_nerf_operator + update_density_grid_mean_and_bitfield
    (testbed_nerf.cu:3533-3658: sample draw, map_positions through the operators in reverse order, NerfNetwork::density, activate_network_density,
    compute_poisson_residual_density, max-splat, EMA merge, mean, grid_to_bitfield, max-pools) with the oracle's density network plugged in, against
    the oracle's update_density_grid — two consecutive updates (reset, then merge on an advanced m_rng), with and without E3 + membrane + affine."""
    from nerfshop_b200.rng import Pcg32

    model, occ = scene
    ops = None
    o = oracle
    if edited:
        cages = e3(model)
        ops = [c.to_op() for c in cages]
        ops.append(editing.AffineDuplication((0.5, 0.5, 0.5), (0.12, 0.12, 0.12), (0.03, 0.0, -0.1), rotation=ROT, hide_original=True, correct_dir=True).to_op())
        o = orc.Oracle(model.desc, model.params, occ, ops)
    plain = oracle

    def density(pos):  # NerfNetwork::density: direction-free, rows = the density network's 16 outputs
        c = np.zeros((pos.shape[0], 7), np.float32)
        c[:, :3] = pos
        c[:, 4:] = 0.5
        return plain.inference(c, density_only=True)

    rng = Pcg32(99)
    us = []
    for step, (n_uni, n_non, reset) in enumerate([(120_000, 0, True), (60_000, 40_000, False)]):
        u = abi.NsbGridUpdate()
        u.n_uniform_samples, u.n_nonuniform_samples, u.reset_grid, u.n_cascades = n_uni, n_non, int(reset), 3
        u.decay, u.ema_step, u.rng_state, u.rng_inc = 0.95, step, rng.state, rng.inc
        u.train_aabb_min[:] = tuple(model.aabb_min)
        u.train_aabb_max[:] = tuple(model.aabb_max)
        u.density_activation, u.apply_operators = abi.NSB_ACT_EXPONENTIAL, int(edited)
        us.append(u)
        rng.advance(); rng.advance()  # m_rng.advance() after each of the two sample-generation launches
    grid0 = np.full(abi.NSB_GRID_CELLS, 0.25, np.float32)  # reset_grid must wipe this

    def reference(us, grid, ops):  # both updates chained on the reference's own grid
        out = []
        for u in us:
            grid, bits, mean = ref_lib.update_density_grid(u, grid, density, ops=ops)
            out.append((grid, bits, mean))
        return out

    def shrink(out):  # per update: the touched set as a digest, the grid at 20,000 of its touched cells, the bitfield, the mean
        res = []
        for grid, bits, mean in out:
            touched = np.nonzero(grid > 0)[0]
            sel = np.sort(np.random.default_rng(7).choice(touched, 20_000, replace=False))
            res += [sha(np.packbits(grid > 0)), touched.size, sel.astype(np.uint32), grid[sel], bits, mean]
        return tuple(res)

    from oracle import ref as ref_lib

    rec = ref.run("update_density_grid x2", reference, us, grid0, ops, shrink=shrink, also=model.params)
    grid_o = grid0
    for step, u in enumerate(us):
        grid_o, bits_o, mean_o = o.update_density_grid(u, grid_o)
        touched_sha, n_touched, sel, grid_r, bits_r, mean_r = rec[6 * step: 6 * step + 6]
        touched = grid_o > 0
        assert sha(np.packbits(touched)) == touched_sha and touched.sum() == n_touched, "same cells touched"
        assert n_touched > 50_000
        bound = lambda m: int(np.ceil(m * sel.size / n_touched))  # a count allowed over all touched cells, at the same rate over the sample
        same = grid_o[sel] == grid_r
        rel = np.abs(grid_o[sel] - grid_r) / np.maximum(grid_r, 1e-12)
        print(f"\n{'E3+affine' if edited else 'no operators'} step {step}: {n_touched} cells touched, {(~same).sum()} of {sel.size} sampled differ (max rel {rel.max():.2e}); "
              f"mean {mean_o:.6g} vs {mean_r:.6g}; bitfield bytes differing {np.count_nonzero(bits_o != bits_r)}")
        # positions may differ by an ulp where the operators map them (gcc vs nvcc contraction of the tet barycentrics, DESIGN.md section 3): the raw
        # fp16 density of such a sample moves by a few fp16 ulps (1 ulp = 1e-3 relative) — a handful of cells in 10^5
        # and a sample within an ulp of a tet face may be mapped by one build and not by the other: at most a few cells in 10^5 differ freely
        assert (~same).sum() <= bound(1e-4 * n_touched + 2) and (rel > 1e-2).sum() <= bound(3)
        assert abs(mean_o - mean_r) <= 1e-6 * max(mean_r, 1e-6) + 1e-9
        assert np.count_nonzero(bits_o != bits_r) <= 2


def test_accumulate_and_tonemap_vs_reference_kernels():
    """Row (f)-4: accumulate_kernel and tonemap_kernel (render_buffer.cu:217-252, 254-332, 471-501), the reference's own, against the oracle's
    accumulate / tonemap (to which nsb_accumulate / nsb_tonemap are pinned): every colour space, every curve, HDR and negative inputs."""
    rng = np.random.default_rng(8)
    H, W = 37, 53
    frame = rng.uniform(-0.2, 3.0, (H, W, 4)).astype(np.float32)
    frame[..., 3] = rng.uniform(0.0, 1.0, (H, W)).astype(np.float32)
    worst_acc = worst_tm = 0.0
    sel = np.sort(np.random.default_rng(9).choice(H * W, 400, replace=False))  # the reference's tonemapped frames are stored at these pixels
    for cs in (abi.NSB_COLOR_LINEAR, abi.NSB_COLOR_SRGB, abi.NSB_COLOR_VISPOSNEG):
        acc_o = acc_r = np.zeros_like(frame)
        for spp in range(3):
            fr = (frame * np.float32(1.0 + 0.1 * spp)).astype(np.float32)
            acc_o = orc.accumulate(fr, acc_o, spp, cs)
            acc_r = ref.accumulate(fr, acc_r, spp, cs)
            worst_acc = max(worst_acc, float(np.abs(acc_o - acc_r).max()))
            assert np.allclose(acc_o, acc_r, rtol=2e-6, atol=2e-7), (cs, spp)
        for curve in (abi.NSB_TONEMAP_IDENTITY, abi.NSB_TONEMAP_ACES, abi.NSB_TONEMAP_HABLE, abi.NSB_TONEMAP_REINHARD):
            for out_cs, clamp, exposure in ((abi.NSB_COLOR_SRGB, 1, 0.0), (abi.NSB_COLOR_LINEAR, 0, 0.7), (abi.NSB_COLOR_SRGB, 0, -1.3)):
                p = abi.NsbTonemap()
                p.color_space, p.output_color_space, p.tonemap_curve, p.clamp_output_color, p.exposure = cs, out_cs, curve, clamp, exposure
                p.background_color[:] = (0.2, 0.4, 0.6, 0.8)
                t_o = orc.tonemap(acc_o, p).reshape(-1, 4)[sel]
                t_r = ref.tonemap(acc_r, exposure, list(p.background_color), cs, out_cs, curve, bool(clamp), shrink=lambda t: t.reshape(-1, 4)[sel])
                err = np.abs(t_o - t_r) / np.maximum(1.0, np.abs(t_r))
                finite = np.isfinite(t_r)
                assert np.array_equal(np.isfinite(t_o), finite)
                worst_tm = max(worst_tm, float(err[finite].max()))
                assert err[finite].max() < 2e-6, (cs, curve, out_cs, clamp, exposure, float(err[finite].max()))
    print(f"\naccumulate max |diff| {worst_acc:.2e}; tonemap max relative diff {worst_tm:.2e}")


def test_membrane_blend_vs_reference_loop():
    """Row (f)-4: the gamma-weighted blend of GrowingSelection::interpolate_poisson_boundary (growing_selection.cu:2363-2392), the reference's own
    statements, against the oracle's membrane_blend (to which nsb_cage_set_membrane's k_membrane_blend is pinned bit for bit)."""
    rng = np.random.default_rng(21)
    nv, ncv = 300, 26
    gamma = rng.uniform(-0.05, 1.0, (nv, ncv)).astype(np.float32)
    gamma /= gamma.sum(1, keepdims=True)  # mean-value-like coordinates: partition of unity, a few negative
    din = rng.uniform(0.0, 40.0, ncv).astype(np.float32)
    dout = rng.uniform(0.05, 60.0, ncv).astype(np.float32)
    din[:3] = 0.0
    shs_in = rng.normal(0, 0.5, (ncv, 27)).astype(np.float32)
    shs_out = rng.normal(0, 0.5, (ncv, 27)).astype(np.float32)
    got = orc.membrane_blend(gamma, din, dout, shs_in, shs_out)
    want = ref.membrane_blend(gamma, din, dout, shs_in, shs_out)
    for name, a, b in zip(("boundary_shs", "outside_density", "residual_density"), got, want):
        d = np.abs(a - b)
        print(f"\n{name}: identical {np.array_equal(a, b)}, max |diff| {d.max():.2e} (values up to {np.abs(b).max():.1f})")
        assert np.allclose(a, b, rtol=3e-6, atol=1e-6), name
    assert (want[2] >= 0).all() and np.abs(want[0]).max() > 0.01


def test_edits_file_objects_through_the_reference_serialisers(tmp_path, scene):
    """Row (f)-3: what nerfshop_b200.edits_io writes for a cage operator (proxy cage with membrane values + interpolation tet mesh) and for an affine
    box is READ by the reference's own from_json into its Cage / TetMesh / AffineBoundingBox classes (cage.h:123-144, tet_mesh.h:156-174,
    affine_bounding_box.cuh:116-126 over json_binding.h:27-87) and WRITTEN back by its to_json: every key the reference reads is present, every array
    survives with its shape convention (vectors as [x, y, z], SH9RGB as 9 rows of 3, index lists flat), and edits_io reads the reference's output back
    into an identical operator."""
    import json

    from nerfshop_b200 import edits_io

    model, _ = scene
    cage = make_cage(model, (0.5, 0.62, 0.78), (0.17, 0.17, 0.17), n_lattice=3)
    rng = np.random.default_rng(5)
    nc = cage.cage_original.shape[0]
    cage.cage_shs = {"inside_shs": rng.normal(0, .3, (nc, 27)).astype(np.float32), "outside_shs": rng.normal(0, .3, (nc, 27)).astype(np.float32),
                     "inside_density": rng.uniform(0, 20, nc).astype(np.float32), "outside_density": rng.uniform(1, 30, nc).astype(np.float32)}
    R = np.array([[0.8, -0.6, 0], [0.6, 0.8, 0], [0, 0, 1]], np.float32)
    aff = edits_io.AffineDuplicationWorld(edits_io.AffineBox((0.9, 0.7, 0.5), (0.2, 0.3, 0.2), R), (0.15, 0.05, -0.1), model.aabb_min, model.aabb_max,
                                          scale=(1.2, 1.0, 0.8), rotation=R, hide_original=True, correct_dir=True)
    path = str(tmp_path / "edits.json")
    edits_io.save_edits(path, [cage, aff])
    j = json.load(open(path))
    cj, aj = j["edit_operators"]

    def same(a, b, what):
        a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
        assert a.shape == b.shape, (what, a.shape, b.shape)
        assert np.array_equal(a.astype(np.float32), b.astype(np.float32)), what

    # Cage: from_json reads all 15 keys with .at() — a missing or mis-shaped one throws inside the reference's code
    cage_back = ref.json_roundtrip(ref.JSON_CAGE, cj["proxy_cage"])
    assert list(cage_back) == ["vertices", "indices", "normals", "initial_normals", "labels", "original_vertices", "colors", "outside_colors", "initial_colors",
                               "new_shs", "initial_shs", "inside_shs", "outside_shs", "inside_density", "outside_density"]  # cage.h:102-121, in that order
    for k in cage_back:
        same(cage_back[k], cj["proxy_cage"][k], f"proxy_cage.{k}")
    assert np.asarray(cage_back["inside_shs"]).shape == (nc, 9, 3)
    # TetMesh
    mesh_back = ref.json_roundtrip(ref.JSON_TET_MESH, cj["interpolation_mesh"])
    assert list(mesh_back) == ["bbox", "original_bbox", "warped_bbox", "original_warped_bbox", "vertices", "indices", "original_vertices", "mvc_coordinates",
                               "gamma_coordinates", "tets", "labels", "colors", "all_indices"]  # tet_mesh.h:139-154
    for k in mesh_back:
        if k.endswith("bbox"):
            same(mesh_back[k]["min"], cj["interpolation_mesh"][k]["min"], k)
            same(mesh_back[k]["max"], cj["interpolation_mesh"][k]["max"], k)
        else:
            same(mesh_back[k], cj["interpolation_mesh"][k], f"interpolation_mesh.{k}")
    # AffineBoundingBox, both of the reference's writers (free function and member)
    for kind in (ref.JSON_AFFINE_BOX, ref.JSON_AFFINE_BOX_MEMBER):
        box_back = ref.json_roundtrip(kind, aj["selection_box"])
        assert set(box_back) == {"min", "max", "rot_matrix", "u", "v", "w", "center", "scale"}
        for k in box_back:
            same(box_back[k], aj["selection_box"][k], f"selection_box.{k}")
    # and the other direction: the file rebuilt from the reference's output loads into an identical operator list
    cj2 = dict(cj, proxy_cage=cage_back, interpolation_mesh=mesh_back)
    aj2 = dict(aj, selection_box=ref.json_roundtrip(ref.JSON_AFFINE_BOX, aj["selection_box"]))
    path2 = str(tmp_path / "edits_ref.json")
    json.dump({"edit_operators": [cj2, aj2]}, open(path2, "w"))
    ops1 = edits_io.load_edits(path, model.aabb_min, model.aabb_max)
    ops2 = edits_io.load_edits(path2, model.aabb_min, model.aabb_max)
    for o1, o2 in zip(ops1, ops2):
        p1, k1 = o1.to_op()
        p2, k2 = o2.to_op()
        cut = abi.NsbEditOp.tet_lut_offsets.offset
        assert bytes(p1)[:cut] == bytes(p2)[:cut] and bytes(p1)[abi.NsbEditOp.selection_box.offset:] == bytes(p2)[abi.NsbEditOp.selection_box.offset:]
        for name in k1:
            assert np.array_equal(k1[name], k2[name]), name


@pytest.mark.parametrize("is_inside", [0, 1])
def test_membrane_boundary_values_vs_reference_compute_poisson_boundary(scene, oracle, is_inside):
    """Row (f)-4: GrowingSelection::compute_poisson_boundary (growing_selection.cu:2220-2348), the reference's own — direction sampling on the
    hemisphere grid, inference, activate_network_output, filter_empty (inside pass), density of each vertex's first sample, Monte-Carlo SH9 fit with
    project_sh9 (sh_utils.cu:30-70) — with the oracle's network plugged in, against the oracle's poisson_boundary fed the SAME jitter: the reference
    draws it with std::rand(), so libc's generator is seeded identically for both (the product draws from a seeded pcg32 instead, DESIGN.md section 7)."""
    import ctypes

    model, occ = scene
    libc = ctypes.CDLL(None)
    libc.rand.restype = ctypes.c_int
    rng = np.random.default_rng(17)
    n, w = 23, 6
    pts = (rng.uniform(0.25, 0.75, (n, 3)) * (np.array(model.aabb_max) - np.array(model.aabb_min)) + np.array(model.aabb_min)).astype(np.float32)
    p = abi.NsbBoundarySampling()
    p.sampling_width, p.hemisphere_width, p.seed = w, 7, 0
    p.train_aabb_min[:] = tuple(model.aabb_min)
    p.train_aabb_max[:] = tuple(model.aabb_max)
    p.rgb_activation, p.density_activation, p.is_inside = abi.NSB_ACT_LOGISTIC, abi.NSB_ACT_EXPONENTIAL, is_inside
    libc.srand(4242)
    uniforms = (np.array([libc.rand() for _ in range(2 * n * w * w)], np.float32) / np.float32(2147483647)).astype(np.float32)  # (float)std::rand() / RAND_MAX
    d_o, sh_o, coords_o = oracle.poisson_boundary_with_jitter(pts, p, uniforms)
    libc.srand(4242)
    d_r, sh_r, coords_r = ref.poisson_boundary(pts, p, occ, lambda c: oracle.inference(c))
    coords_r = coords_r[: n * w * w]  # the reference pads the batch to tcnn::batch_size_granularity
    dpos = np.abs(coords_o[:, :3] - coords_r[:, :3]).max()
    ddir = np.abs(coords_o[:, 4:] - coords_r[:, 4:]).max()
    print(f"\nis_inside {is_inside}: sample positions max |diff| {dpos:.1e}, directions {ddir:.1e}; density identical {np.array_equal(d_o, d_r)} "
          f"(max |diff| {np.abs(d_o - d_r).max():.2e}, {np.count_nonzero(d_r == 0)} filtered); SH max |diff| {np.abs(sh_o - sh_r).max():.2e} of {np.abs(sh_r).max():.2f}")
    assert dpos == 0.0 and ddir < 3e-7  # cos/sin/acos: glibc float vs the reference's double intermediates (std::cos of a float promotes nothing; M_PI is double)
    assert np.array_equal(d_o == 0, d_r == 0)
    assert np.allclose(d_o, d_r, rtol=2e-3, atol=1e-6)   # a direction 1 ulp apart may move the raw fp16 density by an ulp
    assert np.abs(sh_o - sh_r).max() < 2e-3 * max(1.0, float(np.abs(sh_r).max()))
    if is_inside:
        assert np.count_nonzero(d_r == 0) > 0
