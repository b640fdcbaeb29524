"""The reference-facing surface added in round 2, on the GPU: the C++ shim run through a real frame, the show_accel override against the
reference's own CUDA path, the per-operator EditOperator entry points, the device-pointer uploads."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from edit_fixtures import e3
from nerfshop_b200 import abi, editing
from nerfshop_b200 import synthetic as syn
from oracle import oracle as orc
from ref_golden import Recorded, frame_digests, sha

ref = Recorded("gpu_surface")  # outputs of oracle/_ref's CUDA build stored under tests/golden/ref/ (ref_golden.py)

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

SHIM_MAIN = r'''
#include "nerfshop_b200/host/nerfshop_host.hpp"
#include <cuda_runtime.h>
#include <cstdio>
#include <cstring>
#include <vector>
static std::vector<char> slurp(const char* p) { FILE* f = fopen(p, "rb"); fseek(f, 0, SEEK_END); long n = ftell(f); fseek(f, 0, SEEK_SET); std::vector<char> b(n); fread(b.data(), 1, n, f); fclose(f); return b; }
int main(int argc, char** argv) {
  // argv: params.bin occupancy.bin frame.bin out.bin desc.bin
  auto params = slurp(argv[1]); auto occ = slurp(argv[2]); auto fr = slurp(argv[3]); auto ds = slurp(argv[5]);
  NsbModelDesc d; memcpy(&d, ds.data(), sizeof(d));
  NsbFrame frame; memcpy(&frame, fr.data(), sizeof(frame));
  auto ctx = std::make_shared<ngp_b200::Context>(0);
  ngp_b200::NerfNetwork net(ctx, d);
  uint16_t* params_dev; cudaMalloc(&params_dev, params.size()); cudaMemcpy(params_dev, params.data(), params.size(), cudaMemcpyHostToDevice);
  net.set_params_device(params_dev, params.size() / 2);                     // the Trainer's block stays on the device
  uint8_t* occ_dev; cudaMalloc(&occ_dev, occ.size()); cudaMemcpy(occ_dev, occ.data(), occ.size(), cudaMemcpyHostToDevice);
  ngp_b200::check(nsb_upload_occupancy_dev(ctx->get(), occ_dev, occ.size()), "occupancy");
  ngp_b200::NerfTracer tracer(ctx);
  size_t n = (size_t)frame.width * frame.height;
  float *fb, *depth; cudaMalloc(&fb, n * 16); cudaMalloc(&depth, n * 4); cudaMemset(fb, 0, n * 16); cudaMemset(depth, 0, n * 4);
  uint32_t n_hit = ngp_b200::render_nerf(tracer, frame, fb, depth, false, nullptr, true);
  std::vector<float> out(n * 5);
  cudaMemcpy(out.data(), fb, n * 16, cudaMemcpyDeviceToHost); cudaMemcpy(out.data() + n * 4, depth, n * 4, cudaMemcpyDeviceToHost);
  FILE* f = fopen(argv[4], "wb"); fwrite(out.data(), 4, out.size(), f); fclose(f);
  std::printf("%u\n", n_hit);
  return 0;
}
'''


def test_cpp_shim_renders_the_same_frame(scene, renderer, built_lib, tmp_path):
    """ngp_b200::render_nerf / NerfTracer::trace / NerfNetwork::set_params_device through the C ABI from C++, device-pointer uploads, n_hit returned."""
    model, occ = scene
    f = syn.make_frame(model, syn.orbit_cameras(120)[17], 160, 90)
    (tmp_path / "params.bin").write_bytes(np.ascontiguousarray(model.params, np.uint16).tobytes())
    (tmp_path / "occ.bin").write_bytes(np.ascontiguousarray(occ, np.uint8).tobytes())
    (tmp_path / "frame.bin").write_bytes(bytes(f))
    (tmp_path / "desc.bin").write_bytes(bytes(model.desc))
    src = tmp_path / "main.cpp"
    src.write_text(SHIM_MAIN)
    exe = tmp_path / "shim_render"
    libdir = os.path.dirname(built_lib)
    cuda = "/usr/local/cuda"
    subprocess.run(["/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++", "-std=c++17", "-I", ROOT, "-I", f"{cuda}/include", str(src), "-o", str(exe), "-L", libdir, "-lnerfshop_b200",
                    f"-Wl,-rpath,{libdir}", "-L", f"{cuda}/lib64", "-lcudart", f"-Wl,-rpath,{cuda}/lib64"], check=True)
    out = subprocess.run([str(exe), str(tmp_path / "params.bin"), str(tmp_path / "occ.bin"), str(tmp_path / "frame.bin"), str(tmp_path / "out.bin"), str(tmp_path / "desc.bin")], capture_output=True, text=True, check=True)
    got = np.fromfile(tmp_path / "out.bin", np.float32)
    n = 160 * 90
    fb, depth = renderer.render(f)
    st = renderer.stats()
    assert int(out.stdout.strip()) == st.n_hit > 1000
    assert np.array_equal(got[: 4 * n].reshape(90, 160, 4), fb.cpu().numpy())
    assert np.array_equal(got[4 * n:].reshape(90, 160), depth.cpu().numpy())


@pytest.mark.parametrize("mode,level", [(abi.NSB_RENDER_SHADE, 0), (abi.NSB_RENDER_POSITIONS, 1), (abi.NSB_RENDER_POSITIONS, 0)])
def test_show_accel_override_identical_to_reference(scene, renderer, mode, level):
    """m_nerf.show_accel >= 0: alpha = 1 for every sample (testbed_nerf.cu:788-790), Positions mode colours the occupancy cells (:913-923)."""
    import torch

    model, occ = scene
    f = syn.make_frame(model, syn.orbit_cameras(120)[33], 256, 144)
    f.render_mode, f.min_mip, f.show_accel = mode, level, 1
    rc = ref.RefCuda(occ)
    try:
        fb, depth = renderer.render(f)
        fb_r, depth_r, _ = rc.render(f, renderer, shrink=frame_digests)
        g = abi.NsbFrame.from_buffer_copy(f)
        g.show_accel = 0
        fb_off, _ = renderer.render(g)
        torch.cuda.synchronize()
        assert (fb - fb_off).abs().max().item() > 0.1           # the override is visible
        assert sha(fb) == fb_r and sha(depth) == depth_r      # identical to the reference's frame, bit for bit
        fb_o, _, _, _ = orc.Oracle(model.desc, model.params, occ).render(f)
        assert np.abs(fb.cpu().numpy() - fb_o).max() <= 1e-3
    finally:
        rc.close()


def test_per_operator_virtuals_compose_to_the_loops(scene, renderer):
    """EditOperator::map_rays / compute_poisson_full_residuals / map_positions / compute_poisson_residual_density, one operator at a time in reverse list
    order, reproduce the all-operator entry points (and the fused occupancy update's semantics for positions)."""
    import torch

    model, occ = scene
    ops = [c.to_op() for c in e3(model)] + [editing.AffineDuplication((0.5, 0.5, 0.5), (0.12, 0.12, 0.12), (0.03, 0.0, -0.1), hide_original=True, correct_dir=True).to_op()]
    renderer.set_edit_operators(ops)
    try:
        rng = np.random.default_rng(5)
        n = 100_000
        c = np.zeros((n, 7), np.float32)
        c[:, :3] = rng.uniform(0.38, 0.64, (n, 3))
        d = rng.standard_normal((n, 3)).astype(np.float32)
        c[:, 4:] = (d / np.linalg.norm(d, axis=1, keepdims=True) + 1) * 0.5
        want_c, want_m = renderer.map_rays(c)
        want_sh, want_od, want_rd = renderer.poisson_residuals(c)
        lib, ctx = renderer.lib, renderer.ctx
        ct = torch.from_numpy(c).cuda()
        mask = torch.zeros(n, dtype=torch.uint8, device="cuda")
        sh = torch.zeros((n, 27), device="cuda"); od = torch.zeros(n, device="cuda"); rd = torch.zeros(n, device="cuda")
        for i in range(len(ops) - 1, -1, -1):  # testbed_nerf.cu:2868
            abi.check(lib, lib.nsb_poisson_residuals_op(ctx, i, ct.data_ptr(), n, sh.data_ptr(), od.data_ptr(), rd.data_ptr(), None), "poisson op")
        for i in range(len(ops) - 1, -1, -1):  # :2899
            abi.check(lib, lib.nsb_map_rays_op(ctx, i, ct.data_ptr(), mask.data_ptr(), n, None), "map_rays op")
        torch.cuda.synchronize()
        assert np.array_equal(ct.cpu().numpy(), want_c) and np.array_equal(mask.cpu().numpy(), want_m)
        assert np.array_equal(sh.cpu().numpy(), want_sh) and np.array_equal(od.cpu().numpy(), want_od) and np.array_equal(rd.cpu().numpy(), want_rd)
        # positions: same mapped positions as map_rays where a tet / box maps the sample (interpolate_tet_pos has no direction)
        pos = torch.from_numpy(np.ascontiguousarray(c[:, :3])).cuda()
        pmask = torch.zeros(n, dtype=torch.uint8, device="cuda")
        abi.check(lib, lib.nsb_map_positions(ctx, -1, pos.data_ptr(), 3, pmask.data_ptr(), n, None), "map_positions")
        dens = torch.zeros(n, dtype=torch.float16, device="cuda")
        abi.check(lib, lib.nsb_poisson_residual_density(ctx, -1, pos.data_ptr(), 3, dens.data_ptr(), n, None), "residual density")
        torch.cuda.synchronize()
        assert np.array_equal(pos.cpu().numpy(), want_c[:, :3])
        assert (pmask.cpu().numpy() >= want_m).all()            # interpolate_tet_pos masks the vacated region of copy cages too
        nz = dens.cpu().numpy() != 0
        assert 1000 < nz.sum() < n
    finally:
        renderer.set_edit_operators([])
