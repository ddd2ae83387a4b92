"""-m gpu: bfloat16 GRID STORAGE for inference (LrfField.grid_dtype = LRF_GRID_BF16,
TensorBase.set_grid_storage("bf16")).

The kernels gather 16-bit texels (a density texel = one 16-byte load, an appearance texel three) and
compute in fp32; bf16 -> fp32 is exact.  So the claim that is tested is an EQUALITY, not an
approximation: on a field whose grids are bf16-representable the bf16-storage render equals the
fp32-storage render (same arithmetic, same order), and therefore holds the same 1e-4 bar against the
oracle / the unmodified reference evaluated on those parameters.  On arbitrary parameters the
bf16-storage render is the fp32 render of the rounded field."""
import ctypes as C
import json
import os

import numpy as np
import pytest
import torch

import localrf_b200 as L
from localrf_b200 import _lib
from gpu_helpers import module_from_golden, oracle_fields
from helpers import GOLDEN, check_with_ties, load_golden, rel_err, state_digest

pytestmark = pytest.mark.gpu
TOL = 1e-4


def grids(m):
    return [p for plist in (m.density_plane, m.density_line, m.app_plane, m.app_line) for p in plist]


def round_grids_to_bf16(m):
    """In place: every plane / line value becomes bf16-representable (round to nearest even)."""
    with torch.no_grad():
        for p in grids(m):
            p.copy_(p.to(torch.bfloat16).to(torch.float32))
    return m


def rays512(seed=1, n=512):
    g = torch.Generator().manual_seed(seed)
    return torch.cat([0.1 * torch.randn(n, 3, generator=g), torch.randn(n, 3, generator=g)], -1).cuda()


def test_pack_bf16_is_round_to_nearest_even():
    g = torch.Generator().manual_seed(0)
    x = torch.randn(100003, generator=g) * torch.logspace(-6, 6, 100003)
    x[:8] = torch.tensor([0.0, -0.0, 1.0, 1.00390625, 1.001953125, 1.005859375, -3.3895e38, 1e-30])  # ties, range ends
    x = x.cuda()
    out = torch.empty(x.numel(), dtype=torch.bfloat16, device="cuda")
    _lib.check(_lib.lib().lrf_pack_bf16(C.c_void_p(x.data_ptr()), C.c_void_p(out.data_ptr()), x.numel(),
                                        C.c_void_p(torch.cuda.current_stream().cuda_stream)))
    assert torch.equal(out.view(torch.int16), x.to(torch.bfloat16).view(torch.int16))


def test_lookups_from_bf16_grids():
    """lrf_density_feature / lrf_app_feature on bf16 texels == the fp32 lookups of the rounded field."""
    m = round_grids_to_bf16(module_from_golden(load_golden("cfg1_64")))
    g = torch.Generator().manual_seed(3)
    xyz = (torch.rand(20000, 3, generator=g) * 2.2 - 1.1).cuda()           # incl. points beyond the border clamp
    with torch.no_grad():
        d32, a32 = m.compute_densityfeature(xyz), m.compute_appfeature(xyz)
    lib = _lib.lib()
    fs, keep = m._field_struct(None, need_mlp=False, grid16=True)
    assert fs.grid_dtype == _lib.GRID_BF16
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    d16 = torch.empty_like(d32); a16 = torch.empty_like(a32)
    _lib.check(lib.lrf_density_feature(C.byref(fs), C.c_void_p(xyz.data_ptr()), xyz.shape[0], C.c_void_p(d16.data_ptr()), st))
    _lib.check(lib.lrf_app_feature(C.byref(fs), C.c_void_p(xyz.data_ptr()), xyz.shape[0], C.c_void_p(a16.data_ptr()), st))
    torch.cuda.synchronize()
    e_d = float((d16 - d32).abs().max() / d32.abs().max()); e_a = float((a16 - a32).abs().max() / a32.abs().max())
    print(f"bf16 lookups vs fp32 lookups of the rounded field: density {e_d:.1e} (equal: {torch.equal(d16, d32)}), "
          f"appearance {e_a:.1e} (equal: {torch.equal(a16, a32)})")
    assert e_d < 1e-6 and e_a < 1e-6
    # entries that do not read 16-bit grids refuse them instead of mis-reading the pointers
    out = torch.empty(xyz.shape[0], 72, device="cuda")
    with pytest.raises(NotImplementedError):
        _lib.check(lib.lrf_app_products(C.byref(fs), C.c_void_p(xyz.data_ptr()), xyz.shape[0], C.c_void_p(out.data_ptr()), st))


@pytest.mark.parametrize("golden,floater", [("cfg1_64", 0.0), ("cfg1_64", 0.5), ("alphamask_32", 0.0), ("opaque_32", 0.0)])
def test_render_bf16_storage_equals_fp32_storage_and_oracle(golden, floater):
    from oracle import oracle as orc
    m = round_grids_to_bf16(module_from_golden(load_golden(golden)))
    rays = rays512()
    with torch.no_grad():
        rgb32, dep32 = m(rays, floater_thresh=floater, return_weights=True)
        w32 = m.last_weights.clone()
        m.set_grid_storage("bf16")
        rgb16, dep16 = m(rays, floater_thresh=floater, return_weights=True)
        w16 = m.last_weights.clone()
    torch.cuda.synchronize()
    margin = (w32 - float(m.rayMarch_weight_thres)).abs().min(-1).values.cpu().numpy()
    n1, e1 = check_with_ties(rgb16.cpu().numpy(), rgb32.cpu().numpy(), margin, 1e-5, f"{golden} rgb bf16 vs fp32 storage")
    n2, e2 = check_with_ties(dep16.cpu().numpy(), dep32.cpu().numpy(), margin, 1e-5, f"{golden} depth bf16 vs fp32 storage")
    e_w = rel_err(w16.cpu().numpy(), w32.cpu().numpy(), floor=5e-3)
    print(f"{golden} floater {floater}: bf16 vs fp32 storage rgb {e1:.1e} depth {e2:.1e} weights {e_w:.1e} "
          f"(bit-equal rgb: {torch.equal(rgb16, rgb32)}, weights: {torch.equal(w16, w32)})")
    assert e_w < 1e-5 and n2 == 0
    # ... and against the CPU oracle (pinned to the reference) evaluated on the same rounded parameters
    f = oracle_fields(type("S", (), {"tensorfs": [m]})())[0]
    ref = orc.field_forward(f, rays.cpu().numpy(), orc.sample_table(f.n_samples()), floater_thresh=floater)
    margin_o = np.abs(ref["weights"] - float(m.rayMarch_weight_thres)).min(-1)
    n3, e3 = check_with_ties(rgb16.cpu().numpy(), ref["rgb"], margin_o, TOL, f"{golden} rgb bf16 vs oracle", max_tie_frac=0.02)
    assert rel_err(dep16.cpu().numpy(), ref["depth"]) < TOL
    print(f"{golden}: bf16 storage vs oracle on the rounded field: rgb {e3:.1e} ({n3} ties)")


def test_bf16_copies_follow_parameter_updates_and_training_reads_fp32():
    m = module_from_golden(load_golden("cfg1_64"))            # NOT rounded: fp32 and bf16 storage differ here
    rays = rays512(seed=2, n=256)
    m.set_grid_storage("bf16")
    with torch.no_grad():
        a, _ = m(rays)
        for p in grids(m):
            p.mul_(0.5)                                         # in-place update (an optimiser step does the same)
        b, _ = m(rays)
    assert not torch.equal(a, b)                                # the 16-bit copies were refreshed
    m2 = round_grids_to_bf16(module_from_golden(load_golden("cfg1_64")))
    with torch.no_grad():
        for p in grids(m2):
            p.mul_(0.5)                                         # exact (power of two): still the bf16 rounding of 0.5 * p
        c, _ = m2(rays)
    # m renders bf16(0.5 p) = 0.5 bf16(p) = m2's fp32 parameters
    assert int(((b - c).abs().max(-1).values > 1e-5).sum()) <= 2      # (<= 2: room for an exact-threshold tie)
    # a pass that records autograd reads the live fp32 parameters whatever the storage setting
    m3 = module_from_golden(load_golden("cfg1_64"))
    z = m3.sample_table(False, -1, rays.device)
    r = rays.clone().requires_grad_(True)
    rgb_f, dep_f = m3(r, z_vals=z)
    m3.set_grid_storage("bf16")
    rgb_h, dep_h = m3(r, z_vals=z)
    assert rgb_h.requires_grad and torch.equal(rgb_f, rgb_h) and torch.equal(dep_f, dep_h)
    (rgb_h.sum() + dep_h.sum()).backward()
    assert all(p.grad is not None for p in grids(m3))
    with torch.no_grad():
        rgb_e, _ = m3(rays, z_vals=z)                           # eval: the 16-bit copies (unrounded field -> differs)
    assert not torch.equal(rgb_e, rgb_f.detach())


def test_bf16_with_positional_encodings_is_refused():
    m = module_from_golden(load_golden("aniso_pe"))
    with pytest.raises(NotImplementedError):
        m.set_grid_storage("bf16")


def test_local_tensorfs_bf16_plan_path_and_whole_batch_vs_reference():
    """cfg2 at the BASELINE size: LocalTensorfs eval (plan fast path) from bf16 grids against (a) the fp32
    storage of the same rounded field and (b) the UNMODIFIED reference's committed outputs with the rounded parameters."""
    import bench
    wl = bench.Workload("cfg2")
    ours = wl.build(L.LocalTensorfs, quiet=True)
    scenes = json.load(open(os.path.join(GOLDEN, "bench_scenes.json")))
    assert state_digest(ours.state_dict()) == scenes["full"]["cfg2"]      # the reference's scene, before rounding
    ours = ours.to("cuda")
    for rf in ours.tensorfs:
        round_grids_to_bf16(rf)
    ids, views = wl.batches()
    ids = ids.cuda(); view = views[0].cuda()
    kw = wl.call_kwargs(ours, torch.device("cuda"))
    b = 77
    with torch.no_grad():
        rgb32, dep32, _, _ = ours(ids[b], view, 800, 800, **kw)
        ours.set_grid_storage("bf16")
        rgb16, dep16, _, _ = ours(ids[b], view, 800, 800, **kw)
        rgb16b, dep16b, _, _ = ours(ids[b], view, 800, 800, **kw)           # second call: the cached plan
    torch.cuda.synchronize()
    assert torch.equal(rgb16, rgb16b) and torch.equal(dep16, dep16b)
    e_rgb, e_dep = rel_err(rgb16.cpu().numpy(), rgb32.cpu().numpy()), rel_err(dep16.cpu().numpy(), dep32.cpu().numpy())
    n_bad = int((np.abs(rgb16.cpu().numpy() - rgb32.cpu().numpy()).max(-1) > 1e-5).sum())
    print(f"cfg2 batch {b}: bf16 vs fp32 storage rgb {e_rgb:.1e} depth {e_dep:.1e} (rays beyond 1e-5: {n_bad}; "
          f"bit-equal: {torch.equal(rgb16, rgb32)})")
    assert e_dep < 1e-5 and n_bad <= 4          # (a flipped w > 1e-3 decision needs a last-bit difference: none expected)

    g = load_golden("vs_reference")             # the reference on the same rounded field (tests/golden/make_golden.py)
    s, margin = g["bf16.b77.rays"].astype(np.int64), g["bf16.b77.margin"]
    n1, e1 = check_with_ties(rgb16.cpu().numpy()[s], g["bf16.b77.rgb"], margin, TOL, "cfg2 bf16 storage vs reference rgb",
                             n_total=4096)
    n2, e2 = check_with_ties(dep16.cpu().numpy()[s], g["bf16.b77.depth"], margin, TOL,
                             "cfg2 bf16 storage vs reference depth", n_total=4096)
    print(f"cfg2 batch {b}, bf16 grid storage vs the reference (rounded parameters): rgb worst {e1:.2e} "
          f"({n1} threshold ties of 4096, {len(s)} compared), depth worst {e2:.2e}")
    assert n2 == 0
