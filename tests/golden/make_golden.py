"""Generate the golden fixtures by running the UNMODIFIED reference on CPU.

Needs a checkout of facebookresearch/localrf (commit 3905e39); nothing else does:

    LOCALRF_REFERENCE=<checkout> python tests/golden/make_golden.py [fullsize | sched | vs_reference]

Writes tests/golden/*.npz.  Each file holds the inputs (field parameters in the reference's
state_dict layout, rays or ray ids, the sample table z actually used) and the reference's outputs.
The reference never returns per-sample weights, so `alpha2weights` (models/tensorBase.py:23-32) is
wrapped -- not modified -- to capture the last weights it produced.

Recorded environment: see the `meta` entry of every file (torch version, device, reference commit).
"""
import contextlib
import io
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path[:0] = [ROOT, os.path.dirname(HERE)]
from oracle.ref_loader import load_reference  # noqa: E402

TensorVMSplit, AlphaGridMask, LocalTensorfs, ray_utils = load_reference()
import models.tensorBase as ref_tb  # noqa: E402  (the reference's module)

META = f"torch {torch.__version__} cpu; reference facebookresearch/localrf @ 3905e39"

# ---- capture hooks (wrap, don't modify) --------------------------------------------------------
_captured = {}
_orig_a2w = ref_tb.alpha2weights


def _a2w(alpha):
    w, T = _orig_a2w(alpha)
    _captured["weights"] = w.detach().clone()
    if _captured.get("keep_margins"):
        # distance of every ray's closest weight to the w > 1e-3 switch (tensorBase.py:622)
        _captured.setdefault("margins", []).append((w.detach() - 1e-3).abs().min(dim=-1).values)
    return w, T


ref_tb.alpha2weights = _a2w
_orig_sample = ref_tb.TensorBase.sample_ray_contracted


def _sample(self, rays_o, rays_d, is_train=True, N_samples=-1):
    pts, z, valid = _orig_sample(self, rays_o, rays_d, is_train=is_train, N_samples=N_samples)
    _captured.setdefault("z_list", []).append(z.detach().clone().reshape(-1))
    return pts, z, valid


ref_tb.TensorBase.sample_ray_contracted = _sample


def quiet(fn, *a, **k):
    with contextlib.redirect_stdout(io.StringIO()):
        return fn(*a, **k)


def field_kwargs(**over):
    kw = dict(density_n_comp=[8, 8, 8], appearance_n_comp=[24, 24, 24], app_dim=27,
              shadingMode="MLP_Fea_late_view", near_far=[0.1, 1e3], density_shift=-5,
              alphaMask_thres=1e-4, distance_scale=25, rayMarch_weight_thres=1e-3, pos_pe=0,
              view_pe=0, fea_pe=0, featureC=128, step_ratio=0.5, fea2denseAct="softplus")
    kw.update(over)
    return kw


def make_field(grid, seed, **over):
    torch.manual_seed(seed)
    aabb = 2 * torch.tensor([[-1.0, -1, -1], [1, 1, 1]])  # dataLoader/localrf_dataset.py:101
    return quiet(TensorVMSplit, "cpu", aabb, list(grid), **field_kwargs(**over))


def field_to_dict(m, prefix=""):
    d = {}
    for k, v in m.state_dict().items():
        d[prefix + k] = v.detach().cpu().numpy()
    kw = m.get_kwargs()
    for k in ("density_shift", "distance_scale", "rayMarch_weight_thres", "fea_pe", "view_pe",
              "featureC", "app_dim", "step_ratio"):
        d[prefix + k] = np.array(kw[k])
    d[prefix + "fea2denseAct"] = np.array(kw["fea2denseAct"])
    d[prefix + "gridSize"] = np.array(kw["gridSize"])
    d[prefix + "nSamples"] = np.array(m.nSamples)
    return d


def rays_cfg1(n, seed=1):
    g = torch.Generator().manual_seed(seed)  # SURVEY.md §8d config 1
    o = 0.1 * torch.randn(n, 3, generator=g)
    d = torch.randn(n, 3, generator=g)
    return torch.cat([o, d], -1)


def run_field(m, rays, **kw):
    _captured.clear()
    with torch.no_grad():
        rgb, depth = m(rays, **kw)
    return dict(rgb=rgb.numpy(), depth=depth.numpy(), weights=_captured["weights"].numpy(),
                z=_captured["z_list"][-1].numpy())


def save(name, **arrays):
    path = os.path.join(HERE, name + ".npz")
    np.savez(path, meta=np.array(META), **arrays)
    print(f"{name}: {os.path.getsize(path) / 1e6:.2f} MB")


def pack(prefix, out):
    return {f"{prefix}.{k}": v for k, v in out.items()}


# ---- G1/G2: BASELINE config 1 -- 64^3, 512 rays, eval (floater 0 / 0.5) and train (seeded jitter)
def gen_cfg1():
    m = make_field([64, 64, 64], 0)
    rays = rays_cfg1(512)
    arrays = field_to_dict(m)
    arrays["rays"] = rays.numpy()
    arrays.update(pack("eval", run_field(m, rays, is_train=False, floater_thresh=0)))
    arrays.update(pack("eval_floater", run_field(m, rays, is_train=False, floater_thresh=0.5)))
    arrays.update(pack("eval_nobg", run_field(m, rays, is_train=False, white_bg=False)))
    torch.manual_seed(2)
    arrays.update(pack("train", run_field(m, rays, is_train=True)))
    # unit-level vectors for the feature functions
    g = torch.Generator().manual_seed(3)
    xyz = torch.rand(256, 3, generator=g) * 2.2 - 1.1  # a few outside [-1,1] -> border clamp
    xyz[0] = torch.tensor([1.0, -1.0, 0.0]); xyz[1] = torch.tensor([-1.0, 1.0, 1.0])
    with torch.no_grad():
        arrays["unit.xyz"] = xyz.numpy()
        arrays["unit.density_feature"] = m.compute_densityfeature(xyz).numpy()
        app = m.compute_appfeature(xyz)
        arrays["unit.app_feature"] = app.numpy()
        vd = torch.nn.functional.normalize(torch.randn(256, 3, generator=g), dim=-1)
        arrays["unit.viewdirs"] = vd.numpy()
        arrays["unit.mlp_rgb"] = m.renderModule(xyz, vd, app, True).numpy()
        pts = torch.randn(256, 3, generator=g) * 2
        pts[0] = torch.tensor([1.0, 0.5, -1.0]); pts[1] = torch.tensor([0.0, 0.0, 0.0])
        arrays["unit.contract_in"] = pts.numpy()
        arrays["unit.contract_out"] = ray_utils.contract(pts).numpy()
    save("cfg1_64", **arrays)


# ---- G3: anisotropic grid + positional encodings (refine True/False) + floater
def gen_aniso():
    m = make_field([40, 52, 64], 5, fea_pe=2, view_pe=2)
    rays = rays_cfg1(96, seed=6)
    arrays = field_to_dict(m)
    arrays["rays"] = rays.numpy()
    arrays.update(pack("refine", run_field(m, rays, is_train=False, refine=True, floater_thresh=0.5)))
    arrays.update(pack("norefine", run_field(m, rays, is_train=False, refine=False)))
    save("aniso_pe", **arrays)


# ---- G4: "opaque" distribution B (density_shift=+2) -> early termination; and relu activation
def gen_opaque():
    m = make_field([32, 32, 32], 7, density_shift=2)
    rays = rays_cfg1(160, seed=8)
    arrays = field_to_dict(m)
    arrays["rays"] = rays.numpy()
    arrays.update(pack("eval", run_field(m, rays, is_train=False)))
    arrays.update(pack("eval_floater", run_field(m, rays, is_train=False, floater_thresh=0.5)))
    save("opaque_32", **arrays)
    m = make_field([32, 32, 32], 9, fea2denseAct="relu")
    with torch.no_grad():  # larger density features so relu(f) is not ~0 everywhere
        for p in list(m.density_plane) + list(m.density_line):
            p.mul_(4.0)
    arrays = field_to_dict(m)
    arrays["rays"] = rays.numpy()
    arrays.update(pack("eval", run_field(m, rays, is_train=False)))
    save("relu_32", **arrays)


# ---- G5: alpha mask built by the reference's own updateAlphaMask
def gen_alphamask():
    m = make_field([32, 32, 32], 11, density_shift=-7.5)
    with torch.no_grad():
        for p in list(m.density_plane) + list(m.density_line):
            p.mul_(4.0)
    quiet(m.updateAlphaMask, (16, 16, 16))
    frac = float(m.alphaMask.alpha_volume.mean())
    print("alpha mask kept fraction", frac)
    assert 0.1 < frac < 0.9, frac
    rays = rays_cfg1(160, seed=12)
    arrays = field_to_dict(m)
    arrays["rays"] = rays.numpy()
    arrays.update(pack("eval", run_field(m, rays, is_train=False)))
    g = torch.Generator().manual_seed(13)
    pts = torch.rand(512, 3, generator=g) * 4.4 - 2.2
    with torch.no_grad():
        arrays["unit.alpha_pts"] = pts.numpy()
        arrays["unit.alpha_vals"] = m.alphaMask.sample_alpha(pts).numpy()
    save("alphamask_32", **arrays)


# ---- G6: LocalTensorfs -- 3 overlapping fields, explicit blend, exposure, test_id, fov 360, train
def make_local(fov, grid, n_frames, seed):
    torch.manual_seed(seed)
    aabb = 2 * torch.tensor([[-1.0, -1, -1], [1, 1, 1]])
    kw = field_kwargs()
    lt = quiet(LocalTensorfs, camera_prior=None, fov=fov, n_init_frames=n_frames, n_overlap=30,
               WH=(48, 40), n_iters_per_frame=600, n_iters_reg=100, lr_R_init=5e-3, lr_t_init=5e-4,
               lr_i_init=0, lr_exposure_init=1e-3, rf_lr_init=2e-2, rf_lr_basis=1e-3,
               lr_decay_target_ratio=0.1, N_voxel_list={}, update_AlphaMask_list=[],
               lr_upsample_reset=True, device="cpu", aabb=aabb, gridSize=list(grid), **kw)
    return lt


def local_to_dict(lt):
    d = {}
    for k, v in lt.state_dict().items():
        d["sd." + k] = v.detach().cpu().numpy()
    kw = lt.tensorfs[0].get_kwargs()
    for k in ("density_shift", "distance_scale", "rayMarch_weight_thres", "fea_pe", "view_pe",
              "featureC", "app_dim", "step_ratio"):
        d[k] = np.array(kw[k])
    d["fea2denseAct"] = np.array(kw["fea2denseAct"])
    d["gridSize"] = np.array(kw["gridSize"])
    d["n_fields"] = np.array(len(lt.tensorfs))
    d["n_frames"] = np.array(len(lt.r_c2w))
    d["fov"] = np.array(float(lt.fov))
    d["WH"] = np.array([lt.W, lt.H])
    return d


def run_local(lt, ray_ids, view_ids, W, H, **kw):
    _captured.clear()
    with torch.no_grad():
        rgb, depth, dirs, ij = quiet(lt, ray_ids, view_ids, W, H, **kw)
    out = dict(rgb=rgb.numpy(), depth=depth.numpy(), directions=dirs.numpy(), ij=ij.numpy())
    for i, z in enumerate(_captured["z_list"]):
        out[f"z{i}"] = z.numpy()
    return out


def gen_local():
    for fov, name in ((85.6, "local3"), (360, "local3_fov360")):
        lt = make_local(fov, [24, 28, 20], n_frames=4, seed=20)
        # progressive structure built with the reference's own bookkeeping
        quiet(lt.append_rf, 2)
        quiet(lt.append_frame)
        quiet(lt.append_rf, 1)
        quiet(lt.append_frame)
        with torch.no_grad():
            g = torch.Generator().manual_seed(21)
            for i in range(len(lt.r_c2w)):
                lt.r_c2w[i].add_(0.05 * torch.randn(3, 2, generator=g))
                lt.t_c2w[i].add_(0.2 * torch.randn(3, generator=g))
                lt.exposure[i].add_(0.05 * torch.randn(3, 3, generator=g))
            lt.world2rf[1].copy_(torch.tensor([-0.3, 0.0, 0.05]))
            lt.world2rf[2].copy_(torch.tensor([-0.6, 0.1, 0.0]))
            lt.focal_offset.mul_(1.03)
            lt.center_rel.add_(torch.tensor([0.01, -0.02]))
        arrays = local_to_dict(lt)
        W, H = 24, 20
        ids = torch.arange(W * H, dtype=torch.long)
        v = torch.tensor([2])
        bw = torch.tensor([[0.2, 0.5, 0.3]])
        arrays["ray_ids"] = ids.numpy(); arrays["W"] = np.array(W); arrays["H"] = np.array(H)
        arrays["blend3"] = bw.numpy()
        arrays.update(pack("blend3", run_local(lt, ids, v, W, H, is_train=False,
                                               blending_weights=bw.clone(), chunk=256)))
        arrays.update(pack("blend3_testid", run_local(lt, ids, v, W, H, is_train=False,
                                                      blending_weights=bw.clone(), chunk=256,
                                                      test_id=True, floater_thresh=0.5)))
        # natural blending row of every frame (1 or 2 active fields), external pose
        for fr in (0, 3, 5):
            c2w = lt.get_cam2world(torch.tensor([fr])).detach()
            c2w[:, :3, 3] += 0.05
            arrays[f"frame{fr}.cam2world"] = c2w.numpy()
            arrays.update(pack(f"frame{fr}", run_local(lt, ids, torch.tensor([fr]), W, H,
                                                       is_train=False, cam2world=c2w, chunk=128)))
        # training-style call: 4 views x 24 random pixels, ids carry the view offset.
        # (NOT 3 views: utils/utils.py:386 calls torch.cross(b1, b2) without dim, which for a
        #  [3,3] batch crosses over the batch axis -- a reference quirk that exists only at V == 3;
        #  the oracle and the product implement the intended per-view cross product.)
        g = torch.Generator().manual_seed(22)
        tv = torch.tensor([1, 4, 5, 2])
        px = torch.randint(0, W * H, (4, 24), generator=g)
        tid = (px + tv[:, None] * W * H).reshape(-1)
        arrays["train.ray_ids"] = tid.numpy(); arrays["train.view_ids"] = tv.numpy()
        torch.manual_seed(23)
        arrays.update(pack("train", run_local(lt, tid, tv, W, H, is_train=True)))
        save(name, **arrays)


# ---- G7: gradients of the reference (autograd) -- field level and scene level
def gen_grads():
    m = make_field([20, 24, 28], 40)
    rays = rays_cfg1(64, seed=41).requires_grad_(True)
    g = torch.Generator().manual_seed(42)
    c_rgb = torch.randn(64, 3, generator=g)
    c_depth = 0.1 * torch.randn(64, generator=g)
    arrays = field_to_dict(m)
    arrays["rays"] = rays.detach().numpy()
    arrays["c_rgb"] = c_rgb.numpy(); arrays["c_depth"] = c_depth.numpy()
    _captured.clear()
    torch.manual_seed(43)
    rgb, depth = m(rays, is_train=True)
    loss = (rgb * c_rgb).sum() + (depth * c_depth).sum()
    loss.backward()
    arrays["z"] = _captured["z_list"][-1].numpy()
    arrays["out.rgb"] = rgb.detach().numpy(); arrays["out.depth"] = depth.detach().numpy()
    arrays["grad.rays"] = rays.grad.numpy()
    for k, p in m.named_parameters():
        if p.grad is not None:
            arrays["grad." + k] = p.grad.numpy()
    save("grads_field", **arrays)

    lt = make_local(85.6, [24, 28, 20], n_frames=4, seed=20)
    quiet(lt.append_rf, 2); quiet(lt.append_frame); quiet(lt.append_rf, 1); quiet(lt.append_frame)
    with torch.no_grad():
        gg = torch.Generator().manual_seed(21)
        for i in range(len(lt.r_c2w)):
            lt.r_c2w[i].add_(0.05 * torch.randn(3, 2, generator=gg))
            lt.t_c2w[i].add_(0.2 * torch.randn(3, generator=gg))
            lt.exposure[i].add_(0.05 * torch.randn(3, 3, generator=gg))
        lt.world2rf[2].copy_(torch.tensor([-0.6, 0.1, 0.0]))
    arrays = local_to_dict(lt)
    W, H = 24, 20
    gg = torch.Generator().manual_seed(22)
    tv = torch.tensor([1, 4, 5, 2])
    px = torch.randint(0, W * H, (4, 24), generator=gg)
    tid = (px + tv[:, None] * W * H).reshape(-1)
    c_rgb = torch.randn(96, 3, generator=gg); c_depth = 0.1 * torch.randn(96, generator=gg)
    arrays.update({"ray_ids": tid.numpy(), "view_ids": tv.numpy(), "W": np.array(W), "H": np.array(H),
                   "c_rgb": c_rgb.numpy(), "c_depth": c_depth.numpy()})
    _captured.clear()
    torch.manual_seed(44)
    rgb, depth, dirs, ij = quiet(lt, tid, tv, W, H, is_train=True)
    loss = (rgb * c_rgb).sum() + (depth * c_depth).sum()
    loss.backward()
    arrays["z"] = _captured["z_list"][-1].numpy()
    arrays["out.rgb"] = rgb.detach().numpy(); arrays["out.depth"] = depth.detach().numpy()
    for k, p in lt.named_parameters():
        if p.grad is not None and float(p.grad.abs().sum()) > 0:
            arrays["grad." + k] = p.grad.numpy()
    save("grads_local", **arrays)


# ---- G8: BASELINE-size OUTPUT-ONLY goldens (configs 2 and 3, SURVEY.md 8d).  The fields are NOT
# stored (33 MB each): they are regenerated from their seeds by the same constructor calls
# (tests/test_host_logic.py pins "same seed -> same init as the reference").  `margin` is each ray's
# smallest |w - 1e-3| over its samples (and fields): a ray whose margin is below the fp32 noise of
# w sits exactly on the reference's hard w > rayMarch_weight_thres switch (tensorBase.py:622).
FULL_BATCHES = (0, 77, 155)          # first rows, middle, last full batch of the 800x800 frame


def make_scene300(n_fields):
    """== bench.build_scene(...) (+ the cfg-3 extension in tests/test_gpu_fullsize.py)."""
    torch.manual_seed(0)
    aabb = 2 * torch.tensor([[-1.0, -1, -1], [1, 1, 1]])
    lt = quiet(LocalTensorfs, camera_prior=None, fov=85.6, n_init_frames=1, n_overlap=30,
               WH=(800, 800), n_iters_per_frame=600, n_iters_reg=100, lr_R_init=5e-3,
               lr_t_init=5e-4, lr_i_init=0, lr_exposure_init=1e-3, rf_lr_init=2e-2,
               rf_lr_basis=1e-3, lr_decay_target_ratio=0.1, N_voxel_list={},
               update_AlphaMask_list=[], lr_upsample_reset=True, device="cpu", aabb=aabb,
               gridSize=[300] * 3, **field_kwargs())
    for k in range(1, n_fields):
        quiet(lt.append_frame)
        torch.manual_seed(k)
        quiet(lt.append_rf, 1)
    return lt


def run_full(lt, ids, **kw):
    _captured.clear()
    _captured["keep_margins"] = True
    with torch.no_grad():
        rgb, depth, _, _ = quiet(lt, ids, torch.tensor([0]), 800, 800, is_train=False, **kw)
    return rgb.numpy(), depth.numpy(), list(_captured["margins"])


def gen_fullsize():
    lt = make_scene300(1)
    arrays = {"batches": np.array(FULL_BATCHES), "param_checksum": np.array(
        [float(p.double().sum()) for p in lt.tensorfs[0].parameters()])}
    for b in FULL_BATCHES:
        ids = torch.arange(b * 4096, (b + 1) * 4096, dtype=torch.long)
        rgb, depth, margins = run_full(lt, ids, chunk=4096)
        assert len(margins) == 1
        arrays[f"b{b}.rgb"], arrays[f"b{b}.depth"] = rgb, depth
        arrays[f"b{b}.margin"] = margins[0].numpy()
    save("cfg2_300", **arrays)

    lt = make_scene300(3)
    w2rf = [torch.zeros(3), torch.tensor([-0.3, 0.0, 0.0]), torch.tensor([-0.6, 0.0, 0.0])]
    bw = torch.tensor([[0.2, 0.5, 0.3]])
    ids = torch.arange(60 * 4096, 61 * 4096, dtype=torch.long)
    rgb, depth, margins = run_full(lt, ids, world2rf=w2rf, blending_weights=bw, chunk=4096)
    # chunk = 4096 // 3 = 1365 rays (local_tensorfs.py:442): per chunk one alpha2weights call per field
    n_chunks = len(margins) // 3
    per_field = [torch.cat([margins[c * 3 + k] for c in range(n_chunks)]) for k in range(3)]
    arrays = {"batch": np.array(60), "blend": bw.numpy(), "world2rf": torch.stack(w2rf).numpy(),
              "rgb": rgb, "depth": depth, "margin": torch.stack(per_field).min(dim=0).values.numpy(),
              "param_checksum": np.array([float(p.double().sum()) for rf in lt.tensorfs
                                          for p in rf.parameters()])}
    save("cfg3_300", **arrays)


# ---- G9: schedule-time operators (SURVEY.md 8f ranks 2-3) and the AABB sampler, non-cubic grid ----------
def gen_sched():
    from utils.utils import TVLoss               # the reference's regulariser (utils/utils.py:293-312)
    m = make_field([20, 24, 28], 50, density_shift=-7.5)
    with torch.no_grad():
        for p in list(m.density_plane) + list(m.density_line):
            p.mul_(4.0)
    arrays = field_to_dict(m)
    # regularisers + their autograd gradients
    reg = TVLoss()
    for name, fn in (("l1", m.density_L1), ("tv_density", lambda: m.TV_loss_density(reg)),
                     ("tv_app", lambda: m.TV_loss_app(reg))):
        m.zero_grad()
        val = fn()
        val.backward()
        arrays[f"{name}.value"] = val.detach().numpy()
        for k, p_ in m.named_parameters():
            if p_.grad is not None and float(p_.grad.abs().sum()) > 0:
                arrays[f"{name}.grad.{k}"] = p_.grad.clone().numpy()
    m.zero_grad()
    # AABB sampler: eval and seeded train
    rays = rays_cfg1(48, seed=51)
    rays[:, :3] *= 8.0                            # origins in and around the [-2,2]^3 box
    rays[0, 3] = 0.0                              # a zero direction component (the 1e-6 substitution)
    arrays["sr.rays"] = rays.numpy()
    with torch.no_grad():
        pts, z, inside = m.sample_ray(rays[:, :3], rays[:, 3:], is_train=False, N_samples=40)
        arrays["sr.eval.pts"], arrays["sr.eval.z"], arrays["sr.eval.inside"] = pts.numpy(), z.numpy(), inside.numpy()
        torch.manual_seed(52)
        pts, z, inside = m.sample_ray(rays[:, :3], rays[:, 3:], is_train=True, N_samples=-1)
        arrays["sr.train.pts"], arrays["sr.train.z"], arrays["sr.train.inside"] = pts.numpy(), z.numpy(), inside.numpy()
    # occupancy mask: dense alpha, mask, then dense alpha again with the mask in place
    with torch.no_grad():
        arrays["mask.alpha0"] = m.getDenseAlpha((10, 12, 14)).numpy()
        quiet(m.updateAlphaMask, (10, 12, 14))
        arrays["mask.volume"] = m.alphaMask.alpha_volume.numpy()
        frac = float(m.alphaMask.alpha_volume.mean())
        assert 0.05 < frac < 0.95, frac
        arrays["mask.alpha1"] = m.getDenseAlpha((11, 9, 13)).numpy()
        # pooled alpha before thresholding, to identify exact ties on alphaMask_thres in the test
        a = arrays["mask.alpha0"]
        pooled = torch.nn.functional.max_pool3d(torch.from_numpy(a).clamp(0, 1).transpose(0, 2).contiguous()[None, None],
                                                kernel_size=3, padding=1, stride=1)[0, 0]
        arrays["mask.pooled"] = pooled.numpy()
    # upsampling
    quiet(m.upsample_volume_grid, [30, 33, 41])
    for k, v in m.state_dict().items():
        if "plane" in k or "line" in k:
            arrays["up." + k] = v.numpy()
    arrays["up.nSamples"] = np.array(m.nSamples)
    save("sched_nc", **arrays)


# ---- G10: the bench's workloads through the reference (tests/test_gpu_vs_reference.py, test_gpu_bf16.py,
# test_bench_workloads.py).  Scenes are rebuilt from their seeds by bench.Workload; stored are the digests of
# the reference's scenes and, of each compared batch, a fixed seeded sample of SAMPLE_RAYS rays followed by
# every other ray within TIE_MARGIN of the w > 1e-3 switch (so the test counts the batch's threshold ties
# exactly); directions / ij of the sample only.
VS_BATCHES = {"cfg2": (3, 90), "distB": (50,), "incoherent": (0, 7), "cfg3": (60,)}
SAMPLE_RAYS = 512
WEIGHT_ROWS = 64


def ray_sample(margin, seed):
    from helpers import TIE_MARGIN
    s = np.sort(np.random.default_rng(seed).choice(len(margin), SAMPLE_RAYS, replace=False))
    return np.concatenate([s, np.setdiff1d(np.nonzero(margin < TIE_MARGIN)[0], s)]).astype(np.int16)


def gen_vs_reference():
    import json
    import bench
    from helpers import state_digest
    scenes = {"grid12": {}, "full": {}}
    for name in ("cfg2", "distB", "incoherent", "cfg3", "cfg5"):
        scenes["grid12"][name] = state_digest(bench.Workload(name, 12).build(LocalTensorfs, quiet=True).state_dict())
    arrays = {}
    for name, batches in VS_BATCHES.items():
        wl = bench.Workload(name)
        lt = wl.build(LocalTensorfs, quiet=True)
        scenes["full"][name] = state_digest(lt.state_dict())
        ids, views = wl.batches()
        kw = wl.call_kwargs(lt, torch.device("cpu"))
        n_f = len(lt.tensorfs)
        for b in batches:
            _captured.clear()
            _captured["keep_margins"] = True
            with torch.no_grad():
                rgb, depth, dirs, ij = quiet(lt, ids[b], views[b], 800, 800, **kw)
            m = _captured["margins"]                  # alpha2weights calls arrive chunk-major, field-minor
            margin = torch.stack([torch.cat(m[k::n_f]) for k in range(n_f)]).min(0).values.numpy()
            s = ray_sample(margin, b)
            p = f"{name}.b{b}."
            arrays.update({p + "rays": s, p + "rgb": rgb.numpy()[s], p + "depth": depth.numpy()[s],
                           p + "margin": margin[s], p + "directions": dirs.numpy()[s[:SAMPLE_RAYS]],
                           p + "ij": ij.numpy()[s[:SAMPLE_RAYS]].astype(np.int16)})
        if name != "cfg2":
            continue
        # per-sample weights of one field, random rays (white background, the field's own forward)
        g = torch.Generator().manual_seed(4)
        rays = torch.cat([0.1 * torch.randn(4096, 3, generator=g), torch.randn(4096, 3, generator=g)], -1)
        _captured.clear()
        with torch.no_grad():
            rgb, depth = lt.tensorfs[0](rays, is_train=False, white_bg=True, N_samples=-1)
        w = _captured["weights"].numpy()
        margin = np.abs(w - 1e-3).min(-1)
        s = ray_sample(margin, 4)
        arrays.update({"weights.rays": s, "weights.rgb": rgb.numpy()[s], "weights.depth": depth.numpy()[s],
                       "weights.margin": margin[s], "weights.rows": s[:WEIGHT_ROWS], "weights.w": w[s[:WEIGHT_ROWS]]})
        # batch 77 with every plane / line rounded to bfloat16 (the bf16 grid-storage test's field)
        with torch.no_grad():
            for rf in lt.tensorfs:
                for plist in (rf.density_plane, rf.density_line, rf.app_plane, rf.app_line):
                    for q in plist:
                        q.copy_(q.to(torch.bfloat16).to(torch.float32))
        _captured.clear()
        _captured["keep_margins"] = True
        with torch.no_grad():
            rgb, depth, _, _ = quiet(lt, ids[77], views[77], 800, 800, **kw)
        margin = torch.cat(_captured["margins"]).numpy()
        s = ray_sample(margin, 77)
        arrays.update({"bf16.b77.rays": s, "bf16.b77.rgb": rgb.numpy()[s], "bf16.b77.depth": depth.numpy()[s],
                       "bf16.b77.margin": margin[s]})
    path = os.path.join(HERE, "vs_reference.npz")
    np.savez_compressed(path, meta=np.array(META), **arrays)
    print(f"vs_reference: {os.path.getsize(path) / 1e6:.2f} MB")
    with open(os.path.join(HERE, "bench_scenes.json"), "w") as f:
        json.dump({"meta": META, "what": "state_dict digests (tests/helpers.py state_digest) of the reference's "
                   "scenes built by bench.Workload; grid12 at a 12^3 grid, full at the workload's own size",
                   **scenes}, f, indent=1)
        f.write("\n")


if __name__ == "__main__":
    if len(sys.argv) > 1 and sys.argv[1] == "fullsize":
        gen_fullsize()
        sys.exit(0)
    if len(sys.argv) > 1 and sys.argv[1] == "vs_reference":
        gen_vs_reference()
        sys.exit(0)
    if len(sys.argv) > 1 and sys.argv[1] == "sched":
        gen_sched()
        sys.exit(0)
    gen_cfg1()
    gen_aniso()
    gen_opaque()
    gen_alphamask()
    gen_local()
    gen_grads()
    gen_fullsize()
    gen_sched()
