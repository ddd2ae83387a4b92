"""-m gpu: the UNMODIFIED reference's `renderer.render` (renderer.py:15-190, the eval caller of the hot path)
executed on top of dropin/: its imports `local_tensorfs` / `models.*` resolve to this package, everything else
(`utils.utils`: visualize_depth etc.) is the reference's own code.  File / plot I/O is stubbed (no savePath,
draw_poses replaced: it needs matplotlib).  The frames it returns must equal direct forward calls.
Runs in a subprocess because the reference uses top-level module names (`utils`, `models`).
It executes the reference's own renderer module: the bytecode build() compiled into oracle/_ref, or a checkout
named by $LOCALRF_REFERENCE (the repository holds no reference source)."""
import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

SCRIPT = r'''
import sys, types
import numpy as np, torch
ROOT, REF = sys.argv[1], sys.argv[2]
sys.path[:0] = [ROOT + "/dropin", ROOT, REF]
from oracle import ref_loader
for name, attrs in (("kornia", dict(create_meshgrid=None)), ("matplotlib", dict(use=lambda *a, **k: None)),
                    ("matplotlib.pyplot", {}), ("matplotlib.cm", {}), ("plyfile", {}), ("skimage", {}),
                    ("skimage.measure", {}), ("imageio", {}), ("lpips", {})):
    ref_loader._stub(name, **attrs)
import renderer                                     # the reference's module, unmodified
import local_tensorfs, localrf_b200 as L
assert local_tensorfs.LocalTensorfs is L.LocalTensorfs and renderer.__file__.startswith(REF)
import bench
W, H = 64, 48
renderer.draw_poses = lambda poses, colours: np.zeros((H, W, 3), np.uint8)      # matplotlib plot: stubbed I/O
wl = bench.Workload("cfg5", 40)
lt = wl.build(L.LocalTensorfs, quiet=True).to("cuda")
n = len(lt.r_c2w)
train_ds = types.SimpleNamespace(all_fbases={f"{i:04d}": i for i in range(n)})
test_ds = types.SimpleNamespace(all_fbases={"0009": 0, "0030": 1})          # two held-out frames -> test_id exposure rule
args = types.SimpleNamespace(batch_size=4096, device="cuda")
poses = lt.get_cam2world().detach()[4:16]
out = renderer.render(test_ds, poses, lt, args, W=W, H=H, savePath=None, save_video=False, save_frames=False,
                      test=False, train_dataset=train_ds, start=0, floater_thresh=0.5, add_frame_to_list=True)
rgb_maps, depth_maps = out[0], out[1]
assert len(rgb_maps) == 12 and tuple(rgb_maps[0].shape) == (H, W, 3) and tuple(depth_maps[0].shape) == (H, W, 3)
ids = torch.arange(W * H, device="cuda")
is_test = [fb in test_ds.all_fbases for fb in train_ds.all_fbases]
worst = 0.0
with torch.no_grad():
    t = torch.stack(list(lt.t_c2w))
    for i in range(12):
        v = torch.argmin(torch.norm(t - poses[i][None, :, 3], dim=-1))[None]
        rgb, depth, _, _ = lt(ids, v, W, H, is_train=False, cam2world=poses[i][None], test_id=is_test[int(v)],
                              chunk=4096, floater_thresh=0.5)
        worst = max(worst, float((rgb.reshape(H, W, 3).cpu() - rgb_maps[i]).abs().max()))
        ref_vis, _ = renderer.visualize_depth(depth.reshape(H, W).cpu().numpy(), [0, 5])
        want = torch.permute(ref_vis * 255, [1, 2, 0]).byte()
        assert torch.equal(want, depth_maps[i])
assert worst == 0.0, worst
print("RENDER_LOOP_OK", len(rgb_maps))
'''


def test_reference_renderer_loop_runs_on_dropin():
    from oracle import ref_loader
    if not ref_loader.reference_available():
        pytest.skip("no reference (oracle/_ref or $LOCALRF_REFERENCE)")
    ref = ref_loader.REF_PKG
    out = subprocess.run([sys.executable, "-c", SCRIPT, ROOT, ref], capture_output=True, text=True, timeout=900)
    assert out.returncode == 0 and "RENDER_LOOP_OK 12" in out.stdout, (out.stdout[-1500:], out.stderr[-3000:])
