"""-m gpu: the fused path against the UNMODIFIED reference, same parameters, same rays -- whole 4096-ray
batches of the bench's workloads at the BASELINE size.

The reference's outputs are committed (tests/golden/vs_reference.npz, written by tests/golden/make_golden.py
from the reference run on CPU): of every batch a fixed seeded sample of 512 rays plus every ray that could be a
threshold tie; the scenes are rebuilt from their seeds, and their digests (tests/golden/bench_scenes.json) pin
them to the reference's.  The reference's CPU run and the CUDA path each compute alpha = 1 - exp(-x) within an
ulp but not bit-identically, so rays that sit exactly on the reference's hard w > 1e-3 switch are accounted for
one by one (helpers.check_with_ties), and there are at most 1% of them in each whole batch (3% with cfg3's three
fields)."""
import contextlib
import io
import json
import os

import numpy as np
import pytest
import torch

import bench
from helpers import GOLDEN, check_with_ties, load_golden, rel_err, state_digest

pytestmark = pytest.mark.gpu
TOL = 1e-4


@pytest.fixture(scope="module")
def golden():
    return load_golden("vs_reference")


def _ours(wl_name):
    import localrf_b200 as L
    wl = bench.Workload(wl_name)
    lt = wl.build(L.LocalTensorfs, quiet=True)
    scenes = json.load(open(os.path.join(GOLDEN, "bench_scenes.json")))
    assert state_digest(lt.state_dict()) == scenes["full"][wl_name]   # same seed -> the reference's scene
    return wl, lt.to("cuda")


@pytest.mark.parametrize("wl_name,batches", [("cfg2", (3, 90)), ("distB", (50,)), ("incoherent", (0, 7)),
                                             ("cfg3", (60,))])
def test_whole_batches_vs_reference_on_gpu(golden, wl_name, batches):
    wl, ours = _ours(wl_name)
    kw = wl.call_kwargs(ours, torch.device("cuda"))
    ids_all, views = wl.batches()
    for b in batches:
        ids, view = ids_all[b].cuda(), views[b].cuda()
        with torch.no_grad(), contextlib.redirect_stdout(io.StringIO()):
            rgb, depth, dirs, ij = ours(ids, view, 800, 800, **kw)
        p = f"{wl_name}.b{b}."
        s, margin, n = golden[p + "rays"].astype(np.int64), golden[p + "margin"], ids.shape[0]
        # three blended fields, three chances per ray to sit on a switch: the bound of the same batch against
        # the reference in test_gpu_fullsize.py::test_cfg3_three_fields_vs_reference_golden_and_oracle
        ties = 0.03 if wl_name == "cfg3" else 0.01
        n1, e1 = check_with_ties(rgb.cpu().numpy()[s], golden[p + "rgb"], margin, TOL, f"{wl_name} b{b} rgb",
                                 max_tie_frac=ties, n_total=n)
        n2, e2 = check_with_ties(depth.cpu().numpy()[s], golden[p + "depth"], margin, TOL, f"{wl_name} b{b} depth",
                                 n_total=n)
        print(f"{wl_name} batch {b} vs reference: rgb worst {e1:.2e} ({n1} threshold ties of "
              f"{n} rays, {len(s)} compared), depth worst {e2:.2e}")
        assert n2 == 0
        s = s[:len(golden[p + "ij"])]                 # the random sample
        assert np.array_equal(ij.cpu().numpy()[s], golden[p + "ij"])
        np.testing.assert_allclose(dirs.cpu().numpy()[s], golden[p + "directions"], rtol=2e-6, atol=1e-6)


def test_weights_vs_reference_on_gpu(golden):
    """Per-sample weights [4096, 344] of one field against the reference's."""
    wl, ours = _ours("cfg2")
    g = torch.Generator().manual_seed(4)
    rays = torch.cat([0.1 * torch.randn(4096, 3, generator=g), torch.randn(4096, 3, generator=g)], -1).cuda()
    with torch.no_grad():
        rgb, depth = ours.tensorfs[0](rays, is_train=False, return_weights=True)
    w = ours.tensorfs[0].last_weights.cpu().numpy()[golden["weights.rows"]]
    w_ref = golden["weights.w"]
    e_floor = rel_err(w, w_ref, floor=5e-3)
    e_pure = rel_err(w, w_ref, floor=1e-3)
    print(f"weights vs reference: rel err {e_floor:.2e} (floor 5e-3), {e_pure:.2e} (floor 1e-3)")
    assert e_floor < TOL
    s = golden["weights.rays"].astype(np.int64)
    check_with_ties(rgb.cpu().numpy()[s], golden["weights.rgb"], golden["weights.margin"], TOL, "random rays rgb",
                    n_total=rays.shape[0])
    assert rel_err(depth.cpu().numpy()[s], golden["weights.depth"]) < TOL
