"""CPU-only: the bench's workloads build IDENTICAL scenes through the product's constructors and through the
unmodified reference's (same RNG consumption, same append_frame / append_rf bookkeeping), so `bench.py`'s two arms
and `reference_gpu` render the same thing; batches have the advertised shapes.  Small grids; the reference's scenes
are pinned by their state_dict digests (tests/golden/bench_scenes.json, tests/golden/make_golden.py)."""
import json
import os

import pytest
import torch

import bench
from helpers import GOLDEN, state_digest


@pytest.mark.parametrize("name", ["cfg2", "distB", "incoherent", "cfg3", "cfg5"])
def test_workload_scene_equal_for_product_and_reference(name):
    import localrf_b200 as L
    wl = bench.Workload(name, 12)
    ours = wl.build(L.LocalTensorfs, quiet=True)
    assert state_digest(ours.state_dict()) == json.load(open(os.path.join(GOLDEN, "bench_scenes.json")))["grid12"][name]
    assert len(ours.tensorfs) == {"cfg3": 3, "cfg5": 8}.get(name, 1)
    assert float(ours.tensorfs[0].density_shift) == (2 if name == "distB" else -5)
    ids, views = wl.batches()
    assert ids.shape[1] == bench.BATCH and ids.dtype == torch.int64 and len(views) == ids.shape[0]
    if name == "incoherent":
        assert views[0].numel() == 16 and int(ids.max()) < 16 * bench.IMG_W * bench.IMG_H
    else:
        assert all(v.numel() == 1 for v in views) and int(ids.max()) < bench.IMG_W * bench.IMG_H
    if name == "cfg5":      # cross-fade rows: one or two active fields per frame, rows sum to one
        bw = ours.blending_weights
        assert bw.shape == (64, 8) and torch.allclose(bw.sum(1), torch.ones(64))
        assert int((bw > 0).sum(1).max()) == 2 and int((bw > 0).sum(1).min()) == 1


def test_reference_arm_line_shape(monkeypatch, capsys):
    """`--impl reference` prints the contract's JSON keys (tiny grid, 1 step).  It times the reference's own
    code: the bytecode build() compiled into oracle/_ref, or a checkout named by $LOCALRF_REFERENCE."""
    if bench.load_reference_classes() is None:
        pytest.skip("no reference (oracle/_ref or $LOCALRF_REFERENCE)")
    import sys
    monkeypatch.setattr(bench, "_REAL_STDOUT", None)
    monkeypatch.setattr(bench, "quiet_stdout", lambda: None)
    monkeypatch.setattr(sys, "argv", ["bench.py", "--impl", "reference", "--steps", "1", "--warmup", "0", "--grid", "16"])
    bench.main()
    line = json.loads(capsys.readouterr().out.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["cpu_baseline"]["kind"] == "reference"
    assert line["unit"] == "rays/s" and line["value"] > 0 and line["e2e"]["h2d_bytes_per_step"] == 0
