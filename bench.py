#!/usr/bin/env python
"""bench.py -- rays/s of the fused render path (BASELINE.json: 300^3 VM grid, 4096-ray batches).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
                    [--workload cfg2|distB|incoherent|cfg3|cfg5] [--scaling weak|strong|frame]
                    [--exchange fused|nccl] [--lag L] [--grid-storage fp32|bf16] [--dump-outputs DIR]

Workloads (SURVEY.md 8d; fields built by the reference's constructor defaults, random init):
  cfg2        (default, the headline) one TensorVMSplit at 300^3, seed 0, an 800x800 pinhole frame at
              fov 85.6, identity pose, cut into 4096-ray batches; step = one batch
  distB       cfg2 with density_shift = +2 ("opaque": early ray termination)
  incoherent  cfg2's field, training-style batches: 16 views x 256 random pixels each
  cfg3        three 300^3 fields (seeds 0,1,2), world2rf offsets, explicit blend [0.2,0.5,0.3]
  cfg5        slice of config 5: 8 fields at 640^3 (S = 738), 64-frame trajectory along -z with the
              reference's own cross-fade rows, floater_thresh 0.5; step = one 4096-ray batch of a frame

One STEP = one batch through the public API `LocalTensorfs.forward` (one fused launch per active
field: ray generation + march + shading + composite + blend).  Steps walk through different batches.

  value     rays/s with the batch's ray ids already in HBM; each step timed with CUDA events on the
            launching stream; 2 x 256 MiB writes between steps flush the 126 MB L2 (and keep the GPU
            busy while the host prepares the next call, so no host time leaks into the events).
  e2e       the same step from PINNED HOST ray ids to PINNED HOST rgb+depth: the kernel reads the ids
            and stores the finished pixels over PCIe itself (zero-copy; every input / output byte
            crosses the bus inside the timed region), then one stream sync -- every step, wall clock.
  roofline  algorithmic gather bytes (576 B per density sample, 1728 B per shaded sample, 40 B per
            ray; samples counted exactly by the kernel) / event-timed launch duration, against the
            measured HBM copy bandwidth in MEASURED_PEAKS.json; `traffic` = DRAM bytes per launch of
            the committed ncu capture of this workload (profiles/traffic.json), or null.
  cpu_baseline / --impl reference: the UNMODIFIED PyTorch reference (its bytecode, compiled by build() into
            oracle/_ref, or a checkout named by $LOCALRF_REFERENCE; oracle/ref_loader.py) on all host cores,
            4096 rays per step; the CPU oracle port (oracle/lrf_oracle.c) if neither is there.
            `reference_gpu` = the same unmodified reference with device="cuda" on this B200.

N > 1 (torchrun, one rank per GPU), field replicated, rays sharded, no data-path collective:
  --scaling weak    every rank renders its own 4096-ray batch per step (global batch N*4096)
  --scaling strong  each 4096-ray batch is split N ways (BASELINE config 4 as written)
  --scaling frame   the 640 000 rays of a frame are split N ways, one exchange per frame
  The rendered [rays,4] pixels (rgb+depth) are exchanged by the render kernel itself: the thread that
  finishes a ray stores it into every peer's gathered buffer (symmetric memory over NVLink/NVSwitch,
  NVLS multicast when available); the kernel's last CTA publishes the step in every peer's flag array and
  the next launches wait (in their prologue) for the peers' step s-1-lag -- no barrier launch, no collective
  (--exchange fused, --lag 3 default; --lag 0 = same-step barrier kernel); --exchange nccl uses one
  ncclAllGather per step instead.

--dump-outputs DIR: after the timed steps, the arrays the last timed step returned to its caller (rgb, depth,
  directions, ij of LocalTensorfs.forward; rank 0) are written as DIR/<name>.npy in float32 / float64, so two
  builds can be compared output for output: the same arguments give the same inputs.

--grid-storage bf16 (NOT the headline; a separate, labelled line): eval kernels gather bfloat16 copies of the
  grids (LocalTensorfs.set_grid_storage); the roofline then counts 288 / 864 B per density / appearance sample.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

GRID = 300
IMG_W = IMG_H = 800
BATCH = 4096
FOV = 85.6
FALLBACK_HBM_GBS = 6650.0   # B200_PROFILING.md fallback

_REAL_STDOUT = None


def quiet_stdout():
    """Everything libraries print (NCCL's version banner, torchrun notices) goes to stderr; only the
    ONE JSON line reaches the real stdout."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit(line):
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode()); sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


def field_kwargs(**over):
    kw = dict(density_n_comp=[8, 8, 8], appearance_n_comp=[24, 24, 24], app_dim=27,
              shadingMode="MLP_Fea_late_view", near_far=[0.1, 1e3], density_shift=-5,
              alphaMask_thres=1e-4, distance_scale=25, rayMarch_weight_thres=1e-3, pos_pe=0,
              view_pe=0, fea_pe=0, featureC=128, step_ratio=0.5, fea2denseAct="softplus")
    kw.update(over)
    return kw


def _scene(cls, device, grid, n_init_frames=1, **over):
    torch.manual_seed(0)
    aabb = 2 * torch.tensor([[-1.0, -1, -1], [1, 1, 1]])
    return cls(camera_prior=None, fov=FOV, n_init_frames=n_init_frames, n_overlap=30,
               WH=(IMG_W, IMG_H), n_iters_per_frame=600, n_iters_reg=100, lr_R_init=5e-3,
               lr_t_init=5e-4, lr_i_init=0, lr_exposure_init=1e-3, rf_lr_init=2e-2,
               rf_lr_basis=1e-3, lr_decay_target_ratio=0.1, N_voxel_list={},
               update_AlphaMask_list=[], lr_upsample_reset=True, device=device,
               aabb=aabb.to(device) if device != "cpu" else aabb, gridSize=[grid] * 3,
               **field_kwargs(**over))


def build_scene(device, grid=GRID, **over):
    """Product LocalTensorfs with one field, reference constructor defaults, seed 0 (built on the CPU
    so the init draws are the reference's, then moved)."""
    import localrf_b200 as L
    lt = _scene(L.LocalTensorfs, "cpu", grid, **over)
    return lt.to(device) if str(device) != "cpu" else lt


# ---- workloads -----------------------------------------------------------------------------------
class Workload:
    """Scene construction + the batches of one --workload; the SAME code builds the product's scene and
    the unmodified reference's (both constructors consume the RNG identically)."""

    def __init__(self, name, grid=None):
        self.name = name
        self.grid = grid if grid is not None else (640 if name == "cfg5" else GRID)
        self.floater = 0.5 if name == "cfg5" else 0.0
        self.n_frames = {"incoherent": 16, "cfg5": 64}.get(name, 1)

    def build(self, cls, quiet=False):
        import contextlib, io
        ctx = contextlib.redirect_stdout(io.StringIO()) if quiet else contextlib.nullcontext()
        with ctx:
            return self._build(cls)

    def _build(self, cls):
        name, grid = self.name, self.grid
        if name in ("cfg2", "distB"):
            return _scene(cls, "cpu", grid, **({"density_shift": 2} if name == "distB" else {}))
        if name == "incoherent":
            lt = _scene(cls, "cpu", grid, n_init_frames=16)
            g = torch.Generator().manual_seed(5)
            with torch.no_grad():                     # 16 nearby, distinct cameras
                for i in range(16):
                    lt.r_c2w[i].add_(0.05 * torch.randn(3, 2, generator=g))
                    lt.t_c2w[i].add_(0.1 * torch.randn(3, generator=g))
            return lt
        if name == "cfg3":
            lt = _scene(cls, "cpu", grid)
            for k in (1, 2):
                lt.append_frame()                     # append_rf needs >= 2 frames to cross-fade over
                torch.manual_seed(k)
                lt.append_rf(1)
            return lt
        if name == "cfg5":
            # 8 fields, 8 frames per field, camera translating along -z; blending rows and world2rf by
            # the reference's own append_frame / append_rf bookkeeping (local_tensorfs.py:116-177)
            lt = _scene(cls, "cpu", grid)
            for f in range(1, self.n_frames):
                lt.append_frame()
                with torch.no_grad():
                    lt.t_c2w[-1].copy_(torch.tensor([0.0, 0.0, -0.05 * f]))
                if f % 8 == 0:
                    torch.manual_seed(f // 8)
                    lt.append_rf(4)
            return lt
        raise ValueError(name)

    def call_kwargs(self, lt, dev):
        kw = dict(is_train=False, chunk=BATCH)
        if self.floater:
            kw["floater_thresh"] = self.floater
        if self.name == "cfg3":
            kw["world2rf"] = [torch.zeros(3, device=dev), torch.tensor([-0.3, 0.0, 0.0], device=dev),
                              torch.tensor([-0.6, 0.0, 0.0], device=dev)]
            kw["blending_weights"] = torch.tensor([[0.2, 0.5, 0.3]], device=dev)
        return kw

    def batches(self):
        """-> (ids [n_batches, BATCH] int64 (host), views: list of host int64 tensors per batch)"""
        n_full = IMG_W * IMG_H // BATCH
        frame = torch.arange(n_full * BATCH, dtype=torch.int64).view(n_full, BATCH)
        if self.name == "incoherent":
            g = torch.Generator().manual_seed(6)
            px = torch.randint(0, IMG_W * IMG_H, (64, 16, BATCH // 16), generator=g)
            ids = (px + torch.arange(16)[None, :, None] * IMG_W * IMG_H).reshape(64, BATCH)
            return ids, [torch.arange(16)] * 64
        if self.name == "cfg5":
            ids, views = [], []
            for i in range(64):
                ids.append(frame[(i * 37) % n_full])
                views.append(torch.tensor([(i * 11) % self.n_frames]))
            return torch.stack(ids), views
        return frame, [torch.tensor([0])] * n_full

    def describe(self):
        return {
            "cfg2": f"cfg2: TensorVMSplit {self.grid}^3 (reference ctor, seed 0, random init), 800x800 pinhole "
                    "frame fov 85.6 identity pose, 4096-ray batches; step = one batch, steps walk the frame",
            "distB": f"distribution B: cfg2 with density_shift=+2 (opaque, early ray termination), {self.grid}^3",
            "incoherent": f"incoherent: cfg2's {self.grid}^3 field, training-style batches of 16 views x 256 "
                          "random pixels (localrf_dataset.py:273-315), eval arithmetic",
            "cfg3": f"cfg3: 3 fields {self.grid}^3 (seeds 0,1,2), world2rf (0,-.3,-.6), blend [0.2,0.5,0.3], "
                    "4096-ray batches of the 800x800 frame",
            "cfg5": f"cfg5 slice: 8 fields {self.grid}^3, 64-frame -z trajectory, reference cross-fade rows "
                    "(1-2 active fields per frame), floater_thresh 0.5, 4096-ray batches of varying frames",
        }[self.name]


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return FALLBACK_HBM_GBS, "fallback (B200_PROFILING.md)"


def traffic_for(workload):
    """DRAM bytes per launch from the committed ncu capture of this workload (profiles/traffic.json,
    written by profiles/ncu_traffic.py from an `ncu --set full` export), or (None, None)."""
    try:
        t = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))[workload]
        return float(t["dram_bytes_per_launch"]), t["source"]
    except Exception:
        return None, None


class ClockSampler(threading.Thread):
    """SM clock + throttle reasons DURING the timed region (B200_PROFILING.md).  NVML (pynvml) is
    polled every ~2 ms because the timed region is only tens of milliseconds long; nvidia-smi
    (one sample per ~100 ms) is the fallback."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.stop_flag = index, [], False
        self.nvml = None
        try:
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[index]) if vis and vis.split(",")[index].isdigit() else index
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
            self.nvml = pynvml
        except Exception:
            self.nvml = None

    def _sample_nvml(self):
        n = self.nvml
        mhz = float(n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM))
        r = int(n.nvmlDeviceGetCurrentClocksEventReasons(self.handle)) if hasattr(
            n, "nvmlDeviceGetCurrentClocksEventReasons") else int(
            n.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle))
        flags = [bool(r & 0x8), bool(r & 0x40), bool(r & 0x20), bool(r & 0x4)]  # hw_slowdown, hw_thermal, sw_thermal, sw_power_cap
        self.samples.append([mhz, self.max_mhz] + ["Active" if f else "Not Active" for f in flags])

    def run(self):
        while not self.stop_flag:
            try:
                if self.nvml is not None:
                    self._sample_nvml()
                    time.sleep(0.002)
                    continue
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                      "-i", str(self.index)], capture_output=True, text=True, timeout=5).stdout
                parts = [x.strip() for x in out.strip().split(",")]
                if len(parts) >= 6:
                    self.samples.append(parts)
            except Exception:
                self.nvml = None
            time.sleep(0.02)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        sm = sorted(float(s[0]) for s in self.samples)
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(str(s[2 + i]).lower().startswith("active") for s in self.samples)]
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": float(self.samples[0][1]), "reasons": reasons,
                "samples": len(sm), "source": "nvml" if self.nvml is not None else "nvidia-smi"}


# ---- CPU / reference legs ------------------------------------------------------------------------
def frame_ids():
    return torch.arange(IMG_W * IMG_H, dtype=torch.int64)


def oracle_field(lt):
    from oracle import oracle as orc
    rf = lt.tensorfs[0]
    fd = {k: v.detach().cpu().numpy() for k, v in rf.state_dict().items()}
    kw = rf.get_kwargs()
    for k in ("density_shift", "distance_scale", "rayMarch_weight_thres", "fea_pe", "view_pe",
              "featureC", "app_dim", "step_ratio", "fea2denseAct", "gridSize"):
        fd[k] = kw[k]
    return orc.Field(fd)


def oracle_batch(lt, field, ids, n_threads=None):
    """One cfg2 batch through the CPU oracle's LocalTensorfs.forward restatement, on ALL host cores
    (explicit thread count: torchrun exports OMP_NUM_THREADS=1 to its workers)."""
    if n_threads is None:
        n_threads = os.cpu_count() or 1
    from oracle import oracle as orc
    z = orc.sample_table(field.n_samples())
    focal = float(lt.focal(IMG_W).detach().cpu())
    cx, cy = [float(v) for v in lt.center(IMG_W, IMG_H).detach().cpu()]
    c2w = lt.get_cam2world(torch.tensor([0])).detach().cpu().numpy()
    expo = torch.stack(list(lt.exposure))[[0]].detach().cpu().numpy()
    return orc.local_forward([field], [z], ids, IMG_W, IMG_H, False, focal, cx, cy, c2w,
                             np.zeros((1, 3), np.float32), np.ones((1, 1), np.float32),
                             exposure=expo, n_threads=n_threads)


def load_reference_classes():
    """The unmodified reference's LocalTensorfs (oracle/ref_loader.py), or None."""
    try:
        from oracle.ref_loader import load_reference, reference_available
        if not reference_available():
            return None
        return load_reference()[2]
    except Exception as e:  # pragma: no cover
        print(f"bench: reference import failed ({e}); falling back to the oracle port", file=sys.stderr)
        return None


class ReferenceRunner:
    """Steps of a workload through the UNMODIFIED reference's own public API (its stock PyTorch path)."""

    def __init__(self, wl, device):
        cls = load_reference_classes()
        if cls is None:
            raise RuntimeError("reference not available")
        self.wl, self.dev = wl, torch.device(device)
        lt = wl.build(cls, quiet=True)
        if self.dev.type == "cuda":
            # the reference's own device handling: parameters follow .to(), helper tensors follow
            # the `device` attribute (local_tensorfs.py:59,132)
            # every field resident on the GPU (the reference parks older fields on the CPU and
            # shuffles them per frame, local_tensorfs.py:132,432-434,476-479; not reproduced here:
            # this baseline is the reference's arithmetic at its best)
            lt = lt.to(self.dev)
            lt.device = self.dev
            for rf in lt.tensorfs:
                rf.to(self.dev)                      # TensorBase.to also retargets rf.device / stepSize
        self.lt = lt
        ids, views = wl.batches()
        self.ids = ids.to(self.dev)
        self.views = [v.to(self.dev) for v in views]
        self.kw = wl.call_kwargs(lt, self.dev)

    def step(self, i):
        import contextlib, io
        bi = (i * 37) % self.ids.shape[0]
        with torch.no_grad(), contextlib.redirect_stdout(io.StringIO()):
            out = self.lt(self.ids[bi], self.views[bi], IMG_W, IMG_H, **self.kw)
        if self.dev.type == "cuda":
            torch.cuda.synchronize(self.dev)
        return out


def time_reference(wl, device, warmup, steps):
    r = ReferenceRunner(wl, device)
    for i in range(warmup):
        r.step(i)
    t0 = time.perf_counter()
    for i in range(steps):
        r.step(warmup + i)
    dt = time.perf_counter() - t0
    return BATCH * steps / dt, dt


def cpu_baseline(wl, budget_s=20.0):
    """Reported CPU baseline at N=1: the unmodified reference on all host cores (bounded: 1 warm-up +
    as many 4096-ray batches as fit ~budget_s, at least 2); oracle port if it cannot be imported."""
    torch.set_num_threads(os.cpu_count() or 1)
    try:
        r = ReferenceRunner(wl, "cpu")
        t0 = time.perf_counter(); r.step(0); t1 = time.perf_counter() - t0
        steps = int(min(max(budget_s / max(t1, 1e-3), 2), 16))
        t0 = time.perf_counter()
        for i in range(steps):
            r.step(1 + i)
        dt = time.perf_counter() - t0
        return {"value": BATCH * steps / dt, "unit": "rays/s", "cores": torch.get_num_threads(), "kind": "reference",
                "sample": f"{steps} batches of 4096 rays of workload {wl.name}, unmodified PyTorch reference "
                          f"(LocalTensorfs.forward, torch {torch.__version__}, "
                          f"{torch.get_num_threads()} threads), {dt:.2f} s"}
    except Exception as e:
        print(f"bench: reference CPU baseline unavailable ({e}); using the oracle port", file=sys.stderr)
    if wl.name not in ("cfg2", "distB"):
        return None
    lt = wl.build(__import__("localrf_b200").LocalTensorfs, quiet=True)
    field = oracle_field(lt)
    ids = frame_ids().numpy()
    mid = (IMG_W * IMG_H // 2 // BATCH) * BATCH
    oracle_batch(lt, field, ids[mid:mid + 256])
    t0 = time.perf_counter()
    oracle_batch(lt, field, ids[mid:mid + BATCH])
    dt = time.perf_counter() - t0
    return {"value": BATCH / dt, "unit": "rays/s", "cores": os.cpu_count(), "kind": "port",
            "sample": f"one 4096-ray batch (from ray {mid}), oracle/lrf_oracle.c, OpenMP {os.cpu_count()} threads, {dt:.2f} s"}


def run_reference(args):
    """--impl reference: the unmodified PyTorch reference on this box's host cores (rank 0 only),
    4096 rays per step, same workload / metric as our arm."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    wl = Workload(args.workload, args.grid)
    torch.set_num_threads(os.cpu_count() or 1)
    kind, cores = "reference", torch.get_num_threads()
    try:
        value, dt = time_reference(wl, "cpu", args.warmup, args.steps)
        sample = (f"4096 rays per step, unmodified PyTorch reference, LocalTensorfs.forward, "
                  f"torch {torch.__version__}, {cores} threads")
    except Exception as e:
        print(f"bench: reference unavailable ({e}); timing the oracle port", file=sys.stderr)
        if wl.name not in ("cfg2", "distB"):
            emit({"impl": "reference", "unavailable": f"reference not importable and the oracle port covers cfg2 only ({e})"})
            return
        kind, cores = "port", os.cpu_count()
        lt = wl.build(__import__("localrf_b200").LocalTensorfs, quiet=True)
        field = oracle_field(lt)
        ids = frame_ids().numpy()
        n_batches = IMG_W * IMG_H // BATCH
        def step(i):
            lo = (i * 37 % n_batches) * BATCH
            oracle_batch(lt, field, ids[lo:lo + BATCH])
        for i in range(args.warmup):
            step(i)
        t0 = time.perf_counter()
        for i in range(args.steps):
            step(args.warmup + i)
        dt = time.perf_counter() - t0
        value = BATCH * args.steps / dt
        sample = f"4096 rays per step, oracle/lrf_oracle.c, OpenMP {cores} threads"
    emit({
        "impl": "reference", "metric": "rays/sec at 300^3 VM grid, 4096-ray batch", "value": value,
        "unit": "rays/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": args.scaling,
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": wl.describe(), "rays_per_batch": BATCH},
        "cpu_baseline": {"value": value, "unit": "rays/s", "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": value, "unit": "rays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    })


# ---- our arm ---------------------------------------------------------------------------------------
OUTPUT_NAMES = ("rgb", "depth", "directions", "ij")          # LocalTensorfs.forward's return, in order


def dump_outputs(path, outputs):
    """DIR/<name>.npy of every array a step returned: floating point as float32, integers as float64 (exact)."""
    os.makedirs(path, exist_ok=True)
    for name, t in zip(OUTPUT_NAMES, outputs):
        a = t.detach().cpu().numpy()
        np.save(os.path.join(path, name + ".npy"), a.astype(np.float32 if a.dtype.kind == "f" else np.float64))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="cfg2", choices=["cfg2", "distB", "incoherent", "cfg3", "cfg5"])
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong", "frame"])
    ap.add_argument("--exchange", default="fused", choices=["fused", "nccl"])
    ap.add_argument("--lag", type=int, default=3, help="fused exchange: steps of slack between a rank and its "
                    "slowest peer (0 = same-step barrier; L >= 1: step s waits for the peers' step s-1-L, the "
                    "gathered image of step s-1-L is complete after the launch of step s)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-reference-gpu", action="store_true")
    ap.add_argument("--grid", type=int, default=None)
    ap.add_argument("--grid-storage", default="fp32", choices=["fp32", "bf16"],
                    help="storage type the eval kernels gather the plane / line grids from (LocalTensorfs."
                         "set_grid_storage): fp32 = the parameters (the headline, the reference's precision); "
                         "bf16 = bfloat16 copies, half the gather bytes (a separate, labelled line -- it renders "
                         "the bf16-rounded field)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the arrays the last timed step returned as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps is not None and args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    quiet_stdout()
    if args.steps is None:
        args.steps = 20 if args.impl == "reference" else 157
    if args.impl == "reference":
        return run_reference(args)
    if args.warmup < 3:
        args.warmup = 3

    import localrf_b200 as L
    torch.set_grad_enabled(False)               # inference bench: the fused eval path, like renderer.py's @torch.no_grad

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback); use --impl reference for the CPU reference")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)

    wl = Workload(args.workload, args.grid)
    lt = wl.build(L.LocalTensorfs, quiet=True).to(dev)
    bf16 = args.grid_storage == "bf16"
    if bf16:
        lt.set_grid_storage("bf16")
    kw = wl.call_kwargs(lt, dev)
    ids_host, views_host = wl.batches()
    n_batches = ids_host.shape[0]
    scaling = args.scaling if world > 1 else "weak"
    if scaling == "frame":                                   # step = the whole frame, split N ways
        ids_host = frame_ids()[None]
        views_host = [torch.tensor([0])]
        n_batches = 1
    rays_per_step_global = {"weak": world * BATCH, "strong": BATCH, "frame": IMG_W * IMG_H}[scaling]
    ids_dev = ids_host.to(dev)
    views_dev = {id(v): v.to(dev) for v in views_host}      # one device tensor per distinct view list
    stats = torch.zeros(2, dtype=torch.int64, device=dev)

    # ---- multi-GPU plumbing ----------------------------------------------------------------------------
    from localrf_b200.dist import PixelExchange, shard_bounds
    xch, exchange_kind = None, None
    if world > 1:
        exchange_kind = args.exchange
        if args.exchange == "fused":
            try:
                xch = PixelExchange(rays_per_step_global, device=dev, lag=args.lag)
                exchange_kind = ("fused (multimem stores)" if xch.mc_ptr else "fused (peer stores)") + \
                    (f", slack {args.lag} step(s): no barrier launch, step s waits for the peers' step s-{1 + args.lag}"
                     if args.lag >= 1 else ", same-step barrier kernel")
            except Exception as e:
                print(f"bench: symmetric memory unavailable ({e}); using the NCCL all-gather", file=sys.stderr)
                exchange_kind = "nccl (fused unavailable)"
        if xch is None:
            shard = {"weak": BATCH, "strong": -(-BATCH // world // 8) * 8, "frame": -(-IMG_W * IMG_H // world // 8) * 8}[scaling]
            gathered = torch.empty(world * shard, 4, device=dev)
            pix_pad = torch.zeros(shard, 4, device=dev)

    def shard_of(n):
        """(lo, hi, row offset in the gathered buffer) of this rank's rays for one step"""
        if scaling == "weak":
            return 0, n, rank * n
        lo, hi = shard_bounds(n, rank, world)
        return lo, hi, lo

    def batch_index(i):
        return ((i * world + rank) * 37) % n_batches if scaling == "weak" else (i * 37) % n_batches

    def step(i, ids_all, out=None, want_stats=True):
        bi = batch_index(i)
        ids = ids_all[bi]
        lo, hi, row = shard_of(ids.shape[0])
        view = views_dev[id(views_host[bi])]
        if xch is not None:
            return lt(ids[lo:hi], view, IMG_W, IMG_H, stats=stats if want_stats else None,
                      exchange=(xch, row), **kw)
        r = lt(ids[lo:hi], view, IMG_W, IMG_H, stats=stats if want_stats else None, out=out, **kw)
        if world > 1:
            pix_pad[:hi - lo, :3] = r[0]; pix_pad[:hi - lo, 3] = r[1]
            dist.all_gather_into_tensor(gathered, pix_pad)
        return r

    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    for i in range(args.warmup):
        step(i, ids_dev); flush.zero_()
    torch.cuda.synchronize()
    stats.zero_()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    sampler = ClockSampler(local_rank)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    sampler.start()
    for i in range(args.steps):
        flush.zero_(); flush.zero_()         # L2 flush between timed iterations (outside the events)
        ev[i][0].record()
        last = step(args.warmup + i, ids_dev)
        ev[i][1].record()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    sampler.stop_flag = True
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last)
    del last
    times_ms = [a.elapsed_time(c) for a, c in ev]
    total_ms = torch.tensor([sum(times_ms)], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(total_ms, op=dist.ReduceOp.MAX)
    total_ms = float(total_ms)
    st = stats.cpu().tolist()
    value = rays_per_step_global * args.steps / (total_ms * 1e-3)
    launches = [len(p.launches) for p in lt.__dict__.get("_plans", {}).values()]
    # (+ one barrier kernel per step only for the same-step exchange; with slack the render kernel signals itself)
    gpu_launches = args.steps * (max(launches) if launches else 1) + (args.steps if xch is not None and xch.lag == 0 else 0)

    # N > 1: what a step costs on each rank without any exchange (per-rank events, max over ranks): separates
    # the kernel from the exchange / rank-desynchronisation share of ms_per_step
    ms_no_exchange = None
    if world > 1:
        k = max(args.steps // 2, 8)
        evx = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(k)]
        dist.barrier(); torch.cuda.synchronize()
        for i in range(k):
            flush.zero_(); flush.zero_()
            bi = batch_index(args.warmup + i)
            lo, hi, _ = shard_of(ids_dev[bi].shape[0])
            evx[i][0].record()
            lt(ids_dev[bi][lo:hi], views_dev[id(views_host[bi])], IMG_W, IMG_H, **kw)
            evx[i][1].record()
        torch.cuda.synchronize()
        t = torch.tensor([sum(a.elapsed_time(c) for a, c in evx) / k], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_no_exchange = float(t)

    # roofline of the fused kernel (this rank's launches; N=1 only: with N>1 the events also cover the exchange)
    peak, peak_src = peaks()
    roofline = None
    if world == 1:
        rays_total = BATCH * args.steps
        # SURVEY.md 8d: "with 16-bit grid storage halve the 576 / 1728 terms and say so"
        bytes_total = st[0] * (288 if bf16 else 576) + st[1] * (864 if bf16 else 1728) + rays_total * 40
        achieved = bytes_total / (sum(times_ms) * 1e-3) / 1e9
        traffic, traffic_src = traffic_for(wl.name) if not bf16 else (None, None)   # (the captures are of the fp32 kernel)
        n_kern = max(launches) if launches else 1
        roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                    "frac": achieved / peak, "traffic": traffic, "traffic_source": traffic_src,
                    "algorithmic_bytes_per_launch": bytes_total / (args.steps * n_kern),
                    "launches_per_step": n_kern, "peak_source": peak_src,
                    "kernel": "lrf::render_kernel_t<false, true>" if bf16 else "lrf::render_kernel_t<false, false>",
                    "bytes_per_sample": {"density": 288 if bf16 else 576, "appearance": 864 if bf16 else 1728},
                    "bytes_per_ray": bytes_total / rays_total,
                    "density_samples_per_ray": st[0] / rays_total,
                    "app_samples_per_ray": st[1] / rays_total,
                    "note": "algorithmic gather bytes (every texel fetch counted, all active fields); a 300^3 "
                            "field (33 MB) is L2-resident, so DRAM counters read far lower (profiles/)"}

    # ---- e2e: public API from pinned host ids to pinned host pixels, every step ----------------------------
    # Two figures.  `sync`: submit a step, wait for its result, submit the next (a caller that needs
    # each batch before issuing the next one).  `pipelined` (the headline e2e): the renderer's loop --
    # step i+1 is submitted before step i's result is consumed (two pinned result buffers, one CUDA event
    # per step), so the host's share of a step overlaps the GPU's.  Both: every step reads its ray ids
    # from pinned host memory and delivers its pixels to pinned host memory inside the timed region.
    ids_pin = ids_host.pin_memory()
    n_loc = max(shard_of(ids_host.shape[1])[1] - shard_of(ids_host.shape[1])[0], 1)
    bufs = [(torch.empty(n_loc, 3).pin_memory(), torch.empty(n_loc).pin_memory()) for _ in range(2)]
    full_host = [torch.empty(rays_per_step_global, 4).pin_memory() for _ in range(2)] if world > 1 else None
    events = [torch.cuda.Event(), torch.cuda.Event()]
    stream = torch.cuda.current_stream(dev)

    def e2e_submit(i):
        k = i & 1
        if world == 1:
            step(i, ids_pin, out=bufs[k], want_stats=False)
        else:
            step(i, ids_pin, want_stats=False)
            src = xch.gathered(rays_per_step_global) if xch is not None else gathered[:rays_per_step_global]
            full_host[k][:src.shape[0]].copy_(src, non_blocking=True)
        events[k].record(stream)

    def e2e_consume(i):
        k = i & 1
        events[k].synchronize()
        res = bufs[k][0] if world == 1 else full_host[k]
        return float(res[0, 0])                  # the host touches the delivered result

    def e2e_run(pipelined):
        for i in range(args.warmup):
            e2e_submit(i); e2e_consume(i)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        if pipelined:
            e2e_submit(args.warmup)
            for i in range(args.warmup + 1, args.warmup + args.steps):
                e2e_submit(i)
                e2e_consume(i - 1)
            e2e_consume(args.warmup + args.steps - 1)
        else:
            for i in range(args.warmup, args.warmup + args.steps):
                e2e_submit(i); e2e_consume(i)
        torch.cuda.synchronize()
        sec = torch.tensor([time.perf_counter() - t0], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(sec, op=dist.ReduceOp.MAX)
        return rays_per_step_global * args.steps / float(sec)

    e2e_sync_value = e2e_run(False)
    e2e_value = e2e_run(True)
    h2d = n_loc * 8
    d2h = n_loc * 16 if world == 1 else rays_per_step_global * 16

    # ---- whole frame through the API (one fused launch per field for all 640k rays), informational -----------
    frame = None
    if world == 1 and wl.name in ("cfg2", "distB", "cfg3"):
        all_ids = frame_ids().pin_memory()
        view0 = views_dev[id(views_host[0])]
        def frame_call():
            with torch.no_grad():
                r, d, _, _ = lt(all_ids.to(dev, non_blocking=True), view0, IMG_W, IMG_H, **kw)
            r.cpu(); d.cpu()
        frame_call()
        torch.cuda.synchronize(); t0 = time.perf_counter()
        frame_call()
        frame = {"rays_per_s": IMG_W * IMG_H / (time.perf_counter() - t0),
                 "what": "LocalTensorfs.forward on all 640000 rays of the frame incl. H2D/D2H"}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    cpu, ref_gpu = None, None
    if world == 1:
        if not args.no_reference_gpu:
            try:
                del flush
                torch.cuda.empty_cache()
                v, dt = time_reference(wl, dev, 2, 5)
                ref_gpu = {"value": v, "unit": "rays/s", "what": "the unmodified PyTorch reference, "
                           f"device=cuda on this GPU, same workload, 5 batches of 4096 rays after 2 warm-ups, {dt:.3f} s"}
            except Exception as e:
                ref_gpu = {"unavailable": str(e)[:200]}
        if not args.no_cpu_baseline:
            cpu = cpu_baseline(wl)
    line = {
        "metric": "rays/sec at 300^3 VM grid, 4096-ray batch", "value": value, "unit": "rays/s",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": total_ms / args.steps, "higher_is_better": True,
        "scaling": "weak" if scaling == "weak" else "strong",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "dtype_note": ("fp32 storage and arithmetic" if not bf16 else
                       "NOT the headline: fp32 arithmetic on bfloat16 GRID STORAGE (--grid-storage bf16; the render "
                       "equals the fp32 render of the bf16-rounded field, tests/test_gpu_bf16.py)") +
                      "; the two dense MLP layers run on tcgen05 as three bf16 "
                      "products of hi/lo-split fp32 operands with fp32 TMEM accumulators (1e-7 of fp32 on rgb, "
                      "tests/test_gpu_parity.py::test_tensor_core_mlp_vs_torch_fp32)",
        "config": {"workload": wl.describe(), "workload_key": wl.name, "rays_per_batch": BATCH,
                   "grid_storage": args.grid_storage,
                   "rays_per_step_global": rays_per_step_global,
                   "l2": "2 x 256 MiB writes between timed steps",
                   "sharding": {"weak": "every rank its own 4096-ray batch per step",
                                "strong": "each 4096-ray batch split over the ranks (BASELINE config 4)",
                                "frame": "the frame's 640000 rays split over the ranks, one exchange per frame"}[scaling],
                   "exchange": exchange_kind,
                   "ms_per_step_without_exchange": ms_no_exchange,
                   "parallelism": f"ray-batch data parallel x{world}"},
        "clocks": sampler.summary(),
        "e2e": {"value": e2e_value, "unit": "rays/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "sync_per_step_value": e2e_sync_value,
                "how": ("LocalTensorfs.forward per step: pinned host ray ids read and pinned host rgb/depth written "
                        "by the kernel over PCIe (zero-copy)" if world == 1 else
                        "LocalTensorfs.forward per step: pinned host ids (zero-copy), pixel exchange, D2H copy of "
                        "the gathered pixels") + "; value = two steps in flight (two result buffers, one event per "
                        "step, result of step i consumed after step i+1 is submitted); sync_per_step_value = each "
                        "step's result awaited before the next is submitted"},
        "gpu_launches": gpu_launches,
        "roofline": roofline,
        "cpu_baseline": cpu,
        "reference_gpu": ref_gpu,
        "frame_api": frame,
    }
    emit(line)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
