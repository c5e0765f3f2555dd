#!/usr/bin/env python
"""bench.py -- voxel-channels/s of the 8-channel 1 A occupancy path (BASELINE.json metric) on N B200s.

    python bench.py --gpus N --steps K --warmup W            # our CUDA path
    python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU kernel on the host cores
    python bench.py ... --dump-outputs DIR                   # + what the last timed step computed, as DIR/*.npy

A "step" = one pass of the hot path (bin atoms -> scan -> scatter -> tile fill) over one batch of synthetic
pockets: BASELINE.json configs[2] (256 protein pockets x ~3000 atoms, 64^3 grid @ 1 A, 8 channels) PER GPU
(weak scaling: ranks voxelise independent batches, no data-path collective).  One JSON line on stdout (rank 0).

  value     voxel-channels/s, inputs resident in HBM, CUDA-event timed, max over ranks
  e2e       same metric through the public host API (getVoxelDescriptorsBatch): pinned host buffers in,
            pinned host features out, H2D + kernels + D2H inside the timed region
  roofline  algorithmic bytes of the fill kernel / its mean launch duration (CUDA events inside the library,
            recorded on the launch stream) against MEASURED_PEAKS.json hbm_gbs
  cpu_baseline  the reference's compiled Cython kernel (oracle/_ref, kind "reference") or the C port of it
            (kind "port") on a bounded sample of the same pockets, one process per host core
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

METRIC = "voxel-channels/s (8-ch 1A protein grids)"
UNIT = "voxel-channels/s"
HBM_FALLBACK_GBS = 6650.0  # /opt/skills/guides/B200_PROFILING.md fallback when MEASURED_PEAKS.json is absent


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c3", choices=["c3", "c2", "c5"])
    ap.add_argument("--batch", type=int, default=0, help="items per GPU (0 = the config's size)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the side measurements (C2 ligands, C5 fine grids, C4 distances)")
    ap.add_argument("--no-scaling", action="store_true", help="skip the strong-scaling / NCCL gather / config-4 section")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed (rank 0) as DIR/<name>.npy, "
                         "so that two builds can be compared output for output")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    return a


def make_workload(kind: str, batch: int, rank: int):
    from moleculekit_b200 import workloads

    if kind == "c3":
        return workloads.protein_pockets(B=batch or 256, seed=1000 + 100000 * rank)
    if kind == "c2":
        return workloads.ligand_poses(B=batch or 1024, seed=100000 * rank)
    return workloads.fine_grids(B=batch or 8, seed=2000 + 100000 * rank)


# ----------------------------------------------------------------------------------------------------- CPU arm
def host_cores() -> int:
    """Cores this process may really use: scheduler affinity, capped by the cgroup CPU quota (os.cpu_count() reports the
    box's logical CPUs even when a lease grants a fraction of them -- round 1's reference arm oversubscribed 128
    processes onto far fewer cores and hit the driver's time limit)."""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if q != "max":
            n = min(n, max(1, int(float(q) / float(per))))
    except Exception:
        try:
            q = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0:
                n = min(n, max(1, q // per))
        except Exception:
            pass
    return max(1, n)


_CPU_FN = {}


def _cpu_worker(args):
    """One bounded sample item: the leading `nslab` x-planes of one grid of the workload (the reference kernel's cost is
    atoms x centres, so a slab is the same work per voxel-channel)."""
    kind, coords, sigmas, boxsize, center, voxelsize, nslab = args
    if kind not in _CPU_FN:
        sys.path.insert(0, ROOT)
        if kind == "reference":
            from oracle import build_ref

            _CPU_FN[kind] = build_ref.load()[0].calculate_occupancy
        else:
            from oracle import cpu_oracle

            _CPU_FN[kind] = cpu_oracle.calculate_occupancy
    from moleculekit_b200.tools.voxeldescriptors import _centers_from_spec, _grid_spec

    bb_min, nvox = _grid_spec(None, 0, boxsize, center, voxelsize)
    per_plane = int(nvox[1]) * int(nvox[2])
    centers = _centers_from_spec(bb_min, nvox, voxelsize)[: max(1, min(int(nvox[0]), nslab)) * per_plane]
    out = np.zeros((centers.shape[0], sigmas.shape[1]))
    c32 = np.ascontiguousarray(coords, dtype=np.float32)
    s64 = np.ascontiguousarray(sigmas, dtype=np.float64)
    t0 = time.perf_counter()
    _CPU_FN[kind](np.ascontiguousarray(centers), c32, s64, out)
    return time.perf_counter() - t0, out.size


def cpu_kind():
    from oracle import build_ref, cpu_oracle

    try:
        build_ref.build(verbose=False)
    except Exception:
        pass
    if build_ref.load() is not None:
        return "reference"
    cpu_oracle.build()
    return "port"


class CpuArm:
    """The reference's CPU kernel on the host cores: `procs` single-threaded worker processes (the reference kernel is
    single-threaded, setup.py:48), each step = one item per process.  A pilot item sizes the slab so that a step takes
    about `step_seconds` of wall time -- fewer voxels per step, never fewer steps."""

    MAX_PROCS = 32  # beyond this the kernel (a 6 MB centre array streamed per atom) is memory bound: 128 procs were slower than 32

    def __init__(self, w, step_seconds: float):
        import multiprocessing as mp

        self.w, self.kind = w, cpu_kind()
        self.cores = host_cores()
        self.procs = max(1, min(self.cores, self.MAX_PROCS, len(w["coords"])))
        self.pool = mp.get_context("fork").Pool(processes=self.procs)
        # pilot: 2 planes of the first grid on one process
        nx = self._nx()
        t, n = self.pool.apply(_cpu_worker, (self._job(0, 2),))
        rate1 = n / max(t, 1e-6)                                   # voxel-channels/s of one unloaded core
        per_plane = n / 2
        # under load a core delivers maybe half of that (shared memory bandwidth): size for step_seconds of wall time
        self.target = step_seconds
        self.nslab = int(max(1, min(nx, 0.5 * rate1 * step_seconds / per_plane)))
        self.pilot = f"pilot {rate1:.3g} vc/s on 1 core"

    def _nx(self):
        from moleculekit_b200.tools.voxeldescriptors import _grid_spec

        return int(_grid_spec(None, 0, self.w["boxsize"], self.w["centers"][0], self.w["voxelsize"])[1][0])

    def _job(self, b, nslab):
        w = self.w
        return (self.kind, w["coords"][b], w["sigmas"][b], w["boxsize"], w["centers"][b], w["voxelsize"], nslab)

    def step(self):
        t0 = time.perf_counter()
        res = self.pool.map(_cpu_worker, [self._job(b, self.nslab) for b in range(self.procs)], chunksize=1)
        wall = time.perf_counter() - t0
        value = sum(r[1] for r in res) / wall
        if wall > 1.5 * self.target:  # the cores are slower than the pilot promised (shared host): shrink the slab, keep the steps
            self.nslab = max(1, int(self.nslab * self.target / wall))
        return value, wall

    def close(self):
        self.pool.close()
        self.pool.join()

    def describe(self, value):
        return dict(value=value, unit=UNIT, cores=self.procs, kind=self.kind,
                    sample=f"kernel only (centres prebuilt): {self.procs} single-threaded processes (host grants {self.cores} "
                           f"cores), one grid each, leading {self.nslab} of {self._nx()} x-planes per step; {self.pilot}")


def run_reference(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    w = make_workload(a.workload, a.batch, 0)
    n_steps = max(1, a.steps) + max(0, a.warmup)
    arm = CpuArm(w, step_seconds=min(8.0, 150.0 / n_steps))  # the whole run ends within ~3-4 minutes
    for _ in range(a.warmup):
        arm.step()
    vals, walls = [], []
    for _ in range(max(1, a.steps)):
        v, wall = arm.step()
        vals.append(v); walls.append(wall)
    arm.close()
    base = arm.describe(float(np.mean(vals)))
    line = dict(impl="reference", metric=METRIC, value=base["value"], unit=UNIT, n_gpus=a.gpus, steps=len(vals),
                warmup=a.warmup, ms_per_step=float(np.mean(walls)) * 1e3, higher_is_better=True, scaling="weak",
                vs_baseline=None, dtype="f64", data="synthetic",
                config=dict(workload=w["name"], sample_items=arm.procs, sample_x_planes=arm.nslab), cpu_baseline=base,
                e2e=dict(value=base["value"], unit=UNIT, h2d_bytes_per_step=0, d2h_bytes_per_step=0),
                gpu_launches=0)
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------------- clocks
class ClockSampler:
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index: int):
        self.rows, self.proc = [], None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(index)], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), line.strip()))

    def stop(self, t0, t1):
        if not self.proc:
            return None
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for t, row in self.rows:
            f = [x.strip() for x in row.split(",")]
            if len(f) < 7:
                continue
            if t0 - 0.05 <= t <= t1 + 0.15:
                try:
                    sm.append(float(f[0])); mx.append(float(f[1]))
                except ValueError:
                    continue
                for n, v in zip(names, f[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
        if not sm:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=[], samples=0)
        return dict(sm_mhz=float(np.median(sm)), sm_max_mhz=float(max(mx)), reasons=sorted(reasons), samples=len(sm))


# ----------------------------------------------------------------------------------------------------- side measurements
def cpu_next_rows(extra):
    """One core of the reference's own compiled kernels (oracle/_ref; else the C port) on bounded samples of the K9b / K12
    bench workloads (~1 s each), beside the GPU numbers of extra['c6b_wrap_triclinic'] / extra['c10_hbonds']."""
    from oracle import build_ref, cpu_oracle

    mods = build_ref.load()
    kind = "reference" if mods is not None and len(mods) >= 7 else "port"
    rng = np.random.default_rng(3)
    out = {"kind": kind, "cores": 1}
    # wrapping: 6000 atoms (1 solute of 600 + 1800 waters) x 4 frames in a rhombic dodecahedron
    n_prot, n_wat, F, L = 600, 1800, 4, 82.0
    N = n_prot + 3 * n_wat
    xyz = (rng.normal(0, 120, size=(N, 3, F))).astype(np.float32)
    groups = np.concatenate([[0], n_prot + 3 * np.arange(n_wat + 1)]).astype(np.uint32)
    bv = np.repeat(np.array([[L, 0, 0], [0, L, 0], [L / 2, L / 2, L * 2 ** 0.5 / 2]])[:, :, None], F, axis=2)
    cs, zero = np.arange(n_prot, dtype=np.uint32), np.zeros(3, np.float32)
    for name, mode in (("triclinic", None), ("compact", 1), ("rectangular", 0)):
        c = xyz.copy()
        t0 = time.perf_counter()
        if kind == "reference":
            (mods[3].wrap_triclinic_unitcell(groups, c, bv, cs, zero) if mode is None else
             mods[3].wrap_compact_unitcell(groups, c, bv, cs, zero, mode))
        else:
            (cpu_oracle.wrap_triclinic_unitcell(groups, c, bv, cs, zero) if mode is None else
             cpu_oracle.wrap_compact_unitcell(groups, c, bv, cs, zero, mode))
        dt = time.perf_counter() - t0
        g = extra.get("c6b_wrap_triclinic", {}).get(name, {}).get("atom_frames_per_s")
        out[f"wrap_{name}"] = dict(atom_frames_per_s=N * F / dt, sample=f"{N} atoms x {F} frames",
                                   gpu_over_one_core=(g / (N * F / dt)) if g else None)
    # hydrogen bonds: 1 frame, 2400 donor pairs x 1200 acceptors of a periodic water box
    nw = 1200
    O = rng.uniform(0, 33.0, size=(nw, 3, 1))
    h = rng.normal(size=(2, nw, 3, 1)); h /= np.linalg.norm(h, axis=2, keepdims=True)
    c = np.empty((3 * nw, 3, 1), np.float32); c[0::3] = O; c[1::3] = O + 0.96 * h[0]; c[2::3] = O + 0.96 * h[1]
    o = np.arange(0, 3 * nw, 3)
    don = np.concatenate([np.stack([o, o + 1], 1), np.stack([o, o + 2], 1)]).astype(np.uint32)
    acc, ones, box = o.astype(np.uint32), np.ones(3 * nw, np.uint32), np.full((3, 1), 33.0, np.float32)
    t0 = time.perf_counter()
    if kind == "reference":
        mods[6].calculate(don, acc, c, box, ones, ones, dist_threshold=2.5, angle_threshold=120, intra=True, ignore_hs=False)
    else:
        cpu_oracle.hbonds_calculate(don, acc, c, box, ones, ones, 2.5, 120, True, False)
    dt = time.perf_counter() - t0
    g = extra.get("c10_hbonds", {}).get("pair_tests_per_s")
    out["hbonds"] = dict(pair_tests_per_s=len(don) * len(acc) / dt, sample=f"1 frame x {len(don)} donor pairs x {len(acc)} acceptors",
                         gpu_over_one_core=(g / (len(don) * len(acc) / dt)) if g else None)
    # pi-pi: 300 six-rings against themselves, 4 frames
    nr, Fr = 300, 4
    xyz = (rng.uniform(0, 60, size=(6 * nr, 3, Fr))).astype(np.float32)
    ra, st = np.arange(6 * nr, dtype=np.uint32), np.arange(0, 6 * nr + 1, 6, dtype=np.uint32)
    boxr = np.full((3, Fr), 60.0, np.float32)
    t0 = time.perf_counter()
    if kind == "reference" and len(mods) >= 10:
        mods[7].calculate(ra, st, st, xyz, boxr, 4.4, 30.0, 5.5, 60.0)
    else:
        cpu_oracle.ring_interactions(0, ra, st, st, xyz, boxr, 4.4, 30.0, 5.5, 60.0)
    dt = time.perf_counter() - t0
    g = extra.get("c11_ring_detectors", {}).get("pipi_pair_tests_per_s")
    out["pipi"] = dict(pair_tests_per_s=Fr * nr * nr / dt, sample=f"{Fr} frames x {nr} x {nr} rings",
                       gpu_over_one_core=(g / (Fr * nr * nr / dt)) if g else None)
    return out


def _time_cuda(fn, warm=3, steps=10):
    import torch

    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def extra_workloads(dev, peak):
    """Other BASELINE configs on one GPU, device-resident, reported beside the headline (not part of `value`)."""
    import torch

    from moleculekit_b200 import _lib, distance_utils as du, workloads
    from moleculekit_b200.tools import voxeldescriptors as vd

    out = {}
    for key, w, layout in (("c2_ligand_poses", workloads.ligand_poses(B=1024), "xyzc"),
                           ("c5_fine_grids", workloads.fine_grids(B=4), "xyzc"),
                           ("c3_cxyz_layout", workloads.protein_pockets(B=128), "cxyz")):
        vb = vd.VoxelBatch(w["coords"], w["sigmas"], boxsize=w["boxsize"], centers=w["centers"], voxelsize=w["voxelsize"])
        d_c, d_s = vb.to_device(dev)
        o = torch.empty((vb.total_voxels, vb.C), dtype=torch.float32, device=dev)
        ms = _time_cuda(lambda: vb.run(d_c, d_s, o, layout=layout))
        vb.run(d_c, d_s, o, layout=layout)
        _, fill = _lib.get_timing(dev.index)
        nb = workloads.occupancy_algorithmic_bytes(vb.total_voxels, vb.coords.shape[0], vb.C)
        out[key] = dict(workload=w["name"] + (" -> (B,C,X,Y,Z) channel-major output" if layout == "cxyz" else ""),
                        voxel_channels_per_s=vb.total_voxels * vb.C / (ms * 1e-3), ms_per_step=ms,
                        fill_kernel_ms=fill, fill_kernel_gbs=nb / (fill * 1e-3) / 1e9, frac_of_peak=nb / (fill * 1e-3) / 1e9 / peak)
        del o, d_c, d_s
    # C4a: dense periodic distances, 256 x 1024 atoms, 10k frames (only the selected atoms are materialised)
    n1, n2, F = 256, 1024, 10000
    rng = np.random.default_rng(7)
    L = 36.84
    start = rng.uniform(0, L, size=(n1 + n2, 3, 1)).astype(np.float32)
    coords = start + np.cumsum(rng.normal(0, 0.3, size=(n1 + n2, 3, F)).astype(np.float32), axis=2)
    box = np.repeat((L * (1 + 0.002 * rng.normal(size=F))).astype(np.float32)[None, :], 3, axis=0)
    d_c = torch.from_numpy(np.ascontiguousarray(coords)).to(dev); d_b = torch.from_numpy(np.ascontiguousarray(box)).to(dev)
    s1 = torch.arange(0, n1, dtype=torch.int32, device=dev); s2 = torch.arange(n1, n1 + n2, dtype=torch.int32, device=dev)
    ch = torch.ones(n1 + n2, dtype=torch.int32, device=dev); ch[n1:] = 2
    # "distances": bit-identical to the reference's float32 sequence; "distances_fast": exact=False, within 4 ulp of it
    for key, s in (("distances", 4), ("distances_fast", 4), ("contacts", 1)):
        metric = "contacts" if key == "contacts" else "distances"
        kwd = dict(metric=metric, threshold=12.0, exact=(key != "distances_fast"))
        o = torch.empty((F, n1 * n2), dtype=torch.float32 if s == 4 else torch.uint8, device=dev)
        ms = _time_cuda(lambda: du.dist_trajectory_device(d_c, d_b, s1, s2, ch, False, True, out=o, **kwd), steps=5)
        du.dist_trajectory_device(d_c, d_b, s1, s2, ch, False, True, out=o, **kwd)
        prep, main = _lib.get_timing(dev.index)
        nb = F * ((n1 + n2) * 12 + 12 + n1 * n2 * s)
        out[f"c4a_{key}"] = dict(workload=f"C4a: {F} frames x {n1}x{n2} periodic pairs ({key})",
                                    pair_frames_per_s=F * n1 * n2 / (ms * 1e-3), ms_per_step=ms, gather_ms=prep,
                                    kernel_ms=main, kernel_gbs=nb / (main * 1e-3) / 1e9,
                                    frac_of_peak=nb / (main * 1e-3) / 1e9 / peak)
        del o
    # C4b: sparse ordered contacts (calculate_contacts), 1000 frames, 500 x 4500 atoms, <= 12 A
    n1, n2, F = 500, 4500, 1000
    start = rng.uniform(0, L, size=(n1 + n2, 3, 1)).astype(np.float32)
    coords = start + np.cumsum(rng.normal(0, 0.3, size=(n1 + n2, 3, F)).astype(np.float32), axis=2)
    box = np.repeat((L * (1 + 0.002 * rng.normal(size=F))).astype(np.float32)[None, :], 3, axis=0)
    d_c = torch.from_numpy(np.ascontiguousarray(coords)).to(dev); d_b = torch.from_numpy(np.ascontiguousarray(box)).to(dev)
    s1 = torch.arange(0, n1, dtype=torch.int32, device=dev); s2 = torch.arange(n1, n1 + n2, dtype=torch.int32, device=dev)
    ch = torch.ones(n1 + n2, dtype=torch.int32, device=dev); ch[n1:] = 2
    res = {}

    def run_contacts():
        res["off"], res["pairs"] = du.contacts_trajectory_device(d_c, d_b, s1, s2, ch, False, True, 12.0)

    n1c, n2c, Fsh = n1, n2, 1000
    ms = _time_cuda(run_contacts, warm=2, steps=3)
    npairs = int(res["pairs"].shape[0])
    out["c4b_sparse_contacts"] = dict(workload=f"C4b: {F} frames x {n1}x{n2} periodic pair tests <= 12 A, ordered index pairs",
                                      pair_tests_per_s=F * n1 * n2 / (ms * 1e-3), ms_per_step=ms, emitted_pairs=npairs,
                                      output_gbs=(npairs * 8 + F * n1 * 8) / (ms * 1e-3) / 1e9)
    # C4c: residue-level minimum distances (K5, MetricSelfDistance groupsel="residue"): 300 groups of 10 atoms, self
    n_res, per, Fc = 300, 10, 1000
    groups = [list(range(r * per, (r + 1) * per)) for r in range(n_res)]
    gch = torch.arange(n_res, dtype=torch.int32, device=dev) % 2
    masses = torch.ones(n_res * per, dtype=torch.float32, device=dev)
    d_cc = d_c[: n_res * per, :, :Fc].contiguous(); d_bc = d_b[:, :Fc].contiguous()
    ms = _time_cuda(lambda: du.dist_reduction_device(d_cc, d_bc, groups, groups, gch, gch, True, True, masses, 0, 0), warm=1, steps=3)
    npairs = n_res * (n_res - 1) // 2
    out["c4c_residue_mindist"] = dict(workload=f"C4c: {Fc} frames x {npairs} residue pairs ({per}x{per} atoms each), periodic, closest",
                                      ms_per_step=ms, group_pairs_per_s=Fc * npairs / (ms * 1e-3),
                                      atom_pair_tests_per_s=Fc * npairs * per * per / (ms * 1e-3))
    del d_c, d_b, res
    # C6: orthorhombic wrapping (K9) of an unwrapped solvated system: 5k-atom solute + 18k waters, 512 frames
    from moleculekit_b200 import wrapping as wr

    n_prot, n_wat, F = 5000, 18000, 512
    N = n_prot + 3 * n_wat
    g = torch.Generator(device=dev).manual_seed(5)
    L = 82.0
    d_orig = torch.empty((N, 3, F), dtype=torch.float32, device=dev)
    d_orig[:n_prot] = torch.randn((n_prot, 3, 1), generator=g, device=dev) * 9 + torch.randn((1, 3, F), generator=g, device=dev) * 25
    wat_c = (torch.rand((n_wat, 1, 3, F), generator=g, device=dev) - 0.5) * (5 * L)
    d_orig[n_prot:] = (wat_c + torch.randn((n_wat, 3, 3, 1), generator=g, device=dev) * 0.6).reshape(3 * n_wat, 3, F)
    del wat_c
    d_b = torch.full((3, F), L, dtype=torch.float32, device=dev)
    groups = torch.cat([torch.zeros(1, dtype=torch.int32, device=dev),
                        n_prot + 3 * torch.arange(n_wat + 1, dtype=torch.int32, device=dev)])
    csel = torch.arange(0, n_prot, dtype=torch.int32, device=dev)
    d_c = torch.empty_like(d_orig)
    kms, cms, moved = [], [], 0
    for it in range(6):
        d_c.copy_(d_orig)                      # the wrap is in place and idempotent: restore the unwrapped input
        wr.wrap_box_device(d_c, d_b, groups, csel)
        prep, main = _lib.get_timing(dev.index)
        if it:
            kms.append(main); cms.append(prep)
        else:
            moved = int((d_c != d_orig).sum().item())
    main, prep = float(np.mean(kms)), float(np.mean(cms))
    nb = N * 3 * F * 4 + moved * 8 + 3 * F * 8
    out["c6_wrap"] = dict(workload=f"C6: wrap_box, {N} atoms ({n_wat + 1} bonded groups) x {F} frames, centre = {n_prot} solute atoms",
                          atom_frames_per_s=N * F / ((main + prep) * 1e-3), centre_kernel_ms=prep, group_kernel_ms=main,
                          moved_fraction=moved / (N * 3 * F), kernel_gbs=nb / (main * 1e-3) / 1e9,
                          frac_of_peak=nb / (main * 1e-3) / 1e9 / peak,
                          whole_call_gbs=(nb + n_prot * 3 * F * 4) / ((main + prep) * 1e-3) / 1e9,
                          whole_call_frac_of_peak=(nb + n_prot * 3 * F * 4) / ((main + prep) * 1e-3) / 1e9 / peak)
    # C6b: the same system in a rhombic dodecahedron (K9b): every coordinate is centred and rewritten, the group translation
    # is the triclinic / compact / rectangular rule of wrap_triclinic_unitcell / wrap_compact_unitcell
    vec = torch.tensor([[L, 0, 0], [0, L, 0], [L / 2, L / 2, L * 2 ** 0.5 / 2]], dtype=torch.float64, device=dev)
    d_bv = vec[:, :, None].repeat(1, 1, F).contiguous()
    c6b = {}
    for cell in ("triclinic", "compact", "rectangular"):
        kms = []
        for it in range(4):
            d_c.copy_(d_orig)
            wr.wrap_triclinic_device(d_c, d_bv, groups, csel, None, cell)
            prep, main = _lib.get_timing(dev.index)
            if it:
                kms.append(prep + main)
        ms = float(np.mean(kms))
        nbt = 2 * N * 3 * F * 4 + n_prot * 3 * F * 4  # read + write every coordinate, the centre selection read once more
        c6b[cell] = dict(ms_per_call=ms, atom_frames_per_s=N * F / (ms * 1e-3), gbs=nbt / (ms * 1e-3) / 1e9,
                         frac_of_peak=nbt / (ms * 1e-3) / 1e9 / peak)
    out["c6b_wrap_triclinic"] = dict(workload=f"C6b: wrap in a rhombic dodecahedron, {N} atoms ({n_wat + 1} bonded groups) x {F} frames, "
                                              f"centre = {n_prot} solute atoms; unit cells triclinic / compact / rectangular", **c6b)
    del d_bv
    # C10: hydrogen bonds (K12) between the waters of the system: 2 x n_wat donor pairs x n_wat acceptors per frame, 64 frames
    from moleculekit_b200 import hbonds as hbm

    Fh = 64
    ow = n_prot + 3 * torch.arange(n_wat, dtype=torch.int32, device=dev)
    donors = torch.cat([torch.stack([ow, ow + 1], 1), torch.stack([ow, ow + 2], 1)]).contiguous()
    d_wr = d_orig[:, :, :Fh].contiguous()
    wr.wrap_box_device(d_wr, d_b[:, :Fh].contiguous(), groups, csel)
    selw = torch.ones(N, dtype=torch.int32, device=dev)
    resh = {}

    def run_hb():
        resh["r"] = hbm.calculate_device(d_wr, d_b[:, :Fh].contiguous(), donors, ow.contiguous(), selw, selw, 2.5, 120, True, False)

    ms = _time_cuda(run_hb, warm=1, steps=3)
    out["c10_hbonds"] = dict(workload=f"C10: hydrogen bonds, {Fh} frames x {2 * n_wat} donor pairs x {n_wat} acceptors, periodic, "
                                      "count + ordered fill", ms_per_call=ms, pair_tests_per_s=2.0 * Fh * 2 * n_wat * n_wat / (ms * 1e-3),
                             bonds_per_frame=float(resh["r"][1].shape[0]) / Fh)
    # C11: ring detectors (K13): 400 six-rings against themselves (pi-pi) and against 2000 cations (cation-pi), 1000 frames
    from moleculekit_b200 import ringpairs as rp

    nr, nc, Fr = 400, 2000, 1000
    Nr = 6 * nr + nc
    ctr = torch.rand((nr, 1, 3, 1), generator=g, device=dev) * 60 + torch.cumsum(torch.randn((nr, 1, 3, Fr), generator=g, device=dev) * 0.1, dim=3)
    ang = torch.arange(6, device=dev, dtype=torch.float32) * (3.14159265 / 3)
    u = torch.nn.functional.normalize(torch.randn((nr, 3), generator=g, device=dev), dim=1)
    v = torch.nn.functional.normalize(torch.linalg.cross(u, torch.randn((nr, 3), generator=g, device=dev)), dim=1)
    ring_xyz = ctr + 1.39 * (torch.cos(ang)[None, :, None, None] * u[:, None, :, None] + torch.sin(ang)[None, :, None, None] * v[:, None, :, None])
    d_rc = torch.empty((Nr, 3, Fr), dtype=torch.float32, device=dev)
    d_rc[:6 * nr] = ring_xyz.reshape(6 * nr, 3, Fr)
    d_rc[6 * nr:] = torch.rand((nc, 3, 1), generator=g, device=dev) * 60 + torch.cumsum(torch.randn((nc, 3, Fr), generator=g, device=dev) * 0.1, dim=2)
    d_rb = torch.full((3, Fr), 60.0, dtype=torch.float32, device=dev)
    r_atoms = torch.arange(6 * nr, dtype=torch.int32, device=dev)
    r_st = torch.arange(0, 6 * nr + 1, 6, dtype=torch.int32, device=dev)
    cat_idx = 6 * nr + torch.arange(nc, dtype=torch.int32, device=dev)
    resr = {}
    ms_pp = _time_cuda(lambda: resr.__setitem__("pp", rp.calculate_device(rp.PIPI, d_rc, d_rb, r_atoms, r_st, r_st, 4.4, 30.0, 5.5, 60.0)), warm=1, steps=3)
    ms_cp = _time_cuda(lambda: resr.__setitem__("cp", rp.calculate_device(rp.CATIONPI, d_rc, d_rb, r_atoms, r_st, cat_idx, 5.0, 60.0)), warm=1, steps=3)
    out["c11_ring_detectors"] = dict(
        workload=f"C11: {Fr} frames, {nr} rings: pi-pi against themselves and cation-pi against {nc} cations, periodic, count + fill",
        pipi_ms=ms_pp, pipi_pair_tests_per_s=Fr * nr * nr / (ms_pp * 1e-3), pipi_hits_per_frame=float(resr["pp"][1].shape[0]) / Fr,
        cationpi_ms=ms_cp, cationpi_pair_tests_per_s=Fr * nr * nc / (ms_cp * 1e-3), cationpi_hits_per_frame=float(resr["cp"][1].shape[0]) / Fr)
    del d_rc, ring_xyz, ctr
    del d_c, d_orig, d_b, d_wr
    # C7: `within 5 of <solute>` (K10) on one frame of a 96k-atom solvated system (the reference: 96k x 5.5k brute force)
    from moleculekit_b200 import atomselect_utils as asel

    N, n2 = 96000, 5500
    xyz = torch.rand((N, 3), generator=g, device=dev) * 99.5
    xyz[:n2] = torch.randn((n2, 3), generator=g, device=dev) * 11 + 50
    src = torch.arange(n2, dtype=torch.int32, device=dev)
    res = {}

    def run_within():
        res["m"] = asel.within_distance_device(xyz, 5.0, src)

    ms = _time_cuda(run_within, warm=2, steps=10)
    out["c7_within"] = dict(workload=f"C7: within 5 A of {n2} source atoms, {N} query atoms (cell list; reference = brute force)",
                            ms_per_call=ms, selected=int(res["m"].sum().item()), pair_tests_avoided=float(N) * n2,
                            equivalent_pair_tests_per_s=float(N) * n2 / (ms * 1e-3))
    # C4d: MetricShell radial histograms (K8): 500 centres x 4500 partners, 4 shells, 1000 frames of the C4b trajectory
    edges = torch.tensor([0.0, 3.0, 6.0, 9.0, 12.0], dtype=torch.float64, device=dev)
    c4 = start + np.cumsum(rng.normal(0, 0.3, size=(n1c + n2c, 3, Fsh)).astype(np.float32), axis=2)
    d_c4 = torch.from_numpy(np.ascontiguousarray(c4)).to(dev); d_b4 = torch.from_numpy(np.ascontiguousarray(box[:, :Fsh])).to(dev)
    ms = _time_cuda(lambda: du.shell_counts_device(d_c4, d_b4, s1, s2, ch, False, True, edges), warm=1, steps=3)
    out["c4d_metricshell"] = dict(workload=f"C4d: MetricShell, {Fsh} frames x {n1c} centres x {n2c} partners, 4 shells, periodic",
                                  ms_per_step=ms, pair_tests_per_s=Fsh * n1c * n2c / (ms * 1e-3))
    del d_c4, d_b4
    # C1: one getVoxelDescriptors call, host arrays in and out (latency of the drop-in API on a 3PTB-sized molecule)
    import time as _time

    from moleculekit_b200.molecule_lite import MolLite

    w1 = workloads.protein_pockets(B=1, n_atoms=1639, box=60.0, radius=17.0, seed=5)
    mol1 = MolLite(w1["coords"][0])
    vd.getVoxelDescriptors(mol1, userchannels=w1["sigmas"][0], buffer=8, voxelsize=1)
    torch.cuda.synchronize(dev)
    t0 = _time.perf_counter()
    for _ in range(5):
        f1, c1, n1v = vd.getVoxelDescriptors(mol1, userchannels=w1["sigmas"][0], buffer=8, voxelsize=1)
    dt = (_time.perf_counter() - t0) / 5
    out["c1_single_call"] = dict(workload=f"C1-like: one getVoxelDescriptors call, 1639 atoms, grid {list(map(int, n1v))}, host float64 in/out",
                                 ms_per_call=dt * 1e3, voxel_channels_per_s=f1.size / dt)
    # C7b: bond perception (K7) on a 100k-atom solvated system
    from moleculekit_b200.bondguesser import bond_grid_search

    nb_at = 100_000
    xyzb = (rng.uniform(0, 100, size=(nb_at // 3, 1, 3)) + rng.normal(0, 0.6, size=(nb_at // 3, 3, 3))).reshape(-1, 3).astype(np.float32)
    radb = np.tile(np.array([1.52, 1.0, 1.0], np.float32), nb_at // 3)
    ishb = (radb == 1.0).astype(np.uint32)
    bond_grid_search(xyzb, 1.9 * 1.2, ishb, radb)
    t0 = _time.perf_counter()
    bonds = bond_grid_search(xyzb, 1.9 * 1.2, ishb, radb)
    dt = _time.perf_counter() - t0
    out["c7b_bond_search"] = dict(workload=f"K7: bond_grid_search, {len(xyzb)} atoms (host arrays in, sorted pairs out)", ms_per_call=dt * 1e3,
                                  bonds=int(len(bonds)))
    # C8: XTC decode on the device (K11): the 3 frames of tests/golden/xtc/real3.xtc (4507 atoms, re-encoded frames of the
    # reference's test trajectory) repeated to a 3000-frame file
    from moleculekit_b200 import xtc as px

    raw3 = open(os.path.join(ROOT, "tests", "golden", "xtc", "real3.xtc"), "rb").read()
    raw = raw3 * 1000
    idx = px.index_xtc(raw)
    d_bytes = torch.frombuffer(bytearray(raw), dtype=torch.uint8).to(dev)
    nat, Fx = idx["natoms"], len(idx["frames"])
    d_xyz = torch.empty((nat, 3, Fx), dtype=torch.float32, device=dev)
    ms = _time_cuda(lambda: px.decode_xtc_device(d_bytes, idx["frames"], nat, scale=10.0, out=d_xyz), warm=1, steps=3)
    _, kms = _lib.get_timing(dev.index)
    out["c8_xtc_decode"] = dict(workload=f"C8: XTC decode, {Fx} frames x {nat} atoms ({len(raw) / 1e6:.0f} MB compressed -> "
                                         f"{nat * 3 * Fx * 4 / 1e6:.0f} MB frame-minor float32 on the device)",
                                ms_per_call=ms, kernel_ms=kms, frames_per_s=Fx / (ms * 1e-3),
                                atom_frames_per_s=nat * Fx / (ms * 1e-3), output_gbs=nat * 3 * Fx * 4 / (kms * 1e-3) / 1e9)
    # C9: the trajectory pipeline end to end without a host round trip: XTC bytes in pinned host memory -> H2D -> decode
    # (K11) -> wrap around the first 100 atoms (K9, 3-atom groups) -> fused periodic contact map 256 x 1024 (K3) -> per-frame
    # contact counts -> D2H of the counts
    pinned = torch.frombuffer(bytearray(raw) + bytearray(4), dtype=torch.uint8).pin_memory()
    groups = torch.arange(0, nat + 1, 3, dtype=torch.int32, device=dev)
    if int(groups[-1]) != nat:
        groups = torch.cat([groups, torch.tensor([nat], dtype=torch.int32, device=dev)])
    csel = torch.arange(0, 100, dtype=torch.int32, device=dev)
    bx9 = torch.from_numpy(np.ascontiguousarray(idx["box"][[0, 1, 2], [0, 1, 2], :] * np.float32(10.0))).to(dev)
    s1 = torch.arange(0, 256, dtype=torch.int32, device=dev); s2 = torch.arange(256, 1280, dtype=torch.int32, device=dev)
    ch = torch.ones(nat, dtype=torch.int32, device=dev); ch[256:] = 2
    cmap = torch.empty((Fx, 256 * 1024), dtype=torch.uint8, device=dev)
    res = {}

    def pipeline():
        d_b = pinned.to(dev, non_blocking=True)
        xyz = px.decode_xtc_device(d_b, idx["frames"], nat, scale=10.0, out=d_xyz)
        wr.wrap_box_device(xyz, bx9, groups, csel)
        c = du.dist_trajectory_device(xyz, bx9, s1, s2, ch, False, True, metric="contacts", threshold=8.0, out=cmap)
        res["counts"] = c.sum(dim=1, dtype=torch.int32).cpu()

    ms = _time_cuda(pipeline, warm=1, steps=3)
    out["c9_trajectory_pipeline"] = dict(
        workload=f"C9: XTC file ({len(raw) / 1e6:.0f} MB, pinned host) -> H2D -> decode -> wrap -> 256x1024 periodic contact map "
                 f"-> per-frame counts -> D2H; {Fx} frames x {nat} atoms, nothing but the file and the counts crosses PCIe",
        ms_per_call=ms, frames_per_s=Fx / (ms * 1e-3), mean_contacts_per_frame=float(res["counts"].float().mean()))
    return out


# ----------------------------------------------------------------------------------------------------- GPU arm
def bind_to_gpu_numa(index: int):
    from moleculekit_b200 import sharding

    return sharding.bind_to_gpu_numa(index)


def scaling_section(a, dev, world, rank, peak):
    """What SURVEY 8(e) / BASELINE.json's north star describe for N GPUs, measured at every N (so the driver's N=1,2,4,8
    runs give STRONG scaling): (1) the ONE 256-pocket batch of config 3 sharded over the ranks, shards resident;
    (2) the NCCL all_gather that assembles the (256 x 64^3 x 8) tensor on every rank when the caller asks for it;
    (3) the same batch end to end (pinned host in, pinned host out, each rank its slice); (4) config 4: the 10k-frame
    periodic contact map with frames sharded over the ranks, device resident and through MetricDistance.project with
    host arrays.  Times are CUDA events / wall clock per rank, MAX over ranks."""
    import torch
    import torch.distributed as dist

    from moleculekit_b200 import distance_utils as du, sharding, workloads
    from moleculekit_b200.molecule_lite import MolLite
    from moleculekit_b200.projections.metricdistance import MetricDistance
    from moleculekit_b200.tools import voxeldescriptors as vd

    def maxr(x):
        if world == 1:
            return float(x)
        t = torch.tensor([x], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def barrier():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()

    def timed(fn, steps=5, warm=2):
        for _ in range(warm):
            fn()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        torch.cuda.synchronize(dev)
        return maxr(e0.elapsed_time(e1) / steps)

    out = {}
    # ---- (1) strong scaling of the one C3 batch
    B = a.batch or 256
    w = workloads.protein_pockets(B=B, seed=1000)
    off = sharding.partition(B, world)
    b0, b1 = int(off[rank]), int(off[rank + 1])
    vb = vd.VoxelBatch(w["coords"][b0:b1], w["sigmas"][b0:b1], boxsize=w["boxsize"], centers=w["centers"][b0:b1], voxelsize=1.0)
    d_c, d_s = vb.to_device(dev)
    shard = torch.empty((vb.total_voxels, 8), dtype=torch.float32, device=dev)
    ms = timed(lambda: vb.run(d_c, d_s, shard), steps=10, warm=3)
    n_vc = B * 64 ** 3 * 8
    out["c3_strong"] = dict(workload=f"C3: ONE batch of {B} pockets sharded over {world} GPU(s) ({b1 - b0} on rank 0), shards resident",
                            ms_per_step=ms, voxel_channels_per_s=n_vc / (ms * 1e-3))
    # ---- (2) NCCL gather of the shards (only when the caller wants the assembled tensor on every rank)
    if world > 1 and B % world == 0:
        full = torch.empty((B * 64 ** 3, 8), dtype=torch.float32, device=dev)
        ms_g = timed(lambda: dist.all_gather_into_tensor(full, shard), steps=5, warm=2)
        nbytes = full.numel() * 4
        out["c3_gather"] = dict(collective="ncclAllGather (all_gather_into_tensor) of the per-rank grids", ms=ms_g, bytes_assembled=nbytes,
                                algbw_gbs=nbytes / (ms_g * 1e-3) / 1e9, busbw_gbs=nbytes * (world - 1) / world / (ms_g * 1e-3) / 1e9,
                                gather_over_compute=ms_g / ms)
        del full
    # ---- (3) the same batch end to end: every rank uploads its pockets and receives its slice in pinned host memory
    h_c = vd.pinned_array(vb.coords.shape, np.float32); h_c[:] = vb.coords
    h_s = vd.pinned_array(vb.sigmas.shape, np.float64); h_s[:] = vb.sigmas
    h_o = vd.pinned_array((vb.total_voxels, 8), np.float32)
    kw = dict(boxsize=w["boxsize"], centers=w["centers"][b0:b1], voxelsize=1.0, atom_offsets=vb.atom_offsets, device=dev, out=h_o)
    for _ in range(2):
        vd.getVoxelDescriptorsBatch(h_c, h_s, **kw)
    barrier()
    t0 = time.perf_counter()
    for _ in range(5):
        vd.getVoxelDescriptorsBatch(h_c, h_s, **kw)
    torch.cuda.synchronize(dev)
    dt = maxr((time.perf_counter() - t0) / 5)
    out["c3_strong_e2e"] = dict(workload="same batch, pinned host in / out per rank (H2D + kernels + D2H in the timed region)",
                                ms_per_step=dt * 1e3, voxel_channels_per_s=n_vc / dt,
                                d2h_bytes_per_rank=int(vb.total_voxels * 32), h2d_bytes_per_rank=int(h_c.nbytes + h_s.nbytes))
    del h_o, shard, d_c, d_s
    # ---- (4) config 4: 10k frames x (256 x 1024) periodic contacts <= 12 A, frames sharded
    F, n1, n2, nat = (2000 if a.batch else 10000), 256, 1024, 5000
    foff = sharding.partition(F, world)
    f0, f1 = int(foff[rank]), int(foff[rank + 1])
    rng = np.random.default_rng(7)
    L = 36.84
    box = np.repeat((L * (1 + 0.002 * rng.normal(size=F))).astype(np.float32)[None, :], 3, axis=0)[:, f0:f1].copy()
    # selected atoms: random walk (every rank draws the whole walk and keeps its frames); the other 3720 atoms ("water")
    # are never read by the projection -- they only have to be there, as in a real solvated trajectory
    sel = rng.uniform(0, L, size=(n1 + n2, 3, 1)).astype(np.float32) + \
        np.cumsum(rng.normal(0, 0.3, size=(n1 + n2, 3, F)).astype(np.float32), axis=2)
    coords = vd.pinned_array((nat, 3, f1 - f0), np.float32)
    coords[: n1 + n2] = sel[:, :, f0:f1]
    coords[n1 + n2:] = rng.random((nat - n1 - n2, 3, f1 - f0), dtype=np.float32) * L
    del sel
    chain = np.array(["A"] * n1 + ["B"] * n2 + ["W"] * (nat - n1 - n2), dtype=object)
    m1 = np.zeros(nat, bool); m1[:n1] = True
    m2 = np.zeros(nat, bool); m2[n1:n1 + n2] = True
    mol = MolLite(coords, box=box, chain=chain)
    d_c = torch.from_numpy(np.ascontiguousarray(coords[: n1 + n2])).to(dev); d_b = torch.from_numpy(box).to(dev)
    s1 = torch.arange(0, n1, dtype=torch.int32, device=dev); s2 = torch.arange(n1, n1 + n2, dtype=torch.int32, device=dev)
    ch = torch.ones(n1 + n2, dtype=torch.int32, device=dev); ch[n1:] = 2
    o = torch.empty((f1 - f0, n1 * n2), dtype=torch.uint8, device=dev)
    ms4 = timed(lambda: du.dist_trajectory_device(d_c, d_b, s1, s2, ch, False, True, metric="contacts", threshold=12.0, out=o), steps=5, warm=2)
    out["c4_frames_sharded"] = dict(workload=f"C4: {F} frames x {n1}x{n2} periodic contacts <= 12 A, frames sharded over {world} GPU(s), resident",
                                    ms_per_step=ms4, pair_frames_per_s=F * n1 * n2 / (ms4 * 1e-3))
    del o, d_c
    proj = MetricDistance(m1, m2, periodic="selections", metric="contacts", threshold=12)
    proj.device = dev
    for _ in range(2):
        res = proj.project(mol)
    barrier()
    t0 = time.perf_counter()
    for _ in range(3):
        res = proj.project(mol)
    dt4 = maxr((time.perf_counter() - t0) / 3)
    out["c4_project_e2e"] = dict(workload=f"MetricDistance.project (host (N,3,F) float32 in, host (F,P) bool out), {nat} atoms, frames sharded over {world} GPU(s)",
                                 ms_per_step=dt4 * 1e3, pair_frames_per_s=F * n1 * n2 / dt4, result_shape=list(res.shape),
                                 d2h_bytes_per_rank=int(res.size), h2d_bytes_per_rank=int((n1 + n2) * 3 * (f1 - f0) * 4))
    return out


DUMP_ROWS = 1 << 20  # sampled grid rows: 1M rows x 8 channels x 4 B = 32 MB, the whole dump stays under 64 MB


def dump_outputs(path, batch, out):
    """Write what one step of the timed path returns, the float32 grid `out` (total_voxels, C), as .npy files under
    `path`.  The grid of the flagship workload is GBs, so the files hold the rows at a fixed seeded sample of row indices,
    in index order (occupancy_sample.npy, float32, (min(total_voxels, DUMP_ROWS), C)), and the float64 sum of every grid
    and channel over the whole grid (occupancy_sum.npy, (B, C)).  The workloads are seeded, so the same arguments give
    the same inputs."""
    import torch

    os.makedirs(path, exist_ok=True)
    n = batch.total_voxels
    rows = np.sort(np.random.default_rng(0).choice(n, size=min(n, DUMP_ROWS), replace=False))
    np.save(os.path.join(path, "occupancy_sample.npy"), out[torch.from_numpy(rows).to(out.device)].cpu().numpy())
    sums = np.zeros((batch.B, batch.C))
    for b in range(batch.B):
        sums[b] = out[int(batch.out_offsets[b]):int(batch.out_offsets[b + 1])].sum(dim=0, dtype=torch.float64).cpu().numpy()
    np.save(os.path.join(path, "occupancy_sum.npy"), sums)


def run_ours(a):
    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    numa = bind_to_gpu_numa(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    from moleculekit_b200 import _lib, workloads
    from moleculekit_b200.tools import voxeldescriptors as vd

    w = make_workload(a.workload, a.batch, rank)
    batch = vd.VoxelBatch(w["coords"], w["sigmas"], boxsize=w["boxsize"], centers=w["centers"], voxelsize=w["voxelsize"])
    n_vc = batch.total_voxels * batch.C
    n_atoms = batch.coords.shape[0]
    d_coords, d_sig = batch.to_device(dev)
    out = torch.empty((batch.total_voxels, batch.C), dtype=torch.float32, device=dev)

    def barrier():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    # ---- device-resident timing
    _lib.set_timing(True, local)
    for _ in range(max(a.warmup, 3)):
        batch.run(d_coords, d_sig, out)
    barrier()
    clocks = ClockSampler(local) if rank == 0 else None
    time.sleep(0.25 if rank == 0 else 0.0)
    barrier()
    l0 = _lib.launch_count(local)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    fill_ms, prep_ms = [], []
    t_wall0 = time.perf_counter()
    ev0.record()
    for _ in range(a.steps):
        batch.run(d_coords, d_sig, out)
        # reading the library's per-kernel events would synchronise; they are read after the loop for the LAST
        # step and, below, in a second pass for every step
    ev1.record()
    barrier()
    t_wall1 = time.perf_counter()
    launches = _lib.launch_count(local) - l0
    ms_total = ev0.elapsed_time(ev1)
    if a.dump_outputs and rank == 0:
        dump_outputs(a.dump_outputs, batch, out)
    # per-kernel durations (one synchronising read per step, outside the aggregate timing above)
    for _ in range(a.steps):
        batch.run(d_coords, d_sig, out)
        p, m = _lib.get_timing(local)
        prep_ms.append(p); fill_ms.append(m)
    t_wall2 = time.perf_counter()
    clk = clocks.stop(t_wall0, t_wall2) if clocks else None
    ms_step = ms_total / a.steps
    if world > 1:
        t = torch.tensor([ms_step], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_step = float(t.item())
    value = world * n_vc / (ms_step * 1e-3)

    # ---- end to end through the public host API (pinned host in, pinned host out)
    e2e = None
    if not a.no_e2e:
        h_coords = vd.pinned_array(batch.coords.shape, np.float32); h_coords[:] = batch.coords
        h_sig = vd.pinned_array(batch.sigmas.shape, np.float64); h_sig[:] = batch.sigmas
        h_out = vd.pinned_array((batch.total_voxels, batch.C), np.float32)
        kw = dict(boxsize=w["boxsize"], centers=w["centers"], voxelsize=w["voxelsize"], atom_offsets=batch.atom_offsets,
                  device=dev)
        n_e2e = max(3, min(a.steps, 10))

        def e2e_time(n, **extra):
            for _ in range(2):
                vd.getVoxelDescriptorsBatch(h_coords, h_sig, **kw, **extra)
            barrier()
            t0 = time.perf_counter()
            for _ in range(n):
                vd.getVoxelDescriptorsBatch(h_coords, h_sig, **kw, **extra)
            torch.cuda.synchronize(dev)
            dt = (time.perf_counter() - t0) / n
            if world > 1:
                t = torch.tensor([dt], device=dev, dtype=torch.float64)
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                dt = float(t.item())
            return dt

        # the call a user makes: host arrays in, the dense float32 (sum M, 8) host array out.  Default transfer ("auto"):
        # only the 4x4x8 blocks with an atom in reach cross PCIe -- stored by the fill kernel straight into the page-locked
        # result while host threads zero the other blocks (identical bytes to the dense copy)
        dt = e2e_time(n_e2e, out=h_out)
        d2h = int(vd.LAST_TRANSFER.get("d2h_bytes", h_out.nbytes))
        mode = vd.LAST_TRANSFER.get("mode")
        e2e = dict(value=world * n_vc / dt, unit=UNIT, h2d_bytes_per_step=int(h_coords.nbytes + h_sig.nbytes),
                   d2h_bytes_per_step=d2h, ms_per_step=dt * 1e3, steps=n_e2e, transfer=mode,
                   host_bytes_delivered_per_step=int(h_out.nbytes),
                   api="moleculekit_b200.tools.voxeldescriptors.getVoxelDescriptorsBatch(out=pinned float32)")
        if rank == 0 or world > 1:
            dt_dense = e2e_time(3, out=h_out, transfer="dense")
            e2e["dense_transfer"] = dict(ms_per_step=dt_dense * 1e3, value=world * n_vc / dt_dense, d2h_bytes_per_step=int(h_out.nbytes))
            if mode == "direct":  # the staged variant of the same idea: 4 KB block records + host expansion
                dt_c = e2e_time(3, out=h_out, transfer="compact")
                e2e["compact_transfer"] = dict(ms_per_step=dt_c * 1e3, value=world * n_vc / dt_c,
                                               d2h_bytes_per_step=int(vd.LAST_TRANSFER.get("d2h_bytes", 0)))
        if world == 1:  # the reference-typed result: a list of float64 (M, 8) arrays (voxeldescriptors.py:531)
            dt64 = e2e_time(2)
            e2e["float64_lists"] = dict(ms_per_step=dt64 * 1e3, value=n_vc / dt64,
                                        note="dtype=float64 default of the drop-in API; upcast inside the threaded expansion")
        del h_out

    # ---- strong scaling of the one batch, NCCL gather, config 4 frames-sharded (every rank takes part)
    scaling = None
    if not a.no_scaling:
        try:
            peak_s = HBM_FALLBACK_GBS
            del out
            torch.cuda.empty_cache()
            scaling = scaling_section(a, dev, world, rank, peak_s)
            scaling["numa"] = numa
        except Exception as e:  # never let a side measurement break the headline line
            scaling = {"error": repr(e)}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peaks, peak_src = None, "fallback"
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            peaks = json.load(f)
        peak, peak_src = float(peaks["hbm_gbs"]), "measured"
    except Exception:
        peak = HBM_FALLBACK_GBS
    alg_bytes = workloads.occupancy_algorithmic_bytes(batch.total_voxels, n_atoms, batch.C)
    fill_mean = float(np.mean(fill_ms))
    achieved = alg_bytes / (fill_mean * 1e-3) / 1e9
    # DRAM bytes of the fill kernel: measured in THIS run when bench.py is started under `ncu` by
    # profiles/scripts/traffic.sh (it writes the sum next to the report); otherwise taken from the newest committed
    # capture of the same kernel and workload and labelled as such -- never silently attached to another kernel
    traffic, traffic_source = None, None
    kname = _lib.last_fill_kernel(local) if hasattr(_lib, "last_fill_kernel") else "occ_fill_runs_kernel"
    try:
        if a.workload == "c3" and not a.batch:
            fn = os.path.join(ROOT, "profiles", "r02_fill_v10_metrics.txt")  # capture of the shipped (v10) kernel
            tr, kern_ok = 0.0, False
            for ln in open(fn):
                if ln.startswith("# kernel:"):
                    kern_ok = kname.split("<")[0] in ln
                f = ln.split()
                if f and f[0] in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
                    tr += float(f[1]) * {"byte": 1, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}[f[2]]
            if kern_ok and tr:
                traffic, traffic_source = tr, "committed ncu --set full capture of the same kernel and workload (profiles/r02_fill_v10_metrics.txt)"
    except Exception:
        traffic = None
    roofline = dict(bound="hbm", kernel=kname, achieved=achieved, peak=peak, unit="GB/s",
                    frac=achieved / peak, traffic=traffic, traffic_source=traffic_source,
                    peak_source=f"{peak_src} (MEASURED_PEAKS.json hbm_gbs)",
                    algorithmic_bytes_per_launch=int(alg_bytes), kernel_ms_mean=fill_mean,
                    kernel_ms_min=float(np.min(fill_ms)), prep_ms_mean=float(np.mean(prep_ms)),
                    kernel_share_of_step=fill_mean / ms_step)
    extra = None
    if world == 1 and not a.no_extra:
        try:
            extra = extra_workloads(dev, peak)
        except Exception as e:  # never let a side measurement break the headline line
            extra = {"error": repr(e)}
    cpu = None
    if not a.no_cpu and world == 1:
        arm = CpuArm(w, step_seconds=6.0)  # ~10-30 s of CPU work in total (pilot + two bounded steps)
        arm.step()
        v, _ = arm.step()
        arm.close()
        cpu = arm.describe(v)
        if isinstance(extra, dict) and "error" not in extra:
            try:
                extra["cpu_reference_next_rows"] = cpu_next_rows(extra)
            except Exception as e:
                extra["cpu_reference_next_rows"] = {"error": repr(e)}
    line = dict(metric=METRIC, value=value, unit=UNIT, n_gpus=world, steps=a.steps, warmup=max(a.warmup, 3),
                ms_per_step=ms_step, higher_is_better=True, scaling="weak", vs_baseline=None, dtype="f32",
                data="synthetic",
                config=dict(workload=w["name"] + " per GPU", items_per_gpu=batch.B, atoms_per_gpu=int(n_atoms),
                            voxel_channels_per_gpu=int(n_vc),
                            l2="no flush needed: each step streams %.2f GB of grid output, >> 126 MB L2" % (n_vc * 4 / 1e9),
                            parallelism=f"batch sharded over {world} GPU(s), no collective"),
                roofline=roofline, cpu_baseline=cpu, e2e=e2e, gpu_launches=int(launches), clocks=clk, scaling_detail=scaling, extra=extra)
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    args = parse()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)
