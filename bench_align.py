"""Benchmark of K14 (superposition: Molecule.align / molRMSD / MetricRmsd) on a seeded solvated-protein trajectory.

The system is 40 000 atoms (4 000 "protein", the rest 3-atom waters) over 2 000 frames, 960 MB of float32 coordinates,
far above the 126 MB L2.  Every frame is a random rigid motion of one base structure plus 0.5 A of Gaussian noise; the fit
and RMSD selection is 300 CA-like protein atoms.  Printed as one JSON line:

  - kernel times of fit, apply and the fused RMSD (CUDA events, one event pair per repeat, L2 overwritten before each
    repeat so that the 7 MB fit / RMSD working set is read from HBM), algorithmic bytes (apply 24*N*F, fit 12*n_fit*F,
    fused RMSD 12*|fit u rmsd|*F) and their share of the repository's measured copy bandwidth (6478.6 GB/s);
  - a single-frame case (1 M atoms, F = 1, a 100 000-atom fit selection);
  - MetricRmsd.project end to end from host arrays, with and without pbc;
  - the float32 numpy restatement of the reference on the first frames, as the CPU baseline;
  - the GPU name and power limit, read in the same run.

`python bench_align.py [--frames F] [--reps R]`.  Writes nothing.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

COPY_GBPS = 6478.6  # measured device-to-device copy bandwidth the repository's roofline uses


def _gpu_info():
    import torch

    info = {"gpu": torch.cuda.get_device_name(0)}
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30)
        info["power_limit"] = r.stdout.strip() or None
    except Exception as e:  # pragma: no cover - the field says why it is missing
        info["power_limit"] = f"unavailable: {e}"
    return info


def _system(n_atoms, n_protein, F, seed, dev):
    """(N, 3, F) float32 CUDA trajectory, base structure, protein / CA masks, bonds and box."""
    import torch

    rng = np.random.default_rng(seed)
    n_wat = (n_atoms - n_protein) // 3
    N = n_protein + 3 * n_wat
    edge = float(np.cbrt(N / 0.1))  # ~0.1 atoms per cubic Angstrom
    prot = np.cumsum(rng.normal(0, 1.5, size=(n_protein, 3)), axis=0)
    prot = (prot - prot.mean(0)) * (12.0 / prot.std())
    wat_o = rng.uniform(-edge / 2, edge / 2, size=(n_wat, 1, 3))
    wat = (wat_o + rng.normal(0, 0.6, size=(n_wat, 3, 3))).reshape(-1, 3)
    base = np.concatenate([prot, wat])
    rot = np.stack([_rotation(rng) for _ in range(F)])
    shift = rng.uniform(-10, 10, size=(F, 3))
    d_base = torch.from_numpy(base).to(dev)
    traj = torch.empty((N, 3, F), dtype=torch.float32, device=dev)
    g = torch.Generator(device=dev)
    g.manual_seed(seed)
    for f0 in range(0, F, 100):
        f1 = min(F, f0 + 100)
        R = torch.from_numpy(rot[f0:f1]).to(dev)
        t = torch.from_numpy(shift[f0:f1]).to(dev)
        moved = torch.einsum("nd,fed->nef", d_base, R) + t.T[None, :, :]
        noise = torch.randn((N, 3, f1 - f0), generator=g, device=dev, dtype=torch.float64) * 0.5
        traj[:, :, f0:f1] = (moved + noise).float()
    protein = np.zeros(N, bool)
    protein[:n_protein] = True
    ca = np.zeros(N, bool)
    ca[np.linspace(0, n_protein - 1, 300).astype(int)] = True
    chain = np.stack([np.arange(n_protein - 1), np.arange(1, n_protein)], 1)
    o = n_protein + 3 * np.arange(n_wat)
    bonds = np.concatenate([chain, np.stack([o, o + 1], 1), np.stack([o, o + 2], 1)]).astype(np.uint32)
    return traj, protein, ca, bonds, edge


def _rotation(rng):
    q, r = np.linalg.qr(rng.normal(size=(3, 3)))
    q = q * np.sign(np.diag(r))
    if np.linalg.det(q) < 0:
        q[:, 0] = -q[:, 0]
    return q


def _time_kernel(fn, reps, flush):
    """median and mean ms of fn over `reps` repeats, each between its own pair of CUDA events, L2 overwritten before"""
    import torch

    fn()
    torch.cuda.synchronize()
    times = []
    for _ in range(reps):
        flush.zero_()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        times.append(a.elapsed_time(b))
    return statistics.median(times), statistics.fmean(times)


def _roof(name, ms, nbytes):
    return {f"{name}_ms": round(ms, 4), f"{name}_bytes": int(nbytes),
            f"{name}_GBps": round(nbytes / ms / 1e6, 1), f"{name}_copy_bw_share": round(nbytes / ms / 1e6 / COPY_GBPS, 3)}


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--atoms", type=int, default=40000)
    ap.add_argument("--protein", type=int, default=4000)
    ap.add_argument("--frames", type=int, default=2000)
    ap.add_argument("--reps", type=int, default=30)
    ap.add_argument("--single-atoms", type=int, default=1_000_000)
    ap.add_argument("--cpu-frames", type=int, default=20)
    ap.add_argument("--e2e-reps", type=int, default=3)
    ap.add_argument("--seed", type=int, default=7)
    args = ap.parse_args(argv)

    import torch

    if not torch.cuda.is_available():
        raise SystemExit("bench_align.py needs a CUDA device")
    import align_ref
    from moleculekit_b200 import align as al
    from moleculekit_b200.molecule_lite import MolLite
    from moleculekit_b200.projections.metricrmsd import MetricRmsd

    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    res = {"bench": "k14_align", **_gpu_info()}
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # twice the L2

    traj, protein, ca, bonds, edge = _system(args.atoms, args.protein, args.frames, args.seed, dev)
    N, _, F = traj.shape
    sel = np.where(ca)[0]
    res.update({"n_atoms": N, "n_frames": F, "n_fit": int(sel.size), "n_rmsd": int(sel.size),
                "traj_MB": round(traj.numel() * 4 / 1e6, 1)})
    frames = torch.arange(F, device=dev)
    dsel = al.sel_tensor(sel, dev)
    ref = traj[sel][:, :, :1].contiguous()
    xf = al.align_fit_device(traj, frames, dsel, ref)

    ms, _ = _time_kernel(lambda: al.align_fit_device(traj, frames, dsel, ref), args.reps, flush)
    res.update(_roof("fit", ms, 12 * sel.size * F))
    ms, _ = _time_kernel(lambda: al.rmsd_device(traj, frames, dsel, ref, xf), args.reps, flush)
    res.update(_roof("rmsd_fused", ms, 12 * sel.size * F))
    work = traj.clone()
    ms, _ = _time_kernel(lambda: al.align_apply_device(work, frames, xf), args.reps, flush)
    res.update(_roof("apply", ms, 24 * N * F))
    del work

    # single frame, many atoms: parallelism over atoms
    rng = np.random.default_rng(args.seed + 1)
    one = torch.from_numpy(rng.uniform(-200, 200, size=(args.single_atoms, 3, 1)).astype(np.float32)).to(dev)
    sel1 = np.sort(rng.choice(args.single_atoms, args.single_atoms // 10, replace=False))
    dsel1 = al.sel_tensor(sel1, dev)
    ref1 = (one[sel1] * 0.5 + 3.0).contiguous()
    f1 = torch.zeros(1, dtype=torch.int64, device=dev)
    xf1 = al.align_fit_device(one, f1, dsel1, ref1)
    res["single_n_atoms"], res["single_n_fit"] = args.single_atoms, int(sel1.size)
    ms, _ = _time_kernel(lambda: al.align_fit_device(one, f1, dsel1, ref1), args.reps, flush)
    res.update(_roof("single_fit", ms, 12 * sel1.size))
    ms, _ = _time_kernel(lambda: al.align_apply_device(one, f1, xf1), args.reps, flush)
    res.update(_roof("single_apply", ms, 24 * args.single_atoms))

    # MetricRmsd.project from host arrays
    host = traj.cpu().numpy()
    box = np.full((3, F), edge, np.float32)
    mol = MolLite(host, box=box, bonds=bonds, named_selections={"protein": protein, "ca": ca})
    refmol = MolLite(host[:, :, :1].copy(), named_selections={"protein": protein, "ca": ca})
    for pbc in (False, True):
        m = MetricRmsd(refmol, "ca", pbc=pbc)
        out = m.project(mol)
        times = []
        for _ in range(args.e2e_reps):
            t0 = time.perf_counter()
            out = m.project(mol)  # ends in a device-to-host copy: synchronised
            times.append((time.perf_counter() - t0) * 1e3)
        res[f"metricrmsd_pbc_{str(pbc).lower()}_ms"] = round(statistics.median(times), 2)
        if not pbc:
            rmsd_nopbc = out
    res["metricrmsd_mean_rmsd_A"] = round(float(np.mean(rmsd_nopbc)), 4)

    # CPU baseline: the float32 numpy restatement of the reference, first cpu_frames frames, whole trajectory per frame
    nf = min(args.cpu_frames, F)
    sub = np.ascontiguousarray(host[:, :, :nf])
    t0 = time.perf_counter()
    cpu = align_ref.pp_align(sub, sub, sel, sel, range(nf), 0, False, dtype=np.float32)
    cpu_s = time.perf_counter() - t0
    res["cpu_baseline"] = {"what": "float32 numpy restatement of _pp_align, all atoms moved", "frames": nf,
                           "ms_per_frame": round(cpu_s * 1e3 / nf, 3),
                           "extrapolated_ms_all_frames": round(cpu_s * 1e3 / nf * F, 1)}
    gpu = al.align_apply_device(traj[:, :, :nf].contiguous(), torch.arange(nf, device=dev), xf[:nf]).cpu().numpy()
    res["gpu_vs_cpu_float32_max_abs_A"] = float(np.max(np.abs(gpu.astype(np.float64) - cpu)))
    print(json.dumps(res), flush=True)
    return res


if __name__ == "__main__":
    main()
