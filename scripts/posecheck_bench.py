"""Throughput of the pose checks (``posecheck.check_poses``) on the virtual-screening shape of BASELINE.json configs[4]:
one synthetic 100-residue pocket with 5 flexible residues, ligands from ``inputs.with_ligand`` whose sizes follow the
PDBBind test-set law, 10 randomized poses each (random rotation about the centroid, 2 A translation, side chains as in
the input), references = the input ligands and pocket (ligands with more automorphisms than the default cap get no
ligand reference and are screened for clashes only; the JSON counts them).

Reported: the host tables (automorphisms, pair masks, exclusions; once per call), the device work of one call (the two
kernels, CUDA events, warm-up first, then windows of at least 1 s, median of the repeats), the whole ``check_poses`` call
(tables + upload + kernels + one copy back), poses/s and pair tests/s (every pair the three clash sets examine), and the
float64 numpy oracle's clash-screen rate on a subset on the host cores for context.  The card's name and power limit
are read in the same run.  Writes ``profiles/posecheck_bench.json``.

    python scripts/posecheck_bench.py [--ligands 200] [--samples 10] [--repeats 5] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from diffdock_pocket_b200 import inputs, posecheck as pc  # noqa: E402


def card():
    name = torch.cuda.get_device_name(0)
    try:
        limit = subprocess.run(['nvidia-smi', '--query-gpu=power.limit', '--format=csv,noheader', '-i', '0'],
                               capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        limit = 'unknown'
    return name, limit


def random_rotation(rng):
    q = rng.randn(4)
    w, x, y, z = q / np.linalg.norm(q)
    return np.array([[1 - 2 * (y * y + z * z), 2 * (x * y - z * w), 2 * (x * z + y * w)],
                     [2 * (x * y + z * w), 1 - 2 * (x * x + z * z), 2 * (y * z - x * w)],
                     [2 * (x * z - y * w), 2 * (y * z + x * w), 1 - 2 * (x * x + y * y)]])


def oracle_rate(graphs, lig, atoms, n_poses):
    """float64 numpy clash screen (all three sets) of the first n_poses poses -> pair tests / s on the host cores."""
    pairs, t0 = 0, time.perf_counter()
    k = 0
    for g, L in zip(graphs, lig):
        rl = pc.RADIUS_TABLE[pc.ligand_elements(g)].astype(np.float64)
        ra = pc.RADIUS_TABLE[pc.atom_elements(g)].astype(np.float64)
        far = np.triu(pc.far_pairs(len(rl), pc._bonds(g)), 1)
        moved, owner = pc.moved_atoms(g), pc.residue_owner(g)
        excl = pc.bonded_exclusions(g['atom'].pos.numpy(), moved, owner)
        keep = owner[moved][:, None] != owner[None]
        keep[excl[:, 0], excl[:, 1]] = False
        for s in range(L.shape[0]):
            x = L[s].astype(np.float64)
            a = atoms.astype(np.float64)
            for d, sm, m in ((np.linalg.norm(x[:, None] - a[None], axis=-1), rl[:, None] + ra[None], None),
                             (np.linalg.norm(a[moved][:, None] - a[None], axis=-1), ra[moved][:, None] + ra[None], keep),
                             (np.linalg.norm(x[:, None] - x[None], axis=-1), rl[:, None] + rl[None], far)):
                r = d / sm
                r = r[m] if m is not None else r
                count, low = int((r < 0.75).sum()), (r.min() if r.size else np.inf)      # computed to be timed
                pairs += d.size
            k += 1
            if k == n_poses:
                return pairs / (time.perf_counter() - t0), k
    return pairs / (time.perf_counter() - t0), k


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--ligands', type=int, default=200)
    ap.add_argument('--samples', type=int, default=10)
    ap.add_argument('--repeats', type=int, default=5)
    ap.add_argument('--oracle-poses', type=int, default=50)
    ap.add_argument('--out', default=os.path.join(ROOT, 'profiles', 'posecheck_bench.json'))
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit('posecheck_bench: no CUDA device (every rate would be "not measured")')
    dev = torch.device('cuda:0')
    name, limit = card()
    rng = np.random.RandomState(0)
    pocket = inputs.synthetic_complex(0, n_lig=20, n_res=100, flexible_residues=5)
    sizes = inputs.pdbbind_test_sizes()
    graphs, lig = [], []
    for i in range(a.ligands):
        g = inputs.with_ligand(pocket, seed=1000 + i, n_lig=int(sizes[rng.randint(len(sizes))]))
        x = g['ligand'].pos.numpy().astype(np.float64)
        c = x.mean(0)
        lig.append(np.stack([(x - c) @ random_rotation(rng).T + c + rng.randn(3) * 2.0 for _ in range(a.samples)]).astype(np.float32))
        graphs.append(g)
    atoms = pocket['atom'].pos.numpy()
    ref_l = []                              # a ligand above the automorphism cap is screened for clashes only (no RMSD)
    for g in graphs:
        try:
            pc.automorphisms(pc.ligand_elements(g), pc._bonds(g))
            ref_l.append(g['ligand'].pos.numpy())
        except ValueError:
            ref_l.append(None)
    ref_a = [atoms] * len(graphs)
    lig_dev = [torch.from_numpy(l).to(dev) for l in lig]
    n_moved = len(pc.moved_atoms(pocket))
    na = atoms.shape[0]
    pair_tests = sum(l.shape[0] * (l.shape[1] * na + n_moved * na + l.shape[1] * (l.shape[1] - 1) // 2) for l in lig)
    n_poses = sum(l.shape[0] for l in lig)

    t0 = time.perf_counter()
    checks = pc.PoseChecks(graphs, lig_dev, None, ref_l, ref_a)
    torch.cuda.synchronize()
    t_tables = time.perf_counter() - t0
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def window(n):                                               # seconds for n back-to-back calls
        e0.record()
        for _ in range(n):
            checks.launch()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / 1e3

    window(20)                                                   # warm-up: module load, first launches
    iters = max(1, int(np.ceil(1.1 * 20 / window(20))))          # sized from warm calls to last about 1.1 s
    per_call = []
    while len(per_call) < a.repeats:
        t = window(iters)
        if t < 1.0:                                              # every timed window lasts at least 1 s
            iters = int(np.ceil(iters * 1.1 / t))
            continue
        per_call.append(t / iters)
    t_dev = float(np.median(per_call))
    res = checks.result()
    e2e = []
    for _ in range(2):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        pc.check_poses(graphs, lig_dev, None, ref_l, ref_a)
        e2e.append(time.perf_counter() - t0)
    t_e2e = float(np.median(e2e))
    o_rate, o_poses = oracle_rate(graphs, lig, atoms, a.oracle_poses)
    out = dict(
        card=name, power_limit=limit, torch=torch.__version__,
        setup=dict(pocket_residues=100, pocket_atoms=na, moved_sidechain_atoms=n_moved, ligands=a.ligands, samples=a.samples,
                   poses=n_poses, ligands_above_automorphism_cap=sum(r is None for r in ref_l),
                   mean_ligand_atoms=float(np.mean([l.shape[1] for l in lig])), pair_tests_per_call=pair_tests),
        device=dict(seconds_per_call=t_dev, repeats=per_call, launches_per_window=iters, poses_per_s=n_poses / t_dev,
                    pair_tests_per_s=pair_tests / t_dev),
        check_poses_call=dict(seconds=t_e2e, poses_per_s=n_poses / t_e2e, host_tables_seconds_first_call=t_tables),
        oracle_float64_numpy=dict(poses=o_poses, pair_tests_per_s=o_rate, host_cores=os.cpu_count()),
        ligand_pocket_clashes_mean=float(np.mean(np.concatenate([r['ligand_pocket_clashes'] for r in res]))),
    )
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, 'w') as f:
        json.dump(out, f, indent=1)
    print(json.dumps(out))


if __name__ == '__main__':
    main()
