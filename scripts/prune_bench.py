"""Pruned convolutions (``prune_edges``: the atom-aggregating atom-atom / atom-residue convs of the last two interaction
layers run on the edges into atoms whose features are read afterwards) against unpruned plans on BASELINE.json configs[1]:
3dpf ESMFold apo pocket, README big model, 40 samples in mini-batches of 20, 20 reverse-diffusion steps + confidence pass,
bf16 tensor-core convs.  Pruned and unpruned alternate in one process (``--rounds`` times each).
  python scripts/prune_bench.py [--rounds 3] [--mode bf16] [--out FILE]
Per round and setting:
  resident  poses/s of 20 steps + confidence on resident plans (StepRunners built once, captured step graphs, start poses
            reset by device copies) -- the sampler's steady state;
  e2e       poses/s of a whole sampling() call (host graphs in, host poses out; the resident-state cache serves repeats);
  layer_ms  CUDA-event time of the fused TP-conv launch of every interaction layer of one eager score-model forward
            (batch of 20, t = 0.5), and conv_ms their sum;
and once per setting: the live edge count of every layer's conv launch, the live atoms after the last two layers, and the
device memory one batch-20 score-model plan allocates."""
import argparse
import copy
import json
import os
import subprocess
import sys
import time
from functools import partial

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from diffdock_pocket_b200 import diffusion_utils as du, inputs, sampling as ps, utils  # noqa: E402
from diffdock_pocket_b200.hetero import Batch  # noqa: E402

TEMP = dict(temp_sampling=[0.9766, 6.0774, 6.7616, 1.4488], temp_psi=[1.5103, 0.8141, 0.7662, 1.3396], temp_sigma_data=0.48884)   # bench.py


def gpu_info():
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except (OSError, subprocess.SubprocessError, IndexError):
        q = 'unknown'
    return {'device': torch.cuda.get_device_name(0), 'nvidia_smi': q}


def main():
    p = argparse.ArgumentParser()
    p.add_argument('--rounds', type=int, default=3)
    p.add_argument('--mode', default='bf16', choices=['bf16', 'bf16x3', 'fp32'])
    p.add_argument('--samples', type=int, default=40)
    p.add_argument('--batch-size', type=int, default=20)
    p.add_argument('--inference-steps', type=int, default=20)
    p.add_argument('--out', default=None, help='also write the JSON record here')
    args = p.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('prune_bench.py measures on the GPU: no CUDA device')
    dev = torch.device('cuda:0')
    model, conf, sa, ca = utils.build_models(dev, seed=0)
    model.conv_mode = conf.conv_mode = args.mode
    g = inputs.load_graph_npz(os.path.join(ROOT, 'tests', 'golden', '3dpf_apo.npz'), name='3dpf_apo')
    np.random.seed(0)
    torch.manual_seed(0)
    dl0 = [copy.deepcopy(g) for _ in range(args.samples)]
    ps.randomize_position(dl0, False, False, sa.tr_sigma_max, flexible_sidechains=True)
    N, steps = args.samples, args.inference_steps
    sch = du.get_t_schedule('expbeta', steps)
    t2s = partial(du.t_to_sigma, args=sa)
    chunks = [list(range(i, min(i + args.batch_size, N))) for i in range(0, N, args.batch_size)]
    coefs = [ps.step_coefficients(t, steps, (sch,) * 4, t2s, sa, False, TEMP['temp_sampling'], TEMP['temp_psi'],
                                  TEMP['temp_sigma_data'], True) for t in range(steps)]

    def set_mode(prune):
        model.prune_edges = conf.prune_edges = prune

    def e2e(prune, seed=7):
        set_mode(prune)
        dl = copy.deepcopy(dl0)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        torch.manual_seed(seed)
        out, c = ps.sampling(dl, model, steps, sch, sch, sch, sch, dev, t2s, sa, confidence_model=conf, filtering_model_args=ca,
                             batch_size=args.batch_size, **TEMP)
        dt = time.perf_counter() - t0
        return N / dt, torch.stack([o['ligand'].pos for o in out]).cpu(), c.reshape(-1).cpu()

    resident = {}

    def build_resident(prune):
        set_mode(prune)
        streams = [torch.cuda.Stream(device=dev) for _ in range(2)] if len(chunks) > 1 else [None]
        with torch.no_grad():
            rs = [ps.StepRunner(model, [dl0[i] for i in idx], True, False, use_graph=True, stream=streams[k % len(streams)])
                  for k, idx in enumerate(chunks)]
            cps = [conf.make_plan(Batch.from_data_list([dl0[i] for i in idx])) for idx in chunks]
        init = [(r.pl.lig_pos.clone(), r.pl.atom_pos.clone()) for r in rs]
        T_tot, S_tot = sum(r.T for r in rs), sum(r.S for r in rs)
        noise = torch.randn(steps, 6 * N + T_tot + S_tot, generator=torch.Generator().manual_seed(3))
        return rs, cps, init, noise, T_tot

    def resident_pass(prune):
        set_mode(prune)
        rs, cps, init, noise, T_tot = resident[prune]
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        with torch.no_grad():
            for r, (lp, ap) in zip(rs, init):
                r.pl.lig_pos.copy_(lp)
                r.pl.atom_pos.copy_(ap)
                r.sync_in()
            for t_idx in range(steps):
                t, coef = coefs[t_idx]
                z = noise[t_idx]
                s0 = t0_ = c0 = 0
                for idx, r in zip(chunks, rs):
                    b = len(idx)
                    row = torch.cat([z[3 * s0:3 * (s0 + b)], z[3 * N + 3 * s0:3 * N + 3 * (s0 + b)], z[6 * N + t0_:6 * N + t0_ + r.T],
                                     z[6 * N + T_tot + c0:6 * N + T_tot + c0 + r.S]])
                    r.step(t, coef, row)
                    s0, t0_, c0 = s0 + b, t0_ + r.T, c0 + r.S
            cs = []
            for idx, r, cpl in zip(chunks, rs, cps):
                with r.ctx():
                    cpl.lig_pos.copy_(r.pl.lig_pos)
                    cpl.atom_pos.copy_(r.pl.atom_pos)
                    zt = torch.zeros(len(idx))
                    cs.append(conf.run_plan(cpl, {'tr': zt, 'rot': zt, 'tor': zt, 'sc_tor': zt}).reshape(-1).clone())
            for r in rs:
                r.sync_out()
            torch.cuda.synchronize()
        return N / (time.perf_counter() - t0)

    def make_plan(prune):
        set_mode(prune)
        torch.cuda.synchronize()
        m0 = torch.cuda.memory_allocated(dev)
        pl = model.make_plan(Batch.from_data_list([dl0[i] for i in chunks[0]]))
        torch.cuda.synchronize()
        return pl, torch.cuda.memory_allocated(dev) - m0

    ct = {k: torch.full((len(chunks[0]),), 0.5) for k in ('tr', 'rot', 'tor', 'sc_tor')}
    plans = {}

    def layer_ms(prune, reps=5):
        """Event time of each interaction layer's fused conv launch (the first num_conv_layers profiled launches; the
        torsion-head and centre convs follow) and the live edge count of every conv in it."""
        set_mode(prune)
        pl = plans[prune][0]
        nl = model.num_conv_layers
        with torch.no_grad():
            for _ in range(2):
                model.run_plan(pl, ct)
            torch.cuda.synchronize()
            tot = np.zeros(nl)
            for _ in range(reps):
                model.profile = []
                model.run_plan(pl, ct)
                torch.cuda.synchronize()
                tot += np.array([e0.elapsed_time(e1) for e0, e1, _ in model.profile[:nl]]) / reps
            edges = [[int(es.n_dev.item()) for _, es, _ in items] for _, _, items in model.profile[:nl]]
            model.profile = None
        return tot.tolist(), edges

    rec = {'workload': f'3dpf_apo (BASELINE.json configs[1]): {N} samples, batch {args.batch_size}, {steps} steps + confidence, '
                       f'conv_mode {args.mode}, README big model', 'gpu': gpu_info(), 'rounds': []}
    with torch.no_grad():
        make_plan(True)                                               # first plan: packs the weights (not plan memory)
        for prune in (False, True):
            plans[prune] = make_plan(prune)
    for prune in (False, True):                                       # warm-up: plans, graph capture, cache retention
        resident[prune] = build_resident(prune)
        resident_pass(prune)
        resident_pass(prune)
        for _ in range(3):
            e2e(prune)
        layer_ms(prune, reps=1)
    for r in range(args.rounds):
        for prune in (False, True):
            lm, _ = layer_ms(prune)
            row = {'round': r, 'prune': prune, 'resident_poses_s': resident_pass(prune), 'e2e_poses_s': e2e(prune)[0],
                   'layer_ms': lm, 'conv_ms': sum(lm)}
            rec['rounds'].append(row)
            print(json.dumps(row), flush=True)
    for prune in (False, True):
        pl, nbytes = plans[prune]
        _, edges = layer_ms(prune, reps=1)
        key = 'pruned' if prune else 'unpruned'
        rec[key] = {'plan_bytes': nbytes, 'layer_edges': edges, 'layer_edges_total': [sum(e) for e in edges]}
        if prune:
            rec[key]['live_atoms'] = {'last_layer': int(pl.live[0].sum()), 'layer_L-2': int(pl.live[1].sum()), 'atoms': pl.NA}
            rec[key]['pruned_set_bytes'] = sum(t.numel() * t.element_size() for p in pl.pruned.values()
                                               for t in (p.edge, p.n_dev, p.sh, p.emb, p.counts)) + pl.live.numel()
        rows = [x for x in rec['rounds'] if x['prune'] == prune]
        rec['median_' + key] = {k: float(np.median([x[k] for x in rows])) for k in ('resident_poses_s', 'e2e_poses_s', 'conv_ms')}
        rec['median_' + key]['layer_ms'] = np.median(np.array([x['layer_ms'] for x in rows]), 0).tolist()
    set_mode(True)
    line = json.dumps(rec)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as f:
            f.write(line + '\n')


if __name__ == '__main__':
    main()
