"""Cost of the deterministic mode (torch.use_deterministic_algorithms(True): fixed-point scatter-adds in the convolutions)
on BASELINE.json configs[1]: 3dpf ESMFold apo pocket, README big model, 40 samples in mini-batches of 20, 20 reverse-diffusion
steps + confidence pass, bf16 tensor-core convs.  Default and deterministic mode alternate in one process (``--rounds``
times each) so that both see the same clocks and neighbours.
  python scripts/deterministic_bench.py [--rounds 3] [--mode bf16] [--out FILE]
Per round and mode:
  resident  poses/s of 20 steps + confidence on resident plans (StepRunners built once, captured step graphs, start poses
            reset by device copies) -- the sampler's steady state;
  e2e       poses/s of a whole sampling() call (host graphs in, host poses out; the resident-state cache serves repeats);
  conv_ms   summed CUDA-event time of the fused TP-conv launches of one eager score-model forward (batch of 20);
and once: the largest ligand-pose and confidence difference between two default-mode sampling() calls with the same seeds
(information only: how far the fp32 atomics let two identical runs drift), and the same for two deterministic calls (0)."""
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
        raise SystemExit('deterministic_bench.py measures on the GPU: no CUDA device')
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

    def set_mode(det):
        torch.use_deterministic_algorithms(det)

    def e2e(det, seed=7):
        set_mode(det)
        dl = copy.deepcopy(dl0)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        torch.manual_seed(seed)
        out, c = ps.sampling(dl, model, steps, sch, sch, sch, sch, dev, t2s, sa, confidence_model=conf, filtering_model_args=ca,
                             batch_size=args.batch_size, **TEMP)
        dt = time.perf_counter() - t0
        return N / dt, torch.stack([o['ligand'].pos for o in out]).cpu(), c.reshape(-1).cpu()

    resident = {}

    def build_resident(det):
        set_mode(det)
        streams = [torch.cuda.Stream(device=dev) for _ in range(2)] if len(chunks) > 1 else [None]
        with torch.no_grad():
            rs = [ps.StepRunner(model, [dl0[i] for i in idx], True, False, use_graph=True, stream=streams[k % len(streams)])
                  for k, idx in enumerate(chunks)]
            cps = [conf.make_plan(Batch.from_data_list([dl0[i] for i in idx])) for idx in chunks]
        init = [(r.pl.lig_pos.clone(), r.pl.atom_pos.clone()) for r in rs]
        T_tot, S_tot = sum(r.T for r in rs), sum(r.S for r in rs)
        noise = torch.randn(steps, 6 * N + T_tot + S_tot, generator=torch.Generator().manual_seed(3))
        return rs, cps, init, noise, T_tot

    def resident_pass(det):
        set_mode(det)
        rs, cps, init, noise, T_tot = resident[det]
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

    def conv_ms(det, reps=5):
        set_mode(det)
        b = chunks[0]
        with torch.no_grad():
            pl = model.make_plan(Batch.from_data_list([dl0[i] for i in b]))
            ct = {k: torch.full((len(b),), 0.5) for k in ('tr', 'rot', 'tor', 'sc_tor')}
            for _ in range(2):
                model.run_plan(pl, ct)
            torch.cuda.synchronize()
            tot = 0.0
            for _ in range(reps):
                model.profile = []
                model.run_plan(pl, ct)
                torch.cuda.synchronize()
                tot += sum(e0.elapsed_time(e1) for e0, e1, _ in model.profile) / reps
            model.profile = None
        return tot

    rec = {'workload': f'3dpf_apo (BASELINE.json configs[1]): {N} samples, batch {args.batch_size}, {steps} steps + confidence, '
                       f'conv_mode {args.mode}, README big model', 'gpu': gpu_info(), 'rounds': []}
    for det in (False, True):                                         # warm-up: plans, graph capture, cache retention
        resident[det] = build_resident(det)
        resident_pass(det)
        resident_pass(det)
        for _ in range(3):
            e2e(det)
        conv_ms(det, reps=1)
    for r in range(args.rounds):
        for det in (False, True):
            row = {'round': r, 'deterministic': det, 'resident_poses_s': resident_pass(det), 'e2e_poses_s': e2e(det)[0],
                   'conv_ms': conv_ms(det)}
            rec['rounds'].append(row)
            print(json.dumps(row), flush=True)
    # run-to-run differences of two calls with the same seeds
    for det in (False, True):
        _, p1, c1 = e2e(det, seed=11)
        _, p2, c2 = e2e(det, seed=11)
        rec[f'repeat_diff_{"deterministic" if det else "default"}'] = {
            'max_pose_diff_A': float((p1 - p2).abs().max()), 'max_confidence_diff': float((c1 - c2).abs().max()),
            'top1_same': bool(int(c1.argmax()) == int(c2.argmax()))}
    set_mode(False)
    for det in (False, True):
        rows = [x for x in rec['rounds'] if x['deterministic'] == det]
        rec['median_' + ('deterministic' if det else 'default')] = {
            k: float(np.median([x[k] for x in rows])) for k in ('resident_poses_s', 'e2e_poses_s', 'conv_ms')}
    line = json.dumps(rec)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as f:
            f.write(line + '\n')


if __name__ == '__main__':
    main()
