"""Headline benchmark: docked poses/sec for 20-step reverse diffusion (BASELINE.json `metric`).

One bench "step" = one complete pass of the hot path over one batch of synthetic input: `samples` poses of
one complex through `inference_steps` reverse-diffusion steps (score-model forward + fused pose update per
mini-batch per step) plus the confidence pass.  Workload at N=1 is BASELINE.json configs[1] (3dpf ESMFold apo
pocket, explicit centre, 7 flexible residues, 40 samples, batch 20) built from tests/golden/3dpf_apo.npz with
seeded synthetic ESM features and random-init weights of the README big score model (no checkpoint offline).

  python bench.py --gpus N --steps K --warmup W            # this implementation (one rank per GPU under torchrun)
  python bench.py --impl reference ...                      # CPU arm: the oracle port on the host cores

`value`  : poses/s with the batch already resident in HBM (plans built before the timed region).
`e2e`    : poses/s through the public `sampling()` call with HOST graphs: collate + H2D upload of the batch,
           the whole loop, D2H of final poses and confidences inside the timed region.
`roofline`: the fused TP-conv kernel (tcgen05), achieved algorithmic TFLOP/s measured with CUDA events around
           its launches in one instrumented forward, against the measured bf16 peak (MEASURED_PEAKS.json).
Multi-GPU: complexes are sharded (each rank docks its own copy of the workload: weak scaling); the only
collective is one NCCL all-gather of final poses + confidences for ranking, after the loop.
"""
import argparse
import copy
import json
import os
import subprocess
import sys
import threading
import time
from functools import partial

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
GOLD = os.path.join(ROOT, 'tests', 'golden')
TEMP = dict(temp_sampling=[0.9766, 6.0774, 6.7616, 1.4488], temp_psi=[1.5103, 0.8141, 0.7662, 1.3396], temp_sigma_data=0.48884)


def parse():
    p = argparse.ArgumentParser()
    p.add_argument('--gpus', type=int, default=1)
    p.add_argument('--steps', type=int, default=3)
    p.add_argument('--warmup', type=int, default=3)
    p.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    p.add_argument('--mode', default='bf16', choices=['bf16', 'bf16x3', 'fp32'])
    p.add_argument('--samples', type=int, default=40)
    p.add_argument('--batch-size', type=int, default=20)
    p.add_argument('--inference-steps', type=int, default=20)
    p.add_argument('--workload', default='3dpf_apo', choices=['3dpf_apo', '3dpf_holo', 'forward64', 'pdbbind_synth', 'screen'],
                   help='3dpf_apo: BASELINE configs[1] (default, the headline); forward64: configs[2] score-model forward microbench; '
                        'pdbbind_synth: configs[3] complex-sharded set; screen: configs[4] one pocket x many ligands, ligand-sharded')
    p.add_argument('--scaling', default='weak', choices=['weak', 'strong'],
                   help='3dpf workloads under torchrun: weak = every rank docks its own --samples; strong = --samples split over the ranks')
    p.add_argument('--complexes', type=int, default=None, help='pdbbind_synth: complexes (default 48; 363 = the whole test-set law); '
                                                               'screen: ligands (default 192; configs[4] names 10000)')
    p.add_argument('--no-pipeline', action='store_true', help='pdbbind_synth / screen: serial loop over the complexes (A/B of the software pipeline)')
    p.add_argument('--profile-range', action='store_true', help='cudaProfilerStart/Stop around the timed resident steps (for ncu --profile-from-start off)')
    p.add_argument('--no-fp32-grade', action='store_true', help='skip the additional bf16x3 (fp32-grade) resident measurement')
    p.add_argument('--cpu-samples', type=int, default=4)
    p.add_argument('--cpu-steps', type=int, default=3)
    p.add_argument('--no-cpu-baseline', action='store_true')
    p.add_argument('--single-stream', action='store_true', help='run the mini-batches back to back on one stream (A/B of the two-stream overlap)')
    p.add_argument('--no-graph', action='store_true', help='launch kernels eagerly instead of replaying the captured step graph')
    p.add_argument('--dump-outputs', metavar='DIR', default=None,
                   help='after the timed steps, write what the last timed step computed as DIR/<name>.npy (rank 0; float32 / '
                        'float64, at most 64 MB in all: larger outputs are cut to a fixed seeded sample of rows), so that two '
                        'builds can be compared output for output on identical inputs')
    args = p.parse_args()
    if args.steps < 1:
        p.error('--steps must be at least 1')
    if args.dump_outputs is not None and args.impl == 'reference':
        p.error('--dump-outputs records the CUDA path; the reference arm runs a scaled-down sample of the workload')
    return args


DUMP_LIMIT = 64 * 10 ** 6          # bytes of all .npy files together
NPY_HEADER = 128


def dump_outputs(out_dir, arrays):
    """Write ``arrays`` (name -> tensor / array) as ``out_dir/<name>.npy``: float64 stays float64, integers become float64
    (exact), everything else float32.  When the files would exceed DUMP_LIMIT bytes in all, each array keeps the same
    fraction of its leading axis, chosen by a fixed seed, so that arrays with the same leading axis keep the same rows."""
    arrays = {k: (v.detach().cpu().numpy() if torch.is_tensor(v) else np.asarray(v)) for k, v in arrays.items()}
    arrays = {k: v.astype(np.float64 if v.dtype == np.float64 or v.dtype.kind in 'iub' else np.float32) for k, v in arrays.items()}
    total = sum(v.nbytes for v in arrays.values())
    budget = DUMP_LIMIT - NPY_HEADER * len(arrays)
    if total > budget:
        frac = budget / total
        for k, v in arrays.items():
            if v.ndim and v.shape[0] > 1:
                keep = max(1, int(v.shape[0] * frac))
                arrays[k] = v[np.sort(np.random.RandomState(0).choice(v.shape[0], keep, replace=False))]
    os.makedirs(out_dir, exist_ok=True)
    for k, v in arrays.items():
        np.save(os.path.join(out_dir, k + '.npy'), v)


def peaks():
    path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(path):
        d = json.load(open(path))
        return d.get('bf16_tflops_sustained', 1414.3), d.get('hbm_gbs', 6452.2), 'measured (MEASURED_PEAKS.json, sustained bf16)'
    return 1590.0, 6650.0, 'fallback (B200_PROFILING.md)'


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.stop_flag = index, [], False

    def run(self):
        q = ('clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
             'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')
        while not self.stop_flag:
            try:
                out = subprocess.run(['nvidia-smi', f'--query-gpu={q}', '--format=csv,noheader,nounits', '-i', str(self.index)],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.split(',')])
            except Exception:
                pass
            time.sleep(0.2)

    def summary(self):
        if not self.rows:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        sm = sorted(float(r[0]) for r in self.rows if r[0].replace('.', '').isdigit())
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        reasons = [n for i, n in enumerate(names) if any(r[2 + i].lower().startswith('active') for r in self.rows if len(r) > 2 + i)]
        return {'sm_mhz': sm[len(sm) // 2] if sm else None, 'sm_max_mhz': float(self.rows[0][1]) if self.rows else None,
                'reasons': reasons, 'samples': len(self.rows)}


def workload(args, seed):
    from diffdock_pocket_b200 import inputs, sampling as S, utils
    g = inputs.load_graph_npz(os.path.join(GOLD, args.workload + '.npz'), name=args.workload)
    sa = utils.score_model_args()
    np.random.seed(seed)
    torch.manual_seed(seed)
    dl = [copy.deepcopy(g) for _ in range(args.samples)]
    S.randomize_position(dl, False, False, sa.tr_sigma_max, flexible_sidechains=True)
    return g, dl


def conv_flops(ns, w_numel):
    return 2.0 * ((3 * ns) * (3 * ns) + (3 * ns) * w_numel + w_numel)


def conv_bytes(ns, f_in, n_edges):
    """SURVEY 8(d) minimal fused traffic of one conv: per edge 4 * (ns edge embedding + 2 * ns scalar blocks + f_in gathered
    features + 3 edge vector + 2 indices)."""
    return 4.0 * (3 * ns + f_in + 3 + 2) * n_edges


def ncu_traffic(args):
    """dram__bytes_read + dram__bytes_write per launch of the dominant kernel, from the committed ncu --set full capture of
    THIS command (profiles/r2_ncu_traffic.json, written by scripts/ncu_summary.py); None when there is no capture."""
    path = os.path.join(ROOT, 'profiles', 'r2_ncu_traffic.json')
    key = f'{args.workload}:{args.mode}:b{args.batch_size}'
    if os.path.exists(path):
        d = json.load(open(path))
        if key in d:
            return float(d[key]['dram_bytes_per_launch']), d[key].get('source', path)
    return None, None


def cpu_arm(args, n_samples, n_steps, threads):
    """Oracle port (pure PyTorch fp32 on the host cores) on a bounded sample, scaled to poses/s of the full workload."""
    from diffdock_pocket_b200 import so3, torus, utils
    from oracle import diffusion_ref as D, factory, sampling_ref as S
    torch.set_num_threads(threads)
    model, conf, sa, ca = utils.build_models(torch.device('cpu'), seed=0)
    om = factory.oracle_model(sa, model.state_dict(), so3.score_norm_np, torus.score_norm)
    _, dl = workload(args, 0)
    dl = dl[:n_samples]
    sch = D.get_t_schedule(args.inference_steps)
    torch.manual_seed(1)
    t0 = time.time()
    S.sampling(dl, om, args.inference_steps, sch, sch, sch, sch, partial(D.t_to_sigma, args=sa), sa, batch_size=args.batch_size,
               max_steps=n_steps, **TEMP)
    dt = time.time() - t0
    full = dt * (args.samples * args.inference_steps) / (n_samples * n_steps)
    return args.samples / full, dt


def run_reference(args):
    rank = int(os.environ.get('RANK', 0))
    if rank != 0:
        return
    threads = os.cpu_count()
    vals = []
    for _ in range(args.warmup if args.warmup < 1 else 1):
        cpu_arm(args, 1, 1, threads)
    t_all = 0.0
    for _ in range(args.steps):
        v, dt = cpu_arm(args, args.cpu_samples, args.cpu_steps, threads)
        vals.append(v)
        t_all += dt
    value = float(np.mean(vals))
    sample = f'{args.cpu_samples} samples x {args.cpu_steps} of {args.inference_steps} steps per bench step, scaled linearly to {args.samples} x {args.inference_steps}'
    print(json.dumps({
        'impl': 'reference', 'metric': 'docked poses/sec (20-step reverse diffusion)', 'value': value, 'unit': 'poses/s',
        'n_gpus': args.gpus, 'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': 1000.0 * args.samples / value,
        'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
        'config': {'workload': f'{args.workload}: {args.samples} samples, batch {args.batch_size}, {args.inference_steps} steps (BASELINE.json configs[1])'},
        'cpu_baseline': {'value': value, 'unit': 'poses/s', 'cores': threads, 'kind': 'port', 'sample': sample},
        'e2e': {'value': value, 'unit': 'poses/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}}))


def _reduce_max(x, dev, world, dist):
    if world == 1:
        return x
    t = torch.tensor([x], device=dev, dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def bench_forward64(args, model, sa, dev, world, rank, local, dist):
    """BASELINE.json configs[2]: score-model forward microbench, batch of 64 pocket graphs (the 3dpf pocket: receptor_radius 15,
    atom_max_neighbors 8, c_alpha_max_neighbors 24; README big model), at t = 1.0 (every ligand-residue pair is an edge) and
    t = 0.05.  A step = one forward of the resident batch; value = graph-forwards / s at t = 1.0."""
    from diffdock_pocket_b200.hetero import Batch
    args.samples = 64
    g, dl = workload(argparse.Namespace(**{**vars(args), 'workload': '3dpf_apo'}), rank)
    with torch.no_grad():
        pl = model.make_plan(Batch.from_data_list(dl), graphs=dl)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    out, last = {}, {}
    sampler = ClockSampler(local)
    sampler.start()
    for tag, t in (('t1.0', 1.0), ('t0.05', 0.05)):
        ct = {k: torch.full((64,), t) for k in ('tr', 'rot', 'tor', 'sc_tor')}
        with torch.no_grad():
            for _ in range(max(args.warmup, 3)):
                model.run_plan(pl, ct)
            torch.cuda.synchronize()
            ms = []
            for _ in range(args.steps):
                flush.fill_(0)
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                scores = model.run_plan(pl, ct)
                e1.record()
                torch.cuda.synchronize()
                ms.append(e0.elapsed_time(e1))
            if args.dump_outputs is not None:
                last.update({f'{tag}_{k}': v.cpu() for k, v in zip(('tr', 'rot', 'tor', 'sc_tor'), scores)})
            model.profile = []
            model.run_plan(pl, ct)
            torch.cuda.synchronize()
            conv_ms = sum(a.elapsed_time(b) for a, b, _ in model.profile)
            conv_fl = sum(conv_flops(ns, w) * int(es.n_dev.item()) for _, _, convs in model.profile for (w, es, ns) in convs)
            model.profile = None
        m = _reduce_max(float(np.median(ms)), dev, world, dist)
        out[tag] = {'ms_per_forward': m, 'graph_forwards_per_s': world * 64 / (m / 1000.0), 'conv_ms': conv_ms,
                    'conv_tflops': conv_fl / (conv_ms * 1e-3) / 1e12, 'edges': {k: int(pl.es[k].n_dev.item()) for k in ('ll', 'lr', 'la', 'aa', 'rr', 'ar')}}
    sampler.stop_flag = True
    if rank == 0:
        peak_tf, hbm, peak_src = peaks()
        print(json.dumps({
            'metric': 'score-model graph-forwards/sec (batch 64 forward microbench)', 'value': out['t1.0']['graph_forwards_per_s'], 'unit': 'graph-forwards/s',
            'n_gpus': world, 'steps': args.steps, 'warmup': max(args.warmup, 3), 'ms_per_step': out['t1.0']['ms_per_forward'], 'higher_is_better': True,
            'scaling': 'weak', 'vs_baseline': None, 'dtype': args.mode, 'data': 'synthetic',
            'config': {'workload': 'forward64: 64 x 3dpf pocket graph (BASELINE.json configs[2]), README big model, resident batch, t = 1.0 (value) and t = 0.05',
                       'conv_mode': args.mode, 'l2': '256 MiB flush before every timed forward'},
            'clocks': sampler.summary(), 'detail': out,
            'roofline': {'bound': 'tensor', 'achieved': out['t1.0']['conv_tflops'], 'peak': peak_tf, 'unit': 'TFLOP/s', 'frac': out['t1.0']['conv_tflops'] / peak_tf,
                         'traffic': None, 'peak_source': peak_src}}))
        if args.dump_outputs is not None:
            dump_outputs(args.dump_outputs, last)
    if world > 1:
        dist.destroy_process_group()


def bench_set(args, model, conf, sa, ca, dev, world, rank, local, dist):
    """BASELINE.json configs[3] (``pdbbind_synth``: complexes whose ligand sizes follow the PDBBind test set, 40 samples each,
    complexes split over the ranks like np.array_split) and configs[4] (``screen``: one pocket x many procedural ligands x 10
    samples, ligands split over the ranks, final all-gather of the best confidences + global top-k).  The whole job goes
    through the host mirror of inference.py (graphs on the host in, ranked poses on the host out): value == e2e."""
    from diffdock_pocket_b200 import inference, inputs
    screen = args.workload == 'screen'
    n = args.complexes or (192 if screen else 48)
    t_gen = time.time()
    if screen:
        pocket = inputs.synthetic_complex(0, n_lig=30, n_res=139, flexible_residues=7, name='pocket')
        sizes = inputs.pdbbind_test_sizes()
        graphs = [inputs.with_ligand(pocket, 1000 + i, sizes[i % len(sizes)], name=f'ligand{i}') for i in range(n)]
        spc = 10
    else:
        graphs = inputs.pdbbind_synth_set(n)
        spc = args.samples
    t_gen = time.time() - t_gen
    rows = [dict(complex_name=g.name, complex_graph=g) for g in graphs]
    iargs = inference.default_args(samples_per_complex=spc, batch_size=args.batch_size, inference_steps=args.inference_steps)
    sampler = ClockSampler(local)

    def one_pass(sub):
        np.random.seed(1 + rank)
        torch.manual_seed(1 + rank)
        return inference.infer_sharded(sub, model, iargs, sa, dev, filtering_model=conf, filtering_model_args=ca,
                                       batch_complexes=screen, pipeline=not args.no_pipeline)
    for _ in range(max(1, min(args.warmup, 2))):                       # warm-up on a small prefix (lazy init, allocator, weight images)
        one_pass(rows[:max(2 * world, 2)])
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.time()
    e0.record()
    for _ in range(args.steps):
        res, best, ok = one_pass(rows)
    e1.record()
    torch.cuda.synchronize()
    wall = (time.time() - t0) / args.steps
    if world > 1:
        dist.barrier()
    sampler.stop_flag = True
    ms = _reduce_max(e0.elapsed_time(e1) / args.steps, dev, world, dist)
    wall = _reduce_max(wall, dev, world, dist)
    poses = n * spc
    if rank == 0:
        order = torch.argsort(best, descending=True)
        print(json.dumps({
            'metric': 'docked poses/sec (20-step reverse diffusion)', 'value': poses / (ms / 1000.0), 'unit': 'poses/s', 'n_gpus': world,
            'steps': args.steps, 'warmup': max(1, min(args.warmup, 2)), 'ms_per_step': ms, 'higher_is_better': True, 'scaling': 'strong',
            'vs_baseline': None, 'dtype': args.mode, 'data': 'synthetic',
            'config': {'workload': (f'screen: one synthetic pocket (139 residues, 7 flexible) x {n} procedural ligands (PDBBind size law) x {spc} samples, '
                                    f'{args.inference_steps} steps + confidence, ligands split over the ranks, 2 ligands per sampler call (BASELINE.json configs[4]; it names 10000 ligands)'
                                    if screen else
                                    f'pdbbind_synth: {n} synthetic complexes (ligand sizes of the PDBBind test set; 363 = the whole set) x {spc} samples, batch {args.batch_size}, '
                                    f'{args.inference_steps} steps + confidence, complexes split over the ranks (BASELINE.json configs[3])'),
                       'pipeline': not args.no_pipeline, 'conv_mode': args.mode, 'generation_s': t_gen,
                       'l2': 'every complex brings new activations; weights (> 400 MB over the layers) exceed L2'},
            'clocks': sampler.summary(), 'wall_s': wall, 'succeeded_on_rank0': ok,
            'top3': [(int(i), round(float(best[i]), 4)) for i in order[:3]],
            'e2e': {'value': poses / (wall * 1000.0 / 1000.0), 'unit': 'poses/s', 'h2d_bytes_per_step': int(model.static_h2d_bytes), 'd2h_bytes_per_step': None}}))
        if args.dump_outputs is not None:
            # per complex of rank 0's shard, in complex order: samples ranked by confidence, positions in the input frame
            done = [r for r in res if r is not None]
            dump_outputs(args.dump_outputs, {
                'best_confidence': best,
                'confidence': np.concatenate([r['confidence'] for r in done]),
                'ligand_pos': np.concatenate([r['ligand_pos'].reshape(-1, 3) for r in done]),
                'atom_pos': np.concatenate([r['atom_pos'].reshape(-1, 3) for r in done])})
    if world > 1:
        dist.destroy_process_group()


def main():
    args = parse()
    if args.impl == 'reference':
        return run_reference(args)
    import torch.distributed as dist
    from diffdock_pocket_b200 import _lib, diffusion_utils as du, sampling as ps, utils
    from diffdock_pocket_b200.hetero import Batch
    world = int(os.environ.get('WORLD_SIZE', 1))
    rank = int(os.environ.get('RANK', 0))
    local = int(os.environ.get('LOCAL_RANK', 0))
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    if world > 1:
        # NCCL prints its version banner on stdout when the communicator comes up: keep stdout for the one JSON line
        sys.stdout.flush()
        saved = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group('nccl', device_id=dev)
            dist.barrier()
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved, 1)
            os.close(saved)
    model, conf, sa, ca = utils.build_models(dev, seed=0)
    model.conv_mode = conf.conv_mode = args.mode
    if args.workload == 'forward64':
        return bench_forward64(args, model, sa, dev, world, rank, local, dist)
    if args.workload in ('pdbbind_synth', 'screen'):
        return bench_set(args, model, conf, sa, ca, dev, world, rank, local, dist)
    total_samples = args.samples * (world if args.scaling == 'weak' else 1)
    if args.scaling == 'strong':
        # one complex's samples split over the ranks (np.array_split rule); every rank still draws the same initial poses
        from diffdock_pocket_b200.parallel import shard_range
        g, dl_all = workload(args, 0)
        lo, hi = shard_range(args.samples, rank, world)
        dl0 = dl_all[lo:hi]
        args.samples = hi - lo
        assert args.samples > 0, 'more ranks than samples'
    else:
        g, dl0 = workload(args, rank)
    sch = du.get_t_schedule('expbeta', args.inference_steps)
    t2s = partial(du.t_to_sigma, args=sa)
    kw = dict(confidence_model=conf, filtering_model_args=ca, batch_size=args.batch_size, **TEMP)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def gather_rank(poses, confidence):
        """The single collective of the path: all-gather final poses + confidences, rank by confidence
        -> (all poses, all confidences, ranking)."""
        from diffdock_pocket_b200.parallel import gather_and_rank
        return gather_and_rank(poses, confidence)

    # ---- e2e pass through the public API (host graphs in, host poses out) --------------------------------
    def e2e_step(dl):
        torch.manual_seed(7)
        out, c = ps.sampling(dl, model, args.inference_steps, sch, sch, sch, sch, dev, t2s, sa, concurrent_batches=not args.single_stream, **kw)
        poses = torch.stack([o['ligand'].pos for o in out]).to(dev)
        return gather_rank(poses, c.reshape(-1).to(dev))[2].cpu()

    # ---- resident pass: plans + pose states (+ captured step graphs) built once, inputs already in HBM ----------
    chunks = [list(range(i, min(i + args.batch_size, args.samples))) for i in range(0, args.samples, args.batch_size)]
    # independent mini-batches alternate between two streams, exactly as sampling() runs them
    streams = [torch.cuda.Stream(device=dev) for _ in range(2)] if len(chunks) > 1 and not args.single_stream else [None]
    def build_resident():
        with torch.no_grad():
            rs = [ps.StepRunner(model, [dl0[i] for i in idx], True, False, use_graph=not args.no_graph, stream=streams[k % len(streams)])
                  for k, idx in enumerate(chunks)]
            cps = [conf.make_plan(Batch.from_data_list([dl0[i] for i in idx])) for idx in chunks]
        return rs, cps, [r.pl for r in rs], [(r.pl.lig_pos.clone(), r.pl.atom_pos.clone()) for r in rs]
    runners, cplans, plans, init = build_resident()
    N = args.samples
    T_tot, S_tot = sum(r.T for r in runners), sum(r.S for r in runners)
    noise = torch.randn(args.inference_steps, 6 * N + T_tot + S_tot, generator=torch.Generator().manual_seed(3))
    coefs = [ps.step_coefficients(t_idx, args.inference_steps, (sch,) * 4, t2s, sa, False, TEMP['temp_sampling'], TEMP['temp_psi'],
                                  TEMP['temp_sigma_data'], True) for t_idx in range(args.inference_steps)]

    def resident_step(runners=None, cplans=None, plans=None, init=None):
        runners, cplans, plans, init = runners or R0[0], cplans or R0[1], plans or R0[2], init or R0[3]
        with torch.no_grad():
            for pl, (lp, ap) in zip(plans, init):
                pl.lig_pos.copy_(lp)
                pl.atom_pos.copy_(ap)
            for r in runners:
                r.sync_in()
            for t_idx in range(args.inference_steps):
                t, coef = coefs[t_idx]
                z = noise[t_idx]
                s0 = t0 = c0 = 0
                for idx, r in zip(chunks, runners):
                    b = len(idx)
                    row = torch.cat([z[3 * s0:3 * (s0 + b)], z[3 * N + 3 * s0:3 * N + 3 * (s0 + b)], z[6 * N + t0:6 * N + t0 + r.T],
                                     z[6 * N + T_tot + c0:6 * N + T_tot + c0 + r.S]])
                    r.step(t, coef, row)
                    s0, t0, c0 = s0 + b, t0 + r.T, c0 + r.S
            cs = []
            for idx, r, cpl in zip(chunks, runners, cplans):
                with r.ctx():
                    cpl.lig_pos.copy_(r.pl.lig_pos)
                    cpl.atom_pos.copy_(r.pl.atom_pos)
                    zt = torch.zeros(len(idx))
                    cs.append(conf.run_plan(cpl, {'tr': zt, 'rot': zt, 'tor': zt, 'sc_tor': zt}).reshape(-1).clone())
            for r in runners:
                r.sync_out()
            return gather_rank(torch.cat([pl.lig_pos for pl in plans]).reshape(N, -1, 3), torch.cat(cs))

    R0 = (runners, cplans, plans, init)

    # gpu_launches: kernels of ONE bench step, counted on an eager (non-graph) pass of identical work
    eager = [ps.StepRunner(model, [dl0[i] for i in idx], True, False, use_graph=False) for idx in chunks[:1]]
    _lib.COUNTS.clear()
    eager[0].step(*coefs[0], None)
    launches_per_step = _lib.launch_count() * len(chunks) * args.inference_steps
    _lib.COUNTS.clear()
    with torch.no_grad():
        zt = torch.zeros(len(chunks[0]))
        conf.run_plan(cplans[0], {'tr': zt, 'rot': zt, 'tor': zt, 'sc_tor': zt})
    launches_per_step += _lib.launch_count() * len(chunks)
    del eager
    for _ in range(args.warmup):
        resident_step()
    flush.fill_(1)
    sampler = ClockSampler(local)
    sampler.start()
    _lib.COUNTS.clear()
    barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    if args.profile_range:
        torch.cuda.profiler.start()
    ev0.record()
    for _ in range(args.steps):
        last = resident_step()
        flush.fill_(0)                           # L2 flush between timed iterations (256 MiB > 126 MB L2)
    ev1.record()
    barrier()
    if args.profile_range:
        torch.cuda.profiler.stop()
    if rank == 0 and args.dump_outputs is not None:
        # ligand poses and confidences of every rank (the gathered result), side-chain atoms of this rank's samples
        dump_outputs(args.dump_outputs, {'ligand_pos': last[0], 'confidence': last[1], 'rank_order': last[2],
                                         'atom_pos': torch.cat([pl.atom_pos for pl in plans]).reshape(N, -1, 3)})
    ms = ev0.elapsed_time(ev1) / args.steps
    launches = launches_per_step
    sampler.stop_flag = True
    if world > 1:
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    value = total_samples / (ms / 1000.0)

    # ---- roofline of the dominant kernel: instrumented forward (events around every fused conv launch) -----
    roof = None
    if rank == 0:
        peak_tf, hbm, peak_src = peaks()
        pl = plans[0]
        ct = {k: torch.full((len(chunks[0]),), 0.5) for k in ('tr', 'rot', 'tor', 'sc_tor')}
        model.profile = []
        with torch.no_grad():
            model.run_plan(pl, ct)
        torch.cuda.synchronize()
        # the HBM-type kernels of the forward (BASELINE.json's metric names GB/s): events around each launch of a second
        # instrumented forward on ONE stream (the edge-set chains normally run on side streams), algorithmic bytes / time
        prof_conv, model.profile = model.profile, None
        model.profile_small = []
        with torch.no_grad():
            model.run_plan(pl, ct)
        torch.cuda.synchronize()
        small = {}
        for name, a, b, nbytes in model.profile_small:
            d = small.setdefault(name, [0, 0.0, 0.0])
            d[0] += 1
            d[1] += a.elapsed_time(b)
            d[2] += nbytes()
        model.profile_small = None
        model.profile = prof_conv
        hbm_kernels = {k: {'launches': n, 'avg_us': 1e3 * ms_ / n, 'algorithmic_gbs': by / (ms_ * 1e-3) / 1e9, 'frac_of_hbm_peak': by / (ms_ * 1e-3) / 1e9 / hbm}
                       for k, (n, ms_, by) in small.items() if ms_ > 0}
        tot_ms, tot_fl, tot_bytes, n_l, li = 0.0, 0.0, 0.0, 0, 0
        from diffdock_pocket_b200 import tp as tpmod
        dims = [tpmod.irreps_dim(tpmod.parse_irreps(q)) for q in model.irrep_seq]
        for (e0, e1, convs) in model.profile:
            tot_ms += e0.elapsed_time(e1)
            tot_fl += sum(conv_flops(ns, w_numel) * int(es.n_dev.item()) for (w_numel, es, ns) in convs)
            tot_bytes += sum(conv_bytes(ns, dims[min(li, 3)], int(es.n_dev.item())) for (w_numel, es, ns) in convs)
            li += 1
            n_l += 1
        model.profile = None
        ach = tot_fl / (tot_ms * 1e-3) / 1e12 if tot_ms > 0 else 0.0
        # DRAM bytes of one conv launch (dram__bytes_read + write, ncu --set full of the grouped layer-3 launch of this
        # same batch: profiles/r1_ncu_umma_v27_summary.txt); far below the algorithmic 1.2 kB/edge because gathered
        # node rows and the weight image are served by L2
        traffic, traffic_src = ncu_traffic(args)
        roof = {'bound': 'tensor', 'achieved': ach, 'peak': peak_tf, 'unit': 'TFLOP/s', 'frac': ach / peak_tf, 'traffic': traffic,
                'kernel': 'tpconv_umma_kernel' if args.mode != 'fp32' else 'tpconv_fp32_kernel', 'launches_measured': n_l,
                'peak_source': peak_src, 'conv_share_of_forward_ms': tot_ms, 'traffic_source': traffic_src,
                # BASELINE.json's metric also names "TP-conv GB/s": the fused kernel's ALGORITHMIC bytes (SURVEY 8(d): edge
                # embedding + two scalar blocks + gathered features + indices per edge, output rows once) over its time
                'algorithmic_gbs': tot_bytes / (tot_ms * 1e-3) / 1e9 if tot_ms > 0 else 0.0, 'hbm_peak_gbs': hbm,
                'hbm_kernels': hbm_kernels}
    # e2e: same metric through sampling() with host buffers
    n_e2e = max(3, min(args.steps, 5))
    e2e_inputs = [copy.deepcopy(dl0) for _ in range(n_e2e + 2)]      # host graphs (sampling() updates them in place)
    for _ in range(2):                                               # untimed: lazy initialisation, allocator, page cache
        e2e_step(e2e_inputs.pop())
    # the harness keeps n_e2e + 2 deep-copied input sets (hundreds of graphs, thousands of tensor objects) alive; a generation-2
    # pass of Python's cyclic GC over them costs 50-200 ms whenever it happens to fire inside the timed region (measured:
    # scripts/dbg/e2e_calls.py).  They are the harness's objects, not the path's: collect now and freeze them out of the GC.
    import gc
    gc.collect()
    gc.freeze()
    barrier()
    b0 = model.static_h2d_bytes + conf.static_h2d_bytes
    t0 = time.time()
    for _ in range(n_e2e):
        e2e_step(e2e_inputs.pop())
    barrier()
    e2e_ms = (time.time() - t0) * 1000.0 / n_e2e
    static_bytes_per_call = (model.static_h2d_bytes + conf.static_h2d_bytes - b0) / n_e2e
    gc.unfreeze()
    if world > 1:
        t = torch.tensor([e2e_ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_ms = float(t.item())
    # bytes sampling() copies host->device per call: positions + index / edge tensors of every plan, the static node features
    # as counted by the model (once per complex, not per sample), the per-step scalar / noise rows
    # (a call that re-uses the resident state of an earlier call on the same complex -- sampling.LAST_CALL -- uploads only the
    # start poses; the index / edge tensors travel when the plans are built)
    from diffdock_pocket_b200 import sampling as _S
    per_call = (lambda pl: (pl.lig_pos, pl.atom_pos)) if _S.LAST_CALL.get('plan_reused') else \
        (lambda pl: (pl.lig_pos, pl.atom_pos, pl.rec_pos, pl.bond_attr, pl.lig_batch, pl.rec_batch, pl.atom_batch, pl.es['rr'].edge,
                     pl.es['ar'].edge, pl.es['ll'].edge[:pl.Eb]))
    h2d = sum(t.numel() * t.element_size() for pl in plans for t in per_call(pl))
    h2d += static_bytes_per_call + sum(pl.step_in.numel() * 4 for pl in plans) * args.inference_steps
    d2h = sum((pl.NL + pl.NA) * 12 for pl in plans) + N * 4

    # ---- fp32-grade leg: the same resident step with the bf16x3 tensor-core conv (hi/lo split operands, fp32-grade products:
    # the mode that meets the 1e-4 per-layer gate), so that the driver's record carries both numbers
    fp32_grade = None
    if args.mode == 'bf16' and not args.no_fp32_grade:
        model.conv_mode = conf.conv_mode = 'bf16x3'
        R3 = build_resident()
        for _ in range(max(1, min(args.warmup, 2))):
            resident_step(*R3)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        n3 = max(1, min(args.steps, 3))
        e0.record()
        for _ in range(n3):
            resident_step(*R3)
            flush.fill_(0)
        e1.record()
        barrier()
        ms3 = e0.elapsed_time(e1) / n3
        if world > 1:
            t = torch.tensor([ms3], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms3 = float(t.item())
        fp32_grade = {'value': total_samples / (ms3 / 1000.0), 'unit': 'poses/s', 'ms_per_step': ms3, 'conv_mode': 'bf16x3', 'steps': n3}
        del R3
        model.conv_mode = conf.conv_mode = args.mode

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        v, dt = cpu_arm(args, args.cpu_samples, args.cpu_steps, os.cpu_count())
        cpu = {'value': v, 'unit': 'poses/s', 'cores': os.cpu_count(), 'kind': 'port',
               'sample': f'{args.cpu_samples} samples x {args.cpu_steps} of {args.inference_steps} steps ({dt:.1f} s), scaled linearly'}
    if rank == 0:
        print(json.dumps({
            'metric': 'docked poses/sec (20-step reverse diffusion)', 'value': value, 'unit': 'poses/s', 'n_gpus': world,
            'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': ms, 'higher_is_better': True, 'scaling': args.scaling,
            'vs_baseline': None, 'dtype': {'bf16': 'bf16', 'bf16x3': 'bf16x3 (fp32-grade)', 'fp32': 'f32'}[args.mode], 'data': 'synthetic',
            'config': {'workload': (f'{args.workload}: {args.samples} samples, batch {args.batch_size}, {args.inference_steps} reverse-diffusion steps + confidence pass, per GPU (BASELINE.json configs[1])'
                                    if args.scaling == 'weak' else
                                    f'{args.workload}: {total_samples} samples of ONE complex split over {world} GPU(s) ({args.samples} on rank 0), batch {args.batch_size}, {args.inference_steps} steps + confidence pass (BASELINE.json configs[1], strong scaling)'),
                       'weights': 'random init of the README big score model (ns=60 nv=10 6 layers lmax=1) + confidence model (no checkpoint offline)', 'conv_mode': args.mode, 'streams': len(streams),
                       'l2': 'weights + activations (>400 MB) exceed L2; 256 MiB flush between timed iterations'},
            'clocks': sampler.summary(), 'gpu_launches': launches,
            'fp32_grade': fp32_grade,
            'e2e': {'value': total_samples / (e2e_ms / 1000.0), 'unit': 'poses/s', 'h2d_bytes_per_step': int(h2d), 'd2h_bytes_per_step': int(d2h),
                    'resident_state_reused': bool(_S.LAST_CALL.get('plan_reused'))},
            'roofline': roof, 'cpu_baseline': cpu}))
    if world > 1:
        dist.destroy_process_group()


if __name__ == '__main__':
    main()
