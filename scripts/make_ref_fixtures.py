"""Generate ``tests/golden/ref_*.npz`` by EXECUTING THE REFERENCE'S OWN MODULES (run HERE, where /root/reference exists).

``oracle.refshim.load()`` imports the unmodified ``models/layers.py``, ``models/score_model.py``,
``models/all_atom_score_model.py``, ``utils/{geometry,torsion,diffusion_utils,so3,torus,sampling,utils}.py`` from
``/root/reference`` with the oracle's restatements injected for the un-vendored third-party packages; every array
written below is an output of those reference modules.  ``tests/test_reference_pin.py`` (CPU) checks the oracle
against them, ``tests/test_gpu_refpin.py`` (GPU) the CUDA path.

    python scripts/make_ref_fixtures.py [tables] [ops] [conv_grads] [async] [forward] [sampling_small] [sampling_full]

(no argument = everything; ``sampling_full`` is the 20-step big-model run, several minutes of CPU.)
The first run imports ``utils/so3.py`` / ``utils/torus.py`` without their ``.npy`` caches: ~9 minutes.
"""
import copy
import os
import sys
import time
from functools import partial

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from diffdock_pocket_b200 import inputs, torus as ptorus, utils as putils  # noqa: E402  (input graphs, seeded weights)
from oracle import e3nn_mini as E, pyg_mini, refpin, refshim  # noqa: E402

GOLD = os.path.join(ROOT, 'tests', 'golden')


def save(name, d):
    path = os.path.join(GOLD, name)
    np.savez_compressed(path, **d)
    print(f'{name}: {os.path.getsize(path) / 1e6:.2f} MB, {len(d)} arrays', flush=True)


def ref_models(R, sa, ca, seed):
    """Reference models built by the reference's ``get_model`` and loaded (strict) with the product's seeded weights."""
    m, c, sa, ca = putils.build_models(torch.device('cpu'), score_args=sa, conf_args=ca, seed=seed, with_confidence=ca is not None)
    dev = torch.device('cpu')
    rm = R.utils.get_model(sa, dev, partial(R.diffusion_utils.t_to_sigma, args=sa), no_parallel=True)
    rm.load_state_dict(m.state_dict(), strict=True)
    rm.eval()
    rc = None
    if ca is not None:
        rc = R.utils.get_model(ca, dev, partial(R.diffusion_utils.t_to_sigma, args=ca), no_parallel=True, confidence_mode=True)
        rc.load_state_dict(c.state_dict(), strict=True)
        rc.eval()
    return rm, rc, sa, ca, refpin.weight_checksum(m.state_dict()), (refpin.weight_checksum(c.state_dict()) if c is not None else None)


def randomized(R, g, n, sa, seed):
    np.random.seed(seed)
    torch.manual_seed(seed)
    dl = [pyg_mini.from_any(g) for _ in range(n)]
    R.sampling.randomize_position(dl, False, False, sa.tr_sigma_max, flexible_sidechains='flexResidues' in g.node_types)
    return dl


def ref_batch(R, dl, t, sa):
    b = pyg_mini.Batch.from_data_list(copy.deepcopy(dl))
    R.diffusion_utils.set_time(b, None, t, t, t, t, len(dl), True, False, torch.device('cpu'))
    return b


def share_torus_table(R):
    """The reference's torus ``score_norm_`` is a Monte-Carlo table from the unseeded global RNG (utils/torus.py:65-75,
    SURVEY F8): parity runs share ONE table -- the product's seeded one -- by data injection (no code is replaced)."""
    R.torus.score_norm_ = ptorus.score_norm_table().copy()


# ------------------------------------------------------------------------------------------------- tables
def make_tables(R):
    d = dict(so3_exp_score_norms=R.so3._exp_score_norms,
             so3_score_norms_sub=R.so3._score_norms[::50, ::40],
             torus_score_sub=R.torus.score_[::25, ::25], torus_p_sub=R.torus.p_[::25, ::25])
    d['torus_score_norm_seed0'] = R.torus.score_norm_seed0_        # Monte-Carlo table of the import under np.random.seed(0)
    eps = np.array([0.01, 0.03, 0.1, 0.5, 1.0, 1.55, 2.0])
    d['so3_eps'] = eps
    d['so3_score_norm'] = R.so3.score_norm(torch.from_numpy(eps)).numpy()
    sg = np.array([0.0094, 0.03, 0.1, 0.5, 1.0, 3.14, 6.0])
    d['torus_sigma'] = sg
    share_torus_table(R)
    d['torus_score_norm_shared'] = R.torus.score_norm(sg)
    save('ref_tables.npz', d)


# ------------------------------------------------------------------------------------------------- operators
def make_ops(R):
    d = {}
    for i, (in_ir, out_ir) in enumerate(refpin.FTP_CASES):                       # models/layers.py:8-85
        tp = R.layers.FasterTensorProduct(in_ir, '1x0e+1x1o', out_ir)
        x, sh, rng = refpin.ftp_inputs(i)
        w = torch.from_numpy(rng.standard_normal((x.shape[0], tp.weight_numel)).astype(np.float32))
        d[f'ftp{i}_numel'] = tp.weight_numel
        d[f'ftp{i}_out'] = tp(x, sh, w).numpy()
    for case, (in_ir, out_ir, nf, faster, sh_ir) in refpin.CONV_CASES.items():   # models/score_model.py:84-125
        conv = R.score_model.TensorProductConvLayer(in_ir, sh_ir, out_ir, nf, residual=False, batch_norm=True, faster=faster)
        refpin.np_fill(conv, 7).eval()
        x, ei, ea, sh = refpin.conv_inputs(case)
        with torch.no_grad():
            d[f'conv_{case}_out'] = conv(x, ei, ea, sh, out_nodes=x.shape[0] + 3).numpy()
            conv.residual = True
            d[f'conv_{case}_out_residual'] = conv(x, ei, ea, sh).numpy()
    rng = np.random.RandomState(5)                                               # utils/geometry.py
    aa = torch.from_numpy(rng.standard_normal((16, 3)).astype(np.float32))
    aa[0] = 0
    aa[1] *= 1e-4
    d['aa_matrix'] = R.geometry.axis_angle_to_matrix(aa).numpy()
    A = torch.from_numpy(rng.standard_normal((3, 37)).astype(np.float32))
    Rm = R.geometry.axis_angle_to_matrix(torch.tensor([0.3, -1.1, 0.7]))
    B = Rm @ A + torch.tensor([[1.0], [-2.0], [0.5]]) + 0.05 * torch.from_numpy(rng.standard_normal((3, 37)).astype(np.float32))
    kr, kt = R.geometry.rigid_transform_Kabsch_3D_torch(A, B)
    d['kabsch_R'], d['kabsch_t'] = kr.numpy(), kt.numpy()
    sa = putils.score_model_args()                                               # utils/diffusion_utils.py
    ts = np.array([1.0, 0.7, 0.35, 0.05, 0.0])
    d['t_to_sigma'] = np.array([R.diffusion_utils.t_to_sigma(t, t, t, t, sa) for t in ts], dtype=np.float64)
    d['t_schedule_expbeta20'] = np.asarray(R.diffusion_utils.get_t_schedule('expbeta', 20, 1, 1, 1))
    d['t_schedule_beta7'] = np.asarray(R.diffusion_utils.get_t_schedule('expbeta', 7, 2.0, 0.5, 0.9))
    emb = R.diffusion_utils.get_timestep_embedding('sinusoidal', 64, 1000)
    d['sinusoidal'] = emb(torch.tensor(ts, dtype=torch.float32)).numpy()
    g = inputs.load_graph_npz(os.path.join(GOLD, '3dpf_holo.npz'), name='3dpf_holo')            # pose updates
    dl = randomized(R, g, 3, sa, seed=4)
    d['pose_lig0'] = torch.stack([x['ligand'].pos for x in dl]).numpy()
    d['pose_atom0'] = torch.stack([x['atom'].pos for x in dl]).numpy()
    tr, rot, tor, sc = refpin.pose_inputs(g)
    for i, x in enumerate(dl):
        R.diffusion_utils.modify_sidechains(x, sc[i])
        R.diffusion_utils.modify_conformer(x, torch.from_numpy(tr[i:i + 1]), torch.from_numpy(rot[i]), tor[i])
    d['pose_lig1'] = torch.stack([x['ligand'].pos for x in dl]).numpy()
    d['pose_atom1'] = torch.stack([x['atom'].pos for x in dl]).numpy()
    b = ref_batch(R, dl, 0.35, sa)                                               # set_time + collate
    d['set_time_lig_tr'] = b['ligand'].node_t['tr'].numpy()
    d['set_time_complex_sc'] = b.complex_t['sc_tor'].numpy()
    d['collate_ll_index'] = b['ligand', 'ligand'].edge_index.numpy()
    d['collate_ar_index'] = b['atom', 'receptor'].edge_index.numpy()
    d['collate_flex_edge_idx'] = b['flexResidues'].edge_idx.numpy()
    d['collate_flex_batch'] = b['flexResidues'].batch.numpy()
    save('ref_ops.npz', d)


# ------------------------------------------------------------------------------------------------- asynchronous noise schedule
ASYNC_KW = dict(ns=16, nv=4, num_conv_layers=4, sigma_embed_dim=32, distance_embed_dim=32, cross_distance_embed_dim=32,
                asyncronous_noise_schedule=True)


def make_async(R):
    """Forward of the reference's all-atom model built with ``asyncronous_noise_schedule=True`` (sigma embeddings read time
    't' of ``set_time``, models/all_atom_score_model.py:370,450,492,517; utils/diffusion_utils.py:158-165) and a 3-step
    sampler run with a ``t_schedule`` different from the noise schedules (utils/sampling.py:116-117)."""
    share_torus_table(R)
    sa = putils.score_model_args(**ASYNC_KW)
    rm, _, sa, _, ws, _ = ref_models(R, sa, None, seed=5)
    g = inputs.synthetic_complex(3, n_lig=16, n_res=30, flexible_residues=2)
    dl = randomized(R, g, 3, sa, seed=6)
    d = {'weights': np.asarray(ws)}
    b = pyg_mini.Batch.from_data_list(copy.deepcopy(dl))
    R.diffusion_utils.set_time(b, 0.9, 0.4, 0.4, 0.4, 0.4, len(dl), True, True, torch.device('cpu'))
    with torch.no_grad():
        out = rm(b)
    for k, v in zip(('tr', 'rot', 'tor', 'sc'), out):
        d[f'fwd_{k}'] = v.numpy()
    steps = 3
    sch = R.diffusion_utils.get_t_schedule('expbeta', steps, 1, 1, 1)
    t_sch = np.asarray(sch) ** 2 * 0.7 + 0.05
    torch.manual_seed(8)
    out, _ = R.sampling.sampling(copy.deepcopy(dl), rm, steps, sch, sch, sch, sch, torch.device('cpu'),
                                 partial(R.diffusion_utils.t_to_sigma, args=sa), sa, batch_size=2, asyncronous_noise_schedule=True,
                                 t_schedule=t_sch)
    d['t_schedule'] = t_sch
    d['lig_pos'] = torch.stack([o['ligand'].pos for o in out]).numpy()
    d['atom_pos'] = torch.stack([o['atom'].pos for o in out]).numpy()
    save('ref_async.npz', d)


# ------------------------------------------------------------------------------------------------- conv backward
ROW_STRIDE = {'ea': 8, 'w1': 8}


def sums(g):
    g = g.astype(np.float64)
    return np.array([g.sum(), np.abs(g).sum(), (g * g).sum()])


def make_conv_grads(R):
    """Gradients of the reference's own ``TensorProductConvLayer`` (models/score_model.py:84-125 over models/layers.py /
    the FCTP restatement) by PyTorch autograd, as ``loss.backward()`` computes them in utils/training.py:147-191: with
    respect to the node features, edge attributes, edge harmonics and both Linears of the edge MLP.  The [weight_numel,
    hidden] gradient of the second Linear is stored as a strided sample plus its sums (7 MB per case otherwise); those of
    the edge attributes and of the first Linear as every ROW_STRIDE-th row plus their sums and shape (the file stays below
    1 MB)."""
    d = {}
    for case, (in_ir, out_ir, nf, faster, sh_ir) in refpin.CONV_CASES.items():
        conv = R.score_model.TensorProductConvLayer(in_ir, sh_ir, out_ir, nf, residual=False, batch_norm=True, faster=faster)
        refpin.np_fill(conv, 7).eval()
        x, ei, ea, sh = refpin.conv_inputs(case)
        xs, eas, shs = (t.clone().requires_grad_(True) for t in (x, ea, sh))
        out = conv(xs, ei, eas, shs, out_nodes=x.shape[0] + 3)
        probe = torch.from_numpy(np.random.RandomState(11).standard_normal(tuple(out.shape)).astype(np.float32))
        gs = torch.autograd.grad((out * probe).sum(), [xs, eas, shs, conv.fc[0].weight, conv.fc[0].bias, conv.fc[3].weight, conv.fc[3].bias])
        for name, g in zip(('x', 'ea', 'sh', 'w1', 'b1', 'w2', 'b2'), gs):
            g = g.detach().numpy()
            if name == 'w2':
                d[f'grad_{case}_w2_sample'] = g.reshape(-1)[::97].copy()
                d[f'grad_{case}_w2_sums'] = sums(g)
            elif name in ROW_STRIDE:
                key = f'grad_{case}_{name}'
                d[key] = g[::ROW_STRIDE[name]].copy()
                d[key + '_stride'], d[key + '_shape'], d[key + '_sums'] = np.array(ROW_STRIDE[name]), np.array(g.shape), sums(g)
            else:
                d[f'grad_{case}_{name}'] = g
    save('ref_conv_grads.npz', d)


# ------------------------------------------------------------------------------------------------- forward
def run_forward(R, rm, b):
    cap = refpin.Capture(rm)
    with torch.no_grad():
        out = rm(b)
    cap.close()
    return out, cap


def pack_forward(d, tag, out, cap, atom_stride=50, rec_stride=8, lig_stride=2):
    """Per-layer features as every n-th row (strides stored with them) so that each fixture file stays below 1 MB."""
    for k, v in zip(('tr', 'rot', 'tor', 'sc'), out):
        d[f'{tag}_{k}'] = v.numpy()
    for nm in ('ll', 'lr', 'la', 'aa'):
        d[f'{tag}_{nm}'] = cap.rec[nm].numpy().astype(np.int32)
    for l, (lig, atom, rec) in enumerate(cap.layers()):
        d[f'{tag}_lig_L{l}'] = lig[::lig_stride].numpy()
        if atom is not None:
            d[f'{tag}_atom_L{l}'] = atom[::atom_stride].numpy()
        if rec is not None:
            d[f'{tag}_rec_L{l}'] = rec[::rec_stride].numpy()
    d[f'{tag}_strides'] = np.array([atom_stride, rec_stride, lig_stride])


def make_forward(R):
    share_torus_table(R)
    d = {}
    rm, rc, sa, ca, ws, wc = ref_models(R, putils.score_model_args(), putils.confidence_model_args(), seed=0)
    d['big_weight_checksum'], d['conf_weight_checksum'] = ws, wc
    g = inputs.load_graph_npz(os.path.join(GOLD, '3dpf_holo.npz'), name='3dpf_holo')
    dl = randomized(R, g, 2, sa, seed=0)
    d['big_lig_pos'] = torch.stack([x['ligand'].pos for x in dl]).numpy()
    d['big_atom_pos'] = torch.stack([x['atom'].pos for x in dl]).numpy()
    for tag, t in (('t70', 0.7), ('t05', 0.05)):
        t0 = time.time()
        out, cap = run_forward(R, rm, ref_batch(R, dl, t, sa))
        print(f'big forward t={t}: {time.time() - t0:.1f} s', flush=True)
        pack_forward(d, 'big_' + tag, out, cap)
    b = ref_batch(R, dl, 0.0, ca)
    with torch.no_grad():
        d['big_confidence'] = rc(b).numpy()
    b1 = ref_batch(R, dl[:1], 0.3, sa)                                 # forward() side effects on the batch object
    with torch.no_grad():
        rm(b1)
    d['side_lig_node_sigma_emb'] = b1['ligand'].node_sigma_emb.numpy()
    d['side_rec_node_sigma_emb'] = b1['receptor'].node_sigma_emb[:4].numpy()
    d['side_atom_node_sigma_emb'] = b1['atom'].node_sigma_emb[:4].numpy()
    d['side_graph_sigma_emb'] = b1.graph_sigma_emb.numpy()
    d['side_aa_edge_index'] = b1['atom', 'atom'].edge_index.numpy().astype(np.int32)
    save('ref_forward_big.npz', d)

    d = {}
    for name, over, seed in (('small', {}, 0), ('lmax2', dict(sh_lmax=2, num_conv_layers=3), 3)):
        kw = dict(ns=16, nv=4, num_conv_layers=4, sigma_embed_dim=32, distance_embed_dim=32, cross_distance_embed_dim=32)
        kw.update(over)
        ckw = dict(ns=8, nv=2, num_conv_layers=3, sh_lmax=kw.get('sh_lmax', 1))
        rm, rc, sa, ca, ws, wc = ref_models(R, putils.score_model_args(**kw), putils.confidence_model_args(**ckw), seed=seed)
        d[f'{name}_weight_checksum'] = ws
        g = inputs.synthetic_complex(7, n_lig=18, n_res=36, flexible_residues=3)
        dl = randomized(R, g, 3, sa, seed=1)
        d[f'{name}_lig_pos'] = torch.stack([x['ligand'].pos for x in dl]).numpy()
        d[f'{name}_atom_pos'] = torch.stack([x['atom'].pos for x in dl]).numpy()
        out, cap = run_forward(R, rm, ref_batch(R, dl, 0.35, sa))
        pack_forward(d, name, out, cap, atom_stride=2, rec_stride=1, lig_stride=1)
        with torch.no_grad():
            d[f'{name}_confidence'] = rc(ref_batch(R, dl, 0.0, ca)).numpy()
    g = inputs.synthetic_complex(21, n_lig=3, n_res=30, flexible_residues=0)     # rigid ligand, nothing flexible
    rm, rc, sa, ca, ws, wc = ref_models(R, putils.score_model_args(ns=16, nv=4, num_conv_layers=4, sigma_embed_dim=32, distance_embed_dim=32,
                                                                cross_distance_embed_dim=32),
                                        putils.confidence_model_args(ns=8, nv=2, num_conv_layers=3), seed=0)
    dl = randomized(R, g, 3, sa, seed=1)
    out, cap = run_forward(R, rm, ref_batch(R, dl, 0.4, sa))
    d['rigid_lig_pos'] = torch.stack([x['ligand'].pos for x in dl]).numpy()
    for k, v in zip(('tr', 'rot', 'tor', 'sc'), out):
        d[f'rigid_{k}'] = v.numpy()
    save('ref_forward_small.npz', d)


# ------------------------------------------------------------------------------------------------- sampling
def run_sampling(R, rm, rc, sa, ca, dl, steps, batch_size, seed, **kw):
    sch = R.diffusion_utils.get_t_schedule('expbeta', steps, 1, 1, 1)
    rec = refpin.Recorder(rm)
    torch.manual_seed(seed)
    t0 = time.time()
    out, conf = R.sampling.sampling(data_list=copy.deepcopy(dl), model=rec, inference_steps=steps, tr_schedule=sch, rot_schedule=sch,
                                    tor_schedule=sch, sidechain_tor_schedule=sch, device=torch.device('cpu'),
                                    t_to_sigma=partial(R.diffusion_utils.t_to_sigma, args=sa), model_args=sa, confidence_model=rc,
                                    filtering_model_args=ca, batch_size=batch_size, **kw)
    print(f'reference sampling(): {len(dl)} samples x {steps} steps in {time.time() - t0:.1f} s', flush=True)
    nb = (len(dl) + batch_size - 1) // batch_size
    first = [torch.cat([rec.calls[k][i] for k in range(nb)]) for i in range(4)]
    last = [torch.cat([rec.calls[(steps - 1) * nb + k][i] for k in range(nb)]) for i in range(4)]
    d = dict(lig_pos0=torch.stack([x['ligand'].pos for x in dl]).numpy(), atom_pos0=torch.stack([x['atom'].pos for x in dl]).numpy(),
             lig_pos=torch.stack([x['ligand'].pos for x in out]).numpy(), atom_pos=torch.stack([x['atom'].pos for x in out]).numpy(),
             confidence=conf.numpy(), steps=steps, batch_size=batch_size, seed=seed)
    for k, v in zip(('tr', 'rot', 'tor', 'sc'), first):
        d[f'step0_{k}'] = v.numpy()
    for k, v in zip(('tr', 'rot', 'tor', 'sc'), last):
        d[f'last_{k}'] = v.numpy()
    return d


def make_sampling_small(R):
    share_torus_table(R)
    rm, rc, sa, ca, ws, wc = ref_models(R, putils.score_model_args(ns=16, nv=4, num_conv_layers=4, sigma_embed_dim=32, distance_embed_dim=32,
                                                                cross_distance_embed_dim=32),
                                        putils.confidence_model_args(ns=8, nv=2, num_conv_layers=3), seed=0)
    g = inputs.synthetic_complex(5, n_lig=20, n_res=40, flexible_residues=3)
    dl = randomized(R, g, 5, sa, seed=2)
    d = run_sampling(R, rm, rc, sa, ca, dl, 6, 3, 11, **refpin.TEMPS)
    d['weight_checksum'] = ws
    d_ode = run_sampling(R, rm, rc, sa, ca, dl, 4, 2, 12, ode=True)
    d.update({'ode_' + k: v for k, v in d_ode.items() if k in ('lig_pos', 'atom_pos', 'confidence')})
    d_nf = run_sampling(R, rm, rc, sa, ca, dl, 4, 5, 13, no_final_step_noise=True)
    d.update({'nofinal_' + k: v for k, v in d_nf.items() if k in ('lig_pos', 'atom_pos', 'confidence')})
    save('ref_sampling_small.npz', d)


def make_sampling_full(R, n=8):
    """BASELINE configs[1] at reduced sample count: 3dpf ESMFold apo pocket, 7 flexible residues, README big model,
    20 steps, inference.py's default low-temperature parameters, confidence ranking."""
    share_torus_table(R)
    rm, rc, sa, ca, ws, wc = ref_models(R, putils.score_model_args(), putils.confidence_model_args(), seed=0)
    g = inputs.load_graph_npz(os.path.join(GOLD, '3dpf_apo.npz'), name='3dpf_apo')
    dl = randomized(R, g, n, sa, seed=7)
    d = run_sampling(R, rm, rc, sa, ca, dl, 20, 3, 21, **refpin.TEMPS)
    d['weight_checksum'], d['conf_weight_checksum'] = ws, wc
    save('ref_sampling_full.npz', d)


def main():
    what = sys.argv[1:] or ['tables', 'ops', 'conv_grads', 'async', 'forward', 'sampling_small', 'sampling_full']
    torch.set_num_threads(os.cpu_count())
    t0 = time.time()
    R = refshim.load()
    print(f'reference modules imported in {time.time() - t0:.1f} s', flush=True)
    os.makedirs(GOLD, exist_ok=True)
    for w in what:
        {'tables': make_tables, 'ops': make_ops, 'conv_grads': make_conv_grads, 'async': make_async, 'forward': make_forward, 'sampling_small': make_sampling_small,
         'sampling_full': make_sampling_full}[w](R)


if __name__ == '__main__':
    main()
