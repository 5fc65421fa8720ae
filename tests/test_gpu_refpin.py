"""GPU parity against outputs of the REFERENCE'S OWN MODULES (``tests/golden/ref_*.npz``, written by
``scripts/make_ref_fixtures.py`` from the unmodified ``/root/reference`` files; see ``tests/test_reference_pin.py``).

Gates are the north-star ones: edge lists bit-exact; per-layer features and the four scores within 1e-4 (fp32 CUDA-core
conv and the bf16x3 tensor-core conv) or 1e-2 (single-pass bf16 tensor-core conv), measured both against the global
maximum (``rel_err``) and per feature channel (``rel_err_cols``); final poses after a full 20-step run of the README big
model within 0.1 A RMSD.  Nothing here imports ``/root/reference``.
"""
import copy
import os
from functools import partial

import numpy as np
import pytest
import torch

import _common as T
from diffdock_pocket_b200 import diffusion_utils as du, inputs, sampling as ps, utils
from oracle import refpin

pytestmark = pytest.mark.gpu
DEV = torch.device('cuda:0')
TOL = {'fp32': 1e-4, 'bf16x3': 1e-4, 'bf16': 1e-2}
_MODELS = {}


def _z(name):
    return np.load(os.path.join(T.GOLD, name))


def _models(key, sa, ca, seed):
    if key not in _MODELS:
        m, c, sa, ca = utils.build_models(DEV, score_args=sa, conf_args=ca, seed=seed)
        _MODELS[key] = (m, c, sa, ca)
    return _MODELS[key]


def _big():
    return _models('big', utils.score_model_args(), utils.confidence_model_args(), 0)


def _small(**over):
    kw = dict(ns=16, nv=4, num_conv_layers=4, sigma_embed_dim=32, distance_embed_dim=32, cross_distance_embed_dim=32)
    kw.update(over)
    seed = 3 if over else 0
    return _models(('small', tuple(sorted(over.items()))), utils.score_model_args(**kw),
                   utils.confidence_model_args(ns=8, nv=2, num_conv_layers=3, sh_lmax=kw.get('sh_lmax', 1)), seed)


def _lists_from(z, g, prefix):
    dl = []
    for i in range(z[f'{prefix}_lig_pos'].shape[0]):
        x = copy.deepcopy(g)
        x['ligand'].pos = torch.from_numpy(z[f'{prefix}_lig_pos'][i].copy())
        if f'{prefix}_atom_pos' in z:
            x['atom'].pos = torch.from_numpy(z[f'{prefix}_atom_pos'][i].copy())
        dl.append(x)
    return dl


def _run(m, dl, t, mode):
    b = T.batch_at(dl, t)
    m.conv_mode = mode
    try:
        with torch.no_grad():
            pl = m.make_plan(copy.deepcopy(b))
            out = [o.clone() for o in m.run_plan(pl, b.complex_t, return_layers=True)]
    finally:
        m.conv_mode = 'fp32'
    return pl, out


def _check(z, tag, pl, out, mode):
    tol = TOL[mode]
    for nm in ('ll', 'lr', 'la', 'aa'):                                            # graphs bit-exact with the reference run
        assert np.array_equal(pl.es[nm].edge_index().cpu().numpy().astype(np.int32), z[f'{tag}_{nm}']), nm
    sa_, sr_, sl_ = (int(s) for s in z[f'{tag}_strides'])             # rows stored: every sa_-th atom, sr_-th residue, sl_-th ligand atom
    worst = 0.0
    for l, (gl, ga, gr) in enumerate(pl.last_layers):
        want = z[f'{tag}_lig_L{l}']
        e, ec = T.rel_err(gl[::sl_, :want.shape[1]], want), T.rel_err_cols(gl[::sl_, :want.shape[1]], want)
        assert e < tol and ec < 4 * tol, (mode, 'lig', l, e, ec)
        worst = max(worst, e)
        if f'{tag}_atom_L{l}' in z:
            want = z[f'{tag}_atom_L{l}']
            e, ec = T.rel_err(ga[::sa_, :want.shape[1]], want), T.rel_err_cols(ga[::sa_, :want.shape[1]], want)
            assert e < tol and ec < 4 * tol, (mode, 'atom', l, e, ec)
        if f'{tag}_rec_L{l}' in z:
            want = z[f'{tag}_rec_L{l}']
            e, ec = T.rel_err(gr[::sr_, :want.shape[1]], want), T.rel_err_cols(gr[::sr_, :want.shape[1]], want)
            assert e < tol and ec < 4 * tol, (mode, 'rec', l, e, ec)
    for k, v in zip(('tr', 'rot', 'tor', 'sc'), out):
        assert v.numel() == z[f'{tag}_{k}'].size, k
        e = T.rel_err(v, z[f'{tag}_{k}'])
        assert e < tol, (mode, k, e)
    return worst


@pytest.mark.parametrize('mode', ['fp32', 'bf16x3', 'bf16'])
@pytest.mark.parametrize('tag,t', [('t70', 0.7), ('t05', 0.05)])
def test_big_model_forward_vs_reference(tag, t, mode):
    """README big model on two 3dpf holo graphs: models/all_atom_score_model.py:238-436 executed unmodified on the CPU vs the
    CUDA path through the C ABI."""
    z = _z('ref_forward_big.npz')
    m, c, sa, ca = _big()
    np.testing.assert_allclose(refpin.weight_checksum(m.state_dict()), z['big_weight_checksum'], rtol=1e-12)
    dl = _lists_from(z, T.graph('3dpf_holo'), 'big')
    pl, out = _run(m, dl, t, mode)
    _check(z, 'big_' + tag, pl, out, mode)


def test_big_confidence_and_forward_side_effects_vs_reference():
    z = _z('ref_forward_big.npz')
    m, c, sa, ca = _big()
    dl = _lists_from(z, T.graph('3dpf_holo'), 'big')
    with torch.no_grad():
        conf = c(T.batch_at(dl, 0.0))
    assert T.rel_err(conf, z['big_confidence']) < 1e-4
    b = T.batch_at(dl[:1], 0.3)
    with torch.no_grad():
        m(b)
    # what forward() leaves on the batch (all_atom_score_model.py:373,453,495,520,530)
    # (fp32 sin / cos of arguments up to embedding_scale * t = 300: the device's and the host's libm differ by ~1e-5)
    assert T.rel_err(b['ligand'].node_sigma_emb, z['side_lig_node_sigma_emb']) < 1e-4
    assert T.rel_err(b['receptor'].node_sigma_emb[:4], z['side_rec_node_sigma_emb']) < 1e-4
    assert T.rel_err(b['atom'].node_sigma_emb[:4], z['side_atom_node_sigma_emb']) < 1e-4
    assert T.rel_err(b.graph_sigma_emb, z['side_graph_sigma_emb']) < 1e-4
    assert np.array_equal(b['atom', 'atom'].edge_index.cpu().numpy().astype(np.int32), z['side_aa_edge_index'])


@pytest.mark.parametrize('name,mode', [('small', 'fp32'), ('small', 'bf16x3'), ('small', 'bf16'), ('lmax2', 'fp32'), ('lmax2', 'bf16x3'), ('lmax2', 'bf16')])
def test_small_models_forward_vs_reference(name, mode):
    z = _z('ref_forward_small.npz')
    m, c, sa, ca = _small(**(dict(sh_lmax=2, num_conv_layers=3) if name == 'lmax2' else {}))
    np.testing.assert_allclose(refpin.weight_checksum(m.state_dict()), z[f'{name}_weight_checksum'], rtol=1e-12)
    g = inputs.synthetic_complex(7, n_lig=18, n_res=36, flexible_residues=3)
    dl = _lists_from(z, g, name)
    pl, out = _run(m, dl, 0.35, mode)
    _check(z, name, pl, out, mode)
    with torch.no_grad():
        conf = c(T.batch_at(dl, 0.0))
    assert T.rel_err(conf, z[f'{name}_confidence']) < 1e-4


@pytest.mark.parametrize('mode', ['fp32', 'bf16x3', 'bf16'])
@pytest.mark.parametrize('case', list(refpin.CONV_CASES))
def test_conv_operator_vs_reference_score_model_py(case, mode):
    """models/score_model.py:84-125 (TensorProductConvLayer with FasterTensorProduct, and with the e3nn FullyConnectedTensorProduct
    over lmax-2 harmonics) executed unmodified vs the operator-level drop-in in every conv mode.  The tensor-core kernel takes the
    trunk shapes (sh_lmax 1 and 2); 'final' (2x1o + 2x1e outputs) is not a shape it is built for and must fall back to the fp32
    kernel rather than fail."""
    from diffdock_pocket_b200.score_model import TensorProductConvLayer
    from diffdock_pocket_b200 import tp as tpmod
    z = _z('ref_ops.npz')
    in_ir, out_ir, nf, faster, sh_ir = refpin.CONV_CASES[case]
    conv = TensorProductConvLayer(in_ir, sh_ir, out_ir, nf, residual=False, batch_norm=True, faster=faster)
    refpin.np_fill(conv, 7)
    conv = conv.to(DEV).eval()
    assert tpmod.umma_supported(conv.tp.spec, nf // 3) == (case != 'final')
    x, ei, ea, sh = refpin.conv_inputs(case)
    conv.conv_mode = mode
    with torch.no_grad():
        got = conv(x.to(DEV), ei.to(DEV), ea.to(DEV), sh.to(DEV), out_nodes=x.shape[0] + 3)
    want = z[f'conv_{case}_out']
    tol = TOL[mode] if case != 'final' else 1e-4
    assert T.rel_err(got, want) < tol and T.rel_err_cols(got, want) < 4 * tol, (case, mode, T.rel_err(got, want), T.rel_err_cols(got, want))


def test_rigid_ligand_forward_vs_reference():
    z = _z('ref_forward_small.npz')
    m, c, sa, ca = _small()
    g = inputs.synthetic_complex(21, n_lig=3, n_res=30, flexible_residues=0)
    dl = _lists_from(z, g, 'rigid')
    with torch.no_grad():
        out = m(T.batch_at(dl, 0.4))
    assert out[2].numel() == 0 and out[3].numel() == 0
    assert T.rel_err(out[0], z['rigid_tr']) < 1e-4 and T.rel_err(out[1], z['rigid_rot']) < 1e-4


def test_pose_update_kernel_vs_reference_modify_conformer():
    """utils/diffusion_utils.py:37-70 + utils/torsion.py:68-94,251-278 + utils/geometry.py:209-243 executed unmodified vs the
    fused pose-update kernel."""
    z = _z('ref_ops.npz')
    g = T.graph('3dpf_holo')
    dl = []
    for i in range(3):
        x = copy.deepcopy(g)
        x['ligand'].pos = torch.from_numpy(z['pose_lig0'][i].copy())
        x['atom'].pos = torch.from_numpy(z['pose_atom0'][i].copy())
        dl.append(x)
    tr, rot, tor, sc = refpin.pose_inputs(g)
    st = du.PoseState(dl, DEV)
    f = lambda a: torch.from_numpy(a.reshape(-1)).to(DEV)
    st.update((1, 0, 1, 0, 1, 0, 1, 0), f(tr), f(rot), f(tor), f(sc))
    st.write_back(dl)
    for i, x in enumerate(dl):
        assert float(np.abs(x['ligand'].pos.numpy() - z['pose_lig1'][i]).max()) < 2e-4
        assert float(np.abs(x['atom'].pos.numpy() - z['pose_atom1'][i]).max()) < 2e-4


def _rmsd(a, b):
    return float(np.sqrt(((np.asarray(a) - np.asarray(b)) ** 2).sum(-1).mean()))


@pytest.mark.parametrize('mode', ['fp32', 'bf16x3', 'bf16'])
def test_sampler_small_model_vs_reference_sampling_py(mode):
    """utils/sampling.py:70-286 executed unmodified (seeded CPU noise stream incl. the per-step DataLoader seed draw) vs
    ``sampling()`` here: low-temperature SDE, ODE, and no_final_step_noise variants."""
    z = _z('ref_sampling_small.npz')
    m, c, sa, ca = _small()
    np.testing.assert_allclose(refpin.weight_checksum(m.state_dict()), z['weight_checksum'], rtol=1e-12)
    g = inputs.synthetic_complex(5, n_lig=20, n_res=40, flexible_residues=3)
    flex = g['flexResidues'].subcomponents.unique().numpy()
    m.conv_mode = mode
    try:
        for prefix, steps, bs, seed, kw in (('', 6, 3, 11, refpin.TEMPS), ('ode_', 4, 2, 12, dict(ode=True)),
                                            ('nofinal_', 4, 5, 13, dict(no_final_step_noise=True))):
            dl = []
            for i in range(5):
                x = copy.deepcopy(g)
                x['ligand'].pos = torch.from_numpy(z['lig_pos0'][i].copy())
                x['atom'].pos = torch.from_numpy(z['atom_pos0'][i].copy())
                dl.append(x)
            sch = du.get_t_schedule('expbeta', steps)
            torch.manual_seed(seed)
            trace = []
            out, conf = ps.sampling(dl, m, steps, sch, sch, sch, sch, DEV, partial(du.t_to_sigma, args=sa), sa, confidence_model=c,
                                    filtering_model_args=ca, batch_size=bs, trace=trace, **kw)
            for i, x in enumerate(out):
                r1 = _rmsd(x['ligand'].pos.cpu().numpy(), z[prefix + 'lig_pos'][i])
                r2 = _rmsd(x['atom'].pos.cpu().numpy()[flex], z[prefix + 'atom_pos'][i][flex])
                assert r1 < 0.1 and r2 < 0.1, (mode, prefix, i, r1, r2)
            assert T.rel_err(conf, z[prefix + 'confidence']) < 10 * TOL[mode], (mode, prefix)
            if prefix == '':
                for k, v in zip(('tr', 'rot', 'tor', 'sc'), trace[0]):
                    assert T.rel_err(v, z[f'step0_{k}']) < TOL[mode], (mode, k)
    finally:
        m.conv_mode = 'fp32'


@pytest.mark.parametrize('mode', ['fp32', 'bf16x3', 'bf16'])
def test_full_size_sampling_vs_reference(mode):
    """BASELINE configs[1] shape: 3dpf ESMFold apo pocket with 7 flexible residues, README big model (ns=60, nv=10, 6 layers),
    20 reverse-diffusion steps with inference.py's default temperatures, 8 samples in mini-batches of 3 -- the reference's
    own ``sampling()`` on the CPU vs the CUDA path: every final ligand and flexible side-chain pose within 0.1 A RMSD."""
    z = _z('ref_sampling_full.npz')
    m, c, sa, ca = _big()
    np.testing.assert_allclose(refpin.weight_checksum(m.state_dict()), z['weight_checksum'], rtol=1e-12)
    g = T.graph('3dpf_apo')
    flex = g['flexResidues'].subcomponents.unique().numpy()
    n = z['lig_pos0'].shape[0]
    dl = []
    for i in range(n):
        x = copy.deepcopy(g)
        x['ligand'].pos = torch.from_numpy(z['lig_pos0'][i].copy())
        x['atom'].pos = torch.from_numpy(z['atom_pos0'][i].copy())
        dl.append(x)
    steps, bs = int(z['steps']), int(z['batch_size'])
    sch = du.get_t_schedule('expbeta', steps)
    torch.manual_seed(int(z['seed']))
    trace = []
    m.conv_mode = mode
    try:
        out, conf = ps.sampling(dl, m, steps, sch, sch, sch, sch, DEV, partial(du.t_to_sigma, args=sa), sa, confidence_model=c,
                                filtering_model_args=ca, batch_size=bs, trace=trace, **refpin.TEMPS)
    finally:
        m.conv_mode = 'fp32'
    for k, v in zip(('tr', 'rot', 'tor', 'sc'), trace[0]):
        assert T.rel_err(v, z[f'step0_{k}']) < TOL[mode], (mode, k, T.rel_err(v, z[f'step0_{k}']))
    worst = 0.0
    for i, x in enumerate(out):
        r1 = _rmsd(x['ligand'].pos.cpu().numpy(), z['lig_pos'][i])
        r2 = _rmsd(x['atom'].pos.cpu().numpy()[flex], z['atom_pos'][i][flex])
        worst = max(worst, r1, r2)
        assert r1 < 0.1 and r2 < 0.1, (mode, i, r1, r2)
    moved = _rmsd(z['lig_pos'], z['lig_pos0'])
    assert moved > 1.0                                                  # the run did move the ligands by Angstroms
    assert T.rel_err(conf, z['confidence']) < 10 * TOL[mode], (mode, T.rel_err(conf, z['confidence']))
    order_ref = np.argsort(-z['confidence'])
    print(f'full-size sampling [{mode}]: worst RMSD {worst:.4f} A (ligands moved {moved:.2f} A), top-1 {int(order_ref[0])} vs '
          f'{int(np.argsort(-conf.cpu().numpy())[0])}')


@pytest.mark.gpu
@pytest.mark.parametrize('case', list(refpin.CONV_CASES))
def test_conv_backward_vs_reference_autograd(case):
    """Training path (SURVEY 8(f) row 3): gradients of the conv operator -- node features, edge attributes, edge harmonics, both
    Linears of the edge MLP -- from ddp_tp_backward + library GEMMs against PyTorch autograd through the reference's own
    TensorProductConvLayer (models/score_model.py:84-125; fixture tests/golden/ref_conv_grads.npz, scripts/make_ref_fixtures.py)."""
    from diffdock_pocket_b200.score_model import TensorProductConvLayer
    from test_reference_pin import _conv_grads, check_conv_grads
    in_ir, out_ir, nf, faster, sh_ir = refpin.CONV_CASES[case]
    conv = TensorProductConvLayer(in_ir, sh_ir, out_ir, nf, residual=False, batch_norm=True, faster=faster)
    refpin.np_fill(conv, 7)
    conv = conv.to(DEV).eval()
    check_conv_grads(_conv_grads(conv, case), case, 2e-4)


def test_asynchronous_noise_schedule_vs_reference():
    """asyncronous_noise_schedule=True (sigma embeddings at set_time's `t`): forward through forward(data) and a 3-step sampling()
    run with a separate t_schedule against the reference's own model / sampler (tests/golden/ref_async.npz)."""
    from functools import partial
    from test_reference_pin import async_case
    from diffdock_pocket_b200 import diffusion_utils as du, sampling as ps
    from diffdock_pocket_b200.hetero import Batch
    m, sa, dl, z = async_case(DEV)
    m.conv_mode = 'fp32'
    g = inputs.synthetic_complex(3, n_lig=16, n_res=30, flexible_residues=2)
    pl_dl = []
    for o in dl:                                                      # product-side graphs at the oracle-randomised start poses
        x = copy.deepcopy(g)
        x['ligand'].pos, x['atom'].pos = o['ligand'].pos.clone(), o['atom'].pos.clone()
        pl_dl.append(x)
    b = Batch.from_data_list(copy.deepcopy(pl_dl))
    du.set_time(b, 0.9, 0.4, 0.4, 0.4, 0.4, len(dl), True, True, DEV)
    with torch.no_grad():
        out = m(b)
    for k, v in zip(('tr', 'rot', 'tor', 'sc'), out):
        assert T.rel_err(v, z[f'fwd_{k}']) < 1e-4, (k, T.rel_err(v, z[f'fwd_{k}']))
    steps = 3
    sch = du.get_t_schedule('expbeta', steps)
    torch.manual_seed(8)
    got, _ = ps.sampling(copy.deepcopy(pl_dl), m, steps, sch, sch, sch, sch, DEV, partial(du.t_to_sigma, args=sa), sa, batch_size=2,
                         asyncronous_noise_schedule=True, t_schedule=z['t_schedule'])
    assert (torch.stack([o['ligand'].pos.cpu() for o in got]) - torch.from_numpy(z['lig_pos'])).abs().max() < 5e-3
    assert (torch.stack([o['atom'].pos.cpu() for o in got]) - torch.from_numpy(z['atom_pos'])).abs().max() < 5e-3
