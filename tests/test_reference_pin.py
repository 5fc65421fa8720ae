"""The oracle (and the product's host tables / collate) pinned to outputs of the REFERENCE'S OWN MODULES.

``tests/golden/ref_*.npz`` were written by ``scripts/make_ref_fixtures.py``, which imports the unmodified files
of ``/root/reference`` (``oracle/refshim.py``: models/layers.py, models/score_model.py, models/all_atom_score_model.py,
utils/geometry.py, utils/torsion.py, utils/diffusion_utils.py, utils/so3.py, utils/torus.py, utils/sampling.py,
utils/utils.py) and runs them on seeded inputs.  Part 1 re-creates those inputs and checks ``oracle/`` against the
stored reference outputs (runs anywhere).  Part 2 (only where ``/root/reference`` and the table caches exist) executes
the reference live next to the oracle on fresh inputs and verifies that the committed fixtures are reproducible.
"""
import copy
import os
from functools import partial

import numpy as np
import pytest
import torch

import _common as T
from diffdock_pocket_b200 import inputs, so3, torus, utils
from diffdock_pocket_b200.hetero import Batch as ProductBatch
from oracle import diffusion_ref as D, e3nn_mini as E, factory, pyg_mini, refpin, refshim, sampling_ref as S
from oracle.score_model_ref import FasterTensorProduct, TensorProductConvLayer

GOLD = T.GOLD


def _z(name):
    return np.load(os.path.join(GOLD, name))


def _close(a, b, rtol=1e-5, atol=1e-6):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    assert a.shape == b.shape, (a.shape, b.shape)
    np.testing.assert_allclose(a, b, rtol=rtol, atol=atol * max(1.0, float(np.abs(b).max()) if b.size else 1.0))


# =========================================================================================== part 1: fixtures
def test_so3_and_torus_tables_match_the_reference_tables():
    z = _z('ref_tables.npz')
    # utils/so3.py:41-60: the product evaluates the same truncated series with two matmuls
    np.testing.assert_allclose(so3.exp_score_norms(), z['so3_exp_score_norms'], rtol=2e-7)
    np.testing.assert_allclose(so3.score_norm(torch.from_numpy(z['so3_eps'])).numpy(), z['so3_score_norm'], rtol=1e-6)
    # utils/torus.py:19-38: score_ = grad / p on the (sigma, x) grid -- deterministic part, compared on a 201 x 201 sub-grid
    x = 10 ** np.linspace(np.log10(torus.X_MIN), 0, torus.X_N + 1) * np.pi
    sigma = 10 ** np.linspace(np.log10(torus.SIGMA_MIN), np.log10(torus.SIGMA_MAX), torus.SIGMA_N + 1) * np.pi
    shifts = 2 * np.pi * np.arange(-100, 101)
    xs = x[None, ::25] + shifts[:, None]
    for k in range(0, 201, 10):
        s = sigma[25 * k]
        e = np.exp(-xs ** 2 / 2 / s ** 2)
        with np.errstate(invalid='ignore', divide='ignore'):
            row = (xs / s ** 2 * e).sum(0) / e.sum(0)
        ok = np.isfinite(z['torus_score_sub'][k]) & np.isfinite(row)
        assert ok.sum() > 50
        np.testing.assert_allclose(row[ok], z['torus_score_sub'][k][ok], rtol=1e-9, atol=1e-12)
    # utils/torus.py:65-75: score_norm_ is a 10 000-sample Monte-Carlo estimate from the unseeded global RNG (F8); the
    # product's seeded estimator must agree with one seeded draw of the reference's within the estimator's noise
    ref, got = z['torus_score_norm_seed0'], torus.score_norm_table()
    assert ref.shape == got.shape == (5001,)
    rel = np.abs(got - ref) / ref
    assert np.median(rel) < 0.02 and rel.max() < 0.12, (np.median(rel), rel.max())
    # the lookup (utils/torus.py:78-82) on the shared table
    np.testing.assert_allclose(torus.score_norm(z['torus_sigma']), z['torus_score_norm_shared'], rtol=0, atol=0)
    # the oracle's literal restatement of both
    idx = np.array([0, 100, 500, 999])
    np.testing.assert_allclose(D.so3_exp_score_norms(idx), z['so3_exp_score_norms'][idx], rtol=1e-9)


def test_faster_tensor_product_matches_reference_layers_py():
    z = _z('ref_ops.npz')
    for i, (in_ir, out_ir) in enumerate(refpin.FTP_CASES):
        tp = FasterTensorProduct(in_ir, '1x0e+1x1o', out_ir)
        assert tp.weight_numel == int(z[f'ftp{i}_numel'])
        x, sh, rng = refpin.ftp_inputs(i)
        w = torch.from_numpy(rng.standard_normal((x.shape[0], tp.weight_numel)).astype(np.float32))
        _close(tp(x, sh, w).numpy(), z[f'ftp{i}_out'], rtol=1e-5, atol=1e-6)


@pytest.mark.parametrize('case', list(refpin.CONV_CASES))
def test_conv_layer_matches_reference_score_model_py(case):
    z = _z('ref_ops.npz')
    in_ir, out_ir, nf, faster, sh_ir = refpin.CONV_CASES[case]
    conv = TensorProductConvLayer(in_ir, sh_ir, out_ir, nf, residual=False, batch_norm=True, faster=faster)
    refpin.np_fill(conv, 7).eval()
    x, ei, ea, sh = refpin.conv_inputs(case)
    with torch.no_grad():
        _close(conv(x, ei, ea, sh, out_nodes=x.shape[0] + 3).numpy(), z[f'conv_{case}_out'], rtol=2e-5, atol=2e-6)
        conv.residual = True
        _close(conv(x, ei, ea, sh).numpy(), z[f'conv_{case}_out_residual'], rtol=2e-5, atol=2e-6)


def test_geometry_schedules_and_embeddings_match_reference():
    z = _z('ref_ops.npz')
    rng = np.random.RandomState(5)
    aa = torch.from_numpy(rng.standard_normal((16, 3)).astype(np.float32))
    aa[0] = 0
    aa[1] *= 1e-4
    _close(D.axis_angle_to_matrix(aa).numpy(), z['aa_matrix'], rtol=1e-6, atol=1e-7)               # utils/geometry.py:39-86
    A = torch.from_numpy(rng.standard_normal((3, 37)).astype(np.float32))
    Rm = D.axis_angle_to_matrix(torch.tensor([0.3, -1.1, 0.7]))
    B = Rm @ A + torch.tensor([[1.0], [-2.0], [0.5]]) + 0.05 * torch.from_numpy(rng.standard_normal((3, 37)).astype(np.float32))
    kr, kt = D.kabsch(A, B)                                                                        # utils/geometry.py:209-243
    _close(kr.numpy(), z['kabsch_R'], rtol=1e-5, atol=1e-6)
    _close(kt.numpy(), z['kabsch_t'], rtol=1e-5, atol=1e-6)
    sa = utils.score_model_args()
    ts = np.array([1.0, 0.7, 0.35, 0.05, 0.0])
    from diffdock_pocket_b200 import diffusion_utils as du
    for fn in (D.t_to_sigma, du.t_to_sigma):                                                       # utils/diffusion_utils.py:22-34
        np.testing.assert_allclose(np.array([fn(t, t, t, t, sa) for t in ts], dtype=np.float64), z['t_to_sigma'], rtol=1e-14)
    np.testing.assert_allclose(D.get_t_schedule(20), z['t_schedule_expbeta20'], rtol=1e-14)        # :112-117
    np.testing.assert_allclose(du.get_t_schedule('expbeta', 20), z['t_schedule_expbeta20'], rtol=1e-14)
    np.testing.assert_allclose(D.get_t_schedule(7, 2.0, 0.5, 0.9), z['t_schedule_beta7'], rtol=1e-14)
    np.testing.assert_allclose(du.get_t_schedule('expbeta', 7, 2.0, 0.5, 0.9), z['t_schedule_beta7'], rtol=1e-14)
    t32 = torch.tensor(ts, dtype=torch.float32)
    _close(D.sinusoidal_embedding(t32, 64, 1000).numpy(), z['sinusoidal'], rtol=1e-6, atol=1e-7)   # :73-84
    _close(du.sinusoidal_embedding(t32, 64, 1000).numpy(), z['sinusoidal'], rtol=1e-6, atol=1e-7)


def _pose_lists(z):
    g = T.graph('3dpf_holo')
    dl = []
    for i in range(3):
        x = copy.deepcopy(g)
        x['ligand'].pos = torch.from_numpy(z['pose_lig0'][i].copy())
        x['atom'].pos = torch.from_numpy(z['pose_atom0'][i].copy())
        dl.append(x)
    return g, dl


def test_randomize_position_and_pose_updates_match_reference():
    z = _z('ref_ops.npz')
    g = T.graph('3dpf_holo')
    sa = utils.score_model_args()
    dl = T.randomized_list(g, 3, sa, seed=4)                           # utils/sampling.py:16-60 under the same seeds
    for i, x in enumerate(dl):
        _close(x['ligand'].pos.numpy(), z['pose_lig0'][i], rtol=1e-5, atol=1e-6)
        _close(x['atom'].pos.numpy(), z['pose_atom0'][i], rtol=1e-5, atol=1e-6)
    g, dl = _pose_lists(z)
    tr, rot, tor, sc = refpin.pose_inputs(g)
    for i, x in enumerate(dl):                                         # utils/diffusion_utils.py:37-70, utils/torsion.py:68-94,251-278
        D.modify_sidechains(x, sc[i])
        D.modify_conformer(x, torch.from_numpy(tr[i:i + 1]), torch.from_numpy(rot[i]), tor[i])
        assert float(np.abs(x['ligand'].pos.numpy() - z['pose_lig1'][i]).max()) < 2e-5
        assert float(np.abs(x['atom'].pos.numpy() - z['pose_atom1'][i]).max()) < 2e-5
    assert float(np.abs(z['pose_atom1'] - z['pose_atom0']).max()) > 0.5     # the side chains did move


def test_collate_and_set_time_match_reference_run():
    """The product's ``hetero.Batch`` against the batch the reference code saw (``oracle.pyg_mini``: two independent
    restatements of PyG's collate) and the reference's ``set_time``."""
    z = _z('ref_ops.npz')
    g, dl = _pose_lists(z)
    for i, x in enumerate(dl):
        x['ligand'].pos = torch.from_numpy(z['pose_lig1'][i].copy())
        x['atom'].pos = torch.from_numpy(z['pose_atom1'][i].copy())
    from diffdock_pocket_b200 import diffusion_utils as du
    for batch_cls, set_time in ((ProductBatch, lambda b: du.set_time(b, None, 0.35, 0.35, 0.35, 0.35, 3, True, False, torch.device('cpu'))),
                                (pyg_mini.Batch, lambda b: D.set_time(b, 0.35, 0.35, 0.35, 0.35, 3))):
        b = batch_cls.from_data_list(copy.deepcopy(dl))
        set_time(b)
        assert np.array_equal(b['ligand', 'ligand'].edge_index.numpy(), z['collate_ll_index'])
        assert np.array_equal(b['atom', 'receptor'].edge_index.numpy(), z['collate_ar_index'])
        assert np.array_equal(b['flexResidues'].edge_idx.numpy(), z['collate_flex_edge_idx'])
        assert np.array_equal(b['flexResidues'].batch.numpy(), z['collate_flex_batch'])
        assert np.array_equal(b['ligand'].node_t['tr'].numpy(), z['set_time_lig_tr'])
        assert np.array_equal(b.complex_t['sc_tor'].numpy(), z['set_time_complex_sc'])
        assert b.num_graphs == 3


def _oracle_pair(sa, ca, seed):
    m, c, sa, ca = utils.build_models(torch.device('cpu'), score_args=sa, conf_args=ca, seed=seed)
    om = factory.oracle_model(sa, m.state_dict(), so3.score_norm_np, torus.score_norm)
    oc = factory.oracle_model(ca, c.state_dict(), so3.score_norm_np, torus.score_norm, confidence_mode=True)
    return m, om, oc, sa, ca


def _lists_from(z, g, prefix):
    dl = []
    for i in range(z[f'{prefix}_lig_pos'].shape[0]):
        x = copy.deepcopy(g)
        x['ligand'].pos = torch.from_numpy(z[f'{prefix}_lig_pos'][i].copy())
        if f'{prefix}_atom_pos' in z:
            x['atom'].pos = torch.from_numpy(z[f'{prefix}_atom_pos'][i].copy())
        dl.append(x)
    return dl


def _check_forward(z, tag, om, out, strides=(1, 1)):
    dbg = om._debug
    for nm in ('ll', 'lr', 'la', 'aa'):
        assert np.array_equal(dbg[nm].numpy().astype(np.int32), z[f'{tag}_{nm}']), nm
    sa_, sr_, sl_ = (int(s) for s in z[f'{tag}_strides'])             # rows stored: every sa_-th atom, sr_-th residue, sl_-th ligand atom
    for l, (lig, atom, rec) in enumerate(dbg['layers']):
        assert T.rel_err(lig[::sl_], z[f'{tag}_lig_L{l}']) < 1e-5 and T.rel_err_cols(lig[::sl_], z[f'{tag}_lig_L{l}']) < 1e-4, l
        if f'{tag}_atom_L{l}' in z:
            assert T.rel_err(atom[::sa_], z[f'{tag}_atom_L{l}']) < 1e-5, l
        if f'{tag}_rec_L{l}' in z:
            assert T.rel_err(rec[::sr_], z[f'{tag}_rec_L{l}']) < 1e-5, l
    for k, v in zip(('tr', 'rot', 'tor', 'sc'), out):
        assert v.numel() == z[f'{tag}_{k}'].size
        assert T.rel_err(v, z[f'{tag}_{k}']) < 1e-5 and T.rel_err_elem(v, z[f'{tag}_{k}']) < 1e-3, k


@pytest.mark.parametrize('name', ['small', 'lmax2'])
def test_oracle_forward_matches_reference_all_atom_score_model(name):
    """models/all_atom_score_model.py:238-436 executed unmodified (sh_lmax 1 with FasterTensorProduct, sh_lmax 2 with e3nn
    FullyConnectedTensorProduct) vs oracle/score_model_ref.py: edge lists identical, per-layer features and scores to 1e-5."""
    z = _z('ref_forward_small.npz')
    kw = dict(ns=16, nv=4, num_conv_layers=4, sigma_embed_dim=32, distance_embed_dim=32, cross_distance_embed_dim=32)
    seed = 0
    if name == 'lmax2':
        kw.update(sh_lmax=2, num_conv_layers=3)
        seed = 3
    m, om, oc, sa, ca = _oracle_pair(utils.score_model_args(**kw), utils.confidence_model_args(ns=8, nv=2, num_conv_layers=3, sh_lmax=kw.get('sh_lmax', 1)), seed)
    np.testing.assert_allclose(refpin.weight_checksum(m.state_dict()), z[f'{name}_weight_checksum'], rtol=1e-12)
    g = inputs.synthetic_complex(7, n_lig=18, n_res=36, flexible_residues=3)
    dl = _lists_from(z, g, name)
    with torch.no_grad():
        out = om(T.oracle_batch_at(dl, 0.35))
        _check_forward(z, name, om, out)
        conf = oc(T.oracle_batch_at(dl, 0.0))
    assert T.rel_err(conf, z[f'{name}_confidence']) < 1e-5


def test_oracle_forward_rigid_ligand_matches_reference():
    z = _z('ref_forward_small.npz')
    m, om, oc, sa, ca = _oracle_pair(utils.score_model_args(ns=16, nv=4, num_conv_layers=4, sigma_embed_dim=32, distance_embed_dim=32,
                                                            cross_distance_embed_dim=32),
                                     utils.confidence_model_args(ns=8, nv=2, num_conv_layers=3), 0)
    g = inputs.synthetic_complex(21, n_lig=3, n_res=30, flexible_residues=0)
    dl = _lists_from(z, g, 'rigid')
    with torch.no_grad():
        out = om(T.oracle_batch_at(dl, 0.4))
    assert out[2].numel() == 0 and out[3].numel() == 0 and z['rigid_tor'].size == 0 and z['rigid_sc'].size == 0
    assert T.rel_err(out[0], z['rigid_tr']) < 1e-5 and T.rel_err(out[1], z['rigid_rot']) < 1e-5


def test_oracle_forward_big_model_matches_reference():
    """README big model (ns=60, nv=10, 6 layers) on two 3dpf holo graphs at t=0.7 (every lig-residue pair is an edge)."""
    z = _z('ref_forward_big.npz')
    m, om, oc, sa, ca = _oracle_pair(utils.score_model_args(), utils.confidence_model_args(), 0)
    np.testing.assert_allclose(refpin.weight_checksum(m.state_dict()), z['big_weight_checksum'], rtol=1e-12)
    dl = _lists_from(z, T.graph('3dpf_holo'), 'big')
    with torch.no_grad():
        out = om(T.oracle_batch_at(dl, 0.7))
        _check_forward(z, 'big_t70', om, out)
        conf = oc(T.oracle_batch_at(dl, 0.0))
    assert T.rel_err(conf, z['big_confidence']) < 1e-5


def test_oracle_sampling_matches_reference_sampling_py():
    """utils/sampling.py:70-286 executed unmodified (low-temperature parameters of inference.py, ODE mode,
    no_final_step_noise; per-step DataLoader seed draws included) vs oracle/sampling_ref.py under the same seeds."""
    z = _z('ref_sampling_small.npz')
    m, om, oc, sa, ca = _oracle_pair(utils.score_model_args(ns=16, nv=4, num_conv_layers=4, sigma_embed_dim=32, distance_embed_dim=32,
                                                            cross_distance_embed_dim=32),
                                     utils.confidence_model_args(ns=8, nv=2, num_conv_layers=3), 0)
    np.testing.assert_allclose(refpin.weight_checksum(m.state_dict()), z['weight_checksum'], rtol=1e-12)
    g = inputs.synthetic_complex(5, n_lig=20, n_res=40, flexible_residues=3)
    dl = T.randomized_list(g, 5, sa, seed=2)
    _close(torch.stack([x['ligand'].pos for x in dl]).numpy(), z['lig_pos0'], rtol=1e-5, atol=1e-6)
    t2s = partial(D.t_to_sigma, args=sa)
    for prefix, steps, bs, seed, kw in (('', 6, 3, 11, refpin.TEMPS), ('ode_', 4, 2, 12, dict(ode=True)),
                                        ('nofinal_', 4, 5, 13, dict(no_final_step_noise=True))):
        sch = D.get_t_schedule(steps)
        torch.manual_seed(seed)
        trace = []
        out, conf = S.sampling(T.oracle_list(dl), om, steps, sch, sch, sch, sch, t2s, sa, confidence_model=oc, batch_size=bs, trace=trace, **kw)
        lig = torch.stack([x['ligand'].pos for x in out]).numpy()
        atom = torch.stack([x['atom'].pos for x in out]).numpy()
        assert float(np.abs(lig - z[prefix + 'lig_pos']).max()) < 2e-3, prefix
        assert float(np.abs(atom - z[prefix + 'atom_pos']).max()) < 2e-3, prefix
        assert T.rel_err(conf, z[prefix + 'confidence']) < 1e-4, prefix
        if prefix == '':
            for k, v in zip(('tr', 'rot', 'tor', 'sc'), trace[0]):
                assert T.rel_err(v, z[f'step0_{k}']) < 1e-5, k
            for k, v in zip(('tr', 'rot', 'tor', 'sc'), trace[-1]):
                assert T.rel_err(v, z[f'last_{k}']) < 1e-3, k


# =========================================================================================== part 2: live reference
_CACHED = os.path.exists(os.path.join(refshim.CACHE, '.score.npy')) and os.path.exists(os.path.join(refshim.CACHE, '.so3_exp_score_norms2.npy'))
live = pytest.mark.skipif(not (refshim.available() and (_CACHED or os.environ.get('DDP_REF_SLOW'))),
                          reason='needs /root/reference and its so3/torus table caches (python scripts/make_ref_fixtures.py tables: ~9 min)')


@pytest.fixture(scope='module')
def R():
    return refshim.load()


@live
def test_live_reference_modules_are_the_unmodified_files(R):
    for m in R:
        assert m.__file__.startswith(refshim.REF_ROOT + os.sep)


@live
def test_live_faster_tensor_product_and_conv_layer_fresh_inputs(R):
    torch.manual_seed(1234)
    for in_ir, out_ir in refpin.FTP_CASES:
        a, b = R.layers.FasterTensorProduct(in_ir, '1x0e+1x1o', out_ir), FasterTensorProduct(in_ir, '1x0e+1x1o', out_ir)
        assert a.weight_numel == b.weight_numel
        x = torch.randn(7, E.Irreps(in_ir).dim)
        sh = E.spherical_harmonics('1x0e+1x1o', torch.randn(7, 3))
        w = torch.randn(7, a.weight_numel)
        assert torch.allclose(a(x, sh, w), b(x, sh, w), rtol=1e-5, atol=1e-5)
    for case, (in_ir, out_ir, nf, faster, sh_ir) in refpin.CONV_CASES.items():
        a = R.score_model.TensorProductConvLayer(in_ir, sh_ir, out_ir, nf, residual=True, batch_norm=True, faster=faster)
        b = TensorProductConvLayer(in_ir, sh_ir, out_ir, nf, residual=True, batch_norm=True, faster=faster)
        refpin.np_fill(a, 99).eval()
        b.load_state_dict(a.state_dict(), strict=True)
        b.eval()
        x, ei, ea, sh = refpin.conv_inputs(case, n=31, e=200, seed=77)
        with torch.no_grad():
            assert T.rel_err(b(x, ei, ea, sh), a(x, ei, ea, sh)) < 1e-5, case
            assert a(x, ei[:, :0], ea[:0], sh[:0]).item() == 0 and b(x, ei[:, :0], ea[:0], sh[:0]).item() == 0   # score_model.py:109-111


@live
def test_live_geometry_and_torsion_fresh_inputs(R):
    rng = np.random.RandomState(42)
    aa = torch.from_numpy(rng.standard_normal((64, 3)).astype(np.float32) * 2)
    assert torch.allclose(R.geometry.axis_angle_to_matrix(aa), D.axis_angle_to_matrix(aa), atol=1e-6)
    for n in (4, 11, 60):
        A = torch.from_numpy(rng.standard_normal((3, n)).astype(np.float32))
        B = torch.from_numpy(rng.standard_normal((3, n)).astype(np.float32))
        (r1, t1), (r2, t2) = R.geometry.rigid_transform_Kabsch_3D_torch(A, B), D.kabsch(A, B)
        assert torch.allclose(r1, r2, atol=1e-5) and torch.allclose(t1, t2, atol=1e-5)
    g = T.graph('3dpf_apo')
    sa = utils.score_model_args()
    dl = T.randomized_list(g, 2, sa, seed=9)
    a, b = T.oracle_list(dl), T.oracle_list(dl)
    tr, rot, tor, sc = refpin.pose_inputs(g, n=2, seed=3)
    for i in range(2):
        R.diffusion_utils.modify_sidechains(a[i], sc[i])
        R.diffusion_utils.modify_conformer(a[i], torch.from_numpy(tr[i:i + 1]), torch.from_numpy(rot[i]), tor[i])
        D.modify_sidechains(b[i], sc[i])
        D.modify_conformer(b[i], torch.from_numpy(tr[i:i + 1]), torch.from_numpy(rot[i]), tor[i])
        assert (a[i]['ligand'].pos - b[i]['ligand'].pos).abs().max() < 2e-5
        assert (a[i]['atom'].pos - b[i]['atom'].pos).abs().max() < 2e-5


@live
def test_live_fixtures_are_reproducible(R):
    """The committed reference fixtures are what the reference modules produce today (guards against stale files)."""
    z = _z('ref_ops.npz')
    for i, (in_ir, out_ir) in enumerate(refpin.FTP_CASES):
        tp = R.layers.FasterTensorProduct(in_ir, '1x0e+1x1o', out_ir)
        x, sh, rng = refpin.ftp_inputs(i)
        w = torch.from_numpy(rng.standard_normal((x.shape[0], tp.weight_numel)).astype(np.float32))
        assert np.array_equal(tp(x, sh, w).numpy(), z[f'ftp{i}_out'])
    zt = _z('ref_tables.npz')
    assert np.array_equal(R.so3._exp_score_norms, zt['so3_exp_score_norms'])
    assert np.array_equal(R.torus.score_norm_seed0_, zt['torus_score_norm_seed0'])


@live
def test_live_small_model_forward_and_sampler_reference_vs_oracle(R):
    """Reference ``get_model`` + ``forward`` + ``sampling`` next to the oracle on a graph no fixture holds."""
    R.torus.score_norm_ = torus.score_norm_table().copy()             # shared Monte-Carlo table (SURVEY F8)
    sa = utils.score_model_args(ns=16, nv=4, num_conv_layers=3, sigma_embed_dim=32, distance_embed_dim=32, cross_distance_embed_dim=32)
    ca = utils.confidence_model_args(ns=8, nv=2, num_conv_layers=3)
    m, om, oc, sa, ca = _oracle_pair(sa, ca, 5)
    c = utils.build_models(torch.device('cpu'), score_args=sa, conf_args=ca, seed=5)[1]
    dev = torch.device('cpu')
    rm = R.utils.get_model(sa, dev, partial(R.diffusion_utils.t_to_sigma, args=sa), no_parallel=True)
    rm.load_state_dict(m.state_dict(), strict=True)                   # reference key names, strict (inference.py:434-435)
    rc = R.utils.get_model(ca, dev, partial(R.diffusion_utils.t_to_sigma, args=ca), no_parallel=True, confidence_mode=True)
    rc.load_state_dict(c.state_dict(), strict=True)
    rm.eval(), rc.eval()
    g = inputs.synthetic_complex(77, n_lig=15, n_res=28, flexible_residues=2)
    dl = T.randomized_list(g, 4, sa, seed=8)
    steps = 3
    sch = D.get_t_schedule(steps)
    torch.manual_seed(3)
    ref, ref_conf = R.sampling.sampling(data_list=T.oracle_list(dl), model=rm, inference_steps=steps, tr_schedule=sch, rot_schedule=sch,
                                        tor_schedule=sch, sidechain_tor_schedule=sch, device=dev,
                                        t_to_sigma=partial(R.diffusion_utils.t_to_sigma, args=sa), model_args=sa, confidence_model=rc,
                                        filtering_model_args=ca, batch_size=3, **refpin.TEMPS)
    state_ref = torch.random.get_rng_state()
    torch.manual_seed(3)
    out, conf = S.sampling(T.oracle_list(dl), om, steps, sch, sch, sch, sch, partial(D.t_to_sigma, args=sa), sa, confidence_model=oc,
                           batch_size=3, **refpin.TEMPS)
    assert torch.equal(state_ref, torch.random.get_rng_state())      # both consumed the generator identically
    for a, b in zip(out, ref):
        assert (a['ligand'].pos - b['ligand'].pos).abs().max() < 1e-3
        assert (a['atom'].pos - b['atom'].pos).abs().max() < 1e-3
    assert T.rel_err(conf, ref_conf) < 1e-4


# =========================================================================================== conv backward (training path)
def _conv_grads(conv, case):
    x, ei, ea, sh = refpin.conv_inputs(case)
    dev = next(conv.parameters()).device
    xs, eas, shs = (t.clone().to(dev).requires_grad_(True) for t in (x, ea, sh))
    out = conv(xs, ei.to(dev), eas, shs, out_nodes=x.shape[0] + 3)
    probe = torch.from_numpy(np.random.RandomState(11).standard_normal(tuple(out.shape)).astype(np.float32)).to(dev)
    gs = torch.autograd.grad((out * probe).sum(), [xs, eas, shs, conv.fc[0].weight, conv.fc[0].bias, conv.fc[3].weight, conv.fc[3].bias])
    return dict(zip(('x', 'ea', 'sh', 'w1', 'b1', 'w2', 'b2'), [g.detach().cpu().numpy() for g in gs]))


def _sums(g):
    g = g.astype(np.float64)
    return np.array([g.sum(), np.abs(g).sum(), (g * g).sum()])


def check_conv_grads(got, case, rtol):
    """Compare a dict of gradients with tests/golden/ref_conv_grads.npz (autograd through the reference's own layer).
    Gradients the fixture holds as a row sample (``_stride``, ``_shape``, ``_sums``) are compared on those rows and, over
    the whole array, by their absolute and squared sums."""
    z = _z('ref_conv_grads.npz')
    for name in ('x', 'ea', 'sh', 'w1', 'b1', 'b2'):
        key, g = f'grad_{case}_{name}', got[name]
        want = z[key]
        if key + '_stride' in z:
            assert g.shape == tuple(z[key + '_shape'])
            np.testing.assert_allclose(_sums(g)[1:], z[key + '_sums'][1:], rtol=10 * rtol)
            g = g[::int(z[key + '_stride'])]
        assert g.shape == want.shape
        assert T.rel_err(g, want) < rtol, (case, name, T.rel_err(g, want))
    w2 = got['w2']
    assert T.rel_err(w2.reshape(-1)[::97], z[f'grad_{case}_w2_sample']) < rtol
    np.testing.assert_allclose(_sums(w2)[1:], z[f'grad_{case}_w2_sums'][1:], rtol=10 * rtol)


@pytest.mark.parametrize('case', list(refpin.CONV_CASES))
def test_oracle_conv_gradients_match_reference_autograd(case):
    in_ir, out_ir, nf, faster, sh_ir = refpin.CONV_CASES[case]
    conv = TensorProductConvLayer(in_ir, sh_ir, out_ir, nf, residual=False, batch_norm=True, faster=faster)
    refpin.np_fill(conv, 7).eval()
    check_conv_grads(_conv_grads(conv, case), case, 2e-5)


# =========================================================================================== asynchronous noise schedule
ASYNC_KW = dict(ns=16, nv=4, num_conv_layers=4, sigma_embed_dim=32, distance_embed_dim=32, cross_distance_embed_dim=32,
                asyncronous_noise_schedule=True)


def async_case(device):
    """Seeded model / inputs of scripts/make_ref_fixtures.py:make_async -> (product model, score args, sample list, fixture)."""
    sa = utils.score_model_args(**ASYNC_KW)
    m, _, sa, _ = utils.build_models(device, score_args=sa, seed=5, with_confidence=False)
    z = _z('ref_async.npz')
    np.testing.assert_allclose(refpin.weight_checksum(m.state_dict()), z['weights'], rtol=1e-6)
    g = inputs.synthetic_complex(3, n_lig=16, n_res=30, flexible_residues=2)
    np.random.seed(6)
    torch.manual_seed(6)
    dl = [pyg_mini.from_any(g) for _ in range(3)]
    S.randomize_position(dl, False, False, sa.tr_sigma_max, flexible_sidechains=True)
    return m, sa, dl, z


def test_oracle_asynchronous_noise_schedule_matches_reference():
    """all_atom_score_model.py:370,450,492,517 + utils/diffusion_utils.py:158-165 + utils/sampling.py:116-117: the sigma embeddings
    read set_time's `t`; forward and a 3-step sampler run of the reference's own model against the oracle."""
    m, sa, dl, z = async_case(torch.device('cpu'))
    om = factory.oracle_model(sa, m.state_dict(), so3.score_norm_np, torus.score_norm)
    b = pyg_mini.Batch.from_data_list(copy.deepcopy(dl))
    D.set_time(b, 0.4, 0.4, 0.4, 0.4, len(dl), t=0.9)
    with torch.no_grad():
        out = om(b)
    for k, v in zip(('tr', 'rot', 'tor', 'sc'), out):
        _close(v.numpy(), z[f'fwd_{k}'], rtol=2e-4, atol=2e-5)
    D.set_time(b, 0.4, 0.4, 0.4, 0.4, len(dl), t=0.4)                 # the embedding time matters
    with torch.no_grad():
        assert T.rel_err(om(b)[0], z['fwd_tr']) > 1e-3
    steps = 3
    sch = D.get_t_schedule(steps)
    torch.manual_seed(8)
    out, _ = S.sampling(copy.deepcopy(dl), om, steps, sch, sch, sch, sch, partial(D.t_to_sigma, args=sa), sa, batch_size=2,
                        asyncronous_noise_schedule=True, t_schedule=z['t_schedule'])
    assert (torch.stack([o['ligand'].pos for o in out]) - torch.from_numpy(z['lig_pos'])).abs().max() < 2e-3
    assert (torch.stack([o['atom'].pos for o in out]) - torch.from_numpy(z['atom_pos'])).abs().max() < 2e-3
