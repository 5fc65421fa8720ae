"""GPU parity tests: the CUDA path through the C ABI against the CPU oracle on the same seeded inputs.

Gates (BASELINE.md section 5): graphs / edge indices bit-exact; per-layer outputs within 1e-4 relative
(max |a-b| / max |b|) in the fp32-grade modes and 1e-2 in the BF16 edge-MLP mode; final poses within 0.1 A RMSD.
"""
import copy
import os
from functools import partial

import numpy as np
import pytest
import torch

import _common as T
from diffdock_pocket_b200 import diffusion_utils as du, inputs, ops, sampling as ps, utils
from diffdock_pocket_b200.hetero import Batch
from diffdock_pocket_b200.score_model import TensorProductConvLayer
from oracle import cluster, diffusion_ref as D, e3nn_mini as E, sampling_ref as S
from oracle.score_model_ref import TensorProductConvLayer as RefConv

pytestmark = pytest.mark.gpu
DEV = torch.device('cuda:0')


# ------------------------------------------------------------------------------------------- graphs
def _ragged(seed, sizes, scale=4.0):
    rng = np.random.RandomState(seed)
    pts = torch.from_numpy(rng.randn(sum(sizes), 3).astype(np.float32) * scale)
    batch = torch.repeat_interleave(torch.arange(len(sizes)), torch.tensor(sizes))
    return pts, batch


@pytest.mark.parametrize('cap', [2, 32, 10000])
def test_radius_bit_exact(cap):
    x, bx = _ragged(0, [40, 0, 7, 130, 1])
    y, by = _ragged(1, [9, 3, 0, 55, 2])
    ref = cluster.radius(x, y, 5.0, bx, by, cap)
    got = ops.radius(x.to(DEV), y.to(DEV), 5.0, bx.to(DEV), by.to(DEV), cap).cpu()
    assert torch.equal(got, ref)
    c = torch.tensor([3.3, 1.0, 2.0, 0.77, 5.0])
    ref = cluster.radius(x / c[bx][:, None], y / c[by][:, None], 1, bx, by, cap)
    got = ops.radius(x.to(DEV), y.to(DEV), 1, bx.to(DEV), by.to(DEV), cap, inv_scale=c.to(DEV)).cpu()
    assert torch.equal(got, ref)


def test_radius_graph_and_knn_graph_bit_exact():
    x, b = _ragged(2, [37, 1, 64, 300, 5], scale=3.0)
    x[10] = x[11]                                                     # exact duplicates: tie-breaking by index
    x[200:240] = x[200]                                               # > k+1 coincident points
    for r, cap in ((5.0, 32), (3.0, 4)):
        assert torch.equal(ops.radius_graph(x.to(DEV), r, b.to(DEV), max_num_neighbors=cap).cpu(),
                           cluster.radius_graph(x, r, b, max_num_neighbors=cap))
    for k in (8, 12, 5, 32):
        assert torch.equal(ops.knn_graph(x.to(DEV), k, b.to(DEV)).cpu(), cluster.knn_graph(x, k, b))
    assert ops.radius(x[:0].to(DEV), x.to(DEV), 1.0, b[:0].to(DEV), b.to(DEV)).shape == (2, 0)


def test_graphs_on_3dpf_batch_bit_exact():
    m, c, om, oc, sa, ca = T.models(DEV)
    dl = T.randomized_list(T.graph(), 3, sa, seed=0)
    b = T.batch_at(dl, 0.7)
    lig, atom, rec = b['ligand'], b['atom'], b['receptor']
    assert torch.equal(ops.knn_graph(atom.pos.to(DEV), 8, atom.batch.to(DEV)).cpu(), cluster.knn_graph(atom.pos, 8, atom.batch))
    assert torch.equal(ops.radius(atom.pos.to(DEV), lig.pos.to(DEV), 5.0, atom.batch.to(DEV), lig.batch.to(DEV), 10000).cpu(),
                       cluster.radius(atom.pos, lig.pos, 5.0, atom.batch, lig.batch, 10000))
    bonds = b['flexResidues'].edge_idx.T + torch.tensor([0, 1111, 2222])[b['flexResidues'].batch]
    mid = (atom.pos[bonds[0]] + atom.pos[bonds[1]]) / 2
    ref = cluster.radius(atom.pos, mid, 5.0, atom.batch, b['flexResidues'].batch)            # cap 32 binds (SURVEY F10)
    got = ops.radius(atom.pos.to(DEV), mid.to(DEV), 5.0, atom.batch.to(DEV), b['flexResidues'].batch.to(DEV)).cpu()
    assert torch.equal(got, ref) and int(torch.bincount(ref[0]).max()) == 32


# ------------------------------------------------------------------------------------------- conv operator
SEQ = ['60x0e', '60x0e + 10x1o', '60x0e + 10x1o + 10x1e', '60x0e + 10x1o + 10x1e + 60x0o']


def _conv_pair(in_ir, sh_ir, out_ir, n_feat, faster, seed=0):
    torch.manual_seed(seed)
    prod = TensorProductConvLayer(in_ir, sh_ir, out_ir, n_feat, residual=False, batch_norm=True, faster=faster)
    bn = prod.batch_norm
    bn.running_mean.normal_(0, 0.2); bn.running_var.uniform_(0.5, 1.5); bn.weight.data.uniform_(0.7, 1.3); bn.bias.data.normal_(0, 0.2)
    ref = RefConv(in_ir, sh_ir, out_ir, n_feat, residual=False, batch_norm=True, faster=faster)
    ref.load_state_dict(prod.state_dict())
    return prod.to(DEV).eval(), ref.eval()


@pytest.mark.parametrize('case', ['l0', 'l1', 'l2', 'l3', 'final', 'lmax2'])
def test_conv_layer_operator_fp32(case):
    cfg = {'l0': (SEQ[0], SEQ[1], 180, True), 'l1': (SEQ[1], SEQ[2], 180, True), 'l2': (SEQ[2], SEQ[3], 180, True),
           'l3': (SEQ[3], SEQ[3], 180, True), 'final': (SEQ[3], '2x1o + 2x1e', 120, True), 'lmax2': (SEQ[3], SEQ[3], 180, False)}[case]
    in_ir, out_ir, nf, faster = cfg
    sh_ir = '1x0e+1x1o' if faster else '1x0e+1x1o+1x2e'
    prod, ref = _conv_pair(in_ir, sh_ir, out_ir, nf, faster)
    torch.manual_seed(1)
    n, e = 50, 333
    x = torch.randn(n, E.Irreps(in_ir).dim)
    ei = torch.randint(0, n, (2, e))
    ei[0, :40] = 7                                                   # a hub node; nodes without edges exist too
    ea = torch.randn(e, nf)
    sh = E.spherical_harmonics(sh_ir, torch.randn(e, 3))
    with torch.no_grad():
        want = ref(x, ei, ea, sh, out_nodes=n + 3)
        got = prod(x.to(DEV), ei.to(DEV), ea.to(DEV), sh.to(DEV), out_nodes=n + 3)
    assert T.rel_err(got, want) < 1e-4
    assert prod(x.to(DEV), ei[:, :0].to(DEV), ea[:0].to(DEV), sh[:0].to(DEV)).item() == 0       # score_model.py:109-111


# ------------------------------------------------------------------------------------------- full forward
@pytest.mark.parametrize('t', [0.7, 0.05])
def test_score_model_forward_vs_oracle(t):
    m, c, om, oc, sa, ca = T.models(DEV)
    dl = T.randomized_list(T.graph(), 3, sa, seed=0)
    b = T.batch_at(dl, t)
    m.conv_mode = 'fp32'
    with torch.no_grad():
        pl = m.make_plan(copy.deepcopy(b))
        tr, rot, tor, sc = m.run_plan(pl, b.complex_t, return_layers=True)
        want = om(T.oracle_batch_at(dl, t))
    dbg = om._debug
    for nm in ('ll', 'aa', 'lr', 'la'):                               # graphs bit-exact
        assert torch.equal(pl.es[nm].edge_index().cpu(), dbg[nm].long()), nm
    for l, ((gl, ga, gr), (wl, wa, wr)) in enumerate(zip(pl.last_layers, dbg['layers'])):
        assert T.rel_err(gl, wl) < 1e-4 and T.rel_err(ga[:, :wa.shape[1]], wa) < 1e-4, l
        assert T.rel_err(gr[:, :wr.shape[1]], wr) < 1e-4, l
    for got, w, key in ((tr, want[0], 'tr'), (rot, want[1], 'rot'), (tor, want[2], 'tor'), (sc, want[3], 'sc')):
        assert T.rel_err(got, w) < 1e-4, key


def test_forward_drop_in_call_and_confidence():
    m, c, om, oc, sa, ca = T.models(DEV)
    dl = T.randomized_list(T.graph(), 3, sa, seed=0)
    b = T.batch_at(dl, 0.0)
    with torch.no_grad():
        conf = c(copy.deepcopy(b))
        want = oc(T.oracle_batch_at(dl, 0.0))
    assert T.rel_err(conf, want) < 1e-4
    b = T.batch_at(dl[:1], 0.3)                                        # single graph goes through forward()
    b2 = copy.deepcopy(b)
    with torch.no_grad():
        got = m(b2)
        want = om(T.oracle_batch_at(dl[:1], 0.3))
    for g_, w_ in zip(got, want):
        assert T.rel_err(g_, w_) < 1e-4
    assert torch.equal(b2['atom', 'atom'].edge_index.cpu(), om._debug['aa'])      # side effect of all_atom_score_model.py:530


def test_forward_apo_graph_and_empty_cross_edges():
    """Config-2 graph, plus a ligand pushed 60 A away: no ligand-atom edges -> those convs contribute exactly 0."""
    m, c, om, oc, sa, ca = T.models(DEV)
    dl = T.randomized_list(T.graph('3dpf_apo'), 2, sa, seed=3)
    dl[1]['ligand'].pos = dl[1]['ligand'].pos + torch.tensor([60.0, 0, 0])
    b = T.batch_at(dl, 0.2)
    with torch.no_grad():
        got = m(copy.deepcopy(b))
        want = om(T.oracle_batch_at(dl, 0.2))
    for g_, w_ in zip(got, want):
        assert T.rel_err(g_, w_) < 1e-4


# ------------------------------------------------------------------------------------------- pose update + sampler
def test_pose_update_vs_oracle():
    sa = utils.score_model_args()
    g = T.graph()
    dl = T.randomized_list(g, 3, sa, seed=4)
    rng = np.random.RandomState(0)
    tr, rot = rng.randn(3, 3).astype(np.float32), (rng.randn(3, 3) * 0.4).astype(np.float32)
    tor, sc = (rng.randn(3, 5) * 0.5).astype(np.float32), (rng.randn(3, 17) * 0.5).astype(np.float32)
    tor[1, 2] = 0.0                                                   # utils/torsion.py:76 skips exact zeros
    ref = copy.deepcopy(dl)
    for i, d in enumerate(ref):
        D.modify_sidechains(d, sc[i])
        D.modify_conformer(d, torch.from_numpy(tr[i:i + 1]), torch.from_numpy(rot[i]), tor[i])
    got = copy.deepcopy(dl)
    st = du.PoseState(got, DEV)
    f = lambda a: torch.from_numpy(a.reshape(-1)).to(DEV)
    st.update((1, 0, 1, 0, 1, 0, 1, 0), f(tr), f(rot), f(tor), f(sc))
    st.write_back(got)
    for a, r in zip(got, ref):
        assert (a['ligand'].pos - r['ligand'].pos).abs().max() < 2e-4
        assert (a['atom'].pos - r['atom'].pos).abs().max() < 2e-4
    one = copy.deepcopy(dl[0])                                         # single-graph drop-ins
    du.modify_sidechains(one, sc[0])
    du.modify_conformer(one, torch.from_numpy(tr[0:1]), torch.from_numpy(rot[0]), tor[0])
    assert (one['ligand'].pos.cpu() - ref[0]['ligand'].pos).abs().max() < 2e-4
    assert (one['atom'].pos.cpu() - ref[0]['atom'].pos).abs().max() < 2e-4


def test_sampling_parity_small_model():
    """Same weights, same initial poses, same CPU noise stream -> poses within 0.1 A RMSD (north-star gate)."""
    m, c, om, oc, sa, ca = T.models(DEV, small=True)
    g = inputs.synthetic_complex(5, n_lig=20, n_res=40, flexible_residues=3)
    dl = T.randomized_list(g, 5, sa, seed=2)
    steps = 6
    sch = D.get_t_schedule(steps)
    kw = dict(temp_sampling=[0.9766, 6.0774, 6.7616, 1.4488], temp_psi=[1.5103, 0.8141, 0.7662, 1.3396], temp_sigma_data=0.48884)
    torch.manual_seed(11)
    ref, ref_conf = S.sampling(T.oracle_list(dl), om, steps, sch, sch, sch, sch, partial(D.t_to_sigma, args=sa), sa,
                               confidence_model=oc, batch_size=3, **kw)
    torch.manual_seed(11)
    m.conv_mode = 'fp32'
    got, conf = ps.sampling(copy.deepcopy(dl), m, steps, sch, sch, sch, sch, DEV, partial(du.t_to_sigma, args=sa), sa,
                            confidence_model=c, filtering_model_args=ca, batch_size=3, **kw)
    for a, r in zip(got, ref):
        rmsd = float(((a['ligand'].pos.cpu() - r['ligand'].pos) ** 2).sum(-1).mean().sqrt())
        idx = g['flexResidues'].subcomponents.unique()
        rmsd_sc = float(((a['atom'].pos.cpu()[idx] - r['atom'].pos[idx]) ** 2).sum(-1).mean().sqrt())
        assert rmsd < 0.1 and rmsd_sc < 0.1, (rmsd, rmsd_sc)
    assert T.rel_err(conf, ref_conf) < 1e-2


def test_mixed_complex_batch_equals_per_complex_calls():
    """Cross-complex batching: samples of three different complexes (different ligand / pocket sizes, one without
    flexible residues' torsions) in ONE sampler call end where three separate calls end (noise off => deterministic)."""
    from functools import partial
    from diffdock_pocket_b200 import diffusion_utils as du, inputs as inp, sampling as ps
    m, c, om, oc, sa, ca = T.models(DEV, small=True)
    graphs = [inp.synthetic_complex(11, n_lig=12, n_res=30, flexible_residues=2), inp.synthetic_complex(12, n_lig=25, n_res=45, flexible_residues=3),
              inp.synthetic_complex(13, n_lig=9, n_res=26, flexible_residues=1)]
    # (joint == separate only holds while no edge set of any mini-batch is empty: a conv without edges returns 0 and skips
    # its BatchNorm shift, models/score_model.py:109-111, so the reference's output for a graph depends on whether ANOTHER
    # graph of the batch has edges of that type -- reproduced here, see test_mixed_flexible_and_rigid_complexes_in_one_batch)
    lists = [T.randomized_list(g, 3, sa, seed=20 + i) for i, g in enumerate(graphs)]
    steps = 5
    sch = du.get_t_schedule('expbeta', steps)
    kw = dict(temp_sampling=[0.9766, 6.0774, 6.7616, 1.4488], temp_psi=[1.5103, 0.8141, 0.7662, 1.3396], temp_sigma_data=0.48884,
              no_random=True, confidence_model=c, filtering_model_args=ca)
    run = lambda dl, bs: ps.sampling(copy.deepcopy(dl), m, steps, sch, sch, sch, sch, DEV, partial(du.t_to_sigma, args=sa), sa, batch_size=bs, **kw)
    joint, conf_j = run([g for dl in lists for g in dl], 5)                  # mini-batches straddle complexes
    k = 0
    for dl in lists:
        sep, conf_s = run(dl, 3)
        for a, b in zip(joint[k:k + 3], sep):
            assert float((a['ligand'].pos - b['ligand'].pos).abs().max()) < 2e-3
            assert float((a['atom'].pos - b['atom'].pos).abs().max()) < 2e-3
        assert T.rel_err(conf_j[k:k + 3], conf_s) < 1e-3
        k += 3


def test_forward_sh_lmax2_model_vs_oracle():
    """sh_lmax = 2 (the argparse / model default, utils/parsing.py:131): trunk convs are e3nn FullyConnectedTensorProducts
    with 9 spherical harmonics, the torsion heads couple to the 0e, 1o and 1e parts of FullTensorProduct(sh, Y2(bond))."""
    from diffdock_pocket_b200 import inputs as inp, so3, torus, utils
    from oracle import factory
    sa = utils.score_model_args(sh_lmax=2, ns=16, nv=4, num_conv_layers=3, sigma_embed_dim=32, distance_embed_dim=32,
                                cross_distance_embed_dim=32)
    m, _, sa, _ = utils.build_models(DEV, score_args=sa, with_confidence=False, seed=3)
    om = factory.oracle_model(sa, m.state_dict(), so3.score_norm_np, torus.score_norm)
    g = inp.synthetic_complex(7, n_lig=18, n_res=36, flexible_residues=3)
    dl = T.randomized_list(g, 3, sa, seed=1)
    b = T.batch_at(dl, 0.35)
    m.conv_mode = 'fp32'
    with torch.no_grad():
        pl = m.make_plan(copy.deepcopy(b))
        got = m.run_plan(pl, b.complex_t, return_layers=True)
        want = om(T.oracle_batch_at(dl, 0.35))
    for l, ((gl, ga, gr), (wl, wa, wr)) in enumerate(zip(pl.last_layers, om._debug['layers'])):
        assert T.rel_err(gl, wl) < 1e-4 and T.rel_err(ga[:, :wa.shape[1]], wa) < 1e-4, l
    for a, w, key in zip(got, want, ('tr', 'rot', 'tor', 'sc')):
        assert a.numel() > 0 and T.rel_err(a, w) < 1e-4, (key, T.rel_err(a, w))


def test_rigid_ligand_without_flexible_residues():
    """No rotatable bond and no flexible residue: tor / sc scores are empty tensors (all_atom_score_model.py:386-387,
    410-411), the sampler still moves the ligand rigidly and matches the oracle."""
    m, c, om, oc, sa, ca = T.models(DEV, small=True)
    g = inputs.synthetic_complex(21, n_lig=3, n_res=30, flexible_residues=0)
    assert int(g['ligand'].edge_mask.sum()) == 0 and 'flexResidues' not in g
    dl = T.randomized_list(g, 3, sa, seed=1)
    b = T.batch_at(dl, 0.4)
    m.conv_mode = 'fp32'
    with torch.no_grad():
        got = m(copy.deepcopy(b))
        want = om(T.oracle_batch_at(dl, 0.4))
    assert got[2].numel() == 0 and got[3].numel() == 0 and want[2].numel() == 0 and want[3].numel() == 0
    assert T.rel_err(got[0], want[0]) < 1e-4 and T.rel_err(got[1], want[1]) < 1e-4
    steps = 4
    sch = D.get_t_schedule(steps)
    torch.manual_seed(5)
    ref, ref_conf = S.sampling(T.oracle_list(dl), om, steps, sch, sch, sch, sch, partial(D.t_to_sigma, args=sa), sa,
                               confidence_model=oc, batch_size=2)
    torch.manual_seed(5)
    out, conf = ps.sampling(copy.deepcopy(dl), m, steps, sch, sch, sch, sch, DEV, partial(du.t_to_sigma, args=sa), sa,
                            confidence_model=c, filtering_model_args=ca, batch_size=2)
    for a, r in zip(out, ref):
        assert float(((a['ligand'].pos.cpu() - r['ligand'].pos) ** 2).sum(-1).mean().sqrt()) < 0.1
        assert torch.equal(a['atom'].pos.cpu(), r['atom'].pos)                  # nothing flexible: receptor atoms untouched
    assert T.rel_err(conf, ref_conf) < 1e-2


@pytest.mark.parametrize('mode,tol', [('bf16x3', 1e-4), ('bf16', 1e-2)])
def test_forward_batch64_equals_sub_batches(mode, tol):
    """BASELINE.json configs[2] shape (64 pocket graphs, big model, t = 1 so nearly every ligand-residue pair is an edge):
    too large for the oracle, so the check is size-independent -- the 64-graph forward equals four 16-graph forwards
    within the mode's parity gate (the scatter order differs, and in the bf16 mode a last-bit change of a feature can flip
    its bf16 rounding in the next layer)."""
    m, c, om, oc, sa, ca = T.models(DEV)
    dl = T.randomized_list(T.graph('3dpf_apo'), 64, sa, seed=9)
    m.conv_mode = mode
    try:
        with torch.no_grad():
            b = T.batch_at(dl, 1.0)
            pl = m.make_plan(copy.deepcopy(b))
            full = [x.clone() for x in m.run_plan(pl, b.complex_t)]
            assert int(pl.es['lr'].n_dev.item()) > 0.8 * 64 * dl[0]['ligand'].pos.shape[0] * dl[0]['receptor'].pos.shape[0]
            parts = []
            for k in range(0, 64, 16):
                bb = T.batch_at(dl[k:k + 16], 1.0)
                parts.append([x.clone() for x in m.run_plan(m.make_plan(copy.deepcopy(bb)), bb.complex_t)])
    finally:
        m.conv_mode = 'fp32'
    for i in range(4):
        err = T.rel_err(full[i], torch.cat([p[i] for p in parts]))
        assert err < tol, (i, err)


def _calpha_ref(pos, r, k):
    """datasets/process_mols.py:661-677 restated with numpy (float64 distances, as the reference's cdist)."""
    pos = pos.double().numpy()
    dist = np.linalg.norm(pos[:, None] - pos[None], axis=-1)
    src, dst = [], []
    for i in range(len(pos)):
        nb = [j for j in np.where(dist[i] < r)[0] if j != i]
        if len(nb) > k:
            nb = [j for j in np.argsort(dist[i], kind='stable') if j != i][:k]
        if len(nb) == 0:
            nb = [j for j in np.argsort(dist[i], kind='stable') if j != i][:1]
        src += [i] * len(nb)
        dst += [int(j) for j in nb]
    return torch.tensor([src, dst], dtype=torch.long)


def test_calpha_graph_matches_reference_preprocessing():
    """SURVEY 8(f) rank 1 (static per-complex preprocessing on the device): the residue contact graph is bit-exact with
    the host restatement on the 3dpf pockets (cap of 24 active for most residues), on a batch of pockets, and on the
    corner cases (isolated residue -> nearest one; tiny cap; single-residue complex)."""
    for name in ('3dpf_holo', '3dpf_apo'):
        g = T.graph(name)
        got = ops.calpha_graph(g['receptor'].pos.to(DEV), 15.0, 24).cpu()
        assert torch.equal(got, g['receptor', 'receptor'].edge_index), name           # what inputs.py built on the host
        assert torch.equal(got, _calpha_ref(g['receptor'].pos, 15.0, 24)), name
    graphs = [inputs.synthetic_complex(30 + i, n_lig=8, n_res=n, flexible_residues=0) for i, n in enumerate((25, 61, 33))]
    pos = torch.cat([g['receptor'].pos for g in graphs])
    batch = torch.repeat_interleave(torch.arange(3), torch.tensor([g['receptor'].pos.shape[0] for g in graphs]))
    for r, k in ((15.0, 24), (9.0, 5), (4.5, 3)):
        got = ops.calpha_graph(pos.to(DEV), r, k, batch=batch.to(DEV)).cpu()
        off, want = 0, []
        for g in graphs:
            want.append(_calpha_ref(g['receptor'].pos, r, k) + off)
            off += g['receptor'].pos.shape[0]
        assert torch.equal(got, torch.cat(want, 1)), (r, k)
    far = torch.cat([graphs[0]['receptor'].pos, torch.tensor([[400.0, 0.0, 0.0]])])   # one residue with nobody within r
    assert torch.equal(ops.calpha_graph(far.to(DEV), 15.0, 24).cpu(), _calpha_ref(far, 15.0, 24))
    assert ops.calpha_graph(torch.zeros(1, 3, device=DEV), 15.0, 24).shape == (2, 0)


def test_sampler_schedules_agree():
    """The sampler's execution strategies are bookkeeping only: mini-batches on two streams vs one, captured CUDA graphs vs
    eager launches -- same poses and confidences (noise off, fp32 mode; the only freedom left is the order of the scatter
    atomics)."""
    m, c, om, oc, sa, ca = T.models(DEV, small=True)
    g = inputs.synthetic_complex(41, n_lig=16, n_res=34, flexible_residues=3)
    dl = T.randomized_list(g, 7, sa, seed=6)
    steps = 5
    sch = du.get_t_schedule('expbeta', steps)
    kw = dict(temp_sampling=[0.9766, 6.0774, 6.7616, 1.4488], temp_psi=[1.5103, 0.8141, 0.7662, 1.3396], temp_sigma_data=0.48884,
              no_random=True, confidence_model=c, filtering_model_args=ca, batch_size=3)
    m.conv_mode = 'fp32'
    run = lambda **o: ps.sampling(copy.deepcopy(dl), m, steps, sch, sch, sch, sch, DEV, partial(du.t_to_sigma, args=sa), sa, **kw, **o)
    base, conf0 = run(concurrent_batches=False, use_graph=False)
    for opts in (dict(concurrent_batches=True, use_graph=False), dict(concurrent_batches=True, use_graph=True),
                 dict(concurrent_batches=False, use_graph=True)):
        out, conf = run(**opts)
        for a, b in zip(out, base):
            assert float((a['ligand'].pos - b['ligand'].pos).abs().max()) < 2e-3, opts
            assert float((a['atom'].pos - b['atom'].pos).abs().max()) < 2e-3, opts
        assert T.rel_err(conf, conf0) < 1e-3, opts


def test_static_embed_kernel_matches_encoder_arithmetic():
    """``ddp_node_static_embed`` (once-per-complex part of AtomEncoder.forward, models/score_model.py:74-82, and of
    OldAtomEncoder :38-52 with its two Linears folded) against the same arithmetic in PyTorch fp32, for the three node types."""
    from diffdock_pocket_b200.score_model import AtomEncoder, OldAtomEncoder, FEATURE_DIMS, static_embed
    g = T.graph('3dpf_apo')
    torch.manual_seed(0)
    for cls in (AtomEncoder, OldAtomEncoder):
        for kind, key, lm_type in (('lig', 'ligand', None), ('rec_atom', 'atom', None), ('rec_residue', 'receptor', 'esm')):
            enc = cls(60, FEATURE_DIMS[kind], 64, lm_embedding_type=lm_type).to(DEV)
            x = g[key].x
            cat, lm = (x[:, :1], x[:, 1:]) if lm_type else (x, None)
            with torch.no_grad():
                want = enc.static_part(cat.to(DEV), lm.to(DEV).float() if lm is not None else None)
                got = static_embed(enc.static_pack(DEV), cat, lm, DEV)
            assert got.shape == want.shape and T.rel_err(got, want) < 2e-6 and T.rel_err_cols(got, want) < 1e-4, (cls.__name__, kind)


def test_pipelined_and_shared_copy_inference_equals_serial_deepcopy_path():
    """The host mirror of inference.py: (a) samples that share their complex's static tensors (``sample_copies``) and the
    per-complex static cache give the same poses as deep-copied graphs (the reference's inference.py:135) passed straight to
    ``sampling()``; (b) the depth-2 software pipeline over complexes (``defer``) returns exactly what the serial loop returns,
    also with several complexes per sampler call."""
    from diffdock_pocket_b200 import inference
    m, c, om, oc, sa, ca = T.models(DEV, small=True)
    graphs = [inputs.synthetic_complex(50 + i, n_lig=10 + 3 * i, n_res=30 + 4 * i, flexible_residues=i % 3) for i in range(5)]
    rows = [(i, dict(complex_name=g.name, complex_graph=g)) for i, g in enumerate(graphs)]
    args = inference.default_args(samples_per_complex=4, batch_size=8, inference_steps=4, no_random=True)
    sched = du.get_t_schedule('expbeta', 4)
    m.conv_mode = 'fp32'
    run = lambda **kw: inference.infer_multiple_complexes(rows, m, args, sa, filtering_model=c, filtering_model_args=ca, tr_schedule=sched,
                                                          device=DEV, **kw)
    outs = {}
    for name, kw in (('serial', dict(pipeline=False)), ('pipe', dict(pipeline=True)), ('group_serial', dict(pipeline=False, batch_complexes=True)),
                     ('group_pipe', dict(pipeline=True, batch_complexes=True))):
        np.random.seed(3)
        torch.manual_seed(3)
        res, ok = run(**kw)
        assert ok == len(rows), name
        outs[name] = res
    for a, b in zip(outs['serial'], outs['pipe']):                      # identical work, only the host schedule differs
        assert a['name'] == b['name'] and np.abs(a['ligand_pos'] - b['ligand_pos']).max() < 2e-3 and np.abs(a['atom_pos'] - b['atom_pos']).max() < 2e-3
        assert np.abs(a['confidence'] - b['confidence']).max() < 1e-4
    for a, b in zip(outs['group_serial'], outs['group_pipe']):
        assert np.abs(a['ligand_pos'] - b['ligand_pos']).max() < 2e-3 and np.abs(a['confidence'] - b['confidence']).max() < 1e-4
    # (a): the reference-style call on deep copies of complex 1
    np.random.seed(3)
    torch.manual_seed(3)
    for i, g in enumerate(graphs[:2]):                                  # consume the generators exactly like the loop above
        dl = [copy.deepcopy(g) for _ in range(4)]
        ps.randomize_position(dl, sa.no_torsion, True, sa.tr_sigma_max, flexible_sidechains='flexResidues' in g)
        out, conf = ps.sampling(dl, m, 4, sched, sched, sched, sched, DEV, partial(du.t_to_sigma, args=sa), sa, confidence_model=c,
                                filtering_model_args=ca, batch_size=8, no_random=True,
                                temp_sampling=[args.temp_sampling_tr, args.temp_sampling_rot, args.temp_sampling_tor, args.temp_sampling_sc_tor],
                                temp_psi=[args.temp_psi_tr, args.temp_psi_rot, args.temp_psi_tor, args.temp_psi_sc_tor])
    want = outs['serial'][1]
    order = np.argsort(conf.cpu().numpy())[::-1]
    got = np.asarray([out[k]['ligand'].pos.cpu().numpy() + g.original_center.numpy() for k in order])
    assert np.abs(got - want['ligand_pos']).max() < 2e-3


def test_mixed_flexible_and_rigid_complexes_in_one_batch():
    """Cross-complex mini-batch in which only some complexes have flexible residues (PyG cannot even collate such a list; the
    product's collate gives the others zero entries).  Checked against the oracle on the equivalent PyG batch: the rigid
    complexes carry an EMPTY flexResidues store.  Also a batch-composition effect the reference has and this path keeps: a
    ligand with no atom within 5 A gets the ligand-atom convs' BatchNorm shift iff another graph of the batch has such edges."""
    m, c, om, oc, sa, ca = T.models(DEV, small=True)
    g1 = inputs.synthetic_complex(12, n_lig=25, n_res=45, flexible_residues=3)
    g2 = inputs.synthetic_complex(14, n_lig=10, n_res=24, flexible_residues=0)
    g3 = inputs.synthetic_complex(13, n_lig=9, n_res=26, flexible_residues=1)
    assert 'edge_idx' not in g2['flexResidues']
    dl = [T.randomized_list(g1, 1, sa, seed=20)[0], T.randomized_list(g2, 1, sa, seed=21)[0], T.randomized_list(g2, 1, sa, seed=23)[0],
          T.randomized_list(g3, 1, sa, seed=22)[0]]
    odl = T.oracle_list(dl)
    for g in odl:                                                      # the PyG-collatable equivalent
        fr = g['flexResidues']
        if 'edge_idx' not in fr:
            fr.subcomponents, fr.subcomponentsMapping = torch.zeros(0, dtype=torch.long), torch.zeros(0, 2, dtype=torch.long)
            fr.edge_idx, fr.residueNBondsMapping, fr.pdbIds, fr.num_nodes = torch.zeros(0, 2, dtype=torch.long), torch.zeros(0, dtype=torch.long), [], 0
    from oracle import pyg_mini
    ob = pyg_mini.Batch.from_data_list(odl)
    D.set_time(ob, 0.4, 0.4, 0.4, 0.4, 4)
    m.conv_mode = 'fp32'
    with torch.no_grad():
        want = om(ob)
        got = m(T.batch_at(dl, 0.4))
        ob0 = pyg_mini.Batch.from_data_list(odl)
        D.set_time(ob0, 0.0, 0.0, 0.0, 0.0, 4)
        conf_w = oc(ob0)
        conf_g = c(T.batch_at(dl, 0.0))
    for a, w, key in zip(got, want, ('tr', 'rot', 'tor', 'sc')):
        assert a.numel() == w.numel() and T.rel_err(a, w) < 1e-4, (key, T.rel_err(a, w))
    assert T.rel_err(conf_g, conf_w) < 1e-4
    # the pose state of the same mixed list: per-sample side-chain slices line up with the model's bond order
    st = du.PoseState(dl, DEV)
    assert st.S == got[3].numel() and st.T == got[2].numel()


def test_resident_state_cache_reuse_equals_fresh_plans():
    """sampling() keeps the resident state (plans, pose tables, launch programs) of its last inputs keyed by content: a second
    call on the same complex with NEW start poses must reuse it and give exactly what freshly built plans give, a call on a
    complex that differs in one receptor coordinate must not reuse it."""
    m, c, om, oc, sa, ca = T.models(DEV, small=True)
    m.conv_mode = 'fp32'
    g = inputs.synthetic_complex(9, n_lig=18, n_res=36, flexible_residues=2)
    steps = 4
    sch = D.get_t_schedule(steps)

    def run(dl, seed):
        torch.manual_seed(seed)
        out, conf = ps.sampling(copy.deepcopy(dl), m, steps, sch, sch, sch, sch, DEV, partial(du.t_to_sigma, args=sa), sa,
                                confidence_model=c, filtering_model_args=ca, batch_size=3)
        return torch.stack([o['ligand'].pos.cpu() for o in out]), torch.stack([o['atom'].pos.cpu() for o in out]), conf.cpu().clone()

    dl_a, dl_b = T.randomized_list(g, 5, sa, seed=3), T.randomized_list(g, 5, sa, seed=4)
    ps.clear_plan_cache()
    first = run(dl_a, 21)
    assert not ps.LAST_CALL['plan_reused'] and len(ps._PLAN_CACHE) == 0      # a first call keeps nothing alive
    run(dl_a, 21)                               # first repeat: fresh plans once more, kept from here on
    assert not ps.LAST_CALL['plan_reused'] and len(ps._PLAN_CACHE) == 1
    reused = run(dl_b, 22)                      # same complex, other start poses and noise: resident state re-used
    assert ps.LAST_CALL['plan_reused']
    ps.clear_plan_cache()
    fresh = run(dl_b, 22)
    assert not ps.LAST_CALL['plan_reused']
    # (the scatter-adds of the convs are atomic: two runs agree to rounding, not bit for bit)
    close = lambda x, y: float((x.double() - y.double()).abs().max()) < 2e-3
    for a, b in zip(reused, fresh):
        assert close(a, b), float((a.double() - b.double()).abs().max())
    again = run(dl_a, 21)                       # first repeat after the clear: fresh plans, kept; same result as the very first run
    assert not ps.LAST_CALL['plan_reused'] and len(ps._PLAN_CACHE) == 1
    for a, b in zip(again, first):
        assert close(a, b), float((a.double() - b.double()).abs().max())
    g2 = copy.deepcopy(g)
    g2['receptor'].pos[1, 0] += 0.25
    run(T.randomized_list(g2, 5, sa, seed=3), 21)   # same shapes, one receptor coordinate differs: content key misses
    assert not ps.LAST_CALL['plan_reused']
    ps.clear_plan_cache()


# ------------------------------------------------------------------------------------------- conv backward (training path)
@pytest.mark.parametrize('case', ['l1', 'l3', 'final', 'lmax2', 'small'])
@pytest.mark.parametrize('mode', ['fp32', 'bf16x3'])
def test_conv_layer_backward_vs_autograd_of_the_oracle(case, mode):
    """Gradients of the conv operator (node features, edge attributes, edge harmonics, both Linears of the edge MLP) against
    PyTorch autograd through the oracle layer, i.e. what `loss.backward()` computes in the reference's training loop
    (utils/training.py:147-191).  Forward runs on the fused kernels (fp32 CUDA-core / fp32-grade tensor-core), backward on
    ddp_tp_backward + library GEMMs."""
    cfg = {'l1': (SEQ[1], SEQ[2], 180, True), 'l3': (SEQ[3], SEQ[3], 180, True), 'final': (SEQ[3], '2x1o + 2x1e', 120, True),
           'lmax2': (SEQ[3], SEQ[3], 180, False),
           'small': ('16x0e + 4x1o + 4x1e + 16x0o', '16x0e + 4x1o + 4x1e + 16x0o', 48, True)}[case]
    in_ir, out_ir, nf, faster = cfg
    if mode != 'fp32' and case in ('final',):
        pytest.skip('head conv runs on the CUDA-core kernel only')
    sh_ir = '1x0e+1x1o' if faster else '1x0e+1x1o+1x2e'
    prod, ref = _conv_pair(in_ir, sh_ir, out_ir, nf, faster, seed=3)
    prod.conv_mode = mode
    torch.manual_seed(5)
    n, e = 40, 301
    x = torch.randn(n, E.Irreps(in_ir).dim)
    ei = torch.randint(0, n, (2, e))
    ei[0, :30] = 5
    ea = torch.randn(e, nf)
    sh = E.spherical_harmonics(sh_ir, torch.randn(e, 3))
    probe = torch.randn(n + 2, E.Irreps(out_ir).dim)                  # d loss / d out

    def grads(layer, dev):
        xs, eas, shs = (t.clone().to(dev).requires_grad_(True) for t in (x, ea, sh))
        out = layer(xs, ei.to(dev), eas, shs, out_nodes=n + 2)
        params = [layer.fc[0].weight, layer.fc[0].bias, layer.fc[3].weight, layer.fc[3].bias]
        gs = torch.autograd.grad((out * probe.to(dev)).sum(), [xs, eas, shs] + params)
        return out.detach().cpu(), [t.cpu() for t in gs]
    want_out, want = grads(ref, 'cpu')
    got_out, got = grads(prod, DEV)
    assert T.rel_err(got_out, want_out) < 1e-4
    for name, a, b in zip(('x', 'edge_attr', 'edge_sh', 'W1', 'b1', 'W2', 'b2'), got, want):
        assert a.shape == b.shape
        assert T.rel_err(a, b) < 2e-4, (name, T.rel_err(a, b))
    # an optimizer-style in-place update of the weights is seen by the next forward (packed images are re-built)
    with torch.no_grad():
        for lyr in (prod, ref):
            lyr.fc[3].weight.mul_(0.5)
    want2, _ = grads(ref, 'cpu')
    got2, _ = grads(prod, DEV)
    assert T.rel_err(got2, want2) < 1e-4


def test_filtered_knn_graph_bit_exact_on_pockets_and_edge_cases():
    """The atom graph (k = 8 and k = 12) through the filtered search: protein-pocket-like clouds (dense ball + sparse surface
    atoms that need the wider retry radii), an example larger than one shared-memory stage (plain-scan fallback inside the kernel),
    examples smaller than k + 1, coincident points, points far apart -- identical edge lists, order included."""
    g = torch.Generator().manual_seed(7)
    parts = [torch.randn(1100, 3, generator=g) * 9.0,                                  # pocket-sized dense cloud
             torch.cat([torch.randn(600, 3, generator=g) * 6.0, torch.randn(40, 3, generator=g) * 40.0]),   # core + far outliers
             torch.randn(2500, 3, generator=g) * 12.0,                                  # > kKnnStage points
             torch.randn(5, 3, generator=g), torch.randn(1, 3, generator=g),            # fewer than k + 1 points
             torch.rand(200, 3, generator=g) * 400.0,                                   # wide extent: few neighbours within the radii
             torch.zeros(30, 3) + 2.5]                                                  # all coincident
    parts[0][100:120] = parts[0][100]
    x = torch.cat(parts)
    b = torch.cat([torch.full((p.shape[0],), i, dtype=torch.long) for i, p in enumerate(parts)])
    for k in (8, 12):
        assert torch.equal(ops.knn_graph(x.to(DEV), k, b.to(DEV)).cpu(), cluster.knn_graph(x, k, b)), k
