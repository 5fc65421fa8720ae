"""Pruned convolutions (``prune_edges``): the atom-aggregating atom-atom and atom-residue convs of the last two interaction
layers run on the edges into atoms whose features are read afterwards.  The outputs that are read do not change: in the
deterministic mode with the fp32 convolution, which converts every per-edge term to fixed point on its own, pruned and
unpruned runs give the same bits.  The tensor-core kernel pre-reduces runs of edges and splits its last tiles by the
launch's live tile count before that conversion, so there the two agree to rounding only."""
import copy
from functools import partial

import numpy as np
import pytest
import torch

import _common as T
from diffdock_pocket_b200 import diffusion_utils as du, inputs, sampling as ps
from oracle import refpin
from test_gpu_refpin import _big, _small

pytestmark = pytest.mark.gpu
DEV = torch.device('cuda:0')


@pytest.fixture
def deterministic():
    was, warn = torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled()
    torch.use_deterministic_algorithms(True)
    try:
        yield
    finally:
        torch.use_deterministic_algorithms(was, warn_only=warn)


def _forward(m, b, prune, mode='fp32'):
    m.prune_edges, m.conv_mode = prune, mode
    try:
        with torch.no_grad():
            pl = m.make_plan(copy.deepcopy(b))
            out = m.run_plan(pl, b.complex_t)
            out = [o.clone() for o in (out if isinstance(out, tuple) else (out,))]
            torch.cuda.synchronize()
    finally:
        m.prune_edges, m.conv_mode = True, 'fp32'
    return pl, out


def _equal(a, p, what):
    for i, (x, y) in enumerate(zip(a, p)):
        assert x.shape == y.shape and torch.equal(x, y), (what, i, float((x - y).abs().max()) if x.numel() else 0.0)


def _bitwise(m, b, what):
    pl0, a = _forward(m, b, False)
    pl1, p = _forward(m, b, True)
    assert not pl0.prune and pl1.prune
    _equal(a, p, what)
    return pl1


def _apo(n=4, seed=0):
    m, c, sa, ca = _big()
    return m, c, T.randomized_list(T.graph('3dpf_apo'), n, sa, seed=seed)


@pytest.mark.parametrize('t', [1.0, 0.05])
def test_big_model_pruned_bitwise(deterministic, t):
    m, c, dl = _apo()
    pl = _bitwise(m, T.batch_at(dl, t), f'3dpf apo t={t}')
    n_live = pl.live.sum(1).tolist()
    assert 0 < n_live[0] < n_live[1] < pl.NA, n_live                   # something is pruned in both layers


def test_confidence_model_pruned_bitwise(deterministic):
    m, c, dl = _apo()
    pl = _bitwise(c, T.batch_at(dl, 0.0), 'confidence')
    assert torch.equal(pl.live[0].nonzero().flatten().int(), pl.flex_atoms.sort().values)


def test_two_layer_model_pruned_bitwise(deterministic):
    m, c, sa, ca = _small(num_conv_layers=2)
    g = inputs.synthetic_complex(7, n_lig=18, n_res=36, flexible_residues=3)
    pl = _bitwise(m, T.batch_at(T.randomized_list(g, 3, sa, seed=4), 0.6), 'two layers')
    assert pl.prune_layers == [0, 1]


def test_no_flexible_residues_pruned_bitwise(deterministic):
    m, c, sa, ca = _small()
    g = inputs.synthetic_complex(21, n_lig=12, n_res=30, flexible_residues=0)
    dl = T.randomized_list(g, 2, sa, seed=5)
    pl = _bitwise(m, T.batch_at(dl, 0.5), 'no flexible residues')
    assert pl.S == 0 and int(pl.live[0].sum()) == 0
    assert int(pl.pruned[(m.num_conv_layers - 1, 'aa')].n_dev) == 0 and int(pl.es['aa'].n_dev) > 0
    _bitwise(c, T.batch_at(dl, 0.0), 'no flexible residues, confidence')


def test_mixed_complex_batch_pruned_bitwise(deterministic):
    m, c, sa, ca = _small()
    g1 = inputs.synthetic_complex(12, n_lig=25, n_res=45, flexible_residues=3)
    g2 = inputs.synthetic_complex(14, n_lig=10, n_res=24, flexible_residues=0)
    g3 = inputs.synthetic_complex(13, n_lig=9, n_res=26, flexible_residues=1)
    dl = [T.randomized_list(g1, 1, sa, seed=20)[0], T.randomized_list(g2, 1, sa, seed=21)[0], T.randomized_list(g3, 1, sa, seed=22)[0]]
    _bitwise(m, T.batch_at(dl, 0.4), 'mixed batch')
    _bitwise(c, T.batch_at(dl, 0.0), 'mixed batch, confidence')


def test_empty_pruned_set_keeps_batchnorm_shift(deterministic):
    """Live atoms without atom-residue edges: the pruned set of the last layer is empty while the full set is not, and the
    live atoms must still receive that conv's BatchNorm shift (it is added when the FULL set has edges)."""
    m, c, sa, ca = _small()
    g = inputs.synthetic_complex(9, n_lig=18, n_res=36, flexible_residues=2)
    b = T.batch_at(T.randomized_list(g, 1, sa, seed=8), 0.7)
    pl, _ = _forward(m, b, True)
    live = pl.live[0].bool().cpu()
    ar = b['atom', 'receptor'].edge_index
    b['atom', 'receptor'].edge_index = ar[:, ~live[ar[0]]]
    assert b['atom', 'receptor'].edge_index.shape[1] > 0
    pl = _bitwise(m, b, 'empty pruned atom-residue set')
    last = m.num_conv_layers - 1
    assert torch.equal(pl.live[0], live.to(pl.live.device, torch.uint8))
    assert int(pl.pruned[(last, 'ar')].n_dev) == 0 and int(pl.es['ar'].n_dev) > 0


def test_pruned_sets_are_the_filtered_full_sets():
    m, c, dl = _apo()
    pl, _ = _forward(m, T.batch_at(dl, 1.0), True, 'bf16')
    live = pl.live.cpu().numpy().astype(bool)
    for (l, nm), p in pl.pruned.items():
        full = pl.es[nm]
        ei = full.edge_index().cpu().numpy()
        keep = live[m.num_conv_layers - 1 - l][ei[0]]
        n = int(p.n_dev)
        assert n == int(keep.sum()) and 0 < n < ei.shape[1], (l, nm, n, ei.shape[1])
        assert np.array_equal(p.edge_index().cpu().numpy(), ei[:, keep]), (l, nm)
        assert torch.equal(p.sh[:n].cpu(), full.sh[:full.edge_index().shape[1]].cpu()[torch.from_numpy(keep)]), (l, nm)
        assert torch.equal(p.emb[:n].cpu(), full.emb[:full.edge_index().shape[1]].cpu()[torch.from_numpy(keep)]), (l, nm)
        assert p.deg is full.deg


def test_live_atoms_cover_everything_the_heads_read():
    m, c, dl = _apo()
    pl, _ = _forward(m, T.batch_at(dl, 0.3), True, 'bf16')
    live = pl.live.cpu().bool()
    gathered = pl.sc.es.edge_index()[1].cpu()                          # atoms of the side-chain head's radius graph
    assert gathered.numel() > 0 and bool(live[0][gathered].all())
    assert bool(live[0][pl.sc.bonds.long().cpu().flatten()].all())
    assert bool(live[1][live[0]].all())
    la = pl.es['la'].edge_index()[1].cpu()
    assert bool(live[1][la].all())
    aa = pl.es['aa'].edge_index().cpu()
    assert bool(live[1][aa[1][live[0][aa[0]]]].all())


@pytest.mark.parametrize('det', [False, True])
def test_tensor_core_pruned_close(det):
    """bf16 convs: pruned and unpruned agree to the rounding of the accumulation order; in the deterministic mode the pruned
    forward is itself bitwise reproducible."""
    m, c, dl = _apo()
    b = T.batch_at(dl, 1.0)
    was = torch.are_deterministic_algorithms_enabled()
    torch.use_deterministic_algorithms(det)
    try:
        _, a = _forward(m, b, False, 'bf16')
        _, p = _forward(m, b, True, 'bf16')
        _, p2 = _forward(m, b, True, 'bf16')
    finally:
        torch.use_deterministic_algorithms(was)
    for x, y, key in zip(a, p, ('tr', 'rot', 'tor', 'sc')):
        assert T.rel_err(y, x) < 1e-3, (key, T.rel_err(y, x))
    if det:
        _equal(p, p2, 'pruned bf16 repeat')


def test_sampler_pruned_bitwise(deterministic):
    """BASELINE.json configs[1] inputs (3dpf apo, 40 samples, batch 20, 20 steps + confidence) with the fp32 convolution:
    pruned and unpruned runs give the same ligand poses, side-chain atoms and confidences, eager and with graph steps."""
    m, c, sa, ca = _big()
    dl = T.randomized_list(T.graph('3dpf_apo'), 40, sa, seed=0)
    steps = 20
    sch = du.get_t_schedule('expbeta', steps)

    def run(prune, **kw):
        m.prune_edges = c.prune_edges = prune
        torch.manual_seed(7)
        out, conf = ps.sampling(copy.deepcopy(dl), m, steps, sch, sch, sch, sch, DEV, partial(du.t_to_sigma, args=sa), sa,
                                confidence_model=c, filtering_model_args=ca, batch_size=20, **refpin.TEMPS, **kw)
        return (torch.stack([o['ligand'].pos for o in out]).cpu(), torch.stack([o['atom'].pos for o in out]).cpu(), conf.cpu())
    try:
        ps.clear_plan_cache()
        for kw in ({}, {'use_graph': True}):
            _equal(run(False, **kw), run(True, **kw), f'sampling {kw}')
    finally:
        m.prune_edges = c.prune_edges = True
        ps.clear_plan_cache()
