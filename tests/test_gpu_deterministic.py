"""Deterministic mode (torch.use_deterministic_algorithms(True)): the convolutions accumulate in int64 fixed point, so the
same call with the same inputs and seeds returns the same bits on every run -- conv operator (tensor-core bf16 / bf16x3 and
the fp32 kernel), its backward, the big-model forward and the full-size sampler (eager and graph steps, one or two streams,
fresh plans or the resident-state cache) -- while staying within the parity gates of the default mode."""
import copy
from functools import partial

import numpy as np
import pytest
import torch

import _common as T
from diffdock_pocket_b200 import _lib, diffusion_utils as du, sampling as ps
from diffdock_pocket_b200.score_model import TensorProductConvLayer
from oracle import e3nn_mini as E, refpin
from oracle.score_model_ref import TensorProductConvLayer as RefConv
from test_gpu_refpin import TOL, _big, _check, _lists_from, _rmsd, _run, _z

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


def _seq(ns, nv):
    return [f'{ns}x0e', f'{ns}x0e + {nv}x1o', f'{ns}x0e + {nv}x1o + {nv}x1e', f'{ns}x0e + {nv}x1o + {nv}x1e + {ns}x0o']


def _sorted_case(run):
    """The heavy-contention inputs of test_gpu_umma.py::test_conv_operator_sorted_aggregation (runs of ~`run` edges per node)."""
    ns, nv = 60, 10
    seq = _seq(ns, nv)
    torch.manual_seed(1)
    prod = TensorProductConvLayer(seq[3], '1x0e+1x1o', seq[3], 3 * ns, residual=False, batch_norm=True, faster=True)
    ref = RefConv(seq[3], '1x0e+1x1o', seq[3], 3 * ns, residual=False, batch_norm=True, faster=True)
    ref.load_state_dict(prod.state_dict())
    prod, ref = prod.to(DEV).eval(), ref.eval()
    n = 200
    lens = torch.randint(max(run // 2, 1), run * 3 // 2 + 2, (n,))
    agg = torch.repeat_interleave(torch.arange(n), lens)[:4001]
    n_edges = agg.numel()
    ei = torch.stack([agg, torch.randint(0, n, (n_edges,))])
    x = torch.randn(n, E.Irreps(seq[3]).dim)
    ea = torch.randn(n_edges, 3 * ns)
    sh = E.spherical_harmonics('1x0e+1x1o', torch.randn(n_edges, 3))
    return prod, ref, n, (x, ei, ea, sh)


@pytest.mark.parametrize('mode', ['bf16', 'bf16x3', 'fp32'])
@pytest.mark.parametrize('run', [3, 24, 100])
def test_conv_operator_bitwise_reproducible(deterministic, mode, run):
    prod, ref, n, (x, ei, ea, sh) = _sorted_case(run)
    with torch.no_grad():
        want = ref(x, ei, ea, sh, out_nodes=n)
        prod.conv_mode = mode
        args = (x.to(DEV), ei.to(DEV), ea.to(DEV), sh.to(DEV))
        outs = [prod(*args, out_nodes=n).cpu() for _ in range(5)]
    for o in outs[1:]:
        assert torch.equal(o, outs[0]), (mode, run, float((o - outs[0]).abs().max()))
    tol = 1e-4 if mode == 'fp32' else TOL[mode]
    assert T.rel_err(outs[0], want) < tol, (mode, run, T.rel_err(outs[0], want))


@pytest.mark.parametrize('mode', ['fp32', 'bf16x3', 'bf16'])
def test_big_model_forward_bitwise_and_within_gates(deterministic, mode):
    z = _z('ref_forward_big.npz')
    m, c, sa, ca = _big()
    dl = _lists_from(z, T.graph('3dpf_holo'), 'big')
    pl1, out1 = _run(m, dl, 0.7, mode)
    pl2, out2 = _run(m, dl, 0.7, mode)
    assert pl1.deterministic and pl1.sum_arena.dtype == torch.int64 and pl1.g_sum.dtype == torch.int64
    for (a1, b1, c1), (a2, b2, c2) in zip(pl1.last_layers, pl2.last_layers):
        assert torch.equal(a1, a2) and torch.equal(b1, b2) and torch.equal(c1, c2)
    for o1, o2 in zip(out1, out2):
        assert torch.equal(o1, o2)
    _check(z, 'big_t70', pl1, out1, mode)


def test_default_mode_keeps_fp32_sums():
    assert not torch.are_deterministic_algorithms_enabled()
    z = _z('ref_forward_big.npz')
    m, c, sa, ca = _big()
    dl = _lists_from(z, T.graph('3dpf_holo'), 'big')
    pl, out = _run(m, dl, 0.7, 'bf16')
    assert not pl.deterministic and pl.sum_arena.dtype == torch.float32 and pl.g_sum.dtype == torch.float32
    _check(z, 'big_t70', pl, out, 'bf16')


def _full_size_inputs(n=40):
    m, c, sa, ca = _big()
    g = T.graph('3dpf_apo')
    dl = T.randomized_list(g, n, sa, seed=0)
    return m, c, sa, ca, dl


def _sample(m, c, sa, ca, dl, **kw):
    steps = 20
    sch = du.get_t_schedule('expbeta', steps)
    torch.manual_seed(7)
    out, conf = ps.sampling(copy.deepcopy(dl), m, steps, sch, sch, sch, sch, DEV, partial(du.t_to_sigma, args=sa), sa,
                            confidence_model=c, filtering_model_args=ca, batch_size=20, **refpin.TEMPS, **kw)
    return (torch.stack([o['ligand'].pos for o in out]).cpu(), torch.stack([o['atom'].pos for o in out]).cpu(), conf.cpu())


def _equal(a, b, what):
    for x, y, nm in zip(a, b, ('ligand_pos', 'atom_pos', 'confidence')):
        assert torch.equal(x, y), (what, nm, float((x - y).abs().max()))


def test_sampler_bitwise_reproducible_configs1(deterministic):
    """BASELINE.json configs[1]: 3dpf apo, 40 samples, batch 20, 20 steps + confidence, bf16 tensor-core convs."""
    m, c, sa, ca, dl = _full_size_inputs()
    m.conv_mode = c.conv_mode = 'bf16'
    try:
        ps.clear_plan_cache()
        first = _sample(m, c, sa, ca, dl)                              # fresh plans (records the shape signature)
        _equal(first, _sample(m, c, sa, ca, dl), 'fresh vs retained')
        assert not ps.LAST_CALL['plan_reused']
        _equal(first, _sample(m, c, sa, ca, dl), 'fresh vs resident-state cache')
        assert ps.LAST_CALL['plan_reused']
        _equal(first, _sample(m, c, sa, ca, dl, use_graph=True), 'eager vs graph steps')
        _equal(first, _sample(m, c, sa, ca, dl, use_graph=True), 'graph steps, cached')
        _equal(first, _sample(m, c, sa, ca, dl, concurrent_batches=False), 'two streams vs one')
    finally:
        m.conv_mode = c.conv_mode = 'fp32'
        ps.clear_plan_cache()


def test_sampler_cache_never_crosses_modes():
    m, c, sa, ca, dl = _full_size_inputs(n=6)
    m.conv_mode = c.conv_mode = 'bf16'
    try:
        ps.clear_plan_cache()
        for _ in range(3):
            _sample(m, c, sa, ca, dl)                                  # default-mode entry is cached and served
        assert ps.LAST_CALL['plan_reused']
        torch.use_deterministic_algorithms(True)
        try:
            d1 = _sample(m, c, sa, ca, dl)
            assert not ps.LAST_CALL['plan_reused']
            d2 = _sample(m, c, sa, ca, dl)
            d3 = _sample(m, c, sa, ca, dl)
            assert ps.LAST_CALL['plan_reused']
        finally:
            torch.use_deterministic_algorithms(False)
        _equal(d1, d2, 'deterministic fresh vs retained')
        _equal(d1, d3, 'deterministic fresh vs cached')
        entries = list(ps._PLAN_CACHE.values())
        assert sorted(e['deterministic'] for e in entries) == [False, True]
        for e in entries:
            for r in e['runners']:
                assert r.pl.deterministic == e['deterministic']
                assert r.pl.sum_arena.dtype == (torch.int64 if e['deterministic'] else torch.float32)
    finally:
        m.conv_mode = c.conv_mode = 'fp32'
        ps.clear_plan_cache()


def test_full_size_sampling_deterministic_vs_reference(deterministic):
    """tests/golden/ref_sampling_full.npz (the reference's own sampling() on the CPU) in the deterministic mode: every final
    ligand and flexible side-chain pose within 0.1 A RMSD."""
    z = _z('ref_sampling_full.npz')
    m, c, sa, ca = _big()
    g = T.graph('3dpf_apo')
    flex = g['flexResidues'].subcomponents.unique().numpy()
    dl = []
    for i in range(z['lig_pos0'].shape[0]):
        x = copy.deepcopy(g)
        x['ligand'].pos = torch.from_numpy(z['lig_pos0'][i].copy())
        x['atom'].pos = torch.from_numpy(z['atom_pos0'][i].copy())
        dl.append(x)
    steps, bs = int(z['steps']), int(z['batch_size'])
    sch = du.get_t_schedule('expbeta', steps)
    torch.manual_seed(int(z['seed']))
    m.conv_mode = c.conv_mode = 'bf16'
    try:
        out, conf = ps.sampling(dl, m, steps, sch, sch, sch, sch, DEV, partial(du.t_to_sigma, args=sa), sa, confidence_model=c,
                                filtering_model_args=ca, batch_size=bs, **refpin.TEMPS)
    finally:
        m.conv_mode = c.conv_mode = 'fp32'
    for i, x in enumerate(out):
        r1 = _rmsd(x['ligand'].pos.cpu().numpy(), z['lig_pos'][i])
        r2 = _rmsd(x['atom'].pos.cpu().numpy()[flex], z['atom_pos'][i][flex])
        assert r1 < 0.1 and r2 < 0.1, (i, r1, r2)


@pytest.mark.parametrize('case', list(refpin.CONV_CASES))
def test_conv_backward_bitwise_reproducible(deterministic, monkeypatch, case):
    # PyTorch's own rule for cuBLAS under use_deterministic_algorithms (the library GEMMs of the backward)
    monkeypatch.setenv('CUBLAS_WORKSPACE_CONFIG', ':4096:8')
    from test_reference_pin import _conv_grads, check_conv_grads
    in_ir, out_ir, nf, faster, sh_ir = refpin.CONV_CASES[case]
    conv = TensorProductConvLayer(in_ir, sh_ir, out_ir, nf, residual=False, batch_norm=True, faster=faster)
    refpin.np_fill(conv, 7)
    conv = conv.to(DEV).eval()
    g1, g2 = _conv_grads(conv, case), _conv_grads(conv, case)
    for k in g1:
        assert np.array_equal(g1[k], g2[k]), (case, k)
    check_conv_grads(g1, case, 2e-4)


@pytest.mark.parametrize('mode', ['bf16', 'fp32'])
def test_out_of_range_partial_sums_raise_and_clear(deterministic, mode):
    prod, ref, n, (x, ei, ea, sh) = _sorted_case(24)
    prod.conv_mode = mode
    args = (x.to(DEV), ei.to(DEV), ea.to(DEV), sh.to(DEV))
    with torch.no_grad():
        good = prod(*args, out_nodes=n)
        with pytest.raises(RuntimeError, match='fixed-point range'):
            prod(args[0] * 1e12, *args[1:], out_nodes=n)              # finite, but every partial sum is far beyond 2^31
        again = prod(*args, out_nodes=n)                               # the word was cleared: the next call is clean
    assert torch.equal(good, again)
    assert int(_lib.status_word(DEV).item()) == 0
