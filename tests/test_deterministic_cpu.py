"""Host logic of the deterministic mode (no GPU): the accumulation mode is part of the resident-state cache's key and of its
entries, so sampling() never serves a plan, recorded launch program or captured step graph built in the other mode."""
import os
import weakref

import pytest
import torch

from diffdock_pocket_b200 import _lib, inputs, sampling as S

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden')
HEADER = os.path.join(os.path.dirname(GOLD), '..', 'include', 'ddp_b200.h')


class _Model:
    conv_mode, group_convs = 'bf16', True


def _keys(model, conf, det):
    g = inputs.load_graph_npz(os.path.join(GOLD, '3dpf_apo.npz'), name='3dpf_apo')
    gk = [S._graph_key(g, True)] * 3
    return S._cache_key(model, conf, 'cuda:0', 20, True, False, False, True, det, gk)


@pytest.fixture
def cache():
    saved = dict(S._PLAN_CACHE)
    S._PLAN_CACHE.clear()
    try:
        yield S._PLAN_CACHE
    finally:
        S._PLAN_CACHE.clear()
        S._PLAN_CACHE.update(saved)


def _entry(model, conf, det):
    return {'runners': [], 'conf_plans': None, 'streams': [None], 'single': True, 'busy': False, 'sig': None,
            'deterministic': det, 'models': (weakref.ref(model), weakref.ref(conf))}


def test_mode_is_part_of_the_key():
    m, c = _Model(), _Model()
    assert _keys(m, c, False) != _keys(m, c, True)
    assert _keys(m, c, True) == _keys(m, c, True)


@pytest.mark.parametrize('built_det', [False, True])
def test_cache_never_returns_an_entry_of_the_other_mode(cache, built_det):
    m, c = _Model(), _Model()
    cache[_keys(m, c, built_det)] = _entry(m, c, built_det)
    assert S._cache_get(_keys(m, c, built_det), m, c, built_det) is cache[_keys(m, c, built_det)]
    assert S._cache_get(_keys(m, c, not built_det), m, c, not built_det) is None
    # even an entry filed under the other mode's key is refused by the mode it records
    cache[_keys(m, c, not built_det)] = _entry(m, c, built_det)
    assert S._cache_get(_keys(m, c, not built_det), m, c, not built_det) is None


def test_cache_entry_checks_models_and_ownership(cache):
    m, c, other = _Model(), _Model(), _Model()
    k = _keys(m, c, True)
    cache[k] = _entry(m, c, True)
    assert S._cache_get(k, other, c, True) is None
    assert S._cache_get(k, m, other, True) is None
    cache[k]['busy'] = True
    assert S._cache_get(k, m, c, True) is None


def test_mode_follows_the_torch_flag():
    was, warn = torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled()
    try:
        torch.use_deterministic_algorithms(False)
        assert not _lib.deterministic() and _lib.sum_dtype(False) == torch.float32
        torch.use_deterministic_algorithms(True, warn_only=True)
        assert _lib.deterministic() and _lib.sum_dtype(True) == torch.int64
        torch.use_deterministic_algorithms(True)
        assert _lib.deterministic()
    finally:
        torch.use_deterministic_algorithms(was, warn_only=warn)


def test_fixed_point_constants_match_the_header():
    text = open(HEADER).read()
    assert f'#define DDP_ACC_FIXED_SHIFT {_lib.FIXED_SHIFT}' in text
    assert f'#define DDP_STATUS_FIXED_RANGE {_lib.STATUS_FIXED_RANGE}u' in text
    for name in ('ddp_fixed_to_float', 'ddp_tpconv_fp32_fixed', 'ddp_tpconv_umma_fixed', 'ddp_tpconv_umma_group_fixed',
                 'ddp_tp_backward_fixed', 'ddp_node_update_fixed', 'ddp_node_update_multi_fixed'):
        assert name in _lib.EXPORTS and f'{name}(' in text
