"""ESM-2 receptor embeddings, host side: the alphabet and ``encode``, chain sequences of the 3dpf pocket PDB, the
checkpoint loader's key policy, properties of the float64 oracle (``oracle/esm2_ref.py``) and the graph builder with and
without language-model rows.

fair-esm is not installed here: compatibility is pinned to the specification the module documents (vocabulary order,
parameter names after ``upgrade_state_dict``, token-dropout scaling, rotary tables), not to fair-esm itself."""
import os

import numpy as np
import pytest
import torch

from diffdock_pocket_b200 import esm, inputs
from oracle import esm2_ref as R

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden')
PDB = os.path.join(GOLD, '3dpf_pocket', '3dpf_protein.pdb')
SDF = os.path.join(GOLD, '3dpf_pocket', '3dpf_ligand.sdf')


# ------------------------------------------------------------------------------------------------ alphabet
def test_alphabet_order():
    A = esm.Alphabet
    assert A.all_toks[:4] == ['<cls>', '<pad>', '<eos>', '<unk>']
    assert ''.join(A.all_toks[4:31]) == 'LAGVSERTIDPNQKFYMHWCXBUZO.-'
    assert A.all_toks[31:] == ['<null_1>', '<mask>'] and len(A.all_toks) == 33
    assert (A.cls_idx, A.padding_idx, A.eos_idx, A.unk_idx, A.mask_idx) == (0, 1, 2, 3, 32)
    assert (R.PAD, R.MASK) == (A.padding_idx, A.mask_idx)


def test_encode_bos_eos_pad():
    tok, lens = esm.Alphabet().encode(['MK', 'LAGVS'])
    assert lens == [4, 7] and tok.dtype == torch.int64 and tok.shape == (2, 7)
    assert tok[0].tolist() == [0, 20, 17, 2, 1, 1, 1]
    assert tok[1].tolist() == [0, 4, 5, 6, 7, 8, 2]


def test_encode_length_limit():
    a = esm.Alphabet()
    tok, lens = a.encode(['A' * 1022])
    assert tok.shape == (1, 1024) and lens == [1024]
    with pytest.raises(ValueError):
        a.encode(['A' * 10, 'A' * 1023])


# ------------------------------------------------------------------------------------------------ chains
def test_chain_sequences_of_3dpf():
    res = inputs.parse_pdb_heavy(PDB)
    chains = inputs.chain_sequences(res)
    seen = []
    for cid, seq, idx in chains:
        assert len(seq) == len(idx) == sum(r['chain'] == cid for r in res)
        assert all(res[i]['chain'] == cid for i in idx) and idx == sorted(idx)
        assert set(seq) <= set('ACDEFGHIKLMNPQRSTVWY')
        seen += idx
    assert sorted(seen) == list(range(len(res)))
    assert [c for c, _, _ in chains] == list(dict.fromkeys(r['chain'] for r in res))
    assert inputs.chain_sequences([dict(name='MSE', chain='B'), dict(name='GLY', chain='B')])[0][1] == 'MG'


# ------------------------------------------------------------------------------------------------ loader
def _tiny_sd(layers=2, dim=128, heads=2, seed=0):
    torch.manual_seed(seed)
    return esm.ESM2(layers, dim, heads).state_dict()


def _fair_esm_ckpt(sd, token_dropout=True):
    model = {('encoder.sentence_encoder.' if not k.startswith('lm_head') else 'encoder.') + k: v.clone() for k, v in sd.items()}
    model['encoder.lm_head.weight'] = torch.zeros(33, 128)
    model['encoder.lm_head.bias'] = torch.zeros(33)
    model['encoder.sentence_encoder.contact_head.regression.weight'] = torch.zeros(1, 4)
    cfg = dict(model=dict(encoder_layers=2, encoder_embed_dim=128, encoder_attention_heads=2, token_dropout=token_dropout))
    return dict(model=model, cfg=cfg)


def _same(m, sd):
    got = m.state_dict()
    assert set(got) == set(sd) and all(torch.equal(got[k], sd[k]) for k in sd)


def test_load_prefixed_checkpoint_with_cfg(tmp_path):
    sd = _tiny_sd()
    m = esm.load_esm2(_fair_esm_ckpt(sd))
    assert (m.num_layers, m.embed_dim, m.attention_heads) == (2, 128, 2)
    _same(m, sd)
    path = tmp_path / 'esm2_tiny.pt'
    torch.save(_fair_esm_ckpt(sd), path)
    _same(esm.load_esm2(str(path)), sd)


def test_load_plain_state_dict_infers_shape():
    sd = _tiny_sd()
    extra = dict(sd, **{'lm_head.dense.weight': torch.zeros(128, 128), 'contact_head.regression.bias': torch.zeros(1)})
    m = esm.load_esm2(extra)
    assert (m.num_layers, m.embed_dim, m.attention_heads) == (2, 128, 2)
    _same(m, sd)


def test_load_rejects_bad_checkpoints():
    sd = _tiny_sd()
    missing = dict(sd)
    del missing['layers.1.fc2.bias']
    with pytest.raises(KeyError):
        esm.load_esm2(missing)
    with pytest.raises(KeyError):
        esm.load_esm2(dict(sd, **{'layers.0.self_attn.bias_k': torch.zeros(128)}))
    bad = dict(sd)
    bad['layers.0.self_attn.rot_emb.inv_freq'] = bad['layers.0.self_attn.rot_emb.inv_freq'] * 1.001
    with pytest.raises(ValueError):
        esm.load_esm2(bad)
    with pytest.raises(ValueError):
        esm.load_esm2(_fair_esm_ckpt(sd, token_dropout=False))


def test_load_refuses_unrestricted_pickle(tmp_path):
    path = tmp_path / 'pickled.pt'
    torch.save(dict(model=_tiny_sd(), cfg=dict(model=object.__new__(_Opaque))), path)
    with pytest.raises(RuntimeError, match='weights_only'):
        esm.load_esm2(str(path))


class _Opaque:
    pass


def test_module_rejects_other_head_dims():
    with pytest.raises(ValueError):
        esm.ESM2(2, 96, 2)
    with pytest.raises(RuntimeError):
        esm.ESM2(1, 128, 2)(*esm.Alphabet().encode(['MK']))


# ------------------------------------------------------------------------------------------------ oracle properties
def test_oracle_padding_invariance():
    sd = _tiny_sd(seed=1)
    tok, _ = esm.Alphabet().encode(['MKTAYIAKQR', 'LAGVSERTIDPNQKFYMHW'])
    alone, _ = esm.Alphabet().encode(['MKTAYIAKQR'])
    both = R.forward(sd, tok, 2, 2)
    one = R.forward(sd, alone, 2, 2)
    assert torch.allclose(both[0, :12], one[0], rtol=0, atol=1e-12)


def test_oracle_rotary_logits_depend_on_relative_position():
    g = torch.Generator().manual_seed(0)
    q, k = torch.randn(1, 64, generator=g, dtype=torch.float64), torch.randn(1, 64, generator=g, dtype=torch.float64)
    f = R.inv_freq()
    logit = lambda a, b: R.attention_logits(q, k, torch.tensor([a]), torch.tensor([b]), f).item()  # noqa: E731
    qk = float(q.norm() * k.norm())
    for shift in (1, 7, 300):           # exact up to the fp32 rounding of the angles (relative 2^-24 of t * inv_freq)
        assert abs(logit(3 + shift, 10 + shift) - logit(3, 10)) < 2 * 2 ** -24 * (10 + shift) * qk
    assert abs(logit(3, 10) - logit(3, 11)) > 1e-3


def test_oracle_token_dropout_scale():
    sd = _tiny_sd()
    W = sd['embed_tokens.weight'].double()
    tok, _ = esm.Alphabet().encode(['MKTAY', 'LA'])
    x = R.embed(sd['embed_tokens.weight'], tok)
    assert torch.equal(x[0], W[tok[0]] * 0.88)
    assert torch.equal(x[1, :4], W[tok[1, :4]] * 0.88) and not x[1, 4:].any()
    tok[0, 2] = esm.Alphabet.mask_idx                        # 1 of 7 non-pad tokens masked
    x = R.embed(sd['embed_tokens.weight'], tok)
    assert not x[0, 2].any() and torch.equal(x[0, 1], W[tok[0, 1]] * 0.88 / (1 - 1 / 7))


# ------------------------------------------------------------------------------------------------ graph builder
def _graph(**kw):
    atoms, bonds = inputs.parse_sdf(SDF)
    res = inputs.parse_pdb_heavy(PDB)
    return inputs.build_complex_graph(inputs.ligand_graph_from_sdf(atoms, bonds), res, name='3dpf', flexible='auto', **kw), res


def test_build_complex_graph_default_unchanged():
    g, res = _graph()
    n = g['receptor'].x.shape[0]
    want = torch.from_numpy(np.random.RandomState(1234).randn(n, 1280).astype(np.float32) * 0.25)
    assert torch.equal(g['receptor'].x[:, 1:], want)
    g2 = inputs.load_example_3dpf(os.path.dirname(PDB))
    for k in ('receptor', 'atom', 'ligand'):
        assert torch.equal(g[k].x, g2[k].x) and torch.equal(g[k].pos, g2[k].pos)


def test_build_complex_graph_takes_lm_rows():
    g0, res = _graph()
    lm = torch.arange(len(res), dtype=torch.float32)[:, None] + torch.linspace(0, 0.5, 1280)[None]
    g, _ = _graph(lm_embeddings=lm)
    rows = (g['receptor'].x[:, 1] - 0).round().long()
    assert torch.equal(g['receptor'].x[:, 1:], lm[rows])
    assert len(set(rows.tolist())) == g['receptor'].x.shape[0] and rows.tolist() == sorted(rows.tolist())
    assert torch.equal(g['receptor'].x[:, :1], g0['receptor'].x[:, :1])
    assert torch.equal(g['receptor'].pos, g0['receptor'].pos)
    with pytest.raises(ValueError):
        _graph(lm_embeddings=lm[:-1])
