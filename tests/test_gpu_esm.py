"""ESM-2 embeddings on the device: each kernel of ``csrc/esm.cu`` against float64 (``|got - ref| <= 1e-5 max|ref|`` per
row, repeats bitwise equal, argument errors), the whole ``esm.ESM2`` forward against the float64 oracle
(``oracle/esm2_ref.py``, ``|got - ref| <= 1e-4 max|ref row|``) at 2 and 33 layers, and receptor embeddings of the 3dpf
pocket through graph building, the static node embedding, one score-model forward and a short ``sampling()`` call.

fair-esm is not installed here: compatibility is pinned to the specification the module documents, not to fair-esm
itself."""
import copy
import os
from functools import partial

import numpy as np
import pytest
import torch

import _common as T
from diffdock_pocket_b200 import _lib, diffusion_utils as du, esm, inputs, sampling as ps
from diffdock_pocket_b200._lib import ptr
from diffdock_pocket_b200.score_model import static_embed
from oracle import diffusion_ref as D, esm2_ref as R

pytestmark = pytest.mark.gpu
DEV = torch.device('cuda:0')
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden')


def _row_gate(got, ref, tol):
    got, ref = got.double().cpu().reshape(-1, got.shape[-1]), ref.double().cpu().reshape(-1, ref.shape[-1])
    err = (got - ref).abs().max(1).values / ref.abs().max(1).values.clamp(min=1e-30)
    assert float(err.max()) <= tol, float(err.max())


def _st():
    return _lib.stream_ptr()


# ------------------------------------------------------------------------------------------------ kernels
@pytest.mark.parametrize('with_mask', [False, True])
def test_embed_kernel(with_mask):
    g = torch.Generator().manual_seed(0)
    W = torch.randn(33, 1280, generator=g)
    tok, _ = esm.Alphabet().encode(['MKTAYIAKQRQISFVKSHFSRQ', 'LAGV', 'ACDEFGHIKLMNPQRSTVWY' * 2])
    if with_mask:
        tok[0, [3, 5, 9]] = 32
        tok[2, 1] = 32
    W_d, tok_d = W.to(DEV), tok.to(DEV)
    outs = []
    for _ in range(2):
        out = torch.empty(*tok.shape, 1280, device=DEV)
        _lib.check(_lib.lib().ddp_esm_embed(ptr(tok_d), tok.shape[0], tok.shape[1], ptr(W_d), 33, 1280, 1, 32, ptr(out), _st()), 'embed')
        outs.append(out)
    ref = R.embed(W, tok)
    got = outs[0].cpu().double()
    zero = (tok == 1) | (tok == 32)
    assert not got[zero].any() and not ref[zero].any()
    _row_gate(got[~zero], ref[~zero], 1e-5)
    assert torch.equal(outs[0], outs[1])


@pytest.mark.parametrize('in_place,residual', [(False, False), (True, False), (False, True)])   # residual + in place: rejected
def test_layer_norm_kernel(in_place, residual):
    g = torch.Generator().manual_seed(1)
    x = (torch.randn(37, 1280, generator=g) * 3 + 1.5).to(DEV)
    w, b, rb = (torch.randn(1280, generator=g).to(DEV) for _ in range(3))
    want_x = x.double() + (rb.double() if residual else 0)
    ref = R.layer_norm(want_x, w, b)
    runs = []
    for _ in range(2):
        xi = x.clone()
        y = xi if in_place else torch.empty_like(x)
        _lib.check(_lib.lib().ddp_layer_norm(ptr(xi), ptr(rb) if residual else None, ptr(w), ptr(b), 37, 1280, 1e-5, ptr(y), _st()), 'ln')
        runs.append((xi.clone(), y.clone()))
    _row_gate(runs[0][1], ref, 1e-5)
    if residual:
        _row_gate(runs[0][0], want_x, 1e-6)
    assert torch.equal(runs[0][1], runs[1][1])


def test_bias_gelu_kernel():
    g = torch.Generator().manual_seed(2)
    x = (torch.randn(29, 5120, generator=g) * 2).to(DEV)
    b = torch.randn(5120, generator=g).to(DEV)
    v = x.double() + b.double()
    ref = v * 0.5 * (1 + torch.erf(v / np.sqrt(2)))
    runs = []
    for _ in range(2):
        y = x.clone()
        _lib.check(_lib.lib().ddp_bias_gelu(ptr(y), ptr(b), 29, 5120, _st()), 'gelu')
        runs.append(y)
    _row_gate(runs[0], ref, 1e-5)
    assert torch.equal(runs[0], runs[1])


def _attention(q, k, v, lengths, B, T_, H):
    D = H * 64
    out = torch.empty(B * T_, D, device=DEV)
    freq = R.inv_freq().contiguous()
    rc = _lib.lib().ddp_esm_attention(ptr(q), ptr(k), ptr(v), D, ptr(lengths), _lib.C.cast(freq.data_ptr(), _lib.C.POINTER(_lib.f32)),
                                      B, T_, H, 64, ptr(out), D, _st())
    _lib.check(rc, 'attention')
    return out


@pytest.mark.parametrize('H', [2, 20])
@pytest.mark.parametrize('T_', [1, 2, 63, 64, 65, 1024])
def test_attention_kernel(T_, H):
    B, D = 3, H * 64
    g = torch.Generator().manual_seed(T_ * 7 + H)
    lens = [T_, max(1, T_ // 2), max(1, T_ - 5)]
    q, k, v = (torch.randn(B * T_, D, generator=g) for _ in range(3))
    q = q * 0.125 * 4                                   # logits of a few units, as in a trained model
    lens_d = torch.tensor(lens, dtype=torch.int32, device=DEV)
    qd, kd, vd = q.to(DEV), k.to(DEV), v.to(DEV)
    got = _attention(qd, kd, vd, lens_d, B, T_, H)
    again = _attention(qd, kd, vd, lens_d, B, T_, H)
    assert torch.equal(got, again)
    split = lambda y: y.to(DEV, torch.float64).view(B, T_, H, 64).transpose(1, 2)  # noqa: E731
    pad = (torch.arange(T_)[None, :] >= torch.tensor(lens)[:, None]).to(DEV)
    ref = R.attention(split(q), split(k), split(v), pad, R.inv_freq().to(DEV)).transpose(1, 2).reshape(B * T_, D)
    _row_gate(got, ref, 1e-5)


def test_argument_errors():
    L = _lib.lib()
    x = torch.zeros(4 * 128 * 3, device=DEV)
    lens = torch.ones(1, dtype=torch.int32, device=DEV)
    freq = R.inv_freq().contiguous()
    fp = _lib.C.cast(freq.data_ptr(), _lib.C.POINTER(_lib.f32))
    args = lambda **o: dict(dict(q=ptr(x), k=ptr(x), v=ptr(x), ld=128, lens=ptr(lens), f=fp, B=1, T=4, H=2, hd=64, out=ptr(x), ldo=128), **o)  # noqa: E731
    call = lambda a: L.ddp_esm_attention(a['q'], a['k'], a['v'], a['ld'], a['lens'], a['f'], a['B'], a['T'], a['H'], a['hd'], a['out'], a['ldo'], _st())  # noqa: E731
    assert call(args()) == 0
    assert call(args(hd=32, ld=64, ldo=64)) == -3
    assert call(args(T=1025)) < 0
    assert call(args(q=None)) == -1 and call(args(lens=None)) == -1 and call(args(f=None)) == -1
    assert L.ddp_layer_norm(None, None, ptr(x), ptr(x), 1, 128, 1e-5, ptr(x), _st()) == -1
    assert L.ddp_layer_norm(ptr(x), ptr(x), ptr(x), ptr(x), 1, 128, 1e-5, ptr(x), _st()) == -1     # residual + in place
    assert L.ddp_layer_norm(ptr(x), None, ptr(x), ptr(x), 1, 4096, 1e-5, ptr(x), _st()) < 0
    assert L.ddp_bias_gelu(ptr(x), None, 1, 128, _st()) == -1
    assert L.ddp_esm_embed(None, 1, 4, ptr(x), 33, 128, 1, 32, ptr(x), _st()) == -1
    torch.cuda.synchronize()


# ------------------------------------------------------------------------------------------------ whole model
def _model(layers, seed=0):
    torch.manual_seed(seed)
    m = esm.ESM2(layers, 1280, 20)
    with torch.no_grad():                  # non-trivial norms and biases, so every parameter is exercised
        for n, p in m.named_parameters():
            if n.endswith('bias'):
                p.normal_(0, 0.05)
            elif 'layer_norm' in n:
                p.normal_(1, 0.1)
    return m.to(DEV)


def _check_model(m, seqs, mask=None):
    tok, lens = esm.Alphabet().encode(seqs)
    if mask is not None:
        tok[mask] = 32
    got = m(tok, lens)
    again = m(tok, lens)
    assert torch.equal(got, again)
    sd = {k: v.double() for k, v in m.state_dict().items()}
    ref = R.forward(sd, tok.to(DEV), m.num_layers, m.attention_heads)
    err = (got.double() - ref).abs() / ref.abs().max(-1, keepdim=True).values
    assert float(err.max()) <= 1e-4, float(err.max())
    return got


def _seq(n, seed):
    rng = np.random.RandomState(seed)
    return ''.join(rng.choice(list('ACDEFGHIKLMNPQRSTVWY'), n))


def test_model_two_layers():
    _check_model(_model(2), [_seq(150, 0), _seq(61, 1), _seq(7, 2)], mask=(torch.tensor([0, 0, 1]), torch.tensor([5, 40, 3])))


def test_model_full_depth():
    m = _model(33, seed=3)
    one = _check_model(m, [_seq(300, 4)])
    batch = _check_model(m, [_seq(300, 4), _seq(120, 5), _seq(233, 6)])
    assert torch.allclose(batch[0], one[0], rtol=0, atol=1e-4 * float(one[0].abs().max()))


def test_embed_sequences_matches_single_calls():
    m = _model(2, seed=5)
    seqs = [_seq(40, 7), _seq(90, 8), _seq(3, 9)]
    reps = esm.embed_sequences(m, seqs, max_tokens=100)      # forces several batches
    for s, r in zip(seqs, reps):
        tok, lens = esm.Alphabet().encode([s])
        want = m(tok, lens)[0, 1:len(s) + 1]
        assert r.shape == (len(s), 1280)
        assert torch.allclose(r, want, rtol=0, atol=1e-5 * float(want.abs().max()))


# ------------------------------------------------------------------------------------------------ end to end
def test_receptor_embeddings_through_the_score_model():
    lm_model = _model(2, seed=6)
    pdb_dir = os.path.join(GOLD, '3dpf_pocket')
    residues = inputs.parse_pdb_heavy(os.path.join(pdb_dir, '3dpf_protein.pdb'))
    lm = inputs.receptor_embeddings(lm_model, residues)
    assert lm.shape == (len(residues), 1280) and torch.isfinite(lm).all()
    for cid, seq, idx in inputs.chain_sequences(residues):          # rows are the chains' own embeddings
        want = esm.embed_sequences(lm_model, [seq])[0]
        assert torch.allclose(lm[idx], want, rtol=0, atol=1e-5 * float(want.abs().max()))
    g = inputs.load_example_3dpf(pdb_dir, esm_model=lm_model)
    atoms, bonds = inputs.parse_sdf(os.path.join(pdb_dir, '3dpf_ligand.sdf'))
    g2 = inputs.build_complex_graph(inputs.ligand_graph_from_sdf(atoms, bonds), residues, name='3dpf', flexible='auto', lm_embeddings=lm)
    assert torch.equal(g['receptor'].x, g2['receptor'].x)

    m, c, om, oc, sa, ca = T.models(DEV, small=True)
    enc = m.rec_node_embedding
    rx = g['receptor'].x
    got = static_embed(enc.static_pack(DEV), rx[:, :1], rx[:, 1:], DEV)
    want = copy.deepcopy(enc).double().static_part(rx[:, :1].long().to(DEV), rx[:, 1:].double().to(DEV))
    assert T.rel_err(got, want) < 1e-5
    noise = inputs.build_complex_graph(inputs.ligand_graph_from_sdf(atoms, bonds), residues, name='3dpf', flexible='auto')
    other = static_embed(enc.static_pack(DEV), rx[:, :1], noise['receptor'].x[:, 1:], DEV)
    assert T.rel_err(other, got) > 1e-2                              # the rows reach the embedding

    dl = T.randomized_list(g, 2, sa, seed=0)
    m.conv_mode = 'fp32'
    with torch.no_grad():
        outs = m(T.batch_at(dl, 0.5))
    assert all(torch.isfinite(o).all() for o in outs)
    sch = D.get_t_schedule(4)
    torch.manual_seed(0)
    got, conf = ps.sampling(copy.deepcopy(dl), m, 4, sch, sch, sch, sch, DEV, partial(du.t_to_sigma, args=sa), sa,
                            confidence_model=c, filtering_model_args=ca, batch_size=2, max_steps=2)
    assert all(torch.isfinite(d['ligand'].pos).all() for d in got) and torch.isfinite(torch.as_tensor(conf)).all()
