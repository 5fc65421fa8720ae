"""ESM-2 receptor embeddings on the device (DESIGN section 12).

DiffDock-Pocket's receptor nodes read the per-residue representation of the last layer of ESM-2 650M
(``receptor.x[:, 1:]``, 1280 columns; the reference computes it with fair-esm in ``utils/esm.py``).  This module is a
fair-esm-compatible ``ESM2`` for the forward pass: the same parameter names, so a fair-esm checkpoint loads into it
(``load_esm2``), and the same output, ``representations[num_layers]``.  The dense projections are library GEMMs
(``torch.addmm``); embedding, layer norms, bias + GELU and the rotary multi-head attention are the kernels of
``csrc/esm.cu``.  No gradients, no LM / contact head, head dimension 64 only, fp32 throughout.  There is no CPU path:
``forward`` needs a CUDA device.
"""
import re

import torch
from torch import nn

from . import _lib
from ._lib import ptr

HEAD_DIM = 64
MAX_RESIDUES = 1022                   # + BOS + EOS = 1024 tokens, the longest sequence the attention kernel takes
LN_EPS = 1e-5


class Alphabet:
    """The ESM-2 vocabulary (fair-esm ``Alphabet.from_architecture('ESM-1b')``): special tokens, residues, ``<mask>``."""
    all_toks = ['<cls>', '<pad>', '<eos>', '<unk>'] + list('LAGVSERTIDPNQKFYMHWCXBUZO.-') + ['<null_1>', '<mask>']
    tok_to_idx = {t: i for i, t in enumerate(all_toks)}
    cls_idx, padding_idx, eos_idx, unk_idx, mask_idx = 0, 1, 2, 3, 32

    def encode(self, seqs):
        """Sequences of one-letter codes -> (tokens int64 [B, T], lengths [B]): BOS + residues + EOS, padded with
        ``<pad>``; ``T`` = longest length.  Characters outside the vocabulary become ``<unk>``.  A sequence longer than
        1022 residues raises ValueError (it is never truncated)."""
        seqs = list(seqs)
        for s in seqs:
            if len(s) > MAX_RESIDUES:
                raise ValueError(f'sequence of {len(s)} residues: ESM-2 takes at most {MAX_RESIDUES} (no silent truncation)')
        lengths = [len(s) + 2 for s in seqs]
        tokens = torch.full((len(seqs), max(lengths, default=2)), self.padding_idx, dtype=torch.int64)
        for b, s in enumerate(seqs):
            ids = [self.tok_to_idx.get(c, self.unk_idx) for c in s]
            tokens[b, :len(s) + 2] = torch.tensor([self.cls_idx] + ids + [self.eos_idx], dtype=torch.int64)
        return tokens, lengths


def rotary_inv_freq(dim=HEAD_DIM):
    """fair-esm ``RotaryEmbedding.inv_freq``, computed the same way in fp32."""
    return 1.0 / (10000 ** (torch.arange(0, dim, 2).float() / dim))


class _Rotary(nn.Module):
    def __init__(self):
        super().__init__()
        self.register_buffer('inv_freq', rotary_inv_freq())


class _SelfAttention(nn.Module):
    def __init__(self, d):
        super().__init__()
        self.q_proj, self.k_proj, self.v_proj, self.out_proj = (nn.Linear(d, d) for _ in range(4))
        self.rot_emb = _Rotary()


class _Layer(nn.Module):
    def __init__(self, d):
        super().__init__()
        self.self_attn = _SelfAttention(d)
        self.self_attn_layer_norm = nn.LayerNorm(d, eps=LN_EPS)
        self.fc1 = nn.Linear(d, 4 * d)
        self.fc2 = nn.Linear(4 * d, d)
        self.final_layer_norm = nn.LayerNorm(d, eps=LN_EPS)


class ESM2(nn.Module):
    """fair-esm ``esm.model.esm2.ESM2`` (token dropout on) without its LM and contact heads; parameter names as after
    ``upgrade_state_dict``.  ``forward(tokens, lengths) -> [B, T, D]`` is ``representations[num_layers]``."""

    def __init__(self, num_layers=33, embed_dim=1280, attention_heads=20):
        super().__init__()
        if embed_dim != HEAD_DIM * attention_heads:
            raise ValueError(f'embed_dim {embed_dim} != {HEAD_DIM} x attention_heads {attention_heads}: only head dimension '
                             f'{HEAD_DIM} is supported')
        self.num_layers, self.embed_dim, self.attention_heads = num_layers, embed_dim, attention_heads
        self.alphabet = Alphabet()
        self.embed_tokens = nn.Embedding(len(Alphabet.all_toks), embed_dim, padding_idx=Alphabet.padding_idx)
        self.layers = nn.ModuleList(_Layer(embed_dim) for _ in range(num_layers))
        self.emb_layer_norm_after = nn.LayerNorm(embed_dim, eps=LN_EPS)
        self._qkv = None

    def _qkv_weights(self):
        """Per layer the Q, K, V projections stacked into one [3D, D] weight and [3D] bias for ONE GEMM, Q scaled by 1/8
        (fair-esm scales q after its bias; a power of two commutes with rounding), and a host copy of the rotary table
        (the attention takes it by value).  Rebuilt when a parameter or buffer changes."""
        key = tuple((p.data_ptr(), p._version) for p in (*self.parameters(), *self.buffers()))
        if self._qkv is None or self._qkv[0] != key:
            packs = []
            for L in self.layers:
                a = L.self_attn
                w = torch.cat([a.q_proj.weight * 0.125, a.k_proj.weight, a.v_proj.weight]).contiguous()
                b = torch.cat([a.q_proj.bias * 0.125, a.k_proj.bias, a.v_proj.bias]).contiguous()
                packs.append((w, b, a.rot_emb.inv_freq.detach().float().cpu().contiguous()))
            self._qkv = (key, packs)
        return self._qkv[1]

    @torch.no_grad()
    def forward(self, tokens, lengths):
        """tokens int64 [B, T] (``Alphabet.encode``; pads only after EOS), lengths [B] = non-pad tokens per sequence (host
        list or tensor) -> [B, T, D] fp32 on the parameters' device.  Pad rows are computed as fair-esm computes them."""
        dev = self.embed_tokens.weight.device
        if dev.type != 'cuda':
            raise RuntimeError('ESM2.forward runs on a CUDA device (there is no CPU path); move the module with .to("cuda")')
        B, T = tokens.shape
        if not 1 <= T <= MAX_RESIDUES + 2:
            raise ValueError(f'{T} tokens per sequence: 1 .. {MAX_RESIDUES + 2} supported')
        lens = torch.as_tensor(lengths, dtype=torch.int32).cpu()
        if lens.shape != (B,) or int(lens.min()) < 1 or int(lens.max()) > T:
            raise ValueError(f'lengths must be {B} values in 1 .. {T}')
        if tokens.device.type == 'cpu':
            if int(tokens.min()) < 0 or int(tokens.max()) >= len(Alphabet.all_toks):
                raise ValueError('token index outside the ESM-2 vocabulary')
            if not torch.equal((tokens != Alphabet.padding_idx).sum(1).to(torch.int32), lens):
                raise ValueError('lengths must count the non-pad tokens of each sequence')
        D, H, N = self.embed_dim, self.attention_heads, B * T
        L = _lib.lib()
        st = _lib.stream_ptr()
        tok = tokens.to(device=dev, dtype=torch.int64).contiguous()
        lens_d = lens.to(dev)
        f32 = dict(dtype=torch.float32, device=dev)
        x, h, a = (torch.empty(N, D, **f32) for _ in range(3))
        qkv, f = torch.empty(N, 3 * D, **f32), torch.empty(N, 4 * D, **f32)
        _lib.check(L.ddp_esm_embed(ptr(tok), B, T, ptr(self.embed_tokens.weight), self.embed_tokens.num_embeddings, D,
                                   Alphabet.padding_idx, Alphabet.mask_idx, ptr(x), st), 'ddp_esm_embed')
        pending = None                  # bias of the last Linear added into x, applied by the next layer norm
        for layer, (w_qkv, b_qkv, freq) in zip(self.layers, self._qkv_weights()):
            layer_norm(x, pending, layer.self_attn_layer_norm, h)
            torch.addmm(b_qkv, h, w_qkv.t(), out=qkv)
            attention(qkv, lens_d, freq, B, T, H, a)
            x.addmm_(a, layer.self_attn.out_proj.weight.t())
            layer_norm(x, layer.self_attn.out_proj.bias, layer.final_layer_norm, h)
            torch.mm(h, layer.fc1.weight.t(), out=f)
            _lib.check(L.ddp_bias_gelu(ptr(f), ptr(layer.fc1.bias), N, 4 * D, st), 'ddp_bias_gelu')
            x.addmm_(f, layer.fc2.weight.t())
            pending = layer.fc2.bias
        out = torch.empty(N, D, **f32)
        layer_norm(x, pending, self.emb_layer_norm_after, out)
        return out.view(B, T, D)


def layer_norm(x, residual_bias, ln, y):
    """``ddp_layer_norm``: y = ln(x), after x += residual_bias when that is given."""
    _lib.check(_lib.lib().ddp_layer_norm(ptr(x), ptr(residual_bias), ptr(ln.weight), ptr(ln.bias), x.shape[0], x.shape[1],
                                         ln.eps, ptr(y), _lib.stream_ptr()), 'ddp_layer_norm')


def attention(qkv, lengths, freq, B, T, H, out):
    """``ddp_esm_attention`` on the [B * T, 3D] output of the stacked Q / K / V GEMM -> out [B * T, D]; freq: the 32
    inverse frequencies, fp32 on the host."""
    D = H * HEAD_DIM
    base = qkv.data_ptr()
    _lib.check(_lib.lib().ddp_esm_attention(base, base + 4 * D, base + 8 * D, 3 * D, ptr(lengths),
                                            _lib.C.cast(freq.data_ptr(), _lib.C.POINTER(_lib.f32)), B, T, H, HEAD_DIM, ptr(out),
                                            D, _lib.stream_ptr()), 'ddp_esm_attention')


# ------------------------------------------------------------------------------------------------ checkpoints
_PREFIX = re.compile(r'^(encoder\.sentence_encoder\.|encoder\.)')
_DROPPED = ('lm_head.', 'contact_head.')


def _cfg_get(cfg, name):
    return cfg[name] if isinstance(cfg, dict) else getattr(cfg, name)


def load_esm2(source):
    """A fair-esm ESM-2 checkpoint -> ``ESM2`` on the CPU (move it with ``.to('cuda')``).

    ``source``: a checkpoint path (``{'model': state_dict, 'cfg': {'model': {...}}}``, read with
    ``torch.load(weights_only=True)`` only), such a dict, or a plain state dict.  Keys lose the prefixes
    ``encoder.sentence_encoder.`` / ``encoder.``; ``lm_head.*`` and ``contact_head.*`` are dropped; every other key must
    be one of the module's and every one of the module's must be present, and each ``rot_emb.inv_freq`` must equal the
    recomputed table -- anything else raises.  Without ``cfg`` the shape is inferred from the tensors (heads = dim / 64)."""
    if isinstance(source, (str, bytes)) or hasattr(source, '__fspath__'):
        try:
            source = torch.load(source, map_location='cpu', weights_only=True)
        except Exception as e:  # noqa: BLE001 -- any refusal of the restricted unpickler ends here
            raise RuntimeError(f'{source!r} cannot be read with torch.load(weights_only=True) ({e}); if you trust the file, '
                               'load it yourself and pass the resulting dict to load_esm2') from e
    if not isinstance(source, dict):
        raise TypeError(f'load_esm2 takes a path or a dict, not {type(source).__name__}')
    cfg = None
    if 'model' in source and isinstance(source['model'], dict):
        if 'cfg' in source:
            cfg = _cfg_get(source['cfg'], 'model')
        source = source['model']
    sd = {_PREFIX.sub('', k): v for k, v in source.items()}
    sd = {k: v for k, v in sd.items() if not k.startswith(_DROPPED)}
    if cfg is not None:
        if not _cfg_get(cfg, 'token_dropout'):
            raise ValueError('checkpoint has token_dropout = False: only ESM-2 with token dropout is supported')
        layers, dim, heads = (int(_cfg_get(cfg, n)) for n in ('encoder_layers', 'encoder_embed_dim', 'encoder_attention_heads'))
    else:
        if 'embed_tokens.weight' not in sd:
            raise KeyError('state dict has no embed_tokens.weight')
        dim = int(sd['embed_tokens.weight'].shape[1])
        layers = len({int(m.group(1)) for k in sd for m in [re.match(r'layers\.(\d+)\.', k)] if m})
        heads = dim // HEAD_DIM
    model = ESM2(layers, dim, heads)
    want = model.state_dict()
    missing, unexpected = sorted(set(want) - set(sd)), sorted(set(sd) - set(want))
    if missing or unexpected:
        raise KeyError(f'ESM-2 checkpoint does not match ESM2({layers}, {dim}, {heads}): missing {missing[:8]}, '
                       f'unexpected {unexpected[:8]}')
    ref = rotary_inv_freq()
    for k in want:
        if k.endswith('rot_emb.inv_freq') and not torch.equal(sd[k].float().cpu(), ref):
            raise ValueError(f'{k} differs from the rotary table 1 / 10000^(2i / {HEAD_DIM})')
    model.load_state_dict(sd, strict=True)
    return model.eval()


# ------------------------------------------------------------------------------------------------ batching
def embed_sequences(model, seqs, max_tokens=16384):
    """Per sequence the last-layer representation of its residues: a list of [L_i, D] fp32 tensors on the model's
    device (rows 1 .. L_i of the output: BOS and EOS dropped), in input order.  Sequences are sorted by length and packed
    into padded batches of at most ``max_tokens`` tokens (B x T; a single sequence always fits)."""
    seqs = list(seqs)
    alphabet = Alphabet()
    alphabet.encode(seqs)                      # length check of every sequence before any work
    order = sorted(range(len(seqs)), key=lambda i: -len(seqs[i]))
    out = [None] * len(seqs)
    i = 0
    while i < len(order):
        T = len(seqs[order[i]]) + 2
        n = max(1, min(len(order) - i, max_tokens // T))
        idx = order[i:i + n]
        tokens, lengths = alphabet.encode([seqs[j] for j in idx])
        rep = model(tokens, lengths)
        for b, j in enumerate(idx):
            out[j] = rep[b, 1:len(seqs[j]) + 1]
        i += n
    return out
