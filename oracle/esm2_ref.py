"""Float64 restatement of the ESM-2 forward (fair-esm ``esm.model.esm2.ESM2``, last layer's representation), written from
its equations in plain PyTorch for the tests.  It does not import the product package.

    x_0   = E[tok] * (1 - 0.15 * 0.8) / (1 - r),  r = #<mask> / #non-pad tokens of the sequence; <mask> and pad rows = 0
    layer:  h = LN_1(x);  q = (h W_q^T + b_q) / 8,  k = h W_k^T + b_k,  v = h W_v^T + b_v   (per head, head dim 64)
            q, k <- rotary(q), rotary(k) at positions 0 .. T-1 (0 = BOS)
            a = softmax(q k^T + mask) v,  mask = -inf on keys that are pad tokens
            x = x + a W_o^T + b_o;  x = x + W_2 gelu(W_1 LN_2(x) + b_1) + b_2,  gelu(v) = v / 2 (1 + erf(v / sqrt 2))
    out   = LN_after(x)        (LayerNorm eps 1e-5, affine)

Rotary (fair-esm ``RotaryEmbedding``): inv_freq[i] = 1 / 10000^(2i / 64) (fp32 table), angle[t, i] = float32(t * inv_freq[i]),
emb = cat(angle, angle), rotary(x) = x cos(emb) + rotate_half(x) sin(emb), rotate_half(x) = cat(-x[32:], x[:32]).
"""
import math

import torch

PAD, MASK = 1, 32
HEAD_DIM = 64


def inv_freq(dim=HEAD_DIM):
    return 1.0 / (10000 ** (torch.arange(0, dim, 2).float() / dim))


def rotary(x, positions, freq):
    """x [..., T, 64] -> rotated; angles are formed in fp32 (as the table inputs of fair-esm) and applied in x's dtype."""
    ang = (positions.float()[:, None] * freq.float()[None, :]).to(x.dtype)
    emb = torch.cat([ang, ang], -1)
    half = x.shape[-1] // 2
    rot = torch.cat([-x[..., half:], x[..., :half]], -1)
    return x * emb.cos() + rot * emb.sin()


def embed(weight, tokens, dtype=torch.float64):
    x = weight.to(dtype)[tokens]
    pad = tokens == PAD
    is_mask = tokens == MASK
    ratio = is_mask.sum(-1).to(dtype) / (~pad).sum(-1).to(dtype)
    x = x * (1 - 0.15 * 0.8) / (1 - ratio)[:, None, None]
    return x.masked_fill((pad | is_mask)[..., None], 0.0)


def layer_norm(x, w, b, eps=1e-5):
    mu = x.mean(-1, keepdim=True)
    var = ((x - mu) ** 2).mean(-1, keepdim=True)
    return (x - mu) / torch.sqrt(var + eps) * w.to(x.dtype) + b.to(x.dtype)


def attention_logits(q, k, positions_q, positions_k, freq):
    """Rotary logits q_rot . k_rot for q [.., Tq, 64], k [.., Tk, 64] (scaling left to the caller)."""
    return rotary(q, positions_q, freq) @ rotary(k, positions_k, freq).transpose(-1, -2)


def attention(q, k, v, key_pad, freq):
    """q (already / 8), k, v: [B, H, T, 64]; key_pad [B, T] bool -> [B, H, T, 64]."""
    pos = torch.arange(q.shape[2], device=q.device)
    s = attention_logits(q, k, pos, pos, freq)
    s = s.masked_fill(key_pad[:, None, None, :], float('-inf'))
    return torch.softmax(s, -1) @ v


def forward(sd, tokens, num_layers, num_heads, dtype=torch.float64):
    """sd: fair-esm parameter names (after ``upgrade_state_dict``), tensors on the device of ``tokens``.
    -> [B, T, D] representation of the last layer after ``emb_layer_norm_after``."""
    P = lambda k: sd[k].to(dtype)  # noqa: E731
    x = embed(sd['embed_tokens.weight'], tokens, dtype)
    B, T, D = x.shape
    pad = tokens == PAD
    split = lambda y: y.view(B, T, num_heads, HEAD_DIM).transpose(1, 2)  # noqa: E731
    for i in range(num_layers):
        p = f'layers.{i}.'
        h = layer_norm(x, P(p + 'self_attn_layer_norm.weight'), P(p + 'self_attn_layer_norm.bias'))
        lin = lambda y, n: y @ P(p + n + '.weight').T + P(p + n + '.bias')  # noqa: E731
        q = lin(h, 'self_attn.q_proj') * HEAD_DIM ** -0.5
        k, v = lin(h, 'self_attn.k_proj'), lin(h, 'self_attn.v_proj')
        a = attention(split(q), split(k), split(v), pad, sd[p + 'self_attn.rot_emb.inv_freq'])
        x = x + lin(a.transpose(1, 2).reshape(B, T, D), 'self_attn.out_proj')
        h = layer_norm(x, P(p + 'final_layer_norm.weight'), P(p + 'final_layer_norm.bias'))
        f = lin(h, 'fc1')
        x = x + lin(f * 0.5 * (1.0 + torch.erf(f / math.sqrt(2.0))), 'fc2')
    return layer_norm(x, P('emb_layer_norm_after.weight'), P('emb_layer_norm_after.bias'))
