"""Decoder of the tensor-core conv's packed weight image (``ddp_tpconv_pack``) and a float64 replay of the kernel's data
flow on top of it (test infrastructure only).

The replay mirrors ``tpconv_umma_kernel`` step by step: the A operand [emb | p1[i1][:ns] | p2[i2][:ns]] with the constant
one in slot ns, rounded to bf16 (hi, and in mode 1 the bf16 remainder lo) the way ``gather_rows`` rounds it; GEMM1 with
the decoded W1 and ReLU; the hidden activations rounded to bf16 hi / lo the way ``convert_hidden`` does; per weight tile
GEMM2 with exactly the products the kernel issues (hi.hi, plus lo.hi + hi.lo in mode 1); and the basis contraction of
the tile's kind.  Everything after the roundings is float64.  ``replay_edges(..., absolute=True)`` runs the same chain
on the absolute values of every factor: the scale against which the kernel's fp32 accumulation error is measured."""
import struct

import numpy as np
import torch

MAGIC = 0x44445055
HEADER = struct.Struct('<I9i3ii3q2iq')      # umma::Header
TILE = struct.Struct('<HBBHBBHHI')          # umma::TileDesc
assert HEADER.size == 96 and TILE.size == 16
KIND_NAMES = ('x*s0', 'dot(xv,s1)', 'x*s1', 'xv*s0', 'cross(xv,s1)', 'C121(xv,s2)')


def pack(spec, w1, b1, w2, b2, ns, mode, sh_dim=None):
    """``ddp_tpconv_pack`` of a spec with host weights in nn.Linear layout, groups sorted by output block as
    ``PackedConv.umma_image`` hands them over -> (status or image size, image bytes or None)."""
    import ctypes as C
    from diffdock_pocket_b200 import _lib
    L = _lib.lib()
    order = sorted(range(len(spec.groups)), key=lambda i: spec.groups[i]['out_off'])
    groups = (_lib.TpGroup * len(order))(*[_lib.TpGroup(**spec.groups[i]) for i in order])
    cdesc = _lib.TpConv(k1=3 * ns, hid=3 * ns, w_numel=spec.weight_numel, n_emb=ns, ns=ns, n_groups=len(spec.groups),
                        f_in=spec.f_in, f_out=spec.f_out, sh_dim=sh_dim or spec.sh_dim, ctab_len=len(spec.ctab))
    ctab = torch.tensor(spec.ctab, dtype=torch.float32)
    w = [t.detach().float().contiguous().cpu() for t in (w1, b1, w2, b2)]
    args = (C.byref(cdesc), groups, ctab.data_ptr(), *[t.data_ptr() for t in w], mode)
    size = L.ddp_tpconv_pack(*args, None)
    if size <= 0:
        return size, None
    out = torch.zeros(size, dtype=torch.uint8)
    rc = L.ddp_tpconv_pack(*args, out.data_ptr())
    return (rc, None) if rc else (size, out.numpy().tobytes())


def bf16_bits_to_f32(u16):
    return (np.asarray(u16, dtype=np.uint16).astype(np.uint32) << 16).view(np.float32)


def decode_operand(buf, off, n_cols, kp, stage_k, mode):
    """One [n_cols x kp] operand written as K-slabs in UMMA no-swizzle core-matrix order -> (hi, lo, next offset).
    hi / lo are float32 [n_cols, kp]; lo is all zero in mode 0 (the image has no lo part there)."""
    hi = np.zeros((n_cols, kp), dtype=np.float32)
    lo = np.zeros((n_cols, kp), dtype=np.float32)
    n_el = n_cols * stage_k
    for ks in range(kp // stage_k):
        for part, dst in enumerate((hi, lo)[:2 if mode else 1]):
            v = bf16_bits_to_f32(np.frombuffer(buf, dtype=np.uint16, count=n_el, offset=off + 2 * n_el * part))
            cm = v.reshape(stage_k // 8, n_cols // 8, 8, 8)                 # [k-chunk][row group][row][elem]
            dst[:, ks * stage_k:(ks + 1) * stage_k] = cm.transpose(1, 2, 0, 3).reshape(n_cols, stage_k)
        off += 2 * n_el * (2 if mode else 1)
    return hi, lo, off


class Image:
    """Decoded packed image: header fields, tile table, W1 / per-tile W2 (hi and lo kept apart), kind-5 tables."""

    def __init__(self, buf):
        buf = bytes(buf)
        (magic, self.mode, self.ns, self.nv, self.ks, self.kp, self.n1, self.stage_k, self.n_tiles, self.n_slabs_per_edge_tile,
         self.f_in, self.f_out, self.n_parts, self.slab_elems_max, self.tiles_off, self.slabs_off, self.total_bytes,
         self.sh_dim, self.n_ctab5, self.ctab5_off) = HEADER.unpack_from(buf, 0)
        assert magic == MAGIC, hex(magic)
        assert len(buf) == self.total_bytes, (len(buf), self.total_bytes)
        assert self.kp == self.n1 == 3 * self.ks and self.kp % self.stage_k == 0
        self.tiles = []
        for t in range(self.n_tiles):
            n_cols, kind, n_rows, out_off, flags, ctab5, x_off, _, _ = TILE.unpack_from(buf, self.tiles_off + 16 * t)
            # flag bit 1 ("swap the last input irrep into slot 0") is reserved: the packer never sets it and the kernel has
            # no code that honours it, so an image with it set would be computed as if it were clear
            assert not flags & 2, f'tile {t}: reserved flag bit 1 is set'
            assert kind <= 5 and n_cols % 16 == 0 and n_rows > 0, (t, kind, n_cols, n_rows)
            assert kind != 5 or ctab5 < self.n_ctab5, (t, ctab5, self.n_ctab5)
            self.tiles.append(dict(n_cols=n_cols, kind=kind, n_rows=n_rows, out_off=out_off, flags=flags, ctab5=ctab5, x_off=x_off))
        self.ctab5 = np.frombuffer(buf, dtype=np.float32, count=45 * self.n_ctab5, offset=self.ctab5_off).reshape(-1, 3, 5, 3).copy()
        self.w1_hi, self.w1_lo, off = decode_operand(buf, self.slabs_off, self.n1, self.kp, self.stage_k, self.mode)
        self.w2_hi, self.w2_lo = [], []
        for td in self.tiles:
            hi, lo, off = decode_operand(buf, off, td['n_cols'], self.kp, self.stage_k, self.mode)
            self.w2_hi.append(hi)
            self.w2_lo.append(lo)
        assert off == self.total_bytes, (off, self.total_bytes)

    def mul(self, kind):
        return self.ns if kind < 2 else self.nv

    def a_slot(self, s, j):
        """K index of feature j of A source s (0 emb, 1 p1, 2 p2)."""
        return s * self.ks + j


def _bf16_split(v32, mode):
    """float32 -> (hi, lo) as the kernel forms them: hi = RN-even bf16(v), lo = RN-even bf16(v - hi) in mode 1 (0 in mode 0)."""
    hi = v32.to(torch.bfloat16).to(torch.float32)
    lo = (v32 - hi).to(torch.bfloat16).to(torch.float32) if mode else torch.zeros_like(v32)
    return hi, lo


def a_operand(img, emb, p1, i1, p2, i2):
    """[E, kp] float32 A operand of the kernel (before its bf16 rounding)."""
    E, ns = emb.shape[0], img.ns
    A = torch.zeros(E, img.kp, dtype=torch.float32, device=emb.device)
    for s, src in enumerate((emb[:, :ns], p1[i1.long(), :ns], p2[i2.long(), :ns])):
        A[:, s * img.ks:s * img.ks + ns] = src
    A[:, ns] = 1.0
    return A


class Replay:
    """Device copies of one image's operands in float64, ready for ``replay_edges``."""

    def __init__(self, img, device):
        d = lambda a: torch.as_tensor(a, dtype=torch.float64, device=device)
        self.img = img
        self.w1_hi, self.w1_lo = d(img.w1_hi), d(img.w1_lo)
        self.w2_hi = d(np.concatenate(img.w2_hi, 0))              # all tiles stacked: [sum n_cols, kp]
        self.w2_lo = d(np.concatenate(img.w2_lo, 0))
        self.col0 = np.cumsum([0] + [td['n_cols'] for td in img.tiles])
        self.ctab5 = d(img.ctab5)


def hidden(rp, A32, absolute=False):
    """GEMM1 + ReLU + the kernel's bf16 rounding of the hidden activations -> (h_hi, h_lo) float64 [E, n1]."""
    img = rp.img
    a_hi, a_lo = (t.double() for t in _bf16_split(A32, img.mode))
    pre = a_hi @ rp.w1_hi.T
    if img.mode:
        pre = pre + a_lo @ rp.w1_hi.T + a_hi @ rp.w1_lo.T
    h = torch.relu(pre).float()           # fp32 in TMEM (exact for the dyadic grid inputs of the replay tests)
    h_hi, h_lo = (t.double() for t in _bf16_split(h, img.mode))
    if absolute:
        h_hi, h_lo = h_hi.abs(), h_lo.abs()
    return h_hi, h_lo


def replay_edges(rp, A32, x_g, sh, absolute=False):
    """Per-edge kernel output [E, f_out] float64, before the in-degree / out_scale factors and the scatter.
    A32: [E, kp] float32 A operand; x_g: [E, f_in] gathered node features; sh: [E, sh_dim] edge harmonics."""
    img = rp.img
    h_hi, h_lo = hidden(rp, A32, absolute)
    w2_hi, w2_lo = (rp.w2_hi.abs(), rp.w2_lo.abs()) if absolute else (rp.w2_hi, rp.w2_lo)
    w = h_hi @ w2_hi.T
    if img.mode:
        w = w + h_lo @ w2_hi.T + h_hi @ w2_lo.T
    f = (lambda t: t.abs()) if absolute else (lambda t: t)
    x, sh = f(x_g.double()), f(sh.double())
    E = x.shape[0]
    s0, s1 = sh[:, 0], sh[:, 1:4]
    out = torch.zeros(E, img.f_out, dtype=torch.float64, device=x.device)
    for t, td in enumerate(img.tiles):
        kind, nr, mul, xo, oo = td['kind'], td['n_rows'], img.mul(td['kind']), td['x_off'], td['out_off']
        wt = w[:, rp.col0[t]:rp.col0[t] + nr * mul].reshape(E, nr, mul)
        if kind in (0, 2):
            xr = x[:, xo:xo + nr]                                  # [E, nr]
        else:
            xr = x[:, xo:xo + 3 * nr].reshape(E, nr, 3)
        if kind == 0:
            out[:, oo:oo + mul] += torch.einsum('erm,er->em', wt, xr * s0[:, None])
        elif kind == 1:
            out[:, oo:oo + mul] += torch.einsum('erm,er->em', wt, (xr * s1[:, None, :]).sum(-1))
        else:
            if kind == 2:
                b = xr[:, :, None] * s1[:, None, :]
            elif kind == 3:
                b = xr * s0[:, None, None]
            elif kind == 4:
                sv = s1[:, None, :].expand_as(xr)
                if absolute:                                       # |a x b| <= the sums of the absolute products
                    b = torch.stack([xr[..., 1] * sv[..., 2] + xr[..., 2] * sv[..., 1], xr[..., 2] * sv[..., 0] + xr[..., 0] * sv[..., 2],
                                     xr[..., 0] * sv[..., 1] + xr[..., 1] * sv[..., 0]], -1)
                else:
                    b = torch.linalg.cross(xr, sv, dim=-1)
            else:
                c5 = f(rp.ctab5[td['ctab5']])                      # [i][j][k]
                b = torch.einsum('ijk,eri,ej->erk', c5, xr, f(sh[:, 4:9]))
            out[:, oo:oo + 3 * mul] += torch.einsum('erm,erk->emk', wt, b).reshape(E, 3 * mul)
    return out


def replay_chunked(rp, A32, x_g, sh, absolute=False, chunk=8192):
    return torch.cat([replay_edges(rp, A32[c:c + chunk], x_g[c:c + chunk], sh[c:c + chunk], absolute)
                      for c in range(0, A32.shape[0], chunk)]) if A32.shape[0] else \
        torch.zeros(0, rp.img.f_out, dtype=torch.float64, device=A32.device)
