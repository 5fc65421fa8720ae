"""CPU check of the tensor-core weight image (ddp_tpconv_pack): decode the UMMA core-matrix slabs and the tile
table (tests/_umma_image.py), replay the kernel's data flow (A operand with bias slot -> GEMM1 -> ReLU -> per-tile GEMM2 ->
basis contraction, kind-5 coupling tables for sh_lmax = 2) and compare with the oracle conv.  Validates layout, tile
schedule, folded biases and folded path normalisation without a GPU; the kernel itself is covered by the -m gpu tests
(tests/test_gpu_umma_replay.py replays the same decoded image against it)."""
import numpy as np
import pytest
import torch

import _umma_image as U
from diffdock_pocket_b200.score_model import TensorProductConvLayer
from oracle import e3nn_mini as E
from oracle.score_model_ref import TensorProductConvLayer as RefConv


def _irreps(ns, nv, layer):
    seq = [f'{ns}x0e', f'{ns}x0e + {nv}x1o', f'{ns}x0e + {nv}x1o + {nv}x1e', f'{ns}x0e + {nv}x1o + {nv}x1e + {ns}x0o']
    return seq[min(layer, 3)], seq[min(layer + 1, 3)]


@pytest.mark.parametrize('ns,nv,layer,sh_lmax', [(60, 10, 3, 1), (60, 10, 0, 1), (60, 10, 1, 1), (60, 10, 2, 1), (24, 6, 3, 1),
                                                 (16, 4, 3, 1), (16, 4, 3, 2), (16, 4, 1, 2)])
@pytest.mark.parametrize('mode', [0, 1])
def test_packed_image_replays_conv(ns, nv, layer, sh_lmax, mode):
    in_ir, out_ir = _irreps(ns, nv, layer)
    sh_ir = '1x0e+1x1o' if sh_lmax == 1 else '1x0e+1x1o+1x2e'
    faster = sh_lmax == 1                   # sh_lmax = 2: e3nn FullyConnectedTensorProduct, kind-5 tiles
    torch.manual_seed(0)
    prod = TensorProductConvLayer(in_ir, sh_ir, out_ir, 3 * ns, residual=False, batch_norm=False, faster=faster)
    ref = RefConv(in_ir, sh_ir, out_ir, 3 * ns, residual=False, batch_norm=False, faster=faster)
    ref.load_state_dict(prod.state_dict())
    spec = prod.tp.spec
    size, buf = U.pack(spec, prod.fc[0].weight, prod.fc[0].bias, prod.fc[3].weight, prod.fc[3].bias, ns, mode)
    assert buf is not None, size
    img = U.Image(buf)
    assert (img.mode, img.ns, img.nv, img.sh_dim) == (mode, ns, nv, 4 if sh_lmax == 1 else 9)
    kinds = {td['kind'] for td in img.tiles}
    assert (5 in kinds) == (sh_lmax == 2), kinds
    # one accumulation per output block; zero padding columns
    seen_first = set()
    for td, hi, lo in zip(img.tiles, img.w2_hi, img.w2_lo):
        if td['flags'] & 1:
            assert td['out_off'] not in seen_first
            seen_first.add(td['out_off'])
        assert td['n_rows'] * img.mul(td['kind']) <= td['n_cols']
        assert np.all(hi[td['n_rows'] * img.mul(td['kind']):] == 0) and np.all(lo[td['n_rows'] * img.mul(td['kind']):] == 0)
    if mode == 0:
        assert not img.w1_lo.any() and not any(lo.any() for lo in img.w2_lo)
    # the hidden unit `hid` regenerates the constant one for GEMM2's bias row, every unit above it is zero
    rp = U.Replay(img, 'cpu')
    n_e = 9
    g = torch.Generator().manual_seed(1)
    x = torch.randn(n_e, spec.f_in, generator=g)
    ea = torch.randn(n_e, 3 * ns, generator=g)
    sh = E.spherical_harmonics(sh_ir, torch.randn(n_e, 3, generator=g))
    ident = torch.arange(n_e)
    A = U.a_operand(img, ea[:, :ns], ea[:, ns:2 * ns], ident, ea[:, 2 * ns:], ident)
    h_hi, h_lo = U.hidden(rp, A)
    assert torch.all(h_hi[:, 3 * ns] == 1.0) and torch.all(h_lo[:, 3 * ns] == 0) and torch.all(h_hi[:, 3 * ns + 1:] == 0)
    out = U.replay_edges(rp, A, x, sh).numpy()
    with torch.no_grad():
        want = ref.tp(x.double(), sh.double(), ref.double().fc(ea.double())).numpy()
    err = np.abs(out - want).max() / np.abs(want).max()
    assert err < (2e-5 if mode else 2e-2), err
