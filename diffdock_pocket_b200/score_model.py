"""Host mirrors of the shared classes of the reference's ``models/score_model.py``.

Same class names, constructor arguments and ``state_dict`` keys as the reference
(``TensorProductConvLayer`` models/score_model.py:84-125, ``AtomEncoder`` :54-82, ``OldAtomEncoder``
:17-52, ``GaussianSmearing`` :661-671), but every ``forward`` runs on the ddp_b200 CUDA kernels through
the C ABI (``include/ddp_b200.h``); there is no PyTorch/CPU fallback.
"""
import ctypes as C

import numpy as np
import torch
from torch import nn

from . import _lib, tp as tpmod
from ._lib import ptr

FEATURE_DIMS = {  # datasets/process_mols.py:69-97
    'lig': ([119, 4, 12, 12, 8, 10, 6, 6, 2, 8, 2, 2, 2, 2, 2, 2], 0),
    'rec_atom': ([38, 119, 23, 38], 0),
    'rec_residue': ([38], 0),
}


class GaussianSmearing(nn.Module):
    def __init__(self, start=0.0, stop=5.0, num_gaussians=50):
        super().__init__()
        offset = torch.linspace(start, stop, num_gaussians)
        self.coeff = -0.5 / (offset[1] - offset[0]).item() ** 2
        self.register_buffer('offset', offset)


def _static_pack(enc, device, w_emb_t, w_lm_t):
    f32 = dict(dtype=torch.float32, device=device)
    tabs = [e.weight.detach().float() for e in enc.atom_embedding_list]
    off = np.concatenate([[0], np.cumsum([t.shape[0] for t in tabs])[:-1]])
    return dict(table=torch.cat(tabs, 0).to(**f32).contiguous(), table_off=torch.as_tensor(off, dtype=torch.int32, device=device),
                n_cat=len(tabs), ns=enc.emb_dim,
                w_emb_t=None if w_emb_t is None else w_emb_t.to(**f32).contiguous(),
                w_lm_t=None if w_lm_t is None else w_lm_t.to(**f32).contiguous(),
                n_lm=0 if w_lm_t is None else int(w_lm_t.shape[0]))


def static_embed(pack, cat, lm, device):
    """``ddp_node_static_embed`` on one complex: cat [n, n_cat] integer features, lm [n, n_lm] float or None -> [n, ns]."""
    n = cat.shape[0]
    cat_d = cat.to(device=device, dtype=torch.int64).contiguous()
    lm_d = lm.to(device=device, dtype=torch.float32).contiguous() if pack['n_lm'] else None
    out = torch.empty(n, pack['ns'], dtype=torch.float32, device=device)
    _lib.check(_lib.lib().ddp_node_static_embed(ptr(cat_d), n, pack['n_cat'], ptr(pack['table']), ptr(pack['table_off']), ptr(lm_d),
                                                 pack['n_lm'], ptr(pack['w_emb_t']), ptr(pack['w_lm_t']), pack['ns'], ptr(out),
                                                 _lib.stream_ptr()), 'ddp_node_static_embed')
    return out


class AtomEncoder(nn.Module):
    """Parameter holder; the encoder is evaluated as static part (once per complex) + per-graph sigma
    projection (``ddp_graph_sigma_proj`` / ``ddp_node_init``)."""

    def __init__(self, emb_dim, feature_dims, sigma_embed_dim, lm_embedding_type=None):
        super().__init__()
        self.atom_embedding_list = nn.ModuleList()
        self.num_categorical_features = len(feature_dims[0])
        self.lm_embedding_dim = 1280 if lm_embedding_type == 'esm' else 0
        if lm_embedding_type not in (None, 'esm'):
            raise ValueError('LM Embedding type was not correctly determined. LM embedding type: ', lm_embedding_type)
        self.sigma_embed_dim, self.emb_dim = sigma_embed_dim, emb_dim
        self.additional_features_dim = feature_dims[1] + sigma_embed_dim + self.lm_embedding_dim
        for dim in feature_dims[0]:
            emb = nn.Embedding(dim, emb_dim)
            nn.init.xavier_uniform_(emb.weight.data)
            self.atom_embedding_list.append(emb)
        if self.additional_features_dim > 0:
            self.additional_features_embedder = nn.Linear(self.additional_features_dim + emb_dim, emb_dim)

    def _emb_sum(self, cat):
        h = 0
        for i in range(self.num_categorical_features):
            h = h + self.atom_embedding_list[i](cat[:, i].long())
        return h

    def static_part(self, cat, lm=None):
        """Time-independent part of the Linear: W[:, :ns] sum_k Emb_k + W[:, ns:ns+1280] lm."""
        W = self.additional_features_embedder.weight
        ns = self.emb_dim
        out = self._emb_sum(cat) @ W[:, :ns].T
        if self.lm_embedding_dim:
            out = out + lm @ W[:, ns:ns + self.lm_embedding_dim].T
        return out.contiguous()

    def sigma_proj(self):
        """(W_sigma^T [sig, ns], bias) of the per-graph part."""
        W = self.additional_features_embedder.weight
        return W[:, -self.sigma_embed_dim:].T.contiguous(), self.additional_features_embedder.bias

    def static_pack(self, device):
        """Operands of ``ddp_node_static_embed`` (the kernel form of ``static_part``)."""
        W = self.additional_features_embedder.weight.detach().double()
        ns, L = self.emb_dim, self.lm_embedding_dim
        return _static_pack(self, device, W[:, :ns].T, W[:, ns:ns + L].T if L else None)


class OldAtomEncoder(nn.Module):
    def __init__(self, emb_dim, feature_dims, sigma_embed_dim, lm_embedding_type=None):
        super().__init__()
        self.atom_embedding_list = nn.ModuleList()
        self.num_categorical_features = len(feature_dims[0])
        self.num_scalar_features = feature_dims[1] + sigma_embed_dim
        self.lm_embedding_type = lm_embedding_type
        self.sigma_embed_dim, self.emb_dim = sigma_embed_dim, emb_dim
        for dim in feature_dims[0]:
            emb = nn.Embedding(dim, emb_dim)
            nn.init.xavier_uniform_(emb.weight.data)
            self.atom_embedding_list.append(emb)
        if self.num_scalar_features > 0:
            self.linear = nn.Linear(self.num_scalar_features, emb_dim)
        if lm_embedding_type is not None:
            if lm_embedding_type != 'esm':
                raise ValueError('LM Embedding type was not correctly determined. LM embedding type: ', lm_embedding_type)
            self.lm_embedding_dim = 1280
            self.lm_embedding_layer = nn.Linear(self.lm_embedding_dim + emb_dim, emb_dim)

    def _emb_sum(self, cat):
        h = 0
        for i in range(self.num_categorical_features):
            h = h + self.atom_embedding_list[i](cat[:, i].long())
        return h

    def static_part(self, cat, lm=None):
        ns, sd = self.emb_dim, self.sigma_embed_dim
        if self.lm_embedding_type is None:
            return self._emb_sum(cat).contiguous()
        # reference quirk (models/score_model.py:48-51): the "scalar" slice x[:, nc:nc+nsf] of
        # [aa | ESM | sigma] is ESM[:, :sd]; the LM layer sees [ESM[:, sd:] | sigma].
        Wl = self.lm_embedding_layer.weight
        h = self._emb_sum(cat) + lm[:, :sd] @ self.linear.weight.T
        return (h @ Wl[:, :ns].T + lm[:, sd:] @ Wl[:, ns:ns + self.lm_embedding_dim - sd].T).contiguous()

    def static_pack(self, device):
        """Operands of ``ddp_node_static_embed``: the two Linears of ``static_part`` folded (in float64) into one pair
        (W_emb, W_lm) so that the same kernel serves both encoders."""
        ns, sd = self.emb_dim, self.sigma_embed_dim
        if self.lm_embedding_type is None:
            return _static_pack(self, device, None, None)
        Wl = self.lm_embedding_layer.weight.detach().double()
        A = Wl[:, :ns].T                                                        # [ns, ns]
        w_lm = torch.cat([self.linear.weight.detach().double().T @ A, Wl[:, ns:ns + self.lm_embedding_dim - sd].T], 0)
        return _static_pack(self, device, A, w_lm)

    def sigma_proj(self):
        ns, sd = self.emb_dim, self.sigma_embed_dim
        if self.lm_embedding_type is None:
            return self.linear.weight.T.contiguous(), self.linear.bias
        Wl = self.lm_embedding_layer.weight
        return Wl[:, -sd:].T.contiguous(), self.lm_embedding_layer.bias + Wl[:, :ns] @ self.linear.bias


class BatchNorm(nn.Module):
    """Parameter holder with e3nn.nn.BatchNorm's state_dict layout (eval mode is folded into the
    node-update kernel as per-channel scale / shift)."""

    def __init__(self, irreps, eps=1e-5):
        super().__init__()
        self.irreps, self.eps = tpmod.parse_irreps(irreps), eps
        n_scalar = sum(m for m, l, p in self.irreps if l == 0 and p == 1)
        n_feat = sum(m for m, _, _ in self.irreps)
        self.register_buffer('running_mean', torch.zeros(n_scalar))
        self.register_buffer('running_var', torch.ones(n_feat))
        self.weight = nn.Parameter(torch.ones(n_feat))
        self.bias = nn.Parameter(torch.zeros(n_scalar))

    def folded(self):
        sc, sh = tpmod.batch_norm_fold(self.irreps, self.running_mean.detach().cpu().numpy().astype(np.float64),
                                       self.running_var.detach().cpu().numpy().astype(np.float64),
                                       self.weight.detach().cpu().numpy().astype(np.float64),
                                       self.bias.detach().cpu().numpy().astype(np.float64), self.eps)
        return torch.from_numpy(sc), torch.from_numpy(sh)


class _TP(nn.Module):
    """Stands where the reference keeps ``FasterTensorProduct`` / ``o3.FullyConnectedTensorProduct``."""

    def __init__(self, spec):
        super().__init__()
        self.spec = spec
        self.weight_numel = spec.weight_numel


class PackedConv:
    """Device-side, kernel-friendly image of one TensorProductConvLayer (built once per weight load)."""

    def __init__(self, layer, device, n_emb, ns, edge_fold=None, fold_bn=False):
        """``edge_fold`` = (W2e [n_emb, h], b2e [n_emb]) of the edge-embedding MLP's second Linear: folded into the
        first n_emb input columns of fc[0], so that the conv consumes the MLP's hidden activations directly."""
        spec = layer.tp.spec
        f32 = dict(dtype=torch.float32, device=device)
        fc0, fc3 = layer.fc[0], layer.fc[3]
        W1, b1 = fc0.weight.detach().double().cpu(), fc0.bias.detach().double().cpu()
        if edge_fold is not None:
            W2e, b2e = (t.detach().double().cpu() for t in edge_fold)
            assert W2e.shape[0] == n_emb and W2e.shape[1] == n_emb, 'fold keeps the edge-attribute width'
            b1 = b1 + W1[:, :n_emb] @ b2e
            W1 = torch.cat([W1[:, :n_emb] @ W2e, W1[:, n_emb:]], dim=1)
        self.w1_host, self.b1_host = W1.float().contiguous(), b1.float().contiguous()       # nn.Linear layout, for the UMMA pack
        self.w1t = self.w1_host.T.contiguous().to(**f32)
        self.b1 = self.b1_host.to(**f32)
        W2, b2 = fc3.weight.detach().double().cpu(), fc3.bias.detach().double().cpu()
        self.bn_folded = bool(fold_bn and layer.batch_norm is not None)
        if self.bn_folded:
            # the BatchNorm (eval) scale of output channel c multiplies every weight column that feeds c; the shift stays
            # with ddp_node_update.  Scale is constant over the components of an irrep, so one value per (group, o).
            sc, _ = layer.batch_norm.folded()
            col = torch.ones(spec.weight_numel, dtype=torch.float64)
            for g in spec.groups:
                o = torch.arange(g['mul_in'] * g['mul_out']) % g['mul_out']
                col[g['w_off']:g['w_off'] + g['mul_in'] * g['mul_out']] = sc.double()[g['out_off'] + o * g['d_out']]
            W2, b2 = W2 * col[:, None], b2 * col
        self.w2_host, self.b2_host = W2.float().contiguous(), b2.float().contiguous()       # nn.Linear layout, for the UMMA pack
        self.w2t = self.w2_host.T.contiguous().to(**f32)
        self.b2 = self.b2_host.to(**f32)
        self.k1, self.hid = fc0.in_features, fc0.out_features
        garr = (_lib.TpGroup * len(spec.groups))(*[_lib.TpGroup(**g) for g in spec.groups])
        self.groups_host = garr
        self.groups = torch.frombuffer(bytearray(bytes(garr)), dtype=torch.uint8).to(device)
        self.ctab = torch.tensor(spec.ctab, **f32)
        self.col_group = torch.from_numpy(spec.col_group()).to(device)
        self.spec = spec
        if layer.batch_norm is not None:
            sc, sh = layer.batch_norm.folded()
            self.bn_scale, self.bn_shift = sc.to(**f32), sh.to(**f32)
        else:
            self.bn_scale = self.bn_shift = None
        self.cdesc = _lib.TpConv(w1t=ptr(self.w1t), b1=ptr(self.b1), w2t=ptr(self.w2t), b2=ptr(self.b2), k1=self.k1,
                                 hid=self.hid, w_numel=spec.weight_numel, n_emb=n_emb, ns=ns, groups=ptr(self.groups),
                                 ctab=ptr(self.ctab), ctab_len=len(spec.ctab), col_group=ptr(self.col_group),
                                 n_groups=len(spec.groups), f_in=spec.f_in, f_out=spec.f_out, sh_dim=spec.sh_dim)
        self.umma = {}   # mode -> packed device image (tensor-core kernel)

    def umma_image(self, layer, mode, device):
        if mode not in self.umma:
            L = _lib.lib()
            w1, b1 = self.w1_host, self.b1_host
            w2, b2 = self.w2_host, self.b2_host
            ctab = torch.tensor(self.spec.ctab, dtype=torch.float32)
            # the packer builds one accumulation block per run of groups with the same output irrep: hand it the groups
            # sorted by output (e3nn orders FullyConnectedTensorProduct instructions by input irrep, which would split every
            # output into several blocks, i.e. several flushes per edge tile); weight columns are addressed through w_off
            order = sorted(range(len(self.spec.groups)), key=lambda i: self.spec.groups[i]['out_off'])
            garr = (_lib.TpGroup * len(order))(*[_lib.TpGroup(**self.spec.groups[i]) for i in order])
            args = (C.byref(self.cdesc), garr, ptr(ctab), ptr(w1), ptr(b1), ptr(w2), ptr(b2), mode)
            size = L.ddp_tpconv_pack(*args, None)
            if size <= 0:
                raise RuntimeError(f'ddp_tpconv_pack failed ({size}): conv is not tensor-core eligible')
            host = torch.empty(size, dtype=torch.uint8)
            _lib.check(L.ddp_tpconv_pack(*args, ptr(host)), 'ddp_tpconv_pack')
            self.umma[mode] = host.to(device)
            # one-time upload from pageable memory: other streams (the sampler's second mini-batch stream) may launch on
            # this image right away, so make sure the DMA has landed before anybody can
            torch.cuda.current_stream(device).synchronize()
        return self.umma[mode]


class _ConvFn(torch.autograd.Function):
    """Autograd node of one TensorProductConvLayer call (training path, SURVEY 8(f) row 3; the reference differentiates
    ``tp(node_attr[edge_dst], edge_sh, fc(edge_attr))`` + ``scatter(mean)`` with PyTorch / e3nn autograd,
    models/score_model.py:105-125 under utils/training.py:147-191).  Forward = the fused kernels.  Backward: the Linear /
    ReLU gradients and the two weight-gradient GEMMs are library GEMMs; the tensor-product part -- gradients with respect
    to the per-edge weights, the gathered node features and the edge harmonics -- is ``ddp_tp_backward``, on chunks of
    edges whose per-edge weights are re-materialised ([chunk, weight_numel] fp32).  BatchNorm, where present, is the
    eval-mode affine map of the forward (running statistics are constants; its own parameters get no gradient)."""

    @staticmethod
    def forward(ctx, layer, edge_index, out_nodes, edge_weight, node_attr, edge_attr, edge_sh, w1, b1, w2, b2):
        with torch.no_grad():
            out = layer._forward_impl(node_attr, edge_index, edge_attr, edge_sh, out_nodes, edge_weight)
        ctx.layer, ctx.out_nodes = layer, int(out_nodes or node_attr.shape[0])
        ctx.has_ew = torch.is_tensor(edge_weight)
        ctx.save_for_backward(node_attr, edge_attr, edge_sh, w1, b1, w2, b2, edge_index,
                              edge_weight if ctx.has_ew else torch.empty(0))
        return out

    @staticmethod
    def backward(ctx, g):
        node_attr, edge_attr, edge_sh, w1, b1, w2, b2, edge_index, ew = ctx.saved_tensors
        layer, n_out = ctx.layer, ctx.out_nodes
        dev = node_attr.device
        L = _lib.lib()
        E = edge_index.shape[1]
        x, A, sh = node_attr.detach().float().contiguous(), edge_attr.detach().float().contiguous(), edge_sh.detach().float().contiguous()
        W1, B1, W2, B2 = (t.detach().float() for t in (w1, b1, w2, b2))
        agg, src = edge_index[0].long(), edge_index[1].to(torch.int32).contiguous()
        bd = layer._backward_desc(dev)                                # spec only (row groups, coefficient table): no weights
        g = g.detach().float()
        if layer.batch_norm is not None:
            g = g * layer.batch_norm.folded()[0].to(device=dev, dtype=torch.float32)
        deg = torch.bincount(agg, minlength=n_out).clamp(min=1).to(torch.float32)
        g_node = (g / deg[:, None]).contiguous()
        Hpre = torch.addmm(B1, A, W1.T)
        H = torch.relu(Hpre)
        Wn = W2.shape[0]
        det = _lib.deterministic()
        acc_dtype = _lib.sum_dtype(det)                               # deterministic mode: fixed-point g_x / g_sh
        g_x, g_sh = torch.zeros_like(x, dtype=acc_dtype), torch.zeros_like(sh, dtype=acc_dtype)
        g_W2, g_b2, g_H = torch.zeros_like(W2), torch.zeros_like(B2), torch.empty_like(H)
        chunk = max(1024, (1 << 27) // max(Wn, 1))                    # two [chunk, weight_numel] fp32 buffers of <= 0.5 GB each
        for c0 in range(0, E, chunk):
            c1 = min(E, c0 + chunk)
            Wt = torch.addmm(B2, H[c0:c1], W2.T).contiguous()        # per-edge weights of the chunk
            ge = g_node[agg[c0:c1]]
            if ctx.has_ew:
                ge = ge * ew.detach().float().reshape(-1, 1)[c0:c1]
            ge = ge.contiguous()
            g_w = torch.empty_like(Wt)
            if det:
                _lib.check(L.ddp_tp_backward_fixed(C.byref(bd['cdesc']), bd['rows'], ptr(x), src[c0:c1].data_ptr(), x.shape[1],
                                                   sh[c0:c1].data_ptr(), ptr(Wt), ptr(ge), c1 - c0, ptr(g_w), ptr(g_x),
                                                   g_sh[c0:c1].data_ptr(), ptr(_lib.status_word(dev)), _lib.stream_ptr()),
                           'ddp_tp_backward_fixed')
            else:
                _lib.check(L.ddp_tp_backward(C.byref(bd['cdesc']), bd['rows'], ptr(x), src[c0:c1].data_ptr(), x.shape[1], sh[c0:c1].data_ptr(),
                                             ptr(Wt), ptr(ge), c1 - c0, ptr(g_w), ptr(g_x), g_sh[c0:c1].data_ptr(), _lib.stream_ptr()),
                           'ddp_tp_backward')
            g_W2.addmm_(g_w.T, H[c0:c1])
            g_b2 += g_w.sum(0)
            g_H[c0:c1] = g_w @ W2
        if det:
            q_x, q_sh = g_x, g_sh
            g_x, g_sh = torch.empty_like(x), torch.empty_like(sh)
            for q, f in ((q_x, g_x), (q_sh, g_sh)):
                _lib.check(L.ddp_fixed_to_float(ptr(q), q.numel(), ptr(f), _lib.stream_ptr()), 'ddp_fixed_to_float')
            _lib.check_status(dev)
        g_pre = g_H * (Hpre > 0)
        g_W1, g_b1, g_A = g_pre.T @ A, g_pre.sum(0), g_pre @ W1
        need = ctx.needs_input_grad
        cast = lambda t, like: t.to(like.dtype)
        return (None, None, None, None, cast(g_x, node_attr) if need[4] else None, cast(g_A, edge_attr) if need[5] else None,
                cast(g_sh, edge_sh) if need[6] else None, g_W1 if need[7] else None, g_b1 if need[8] else None,
                g_W2 if need[9] else None, g_b2 if need[10] else None)


class TensorProductConvLayer(nn.Module):
    """models/score_model.py:84-125 (operator-level drop-in)."""

    def __init__(self, in_irreps, sh_irreps, out_irreps, n_edge_features, residual=True, batch_norm=True, dropout=0.0,
                 hidden_features=None, faster=False):
        super().__init__()
        self.in_irreps, self.out_irreps, self.sh_irreps = in_irreps, out_irreps, sh_irreps
        self.residual = residual
        if hidden_features is None:
            hidden_features = n_edge_features
        sh_ir = tpmod.parse_irreps(sh_irreps) if isinstance(sh_irreps, str) else list(sh_irreps)
        if faster:
            assert [tuple(t) for t in sh_ir] == [(1, 0, 1), (1, 1, -1)], "sh_irreps don't look like 1st order spherical harmonics"
            spec = tpmod.faster_tp_spec(in_irreps, out_irreps)
        else:
            spec = tpmod.fctp_spec(in_irreps, sh_ir, out_irreps)
        self.tp = _TP(spec)
        self.fc = nn.Sequential(nn.Linear(n_edge_features, hidden_features), nn.ReLU(), nn.Dropout(dropout),
                                nn.Linear(hidden_features, spec.weight_numel))
        self.batch_norm = BatchNorm(out_irreps) if batch_norm else None
        self._packed = None
        self.conv_mode = 'fp32'      # stand-alone operator calls: 'fp32' | 'bf16' | 'bf16x3'

    def _load_from_state_dict(self, *a, **k):
        self._packed = None
        return super()._load_from_state_dict(*a, **k)

    def _backward_desc(self, device):
        """Descriptor of ``ddp_tp_backward``: the row groups and coefficient table of the spec on the device (weight-free, so it
        survives optimizer steps) + the number of basis rows per edge."""
        bd = getattr(self, '_bwd', None)
        if bd is None or bd['device'] != torch.device(device):
            spec = self.tp.spec
            if any(max(g['d1'], g['d2'], g['d_out']) > 5 for g in spec.groups):
                raise NotImplementedError('ddp_tp_backward handles irreps up to l = 2')
            garr = (_lib.TpGroup * len(spec.groups))(*[_lib.TpGroup(**g) for g in spec.groups])
            groups = torch.frombuffer(bytearray(bytes(garr)), dtype=torch.uint8).to(device)
            ctab = torch.tensor(spec.ctab, dtype=torch.float32, device=device)
            cdesc = _lib.TpConv(w1t=None, b1=None, w2t=None, b2=None, k1=self.fc[0].in_features, hid=self.fc[0].out_features,
                                w_numel=spec.weight_numel, n_emb=self.fc[0].in_features, ns=0, groups=ptr(groups), ctab=ptr(ctab),
                                ctab_len=len(spec.ctab), col_group=None, n_groups=len(spec.groups), f_in=spec.f_in, f_out=spec.f_out,
                                sh_dim=spec.sh_dim)
            bd = self._bwd = dict(device=torch.device(device), groups=groups, ctab=ctab, cdesc=cdesc,
                                  rows=int(sum(g['mul_in'] for g in spec.groups)))
        return bd

    def packed(self, device, n_emb, ns, edge_fold=None, fold_bn=False):
        # (parameter versions: an optimizer step between two training forwards invalidates the packed image)
        key = (None if edge_fold is None else tuple(id(t) for t in edge_fold), bool(fold_bn),
               tuple(p._version for p in self.fc.parameters()))
        if self._packed is None or self._packed.w1t.device != torch.device(device) or self._packed.cdesc.n_emb != n_emb \
                or self._packed.fold_key != key:
            self._packed = PackedConv(self, device, n_emb, ns, edge_fold, fold_bn)
            self._packed.fold_key = key
        return self._packed

    def forward(self, node_attr, edge_index, edge_attr, edge_sh, out_nodes=None, reduce='mean', edge_weight=1.0):
        """Stand-alone operator call: edge_attr is the already concatenated [E, n_edge_features].  With autograd enabled and
        something to differentiate (inputs or the edge-MLP parameters) the call is recorded as one ``_ConvFn`` node."""
        if edge_index.numel() == 0:
            return torch.tensor(0, dtype=node_attr.dtype, device=node_attr.device)
        assert reduce == 'mean' and not self.residual
        fc0, fc3 = self.fc[0], self.fc[3]
        if torch.is_grad_enabled() and any(t.requires_grad for t in (node_attr, edge_attr, edge_sh, fc0.weight, fc0.bias, fc3.weight, fc3.bias)):
            if self.training and self.fc[2].p > 0:
                raise NotImplementedError('dropout inside the fused edge MLP is not differentiated (train with dropout = 0 or eval())')
            return _ConvFn.apply(self, edge_index, out_nodes, edge_weight, node_attr, edge_attr, edge_sh, fc0.weight, fc0.bias,
                                 fc3.weight, fc3.bias)
        return self._forward_impl(node_attr, edge_index, edge_attr, edge_sh, out_nodes, edge_weight)

    def _forward_impl(self, node_attr, edge_index, edge_attr, edge_sh, out_nodes=None, edge_weight=1.0):
        dev = node_attr.device
        if dev.type != 'cuda':
            raise RuntimeError('TensorProductConvLayer runs on CUDA only (no CPU fallback)')
        L = _lib.lib()
        E = edge_index.shape[1]
        out_nodes = int(out_nodes or node_attr.shape[0])
        ei = edge_index.to(torch.int32).contiguous()
        x = node_attr.float().contiguous()
        ea, sh = edge_attr.float().contiguous(), edge_sh.float().contiguous()
        ew = None
        if torch.is_tensor(edge_weight):
            ew = edge_weight.float().reshape(-1).contiguous()
        n_dev = torch.tensor([E], dtype=torch.int32, device=dev)
        k1 = self.fc[0].in_features
        use_tc = self.conv_mode != 'fp32' and k1 % 3 == 0 and ew is None and tpmod.umma_supported(self.tp.spec, k1 // 3)
        if use_tc:
            ns = k1 // 3
            pk = self.packed(dev, ns, ns)
            parts = [ea[:, i * ns:(i + 1) * ns].contiguous() for i in range(3)]
            ident = torch.arange(E, dtype=torch.int32, device=dev)
            ed = _lib.TpEdges(emb=ptr(parts[0]), p1=ptr(parts[1]), i1=ptr(ident), ld1=ns, p2=ptr(parts[2]), i2=ptr(ident), ld2=ns,
                              x=ptr(x), gather=ei[1].data_ptr(), ldx=x.shape[1], sh=ptr(sh), agg=ei[0].data_ptr(), ew=None,
                              n_edges_dev=ptr(n_dev), edge_cap=E)
        else:
            pk = self.packed(dev, k1, 0)
            ed = _lib.TpEdges(emb=ptr(ea), p1=None, i1=None, ld1=0, p2=None, i2=None, ld2=0, x=ptr(x), gather=ei[1].data_ptr(),
                              ldx=x.shape[1], sh=ptr(sh), agg=ei[0].data_ptr(), ew=ptr(ew), n_edges_dev=ptr(n_dev), edge_cap=E)
        f_out = pk.spec.f_out
        det = _lib.deterministic()                                    # fixed-point sums: bitwise reproducible
        s = torch.zeros(out_nodes, f_out, device=dev, dtype=_lib.sum_dtype(det))
        status = ptr(_lib.status_word(dev)) if det else None
        if use_tc:
            mode = 0 if self.conv_mode == 'bf16' else 1
            img = pk.umma_image(self, mode, dev)
            if det:
                _lib.check(L.ddp_tpconv_umma_fixed(C.byref(pk.cdesc), ptr(img), mode, C.byref(ed), ptr(s), status, _lib.stream_ptr()),
                           'ddp_tpconv_umma_fixed')
            else:
                _lib.check(L.ddp_tpconv_umma(C.byref(pk.cdesc), ptr(img), mode, C.byref(ed), ptr(s), _lib.stream_ptr()), 'ddp_tpconv_umma')
        elif det:
            _lib.check(L.ddp_tpconv_fp32_fixed(C.byref(pk.cdesc), C.byref(ed), ptr(s), status, _lib.stream_ptr()), 'ddp_tpconv_fp32_fixed')
        else:
            _lib.check(L.ddp_tpconv_fp32(C.byref(pk.cdesc), C.byref(ed), ptr(s), _lib.stream_ptr()), 'ddp_tpconv_fp32')
        deg = torch.zeros(out_nodes, dtype=torch.int32, device=dev)
        _lib.check(L.ddp_degree(ei[0].data_ptr(), ptr(n_dev), E, ptr(deg), _lib.stream_ptr()), 'ddp_degree')
        up = _lib.Update(sum=ptr(s), deg=ptr(deg), scale=ptr(pk.bn_scale), shift=ptr(pk.bn_shift), n_edges_dev=ptr(n_dev))
        out = torch.empty(out_nodes, f_out, device=dev)
        update = L.ddp_node_update_fixed if det else L.ddp_node_update
        _lib.check(update(None, 0, 0, C.byref(up), 1, out_nodes, f_out, ptr(out), f_out, _lib.stream_ptr()), 'ddp_node_update')
        if det:
            _lib.check_status(dev)                                    # (synchronises: a stand-alone call returns checked results)
        return out
