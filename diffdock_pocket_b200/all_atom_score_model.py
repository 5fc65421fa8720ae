"""All-atom score / confidence model: host mirror of ``models/all_atom_score_model.py``.

``TensorProductScoreModel`` keeps the reference constructor signature (all_atom_score_model.py:22-32),
module attribute names (so reference checkpoints load, SURVEY.md App. A.5) and ``forward(data)``
contract (:238-436), but evaluates everything through the ddp_b200 CUDA kernels:

* ``make_plan(data)`` uploads one collated batch once and allocates every workspace (static tensors,
  fixed-capacity dynamic edge buffers with device-side counts);
* ``run_plan(plan, t)`` launches the forward without a single host synchronisation, which is what lets
  ``sampling()`` keep the batch resident on the GPU for all steps.

Supported configuration: ``parallel == 1``, no affinity head, ``separate_noise_schedule`` /
``odd_parity`` off (the reference inference path, SURVEY.md App. A.1).
The per-graph diffusion time is read from ``data.complex_t['tr']`` (``set_time`` broadcasts the same
value to every node of a graph, utils/diffusion_utils.py:124-149).
"""
import ctypes as C
import os

import numpy as np
import torch
from torch import nn

from . import _lib, so3, torus, tp as tpmod
from ._lib import ptr
from .score_model import (FEATURE_DIMS, AtomEncoder, GaussianSmearing, OldAtomEncoder, TensorProductConvLayer, _TP, static_embed)


STATIC_KEYS = (('ligand', 'x'), ('receptor', 'x'), ('atom', 'x'))      # collate skips these when the plan gets ``graphs``


def _mlp(i, h, o, dropout):
    return nn.Sequential(nn.Linear(i, h), nn.ReLU(), nn.Dropout(dropout), nn.Linear(h, o))


class _EdgeSet:
    """Fixed-capacity device edge buffer: row 0 = edge[:cap], row 1 = edge[cap:], live count on device."""

    def __init__(self, cap, ns, sh_dim, device, with_slab=None):
        self.cap = max(int(cap), 1)
        self.edge = torch.zeros(2 * self.cap, dtype=torch.int32, device=device)
        self.n_dev = torch.zeros(1, dtype=torch.int32, device=device)
        self.sh = torch.zeros(self.cap, sh_dim, device=device)
        self.emb = torch.zeros(self.cap, ns, device=device)
        self.deg = {}
        if with_slab is not None:
            n_q, w = with_slab
            self.slab_w = max(int(w), 1)
            self.slab = torch.zeros(max(int(n_q), 1) * self.slab_w, dtype=torch.int32, device=device)
            self.counts = torch.zeros(max(int(n_q), 1) + 1, dtype=torch.int32, device=device)

    def row(self, r):
        return self.edge.data_ptr() + 4 * self.cap * r

    def set_static(self, ei):
        n = ei.shape[1]
        self.edge[:n] = ei[0].to(torch.int32)
        self.edge[self.cap:self.cap + n] = ei[1].to(torch.int32)
        self.n_dev.fill_(n)

    def live_copy(self, ns, sh_dim, device):
        """Buffer of the same capacity for the edges of this set whose aggregation node is live (``ddp_live_edges``).  It
        shares the in-degrees of the full set: a live node keeps all of its edges, so its mean keeps its normaliser."""
        c = _EdgeSet(self.cap, ns, sh_dim, device)
        c.deg = self.deg
        c.counts = torch.zeros((self.cap + 255) // 256 + 1, dtype=torch.int32, device=device)
        return c

    def edge_index(self):
        """Host-synchronising view [2, E] int64 (tests / drop-in side effects only)."""
        n = int(self.n_dev.item())
        return torch.stack([self.edge[:n], self.edge[self.cap:self.cap + n]]).long()


class Plan:
    pass


class _Branches:
    """Fork / join of independent kernel chains onto side streams (works eagerly and under CUDA-graph capture:
    the side streams join the capture through the fork event and are joined back before the forward returns)."""

    def __init__(self, device, n=4):
        self.side = [torch.cuda.Stream(device=device) for _ in range(n)]

    def fork(self, k):
        main = torch.cuda.current_stream()
        ev = torch.cuda.Event()
        ev.record(main)
        for s in self.side[:k]:
            s.wait_event(ev)
        return main

    def join(self, main, k):
        for s in self.side[:k]:
            ev = torch.cuda.Event()
            ev.record(s)
            main.wait_event(ev)


class TensorProductScoreModel(nn.Module):
    def __init__(self, t_to_sigma, device, timestep_emb_func, in_lig_edge_features=4, sigma_embed_dim=32, sh_lmax=2,
                 ns=16, nv=4, num_conv_layers=2, lig_max_radius=5, rec_max_radius=30, cross_max_distance=250,
                 center_max_distance=30, distance_embed_dim=32, cross_distance_embed_dim=32, no_torsion=False,
                 scale_by_sigma=True, norm_by_sigma=True, use_second_order_repr=False, batch_norm=True,
                 dynamic_max_cross=False, dropout=0.0, smooth_edges=False, odd_parity=False,
                 separate_noise_schedule=False, lm_embedding_type=False, confidence_mode=False,
                 confidence_dropout=0, confidence_no_batchnorm=False, asyncronous_noise_schedule=False,
                 affinity_prediction=False, parallel=1, parallel_aggregators="mean max min std",
                 num_confidence_outputs=1, fixed_center_conv=False, atom_max_neighbors=None,
                 no_aminoacid_identities=False, flexible_sidechains=False, include_miscellaneous_atoms=False,
                 use_old_atom_encoder=False):
        super().__init__()
        if parallel != 1 or affinity_prediction or separate_noise_schedule or odd_parity \
                or smooth_edges or include_miscellaneous_atoms:
            raise NotImplementedError('configuration outside the accelerated inference path (see module docstring)')
        if not lm_embedding_type:
            lm_embedding_type = None
        self.t_to_sigma, self.timestep_emb_func = t_to_sigma, timestep_emb_func
        self.asyncronous_noise_schedule = bool(asyncronous_noise_schedule)
        self.in_lig_edge_features, self.sigma_embed_dim = in_lig_edge_features, sigma_embed_dim
        self.lig_max_radius, self.rec_max_radius = lig_max_radius, rec_max_radius
        self.cross_max_distance, self.dynamic_max_cross = cross_max_distance, dynamic_max_cross
        self.center_max_distance, self.distance_embed_dim = center_max_distance, distance_embed_dim
        self.cross_distance_embed_dim = cross_distance_embed_dim
        self.sh_lmax = sh_lmax
        self.sh_irreps = [(1, l, (-1) ** l) for l in range(sh_lmax + 1)]
        self.sh_dim = (sh_lmax + 1) ** 2
        self.ns, self.nv = ns, nv
        self.scale_by_sigma, self.device, self.no_torsion = scale_by_sigma, device, no_torsion
        self.num_conv_layers, self.confidence_mode = num_conv_layers, confidence_mode
        self.fixed_center_conv, self.atom_max_neighbors = fixed_center_conv, atom_max_neighbors
        self.no_aminoacid_identities, self.flexible_sidechains = no_aminoacid_identities, flexible_sidechains
        self.lm_embedding_type = lm_embedding_type
        self.conv_mode = 'fp32'          # 'fp32' | 'bf16' | 'bf16x3'  (tensor-core modes need FasterTP convs)

        enc = OldAtomEncoder if use_old_atom_encoder else AtomEncoder
        self.lig_node_embedding = enc(ns, FEATURE_DIMS['lig'], sigma_embed_dim)
        self.lig_edge_embedding = _mlp(in_lig_edge_features + sigma_embed_dim + distance_embed_dim, ns, ns, dropout)
        self.rec_node_embedding = enc(ns, FEATURE_DIMS['rec_residue'], sigma_embed_dim, lm_embedding_type)
        self.rec_edge_embedding = _mlp(sigma_embed_dim + distance_embed_dim, ns, ns, dropout)
        self.atom_node_embedding = enc(ns, FEATURE_DIMS['rec_atom'], sigma_embed_dim)
        self.atom_edge_embedding = _mlp(sigma_embed_dim + distance_embed_dim, ns, ns, dropout)
        self.lr_edge_embedding = _mlp(sigma_embed_dim + cross_distance_embed_dim, ns, ns, dropout)
        self.ar_edge_embedding = _mlp(sigma_embed_dim + distance_embed_dim, ns, ns, dropout)
        self.la_edge_embedding = _mlp(sigma_embed_dim + cross_distance_embed_dim, ns, ns, dropout)
        self.lig_distance_expansion = GaussianSmearing(0.0, lig_max_radius, distance_embed_dim)
        self.rec_distance_expansion = GaussianSmearing(0.0, rec_max_radius, distance_embed_dim)
        self.cross_distance_expansion = GaussianSmearing(0.0, cross_max_distance, cross_distance_embed_dim)

        if use_second_order_repr:
            seq = [f'{ns}x0e', f'{ns}x0e + {nv}x1o + {nv}x2e', f'{ns}x0e + {nv}x1o + {nv}x2e + {nv}x1e + {nv}x2o',
                   f'{ns}x0e + {nv}x1o + {nv}x2e + {nv}x1e + {nv}x2o + {ns}x0o']
        else:
            seq = [f'{ns}x0e', f'{ns}x0e + {nv}x1o', f'{ns}x0e + {nv}x1o + {nv}x1e', f'{ns}x0e + {nv}x1o + {nv}x1e + {ns}x0o']
        self.irrep_seq = seq
        faster = sh_lmax == 1 and not use_second_order_repr
        self.faster = faster
        convs = []
        for i in range(num_conv_layers):
            for _ in range(9):
                convs.append(TensorProductConvLayer(seq[min(i, 3)], self.sh_irreps, seq[min(i + 1, 3)], 3 * ns, residual=False,
                                                    batch_norm=batch_norm, dropout=dropout, faster=faster))
        self.conv_layers = nn.ModuleList(convs)
        last = seq[min(num_conv_layers, 3)]
        if confidence_mode:
            cin = (2 * ns if num_conv_layers >= 3 else ns) * (2 if flexible_sidechains else 1)
            bn = (lambda: nn.Identity()) if confidence_no_batchnorm else (lambda: nn.BatchNorm1d(ns))
            self.confidence_predictor = nn.Sequential(
                nn.Linear(cin, ns), bn(), nn.ReLU(), nn.Dropout(confidence_dropout),
                nn.Linear(ns, ns), bn(), nn.ReLU(), nn.Dropout(confidence_dropout),
                nn.Linear(ns, num_confidence_outputs))
        else:
            self.center_distance_expansion = GaussianSmearing(0.0, center_max_distance, distance_embed_dim)
            self.center_edge_embedding = _mlp(distance_embed_dim + sigma_embed_dim, ns, ns, dropout)
            self.final_conv = TensorProductConvLayer(last, self.sh_irreps, '2x1o + 2x1e', 2 * ns, residual=False,
                                                     dropout=dropout, batch_norm=batch_norm, faster=faster)
            self.tr_final_layer = nn.Sequential(nn.Linear(1 + sigma_embed_dim, ns), nn.Dropout(dropout), nn.ReLU(), nn.Linear(ns, 1))
            self.rot_final_layer = nn.Sequential(nn.Linear(1 + sigma_embed_dim, ns), nn.Dropout(dropout), nn.ReLU(), nn.Linear(ns, 1))
            tor_sh = tpmod.full_tp_out_irreps(self.sh_irreps, '1x2e')
            self._tor_ftp = self._tor_ftp_table(last, tor_sh, ns)
            if not no_torsion:
                self.final_edge_embedding = _mlp(distance_embed_dim, ns, ns, dropout)
                self.final_tp_tor = nn.Module()          # o3.FullTensorProduct has no parameters
                self.tor_bond_conv = self._tor_conv(last, tor_sh, ns, dropout, batch_norm, self._tor_ftp)
                self.tor_final_layer = nn.Sequential(nn.Linear(2 * ns, ns, bias=False), nn.Tanh(), nn.Dropout(dropout),
                                                     nn.Linear(ns, 1, bias=False))
            if flexible_sidechains:
                self.sidechain_final_edge_embedding = _mlp(distance_embed_dim, ns, ns, dropout)
                self.final_tp_sc_tor = nn.Module()
                self.sc_tor_bond_conv = self._tor_conv(last, tor_sh, ns, dropout, batch_norm, self._tor_ftp)
                self.sc_tor_final_layer = nn.Sequential(nn.Linear(2 * ns, ns, bias=False), nn.Tanh(), nn.Dropout(dropout),
                                                        nn.Linear(ns, 1, bias=False))
        self._packed = None

    def _tor_ftp_table(self, last, tor_sh, ns):
        """Which irreps of sh_tor = FullTensorProduct(sh_edge, Y2(bond)) the torsion convs read, and how to compute them.
        lmax 1: only the 1o part, laid out [1 | 1o] so the conv looks FasterTensorProduct-shaped (tensor-core eligible,
        ``ddp_tor_edge_sh``).  lmax 2: 0e, 1o, 1e via the generic path table of ``ddp_tor_edge_sh_generic``."""
        used = tpmod.fctp_used_sh(last, tor_sh, f'{ns}x0o + {ns}x0e')
        if self.sh_lmax == 1:
            assert used == [0]
            return dict(keep=[0], base=1, dim=4, paths=None, ctab=None)
        prov = tpmod.full_tp_paths(self.sh_irreps, '1x2e')
        sh_off = tpmod.irreps_offsets(self.sh_irreps)
        paths, ctab, o = [], [], 0
        for k in used:
            lo, _, i1, _ = prov[k]
            l1 = self.sh_irreps[i1][1]
            cg = tpmod.wigner_3j(l1, 2, lo) * np.sqrt(2 * lo + 1)             # e3nn FullTensorProduct, component normalisation
            paths.append(dict(in_off=sh_off[i1], d_in=2 * l1 + 1, out_off=o, d_out=2 * lo + 1, c_off=len(ctab)))
            ctab += [float(v) for v in cg.reshape(-1)]
            o += 2 * lo + 1
        return dict(keep=used, base=0, dim=o, paths=paths, ctab=ctab)

    @staticmethod
    def _tor_conv(last, tor_sh, ns, dropout, batch_norm, ftp):
        conv = TensorProductConvLayer(last, tor_sh, f'{ns}x0o + {ns}x0e', 3 * ns, residual=False, dropout=dropout,
                                      batch_norm=batch_norm)
        # only the sh_tor irreps the conv can couple to are materialised (valid while node irreps have l <= 1)
        spec = tpmod.fctp_spec(last, tor_sh, f'{ns}x0o + {ns}x0e', sh_keep=ftp['keep'], sh_base=ftp['base'])
        assert spec.weight_numel == conv.tp.weight_numel
        spec.tc_eligible = ftp['paths'] is None and all(l <= 1 for _, l, _ in tpmod.parse_irreps(last))
        conv.tp = _TP(spec)
        return conv

    # ------------------------------------------------------------------------------------------ packing
    def _load_from_state_dict(self, *a, **k):
        self._packed = None
        return super()._load_from_state_dict(*a, **k)

    @staticmethod
    def _is_e3nn_constant(key, value):
        """Keys an e3nn 0.5.1 module contributes to a reference checkpoint that carry no learned state: the persistent
        buffers of ``o3.TensorProduct`` (``output_mask``, the Wigner-3j constants ``_w3j_*`` inside the TorchScript-compiled
        ``_compiled_main_*`` sub-modules) and the EMPTY ``weight`` buffer it registers when ``internal_weights`` is off.
        They belong to ``conv.tp`` of the non-``faster`` convs, ``tor_bond_conv.tp`` / ``sc_tor_bond_conv.tp`` and
        ``final_tp_tor`` / ``final_tp_sc_tor`` (models/all_atom_score_model.py:193-228, models/score_model.py:98)."""
        parts = key.split('.')
        owner_is_tp = 'tp' in parts[:-1] or any(p.startswith('final_tp') for p in parts[:-1])
        if not owner_is_tp:
            return False
        last = parts[-1]
        if last == 'output_mask' or last.startswith('_w3j') or any(p.startswith('_compiled_main') for p in parts[:-1]):
            return True
        return last == 'weight' and torch.is_tensor(value) and value.numel() == 0

    def load_state_dict(self, state_dict, strict=True, **kw):
        """``strict=True`` like the reference (inference.py:434-435,447-448) on everything learned; the constant e3nn
        buffers listed in ``_is_e3nn_constant`` are the ONLY keys that are dropped.  A ``module.``-prefixed checkpoint
        (saved from ``DataParallel``, utils/utils.py:110-111) is accepted as the reference's wrapped model would."""
        sd = state_dict
        if sd and all(k.startswith('module.') for k in sd):
            sd = {k[len('module.'):]: v for k, v in sd.items()}
        sd = type(sd)((k, v) for k, v in sd.items() if not self._is_e3nn_constant(k, v)) if not isinstance(sd, dict) \
            else {k: v for k, v in sd.items() if not self._is_e3nn_constant(k, v)}
        return super().load_state_dict(sd, strict=strict, **kw)

    def _edge_mlp_pack(self, seq, rbf, dev, layout):
        """layout: tuple of ('pre', n) / ('sig', n) / ('rbf', n) giving the column order of Linear 0."""
        W, b1 = seq[0].weight.detach(), seq[0].bias.detach()
        cols, o = {}, 0
        for kind, n in layout:
            cols[kind] = W[:, o:o + n]
            o += n
        assert o == W.shape[1]
        f32 = dict(dtype=torch.float32, device=dev)
        pk = dict(w_pre=cols['pre'].T.contiguous().to(**f32) if 'pre' in cols else None,
                  w_rbf=cols['rbf'].T.contiguous().to(**f32),
                  w_sig=cols['sig'].T.contiguous().to(**f32) if 'sig' in cols else None,
                  b1=b1.contiguous().to(**f32), w2=seq[3].weight.detach().T.contiguous().to(**f32),
                  b2=seq[3].bias.detach().contiguous().to(**f32), offset=rbf.offset.detach().contiguous().to(**f32))
        # the second Linear is folded into the W1 of every conv that consumes this embedding (PackedConv edge_fold)
        pk['fold'] = (seq[3].weight, seq[3].bias)
        pk['desc'] = _lib.EdgeMlp(w_pre=ptr(pk['w_pre']), w_rbf=ptr(pk['w_rbf']), w2=None, b2=ptr(pk['b2']),
                                  b1=ptr(pk['b1']), rbf_offset=ptr(pk['offset']), rbf_coeff=float(rbf.coeff),
                                  n_pre=cols['pre'].shape[1] if 'pre' in cols else 0, n_rbf=cols['rbf'].shape[1],
                                  ns=self.ns, sh_dim=self.sh_dim)
        return pk

    def packed(self):
        dev = next(self.parameters()).device
        if self._packed is not None and self._packed['device'] == dev:
            return self._packed
        if dev.type != 'cuda':
            raise RuntimeError('the ddp_b200 score model runs on CUDA only (no CPU fallback); call model.to("cuda")')
        P = dict(device=dev)
        sd, dd, cd, ns = self.sigma_embed_dim, self.distance_embed_dim, self.cross_distance_embed_dim, self.ns
        f32 = dict(dtype=torch.float32, device=dev)
        em = {}
        em['ll'] = self._edge_mlp_pack(self.lig_edge_embedding, self.lig_distance_expansion, dev,
                                       (('pre', self.in_lig_edge_features), ('sig', sd), ('rbf', dd)))
        em['rr'] = self._edge_mlp_pack(self.rec_edge_embedding, self.rec_distance_expansion, dev, (('sig', sd), ('rbf', dd)))
        em['aa'] = self._edge_mlp_pack(self.atom_edge_embedding, self.lig_distance_expansion, dev, (('sig', sd), ('rbf', dd)))
        em['lr'] = self._edge_mlp_pack(self.lr_edge_embedding, self.cross_distance_expansion, dev, (('sig', sd), ('rbf', cd)))
        em['la'] = self._edge_mlp_pack(self.la_edge_embedding, self.cross_distance_expansion, dev, (('sig', sd), ('rbf', cd)))
        em['ar'] = self._edge_mlp_pack(self.ar_edge_embedding, self.rec_distance_expansion, dev, (('sig', sd), ('rbf', dd)))
        proj_names = ['lig_node', 'rec_node', 'atom_node', 'll', 'rr', 'aa', 'lr', 'la', 'ar']
        ws, bs = [], []
        for enc in (self.lig_node_embedding, self.rec_node_embedding, self.atom_node_embedding):
            w, b = enc.sigma_proj()
            ws.append(w.detach().to(**f32))
            bs.append(b.detach().to(**f32))
        for k in ('ll', 'rr', 'aa', 'lr', 'la', 'ar'):
            ws.append(em[k]['w_sig'])
            bs.append(em[k]['b1'])
        if not self.confidence_mode:
            em['center'] = self._edge_mlp_pack(self.center_edge_embedding, self.center_distance_expansion, dev,
                                               (('rbf', dd), ('sig', sd)))
            proj_names.append('center')
            ws.append(em['center']['w_sig'])
            bs.append(em['center']['b1'])
            if not self.no_torsion:
                em['tor'] = self._edge_mlp_pack(self.final_edge_embedding, self.lig_distance_expansion, dev, (('rbf', dd),))
            if self.flexible_sidechains:
                em['sc'] = self._edge_mlp_pack(self.sidechain_final_edge_embedding, self.lig_distance_expansion, dev, (('rbf', dd),))
        P['em'], P['proj_names'] = em, proj_names
        P['static'] = {k: enc.static_pack(dev) for k, enc in (('lig', self.lig_node_embedding), ('rec', self.rec_node_embedding),
                                                               ('atom', self.atom_node_embedding))}
        self._static_cache = {}
        P['proj_w'], P['proj_b'] = torch.stack(ws).contiguous(), torch.stack(bs).contiguous()
        half = sd // 2
        P['freq'] = torch.exp(torch.arange(half, dtype=torch.float32) * -(np.log(10000) / (half - 1))).to(dev)
        conv_edges = ('ll', 'lr', 'la', 'aa', 'la', 'ar', 'rr', 'lr', 'ar')       # edge embedding each of a layer's 9 convs reads
        P['convs'] = [c.packed(dev, ns, ns, em[conv_edges[i % 9]]['fold'], fold_bn=True) for i, c in enumerate(self.conv_layers)]
        if not self.confidence_mode:
            P['final_conv'] = self.final_conv.packed(dev, ns, ns, em['center']['fold'])
            def lin(l):
                return l.weight.detach().T.contiguous().to(**f32), (l.bias.detach().contiguous().to(**f32) if l.bias is not None else None)
            P['tr'] = lin(self.tr_final_layer[0]) + lin(self.tr_final_layer[3])
            P['rot'] = lin(self.rot_final_layer[0]) + lin(self.rot_final_layer[3])
            P['c121'] = torch.tensor((tpmod.wigner_3j(1, 2, 1) * np.sqrt(3.0)).reshape(-1), **f32)
            if self._tor_ftp['paths'] is not None:
                P['ftp_ctab'] = torch.tensor(self._tor_ftp['ctab'], **f32)
                P['ftp_paths'] = (_lib.FtpPath * len(self._tor_ftp['paths']))(*[_lib.FtpPath(**q) for q in self._tor_ftp['paths']])
            if not self.no_torsion:
                P['tor_conv'] = self.tor_bond_conv.packed(dev, ns, ns, em['tor']['fold'])
                P['tor_mlp'] = [lin(self.tor_final_layer[0]), lin(self.tor_final_layer[3])]
            if self.flexible_sidechains:
                P['sc_conv'] = self.sc_tor_bond_conv.packed(dev, ns, ns, em['sc']['fold'])
                P['sc_mlp'] = [lin(self.sc_tor_final_layer[0]), lin(self.sc_tor_final_layer[3])]
        else:
            cp = self.confidence_predictor
            layers = []
            for li, bi in ((0, 1), (4, 5), (8, None)):
                W, b = cp[li].weight.detach().double(), cp[li].bias.detach().double()
                if bi is not None and isinstance(cp[bi], nn.BatchNorm1d):
                    bnm = cp[bi]
                    s = bnm.weight.detach().double() / torch.sqrt(bnm.running_var.detach().double() + bnm.eps)
                    W, b = W * s[:, None], (b - bnm.running_mean.detach().double()) * s + bnm.bias.detach().double()
                layers.append((W.T.float().contiguous().to(dev), b.float().contiguous().to(dev)))
            P['conf_mlp'] = layers
        self._packed = P
        return P

    # ------------------------------------------------------------------------------------------ plan
    STATIC_CACHE_SIZE = 256
    # Plans built while this is set run the atom-aggregating convs of the last two interaction layers on the edges into
    # atoms whose features are read afterwards only (_live_edges); the outputs that are read are the same.  Off: A/B runs.
    prune_edges = True
    LIVE_RADIUS_MARGIN = 0.01      # Å added to the torsion head's radius: the live set may be larger, never smaller

    def static_for(self, graph):
        """Time-independent node embeddings of ONE complex (``ddp_node_static_embed``: AtomEncoder sums + the part of its
        Linear that does not see sigma, incl. the 1280-wide ESM product) on the device: (ligand, atom, receptor) parts, each
        cached on its own -- a screening run re-uses the pocket's atom / residue embeddings across all ligands."""
        P = self.packed()
        rx = graph['receptor'].x
        return (self._static_one('lig', graph['ligand'].x, lambda x: (x, None)),
                self._static_one('atom', graph['atom'].x, lambda x: (x, None)),
                self._static_one('rec', rx, lambda x: ((x * 0 if self.no_aminoacid_identities else x)[:, :1],
                                                      (x * 0 if self.no_aminoacid_identities else x)[:, 1:] if self.lm_embedding_type else None)))

    static_h2d_bytes = 0          # bytes of static node features uploaded so far (bench.py's e2e accounting)

    def _static_one(self, kind, x, split):
        """Cache levels: (1) identity of the feature tensor (samples made by ``hetero.sample_copies`` share it; the entry
        keeps the tensor alive, so its address cannot be reused by another complex while it is cached); (2) content --
        deep-copied samples (the reference's inference.py:135) have equal values in different storage: same shape and
        fingerprint, then verified exactly with ``torch.equal`` (host reads instead of an upload + embedding per sample)."""
        P = self.packed()
        cache = self._static_cache.setdefault(kind, {})
        key = (x.data_ptr(), tuple(x.shape), x._version)
        hit = cache.get(key)
        if hit is not None:
            cache[key] = cache.pop(key)                                # most recently used last
            return hit[0]
        f = x.reshape(-1)
        fp = (tuple(x.shape), tuple(f[::max(1, f.numel() // 61)][:64].tolist()))
        out = None
        for out2, keep2, fp2 in reversed(list(cache.values())):
            if fp2 == fp and torch.equal(keep2, x):
                out = out2
                break
        if out is None:
            cat, lm = split(x)
            with torch.no_grad():
                out = static_embed(P['static'][kind], cat, lm, P['device'])
            self.static_h2d_bytes += 8 * cat.numel() + (4 * lm.numel() if lm is not None else 0)
        cache[key] = (out, x, fp)
        while len(cache) > self.STATIC_CACHE_SIZE:
            cache.pop(next(iter(cache)))
        return out

    def make_plan(self, data, extra_step_floats=0, graphs=None):
        """Upload one collated batch and allocate all workspaces (no per-step allocation afterwards).
        ``graphs``: the per-sample graphs ``data`` was collated from -- their static node features are then taken per
        complex from ``static_for`` (uploaded and embedded once per complex, not once per sample) and ``data`` may have
        been collated without the ``x`` matrices (``Batch.from_data_list(..., skip=STATIC_KEYS)``)."""
        P = self.packed()
        dev = P['device']
        ns, sh_dim = self.ns, self.sh_dim
        i32 = dict(dtype=torch.int32, device=dev)
        f32 = dict(dtype=torch.float32, device=dev)
        pl = Plan()
        pl.device = dev
        # accumulation mode, fixed for the plan's lifetime: int64 fixed-point sums under torch.use_deterministic_algorithms
        pl.deterministic = _lib.deterministic()
        sum_t = dict(dtype=_lib.sum_dtype(pl.deterministic), device=dev)
        pl.status = _lib.status_word(dev) if pl.deterministic else None
        lig, rec, atom = data['ligand'], data['receptor'], data['atom']
        B = int(data.num_graphs) if hasattr(data, 'num_graphs') or 'num_graphs' in data else 1
        pl.B = B

        def batch_of(store):
            return store.batch if 'batch' in store else torch.zeros(store.pos.shape[0], dtype=torch.long)

        def ptr_of(batch):
            cnt = torch.bincount(batch.cpu(), minlength=B)
            return torch.cat([torch.zeros(1, dtype=torch.long), cnt.cumsum(0)])
        lb, rb, ab = batch_of(lig).cpu(), batch_of(rec).cpu(), batch_of(atom).cpu()
        lp, rp, ap = ptr_of(lb), ptr_of(rb), ptr_of(ab)
        pl.NL, pl.NR, pl.NA = int(lp[-1]), int(rp[-1]), int(ap[-1])
        pl.lig_ptr_h, pl.rec_ptr_h, pl.atom_ptr_h = lp, rp, ap
        pl.lig_ptr, pl.rec_ptr, pl.atom_ptr = lp.to(**i32), rp.to(**i32), ap.to(**i32)
        pl.lig_batch, pl.rec_batch, pl.atom_batch = lb.to(**i32), rb.to(**i32), ab.to(**i32)
        pl.lig_pos = lig.pos.to(**f32).contiguous().clone()
        pl.rec_pos = rec.pos.to(**f32).contiguous().clone()
        pl.atom_pos = atom.pos.to(**f32).contiguous().clone()
        # static node-embedding parts (time independent, once per complex)
        with torch.no_grad():
            if graphs is not None:
                assert len(graphs) == B
                parts = [self.static_for(g) for g in graphs]
                pl.lig_static, pl.atom_static, pl.rec_static = (torch.cat([q[i] for q in parts], 0) if B > 1 else parts[0][i] for i in range(3))
                pl.static_h2d_bytes = 0
            else:
                rx = rec.x
                if self.no_aminoacid_identities:
                    rx = rx * 0
                pl.lig_static = static_embed(P['static']['lig'], lig.x, None, dev)
                pl.atom_static = static_embed(P['static']['atom'], atom.x, None, dev)
                pl.rec_static = static_embed(P['static']['rec'], rx[:, :1], rx[:, 1:] if self.lm_embedding_type else None, dev)
                pl.static_h2d_bytes = 8 * (lig.x.numel() + atom.x.numel() + rx.shape[0]) + 4 * rx.shape[0] * (rx.shape[1] - 1)
                self.static_h2d_bytes += pl.static_h2d_bytes
            assert pl.lig_static.shape[0] == pl.NL and pl.atom_static.shape[0] == pl.NA and pl.rec_static.shape[0] == pl.NR
        F = tpmod.irreps_dim(tpmod.parse_irreps(self.irrep_seq[3]))
        pl.F = F
        pl.x = {k: [torch.zeros(n, F, **f32), torch.zeros(n, F, **f32)] for k, n in (('l', pl.NL), ('r', pl.NR), ('a', pl.NA))}
        # ---- edge sets ---------------------------------------------------------------------------
        nl_g, nr_g, na_g = (lp[1:] - lp[:-1]), (rp[1:] - rp[:-1]), (ap[1:] - ap[:-1])
        bond_ei = data['ligand', 'ligand'].edge_index
        Eb = bond_ei.shape[1]
        pl.Eb = Eb
        es = {}
        es['ll'] = _EdgeSet(Eb + int(torch.minimum(nl_g - 1, torch.tensor(32)).clamp(min=0).mul(nl_g).sum()), ns, sh_dim, dev,
                            with_slab=(pl.NL, 33))
        es['ll'].edge[:Eb] = bond_ei[0].to(**i32)
        es['ll'].edge[es['ll'].cap:es['ll'].cap + Eb] = bond_ei[1].to(**i32)
        pl.bond_attr = data['ligand', 'ligand'].edge_attr.to(**f32).contiguous()
        k = self.atom_max_neighbors if self.atom_max_neighbors else 32
        pl.knn_k = k
        es['aa'] = _EdgeSet(int(torch.minimum(na_g - 1, torch.tensor(k + 1)).clamp(min=0).mul(na_g).sum()), ns, sh_dim, dev,
                            with_slab=(pl.NA, k + 1))
        es['lr'] = _EdgeSet(int((nl_g * nr_g).sum()), ns, sh_dim, dev, with_slab=(pl.NL, int(nr_g.max())))
        es['la'] = _EdgeSet(int((nl_g * na_g).sum()), ns, sh_dim, dev, with_slab=(pl.NL, int(na_g.max())))
        rr = data['receptor', 'receptor'].edge_index
        es['rr'] = _EdgeSet(rr.shape[1], ns, sh_dim, dev)
        es['rr'].set_static(rr.to(dev))
        ar = data['atom', 'receptor'].edge_index
        es['ar'] = _EdgeSet(ar.shape[1], ns, sh_dim, dev)
        es['ar'].set_static(ar.to(dev))
        pl.es = es
        # degree buffers: (edge set, row) -> int32 [n nodes of that side]
        sides = {('ll', 0): pl.NL, ('lr', 0): pl.NL, ('lr', 1): pl.NR, ('la', 0): pl.NL, ('la', 1): pl.NA, ('aa', 0): pl.NA,
                 ('ar', 0): pl.NA, ('ar', 1): pl.NR, ('rr', 0): pl.NR}
        pl.deg_arena = torch.zeros(sum(sides.values()), **i32)
        o = 0
        pl.deg_static = {}
        for (nm, r), n in sides.items():
            es[nm].deg[r] = pl.deg_arena[o:o + n]
            o += n
        # static part of the degrees (receptor-receptor, atom-receptor, ligand bond edges): counted once per complex
        pl.deg_base = torch.zeros_like(pl.deg_arena)
        o = 0
        for (nm, r), n in sides.items():
            if nm in ('rr', 'ar'):
                src = (rr if nm == 'rr' else ar)[r]
                pl.deg_base[o:o + n] = torch.bincount(src.cpu(), minlength=n).to(**i32)
            elif nm == 'll' and Eb > 0:
                pl.deg_base[o:o + n] = torch.bincount(bond_ei[r].cpu(), minlength=n).to(**i32)
            o += n
        dyn = [(nm, r) for (nm, r) in sides if nm not in ('rr', 'ar')]
        pl.deg_jobs = (_lib.DegreeJob * len(dyn))(*[
            _lib.DegreeJob(idx=es[nm].row(r), n_edges_dev=ptr(es[nm].n_dev), edge_cap=es[nm].cap,
                           start=Eb if nm == 'll' else 0, deg=ptr(es[nm].deg[r])) for (nm, r) in dyn])
        # scatter-sum arena: three updates per node type
        pl.sum_arena = torch.zeros((pl.NL + pl.NA + pl.NR) * F + 64, **sum_t)
        pl.sum_used = [min(pl.sum_arena.numel(), (pl.NL + pl.NA + pl.NR) * d + 16) for d in [tpmod.irreps_dim(tpmod.parse_irreps(q)) for q in self.irrep_seq]]
        pl.ones_F = torch.ones(F, **f32)
        pl.one_i32 = torch.ones(1, **i32)
        pl.sig = torch.zeros(B, self.sigma_embed_dim, **f32)
        pl.U = torch.zeros(len(P['proj_names']), B, ns, **f32)
        # ---- per-forward host scalars -> one pinned staging buffer ------------------------------
        T = 0 if self.no_torsion or self.confidence_mode else int(lig.edge_mask.sum())
        pl.T = T
        S = 0
        has_flex = self.flexible_sidechains and 'flexResidues' in data and len(data['flexResidues']) > 0 \
            and 'edge_idx' in data['flexResidues']
        if has_flex:
            S = int(data['flexResidues'].edge_idx.shape[0])
        pl.S = S
        pl.n_scal = 4 * B + T + S
        pl.step_in = torch.zeros(pl.n_scal + extra_step_floats, **f32)      # [per-graph scalars | caller's step inputs]
        pl.scal = pl.step_in[:pl.n_scal]
        if not self.confidence_mode:
            ce = torch.stack([lb, torch.arange(pl.NL)])
            es['center'] = _EdgeSet(pl.NL, ns, sh_dim, dev)
            es['center'].set_static(ce.to(dev))
            pl.center = torch.zeros(B, 3, **f32)
            pl.center_deg = (lp[1:] - lp[:-1]).to(**i32)
            pl.g_sum = torch.zeros(B, 12, **sum_t)
            pl.g = torch.zeros(B, 12, **f32)
            pl.tr_out, pl.rot_out = torch.zeros(B, 3, **f32), torch.zeros(B, 3, **f32)
            if T > 0:
                bonds = bond_ei[:, lig.edge_mask.bool()].long()
                pl.tor_batch_h = lb[bonds[0]]
                pl.tor = self._bond_head_plan(bonds, pl.tor_batch_h, B, pl.NL, int(nl_g.max()), dev, pl.deterministic)
            if S > 0:
                fr = data['flexResidues']
                frb = fr.batch.cpu() if 'batch' in fr else torch.zeros(S, dtype=torch.long)
                bonds = ap[:-1][frb] + fr.edge_idx.T.long().cpu()          # get_sc_tor_bonds, :638-652
                pl.sc_batch_h = frb
                pl.sc = self._bond_head_plan(bonds, frb, B, pl.NA, int(na_g.max()), dev, pl.deterministic)
            pl.tor_out = torch.zeros(max(T, 1), **f32)
            pl.sc_out = torch.zeros(max(S, 1), **f32)
        else:
            w = 2 * ns if self.num_conv_layers >= 3 else ns
            pl.conf_in = torch.zeros(B, w * (2 if self.flexible_sidechains else 1), **f32)
            nout = self.confidence_predictor[8].out_features
            pl.conf_out = torch.zeros(B, nout, **f32)
            if self.flexible_sidechains and S > 0:
                fr = data['flexResidues']
                frb = fr.batch.cpu() if 'batch' in fr else torch.zeros(S, dtype=torch.long)
                bonds = ap[:-1][frb] + fr.edge_idx.T.long().cpu()
                fa = bonds.unique()
                fcnt = torch.bincount(ab[fa], minlength=B)
                pl.flex_atoms = fa.to(**i32)
                pl.flex_ptr = torch.cat([torch.zeros(1, dtype=torch.long), fcnt.cumsum(0)]).to(**i32)
                bcnt = torch.bincount(frb, minlength=B)
                pl.live_bonds = (bonds.to(**i32).contiguous(), torch.cat([torch.zeros(1, dtype=torch.long), bcnt.cumsum(0)]).to(**i32), 0.0)
        # live atoms and pruned atom-aggregating edge sets of the last two interaction layers (_live_edges)
        nl = self.num_conv_layers
        pl.prune_layers = [l for l in (nl - 2, nl - 1) if l >= 0 and (self.flexible_sidechains or l < nl - 1)] if self.prune_edges else []
        pl.prune = bool(pl.prune_layers)
        if pl.prune:
            if not hasattr(pl, 'live_bonds'):
                pl.live_bonds = (pl.sc.bonds, pl.sc.ptr, self.lig_max_radius + self.LIVE_RADIUS_MARGIN) if S > 0 and not self.confidence_mode else None
            pl.live = torch.zeros(2, pl.NA, dtype=torch.uint8, device=dev)
            pl.pruned = {(l, nm): es[nm].live_copy(ns, sh_dim, dev) for l in pl.prune_layers for nm in ('aa', 'ar')}
        return pl

    def _bond_head_plan(self, bonds, bond_batch, B, n_nodes, max_seg, dev, det=False):
        i32 = dict(dtype=torch.int32, device=dev)
        f32 = dict(dtype=torch.float32, device=dev)
        h = Plan()
        n = bonds.shape[1]
        h.n = n
        h.bonds = bonds.to(**i32).contiguous()                      # [2, n]
        cnt = torch.bincount(bond_batch, minlength=B)
        h.ptr = torch.cat([torch.zeros(1, dtype=torch.long), cnt.cumsum(0)]).to(**i32)
        h.batch = bond_batch.to(**i32)
        h.mid, h.y2, h.attr = torch.zeros(n, 3, **f32), torch.zeros(n, 5, **f32), torch.zeros(n, self.ns, **f32)
        h.es = _EdgeSet(n * min(32, max_seg), self.ns, self.sh_dim, dev, with_slab=(n, min(32, max_seg)))
        h.sh_tor = torch.zeros(h.es.cap, self._tor_ftp['dim'], **f32)
        h.deg = torch.zeros(n, **i32)
        h.sum = torch.zeros(n, 2 * self.ns, dtype=_lib.sum_dtype(det), device=dev)
        h.feat = torch.zeros(n, 2 * self.ns, **f32)
        return h

    # ------------------------------------------------------------------------------------------ scalars
    def _host_scalars(self, pl, complex_t, out=None):
        """t, sigma, score norms and cutoffs per graph, computed on the host exactly like the reference
        (all_atom_score_model.py:243-245, 263, 383-384, 405-407, 432-433) and staged in one pinned buffer."""
        B, T, S = pl.B, pl.T, pl.S
        ct = [torch.as_tensor(complex_t[k]).detach().float().cpu().reshape(-1)[:B] for k in ('tr', 'rot', 'tor', 'sc_tor')]
        if self.confidence_mode:
            tr_s, rot_s, tor_s, sc_s = ct
        else:
            tr_s, rot_s, tor_s, sc_s = self.t_to_sigma(*ct)
        h = torch.zeros(pl.n_scal, dtype=torch.float32) if out is None else out
        # time of the sigma embedding: 'tr', or 't' under the asynchronous noise schedule (all_atom_score_model.py:370,450,492,517)
        h[0:B] = torch.as_tensor(complex_t['t']).detach().float().cpu().reshape(-1)[:B] if self.asyncronous_noise_schedule else ct[0]
        h[B:2 * B] = tr_s
        if not self.confidence_mode:
            h[2 * B:3 * B] = so3.score_norm(rot_s.float())
        h[3 * B:4 * B] = (tr_s * 3 + 20) if self.dynamic_max_cross else float(self.cross_max_distance)
        if T > 0:
            es = tor_s[pl.tor_batch_h]
            h[4 * B:4 * B + T] = torch.sqrt(torch.tensor(torus.score_norm(es.numpy()))).float()
        if S > 0 and not self.confidence_mode:
            es = sc_s[pl.sc_batch_h]
            h[4 * B + T:4 * B + T + S] = torch.sqrt(torch.tensor(torus.score_norm(es.numpy()))).float()
        if out is None:
            # fresh pinned staging buffer per call: the caching host allocator keeps it alive until the async copy ran
            pl.scal.copy_(h.pin_memory(), non_blocking=True)
        return h

    # ------------------------------------------------------------------------------------------ forward
    @staticmethod
    def _edges_desc(es, flip, x, p1, i1_row, p2, i2_row, out_scale=None, agg_deg=None):
        """ddp_tpconv_edges_t of one conv: agg / gather rows follow ``flip`` (torch.flip of edge_index).  With
        ``out_scale`` / ``agg_deg`` the conv accumulates mean- and BatchNorm-scaled contributions."""
        agg_r, gat_r = (1, 0) if flip else (0, 1)
        return _lib.TpEdges(emb=ptr(es.emb), p1=ptr(p1) if p1 is not None else None,
                            i1=es.row(i1_row) if p1 is not None else None, ld1=p1.shape[1] if p1 is not None else 0,
                            p2=ptr(p2) if p2 is not None else None, i2=es.row(i2_row) if p2 is not None else None,
                            ld2=p2.shape[1] if p2 is not None else 0, x=ptr(x), gather=es.row(gat_r), ldx=x.shape[1],
                            sh=ptr(es.sh_conv if hasattr(es, 'sh_conv') else es.sh), agg=es.row(agg_r), ew=None,
                            n_edges_dev=ptr(es.n_dev), edge_cap=es.cap, out_scale=ptr(out_scale), agg_deg=ptr(agg_deg))

    def _conv_group(self, L, st, items, status=None):
        """Fused tensor-product convolutions that share irreps (the convs of one interaction layer, or a single
        head conv).  items: (layer, packed, edge set, flip, x, p1, i1_row, p2, i2_row, sum_buf[, out_scale, agg_deg]).  On the tensor-core
        path they run as ONE persistent kernel over the union of their edge tiles (ddp_tpconv_umma_group).  ``status``: the
        plan's status word in the deterministic mode (int64 fixed-point sum buffers, the *_fixed kernels), else None."""
        if len(items) > 1 and not getattr(self, 'group_convs', True):      # one launch per conv (per-conv timing)
            for it in items:
                self._conv_group(L, st, [it], status)
            return
        det = status is not None
        prof = getattr(self, 'profile', None)
        if prof is not None:
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            ev0.record()
        tc = self.conv_mode != 'fp32' and all(tpmod.umma_supported(it[1].spec, self.ns) and it[5] is not None and it[7] is not None for it in items)
        eds = [self._edges_desc(*it[2:9], *it[10:12]) for it in items]
        if _lib.RECORD is not None:
            _lib.RECORD.append((None, None, eds))       # the grouped launch receives raw ADDRESSES of these: keep them alive with the record
        if tc:
            mode = 0 if self.conv_mode == 'bf16' else 1
            n = len(items)
            convs = (C.c_void_p * n)(*[C.addressof(it[1].cdesc) for it in items])
            imgs = (C.c_void_p * n)(*[ptr(it[1].umma_image(it[0], mode, it[4].device)) for it in items])
            edp = (C.c_void_p * n)(*[C.addressof(e) for e in eds])
            sums = (C.c_void_p * n)(*[ptr(it[9]) for it in items])
            if det:
                _lib.check(L.ddp_tpconv_umma_group_fixed(convs, imgs, mode, edp, sums, n, ptr(status), st), 'ddp_tpconv_umma_group_fixed')
            else:
                _lib.check(L.ddp_tpconv_umma_group(convs, imgs, mode, edp, sums, n, st), 'ddp_tpconv_umma_group')
        else:
            for it, e in zip(items, eds):
                if det:
                    _lib.check(L.ddp_tpconv_fp32_fixed(C.byref(it[1].cdesc), C.byref(e), ptr(it[9]), ptr(status), st), 'ddp_tpconv_fp32_fixed')
                else:
                    _lib.check(L.ddp_tpconv_fp32(C.byref(it[1].cdesc), C.byref(e), ptr(it[9]), st), 'ddp_tpconv_fp32')
        if prof is not None:
            ev1.record()
            if tc:
                prof.append((ev0, ev1, [(it[1].spec.weight_numel, it[2], self.ns) for it in items]))

    def run_plan(self, pl, complex_t, return_layers=False):
        """Forward on a resident plan.  Returns device tensors; performs no host synchronisation."""
        self._host_scalars(pl, complex_t)
        return self.launch_plan(pl, return_layers)

    def _branches(self, device):
        """Side streams of the launching stream (one set per stream, so that forwards issued on different streams --
        the sampler's concurrent mini-batches -- do not serialise on shared side streams)."""
        if getattr(self, '_br', None) is None:
            self._br = {}
        key = (str(device), torch.cuda.current_stream().cuda_stream)
        if key not in self._br:
            self._br[key] = _Branches(device)
        return self._br[key]

    replay_launches = os.environ.get('DDP_NO_REPLAY', '') == ''     # A/B switch of the recorded launch sequences

    def launch_plan(self, pl, return_layers=False):
        """Kernel launches only (per-graph scalars already staged in ``pl.scal``): CUDA-graph capturable.

        Nothing in the launch sequence of a resident plan changes from step to step (every pointer, count and descriptor is
        fixed; the per-step scalars live in device buffers), so the first launch RECORDS it -- the C-ABI calls with their
        marshalled arguments, the few torch fills in between, the stream forks / joins -- and later launches replay the
        record: ~0.5 ms of host time per forward instead of ~2.8 ms of Python descriptor building.  (The recorded closures
        capture tensors, never the plan itself: a plan -> record -> plan cycle would keep freed plans away from the caching
        allocator until the cyclic GC runs, and every new plan would pay cudaMalloc.)"""
        key = (self.conv_mode, torch.cuda.current_stream().cuda_stream, getattr(self, 'group_convs', True), id(self.packed()),
               pl.deterministic, pl.prune)
        debug = return_layers or getattr(self, 'profile', None) is not None or getattr(self, 'profile_small', None) is not None or not self.replay_launches
        prog = getattr(pl, 'program', None)
        if prog is not None and prog[0] == key and not debug:
            base = torch.cuda.current_stream()
            for name, fn, args in prog[1]:
                if name is None:                                   # torch op recorded with the stream it ran on
                    if fn is None:
                        continue                                   # keep-alive entry
                    if args is None or args == base:
                        fn()
                    else:
                        with torch.cuda.stream(args):
                            fn()
                elif fn(*args) != 0:
                    raise RuntimeError(f'{name} failed in a replayed launch')
            return prog[2]
        if debug:
            return self._launch_plan_body(pl, return_layers)
        assert _lib.RECORD is None, 'nested launch recording'
        _lib.RECORD = rec = []
        try:
            out = self._launch_plan_body(pl, False)
        finally:
            _lib.RECORD = None
        pl.program = (key, rec, out)
        return out

    def _small_begin(self):
        """Instrumented forwards only (``model.profile_small = []``): CUDA events around the HBM-type kernels."""
        if getattr(self, 'profile_small', None) is None:
            return None
        ev = torch.cuda.Event(enable_timing=True)
        ev.record()
        return ev

    def _small_end(self, ev0, name, nbytes):
        if ev0 is not None:
            ev1 = torch.cuda.Event(enable_timing=True)
            ev1.record()
            self.profile_small.append((name, ev0, ev1, nbytes))

    @staticmethod
    def _py(fn):
        """Run a torch-side step of the launch sequence (fill, copy, fork / join) and record it with its stream."""
        fn()
        if _lib.RECORD is not None:
            _lib.RECORD.append((None, fn, torch.cuda.current_stream()))

    def _live_edges(self, pl, L, st):
        """Live atoms and the pruned edge sets of ``pl.prune_layers``, on stream ``st``.  live[0]: the atoms whose
        last-layer features are read -- the side-chain torsion head's bond endpoints and every atom closer than
        lig_max_radius (+ margin) to a bond midpoint (its radius graph takes the first 32 of those), or the confidence
        model's flexible-bond atoms.  live[1]: the atoms whose layer L-2 features the last layer reads -- live[0] (the
        residual), the k-NN neighbours its atom-atom conv gathers into live[0] and every atom of a ligand-atom edge (the
        ligand-side conv gathers them).  Receptor features are not pruned: at t = 1 every ligand-residue pair is an edge."""
        es, live, chk = pl.es, pl.live, _lib.check
        bonds, bptr, r = pl.live_bonds if pl.live_bonds is not None else (None, None, 0.0)
        chk(L.ddp_mark_bond_nodes(ptr(pl.atom_pos), ptr(pl.atom_ptr), pl.B, pl.NA, ptr(bonds), 0 if bonds is None else bonds.shape[1],
                                  ptr(bptr), float(r), ptr(live[0]), st), 'ddp_mark_bond_nodes')
        self._py(lambda a=live[1], b=live[0]: a.copy_(b))
        aa, la = es['aa'], es['la']
        chk(L.ddp_mark_gathered(aa.row(0), aa.row(1), ptr(aa.n_dev), aa.cap, ptr(live[0]), ptr(live[1]), st), 'ddp_mark_gathered(aa)')
        chk(L.ddp_mark_gathered(None, la.row(1), ptr(la.n_dev), la.cap, None, ptr(live[1]), st), 'ddp_mark_gathered(la)')
        for (l, nm), p in pl.pruned.items():
            e = es[nm]
            chk(L.ddp_live_edges(ptr(e.edge), e.cap, ptr(e.n_dev), 0, ptr(e.sh), self.sh_dim, ptr(e.emb), self.ns,
                                 ptr(live[self.num_conv_layers - 1 - l]), ptr(p.counts), ptr(p.edge), p.cap, ptr(p.n_dev), ptr(p.sh),
                                 ptr(p.emb), st), f'ddp_live_edges({nm})')

    def _launch_plan_body(self, pl, return_layers=False):
        P = self.packed()
        L = _lib.lib()
        st = _lib.stream_ptr()
        B, ns, F = pl.B, self.ns, pl.F
        es = pl.es
        t_dev, tr_sigma, so3n, cutoff = pl.scal[0:B], pl.scal[B:2 * B], pl.scal[2 * B:3 * B], pl.scal[3 * B:4 * B]
        chk = _lib.check
        # readers of the conv sums: the fixed-point forms in the deterministic mode (int64 sum buffers)
        node_update = L.ddp_node_update_fixed if pl.deterministic else L.ddp_node_update
        node_update_multi = L.ddp_node_update_multi_fixed if pl.deterministic else L.ddp_node_update_multi
        names = P['proj_names']
        scale = float(self.timestep_emb_func.keywords.get('scale', 1.0)) if hasattr(self.timestep_emb_func, 'keywords') else float(getattr(self.timestep_emb_func, 'scale', 1.0))
        chk(L.ddp_graph_sigma_proj(ptr(t_dev), B, scale, ptr(P['freq']), self.sigma_embed_dim, ptr(P['proj_w']), ptr(P['proj_b']),
                                   len(names), ns, ptr(pl.sig), ptr(pl.U), st), 'ddp_graph_sigma_proj')
        U = {n: pl.U[i] for i, n in enumerate(names)}
        cur = {k: 0 for k in 'lra'}
        xl, xr, xa = pl.x['l'][0], pl.x['r'][0], pl.x['a'][0]
        chk(L.ddp_node_init(ptr(pl.lig_static), ptr(U['lig_node']), ptr(pl.lig_batch), pl.NL, ns, ptr(xl), F, st), 'node_init')
        chk(L.ddp_node_init(ptr(pl.rec_static), ptr(U['rec_node']), ptr(pl.rec_batch), pl.NR, ns, ptr(xr), F, st), 'node_init')
        chk(L.ddp_node_init(ptr(pl.atom_static), ptr(U['atom_node']), ptr(pl.atom_batch), pl.NA, ns, ptr(xa), F, st), 'node_init')
        # ---- dynamic graphs + edge geometry / embeddings: one independent chain per edge set, on side streams ------
        em = P['em']
        geo = {'ll': (pl.lig_pos, pl.lig_pos, pl.lig_batch), 'rr': (pl.rec_pos, pl.rec_pos, pl.rec_batch),
               'aa': (pl.atom_pos, pl.atom_pos, pl.atom_batch), 'lr': (pl.lig_pos, pl.rec_pos, pl.lig_batch),
               'la': (pl.lig_pos, pl.atom_pos, pl.lig_batch), 'ar': (pl.atom_pos, pl.rec_pos, pl.atom_batch)}

        def embed(nm, st_):
            pa, pb, ga = geo[nm]
            e_ = es[nm]
            pre, npre = (pl.bond_attr, pl.Eb) if nm == 'll' else (None, 0)
            t0 = self._small_begin()
            chk(L.ddp_edge_embed(ptr(pa), ptr(pb), ptr(e_.edge), e_.cap, ptr(e_.n_dev), ptr(ga), ptr(pre), npre, ptr(U[nm]),
                                 C.byref(em[nm]['desc']), ptr(e_.sh), ptr(e_.emb), st_), f'ddp_edge_embed({nm})')
            # algorithmic bytes per edge: two positions + two indices in, harmonics + hidden activations out
            self._small_end(t0, 'edge_embed_fold', lambda: int(e_.n_dev.item()) * (24 + 8 + 4 * (self.sh_dim + ns)))

        def build(nm, st_):
            e = es[nm]
            if nm == 'll':
                chk(L.ddp_radius(ptr(pl.lig_pos), ptr(pl.lig_pos), ptr(pl.lig_ptr), ptr(pl.lig_ptr), B, pl.NL, None,
                                 float(self.lig_max_radius), 33, 1, pl.Eb, ptr(e.slab), e.slab_w, ptr(e.counts), ptr(e.edge), e.cap,
                                 ptr(e.n_dev), st_), 'ddp_radius(ll)')
            elif nm == 'aa':
                chk(L.ddp_knn_graph(ptr(pl.atom_pos), ptr(pl.atom_ptr), B, pl.NA, pl.knn_k, ptr(e.slab), e.slab_w, ptr(e.counts),
                                    ptr(e.edge), e.cap, ptr(e.n_dev), st_), 'ddp_knn_graph')
            elif nm == 'lr' and self.dynamic_max_cross:
                chk(L.ddp_radius(ptr(pl.rec_pos), ptr(pl.lig_pos), ptr(pl.rec_ptr), ptr(pl.lig_ptr), B, pl.NL, ptr(cutoff), 1.0, 10000,
                                 0, 0, ptr(e.slab), e.slab_w, ptr(e.counts), ptr(e.edge), e.cap, ptr(e.n_dev), st_), 'ddp_radius(lr)')
            elif nm == 'lr':
                chk(L.ddp_radius(ptr(pl.rec_pos), ptr(pl.lig_pos), ptr(pl.rec_ptr), ptr(pl.lig_ptr), B, pl.NL, None,
                                 float(self.cross_max_distance), 10000, 0, 0, ptr(e.slab), e.slab_w, ptr(e.counts), ptr(e.edge), e.cap,
                                 ptr(e.n_dev), st_), 'ddp_radius(lr)')
            else:
                chk(L.ddp_radius(ptr(pl.atom_pos), ptr(pl.lig_pos), ptr(pl.atom_ptr), ptr(pl.lig_ptr), B, pl.NL, None,
                                 float(self.lig_max_radius), 10000, 0, 0, ptr(e.slab), e.slab_w, ptr(e.counts), ptr(e.edge), e.cap,
                                 ptr(e.n_dev), st_), 'ddp_radius(la)')
            embed(nm, st_)

        br = self._branches(pl.device)
        main = torch.cuda.current_stream()
        self._py(lambda: br.fork(3))
        for side, nm in zip(br.side, ('aa', 'lr', 'la')):
            with torch.cuda.stream(side):
                build(nm, _lib.stream_ptr())
        build('ll', st)
        embed('rr', st)
        embed('ar', st)
        self._py(lambda: br.join(main, 3))
        self._py(lambda a=pl.deg_arena, b=pl.deg_base: a.copy_(b))   # static edge sets + ligand bond edges
        chk(L.ddp_degree_multi(pl.deg_jobs, len(pl.deg_jobs), st), 'ddp_degree_multi')   # dynamic ones, one launch
        # per-layer outputs of every node are returned unpruned
        prune = pl.prune and not return_layers
        if prune:
            self._py(lambda: br.fork(1))                                 # joined before the first pruned layer
            with torch.cuda.stream(br.side[0]):
                self._live_edges(pl, L, _lib.stream_ptr())
        # ---- interaction layers (all_atom_score_model.py:271-324) --------------------------------
        layers_out = []
        seq_dims = [tpmod.irreps_dim(tpmod.parse_irreps(s)) for s in self.irrep_seq]
        for l in range(self.num_conv_layers):
            last = l == self.num_conv_layers - 1
            f_old, f_new = seq_dims[min(l, 3)], seq_dims[min(l + 1, 3)]
            Cv, Pk = self.conv_layers, P['convs']
            self._py(lambda a=pl.sum_arena[:pl.sum_used[min(l + 1, 3)]]: a.zero_())
            o = 0

            def take(n):
                nonlocal o
                v = pl.sum_arena[o:o + n * f_new].view(n, f_new)
                o += (n * f_new + 3) // 4 * 4                                # keep every slice 16-byte aligned
                return v

            # One accumulation buffer per node type: every conv adds out * bn_scale / in-degree (its scatter-mean and
            # BatchNorm scale, all_atom_score_model.py:315-324 + score_model.py:117,123) straight into it.
            def job(ci, nm, flip, x, p1, i1, p2, i2, buf):
                agg_r = 1 if flip else 0
                # atom-aggregating aa / ar convs of a pruned layer: the edges into live atoms; degrees of the full set
                e_ = pl.pruned[(l, nm)] if prune and not flip and (l, nm) in pl.pruned else es[nm]
                # BatchNorm scale lives in the packed weights (PackedConv fold_bn); without BatchNorm out_scale stays NULL
                return (Cv[ci], Pk[ci], e_, flip, x, p1, i1, p2, i2, buf, None, es[nm].deg[agg_r])
            s_l = take(pl.NL)
            grp = [job(9 * l, 'll', False, xl, xl, 0, xl, 1, s_l), job(9 * l + 1, 'lr', False, xr, xl, 0, xr, 1, s_l),
                   job(9 * l + 2, 'la', False, xa, xl, 0, xa, 1, s_l)]
            do_atom = self.flexible_sidechains or not last
            if do_atom:
                s_a = take(pl.NA)
                grp += [job(9 * l + 3, 'aa', False, xa, xa, 0, xa, 1, s_a), job(9 * l + 4, 'la', True, xl, xa, 1, xl, 0, s_a),
                        job(9 * l + 5, 'ar', False, xr, xa, 0, xr, 1, s_a)]
                if not last:
                    s_r = take(pl.NR)
                    grp += [job(9 * l + 6, 'rr', False, xr, xr, 0, xr, 1, s_r), job(9 * l + 7, 'lr', True, xl, xr, 1, xl, 0, s_r),
                            job(9 * l + 8, 'ar', True, xa, xr, 1, xa, 0, s_r)]
            # largest edge sets first: the round-robin tile walk then ends on the small ones
            grp.sort(key=lambda it: -it[2].cap)
            if prune and l == pl.prune_layers[0]:
                self._py(lambda: br.join(main, 1))
            self._conv_group(L, st, grp, pl.status)

            def update(key, x_old, n, buf, items):
                # the buffer is already normalised (deg = NULL); every live conv still contributes its BatchNorm shift
                # (empty edge sets: `return 0`, score_model.py:109-111); the buffer itself is always read
                x_new = pl.x[key][1 - cur[key]]
                cur[key] = 1 - cur[key]
                J = _lib.NodeUpdateJob(old_x=ptr(x_old), f_old=f_old, ld_old=F, n_updates=len(items) + 1, n=n, f_new=f_new,
                                       new_x=ptr(x_new), ld_new=F)
                J.updates[0] = _lib.Update(sum=ptr(buf), deg=None, scale=None, shift=None, n_edges_dev=ptr(pl.one_i32))
                for k, (nm, ci) in enumerate(items):
                    J.updates[k + 1] = _lib.Update(sum=None, deg=None, scale=None, shift=ptr(Pk[ci].bn_shift), n_edges_dev=ptr(es[nm].n_dev))
                return x_new, J
            xl_new, Jl = update('l', xl, pl.NL, s_l, [('ll', 9 * l), ('la', 9 * l + 2), ('lr', 9 * l + 1)])
            node_jobs = [Jl]
            if do_atom:
                xa_new, Ja = update('a', xa, pl.NA, s_a, [('aa', 9 * l + 3), ('la', 9 * l + 4), ('ar', 9 * l + 5)])
                node_jobs.append(Ja)
                if not last:
                    xr, Jr = update('r', xr, pl.NR, s_r, [('rr', 9 * l + 6), ('ar', 9 * l + 8), ('lr', 9 * l + 7)])
                    node_jobs.append(Jr)
                xa = xa_new
            t0 = self._small_begin()
            chk(node_update_multi((_lib.NodeUpdateJob * len(node_jobs))(*node_jobs), len(node_jobs), st), 'ddp_node_update_multi')
            # algorithmic bytes per node: old features + the accumulated update in, new features out
            self._small_end(t0, 'node_update_multi', lambda jobs_=tuple((J.n, J.f_old, J.f_new) for J in node_jobs): sum(4 * n * (fo + 2 * fn) for n, fo, fn in jobs_))
            xl = xl_new
            if return_layers:
                layers_out.append((xl[:, :f_new].clone(), xa[:, :f_new if do_atom else f_old].clone(), xr.clone()))
        pl.last_layers = layers_out
        f_last = seq_dims[min(self.num_conv_layers, 3)]

        if self.confidence_mode:                                       # :329-353
            w = 2 * ns if self.num_conv_layers >= 3 else ns
            ld = pl.conf_in.shape[1]
            chk(L.ddp_segment_mean(ptr(xl), None, ptr(pl.lig_ptr), B, ns, F, ptr(pl.conf_in), ld, st), 'segment_mean')
            if self.num_conv_layers >= 3:
                chk(L.ddp_segment_mean(xl.data_ptr() + 4 * (f_last - ns), None, ptr(pl.lig_ptr), B, ns, F,
                                       pl.conf_in.data_ptr() + 4 * ns, ld, st), 'segment_mean')
            if self.flexible_sidechains:
                if pl.S > 0:
                    chk(L.ddp_segment_mean(ptr(xa), ptr(pl.flex_atoms), ptr(pl.flex_ptr), B, ns, F, pl.conf_in.data_ptr() + 4 * w, ld, st), 'segment_mean')
                    if self.num_conv_layers >= 3:
                        chk(L.ddp_segment_mean(xa.data_ptr() + 4 * (f_last - ns), ptr(pl.flex_atoms), ptr(pl.flex_ptr), B, ns, F,
                                               pl.conf_in.data_ptr() + 4 * (w + ns), ld, st), 'segment_mean')
                else:
                    self._py(lambda a=pl.conf_in[:, w:]: a.zero_())
            lay = P['conf_mlp']
            arr = (_lib.MlpLayer * 3)(*[_lib.MlpLayer(wt=ptr(wt), b=ptr(b), n_in=wt.shape[0], n_out=wt.shape[1], act=a)
                                       for (wt, b), a in zip(lay, (1, 1, 0))])
            chk(L.ddp_row_mlp(ptr(pl.conf_in), B, ld, arr, 3, None, ptr(pl.conf_out), pl.conf_out.shape[1], st), 'row_mlp')
            return pl.conf_out.squeeze(dim=-1)

        # ---- heads: the two torsion heads run on side streams next to the translation / rotation head --------------
        def tor_head(key, n, pos, xn, nptr, conv, mlp_key, emk, out, soff, st_):           # :386-434
            h = getattr(pl, key)
            e = h.es
            chk(L.ddp_bond_geometry(ptr(pos), ptr(h.bonds), n, ptr(xn), F, ns, ptr(h.mid), ptr(h.y2), ptr(h.attr), st_), 'bond_geometry')
            chk(L.ddp_radius(ptr(pos), ptr(h.mid), ptr(nptr), ptr(h.ptr), B, n, None, float(self.lig_max_radius), 32, 0, 0,
                             ptr(e.slab), e.slab_w, ptr(e.counts), ptr(e.edge), e.cap, ptr(e.n_dev), st_), f'ddp_radius({key})')
            chk(L.ddp_edge_embed(ptr(h.mid), ptr(pos), ptr(e.edge), e.cap, ptr(e.n_dev), ptr(h.batch), None, 0, None,
                                 C.byref(em[emk]['desc']), ptr(e.sh), ptr(e.emb), st_), f'ddp_edge_embed({key})')
            if self._tor_ftp['paths'] is None:
                chk(L.ddp_tor_edge_sh(ptr(e.sh), self.sh_dim, ptr(h.y2), ptr(P['c121']), ptr(e.edge), ptr(e.n_dev), e.cap, ptr(h.sh_tor), st_), 'tor_edge_sh')
            else:
                chk(L.ddp_tor_edge_sh_generic(ptr(e.sh), self.sh_dim, ptr(h.y2), P['ftp_paths'], len(P['ftp_paths']), ptr(P['ftp_ctab']),
                                              ptr(e.edge), ptr(e.n_dev), e.cap, ptr(h.sh_tor), self._tor_ftp['dim'], st_), 'tor_edge_sh_generic')
            e.sh_conv = h.sh_tor
            self._py(lambda a=h.sum, b=h.deg: (a.zero_(), b.zero_()))
            chk(L.ddp_degree(e.row(0), ptr(e.n_dev), e.cap, ptr(h.deg), st_), 'ddp_degree')
            pk = P[key + '_conv']
            self._conv_group(L, st_, [(conv, pk, e, False, xn, xn, 1, h.attr, 0, h.sum)], pl.status)
            up = _lib.Update(sum=ptr(h.sum), deg=ptr(h.deg), scale=ptr(pk.bn_scale), shift=ptr(pk.bn_shift), n_edges_dev=ptr(e.n_dev))
            chk(node_update(None, 0, 0, C.byref(up), 1, n, 2 * ns, ptr(h.feat), 2 * ns, st_), 'ddp_node_update')
            (w1, _), (w2, _) = P[mlp_key]
            arr = (_lib.MlpLayer * 2)(_lib.MlpLayer(wt=ptr(w1), b=None, n_in=2 * ns, n_out=ns, act=2),
                                      _lib.MlpLayer(wt=ptr(w2), b=None, n_in=ns, n_out=1, act=0))
            rs = pl.scal[soff:soff + n] if self.scale_by_sigma else None
            chk(L.ddp_row_mlp(ptr(h.feat), n, 2 * ns, arr, 2, ptr(rs), ptr(out), 1, st_), 'row_mlp')
            return out[:n]

        heads = (('tor', pl.T, pl.lig_pos, xl, pl.lig_ptr, getattr(self, 'tor_bond_conv', None), 'tor_mlp', 'tor', pl.tor_out, 4 * B),
                 ('sc', pl.S, pl.atom_pos, xa, pl.atom_ptr, getattr(self, 'sc_tor_bond_conv', None), 'sc_mlp', 'sc', pl.sc_out, 4 * B + pl.T))
        self._py(lambda: br.fork(2))
        outs = []
        for side, hd in zip(br.side, heads):
            if hd[1] == 0:
                outs.append(torch.empty(0, device=pl.device))
                continue
            with torch.cuda.stream(side):
                outs.append(tor_head(*hd, _lib.stream_ptr()))
        # translation / rotation head (:357-384)
        ec = es['center']
        chk(L.ddp_segment_mean(ptr(pl.lig_pos), None, ptr(pl.lig_ptr), B, 3, 3, ptr(pl.center), 3, st), 'segment_mean')
        chk(L.ddp_edge_embed(ptr(pl.center), ptr(pl.lig_pos), ptr(ec.edge), ec.cap, ptr(ec.n_dev), None, None, 0, ptr(U['center']),
                             C.byref(em['center']['desc']), ptr(ec.sh), ptr(ec.emb), st), 'ddp_edge_embed(center)')
        self._py(lambda a=pl.g_sum: a.zero_())
        self._conv_group(L, st, [(self.final_conv, P['final_conv'], ec, False, xl, xl, 1 if self.fixed_center_conv else 0, None, 0, pl.g_sum)],
                         pl.status)
        fc = P['final_conv']
        up = _lib.Update(sum=ptr(pl.g_sum), deg=ptr(pl.center_deg), scale=ptr(fc.bn_scale), shift=ptr(fc.bn_shift), n_edges_dev=ptr(ec.n_dev))
        chk(node_update(None, 0, 0, C.byref(up), 1, B, 12, ptr(pl.g), 12, st), 'ddp_node_update')
        (tw1, tb1, tw2, tb2), (rw1, rb1, rw2, rb2) = P['tr'], P['rot']
        if self.scale_by_sigma:
            trs, son = tr_sigma, so3n
        else:
            trs = son = pl.ones_F[:B] if B <= pl.ones_F.numel() else torch.ones(B, device=pl.device)
        chk(L.ddp_tr_rot_head(ptr(pl.g), ptr(pl.sig), self.sigma_embed_dim, B, ptr(tw1), ptr(tb1), ptr(tw2), ptr(tb2), ptr(rw1),
                              ptr(rb1), ptr(rw2), ptr(rb2), ns, ptr(trs), ptr(son), ptr(pl.tr_out), ptr(pl.rot_out), st), 'tr_rot_head')
        self._py(lambda: br.join(main, 2))
        return pl.tr_out, pl.rot_out, outs[0], outs[1]

    def forward(self, data):
        """Drop-in ``model(data)`` on a collated batch (uploads the batch, runs, returns device tensors)."""
        pl = self.make_plan(data)
        out = self.run_plan(pl, data.complex_t)
        # side effects the reference's forward leaves on ``data`` (all_atom_score_model.py:373,453,495,520,530)
        data['atom', 'atom'].edge_index = pl.es['aa'].edge_index()
        data.graph_sigma_emb = pl.sig
        for key in ('ligand', 'receptor', 'atom'):
            node_t = getattr(data[key], 'node_t', None)
            if node_t is not None:
                data[key].node_sigma_emb = self.timestep_emb_func(torch.as_tensor(node_t['t' if self.asyncronous_noise_schedule else 'tr'], dtype=torch.float32).to(pl.device))
        self._last_plan = pl
        if pl.deterministic:
            _lib.check_status(pl.device)          # (the k-NN edge list above was already read back: no extra stall)
        return out
