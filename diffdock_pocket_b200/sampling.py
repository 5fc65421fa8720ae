"""Reverse-diffusion sampler: host mirror of ``utils/sampling.py``.

``sampling()`` keeps the reference signature and return values (utils/sampling.py:70-286) and draws
its noise from the same generators in the same order (``torch.normal`` on the CPU default generator:
tr_z, rot_z, tor_z, sidechain_tor_z per step), but the loop body is restructured for the GPU:

* every mini-batch of ``batch_size`` samples is collated and uploaded ONCE (``model.make_plan``) and
  stays resident; the reference re-collates and re-uploads every step (utils/sampling.py:100,114);
* per step and batch: one H2D copy of the step's noise slice, the score-model forward
  (``model.run_plan``, no host sync) and one fused pose-update launch (``ddp_pose_update``) that turns
  scores + noise into the new ligand / side-chain coordinates on the device; the reference makes
  N x (n_sc + 1) CPU round trips per step (utils/sampling.py:245-251);
* poses return to the host once, after the last step (and the confidence pass).

``use_graph=True`` additionally captures each mini-batch's whole step as a CUDA graph (worth it only when the
plans outlive many calls or the batch is so small that launches dominate: capture + instantiation cost ~40 ms per
mini-batch, while at batch 20 the eager launch stream already runs ~4x ahead of the GPU).

Resident state outlives the call when calls repeat: from the first REPEAT of an input's shape signature on, the runners
(plans, workspaces, pose tables, recorded launch programs) and the confidence plans of the last ``PLAN_CACHE_SIZE`` distinct
inputs are kept, keyed by the CONTENT of everything the plans were built from (topology, static features, receptor coordinates -- everything but the moving ligand / atom
coordinates).  A later call on the same complex(es) -- re-docking, more samples, a screening loop over one pocket with a
recurring ligand -- only uploads the new start poses: the ~50 ms of host-side collation and plan building of the first
call, during which the GPU starves inside step 0, are gone (``DDP_PLAN_CACHE=0`` disables the cache).

SVGD (svgd_weight > 0) and ``pivot`` are outside the accelerated path and raise NotImplementedError; the asynchronous
noise schedule (``asyncronous_noise_schedule=True`` with ``t_schedule``, utils/sampling.py:116-117) is supported: the step's
``t_schedule[t_idx]`` becomes the time of the sigma embeddings.
"""
import collections
import contextlib
import copy
import gc
import os

import numpy as np
import torch
from scipy.spatial.transform import Rotation as R

from .diffusion_utils import PoseState, modify_conformer, modify_sidechains
from .all_atom_score_model import STATIC_KEYS
from .hetero import Batch
from . import _lib


def randomize_position(data_list, no_torsion, no_random, tr_sigma_max, pocket_knowledge=False, pocket_cutoff=7,
                       flexible_sidechains=False):
    """utils/sampling.py:16-60 (in-place).  Host-side initial-state generator (once per complex)."""
    from .torsion import modify_conformer_torsion_angles
    center_pocket = 0
    if pocket_knowledge:
        g = data_list[0]
        d = torch.cdist(g['receptor'].pos, torch.from_numpy(g['ligand'].orig_pos[0]).float() - g.original_center)
        label = torch.any(d < pocket_cutoff, dim=1)
        center_pocket = g['receptor'].pos[label].mean(dim=0) if torch.any(label) else \
            g['receptor'].pos[torch.argmin(torch.min(d, dim=1)[0])]
    if not no_torsion:
        for g in data_list:
            upd = np.random.uniform(low=-np.pi, high=np.pi, size=int(g['ligand'].edge_mask.sum()))
            mr = g['ligand'].mask_rotate
            mr = mr if isinstance(mr, np.ndarray) else mr[0]
            g['ligand'].pos = modify_conformer_torsion_angles(
                g['ligand'].pos, g['ligand', 'ligand'].edge_index.T[g['ligand'].edge_mask], mr, upd)
    if flexible_sidechains:
        from .torsion import modify_sidechains_host
        for g in data_list:
            if 'flexResidues' not in g or 'edge_idx' not in g['flexResidues']:
                continue                                  # complex without flexible residues in a mixed list (draws nothing)
            upd = np.random.uniform(low=-np.pi, high=np.pi, size=len(g['flexResidues'].edge_idx))
            modify_sidechains_host(g, upd)
    for g in data_list:
        center = torch.mean(g['ligand'].pos, dim=0, keepdim=True)
        rot = torch.from_numpy(R.random().as_matrix()).float()
        g['ligand'].pos = (g['ligand'].pos - center) @ rot.T + center_pocket
        if not no_random:
            g['ligand'].pos += torch.normal(mean=0, std=tr_sigma_max, size=(1, 3))


# ------------------------------------------------------------------------------------------ resident-state cache
PLAN_CACHE_SIZE = int(os.environ.get('DDP_PLAN_CACHE', 2))      # inputs (lists of complexes) whose resident state is kept; 0: off
_PLAN_CACHE = collections.OrderedDict()                         # key -> {'runners', 'conf_plans', 'busy'}
_SEEN_SIGS = collections.OrderedDict()                          # shape signatures of recent calls (retention starts at the first repeat)
LAST_CALL = {'plan_reused': False}                              # bench.py's H2D accounting reads this


def _bytes_key(t):
    if t is None:
        return None
    if torch.is_tensor(t):
        t = t.detach().cpu().contiguous()
        return (tuple(t.shape), str(t.dtype), hash(t.numpy().tobytes()))
    a = np.ascontiguousarray(np.asarray(t))
    return (a.shape, str(a.dtype), hash(a.tobytes()))


def _graph_key(g, flexible_sidechains):
    """Content key of everything a plan / pose state is built from in one complex graph, except the ligand and atom
    coordinates (the only per-call inputs).  Exact (hash of the bytes) for the index / feature tables; the receptor's
    wide language-model features are keyed by a strided sample next to the exact receptor coordinates."""
    lig, rec, atom = g['ligand'], g['receptor'], g['atom']
    mr = lig.mask_rotate if 'mask_rotate' in lig else None
    if mr is not None and not isinstance(mr, np.ndarray):
        mr = mr[0]
    rx = rec.x.reshape(-1)
    key = [tuple(lig.pos.shape), tuple(atom.pos.shape), _bytes_key(lig.x), _bytes_key(lig.edge_mask if 'edge_mask' in lig else None),
           _bytes_key(mr), _bytes_key(g['ligand', 'ligand'].edge_index), _bytes_key(g['ligand', 'ligand'].edge_attr),
           _bytes_key(rec.pos), tuple(rec.x.shape), tuple(rx[::max(1, rx.numel() // 251)][:256].tolist()),
           _bytes_key(g['receptor', 'receptor'].edge_index), _bytes_key(atom.x), _bytes_key(g['atom', 'receptor'].edge_index)]
    if flexible_sidechains and 'flexResidues' in g and 'edge_idx' in g['flexResidues']:
        fr = g['flexResidues']
        key += [_bytes_key(fr.edge_idx), _bytes_key(fr.subcomponents), _bytes_key(fr.subcomponentsMapping)]
    else:
        key.append(None)
    return tuple(key)


def _graph_tables(g, flexible_sidechains):
    lig, rec, atom = g['ligand'], g['receptor'], g['atom']
    mr = lig.mask_rotate if 'mask_rotate' in lig else None
    if mr is not None and not isinstance(mr, np.ndarray):
        mr = mr[0]
    rx = rec.x.reshape(-1)                                         # wide language-model features: strided sample, as in _graph_key
    t = [lig.x, lig.edge_mask if 'edge_mask' in lig else None, mr, g['ligand', 'ligand'].edge_index, g['ligand', 'ligand'].edge_attr,
         rec.pos, rx[::max(1, rx.numel() // 251)][:256], g['receptor', 'receptor'].edge_index, atom.x, g['atom', 'receptor'].edge_index]
    if flexible_sidechains and 'flexResidues' in g and 'edge_idx' in g['flexResidues']:
        fr = g['flexResidues']
        t += [fr.edge_idx, fr.subcomponents, fr.subcomponentsMapping]
    return t


def _same_tables(a, b):
    if len(a) != len(b):
        return False
    for x, y in zip(a, b):
        if x is y:
            continue
        if x is None or y is None:
            return False
        if torch.is_tensor(x) and torch.is_tensor(y):
            if x.shape != y.shape or x.dtype != y.dtype or not torch.equal(x, y):
                return False
        elif not np.array_equal(np.asarray(x), np.asarray(y)):
            return False
    return True


def _cache_key(model, confidence_model, device, batch_size, flexible_sidechains, no_torsion, use_graph, concurrent_batches,
               deterministic, graph_keys):
    """Key of one resident-state entry: everything its plans, recorded launch programs and captured step graphs were
    built for -- including the accumulation mode, so that state built in one mode is never replayed in the other."""
    return (id(model), id(confidence_model), getattr(model, 'conv_mode', None), getattr(model, 'group_convs', None), str(device),
            batch_size, bool(flexible_sidechains), bool(no_torsion), bool(use_graph), bool(concurrent_batches), bool(deterministic),
            tuple(graph_keys))


def _cache_get(key, model, confidence_model, deterministic):
    """The cached entry for ``key`` if it may be used now: not owned by an unfinished (deferred) call, built for these
    model objects (ids can be recycled) and in this accumulation mode."""
    e = _PLAN_CACHE.get(key)
    if e is None or e['busy'] or e['models'][0]() is not model or e['deterministic'] != bool(deterministic):
        return None
    if confidence_model is not None and e['models'][1]() is not confidence_model:
        return None
    return e


def clear_plan_cache():
    _PLAN_CACHE.clear()
    _SEEN_SIGS.clear()


def is_iterable(arr):
    try:
        iter(arr)
        return True
    except TypeError:
        return False


def step_coefficients(t_idx, inference_steps, schedules, t_to_sigma, model_args, ode, temp_sampling, temp_psi,
                      temp_sigma_data, flexible_sidechains):
    """Host scalars of one step (utils/sampling.py:94-98, 110, 129-195): perturb = a * score + b * z."""
    ma = model_args
    tr_s, rot_s, tor_s, sc_s = schedules
    last = t_idx == inference_steps - 1
    t = [s[t_idx] for s in schedules]
    dt = [s[t_idx] - s[t_idx + 1] if not last else s[t_idx] for s in schedules]
    sig = t_to_sigma(*t)
    rng = [(ma.tr_sigma_max, ma.tr_sigma_min), (ma.rot_sigma_max, ma.rot_sigma_min), (ma.tor_sigma_max, ma.tor_sigma_min),
           (getattr(ma, 'sidechain_tor_sigma_max', 1.0), getattr(ma, 'sidechain_tor_sigma_min', 1.0))]
    g = [sig[0] * np.sqrt(2 * np.log(rng[0][0] / rng[0][1])), 2 * sig[1] * np.sqrt(np.log(rng[1][0] / rng[1][1])),
         sig[2] * np.sqrt(2 * np.log(rng[2][0] / rng[2][1])), sig[3] * np.sqrt(2 * np.log(rng[3][0] / rng[3][1]))]
    ts = list(temp_sampling) if is_iterable(temp_sampling) else [temp_sampling] * 4
    tp = list(temp_psi) if is_iterable(temp_psi) else [temp_psi] * 4
    assert len(ts) == 4 and len(tp) == 4
    coef = []
    for k in range(4):
        if ode:
            a, b = 0.5 * g[k] ** 2 * dt[k], 0.0
        else:
            a, b = g[k] ** 2 * dt[k], g[k] * np.sqrt(dt[k])
        active = (k < 2) or (k == 2 and not ma.no_torsion) or (k == 3 and flexible_sidechains)
        if ts[k] != 1.0 and active:
            sd = np.exp(temp_sigma_data * np.log(rng[k][0]) + (1 - temp_sigma_data) * np.log(rng[k][1]))
            lam = (sd + sig[k]) / (sd + sig[k] / ts[k])
            a, b = g[k] ** 2 * dt[k] * (lam + ts[k] * tp[k] / 2), g[k] * np.sqrt(dt[k] * (1 + tp[k]))
        coef += [float(a), float(b)]
    return t, coef


class StepRunner:
    """One resident mini-batch: plan + pose state + (optionally) the captured CUDA graph of one whole
    reverse-diffusion step (score-model forward + fused pose update).  Per step the host stages ONE pinned row
    [per-graph scalars | 8 step coefficients | tr_z | rot_z | tor_z | sc_z], copies it to the device with one
    async H2D and replays the graph: no other host work, no synchronisation."""

    def __init__(self, model, data_sub, flexible_sidechains, no_torsion, use_graph=True, stream=None):
        b = len(data_sub)
        self.model, self.b = model, b
        self.stream = stream                     # None: the caller's current stream
        n_tor = 0 if no_torsion else sum(int(g['ligand'].edge_mask.sum()) for g in data_sub)
        n_sc = sum(int(g['flexResidues'].edge_idx.shape[0]) for g in data_sub
                   if flexible_sidechains and 'flexResidues' in g and 'edge_idx' in g['flexResidues'])
        self.n_extra = 8 + 6 * b + n_tor + n_sc
        self.pl = model.make_plan(Batch.from_data_list(data_sub, skip=STATIC_KEYS), extra_step_floats=self.n_extra, graphs=data_sub)
        pl = self.pl
        # the pose state (host loops over the samples' bond tables) is only needed by the pose update that FOLLOWS the first
        # forward: it is built after that forward has been launched, i.e. while the GPU already works (see _launch)
        self._ps_args = (data_sub, pl.device, flexible_sidechains, no_torsion)
        self._ps = None
        self.T, self.S = n_tor, n_sc
        o = pl.n_scal
        x = pl.step_in
        self.coef_dev = x[o:o + 8]
        o += 8
        self.z = (x[o:o + 3 * b], x[o + 3 * b:o + 6 * b], x[o + 6 * b:o + 6 * b + self.T],
                  x[o + 6 * b + self.T:o + 6 * b + self.T + self.S])
        self.use_sc = flexible_sidechains and n_sc > 0
        self.graph = None
        self.use_graph = use_graph
        self.out = None
        self.calls = 0

    def reset(self, data_sub):
        """Re-use this runner for another call on the same complexes: only the start poses change (two H2D copies)."""
        lp = torch.cat([g['ligand'].pos for g in data_sub]).float().pin_memory()
        ap = torch.cat([g['atom'].pos for g in data_sub]).float().pin_memory()
        assert lp.shape == self.pl.lig_pos.shape and ap.shape == self.pl.atom_pos.shape
        self.pl.lig_pos.copy_(lp, non_blocking=True)
        self.pl.atom_pos.copy_(ap, non_blocking=True)
        self._keep = (lp, ap)                    # pinned sources stay alive until the copies have run
        if self._ps is not None:
            self._ps._host = None
        self.out = None

    @property
    def ps(self):
        if self._ps is None:
            data_sub, dev, flex, no_tor = self._ps_args
            self._ps = PoseState(data_sub, dev, lig_pos=self.pl.lig_pos, atom_pos=self.pl.atom_pos, flexible_sidechains=flex, no_torsion=no_tor)
            assert (self._ps.T, self._ps.S) == (self.T, self.S)
            self._ps_args = None
        return self._ps

    def _launch(self):
        tr, rot, tor, sc = self.model.launch_plan(self.pl)
        self.out = (tr, rot, tor, sc)
        self.ps.update(self.coef_dev, tr, rot, tor if self.ps.has_tor else None, sc if self.use_sc else None,
                       tr_z=self.z[0], rot_z=self.z[1], tor_z=self.z[2] if self.ps.has_tor else None,
                       sc_z=self.z[3] if self.use_sc else None)

    def stage(self, t4, coef, noise_row=None):
        """Host side of one step: scalars + coefficients + this batch's noise -> one pinned row -> one H2D.
        ``t4``: (t_tr, t_rot, t_tor, t_sc[, t]) -- the fifth entry is the embedding time of the asynchronous noise schedule."""
        pl, b = self.pl, self.b
        row = torch.zeros(pl.n_scal + self.n_extra, dtype=torch.float32).pin_memory()
        ct = {k: torch.full((b,), float(v)) for k, v in zip(('tr', 'rot', 'tor', 'sc_tor', 't'), t4)}
        self.model._host_scalars(pl, ct, out=row[:pl.n_scal])
        row[pl.n_scal:pl.n_scal + 8] = torch.tensor([float(c) for c in coef])
        if noise_row is not None:
            row[pl.n_scal + 8:] = noise_row
        pl.step_in.copy_(row, non_blocking=True)

    def ctx(self):
        """Context that makes this runner's stream current (mini-batches are independent through the whole loop, so
        the sampler puts them on different streams: one mini-batch's graph-building front and pose-update tail, which
        cannot fill the GPU, overlap the other's convolutions)."""
        return torch.cuda.stream(self.stream) if self.stream is not None else contextlib.nullcontext()

    def sync_in(self):
        if self.stream is not None:
            self.stream.wait_stream(torch.cuda.current_stream())

    def sync_out(self):
        if self.stream is not None:
            torch.cuda.current_stream().wait_stream(self.stream)

    def step(self, t4, coef, noise_row=None):
        with self.ctx():
            return self._step(t4, coef, noise_row)

    def _step(self, t4, coef, noise_row):
        self.stage(t4, coef, noise_row)
        self.calls += 1
        if not self.use_graph or self.calls == 1:
            return self._launch()                # first step runs eagerly (lazy kernel attributes, allocator warm-up)
        if self.graph is None:                   # second step: capture (does not execute), then replay from here on
            torch.cuda.synchronize()
            self.graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(self.graph):
                self._launch()
        self.graph.replay()


def sampling(data_list, model, inference_steps, tr_schedule, rot_schedule, tor_schedule, sidechain_tor_schedule, device,
             t_to_sigma, model_args, no_random=False, ode=False, visualization_list=None, sidechain_visualization_list=None,
             confidence_model=None, filtering_data_list=None, filtering_model_args=None, asyncronous_noise_schedule=False,
             t_schedule=None, batch_size=32, no_final_step_noise=False, pivot=None, return_full_trajectory=False,
             svgd_weight=0.0, svgd_repulsive_weight=1.0, svgd_only=False, svgd_rot_rel_weight=1.0, svgd_tor_rel_weight=1.0,
             svgd_sidechain_tor_rel_weight=1.0, temp_sampling=1.0, temp_psi=0.0, temp_sigma_data=0.5,
             flexible_sidechains=None, max_steps=None, trace=None, use_graph=False, concurrent_batches=True,
             loader_seed_draws=True, defer=False):
    """Reference signature and return values (utils/sampling.py:70-286); see the module docstring for what runs where.

    The cyclic garbage collector is paused for the duration of the call (and restored afterwards): the launch loop creates
    no reference cycles, but a generation-2 collection triggered in the middle of it walks every graph / tensor object the
    CALLER keeps alive and stalls the launch stream for 30-90 ms while the GPU idles (measured: 12 consecutive calls take
    270-276 ms each with the collector paused, 270-360 ms with it running)."""
    kw = dict(locals())
    gc_was_enabled = gc.isenabled()
    gc.disable()
    try:
        return _sampling(**kw)
    finally:
        if gc_was_enabled:
            gc.enable()


def _sampling(data_list, model, inference_steps, tr_schedule, rot_schedule, tor_schedule, sidechain_tor_schedule, device,
             t_to_sigma, model_args, no_random=False, ode=False, visualization_list=None, sidechain_visualization_list=None,
             confidence_model=None, filtering_data_list=None, filtering_model_args=None, asyncronous_noise_schedule=False,
             t_schedule=None, batch_size=32, no_final_step_noise=False, pivot=None, return_full_trajectory=False,
             svgd_weight=0.0, svgd_repulsive_weight=1.0, svgd_only=False, svgd_rot_rel_weight=1.0, svgd_tor_rel_weight=1.0,
             svgd_sidechain_tor_rel_weight=1.0, temp_sampling=1.0, temp_psi=0.0, temp_sigma_data=0.5,
             flexible_sidechains=None, max_steps=None, trace=None, use_graph=False, concurrent_batches=True,
             loader_seed_draws=True, defer=False):
    if svgd_weight > 0 or pivot is not None:
        raise NotImplementedError('SVGD / pivot are outside the accelerated path')
    if asyncronous_noise_schedule and t_schedule is None:
        raise ValueError('asyncronous_noise_schedule needs t_schedule (utils/sampling.py:116)')
    flexible_sidechains = model_args.flexible_sidechains if flexible_sidechains is None else flexible_sidechains
    no_sidechains_in_batch = False
    if flexible_sidechains:
        # (graphs without any 'flexResidues' store count as zero flexible atoms; the reference would raise on them)
        has_sc = lambda c: 'flexResidues' in c and 'subcomponents' in c['flexResidues']
        no_sidechains_in_batch = sum(len(c['flexResidues'].subcomponents) for c in data_list if has_sc(c)) == 0
        if no_sidechains_in_batch:
            data_list = copy.deepcopy(data_list)
            for c in data_list:
                if 'flexResidues' in c:
                    del c['flexResidues']
    N = len(data_list)
    ma = model_args
    device = torch.device(device) if not isinstance(device, torch.device) else device
    trajectory, sidechain_trajectory = [], []
    schedules = (tr_schedule, rot_schedule, tor_schedule, sidechain_tor_schedule)

    # one resident plan + pose state (+ optionally a captured step graph) per mini-batch; the plans are built lazily
    # inside step 0 so that the GPU already works on mini-batch k while the host collates mini-batch k + 1
    chunks = [list(range(i, min(i + batch_size, N))) for i in range(0, N, batch_size)]
    use_graph = bool(use_graph) and trace is None
    runners = [None] * len(chunks)
    # accumulation mode of this call's plans (fixed-point sums under torch.use_deterministic_algorithms: bitwise reproducible)
    det = bool(torch.are_deterministic_algorithms_enabled())
    # resident state of an earlier call on the same input (see the module docstring)
    cache_key = cached = full_key = cache_sig = None
    LAST_CALL['plan_reused'] = False
    if PLAN_CACHE_SIZE > 0 and trace is None and filtering_data_list is None and N > 0:
        memo = []                                                     # (tables, key) of the distinct complexes seen so far

        def gkey(g):
            # samples of one complex share (or are deep copies of) the same tables: hash each distinct complex once, the
            # others are compared with it exactly (memcmp speed)
            tabs = _graph_tables(g, flexible_sidechains)
            shape = (tuple(g['ligand'].pos.shape), tuple(g['atom'].pos.shape))
            for tabs2, shape2, key2 in memo:
                if shape2 == shape and _same_tables(tabs, tabs2):
                    return key2
            memo.append((tabs, shape, _graph_key(g, flexible_sidechains)))
            return memo[-1][2]
        def full_key():
            return _cache_key(model, confidence_model, device, batch_size, flexible_sidechains, ma.no_torsion, use_graph,
                              concurrent_batches, det, (gkey(g) for g in data_list))
        # the content key costs ~0.1 ms per graph: on the critical path only when an entry of the same shape signature exists
        # (a possible hit); otherwise it is computed after this call's launches are enqueued, under the GPU work
        cache_sig = (N, tuple((g['ligand'].pos.shape[0], g['atom'].pos.shape[0], g['receptor'].pos.shape[0]) for g in data_list))
        # Retention is adaptive: a run that docks every complex once (the usual inference loop) must not pay for it -- state kept
        # alive delays the re-use of its device memory by the next complex's plans.  The first call of a shape signature only
        # records the signature; from the first repeat on the call's resident state is kept.
        retain = cache_sig in _SEEN_SIGS
        _SEEN_SIGS[cache_sig] = True
        _SEEN_SIGS.move_to_end(cache_sig)
        while len(_SEEN_SIGS) > 64:
            _SEEN_SIGS.popitem(last=False)
        if not retain:
            full_key = None
        if retain and any(e['sig'] == cache_sig for e in _PLAN_CACHE.values()):
            cache_key = full_key()
            cached = _cache_get(cache_key, model, confidence_model, det)
    # independent mini-batches alternate between two streams (see StepRunner.ctx); host-visible intermediates
    # (trace, trajectories, visualisation) keep the single-stream order
    single = len(chunks) < 2 or trace is not None or return_full_trajectory or visualization_list is not None \
        or sidechain_visualization_list is not None or not concurrent_batches
    if cached is not None and cached['single'] != single:
        cached = None
    streams = [None] if single else [torch.cuda.Stream(device=device) for _ in range(2)]
    if cached is not None:
        cached['busy'] = True
        _PLAN_CACHE.move_to_end(cache_key)
        runners, streams = list(cached['runners']), cached['streams']
        for idx, r in zip(chunks, runners):
            r.reset([data_list[i] for i in idx])
            r.sync_in()                                               # the start poses were uploaded on the caller's stream
        LAST_CALL['plan_reused'] = True
    n_tor = [0 if ma.no_torsion else sum(int(data_list[i]['ligand'].edge_mask.sum()) for i in idx) for idx in chunks]
    n_sc = [sum(int(data_list[i]['flexResidues'].edge_idx.shape[0]) for i in idx
                if flexible_sidechains and 'flexResidues' in data_list[i] and 'edge_idx' in data_list[i]['flexResidues'])
            for idx in chunks]
    T_tot, S_tot = sum(n_tor), sum(n_sc)
    n_steps = inference_steps if max_steps is None else min(max_steps, inference_steps)
    M = 6 * N + T_tot + S_tot
    # Noise for all steps is drawn up front, in the reference's order (per step: tr_z, rot_z, tor_z,
    # sidechain_tor_z; utils/sampling.py:136-163) -- nothing else consumes the CPU generator in between, so the
    # stream is identical; each step's slice travels to the device inside that step's single H2D copy.
    # The reference also builds a torch DataLoader every step (utils/sampling.py:100) whose iterator draws its
    # ``_base_seed`` (one int64 ``random_()``) from the same default generator before the step's noise; the draw is
    # repeated here so that a seeded run consumes the identical stream (``loader_seed_draws=False`` skips it).
    noise_host = torch.zeros(max(n_steps, 1), M)
    for t_idx in range(n_steps):
        if loader_seed_draws:
            torch.empty((), dtype=torch.int64).random_()
        if not ode:
            zero_noise = no_random or (no_final_step_noise and t_idx == inference_steps - 1)
            draw = (lambda shape: torch.zeros(shape)) if zero_noise else (lambda shape: torch.normal(mean=0, std=1, size=shape))
            noise_host[t_idx, :3 * N] = draw((N, 3)).reshape(-1)
            noise_host[t_idx, 3 * N:6 * N] = draw((N, 3)).reshape(-1)
            if not ma.no_torsion:
                noise_host[t_idx, 6 * N:6 * N + T_tot] = draw((T_tot,))
            if flexible_sidechains:
                noise_host[t_idx, 6 * N + T_tot:] = draw((S_tot,))
    if loader_seed_draws and confidence_model is not None and n_steps == inference_steps:
        for _ in range(2):                                            # the two loaders of utils/sampling.py:265-266
            torch.empty((), dtype=torch.int64).random_()

    conf_plans = cached['conf_plans'] if cached is not None else None
    max_ahead = int(os.environ.get('DDP_MAX_AHEAD', 2))
    pace = [[] for _ in chunks]

    def conf_plan(idx):
        sub = [(filtering_data_list if filtering_data_list is not None else data_list)[i] for i in idx]
        return confidence_model.make_plan(Batch.from_data_list(sub, skip=STATIC_KEYS), graphs=sub)

    def write_back_all():
        for idx, r in zip(chunks, runners):
            if r is not None:
                r.ps.write_back([data_list[i] for i in idx])

    with torch.no_grad():
        for t_idx in range(n_steps):
            t, coef = step_coefficients(t_idx, inference_steps, schedules, t_to_sigma, ma, ode, temp_sampling, temp_psi,
                                        temp_sigma_data, flexible_sidechains)
            if asyncronous_noise_schedule:
                t = list(t) + [t_schedule[t_idx]]                     # embedding time (set_time's `t`, utils/sampling.py:116)
            if return_full_trajectory:
                write_back_all()
                trajectory.append(np.asarray([g['ligand'].pos.cpu().numpy() for g in data_list]))
                sidechain_trajectory.append(np.asarray([]) if no_sidechains_in_batch or not flexible_sidechains else np.asarray(
                    [g['atom'].pos.cpu().numpy()[g['flexResidues'].subcomponents.unique().cpu().numpy()] for g in data_list]))
            z = noise_host[t_idx]
            s0 = t0 = c0 = 0
            step_scores = []
            for k, idx in enumerate(chunks):
                if runners[k] is None:
                    runners[k] = StepRunner(model, [data_list[i] for i in idx], flexible_sidechains, ma.no_torsion, use_graph=use_graph,
                                            stream=streams[k % len(streams)])
                    assert (runners[k].T, runners[k].S) == (n_tor[k], n_sc[k])
                    runners[k].sync_in()                              # plan + pose state were uploaded on the caller's stream
                r = runners[k]
                b = len(idx)
                row = torch.cat([z[3 * s0:3 * (s0 + b)], z[3 * N + 3 * s0:3 * N + 3 * (s0 + b)], z[6 * N + t0:6 * N + t0 + r.T],
                                 z[6 * N + T_tot + c0:6 * N + T_tot + c0 + r.S]])
                r.step(t, coef, row)
                if trace is not None:
                    step_scores.append(tuple(o.clone() for o in r.out))
                s0, t0, c0 = s0 + b, t0 + r.T, c0 + r.S
                if max_ahead > 0 and len(streams) > 1:
                    # concurrent mini-batches: keep the host at most ``max_ahead`` steps in front of each stream, so that the
                    # two streams advance in step (one's small kernels under the other's convolutions) instead of one
                    # stream racing through its queue first
                    ev = torch.cuda.Event()
                    ev.record(r.stream)
                    pace[k].append(ev)
                    if len(pace[k]) > max_ahead:
                        pace[k].pop(0).synchronize()
            if trace is not None:
                trace.append(tuple(torch.cat([s[k] for s in step_scores]).cpu() for k in range(4)))
            if conf_plans is None and confidence_model is not None:
                # confidence plans (static tensors, workspaces) are collated and uploaded while the GPU runs step 0;
                # the final poses reach them by device-to-device copies after the last step
                conf_plans = [conf_plan(idx) for idx in chunks]
            if visualization_list is not None or sidechain_visualization_list is not None:
                write_back_all()
                if visualization_list is not None:
                    for i, v in enumerate(visualization_list):
                        v.add((data_list[i]['ligand'].pos + data_list[i].original_center).detach().cpu(), part=1, order=t_idx + 2)
                if sidechain_visualization_list is not None:
                    for i, v in enumerate(sidechain_visualization_list):
                        v.append(data_list[i]['atom'].pos + data_list[i]['original_center'])

        confidence = None
        if confidence_model is not None:                              # utils/sampling.py:263-281
            if conf_plans is None:                                    # n_steps == 0
                conf_plans = [conf_plan(idx) for idx in chunks]
            conf = []
            cur = torch.cuda.current_stream()
            for idx, r, cpl in zip(chunks, runners, conf_plans):
                zt = torch.zeros(len(idx))
                if r is None:
                    conf.append(confidence_model.run_plan(cpl, {'tr': zt, 'rot': zt, 'tor': zt, 'sc_tor': zt, 't': zt}).clone())
                    continue
                r.sync_in()                                           # the confidence plans were uploaded on the caller's stream
                with r.ctx():
                    cpl.lig_pos.copy_(r.pl.lig_pos)
                    if filtering_data_list is None:                   # filtering graphs keep their own receptor atoms
                        cpl.atom_pos.copy_(r.pl.atom_pos)
                    conf.append(confidence_model.run_plan(cpl, {'tr': zt, 'rot': zt, 'tor': zt, 'sc_tor': zt, 't': zt}).clone())
                    conf[-1].record_stream(cur)
            for r in runners:
                if r is not None:
                    r.sync_out()
            confidence = torch.cat(conf, dim=0)
        for r in runners:
            if r is not None:
                r.sync_out()
        staged = None
        if defer:
            # asynchronous device->host copies into pinned buffers + one event: finish() waits for THIS call's work only,
            # not for whatever the caller has enqueued behind it in the meantime
            for r in runners:
                if r is not None:
                    r.ps.stage_to_host()
            conf_host = None
            if confidence is not None:
                conf_host = torch.empty(confidence.shape, dtype=confidence.dtype, pin_memory=True)
                conf_host.copy_(confidence, non_blocking=True)
            status_host = None
            if det:                                                   # the status word travels with the results
                status_host = torch.empty(1, dtype=torch.int32, pin_memory=True)
                status_host.copy_(_lib.status_word(device), non_blocking=True)
            staged = (torch.cuda.Event(), conf_host, status_host)
            staged[0].record()

    if full_key is not None and cache_key is None and n_steps > 0:
        cache_key = full_key()                                        # (everything is enqueued: this overlaps the GPU work)

    def finish():
        nonlocal confidence
        if staged is not None:
            staged[0].synchronize()
            confidence = staged[1]
        write_back_all()                                              # the one device->host read of the poses
        if det:                                                       # fixed-point range / NaN errors of the whole call
            _lib.check_status(device, None if staged is None else int(staged[2][0]))
        if cache_key is not None and all(r is not None for r in runners) and n_steps > 0:
            # hand the resident state to the cache (or back to it): the next call on this input starts from here
            import weakref
            _PLAN_CACHE[cache_key] = {'runners': runners, 'conf_plans': conf_plans, 'streams': streams, 'single': single, 'busy': False, 'sig': cache_sig,
                                      'deterministic': det,
                                      'models': (weakref.ref(model), weakref.ref(confidence_model) if confidence_model is not None else None)}
            _PLAN_CACHE.move_to_end(cache_key)
            while len(_PLAN_CACHE) > PLAN_CACHE_SIZE:
                _PLAN_CACHE.popitem(last=False)
        if filtering_data_list is not None:
            for i, g in enumerate(filtering_data_list):
                g['ligand'].pos = data_list[i]['ligand'].pos
        if return_full_trajectory:
            return data_list, confidence, trajectory, sidechain_trajectory
        return data_list, confidence
    if defer:
        # everything is enqueued; nothing has been waited for.  The caller overlaps its next complex's host work (graph
        # copies, randomize_position, collation, plan upload) with this one's GPU work and calls finish() later.
        return finish
    return finish()
