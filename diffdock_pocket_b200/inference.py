"""Host mirror of the docking driver in ``inference.py`` (boundary only: no RDKit / Biopython file I/O).

``infer_single_complex`` follows inference.py:106-291 up to the ranking step (:135 copy the complex graph
``samples_per_complex`` times, :140 ``randomize_position``, :177 ``sampling``, :198-219 gather poses in the original
frame and sort by confidence, descending); the ranked SDF / PDB files (:221-240) are written by ``writer.AsyncWriter``
(text-level, on worker threads) when the rows carry the template files' lines; relaxation (:242-262) stays with the
reference's OpenMM code.  ``infer_multiple_complexes`` is the per-device loop (:294-304) with
the reference's per-complex failure isolation (:282-287: a failing complex is reported and skipped).

Multi-GPU: the reference splits the complex table with ``np.array_split`` over a spawn pool (inference.py:466-488).
``infer_sharded`` does the same split over ``torch.distributed`` ranks (one process per GPU) and adds the path's single
collective: an all-gather of every complex's best confidence so that all ranks hold the global ranking
(virtual-screening use, BASELINE.json configs[4]).
"""
import copy
import os
import traceback
from argparse import Namespace
from functools import partial

import numpy as np
import torch
import torch.distributed as dist

from .diffusion_utils import get_t_schedule, t_to_sigma as t_to_sigma_compl
from .parallel import shard_range
from .posecheck import check_poses
from .hetero import sample_copies
from .sampling import randomize_position, sampling


def default_args(**over):
    """Sampler flags of inference.py's parser (:49-103) that reach the hot path."""
    a = dict(samples_per_complex=10, batch_size=32, inference_steps=30, actual_steps=None, no_random=False, ode=False,
             no_final_step_noise=False, rigid=False, inf_sched_alpha=1.0, inf_sched_beta=1.0,
             temp_sampling_tr=0.9766350103728372, temp_psi_tr=1.5102572175711826,
             temp_sampling_rot=6.077432837220868, temp_psi_rot=0.8141168207563049,
             temp_sampling_tor=6.761568162335063, temp_psi_tor=0.7661845361370018,
             temp_sampling_sc_tor=1.4487910576602347, temp_psi_sc_tor=1.339614553802453,
             temp_sigma_data=0.48884149503636976)
    a.update(over)
    return Namespace(**a)


def infer_single_complex(idx, protein_ligand_info_row, model, args, score_model_args, filtering_args=None,
                         filtering_model=None, filtering_model_args=None, filtering_complex_dict=None, t_schedule=None,
                         tr_schedule=None, device=None, defer=False, writer=None, out_dir=None, pose_checks=False):
    """-> dict(name, ligand_pos [spc, N_l, 3], atom_pos [spc, N_a, 3], confidence [spc] or None), poses in the original
    frame and sorted by confidence (descending); ``None`` if the complex failed (the reference returns 0 and goes on).
    ``pose_checks=True`` adds ``checks``: ``posecheck.check_poses`` of the ranked poses (clash counts and minimum ratios,
    and ``rmsd`` / ``sc_rmsd`` against the row's ``ref_ligand_pos`` / ``ref_atom_pos``, original frame, when it has them;
    see ``_pose_checks`` for how a failing check is reported without touching the poses).
    ``defer=True`` returns a zero-argument callable producing that result instead: all GPU work is enqueued, nothing has
    been waited for, so the caller can prepare the next complex meanwhile (``infer_multiple_complexes`` does)."""
    orig = protein_ligand_info_row['complex_graph']
    spc = args.samples_per_complex
    t_to_sigma = partial(t_to_sigma_compl, args=score_model_args)
    flex = False if args.rigid else score_model_args.flexible_sidechains

    def failed(e):                                                  # inference.py:282-287
        print('Failed on', getattr(orig, 'name', idx), e)
        traceback.print_exc()
        return None
    try:
        # inference.py:135 deep-copies the graph per sample; here the samples share the static tensors of the complex
        # (features, receptor graph) and own only the coordinates the sampler moves
        data_list = sample_copies(orig, spc)
        randomize_position(data_list, score_model_args.no_torsion, args.no_random, score_model_args.tr_sigma_max,
                           flexible_sidechains=flex)
        filtering_data_list = None
        if filtering_model is not None and filtering_complex_dict is not None and not (
                getattr(filtering_args, 'use_original_model_cache', True) or getattr(filtering_args, 'transfer_weights', False)):
            filtering_data_list = sample_copies(filtering_complex_dict[orig.name], spc)
        steps = args.actual_steps if args.actual_steps is not None else args.inference_steps
        pending = sampling(
            data_list=data_list, model=model, inference_steps=steps, tr_schedule=tr_schedule, rot_schedule=tr_schedule,
            tor_schedule=tr_schedule, sidechain_tor_schedule=tr_schedule, t_schedule=t_schedule, t_to_sigma=t_to_sigma,
            model_args=score_model_args, confidence_model=filtering_model, device=device, no_random=args.no_random,
            ode=args.ode, filtering_data_list=filtering_data_list, filtering_model_args=filtering_model_args,
            asyncronous_noise_schedule=getattr(score_model_args, 'asyncronous_noise_schedule', False),
            batch_size=args.batch_size, no_final_step_noise=args.no_final_step_noise,
            temp_sampling=[args.temp_sampling_tr, args.temp_sampling_rot, args.temp_sampling_tor, args.temp_sampling_sc_tor],
            temp_psi=[args.temp_psi_tr, args.temp_psi_rot, args.temp_psi_tor, args.temp_psi_sc_tor],
            flexible_sidechains=flex, defer=True)     # reference quirk kept: --temp_sigma_data is parsed (:101) but never
        #                                               passed to sampling() (:177-196), so its default 0.5 applies
    except Exception as e:
        failed(e)
        return (lambda: None) if defer else None

    def finish():
        try:
            graphs, confidence = pending()
            res = _rank(orig, idx, graphs, confidence)              # inference.py:198-219
            _submit_write(writer, out_dir, protein_ligand_info_row, res, flex)
        except Exception as e:
            return failed(e)
        if pose_checks:
            _pose_checks([(protein_ligand_info_row, res)])
        return res
    return finish if defer else finish()


def _submit_write(writer, out_dir, row, res, flex):
    """inference.py:221-240 handed to ``writer.AsyncWriter`` (rows carry the template files' lines: 'ligand_sdf_lines' and,
    for flexible side chains, 'protein_pdb_lines'); the files are written while the next complex is docked."""
    if writer is None or res is None or 'ligand_sdf_lines' not in row:
        return
    g = row['complex_graph']
    fr = g['flexResidues'] if flex and 'flexResidues' in g and 'edge_idx' in g['flexResidues'] else None
    writer.submit(os.path.join(out_dir or '.', str(res['name'])), res, row['ligand_sdf_lines'],
                  row.get('protein_pdb_lines') if fr is not None else None, fr)


_CHECK_STREAMS = {}


def _pose_checks(items):
    """One ``check_poses`` call over the ranked poses of [(row, result), ...] (results of failed complexes skipped); adds
    ``result['checks']``.  The checks are a diagnostic: they never change or drop a docking result.  A ligand above the
    automorphism cap gets checks without RMSD (``rmsd_error``); any other failure is reported as ``checks = {'error': msg}``.
    They run on a side stream of their own, from the host copies of the ranked poses, so that they do not wait for the
    sampler work the pipeline of ``infer_multiple_complexes`` has already enqueued behind them."""
    items = [(row, res) for row, res in items if res is not None]
    if not items:
        return
    dev = torch.cuda.current_device()
    if dev not in _CHECK_STREAMS:
        _CHECK_STREAMS[dev] = torch.cuda.Stream(dev)
    try:
        with torch.cuda.stream(_CHECK_STREAMS[dev]):
            out = check_poses([row['complex_graph'] for row, _ in items], [res['ligand_pos'] for _, res in items],
                              [res['atom_pos'] for _, res in items], [row.get('ref_ligand_pos') for row, _ in items],
                              [row.get('ref_atom_pos') for row, _ in items], strict=False)
    except Exception as e:
        print('Pose checks failed for', [getattr(row['complex_graph'], 'name', None) for row, _ in items], e)
        out = [{'error': str(e)}] * len(items)
    for (_, res), checks in zip(items, out):
        res['checks'] = checks


def _rank(orig, idx, graphs, confidence):
    center = np.asarray(orig.original_center.cpu().numpy() if torch.is_tensor(orig.original_center) else orig.original_center)
    ligand_pos = np.asarray([g['ligand'].pos.cpu().numpy() + center for g in graphs])
    atom_pos = np.asarray([g['atom'].pos.cpu().numpy() + center for g in graphs])
    if confidence is not None:
        if confidence.dim() == 2:
            confidence = confidence[:, 0]
        confidence = confidence.cpu().numpy()
        order = np.argsort(confidence)[::-1]
        confidence, ligand_pos, atom_pos = confidence[order], ligand_pos[order], atom_pos[order]
    return dict(name=orig.name, index=idx, ligand_pos=ligand_pos, atom_pos=atom_pos, confidence=confidence)


def infer_complex_group(group, model, args, score_model_args, filtering_model=None, filtering_model_args=None,
                        tr_schedule=None, t_schedule=None, device=None, defer=False, writer=None, out_dir=None, pose_checks=False):
    """Cross-complex batching (SURVEY.md 8(f)-1; the reference's sampler assumes one complex per call, F9): the samples
    of several complexes share one ``sampling()`` call, so that small ``samples_per_complex`` still fill the mini-batch
    (virtual screening).  ``group``: [(idx, row), ...].  Falls back to one call per complex if the joint call fails.
    ``defer`` and ``pose_checks`` as in ``infer_single_complex`` (the callable returns the list of per-complex results; the
    checks of the whole group run as one ``check_poses`` call)."""
    spc = args.samples_per_complex
    flex = False if args.rigid else score_model_args.flexible_sidechains

    def one_by_one(e):
        print('Joint call failed for', [row['complex_graph'].name for _, row in group], e, '- retrying one complex at a time')
        return [infer_single_complex(idx, row, model, args, score_model_args, filtering_model=filtering_model,
                                     filtering_model_args=filtering_model_args, tr_schedule=tr_schedule, t_schedule=t_schedule,
                                     device=device, writer=writer, out_dir=out_dir, pose_checks=pose_checks) for idx, row in group]
    try:
        data_list = []
        for _, row in group:
            dl = sample_copies(row['complex_graph'], spc)
            randomize_position(dl, score_model_args.no_torsion, args.no_random, score_model_args.tr_sigma_max, flexible_sidechains=flex)
            data_list += dl
        steps = args.actual_steps if args.actual_steps is not None else args.inference_steps
        pending = sampling(
            data_list=data_list, model=model, inference_steps=steps, tr_schedule=tr_schedule, rot_schedule=tr_schedule,
            tor_schedule=tr_schedule, sidechain_tor_schedule=tr_schedule, t_schedule=t_schedule,
            t_to_sigma=partial(t_to_sigma_compl, args=score_model_args), model_args=score_model_args,
            confidence_model=filtering_model, device=device, no_random=args.no_random, ode=args.ode,
            filtering_model_args=filtering_model_args, batch_size=args.batch_size, no_final_step_noise=args.no_final_step_noise,
            temp_sampling=[args.temp_sampling_tr, args.temp_sampling_rot, args.temp_sampling_tor, args.temp_sampling_sc_tor],
            temp_psi=[args.temp_psi_tr, args.temp_psi_rot, args.temp_psi_tor, args.temp_psi_sc_tor], flexible_sidechains=flex,
            defer=True)
    except Exception as e:
        res = one_by_one(e)
        return (lambda: res) if defer else res

    def finish():
        try:
            graphs, confidence = pending()
            out = [_rank(row['complex_graph'], idx, graphs[k * spc:(k + 1) * spc],
                         confidence[k * spc:(k + 1) * spc] if confidence is not None else None) for k, (idx, row) in enumerate(group)]
            for (idx, row), res in zip(group, out):
                _submit_write(writer, out_dir, row, res, flex)
        except Exception as e:
            return one_by_one(e)
        if pose_checks:
            _pose_checks([(row, res) for (_, row), res in zip(group, out)])
        return out
    return finish if defer else finish()


def infer_multiple_complexes(rows, *a, batch_complexes=False, pipeline=True, **kw):
    """inference.py:294-304 over a list of (idx, row) (rows: dicts with 'complex_graph'); -> (results, count_succeeded).
    ``batch_complexes``: pack floor(batch_size / samples_per_complex) complexes into each sampler call.
    ``pose_checks``, like the other keyword arguments, is passed to every call.
    ``pipeline``: software pipeline of depth 2 -- the host prepares and enqueues call k + 1 (graph copies,
    ``randomize_position``, collation, plan upload, kernel launches) while the GPU still runs call k, and only then
    collects call k's poses; without it the GPU idles during every complex's host work (the reference's loop is serial)."""
    args = a[1] if len(a) > 1 else kw['args']
    per_call = max(1, args.batch_size // args.samples_per_complex) if batch_complexes else 1
    if per_call == 1:
        launch = lambda item: infer_single_complex(item[0], item[1], *a, defer=True, **kw)
        items, wrap = list(rows), (lambda r: [r])
    else:
        model, score_model_args = (a[0] if a else kw['model']), (a[2] if len(a) > 2 else kw['score_model_args'])
        passthrough = {k: kw[k] for k in ('filtering_model', 'filtering_model_args', 'tr_schedule', 't_schedule', 'device', 'writer', 'out_dir',
                                          'pose_checks') if k in kw}
        launch = lambda grp: infer_complex_group(grp, model, args, score_model_args, defer=True, **passthrough)
        items, wrap = [rows[j:j + per_call] for j in range(0, len(rows), per_call)], (lambda r: r)
    results, pending = [], None
    for item in items:
        fin = launch(item)
        if not pipeline:
            results += wrap(fin())
            continue
        if pending is not None:
            results += wrap(pending())
        pending = fin
    if pending is not None:
        results += wrap(pending())
    return results, sum(r is not None for r in results)


def infer_sharded(rows, model, args, score_model_args, device, filtering_model=None, filtering_model_args=None, group=None,
                  batch_complexes=False, pipeline=True, pose_checks=False):
    """Complexes split over the ranks like ``np.array_split`` (inference.py:468); every rank docks its shard with no
    communication; one all-gather of (complex index, best confidence) at the end -> global ranking on every rank.
    ``pose_checks`` as in ``infer_single_complex`` (each rank checks its own shard)."""
    world = dist.get_world_size(group) if dist.is_initialized() else 1
    rank = dist.get_rank(group) if dist.is_initialized() else 0
    lo, hi = shard_range(len(rows), rank, world)
    sched = get_t_schedule('expbeta', args.inference_steps, inf_sched_alpha=args.inf_sched_alpha, inf_sched_beta=args.inf_sched_beta)   # inference.py:457-459
    local, ok = infer_multiple_complexes([(i, rows[i]) for i in range(lo, hi)], model, args, score_model_args,
                                         filtering_model=filtering_model, filtering_model_args=filtering_model_args,
                                         tr_schedule=sched, device=device, batch_complexes=batch_complexes, pipeline=pipeline,
                                         pose_checks=pose_checks)
    # the single collective of the path: all-gather of the shards' best confidences (padded to the largest shard)
    width = -(-len(rows) // world) if len(rows) else 1
    mine = torch.full((width,), float('-inf'), device=device)
    for r in local:
        if r is not None and r['confidence'] is not None:
            mine[r['index'] - lo] = float(r['confidence'][0])
    if world > 1:
        parts = [torch.empty_like(mine) for _ in range(world)]
        dist.all_gather(parts, mine, group=group)
    else:
        parts = [mine]
    best = torch.cat([parts[r][:shard_range(len(rows), r, world)[1] - shard_range(len(rows), r, world)[0]] for r in range(world)])
    return local, best.cpu(), ok
