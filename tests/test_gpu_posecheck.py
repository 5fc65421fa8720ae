"""Pose checks on the device (``ddp_pose_rmsd``, ``ddp_clash_screen`` through ``posecheck.check_poses``) against a float64
oracle kept in this file: symmetry-corrected ligand RMSD and side-chain RMSD within 1 fp32 ulp, clash counts equal
outside a 1e-5 relative band around the threshold (pairs inside it are ambiguous in fp32), minimum ratios within 1e-6
relative.  Also: the 3dpf anchors, symmetry, bitwise reproducibility and packing independence, and the opt-in
``pose_checks`` of the inference driver."""
import numpy as np
import pytest
import torch
from networkx.algorithms.isomorphism import GraphMatcher
import networkx as nx

import _common as T
from diffdock_pocket_b200 import _lib, diffusion_utils as du, inference, inputs, posecheck as pc

pytestmark = pytest.mark.gpu
DEV = torch.device('cuda:0')
SETS = ('ligand_pocket', 'sidechain_pocket', 'ligand_internal')
AMBIGUOUS = 1e-5


# ------------------------------------------------------------------------------------------------ float64 oracle
def _oracle_tables(g, with_autos=True):
    xl = g['ligand'].x[:, 0].numpy()
    ei = g['ligand', 'ligand'].edge_index.numpy()
    G = nx.Graph()
    G.add_nodes_from((i, {'z': int(z)}) for i, z in enumerate(xl))
    G.add_edges_from(zip(ei[0].tolist(), ei[1].tolist()))
    autos = [np.array([m[i] for i in range(len(xl))]) for m in
             GraphMatcher(G, G, node_match=lambda a, b: a['z'] == b['z']).isomorphisms_iter()] if with_autos else None
    sp = dict(nx.all_pairs_shortest_path_length(G))
    n = len(xl)
    far = np.array([[j > i and sp[i].get(j, np.inf) >= 4 for j in range(n)] for i in range(n)])
    own = np.full(g['atom'].pos.shape[0], -1)
    aei = g['atom', 'receptor'].edge_index.numpy()
    own[aei[0]] = aei[1]
    moved = None
    if 'flexResidues' in g and g['flexResidues'].subcomponents.numel():
        moved = np.unique(g['flexResidues'].subcomponents.numpy())
    return autos, far, own, moved


def oracle(g, lig, atoms, ref_l=None, ref_a=None, ratio=0.75):
    """-> dict per check: (clear count, ambiguous count) per set and pose, min ratio per set and pose, rmsd, sc_rmsd."""
    autos, far, own, moved = _oracle_tables(g, with_autos=ref_l is not None)
    lig = np.asarray(lig, np.float32).astype(np.float64)
    atoms = np.asarray(atoms, np.float32).astype(np.float64)
    rl = pc.RADIUS_TABLE[g['ligand'].x[:, 0].numpy()].astype(np.float64)
    ra = pc.RADIUS_TABLE[g['atom'].x[:, 1].numpy()].astype(np.float64)
    inp = g['atom'].pos.numpy().astype(np.float64)
    out = {k: [] for k in ('clear', 'amb', 'min')}
    for s in range(lig.shape[0]):
        sets = [(np.linalg.norm(lig[s][:, None] - atoms[s][None], axis=-1), rl[:, None] + ra[None], None)]
        if moved is not None:
            d = np.linalg.norm(atoms[s][moved][:, None] - atoms[s][None], axis=-1)
            keep = (own[moved][:, None] != own[None]) & (np.linalg.norm(inp[moved][:, None] - inp[None], axis=-1) >= pc.BONDED_CUTOFF)
            sets.append((d, ra[moved][:, None] + ra[None], keep))
        else:
            sets.append((np.zeros((0, 0)), np.ones((0, 0)), None))
        sets.append((np.linalg.norm(lig[s][:, None] - lig[s][None], axis=-1), rl[:, None] + rl[None], far))
        clear, amb, mn = [], [], []
        for d, sm, keep in sets:
            if keep is not None:
                d, sm = d[keep], sm[keep]
            thr = ratio * sm
            a = np.abs(d - thr) <= AMBIGUOUS * thr
            clear.append(int(((d < thr) & ~a).sum()))
            amb.append(int(a.sum()))
            mn.append(float((d / sm).min()) if d.size else np.inf)
        out['clear'].append(clear)
        out['amb'].append(amb)
        out['min'].append(mn)
    out = {k: np.array(v) for k, v in out.items()}
    if ref_l is not None:
        r = np.asarray(ref_l, np.float32).astype(np.float64)
        out['rmsd'] = np.array([min(np.sqrt(((lig[s] - r[p]) ** 2).sum(-1).mean()) for p in autos) for s in range(lig.shape[0])])
    if ref_a is not None:
        r = np.asarray(ref_a, np.float32).astype(np.float64)
        out['sc_rmsd'] = None if moved is None else \
            np.array([np.sqrt(((atoms[s][moved] - r[moved]) ** 2).sum(-1).mean()) for s in range(lig.shape[0])])
    return out


def _ulp_close(got, ref):
    r32 = np.float32(ref)
    return np.abs(got.astype(np.float64) - r32.astype(np.float64)) <= np.spacing(np.abs(r32)).astype(np.float64)


def assert_matches(got, ref, what):
    for k, name in enumerate(SETS):
        cnt = got[name + '_clashes']
        lo, hi = ref['clear'][:, k], ref['clear'][:, k] + ref['amb'][:, k]
        assert ((lo <= cnt) & (cnt <= hi)).all(), (what, name, cnt, lo, hi)
        mg, mr = got[name + '_min_ratio'].astype(np.float64), ref['min'][:, k]
        inf = np.isinf(mr)
        assert (np.isinf(mg) == inf).all(), (what, name, mg, mr)
        assert (np.abs(mg[~inf] - mr[~inf]) <= 1e-6 * mr[~inf]).all(), (what, name, np.abs(mg - mr) / mr)
    for key in ('rmsd', 'sc_rmsd'):
        if key in ref:
            if ref[key] is None:
                assert got[key] is None, what
            else:
                assert got[key].dtype == np.float32 and _ulp_close(got[key], ref[key]).all(), (what, key, got[key], ref[key])
        else:
            assert key not in got, (what, key)


# ------------------------------------------------------------------------------------------------ poses
def _rot(axis, theta):
    axis = axis / np.linalg.norm(axis)
    K = np.array([[0, -axis[2], axis[1]], [axis[2], 0, -axis[0]], [-axis[1], axis[0], 0]])
    return np.eye(3) + np.sin(theta) * K + (1 - np.cos(theta)) * K @ K


def poses(g, S, seed, rigid=1.0, torsion=1.0, sidechain=1.0):
    """S perturbed copies of the input ligand and pocket: pose 0 unperturbed; then random rigid moves (rotation about the
    centroid, translation in A), torsion rotations of the rotatable bonds, side-chain torsions of the flexible residues."""
    rng = np.random.RandomState(seed)
    lig0, at0 = g['ligand'].pos.numpy().astype(np.float64), g['atom'].pos.numpy().astype(np.float64)
    ei = g['ligand', 'ligand'].edge_index.numpy().T[np.asarray(g['ligand'].edge_mask, bool)]
    mr = np.asarray(g['ligand'].mask_rotate, bool)
    fr = g['flexResidues'] if 'flexResidues' in g and 'edge_idx' in g['flexResidues'] else None
    L, A = [lig0.copy()], [at0.copy()]
    for _ in range(S - 1):
        l, a = lig0.copy(), at0.copy()
        for (u, v), m in zip(ei, mr):
            if torsion:
                l[m] = (l[m] - l[v]) @ _rot(l[u] - l[v], rng.uniform(-np.pi, np.pi) * torsion).T + l[v]
        if rigid:
            c = l.mean(0)
            l = (l - c) @ _rot(rng.randn(3), rng.uniform(0, np.pi) * rigid).T + c + rng.randn(3) * rigid
        if fr is not None and sidechain:
            sub, mp = fr.subcomponents.numpy(), fr.subcomponentsMapping.numpy()
            for (u, v), (s0, s1) in zip(fr.edge_idx.numpy(), mp):
                idx = sub[s0:s1]
                a[idx] = (a[idx] - a[v]) @ _rot(a[u] - a[v], rng.uniform(-np.pi, np.pi) * sidechain).T + a[v]
        L.append(l)
        A.append(a)
    return np.asarray(L, np.float32), np.asarray(A, np.float32)


def _synthetic(n_lig, seed):
    g = inputs.synthetic_complex(seed, n_lig=n_lig, n_res=40, flexible_residues=3)
    if n_lig > 150:           # random elements: a 512-atom tree of three elements has far more automorphisms than the cap
        g['ligand'].x = g['ligand'].x.clone()
        g['ligand'].x[:, 0] = torch.from_numpy(np.random.RandomState(seed).choice([5, 6, 7, 8, 14, 15, 16, 33, 34, 52, 118], n_lig))
    return g


def _ref(g):
    return g['ligand'].pos.numpy(), g['atom'].pos.numpy()


def _case(name):
    if name.startswith('3dpf'):
        return T.graph(name)
    return _synthetic(int(name[3:]), {'lig7': 1, 'lig29': 2, 'lig147': 3, 'lig512': 4}[name])


# ------------------------------------------------------------------------------------------------ tests
@pytest.mark.parametrize('name', ['3dpf_holo', '3dpf_apo', 'lig7', 'lig29', 'lig147', 'lig512'])
@pytest.mark.parametrize('kind', ['rigid', 'torsion', 'all'])
def test_oracle_agreement(name, kind):
    g = _case(name)
    S = 40 if kind == 'all' else 8
    lig, at = poses(g, S, seed=sum(map(ord, name + kind)), rigid=1.0 if kind != 'torsion' else 0,
                    torsion=1.0 if kind != 'rigid' else 0, sidechain=1.0 if kind == 'all' else 0)
    rl, ra = _ref(g)
    got = pc.check_poses([g], [lig], [at], [rl], [ra])[0]
    assert_matches(got, oracle(g, lig, at, rl, ra), (name, kind))
    assert (got['rmsd'][0] == 0) and (got['sc_rmsd'][0] == 0)


@pytest.mark.parametrize('ratio', [0.5, 1.0])
def test_ratio_and_device_inputs(ratio):
    """Other ratios; CUDA tensors in, pocket taken from the graph when atom_pos is None, no references -> no RMSD keys."""
    g = T.graph('3dpf_apo')
    lig, at = poses(g, 6, seed=3, sidechain=0)
    got = pc.check_poses([g], [torch.from_numpy(lig).to(DEV)], ratio=ratio)[0]
    assert 'rmsd' not in got and 'sc_rmsd' not in got
    assert_matches(got, oracle(g, lig, at, ratio=ratio), ratio)


def test_rigid_complex_has_no_sidechain_set():
    g = inputs.synthetic_complex(5, n_lig=20, n_res=30, flexible_residues=0)
    lig, at = poses(g, 4, seed=1)
    rl, ra = _ref(g)
    got = pc.check_poses([g], [lig], [at], [rl], [ra])[0]
    assert got['sc_rmsd'] is None
    assert (got['sidechain_pocket_clashes'] == 0).all() and np.isinf(got['sidechain_pocket_min_ratio']).all()
    assert_matches(got, oracle(g, lig, at, rl, ra), 'rigid')


def test_anchors_3dpf():
    holo, apo = T.graph('3dpf_holo'), T.graph('3dpf_apo')
    rl = holo['ligand'].pos.numpy()[None]
    h, a = pc.check_poses([holo, apo], [rl, apo['ligand'].pos.numpy()[None]], None, [rl[0], apo['ligand'].pos.numpy()])
    assert h['rmsd'][0] == 0 and a['rmsd'][0] == 0
    assert h['ligand_pocket_clashes'][0] == 0 and a['ligand_pocket_clashes'][0] == 57
    assert abs(h['ligand_pocket_min_ratio'][0] - 0.881) < 5e-4 and abs(a['ligand_pocket_min_ratio'][0] - 0.154) < 5e-4


def test_symmetry():
    g = T.graph('3dpf_holo')
    A = pc.automorphisms(pc.ligand_elements(g), pc._bonds(g))
    assert len(A) == 2
    x = g['ligand'].pos.numpy()
    swapped = x[A[1]]                                           # equivalent atoms exchanged in the reference
    plain = np.sqrt(((x.astype(np.float64) - swapped) ** 2).sum(-1).mean())
    assert plain > 0.1
    got = pc.check_poses([g], [x[None]], ref_ligand_pos=[swapped])[0]
    assert got['rmsd'][0] == 0 and got['rmsd_automorphism'][0] == 1


def _bitwise(a, b):
    assert a.keys() == b.keys()
    for k in a:
        if a[k] is None:
            assert b[k] is None, k
        else:
            assert a[k].dtype == b[k].dtype and a[k].tobytes() == b[k].tobytes(), k


def test_reproducible_and_packing_independent():
    gs = [T.graph('3dpf_holo'), T.graph('3dpf_apo'), _case('lig29'), _case('lig147'),
          inputs.synthetic_complex(5, n_lig=20, n_res=30, flexible_residues=0)]
    ps = [poses(g, S, seed=10 + k) for k, (g, S) in enumerate(zip(gs, (12, 40, 5, 9, 3)))]
    refs = [_ref(g) for g in gs]
    args = ([g for g in gs], [p[0] for p in ps], [p[1] for p in ps], [r[0] for r in refs], [r[1] for r in refs])
    one = pc.check_poses(*args)
    two = pc.check_poses(*args)
    for a, b in zip(one, two):
        _bitwise(a, b)
    for c, g in enumerate(gs):
        _bitwise(one[c], pc.check_poses([g], [ps[c][0]], [ps[c][1]], [refs[c][0]], [refs[c][1]])[0])
        assert_matches(one[c], oracle(g, ps[c][0], ps[c][1], *refs[c]), c)
    # a complex without references in the same call keeps the others' results
    mixed = pc.check_poses(args[0], args[1], args[2], [None] + args[3][1:], [None] + args[4][1:])
    assert 'rmsd' not in mixed[0] and 'sc_rmsd' not in mixed[0]
    for c in range(1, len(gs)):
        _bitwise(mixed[c], one[c])


def test_argument_errors():
    g = T.graph('3dpf_holo')
    x = g['ligand'].pos.numpy()
    with pytest.raises(ValueError):
        pc.check_poses([g], [x[None, :10]])
    with pytest.raises(ValueError):
        pc.check_poses([g], [x[None]], ref_ligand_pos=[x[:10]])
    with pytest.raises(ValueError, match='max_automorphisms'):
        pc.check_poses([g], [x[None]], ref_ligand_pos=[x], max_automorphisms=1)
    L = _lib.lib()
    assert L.ddp_pose_rmsd(None, None, None, 1, None, None, None, None, None, None, None, None) == -1
    assert L.ddp_clash_screen(None, None) == -1


# ------------------------------------------------------------------------------------------------ inference
@pytest.fixture
def deterministic():
    was, warn = torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled()
    torch.use_deterministic_algorithms(True)
    try:
        yield
    finally:
        torch.use_deterministic_algorithms(was, warn_only=warn)


def _row(g):
    c = g.original_center.numpy().reshape(1, 3)
    return dict(complex_graph=g, ref_ligand_pos=g['ligand'].pos.numpy() + c, ref_atom_pos=g['atom'].pos.numpy() + c)


def _dock(fn, *a, **kw):
    np.random.seed(7)
    torch.manual_seed(7)
    return fn(*a, **kw)


def test_infer_single_complex_pose_checks(deterministic):
    m, c, _, _, sa, ca = T.models(DEV, small=True)
    args = inference.default_args(samples_per_complex=4, batch_size=4, inference_steps=3)
    sched = du.get_t_schedule('expbeta', args.inference_steps)
    g = T.graph('3dpf_apo')
    row = _row(g)
    kw = dict(filtering_model=c, filtering_model_args=ca, tr_schedule=sched, device=DEV)
    on = _dock(inference.infer_single_complex, 0, row, m, args, sa, pose_checks=True, **kw)
    off = _dock(inference.infer_single_complex, 0, row, m, args, sa, **kw)
    assert set(off) == {'name', 'index', 'ligand_pos', 'atom_pos', 'confidence'}
    assert set(on) == set(off) | {'checks'}
    for k in off:
        assert np.array_equal(np.asarray(on[k]), np.asarray(off[k])), k
    assert_matches(on['checks'], oracle(g, on['ligand_pos'], on['atom_pos'], row['ref_ligand_pos'], row['ref_atom_pos']), 'infer')
    assert (on['checks']['sc_rmsd'] > 0).all()


def test_infer_complex_group_one_launch_per_kernel(deterministic):
    m, c, _, _, sa, ca = T.models(DEV, small=True)
    args = inference.default_args(samples_per_complex=3, batch_size=9, inference_steps=2)
    sched = du.get_t_schedule('expbeta', args.inference_steps)
    gs = [T.graph('3dpf_apo'), inputs.synthetic_complex(2, n_lig=18, n_res=40, flexible_residues=2),
          inputs.synthetic_complex(3, n_lig=12, n_res=30, flexible_residues=0)]
    rows = [_row(g) for g in gs]
    rows[2].pop('ref_atom_pos')
    before = dict(_lib.COUNTS)
    out = _dock(inference.infer_complex_group, list(enumerate(rows)), m, args, sa, filtering_model=c, filtering_model_args=ca,
                tr_schedule=sched, device=DEV, pose_checks=True)
    for k in ('ddp_clash_screen', 'ddp_pose_rmsd'):
        assert _lib.COUNTS.get(k, 0) - before.get(k, 0) == 1, k
    for row, res in zip(rows, out):
        g = row['complex_graph']
        assert_matches(res['checks'], oracle(g, res['ligand_pos'], res['atom_pos'], row['ref_ligand_pos'], row.get('ref_atom_pos')),
                       g.name)


def _symmetric_ligand_complex(pocket):
    """``pocket`` with tetra-tert-butylmethane (17 carbons) as its ligand: 4! (3!)^4 = 31104 automorphisms, far above the
    default cap of 4096."""
    d = np.array([[1, 1, 1], [1, -1, -1], [-1, 1, -1], [-1, -1, 1]], float) / np.sqrt(3)
    atoms, bonds = [(0.0, 0.0, 0.0, 'C', 0)], []
    for k in range(4):
        q = 1.54 * d[k]
        atoms.append((*q, 'C', 0))
        bonds.append((0, len(atoms) - 1, 1))
        for m in range(4):
            if m != k:
                atoms.append((*(q - 1.54 * d[m]), 'C', 0))
                bonds.append((1 + 4 * k, len(atoms) - 1, 1))
    g = inputs.with_ligand(pocket, seed=0, n_lig=17, name='tetra_tert_butylmethane')
    x, pos, ei, ea = inputs.ligand_graph_from_sdf(atoms, bonds)
    g['ligand'].x, g['ligand'].pos = x, pos - pos.mean(0, keepdim=True)
    g['ligand', 'lig_bond', 'ligand'].edge_index, g['ligand', 'lig_bond', 'ligand'].edge_attr = ei, ea
    em, mr = inputs.rotatable_bond_masks(x.shape[0], ei)
    g['ligand'].edge_mask, g['ligand'].mask_rotate = torch.tensor(em), mr
    return g


def _same_poses(on, off):
    assert set(on) == set(off) | {'checks'}
    for k in off:
        assert np.array_equal(np.asarray(on[k]), np.asarray(off[k])), k


def test_ligand_above_cap_keeps_poses_and_other_checks(deterministic):
    """A failing check never changes docking: a group with a ligand above the automorphism cap keeps the poses of every
    complex; that complex gets the clash sets and sc_rmsd but no RMSD (rmsd_error instead), the others full checks."""
    m, c, _, _, sa, ca = T.models(DEV, small=True)
    args = inference.default_args(samples_per_complex=3, batch_size=9, inference_steps=2)
    sched = du.get_t_schedule('expbeta', args.inference_steps)
    pocket = inputs.synthetic_complex(2, n_lig=18, n_res=40, flexible_residues=2)
    gs = [T.graph('3dpf_apo'), pocket, _symmetric_ligand_complex(pocket)]
    with pytest.raises(ValueError, match='max_automorphisms'):
        pc.check_poses([gs[2]], [gs[2]['ligand'].pos.numpy()[None]], ref_ligand_pos=[gs[2]['ligand'].pos.numpy()])
    rows = [_row(g) for g in gs]
    kw = dict(filtering_model=c, filtering_model_args=ca, tr_schedule=sched, device=DEV)
    on = _dock(inference.infer_complex_group, list(enumerate(rows)), m, args, sa, pose_checks=True, **kw)
    off = _dock(inference.infer_complex_group, list(enumerate(rows)), m, args, sa, **kw)
    for k, (row, a, b) in enumerate(zip(rows, on, off)):
        _same_poses(a, b)
        ref_l = row['ref_ligand_pos'] if k < 2 else None
        assert_matches(a['checks'], oracle(gs[k], a['ligand_pos'], a['atom_pos'], ref_l, row['ref_atom_pos']), k)
    assert 'rmsd' not in on[2]['checks'] and 'max_automorphisms' in on[2]['checks']['rmsd_error']
    assert all('rmsd_error' not in r['checks'] for r in on[:2])
    one_on = _dock(inference.infer_single_complex, 2, rows[2], m, args, sa, pose_checks=True, **kw)
    one_off = _dock(inference.infer_single_complex, 2, rows[2], m, args, sa, **kw)
    _same_poses(one_on, one_off)
    assert 'rmsd' not in one_on['checks'] and 'rmsd_error' in one_on['checks']
