"""Host tables of the pose checks (``diffdock_pocket_b200.posecheck``): automorphisms, the >= 4-bond pair mask, radii from
the element columns, residue owners and bonded exclusions.  No GPU."""

import networkx as nx
import numpy as np
import pytest

import _common as T
from diffdock_pocket_b200 import inputs, posecheck as pc

C = 5                                   # element index of carbon (Z - 1)


def _ring(n):
    return np.array([(i, (i + 1) % n) for i in range(n)])


def test_automorphism_counts():
    assert len(pc.automorphisms([C] * 6, _ring(6))) == 12                                      # benzene skeleton
    assert len(pc.automorphisms([C] * 5, [(0, 1), (0, 2), (0, 3), (0, 4)])) == 24              # neopentane
    g = T.graph('3dpf_holo')
    assert len(pc.automorphisms(pc.ligand_elements(g), pc._bonds(g))) == 2


def test_automorphisms_identity_first_and_element_preserving():
    cases = [([C] * 6, _ring(6)), ([C] * 5, [(0, 1), (0, 2), (0, 3), (0, 4)]),
             ([C, 7, C, 7, C, C], _ring(6)),                                       # pyrimidine-like: elements cut the group
             ([C, C, 7], [])]                                                      # no bonds: only same-element swaps
    g = T.graph('3dpf_apo')
    cases.append((pc.ligand_elements(g), pc._bonds(g)))
    for el, bonds in cases:
        el = np.asarray(el)
        A = pc.automorphisms(el, bonds)
        assert A.dtype == np.int16 and (A[0] == np.arange(len(el))).all()
        assert [tuple(r) for r in A[1:]] == sorted({tuple(r) for r in A[1:]})        # distinct, ordered
        E = {tuple(sorted(b)) for b in np.asarray(bonds).reshape(-1, 2).tolist()}
        for r in A:
            assert (el[r] == el).all()
            assert {tuple(sorted((int(r[a]), int(r[b])))) for a, b in E} == E
    assert len(pc.automorphisms([C, C, 7], [])) == 2
    assert len(pc.automorphisms([C, 7, C, 7, C, C], _ring(6))) == 2


def test_automorphism_cap_raises():
    with pytest.raises(ValueError, match='max_automorphisms = 11'):
        pc.automorphisms([C] * 6, _ring(6), max_automorphisms=11)
    assert len(pc.automorphisms([C] * 6, _ring(6), max_automorphisms=12)) == 12


def _far_networkx(n, bonds):
    G = nx.Graph()
    G.add_nodes_from(range(n))
    G.add_edges_from(map(tuple, np.asarray(bonds).reshape(-1, 2).tolist()))
    sp = dict(nx.all_pairs_shortest_path_length(G))
    return np.array([[i != j and sp[i].get(j, np.inf) >= 4 for j in range(n)] for i in range(n)])


@pytest.mark.parametrize('case', ['3dpf', 'tree29', 'tree147', 'ring', 'disconnected'])
def test_far_pair_mask_equals_shortest_paths(case):
    if case == '3dpf':
        g = T.graph('3dpf_holo')
        n, bonds = g['ligand'].pos.shape[0], pc._bonds(g)
    elif case.startswith('tree'):
        g = inputs.synthetic_complex(3, n_lig=int(case[4:]), n_res=12, flexible_residues=0)
        n, bonds = g['ligand'].pos.shape[0], pc._bonds(g)
    elif case == 'ring':
        n, bonds = 9, _ring(9)
    else:
        n, bonds = 7, np.array([(0, 1), (1, 2), (2, 3), (3, 4)])              # atoms 5, 6 unbonded
    far = pc.far_pairs(n, bonds)
    assert (far == _far_networkx(n, bonds)).all()
    packed = pc.pack_pair_mask(far)
    assert packed.dtype == np.uint32 and packed.shape == (n, (n + 31) // 32)
    j = np.arange(n)
    assert (((packed[:, j // 32] >> (j % 32).astype(np.uint32)) & 1).astype(bool) == far).all()


def test_radius_from_element_columns():
    g = T.graph('3dpf_holo')
    assert (pc.ligand_elements(g) == g['ligand'].x[:, 0].numpy()).all()
    assert (pc.atom_elements(g) == g['atom'].x[:, 1].numpy()).all()
    table = {1: 2.0, 5: 1.92, 6: 1.70, 7: 1.55, 8: 1.52, 9: 1.47, 15: 1.80, 16: 1.80, 17: 1.75, 34: 1.90, 35: 1.85, 53: 1.98,
             26: 2.0, 119: 2.0}                                              # H, Fe and "other" (119) get 2.00
    for z, r in table.items():
        assert pc.RADIUS_TABLE[z - 1] == np.float32(r), z
    assert pc.RADIUS_TABLE.shape == (119,) and pc.RADIUS_TABLE.dtype == np.float32
    # the SDF reader maps an unknown element to index 118 ("other")
    x, *_ = inputs.ligand_graph_from_sdf([(0, 0, 0, 'C', 0), (1.5, 0, 0, 'XX', 0), (3, 0, 0, 'SE', 0)], [(0, 1, 1), (1, 2, 1)])
    assert x[:, 0].tolist() == [5, 118, 33]
    assert pc.RADIUS_TABLE[x[:, 0].numpy()].tolist() == [np.float32(1.70), np.float32(2.0), np.float32(1.90)]
    bad = T.graph('3dpf_holo')
    bad['ligand'].x = bad['ligand'].x.clone()
    bad['ligand'].x[0, 0] = 119
    with pytest.raises(ValueError):
        pc.ligand_elements(bad)


def test_sidechain_tables():
    g = T.graph('3dpf_apo')
    moved = pc.moved_atoms(g)
    assert len(moved) == 37 and (moved == np.unique(g['flexResidues'].subcomponents.numpy())).all()
    owner = pc.residue_owner(g)
    ei = g['atom', 'receptor'].edge_index.numpy()
    assert (owner[ei[0]] == ei[1]).all()
    assert pc.bonded_exclusions(g['atom'].pos.numpy(), moved, owner).shape == (0, 2)
    assert pc.moved_atoms(inputs.synthetic_complex(1, n_lig=8, n_res=10, flexible_residues=0)) is None
    # two residues whose atoms 1 and 3 are 2.0 A apart (a disulfide-like bond); atom 0 moves
    pos = np.array([[0, 0, 0], [1.5, 0, 0], [5, 0, 0], [3.5, 0, 0]], float)
    owner = np.array([0, 0, 1, 1], np.int32)
    ex = pc.bonded_exclusions(pos, np.array([0, 1], np.int32), owner)
    assert ex.tolist() == [[1, 3]]
