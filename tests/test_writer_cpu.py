"""Ranked-pose writer (SURVEY.md 8(f)-2; inference.py:198-240, process_mols.py:726-733, utils/visualise.py:62-132): text-level
SDF / PDB output, checked by reading the files back.  Input: the 3dpf holo ligand (with hydrogens) and its pocket, written
from tests/golden/3dpf_holo.npz by ``scripts/make_fixtures.py pocket``."""
import os

import numpy as np
import pytest

from diffdock_pocket_b200 import inputs, writer

EX = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', '3dpf_pocket')


def test_ranked_sdf_and_flexible_protein_pdb_round_trip(tmp_path):
    g = inputs.load_example_3dpf(EX, apo=False, flexible='auto')
    center = g.original_center.numpy()
    sdf = open(os.path.join(EX, '3dpf_ligand.sdf')).read().splitlines()
    pdb = open(os.path.join(EX, '3dpf_protein.pdb')).read().splitlines()
    rng = np.random.RandomState(0)
    n = 3
    lig = np.stack([g['ligand'].pos.numpy() + center + rng.randn(1, 3) for _ in range(n)])
    atom = np.stack([g['atom'].pos.numpy() + center for _ in range(n)])
    flex = np.unique(g['flexResidues'].subcomponents.numpy())
    atom[:, flex] += rng.randn(n, len(flex), 3) * 0.5
    conf = np.array([1.234, -0.5, -2.0])
    res = dict(name='3dpf', index=0, ligand_pos=lig, atom_pos=atom, confidence=conf)
    w = writer.AsyncWriter()
    w.submit(str(tmp_path), res, sdf, pdb, g['flexResidues'])
    files = w.close()[0]
    assert sorted(files) == sorted(['rank1.sdf', 'rank1_confidence1.23.sdf', 'rank2_confidence-0.50.sdf', 'rank3_confidence-2.00.sdf',
                                    'rank1_protein.pdb', 'rank1_confidence1.23_protein.pdb', 'rank2_confidence-0.50_protein.pdb',
                                    'rank3_confidence-2.00_protein.pdb'])
    # ligand: heavy atoms only, same bond graph, coordinates of the pose
    atoms0, bonds0 = inputs.parse_sdf(os.path.join(EX, '3dpf_ligand.sdf'))
    heavy0 = [a for a in atoms0 if a[3] != 'H']
    for r, nm in enumerate(['rank1.sdf', 'rank2_confidence-0.50.sdf', 'rank3_confidence-2.00.sdf']):
        atoms, bonds = inputs.parse_sdf(str(tmp_path / nm))
        assert [a[3] for a in atoms] == [a[3] for a in heavy0] and len(atoms) == lig.shape[1]
        assert np.abs(np.array([a[:3] for a in atoms]) - lig[r]).max() < 1e-4
        x, pos, ei, ea = inputs.ligand_graph_from_sdf(atoms, bonds)
        assert ei.shape == g['ligand', 'ligand'].edge_index.shape and (ei == g['ligand', 'ligand'].edge_index).all()
    # protein: same records, flexible atoms at their predicted positions, everything else untouched
    out = open(tmp_path / 'rank2_confidence-0.50_protein.pdb').read().splitlines()
    assert len(out) == len(pdb)
    changed = [i for i, (a, b) in enumerate(zip(pdb, out)) if a != b]
    assert 0 < len(changed) <= len(flex)
    res_out = inputs.parse_pdb_heavy(str(tmp_path / 'rank2_confidence-0.50_protein.pdb'))
    g2 = inputs.build_complex_graph(inputs.ligand_graph_from_sdf(atoms0, bonds0), res_out, name='x', flexible='auto')
    assert g2['atom'].pos.shape == g['atom'].pos.shape
    moved = g2['atom'].pos.numpy() + g2.original_center.numpy()
    assert np.abs(moved[flex] - atom[1][flex]).max() < 2e-3                      # PDB columns carry 3 decimals
    rest = np.setdiff1d(np.arange(atom.shape[1]), flex)
    assert np.abs(moved[rest] - atom[1][rest]).max() < 2e-3


def test_mol_block_drops_hydrogens_and_renumbers_bonds():
    tpl = ['mol', '  test', '', '  4  3  0  0  0  0  0  0  0  0999 V2000',
           '    0.0000    0.0000    0.0000 C   0  0  0  0  0  0  0  0  0  0  0  0',
           '    1.0000    0.0000    0.0000 H   0  0  0  0  0  0  0  0  0  0  0  0',
           '    0.0000    1.5000    0.0000 O   0  0  0  0  0  0  0  0  0  0  0  0',
           '    0.0000    2.5000    0.0000 N   0  0  0  0  0  0  0  0  0  0  0  0',
           '  1  2  1  0', '  1  3  2  0', '  3  4  1  0', 'M  END']
    out = writer.mol_block_with_coords(tpl, np.array([[1.0, 2.0, 3.0], [4.0, 5.0, 6.0], [7.0, 8.0, 9.0]]))
    assert out[3].startswith('  3  2') and out[-1] == 'M  END'
    assert out[4].startswith('    1.0000    2.0000    3.0000 C') and out[6].startswith('    7.0000    8.0000    9.0000 N')
    assert out[7].startswith('  1  2  2') and out[8].startswith('  2  3  1')
    with pytest.raises(ValueError):
        writer.mol_block_with_coords(tpl, np.zeros((2, 3)))
