"""Generate the committed fixtures under tests/golden/ (run HERE, where /root/reference exists).

1. ``3dpf_holo.npz`` / ``3dpf_apo.npz``: the reference's only real input fixture
   (example_data/3dpf_*), converted to the HeteroData field layout by diffdock_pocket_b200.inputs
   (ESM features are NOT stored: they are regenerated from a seed at load time).
2. ``python scripts/make_fixtures.py pocket``: ``3dpf_pocket/3dpf_ligand.sdf`` and ``3dpf_pocket/3dpf_protein.pdb``, text
   files written back from ``3dpf_holo.npz`` alone (the ligand with its hydrogens, the residues within 8 A of it) for the
   tests of the SDF / PDB writer.
Reference OUTPUT fixtures (``ref_*.npz``) come from ``scripts/make_ref_fixtures.py``, which executes the reference's own modules.
"""
import copy
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from diffdock_pocket_b200 import inputs, so3, torus, utils  # noqa: E402
from diffdock_pocket_b200.hetero import Batch  # noqa: E402
from oracle import diffusion_ref as D, factory, sampling_ref as S  # noqa: E402

GOLD = os.path.join(ROOT, 'tests', 'golden')
EX = '/root/reference/example_data'


def main():
    os.makedirs(GOLD, exist_ok=True)
    holo = inputs.load_example_3dpf(EX, apo=False, flexible='auto')
    inputs.save_graph_npz(holo, os.path.join(GOLD, '3dpf_holo.npz'))
    # README.md:47 flexible list is in holo numbering (80..242); the ESMFold file is numbered from 1
    flex = [f'A:{int(r) - 79}' for r in (160, 193, 197, 198, 222, 224, 227)]
    apo = inputs.load_example_3dpf(EX, apo=True, flexible=flex, pocket_center=[9.7742, 27.2863, 14.6573])
    inputs.save_graph_npz(apo, os.path.join(GOLD, '3dpf_apo.npz'))
    print('holo', holo['ligand'].pos.shape, holo['receptor'].pos.shape, holo['atom'].pos.shape, holo['flexResidues'].edge_idx.shape)
    print('apo ', apo['ligand'].pos.shape, apo['receptor'].pos.shape, apo['atom'].pos.shape, apo['flexResidues'].edge_idx.shape)


def pocket_files(cutoff=8.0):
    """SDF + PDB of the holo complex from the stored graph: elements, formal charges, bond orders and H counts come from
    the ligand features (hydrogens placed 1 A from their atom), residue and atom names from the atom features; residues
    are numbered by their pocket index."""
    z = np.load(os.path.join(GOLD, '3dpf_holo.npz'))
    out = os.path.join(GOLD, '3dpf_pocket')
    os.makedirs(out, exist_ok=True)
    symbol = {v: k for k, v in inputs.Z_OF.items()}
    c = z['original_center'][0].astype(np.float64)
    lx, lp = z['ligand.x'], z['ligand.pos'] + c
    ei, ea = z['lig_bond.edge_index'], z['lig_bond.edge_attr'].argmax(1)
    charge_code = {0: 0, 1: 3, 2: 2, 3: 1, -1: 5, -2: 6, -3: 7}
    atoms = [(p, symbol[int(x[0]) + 1], charge_code[[-5, -4, -3, -2, -1, 0, 1, 2, 3, 4, 5][x[3]]]) for x, p in zip(lx, lp)]
    bonds = [(int(ei[0, k]), int(ei[1, k]), int(ea[k]) + 1) for k in range(0, ei.shape[1], 2)]
    dirs = np.array([[1, 0, 0], [0, 1, 0], [0, 0, 1]], dtype=np.float64)
    for i, x in enumerate(lx):
        for h in range(int(x[5])):
            bonds.append((i, len(atoms), 1))
            atoms.append((lp[i] + dirs[h], 'H', 0))
    sdf = ['3dpf', '  make_fixtures', 'ligand of tests/golden/3dpf_holo.npz', f'{len(atoms):3d}{len(bonds):3d}  0  0  0  0  0  0  0  0999 V2000']
    sdf += [f'{p[0]:10.4f}{p[1]:10.4f}{p[2]:10.4f} {el:<3} 0{q:3d}  0  0  0  0  0  0  0  0  0  0' for p, el, q in atoms]
    sdf += [f'{a + 1:3d}{b + 1:3d}{t:3d}  0' for a, b, t in bonds] + ['M  END', '$$$$']
    with open(os.path.join(out, '3dpf_ligand.sdf'), 'w') as f:
        f.write('\n'.join(sdf) + '\n')
    ax, ap, owner = z['atom.x'], z['atom.pos'] + c, z['atom_rec_contact.edge_index'][1]
    near = np.unique(owner[np.linalg.norm(ap[:, None] - lp[None], axis=-1).min(1) < cutoff])
    pdb = ['REMARK   1 POCKET OF tests/golden/3dpf_holo.npz: RESIDUES WITHIN 8 A OF THE LIGAND']
    for i in np.flatnonzero(np.isin(owner, near)):
        name, el = inputs.ATOM_TYPE_3[ax[i, 3]], symbol[int(ax[i, 1]) + 1]
        x, y, zz = ap[i]
        pdb.append(f'ATOM  {len(pdb):5d} {name if len(name) == 4 else " " + name:<4} {inputs.AMINO_ACIDS[ax[i, 0]]:3s} A{int(owner[i]) + 1:4d}    '
                   f'{x:8.3f}{y:8.3f}{zz:8.3f}  1.00  0.00          {el:>2s}')
    with open(os.path.join(out, '3dpf_protein.pdb'), 'w') as f:
        f.write('\n'.join(pdb + ['END']) + '\n')


if __name__ == '__main__':
    pocket_files() if sys.argv[1:] == ['pocket'] else main()
