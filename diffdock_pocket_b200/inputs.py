"""Host-side input builders: reference-shaped HeteroData graphs without RDKit / Biopython / ESM.

Preprocessing is outside the accelerated path (SURVEY.md section 2, ``datasets/*`` rows are out of
scope); the hot path only needs graphs with the field layout of SURVEY.md App. C.  This module
provides (a) a plain-text PDB / SDF reader that rebuilds that layout for the ``example_data/3dpf_*``
files following the reference's rules (pocket selection datasets/pdbbind.py:324-339,585-603,775-784;
C-alpha graph and atom->residue edges datasets/process_mols.py:650-724; ligand bond graph :435-454;
rotatable-bond masks utils/torsion.py:16-65; side-chain masks utils/torsion.py:163-248), (b) an
``.npz`` round trip so fixtures travel to machines without the reference tree, and (c) procedural
synthetic complexes for the benchmark configurations.  Ligand categorical features use only what a
text SDF gives (element, degree, H count, charge, ring membership).  The receptor's ESM-2 embeddings
come from ``receptor_embeddings`` (``esm.ESM2`` on the device) when the caller passes a model or
precomputed rows; otherwise they are seeded N(0, 0.25^2) features.
"""
import numpy as np
import torch

from .hetero import HeteroData

AMINO_ACIDS = ['ALA', 'ARG', 'ASN', 'ASP', 'CYS', 'GLN', 'GLU', 'GLY', 'HIS', 'ILE', 'LEU', 'LYS', 'MET', 'PHE', 'PRO',
               'SER', 'THR', 'TRP', 'TYR', 'VAL', 'HIP', 'HIE', 'TPO', 'HID', 'LEV', 'MEU', 'PTR', 'GLV', 'CYT', 'SEP',
               'HIZ', 'CYM', 'GLM', 'ASQ', 'TYS', 'CYX', 'GLZ', 'misc']
ATOM_TYPE_2 = ['C*', 'CA', 'CB', 'CD', 'CE', 'CG', 'CH', 'CZ', 'N*', 'ND', 'NE', 'NH', 'NZ', 'O*', 'OD', 'OE', 'OG', 'OH',
               'OX', 'S*', 'SD', 'SG', 'misc']
ATOM_TYPE_3 = ['C', 'CA', 'CB', 'CD', 'CD1', 'CD2', 'CE', 'CE1', 'CE2', 'CE3', 'CG', 'CG1', 'CG2', 'CH2', 'CZ', 'CZ2',
               'CZ3', 'N', 'ND1', 'ND2', 'NE', 'NE1', 'NE2', 'NH1', 'NH2', 'NZ', 'O', 'OD1', 'OD2', 'OE1', 'OE2', 'OG',
               'OG1', 'OH', 'OXT', 'SD', 'SG', 'misc']
RESIDUE_ATOM_ORDER = {
    'ALA': ['N', 'CA', 'C', 'O', 'CB'], 'ARG': ['N', 'CA', 'C', 'O', 'CB', 'CG', 'CD', 'NE', 'CZ', 'NH1', 'NH2'],
    'ASN': ['N', 'CA', 'C', 'O', 'CB', 'CG', 'OD1', 'ND2'], 'ASP': ['N', 'CA', 'C', 'O', 'CB', 'CG', 'OD1', 'OD2'],
    'CYS': ['N', 'CA', 'C', 'O', 'CB', 'SG'], 'GLN': ['N', 'CA', 'C', 'O', 'CB', 'CG', 'CD', 'OE1', 'NE2'],
    'GLU': ['N', 'CA', 'C', 'O', 'CB', 'CG', 'CD', 'OE1', 'OE2'], 'GLY': ['N', 'CA', 'C', 'O'],
    'HIS': ['N', 'CA', 'C', 'O', 'CB', 'CG', 'ND1', 'CD2', 'CE1', 'NE2'],
    'ILE': ['N', 'CA', 'C', 'O', 'CB', 'CG1', 'CG2', 'CD1'], 'LEU': ['N', 'CA', 'C', 'O', 'CB', 'CG', 'CD1', 'CD2'],
    'LYS': ['N', 'CA', 'C', 'O', 'CB', 'CG', 'CD', 'CE', 'NZ'], 'MET': ['N', 'CA', 'C', 'O', 'CB', 'CG', 'SD', 'CE'],
    'MSE': ['N', 'CA', 'C', 'O', 'CB', 'CG', 'SE', 'CE'],
    'PHE': ['N', 'CA', 'C', 'O', 'CB', 'CG', 'CD1', 'CD2', 'CE1', 'CE2', 'CZ'], 'PRO': ['N', 'CA', 'C', 'O', 'CB', 'CG', 'CD'],
    'SER': ['N', 'CA', 'C', 'O', 'CB', 'OG'], 'THR': ['N', 'CA', 'C', 'O', 'CB', 'OG1', 'CG2'],
    'TRP': ['N', 'CA', 'C', 'O', 'CB', 'CG', 'CD1', 'CD2', 'NE1', 'CE2', 'CE3', 'CZ2', 'CZ3', 'CH2'],
    'TYR': ['N', 'CA', 'C', 'O', 'CB', 'CG', 'CD1', 'CD2', 'CE1', 'CE2', 'CZ', 'OH'],
    'VAL': ['N', 'CA', 'C', 'O', 'CB', 'CG1', 'CG2'],
}
NO_TORSION_RES = {'ALA', 'GLY', 'PRO'}
ONE_LETTER = {'ALA': 'A', 'ARG': 'R', 'ASN': 'N', 'ASP': 'D', 'CYS': 'C', 'GLN': 'Q', 'GLU': 'E', 'GLY': 'G', 'HIS': 'H',
              'ILE': 'I', 'LEU': 'L', 'LYS': 'K', 'MET': 'M', 'PHE': 'F', 'PRO': 'P', 'SER': 'S', 'THR': 'T', 'TRP': 'W',
              'TYR': 'Y', 'VAL': 'V', 'MSE': 'M'}
Z_OF = {'H': 1, 'B': 5, 'C': 6, 'N': 7, 'O': 8, 'F': 9, 'P': 15, 'S': 16, 'CL': 17, 'SE': 34, 'BR': 35, 'I': 53}


def _safe_index(lst, v):
    return lst.index(v) if v in lst else len(lst) - 1


# --------------------------------------------------------------------------------------- text readers
def parse_sdf(path):
    lines = open(path).read().splitlines()
    na, nb = int(lines[3][0:3]), int(lines[3][3:6])
    atoms = []
    for ln in lines[4:4 + na]:
        chg_code = int(ln[36:39]) if len(ln) >= 39 and ln[36:39].strip() else 0
        atoms.append((float(ln[0:10]), float(ln[10:20]), float(ln[20:30]), ln[31:34].strip().upper(),
                      {0: 0, 1: 3, 2: 2, 3: 1, 4: 0, 5: -1, 6: -2, 7: -3}[chg_code]))
    bonds = [(int(ln[0:3]) - 1, int(ln[3:6]) - 1, int(ln[6:9])) for ln in lines[4 + na:4 + na + nb]]
    return atoms, bonds


def parse_pdb_heavy(path):
    """-> list of residues: dict(name, chain, resseq, atoms=[(atom_name, element, xyz)]) in file order."""
    residues, key = [], None
    for ln in open(path):
        if not ln.startswith('ATOM'):
            continue
        name, resn, chain, resseq = ln[12:16].strip(), ln[17:20].strip(), ln[21], ln[22:27].strip()
        elem = ln[76:78].strip().upper() or name[0]
        if elem == 'H' or elem == 'D':
            continue
        if (chain, resseq) != key:
            key = (chain, resseq)
            residues.append(dict(name=resn, chain=chain, resseq=resseq, atoms=[]))
        residues[-1]['atoms'].append((name, elem, np.array([float(ln[30:38]), float(ln[38:46]), float(ln[46:54])])))
    out = []
    for r in residues:
        order = RESIDUE_ATOM_ORDER.get(r['name'])
        names = [a[0] for a in r['atoms']]
        if order is None or not {'N', 'CA', 'C'} <= set(names):
            continue
        r['atoms'].sort(key=lambda a: 999 if a[0] == 'OXT' else (order.index(a[0]) if a[0] in order else 998))
        out.append(r)
    return out


# --------------------------------------------------------------------------------------- receptor language-model features
def chain_sequences(residues):
    """-> [(chain_id, sequence, residue_indices)]: one-letter sequence of every chain of ``parse_pdb_heavy``'s residues
    (chains and residues in file order, MSE read as M) and the indices of its residues in ``residues``.

    ``parse_pdb_heavy`` keeps ATOM records of standard residues (and MSE) only, so a chain with HETATM residues (MSE
    written as HETATM, modified residues) gives a shorter sequence than the reference's walk over every residue with
    N / CA / C atoms (DESIGN section 12)."""
    chains = {}
    for i, r in enumerate(residues):
        chains.setdefault(r['chain'], []).append(i)
    return [(c, ''.join(ONE_LETTER.get(residues[i]['name'], 'X') for i in idx), idx) for c, idx in chains.items()]


def receptor_embeddings(esm_model, residues):
    """ESM-2 last-layer embeddings of ``residues`` (``parse_pdb_heavy`` order) -> [len(residues), D] fp32 on the model's
    device.  Every chain is embedded as its own sequence with BOS / EOS, as the reference does, all chains in one
    ``esm.embed_sequences`` call; rows go back to residue order.  See ``chain_sequences`` for the HETATM deviation."""
    from . import esm
    chains = chain_sequences(residues)
    reps = esm.embed_sequences(esm_model, [s for _, s, _ in chains])
    out = torch.empty(len(residues), esm_model.embed_dim, dtype=torch.float32, device=reps[0].device if reps else 'cpu')
    for (_, _, idx), rep in zip(chains, reps):
        out[torch.as_tensor(idx, device=out.device)] = rep
    return out


# --------------------------------------------------------------------------------------- ligand
def _ring_sizes(n, bonds):
    import networkx as nx
    G = nx.Graph()
    G.add_nodes_from(range(n))
    G.add_edges_from([(a, b) for a, b, _ in bonds])
    sizes = [set() for _ in range(n)]
    for cyc in nx.minimum_cycle_basis(G):
        for a in cyc:
            sizes[a].add(len(cyc))
    return sizes


def rotatable_bond_masks(n_nodes, edge_index):
    """utils/torsion.py:16-65 on the directed bond list (both directions, consecutive)."""
    import networkx as nx
    edges = edge_index.T.numpy()
    G = nx.Graph()
    G.add_nodes_from(range(n_nodes))
    G.add_edges_from([tuple(e) for e in edges])
    to_rotate = []
    for i in range(0, edges.shape[0], 2):
        assert edges[i, 0] == edges[i + 1, 1]
        G2 = G.copy()
        G2.remove_edge(*edges[i])
        if not nx.is_connected(G2):
            comp = list(sorted(nx.connected_components(G2), key=len)[0])
            if len(comp) > 1:
                if edges[i, 0] in comp:
                    to_rotate += [[], comp]
                else:
                    to_rotate += [comp, []]
                continue
        to_rotate += [[], []]
    mask_edges = np.asarray([len(c) > 0 for c in to_rotate], dtype=bool)
    mask_rotate = np.zeros((int(mask_edges.sum()), n_nodes), dtype=bool)
    k = 0
    for i, c in enumerate(to_rotate):
        if mask_edges[i]:
            mask_rotate[k][np.asarray(c, dtype=int)] = True
            k += 1
    return mask_edges, mask_rotate


def ligand_graph_from_sdf(atoms, bonds):
    heavy = [i for i, a in enumerate(atoms) if a[3] != 'H']
    remap = {old: new for new, old in enumerate(heavy)}
    nh = [0] * len(atoms)
    deg = [0] * len(atoms)
    for a, b, _ in bonds:
        deg[a] += 1
        deg[b] += 1
        if atoms[b][3] == 'H':
            nh[a] += 1
        if atoms[a][3] == 'H':
            nh[b] += 1
    hb = [(remap[a], remap[b], t) for a, b, t in bonds if a in remap and b in remap]
    rings = _ring_sizes(len(heavy), hb)
    unsat = [False] * len(heavy)
    arom = [False] * len(heavy)
    for a, b, t in hb:
        if t in (2, 3, 4):
            unsat[a] = unsat[b] = True
        if t == 4:
            arom[a] = arom[b] = True
    x = []
    charges = [-5, -4, -3, -2, -1, 0, 1, 2, 3, 4, 5]
    for new, old in enumerate(heavy):
        z = Z_OF.get(atoms[old][3], 119)
        x.append([min(z - 1, 118), 0, min(deg[old], 11), _safe_index(charges + ['misc'], atoms[old][4]), 0, min(nh[old], 9), 0,
                  1 if unsat[new] else 2, int(arom[new]), min(len(rings[new]), 7),
                  int(3 in rings[new]), int(4 in rings[new]), int(5 in rings[new]), int(6 in rings[new]),
                  int(7 in rings[new]), int(8 in rings[new])])
    pos = np.array([[atoms[o][0], atoms[o][1], atoms[o][2]] for o in heavy], dtype=np.float32)
    row, col, et = [], [], []
    for a, b, t in hb:
        row += [a, b]
        col += [b, a]
        et += 2 * [{1: 0, 2: 1, 3: 2, 4: 3}.get(t, 0)]
    edge_index = torch.tensor([row, col], dtype=torch.long)
    edge_attr = torch.nn.functional.one_hot(torch.tensor(et, dtype=torch.long), num_classes=4).float()
    return torch.tensor(x, dtype=torch.long), torch.from_numpy(pos), edge_index, edge_attr


# --------------------------------------------------------------------------------------- side chains
def _sidechain_bonds(res_atom_names):
    """utils/torsion.py:163-248: rotatable side-chain bonds, C-alpha outwards (BFS), with the atoms each one moves."""
    import networkx as nx
    keep = [i for i, n in enumerate(res_atom_names) if n not in ('OXT', 'C', 'O', 'N')]
    nodes = [res_atom_names[i] for i in keep]
    nxt = {'A': 'B', 'B': 'G', 'G': 'D', 'D': 'E', 'E': 'Z', 'Z': 'H', 'H': ''}
    G = nx.DiGraph()
    G.add_nodes_from(nodes)
    for i in range(len(nodes) - 1):
        for j in range(i + 1, len(nodes)):
            a, b = nodes[i], nodes[j]
            if (a, b) in (('CE1', 'NE2'), ('NE1', 'CE2'), ('CD2', 'CE3'), ('CZ3', 'CH2')):
                G.add_edge(a, b)
            if len(a) < 2 or len(b) < 2:
                continue
            if len(a) == len(b) == 3:
                if nxt.get(a[1]) == b[1] and a[2] == b[2]:
                    G.add_edge(a, b)
            elif nxt.get(a[1]) == b[1]:
                G.add_edge(a, b)
    out = []
    if 'CA' not in G:
        return out
    for e in nx.bfs_tree(G, 'CA').edges():
        G2 = G.to_undirected()
        G2.remove_edge(*e)
        if not nx.is_connected(G2):
            comp = [c for c in nx.connected_components(G2) if e[1] in c][0]
            if len(comp) > 1:
                g2n = list(G2.nodes)
                out.append(([keep[g2n.index(v)] for v in comp], [keep[g2n.index(e[0])], keep[g2n.index(e[1])]]))
    return out


# --------------------------------------------------------------------------------------- complex graph
def build_complex_graph(lig, residues, name='complex', pocket_center=None, flexible=None, flexdist=3.5,
                        receptor_radius=15.0, c_alpha_max_neighbors=24, pocket_buffer=10.0, pocket_cutoff=5.0,
                        esm_seed=1234, lm_embeddings=None):
    """``lig`` = (x, pos, edge_index, edge_attr); ``flexible``: None -> no flexResidues store,
    'auto' -> prism/flexdist rule, or an explicit list like ['A:160', 'A:193'].  ``lm_embeddings``: [len(residues), 1280]
    rows aligned to ``residues`` (``receptor_embeddings``); the pocket residues take theirs as ``receptor.x[:, 1:]``.
    Without it those columns are seeded N(0, 0.25^2) noise (``esm_seed``)."""
    lig_x, lig_pos, lig_ei, lig_ea = lig
    g = HeteroData()
    g['name'] = name
    g['ligand'].x, g['ligand'].pos = lig_x, lig_pos.clone().float()
    g['ligand', 'lig_bond', 'ligand'].edge_index = lig_ei
    g['ligand', 'lig_bond', 'ligand'].edge_attr = lig_ea
    em, mr = rotatable_bond_masks(lig_x.shape[0], lig_ei)
    g['ligand'].edge_mask, g['ligand'].mask_rotate = torch.tensor(em), mr

    ca_all = torch.tensor(np.array([[a[2] for a in r['atoms'] if a[0] == 'CA'][0] for r in residues]), dtype=torch.float32)
    if pocket_center is None:                                             # datasets/pdbbind.py:324-339
        d = torch.cdist(ca_all, g['ligand'].pos)
        label = torch.any(d < pocket_cutoff, dim=1)
        center = ca_all[label].mean(0) if label.any() else ca_all[d.min(1)[0].argmin()]
        radius = torch.linalg.norm(g['ligand'].pos - center[None], dim=1).max()
    else:                                                                 # datasets/pdbbind.py:586-590
        center = torch.as_tensor(pocket_center, dtype=torch.float32)
        radius = torch.linalg.vector_norm(g['ligand'].pos - g['ligand'].pos.mean(0, keepdim=True), dim=1).max()
    radius = float(radius) + pocket_buffer
    cen = center.numpy().astype(np.float64)
    pocket_idx = [i for i, r in enumerate(residues)
                  if (np.linalg.norm(np.array([a[2] for a in r['atoms']]) - cen, axis=1) < radius).any()]
    pocket = [residues[i] for i in pocket_idx]
    ca = np.array([[a[2] for a in r['atoms'] if a[0] == 'CA'][0] for r in pocket])
    n_res = len(pocket)
    dist = np.linalg.norm(ca[:, None] - ca[None], axis=-1)
    src, dst = [], []
    for i in range(n_res):                                                # datasets/process_mols.py:661-677
        nb = list(np.where(dist[i] < receptor_radius)[0])
        nb.remove(i)
        if c_alpha_max_neighbors is not None and len(nb) > c_alpha_max_neighbors:
            nb = list(np.argsort(dist[i]))[1:c_alpha_max_neighbors + 1]
        if len(nb) == 0:
            nb = list(np.argsort(dist[i]))[1:2]
        src += [i] * len(nb)
        dst += [int(j) for j in nb]
    aa = torch.tensor([[_safe_index(AMINO_ACIDS, r['name'])] for r in pocket], dtype=torch.float32)
    if lm_embeddings is None:
        esm = torch.from_numpy(np.random.RandomState(esm_seed).randn(n_res, 1280).astype(np.float32) * 0.25)
    else:
        lm = torch.as_tensor(lm_embeddings)
        if lm.shape != (len(residues), 1280):
            raise ValueError(f'lm_embeddings must be [{len(residues)}, 1280] (one row per residue), got {tuple(lm.shape)}')
        esm = lm[torch.as_tensor(pocket_idx, dtype=torch.long, device=lm.device)].detach().to('cpu', torch.float32)
    g['receptor'].x = torch.cat([aa, esm], 1)
    g['receptor'].pos = torch.from_numpy(ca).float()
    g['receptor', 'rec_contact', 'receptor'].edge_index = torch.tensor([src, dst], dtype=torch.long)
    ax, ap, owner, res_start = [], [], [], []
    for ri, r in enumerate(pocket):
        res_start.append(len(ax))
        for (an, el, xyz) in r['atoms']:
            ax.append([_safe_index(AMINO_ACIDS, r['name']), min(Z_OF.get(el, 119) - 1, 118),
                       _safe_index(ATOM_TYPE_2, (an + '*')[:2]), _safe_index(ATOM_TYPE_3, an)])
            ap.append(xyz)
            owner.append(ri)
    g['atom'].x = torch.tensor(ax, dtype=torch.long)
    g['atom'].pos = torch.from_numpy(np.array(ap)).float()
    g['atom', 'atom_rec_contact', 'receptor'].edge_index = torch.tensor([list(range(len(ax))), owner], dtype=torch.long)

    if flexible is not None:                                              # datasets/process_mols.py:773-914
        lp = g['ligand'].pos.numpy().astype(np.float64)
        lo, hi = lp.min(0) - flexdist, lp.max(0) + flexdist
        sub, mapping, eidx, nb_per_res, ids = [], [], [], [], []
        for ri, r in enumerate(pocket):
            if r['name'] in NO_TORSION_RES or r['name'] not in RESIDUE_ATOM_ORDER:
                continue
            if flexible == 'auto':
                ok = False
                for (an, el, xyz) in r['atoms']:
                    if an in ('CA', 'N', 'C', 'O', 'OXT'):
                        continue
                    if np.all(xyz >= lo) and np.all(xyz <= hi) and (np.linalg.norm(lp - xyz, axis=1) < flexdist).any():
                        ok = True
                        break
            else:
                ok = f"{r['chain']}:{r['resseq']}" in flexible
            if not ok:
                continue
            bonds = _sidechain_bonds([a[0] for a in r['atoms']])
            nb_per_res.append(len(bonds))
            ids.append((r['chain'], r['resseq']))
            for comp, e in bonds:
                mapping.append([len(sub), len(sub) + len(comp)])
                sub += [res_start[ri] + c for c in comp]
                eidx.append([res_start[ri] + e[0], res_start[ri] + e[1]])
        fr = g['flexResidues']
        fr.subcomponents = torch.tensor(sub, dtype=torch.long)
        fr.subcomponentsMapping = torch.tensor(mapping, dtype=torch.long).reshape(-1, 2)
        fr.edge_idx = torch.tensor(eidx, dtype=torch.long).reshape(-1, 2)
        fr.residueNBondsMapping = torch.tensor(nb_per_res, dtype=torch.long)
        fr.pdbIds = ids
        fr.num_nodes = fr.edge_idx.shape[0]
    for k in ('receptor', 'atom', 'ligand'):                              # datasets/pdbbind.py:714-731
        g[k].pos = g[k].pos - center[None]
    g.original_center = center[None].clone()
    return g


def load_example_3dpf(example_dir, apo=False, flexible='auto', pocket_center=None, esm_model=None):
    """``esm_model``: an ``esm.ESM2`` on the device; given, the receptor features are its embeddings of the protein's
    chains (``receptor_embeddings``) instead of seeded noise."""
    atoms, bonds = parse_sdf(f'{example_dir}/3dpf_ligand.sdf')
    residues = parse_pdb_heavy(f"{example_dir}/{'3dpf_protein_esm.pdb' if apo else '3dpf_protein.pdb'}")
    lm = None if esm_model is None else receptor_embeddings(esm_model, residues)
    return build_complex_graph(ligand_graph_from_sdf(atoms, bonds), residues, name='3dpf', pocket_center=pocket_center,
                               flexible=flexible, lm_embeddings=lm)


# --------------------------------------------------------------------------------------- npz round trip
_FIELDS = [('ligand', 'x'), ('ligand', 'pos'), ('ligand', 'edge_mask'), ('receptor', 'x'), ('receptor', 'pos'),
           ('atom', 'x'), ('atom', 'pos')]


def save_graph_npz(g, path, drop_esm=True):
    d = {f'{a}.{b}': getattr(g[a], b).numpy() for a, b in _FIELDS}
    if drop_esm:
        d['receptor.x'] = d['receptor.x'][:, :1]
    d['ligand.mask_rotate'] = g['ligand'].mask_rotate
    d['lig_bond.edge_index'] = g['ligand', 'ligand'].edge_index.numpy()
    d['lig_bond.edge_attr'] = g['ligand', 'ligand'].edge_attr.numpy()
    d['rec_contact.edge_index'] = g['receptor', 'receptor'].edge_index.numpy()
    d['atom_rec_contact.edge_index'] = g['atom', 'receptor'].edge_index.numpy()
    d['original_center'] = g.original_center.numpy()
    if 'flexResidues' in g:
        fr = g['flexResidues']
        for k in ('subcomponents', 'subcomponentsMapping', 'edge_idx', 'residueNBondsMapping'):
            d[f'flexResidues.{k}'] = getattr(fr, k).numpy()
    np.savez_compressed(path, **d)


def load_graph_npz(path, esm_seed=1234, name='complex'):
    z = np.load(path)
    g = HeteroData()
    g['name'] = name
    for a, b in _FIELDS:
        setattr(g[a], b, torch.from_numpy(z[f'{a}.{b}']))
    if g['receptor'].x.shape[1] == 1:
        esm = np.random.RandomState(esm_seed).randn(g['receptor'].x.shape[0], 1280).astype(np.float32) * 0.25
        g['receptor'].x = torch.cat([g['receptor'].x.float(), torch.from_numpy(esm)], 1)
    g['ligand'].mask_rotate = z['ligand.mask_rotate']
    g['ligand', 'lig_bond', 'ligand'].edge_index = torch.from_numpy(z['lig_bond.edge_index'])
    g['ligand', 'lig_bond', 'ligand'].edge_attr = torch.from_numpy(z['lig_bond.edge_attr'])
    g['receptor', 'rec_contact', 'receptor'].edge_index = torch.from_numpy(z['rec_contact.edge_index'])
    g['atom', 'atom_rec_contact', 'receptor'].edge_index = torch.from_numpy(z['atom_rec_contact.edge_index'])
    g.original_center = torch.from_numpy(z['original_center'])
    if 'flexResidues.edge_idx' in z:
        fr = g['flexResidues']
        for k in ('subcomponents', 'subcomponentsMapping', 'edge_idx', 'residueNBondsMapping'):
            setattr(fr, k, torch.from_numpy(z[f'flexResidues.{k}']))
        fr.num_nodes = fr.edge_idx.shape[0]
    return g


# --------------------------------------------------------------------------------------- synthetic
def _random_tree_ligand(rng, n_lig):
    """Random-tree ligand with 1.5 A bonds -> (x, pos, edge_index, edge_attr)."""
    pos = [np.zeros(3)]
    bonds = []
    while len(pos) < n_lig:
        a = rng.randint(len(pos))
        d = rng.randn(3)
        p = pos[a] + d * 1.5 / np.linalg.norm(d)
        if np.min(np.linalg.norm(np.array(pos) - p, axis=1)) < 1.2:
            continue
        bonds.append((a, len(pos), 1))
        pos.append(p)
    atoms = [(p[0], p[1], p[2], 'C' if rng.rand() < 0.7 else ('N' if rng.rand() < 0.5 else 'O'), 0) for p in pos]
    return ligand_graph_from_sdf(atoms, bonds)


def with_ligand(pocket_graph, seed, n_lig, name=None):
    """A complex made of ``pocket_graph``'s receptor (its stores are SHARED, not copied) and a new procedural ligand:
    the virtual-screening shape of BASELINE.json configs[4] (one pocket, many ligands)."""
    lig_x, lig_pos, lig_ei, lig_ea = _random_tree_ligand(np.random.RandomState(seed), n_lig)
    g = HeteroData()
    for k, st in pocket_graph._nodes.items():
        if k != 'ligand':
            g._nodes[k] = st
    for k, st in pocket_graph._edges.items():
        if k[0] != 'ligand':
            g._edges[k] = st
    g._glob.update(pocket_graph._glob)
    g['name'] = name or f'lig{seed}'
    g['ligand'].x = lig_x
    g['ligand'].pos = (lig_pos - lig_pos.mean(0, keepdim=True)).float()
    g['ligand', 'lig_bond', 'ligand'].edge_index = lig_ei
    g['ligand', 'lig_bond', 'ligand'].edge_attr = lig_ea
    em, mr = rotatable_bond_masks(lig_x.shape[0], lig_ei)
    g['ligand'].edge_mask, g['ligand'].mask_rotate = torch.tensor(em), mr
    return g


def pdbbind_test_sizes():
    """Heavy-atom counts of the 363 PDBBind test ligands (tests/golden/pdbbind_test_ligand_sizes.txt, written by
    scripts/make_size_law.py from the reference's data/test_ligands_smiles.txt): min 7, median 29, mean 35.9, max 147."""
    import os
    path = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), 'tests', 'golden', 'pdbbind_test_ligand_sizes.txt')
    return [int(l) for l in open(path) if l.strip()]


def pdbbind_synth_set(n=None, seed=0, flexible_residues=5):
    """BASELINE.json configs[3]: synthetic complexes whose ligand sizes follow the PDBBind test set; the pocket grows with
    the ligand (the reference cuts it at ligand radius + 10 A, datasets/pdbbind.py:597)."""
    sizes = pdbbind_test_sizes()
    sizes = sizes if n is None else [sizes[i % len(sizes)] for i in range(n)]
    return [synthetic_complex(seed + i, n_lig=int(k), n_res=int(min(200, 70 + 2 * k)), flexible_residues=flexible_residues, name=f'pdbbind_synth{i}')
            for i, k in enumerate(sizes)]


def synthetic_complex(seed, n_lig=37, n_res=139, flexible_residues=7, name=None):
    """Procedural pocket + ligand of reference shape: a random-walk C-alpha trace folded into a ball
    around the origin (3.8 A steps), ~8 heavy atoms per residue with real residue templates, and a
    random-tree ligand with 1.5 A bonds (SURVEY.md 8(d) configs 3-5)."""
    rng = np.random.RandomState(seed)
    names = [k for k in RESIDUE_ATOM_ORDER if k != 'MSE']
    R = 3.8 * (n_res ** (1 / 3)) * 0.9 + 4.0
    ca = [rng.randn(3) * 2 + np.array([R * 0.5, 0, 0])]
    while len(ca) < n_res:
        step = rng.randn(3)
        step *= 3.8 / np.linalg.norm(step)
        p = ca[-1] + step
        if np.linalg.norm(p) > R or np.linalg.norm(p) < 5.0 or (len(ca) > 2 and np.min(np.linalg.norm(np.array(ca[:-1]) - p, axis=1)) < 3.0):
            continue
        ca.append(p)
    residues = []
    for i, c in enumerate(ca):
        rn = names[rng.randint(len(names))]
        atoms = []
        prev = c
        for an in RESIDUE_ATOM_ORDER[rn]:
            if an == 'CA':
                xyz = c
            else:
                d = rng.randn(3)
                xyz = prev + d * 1.5 / np.linalg.norm(d)
            atoms.append((an, an[0], xyz.copy()))
            if an not in ('N', 'C', 'O'):
                prev = xyz
        residues.append(dict(name=rn, chain='A', resseq=str(i + 1), atoms=atoms))
    lig = _random_tree_ligand(rng, n_lig)
    flex = None
    if flexible_residues:
        cand = [r for r in residues if r['name'] not in NO_TORSION_RES]
        cand.sort(key=lambda r: np.linalg.norm([a[2] for a in r['atoms'] if a[0] == 'CA'][0]))
        flex = [f"A:{r['resseq']}" for r in cand[:flexible_residues]]
    return build_complex_graph(lig, residues, name=name or f'synthetic{seed}', pocket_center=np.zeros(3), flexible=flex,
                               pocket_buffer=1e6, esm_seed=seed + 1234)
