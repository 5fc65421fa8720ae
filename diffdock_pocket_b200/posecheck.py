"""Pose checks of docked poses on the device: symmetry-corrected ligand RMSD, flexible side-chain RMSD and steric clashes.

Definitions (DESIGN section 11).  All positions are in one frame, the caller's; no superposition is done.
  * Elements: ligand atom i has Z = ligand.x[i, 0] + 1, pocket atom j has Z = atom.x[j, 1] + 1; index 118 means "other".
    Van der Waals radii: ``VDW_RADII`` (2.00 A for every other element), tabulated once in ``RADIUS_TABLE``.
  * Ligand RMSD: min over the element-preserving automorphisms pi of the heavy-atom bond graph (edges unlabelled, so
    Kekule and aromatic input give the same answer) of sqrt(mean_i |x_i - ref_pi(i)|^2).  The automorphisms are enumerated
    on the host (networkx GraphMatcher), identity first; more than ``max_automorphisms`` raises ValueError.
  * Side-chain RMSD: by-index RMSD over the moved atoms ``flexResidues.subcomponents.unique()`` (no ring-flip or
    carboxylate symmetry); None for a complex without flexible residues.
  * Clash: d_ij < ratio (R_i + R_j), evaluated in fp32 as d^2 < (ratio (R_i + R_j))^2.  Three sets, each giving a count
    and the minimum of d_ij / (R_i + R_j) (+inf for an empty set): ligand x pocket of the same pose; moved side-chain
    atom x pocket atom of another residue (ordered pairs), without the pairs closer than ``BONDED_CUTOFF`` in the input
    receptor (disulfides); ligand pairs at least ``FAR_BONDS`` bonds apart (or disconnected).
"""
import numpy as np
import torch

from . import _lib

VDW_RADII = {6: 1.70, 7: 1.55, 8: 1.52, 9: 1.47, 15: 1.80, 16: 1.80, 17: 1.75, 35: 1.85, 53: 1.98, 5: 1.92, 34: 1.90}
OTHER_RADIUS = 2.00
N_ELEMENTS = 119                  # element indices 0..118 (Z - 1); 118 = "other"
RADIUS_TABLE = np.array([VDW_RADII.get(e + 1, OTHER_RADIUS) for e in range(N_ELEMENTS)], dtype=np.float32)
BONDED_CUTOFF = 2.3
FAR_BONDS = 4
MAX_ROWS = 512                    # ddp_pose_max_ligand_atoms(): ligand atoms, and moved side-chain atoms, per pose

_SETS = ('ligand_pocket', 'sidechain_pocket', 'ligand_internal')


# ------------------------------------------------------------------------------------------------ host tables
def _elements(col, what):
    e = np.asarray(torch.as_tensor(col).cpu().numpy(), dtype=np.int64)
    if e.size and (e.min() < 0 or e.max() >= N_ELEMENTS):
        raise ValueError(f'{what}: element index outside [0, {N_ELEMENTS - 1}]')
    return e.astype(np.int32)


def ligand_elements(g):
    """Radius-table index (Z - 1) of every ligand atom: ``ligand.x[:, 0]``."""
    return _elements(g['ligand'].x[:, 0], 'ligand.x[:, 0]')


def atom_elements(g):
    """Radius-table index (Z - 1) of every pocket atom: ``atom.x[:, 1]``."""
    return _elements(g['atom'].x[:, 1], 'atom.x[:, 1]')


def _bonds(g):
    ei = np.asarray(g['ligand', 'ligand'].edge_index.cpu().numpy(), dtype=np.int64)
    return np.unique(np.sort(ei.T, axis=1), axis=0) if ei.size else np.zeros((0, 2), np.int64)


def automorphisms(elements, bonds, max_automorphisms=4096, name='ligand'):
    """Element-preserving automorphisms of the bond graph -> int16 [A, N], row a maps atom i to perm[a, i]; row 0 is the
    identity, the others follow in lexicographic order.  ``bonds``: [E, 2] (either direction, repeats allowed)."""
    import networkx as nx
    from networkx.algorithms.isomorphism import GraphMatcher
    n = len(elements)
    G = nx.Graph()
    G.add_nodes_from((i, {'z': int(z)}) for i, z in enumerate(elements))
    G.add_edges_from((int(a), int(b)) for a, b in np.asarray(bonds).reshape(-1, 2))
    out = []
    for m in GraphMatcher(G, G, node_match=lambda a, b: a['z'] == b['z']).isomorphisms_iter():
        out.append([m[i] for i in range(n)])
        if len(out) > max_automorphisms:
            raise ValueError(f'{name}: more than max_automorphisms = {max_automorphisms} automorphisms '
                             f'({len(out)} enumerated before stopping)')
    ident = list(range(n))
    rest = sorted(p for p in out if p != ident)
    return np.asarray([ident] + rest, dtype=np.int16).reshape(-1, n)


def far_pairs(n, bonds):
    """bool [N, N]: pairs at least FAR_BONDS bonds apart in the bond graph, or disconnected (the diagonal is False)."""
    from scipy.sparse import coo_matrix
    from scipy.sparse.csgraph import shortest_path
    b = np.asarray(bonds, dtype=np.int64).reshape(-1, 2)
    adj = coo_matrix((np.ones(len(b)), (b[:, 0], b[:, 1])), shape=(n, n))
    d = shortest_path(adj, method='D', directed=False, unweighted=True)
    return d >= FAR_BONDS


def pack_pair_mask(mask):
    """bool [N, N] -> uint32 [N, ceil(N / 32)]: bit j % 32 of word j // 32 in row i is mask[i, j]."""
    n = mask.shape[0]
    w = (n + 31) // 32
    padded = np.zeros((n, 32 * w), dtype=np.uint64)
    padded[:, :n] = mask
    return (padded.reshape(n, w, 32) << np.arange(32, dtype=np.uint64)).sum(-1).astype(np.uint32)


def moved_atoms(g):
    """Pocket atoms moved by the side-chain torsions (sorted), or None without flexible residues."""
    if 'flexResidues' not in g or 'subcomponents' not in g['flexResidues']:
        return None
    sub = g['flexResidues'].subcomponents
    return np.unique(np.asarray(sub.cpu().numpy(), dtype=np.int64)).astype(np.int32) if sub.numel() else None


def residue_owner(g):
    """Residue of every pocket atom (``('atom', 'receptor').edge_index[1]``); -1 for an atom without one."""
    ei = np.asarray(g['atom', 'receptor'].edge_index.cpu().numpy(), dtype=np.int64)
    owner = np.full(g['atom'].pos.shape[0], -1, dtype=np.int32)
    owner[ei[0]] = ei[1]
    return owner


def bonded_exclusions(pos, moved, owner):
    """int32 [E, 2] pairs (k, j): moved atom k (position in ``moved``) and pocket atom j of another residue closer than
    BONDED_CUTOFF in ``pos`` (the input receptor): covalent bonds between residues, left out of the side-chain set."""
    if moved is None or len(moved) == 0:
        return np.zeros((0, 2), np.int32)
    p = np.asarray(pos, dtype=np.float64)
    d = np.linalg.norm(p[moved][:, None] - p[None], axis=-1)
    k, j = np.nonzero((d < BONDED_CUTOFF) & (owner[moved][:, None] != owner[None]))
    return np.stack([k, j], 1).astype(np.int32).reshape(-1, 2)


# ------------------------------------------------------------------------------------------------ packing
class _Tables:
    """The index tables of one call, packed for one upload each: int32 tables (sections 16-byte aligned), a parallel
    int32 array holding the residue owners at the offsets of the pocket radius indices, and the int16 automorphisms.
    Complexes with equal ligand topologies, or equal pockets, share their tables."""

    def __init__(self, max_automorphisms):
        self.ints, self.owners, self.n = [], [], 0
        self.autos, self.n16 = [], 0
        self.max_automorphisms = max_automorphisms
        self._topo, self._pocket, self._ident = {}, {}, {}

    def add(self, a, owner=None):
        a = np.asarray(a)
        a = np.ascontiguousarray(a.view(np.int32) if a.dtype == np.uint32 else a.astype(np.int32)).reshape(-1)
        off, size = self.n, len(a) + (-len(a)) % 4
        self.ints.append(np.pad(a, (0, size - len(a))))
        self.owners.append(np.pad(np.asarray(owner, np.int32), (0, size - len(a))) if owner is not None else np.zeros(size, np.int32))
        self.n += size
        return off

    def _add16(self, a):
        off = self.n16
        self.autos.append(np.asarray(a, np.int16).reshape(-1))
        self.n16 += self.autos[-1].size
        return off

    def ligand(self, g):
        """-> dict(el, far: offsets of the radius indices and the pair mask, elements, bonds, autos) of g's topology."""
        el, bonds = ligand_elements(g), _bonds(g)
        key = (el.tobytes(), bonds.tobytes())
        t = self._topo.get(key)
        if t is None:
            t = self._topo[key] = dict(el=self.add(el), far=self.add(pack_pair_mask(far_pairs(len(el), bonds))), elements=el,
                                       bonds=bonds, autos=None)
        return t

    def automorphisms(self, t, name):
        """-> (offset, count) of the automorphism table of topology t; ValueError above the cap (enumerated once)."""
        if t['autos'] is None:
            try:
                A = automorphisms(t['elements'], t['bonds'], self.max_automorphisms, name)
                t['autos'] = (self._add16(A), len(A))
            except ValueError as e:
                t['autos'] = e
        if isinstance(t['autos'], ValueError):
            raise t['autos']
        return t['autos']

    def identity(self, n):
        if n not in self._ident:
            self._ident[n] = self._add16(np.arange(n))
        return self._ident[n]

    def pocket(self, g, c):
        """-> dict(atom, moved_off, n_moved, excl, n_excl: offsets and counts, moved: atom indices or None) of g's pocket."""
        fr = g['flexResidues'] if 'flexResidues' in g and 'subcomponents' in g['flexResidues'] else None
        parts = (g['atom'].x[:, 1], g['atom'].pos, g['atom', 'receptor'].edge_index, fr.subcomponents if fr is not None else None)
        key = tuple(b'' if t is None else np.ascontiguousarray(t.cpu().numpy()).tobytes() for t in parts)
        p = self._pocket.get(key)
        if p is None:
            moved = moved_atoms(g)
            if moved is not None and len(moved) > MAX_ROWS:
                raise ValueError(f'complex {c}: {len(moved)} moved side-chain atoms, more than {MAX_ROWS}')
            owner = residue_owner(g)
            excl = bonded_exclusions(np.asarray(g['atom'].pos.cpu().numpy()), moved, owner)
            p = self._pocket[key] = dict(atom=self.add(atom_elements(g), owner), moved=moved,
                                         moved_off=self.add(moved) if moved is not None else 0,
                                         n_moved=0 if moved is None else len(moved), excl=self.add(excl) // 2, n_excl=len(excl))
        return p


def _device(*lists):
    for lst in lists:
        for a in lst:
            if torch.is_tensor(a) and a.is_cuda:
                return a.device
    return torch.device('cuda', torch.cuda.current_device())


def _rows(arrays, device):
    """Concatenate [S, N, 3] arrays (host or CUDA) to one fp32 device tensor [sum S N, 3]."""
    if not arrays:
        return torch.zeros(0, 3, device=device)
    if all(not torch.is_tensor(a) for a in arrays):
        return torch.from_numpy(np.concatenate([np.asarray(a, dtype=np.float32).reshape(-1, 3) for a in arrays])).to(device)
    return torch.cat([torch.as_tensor(a).to(device=device, dtype=torch.float32).reshape(-1, 3) for a in arrays]).contiguous()


def _expect(a, shape, what):
    if tuple(a.shape) != shape:
        raise ValueError(f'{what}: shape {tuple(a.shape)}, expected {list(shape)}')


class PoseChecks:
    """The tables and device buffers of one ``check_poses`` call: ``launch()`` enqueues the two kernels (one launch each for
    all complexes), ``result()`` copies the outputs to the host once and splits them per complex.  Everything runs on the
    device of the CUDA inputs (else the current device) and on that device's current stream."""

    def __init__(self, graphs, ligand_pos, atom_pos=None, ref_ligand_pos=None, ref_atom_pos=None, ratio=0.75,
                 max_automorphisms=4096, strict=True):
        nc = len(graphs)
        per = [list(x) if x is not None else [None] * nc for x in (ligand_pos, atom_pos, ref_ligand_pos, ref_atom_pos)]
        if any(len(x) != nc for x in per):
            raise ValueError('ligand_pos / atom_pos / ref_ligand_pos / ref_atom_pos: one entry per complex')
        self.device = _device(*per)
        with torch.cuda.device(self.device):
            self._build(graphs, *per, float(ratio), _Tables(max_automorphisms), strict)

    def _build(self, graphs, ligand_pos, atom_pos, ref_ligand_pos, ref_atom_pos, ratio, T, strict):
        dev = self.device
        cplx, pose_complex, lig_ptr, atom_ptr, atom_rows = [], [], [0], [0], []
        entries = []             # RMSD entries: (result key, complex, moved atoms or None, reference rows, auto offset, count)
        self.spans, self.rmsd_errors, self.no_sidechains = [], {}, set()
        for c, g in enumerate(graphs):
            lp, ap = ligand_pos[c], atom_pos[c]
            nl, na = g['ligand'].pos.shape[0], g['atom'].pos.shape[0]
            s = lp.shape[0]
            _expect(lp, (s, nl, 3), f'ligand_pos[{c}]')
            if nl > MAX_ROWS:
                raise ValueError(f'complex {c}: {nl} ligand atoms, more than {MAX_ROWS}')
            if ap is None:
                ap = torch.as_tensor(g['atom'].pos).to(device=dev, dtype=torch.float32)[None].expand(s, na, 3)
            _expect(ap, (s, na, 3), f'atom_pos[{c}]')
            atom_rows.append(ap)
            topo, pk = T.ligand(g), T.pocket(g, c)
            cplx.append([topo['el'], topo['far'], pk['atom'], pk['moved_off'], pk['n_moved'], pk['excl'], pk['n_excl']])
            self.spans.append((len(pose_complex), len(pose_complex) + s))
            pose_complex += [c] * s
            lig_ptr += [lig_ptr[-1] + nl * (k + 1) for k in range(s)]
            atom_ptr += [atom_ptr[-1] + na * (k + 1) for k in range(s)]
            if ref_ligand_pos[c] is not None:
                _expect(ref_ligand_pos[c], (nl, 3), f'ref_ligand_pos[{c}]')
                try:
                    a_off, n_auto = T.automorphisms(topo, f'ligand of complex {c} ({getattr(g, "name", c)})')
                    entries.append(('rmsd', c, None, torch.as_tensor(ref_ligand_pos[c]), a_off, n_auto))
                except ValueError as e:
                    if strict:
                        raise
                    self.rmsd_errors[c] = str(e)
            if ref_atom_pos[c] is not None:
                _expect(ref_atom_pos[c], (na, 3), f'ref_atom_pos[{c}]')
                if pk['moved'] is None:
                    self.no_sidechains.add(c)
                else:
                    ref = torch.as_tensor(ref_atom_pos[c])
                    moved = torch.as_tensor(pk['moved'], dtype=torch.long, device=ref.device)
                    entries.append(('sc_rmsd', c, moved, ref[moved], T.identity(pk['n_moved']), 1))
        self.n_poses = P = len(pose_complex)
        self.max_l = max((g['ligand'].pos.shape[0] for g in graphs), default=0)
        self.max_a = max((g['atom'].pos.shape[0] for g in graphs), default=0)
        self.ratio = ratio
        self.lig = _rows(list(ligand_pos), dev)
        self.atoms = _rows(atom_rows, dev)
        # RMSD rows: the ligand rows of the poses with a reference, the moved side-chain rows of those with a pocket one
        r_complex, r_ptr, ref_off, auto_off, n_auto, rows, refs = [], [0], [], [], [], [], []
        self.entries = []
        for t, (key, c, moved, ref, a_off, na_) in enumerate(entries):
            p0, p1 = self.spans[c]
            if moved is None:
                rows.append(self.lig[lig_ptr[p0]:lig_ptr[p1]])
            else:
                rows.append(self.atoms[atom_ptr[p0]:atom_ptr[p1]].view(p1 - p0, -1, 3)[:, moved.to(dev)].reshape(-1, 3))
            n = len(ref)
            r_complex += [t] * (p1 - p0)
            r_ptr += [r_ptr[-1] + n * (k + 1) for k in range(p1 - p0)]
            ref_off.append(sum(len(r) for r in refs))
            refs.append(ref.to(device=dev, dtype=torch.float32))
            auto_off.append(a_off)
            n_auto.append(na_)
            self.entries.append((key, c, p1 - p0))
        self.R = R = len(r_complex)
        self.rpos = torch.cat(rows).contiguous() if rows else torch.zeros(0, 3, device=dev)
        self.ref = torch.cat(refs).contiguous() if refs else torch.zeros(0, 3, device=dev)
        if max(T.n16, r_ptr[-1], lig_ptr[-1], atom_ptr[-1]) >= 2 ** 31:
            raise ValueError('pose checks: more than 2^31 rows or automorphism entries in one call')
        self.off = {k: T.add(v) for k, v in dict(cplx=np.asarray(cplx, np.int32).reshape(-1, 7), pose_complex=pose_complex,
                                                  lig_ptr=lig_ptr, atom_ptr=atom_ptr, r_complex=r_complex, r_ptr=r_ptr,
                                                  ref_off=ref_off, auto_off=auto_off, n_auto=n_auto).items()}
        self.owner_base = 4 * T.n
        self.ints = torch.from_numpy(np.concatenate(T.ints + T.owners)).to(dev)
        self.autos = torch.from_numpy(np.concatenate(T.autos) if T.autos else np.zeros(2, np.int16)).to(dev)
        self.radius = torch.from_numpy(RADIUS_TABLE).to(dev)
        # outputs: counts [P][3] | min ratios [P][3] | rmsd [R] | automorphism [R], one int32 buffer, one copy back
        self.out = torch.empty(6 * P + 2 * R, dtype=torch.int32, device=dev)

    def _p(self, name):
        return self.ints.data_ptr() + 4 * self.off[name]

    def launch(self):
        """Enqueue the clash screen and the RMSD kernel on the current stream of the device (no synchronisation)."""
        P, R = self.n_poses, self.R
        with torch.cuda.device(self.device):
            L = _lib.lib()
            self.out[:3 * P].zero_()
            self.out[3 * P:6 * P].fill_(0x7f800000)                  # +inf
            base = self.ints.data_ptr()
            if P:
                A = _lib.ClashScreen(
                    n_poses=P, max_lig_atoms=self.max_l, max_atoms=self.max_a, pose_complex=self._p('pose_complex'),
                    lig_pos=_lib.ptr(self.lig), lig_ptr=self._p('lig_ptr'), atom_pos=_lib.ptr(self.atoms),
                    atom_ptr=self._p('atom_ptr'), complexes=self._p('cplx'), lig_type=base, atom_type=base,
                    atom_owner=base + self.owner_base, moved=base, excl=base, far_mask=base, radius=_lib.ptr(self.radius),
                    ratio=self.ratio, count=self.out.data_ptr(), min_ratio=self.out.data_ptr() + 4 * 3 * P)
                _lib.check(L.ddp_clash_screen(A, _lib.stream_ptr()), 'ddp_clash_screen')
            if R:
                _lib.check(L.ddp_pose_rmsd(_lib.ptr(self.rpos), self._p('r_ptr'), self._p('r_complex'), R, _lib.ptr(self.ref),
                                           self._p('ref_off'), _lib.ptr(self.autos), self._p('auto_off'), self._p('n_auto'),
                                           self.out.data_ptr() + 4 * 6 * P, self.out.data_ptr() + 4 * (6 * P + R),
                                           _lib.stream_ptr()), 'ddp_pose_rmsd')

    def result(self):
        """-> one dict per complex of host arrays (see ``check_poses``)."""
        P, R = self.n_poses, self.R
        with torch.cuda.device(self.device):
            host = self.out.cpu().numpy()
        count = host[:3 * P].reshape(P, 3)
        minr = host[3 * P:6 * P].view(np.float32).reshape(P, 3)
        rmsd = host[6 * P:6 * P + R].view(np.float32)
        best = host[6 * P + R:]
        out = []
        for p0, p1 in self.spans:
            d = {}
            for k, name in enumerate(_SETS):
                d[name + '_clashes'] = count[p0:p1, k].copy()
                d[name + '_min_ratio'] = minr[p0:p1, k].copy()
            out.append(d)
        r0 = 0
        for key, c, s in self.entries:
            out[c][key] = rmsd[r0:r0 + s].copy()
            if key == 'rmsd':
                out[c]['rmsd_automorphism'] = best[r0:r0 + s].copy()
            r0 += s
        for c in self.no_sidechains:
            out[c]['sc_rmsd'] = None
        for c, msg in self.rmsd_errors.items():
            out[c]['rmsd_error'] = msg
        return out


def check_poses(graphs, ligand_pos, atom_pos=None, ref_ligand_pos=None, ref_atom_pos=None, ratio=0.75, max_automorphisms=4096,
                strict=True):
    """Pose checks of the samples of several complexes in one launch per kernel.

    ``graphs``: one complex graph per complex (its bond graph, elements, residues and flexible residues are read);
    ``ligand_pos[c]``: [S_c, N_l, 3] poses, ``atom_pos[c]``: [S_c, N_a, 3] pocket atoms of the same poses (None: the
    graph's ``atom.pos`` for every pose); ``ref_ligand_pos[c]`` [N_l, 3] / ``ref_atom_pos[c]`` [N_a, 3]: references (None:
    no RMSD keys).  Arrays may be host arrays or CUDA tensors, all in one frame.  Returns per complex a dict of host arrays
    over its S_c poses: ``{ligand_pocket, sidechain_pocket, ligand_internal}_clashes`` (int32) and ``..._min_ratio``
    (float32, +inf for an empty set); with a ligand reference ``rmsd`` (float32) and ``rmsd_automorphism`` (int32, the
    row of the minimising automorphism, 0 = identity); with a pocket reference ``sc_rmsd`` (float32, None without flexible
    residues).  A ligand with more than ``max_automorphisms`` automorphisms raises ValueError, or with ``strict=False``
    gets no ``rmsd`` keys but ``rmsd_error`` (the message) while the other checks and complexes are unaffected.  More than
    ``MAX_ROWS`` ligand or moved atoms raises ValueError."""
    pc = PoseChecks(graphs, ligand_pos, atom_pos, ref_ligand_pos, ref_atom_pos, ratio, max_automorphisms, strict)
    pc.launch()
    return pc.result()
