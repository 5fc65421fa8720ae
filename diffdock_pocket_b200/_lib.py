"""ctypes binding of ``libddp_b200.so`` (the C ABI declared in ``include/ddp_b200.h``).

There is no CPU fallback: if the shared library is missing or a call returns non-zero the caller
gets an exception.  ``build()`` compiles the CUDA sources in-tree for sm_100a with nvcc.
"""
import ctypes as C
import os
import subprocess

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
SO_PATH = os.environ.get('DDP_LIB', os.path.join(_HERE, 'libddp_b200.so'))     # DDP_LIB: A/B runs of two builds
CSRC = os.path.join(_HERE, 'csrc')
SOURCES = ['graph.cu', 'embed.cu', 'tpconv_fp32.cu', 'tpconv_umma.cu', 'tpconv_bwd.cu', 'pose.cu', 'capi.cu']
NVCC_FLAGS = ['-gencode', 'arch=compute_100a,code=sm_100a', '-lineinfo', '-O3', '-std=c++17',
              '-Xcompiler', '-fPIC', '-shared']

i32, f32, vp = C.c_int32, C.c_float, C.c_void_p


class EdgeMlp(C.Structure):
    _fields_ = [('w_pre', vp), ('w_rbf', vp), ('w2', vp), ('b2', vp), ('b1', vp), ('rbf_offset', vp),
                ('rbf_coeff', f32), ('n_pre', i32), ('n_rbf', i32), ('ns', i32), ('sh_dim', i32)]


class TpGroup(C.Structure):
    _fields_ = [('d1', i32), ('d2', i32), ('d_out', i32), ('x_off', i32), ('mul_in', i32), ('sh_off', i32),
                ('w_off', i32), ('out_off', i32), ('mul_out', i32), ('c_off', i32)]


class TpConv(C.Structure):
    _fields_ = [('w1t', vp), ('b1', vp), ('w2t', vp), ('b2', vp), ('k1', i32), ('hid', i32), ('w_numel', i32),
                ('n_emb', i32), ('ns', i32), ('groups', vp), ('ctab', vp), ('ctab_len', i32), ('col_group', vp),
                ('n_groups', i32), ('f_in', i32), ('f_out', i32), ('sh_dim', i32)]


class TpEdges(C.Structure):
    _fields_ = [('emb', vp), ('p1', vp), ('i1', vp), ('ld1', i32), ('p2', vp), ('i2', vp), ('ld2', i32),
                ('x', vp), ('gather', vp), ('ldx', i32), ('sh', vp), ('agg', vp), ('ew', vp),
                ('n_edges_dev', vp), ('edge_cap', i32), ('out_scale', vp), ('agg_deg', vp)]


class Update(C.Structure):
    _fields_ = [('sum', vp), ('deg', vp), ('scale', vp), ('shift', vp), ('n_edges_dev', vp)]


class NodeUpdateJob(C.Structure):
    _fields_ = [('old_x', vp), ('f_old', i32), ('ld_old', i32), ('updates', Update * 4), ('n_updates', i32), ('n', i32),
                ('f_new', i32), ('new_x', vp), ('ld_new', i32)]


class DegreeJob(C.Structure):
    _fields_ = [('idx', vp), ('n_edges_dev', vp), ('edge_cap', i32), ('start', i32), ('deg', vp)]


class MlpLayer(C.Structure):
    _fields_ = [('wt', vp), ('b', vp), ('n_in', i32), ('n_out', i32), ('act', i32)]


class FtpPath(C.Structure):
    _fields_ = [('in_off', i32), ('d_in', i32), ('out_off', i32), ('d_out', i32), ('c_off', i32)]


class StepCoef(C.Structure):
    _fields_ = [(k, f32) for k in ('a_tr', 'b_tr', 'a_rot', 'b_rot', 'a_tor', 'b_tor', 'a_sc', 'b_sc')]


class Pose(C.Structure):
    _fields_ = [('n_samples', i32), ('lig_pos', vp), ('lig_ptr', vp), ('tor_ptr', vp), ('tor_bonds', vp),
                ('mask_rotate', vp), ('mask_ptr', vp), ('atom_pos', vp), ('sc_ptr', vp), ('sc_bonds', vp),
                ('sc_sub_ptr', vp), ('sc_sub', vp), ('tr_score', vp), ('rot_score', vp), ('tor_score', vp),
                ('sc_score', vp), ('tr_z', vp), ('rot_z', vp), ('tor_z', vp), ('sc_z', vp)]


_SIGS = {
    'ddp_version': (C.c_char_p, []),
    'ddp_radius': (i32, [vp, vp, vp, vp, i32, i32, vp, f32, i32, i32, i32, vp, i32, vp, vp, i32, vp, vp]),
    'ddp_knn_graph': (i32, [vp, vp, i32, i32, i32, vp, i32, vp, vp, i32, vp, vp]),
    'ddp_knn_set_grid': (i32, [i32]),
    'ddp_calpha_graph': (i32, [vp, vp, i32, i32, f32, i32, vp, i32, vp, vp, i32, vp, vp]),
    'ddp_degree': (i32, [vp, vp, i32, vp, vp]),
    'ddp_edge_embed': (i32, [vp, vp, vp, i32, vp, vp, vp, i32, vp, C.POINTER(EdgeMlp), vp, vp, vp]),
    'ddp_graph_sigma_proj': (i32, [vp, i32, f32, vp, i32, vp, vp, i32, i32, vp, vp, vp]),
    'ddp_node_init': (i32, [vp, vp, vp, i32, i32, vp, i32, vp]),
    'ddp_node_static_embed': (i32, [vp, i32, i32, vp, vp, vp, i32, vp, vp, i32, vp, vp]),
    'ddp_tpconv_fp32': (i32, [C.POINTER(TpConv), C.POINTER(TpEdges), vp, vp]),
    'ddp_tpconv_pack': (C.c_int64, [C.POINTER(TpConv), C.POINTER(TpGroup), vp, vp, vp, vp, vp, i32, vp]),
    'ddp_tpconv_umma': (i32, [C.POINTER(TpConv), vp, i32, C.POINTER(TpEdges), vp, vp]),
    'ddp_tpconv_umma_group': (i32, [vp, vp, i32, vp, vp, i32, vp]),
    'ddp_tpconv_umma_set_trace': (i32, [vp]),
    'ddp_tp_backward': (i32, [C.POINTER(TpConv), i32, vp, vp, i32, vp, vp, vp, i32, vp, vp, vp, vp]),
    'ddp_node_update': (i32, [vp, i32, i32, C.POINTER(Update), i32, i32, i32, vp, i32, vp]),
    'ddp_node_update_multi': (i32, [C.POINTER(NodeUpdateJob), i32, vp]),
    'ddp_degree_multi': (i32, [C.POINTER(DegreeJob), i32, vp]),
    'ddp_segment_mean': (i32, [vp, vp, vp, i32, i32, i32, vp, i32, vp]),
    'ddp_bond_geometry': (i32, [vp, vp, i32, vp, i32, i32, vp, vp, vp, vp]),
    'ddp_tor_edge_sh': (i32, [vp, i32, vp, vp, vp, vp, i32, vp, vp]),
    'ddp_tor_edge_sh_generic': (i32, [vp, i32, vp, C.POINTER(FtpPath), i32, vp, vp, vp, i32, vp, i32, vp]),
    'ddp_row_mlp': (i32, [vp, i32, i32, C.POINTER(MlpLayer), i32, vp, vp, i32, vp]),
    'ddp_tr_rot_head': (i32, [vp, vp, i32, i32, vp, vp, vp, vp, vp, vp, vp, vp, i32, vp, vp, vp, vp, vp]),
    'ddp_pose_update': (i32, [C.POINTER(Pose), C.POINTER(StepCoef), vp]),
    'ddp_pose_max_ligand_atoms': (i32, []),
    'ddp_pose_update_dev': (i32, [C.POINTER(Pose), vp, vp]),
    # deterministic mode (fixed-point accumulation, DDP_ACC_FIXED_SHIFT)
    'ddp_fixed_to_float': (i32, [vp, C.c_int64, vp, vp]),
    'ddp_tpconv_fp32_fixed': (i32, [C.POINTER(TpConv), C.POINTER(TpEdges), vp, vp, vp]),
    'ddp_tpconv_umma_fixed': (i32, [C.POINTER(TpConv), vp, i32, C.POINTER(TpEdges), vp, vp, vp]),
    'ddp_tpconv_umma_group_fixed': (i32, [vp, vp, i32, vp, vp, i32, vp, vp]),
    'ddp_tp_backward_fixed': (i32, [C.POINTER(TpConv), i32, vp, vp, i32, vp, vp, vp, i32, vp, vp, vp, vp, vp]),
    'ddp_node_update_fixed': (i32, [vp, i32, i32, C.POINTER(Update), i32, i32, i32, vp, i32, vp]),
    'ddp_node_update_multi_fixed': (i32, [C.POINTER(NodeUpdateJob), i32, vp]),
}
EXPORTS = sorted(_SIGS)
_LIB = None
# kernels launched per C-ABI call (for the bench's gpu_launches claim)
KERNELS_PER_CALL = {'ddp_radius': 3, 'ddp_knn_graph': 3, 'ddp_calpha_graph': 3, 'ddp_version': 0, 'ddp_pose_max_ligand_atoms': 0, 'ddp_tpconv_pack': 0, 'ddp_tpconv_umma_set_trace': 0, 'ddp_knn_set_grid': 0}
COUNTS = {}


def launch_count():
    return sum(n * KERNELS_PER_CALL.get(k, 1) for k, n in COUNTS.items())


# While a list is installed here every C call is also appended to it as (name, fn, args): the score model records the
# launch sequence of a resident plan once and replays it on later steps without re-marshalling ~60 descriptors
# (all_atom_score_model.launch_plan).
RECORD = None


class _Counted:
    def __init__(self, name, fn):
        self.name, self.fn = name, fn

    def __call__(self, *a):
        COUNTS[self.name] = COUNTS.get(self.name, 0) + 1
        if RECORD is not None and KERNELS_PER_CALL.get(self.name, 1) > 0:     # launches only (not ddp_tpconv_pack & co.)
            RECORD.append((self.name, self.fn, a))
        return self.fn(*a)


class _Lib:
    pass


def build(verbose=False):
    """Compile every CUDA source in-tree for sm_100a (nvcc cross-compiles without a GPU)."""
    srcs = [os.path.join(CSRC, s) for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]
    newest = max(os.path.getmtime(p) for p in srcs + [os.path.join(CSRC, 'ddp_common.cuh'),
                                                     os.path.join(_HERE, '..', 'include', 'ddp_b200.h')]
                 + [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith('.cuh')])
    if os.path.exists(SO_PATH) and os.path.getmtime(SO_PATH) >= newest:
        return SO_PATH
    cmd = ['nvcc'] + NVCC_FLAGS + os.environ.get('DDP_NVCC_FLAGS', '').split() + srcs + ['-o', SO_PATH]
    if verbose:
        print(' '.join(cmd))
    subprocess.check_call(cmd)
    return SO_PATH


def lib():
    global _LIB
    if _LIB is None:
        if not os.path.exists(SO_PATH):
            raise RuntimeError(f'{SO_PATH} is missing: run `python -c "import __graft_entry__ as g; g.build()"` '
                               '(there is no CPU fallback for the ddp_b200 kernels)')
        dll = C.CDLL(SO_PATH)
        L = _Lib()
        for name, (res, args) in _SIGS.items():
            fn = getattr(dll, name)
            fn.restype, fn.argtypes = res, args
            setattr(L, name, _Counted(name, fn))
        L.dll = dll
        _LIB = L
    return _LIB


def check(status, what):
    if status != 0:
        raise RuntimeError(f'{what} failed with status {status}')


def ptr(t):
    """Device pointer of a tensor (or NULL)."""
    if t is None:
        return None
    assert t.is_contiguous(), 'non-contiguous tensor passed to the C ABI'
    return t.data_ptr()


def stream_ptr():
    return torch.cuda.current_stream().cuda_stream


# ------------------------------------------------------------------------------------------ deterministic mode
FIXED_SHIFT = 32                  # DDP_ACC_FIXED_SHIFT (include/ddp_b200.h)
STATUS_FIXED_RANGE = 1            # DDP_STATUS_FIXED_RANGE


def deterministic():
    """The accumulation mode callers get: fixed point (bitwise reproducible) under
    ``torch.use_deterministic_algorithms(True)`` (also with ``warn_only=True``), fp32 atomics otherwise."""
    return torch.are_deterministic_algorithms_enabled()


def sum_dtype(det):
    return torch.int64 if det else torch.float32


_STATUS = {}


def _cuda_device(device):
    device = torch.device(device)
    return torch.device('cuda', torch.cuda.current_device()) if device.index is None else device


def status_word(device):
    """The sticky device status word of the fixed-point kernels on ``device`` (one int32 per device, allocated once, so
    recorded launch sequences and captured graphs may hold its address)."""
    device = _cuda_device(device)
    w = _STATUS.get(device)
    if w is None:
        w = _STATUS[device] = torch.zeros(1, dtype=torch.int32, device=device)
    return w


def check_status(device, value=None):
    """Read (and clear) the status word after a synchronisation: raises RuntimeError if a fixed-point accumulation saw a
    non-finite partial sum or one outside the representable range since the last check.  ``value``: the word's content
    already copied to the host with the results (otherwise it is read here).  The word is cleared before the exception,
    so the next call on the same device starts clean."""
    w = _STATUS.get(_cuda_device(device))
    if w is None:
        return
    v = int(w.item()) if value is None else int(value)
    if v:
        w.zero_()
        raise RuntimeError('deterministic accumulation: a partial sum was not finite or outside the fixed-point range '
                           f'(|v| < 2^{63 - FIXED_SHIFT}); status word 0x{v:x}')
