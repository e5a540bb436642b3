"""ctypes binding of the C ABI in include/professad_b200.h.

PyTorch is used for device memory, streams and autograd plumbing only: every pointer that crosses
this boundary is a raw ``data_ptr()`` and every entry point is ``extern "C"``.  There is no CPU
fallback: if the library is missing or no CUDA device is visible, calls raise ``RuntimeError``.
"""
import ctypes
import os
import threading

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, 'libprofessad_b200.so')

_c_double_p = ctypes.POINTER(ctypes.c_double)
_vp = ctypes.c_void_p
_int = ctypes.c_int
_dbl = ctypes.c_double
# pad_comm_fn (include/professad_b200.h): int fn(void* user, int op, long long count, void* stream)
COMM_FN = ctypes.CFUNCTYPE(ctypes.c_int, ctypes.c_void_p, ctypes.c_int, ctypes.c_longlong, ctypes.c_void_p)

# name -> (restype, argtypes); must list every symbol include/professad_b200.h declares
SIGNATURES = {
    'pad_version': (ctypes.c_char_p, []),
    'pad_last_error': (ctypes.c_char_p, []),
    'pad_launch_count': (ctypes.c_ulonglong, []),
    'pad_fft_exec_count': (ctypes.c_ulonglong, []),
    'pad_plan_create': (_int, [ctypes.POINTER(_vp), _c_double_p, ctypes.POINTER(_int), _int]),
    'pad_plan_create_slab': (_int, [ctypes.POINTER(_vp), ctypes.POINTER(_dbl), ctypes.POINTER(_int), _int, _int, _int, _vp, _vp, _vp, COMM_FN, _vp]),
    'pad_plan_set_overlap_buffers': (_int, [_vp, _vp, _vp]),
    'pad_slab_fast_elements': (ctypes.c_size_t, [_vp]),
    'pad_plan_set_slab_fast_buffers': (_int, [_vp, ctypes.POINTER(_vp)]),
    'pad_plan_set_slab_peer_buffers': (_int, [_vp, ctypes.POINTER(_vp), _int]),
    'pad_plan_set_slab_peer_recv': (_int, [_vp, ctypes.POINTER(_vp), ctypes.POINTER(_vp), _int]),
    'pad_plan_destroy': (_int, [_vp]),
    'pad_plan_set_box': (_int, [_vp, _c_double_p]),
    'pad_graph_stats': (_int, [ctypes.POINTER(ctypes.c_ulonglong), ctypes.POINTER(ctypes.c_ulonglong)]),
    'pad_plan_workspace_bytes': (ctypes.c_size_t, [_vp]),
    'pad_eval_local': (_int, [_vp, _vp, _vp, _int, _vp, _vp, _int, _vp]),
    'pad_eval_hartree': (_int, [_vp, _vp, _vp, _vp, _int, _vp]),
    'pad_eval_weizsaecker': (_int, [_vp, _vp, _vp, _vp, _int, _vp]),
    'pad_eval_wt': (_int, [_vp, _vp, _dbl, _dbl, _int, _vp, _vp, _int, _vp]),
    'pad_eval_wt_components': (_int, [_vp, _vp, _dbl, _dbl, _vp, _vp, _vp]),
    'pad_eval_wgc99': (_int, [_vp, _vp, _dbl, _dbl, _dbl, _dbl, _vp, _vp, _int, _vp]),
    'pad_eval_pbe': (_int, [_vp, _vp, _int, _vp, _vp, _int, _vp]),
    'pad_eval_semilocal_kinetic': (_int, [_vp, _vp, _int, _dbl, _dbl, _vp, _vp, _int, _vp]),
    'pad_eval_hc': (_int, [_vp, _vp, _int, _dbl, _dbl, _dbl, _dbl, _int, _vp, _int, _vp, _vp, _int, _vp, _vp]),
    'pad_set_fast_fft': (_int, [_int]),
    'pad_set_option': (_int, [ctypes.c_char_p, _int]),
    'pad_dbg_fastmath': (_int, [_vp, ctypes.c_size_t, _dbl, _vp, _vp, _vp]),
    'pad_profile_begin': (_int, []),
    'pad_profile_end': (_int, [ctypes.c_char_p, ctypes.POINTER(ctypes.c_double), _int, ctypes.POINTER(_int), ctypes.POINTER(_int)]),
    'pad_fft_axis_fast': (_int, [_vp, _vp, _int, _int, _vp]),
    'pad_fast_fft_supported': (_int, [_vp]),
    'pad_pipe_supported': (_int, [_vp]),
    'pad_pipe_status': (_int, [_vp, _vp]),
    'pad_rfft3_fast': (_int, [_vp, _vp, _vp, _vp, _vp]),
    'pad_irfft3_fast': (_int, [_vp, _vp, _vp, _vp]),
    'pad_gradient': (_int, [_vp, _vp, _vp, _vp, _vp, _vp]),
    'pad_laplacian': (_int, [_vp, _vp, _vp, _vp]),
    # struct pointers (pad_terms*, pad_denopt_params*, pad_denopt_result*) are passed with ctypes.byref
    'pad_eval_total': (_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    # pad_species* is passed as a ctypes array of _density_opt-style Structures
    'pad_ionic_potential': (_int, [_vp, _vp, _int, _vp, _vp]),
    'pad_ionic_potential_pme': (_int, [_vp, _vp, _int, _int, _vp, _vp]),
    'pad_pme_structure_factor': (_int, [_vp, _vp, _int, _int, _vp, _vp]),
    'pad_ion_forces': (_int, [_vp, _vp, _int, _vp, _vp, _vp]),
    'pad_ion_stress': (_int, [_vp, _vp, _int, _vp, _vp, _int, _vp]),
    'pad_ion_forces_pme': (_int, [_vp, _vp, _int, _int, _vp, _vp, _vp]),
    'pad_ion_stress_pme': (_int, [_vp, _vp, _int, _int, _vp, _vp, _int, _vp]),
    'pad_stress_terms': (_int, [_vp, _vp, _vp, _vp, _vp]),
    'pad_ion_ion_work_doubles': (ctypes.c_size_t, [_c_double_p, _int, _dbl]),
    'pad_ion_ion': (_int, [_c_double_p, _vp, _vp, _int, _dbl, _dbl, _dbl, _vp, _vp, _vp, _vp, _int, _vp]),
    'pad_chi_to_density': (_int, [_vp, _vp, _dbl, _vp, _vp]),
    'pad_chi_project': (_int, [_vp, _vp, _vp, _vp, _dbl, _vp, _vp, _vp]),
    'pad_denopt_create': (_int, [ctypes.POINTER(_vp), _vp, _vp, _vp]),
    'pad_denopt_run': (_int, [_vp, _vp, _vp, _vp, _vp, _vp]),
    'pad_denopt_destroy': (_int, [_vp]),
}

PART_TF, PART_VW, PART_NL, PART_ALL = 1, 2, 4, 7
LOCAL_TF, LOCAL_LDAX, LOCAL_PZC, LOCAL_IONEL = 1, 2, 4, 8
SEMILOCAL_LKT, SEMILOCAL_PG = 0, 1

_lib = None
_lock = threading.Lock()


def load_library():
    """Load (building first if the sources are newer) the shared library and declare signatures."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is not None:
            return _lib
        if not os.path.exists(LIB_PATH):
            from . import build as _build
            _build.build()
        lib = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)       # AttributeError here = header/library mismatch
            fn.restype = res
            fn.argtypes = args
        for env, opt in (('PAD_FAST_FFT', b'fast_fft'), ('PAD_OWN_XY', b'own_xy'), ('PAD_PIPE', b'pipe'),
                         ('PAD_PIPE_LPI', b'pipe_lpi'), ('PAD_PIPE_TPI', b'pipe_tpi'), ('PAD_FUSE_TERMS', b'fuse_terms'),
                         ('PAD_ZINV_STREAM', b'zinv_stream'), ('PAD_FUSE_MID', b'fuse_mid'), ('PAD_FOLD_TABLE', b'fold_table'),
                         ('PAD_GRAPHS', b'graphs'), ('PAD_YWIDE', b'ywide'), ('PAD_XONE', b'xone'), ('PAD_PBE_FAST', b'pbe_fast'), ('PAD_LOCAL_TAIL', b'local_tail')):
            if os.environ.get(env, '').lstrip('-').isdigit():
                lib.pad_set_option(opt, int(os.environ[env]))
        _lib = lib
    return _lib


def check(rc):
    if rc != 0:
        raise RuntimeError('professad_b200: ' + load_library().pad_last_error().decode())


def require_cuda(t, what='den'):
    if not isinstance(t, torch.Tensor) or t.device.type != 'cuda':
        dev = getattr(t, 'device', type(t).__name__)
        raise RuntimeError(
            f'professad_b200: `{what}` must be a CUDA tensor (got {dev}). This build runs the functional '
            'kernels on a B200 only; there is no CPU fallback.')
    if t.dtype != torch.double:
        raise TypeError(f'professad_b200: `{what}` must be torch.double (got {t.dtype})')


def stream_ptr(device):
    return ctypes.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def ptr(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else ctypes.c_void_p(0)


class Plan:
    """Owns one ``pad_plan`` (cuFFT plans, scratch fields, cached kernels) for (shape, device)."""

    def __init__(self, box_host, shape, device_index):
        self.lib = load_library()
        self.shape = tuple(int(s) for s in shape)
        self.device_index = device_index
        self.handle = _vp()
        self.box = None
        box_arr = (ctypes.c_double * 9)(*box_host)
        shp = (ctypes.c_int * 3)(*self.shape)
        check(self.lib.pad_plan_create(ctypes.byref(self.handle), box_arr, shp, device_index))
        self.box = tuple(box_host)
        self._set_geometry()

    def _set_geometry(self):
        b = self.box
        det = (b[0] * (b[4] * b[8] - b[5] * b[7]) - b[1] * (b[3] * b[8] - b[5] * b[6])
               + b[2] * (b[3] * b[7] - b[4] * b[6]))
        self.vol = abs(det)
        self.npts = self.shape[0] * self.shape[1] * self.shape[2]
        self.dV = self.vol / self.npts

    def set_box(self, box_host):
        box_host = tuple(box_host)
        if box_host != self.box:
            check(self.lib.pad_plan_set_box(self.handle, (ctypes.c_double * 9)(*box_host)))
            self.box = box_host
            self._set_geometry()

    def workspace_bytes(self):
        return int(self.lib.pad_plan_workspace_bytes(self.handle))

    def close(self):
        if self.handle:
            self.lib.pad_plan_destroy(self.handle)
            self.handle = _vp()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


_plans = {}
_box_cache = {}


def box_to_host(box_vecs):
    """9 host floats for a (3,3) lattice tensor.  The device->host copy (a sync) happens once per
    tensor version: the cache holds a reference, so the address cannot be recycled under us."""
    key = (box_vecs.data_ptr(), box_vecs._version, box_vecs.device)
    hit = _box_cache.get(key)
    if hit is not None and hit[0] is box_vecs:
        return hit[1]
    if box_vecs.shape != (3, 3):
        raise ValueError('box_vecs must have shape (3, 3)')
    host = tuple(box_vecs.detach().double().cpu().reshape(-1).tolist())
    if len(_box_cache) > 64:
        _box_cache.clear()
    _box_cache[key] = (box_vecs, host)
    return host


def get_plan(box_vecs, den):
    """Plan for (den.shape, den.device), with its lattice updated to ``box_vecs``.  Inside a
    ``parallel.slab(...)`` context: the rank's slab plan of the global grid."""
    require_cuda(den)
    if den.dim() != 3:
        raise ValueError('den must be a 3-D grid')
    from . import parallel
    ctx = parallel.current()
    if ctx is not None:
        return ctx.plan_for(box_vecs, den)
    dev = den.device.index if den.device.index is not None else torch.cuda.current_device()
    key = (tuple(den.shape), dev)
    host = box_to_host(box_vecs)
    plan = _plans.get(key)
    if plan is None:
        plan = Plan(host, den.shape, dev)
        _plans[key] = plan
    else:
        plan.set_box(host)
    return plan


def release_plans():
    """Free every cached plan (device scratch, cuFFT plans)."""
    for p in _plans.values():
        p.close()
    _plans.clear()
    _box_cache.clear()
