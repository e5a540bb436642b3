"""Binding of the fused evaluator and the device-resident density optimiser
(pad_eval_total / pad_chi_project / pad_denopt_* in include/professad_b200.h).

``describe_terms`` turns a reference-style ``terms`` list (callables dispatched on by name,
system.py:759-772) into one ``pad_terms`` descriptor when every term is a native functional;
otherwise it returns ``None`` and System uses the generic autograd closure.
"""
import ctypes

import torch

from . import _native
from ._native import check, ptr, stream_ptr


class PadTerms(ctypes.Structure):
    _fields_ = [('local_mask', ctypes.c_int), ('hartree', ctypes.c_int), ('kinetic', ctypes.c_int),
                ('kinetic_parts', ctypes.c_int), ('pbe', ctypes.c_int),
                ('alpha', ctypes.c_double), ('beta', ctypes.c_double), ('gamma', ctypes.c_double),
                ('kappa', ctypes.c_double),
                ('hc_variant', ctypes.c_int), ('hc_geometric', ctypes.c_int), ('hc_n_eta', ctypes.c_int),
                ('hc_p0', ctypes.c_double), ('hc_p1', ctypes.c_double), ('hc_table_dev', ctypes.c_void_p),
                ('sl_variant', ctypes.c_int), ('sl_p0', ctypes.c_double), ('sl_p1', ctypes.c_double)]


class PadDenoptParams(ctypes.Structure):
    _fields_ = [('n_elec', ctypes.c_double), ('ntol', ctypes.c_double), ('n_conv_cond_count', ctypes.c_int),
                ('method', ctypes.c_int), ('step_size', ctypes.c_double), ('n_maxiter', ctypes.c_int),
                ('conv_target', ctypes.c_int), ('history', ctypes.c_int), ('max_iter', ctypes.c_int),
                ('tolerance_grad', ctypes.c_double), ('tolerance_change', ctypes.c_double)]


class PadDenoptResult(ctypes.Structure):
    _fields_ = [('iterations', ctypes.c_int), ('converged', ctypes.c_int), ('closures', ctypes.c_int),
                ('energy', ctypes.c_double), ('last_dE_eV', ctypes.c_double), ('last_dEdchi', ctypes.c_double),
                ('last_euler', ctypes.c_double)]


_vp = ctypes.c_void_p


def describe_terms(terms, device=None):
    """pad_terms for a list of native functionals (IonIon is skipped, as in the density optimisation),
    or None if a term is not native or the combination is not representable.  ``device``: the CUDA device the
    described terms will be evaluated on (tables that travel as raw pointers are moved there); default: current."""
    T = PadTerms()
    for f in terms:
        name = getattr(f, '__qualname__', '') or getattr(f, '__name__', '')
        if name == 'IonIon':
            continue
        spec = getattr(f, '_pad_term', None)
        owner = getattr(f, '__self__', None)
        if spec is None and owner is not None:
            maker = getattr(owner, '_pad_term_of', None)
            spec = maker(device) if maker is not None else None
        if spec is None:
            return None
        kind = spec[0]
        if kind == 'local':
            if T.local_mask & spec[1]:
                return None
            T.local_mask |= spec[1]
        elif kind == 'hartree':
            if T.hartree:
                return None
            T.hartree = 1
        elif kind == 'pbe':
            if T.pbe & spec[1]:
                return None
            T.pbe |= spec[1]
        elif kind == 'wt':
            if T.kinetic:
                return None
            T.kinetic, T.alpha, T.beta, T.kinetic_parts = 1, spec[1], spec[2], spec[3]
        elif kind == 'wgc99':
            if T.kinetic:
                return None
            T.kinetic = 2
            T.alpha, T.beta, T.gamma, T.kappa = spec[1:5]
        elif kind == 'hc':
            if T.kinetic:
                return None
            T.kinetic = 3
            _, T.hc_variant, T.hc_p0, T.hc_p1, T.beta, T.kappa, T.hc_geometric, table = spec
            T.hc_n_eta = int(table.shape[1])
            T.hc_table_dev = table.data_ptr()
            T._keep = table             # the descriptor holds a raw device pointer: keep the tensor alive with it
        elif kind == 'semilocal':
            if T.kinetic:
                return None
            T.kinetic = 4
            T.sl_variant, T.sl_p0, T.sl_p1 = spec[1:4]
        else:
            return None
    if not (T.local_mask or T.hartree or T.kinetic or T.pbe):
        return None
    return T


def eval_total(box_vecs, den, v_ext, T, want_potential=True):
    """E (0-dim device tensor) and total dE/dn of a described term list, one C-ABI call."""
    _native.require_cuda(den)
    den = den.detach().contiguous()
    plan = _native.get_plan(box_vecs, den)
    E = torch.empty((), dtype=torch.double, device=den.device)
    v = torch.empty_like(den) if want_potential else None
    vx = v_ext.detach().contiguous() if v_ext is not None else None
    check(plan.lib.pad_eval_total(plan.handle, ctypes.byref(T), ptr(den), ptr(vx), ptr(E), ptr(v),
                                  stream_ptr(den.device)))
    return E, v


def stress_terms(box_vecs, den, T):
    """Analytic stress (3, 3) in Ha/bohr^3 of a described term list without its IonElectron part (pad_stress_terms)."""
    _native.require_cuda(den)
    den = den.detach().contiguous()
    plan = _native.get_plan(box_vecs, den)
    out = torch.empty(9, dtype=torch.double, device=den.device)
    check(plan.lib.pad_stress_terms(plan.handle, ctypes.byref(T), ptr(den), ptr(out), stream_ptr(den.device)))
    return out.reshape(3, 3)


def chi_to_density(box_vecs, chi, n_elec):
    chi = chi.detach().contiguous()
    plan = _native.get_plan(box_vecs, chi)
    den = torch.empty_like(chi)
    check(plan.lib.pad_chi_to_density(plan.handle, ptr(chi), float(n_elec), ptr(den), stream_ptr(chi.device)))
    return den


def chi_project(box_vecs, chi, den, v, n_elec):
    """dE/dchi_ijk (autograd convention) and [|g|_1, g.g, max|dE/dchi|, max|mu - v|] on the device."""
    chi = chi.detach().contiguous()
    plan = _native.get_plan(box_vecs, chi)
    g = torch.empty_like(chi)
    stats = torch.empty(4, dtype=torch.double, device=chi.device)
    check(plan.lib.pad_chi_project(plan.handle, ptr(chi), ptr(den.contiguous()), ptr(v.contiguous()), float(n_elec),
                                   ptr(g), ptr(stats), stream_ptr(chi.device)))
    return g, stats


CONV_TARGETS = {'dE': 0, 'dEdchi': 1, 'euler': 2}
METHODS = {'LBFGS': 0, 'TPGD': 1}


def run(box_vecs, den, v_ext, T, n_elec, ntol, n_conv_cond_count, n_method, n_step_size, n_maxiter, conv_target):
    """Device-resident optimize_density.  ``den`` is replaced by the optimised density (in place).
    Returns (result dict, trace tensor (iterations, 4))."""
    _native.require_cuda(den)
    assert den.is_contiguous()
    plan = _native.get_plan(box_vecs, den)
    n_maxiter = int(round(n_maxiter))
    prm = PadDenoptParams(float(n_elec), float(ntol), int(n_conv_cond_count), METHODS[n_method], float(n_step_size),
                          n_maxiter, CONV_TARGETS[conv_target], 8, 6, 1e-5, 1e-9)
    handle = _vp()
    check(plan.lib.pad_denopt_create(ctypes.byref(handle), plan.handle, ctypes.byref(T), ctypes.byref(prm)))
    try:
        res = PadDenoptResult()
        trace = torch.zeros((max(n_maxiter, 1), 4), dtype=torch.double).pin_memory()
        vx = v_ext.detach().contiguous() if v_ext is not None else None
        check(plan.lib.pad_denopt_run(handle, ptr(den), ptr(vx), ctypes.byref(res), ctypes.c_void_p(trace.data_ptr()),
                                      stream_ptr(den.device)))
    finally:
        plan.lib.pad_denopt_destroy(handle)
    out = {'iterations': res.iterations, 'converged': bool(res.converged), 'closures': res.closures,
           'energy': res.energy, 'dE_eV': res.last_dE_eV, 'dEdchi': res.last_dEdchi, 'euler': res.last_euler}
    return out, trace[:res.iterations].clone()
