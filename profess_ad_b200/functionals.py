"""Energy functionals with the reference's names and call contract (src/professad/functionals.py):

    f(box_vecs, den) -> scalar energy tensor [Hartree],  differentiable w.r.t. ``den`` by autograd
    IonElectron(box_vecs, den, v_ext)

Each functional is ONE C-ABI call that produces the energy and, when ``den.requires_grad``, the
analytic potential dE/dn in the same pass; ``backward`` just scales the stored potential by
``grad_out * dV`` (autograd's dE/dn_ijk is the un-normalised partial: callers divide by dV,
system.py:434-435, functional_tools.py:31).  Differentiation w.r.t. ``box_vecs`` (stress) and
double-backward are not part of this path and raise.
"""
import ctypes
import math

import numpy as np
import torch

from . import _native
from ._native import check, ptr, stream_ptr

J_per_Ha = 4.3597447222071e-18
eV_per_Ha = J_per_Ha / 1.602176634e-19


# ----------------------------------------------------------------------------------------------
#  autograd plumbing
# ----------------------------------------------------------------------------------------------
class _NativeEnergy(torch.autograd.Function):
    """forward: E = launch(plan, den, E_ptr, v_ptr); backward: grad_out * v * dV."""

    @staticmethod
    def forward(ctx, den, box_vecs, launch, extra):
        _native.require_cuda(den)
        if box_vecs.requires_grad:
            raise NotImplementedError('professad_b200: derivatives w.r.t. box_vecs (stress) are not on the B200 '
                                      'hot path; use the reference for cell derivatives')
        d = den.detach()
        if not d.is_contiguous():
            d = d.contiguous()
        if d.data_ptr() % 16:           # views at odd offsets: cuFFT operands need 16-byte alignment
            d = d.clone()
        plan = _native.get_plan(box_vecs, d)
        need_v = ctx.needs_input_grad[0]
        E = torch.empty((), dtype=torch.double, device=d.device)
        v = torch.empty_like(d) if need_v else None
        launch(plan, d, extra, E, v, stream_ptr(d.device))
        ctx.dV = plan.dV
        if need_v:
            ctx.save_for_backward(v)
        return E

    @staticmethod
    @torch.autograd.function.once_differentiable      # the potential is a constant here: a second derivative must raise,
    def backward(ctx, grad_out):                      # not silently drop the native terms (create_graph=True)
        (v,) = ctx.saved_tensors
        return v * (grad_out * ctx.dV), None, None, None


def _evaluate(box_vecs, den, launch, extra=None):
    return _NativeEnergy.apply(den, box_vecs, launch, extra)


def energy_and_potential(box_vecs, den, functional):
    """Convenience: (E, delta E/delta n) of a native or user functional in one go."""
    d = den.detach().clone().requires_grad_(True)
    E = functional(box_vecs, d)
    (g,) = torch.autograd.grad(E, d)
    dV = torch.abs(torch.linalg.det(box_vecs)) / den.numel()
    return E.detach(), g / dV


# ----------------------------------------------------------------------------------------------
#  ion / electron terms
# ----------------------------------------------------------------------------------------------
def IonIon():
    """Ion-ion interaction marker (functionals.py:21-28).  Dispatched on by name in System."""
    return None


def _launch_local(terms):
    def launch(plan, den, v_ext, E, v, stream):
        check(plan.lib.pad_eval_local(plan.handle, ptr(den), ptr(v_ext), terms, ptr(E), ptr(v), 0, stream))
    return launch


_L_IONEL = _launch_local(_native.LOCAL_IONEL)
_L_TF = _launch_local(_native.LOCAL_TF)
_L_LDAX = _launch_local(_native.LOCAL_LDAX)
_L_PZC = _launch_local(_native.LOCAL_PZC)
_L_PZ = _launch_local(_native.LOCAL_LDAX | _native.LOCAL_PZC)


def IonElectron(box_vecs, den, v_ext):
    """U = int n v_ext (functionals.py:31-46)."""
    _native.require_cuda(v_ext, 'v_ext')
    return _evaluate(box_vecs, den, _L_IONEL, v_ext.detach().contiguous())


def Hartree(box_vecs, den):
    """Hartree energy (functionals.py:49-72): 2 FFTs, Coulomb multiply fused in reciprocal space."""
    def launch(plan, d, _, E, v, stream):
        check(plan.lib.pad_eval_hartree(plan.handle, ptr(d), ptr(E), ptr(v), 0, stream))
    return _evaluate(box_vecs, den, launch)


# ----------------------------------------------------------------------------------------------
#  kinetic functionals
# ----------------------------------------------------------------------------------------------
class KineticFunctional(torch.nn.Module):
    """Template class (functionals.py:83-200).  Only what the hot path needs is kept: parameter
    storage and device handling.  The ML-training helpers of the reference are out of scope."""

    def __init__(self, init_args=None):
        super().__init__()
        self.init_args = init_args
        self.device = torch.device('cpu')

    def initialize(self):
        self.param_grad(False)

    def set_device(self, device=None):
        self.device = torch.device('cuda') if device is None else device
        for p in self.parameters():
            p.data = p.data.to(self.device)

    def param_grad(self, requires_grad=True):
        for p in self.parameters():
            p.requires_grad_(requires_grad)


def ThomasFermi(box_vecs, den):
    """T_TF = int (3/10)(3 pi^2)^(2/3) n^(5/3) (functionals.py:207-224)."""
    return _evaluate(box_vecs, den, _L_TF)


def _launch_wt(alpha, beta, parts):
    def launch(plan, d, _, E, v, stream):
        check(plan.lib.pad_eval_wt(plan.handle, ptr(d), alpha, beta, parts, ptr(E), ptr(v), 0, stream))
    return launch


_L_VW = _launch_wt(1.0, 1.0, _native.PART_VW)


def Weizsaecker(box_vecs, den):
    """T_vW = int |grad n|^2 / (8 n) evaluated as -1/2 int sqrt(n) lap sqrt(n) (functionals.py:227-246)."""
    return _evaluate(box_vecs, den, _L_VW)


def G_inv_lind_analytical(eta):
    """functionals.py:617-618"""
    return 0.5 + ((1 - eta.pow(2)) / (4 * eta)) * torch.log(torch.abs((1 + eta) / (1 - eta)))


def G_inv_lind(eta):
    """functionals.py:621-628"""
    out = torch.where((eta == 0) | (eta == 1), torch.ones_like(eta), G_inv_lind_analytical(eta))
    return torch.where(eta == 1, torch.full_like(eta, 0.5), out)


def G_inv_lindhard(box_vecs, den):
    """functionals.py:631-639 (compatibility helper; the kernels evaluate the Lindhard function on the fly)."""
    from .functional_tools import wavevecs
    kx, ky, kz, k2 = wavevecs(box_vecs, den.shape)
    vol = torch.abs(torch.linalg.det(box_vecs))
    n0 = (torch.mean(den) * vol).item() / vol
    k_F = (3 * np.pi * np.pi * n0).pow(1 / 3)
    eta = torch.sqrt(k2) / (2 * k_F)
    return eta, G_inv_lind(eta)


def non_local_KEF(box_vecs, den, alpha, beta):
    """Non-local part of a Wang-Teter style functional (functionals.py:644-652)."""
    return _evaluate(box_vecs, den, _launch_wt(float(alpha), float(beta), _native.PART_NL))


_A98 = (5 + math.sqrt(5)) / 6
_B98 = (5 - math.sqrt(5)) / 6
_L_WT = _launch_wt(5 / 6, 5 / 6, _native.PART_ALL)
_L_PERROT = _launch_wt(1.0, 1.0, _native.PART_ALL)
_L_SM = _launch_wt(0.5, 0.5, _native.PART_ALL)
_L_WGC98 = _launch_wt(_A98, _B98, _native.PART_ALL)


def WangTeter(box_vecs, den):
    """Wang-Teter functional, (alpha, beta) = (5/6, 5/6) (functionals.py:655-670): 4 FFTs."""
    return _evaluate(box_vecs, den, _L_WT)


def Perrot(box_vecs, den):
    """Perrot functional, (1, 1) (functionals.py:673-689)."""
    return _evaluate(box_vecs, den, _L_PERROT)


def SmargiassiMadden(box_vecs, den):
    """Smargiassi-Madden functional, (1/2, 1/2) (functionals.py:692-707)."""
    return _evaluate(box_vecs, den, _L_SM)


def WangGovindCarter98(box_vecs, den):
    """WGC98, ((5+sqrt5)/6, (5-sqrt5)/6) (functionals.py:710-725): 6 FFTs."""
    return _evaluate(box_vecs, den, _L_WGC98)


class WangTeterStyleFunctional(KineticFunctional):
    """vW + TF * f(T_NL / f'(0) / TF) with user (alpha, beta, f) (functionals.py:728-782).

    ``f`` is an arbitrary Python callable, so its value and derivative are taken on the host from the
    three component energies (one small device->host read per call)."""

    def __init__(self, init_args=None):
        super().__init__()
        if init_args is None:
            alpha, beta, f = 5 / 6, 5 / 6, lambda x: 1 + x
        else:
            alpha, beta, f = init_args
        self.alpha = torch.nn.Parameter(torch.tensor([alpha], dtype=torch.double))
        self.beta = torch.nn.Parameter(torch.tensor([beta], dtype=torch.double))
        self.f = f
        zero = torch.zeros((1,), dtype=torch.double, requires_grad=True)
        assert self.f(zero).item() == 1.0, 'Requires f(0) = 1'
        self.fprime0 = torch.autograd.grad(self.f(zero), zero)[0].item()
        self.initialize()

    def forward(self, box_vecs, den):
        alpha, beta = float(self.alpha.item()), float(self.beta.item())
        f, fprime0 = self.f, self.fprime0

        def launch(plan, d, _, E, v, stream):
            E3 = torch.empty(3, dtype=torch.double, device=d.device)
            v3 = torch.empty((3,) + tuple(d.shape), dtype=torch.double, device=d.device) if v is not None else None
            check(plan.lib.pad_eval_wt_components(plan.handle, ptr(d), alpha, beta, ptr(E3), ptr(v3), stream))
            tf, vw, tnl = E3.tolist()
            with torch.enable_grad():       # autograd.Function.forward runs with grad mode off
                x = torch.tensor([tnl / fprime0 / tf], dtype=torch.double, requires_grad=True)
                fx = f(x)
                dfx = torch.autograd.grad(fx, x)[0].item()
            fx, x = fx.item(), x.item()
            E.fill_(vw + tf * fx)
            if v is not None:
                torch.add(v3[1], v3[0], alpha=fx - x * dfx, out=v)
                v.add_(v3[2], alpha=dfx / fprime0)
        return _evaluate(box_vecs, den, launch).reshape(1)


class WangGovindCarter99(KineticFunctional):
    """WGC99 functional with Taylor-expanded density-dependent kernel (functionals.py:787-985).

    Evaluated in the 14-FFT analytic form (SURVEY.md section 8, a10); the kernel series of
    ``generate_kernel`` (functionals.py:845-939) is summed on the device and cached in the plan."""

    def __init__(self, init_args=None):
        super().__init__()
        if init_args is None:
            alpha, beta, gamma, kappa = _A98, _B98, 2.7, 1.0
        else:
            alpha, beta, gamma, kappa = init_args
        for name, val in (('alpha', alpha), ('beta', beta), ('gamma', gamma), ('kappa', kappa)):
            setattr(self, name, torch.nn.Parameter(torch.tensor([val], dtype=torch.double)))
        self.initialize()

    @property
    def _args(self):
        """(alpha, beta, gamma, kappa) as they are NOW (load_state_dict / .data edits count, as in the reference)"""
        return tuple(float(p.item()) for p in (self.alpha, self.beta, self.gamma, self.kappa))

    def forward(self, box_vecs, den):
        a, b, g, k = self._args

        def launch(plan, d, _, E, v, stream):
            check(plan.lib.pad_eval_wgc99(plan.handle, ptr(d), a, b, g, k, ptr(E), ptr(v), 0, stream))
        return _evaluate(box_vecs, den, launch).reshape(1)


# Semilocal kinetic functionals T = int C_TF n^(5/3) F(p, q) with p = s^2 and q the reduced gradient / Laplacian of
# functional_tools.py:122-135.  The constants are the published ones; they travel through the C ABI as arguments.
LKT_A = 1.3                          # Luo, Karasiev, Trickey, PRB 98, 041111 (2018)
PG_MU, PG_BETA = 40 / 27, 0.25       # PGSL0.25: Constantin, Fabiano, Della Sala, JPCL 9, 4385 (2018)


def _launch_semilocal(variant, p0, p1):
    def launch(plan, d, _, E, v, stream):
        check(plan.lib.pad_eval_semilocal_kinetic(plan.handle, ptr(d), variant, p0, p1, ptr(E), ptr(v), 0, stream))
    return launch


_L_LKT = _launch_semilocal(_native.SEMILOCAL_LKT, LKT_A, 0.0)
_L_PG = _launch_semilocal(_native.SEMILOCAL_PG, PG_MU, PG_BETA)


def LuoKarasievTrickey(box_vecs, den):
    """LKT (functionals.py:309): F = 1 / cosh(a s) + (5/3) s^2, a = 1.3.  8 FFTs."""
    return _evaluate(box_vecs, den, _L_LKT)


def PauliGaussian(box_vecs, den):
    """Pauli-Gaussian PGSL0.25 (functionals.py:336): F = (5/3) p + exp(-mu p) + beta q^2, mu = 40/27, beta = 0.25.
    10 FFTs: the Laplacian travels with the gradient."""
    return _evaluate(box_vecs, den, _L_PG)


# ----------------------------------------------------------------------------------------------
#  exchange-correlation
# ----------------------------------------------------------------------------------------------
def lda_exchange(box_vecs, den):
    """functionals.py:1510-1512"""
    return _evaluate(box_vecs, den, _L_LDAX)


def perdew_zunger_correlation(box_vecs, den):
    """functionals.py:1515-1521"""
    return _evaluate(box_vecs, den, _L_PZC)


def PerdewZunger(box_vecs, den):
    """Perdew-Zunger LDA (functionals.py:1540-1554): exchange + correlation in one pass over n."""
    return _evaluate(box_vecs, den, _L_PZ)


def _launch_pbe(which):
    def launch(plan, d, _, E, v, stream):
        check(plan.lib.pad_eval_pbe(plan.handle, ptr(d), which, ptr(E), ptr(v), 0, stream))
    return launch


_L_PBEX, _L_PBEC, _L_PBE = _launch_pbe(1), _launch_pbe(2), _launch_pbe(3)


def pbe_exchange(box_vecs, den):
    """functionals.py:1597-1603"""
    return _evaluate(box_vecs, den, _L_PBEX)


def pbe_correlation(box_vecs, den):
    """functionals.py:1606-1618"""
    return _evaluate(box_vecs, den, _L_PBEC)


def PerdewBurkeErnzerhof(box_vecs, den):
    """PBE exchange-correlation (functionals.py:1621-1635): 8 FFTs, gradient shared by x and c."""
    return _evaluate(box_vecs, den, _L_PBE)


# ----------------------------------------------------------------------------------------------
#  descriptors for the fused evaluator / device-resident optimiser (see _density_opt.describe_terms)
# ----------------------------------------------------------------------------------------------
IonElectron._pad_term = ('local', _native.LOCAL_IONEL)
ThomasFermi._pad_term = ('local', _native.LOCAL_TF)
lda_exchange._pad_term = ('local', _native.LOCAL_LDAX)
perdew_zunger_correlation._pad_term = ('local', _native.LOCAL_PZC)
PerdewZunger._pad_term = ('local', _native.LOCAL_LDAX | _native.LOCAL_PZC)
Hartree._pad_term = ('hartree',)
Weizsaecker._pad_term = ('wt', 1.0, 1.0, _native.PART_VW)
WangTeter._pad_term = ('wt', 5 / 6, 5 / 6, _native.PART_ALL)
Perrot._pad_term = ('wt', 1.0, 1.0, _native.PART_ALL)
SmargiassiMadden._pad_term = ('wt', 0.5, 0.5, _native.PART_ALL)
WangGovindCarter98._pad_term = ('wt', _A98, _B98, _native.PART_ALL)
pbe_exchange._pad_term = ('pbe', 1)
pbe_correlation._pad_term = ('pbe', 2)
PerdewBurkeErnzerhof._pad_term = ('pbe', 3)
WangGovindCarter99._pad_term_of = lambda self, device=None: ('wgc99',) + self._args
LuoKarasievTrickey._pad_term = ('semilocal', _native.SEMILOCAL_LKT, LKT_A, 0.0)
PauliGaussian._pad_term = ('semilocal', _native.SEMILOCAL_PG, PG_MU, PG_BETA)


# ----------------------------------------------------------------------------------------------
#  Huang-Carter family (functionals.py:1176-1365): field-dependent kernel by a spline over xi
# ----------------------------------------------------------------------------------------------
def huang_carter_kernel_table(beta, eta_max=50, N_eta=10000, rtol=1e-12, atol=1e-14):
    """omega(eta) on linspace(0, eta_max, N_eta) (functionals.py:1204-1230): the ODE
    w' = -[(5/3)(1/Ginv - 3 eta^2 - 1) - (5 - 3 beta) beta w] / (beta eta) integrated from eta_max
    down to the first grid point with w(eta_max) = -(8/3)/((5 - 3 beta) beta); omega(0) = 0.
    The reference integrates with xitorch.solve_ivp defaults (un-pinned dependency); here an
    8th-order Dormand-Prince integrator at tight tolerance is used (DESIGN.md: parity unpinned at
    this boundary -- for parity runs inject the same table into both sides via ``.kernel``)."""
    from scipy.integrate import solve_ivp

    def lind(e):
        if e == 0:
            return 1.0
        if e == 1:
            return 2.0
        return 1.0 / (0.5 + (1 - e * e) / (4 * e) * math.log(abs((1 + e) / (1 - e))))

    def rhs(e, w):
        return [-((5.0 / 3.0) * (lind(e) - 3 * e * e - 1) - (5 - 3 * beta) * beta * w[0]) / beta / e]
    etas = np.linspace(0.0, float(eta_max), int(N_eta))
    w_inf = -(8.0 / 3.0) / ((5 - 3 * beta) * beta)
    sol = solve_ivp(rhs, (etas[-1], etas[1]), [w_inf], t_eval=etas[1:][::-1], method='DOP853', rtol=rtol, atol=atol)
    w = np.concatenate([[0.0], sol.y[0][::-1]])
    return torch.from_numpy(np.stack([etas, w]))


class _HuangCarterFamily(KineticFunctional):
    mode = 'geometric'
    _variant = 0

    def _pad_term_of(self, device=None):
        """Descriptor for the fused evaluator / device-resident optimiser (_density_opt.describe_terms).  The table
        travels as a raw device pointer: it must live on the device the terms are evaluated on."""
        if self.mode not in ('geometric', 'arithmetic'):
            return None
        if device is None:
            if not torch.cuda.is_available():
                return None
            device = torch.device('cuda', torch.cuda.current_device())
        device = torch.device(device)
        if device.type != 'cuda':
            return None
        if device.index is None:
            device = torch.device('cuda', torch.cuda.current_device())
        table = self.kernel
        if table.device != device or table.dtype != torch.double or not table.is_contiguous():
            table = table.to(device=device, dtype=torch.double).contiguous()
            self.kernel = table
        p0, p1 = self._params()
        return ('hc', self._variant, p0, p1, float(self.beta.item()), float(self.kappa),
                1 if self.mode == 'geometric' else 0, table)

    def generate_kernel(self, eta_max=50, N_eta=10000):
        self.kernel = huang_carter_kernel_table(float(self.beta.item()), eta_max, N_eta)

    def _params(self):
        raise NotImplementedError

    def forward(self, box_vecs, den):
        p0, p1 = self._params()
        beta, kappa, variant = float(self.beta.item()), float(self.kappa), self._variant
        geometric = 1 if self.mode == 'geometric' else 0
        if self.mode not in ('geometric', 'arithmetic'):
            raise ValueError('Parameter \'mode\' can only be \'arithmetic\' or \'geometric\'')
        if geometric:
            assert kappa > 1, 'κ > 1 for geometric progression based spline for field_dependent_convolution'
        table = self.kernel
        if table.device != den.device or table.dtype != torch.double or not table.is_contiguous():
            table = table.to(device=den.device, dtype=torch.double).contiguous()
            self.kernel = table
        n_eta = int(table.shape[1])
        owner = self

        def launch(plan, d, _, E, v, stream):
            n_nodes = ctypes.c_int(0)
            check(plan.lib.pad_eval_hc(plan.handle, ptr(d), variant, p0, p1, beta, kappa, geometric, ptr(table), n_eta,
                                       ptr(E), ptr(v), 0, ctypes.byref(n_nodes), stream))
            owner.last_n_nodes = n_nodes.value
        return _evaluate(box_vecs, den, launch).reshape(1)


class HuangCarter(_HuangCarterFamily):
    """Huang-Carter functional (functionals.py:1176-1269), init_args = (lambda, beta, kappa).
    xi = 2 kF(n) (1 + lambda |grad n|^2 / n^{8/3})."""
    _variant = 0

    def __init__(self, init_args, kernel=None):
        super().__init__()
        lamb, beta, kappa = init_args
        self.lamb = torch.nn.Parameter(torch.tensor([lamb], dtype=torch.double))
        self.beta = torch.nn.Parameter(torch.tensor([beta], dtype=torch.double))
        self.kappa = kappa
        self.debug = False          # the reference forgets to set this (functionals.py:1247)
        self.initialize()
        if kernel is None:
            self.generate_kernel()
        else:
            self.kernel = kernel

    def _params(self):
        return float(self.lamb.item()), 0.0


class RevisedHuangCarter(_HuangCarterFamily):
    """revised Huang-Carter functional (functionals.py:1272-1365), init_args = (a, b, beta, kappa).
    xi = 2 kF(n) (1 + a s^2 / (1 + b s^2)) with s the reduced gradient."""
    _variant = 1

    def __init__(self, init_args, kernel=None):
        super().__init__()
        a, b, beta, kappa = init_args
        self.a = torch.nn.Parameter(torch.tensor([a], dtype=torch.double))
        self.b = torch.nn.Parameter(torch.tensor([b], dtype=torch.double))
        self.beta = torch.nn.Parameter(torch.tensor([beta], dtype=torch.double))
        self.kappa = kappa
        self.initialize()
        if kernel is None:
            self.generate_kernel()
        else:
            self.kernel = kernel

    def _params(self):
        return float(self.a.item()), float(self.b.item())
