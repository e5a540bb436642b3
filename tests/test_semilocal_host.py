"""Host-side checks of the semilocal kinetic functionals (LuoKarasievTrickey, PauliGaussian): the analytic point math,
potential and stress that csrc/xc.cuh, csrc/functionals.cu / fftz.cu and csrc/stress.cu implement, restated in torch and
checked against autograd (tests/semilocal_oracle.py, on the oracle's grid) on even, odd and mixed skewed grids; and the term-list descriptor."""
import pytest
import torch

import analytic_model as am
import semilocal_oracle as so
from oracle import ofdft_oracle as orc

C = 0.25 * (3.0 * am.PI * am.PI) ** (-2.0 / 3.0)
LKT = (0, 1.3, 0.0)
PG = (1, 40.0 / 27.0, 0.25)
SHAPES = [((8, 10, 12), 1), ((9, 7, 11), 2), ((8, 9, 10), 3)]


def point(den, sig, lap, variant, p0, p1):
    """e, e_n, e_sigma, e_L of semilocal_kinetic_point (xc.cuh)"""
    n23 = den.pow(2.0 / 3.0)
    p = C * sig / den.pow(8.0 / 3.0)
    if variant == 0:
        x = p0 * torch.sqrt(p)
        sech = 1.0 / torch.cosh(x)
        F = sech + 5.0 / 3.0 * p
        Fp = 5.0 / 3.0 - 0.5 * p0 * p0 * sech * torch.tanh(x) / x
        qFq, e_l = torch.zeros_like(den), torch.zeros_like(den)
    else:
        q = C * lap / (den * n23)
        g = torch.exp(-p0 * p)
        F = 5.0 / 3.0 * p + g + p1 * q * q
        Fp = 5.0 / 3.0 - p0 * g
        qFq = 2.0 * p1 * q * q
        e_l = am.C_TF * C * 2.0 * p1 * q
    e = am.C_TF * den * n23 * F
    e_n = am.C_TF * n23 * (5.0 / 3.0 * F - 8.0 / 3.0 * p * Fp - 5.0 / 3.0 * qFq)
    e_s = am.C_TF * C * Fp / den
    return e, e_n, e_s, e_l


def _fields(g, den):
    ik = [g.sym(lambda kx, ky, kz, c=c: 1j * (kx, ky, kz)[c]) for c in range(3)]
    mk2 = g.sym(lambda kx, ky, kz: -(kx * kx + ky * ky + kz * kz))
    R = g.fwd(den)
    return ik, mk2, [g.inv(m * R) for m in ik], g.inv(mk2 * R)


def energy_potential(box, den, variant, p0, p1):
    """E and v = e_n - div(2 e_sigma grad n) + lap(e_L), with the Hermitian multipliers of the kernels"""
    g = am.KGrid(box, den.shape)
    ik, mk2, gr, lap = _fields(g, den)
    sig = gr[0] ** 2 + gr[1] ** 2 + gr[2] ** 2
    e, e_n, e_s, e_l = point(den, sig, lap, variant, p0, p1)
    div = sum(g.inv(ik[c] * g.fwd(2.0 * e_s * gr[c])) for c in range(3))
    return g.integ(e), e_n - div + g.inv(mk2 * g.fwd(e_l))


def stress(box, den, variant, p0, p1):
    """delta_ij mean(e - n e_n - 2 sigma e_sigma - L e_L) - 2 mean(e_sigma g_i g_j) + 2 sum_k w Re(conj(l_k) c_k) k_i k_j"""
    g = am.KGrid(box, den.shape)
    _, _, gr, lap = _fields(g, den)
    sig = gr[0] ** 2 + gr[1] ** 2 + gr[2] ** 2
    e, e_n, e_s, e_l = point(den, sig, lap, variant, p0, p1)
    out = float((e - den * e_n - 2.0 * sig * e_s - lap * e_l).mean()) * torch.eye(3, dtype=torch.double)
    for i in range(3):
        for j in range(3):
            out[i, j] -= 2.0 * float((e_s * gr[i] * gr[j]).mean())
    lk, ck = g.fwd(e_l) / g.N, g.fwd(den) / g.N
    return out + 2.0 * am._tensor_sum(g, am._weights(g) * (lk.conj() * ck).real)


def _oracle(variant):
    return so.LuoKarasievTrickey if variant == 0 else so.PauliGaussian


@pytest.mark.parametrize('shape,seed', SHAPES)
@pytest.mark.parametrize('params', [LKT, PG], ids=['LKT', 'PG'])
def test_analytic_potential_equals_autograd(shape, seed, params):
    box, den = orc.synth_rough(shape, seed=seed)
    E, V = orc.energy_and_potential(box, den, _oracle(params[0]))
    e, v = energy_potential(box, den, *params)
    assert abs(E.item() - e) < 1e-12 * abs(e)
    assert ((V - v).abs().max() / V.abs().max()).item() < 1e-12


@pytest.mark.parametrize('shape,seed', SHAPES)
@pytest.mark.parametrize('params', [LKT, PG], ids=['LKT', 'PG'])
def test_analytic_stress_equals_autograd(shape, seed, params):
    """the formula of csrc/stress.cu (kinetic == 4) against autograd through box_vecs"""
    box, den = orc.synth_rough(shape, seed=seed)
    ref = orc.stress(box, den, _oracle(params[0]))
    got = stress(box, den, *params)
    assert float((got - ref).abs().max() / ref.abs().max()) <= 1e-13


def test_lkt_small_gradient_series():
    """sigma = 0 and tiny gradients: tanh(x)/x from its series agrees with the closed form and has no 0/0"""
    x = torch.tensor([0.0, 1e-8, 1e-3, 0.03, 0.0624], dtype=torch.double)
    x2 = x * x
    series = 1.0 + x2 * (-1.0 / 3.0 + x2 * (2.0 / 15.0 + x2 * (-17.0 / 315.0 + x2 * (62.0 / 2835.0))))
    closed = torch.where(x > 0, torch.tanh(x) / torch.where(x > 0, x, torch.ones_like(x)), torch.ones_like(x))
    assert float((series - closed).abs().max()) < 1e-14


def test_describe_terms_maps_semilocal_kinetic():
    import profess_ad_b200.functionals as F
    from profess_ad_b200 import _density_opt as D, _native
    T = D.describe_terms([F.IonElectron, F.Hartree, F.LuoKarasievTrickey, F.PerdewBurkeErnzerhof])
    assert (T.kinetic, T.sl_variant, T.sl_p0, T.pbe) == (4, _native.SEMILOCAL_LKT, 1.3, 3)
    assert T.local_mask == _native.LOCAL_IONEL and T.hartree == 1
    T = D.describe_terms([F.PauliGaussian, F.PerdewZunger])
    assert (T.kinetic, T.sl_variant, T.sl_p0, T.sl_p1) == (4, _native.SEMILOCAL_PG, 40 / 27, 0.25)
    # one kinetic term per list
    assert D.describe_terms([F.LuoKarasievTrickey, F.PauliGaussian]) is None
    assert D.describe_terms([F.PauliGaussian, F.WangTeter]) is None
    assert D.describe_terms([F.WangGovindCarter99().forward, F.LuoKarasievTrickey]) is None


def test_pad_terms_fields_appended():
    """the semilocal fields sit after every earlier field of pad_terms: existing offsets do not move"""
    from profess_ad_b200._density_opt import PadTerms
    names = [f[0] for f in PadTerms._fields_]
    assert names[-3:] == ['sl_variant', 'sl_p0', 'sl_p1']
    assert PadTerms.hc_table_dev.offset < PadTerms.sl_variant.offset
