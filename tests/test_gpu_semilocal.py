"""GPU checks of the semilocal kinetic functionals LuoKarasievTrickey and PauliGaussian (pad_eval_semilocal_kinetic,
pad_terms kinetic == 4): both routes against the autograd restatement (tests/semilocal_oracle.py), fused route against cuFFT route, term lists with PBE,
stress, size-independent properties at 256^3, density optimisation and slab plans.

The constants are those of the papers (LKT: PRB 98, 041111 (2018); PGSL0.25: JPCL 9, 4385 (2018)); parity with the
reference's own implementation is not pinned by golden vectors (DESIGN.md section 1)."""
import os
import threading

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

E_RTOL = 1e-10
V_RTOL = 1e-9
EV = 27.211386245988


def _pairs():
    import profess_ad_b200.functionals as F
    import semilocal_oracle as so
    return [('LKT', F.LuoKarasievTrickey, so.LuoKarasievTrickey), ('PG', F.PauliGaussian, so.PauliGaussian)]


class _Route:
    """fast = 1: fused passes where the grid allows them, 0: cuFFT everywhere"""

    def __init__(self, fast):
        from profess_ad_b200 import _native
        self.lib, self.fast = _native.load_library(), fast

    def __enter__(self):
        self.old = self.lib.pad_set_fast_fft(self.fast)

    def __exit__(self, *exc):
        self.lib.pad_set_fast_fft(self.old)


def _rel(a, b):
    return ((a - b).abs().max() / b.abs().max()).item()


def _golden_input(case, golden_dir):
    g = np.load(os.path.join(golden_dir, f'functionals_{case}.npz'))
    return torch.from_numpy(g['box']), torch.from_numpy(g['den'])


@pytest.mark.parametrize('fast', [1, 0], ids=['fused', 'cufft'])
@pytest.mark.parametrize('case', ['rough_even', 'rough_odd', 'rough_mixed', 'smooth16'])
def test_match_oracle(case, fast, golden_dir):
    from oracle import ofdft_oracle as orc
    from profess_ad_b200.functionals import energy_and_potential
    box, den = _golden_input(case, golden_dir)
    dev = torch.device('cuda:0')
    for name, f, fo in _pairs():
        E_ref, V_ref = orc.energy_and_potential(box, den, fo)
        with _Route(fast):
            E, V = energy_and_potential(box.to(dev), den.to(dev), f)
        assert abs(E.item() - E_ref.item()) <= E_RTOL * max(1.0, abs(E_ref.item())), (case, name, E.item(), E_ref.item())
        assert _rel(V.cpu(), V_ref) <= V_RTOL, (case, name)


@pytest.mark.parametrize('shape', [(64, 128, 128), (128, 128, 128)])
def test_fused_route_equals_cufft_route(shape):
    from oracle import ofdft_oracle as orc
    from profess_ad_b200 import _native
    from profess_ad_b200.functionals import energy_and_potential
    box, den = orc.synth_rough(shape, seed=4, L=12.0)
    dev = torch.device('cuda:0')
    box, den = box.to(dev), den.to(dev)
    lib = _native.load_library()
    for name, f, _ in _pairs():
        c0 = lib.pad_launch_count()
        with _Route(1):
            E1, V1 = energy_and_potential(box, den, f)
        torch.cuda.synchronize()
        n_fused = lib.pad_launch_count() - c0
        f0 = lib.pad_fft_exec_count()
        with _Route(0):
            E0, V0 = energy_and_potential(box, den, f)
        torch.cuda.synchronize()
        assert lib.pad_fft_exec_count() > f0            # the cuFFT route ran cuFFT ...
        assert n_fused > 0
        assert abs(E1.item() - E0.item()) <= 1e-12 * abs(E0.item()), (name, E1.item(), E0.item())
        assert _rel(V1, V0) <= 1e-11, name


def test_fused_route_runs_no_cufft():
    from oracle import ofdft_oracle as orc
    from profess_ad_b200 import _native
    from profess_ad_b200.functionals import energy_and_potential
    box, den = orc.synth_rough((64, 128, 128), seed=6, L=12.0)
    dev = torch.device('cuda:0')
    lib = _native.load_library()
    for _, f, _ in _pairs():
        energy_and_potential(box.to(dev), den.to(dev), f)      # plan, buffers
        torch.cuda.synchronize()
        f0 = lib.pad_fft_exec_count()
        energy_and_potential(box.to(dev), den.to(dev), f)
        torch.cuda.synchronize()
        assert lib.pad_fft_exec_count() == f0


@pytest.mark.parametrize('shape', [(64, 128, 128), (17, 20, 22)])
def test_term_list_with_pbe_equals_separate_calls(shape):
    """pad_eval_total with the kinetic term and PBE (one shared round trip) == the sum of the separate calls"""
    import profess_ad_b200.functionals as F
    from oracle import ofdft_oracle as orc
    from profess_ad_b200 import _density_opt as D
    box, den = orc.synth_rough(shape, seed=8, L=10.0)
    dev = torch.device('cuda:0')
    box, den = box.to(dev), den.to(dev)
    for name, f, _ in _pairs():
        for fast in (1, 0):
            with _Route(fast):
                T = D.describe_terms([F.Hartree, f, F.PerdewBurkeErnzerhof])
                E, v = D.eval_total(box, den, None, T)
                parts = [F.energy_and_potential(box, den, g) for g in (F.Hartree, f, F.PerdewBurkeErnzerhof)]
            E_sum = sum(p[0].item() for p in parts)
            v_sum = sum(p[1] for p in parts)
            assert abs(E.item() - E_sum) <= 1e-12 * abs(E_sum), (name, fast, E.item(), E_sum)
            assert _rel(v, v_sum) <= 1e-11, (name, fast)


@pytest.mark.parametrize('shape,seed', [((8, 10, 12), 1), ((9, 7, 11), 2), ((64, 128, 128), 3)])
def test_stress_matches_oracle(shape, seed):
    from oracle import ofdft_oracle as orc
    from profess_ad_b200.functional_tools import get_stress
    box, den = orc.synth_rough(shape, seed=seed)
    dev = torch.device('cuda:0')
    for name, f, fo in _pairs():
        ref = orc.stress(box, den, fo)
        got = get_stress(box.to(dev), den.to(dev), f).cpu()
        assert _rel(got, ref) <= 1e-10, (name, got, ref)


def test_full_size_properties_256():
    """256^3: tiling a 128^3 cell twice per axis multiplies E by 8 and tiles v; a translation by whole grid points
    leaves E unchanged and translates v; v is the derivative of E along a number-conserving direction."""
    import profess_ad_b200.functionals as F
    from profess_ad_b200.synthetic import smooth_supercell
    dev = torch.device('cuda:0')
    box1, den1 = smooth_supercell(128, 2, device=dev)
    gen = torch.Generator().manual_seed(3)
    den1 = den1 * (1 + 0.05 * torch.rand(128, 128, 128, dtype=torch.double, generator=gen).to(dev))
    box2, den2 = 2 * box1, den1.repeat(2, 2, 2).contiguous()
    dV = abs(torch.linalg.det(box2).item()) / den2.numel()
    for name, f, _ in _pairs():
        E1, V1 = F.energy_and_potential(box1, den1, f)
        E2, V2 = F.energy_and_potential(box2, den2, f)
        assert abs(E2.item() - 8 * E1.item()) <= 2e-12 * abs(E2.item()), (name, E2.item(), 8 * E1.item())
        assert _rel(V2, V1.repeat(2, 2, 2)) < 1e-10, name
        shift = (37, 101, 6)
        E3, V3 = F.energy_and_potential(box2, torch.roll(den2, shift, (0, 1, 2)).contiguous(), f)
        assert abs(E3.item() - E2.item()) <= 2e-12 * abs(E2.item()), name
        assert _rel(V3, torch.roll(V2, shift, (0, 1, 2))) < 1e-10, name
        W = V2 / V2.abs().max()
        delta = 0.01 * den2.mean() * (W - W.mean())
        eps = 1e-3
        Ep = f(box2, (den2 + eps * delta).contiguous()).item()
        Em = f(box2, (den2 - eps * delta).contiguous()).item()
        lhs = (Ep - Em) / (2 * eps)
        rhs = (V2 * delta).sum().item() * dV
        assert abs(lhs - rhs) <= 1e-7 * abs(rhs) + 1e-12, (name, lhs, rhs)


def _lkt_user_term(box_vecs, den):
    """LKT as a plain torch user term (the host-driven generic path, autograd for the potential)"""
    from profess_ad_b200.functional_tools import reduced_gradient_squared, wavevecs
    kx, ky, kz, _ = wavevecs(box_vecs, den.shape)
    p = reduced_gradient_squared(kx, ky, kz, den)
    s = torch.sqrt(p + 1e-300)        # finite autograd at the uniform start (grad n = 0)
    c_tf = 0.3 * (3 * np.pi ** 2) ** (2 / 3)
    vol = torch.abs(torch.linalg.det(box_vecs))
    return torch.mean(c_tf * den.pow(5 / 3) * (1 / torch.cosh(1.3 * s) + 5 / 3 * p)) * vol


def _al_system(golden_dir, potentials_dir, terms, reps=1, shape=None):
    from profess_ad_b200.system import System
    g = np.load(os.path.join(golden_dir, 'denopt_al_fcc4_config1.npz'))
    frac = torch.from_numpy(g['frac'])
    if reps > 1:
        cells = [frac + torch.tensor([i, j, k], dtype=torch.double) for i in range(reps) for j in range(reps) for k in range(reps)]
        frac = torch.cat(cells) / reps
    box = reps * torch.from_numpy(g['box_bohr'])
    shape = shape or tuple(int(s) for s in g['shape'])
    ions = [['Al', os.path.join(potentials_dir, 'al.gga.recpot'), frac]]
    return System(box, shape, ions, terms, units='b', coord_type='fractional'), frac.shape[0]


@pytest.mark.parametrize('reps,shape', [(1, None), (2, (32, 32, 32))], ids=['fcc4', 'fcc32_32cubed'])
def test_density_optimisation_lkt(reps, shape, golden_dir, potentials_dir, monkeypatch):
    """fcc Al, LKT + Hartree + PZ + IonElectron: the device-resident loop == the host-driven generic path with LKT as a
    torch user term (and == the CPU oracle on the 4-atom cell), within 1e-6 eV/atom"""
    import profess_ad_b200.functionals as F
    import semilocal_oracle as so
    from oracle import ofdft_oracle as orc
    from profess_ad_b200.system import System
    native, natoms = _al_system(golden_dir, potentials_dir, [F.IonElectron, F.Hartree, F.LuoKarasievTrickey, F.PerdewZunger],
                                reps, shape)
    native.optimize_density(ntol=1e-9, from_uniform=True)
    assert native.last_optimization.get('native') and native.last_optimization['converged']
    generic, _ = _al_system(golden_dir, potentials_dir, [F.IonElectron, F.Hartree, _lkt_user_term, F.PerdewZunger], reps, shape)
    monkeypatch.setattr(System, 'use_native_optimizer', False)
    generic.optimize_density(ntol=1e-9, from_uniform=True)
    e_native, e_generic = native.energy('eV'), generic.energy('eV')
    assert abs(e_native - e_generic) / natoms < 1e-6, (e_native, e_generic)
    if reps == 1:                   # no IonIon term: energy() is the functional energy the oracle minimises
        v_ext = native.ionic_potential().cpu()
        box = native.lattice_vectors('b').cpu()
        n_elec = float(native.electron_count())
        den0 = torch.full(tuple(v_ext.shape), n_elec / abs(torch.linalg.det(box).item()), dtype=torch.double)
        ref = orc.optimize_density(box, den0, n_elec, [orc.IonElectron, orc.Hartree, so.LuoKarasievTrickey, orc.PerdewZunger],
                                   v_ext=v_ext, ntol=1e-9)
        assert abs(e_native - ref['energy'] * EV) / natoms < 1e-6, (e_native, ref['energy'] * EV)
    assert native.stress().shape == (3, 3)
    native.pressure()


def _slab_rank(comm, shape, box, den_global, f, out, idx, errors):
    from profess_ad_b200 import parallel
    from profess_ad_b200.functional_tools import get_stress
    try:
        dev = torch.device('cuda:0')
        with torch.cuda.stream(torch.cuda.Stream(dev)):
            with parallel.slab(shape, comm=comm):
                d = parallel.local_slab(den_global.to(dev)).requires_grad_(True)
                E = f(box.to(dev), d)
                (g,) = torch.autograd.grad(E, d)
                sig = get_stress(box.to(dev), d.detach(), f)
                torch.cuda.current_stream(dev).synchronize()
                out[idx] = (E.item(), g.cpu(), sig.cpu())
    except BaseException as e:      # noqa: BLE001
        errors.append(e)
        try:
            comm.shared.barrier.abort()
        except Exception:
            pass


@pytest.mark.parametrize('world,shape', [(2, (8, 6, 10)), (4, (8, 12, 6)), (2, (64, 64, 128))])
def test_slabs_match_single_gpu(world, shape):
    from oracle import ofdft_oracle as orc
    from profess_ad_b200 import parallel
    from profess_ad_b200.functional_tools import get_stress
    from profess_ad_b200.functionals import energy_and_potential
    box, den = orc.synth_rough(shape, seed=21 + world, L=8.5)
    dev = torch.device('cuda:0')
    dV = abs(torch.linalg.det(box).item()) / den.numel()
    for name, f, _ in _pairs():
        E1, V1 = energy_and_potential(box.to(dev), den.to(dev), f)
        S1 = get_stress(box.to(dev), den.to(dev), f).cpu()
        out, errors = [None] * world, []
        shared = parallel.ThreadComm.Shared(world)
        threads = [threading.Thread(target=_slab_rank, args=(parallel.ThreadComm(shared, r), shape, box, den, f, out, r, errors))
                   for r in range(world)]
        for t in threads:
            t.start()
        for t in threads:
            t.join(timeout=300)
        if errors:
            raise errors[0]
        for E, _, S in out:
            assert abs(E - E1.item()) <= 1e-12 * abs(E1.item()), (name, world, E, E1.item())
            assert _rel(S, S1) <= 1e-11, (name, world)
        g = torch.cat([o[1] for o in out], dim=0)
        assert _rel(g / dV, V1.cpu()) <= 1e-11, (name, world)


def test_optimize_geometry_with_lkt(golden_dir, potentials_dir):
    """cell + ions relaxation with LKT as the kinetic term: the analytic forces and the kinetic == 4 stress drive the
    reference's optimisers to a point where both are below the tolerances"""
    import profess_ad_b200.functionals as F
    from profess_ad_b200.system import System
    g = np.load(os.path.join(golden_dir, 'geometry_li2_full.npz'))
    terms = [F.IonIon, F.IonElectron, F.Hartree, F.LuoKarasievTrickey, F.PerdewBurkeErnzerhof]
    ions = [['Li', os.path.join(potentials_dir, 'li.gga.recpot'), torch.from_numpy(g['frac0'])]]
    s = System(torch.from_numpy(g['box0_A']), tuple(int(n) for n in g['shape']), ions, terms, units='a', coord_type='fractional')
    assert s.optimize_geometry(g_maxiter=60, ntol=1e-9, ftol=0.02, stol=0.002)
    assert s.forces('eV/a').abs().max().item() < 0.02
    assert s.stress('eV/a3').abs().max().item() < 0.002
