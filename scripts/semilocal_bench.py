"""E + V of the semilocal kinetic functionals at 256^3 on one GPU: LuoKarasievTrickey, PauliGaussian, PBE and LKT + PBE
(one term list, one shared gradient / divergence round trip), timed with CUDA events in one process.

    python scripts/semilocal_bench.py [--n 256] [--reps 50] [--out path.json]

Prints one JSON line per case: median ms per E + V, the route taken (fused passes or cuFFT), the algorithmic bytes
B_alg = 16 N n_fft + 16 N (every 3-D transform reads and writes N doubles; the density in and the potential out) and the
rate B_alg / time, with the device name and power limit.  The working set (several 134 MB fields) exceeds the L2."""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import profess_ad_b200.functionals as F  # noqa: E402
from profess_ad_b200 import _density_opt as D, _native  # noqa: E402
from profess_ad_b200.synthetic import smooth_supercell  # noqa: E402

CASES = [('LKT', [F.LuoKarasievTrickey], 8), ('PG', [F.PauliGaussian], 10), ('PBE', [F.PerdewBurkeErnzerhof], 8),
         ('LKT+PBE', [F.LuoKarasievTrickey, F.PerdewBurkeErnzerhof], 8)]


def power_limit_w(index):
    try:
        r = subprocess.run(['nvidia-smi', '-i', str(index), '--query-gpu=power.limit', '--format=csv,noheader,nounits'],
                           capture_output=True, text=True, timeout=30)
        return float(r.stdout.strip().splitlines()[0])
    except Exception:      # noqa: BLE001
        return None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--n', type=int, default=256)
    ap.add_argument('--reps', type=int, default=50)
    ap.add_argument('--out', default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('semilocal_bench: needs a CUDA device')
    dev = torch.device('cuda:0')
    box, den = smooth_supercell(a.n, a.n // 64, device=dev)
    gen = torch.Generator().manual_seed(3)
    den = (den * (1 + 0.05 * torch.rand(den.shape, dtype=torch.double, generator=gen).to(dev))).contiguous()
    lib = _native.load_library()
    N = den.numel()
    head = {'device': torch.cuda.get_device_name(dev), 'power_limit_w': power_limit_w(dev.index or 0), 'shape': [a.n] * 3}
    rows = []
    Ts = {name: D.describe_terms(terms) for name, terms, _ in CASES}
    for _ in range(3):                          # warm-up: plans, buffers, module loads, cuFFT plans of every case
        for name, _, _ in CASES:
            D.eval_total(box, den, None, Ts[name])
    torch.cuda.synchronize()
    times = {name: [] for name, _, _ in CASES}
    routes, launches = {}, {}
    for name, _, _ in CASES:
        f0, l0 = lib.pad_fft_exec_count(), lib.pad_launch_count()
        D.eval_total(box, den, None, Ts[name])
        torch.cuda.synchronize()
        routes[name] = 'fused' if lib.pad_fft_exec_count() == f0 else 'cufft'
        launches[name] = lib.pad_launch_count() - l0
    for _ in range(a.reps):                     # the cases alternate, so drifts of the shared host hit all of them alike
        for name, _, _ in CASES:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            D.eval_total(box, den, None, Ts[name])
            e1.record()
            e1.synchronize()
            times[name].append(e0.elapsed_time(e1))
    for name, _, n_fft in CASES:
        t = sorted(times[name])
        ms = t[len(t) // 2]
        b_alg = 16 * N * n_fft + 16 * N
        rows.append(dict(head, case=name, route=routes[name], launches=launches[name], ms_median=ms, ms_min=t[0], ms_max=t[-1], n_fft=n_fft,
                         B_alg=b_alg, B_alg_per_s=b_alg / (ms * 1e-3)))
    pbe = next(r['ms_median'] for r in rows if r['case'] == 'PBE')
    for r in rows:
        r['over_pbe'] = r['ms_median'] / pbe
        print(json.dumps(r))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, 'w') as fh:
            json.dump(rows, fh, indent=1)


if __name__ == '__main__':
    main()
