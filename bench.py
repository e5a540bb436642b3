#!/usr/bin/env python
"""Headline benchmark: WangGovindCarter99 energy + potential evaluations per second at 256^3.

    python bench.py --gpus N --steps K --warmup W            # B200 arm (this repo's CUDA path)
    python bench.py --impl reference --gpus N --steps K --warmup W   # the reference algorithm on host cores
    python bench.py --gpus 1 --steps K --warmup W --dump-outputs DIR  # B200 arm, then DIR/*.npy: outputs of the last timed step

One "step" = one evaluation of E[n] and dE/dn for the full kinetic functional WangGovindCarter99
(TF + vW + non-local term, kernel cached) on the synthetic 256-atom Al supercell density of
BASELINE.md section 4 (`synth(256, side=4)`), i.e. BASELINE.json configs[1].

  value     : whole-job evals/s, density resident in HBM, timed with CUDA events on the launch stream
  e2e       : same metric through the public Python API from PINNED HOST buffers: H2D of the density,
              evaluation, D2H of the energy and the potential, all inside the timed region
  roofline  : algorithmic bytes per evaluation (SURVEY.md section 8d: 16 N n_fft + 16 N, n_fft = 14)
              / measured time per evaluation, against MEASURED_PEAKS.json hbm_gbs
  cpu_baseline : the UNMODIFIED reference (oracle/_ref, built by oracle/make_ref.py; kind "reference") -- or, if that
              directory is absent, the oracle port (oracle/ofdft_oracle.py, kind "port") -- torch CPU fp64 on all host
              threads, bounded sample, N=1 rank 0 only; its E and dE/dn at 256^3 are compared with the GPU's (`parity`)

Multi-GPU (torchrun): the headline line is independent systems, one per GPU (BASELINE.json configs[3] style weak
scaling, no data-path collective).  For N > 1 the same line carries a `slab` block: ONE grid slab-decomposed over the N
GPUs (all-to-all over NVLink inside every 3-D transform, strong scaling) for BASELINE.json configs[2] and [4].
"""
import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = 'WGC99 energy+potential evaluations per second at 256^3'
UNIT = 'evals/s'
GRID = int(os.environ.get('PAD_BENCH_GRID', '256'))
SIDE = 4
N_FFT = 14
# dram__bytes_read.sum + dram__bytes_write.sum from an ncu capture of this pipeline at 256^3 -- NOT measured in the bench
# run (a run under ncu is never a bench value): per launch of the dominant stage, and summed over one evaluation
NCU_TRAFFIC_256 = {'x-fwd * kernel-mix * x-inv (3 fields)': 0.9278e9, 'evaluation': 8.936e9}
NCU_TRAFFIC_SOURCE = 'profiles/r02_ncu_full_wgc99_256_final.md (ncu --set full of one evaluation; not measured in this run)'
DUMP_POINTS = 1 << 22          # grid points of dE/dn written by --dump-outputs: 32 MB of float64
DUMP_SEED = 0


def workload_config():
    """`config` of the JSON line: identical in the B200 arm and in the reference arm."""
    return {'workload': f'Al 256-atom supercell, WangGovindCarter99 E+V, {GRID}^3 grid (BASELINE.json configs[1])',
            'grid': [GRID] * 3, 'functional': 'WangGovindCarter99 (TF + vW + non-local, kernel cached)',
            'density': f'synthetic smooth_supercell({GRID}, side={SIDE})'}


def algorithmic_bytes(n):
    npts = n ** 3
    return 16 * npts * N_FFT + 16 * npts


def stage_bytes(name, n, ns):
    """Bytes one launch of a pipeline stage has to move (its own inputs and outputs once): n real points
    (8 B), ns live half-spectrum points (16 B)."""
    table = {
        'sum(n) -> n_ref, kernel cache check': 8 * n,
        'gen a,a.th,a.th2,chi + z-r2c (4 fields)': 8 * n + 4 * 16 * ns,
        'y-fwd (4 fields)': 2 * 4 * 16 * ns, 'y-inv (4 fields)': 2 * 4 * 16 * ns,
        'y-fwd (3 fields)': 2 * 3 * 16 * ns, 'y-inv (3 fields)': 2 * 3 * 16 * ns,
        'x-fwd * kernel-mix * x-inv (3 fields)': 2 * 3 * 16 * ns + 32 * ns,
        'x-fwd * (-k^2) * x-inv (1 field)': 2 * 16 * ns,
        'z-c2r (4 fields) + energy/v1/P': 4 * 16 * ns + 8 * n + 16 * n,
        'gen P,P.th,P.th2 + z-r2c (3 fields)': 16 * n + 3 * 16 * ns,
        'z-c2r (3 fields) + v2': 3 * 16 * ns + 8 * n + 16 * n,
    }
    return table.get(name)


def measured_peak():
    path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    try:
        with open(path) as f:
            return float(json.load(f)['hbm_gbs']), 'measured (MEASURED_PEAKS.json hbm_gbs)'
    except Exception:
        return 6650.0, 'fallback (B200_PROFILING.md)'


class ClockSampler:
    """SM clock / throttle reasons sampled through NVML while the timed region runs (nvidia-smi polling is too slow for a
    sub-second region).  NVML is initialised BEFORE the region and polled every 25 ms: every query takes the driver's lock, so
    a tighter loop (5 ms in earlier rounds) -- or nvmlInit inside the region -- showed up as stalled kernel launches on some
    boxes (3.8 instead of 2.2 ms per step with one sample taken)."""
    REASONS = {0x8: 'hw_slowdown', 0x40: 'hw_thermal_slowdown', 0x20: 'sw_thermal_slowdown', 0x4: 'sw_power_cap'}
    PERIOD = 0.025

    def __init__(self, index):
        self.index = index
        self.samples = []
        self.mask = 0
        self.stop_flag = False
        self.thread = None
        self.err = None
        self.max_mhz = None
        self.power = []
        self.nvml = self.handle = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nvml = pynvml
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
        except Exception as e:      # noqa: BLE001
            self.err = repr(e)

    def _sample(self):
        pynvml, h = self.nvml, self.handle
        self.samples.append(float(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)))
        try:
            self.mask |= int(pynvml.nvmlDeviceGetCurrentClocksEventReasons(h))
        except Exception:
            self.mask |= int(pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(h))
        try:
            self.power.append(pynvml.nvmlDeviceGetPowerUsage(h) / 1000.0)
        except Exception:
            pass

    def _run(self):
        try:
            while not self.stop_flag:
                time.sleep(self.PERIOD)
                if not self.stop_flag:
                    self._sample()
        except Exception as e:      # noqa: BLE001
            self.err = repr(e)

    def start(self):
        """No sampling thread any more: an NVML query takes the driver's lock, and a query that lands while the host is still
        queueing the timed steps stalls the launches (seen as a 20-30 ms hole at the start of 1 run in 5).  The samples are taken
        in stop() instead -- the launch loop is finished after ~10 ms of host time while the GPU works through the queued steps
        for >= 100 ms, so they still fall inside the timed work."""
        return

    def stop(self):
        """Call while the GPU is still busy with the last timed steps (before the closing synchronise): takes a final sample."""
        self.stop_flag = True
        if self.thread is not None:
            self.thread.join(timeout=2)
        if self.handle is not None:
            try:
                for i in range(5):          # the launch loop runs far ahead of the GPU: these fall into the timed work
                    self._sample()
                    time.sleep(0.008)
            except Exception as e:      # noqa: BLE001
                self.err = repr(e)
        if not self.samples:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvml unavailable: ' + str(self.err)]}
        sm = sorted(self.samples)
        return {'sm_mhz': sm[len(sm) // 2], 'sm_min_mhz': sm[0], 'sm_max_mhz': self.max_mhz,
                'reasons': sorted(v for k, v in self.REASONS.items() if self.mask & k),
                'power_w_max': max(self.power) if self.power else None, 'samples': len(sm)}


def host_cores():
    """Physical cores this process may run on (what torch picks by default when OMP_NUM_THREADS is not set)."""
    try:
        allowed = len(os.sched_getaffinity(0))
    except AttributeError:
        allowed = os.cpu_count() or 1
    try:
        import psutil
        physical = psutil.cpu_count(logical=False) or allowed
    except Exception:      # noqa: BLE001
        physical = allowed
    return max(1, min(allowed, physical))


def dist_env():
    rank = int(os.environ.get('RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    return rank, world, local


# --------------------------------------------------------------------------------------------------
#  CPU reference arm / cpu_baseline
# --------------------------------------------------------------------------------------------------
def reference_functional():
    """(callable (box, den) -> (E, dE/dn), kind, label): the unmodified reference from oracle/_ref when it is there
    (WangGovindCarter99.forward differentiated by torch.autograd, functional_tools.get_functional_derivative), else the
    oracle port."""
    import torch
    from oracle import ref_loader
    ref = ref_loader.load_reference()
    if ref is not None:
        wgc = ref.functionals.WangGovindCarter99()

        def run(box, den):
            d = den.clone().requires_grad_(True)
            E = wgc.forward(box, d)
            (g,) = torch.autograd.grad(E, d)
            dV = torch.abs(torch.linalg.det(box)) / den.numel()
            return E.detach().reshape(()), g / dV
        return run, 'reference', 'unmodified reference (oracle/_ref: professad.functionals.WangGovindCarter99 + autograd)'
    from oracle import ofdft_oracle as orc
    wgc = orc.WangGovindCarter99()
    return (lambda box, den: orc.energy_and_potential(box, den, wgc)), 'port', 'oracle port (oracle/ofdft_oracle.py)'


def cpu_reference_run(steps, warmup, sample_grid=None, threads=None, max_timed=3, keep=False):
    """The reference's own CPU implementation of the path (torch CPU fp64, all host threads) on the SAME workload.
    Bounded sample: at most `max_timed` timed evaluations after one warm-up that also builds and caches the kernel
    (not timed, as on the GPU).  Returns a dict; with keep=True it also holds the last E and dE/dn."""
    import torch
    from oracle import ofdft_oracle as orc
    # torchrun exports OMP_NUM_THREADS=1 to its workers: the CPU arm is meant to use every host core it can
    torch.set_num_threads(threads or host_cores())
    cores = torch.get_num_threads()
    n = sample_grid or GRID
    n_timed = max(1, min(steps, max_timed))
    box, den = orc.synth_smooth(n, SIDE)
    run, kind, label = reference_functional()
    t0 = time.perf_counter()
    run(box, den)
    t_first = time.perf_counter() - t0
    t0 = time.perf_counter()
    for _ in range(n_timed):
        E, V = run(box, den)
    dt = (time.perf_counter() - t0) / n_timed
    scale = (GRID ** 3 * math.log2(GRID ** 3)) / (n ** 3 * math.log2(n ** 3))
    sec_per_eval = dt * scale
    sample = (f'{n_timed} evals (+1 warm-up of {t_first:.1f} s that builds the kernel) of the {label} at {n}^3 on {cores} threads'
              + ('' if n == GRID else f', scaled x{scale:.2f} (N log N) to {GRID}^3'))
    out = {'value': 1.0 / sec_per_eval, 'ms': sec_per_eval * 1e3, 'cores': cores, 'sample': sample, 'kind': kind,
           'n_timed': n_timed}
    if keep:
        out['E'], out['V'] = float(E), V
    return out


def run_reference(args):
    rank, world, _ = dist_env()
    if rank != 0:
        return
    r = cpu_reference_run(args.steps, args.warmup)
    line = {
        'impl': 'reference', 'metric': METRIC, 'value': r['value'], 'unit': UNIT, 'n_gpus': args.gpus,
        'steps': r['n_timed'], 'warmup': 1, 'steps_requested': args.steps, 'warmup_requested': args.warmup,
        'ms_per_step': r['ms'], 'higher_is_better': True,
        'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f64', 'data': 'synthetic',
        'config': workload_config(),
        'cpu_baseline': {'value': r['value'], 'unit': UNIT, 'cores': r['cores'], 'kind': r['kind'], 'sample': r['sample']},
        'e2e': {'value': r['value'], 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'gpu_launches': 0,
    }
    print(json.dumps(line), flush=True)


def bind_to_gpu_numa(index):
    """Pin this rank to the CPU cores of the NUMA node its GPU hangs off, BEFORE any pinned host buffer is allocated
    (first-touch puts the pages there): with 8 ranks staging 134 MB per step each through host memory, buffers on the
    far socket halve the per-rank PCIe rate.  Returns what was done, for the JSON line."""
    info = {'gpu': index}
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        bus = pynvml.nvmlDeviceGetPciInfo(h).busId
        bus = bus.decode() if isinstance(bus, bytes) else bus
        bus = bus.lower()
        if len(bus.split(':')[0]) == 8:          # NVML prints an 8-digit PCI domain, sysfs a 4-digit one
            bus = bus[4:]
        node = int(open(f'/sys/bus/pci/devices/{bus}/numa_node').read().strip())
        info['numa_node'] = node
        if node >= 0:
            cpus = set()
            for part in open(f'/sys/devices/system/node/node{node}/cpulist').read().strip().split(','):
                a, _, b = part.partition('-')
                cpus.update(range(int(a), int(b or a) + 1))
            allowed = cpus & set(os.sched_getaffinity(0))
            if allowed:
                os.sched_setaffinity(0, allowed)
                info['cpus_bound'] = len(allowed)
    except Exception as e:      # noqa: BLE001 -- placement is an optimisation, never a failure
        info['error'] = repr(e)
    return info


# --------------------------------------------------------------------------------------------------
#  B200 arm
# --------------------------------------------------------------------------------------------------
def run_gpu(args):
    import torch
    import torch.distributed as dist
    rank, world, local = dist_env()
    if not torch.cuda.is_available():
        raise RuntimeError('bench.py: no CUDA device; the B200 arm has no CPU fallback (use --impl reference)')
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    numa = bind_to_gpu_numa(local) if world > 1 else None
    if world > 1:
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        # high-priority NCCL stream: in the slab block the exchange of one field runs while the FFT kernels of the next one
        # fill the SMs; its CTAs must not queue behind them
        opts = dist.ProcessGroupNCCL.Options(is_high_priority_stream=True)
        dist.init_process_group('nccl', device_id=dev, pg_options=opts)

    import profess_ad_b200.functionals as F
    from profess_ad_b200.synthetic import smooth_supercell
    from profess_ad_b200 import _native
    lib = _native.load_library()

    box_h, den_h = smooth_supercell(GRID, SIDE)
    box = box_h.to(dev)
    den = den_h.to(dev)
    wgc = F.WangGovindCarter99()
    npts = den.numel()

    def step_device():
        d = den.requires_grad_(True)
        E = wgc.forward(box, d)
        (g,) = torch.autograd.grad(E, d)
        den.requires_grad_(False)
        return E, g

    def barrier():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize(dev)

    # ---- device-resident timing -------------------------------------------------------------------
    import ctypes

    def graph_stats():
        c, r = ctypes.c_ulonglong(0), ctypes.c_ulonglong(0)
        lib.pad_graph_stats(ctypes.byref(c), ctypes.byref(r))
        return c.value, r.value

    n_warm = 0
    for _ in range(max(3, args.warmup)):
        step_device()
        n_warm += 1
    # The library captures an evaluation as a CUDA graph the second time it sees an argument set, and the framework's allocator
    # cycles the potential through a few addresses: keep warming up (untimed, at most 16 more steps) until three consecutive steps
    # were pure replays, so that no capture / instantiation (tens of ms of host time) falls into the timed region.
    streak = 0
    while streak < 3 and n_warm < max(3, args.warmup) + 16:
        c0, r0 = graph_stats()
        step_device()
        n_warm += 1
        c1, r1 = graph_stats()
        streak = streak + 1 if (c1 == c0 and r1 > r0) else 0
        if c1 == 0 and r1 == 0 and n_warm >= max(3, args.warmup) + 4:
            break          # graphs are off
    # A freshly started box serves this process's code pages (libcuda, libtorch, the interpreter) from a cold page cache: the
    # first seconds of ANY launch loop see host stalls of milliseconds (measured on fresh boxes: 1.4-2.4 ms of host time per step
    # in the first two bench processes, 0.17-0.2 ms from the third on).  Settle, untimed: blocks of 5 steps until three blocks in
    # a row queue within 25 % of the fastest block seen (at most 3 s / 300 steps).
    best, good, t_settle = float('inf'), 0, time.perf_counter()
    while good < 3 and n_warm < 300 and time.perf_counter() - t_settle < 3.0:
        t0 = time.perf_counter()
        for _ in range(5):
            step_device()
        host = (time.perf_counter() - t0) / 5
        torch.cuda.synchronize(dev)
        n_warm += 5
        best = min(best, host)
        good = good + 1 if host <= 1.25 * best else 0
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    import gc
    # The timed region -- EXACTLY K steps between barrier + synchronise on both sides, max over the ranks -- is taken three times
    # back to back and the MEDIAN region is reported (all three in `repeats_ms_per_step`): one region in five on a freshly
    # started box showed host-side holes (1.5x - 2x the step time with every kernel at its usual duration).
    regions = []
    for rep in range(3):
        gc.collect()
        gc.disable()          # (as timeit does: a collector pass in the middle of the launch loop is host jitter, not the workload)
        gc0 = graph_stats()
        l0, f0 = lib.pad_launch_count(), lib.pad_fft_exec_count()
        ev0.record()
        t_host = time.perf_counter()
        for _ in range(args.steps):
            E, g = step_device()
        ev1.record()
        gc.enable()
        gc1 = graph_stats()
        host_ms = (time.perf_counter() - t_host) * 1e3 / args.steps       # CPU time to queue one step (no sync inside)
        clk = sampler.stop()      # every rank: the queue still holds timed steps, so these samples are taken under load
        barrier()
        own_ms = ev0.elapsed_time(ev1)
        t = torch.tensor([own_ms], dtype=torch.double, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        regions.append({'ms_total': t.item(), 'own_ms': own_ms, 'host_ms': host_ms, 'clocks': clk,
                        'launches': int(lib.pad_launch_count() - l0), 'fft_execs': int(lib.pad_fft_exec_count() - f0),
                        'caps': gc1[0] - gc0[0], 'reps': gc1[1] - gc0[1]})
        sampler = ClockSampler(local)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, E, g)
    pick = sorted(range(3), key=lambda i: regions[i]['ms_total'])[1]
    R = regions[pick]
    graph_caps_timed, graph_reps_timed = R['caps'], R['reps']
    host_enqueue_ms, clocks, launches, fft_execs, ms_total, own_region_ms = R['host_ms'], R['clocks'], R['launches'], R['fft_execs'], R['ms_total'], R['own_ms']
    repeats_ms_per_step = [r['ms_total'] / args.steps for r in regions]
    t = torch.tensor([host_enqueue_ms], dtype=torch.double, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    host_enqueue_ms = t.item()
    per_rank = None
    if world > 1:
        # the reported time is the MAX over the ranks; keep every rank's own figures beside it (which GPU was slow, and was it
        # the GPU -- clock -- or its host process -- enqueue time)
        mine = torch.tensor([own_region_ms / args.steps, float(clocks.get('sm_mhz') or 0.0)], dtype=torch.double, device=dev)
        allr = [torch.empty_like(mine) for _ in range(world)]
        dist.all_gather(allr, mine)
        per_rank = {'ms_per_step': [round(a[0].item(), 4) for a in allr], 'sm_mhz': [a[1].item() for a in allr]}
    ms_per_step = ms_total / args.steps
    value = world * args.steps / (ms_total * 1e-3)

    # ---- live per-kernel timing (CUDA events on the launch stream between the pipeline stages) ----
    stages = []
    if rank == 0:
        import ctypes
        lib.pad_profile_begin()
        for _ in range(5):
            step_device()
        torch.cuda.synchronize(dev)
        names = ctypes.create_string_buffer(48 * 256)
        ms = (ctypes.c_double * 256)()
        n_st, n_ev = ctypes.c_int(0), ctypes.c_int(0)
        lib.pad_profile_end(names, ms, 256, ctypes.byref(n_st), ctypes.byref(n_ev))
        agg = {}
        for i in range(n_st.value):
            nm = names.raw[48 * i:48 * i + 48].split(b'\0')[0].decode()
            a = agg.setdefault(nm, [0.0, 0])
            a[0] += ms[i]
            a[1] += 1
        ns = GRID * GRID * (GRID // 2 + 1)
        for nm, (t_ms, cnt) in agg.items():
            b = stage_bytes(nm, npts, ns)
            if b and nm.startswith('x-fwd * kernel-mix'):
                b *= 2          # both convolutions of an evaluation run this stage over the whole grid
            stages.append({'stage': nm, 'launches_per_eval': cnt, 'ms_per_eval': t_ms,
                           'alg_bytes_per_eval': b,
                           'GBps': (b / (t_ms * 1e-3) / 1e9) if b and t_ms > 0 else None})

    # ---- end to end: pinned host -> device -> E, V -> pinned host ---------------------------------
    # Every step copies its density from pinned host memory and returns E and the potential to pinned host
    # memory.  HostPipeline overlaps the copies of neighbouring steps with the kernels (3 streams); the
    # strictly serial figure (copy in, evaluate, copy out, one stream) is reported next to it.
    from profess_ad_b200.streaming import HostPipeline
    n_e2e = max(6, min(args.steps, 30))
    den_pin = den_h.pin_memory()
    v_pins = [torch.empty_like(den_pin).pin_memory() for _ in range(2)]
    e_pin = torch.empty(n_e2e, dtype=torch.double).pin_memory()
    pipe = HostPipeline(wgc.forward, box, tuple(den.shape), dev, depth=2)
    ins = [den_pin] * n_e2e
    outs = [v_pins[i % 2] for i in range(n_e2e)]
    pipe.run(ins[:4], outs[:4], e_pin[:4])
    barrier()
    # the host link is shared with whatever else runs on the box: three repetitions, the MEDIAN is reported
    # (all three are kept in e2e.repeats)
    e2e_repeats = []
    for _ in range(3):
        ev0.record()
        pipe.run(ins, outs, e_pin)
        ev1.record()
        barrier()
        t = torch.tensor([ev0.elapsed_time(ev1)], dtype=torch.double, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_repeats.append(world * n_e2e / (t.item() * 1e-3))
    e2e_value = sorted(e2e_repeats)[len(e2e_repeats) // 2]
    e_check = float(e_pin[-1])

    den_in = torch.empty_like(den)
    v_pin = v_pins[0]

    def step_e2e():
        den_in.copy_(den_pin, non_blocking=True)
        d = den_in.requires_grad_(True)
        E = wgc.forward(box, d)
        (g,) = torch.autograd.grad(E, d)
        den_in.requires_grad_(False)
        v_pin.copy_(g, non_blocking=True)
        e_pin[0:1].copy_(E.detach().reshape(1), non_blocking=True)

    for _ in range(2):
        step_e2e()
    barrier()
    ev0.record()
    for _ in range(6):
        step_e2e()
    ev1.record()
    barrier()
    t = torch.tensor([ev0.elapsed_time(ev1)], dtype=torch.double, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_serial = world * 6 / (t.item() * 1e-3)
    dV = abs(torch.linalg.det(box_h).item()) / npts

    slab = None
    if world > 1 and not args.no_slab:
        # free the per-GPU 256^3 working set first: the slab plans of a 512^3 / 1024^3 grid want the memory
        del pipe, den_in
        from profess_ad_b200 import _native as _nat
        _nat.release_plans()
        torch.cuda.empty_cache()
        slab = slab_block(world, args.steps, args.warmup)

    if rank == 0:
        peak, peak_src = measured_peak()
        balg = algorithmic_bytes(GRID)
        achieved = balg / (ms_per_step * 1e-3) / 1e9
        line = {
            'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': world, 'steps': args.steps,
            'warmup': n_warm, 'warmup_requested': args.warmup, 'ms_per_step': ms_per_step, 'repeats_ms_per_step': repeats_ms_per_step,
            'higher_is_better': True, 'scaling': 'weak',
            'vs_baseline': None, 'dtype': 'f64', 'data': 'synthetic',
            'config': workload_config(),
            'config_detail': {'per_gpu': 'one independent system per GPU',
                              'l2': 'working set per evaluation (>= 2 GB of fields) exceeds the 126 MB L2',
                              'energy_Ha': e_check, 'per_rank': per_rank},
            'clocks': clocks,
            'e2e': {'value': e2e_value, 'unit': UNIT, 'h2d_bytes_per_step': npts * 8, 'd2h_bytes_per_step': npts * 8 + 8,
                    'how': 'profess_ad_b200.streaming.HostPipeline: H2D / evaluate / D2H of consecutive steps on 3 streams, 2 device buffers',
                    'serial_value': e2e_serial, 'repeats': e2e_repeats,
                    'per_rank_host_link_GBps_each_way': (e2e_value / world) * npts * 8 / 1e9,
                    'numa': numa},
            'gpu_launches': launches + fft_execs,
            'launch_detail': {'own_kernels': launches, 'cufft_execs': fft_execs, 'host_enqueue_ms_per_step': host_enqueue_ms,
                              'graph_captures_in_timed_region': graph_caps_timed, 'graph_replays_in_timed_region': graph_reps_timed},
            'roofline': {'bound': 'hbm', 'achieved': achieved, 'peak': peak, 'unit': 'GB/s', 'frac': achieved / peak,
                         'traffic': NCU_TRAFFIC_256['evaluation'] if GRID == 256 else None,
                         'traffic_source': NCU_TRAFFIC_SOURCE,
                         'peak_source': peak_src,
                         'kernel': 'whole WGC99 E+V evaluation (14 FFTs + fused elementwise passes)',
                         'algorithmic_bytes_per_eval': balg,
                         'kernels': stages},
        }
        if stages:
            dom = max(stages, key=lambda r: r['ms_per_eval'])
            line['roofline']['dominant_kernel'] = {
                'stage': dom['stage'], 'ms_per_eval': dom['ms_per_eval'], 'achieved': dom['GBps'],
                'frac': (dom['GBps'] / peak) if dom['GBps'] else None,
                'traffic_per_launch': NCU_TRAFFIC_256.get(dom['stage']) if GRID == 256 else None,
                'launches_per_eval': dom['launches_per_eval'],
                'note': 'CUDA events on the launch stream around this stage, mean of 5 evaluations'}
        if slab is not None:
            line['slab'] = slab
        if world == 1:
            line['also'] = also_reported(dev, box, den)
        if world == 1 and not args.no_denopt:
            # a fresh start for the second metric: the evaluation legs above leave ~10 GB of plans, staging buffers and cached
            # allocator blocks behind
            del pipe, den_in, v_pins, den_pin
            _native.release_plans()
            torch.cuda.empty_cache()
            line['density_optimization'] = density_optimization_leg(dev, with_cpu=not args.no_cpu_baseline)
        if world == 1 and not args.no_cpu_baseline:
            r = cpu_reference_run(2, 1, max_timed=2, keep=True)
            line['cpu_baseline'] = {'value': r['value'], 'unit': UNIT, 'cores': r['cores'], 'kind': r['kind'], 'sample': r['sample']}
            # parity at the headline size: E and dE/dn of the CPU leg just timed against the GPU's (north_star tolerances:
            # 1e-8 Ha/atom, 1e-9 relative max-abs)
            try:
                E_g, V_g = step_device()
                V_g = (V_g / dV).cpu()
                line['parity'] = {'against': r['kind'], 'grid': [GRID] * 3,
                                  'dE_Ha_per_atom': abs(E_g.item() - r['E']) / (4 * SIDE ** 3),
                                  'dV_rel': ((V_g - r['V']).abs().max() / r['V'].abs().max()).item(),
                                  'E_gpu_Ha': E_g.item(), 'E_cpu_Ha': r['E'],
                                  'tolerance': {'dE_Ha_per_atom': 1e-8, 'dV_rel': 1e-9}}
            except Exception as e:      # noqa: BLE001
                line['parity'] = {'error': repr(e)}
            try:        # SURVEY.md section 8(d): also at one thread (bounded: 2 evaluations at 128^3, scaled N log N)
                r1 = cpu_reference_run(2, 1, sample_grid=min(GRID, 128), threads=1, max_timed=2)
                line['cpu_baseline']['one_thread'] = {'value': r1['value'], 'unit': UNIT, 'cores': 1, 'sample': r1['sample']}
            except Exception as e:      # noqa: BLE001
                line['cpu_baseline']['one_thread'] = {'error': repr(e)}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def dump_outputs(out_dir, E, g):
    """--dump-outputs: what the last timed step handed its caller, as float64 .npy files, so that two builds can be compared
    output for output.  energy.npy is E (Ha); grad_sample.npy is dE/dn (the autograd gradient with respect to the density) at
    DUMP_POINTS grid points drawn with a fixed seed, in ascending flat (C-order) index -- the whole field if the grid is smaller
    (at 256^3 the field alone is 128 MB)."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    flat = g.detach().reshape(-1)
    if flat.numel() > DUMP_POINTS:
        idx = torch.randperm(flat.numel(), generator=torch.Generator().manual_seed(DUMP_SEED))[:DUMP_POINTS].sort().values
        flat = flat[idx.to(flat.device)]
    np.save(os.path.join(out_dir, 'energy.npy'), np.array([E.item()], dtype=np.float64))
    np.save(os.path.join(out_dir, 'grad_sample.npy'), flat.double().cpu().numpy())


def also_reported(dev, box, den):
    """SURVEY.md section 8(d), "also reported": E+V evaluations per second of the other non-local kinetic functionals and
    of the full term stack at 256^3, and of WGC99 at 128^3 (device-resident inputs, CUDA events, 20 evaluations each)."""
    import torch
    import profess_ad_b200.functionals as F
    from profess_ad_b200 import _density_opt as D
    from profess_ad_b200.synthetic import smooth_supercell

    def rate(fn, n=20):
        for _ in range(3):
            fn()
        torch.cuda.synchronize(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            fn()
        e1.record()
        torch.cuda.synchronize(dev)
        return n / (e0.elapsed_time(e1) * 1e-3)

    def ev(f, b, d):
        def go():
            x = d.requires_grad_(True)
            E = f(b, x)
            torch.autograd.grad(E, x)
            d.requires_grad_(False)
        return go
    out = {}
    try:
        out['WangTeter E+V, 256^3'] = rate(ev(F.WangTeter, box, den))
        out['WangGovindCarter98 E+V, 256^3'] = rate(ev(F.WangGovindCarter98, box, den))
        out['PerdewBurkeErnzerhof E+V, 256^3'] = rate(ev(F.PerdewBurkeErnzerhof, box, den))
        terms = [F.IonElectron, F.Hartree, F.WangGovindCarter99().forward, F.PerdewZunger]
        T = D.describe_terms(terms)
        v_ext = -0.1 * den / den.mean()
        out['IonElectron + Hartree + WGC99 + PerdewZunger E+V (fused term list), 256^3'] = rate(lambda: D.eval_total(box, den, v_ext, T))
        b128, d128 = smooth_supercell(128, 2, device=dev)
        out['WangGovindCarter99 E+V, 128^3'] = rate(ev(F.WangGovindCarter99().forward, b128, d128), 50)
    except Exception as e:      # noqa: BLE001 -- the headline line must still be printed
        out['error'] = repr(e)
    return {'unit': UNIT, 'values': out}


def _denopt_workloads():
    """(name, box_bohr, shape, frac, terms-as-names): BASELINE.json metric 2 workloads.  The first two are small enough for the
    reference's CPU path to run next to the GPU in the default bench (SURVEY.md section 8d); the 256^3 one is GPU only."""
    import torch
    from profess_ad_b200.synthetic import fcc_supercell
    a0 = 0.529177210903
    box1 = (4 * 16.8) ** (1.0 / 3.0) / a0 * torch.eye(3, dtype=torch.double)          # crystal_tools.get_cell('fcc-c', 16.8 A^3/atom)
    frac1 = torch.tensor([[0.0, 0.0, 0.0], [0.0, 0.5, 0.5], [0.5, 0.0, 0.5], [0.5, 0.5, 0.0]], dtype=torch.double)
    box4, frac4 = fcc_supercell(4)
    cfg1 = ['IonElectron', 'Hartree', 'ThomasFermi', 'Weizsaecker', 'PerdewZunger']
    wgc = ['IonElectron', 'Hartree', 'WangGovindCarter99', 'PerdewZunger']
    return [
        ('BASELINE.json configs[0]: fcc Al 4-atom cell, ecut2shape(1600 eV), TF + vW + Hartree + PZ + IonElectron', box1, None, frac1, cfg1, True),
        ('Al 256-atom fcc supercell, 64^3 grid, IonElectron + Hartree + WGC99 + PZ', box4, (64,) * 3, frac4, wgc, True),
        ('Al 256-atom fcc supercell, 128^3 grid, IonElectron + Hartree + WGC99 + PZ', box4, (128,) * 3, frac4, wgc, False),
        ('Al 256-atom fcc supercell, 256^3 grid, IonElectron + Hartree + WGC99 + PZ', box4, (256,) * 3, frac4, wgc, False),
    ]


def _terms(F, names):
    return [F.WangGovindCarter99().forward if n == 'WangGovindCarter99' else getattr(F, n) for n in names]


def density_optimization_leg(dev, with_cpu=True):
    """BASELINE.json metric 2, "s per density optimisation": System.optimize_density(ntol=1e-7, LBFGS, from uniform) with the
    tests/potentials/al.gga.recpot local pseudopotential; wall clock around the public call, the faster of the last two of three runs on the GPU (garbage collector off inside a run).
    For the two small workloads the UNMODIFIED reference's System (oracle/_ref) runs the same call on the host cores."""
    import torch
    import profess_ad_b200.functionals as F
    from profess_ad_b200.system import System
    pot = os.path.join(ROOT, 'tests', 'potentials', 'al.gga.recpot')
    ref = None
    if with_cpu:
        try:
            from oracle import ref_loader
            ref = ref_loader.load_reference()
        except Exception:      # noqa: BLE001
            ref = None
    out = []
    for name, box, shape, frac, term_names, cpu_ok in _denopt_workloads():
        row = {'workload': name}
        try:
            shp = tuple(shape) if shape is not None else tuple(int(x) for x in System.ecut2shape(1600, box * 0.529177210903))
            row['grid'] = list(shp)
            s = System(box, shp, [['Al', pot, frac]], _terms(F, term_names), units='b', coord_type='fractional', device=dev)
            dt = None
            import gc
            for _ in range(3):          # minimum of the last two of three runs; the collector is off inside a run (as timeit does):
                gc.collect()            # the loop is host-driven, a generation-2 pass over this process's objects shows up in it
                gc.disable()
                try:
                    torch.cuda.synchronize(dev)
                    t0 = time.perf_counter()
                    s.optimize_density(ntol=1e-7, n_method='LBFGS', from_uniform=True)
                    torch.cuda.synchronize(dev)
                    t_run = time.perf_counter() - t0
                finally:
                    gc.enable()
                dt = t_run if (dt is None or _ == 1) else min(dt, t_run)
            info = s.last_optimization
            n_at = frac.shape[0]
            row.update({'seconds': dt, 'iterations': info.get('iterations'), 'closures': info.get('closures'),
                        'converged': bool(info.get('converged')), 'energy_eV_per_atom': s.energy('eV') / n_at,
                        'optimizer': 'device-resident L-BFGS' if info.get('native') else 'host-driven L-BFGS'})
            del s
        except Exception as e:      # noqa: BLE001 -- the headline line must still be printed
            row['error'] = repr(e)
        row['_cpu'] = (box, shp, frac, term_names, cpu_ok) if 'error' not in row else None
        out.append(row)
    # the CPU references AFTER all GPU runs: their 16 OpenMP workers keep spinning for a while after a parallel region and
    # would compete with the host thread that drives the next GPU optimisation (measured: 128^3 0.14 -> 0.56 s)
    for row in out:
        cpu = row.pop('_cpu', None)
        if cpu is None:
            continue
        box, shp, frac, term_names, cpu_ok = cpu
        dt, n_at = row['seconds'], frac.shape[0]
        try:
            if cpu_ok and ref is not None:
                torch.set_num_threads(host_cores())
                RF = ref.functionals
                rs = ref.system.System(box.clone(), shp, [['Al', pot, frac.clone()]], _terms(RF, term_names), units='b',
                                       coord_type='fractional')
                t0 = time.perf_counter()
                rs.optimize_density(ntol=1e-7, n_method='LBFGS', from_uniform=True)
                cpu_dt = time.perf_counter() - t0
                e_ref = rs.energy('eV') / n_at
                row['cpu_reference'] = {'seconds': cpu_dt, 'cores': torch.get_num_threads(), 'kind': 'reference',
                                        'energy_eV_per_atom': e_ref, 'sample': 'one full System.optimize_density of the unmodified reference (oracle/_ref), all host threads'}
                row['dE_eV_per_atom_vs_reference'] = abs(row['energy_eV_per_atom'] - e_ref)
                row['speedup_vs_cpu_reference'] = cpu_dt / dt
                del rs
        except Exception as e:      # noqa: BLE001 -- the headline line must still be printed
            row['cpu_reference'] = {'error': repr(e)}
    return out


# --------------------------------------------------------------------------------------------------
#  one large grid over N GPUs (slab-decomposed FFT, all-to-all over NVLink): strong scaling
# --------------------------------------------------------------------------------------------------
def slab_measure(n, functional, steps, warmup, overlap=None):
    """One strong-scaling measurement (torch.distributed must be initialised): dict for the JSON line."""
    import torch
    import torch.distributed as dist
    import profess_ad_b200.functionals as F
    from profess_ad_b200 import parallel
    from profess_ad_b200.synthetic import smooth_supercell
    rank, world = dist.get_rank(), dist.get_world_size()
    dev = torch.device('cuda', torch.cuda.current_device())
    side = max(1, n // 64)
    lo, hi = parallel.slab_bounds(n, rank, world)
    box, den = smooth_supercell(n, side, device=dev, x_range=(lo, hi))
    n_fft = N_FFT
    hc = None
    if functional == 'wgc99':
        fun, label = F.WangGovindCarter99().forward, 'WangGovindCarter99'
    elif functional == 'pbe':
        fun, label, n_fft = F.PerdewBurkeErnzerhof, 'PerdewBurkeErnzerhof', 8
    else:       # BASELINE.json configs[2]: Huang-Carter field-dependent spline kernel
        hc = F.RevisedHuangCarter((0.45, 0.10, 2.0 / 3.0, 1.15)) if functional == 'revhc' else F.HuangCarter((0.01177, 0.7143, 1.2))
        fun, label = hc.forward, type(hc).__name__
    if overlap is None:
        overlap = os.environ.get('PAD_SLAB_OVERLAP', '1') != '0'
    path = {}
    with parallel.slab((n, n, n), overlap=overlap) as ctx:
        def step():
            d = den.requires_grad_(True)
            E = fun(box, d)
            (g,) = torch.autograd.grad(E, d)
            den.requires_grad_(False)
            return E, g
        for _ in range(max(3, warmup)):
            E, g = step()
        torch.cuda.synchronize(dev)
        dist.barrier()
        torch.cuda.synchronize(dev)
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        for _ in range(steps):
            E, g = step()
        ev1.record()
        torch.cuda.synchronize(dev)
        dist.barrier()
        t = torch.tensor([ev0.elapsed_time(ev1)], dtype=torch.double, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = t.item() / steps
        e_val = E.item()
        plan = next(iter(ctx.plans.values()), None)
        lib = plan.lib if plan is not None else None
        fused = bool(plan is not None and lib.pad_fast_fft_supported(plan.handle)) and functional in ('wgc99',)
        if fused and plan.peer is not None:
            path = {'transforms': 'own z / y / x FFT passes per rank; the forward y pass stores its rows into the owner ranks\' transposed '
                                  'buffers and the fused x pass (kernel mix inside) stores its planes into the owners\' local buffers '
                                  'over NVLink (symmetric memory), barriers instead of all-to-alls', 'exchange': 'peer stores'}
        elif fused:
            path = {'transforms': 'own z / y / x FFT passes per rank, y pass stores rows blocked by destination rank, NCCL all-to-all '
                                  'pipelined over two stagings', 'exchange': 'all_to_all_single'}
        elif plan is not None and getattr(plan, 'recv_sym', None) is not None:
            path = {'transforms': 'batched 2-D (y,z) cuFFT, pack kernel that stores straight into the owner ranks\' receive buffers over '
                                  'NVLink (symmetric memory) + barrier, strided 1-D (x) cuFFT per 3-D transform', 'exchange': 'peer stores'}
        else:
            path = {'transforms': 'batched 2-D (y,z) cuFFT + NCCL all-to-all + strided 1-D (x) cuFFT per 3-D transform',
                    'exchange': 'all_to_all_single'}
    npts = n ** 3
    if hc is not None:
        n_fft = 12 + 2 * int(getattr(hc, 'last_n_nodes', 0))
    balg = 16 * npts * n_fft + 16 * npts
    peak, peak_src = measured_peak()
    nk = n * n * (n // 2 + 1)
    a2a_bytes = n_fft * (world - 1) / world ** 2 * nk * 16       # per GPU and direction, per evaluation
    return {
        'metric': f'{"WGC99" if functional == "wgc99" else label} energy+potential evaluations per second at {n}^3, one grid slab-decomposed over the GPUs',
        'value': 1e3 / ms, 'unit': UNIT, 'n_gpus': world, 'steps': steps, 'warmup': max(3, warmup),
        'ms_per_step': ms, 'higher_is_better': True, 'scaling': 'strong', 'vs_baseline': None, 'dtype': 'f64',
        'data': 'synthetic',
        'config': {'workload': f'Al {4 * side ** 3}-atom supercell, {label} E+V, {n}^3 grid, slabs of {n // world} planes per GPU',
                   'n_fft': n_fft, 'grid': [n] * 3, 'energy_Ha': e_val,
                   'transforms': path.get('transforms'), 'exchange': path.get('exchange'), 'exchange_overlap': bool(overlap)},
        'roofline': {'bound': 'hbm', 'achieved': balg / (ms * 1e-3) / 1e9 / world, 'peak': peak, 'unit': 'GB/s',
                     'frac': balg / (ms * 1e-3) / 1e9 / world / peak, 'traffic': None, 'peak_source': peak_src,
                     'algorithmic_bytes_per_eval': balg, 'per': 'GPU',
                     'nvlink_bytes_per_gpu_per_eval_each_way': a2a_bytes,
                     'nvlink_GBps_each_way': a2a_bytes / (ms * 1e-3) / 1e9},
    }


def slab_geometry_step(n, steps=2):
    """BASELINE.json configs[4]: one geometry-optimisation step's worth of derivatives on ONE n^3 grid over the ranks for a bcc Li
    supercell: PerdewBurkeErnzerhof E + dE/dn, its stress, the ion-electron forces of every atom and the ion-electron stress
    (everything that scales with the grid; v_ext is built once per geometry and timed separately)."""
    import torch
    import torch.distributed as dist
    import profess_ad_b200.functionals as F
    from profess_ad_b200 import parallel, ion_utils as IU
    from profess_ad_b200.functional_tools import get_stress
    from profess_ad_b200.synthetic import smooth_supercell
    rank, world = dist.get_rank(), dist.get_world_size()
    dev = torch.device('cuda', torch.cuda.current_device())
    side = max(1, n // 64)
    lo, hi = parallel.slab_bounds(n, rank, world)
    box, den = smooth_supercell(n, side, device=dev, x_range=(lo, hi))           # smooth density on the same cubic cell
    den = den * (2.0 / 12.0)                                                     # 2 atoms x 1 e- per cell instead of 4 x 3
    r = torch.arange(side, dtype=torch.double)
    cells = torch.stack(torch.meshgrid(r, r, r, indexing='ij'), dim=-1).reshape(-1, 1, 3)
    basis = torch.tensor([[0.0, 0.0, 0.0], [0.5, 0.5, 0.5]], dtype=torch.double)
    frac = ((cells + basis[None]) / side).reshape(-1, 3).to(dev)
    pot = os.path.join(ROOT, 'tests', 'potentials', 'li.gga.recpot')
    species = [(pot, frac)]

    def timed(fn, reps):
        fn()
        torch.cuda.synchronize(dev)
        dist.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            out = fn()
        e1.record()
        torch.cuda.synchronize(dev)
        t = torch.tensor([e0.elapsed_time(e1) / reps], dtype=torch.double, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t.item(), out
    with parallel.slab((n, n, n)) as ctx:
        def ev():
            d = den.requires_grad_(True)
            E = F.PerdewBurkeErnzerhof(box, d)
            (g,) = torch.autograd.grad(E, d)
            den.requires_grad_(False)
            return E
        ms_vext, _ = timed(lambda: IU.ionic_potential(box, ctx.local_shape, species), 1)
        ms_ev, E = timed(ev, max(steps, 3))
        ms_st, _ = timed(lambda: get_stress(box, den, F.PerdewBurkeErnzerhof), steps)
        ms_f, _ = timed(lambda: IU.ion_electron_forces(box, den, species), 1)
        ms_is, _ = timed(lambda: IU.ion_electron_stress(box, den, species), 1)
        # the same three with the particle-mesh Ewald structure factor of order 8 (System(pme_order=8)): O(N log N + N_ion 8^3)
        # instead of O(N_k N_ion) -- what a run of this size uses in the reference as well (the exact structure factor of 8192 ions
        # on 1024^3 is a 34-TB phase tensor there)
        pme = {}
        try:
            pme['v_ext build (once per geometry)'], _ = timed(lambda: IU.ionic_potential(box, ctx.local_shape, species, pme_order=8), 2)
            pme['ion-electron forces'], f_pme = timed(lambda: IU.ion_electron_forces(box, den, species, pme_order=8), 2)
            pme['ion-electron stress'], _ = timed(lambda: IU.ion_electron_stress(box, den, species, pme_order=8), 2)
            f_exact = IU.ion_electron_forces(box, den, species)
            # (ions on perfect lattice sites in a density with the lattice's symmetry: the exact forces vanish up to rounding, so
            #  the numbers below are absolute, Ha/bohr -- what is left in F_pme is the order-8 mesh error)
            pme['max |F_exact| Ha/bohr'] = f_exact.abs().max().item()
            pme['max |F_pme| Ha/bohr'] = f_pme.abs().max().item()
        except Exception as e:      # noqa: BLE001
            pme['error'] = repr(e)
        e_val = E.item()
    npts = n ** 3
    peak, _ = measured_peak()
    balg = 16 * npts * 8 + 16 * npts
    nk = n * n * (n // 2 + 1)
    a2a = 8 * (world - 1) / world ** 2 * nk * 16
    return {'workload': f'bcc Li {frac.shape[0]}-atom supercell, {n}^3 grid: PBE E+V, PBE stress, ion-electron forces + stress (BASELINE.json configs[4])',
            'n_gpus': world, 'grid': [n] * 3, 'atoms': int(frac.shape[0]),
            'ms': {'PBE E+V': ms_ev, 'PBE stress': ms_st, 'ion-electron forces': ms_f, 'ion-electron stress': ms_is,
                   'v_ext build (once per geometry)': ms_vext},
            'ms_pme_order_8': pme,
            'ms_per_step': ms_ev + ms_st + ms_f + ms_is,
            'ms_per_step_pme_order_8': (ms_ev + ms_st + pme['ion-electron forces'] + pme['ion-electron stress']) if 'error' not in pme else None,
            'energy_Ha': e_val,
            'PBE_E+V_hbm_frac_per_gpu': balg / (ms_ev * 1e-3) / 1e9 / world / peak,
            'PBE_E+V_nvlink_GBps_each_way': a2a / (ms_ev * 1e-3) / 1e9}


def slab_block(world, steps, warmup):
    """`slab` entries of the N > 1 line: one grid over the N GPUs (strong scaling).  512^3 WangGovindCarter99 and
    RevisedHuangCarter (BASELINE.json configs[2]) at every N; the 1024^3 PBE geometry step (configs[4]) where it fits."""
    import torch
    out = []
    plan = [('wgc99', 512, min(steps, 10)), ('revhc', 512, min(steps, 5))]
    for fun, n, k in plan:
        try:
            m = slab_measure(n, fun, max(2, k), min(warmup, 3))
            out.append({'workload': m['config']['workload'], 'metric': m['metric'], 'n_gpus': world, 'grid': [n] * 3,
                        'ms_per_eval': m['ms_per_step'], 'evals_per_s': m['value'], 'n_fft': m['config']['n_fft'],
                        'energy_Ha': m['config']['energy_Ha'],
                        'hbm_frac_per_gpu': m['roofline']['frac'], 'hbm_GBps_per_gpu': m['roofline']['achieved'],
                        'nvlink_GBps_each_way': m['roofline']['nvlink_GBps_each_way'],
                        'nvlink_frac_of_900': m['roofline']['nvlink_GBps_each_way'] / 900.0,
                        'transforms': m['config']['transforms'], 'exchange': m['config']['exchange'],
                        'exchange_overlap': m['config']['exchange_overlap']})
        except Exception as e:      # noqa: BLE001 -- the headline line must still be printed
            out.append({'workload': f'{fun} {n}^3', 'error': repr(e)})
        torch.cuda.empty_cache()
    if world >= 8:
        try:
            out.append(slab_geometry_step(1024))
        except Exception as e:      # noqa: BLE001
            out.append({'workload': 'PBE geometry step 1024^3', 'error': repr(e)})
        torch.cuda.empty_cache()
    return out


def slab_init():
    import torch
    import torch.distributed as dist
    rank, world, local = dist_env()
    if not torch.cuda.is_available():
        raise RuntimeError('bench.py: no CUDA device; the B200 arm has no CPU fallback (use --impl reference)')
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
    os.environ.setdefault('MASTER_PORT', '29533')
    if not dist.is_initialized():
        # high-priority NCCL stream: the exchange of one field is meant to run WHILE the FFT kernels of the next one
        # fill the SMs (pipelined batches in csrc/plan.cu); its CTAs must not queue behind them
        opts = dist.ProcessGroupNCCL.Options(is_high_priority_stream=True)
        dist.init_process_group('nccl', rank=rank, world_size=world, device_id=dev, pg_options=opts)
    return rank, world


def run_slab(args):
    import torch.distributed as dist
    rank, world = slab_init()
    line = slab_measure(args.slab_grid, args.slab_functional, args.steps, args.warmup)
    if rank == 0:
        print(json.dumps(line), flush=True)
    dist.destroy_process_group()


class CleanStdout:
    """The driver reads ONE JSON line from stdout.  Libraries write there too (NCCL prints its version banner from
    inside ncclCommInit whatever NCCL_DEBUG says): while the benchmark runs, file descriptor 1 points at stderr, and
    print() of the result line goes to the real stdout."""

    def __enter__(self):
        sys.stdout.flush()
        self.real = os.dup(1)
        os.dup2(2, 1)
        self.prev = sys.stdout
        sys.stdout = os.fdopen(self.real, 'w', buffering=1, closefd=False)
        return self

    def __exit__(self, *exc):
        sys.stdout.flush()
        sys.stdout = self.prev
        os.dup2(self.real, 1)
        os.close(self.real)
        return False


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=50,
                    help='evaluations in each timed region (three regions back to back, the median one is reported)')
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-denopt', action='store_true', help='skip the density-optimisation timing leg')
    ap.add_argument('--no-slab', action='store_true', help='N > 1: skip the one-grid-over-N-GPUs (slab) block')
    ap.add_argument('--slab-functional', default='wgc99', choices=['wgc99', 'hc', 'revhc', 'pbe'],
                    help='functional evaluated in --slab-grid mode')
    ap.add_argument('--slab-grid', type=int, default=0,
                    help='strong-scaling mode: ONE n^3 grid slab-decomposed over the --gpus ranks (e.g. 512)')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='after the timed steps, write what the last one returned (energy, seeded sample of dE/dn) as DIR/<name>.npy')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and (args.impl != 'b200' or args.slab_grid):
        ap.error('--dump-outputs writes the outputs of the headline B200 run only')
    with CleanStdout():
        if args.impl == 'reference':
            run_reference(args)
        elif args.slab_grid:
            run_slab(args)
        else:
            run_gpu(args)


if __name__ == '__main__':
    main()
