"""Benchmark of the Shamir hot path: BASELINE.json's metric "GF(p) Shamir share+recombine pairs/sec".

    python bench.py --gpus 1 --steps 10 --warmup 3             (N > 1: launched with torch.distributed.run)
    python bench.py --impl reference --steps 3 --warmup 1       (CPU port of the reference's algorithm)

One step = one pass of the hot path over one batch: share generation of n secrets (degree t, m
parties; coefficient matrix resident in HBM, "parity mode") followed by Lagrange recombination of
t+1 of the resulting share rows.  One *pair* = one secret split + recombined.

Workloads (--workload):
    c3   (default, BASELINE.json configs[2]) p = 2^128-173, m=5, t=2, n = 10^8 per GPU
    ns64 (north_star's 64-bit case)          p = 2^64-189,  m=3, t=1, n = 2*10^8 per GPU
    c5   (configs[4] field/shape)            p = 2^256-189, m=7, t=3, n = 2*10^7 per GPU, recombine 2t+1
    modmul (configs[1])                      p = 2^64-189 elementwise a*b, n = 10^8 (value = elem/s)

The element axis is sharded over the GPUs with no data-path collective (weak scaling: n per GPU fixed).
Printed JSON line: see the driver's contract; extra keys `roofline`, `cpu_baseline`, `e2e`, `clocks`, and
    sustained        the same step repeated for >= 2 s after the K timed steps (clocks / power under sustained load)
    extra            (N = 1, default workload) short full-size passes of the other configurations in the SAME process:
                     ns64, c5, c3g, c4, modmul, modmul_generic, prss -- kernel times and roofline fractions
    multi_selftest   (N > 1) sharded == single-GPU, NCCL gather, both co-located reshare forms, checked before timing
    gather           (N > 1) the one collective of the path (SURVEY 8e): all-gather of the recombined vector, timed
    numa             the NUMA node / CPU set this rank bound itself to before allocating pinned memory
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    'c3': dict(p=2**128 - 173, m=5, t=2, k=3, n=100_000_000, name='shamir split+recombine p=2^128-173 m=5 t=2 n=1e8/GPU (BASELINE configs[2])'),
    'ns64': dict(p=2**64 - 189, m=3, t=1, k=2, n=200_000_000, name='shamir split+recombine p=2^64-189 m=3 t=1 n=2e8/GPU (north_star 64-bit case)'),
    'c5': dict(p=2**256 - 189, m=7, t=3, k=7, n=20_000_000, name='shamir reshare p=2^256-189 m=7 t=3 recombine 2t+1 n=2e7/GPU (configs[4] shape)'),
    'modmul': dict(p=2**64 - 189, m=0, t=0, k=0, n=100_000_000, name='elementwise modmul p=2^64-189 n=1e8/GPU (BASELINE configs[1])'),
    'modmul_generic': dict(p=9409569905028393239, m=0, t=0, k=0, n=100_000_000, name='elementwise modmul generic 64-bit prime 9409569905028393239 (Montgomery) n=1e8/GPU (BASELINE configs[1])'),
    'c3g': dict(p=0x800000000000000000000000000000fb, m=5, t=2, k=3, n=100_000_000, name='shamir split+recombine GENERIC 128-bit prime (Montgomery path) m=5 t=2 n=1e8/GPU'),
    'prss': dict(p=2**256 - 189, m=7, t=3, k=0, n=1 << 21, prss=True, name='PRSS np_pseudorandom_share p=2^256-189 m=7 t=3 (20 key subsets, 48-byte PRF chunks): combine kernel on n=2^21 resident bytes; e2e at np_cnnmnist call size n=213,248 (configs[4] shape)'),
    'c4': dict(p=283, binary=True, m=3, t=1, k=3, n=1 << 28, name='GF(2^8) reshare (np_aes field, modulus 283) m=3 t=1 recombine 2t+1, batched n=2^28 bytes/GPU + per-call latency at n=16 (BASELINE configs[3] shape)'),
}
METRIC = 'GF(p) Shamir share+recombine pairs/sec'


def peaks():
    path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(path):
        try:
            return float(json.load(open(path))['hbm_gbs']), 'measured (MEASURED_PEAKS.json)'
        except Exception:
            pass
    return 6650.0, 'fallback (B200_PROFILING.md)'


def ncu_traffic(workload, kernel):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernel, from the committed
    `ncu --set full` summary of the same workload (profiles/), or (None, None)."""
    import glob
    import re
    for path in sorted(glob.glob(os.path.join(ROOT, 'profiles', f'r*_ncu_{kernel}_{workload}.txt')), reverse=True):
        total, units = 0.0, {'Gbyte': 1e9, 'Mbyte': 1e6, 'Kbyte': 1e3, 'byte': 1.0, 'Tbyte': 1e12}
        for line in open(path):
            mt = re.match(r'\s*dram__bytes_(read|write)\.sum\s+([0-9.]+)\s+(\w+)', line)
            if mt:
                total += float(mt.group(2)) * units.get(mt.group(3), 1.0)
        if total:
            return total, os.path.relpath(path, ROOT)
    return None, None


class ClockSampler:
    """SM clock, power and throttle reasons polled from a thread every ~2 ms (NVML through nvidia_ml_py).  The thread is
    started BEFORE the warm-up so that it is certainly running when the timed region begins; report(t0, t1) keeps the
    samples whose time stamp lies inside [t0, t1] (perf_counter), so a 30 ms region still gets its own samples."""
    BAD = {0x8: 'hw_slowdown', 0x40: 'hw_thermal_slowdown', 0x20: 'sw_thermal_slowdown', 0x4: 'sw_power_cap'}

    def __init__(self, index):
        self.index, self.rows, self.stop_flag, self.thread, self.max = index, [], False, None, None

    def _poll(self):
        import pynvml as nv
        h = nv.nvmlDeviceGetHandleByIndex(self.index)
        self.max = float(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM))
        while not self.stop_flag:
            mhz = float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
            try:
                power = nv.nvmlDeviceGetPowerUsage(h) / 1000.0
                mask = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
            except Exception:   # noqa: BLE001
                power, mask = None, 0
            self.rows.append((time.perf_counter(), mhz, power, mask))
            time.sleep(0.002)

    def start(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            self.thread = threading.Thread(target=self._poll, daemon=True)
            self.thread.start()
            time.sleep(0.02)
        except Exception as exc:   # noqa: BLE001
            self.thread = None
            self.error = repr(exc)

    def report(self, t0, t1):
        if self.thread is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvml unavailable: ' + getattr(self, 'error', '?')]}
        rows = [r for r in list(self.rows) if t0 <= r[0] <= t1]
        inside = len(rows)
        if not rows:                # region shorter than one polling interval: the nearest samples on either side
            rows = sorted(list(self.rows), key=lambda r: min(abs(r[0] - t0), abs(r[0] - t1)))[:2]
        sm = sorted(r[1] for r in rows)
        power = [r[2] for r in rows if r[2] is not None]
        reasons = set()
        for r in rows:
            for bit, name in self.BAD.items():
                if r[3] & bit:
                    reasons.add(name)
        return {'sm_mhz': sm[len(sm) // 2] if sm else None, 'sm_max_mhz': self.max, 'samples': len(rows),
                'samples_inside_region': inside, 'power_w_max': max(power) if power else None,
                'reasons': sorted(reasons), 'source': 'nvml'}

    def stop(self):
        self.stop_flag = True
        if self.thread is not None:
            self.thread.join(timeout=2)


def bind_to_gpu_numa(index):
    """Pin this process to the CPUs of the NUMA node its GPU hangs off (before CUDA is initialised and before any
    pinned host memory is allocated: first-touch then puts the staging buffers next to the GPU's PCIe root port).
    Round 1's 8-GPU e2e curve (0.63) came from ranks 4-7 pinning memory on the far socket."""
    info = {'bound': False}
    try:
        import pynvml as nv
        nv.nvmlInit()
        bus = nv.nvmlDeviceGetPciInfo(nv.nvmlDeviceGetHandleByIndex(index)).busId
        bus = bus.decode() if isinstance(bus, bytes) else bus
        dom, rest = bus.split(':', 1)
        path = f'/sys/bus/pci/devices/{dom[-4:].lower()}:{rest.lower()}/numa_node'
        node = int(open(path).read().strip())
        info['pci'] = bus
        info['node'] = node
        if node < 0:
            return info
        cpus = set()
        for part in open(f'/sys/devices/system/node/node{node}/cpulist').read().strip().split(','):
            lo, _, hi = part.partition('-')
            cpus.update(range(int(lo), int(hi or lo) + 1))
        allowed = os.sched_getaffinity(0) & cpus
        if allowed:
            os.sched_setaffinity(0, allowed)
            info.update(bound=True, cpus=len(allowed))
    except Exception as exc:   # noqa: BLE001
        info['error'] = repr(exc)[:200]
    return info


# ---------------------------------------------------------------------------------------------------
# CPU arm: the oracle port of the reference's NumPy-object path (np_random_split + np_recombine)
# ---------------------------------------------------------------------------------------------------

def reference_path():
    """Where the UNMODIFIED reference is importable from on this box: $MPYC_REFERENCE, or baseline/_ref (pip install
    --target of the checkout, tools/install_reference.sh; git-ignored, travels with gpurun).  None: only the oracle
    port (oracle/shamir_oracle.py) is available."""
    for cand in (os.environ.get('MPYC_REFERENCE'), os.path.join(ROOT, 'baseline', '_ref')):
        if cand and os.path.isfile(os.path.join(cand, 'mpyc', 'thresha.py')):
            return cand
    return None


_REFMOD = {}


def _reference_modules():
    """(finfields, thresha) of the real reference, imported once per process (MPyC parses sys.argv at import)."""
    if not _REFMOD:
        path = reference_path()
        if path is None:
            _REFMOD['mods'] = None
        else:
            argv, sys.argv = sys.argv, [sys.argv[0], '--no-log']
            sys.path.insert(0, path)
            try:
                from mpyc import finfields, thresha
                _REFMOD['mods'] = (finfields, thresha)
            except Exception:   # noqa: BLE001
                _REFMOD['mods'] = None
            finally:
                sys.argv = argv
    return _REFMOD['mods']


def _cpu_pairs(args):
    """One process: split + recombine `n` pairs `reps` times on the CPU.  With the reference importable this is
    thresha.np_random_split + thresha.np_recombine themselves (stock code path: secrets.randbelow per coefficient,
    NumPy object matmul); otherwise the oracle port of the same two functions."""
    p, m, t, k, n, reps, with_rng = args
    import secrets
    import numpy as np
    from oracle import shamir_oracle as orc
    vals = orc.synth_elements(p, n, 20260923)
    s = np.array(vals, dtype=object)
    mods = _reference_modules() if with_rng else None
    if mods is not None:
        finfields, thresha = mods
        F = finfields.GF(p)
        a = F.array(s)
        t0 = time.perf_counter()
        for _ in range(reps):
            sh = thresha.np_random_split(F, a, t, m)
            out = thresha.np_recombine(F, [(i + 1, sh[i]) for i in range(k)])
        dt = time.perf_counter() - t0
        assert out.value.tolist() == vals
        return n * reps, dt, 'reference'
    C = np.array(orc.np_stream_to_C(orc.synth_elements(p, t * n, 7, stream=2), t, n), dtype=object) if t else np.empty((0, n), dtype=object)
    xs = tuple(range(1, k + 1))
    t0 = time.perf_counter()
    for _ in range(reps):
        Cr = orc.np_draw_coefficients(p, t, n, secrets.randbelow) if with_rng else C
        sh = orc.np_split(p, s, Cr, m)
        out = orc.np_recombine(p, xs, sh[:k])
    dt = time.perf_counter() - t0
    assert out.tolist() == vals
    return n * reps, dt, 'port'


def cpu_baseline(w, n=20000, target_s=12.0):
    """1 core, bounded sample; returns the cpu_baseline object.  kind 'reference': mpyc.thresha itself (baseline/_ref
    or $MPYC_REFERENCE); kind 'port': oracle/shamir_oracle.py, its restatement pinned by the golden fixtures."""
    pairs, dt, kind = _cpu_pairs((w['p'], w['m'], w['t'], w['k'], n, 1, True))
    reps = max(1, int(target_s * 0.7 / max(dt, 1e-3)))
    pairs, dt, kind = _cpu_pairs((w['p'], w['m'], w['t'], w['k'], n, reps, True))
    pairs2, dt2, _ = _cpu_pairs((w['p'], w['m'], w['t'], w['k'], n, max(1, reps // 2), False))
    what = ('mpyc.thresha.np_random_split + np_recombine of the unmodified reference (gmpy2 absent: its own stubs)' if kind == 'reference'
            else 'oracle port np_split+np_recombine (NumPy object arrays, coefficients via secrets.randbelow as the reference does)')
    return {'value': pairs / dt, 'unit': 'pairs/s', 'cores': 1, 'kind': kind,
            'sample': f'{what} on {n} elements x {reps} reps, 1 process', 'value_without_rng_port': pairs2 / dt2}


_REF = {}


def _ref_init(p, m, t, k, n):
    """Pool initializer: every worker builds its inputs once (outside the timed steps)."""
    import numpy as np
    from oracle import shamir_oracle as orc
    vals = orc.synth_elements(p, n, 20260923 + os.getpid() % 1000)
    _REF.update(p=p, m=m, t=t, k=k, n=n, s=np.array(vals, dtype=object), first=vals[0])
    mods = _reference_modules()
    if mods is not None:
        F = mods[0].GF(p)
        _REF.update(F=F, a=F.array(_REF['s']))


def _ref_step(_):
    """One worker's share of a step: draw coefficients as the reference does, split, recombine t+1 shares."""
    import secrets
    r = _REF
    if 'F' in r:
        thresha = _reference_modules()[1]
        sh = thresha.np_random_split(r['F'], r['a'], r['t'], r['m'])
        out = thresha.np_recombine(r['F'], [(i + 1, sh[i]) for i in range(r['k'])])
        assert out.value[0] == r['first']
        return r['n']
    from oracle import shamir_oracle as orc
    C = orc.np_draw_coefficients(r['p'], r['t'], r['n'], secrets.randbelow)
    sh = orc.np_split(r['p'], r['s'], C, r['m'])
    out = orc.np_recombine(r['p'], tuple(range(1, r['k'] + 1)), sh[:r['k']])
    assert out[0] == r['first']
    return r['n']


def workload_config(w, n, world):
    return {'workload': w['name'], 'p_bits': w['p'].bit_length(), 'm': w['m'], 't': w['t'], 'recombine_k': w['k'],
            'n_per_gpu': n}


def run_reference_arm(a, w):
    """CPU arm: the reference's own thresha.np_random_split + np_recombine (NumPy object arrays, per-element
    secrets.randbelow) on all host cores, one independent process per core -- the UNMODIFIED reference when it is
    importable on this box (baseline/_ref or $MPYC_REFERENCE: kind 'reference'), else the oracle port (kind 'port').
    Each step is a bounded sample of the workload: 20 000 pairs per process."""
    import multiprocessing as mp
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    cores = len(os.sched_getaffinity(0)) or os.cpu_count() or 1
    n = 20000
    kind = 'reference' if _reference_modules() is not None else 'port'
    done = []
    with mp.get_context('fork').Pool(cores, initializer=_ref_init, initargs=(w['p'], w['m'], w['t'], w['k'], n)) as pool:
        pool.map(_ref_step, range(cores))          # make sure every worker is up before timing
        for step in range(a.warmup + a.steps):
            t0 = time.perf_counter()
            res = pool.map(_ref_step, range(cores), chunksize=1)
            dt = time.perf_counter() - t0
            if step >= a.warmup:
                done.append((sum(res), dt))
    pairs = sum(x for x, _ in done)
    dt = sum(y for _, y in done)
    val = pairs / dt
    what = 'mpyc.thresha.np_random_split+np_recombine (unmodified reference)' if kind == 'reference' else \
        'oracle port of thresha.np_random_split+np_recombine incl. secrets.randbelow'
    sample = f'{cores} independent processes x {n} pairs per step ({what})'
    cfg = workload_config(w, a.n or w['n'], a.gpus)     # the same dict as the product arm prints
    line = {'metric': METRIC, 'impl': 'reference', 'value': val, 'unit': 'pairs/s', 'n_gpus': a.gpus, 'steps': a.steps,
            'warmup': a.warmup, 'ms_per_step': 1e3 * dt / max(a.steps, 1), 'higher_is_better': True, 'scaling': 'weak',
            'vs_baseline': None, 'dtype': 'python-int (exact)', 'data': 'synthetic', 'config': cfg,
            'cpu_baseline': {'value': val, 'unit': 'pairs/s', 'cores': cores, 'kind': kind, 'sample': sample},
            'sample_per_step': f'{n} pairs x {cores} processes',
            'e2e': {'value': val, 'unit': 'pairs/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
            'gpu_launches': 0}
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------------------------------

def dropin_rate(w, device, n=200_000):
    """The rate an unmodified MPyC caller sees: mpyc_b200.thresha.np_random_split + np_recombine on NumPy
    object arrays of Python ints (conversion to limbs, CSPRNG draw, PCIe and kernels all inside)."""
    import random
    import numpy as np
    from mpyc_b200 import thresha
    p, m, t, k = w['p'], w['m'], w['t'], w['k']

    class Arr:
        def __init__(self, value, check=True):
            self.value = value

    class Field:
        modulus = order = characteristic = p
        ext_deg = 1
        array = Arr
    thresha.device = device
    rnd = random.Random(20260923)
    s = np.array([rnd.randrange(p) for _ in range(n)], dtype=object)
    thresha.np_random_split(Field, s[:1000], t, m)                     # warm-up (tables, workspace)
    t0 = time.perf_counter()
    sh = thresha.np_random_split(Field, s, t, m)
    out = thresha.np_recombine(Field, [(i + 1, sh[i]) for i in range(k)])
    dt = time.perf_counter() - t0
    assert out.value.tolist() == s.tolist()
    # limb wire (mpyc_b200.wire): rows stay limb buffers; as in runtime.py:655-665 every row is pickled for its
    # peer and the k received rows are unpickled before np_recombine -- pickling is INSIDE this timed region
    import pickle
    thresha.limb_wire = True
    try:
        t0 = time.perf_counter()
        sh = thresha.np_random_split(Field, s, t, m)
        sent = [pickle.dumps(row) for row in sh]
        out = thresha.np_recombine(Field, [(i + 1, pickle.loads(sent[i])) for i in range(k)])
        dt_lw = time.perf_counter() - t0
    finally:
        thresha.limb_wire = False
    assert out.value.tolist() == s.tolist()
    return {'value': n / dt, 'unit': 'pairs/s', 'n': n,
            'path': 'mpyc_b200.thresha.np_random_split + np_recombine on dtype=object arrays (what runtime.py calls)',
            'limb_wire': {'value': n / dt_lw, 'unit': 'pairs/s',
                          'path': 'same calls with install(limb_wire=True): ShareRow rows, pickle.dumps of all m rows and '
                                  'pickle.loads of the k recombined ones inside the timed region',
                          'wire_bytes_per_row': len(sent[0])}}


def measure_prss(w, n, steps, warmup, local, rank, peak, with_e2e=True, dump_dir=None, dump_suffix=''):
    """K4 on PRF bytes resident in HBM (CUDA events), and -- with_e2e -- the host pipeline mpyc_b200_prss_host and the
    drop-in call at np_cnnmnist's largest per-call size.  dump_dir: write the shares of the last timed step there."""
    import itertools
    import numpy as np
    import torch
    import mpyc_b200
    from mpyc_b200 import _cabi, thresha
    from mpyc_b200._cabi import lib, check
    p, m, t = w['p'], w['m'], w['t']
    ctx = mpyc_b200.context_for(p)
    L, eb = ctx.nlimbs, ctx.elem_bytes
    party = 1
    subsets = [S for S in itertools.combinations(range(m), m - t) if party in S]
    nsub, d = len(subsets), 1
    prf = {S: thresha.PRF(bytes([(31 * a_ + 7) % 256 for a_ in S] + [0] * (16 - len(S))), p) for S in subsets}
    chunk = next(iter(prf.values())).byte_length
    stride = (n * d * chunk + 15) // 16 * 16
    # device-resident PRF bytes: random bytes stand in for the XOF output (the kernel's work does not depend on them)
    g = torch.Generator(device='cuda')
    g.manual_seed(20260923 + rank)
    d_bytes = torch.randint(0, 256, (nsub, stride), dtype=torch.uint8, device='cuda', generator=g)
    d_out = torch.empty((n, L), dtype=torch.int64, device='cuda')
    coef = []
    for S in subsets:
        coef.extend(_cabi.int_to_limbs(int(thresha._f_S_i(_PrssField(p), m, party, S)), L))
    wl = _cabi.int_to_limbs(1, L)
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)

    def step():
        check(lib.mpyc_b200_prss_combine(ctx.handle, ctypes.c_void_p(d_bytes.data_ptr()), stride, nsub, d, chunk, 0,
                                         _cabi.u64_array(coef), _cabi.u64_array(wl), ctypes.c_void_p(d_out.data_ptr()), n, st))
    for _ in range(warmup):
        step()
    torch.cuda.synchronize()
    launches0 = mpyc_b200.launch_count()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(steps + 1)]
    t_start = time.perf_counter()
    ev[0].record()
    for i in range(steps):
        step()
        ev[i + 1].record()
    torch.cuda.synchronize()
    t_end = time.perf_counter()
    launches = mpyc_b200.launch_count() - launches0
    ms = ev[0].elapsed_time(ev[-1]) / steps
    if dump_dir:
        dump_outputs(dump_dir, {'prss_shares': d_out.unsqueeze(0)}, n, dump_suffix)
    alg = n * (nsub * d * chunk + eb)
    ach = alg / (ms * 1e-3) / 1e9
    out = {'kernel': 'k_prss_tiles', 'n': n, 'subsets': nsub, 'chunk_bytes': chunk, 'ms': ms, 'algorithmic_bytes': alg,
           'achieved': ach, 'frac': ach / peak, 'value': n / (ms * 1e-3), 'unit': 'shares/s', 'gpu_launches': int(launches),
           'window': (t_start, t_end), 'prf': prf, 'ctx': ctx, 'coef': coef, 'wl': wl, 'nsub': nsub, 'chunk': chunk, 'party': party}
    del d_bytes, d_out
    if with_e2e:
        ne = 213_248      # the largest per-call size of np_cnnmnist
        F = _PrssField(p)
        thresha.device = local
        thresha.np_pseudorandom_share(F, m, party, prf, b'warm', 4096)
        reps, t0 = 3, time.perf_counter()
        for r in range(reps):
            thresha.np_pseudorandom_share(F, m, party, prf, b'uci%d' % r, ne)
        dt = (time.perf_counter() - t0) / reps
        out_limbs = np.empty((ne, L), dtype=np.uint64)
        keys = b''.join(f.key for f in prf.values())
        t0 = time.perf_counter()
        for r in range(reps):
            check(lib.mpyc_b200_prss_host(ctx.handle, keys, 16, b'uci%d' % r, 4, nsub, d, chunk, 0, _cabi.u64_array(coef),
                                          _cabi.u64_array(wl), ctypes.c_void_p(out_limbs.ctypes.data), ne, local, 0))
        dt_abi = (time.perf_counter() - t0) / reps
        out['e2e'] = {'value': ne / dt_abi, 'unit': 'shares/s', 'h2d_bytes_per_step': ne * nsub * d * chunk, 'd2h_bytes_per_step': ne * eb,
                      'n_per_step': ne, 'ms_per_step': dt_abi * 1e3,
                      'path': 'mpyc_b200_prss_host: SHAKE128 sponges on host threads -> pinned chunks -> H2D -> K4 -> D2H (host buffers in and out)',
                      'xof_bytes_per_step': ne * nsub * d * chunk, 'xof_MBps': ne * nsub * d * chunk / dt_abi / 1e6,
                      'host_threads': min(nsub, len(os.sched_getaffinity(0))),
                      'dropin': {'value': ne / dt, 'unit': 'shares/s', 'path': 'mpyc_b200.thresha.np_pseudorandom_share (field.array of Python ints out)'}}
    return out


def run_prss_arm(a, w):
    """PRSS (thresha.np_pseudorandom_share, mpyc/thresha.py:163-173) at the np_cnnmnist shape.  value: elements/s of the
    combine kernel K4 on PRF bytes resident in HBM; e2e: the host pipeline (SHAKE128 sponges on host threads,
    pinned chunks, H2D, K4, D2H) at the largest per-call size of the demo; cpu_baseline: the oracle port."""
    import torch
    from mpyc_b200 import thresha
    if not torch.cuda.is_available():
        raise SystemExit('bench.py: no CUDA device (there is no CPU fallback for the product arm)')
    local = int(os.environ.get('LOCAL_RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    torch.cuda.set_device(local)
    dist = _dist_init(local) if world > 1 else None
    p, m, t, n = w['p'], w['m'], w['t'], a.n or w['n']
    peak, peak_src = peaks()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    r = measure_prss(w, n, a.steps, a.warmup, local, rank, peak, dump_dir=a.dump_outputs, dump_suffix=rank_suffix(world, rank))
    ms = r['ms']
    if world > 1:
        tt = torch.tensor([ms], device='cuda')
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        ms = float(tt.item())
    clocks = sampler.report(*r['window']) if rank == 0 else None
    sampler.stop()
    roofline = {'bound': 'hbm', 'kernel': 'k_prss_tiles', 'achieved': r['algorithmic_bytes'] / (ms * 1e-3) / 1e9, 'peak': peak,
                'peak_source': peak_src, 'unit': 'GB/s', 'frac': r['algorithmic_bytes'] / (ms * 1e-3) / 1e9 / peak,
                'traffic': ncu_traffic('prss', 'prss')[0], 'ms': ms, 'algorithmic_bytes': r['algorithmic_bytes'],
                'note': 'subset constants are cached in the field handle: a call costs no allocation, upload or synchronisation'}
    e2e = r['e2e']
    e2e['value'] *= world
    cpu = None
    prf, party = r['prf'], r['party']
    if rank == 0 and not a.no_cpu:
        from oracle import shamir_oracle as orc
        Fo = orc.field_of(p)
        F = _PrssField(p)
        nc = 10_000
        t0 = time.perf_counter()
        got = orc.prss_share(Fo, m, party, {S: orc.prf_values(f.key, p, b'uci0', nc) for S, f in prf.items()}, nc)
        dtc = time.perf_counter() - t0
        chk = thresha.np_pseudorandom_share(F, m, party, prf, b'uci0', nc)
        assert got == chk.value.tolist(), 'PRSS differs from the oracle'
        cpu = {'value': nc / dtc, 'unit': 'shares/s', 'cores': 1, 'kind': 'port',
               'sample': f'oracle port of np_pseudorandom_share (hashlib SHAKE128 + Python ints) on {nc} elements, 1 process'}
    if rank == 0:
        line = {'metric': 'PRSS pseudorandom shares/sec', 'value': world * n / (ms * 1e-3), 'unit': 'shares/s', 'n_gpus': world,
                'steps': a.steps, 'warmup': a.warmup, 'ms_per_step': ms, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
                'dtype': f'u64x{r["ctx"].nlimbs} limbs (exact integer arithmetic mod p)', 'data': 'synthetic',
                'config': {'workload': w['name'], 'p_bits': p.bit_length(), 'm': m, 't': t, 'subsets': r['nsub'], 'chunk_bytes': r['chunk'], 'n_per_gpu': n,
                           'l2_policy': 'PRF bytes (2 GB) far larger than the 126 MB L2; no flush needed'},
                'roofline': roofline, 'cpu_baseline': cpu, 'e2e': e2e, 'gpu_launches': r['gpu_launches'], 'clocks': clocks}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


class _PrssArr:
    def __init__(self, value, check=True):
        self.value = value


def _PrssField(p):
    class Field:
        modulus = order = characteristic = p
        ext_deg = 1
        array = _PrssArr
    return Field


def _dist_init(local):
    import torch
    import torch.distributed as dist
    os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
    dist.init_process_group('nccl', device_id=torch.device('cuda', local))
    return dist


DUMP_SAMPLE = 1 << 16       # elements per output written by --dump-outputs (at most ~34 MB in all, for c5)


def dump_outputs(directory, arrays, n, suffix=''):
    """--dump-outputs: write device outputs as DIR/<name><suffix>.npy.  `arrays` maps names to tensors whose axis 1 is
    the element axis: int64 limbs (rows, n, L) or GF(2^8) bytes (rows, n).  Limbs become float64 words, exactly: each
    64-bit limb is split into two 32-bit words, least significant first, so an element is 2L words.  GF(2^8) bytes
    become float32.  Outputs longer than DUMP_SAMPLE elements are sampled at seeded element indices, the same in every
    run and every array, and element_index<suffix>.npy records them."""
    import numpy as np
    import torch
    os.makedirs(directory, exist_ok=True)
    if n > DUMP_SAMPLE:
        idx = np.unique(np.random.default_rng(20260923).integers(0, n, size=DUMP_SAMPLE))
    else:
        idx = np.arange(n)
    np.save(os.path.join(directory, f'element_index{suffix}.npy'), idx.astype(np.float64))
    for name, t in arrays.items():
        x = t.index_select(1, torch.from_numpy(idx).to(t.device)).cpu().numpy()
        x = x.astype(np.float32) if x.dtype == np.uint8 else x.view(np.uint32).astype(np.float64)
        np.save(os.path.join(directory, f'{name}{suffix}.npy'), x[0] if x.shape[0] == 1 else x)


def measure_device(w, n, steps, warmup, seed_rank=0, sustain_s=0.0, keep=False, dump_dir=None, dump_suffix=''):
    """K steps of the hot path on device-resident inputs, timed with CUDA events on the launching stream.
    Returns a dict with per-kernel milliseconds, launches and (keep=True) the buffers for later checks.
    dump_dir: write the outputs of the last timed step there (dump_outputs)."""
    import torch
    import mpyc_b200
    from mpyc_b200 import _cabi, device as dev
    from mpyc_b200._cabi import lib, check
    p, m, t, k = w['p'], w['m'], w['t'], w['k']
    ctx = mpyc_b200.context_for(p, binary=bool(w.get('binary')))
    is_mul = m == 0
    S = dev.DeviceArray.random(ctx, n, seed=20260923 + seed_rank, stream_id=1)
    if is_mul:
        B = dev.DeviceArray.random(ctx, n, seed=77 + seed_rank, stream_id=2)
        OUT = dev.DeviceArray.empty(ctx, n)
    else:
        C = dev.DeviceMatrix.empty(ctx, t, n)
        for j in range(t):
            C.t[j].copy_(dev.DeviceArray.random(ctx, n, seed=100 + j + 10 * seed_rank, stream_id=3).t)
        SH = dev.DeviceMatrix.empty(ctx, m, n)
        REC = dev.DeviceMatrix.empty(ctx, 1, n)
        xs = list(range(1, k + 1))
        rows = [SH.row(x - 1) for x in xs]
    torch.cuda.synchronize()

    def split():
        if is_mul:
            check(lib.mpyc_b200_ff_binop(ctx.handle, _cabi.OP_MUL, S.ptr, B.ptr, OUT.ptr, n, dev._stream_ptr()))
        else:
            dev.shamir_split(ctx, S, C, t, m, out=SH)

    def recombine():
        if not is_mul:
            dev.shamir_recombine(ctx, xs, rows, 0, out=REC)

    for _ in range(warmup):
        split()
        recombine()
    torch.cuda.synchronize()
    if not is_mul:   # correctness guard inside the bench: the recombined secrets are the inputs
        assert REC.row(0).count_mismatch(S) == 0, 'recombined secrets differ from inputs'

    def timed(count):
        launches0 = mpyc_b200.launch_count()
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(2 * count + 1)]
        t_start = time.perf_counter()
        ev[0].record()
        for i in range(count):
            split()
            ev[2 * i + 1].record()
            recombine()
            ev[2 * i + 2].record()
        torch.cuda.synchronize()
        t_end = time.perf_counter()
        return {'total_ms': ev[0].elapsed_time(ev[-1]),
                'split_ms': sum(ev[2 * i].elapsed_time(ev[2 * i + 1]) for i in range(count)) / count,
                'rec_ms': 0.0 if is_mul else sum(ev[2 * i + 1].elapsed_time(ev[2 * i + 2]) for i in range(count)) / count,
                'launches': mpyc_b200.launch_count() - launches0, 'window': (t_start, t_end), 'count': count}
    common = dict(ctx=ctx, is_mul=is_mul, eb=ctx.elem_bytes, L=max(ctx.nlimbs, 1))
    res = timed(steps)
    res.update(common)
    if dump_dir:
        outputs = {'product': OUT.t.unsqueeze(0)} if is_mul else {'shares': SH.t, 'recombined': REC.t}
        dump_outputs(dump_dir, outputs, n, dump_suffix)
    if sustain_s > 0:
        per = max(res['total_ms'] / steps, 1e-3)
        res['sustained'] = timed(max(steps, int(sustain_s * 1e3 / per) + 1))
        res['sustained'].update(common)
    if keep:
        res['buffers'] = dict(S=S, B=B, OUT=OUT) if is_mul else dict(S=S, C=C, SH=SH, REC=REC, rows=rows, xs=xs)
    return res


def kernel_rooflines(w, n, res, peak):
    """Algorithmic bytes (SURVEY 8d) / measured duration for the kernels of one measure_device() result."""
    eb, m, t, k = res['eb'], w['m'], w['t'], w['k']
    if res['is_mul']:
        b = 3 * eb * n
        return {'k_binop<mul>': {'achieved': b / (res['split_ms'] * 1e-3) / 1e9, 'frac': b / (res['split_ms'] * 1e-3) / 1e9 / peak,
                                 'ms': res['split_ms'], 'algorithmic_bytes': b}}
    sb, rb = (1 + t + m) * eb * n, (k + 1) * eb * n
    step_ms = res['total_ms'] / res['count']
    return {'k_split': {'achieved': sb / (res['split_ms'] * 1e-3) / 1e9, 'frac': sb / (res['split_ms'] * 1e-3) / 1e9 / peak,
                        'ms': res['split_ms'], 'algorithmic_bytes': sb},
            'k_recombine': {'achieved': rb / (res['rec_ms'] * 1e-3) / 1e9, 'frac': rb / (res['rec_ms'] * 1e-3) / 1e9 / peak,
                            'ms': res['rec_ms'], 'algorithmic_bytes': rb},
            'step_total': {'achieved': (sb + rb) / (step_ms * 1e-3) / 1e9, 'frac': (sb + rb) / (step_ms * 1e-3) / 1e9 / peak,
                           'bytes_per_pair': (sb + rb) / n, 'ms': step_ms}}


def run_extras(peak, local):
    """Short full-size passes of the other configurations in the same process (5 timed steps each after 3 warm-up
    steps): what round 1 could only show in builder-run lines."""
    import gc
    import torch
    out = {}
    for name in ('ns64', 'c5', 'c3g', 'c4', 'modmul', 'modmul_generic'):
        w = WORKLOADS[name]
        try:
            res = measure_device(w, w['n'], steps=5, warmup=3)
            rl = kernel_rooflines(w, w['n'], res, peak)
            unit = 'elem/s' if res['is_mul'] else 'pairs/s'
            out[name] = {'workload': w['name'], 'value': w['n'] / (res['total_ms'] / res['count'] * 1e-3), 'unit': unit,
                         'kernels': {k: {kk: (round(vv, 4) if isinstance(vv, float) else vv) for kk, vv in v.items()} for k, v in rl.items()},
                         'gpu_launches': int(res['launches'])}
        except Exception as exc:   # noqa: BLE001
            out[name] = {'error': repr(exc)[:300]}
        gc.collect()
        torch.cuda.empty_cache()
    try:
        r = measure_prss(WORKLOADS['prss'], WORKLOADS['prss']['n'], steps=5, warmup=3, local=local, rank=0, peak=peak)
        out['prss'] = {k: v for k, v in r.items() if k not in ('window', 'prf', 'ctx', 'coef', 'wl', 'party')}
    except Exception as exc:   # noqa: BLE001
        out['prss'] = {'error': repr(exc)[:300]}
    try:
        out['local'] = measure_local(peak)
    except Exception as exc:   # noqa: BLE001
        out['local'] = {'error': repr(exc)[:300]}
    return out


def measure_local(peak, steps=5, warmup=3):
    """The protocol-local kernels (csrc/local.cuh, SURVEY 8f N3/N4) at sizes beyond L2, CUDA events on the launching
    stream: algorithmic bytes / duration against the copy peak.  np_sgn's shape: l = 37 bit positions per element."""
    import torch
    import mpyc_b200
    from mpyc_b200 import device as dev
    from mpyc_b200.device import DeviceArray
    out = {}

    def timed(fn):
        for _ in range(warmup):
            fn()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(steps):
            fn()
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / steps

    def entry(bytes_, ms, **kw):
        g = bytes_ / ms / 1e6
        return {'ms': round(ms, 4), 'algorithmic_bytes': bytes_, 'achieved': round(g, 1), 'frac': round(g / peak, 4), **kw}

    for label, p in (('p128', 2**128 - 173), ('p64', 2**64 - 189), ('p256', 2**256 - 189)):
        ctx = mpyc_b200.context_for(p)
        E = 8 * ctx.nlimbs
        n = (1 << 30) // E                                   # 1 GiB per operand
        A = DeviceArray.random(ctx, n, seed=5, stream_id=1)
        C = DeviceArray.random(ctx, n, seed=5, stream_id=3)
        res = {'fma_square_add': entry(3 * E * n, timed(lambda: dev.fma(A, None, C)), n=n),
               'axpb': entry(2 * E * n, timed(lambda: dev.axpb(A, (p + 1) >> 1, 12345)), n=n),
               'low_bits': entry(2 * E * n, timed(lambda: dev.low_bits(A, 37)), n=n)}
        for f in (6, 37):
            rows = n // f
            bits = DeviceArray(ctx, A.t[:rows * f])
            res[f'bits_compose_f{f}'] = entry((f + 1) * E * rows, timed(lambda: dev.bits_compose(bits, rows, f, descending=(f == 37))),
                                              n=rows, f=f)
        rows = n // 37
        c = DeviceArray(ctx, C.t[:rows])
        res['bits_decompose_l37'] = entry(38 * E * rows, timed(lambda: dev.bits_decompose(c, 37, descending=True)), n=rows, l=37)
        out[label] = res
        del A, C, bits, c
        torch.cuda.empty_cache()
    return out


def multi_selftest(world, rank, local):
    """N > 1 pre-flight (the checks of tests/test_gpu_multi.py, which a 1-GPU test box skips): the sharded path equals
    the single-GPU result, the NCCL gather reassembles the element axis (all-gather and gather-to-one), and one
    co-located secure multiplication is reshared GPU to GPU in both forms (grouped ncclSend/ncclRecv; K2 storing into
    the peer GPU) and opens to the product."""
    import torch
    import torch.distributed as dist
    import mpyc_b200
    from mpyc_b200 import device as dev, sharding, exchange
    from mpyc_b200.device import DeviceArray, DeviceMatrix
    p, m, t, n = 2**128 - 173, 5, 2, 1_000_003
    ctx = mpyc_b200.context_for(p)
    S = DeviceArray.random(ctx, n, seed=11, stream_id=1)
    C = DeviceMatrix.empty(ctx, t, n)
    for j in range(t):
        C.t[j].copy_(DeviceArray.random(ctx, n, seed=20 + j, stream_id=2).t)
    lo, hi = sharding.shard_bounds(n, world, rank)
    S_loc = DeviceArray(ctx, S.t[lo:hi].contiguous())
    C_loc = DeviceMatrix.empty(ctx, t, hi - lo)
    for j in range(t):
        C_loc.t[j].copy_(C.t[j, lo:hi])
    sh_loc = dev.shamir_split(ctx, S_loc, C_loc, t, m)
    rec_loc = dev.shamir_recombine(ctx, [1, 2, 3], [sh_loc.row(i) for i in range(3)])
    assert rec_loc.count_mismatch(S_loc) == 0, 'sharded recombination differs'
    assert torch.equal(sharding.gather(rec_loc.t.contiguous(), n), S.t), 'all-gather differs'
    row3 = sharding.gather(sh_loc.t[3].contiguous(), n, dst=0)
    if rank == 0:
        assert torch.equal(row3, dev.shamir_split(ctx, S, C, t, m).t[3]), 'gather-to-one differs from the single-GPU shares'
    forms = ['nccl']
    if os.environ.get('MPYC_B200_BENCH_PEER', '1') == '1':
        forms.append('peer')
    nn = 200_003
    A = DeviceArray.random(ctx, nn, seed=3, stream_id=1)
    Bv = DeviceArray.random(ctx, nn, seed=4, stream_id=1)
    CA, CB = DeviceMatrix.empty(ctx, t, nn), DeviceMatrix.empty(ctx, t, nn)
    for j in range(t):
        CA.t[j].copy_(DeviceArray.random(ctx, nn, seed=30 + j, stream_id=2).t)
        CB.t[j].copy_(DeviceArray.random(ctx, nn, seed=40 + j, stream_id=2).t)
    sa, sb = dev.shamir_split(ctx, A, CA, t, m), dev.shamir_split(ctx, Bv, CB, t, m)
    mine = exchange.local_parties(m, world, rank)
    prod = {j: (sa.row(j) * sb.row(j)).t for j in mine}
    want = A * Bv
    for form in forms:
        if form == 'peer':
            peer = exchange.PeerReshare(ctx, m, t, nn, first_dealer=1)
            new = peer.reshare(prod)
            torch.cuda.synchronize()
            dist.barrier()
        else:
            new = exchange.reshare(exchange.DeviceEngine(ctx), prod, t, m, first_dealer=1)
        full = [None] * m
        for i in range(m):
            buf = new[i].contiguous() if i in new else torch.empty((nn, ctx.nlimbs), dtype=torch.int64, device='cuda')
            dist.broadcast(buf, src=exchange.owner(i, world))
            full[i] = DeviceArray(ctx, buf)
        for xs in (list(range(1, t + 2)), list(range(m - t, m + 1))):
            assert dev.shamir_recombine(ctx, xs, [full[x - 1] for x in xs]).count_mismatch(want) == 0, f'reshare ({form}) differs'
        if form == 'peer':
            dist.barrier()
            peer.close()
    return 'ok: sharded==single, all-gather, gather-to-one, reshare ' + '+'.join(forms)


def time_gather(REC_row, n, world):
    """The single collective of the path (SURVEY 8e): all-gather of the sharded, recombined vector."""
    import torch
    from mpyc_b200 import sharding
    loc = REC_row.t.contiguous()
    sharding.gather(loc, n * world)                      # warm-up (NCCL channel setup)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = 3
    e0.record()
    for _ in range(reps):
        full = sharding.gather(loc, n * world)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps
    out_bytes = full.numel() * full.element_size()
    del full
    return {'collective': 'ncclAllGather of the recombined vector (sharding.gather)', 'ms': ms, 'bytes_out_per_rank': out_bytes,
            'algbw_GBps': out_bytes / (ms * 1e-3) / 1e9, 'busbw_GBps': out_bytes * (world - 1) / world / (ms * 1e-3) / 1e9}


def pcie_probe(nbytes=1 << 29, reps=3):
    """What the host link gives this rank: pinned cudaMemcpyAsync H2D alone, D2H alone, and both directions at once
    (GB/s per direction).  The e2e step moves h2d_bytes + d2h_bytes per step through exactly this link, so the
    bidirectional figure is its ceiling."""
    import torch
    h_in = torch.empty(nbytes, dtype=torch.uint8).pin_memory()
    h_out = torch.empty(nbytes, dtype=torch.uint8).pin_memory()
    d_a = torch.empty(nbytes, dtype=torch.uint8, device='cuda')
    d_b = torch.empty(nbytes, dtype=torch.uint8, device='cuda')
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()

    def run(up, down):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(reps):
            if up:
                with torch.cuda.stream(s1):
                    d_a.copy_(h_in, non_blocking=True)
            if down:
                with torch.cuda.stream(s2):
                    h_out.copy_(d_b, non_blocking=True)
        torch.cuda.synchronize()
        return reps * nbytes / (time.perf_counter() - t0) / 1e9
    run(True, True)
    return {'h2d_alone_GBps': run(True, False), 'd2h_alone_GBps': run(False, True), 'bidirectional_GBps_per_direction': run(True, True),
            'bytes_per_copy': nbytes}


def rank_suffix(world, rank):
    """With N > 1 every rank dumps its own shard of the element axis."""
    return f'_rank{rank}' if world > 1 else ''


def run_gpu_arm(a, w):
    local = int(os.environ.get('LOCAL_RANK', '0'))
    numa = bind_to_gpu_numa(local)       # before CUDA initialisation and any pinned allocation
    if w.get('prss'):
        return run_prss_arm(a, w)
    import torch
    import mpyc_b200
    from mpyc_b200 import _cabi
    from mpyc_b200._cabi import lib, check

    rank = int(os.environ.get('RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    if not torch.cuda.is_available():
        raise SystemExit('bench.py: no CUDA device (there is no CPU fallback for the product arm)')
    torch.cuda.set_device(local)
    dist = _dist_init(local) if world > 1 else None
    p, m, t, k, n = w['p'], w['m'], w['t'], w['k'], a.n or w['n']
    if w.get('binary'):
        a.no_e2e = True   # host-buffer pipeline is exercised by the prime-field workloads
    peak, peak_src = peaks()

    selftest = None
    if world > 1 and not a.no_selftest:
        try:
            selftest = multi_selftest(world, rank, local)
        except Exception as exc:   # noqa: BLE001
            selftest = 'FAILED: ' + repr(exc)[:300]
        torch.cuda.empty_cache()

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()              # before the warm-up: certainly polling when the timed region starts
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    res = measure_device(w, n, a.steps, a.warmup, seed_rank=rank, sustain_s=a.sustain, keep=True,
                         dump_dir=a.dump_outputs, dump_suffix=rank_suffix(world, rank))
    if world > 1:
        dist.barrier()
    is_mul, eb, L, ctx = res['is_mul'], res['eb'], res['L'], res['ctx']
    buf = res['buffers']
    launches = int(res['launches'])
    total_ms = res['total_ms']
    if world > 1:
        tl = torch.tensor([launches], device='cuda', dtype=torch.int64)
        dist.all_reduce(tl)
        launches = int(tl.item())
        tt = torch.tensor([total_ms], device='cuda', dtype=torch.float64)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        total_ms = float(tt.item())
    clocks = sampler.report(*res['window']) if rank == 0 else None
    ms_per_step = total_ms / a.steps
    value = world * n / (ms_per_step * 1e-3)
    sustained = None
    if 'sustained' in res:
        sres = res['sustained']
        sms = sres['total_ms']
        if world > 1:
            tt = torch.tensor([sms], device='cuda', dtype=torch.float64)
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            sms = float(tt.item())
        if rank == 0:
            rl_s = kernel_rooflines(w, n, sres, peak)
            dom = 'k_binop<mul>' if is_mul else 'k_split'
            sustained = {'seconds': sms / 1e3, 'steps': sres['count'], 'ms_per_step': sms / sres['count'],
                         'value': world * n / (sms / sres['count'] * 1e-3), 'unit': 'pairs/s' if not is_mul else 'elem/s',
                         'dominant_kernel_frac': rl_s[dom]['frac'], 'dominant_kernel_ms': rl_s[dom]['ms'],
                         'clocks': sampler.report(*sres['window'])}

    # ---- roofline of the dominant kernel (share generation), algorithmic bytes / measured duration ----
    rl = kernel_rooflines(w, n, res, peak)
    dom_name = 'k_binop<mul>' if is_mul else 'k_split'
    sec = {} if is_mul else {'recombine': dict(kernel='k_recombine', unit='GB/s', **rl['k_recombine']),
                             'step_total': dict(unit='GB/s', **rl['step_total'])}
    traffic, traffic_src = ncu_traffic(a.workload, 'binop' if is_mul else 'split') if n == w['n'] else (None, None)
    roofline = {'bound': 'hbm', 'kernel': dom_name, 'achieved': rl[dom_name]['achieved'], 'peak': peak, 'peak_source': peak_src,
                'unit': 'GB/s', 'frac': rl[dom_name]['frac'], 'traffic': traffic, 'traffic_source': traffic_src,
                'ms': rl[dom_name]['ms'], 'algorithmic_bytes': rl[dom_name]['algorithmic_bytes'], **sec}

    gather = None
    if world > 1 and not is_mul and not a.no_selftest:
        try:
            gather = time_gather(buf['REC'].row(0), n, world)
        except Exception as exc:   # noqa: BLE001
            gather = {'error': repr(exc)[:300]}

    # ---- e2e: same path through the C ABI's host-buffer entry points, pinned host memory ----------------
    e2e = None
    if not a.no_e2e:
        ne = a.e2e_n
        S = buf['S']
        hs = torch.empty((ne, L), dtype=torch.int64).pin_memory()
        hs.copy_(S.t[:ne].cpu())
        if is_mul:
            hb = torch.empty((ne, L), dtype=torch.int64).pin_memory()
            hb.copy_(buf['B'].t[:ne].cpu())
            ho = torch.empty((ne, L), dtype=torch.int64).pin_memory()

            def e2e_run(count):
                for _ in range(count):
                    check(lib.mpyc_b200_ff_binop_host(ctx.handle, _cabi.OP_MUL, hs.data_ptr(), hb.data_ptr(), ho.data_ptr(), ne, local))
            h2d, d2h = 2 * eb * ne, eb * ne
            path = 'mpyc_b200_ff_binop_host (pinned host buffers, copies inside)'
            serial_ms = explicit_ms = explicit_h2d = None
        else:
            xs = buf['xs']
            hc = torch.empty((t, ne, L), dtype=torch.int64).pin_memory()
            hc.copy_(buf['C'].t[:, :ne].cpu())
            hsh = [torch.empty((m, ne, L), dtype=torch.int64).pin_memory() for _ in range(2)]   # double-buffered share rows
            hout = torch.empty((1, ne, L), dtype=torch.int64).pin_memory()
            rowp = [_cabi.ptr_array([h[x - 1].data_ptr() for x in xs]) for h in hsh]
            xs_c, xr_c = _cabi.i64_array(xs), _cabi.i64_array([0])

            import ctypes
            import os as _os
            key32 = (ctypes.c_uint8 * 32).from_buffer_copy(_os.urandom(32))
            nonce = [0]

            def do_split_explicit(b):
                check(lib.mpyc_b200_shamir_split_host(ctx.handle, hs.data_ptr(), hc.data_ptr(), ne, hsh[b].data_ptr(), ne, ne, t, m, local))

            def do_split(b):
                # what thresha.np_random_split(field, s, t, m) is: secrets in, shares out -- the coefficients are the callee's
                # own randomness (mpyc/thresha.py:58-60 draws them with secrets.randbelow; here an in-kernel ChaCha20 stream
                # keyed with OS randomness), so only the secrets cross PCIe on the way up
                nonce[0] += 1
                check(lib.mpyc_b200_shamir_split_generate_host(ctx.handle, hs.data_ptr(), hsh[b].data_ptr(), ne, ne, t, m, key32,
                                                               nonce[0], local))

            def do_rec(b):
                check(lib.mpyc_b200_shamir_recombine_host(ctx.handle, rowp[b], xs_c, k, xr_c, 1, hout.data_ptr(), ne, ne, local))

            def e2e_serial(count):
                for _ in range(count):
                    do_split(0)
                    do_rec(0)

            def e2e_run(count):
                # software pipeline over successive batches: while batch j's shares are recombined (H2D-heavy), batch
                # j+1 is split from a second host thread (D2H-heavy); the two entry points use separate workspaces in
                # the library.  `count` splits and `count` recombinations in total.  (Measured on the B200 box with
                # 32 MiB pipeline chunks this, the serial two-call form and the single-thread
                # mpyc_b200_shamir_reshare_step_host were within 4 % of each other -- 41.3 / 42.4 / 44.3 ms; with
                # call-sized chunks (128 MiB here) 37.6 / 42.3 ms: the step is bound by the PCIe throughput the
                # chunked bidirectional copy pattern reaches, see pcie_probe.)
                for j in range(count + 1):
                    th = None
                    if j < count:
                        th = threading.Thread(target=do_split, args=(j % 2,))
                        th.start()
                    if j >= 1:
                        do_rec((j - 1) % 2)
                    if th is not None:
                        th.join()
            h2d, d2h = eb * ne + k * eb * ne, m * eb * ne + eb * ne
            path = ('mpyc_b200_shamir_split_generate_host (secrets in, shares out: np_random_split\'s signature) + '
                    'mpyc_b200_shamir_recombine_host on pinned host buffers, copies inside; successive batches pipelined from '
                    'two host threads (split of batch j+1 overlaps recombination of batch j)')
            e2e_serial(2)
            t0 = time.perf_counter()
            e2e_serial(max(2, a.steps // 4))
            serial_ms = 1e3 * (time.perf_counter() - t0) / max(2, a.steps // 4)
            # the same step with the coefficients supplied by the caller (parity mode: t more rows go up)
            generate_split = do_split
            do_split = do_split_explicit
            e2e_run(1)
            if world > 1:
                dist.barrier()
            t0 = time.perf_counter()
            e2e_run(max(2, a.steps // 2))
            explicit_ms = 1e3 * (time.perf_counter() - t0) / max(2, a.steps // 2)
            do_split = generate_split
            explicit_h2d = (1 + t) * eb * ne + k * eb * ne
        e2e_run(max(1, min(a.warmup, 2)))
        if world > 1:
            dist.barrier()
        t0 = time.perf_counter()
        e2e_run(a.steps)
        dt = time.perf_counter() - t0
        if world > 1:   # every rank drives its own GPU over its own PCIe link; the job time is the slowest rank
            td = torch.tensor([dt], device='cuda', dtype=torch.float64)
            dist.all_reduce(td, op=dist.ReduceOp.MAX)
            dt = float(td.item())
        if not is_mul:
            assert torch.equal(hout[0], hs), 'e2e: recombined secrets differ from inputs'
        if world > 1:
            dist.barrier()
        probe = pcie_probe()                      # all ranks at once: what the shared host links give concurrently
        if world > 1:
            tp = torch.tensor([probe['bidirectional_GBps_per_direction']], device='cuda', dtype=torch.float64)
            dist.all_reduce(tp, op=dist.ReduceOp.MIN)
            probe['bidirectional_GBps_per_direction_min_over_ranks'] = float(tp.item())
        e2e = {'value': world * ne * a.steps / dt, 'unit': 'pairs/s' if not is_mul else 'elem/s', 'h2d_bytes_per_step': h2d,
               'd2h_bytes_per_step': d2h, 'n_per_step': ne, 'ms_per_step': 1e3 * dt / a.steps, 'path': path,
               'serial_two_call_ms_per_step': serial_ms,
               'explicit_coefficients_ms_per_step': explicit_ms, 'explicit_coefficients_h2d_bytes_per_step': explicit_h2d,
               'pcie_GBps_per_direction': {'h2d': h2d / (dt / a.steps) / 1e9, 'd2h': d2h / (dt / a.steps) / 1e9},
               'pcie_probe': probe,
               'note': 'all ranks concurrently, max over ranks of the host wall clock around the blocking C-ABI calls'}
        del hs

    if rank != 0:
        sampler.stop()
        if world > 1:
            dist.destroy_process_group()
        return
    kind_cpu = None if (a.no_cpu or is_mul or world > 1 or w.get('binary')) else cpu_baseline(w)
    small_call = None
    if w.get('binary'):
        from mpyc_b200 import device as dev
        # np_aes.py shape: calls on n = 16 bytes; launch latency, not bandwidth, is what counts there
        s16 = dev.DeviceArray.random(ctx, 16, seed=1, stream_id=1)
        c16 = dev.DeviceMatrix.empty(ctx, t, 16)
        c16.t[0].copy_(dev.DeviceArray.random(ctx, 16, seed=2, stream_id=2).t)
        sh16 = dev.DeviceMatrix.empty(ctx, m, 16)
        r16 = dev.DeviceMatrix.empty(ctx, 1, 16)
        rows16 = [sh16.row(i) for i in range(k)]
        for _ in range(20):
            dev.shamir_split(ctx, s16, c16, t, m, out=sh16)
            dev.shamir_recombine(ctx, list(range(1, k + 1)), rows16, 0, out=r16)
        torch.cuda.synchronize()
        reps = 2000
        t0 = time.perf_counter()
        for _ in range(reps):
            dev.shamir_split(ctx, s16, c16, t, m, out=sh16)
            dev.shamir_recombine(ctx, list(range(1, k + 1)), rows16, 0, out=r16)
        torch.cuda.synchronize()
        small_call = {'n': 16, 'us_per_split_plus_recombine': 1e6 * (time.perf_counter() - t0) / reps,
                      'note': 'device-resident, two kernel launches per pair, host-side issue rate included'}
    dropin = None
    if not (a.no_e2e or is_mul or world > 1 or w.get('binary')):
        dropin = dropin_rate(w, local)
    extra = None
    if world == 1 and a.workload == 'c3' and not a.no_extras and n == w['n']:
        import gc
        res = buf = None
        gc.collect()
        torch.cuda.empty_cache()
        extra = run_extras(peak, local)
    sampler.stop()
    cfg = workload_config(w, n, world)
    line = {'metric': METRIC if not is_mul else 'GF(p) modmul elem/sec', 'value': value,
            'unit': 'pairs/s' if not is_mul else 'elem/s', 'n_gpus': world, 'steps': a.steps, 'warmup': a.warmup,
            'ms_per_step': ms_per_step, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
            'dtype': ('u8 (GF(2^8) polynomial arithmetic)' if w.get('binary') else f'u64x{L} limbs (exact integer arithmetic mod p)'), 'data': 'synthetic',
            'config': cfg, 'parallelism': f'element axis sharded over {world} GPU(s), no data-path collective',
            'l2_policy': 'inputs (>= 1.6 GB) far larger than the 126 MB L2; no flush needed',
            'coefficients': 'resident in HBM (parity mode)',
            'roofline': roofline, 'cpu_baseline': kind_cpu, 'e2e': e2e, 'e2e_dropin': dropin, 'small_call': small_call,
            'sustained': sustained, 'extra': extra, 'multi_selftest': selftest, 'gather': gather, 'numa': numa,
            'gpu_launches': int(launches), 'clocks': clocks}
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=10)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--workload', default='c3', choices=sorted(WORKLOADS))
    ap.add_argument('--n', type=int, default=0, help='elements per GPU (default: the workload size)')
    ap.add_argument('--e2e-n', type=int, default=1 << 24)
    ap.add_argument('--no-e2e', action='store_true')
    ap.add_argument('--no-cpu', action='store_true')
    ap.add_argument('--no-extras', action='store_true', help='skip the short passes of the other configurations (N = 1)')
    ap.add_argument('--no-selftest', action='store_true', help='skip the multi-GPU pre-flight and the gather timing (N > 1)')
    ap.add_argument('--sustain', type=float, default=2.0, help='seconds of the sustained pass after the K timed steps (0 = off)')
    ap.add_argument('--config', dest='workload_alias', default=None, help='alias of --workload')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='write the outputs of the last timed step to DIR/<name>.npy (GPU arm; see dump_outputs)')
    a = ap.parse_args()
    if a.dump_outputs and a.impl != 'ours':
        ap.error('--dump-outputs applies to the GPU arm (--impl ours)')
    if a.workload_alias:
        a.workload = a.workload_alias
    a.warmup = max(a.warmup, 3) if a.impl == 'ours' else a.warmup
    w = WORKLOADS[a.workload]
    if a.impl == 'reference':
        run_reference_arm(a, w)
    else:
        run_gpu_arm(a, w)


if __name__ == '__main__':
    main()
