"""The JSON-line contract of bench.py that can be checked without a GPU: the reference arm (`--impl reference`: the
unmodified reference where it is importable -- baseline/_ref or $MPYC_REFERENCE --, else the oracle port) prints one line
with the keys the driver reads, on the same `config` as the GPU arm, with an `e2e` that moves no bytes over PCIe.
With a GPU: what the product arm's --dump-outputs writes."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_the_contract_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--steps', '1', '--warmup', '1'],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    for key in ('metric', 'value', 'unit', 'n_gpus', 'steps', 'warmup', 'ms_per_step', 'higher_is_better', 'scaling', 'vs_baseline',
                'dtype', 'data', 'config', 'cpu_baseline', 'e2e', 'impl'):
        assert key in line, key
    assert line['impl'] == 'reference' and line['unit'] == 'pairs/s' and line['higher_is_better'] is True
    assert line['value'] > 0 and line['steps'] == 1 and line['n_gpus'] == 1 and line['vs_baseline'] is None
    cfg = line['config']
    assert 'workload' in cfg and cfg['p_bits'] == 128 and cfg['m'] == 5 and cfg['t'] == 2 and cfg['recombine_k'] == 3
    cb = line['cpu_baseline']
    assert cb['kind'] in ('reference', 'port') and cb['cores'] >= 1 and cb['value'] == line['value'] and cb['sample']
    e2e = line['e2e']
    assert e2e['value'] == line['value'] and e2e['h2d_bytes_per_step'] == 0 and e2e['d2h_bytes_per_step'] == 0


def _words_to_ints(words):
    """float64 32-bit words, least significant first (bench.dump_outputs) -> Python ints."""
    return [sum(int(w) << (32 * j) for j, w in enumerate(row)) for row in words.tolist()]


@pytest.mark.gpu
def test_dump_outputs_are_the_last_steps_shares_and_independent_of_steps(tmp_path):
    """--dump-outputs on the default workload at a small n: the sampled shares and recombined secrets equal the oracle's
    split of the bench's seeded inputs, two runs with different --steps write identical arrays, and --steps sets the
    number of timed steps (the launch count scales with it)."""
    import numpy as np
    from oracle import shamir_oracle as orc
    torch = pytest.importorskip('torch')
    if not torch.cuda.is_available():
        pytest.skip('no CUDA device')
    n, lines = 100_000, {}
    for steps in (2, 3):
        out = tmp_path / f'steps{steps}'
        r = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--gpus', '1', '--steps', str(steps), '--warmup', '1',
                            '--n', str(n), '--no-e2e', '--no-cpu', '--sustain', '0', '--dump-outputs', str(out)],
                           capture_output=True, text=True, timeout=600, cwd=tmp_path)
        assert r.returncode == 0, r.stderr[-2000:]
        lines[steps] = json.loads(r.stdout.strip().splitlines()[-1])
        assert lines[steps]['steps'] == steps
    assert lines[3]['gpu_launches'] * 2 == lines[2]['gpu_launches'] * 3 > 0
    names = sorted(f.name for f in (tmp_path / 'steps2').iterdir())
    assert names == ['element_index.npy', 'recombined.npy', 'shares.npy']
    assert names == sorted(f.name for f in (tmp_path / 'steps3').iterdir())
    arrays = {}
    for name in names:
        a, b = np.load(tmp_path / 'steps2' / name), np.load(tmp_path / 'steps3' / name)
        assert a.dtype == np.float64 and np.array_equal(a, b), name
        arrays[name[:-4]] = a
    assert sum(a.nbytes for a in arrays.values()) <= 64 << 20
    idx = arrays['element_index'].astype(np.int64)
    assert 0 < len(idx) < n and (np.diff(idx) > 0).all() and idx[-1] < n
    p, m, t = 2**128 - 173, 5, 2
    s, *C = ([row[h] for h in idx] for row in [orc.synth_elements(p, n, 20260923, stream=1)] +
             [orc.synth_elements(p, n, 100 + j, stream=3) for j in range(t)])
    assert arrays['shares'].shape == (m, len(idx), 4) and arrays['recombined'].shape == (len(idx), 4)
    assert [_words_to_ints(row) for row in arrays['shares']] == orc.split_np_order(orc.field_of(p), s, C, m)
    assert _words_to_ints(arrays['recombined']) == s
