"""Generate tests/golden/random_instances.json by running the UNMODIFIED reference (lschoe/mpyc) on the seeded random
instances of tests/test_oracle_vs_reference.py.

    MPYC_REFERENCE=<reference checkout> python tests/golden/make_golden_random.py

secrets.randbelow is replaced, for the duration of each split, by the instance's fixed stream (as in make_golden.py).
Only the reference's outputs are stored: the test regenerates the inputs from the same seeds.  Integers are hex strings,
0/1 matrices one string of digits per row.
"""
import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
TESTS = os.path.dirname(HERE)
REF = os.environ['MPYC_REFERENCE']
sys.dont_write_bytecode = True
sys.path[:0] = [REF, os.path.dirname(TESTS), TESTS]
_argv, sys.argv = sys.argv, [sys.argv[0], '--no-log']   # mpyc parses sys.argv at import
from mpyc import finfields, thresha   # noqa: E402
import numpy as np   # noqa: E402
sys.argv = _argv

from test_oracle_vs_reference import PRIMES, bit_rows, local_instances, operator_instance, split_instances   # noqa: E402


def hx(v):
    if isinstance(v, (list, tuple)):
        return [hx(x) for x in v]
    if isinstance(v, np.ndarray):
        return hx(v.tolist())
    return hex(int(v))


class injected:
    """Context manager: secrets.randbelow -> next value of a fixed stream (restored on exit)."""

    def __init__(self, stream):
        self.it = iter(stream)

    def __enter__(self):
        self.orig = thresha.secrets.randbelow
        thresha.secrets.randbelow = lambda order: next(self.it)

    def __exit__(self, *exc):
        thresha.secrets.randbelow = self.orig


def split_cases(p):
    F = finfields.GF(p)
    out = []
    for inst in split_instances(p):
        m, t, n, s, stream, xs, i, keys, uci = (inst[k] for k in ('m', 't', 'n', 's', 'stream', 'xs', 'i', 'keys', 'uci'))
        with injected(stream):
            sh_np = thresha.np_random_split(F, F.array(np.array(s, dtype=object)), t, m)
        with injected(stream):
            sh_li = thresha.random_split(F, [F(x) for x in s], t, m)
        lam = [[int(v) % p for v in thresha._recombination_vector(F, tuple(xs), x_r)] for x_r in (0, m + 1)]
        y = thresha.np_recombine(F, [(x, sh_np[x - 1]) for x in xs])
        prfs = {S: thresha.PRF(k, p) for S, k in keys.items()}
        case = {'shares_np': hx(sh_np), 'shares_list': hx(sh_li), 'lambda': hx(lam), 'recombined': hx(y.value),
                'f_S_i': {','.join(map(str, S)): hex(int(thresha._f_S_i(F, m, i, S)) % p) for S in keys},
                'prss': hx(thresha.np_pseudorandom_share(F, m, i, prfs, uci, n).value)}
        if t:
            case['zero_np'] = hx(thresha.np_pseudorandom_share_0(F, m, i, prfs, uci, n).value)
            case['zero_list'] = hx([a.value for a in thresha.pseudorandom_share_zero(F, m, i, prfs, uci, n)])
        out.append(case)
    return out


def operator_case(p):
    F = finfields.GF(p)
    a, b = operator_instance(p)
    A, B = F.array(np.array(a, dtype=object)), F.array(np.array(b, dtype=object))
    ops = {'add': A + B, 'sub': A - B, 'mul': A * B, 'neg': -A, 'reciprocal': B.reciprocal(), 'div': A / B,
           'lshift5': A << 5, 'rshift5': A >> 5, 'pow7': A ** 7}
    return {k: hx(v.value) for k, v in ops.items()}


def local_cases(p):
    """The raw-value expressions of np_random_bits / np_trunc / np_sgn / np_to_bits (mpyc/runtime.py:860, 870,
    3646-3660, 4252-4271, 4415) on the reference's field arrays."""
    Zp = finfields.GF(p)
    arr = lambda v: Zp.array(np.array(v, dtype=object))   # noqa: E731
    out = []
    for inst in local_instances(p):
        n, f, l = inst['n'], inst['f'], inst['l']
        A, B, C, R = arr(inst['a']), arr(inst['b']), arr(inst['c']), arr(inst['bits'])
        out.append({'square_add': hx(Zp.array(A.value**2 + C.value).value),
                    'fma': hx(Zp.array(A.value * B.value + C.value).value),
                    'axpb': hx(Zp.array(A.value * inst['s'] + inst['t']).value),
                    'low_bits': hx(C.value & ((1 << inst['nb']) - 1)),
                    'nonzero': (A.value != 0).tolist(),
                    'compose_asc': hx(Zp.array(np.sum(R.value.reshape((n, f)) << np.arange(f), axis=1)).value),
                    'compose_desc': hx(Zp.array(np.sum(R.value.reshape((n, f)) << np.arange(f - 1, -1, -1), axis=1)).value),
                    'decompose_desc': bit_rows((np.right_shift.outer(C.value, np.arange(l - 1, -1, -1)).T & 1).tolist()),
                    'decompose_asc': bit_rows((np.right_shift.outer(C.value, np.arange(l)).T & 1).tolist())})
    return out


def main():
    obj = {'meta': {'reference': 'lschoe/mpyc v0.11.2 (unmodified)'},
           'primes': {hex(p): {'split': split_cases(p), 'operators': operator_case(p), 'local': local_cases(p)} for p in PRIMES}}
    path = os.path.join(HERE, 'random_instances.json')
    with open(path, 'w') as fh:
        json.dump(obj, fh, separators=(',', ':'))
    print(path, os.path.getsize(path), 'bytes')


if __name__ == '__main__':
    main()
