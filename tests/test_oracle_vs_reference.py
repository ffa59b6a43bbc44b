"""Cross-check of the oracle against the UNMODIFIED reference on randomised (p, m, t, n) instances of every function on
the path, beyond the edge cases of the other golden fixtures -- split (np and list order), recombination vectors and
recombination, f_S(i), PRF, PRSS shares and zero-shares, the field-array operators and the protocols' local algebra.
The instances come from the seeded generators below; what the reference returned on them (secrets.randbelow replaced
by the instance's fixed stream for the duration of each call) is stored in tests/golden/random_instances.json, written
by tests/golden/make_golden_random.py."""
import itertools
import random

import pytest

from golden_util import load, unhex
from oracle import shamir_oracle as orc

PRIMES = [2**61 - 1, 2**64 - 189, 2**69 - 93, 2**128 - 173, 2**256 - 189, 9409569905028393239, 101, 2**89 - 1]


def split_instances(p):
    rnd = random.Random(p % 10007)
    for m, t in ((1, 0), (3, 1), (4, 1), (5, 2), (7, 3), (6, 5)):
        n = rnd.randrange(1, 9)
        s = [rnd.randrange(p) for _ in range(n)]
        stream = [rnd.randrange(p) for _ in range(t * n)]
        xs = sorted(rnd.sample(range(1, m + 1), min(m, t + 1)))
        i = rnd.randrange(m)
        subsets = [S for S in itertools.combinations(range(m), m - t) if i in S]
        keys = {S: bytes(rnd.randrange(256) for _ in range(16)) for S in subsets}
        uci = bytes(rnd.randrange(256) for _ in range(5))
        yield dict(m=m, t=t, n=n, s=s, stream=stream, xs=xs, i=i, keys=keys, uci=uci)


def operator_instance(p):
    rnd = random.Random(p % 7919)
    a = [rnd.randrange(p) for _ in range(12)]
    b = [rnd.randrange(1, p) for _ in range(12)]
    return a, b


def local_instances(p):
    rnd = random.Random(p % 9973)
    for _ in range(6):
        n, f = rnd.randrange(1, 7), rnd.randrange(1, 75)
        a, b, c = ([rnd.randrange(p) for _ in range(n)] for _ in range(3))
        s, t = rnd.randrange(p), rnd.randrange(p)
        nb = rnd.randrange(0, p.bit_length() + 3)
        bits = [rnd.randrange(p) for _ in range(n * f)]
        l = rnd.randrange(1, p.bit_length() + 1)
        yield dict(n=n, f=f, a=a, b=b, c=c, s=s, t=t, nb=nb, bits=bits, l=l)


def bit_rows(rows):
    """A 0/1 matrix as stored in the fixture: one string of '0' and '1' per row."""
    return [''.join(map(str, r)) for r in rows]


@pytest.fixture(scope='module')
def golden():
    return load('random_instances.json')['primes']


@pytest.mark.parametrize('p', PRIMES, ids=lambda p: f'p{p.bit_length()}')
def test_split_recombine_prss_random_instances(golden, p):
    Fo = orc.field_of(p)
    cases = golden[hex(p)]['split']
    instances = list(split_instances(p))
    assert len(cases) == len(instances)
    for inst, g in zip(instances, cases):
        m, t, n, s, stream, xs, i = (inst[k] for k in ('m', 't', 'n', 's', 'stream', 'xs', 'i'))
        sh_np = unhex(g['shares_np'])
        assert sh_np == orc.split_np_order(Fo, s, orc.np_stream_to_C(stream, t, n), m)
        assert unhex(g['shares_list']) == orc.split_list_order(Fo, s, orc.list_stream_to_c(stream, t, n), m)
        for x_r, want in zip((0, m + 1), g['lambda']):
            assert unhex(want) == orc.recombination_vector(Fo, xs, x_r)
        assert unhex(g['recombined']) == orc.recombine(Fo, xs, [sh_np[x - 1] for x in xs]) == s
        # PRSS for one party
        keys, uci = inst['keys'], inst['uci']
        for S in keys:
            assert unhex(g['f_S_i'][','.join(map(str, S))]) == orc.f_S_i(Fo, m, i, S) % p
        assert unhex(g['prss']) == orc.prss_share(Fo, m, i, {S: orc.prf_values(k, p, uci, n) for S, k in keys.items()}, n)
        if t:
            prl = {S: orc.prf_values(k, p, uci, n * t) for S, k in keys.items()}
            assert unhex(g['zero_np']) == orc.prss_share_zero_np_order(Fo, m, i, prl, n)
            assert unhex(g['zero_list']) == orc.prss_share_zero_list_order(Fo, m, i, prl, n)


@pytest.mark.parametrize('p', PRIMES, ids=lambda p: f'p{p.bit_length()}')
def test_field_array_operators_random_instances(golden, p):
    a, b = operator_instance(p)
    g = {k: unhex(v) for k, v in golden[hex(p)]['operators'].items()}
    assert g['add'] == orc.ff_add(p, a, b)
    assert g['sub'] == orc.ff_sub(p, a, b)
    assert g['mul'] == orc.ff_mul(p, a, b)
    assert g['neg'] == orc.ff_neg(p, a)
    assert g['reciprocal'] == orc.ff_inv(p, b)
    assert g['div'] == orc.ff_div(p, a, b)
    assert g['lshift5'] == orc.ff_lshift(p, a, 5)
    assert g['rshift5'] == orc.ff_rshift(p, a, 5)
    assert g['pow7'] == orc.ff_pow(p, a, 7)


@pytest.mark.parametrize('p', PRIMES, ids=lambda p: f'p{p.bit_length()}')
def test_local_algebra_random_instances(golden, p):
    """oracle.local_* against the expressions of np_random_bits / np_trunc / np_sgn / np_to_bits (mpyc/runtime.py:860,
    870, 3646-3660, 4252-4271, 4415) evaluated on the reference's field arrays, random sizes and bit counts."""
    cases = golden[hex(p)]['local']
    instances = list(local_instances(p))
    assert len(cases) == len(instances)
    for inst, g in zip(instances, cases):
        n, f, a, b, c, bits, l = (inst[k] for k in ('n', 'f', 'a', 'b', 'c', 'bits', 'l'))
        assert unhex(g['square_add']) == orc.local_fma(p, a, a, c)
        assert unhex(g['fma']) == orc.local_fma(p, a, b, c)
        assert unhex(g['axpb']) == orc.local_axpb(p, a, inst['s'], inst['t'])
        assert unhex(g['low_bits']) == orc.local_low_bits(c, inst['nb'])
        assert g['nonzero'] == orc.local_nonzero(a)
        assert unhex(g['compose_asc']) == orc.local_bits_compose(p, bits, n, f)
        assert unhex(g['compose_desc']) == orc.local_bits_compose(p, bits, n, f, descending=True)
        assert g['decompose_desc'] == bit_rows(orc.local_bits_decompose(c, l, descending=True))
        assert g['decompose_asc'] == bit_rows(orc.local_bits_decompose(c, l))
