"""The lane-0 recurrence of the t = 3 partial rounds (csrc/poseidon_host.hpp derive_recurrence, csrc/poseidon.cuh
pos_partial_recur): the device code compiled for the CPU with the schedule as the library passes it to the kernels, bit-exact
against the oracle through CRH, two-to-one, sponge and bare permutation; the fallback when the recurrence does not exist; the
schedule's coefficients against Cayley-Hamilton and a dense trace; and the exact bounds behind the unreduced history."""
import ctypes as C
import random
from fractions import Fraction as Fr

import numpy as np
import pytest

from helpers import ALL_CONFIGS, build_host_shim, crafted_sbox_inputs, oracle_config, synth_elems
from oracle import cref, fields as OF, poseidon as OP

u64p = C.POINTER(C.c_uint64)
FID = {"bls12_381_fr": 0, "bn254_fr": 1, "jubjub_fr": 2, "bls12_377_fr": 3}
PRIMES = ((OF.BLS12_381_FR, 0), (OF.BN254_FR, 1), (OF.JUBJUB_FR, 2), (OF.BLS12_377_FR, 3))


@pytest.fixture(scope="module")
def shim():
    return build_host_shim("poseidon_recur_shim")


def _P(a):
    return a.ctypes.data_as(u64p)


def _mont(cfg):
    p = cfg.p
    return cref.ints_to_mont([x for r in cfg.ark for x in r], p), cref.ints_to_mont([x for r in cfg.mds for x in r], p)


def run(shim, fid, cfg, mode, inp, n_out=1):
    """mode 0: CRH (one hinted permutation when len <= rate), 1: generic sponge, 2: bare permutation.  -> (recur, out)"""
    ark, mds = _mont(cfg)
    n, L = inp.shape[0], inp.shape[1]
    out = np.zeros((n, inp.shape[1] if mode == 2 else n_out, 4), dtype=np.uint64)
    rc = shim.recur_run(fid, mode, cfg.rate, cfg.capacity, cfg.full_rounds, cfg.partial_rounds, C.c_ulonglong(cfg.alpha), _P(ark),
                        _P(mds), _P(np.ascontiguousarray(inp)), C.c_long(L), C.c_long(n_out), C.c_long(n), _P(out))
    assert rc >= 0
    return rc, out


def schedule(shim, fid, cfg):
    ark, mds = _mont(cfg)
    rows, ck, rr = (np.zeros((k, 4), dtype=np.uint64) for k in (15, max(cfg.partial_rounds, 1), 10))
    flags = (C.c_int * 2)()
    assert shim.recur_schedule(fid, cfg.rate, cfg.capacity, cfg.full_rounds, cfg.partial_rounds, C.c_ulonglong(cfg.alpha), _P(ark),
                               _P(mds), _P(rows), _P(ck), _P(rr), flags) == 0
    p = cfg.p
    return flags[0], flags[1], cref.mont_to_ints(rows, p), cref.mont_to_ints(ck, p), cref.mont_to_ints(rr, p)


def check_all(shim, fid, cfg, expect_recur, n=6, extra=None):
    """CRH at several lengths (one-permutation and multi-block), two-to-one, sponge with several outputs, bare permutation."""
    p, t = cfg.p, cfg.rate + cfg.capacity
    O = cref.Poseidon(cfg)
    for L in (0, 1, 2, 3, 5):
        inp = np.ascontiguousarray(synth_elems(40 + L, (n, max(L, 1)), p)[:, :L])
        if L:
            inp[0, :] = cref.ints_to_mont([p - 1] * L, p)
        rc, out = run(shim, fid, cfg, 0, inp)
        assert rc == expect_recur
        assert (out[:, 0] == O.crh_batch(inp)).all(), L
    pairs = synth_elems(7, (n, 2), p) if extra is None else extra
    assert (run(shim, fid, cfg, 0, pairs)[1][:, 0] == O.compress_batch(pairs)).all()
    for L, K in ((0, 1), (2, 3), (3, 2)):
        inp = np.ascontiguousarray(synth_elems(60 + L, (3, max(L, 1)), p)[:, :L])
        _, out = run(shim, fid, cfg, 1, inp, n_out=K)
        ints = cref.mont_to_ints(inp, p)
        for i in range(3):
            s = OP.PoseidonSponge(cfg)
            s.absorb(ints[i * L:(i + 1) * L])
            assert cref.mont_to_ints(out[i], p) == s.squeeze_native_field_elements(K), (L, K)
    states = synth_elems(80, (3, t), p)
    states[0] = cref.ints_to_mont([p - 1] * t, p)
    _, out = run(shim, fid, cfg, 2, states)
    for i in range(3):
        assert cref.mont_to_ints(out[i], p) == OP.permute(cfg, cref.mont_to_ints(states[i], p))


@pytest.mark.parametrize("which", ALL_CONFIGS)
def test_named_configs(shim, which):
    """Every named t = 3 configuration (all four fields) derives the recurrence and matches the oracle everywhere."""
    fname, cfg = oracle_config(which)
    check_all(shim, FID[fname], cfg, expect_recur=1)


@pytest.mark.parametrize("rf,rp", [(8, 3), (8, 4), (3, 4), (5, 3), (7, 9), (1, 5)])
def test_short_and_odd_schedules(shim, rf, rp):
    """The fewest partial rounds the recurrence takes (two bootstrap rounds + one), odd RF, random parameters, every field."""
    rnd = random.Random(rf * 100 + rp)
    for p, fid in PRIMES:
        for alpha in (5, 17):
            ark = [[rnd.randrange(p) for _ in range(3)] for _ in range(rf + rp)]
            mds = [[rnd.randrange(p) for _ in range(3)] for _ in range(3)]
            cfg = OP.PoseidonConfig(p, rf, rp, alpha, ark, mds, 2, 1)
            check_all(shim, fid, cfg, expect_recur=1 if rf >= 3 else 0, n=4)


def test_bn254_largest_unreduced_values(shim):
    """BN254 Fr, alpha = 5 keeps x = d + c and the S-box outputs unreduced in the history: round constants at p-1 (x up to 2p-2),
    inputs at p-1 / 0 / 1 and crafted S-box operands, many random inputs."""
    rnd = random.Random(5)
    p = OF.BN254_FR
    for rf, rp in ((8, 57), (8, 3), (4, 4)):
        ark = [[p - 1 - rnd.randrange(3) for _ in range(3)] for _ in range(rf + rp)]
        mds = [[rnd.randrange(p) for _ in range(3)] for _ in range(3)]
        cfg = OP.PoseidonConfig(p, rf, rp, 5, ark, mds, 2, 1)
        inp = synth_elems(9 + rp, (128, 2), p)
        inp[0] = cref.ints_to_mont([p - 1] * 2, p)
        inp[1] = cref.ints_to_mont([0, 0], p)
        inp[2] = cref.ints_to_mont([1, 1], p)
        rc, out = run(shim, 1, cfg, 0, inp)
        assert rc == 1 and (out[:, 0] == cref.Poseidon(cfg).compress_batch(inp)).all(), (rf, rp)
    for which in ("bn254_r2", "bls_default_r2", "bls377_random"):
        fname, cfg = oracle_config(which)
        inp = crafted_sbox_inputs(cfg, 300)
        rc, out = run(shim, FID[fname], cfg, 0, inp)
        assert rc == 1 and (out[:, 0] == cref.Poseidon(cfg).crh_batch(inp)).all(), which


def test_fallback_without_recurrence(shim):
    """A sparse schedule whose lane 2 never reaches lane 0 (M[0][2] = 0, lower block the identity): lanes 1, 2 cannot be rebuilt from
    lane 0, so recur = 0 and the sparse rounds run -- still the oracle's digests.  Likewise t = 2, t = 4 and rp < 3."""
    rnd = random.Random(8)
    for p, fid in PRIMES:
        ark = [[rnd.randrange(p) for _ in range(3)] for _ in range(8 + 9)]
        cfg = OP.PoseidonConfig(p, 8, 9, 5, ark, [[7, 1, 0], [3, 1, 0], [5, 0, 1]], 2, 1)
        sparse, recur, *_ = schedule(shim, fid, cfg)
        assert (sparse, recur) == (1, 0)
        check_all(shim, fid, cfg, expect_recur=0, n=4)
    p = OF.BLS12_381_FR
    for rate, rp in ((1, 9), (3, 9), (2, 2)):
        t = rate + 1
        cfg = OP.PoseidonConfig(p, 8, rp, 5, [[rnd.randrange(p) for _ in range(t)] for _ in range(8 + rp)],
                                [[rnd.randrange(p) for _ in range(t)] for _ in range(t)], rate, 1)
        assert schedule(shim, 0, cfg)[:2] == (1, 0)
        check_all(shim, 0, cfg, expect_recur=0, n=4)


@pytest.mark.parametrize("which", ["bn254_r2", "bls_default_r2"])
def test_schedule_algebra(shim, which):
    """Rounds >= 2 use [m00, b1, b2, -d1, -d2] of Cayley-Hamilton on the lower 2x2 block B of the MDS (z^2 + d1 z + d2), and with the
    schedule's constants they reproduce lane 0 of a dense trace of the reference's permutation."""
    fname, cfg = oracle_config(which)
    p, M = cfg.p, cfg.mds
    sparse, recur, rows, ck, rr = schedule(shim, FID[fname], cfg)
    assert (sparse, recur) == (1, 1)
    m00, a, b = M[0][0], (M[0][1], M[0][2]), (M[1][0], M[2][0])
    B = ((M[1][1], M[1][2]), (M[2][1], M[2][2]))
    d1 = -(B[0][0] + B[1][1]) % p
    d2 = (B[0][0] * B[1][1] - B[0][1] * B[1][0]) % p
    ab = (a[0] * b[0] + a[1] * b[1]) % p
    Bb = [(B[i][0] * b[0] + B[i][1] * b[1]) % p for i in range(2)]
    aBb = (a[0] * Bb[0] + a[1] * Bb[1]) % p
    beta1 = (ab + d1 * m00) % p
    beta2 = (aBb + d1 * ab + d2 * m00) % p
    assert rows[10:15] == [m00, beta1, beta2, -d1 % p, -d2 % p]
    # dense trace: x_k = lane 0 after the constant addition of partial round k
    half, rp = cfg.full_rounds // 2, cfg.partial_rounds
    rnd = random.Random(1)
    for _ in range(3):
        st = [rnd.randrange(p) for _ in range(3)]
        xs, ys = [], []
        for r in range(half + rp):
            st = [(st[i] + cfg.ark[r][i]) % p for i in range(3)]
            if r < half:
                st = [pow(v, cfg.alpha, p) for v in st]
            else:
                xs.append(st[0])
                st[0] = pow(st[0], cfg.alpha, p)
                ys.append(st[0])
            st = [sum(st[j] * M[i][j] for j in range(3)) % p for i in range(3)]
        for k in range(2, rp - 1):
            h = (ys[k], ys[k - 1], ys[k - 2], xs[k], xs[k - 1])
            assert (sum(c * v for c, v in zip(rows[10:15], h)) + ck[k]) % p == xs[k + 1], k


# ---------------------------------------------------------------------------------------------------- exact bounds (BN254 Fr)
P = OF.BN254_FR
R = 1 << 256
rho = Fr(P, R)
TOP = P >> 224


def mont(a, b):
    """upper bound (in units of p) of the unreduced Montgomery product of values below a*p and b*p"""
    return a * b * rho + 1


def needs_x(terms):
    """fp.cuh dot_needs_x<F, terms>"""
    return (terms + 1) * (TOP + 1) > (1 << 32)


def reduce_passes(terms):
    """fp.cuh dot_reduce_passes<F, terms>: conditional subtractions are K + 1"""
    k = 0
    while terms * (TOP + 1) > ((2 << k) - 1) * (1 << 32):
        k += 1
    return k


def test_recurrence_bounds_bn254():
    x = Fr(2)                                                   # x = d + c: d canonical (the dot reduces fully), c canonical
    assert x * rho < 1                                          # fits 256 bits
    assert x * x * rho < 1                                      # fp_sqr<LAZY> precondition: x^2 < R*p
    x2 = mont(x, x)
    x4 = mont(x2, x2)
    assert x2 * x2 * rho < 1 and x4 + 1 < 1 / rho               # second squaring; fp_mul(x4, x): full operand x4 + p < R
    y = mont(x4, x)
    assert y < Fr(16, 10)                                       # S-box output below 1.6p
    # history (y_k, y_k-1, y_k-2, x_k, x_k-1); at round 0 (y_0, s1, s2, x_0, 0) and round 1 (y_1, y_0, s1, x_1, x_0) are smaller
    hist = 3 * y + 2 * x
    assert hist < 5 + 4                                         # what fp_dot<F, 5, EX = 4> declares
    assert needs_x(5) and needs_x(9)                            # the overflow word is kept: the code is that of any 5-term dot
    assert (hist + 1) * rho * (1 << 32) < (1 << 64)             # running value < (sum + 1) p 2^32 fits the 9 limbs + X
    k = reduce_passes(9)
    assert hist * rho + 1 <= (2 << k) and k == 1                # result < 2.67p: two conditional subtractions give canonical d
    # rebuild of lanes 1, 2 from (y_rp-1, y_rp-2, lane 0 (reduced after the last round), x_rp-1)
    reb = 2 * y + 1 + x
    assert reb < 4 + 3
    k = reduce_passes(7)
    assert reb * rho + 1 <= (2 << k)


def test_recurrence_bounds_other_fields():
    """Without the lazy form every history value is canonical: five terms below 5p, the plain fp_dot<F, 5> contract."""
    for p in (OF.BLS12_381_FR, OF.BLS12_377_FR, OF.JUBJUB_FR):
        r = Fr(p, R)
        assert 5 * r * (1 << 32) < (1 << 64)
        assert 5 * r + 1 < 4                                    # at most two conditional subtractions
