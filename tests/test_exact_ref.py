"""Self-checks of tests/exact_ref.py, the exact integer reference the GPU FP64 tests compare with (CPU only: the oracle
library is built by __graft_entry__.build(), no GPU is needed).

  * its two product routes (uint64 matrices, float FFT on small-norm operands) agree bit for bit;
  * its decompositions equal the oracle's (tfhe-rs rule) and the kernels' (2^8, 5) byte recoding;
  * external_product_add is bit-exact against the oracle on small-norm GGSWs (the oracle's FFT rounds exactly there too);
  * with the oracle's real keys, where the oracle's FFT rounding is noise, blind rotation and vertical packing agree with
    the oracle on the phase and decrypt to the LUT entry the secret key selects."""
import numpy as np
import pytest

import exact_ref as X

N = 512


def _dist(a, b):
    with np.errstate(over="ignore"):
        return int(np.abs((X.as_u64(a) - X.as_u64(b)).view(np.int64).astype(np.float64)).max())


def test_float_route_equals_matrix_route():
    rng = np.random.default_rng(0)
    for K, bl, lv, wlog in ((1, 8, 5, 16), (4, 8, 5, 16), (4, 15, 1, 16)):
        ggsw = rng.integers(-2 ** wlog, 2 ** wlog + 1, (lv, K + 1, K + 1, N))
        glwe = rng.integers(0, 2 ** 64, (3, K + 1, N), dtype=np.uint64)
        fast = X.external_product(ggsw, glwe, bl, lv)
        slow = np.zeros_like(fast)
        dig = X.kernel_digits(glwe, bl, lv)
        with np.errstate(over="ignore"):
            for lev in range(lv):
                for r in range(K + 1):
                    for c in range(K + 1):
                        slow[:, c] += X.negacyclic_mul(dig[lev][:, r], ggsw[lev, r, c])
        assert np.array_equal(fast, slow), (K, bl, lv)
    # full-range words take the matrix route
    ggsw = rng.integers(0, 2 ** 64, (1, 2, 2, N), dtype=np.uint64)
    glwe = rng.integers(0, 2 ** 64, (2, N), dtype=np.uint64)
    got = X.external_product(ggsw, glwe, 15, 1)
    d = X.signed_digits(glwe, 15, 1)[0]
    with np.errstate(over="ignore"):
        want = [X.negacyclic_mul(d[0], ggsw[0, 0, c]) + X.negacyclic_mul(d[1], ggsw[0, 1, c]) for c in range(2)]
    assert np.array_equal(got, np.stack(want))


def test_negacyclic_mul_by_monomial():
    rng = np.random.default_rng(1)
    p = rng.integers(0, 2 ** 64, N, dtype=np.uint64)
    for deg in (0, 1, 511, 512, 513, 1023):
        mono = np.zeros(N, dtype=np.int64)
        mono[deg % N] = -1 if deg >= N else 1
        assert np.array_equal(X.negacyclic_mul(mono, p), X.monomial_mul(p, deg)), deg
    assert np.array_equal(X.monomial_mul(X.monomial_mul(p, 300), -300), p)


def test_decompositions_match_oracle_and_kernel_recoding(orc):
    rng = np.random.default_rng(2)
    x = rng.integers(0, 2 ** 64, 3000, dtype=np.uint64)
    # exact ties at every level of both bases, and the words next to the wrap
    x[:8] = [0, (1 << 64) - 1, 1 << 63, 0x0000008000800000, 0x7F7F7F7F7F800000, 0x8080808080800000, 1 << 48, 3 << 48]
    for bl, lv in ((8, 5), (15, 1), (12, 3), (2, 6)):
        mine = X.signed_digits(x, bl, lv)
        for i in range(x.size):
            ref = orc.decompose(int(x[i]), bl, lv)                 # index 0 = level lv (least significant)
            assert list(mine[::-1, i]) == [int(v) for v in ref], (bl, lv, hex(int(x[i])))
    k = X.signed_digits_85(x)
    t = X.signed_digits(x, 8, 5)
    assert k.min() >= -128 and k.max() <= 127
    with np.errstate(over="ignore"):
        val = lambda d: sum(X.as_u64(d[lev - 1]) << np.uint64(64 - 8 * lev) for lev in range(1, 6))
        assert np.array_equal(val(k), val(t))
    assert (k != t).any(), "the inputs must contain ties the two rules resolve differently"


@pytest.mark.parametrize("K", [1, 4])
def test_external_product_bit_exact_against_oracle(orc, K):
    """Small-norm GGSWs: the oracle's double-precision FFT rounds to the exact integers as well, so its words equal the
    reference's exactly (with the oracle's tie rule; the (2^8, 5) kernel recoding differs from it on ties)."""
    o = orc.Oracle(orc.param_opt() if K == 4 else orc.param_test())       # no keys needed
    rng = np.random.default_rng(3 + K)
    for bl, lv in ((8, 5), (15, 1)):
        ggsw = rng.integers(-2 ** 16, 2 ** 16 + 1, (lv, K + 1, K + 1, N)).astype(np.int64)
        glwe = rng.integers(0, 2 ** 64, (K + 1) * N, dtype=np.uint64)
        glwe[:4] = [0, (1 << 64) - 1, 1 << 63, 0x8080808080800000]
        acc = rng.integers(0, 2 ** 64, (K + 1) * N, dtype=np.uint64)
        ref = o.external_product_add(ggsw.view(np.uint64).reshape(lv, K + 1, (K + 1) * N), bl, lv, glwe, acc)
        got = X.external_product_add(ggsw, glwe.reshape(K + 1, N), acc.reshape(K + 1, N), bl, lv, X.signed_digits)
        assert np.array_equal(got.ravel(), ref), (K, bl, lv)


def test_blind_rotation_matches_oracle_bootstrap(oracle_test):
    """Real keys at the test parameters: the oracle's FFT rounding (~2^26 per step) is noise, the tolerance 2^36 is that of
    test_gpu_parity.  With the secret key, the phase is the LUT coefficient the modulus-switched phase selects."""
    o = oracle_test
    rng = np.random.default_rng(5)
    lut = rng.integers(0, 2 ** 64, N, dtype=np.uint64)
    lwe = o.encrypt_lwe_small(rng.integers(0, 2 ** 64, 6, dtype=np.uint64))
    bsk = o.bsk().reshape(o.n, 5, o.k + 1, o.k + 1, N)
    got = X.blind_rotate(lwe, lut, bsk, digits=X.signed_digits)
    ref = o.bootstrap(lwe, lut)
    assert _dist(o.phase_big(got), o.phase_big(ref)) < 2 ** 36
    s = o.lwe_sk().astype(np.int64)
    idx = (X.mod_switch(lwe[:, -1]) - (X.mod_switch(lwe[:, :-1]) * s).sum(axis=1)) % (2 * N)
    want = np.array([X.monomial_mul(lut, -int(i))[0] for i in idx], dtype=np.uint64)
    assert _dist(o.phase_big(got), want) < 2 ** 40      # the PBS noise of the oracle's key (std 2^-50 on the GLWE side)
    # pre_add / post_add: the same as adding them to the input body and to the output body
    lwe2 = lwe.copy()
    lwe2[:, -1] += np.uint64(1 << 62)
    got2 = X.blind_rotate(lwe, lut, bsk, pre_add=1 << 62, post_add=12345, digits=X.signed_digits)
    ref2 = X.blind_rotate(lwe2, lut, bsk, digits=X.signed_digits)
    ref2[:, -1] += np.uint64(12345)
    assert np.array_equal(got2, ref2)


@pytest.mark.parametrize("nbits,npoly", [(3, 1), (4, 2), (5, 4)])
def test_vertical_packing_matches_oracle(oracle_test, nbits, npoly):
    """Tree depth 0, 1, 2 at K = 1 with circuit-bootstrapped GGSWs: phase within 2^36 of the oracle (its level-1 FFT
    rounding is ~2^31 per CMux, test_emulation), and the result decrypts to the LUT entry of the encrypted index."""
    o = oracle_test
    rng = np.random.default_rng(10 * nbits + npoly)
    value = int(rng.integers(0, 2 ** nbits))
    bits = [(value >> (nbits - 1 - i)) & 1 for i in range(nbits)]
    lwe = o.encrypt_lwe_small(np.array(bits, dtype=np.uint64) << np.uint64(63))
    ggsw = np.stack([o.circuit_bootstrap_boolean(l) for l in lwe])          # [nbits][1][2][1024]
    lut = rng.integers(0, 2, (2, npoly, N)).astype(np.uint64) << np.uint64(63)
    got = X.vertical_packing(lut, ggsw.reshape(nbits, 1, 2, 2, N), 2)
    for j in range(2):
        assert _dist(o.phase_big(got[j]), o.phase_big(o.vertical_packing(lut[j], ggsw))) < 2 ** 36
    nrot = nbits - int(np.log2(npoly))            # the tree bits pick the polynomial, the others the coefficient
    entry = (value >> nrot) * N + (value & ((1 << nrot) - 1))
    assert np.array_equal(o.decrypt_bits(got), (lut.reshape(2, -1)[:, entry] >> np.uint64(63)).astype(np.uint8))
