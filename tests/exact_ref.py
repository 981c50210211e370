"""Exact integer reference of the FP64 stages (blind rotation, external product, CMux, vertical packing), plain numpy.

Everything here is arithmetic modulo 2^64 on integers: no FFT rounding reaches a result.  Products of a digit polynomial
and a key polynomial are taken either as uint64 wrapping matrix products (any key words), or, when the operands are small
enough that every exact coefficient of the sum is far below 2^53, through a float FFT whose result is rounded back to the
integer it approximates; that route asserts both the size bound and that every value it rounds lies within 1/8 of an
integer.  This module imports neither the product nor the oracle.

Conventions (those of the C ABI and of the CPU oracle):
  * polynomials have N = 512 coefficients, negacyclic (X^N = -1);
  * a GLWE is [K + 1][N] (K mask polynomials, then the body), an LWE under the big key is [K * N + 1];
  * a GGSW is [level][row][col][N], level index 0 = level 1 (the most significant digit);
  * a bootstrap key is [n][pbs_level][K + 1][K + 1][N];
  * vertical-packing GGSW lists are [nbits][...] with index 0 = the most significant selector bit.
"""
import numpy as np

N = 512
_U = np.uint64
_MASK64 = (1 << 64) - 1
FLOAT_ROUTE_BOUND = 2 ** 44   # largest exact |coefficient| of a digit-key sum taken through the float FFT (see _float_sum)


def as_u64(x):
    """uint64 view of integer words (negative int64 values wrap modulo 2^64)"""
    x = np.asarray(x)
    if x.dtype == np.uint64:
        return x
    return np.ascontiguousarray(x, dtype=np.int64).view(np.uint64)


def as_i64(x):
    """uint64 words read as signed (two's complement) integers"""
    return as_u64(x).view(np.int64)


# ---- signed decomposition ------------------------------------------------------------------------------------------
def signed_digits(x, base_log, level):
    """Balanced signed decomposition with closest-representable rounding, as tfhe-rs' SignedDecomposer and the oracle
    (decomp_init_state / decomp_next) do it: a digit equal to +-B/2 is +B/2 when the next state bit is 0, -B/2 (carry 1)
    otherwise.  Returns int64 [level, *x.shape], index l - 1 = level l (level 1 most significant); sum_l d_l 2^(64 - l
    base_log) = closest(x) mod 2^64."""
    assert 0 < base_log * level < 64
    x = as_u64(x)
    r = 64 - base_log * level
    with np.errstate(over="ignore"):
        v = ((x >> _U(r)) + ((x >> _U(r - 1)) & _U(1))) & _U(_MASK64 >> r)
        mask = _U((1 << base_log) - 1)
        out = np.empty((level,) + x.shape, dtype=np.int64)
        for lev in range(level, 0, -1):
            res = v & mask
            v = v >> _U(base_log)
            carry = (((res - _U(1)) | v) & res) >> _U(base_log - 1)
            v = v + carry
            out[lev - 1] = res.astype(np.int64) - (carry << _U(base_log)).astype(np.int64)
    return out


def signed_digits_85(x):
    """The (2^8, 5) recoding of the PBS kernels (cmux_core.cuh decomp85_*, pbs_cl2_kernel.cu digit_of_level, the digit
    parking of pbs_ws2_kernel.cu): one addition of 2^23 + 128 * (2^24 + 2^32 + .. + 2^56) and a byte per level, so a tie
    (+-128) always becomes -128 with a carry.  Same value as signed_digits(x, 8, 5), digits in [-128, 127]."""
    x = as_u64(x)
    with np.errstate(over="ignore"):
        y = x + _U(0x8080808080800000)
    out = np.empty((5,) + x.shape, dtype=np.int64)
    for lev in range(1, 6):
        out[lev - 1] = ((y >> _U(24 + 8 * (5 - lev))) & _U(0xFF)).astype(np.int64) - 128
    return out


def kernel_digits(x, base_log, level):
    """The decomposition the CUDA kernels apply: the byte recoding at (2^8, 5), the tfhe-rs rule otherwise."""
    if (base_log, level) == (8, 5):
        return signed_digits_85(x)
    return signed_digits(x, base_log, level)


# ---- negacyclic products ------------------------------------------------------------------------------------------------
def negacyclic_matrix(p):
    """T (uint64 [N][N]) with (T @ d)[i] = sum_j d[j] p[i - j] (negacyclic), exact modulo 2^64 in uint64 arithmetic."""
    p = as_u64(p)
    n = p.size
    i, j = np.meshgrid(np.arange(n), np.arange(n), indexing="ij")
    with np.errstate(over="ignore"):
        return np.where(i >= j, p[(i - j) % n], _U(0) - p[(i - j) % n])


def negacyclic_mul(d, p):
    """d * p mod (X^N + 1, 2^64) for integer digits d [..., N] and u64 words p [N], in uint64 wrapping arithmetic."""
    t = negacyclic_matrix(p)
    with np.errstate(over="ignore"):
        return (as_u64(np.asarray(d, dtype=np.int64)) @ t.T).astype(np.uint64)


def _spectrum(a):
    return np.fft.rfft(np.asarray(a, dtype=np.float64), n=2 * N)


def _float_sum(spec, bound):
    """Round the negacyclic sum whose length-2N spectrum is spec back to exact integers.  Why this is exact: every
    coefficient of the exact sum is an integer of magnitude <= bound <= 2^44; the double-precision FFT of length 2N = 1024
    errs by at most ~ bound * 2^-53 * 4 log2(1024) = bound * 2^-47.7 < 2^-3, so nearest-integer rounding returns the exact
    value.  The assertion on the rounding residual checks this on every coefficient."""
    assert bound <= FLOAT_ROUTE_BOUND, f"operands too large for the float route: bound 2^{np.log2(bound):.1f}"
    t = np.fft.irfft(spec, n=2 * N)
    r = t[..., :N] - t[..., N:]
    ri = np.rint(r)
    assert np.abs(r - ri).max(initial=0.0) < 0.125, "float route not exact"
    return ri.astype(np.int64)


# ---- external product, CMux ---------------------------------------------------------------------------------------------
def external_product(ggsw, glwe, base_log, level, digits=kernel_digits):
    """GGSW (x) glwe modulo 2^64: sum over level l and row r of digit_l(glwe[r]) * ggsw[l][r][c] for every output column c.
    ggsw [level][K+1][K+1][N] (u64 words, or signed integers), glwe u64 [..., K+1, N] -> u64 [..., K+1, N]."""
    ggsw = np.asarray(ggsw)
    kp1 = ggsw.shape[1]
    assert ggsw.shape == (level, kp1, kp1, N)
    glwe = as_u64(glwe)
    dig = digits(glwe, base_log, level)                                   # [level, ..., K+1, N]
    w = as_i64(ggsw) if ggsw.dtype == np.uint64 else ggsw.astype(np.int64)
    wmax = int(np.abs(w.astype(np.float64)).max(initial=0))
    dmax = int(np.abs(dig).max(initial=0))
    bound = level * kp1 * N * dmax * wmax
    batch = glwe.shape[:-2]
    if bound <= FLOAT_ROUTE_BOUND:
        ds = _spectrum(dig)                                               # [level, ..., K+1, N+1]
        ws = _spectrum(w)                                                 # [level, K+1, K+1, N+1]
        ds = np.moveaxis(ds, 0, -3).reshape(batch + (level * kp1, N + 1))        # [..., level*row, f]
        spec = np.einsum("...kf,kcf->...cf", ds, ws.reshape(level * kp1, kp1, N + 1), optimize=True)
        return _float_sum(spec, bound).view(np.uint64)
    out = np.zeros(batch + (kp1, N), dtype=np.uint64)
    with np.errstate(over="ignore"):
        for lev in range(level):
            for r in range(kp1):
                d = as_u64(dig[lev][..., r, :])   # digits as two's-complement words: the sum wraps like the exact one
                for c in range(kp1):
                    out[..., c, :] += d @ negacyclic_matrix(ggsw[lev, r, c]).T
    return out


def external_product_add(ggsw, glwe, acc, base_log, level, digits=kernel_digits):
    """acc + GGSW (x) glwe (the oracle's external_product_add)"""
    with np.errstate(over="ignore"):
        return as_u64(acc) + external_product(ggsw, glwe, base_log, level, digits)


def cmux(ggsw, c0, c1, base_log, level, digits=kernel_digits):
    """c0 + GGSW (x) (c1 - c0): c1 when the GGSW encrypts 1, c0 when it encrypts 0"""
    with np.errstate(over="ignore"):
        return external_product_add(ggsw, as_u64(c1) - as_u64(c0), c0, base_log, level, digits)


# ---- monomials, sample extraction ---------------------------------------------------------------------------------------
def monomial_mul(poly, deg):
    """poly * X^deg (negacyclic).  poly u64 [..., N]; deg an int or an int array broadcasting against poly[..., 0]."""
    poly = as_u64(poly)
    deg = np.asarray(deg, dtype=np.int64)[..., None] % (2 * N)
    s = (np.arange(N) - deg) % (2 * N)                                    # source index of coefficient j, in [0, 2N)
    src = np.take_along_axis(poly, np.broadcast_to(s % N, poly.shape), axis=-1)
    with np.errstate(over="ignore"):
        return np.where(np.broadcast_to(s >= N, poly.shape), _U(0) - src, src)


def sample_extract(glwe, post_add=0):
    """LWE of coefficient 0 of glwe [..., K+1, N] -> [..., K*N + 1]: mask r = (a_r[0], -a_r[N-1], .., -a_r[1])"""
    glwe = as_u64(glwe)
    mask = glwe[..., :-1, :]
    with np.errstate(over="ignore"):
        rev = np.concatenate([mask[..., :1], _U(0) - mask[..., :0:-1]], axis=-1)
        body = glwe[..., -1, 0] + _U(post_add & _MASK64)
    return np.concatenate([rev.reshape(glwe.shape[:-2] + (-1,)), body[..., None]], axis=-1)


# ---- blind rotation (PBS) -----------------------------------------------------------------------------------------------
def mod_switch(x, in_scale=1, add=0):
    """(x * in_scale + add + 2^53) >> 54 mod 2N, wrapping modulo 2^64 (ws_mod_switch_2n in ws_common.cuh)"""
    with np.errstate(over="ignore"):
        y = as_u64(x) * _U(in_scale & _MASK64) + _U(add & _MASK64) + _U(1 << 53)
    return ((y >> _U(54)) & _U(2 * N - 1)).astype(np.int64)


def blind_rotate(lwe, lut, bsk, pre_add=0, post_add=0, in_scale=1, base_log=8, level=5, digits=kernel_digits):
    """PBS of every row of lwe [B][n+1] with the trivial accumulator (0, .., 0, X^-b~ lut) and the bootstrap key bsk
    [n][level][K+1][K+1][N]: acc += BSK_i (x) (acc * X^a~_i - acc) for i = 0 .. n-1, then sample extract of coefficient 0,
    post_add on the body.  pre_add is added to the body before its modulus switch.  Returns u64 [B][K*N + 1]."""
    lwe = np.atleast_2d(as_u64(lwe))
    bsk = np.asarray(bsk)
    n, kp1 = bsk.shape[0], bsk.shape[2]
    assert lwe.shape[1] == n + 1 and bsk.shape == (n, level, kp1, kp1, N)
    b = mod_switch(lwe[:, n], in_scale, pre_add)
    acc = np.zeros((lwe.shape[0], kp1, N), dtype=np.uint64)
    acc[:, -1] = monomial_mul(np.broadcast_to(as_u64(lut), (lwe.shape[0], N)), -b)
    for i in range(n):
        a = mod_switch(lwe[:, i], in_scale)
        with np.errstate(over="ignore"):
            diff = monomial_mul(acc, a[:, None]) - acc
        acc = external_product_add(bsk[i], diff, acc, base_log, level, digits)
    return sample_extract(acc, post_add)


# ---- vertical packing ---------------------------------------------------------------------------------------------------
def vertical_packing(lut, ggsw, kp1, base_log=15, level=1, digits=kernel_digits):
    """tfhe-rs vertical_packing (and tfa_vertical_packing) for every output at once.
    lut u64 [nouts][npoly][N] (npoly a power of two), ggsw [nbits][level][K+1][K+1][N], index 0 = most significant bit.
    CMux tree over the top log2(npoly) bits (when there are that many), least significant tree bit first, leaves = trivial
    GLWEs of the LUT polynomials; then a blind rotation over the remaining bits, least significant first, by X^-(2^t);
    then sample extract.  Returns u64 [nouts][K*N + 1]."""
    lut = as_u64(lut)
    nouts, npoly = lut.shape[:2]
    nbits = len(ggsw)
    tree = int(np.log2(npoly))
    assert 1 << tree == npoly
    if tree > nbits:
        tree = 0
    cur = np.zeros((nouts, 1 << tree, kp1, N), dtype=np.uint64)
    cur[:, :, -1] = lut[:, :1 << tree]
    for layer in range(tree - 1, -1, -1):
        cur = cmux(ggsw[layer], cur[:, 0::2], cur[:, 1::2], base_log, level, digits)
    acc = cur[:, 0]
    for t, g in enumerate(range(nbits - 1, tree - 1, -1)):
        with np.errstate(over="ignore"):
            diff = monomial_mul(acc, -(1 << t)) - acc
        acc = external_product_add(ggsw[g], diff, acc, base_log, level, digits)
    return sample_extract(acc)
