// cmux_core.cuh — one CMux step  acc += GGSW (x) ct1  for G ciphertexts resident in one CTA.
//
// This is the inner loop of every FP64 stage of the reference's per-byte chain:
//   * blind rotation inside the PBS of circuit_bootstrap_boolean (many_wopbs.rs:253; 669 steps
//     with the bootstrap key, beta = 2^8, l = 5) and of the general extract_bits loop (:194),
//   * the blind-rotation half of vertical_packing (many_wopbs.rs:277; 8-9 steps with the
//     circuit-bootstrapped GGSWs, beta = 2^15, l = 1),
//   * the CMux tree of vertical_packing when a LUT spans several polynomials.
// Arithmetic follows SURVEY.md §9.3-9.6 (signed decomposition, forward FFT of the digits,
// multiply-accumulate against the Fourier GGSW, inverse FFT, round, add).
//
// CTA organisation (256 threads = 16 groups of 16 lanes):
//   FFT phases:  group g handles polynomial r = g % (K+1) of ciphertext ct = g / (K+1)
//                (G*(K+1) <= 16 groups busy).  Lane n2 owns coefficients 16 n1 + n2 (+256).
//   MAC phase:   thread p owns Fourier point p of all G ciphertexts and all K+1 output
//                polynomials; the GGSW value for (level, row, *, p) is loaded once and used G times.
// Fourier GGSW layout: [level slot][row][col][p] complex, slot 0 = level LEVELS (the order in which the
// decomposition produces the digits, SURVEY §9.3), p = natural DFT index.
// The phases below are separate __host__ __device__ functions so that emu.cu can run them on the CPU
// thread by thread; the kernels call them with barriers in between.
#pragma once
#include "fft_core.cuh"

#define CMUX_THREADS 256
#define CMUX_GROUPS 16
#define POLY_N 512
#define POLY_M 256

enum { DIFF_ROTATE = 0, DIFF_EXTERNAL = 1 };

template <int K, int G>
struct CmuxSmem {
    uint64_t acc[G][K + 1][POLY_N];      // the G accumulators (GLWE, standard domain)
    cd xb[G * (K + 1)][XB_ELEMS];        // exchange / hand-over buffers, one per busy 16-lane group
    cd tw[256];                          // mid twiddles, swizzled (fft_core.cuh)
    int rot[G];                          // per-ciphertext rotation amount of the current step, in [0, 2N)
};

template <int K, int G>
struct CmuxRegs {
    cd v[16];              // FFT working set
    uint32_t st_re[16];    // decomposition state of coefficient 16 n1 + lane
    uint32_t st_im[16];    // decomposition state of coefficient 16 n1 + lane + 256
    cd facc[G][K + 1];     // Fourier accumulators of point p = tid
};

// theta^(e) = exp(2 pi i e / 1024); used once per CTA to fill the twiddle tables
HD cd theta_pow(int e, const double *cos1024 /* [1024] */, const double *sin1024) {
    e &= 1023;
    return cmk(cos1024[e], sin1024[e]);
}

// coefficient j of (acc * X^rot): rot in [0, 2N)
HD uint64_t rotated_coef(const uint64_t *poly, int j, int rot) {
    int s = (j - rot) & (2 * POLY_N - 1);
    uint64_t x = poly[s & (POLY_N - 1)];
    return (s & POLY_N) ? (uint64_t)0 - x : x;
}

// First decomposition step from the full 64-bit value: returns the digit of level LEVELS and leaves
// the (<= 32-bit) state for the remaining levels (SURVEY §9.3).
template <int BASE_LOG, int LEVELS>
HD int decomp_first(uint64_t x, uint32_t &state) {
    constexpr int R = 64 - BASE_LOG * LEVELS;
    uint64_t s = ((x >> R) + ((x >> (R - 1)) & 1)) & (~0ull >> R);
    uint32_t res = (uint32_t)s & ((1u << BASE_LOG) - 1);
    uint32_t st = (uint32_t)(s >> BASE_LOG);
    uint32_t carry = (((res - 1u) | st) & res) >> (BASE_LOG - 1);
    state = st + carry;
    return (int)res - (int)(carry << BASE_LOG);
}
template <int BASE_LOG>
HD int decomp_next(uint32_t &state) {
    uint32_t res = state & ((1u << BASE_LOG) - 1);
    uint32_t st = state >> BASE_LOG;
    uint32_t carry = (((res - 1u) | st) & res) >> (BASE_LOG - 1);
    state = st + carry;
    return (int)res - (int)(carry << BASE_LOG);
}

// ---- signed decomposition for (beta, l) = (2^8, 5), the bootstrap-key decomposition (client.rs:42-43) ----
// All five digits at once: with r = 64 - 40 = 24, x' = x + 2^23 (closest representable, SURVEY §9.3) plus the
// offset 128 * (1 + 2^8 + .. + 2^32) << 24 has, in bits 24..63, the bytes  d_j + 128  of a balanced digit set
// d_j in [-128, 127] with  sum_j d_j 2^(8j) = closest(x) >> 24  (mod 2^40): adding 128 per byte lets the
// carries of the signed recoding ripple in ONE 64-bit addition.  Digit of level 5 (least significant,
// consumed first) = byte 3 of the low word; the high word holds levels 4, 3, 2, 1 in bytes 0..3.
// Byte -> double without a conversion instruction (I2F.F64 issues at 1/4 of the FP64 rate on B200,
// scratch/mb_xu.cu): the byte becomes the low mantissa bits of 2^52, and one exact subtraction of 2^52 + 128
// leaves d_j.
// Difference from tfhe-rs' iterator: an exact tie (digit = +-128) is always resolved to -128 (+1 carry)
// where tfhe-rs picks by a state bit; both recodings represent the same value, so the external product is
// the same up to the noise realisation (DESIGN.md §4).
#ifndef USE_DECOMP85
#define USE_DECOMP85 1
#endif
#define DECOMP85_ADD 0x8080808080800000ull
HD double digit85(uint32_t w, int b) {
#ifdef __CUDA_ARCH__
    const uint32_t byte = __byte_perm(w, 0, 0x4440 + b);
    return __hiloint2double(0x43300000, (int)byte) - 4503599627370624.0;   // (2^52 + byte) - (2^52 + 128)
#else
    return (double)(int)((w >> (8 * b)) & 0xFF) - 128.0;
#endif
}
// first digit (level 5) and the state word holding the other four
HD double decomp85_first(uint64_t x, uint32_t &state) {
    const uint64_t y = x + DECOMP85_ADD;
    state = (uint32_t)(y >> 32);
    return digit85((uint32_t)y, 3);
}
// digit of level lev in 4..1
HD double decomp85_level(uint32_t state, int lev) { return digit85(state, 4 - lev); }

// ---- phase A: build ct1 = (acc * X^rot - acc) [DIFF_ROTATE] or (ext - acc) [DIFF_EXTERNAL] for the
// 32 coefficients this lane owns, start the decomposition, emit the digits of the first level into v.
template <int K, int G, int BASE_LOG, int LEVELS, int MODE>
HD void phase_load_decompose(int tid, CmuxSmem<K, G> &sm, CmuxRegs<K, G> &rg, const uint64_t *const *ext /* [G] GLWE pointers */) {
    const int gid = tid >> 4, lane = tid & 15;
#pragma unroll
    for (int ct = 0; ct < G; ct++)
#pragma unroll
        for (int c = 0; c <= K; c++) rg.facc[ct][c] = cmk(0.0, 0.0);
    if (gid >= G * (K + 1)) return;
    const int ct = gid / (K + 1), r = gid % (K + 1);
    const uint64_t *poly = sm.acc[ct][r];
    const int s0 = (lane - sm.rot[ct]) & (2 * POLY_N - 1);
#pragma unroll
    for (int n1 = 0; n1 < 16; n1++) {
        const int j = 16 * n1 + lane;
        uint64_t a0, a1;
        if (MODE == DIFF_ROTATE) {
            // (acc * X^rot)[j] and [j + 256]: source index s = j - rot mod 2N, sign flips when s >= N;
            // adding 256 to j toggles bit 8 of s and carries into the sign bit
            const int s = (s0 + 16 * n1) & (2 * POLY_N - 1);
            const int i0 = s & (POLY_N - 1);
            const uint64_t x0 = poly[i0], x1 = poly[i0 ^ POLY_M];
            const uint64_t m0 = (uint64_t)0 - (uint64_t)((s >> 9) & 1);
            const uint64_t m1 = (uint64_t)0 - (uint64_t)(((s >> 9) ^ (s >> 8)) & 1);
            a0 = ((x0 ^ m0) - m0) - poly[j];
            a1 = ((x1 ^ m1) - m1) - poly[j + POLY_M];
        } else {
            const uint64_t *e = ext[ct] + (size_t)r * POLY_N;
            a0 = e[j] - poly[j];
            a1 = e[j + POLY_M] - poly[j + POLY_M];
        }
        double d0, d1;
        if (USE_DECOMP85 && BASE_LOG == 8 && LEVELS == 5) {
            d0 = decomp85_first(a0, rg.st_re[n1]);
            d1 = decomp85_first(a1, rg.st_im[n1]);
        } else {
            d0 = (double)decomp_first<BASE_LOG, LEVELS>(a0, rg.st_re[n1]);
            d1 = (double)decomp_first<BASE_LOG, LEVELS>(a1, rg.st_im[n1]);
        }
        rg.v[n1] = cmk(d0, d1);
    }
}
// register-only forms used by the warp-specialised PBS kernel (no Fourier accumulators in the FFT warps)
template <int BASE_LOG, int LEVELS>
HD void load_decompose_rot(const uint64_t *poly, int lane, int rot, cd (&v)[16], uint32_t (&st_re)[16], uint32_t (&st_im)[16]) {
    const int s0 = (lane - rot) & (2 * POLY_N - 1);
#pragma unroll
    for (int n1 = 0; n1 < 16; n1++) {
        const int j = 16 * n1 + lane;
        const int s = (s0 + 16 * n1) & (2 * POLY_N - 1);
        const int i0 = s & (POLY_N - 1);
        const uint64_t x0 = poly[i0], x1 = poly[i0 ^ POLY_M];
        const uint64_t m0 = (uint64_t)0 - (uint64_t)((s >> 9) & 1);
        const uint64_t m1 = (uint64_t)0 - (uint64_t)(((s >> 9) ^ (s >> 8)) & 1);
        const uint64_t a0 = ((x0 ^ m0) - m0) - poly[j];
        const uint64_t a1 = ((x1 ^ m1) - m1) - poly[j + POLY_M];
        double d0, d1;
        if (USE_DECOMP85 && BASE_LOG == 8 && LEVELS == 5) {
            d0 = decomp85_first(a0, st_re[n1]);
            d1 = decomp85_first(a1, st_im[n1]);
        } else {
            d0 = (double)decomp_first<BASE_LOG, LEVELS>(a0, st_re[n1]);
            d1 = (double)decomp_first<BASE_LOG, LEVELS>(a1, st_im[n1]);
        }
        v[n1] = cmk(d0, d1);
    }
}
// digits of level lev (LEVELS-1 .. 1; levels are consumed in decreasing order)
template <int BASE_LOG, int LEVELS>
HD void next_digits(cd (&v)[16], uint32_t (&st_re)[16], uint32_t (&st_im)[16], int lev) {
#pragma unroll
    for (int n1 = 0; n1 < 16; n1++) {
        double d0, d1;
        if (USE_DECOMP85 && BASE_LOG == 8 && LEVELS == 5) {
            d0 = decomp85_level(st_re[n1], lev);
            d1 = decomp85_level(st_im[n1], lev);
        } else {
            d0 = (double)decomp_next<BASE_LOG>(st_re[n1]);
            d1 = (double)decomp_next<BASE_LOG>(st_im[n1]);
        }
        v[n1] = cmk(d0, d1);
    }
}
template <int K, int G, int BASE_LOG, int LEVELS>
HD void phase_next_digits(int tid, CmuxRegs<K, G> &rg, int lev) {
    if ((tid >> 4) >= G * (K + 1)) return;
    next_digits<BASE_LOG, LEVELS>(rg.v, rg.st_re, rg.st_im, lev);
}
// ---- forward FFT of the digit polynomial held in v -------------------------------------------
// The *_b variants take the base of a [16][XB_ELEMS] exchange / hand-over buffer and the twiddle table
// explicitly (the warp-specialised PBS kernel double-buffers it); the CmuxSmem forms use sm.xb.
template <int K, int G>
HD void phase_fwd1_b(int tid, cd (*xb)[XB_ELEMS], const cd *tw, cd (&v)[16]) {
    const int gid = tid >> 4, lane = tid & 15;
    if (gid >= G * (K + 1)) return;
    fft256_fwd_pass1(v, lane, tw, xb[gid]);
}
template <int K, int G>
HD void phase_fwd2_b(int tid, cd (*xb)[XB_ELEMS], cd (&v)[16]) {
    const int gid = tid >> 4, lane = tid & 15;
    if (gid >= G * (K + 1)) return;
    fft256_fwd_pass2(v, lane, xb[gid]);
}
template <int K, int G>
HD void phase_fwd3_b(int tid, cd (*xb)[XB_ELEMS], cd (&v)[16]) {
    const int gid = tid >> 4, lane = tid & 15;
    if (gid >= G * (K + 1)) return;
#pragma unroll
    for (int k2 = 0; k2 < 16; k2++) xb[gid][lane + 16 * k2] = v[rev4(k2)];
}
template <int K, int G>
HD void phase_fwd1(int tid, CmuxSmem<K, G> &sm, CmuxRegs<K, G> &rg) { phase_fwd1_b<K, G>(tid, sm.xb, sm.tw, rg.v); }
template <int K, int G>
HD void phase_fwd2(int tid, CmuxSmem<K, G> &sm, CmuxRegs<K, G> &rg) { phase_fwd2_b<K, G>(tid, sm.xb, rg.v); }
template <int K, int G>
HD void phase_fwd3(int tid, CmuxSmem<K, G> &sm, CmuxRegs<K, G> &rg) { phase_fwd3_b<K, G>(tid, sm.xb, rg.v); }
// ---- multiply-accumulate of one level against the Fourier GGSW -------------------------------
// ggsw_level points at [row r][col c][point p] complex of this level.
template <int K, int G>
HD void phase_mac(int tid, CmuxSmem<K, G> &sm, CmuxRegs<K, G> &rg, const cd *__restrict__ ggsw_level) {
    const int p = tid;
#pragma unroll
    for (int r = 0; r <= K; r++) {
        cd w[K + 1];
        const cd *g = ggsw_level + (size_t)r * (K + 1) * POLY_M + p;
#pragma unroll
        for (int c = 0; c <= K; c++) {
#ifdef __CUDA_ARCH__
            w[c] = __ldg(g + c * POLY_M);
#else
            w[c] = g[c * POLY_M];
#endif
        }
#pragma unroll
        for (int ct = 0; ct < G; ct++) {
            const cd x = sm.xb[ct * (K + 1) + r][p];
#pragma unroll
            for (int c = 0; c <= K; c++) cmac(rg.facc[ct][c], x, w[c]);
        }
    }
}
// software-pipelined form: operands of the NEXT row are fetched while the current row is computed
template <int K, int G>
struct MacOperands { cd w[K + 1]; cd x[G]; };
template <int K, int G>
HD void mac_fetch(int tid, const CmuxSmem<K, G> &sm, int r, const cd *w_ptr, MacOperands<K, G> &o) {
#pragma unroll
    for (int c = 0; c <= K; c++) o.w[c] = w_ptr[c * POLY_M];
#pragma unroll
    for (int ct = 0; ct < G; ct++) o.x[ct] = sm.xb[ct * (K + 1) + r][tid];
}
template <int K, int G>
HD void mac_compute(CmuxRegs<K, G> &rg, const MacOperands<K, G> &o) {
#pragma unroll
    for (int ct = 0; ct < G; ct++)
#pragma unroll
        for (int c = 0; c <= K; c++) cmac(rg.facc[ct][c], o.x[ct], o.w[c]);
}
// ---- inverse transform of the K+1 accumulators of every ciphertext and update of acc ----------
template <int K, int G>
HD void phase_inv0(int tid, CmuxSmem<K, G> &sm, CmuxRegs<K, G> &rg) {
    const int p = tid;
#pragma unroll
    for (int ct = 0; ct < G; ct++)
#pragma unroll
        for (int c = 0; c <= K; c++) sm.xb[ct * (K + 1) + c][p] = rg.facc[ct][c];
}
template <int K, int G>
HD void phase_inv1_b(int tid, cd (*xb)[XB_ELEMS], cd (&v)[16]) {
    const int gid = tid >> 4, lane = tid & 15;
    if (gid >= G * (K + 1)) return;
#pragma unroll
    for (int k2 = 0; k2 < 16; k2++) v[k2] = xb[gid][lane + 16 * k2];
    fft256_inv_pass1_compute(v);
}
template <int K, int G>
HD void phase_inv2_b(int tid, cd (*xb)[XB_ELEMS], const cd *tw, cd (&v)[16]) {
    const int gid = tid >> 4, lane = tid & 15;
    if (gid >= G * (K + 1)) return;
    fft256_inv_pass1_store(v, lane, tw, xb[gid]);
}
// acc: base of the [G][K+1][512] accumulator array
template <int K, int G>
HD void phase_inv3_b(int tid, cd (*xb)[XB_ELEMS], uint64_t (*acc)[K + 1][POLY_N], cd (&v)[16]) {
    const int gid = tid >> 4, lane = tid & 15;
    if (gid >= G * (K + 1)) return;
    const int ct = gid / (K + 1), c = gid % (K + 1);
    fft256_inv_pass2(v, lane, xb[gid]);
    uint64_t *poly = acc[ct][c];
#pragma unroll
    for (int n1 = 0; n1 < 16; n1++) {
        const int j = 16 * n1 + lane;
        poly[j] += f64_to_torus(v[n1].x);
        poly[j + POLY_M] += f64_to_torus(v[n1].y);
    }
}
template <int K, int G>
HD void phase_inv1(int tid, CmuxSmem<K, G> &sm, CmuxRegs<K, G> &rg) { phase_inv1_b<K, G>(tid, sm.xb, rg.v); }
template <int K, int G>
HD void phase_inv2(int tid, CmuxSmem<K, G> &sm, CmuxRegs<K, G> &rg) { phase_inv2_b<K, G>(tid, sm.xb, sm.tw, rg.v); }
template <int K, int G>
HD void phase_inv3(int tid, CmuxSmem<K, G> &sm, CmuxRegs<K, G> &rg) { phase_inv3_b<K, G>(tid, sm.xb, sm.acc, rg.v); }

// ---- forward transform of a torus polynomial (key conversion, SURVEY §9.4(6)) -----------------
// lane loads 32 coefficients as signed 64-bit -> f64 (53-bit rounding, SURVEY §9.6)
HD void load_torus_poly(cd (&v)[16], int lane, const uint64_t *poly) {
#pragma unroll
    for (int n1 = 0; n1 < 16; n1++) {
        const int j = 16 * n1 + lane;
        v[n1] = cmk((double)(int64_t)poly[j], (double)(int64_t)poly[j + POLY_M]);
    }
}
