// pbs_ws_kernel.cu — warp-specialised PBS (blind rotation + sample extract), sm_100a.
//
// The CMux arithmetic of cmux_core.cuh, in a warp-specialised schedule.  One CTA of 512
// threads holds G ciphertexts for all n CMux steps:
//   warps 8-15 "FFT warps" : per step: rotate-subtract + signed decomposition, per level a forward FFT of
//                            every digit polynomial into its hand-over slot, then the K+1 inverse FFTs and the
//                            accumulator update.  Each 16-lane group owns polynomial (ct, r) and only ever
//                            touches its own accumulator polynomial and its own slot, so FFT groups never wait
//                            for each other (warp-level syncs only).
//   warps 0-7  "MAC warps" : thread p owns Fourier point p of all G ciphertexts and multiplies row r of the
//                            current level as soon as the G slots (*, r) are full, while the FFT warps already
//                            work on the next level (the first pass of the next FFT runs in registers before
//                            the slot is free).
// The FFT phases are FP64-pipe bound and the multiply-accumulate is shared-memory bound (it reads 52 KB per row
// for 60 FMAs per thread), so the two roles use complementary resources; run in separate warps they overlap
// instead of alternating, with four warps per scheduler instead of two.  The roles have different register
// needs (FFT: 16 complex + 32 decomposition states; MAC: G*(K+1) complex accumulators), so the register file
// is re-balanced with setmaxnreg (144 / 112 per thread at G = 3).
//
// Bootstrap key: rows [col][p] of (K+1) x 4 KB, stored in consumption order, streamed L2 -> shared memory by
// the TMA engine (cp.async.bulk, one lane per row) into a ring of K+1 slots (one level); BFULL[0/1] count the
// bytes of the first / second half of the rows of a level, BEMPTY[r] one arrival per MAC warp; the producer role rotates over the MAC warps and refills
// the slot released one row earlier.
// Hand-shake per row r (mbarriers in shared memory): RFULL[r] (one arrival per FFT group (ct, r), MAC threads
// wait), REMPTY[r] (one arrival per MAC warp, the FFT lanes of row r wait before they overwrite their slot),
// INV (MAC warps arrive after leaving the Fourier accumulators in the slots, FFT lanes wait).
#include "ws_common.cuh"

// scratch/pbs_lab builds several variants of this file into one binary: each gets its own namespace and launcher name
#ifndef PBS_WS_NS
#define PBS_WS_NS ws_default
#endif
#ifndef PBS_WS_LAUNCH_NAME
#define PBS_WS_LAUNCH_NAME launch_pbs_ws
#endif
// Tuning switches.  The defaults are the configuration measured best on B200 with scratch/pbs_lab (one wave of 444 ciphertexts,
// every variant checked bit for bit against the round-1 kernel): 10.12 ms against 10.59 ms.  DESIGN.md §7 lists what was measured
// for each of them and for the schedules that lost (row-ahead barrier probes, software-pipelined MAC rows, twiddles on the pass-2 side).
#ifndef WS_MAC_REUSE
#define WS_MAC_REUSE 1    // FMAs of one key value ordered so that consecutive DFMAs share an operand (a DFMA with three distinct
#endif                    // register operands issues every 3 cycles on B200, every 2 with one operand reused: scratch/mb_fp64ops.cu)
#ifndef WS_REVMAP
#define WS_REVMAP 1       // FFT groups in reverse warp order: the issue arbiter favours high warp ids and the MAC role consumes row 0 first
#endif
#ifndef WS_TWB_INV
#define WS_TWB_INV 8      // inverse pass 1: mid twiddles fetched in batches of 8 (0: one by one, each load behind the previous store)
#endif
#ifndef WS_ROT_LATE
#define WS_ROT_LATE 1     // the next mask element is fetched before the inverse FFT and mod-switched after it
#endif
#ifndef WS_TMEM_ST
#define WS_TMEM_ST 1      // the digits of the levels still to come are parked in tensor memory (tcgen05.st / tcgen05.ld, 32 columns per thread)
#endif                    // instead of 32 registers per FFT thread: no spills, and ptxas keeps several twiddle loads in flight (10.40 -> 10.12 ms)
#ifndef WS_DIAG
#define WS_DIAG 0         // diagnostics of scratch/pbs_lab: each bit removes one piece of work (results are WRONG when != 0)
#endif
#ifndef WS_TIMING
#define WS_TIMING 0       // scratch/pbs_lab: per-activity clock64() sums of CTA 0 (FFT thread 0, MAC thread 0) into PbsArgs::dbg[0..WT_COUNT)
#endif
namespace PBS_WS_NS {

template <int K, int G>
struct WsSmem {
    uint64_t acc[G][K + 1][POLY_N];      // the G accumulators (GLWE, standard domain)
    cd hs[(K + 1) * G][XB_ELEMS];        // hand-over slots: spectrum / Fourier accumulator of (ct, r) at [r * G + ct]
    cd tw[256];                          // mid twiddles, swizzled (fft_core.cuh)
    cd ring[K + 1][K + 1][POLY_M];       // one level of the Fourier bootstrap key: [row][col][p]
    uint64_t rfull[K + 1];
    uint64_t rempty[K + 1];
    uint64_t bfull[2];                   // key rows 0..BSPLIT-1 / BSPLIT..K of a level have landed
    uint64_t bempty[K + 1];
    uint64_t inv;
    uint32_t tmem_base;                  // WS_TMEM_ST: base address of the allocated tensor-memory columns
    uint32_t pad_;
};

// facc[g][c] += x[g] * w for all g, in an order that lets consecutive DFMAs share the key component as one operand: a DFMA with
// three distinct register operands issues every 3 cycles on B200, with one operand from the reuse cache every 2
// (scratch/mb_fp64ops.cu).  Per accumulator the order of the two updates is that of cmac (bit-identical results).
template <int G, int KP1>
__device__ __forceinline__ void cmac_cols(cd (&facc)[G][KP1], int c, const cd (&x)[G], cd w) {
#pragma unroll
    for (int g = 0; g < G; g++) facc[g][c].x = fma(x[g].x, w.x, facc[g][c].x);
#pragma unroll
    for (int g = 0; g < G; g++) facc[g][c].y = fma(x[g].x, w.y, facc[g][c].y);
#pragma unroll
    for (int g = 0; g < G; g++) facc[g][c].x = fma(-x[g].y, w.y, facc[g][c].x);
#pragma unroll
    for (int g = 0; g < G; g++) facc[g][c].y = fma(x[g].y, w.x, facc[g][c].y);
}

enum { WT_F_DECOMP, WT_F_PASS1, WT_F_WAIT_EMPTY, WT_F_POST, WT_F_WAIT_INV, WT_F_INV, WT_M_WAIT, WT_M_MAC, WT_M_HANDOVER, WT_COUNT };
template <int K, int G, int BASE_LOG, int LEVELS>
__global__ void __launch_bounds__(WS_THREADS, 1) pbs_ws_kernel(PbsArgs a) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    long long tacc[6] = {0, 0, 0, 0, 0, 0};
    long long tlast = WS_TIMING ? clock64() : 0;
#define WT(k) do { if (WS_TIMING) { const long long t_ = clock64(); tacc[(k) % 6] += t_ - tlast; tlast = t_; } } while (0)
    WsSmem<K, G> &sm = *reinterpret_cast<WsSmem<K, G> *>(smem_raw);
    const int tid = threadIdx.x;
    const int n = a.lwe_dim;
    const int ct0 = blockIdx.x * G;
    constexpr int RING = K + 1;
    constexpr int ROWS = LEVELS * (K + 1);
    constexpr int ROW_ELEMS = POLY_M * (K + 1);
    constexpr unsigned ROW_BYTES = (unsigned)(ROW_ELEMS * sizeof(cd));
    const int nrows = n * ROWS;
    // register split (per thread, 8 + 8 warps, 128 on average): the MAC role holds G*(K+1) complex accumulators
    // The key ring is watched by two barriers per level (a try_wait costs ~95 cycles on the barrier unit even when
    // the phase is long complete, and they serialise): rows [0, BSPLIT) are waited for when the level starts, rows
    // [BSPLIT, K] just before row BSPLIT (the slot of the last row is only refilled at row 0 of the next level).
    constexpr int BSPLIT = (K + 2) / 2;
    constexpr int MAC_REGS = G >= 3 ? WS_MAC_REGS3 : (G == 2 ? 96 : 72);

    // ---- prologue (all 512 threads) ---------------------------------------------------------------
    for (int i = tid; i < 256; i += WS_THREADS) sm.tw[i] = a.tw[i];
    if (tid == 0) {
        for (int r = 0; r <= K; r++) {
            // spectra-ready barriers are shared by pairs of rows (0,1), (2,3), (4): the barrier unit serialises try_waits
            // at ~95 cycles each, and in steady state the FFT role is far enough ahead for the pair to be complete
            ws_mbar_init(&sm.rfull[r], G * ((r | 1) <= K ? 2 : 1));
            ws_mbar_init(&sm.rempty[r], WS_MAC_WARPS);
            ws_mbar_init(&sm.bempty[r], WS_MAC_WARPS);
        }
        ws_mbar_init(&sm.bfull[0], BSPLIT);
        ws_mbar_init(&sm.bfull[1], K + 1 - BSPLIT);
        ws_mbar_init(&sm.inv, WS_MAC_WARPS);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
#if WS_TMEM_ST
    if (tid < 32) {   // warp 0: 64 columns = 32 per FFT warp, two FFT warps per lane quarter
#if WS_DIAG & 256
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(ws_smem_u32(&sm.tmem_base)) : "memory");
#else
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 64;" ::"r"(ws_smem_u32(&sm.tmem_base)) : "memory");
#endif
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
#endif
    for (int g = 0; g < G; g++) {
        const int rot = (2 * POLY_N - ws_mod_switch_2n(a, min(ct0 + g, a.count - 1), n)) & (2 * POLY_N - 1);
        for (int idx = tid; idx < (K + 1) * POLY_N; idx += WS_THREADS) {
            const int r = idx / POLY_N, j = idx % POLY_N;
            sm.acc[g][r][j] = (r == K) ? rotated_coef(a.lut, j, rot) : 0;
        }
    }
    __syncthreads();

    // Role by warp index: the MAC role takes warps 0-7 and the FFT role warps 8-15.  The FFT warps are the critical
    // path (they carry 64 % of the FP64 work plus all integer work), and the issue arbiter favours the higher
    // warp ids when several warps of a scheduler are eligible.
#ifndef WS_FFT_HIGH
#define WS_FFT_HIGH 1
#endif
    if (WS_FFT_HIGH ? (tid >= WS_THREADS - WS_FFT_THREADS) : (tid < WS_FFT_THREADS)) {
        // ================================ FFT warps ================================================
        if (MAC_REGS <= 128) asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(256 - MAC_REGS));
        else asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(256 - MAC_REGS));
        const int ftid = WS_FFT_HIGH ? tid - (WS_THREADS - WS_FFT_THREADS) : tid;
#if WS_REVMAP   // groups in reverse warp order: the issue arbiter favours high warp ids, and the MAC role consumes row 0 first
        const int gid = 15 - (ftid >> 4), lane = ftid & 15;
#else
        const int gid = ftid >> 4, lane = ftid & 15;
#endif
        const bool active = gid < G * (K + 1);
        // group -> polynomial: row-major (r = gid / G, ct = gid % G), so that the two groups of a warp own the same
        // or adjacent rows and the warp-uniform wait below never holds a row-r group back until row r+2 is consumed
        const int ct = active ? gid % G : 0, r = active ? gid / G : 0;
        // Both 16-lane groups of a warp execute ONE instruction stream (a diverged half-warp would pay a full
        // issue slot and a full FP64 pipe pass for 16 lanes): waits are made warp-uniform by waiting for the
        // later row of the two groups; an idle group (gid >= G*(K+1)) runs along with its stores predicated off.
#if WS_REVMAP
        const int gid_a = 14 - (ftid >> 5) * 2, gid_b = gid_a + 1;
#else
        const int gid_a = (ftid >> 5) * 2, gid_b = gid_a + 1;
#endif
        const int r_a = gid_a / G;
        const int r_b = (gid_b < G * (K + 1)) ? gid_b / G : r_a;
        cd *slot = sm.hs[active ? gid : 0];
        const int my_ct = min(ct0 + ct, a.count - 1);
        cd v[16];
        uint32_t st_re[16], st_im[16];
#if WS_TMEM_ST
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        // this warp's lane quarter is (tid / 32) % 4; the two FFT warps that share a quarter use columns 0..31 / 32..63
        const unsigned taddr = sm.tmem_base + ((unsigned)(((tid >> 5) & 3) * 32) << 16) + (unsigned)((ftid >> 7) * 32);
#endif
        unsigned produced = 0;                    // levels this group has produced so far
        if (gid_a < G * (K + 1)) {
            int rot = ws_mod_switch_2n(a, my_ct, 0);
#pragma unroll 1
            for (int i = 0; i < n; i++) {
                // the mask element of the next step is fetched one step ahead (its latency hides behind a CMux)
#if !WS_ROT_LATE
                const int rot_next = (i + 1 < n) ? ws_mod_switch_2n(a, my_ct, i + 1) : 0;
#endif
                load_decompose_rot<BASE_LOG, LEVELS>(sm.acc[ct][r], lane, rot, v, st_re, st_im);
#if WS_TMEM_ST
                // park the digits of levels 4..1: per level one word per four coefficients (8 words), 32 columns per thread
#pragma unroll
                for (int b = 0; b < 4; b++) {
                    uint32_t pk[8];
#pragma unroll
                    for (int j = 0; j < 4; j++) {
                        pk[j] = ws_gather_byte(st_re[4 * j], st_re[4 * j + 1], st_re[4 * j + 2], st_re[4 * j + 3], b);
                        pk[4 + j] = ws_gather_byte(st_im[4 * j], st_im[4 * j + 1], st_im[4 * j + 2], st_im[4 * j + 3], b);
                    }
                    ws_tmem_st8(taddr + b * 8, pk);
                }
                ws_tmem_wait_st();
#endif
#if !WS_ROT_LATE
                rot = rot_next;
#endif
                WT(WT_F_DECOMP);
#pragma unroll 1
                for (int lev = LEVELS; lev >= 1; lev--) {
#if WS_TMEM_ST
                    if (lev != LEVELS) {
                        uint32_t pk[8];
                        ws_tmem_ld8(taddr + (4 - lev) * 8, pk);
#pragma unroll
                        for (int n1 = 0; n1 < 16; n1++) v[n1] = cmk(digit85(pk[n1 >> 2], n1 & 3), digit85(pk[4 + (n1 >> 2)], n1 & 3));
                    }
#else
                    if (lev != LEVELS) next_digits<BASE_LOG, LEVELS>(v, st_re, st_im, lev);
#endif
                    // first pass in registers; only then wait until the MAC warps have consumed the previous
                    // occupant of the slot (rows of the previous production)
#if WS_DIAG & 64           // diagnostic (wrong results): no first-pass arithmetic
                    v[0].x += 1.0;
#else
                    fft256_fwd_pass1_compute(v, lane, sm.tw);
#endif
                    WT(WT_F_PASS1);
                    // (every MAC warp releases the rows of a level in order, so the release of row r_b >= r_a implies r_a's)
#if !(WS_DIAG & 128)
                    if (produced > 0) ws_mbar_wait(&sm.rempty[r_b], (produced - 1) & 1);
#endif
                    WT(WT_F_WAIT_EMPTY);
                    if (active) fft256_fwd_pass1_store(v, lane, slot);
                    __syncwarp();
#if WS_DIAG & 8            // diagnostic (wrong results): loads of pass 2 without its arithmetic
#pragma unroll
                    for (int n2 = 0; n2 < 16; n2++) v[n2] = slot[xb_idx(lane, n2)];
#elif WS_DIAG & 16         // diagnostic (wrong results): arithmetic of pass 2 without its loads
                    fft16<1>(v);
#else
                    fft256_fwd_pass2(v, lane, slot);
#endif
                    __syncwarp();
                    if (active) {
#pragma unroll
                        for (int k2 = 0; k2 < 16; k2++) slot[lane + 16 * k2] = v[rev4(k2)];
                    }
                    __syncwarp();
#if !(WS_DIAG & 128)
                    if (active && lane == 0) ws_mbar_arrive(&sm.rfull[r & ~1]);
#endif
                    produced++;
                    WT(WT_F_POST);
                }
#if WS_ROT_LATE
                // raw mask element of the next step: loaded here (registers are free once the digits are consumed), used
                // after the inverse transform, so that neither its latency nor its registers sit in the decomposition
                const uint64_t raw_next = a.lwe_in[(size_t)my_ct * (n + 1) + min(i + 1, n - 1)];
#endif
                // inverse transform of the Fourier accumulator the MAC warps left in this group's slot
#if !(WS_DIAG & 128)
                ws_mbar_wait(&sm.inv, i & 1);
#endif
                WT(WT_F_WAIT_INV);
#pragma unroll
                for (int k2 = 0; k2 < 16; k2++) v[k2] = slot[lane + 16 * k2];
                fft256_inv_pass1_compute(v);
                __syncwarp();
#if WS_TWB_INV
                if (active) fft256_inv_pass1_store_b<WS_TWB_INV>(v, lane, sm.tw, slot);
#else
                if (active) fft256_inv_pass1_store(v, lane, sm.tw, slot);
#endif
                __syncwarp();
                fft256_inv_pass2(v, lane, slot);
                if (active) {
                    uint64_t *poly = sm.acc[ct][r];
#pragma unroll
                    for (int n1 = 0; n1 < 16; n1++) {
                        const int j = 16 * n1 + lane;
                        poly[j] += f64_to_torus(v[n1].x);
                        poly[j + POLY_M] += f64_to_torus(v[n1].y);
                    }
                }
                __syncwarp();
#if WS_ROT_LATE
                rot = (int)((raw_next * a.in_scale + (1ull << 53)) >> 54) & (2 * POLY_N - 1);
#endif
                WT(WT_F_INV);
            }
            if (WS_TIMING && a.dbg && blockIdx.x == 0 && ftid == 0)
                for (int k = 0; k < 6; k++) a.dbg[k] = (uint64_t)tacc[k];
        }
    } else {
        // ================================ MAC warps ================================================
        if (MAC_REGS <= 128) asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(MAC_REGS));
        else asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(MAC_REGS));
        const int p = WS_FFT_HIGH ? tid : tid - WS_FFT_THREADS;
        const int mwarp = p >> 5, mlane = p & 31;
        auto produce = [&](int q) {               // fetch key row q into slot q % RING (the caller knows it is free)
            const int s = q % RING;
            uint64_t *bar = &sm.bfull[s < BSPLIT ? 0 : 1];
#if WS_DIAG & 2          // diagnostic (wrong results): 16 bytes per key row instead of 20 KB
            ws_mbar_arrive_expect_tx(bar, 16);
            ws_bulk_copy_g2s(&sm.ring[s][0][0], a.bsk + (size_t)q * ROW_ELEMS, 16, bar);
#else
            ws_mbar_arrive_expect_tx(bar, ROW_BYTES);
            ws_bulk_copy_g2s(&sm.ring[s][0][0], a.bsk + (size_t)q * ROW_ELEMS, ROW_BYTES, bar);
#endif
        };
        if (p == 0)
            for (int q = 0; q < RING; q++) produce(q);   // nrows >= RING always
        cd facc[G][K + 1];
        const int n_mac = (WS_DIAG & 128) ? 0 : n;   // diagnostic: no MAC role at all
        unsigned level_count = 0;
        int q = 0;                                // next key row to consume
#pragma unroll 1
        for (int i = 0; i < n_mac; i++) {
#pragma unroll
            for (int g = 0; g < G; g++)
#pragma unroll
                for (int c = 0; c <= K; c++) facc[g][c] = cmk(0.0, 0.0);
#pragma unroll 1
            for (int lev = LEVELS; lev >= 1; lev--) {
                const unsigned parity = level_count & 1;
#pragma unroll
                for (int r = 0; r <= K; r++, q++) {
                    if (r == 0) ws_mbar_wait2(&sm.bfull[0], parity, &sm.rfull[0], parity);
                    else if (r == BSPLIT && (r & 1) == 0) ws_mbar_wait2(&sm.bfull[1], parity, &sm.rfull[r], parity);
                    else if (r == BSPLIT) ws_mbar_wait(&sm.bfull[1], parity);
                    else if ((r & 1) == 0) ws_mbar_wait(&sm.rfull[r], parity);
                    WT(WT_M_WAIT);
#if WS_DIAG & 32           // diagnostic (wrong results): the MAC role only runs the barrier protocol
                    if (0) {
#else
                    {
#endif
                    cd x[G];
#pragma unroll
                    for (int g = 0; g < G; g++) x[g] = sm.hs[r * G + g][p];
#pragma unroll
                    for (int c = 0; c <= K; c++) {   // key values are streamed one at a time (register budget)
#if WS_DIAG & 256    // diagnostic (wrong results): key values read from tensor memory (whatever it holds) instead of the shared-memory ring
                        cd w;
                        {
                            uint32_t t0, t1, t2, t3;
                            const unsigned ta = sm.tmem_base + ((unsigned)(((tid >> 5) & 3) * 32) << 16) + 64u + (unsigned)(r * 40 + (p >> 7) * 20 + c * 4);
                            asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0,%1,%2,%3}, [%4];" : "=r"(t0), "=r"(t1), "=r"(t2), "=r"(t3) : "r"(ta));
                            asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
                            w = cmk(__hiloint2double((int)t1, (int)t0), __hiloint2double((int)t3, (int)t2));
                        }
#elif WS_DIAG & 1      // diagnostic (wrong results): one key load per row instead of K+1
                        const cd w = sm.ring[r][0][p];
#else
                        const cd w = sm.ring[r][c][p];
#endif
#if WS_DIAG & 4      // diagnostic (wrong results): a quarter of the FMAs
                        if (c == 0) cmac(facc[0][c], x[0], w);
                        else { facc[0][c].x += w.x; }
#else
#if WS_MAC_REUSE
                        cmac_cols<G, K + 1>(facc, c, x, w);
#else
#pragma unroll
                        for (int g = 0; g < G; g++) cmac(facc[g][c], x[g], w);
#endif
#endif
                    }
                    }
                    __syncwarp();
                    if (mlane == 0) {
                        // this warp's reads of the row are complete (their values fed the FMAs above)
                        ws_mbar_arrive(&sm.bempty[r]);
                        if (lev > 1) ws_mbar_arrive(&sm.rempty[r]);   // after the last level the slot is released below
                        // refill the key slot released one row earlier, once every MAC warp is done with it
                        if (mwarp == (q & (WS_MAC_WARPS - 1)) && q >= 1 && q - 1 + RING < nrows) {
                            const int ps = (r + K) % RING;                              // slot of row q - 1
                            const unsigned pp = (r == 0) ? (parity ^ 1) : parity;       // its level
                            ws_mbar_wait(&sm.bempty[ps], pp);
                            produce(q - 1 + RING);
                        }
                    }
                    WT(WT_M_MAC);
                }
                level_count++;
            }
            // hand over through the slots: thread p only ever reads and writes element p of a slot, so no
            // MAC-side synchronisation is needed; the FFT lanes read after INV completes
#pragma unroll
            for (int g = 0; g < G; g++)
#pragma unroll
                for (int c = 0; c <= K; c++) sm.hs[c * G + g][p] = facc[g][c];
            __syncwarp();
            if (mlane == 0) {
                ws_mbar_arrive(&sm.inv);
                // the slots are free again once the FFT lanes have read them (they wait on INV first, and only
                // the owner group of a slot ever writes it)
#pragma unroll
                for (int r = 0; r <= K; r++) ws_mbar_arrive(&sm.rempty[r]);
            }
            WT(WT_M_HANDOVER);
        }
        if (WS_TIMING && a.dbg && blockIdx.x == 0 && p == 0)
            for (int k = 6; k < WT_COUNT; k++) a.dbg[k] = (uint64_t)tacc[k % 6];
    }
#undef WT
    __syncthreads();
#if WS_TMEM_ST
#if WS_DIAG & 256
    if (tid < 32) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(sm.tmem_base) : "memory");
#else
    if (tid < 32) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 64;" ::"r"(sm.tmem_base) : "memory");
#endif
#endif
    // sample extract of coefficient 0 (SURVEY §9.4(3))
    for (int g = 0; g < G; g++) {
        if (ct0 + g >= a.count) continue;
        uint64_t *out = a.out + (size_t)(ct0 + g) * (K * POLY_N + 1);
        for (int idx = tid; idx < K * POLY_N; idx += WS_THREADS) {
            const int r = idx / POLY_N, j = idx % POLY_N;
            out[idx] = (j == 0) ? sm.acc[g][r][0] : (uint64_t)0 - sm.acc[g][r][POLY_N - j];
        }
        if (tid == 0) out[K * POLY_N] = sm.acc[g][K][0] + a.post_add;
    }
}

}  // namespace PBS_WS_NS
using namespace PBS_WS_NS;

#define LAUNCH_WS(k, g, bl, lv)                                                                         \
    if (K == k && G == g && base_log == bl && levels == lv) {                                           \
        const size_t smem = sizeof(WsSmem<k, g>);                                                       \
        cudaError_t e = cudaFuncSetAttribute(pbs_ws_kernel<k, g, bl, lv>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); \
        if (e != cudaSuccess) return e;                                                                 \
        pbs_ws_kernel<k, g, bl, lv><<<(a.count + g - 1) / g, WS_THREADS, smem, s>>>(a);                 \
        return cudaGetLastError();                                                                      \
    }
cudaError_t PBS_WS_LAUNCH_NAME(int K, int G, int base_log, int levels, const PbsArgs &a, cudaStream_t s) {
    LAUNCH_WS(4, 1, 8, 5) LAUNCH_WS(4, 2, 8, 5) LAUNCH_WS(4, 3, 8, 5)
    LAUNCH_WS(1, 1, 8, 5) LAUNCH_WS(1, 4, 8, 5) LAUNCH_WS(1, 8, 8, 5)
    return cudaErrorInvalidValue;
}
