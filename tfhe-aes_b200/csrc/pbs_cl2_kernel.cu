// pbs_cl2_kernel.cu — one PBS (blind rotation + sample extract) per thread-block CLUSTER of two CTAs, sm_100a.
//
// The batched kernel (pbs_ws_kernel.cu) keeps G ciphertexts in one CTA for all n CMux steps; a wave of at most 148 single-
// ciphertext CTAs takes 7.5 ms whatever its size, because one CTA transforms the five decomposition levels of a polynomial one
// after the other and multiplies 25 key rows through one shared-memory pipe.  Key expansion (50 dependent stages of 32
// bootstraps, server.rs:107-167), the carry chain of add_scalar on few blocks (server.rs:172-275) and a single CTR block
// (BASELINE config 1) are made of such waves.  Here the K+1 = 5 polynomials of ONE ciphertext are split over the two CTAs of a
// cluster (CTA 0: polynomials 0-2, CTA 1: polynomials 3-4):
//   * every (level, polynomial) pair has its own 16-lane FFT group, so the five levels are transformed in parallel (each group
//     re-derives the rotated difference and keeps only its own digit: no digit state, no hand-over between groups);
//   * each CTA multiplies only the key rows of its own polynomials (15 / 10 of the 25 rows) into partial Fourier accumulators of
//     all K+1 output columns; with one ciphertext every key value is used once per CTA, so the rows are not staged in shared
//     memory: each MAC thread reads its five values of a row straight from L2, CL_PF = 5 rows ahead in registers;
//   * the partial sums of the columns the other CTA owns go to its shared memory with st.async (8 / 12 KB per step, byte-counted on
//     the receiver's mbarrier: no release fence, no arrival, the sender does not wait for the round trip), and the owner adds the
//     two halves, inverse-transforms and updates its polynomials.
// Arithmetic, decomposition (tie rule included) and FFT are those of pbs_ws_kernel (cmux_core.cuh / fft_core.cuh); only the order
// in which the 25 products are summed differs (per CTA, then across), i.e. the last bits of the floating-point sums.
#include <cuda.h>
#include "ws_common.cuh"

namespace {

constexpr int CL_K = 4;
constexpr int CL_LEVELS = 5;
constexpr int CL_MAXP = 3;                      // polynomials of CTA 0 (CTA 1 has 2)
constexpr int CL_ROWS = CL_MAXP * CL_LEVELS;    // 15 (level, polynomial) pairs / key rows per step in CTA 0
#ifndef CL_PF_ROWS
#define CL_PF_ROWS 5
#endif
constexpr int CL_PF = CL_PF_ROWS;               // key rows in flight per MAC thread (registers; setmaxnreg 112 / 144 above 4).  Measured per wave of 32: 4 rows 5.01 ms, 5 rows 4.73 ms, 6 rows 4.96 ms
constexpr int CL_THREADS = 512;                 // warps 0-7: FFT groups, warps 8-15: MAC role (point p = tid - 256)
constexpr int CL_MAC_WARPS = (CL_THREADS - 256) / 32;

struct ClSmem {
    uint64_t acc[CL_MAXP][POLY_N];              // own polynomials of the accumulator (standard domain)
    cd hs[CL_ROWS][XB_ELEMS];                   // slot of group g = level_slot * np + local polynomial: exchange, spectrum, and (slots 0..np-1) Fourier sums
    cd rx[2][CL_MAXP][POLY_M];                  // partial sums of own columns from the peer CTA, double-buffered by step parity
    cd tw[256];
    uint64_t allspec;                           // every spectrum of the step is in its slot (FFT groups -> MAC role)
    uint64_t rxfull;                            // the peer's partial sums of the step have landed in rx (byte count of its st.async stores)
    uint64_t inv;                               // Fourier sums of the own columns in slots 0..np-1 (MAC role -> owner groups)
    uint64_t accready[CL_MAXP];                 // polynomial updated (owner group -> the 5 groups of that polynomial)
};

__device__ __forceinline__ unsigned cluster_ctarank() { unsigned r; asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r)); return r; }
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ unsigned map_to_peer(const void *local_addr, unsigned peer) {
    unsigned la = ws_smem_u32(local_addr), ra;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(ra) : "r"(la), "r"(peer));
    return ra;
}
// asynchronous remote store: the 16 bytes are counted on the receiver's mbarrier when they land (no release fence, the sender
// does not wait for the round trip)
__device__ __forceinline__ void st_async_cd(unsigned remote_addr, cd v, unsigned remote_bar) {
    asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.v2.f64 [%0], {%1, %2}, [%3];" ::"r"(remote_addr), "d"(v.x), "d"(v.y),
                 "r"(remote_bar)
                 : "memory");
}
// arrive on the peer's barrier; release at cluster scope orders this thread's (and, after __syncwarp, its warp's) remote stores before it
__device__ __forceinline__ void mbar_arrive_remote(unsigned remote_bar) {
    asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(remote_bar) : "memory");
}
__device__ __forceinline__ void mbar_wait_cluster(uint64_t *bar, unsigned parity) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "WAITC_LOOP:\n\t"
        "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra.uni WAITC_DONE;\n\t"
        "bra.uni WAITC_LOOP;\n\t"
        "WAITC_DONE:\n\t}" ::"r"(ws_smem_u32(bar)), "r"(parity) : "memory");
}

// digit of level `lev` (5 = least significant) of the rotated difference, as a double (decomposition (2^8, 5) of cmux_core.cuh)
__device__ __forceinline__ double digit_of_level(uint64_t x, int lev) {
    const uint64_t y = x + DECOMP85_ADD;
    const uint32_t byte = (uint32_t)(y >> (24 + 8 * (5 - lev))) & 0xFFu;
    return __hiloint2double(0x43300000, (int)byte) - 4503599627370624.0;
}

// NP = own polynomials of this CTA (3 for rank 0, 2 for rank 1)
template <int NP>
__device__ __forceinline__ void cl2_body(const PbsArgs &a, ClSmem &sm, const unsigned rank) {
    const int tid = threadIdx.x;
    const unsigned peer = rank ^ 1u;
    constexpr int PEER_NP = 5 - NP;
    const int pbase = rank == 0 ? 0 : 3, peer_pbase = rank == 0 ? 3 : 0;
    constexpr int NROWS = NP * CL_LEVELS;
    const int ct = blockIdx.x >> 1;
    const int n = a.lwe_dim;
    constexpr int ROW_ELEMS = (CL_K + 1) * POLY_M;

    if (tid < 256) {
        // ================================ FFT groups ========================================================================
        if (CL_PF > 4) asm volatile("setmaxnreg.dec.sync.aligned.u32 112;");
        const int gid = tid >> 4, lane = tid & 15;
        const bool active = gid < NROWS;
        const int ls = active ? gid / NP : 0, lp = active ? gid % NP : 0;
        const int lev = CL_LEVELS - ls;                                  // decomposition level of this group (5 first)
        const bool owner = active && ls == 0;                            // also inverse-transforms column / polynomial lp
        const int gid_a = (tid >> 5) * 2;
        const bool warp_active = gid_a < NROWS, warp_owner = gid_a < NP;        // owners are groups 0..NP-1
        cd *slot = sm.hs[active ? gid : 0];
        uint64_t *poly = sm.acc[lp];
        cd v[16];
        int rot = ws_mod_switch_2n(a, ct, 0);
        if (warp_active) {
#pragma unroll 1
            for (int i = 0; i < n; i++) {
                const uint64_t raw_next = a.lwe_in[(size_t)ct * (n + 1) + min(i + 1, n - 1)];
                if (i > 0) ws_mbar_wait_lane(&sm.accready[lp], (unsigned)(i - 1) & 1);   // lanes of one warp may belong to two polynomials
                __syncwarp();
                // rotated difference acc * X^rot - acc, digit of this group's level only (load_decompose_rot of cmux_core.cuh)
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
                    v[n1] = cmk(digit_of_level(a0, lev), digit_of_level(a1, lev));
                }
                fft256_fwd_pass1_compute(v, lane, sm.tw);
                if (active) fft256_fwd_pass1_store(v, lane, slot);
                __syncwarp();
                fft256_fwd_pass2(v, lane, slot);
                __syncwarp();
                if (active) {
#pragma unroll
                    for (int k2 = 0; k2 < 16; k2++) slot[lane + 16 * k2] = v[rev4(k2)];
                }
                __syncwarp();
                if (active && lane == 0) ws_mbar_arrive(&sm.allspec);
                rot = (int)((raw_next * a.in_scale + (1ull << 53)) >> 54) & (2 * POLY_N - 1);
                if (warp_owner) {
                    ws_mbar_wait(&sm.inv, (unsigned)i & 1);
#pragma unroll
                    for (int k2 = 0; k2 < 16; k2++) v[k2] = slot[lane + 16 * k2];
                    fft256_inv_pass1_compute(v);
                    __syncwarp();
                    if (owner) fft256_inv_pass1_store_b<8>(v, lane, sm.tw, slot);
                    __syncwarp();
                    fft256_inv_pass2(v, lane, slot);
                    if (owner) {
#pragma unroll
                        for (int n1 = 0; n1 < 16; n1++) {
                            const int j = 16 * n1 + lane;
                            poly[j] += f64_to_torus(v[n1].x);
                            poly[j + POLY_M] += f64_to_torus(v[n1].y);
                        }
                    }
                    __syncwarp();
                    if (owner && lane == 0) ws_mbar_arrive(&sm.accready[lp]);
                }
            }
        }
    } else {
        // ================================ MAC role ==========================================================================
        // One ciphertext per cluster: every key value is used exactly once per CTA, so the key rows are not staged in shared
        // memory; thread p reads its K+1 values of a row straight from L2 (all clusters walk the key together), CL_PF rows ahead.
        if (CL_PF > 4) asm volatile("setmaxnreg.inc.sync.aligned.u32 144;");
        const int p = tid - 256, mlane = p & 31;
        const unsigned remote_rx = map_to_peer(&sm.rx[0][0][p], peer), remote_bar = map_to_peer(&sm.rxfull, peer);
        // row g = level_slot * NP + local polynomial of step i in the key stream [i][level slot][row][col][p]
        auto row_ptr = [&](int i, int g) {
            return a.bsk + ((size_t)(i * CL_LEVELS + g / NP) * (CL_K + 1) + (pbase + g % NP)) * ROW_ELEMS + p;
        };
        cd wbuf[CL_PF][CL_K + 1];
        auto fetch = [&](int slot, const cd *src) {
#pragma unroll
            for (int c = 0; c <= CL_K; c++) {
                const double2 t = __ldg(reinterpret_cast<const double2 *>(src + c * POLY_M));
                wbuf[slot][c] = t;
            }
        };
#pragma unroll
        for (int g = 0; g < CL_PF; g++) fetch(g, row_ptr(0, g));
#pragma unroll 1
        for (int i = 0; i < n; i++) {
            cd facc[CL_K + 1];
#pragma unroll
            for (int c = 0; c <= CL_K; c++) facc[c] = cmk(0.0, 0.0);
            ws_mbar_wait(&sm.allspec, (unsigned)i & 1);
            const int inext = min(i + 1, n - 1);          // the last step prefetches rows it never uses
#pragma unroll
            for (int g = 0; g < NROWS; g++) {
                const cd x = sm.hs[g][p];
#pragma unroll
                for (int c = 0; c <= CL_K; c++) cmac(facc[c], x, wbuf[g % CL_PF][c]);
                // refill the register slot with the row CL_PF ahead (the first rows of the next step when this one runs out)
                const int gn = g + CL_PF;
                fetch(g % CL_PF, gn < NROWS ? row_ptr(i, gn) : row_ptr(inext, gn - NROWS));
            }
            if (NROWS % CL_PF != 0) {
                // row r of the next step sits in register slot (NROWS + r) % CL_PF: rotate so that it is in slot r again (register moves)
                cd t[CL_PF][CL_K + 1];
#pragma unroll
                for (int r = 0; r < CL_PF; r++)
#pragma unroll
                    for (int c = 0; c <= CL_K; c++) t[r][c] = wbuf[(NROWS + r) % CL_PF][c];
#pragma unroll
                for (int r = 0; r < CL_PF; r++)
#pragma unroll
                    for (int c = 0; c <= CL_K; c++) wbuf[r][c] = t[r][c];
            }
            // partial sums of the peer's columns -> its shared memory; the bytes complete its rxfull barrier as they land
#pragma unroll
            for (int c = 0; c < PEER_NP; c++)
                st_async_cd(remote_rx + (unsigned)(((i & 1) * CL_MAXP + c) * POLY_M * sizeof(cd)), facc[peer_pbase + c], remote_bar);
            mbar_wait_cluster(&sm.rxfull, (unsigned)i & 1);
            // the next phase expects the peer's NP columns again (posted thousands of cycles before the peer can send them)
            if (p == 0) ws_mbar_arrive_expect_tx(&sm.rxfull, (unsigned)(NP * POLY_M * sizeof(cd)));
#pragma unroll
            for (int c = 0; c < NP; c++) {
                const cd r = sm.rx[i & 1][c][p];
                sm.hs[c][p] = cmk(facc[pbase + c].x + r.x, facc[pbase + c].y + r.y);
            }
            __syncwarp();
            if (mlane == 0) ws_mbar_arrive(&sm.inv);
        }
    }
}

__global__ void __launch_bounds__(CL_THREADS, 1) pbs_cl2_kernel(PbsArgs a) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    ClSmem &sm = *reinterpret_cast<ClSmem *>(smem_raw);
    const int tid = threadIdx.x;
    const unsigned rank = cluster_ctarank();
    const int np = rank == 0 ? 3 : 2, pbase = rank == 0 ? 0 : 3;
    const int ct = blockIdx.x >> 1;
    const int n = a.lwe_dim;
    // ---- prologue ------------------------------------------------------------------------------------------------------
    for (int i = tid; i < 256; i += CL_THREADS) sm.tw[i] = a.tw[i];
    if (tid == 0) {
        ws_mbar_init(&sm.allspec, np * CL_LEVELS);
        ws_mbar_init(&sm.rxfull, 1);
        ws_mbar_arrive_expect_tx(&sm.rxfull, (unsigned)(np * POLY_M * sizeof(cd)));   // step 0: np columns of 4 KB from the peer
        ws_mbar_init(&sm.inv, CL_MAC_WARPS);
        for (int lp = 0; lp < CL_MAXP; lp++) ws_mbar_init(&sm.accready[lp], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    {
        const int rot = (2 * POLY_N - ws_mod_switch_2n(a, ct, n)) & (2 * POLY_N - 1);
        for (int idx = tid; idx < np * POLY_N; idx += CL_THREADS) {
            const int lp = idx / POLY_N, j = idx % POLY_N;
            sm.acc[lp][j] = (pbase + lp == CL_K) ? rotated_coef(a.lut, j, rot) : 0;
        }
    }
    __syncthreads();
    cluster_sync_all();                               // both CTAs are resident and their barriers initialised before any remote access
    if (rank == 0) cl2_body<3>(a, sm, rank);
    else cl2_body<2>(a, sm, rank);
    __syncthreads();
    cluster_sync_all();                               // no CTA leaves while its peer may still write into its shared memory
    // sample extract of coefficient 0 (SURVEY §9.4(3)): mask segment r from polynomial r, body from polynomial K
    uint64_t *out = a.out + (size_t)ct * (CL_K * POLY_N + 1);
    for (int idx = tid; idx < np * POLY_N; idx += CL_THREADS) {
        const int lp = idx / POLY_N, j = idx % POLY_N, r = pbase + lp;
        if (r < CL_K) out[r * POLY_N + j] = (j == 0) ? sm.acc[lp][0] : (uint64_t)0 - sm.acc[lp][POLY_N - j];
        else if (j == 0) out[CL_K * POLY_N] = sm.acc[lp][0] + a.post_add;
    }
}

}  // namespace

// one cluster of two CTAs per ciphertext: worthwhile for count <= 74 (one wave)
cudaError_t launch_pbs_cl2(const PbsArgs &a, cudaStream_t s) {
    const size_t smem = sizeof(ClSmem);
    cudaError_t e = cudaFuncSetAttribute(pbs_cl2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(2 * a.count);
    cfg.blockDim = dim3(CL_THREADS);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = s;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 2; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, pbs_cl2_kernel, a);
}
