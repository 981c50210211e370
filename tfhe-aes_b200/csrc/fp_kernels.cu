// fp_kernels.cu — the FP64 kernels of the WoPBS chain other than the PBS (sm_100a).  The PBS, K3 of SURVEY.md §2.2,
// has kernels of its own: pbs_ws_kernel.cu, pbs_ws2_kernel.cu and pbs_cl2_kernel.cu.
//   vp_kernel             blind-rotation half of vertical_packing + sample extract — K6 (many_wopbs.rs:277)
//   cmux_tree_kernel      one layer of the vertical-packing CMux tree (LUT larger than N) — K6 general form
//   fourier_convert_kernel standard GGSW -> Fourier layout — K5 (fill_with_forward_fourier, many_wopbs.rs:263)
//                         and the one-time bootstrap-key conversion at key load.
// All of them run the CTA-level phases of cmux_core.cuh.
#include "cmux_core.cuh"
#include "kernels.h"

template <int K, int G>
__device__ __forceinline__ CmuxSmem<K, G> &smem_view(unsigned char *raw) {
    return *reinterpret_cast<CmuxSmem<K, G> *>(raw);
}

template <int K, int G>
__device__ __forceinline__ void load_twiddles(CmuxSmem<K, G> &sm, const cd *tw, int tid) {
    for (int i = tid; i < 256; i += CMUX_THREADS) sm.tw[i] = tw[i];
}

// One full CMux step on the resident accumulators (all barriers included).
template <int K, int G, int BASE_LOG, int LEVELS, int MODE>
__device__ __forceinline__ void cmux_step(int tid, CmuxSmem<K, G> &sm, CmuxRegs<K, G> &rg, const cd *__restrict__ ggsw,
                                          const uint64_t *const *ext) {
    phase_load_decompose<K, G, BASE_LOG, LEVELS, MODE>(tid, sm, rg, ext);
#pragma unroll 1
    for (int lev = LEVELS; lev >= 1; lev--) {
        if (lev != LEVELS) phase_next_digits<K, G, BASE_LOG, LEVELS>(tid, rg, lev);
        phase_fwd1<K, G>(tid, sm, rg);
        __syncwarp();
        phase_fwd2<K, G>(tid, sm, rg);
        __syncwarp();
        phase_fwd3<K, G>(tid, sm, rg);
        __syncthreads();
        phase_mac<K, G>(tid, sm, rg, ggsw + (size_t)(LEVELS - lev) * (K + 1) * POLY_M * (K + 1));
        __syncthreads();
    }
    phase_inv0<K, G>(tid, sm, rg);
    __syncthreads();
    phase_inv1<K, G>(tid, sm, rg);
    __syncwarp();
    phase_inv2<K, G>(tid, sm, rg);
    __syncwarp();
    phase_inv3<K, G>(tid, sm, rg);
    __syncthreads();
}

// sample extract of coefficient 0 (SURVEY §9.4(3)) from the resident accumulator g
template <int K, int G>
__device__ __forceinline__ void sample_extract(int tid, const CmuxSmem<K, G> &sm, int g, uint64_t *out, uint64_t post_add) {
    for (int idx = tid; idx < K * POLY_N; idx += CMUX_THREADS) {
        const int r = idx / POLY_N, j = idx % POLY_N;
        out[idx] = (j == 0) ? sm.acc[g][r][0] : (uint64_t)0 - sm.acc[g][r][POLY_N - j];
    }
    if (tid == 0) out[K * POLY_N] = sm.acc[g][K][0] + post_add;
}

// ------------------------------------------------------------------------------------------------
// Vertical packing, blind-rotation half: for GGSW bit t = 0 (LSB) .. nrot-1:
//   acc += GGSW_t (x) (acc * X^-(2^t) - acc);  then sample extract.
// blockIdx.y = job (one encrypted byte = one GGSW list), blockIdx.x = chunk of G outputs.
// ------------------------------------------------------------------------------------------------
template <int K, int G, int BASE_LOG, int LEVELS>
__global__ void __launch_bounds__(CMUX_THREADS, 1) vp_kernel(VpArgs a) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    CmuxSmem<K, G> &sm = smem_view<K, G>(smem_raw);
    CmuxRegs<K, G> rg;
    const int tid = threadIdx.x;
    const int job = blockIdx.y, o0 = blockIdx.x * G;
    load_twiddles<K, G>(sm, a.tw, tid);
    for (int g = 0; g < G; g++) {
        const int o = min(o0 + g, a.nouts - 1);
        for (int idx = tid; idx < (K + 1) * POLY_N; idx += CMUX_THREADS) {
            const int r = idx / POLY_N, j = idx % POLY_N;
            uint64_t v;
            if (a.glwe_init) v = a.glwe_init[((size_t)job * a.nouts + o) * (K + 1) * POLY_N + idx];
            else v = (r == K) ? a.lut[(size_t)job * a.lut_job_stride + (size_t)o * a.lut_out_stride + j] : 0;
            sm.acc[g][r][j] = v;
        }
    }
    __syncthreads();
    const size_t ggsw_size = (size_t)LEVELS * (K + 1) * POLY_M * (K + 1);
    const cd *ggsw_job = a.ggsw_f + (size_t)job * (a.nbits - a.nshared) * ggsw_size;
    const cd *ggsw_shared = a.shared_set ? a.ggsw_shared + (size_t)a.shared_set[job] * a.shared_set_stride : a.ggsw_shared;
#pragma unroll 1
    for (int t = 0; t < a.nrot; t++) {
        const int deg = (t < 31 ? (1 << t) : 0) & (2 * POLY_N - 1);
        if (tid < G) sm.rot[tid] = (2 * POLY_N - deg) & (2 * POLY_N - 1);
        __syncthreads();
        const cd *ggsw_t = t < a.nshared ? ggsw_shared + (size_t)t * ggsw_size : ggsw_job + (size_t)(t - a.nshared) * ggsw_size;
        cmux_step<K, G, BASE_LOG, LEVELS, DIFF_ROTATE>(tid, sm, rg, ggsw_t, nullptr);
    }
    for (int g = 0; g < G; g++)
        if (o0 + g < a.nouts)
            sample_extract<K, G>(tid, sm, g, a.out + ((size_t)job * a.nouts + o0 + g) * (K * POLY_N + 1), 0);
}

// ------------------------------------------------------------------------------------------------
// One layer of the CMux tree: out[q] = c0[q] + GGSW (x) (c1[q] - c0[q]),  c0 = in[2q], c1 = in[2q+1].
// blockIdx.y = job, blockIdx.x = chunk of G pairs (pairs enumerate (output, pair-in-output)).
// ------------------------------------------------------------------------------------------------
template <int K, int G, int BASE_LOG, int LEVELS>
__global__ void __launch_bounds__(CMUX_THREADS, 1) cmux_tree_kernel(TreeArgs a) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    CmuxSmem<K, G> &sm = smem_view<K, G>(smem_raw);
    __shared__ const uint64_t *ext[G];
    CmuxRegs<K, G> rg;
    const int tid = threadIdx.x;
    const int job = blockIdx.y, q0 = blockIdx.x * G;
    const size_t gsz = (size_t)(K + 1) * POLY_N;
    load_twiddles<K, G>(sm, a.tw, tid);
    for (int g = 0; g < G; g++) {
        const int q = min(q0 + g, a.npairs - 1);
        const uint64_t *c0 = a.in + ((size_t)job * a.npairs * 2 + 2 * q) * gsz;
        if (tid == 0) ext[g] = c0 + gsz;
        for (int idx = tid; idx < (int)gsz; idx += CMUX_THREADS) sm.acc[g][idx / POLY_N][idx % POLY_N] = c0[idx];
    }
    __syncthreads();
    const size_t ggsw_size = (size_t)LEVELS * (K + 1) * POLY_M * (K + 1);
    const cd *ggsw = a.ggsw_f + ((size_t)job * a.nbits + a.bit_index) * ggsw_size;
    cmux_step<K, G, BASE_LOG, LEVELS, DIFF_EXTERNAL>(tid, sm, rg, ggsw, ext);
    for (int g = 0; g < G; g++)
        if (q0 + g < a.npairs) {
            uint64_t *o = a.out + ((size_t)job * a.npairs + q0 + g) * gsz;
            for (int idx = tid; idx < (int)gsz; idx += CMUX_THREADS) o[idx] = sm.acc[g][idx / POLY_N][idx % POLY_N];
        }
}

// ------------------------------------------------------------------------------------------------
// standard-domain GGSW list [g][level][row][col][N] (u64) -> Fourier layout [g][level][row][col][p]
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(CMUX_THREADS, 2) fourier_convert_kernel(ConvertArgs a) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    cd *xb_all = reinterpret_cast<cd *>(smem_raw);
    cd *tw = xb_all + CMUX_GROUPS * XB_ELEMS;
    const int tid = threadIdx.x, gid = tid >> 4, lane = tid & 15;
    for (int i = tid; i < 256; i += CMUX_THREADS) tw[i] = a.tw[i];
    __syncthreads();
    const long q = (long)blockIdx.x * CMUX_GROUPS + gid;
    const bool active = q < a.npoly;
    cd *xb = xb_all + gid * XB_ELEMS;
    cd v[16];
    if (active) {
        load_torus_poly(v, lane, a.in + (size_t)q * POLY_N);
        fft256_fwd_pass1(v, lane, tw, xb);
    }
    __syncwarp();
    if (active) {
        fft256_fwd_pass2(v, lane, xb);
        // [g][level][row][col] -> [g][level slot = levels-1-level][row][col][p]
        const long per_level = (long)(a.glwe_dim + 1) * (a.glwe_dim + 1);
        const long rc = q % per_level, gl = q / per_level;
        const long lev = gl % a.levels, g = gl / a.levels;
        cd *dst = a.out + (size_t)((g * a.levels + (a.levels - 1 - lev)) * per_level + rc) * POLY_M;
#pragma unroll
        for (int k2 = 0; k2 < 16; k2++) dst[lane + 16 * k2] = v[rev4(k2)];
    }
}

// ------------------------------------------------------------------------------------------------
// host launchers
// ------------------------------------------------------------------------------------------------
template <typename F>
static cudaError_t set_smem(F f, size_t bytes) {
    return cudaFuncSetAttribute(f, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
}

#define LAUNCH_VP(k, g, bl, lv)                                                      \
    if (K == k && G == g && base_log == bl && levels == lv) {                        \
        size_t smem = sizeof(CmuxSmem<k, g>);                                        \
        cudaError_t e = set_smem(vp_kernel<k, g, bl, lv>, smem);                     \
        if (e != cudaSuccess) return e;                                              \
        dim3 grid((a.nouts + g - 1) / g, a.njobs);                                   \
        vp_kernel<k, g, bl, lv><<<grid, CMUX_THREADS, smem, s>>>(a);                 \
        return cudaGetLastError();                                                   \
    }
cudaError_t launch_vp(int K, int G, int base_log, int levels, const VpArgs &a, cudaStream_t s) {
    LAUNCH_VP(4, 1, 15, 1) LAUNCH_VP(4, 2, 15, 1) LAUNCH_VP(4, 3, 15, 1)
    LAUNCH_VP(1, 1, 15, 1) LAUNCH_VP(1, 4, 15, 1) LAUNCH_VP(1, 8, 15, 1)
    return cudaErrorInvalidValue;
}
#define LAUNCH_TREE(k, g, bl, lv)                                                    \
    if (K == k && G == g && base_log == bl && levels == lv) {                        \
        size_t smem = sizeof(CmuxSmem<k, g>);                                        \
        cudaError_t e = set_smem(cmux_tree_kernel<k, g, bl, lv>, smem);              \
        if (e != cudaSuccess) return e;                                              \
        dim3 grid((a.npairs + g - 1) / g, a.njobs);                                  \
        cmux_tree_kernel<k, g, bl, lv><<<grid, CMUX_THREADS, smem, s>>>(a);          \
        return cudaGetLastError();                                                   \
    }
cudaError_t launch_cmux_tree(int K, int G, int base_log, int levels, const TreeArgs &a, cudaStream_t s) {
    LAUNCH_TREE(4, 3, 15, 1) LAUNCH_TREE(4, 1, 15, 1) LAUNCH_TREE(1, 1, 15, 1) LAUNCH_TREE(1, 8, 15, 1)
    return cudaErrorInvalidValue;
}
cudaError_t launch_fourier_convert(const ConvertArgs &a, cudaStream_t s) {
    size_t smem = (size_t)(CMUX_GROUPS * XB_ELEMS + 256) * sizeof(cd);
    cudaError_t e = set_smem(fourier_convert_kernel, smem);
    if (e != cudaSuccess) return e;
    long blocks = (a.npoly + CMUX_GROUPS - 1) / CMUX_GROUPS;
    fourier_convert_kernel<<<(unsigned)blocks, CMUX_THREADS, smem, s>>>(a);
    return cudaGetLastError();
}
