// kernels.h — argument blocks and host launchers of the sm_100a kernels (internal to the library).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

struct PbsArgs {
    const uint64_t *lwe_in;   // [count][lwe_dim+1]
    const double2 *bsk;       // Fourier BSK [lwe_dim][level][row][col][p]
    const double2 *tw;        // 256 mid twiddles (make_twiddle_table)
    const uint64_t *lut;      // [N] body of the trivial accumulator
    uint64_t *out;            // [count][k*N+1]
    uint64_t in_scale;        // cleartext multiplier applied to the input before the modulus switch
    uint64_t pre_add_body;    // added to the input body before the modulus switch (q/4 centring)
    uint64_t post_add;        // added to the output body
    int lwe_dim;
    int count;
    uint64_t *dbg;            // per-activity cycle counters of CTA 0 in the WS_TIMING / WS2_TIMING builds of scratch/pbs_lab (nullptr otherwise)
};
struct VpArgs {
    const double2 *ggsw_f;    // [njobs][nbits][level][row][col][p], bit 0 = LSB
    const double2 *tw;
    const uint64_t *lut;      // [.. job*lut_job_stride + out*lut_out_stride + j ..] LUT polynomial per output (if glwe_init == 0)
    const uint64_t *glwe_init;// or [njobs][nouts][(k+1)N] start accumulators (root of the CMux tree)
    uint64_t *out;            // [njobs][nouts][k*N+1]
    size_t lut_job_stride;
    size_t lut_out_stride;
    int nbits;                // selector bits (GGSWs) per job, of which the first nshared come from ggsw_shared
    int nrot;                 // GGSWs consumed by the blind rotation (bits 0..nrot-1)
    const double2 *ggsw_shared;  // [nshared][level][row][col][p]: GGSWs common to all jobs (bits 0..nshared-1), or nullptr
    int nshared;              // ggsw_f then holds nbits - nshared GGSWs per job
    const int32_t *shared_set;   // [njobs] or nullptr: job j reads its shared GGSWs at ggsw_shared + shared_set[j] * shared_set_stride
    size_t shared_set_stride;    // in double2
    int nouts;
    int njobs;
};
struct TreeArgs {
    const double2 *ggsw_f;    // [njobs][nbits][...]
    const double2 *tw;
    const uint64_t *in;       // [njobs][2*npairs][(k+1)N]
    uint64_t *out;            // [njobs][npairs][(k+1)N]
    int nbits;
    int bit_index;            // which GGSW of the job drives this layer
    int npairs;
    int njobs;
};
struct ConvertArgs {
    const uint64_t *in;       // [npoly][N], polys ordered [g][level][row][col]
    double2 *out;             // [g][level][row][col][p]
    const double2 *tw;
    long npoly;
    int glwe_dim;
    int levels;               // levels per GGSW (output slot order is reversed: slot 0 = last level)
};

struct ImmaGemvArgs {
    const int8_t *dl;         // [count][rows_pad] low digit limbs
    const int8_t *dh;         // [count][rows_pad] high digit limbs (nullptr when digits fit one limb)
    const uint8_t *kp;        // prepared key [nkeys][ntiles][kchunks][2048]
    uint64_t *out;            // [count][out_stride], pre-initialised; the product is subtracted
    int out_stride;
    int rows_pad;             // kchunks * 32
    int kchunks;
    int ntiles;               // ceil(ncols / 8)
    int ncols;
    int nkeys;
    int count;
};
cudaError_t launch_imma_prepare_key(const uint64_t *key, size_t key_stride, int nkeys, int rows, int ncols, int row_stride, uint8_t *kp,
                                    cudaStream_t s);
cudaError_t launch_imma_decompose(const uint64_t *in, int in_stride, int nelem, int count, int base_log, int levels, int rows_pad,
                                  int8_t *dl, int8_t *dh, cudaStream_t s);
cudaError_t launch_imma_gemv(const ImmaGemvArgs &a, int digit_limbs, cudaStream_t s);

// tcgen05 PFKS (tc5_kernels.cu): key in its standard layout [nkeys][rows][ncols] u64
bool tc5_pfks_supported(int ncols, int rows_pad);
cudaError_t launch_tc5_pfks(const int8_t *dl, const int8_t *dh, int rows_pad, const uint64_t *key, int nkeys, int rows, int ncols, int count,
                            uint64_t *out, int out_stride, cudaStream_t s);
bool tc5_ks_supported(int ncols, int key_pitch_cols, int rows_pad);
cudaError_t launch_tc5_keyswitch(const int8_t *dl, int rows_pad, const uint64_t *key, int rows, int ncols, int key_pitch_cols, int count,
                                 const uint64_t *in, int in_stride, int body_index, uint64_t *out, int out_stride, cudaStream_t s);

cudaError_t launch_pbs_ws(int K, int G, int base_log, int levels, const PbsArgs &a, cudaStream_t s);
cudaError_t launch_pbs_ws2(int K, int G, int base_log, int levels, const PbsArgs &a, cudaStream_t s);   // K = 4, G = 3, (2^8, 5): two sets of G per CTA (large batches)
cudaError_t launch_pbs_cl2(const PbsArgs &a, cudaStream_t s);   // K = 4, (2^8, 5): one ciphertext per cluster of two CTAs (small batches)
cudaError_t launch_vp(int K, int G, int base_log, int levels, const VpArgs &a, cudaStream_t s);
cudaError_t launch_cmux_tree(int K, int G, int base_log, int levels, const TreeArgs &a, cudaStream_t s);
cudaError_t launch_fourier_convert(const ConvertArgs &a, cudaStream_t s);

// integer kernels (int_kernels.cu)
// out[b][c] = offset*colsum[c] (+ body of in for the keyswitch when body_src != nullptr)
cudaError_t launch_gemv_init(uint64_t *out, int out_stride, int total_cols, int count, const uint64_t *colsum,
                             uint64_t offset, const uint64_t *body_src, int body_src_stride, int body_src_index,
                             int body_dst_col, cudaStream_t s);
struct SumEntry {
    const uint64_t *src[5];
    uint64_t *dst;
    int nsrc;
    int _pad;
};
cudaError_t launch_lwe_sum(const SumEntry *entries, int nentries, int unit_words, cudaStream_t s);
// gather-sum of a SumEntry plus a clear byte XORed into the encrypted destination byte (1-bit blocks): bit j of
// (clear ^ *clear_src) adds bit << 63 to the body of LWE j
struct SumXorEntry {
    const uint64_t *src[5];
    uint64_t *dst;
    const uint8_t *clear_src;   // device byte, or nullptr
    int nsrc;
    uint32_t clear;
};
cudaError_t launch_lwe_sum_xor(const SumXorEntry *entries, int nentries, int lw, cudaStream_t s);
cudaError_t launch_scale_lwe(const uint64_t *in, uint64_t *out, long nwords, uint64_t mul, cudaStream_t s);
cudaError_t launch_sub_lwe(uint64_t *inout, const uint64_t *sub, long nwords, cudaStream_t s);
cudaError_t launch_add_body(uint64_t *lwe, int lwe_words, int count, uint64_t add, cudaStream_t s);
cudaError_t launch_fill_u64(uint64_t *dst, long n, uint64_t v, cudaStream_t s);
cudaError_t launch_xor_clear(uint64_t *states, const uint8_t *data, int lw, long nbits, cudaStream_t s);
// trivial GLWE leaves for the CMux tree: out[job][out][leaf][(k+1)N] from lut[job*js + out*os + leaf*N + j]
cudaError_t launch_tree_leaves(const uint64_t *lut, size_t lut_job_stride, size_t lut_out_stride, int njobs, int nouts,
                               int nleaf, int glwe_dim, uint64_t *out, cudaStream_t s);
// counter-add LUTs of Server::add_scalar (server.rs:181-248), generated on the device
cudaError_t launch_add_scalar_luts(const uint64_t *counters_lo_hi, int nblk, int byte_index, int nbits, uint64_t *luts,
                                   cudaStream_t s);
// packed[g][r][c] (g < ceil(count / 512)) = round(x / 2^48) mod 2^16 of x = sum_i X^i pfks[512 g + i][r][c] over the inputs of
// GLWE g; pfks [count][(glwe_dim + 1) * 512]: the PFKS outputs under the last circuit-bootstrap key
cudaError_t launch_glwe_pack(const uint64_t *pfks, int count, int glwe_dim, uint16_t *packed, cudaStream_t s);
// out [count][glwe_dim * 512 + 1]: LWE i = sample extraction of coefficient i % 512 of GLWE i / 512, words widened as v << 48
cudaError_t launch_glwe_unpack(const uint16_t *packed, int count, int glwe_dim, uint64_t *out, cudaStream_t s);
