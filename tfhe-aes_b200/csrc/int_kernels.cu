// int_kernels.cu — elementwise integer (u64 wrapping) kernels of the WoPBS chain (sm_100a):
//   lwe_sum            fused ShiftRows / MixColumns / AddRoundKey additions (K7; server.rs:278-282,
//                      mix_columns.rs:4-78, inv_mix_columns.rs:4-58)
//   lwe_sum_xor        the same plus a clear byte XORed in (public-IV CTR: counter bytes, data bytes)
//   gemv_init          output initialisation of the keyswitch / PFKS products (imma_kernels.cu)
//   helpers of the general extract_bits loop, CMux-tree leaves, add_scalar LUT generation.
#include "kernels.h"

__global__ void gemv_init_kernel(uint64_t *out, int out_stride, int total_cols, long total, const uint64_t *colsum, uint64_t offset,
                                 const uint64_t *body_src, int body_src_stride, int body_src_index, int body_dst_col) {
    long idx = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= total) return;
    const long b = idx / total_cols;
    const int c = (int)(idx % total_cols);
    uint64_t v = colsum ? offset * colsum[c] : 0;
    if (body_src && c == body_dst_col) v += body_src[b * body_src_stride + body_src_index];
    out[b * out_stride + c] = v;
}
cudaError_t launch_gemv_init(uint64_t *out, int out_stride, int total_cols, int count, const uint64_t *colsum, uint64_t offset,
                             const uint64_t *body_src, int body_src_stride, int body_src_index, int body_dst_col, cudaStream_t s) {
    long total = (long)count * total_cols;
    gemv_init_kernel<<<(unsigned)((total + 255) / 256), 256, 0, s>>>(out, out_stride, total_cols, total, colsum, offset, body_src,
                                                                    body_src_stride, body_src_index, body_dst_col);
    return cudaGetLastError();
}

// ---- fused linear layer: dst = sum of up to 5 encrypted bytes (wrapping u64 adds); consecutive threads read consecutive u64 words
// (a byte is 8 x 2049 words: not 16-byte aligned from one LWE to the next, so no 128-bit accesses); 87 % of the HBM copy peak
__global__ void lwe_sum_kernel(const SumEntry *__restrict__ entries, int unit_words) {
    const SumEntry e = entries[blockIdx.y];
    for (int w = blockIdx.x * blockDim.x + threadIdx.x; w < unit_words; w += gridDim.x * blockDim.x) {
        uint64_t s = e.src[0][w];
        for (int t = 1; t < e.nsrc; t++) s += e.src[t][w];
        e.dst[w] = s;
    }
}
cudaError_t launch_lwe_sum(const SumEntry *entries, int nentries, int unit_words, cudaStream_t s) {
    dim3 grid((unit_words + 1023) / 1024, nentries);
    lwe_sum_kernel<<<grid, 256, 0, s>>>(entries, unit_words);
    return cudaGetLastError();
}
// the same over one encrypted byte (8 LWEs of lw words) per entry, plus the clear byte on the 8 body words: with one message
// bit per LWE at 2^63, adding the encoded bit is the XOR (no bootstrap, no added noise)
__global__ void lwe_sum_xor_kernel(const SumXorEntry *__restrict__ entries, int lw) {
    const SumXorEntry e = entries[blockIdx.y];
    const uint32_t clear = e.clear ^ (e.clear_src ? *e.clear_src : 0u);
    const int unit_words = 8 * lw;
    for (int w = blockIdx.x * blockDim.x + threadIdx.x; w < unit_words; w += gridDim.x * blockDim.x) {
        uint64_t s = e.src[0][w];
        for (int t = 1; t < e.nsrc; t++) s += e.src[t][w];
        const uint32_t j = (uint32_t)w / (uint32_t)lw;
        if ((uint32_t)w - j * (uint32_t)lw == (uint32_t)lw - 1) s += (uint64_t)((clear >> j) & 1) << 63;
        e.dst[w] = s;
    }
}
cudaError_t launch_lwe_sum_xor(const SumXorEntry *entries, int nentries, int lw, cudaStream_t s) {
    dim3 grid((8 * lw + 1023) / 1024, nentries);
    lwe_sum_xor_kernel<<<grid, 256, 0, s>>>(entries, lw);
    return cudaGetLastError();
}

// ---- small elementwise helpers used by the general extract_bits loop --------------------------------
__global__ void scale_kernel(const uint64_t *in, uint64_t *out, long n, uint64_t mul) {
    long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = in[i] * mul;
}
cudaError_t launch_scale_lwe(const uint64_t *in, uint64_t *out, long n, uint64_t mul, cudaStream_t s) {
    scale_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(in, out, n, mul);
    return cudaGetLastError();
}
__global__ void sub_kernel(uint64_t *inout, const uint64_t *sub, long n) {
    long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) inout[i] -= sub[i];
}
cudaError_t launch_sub_lwe(uint64_t *inout, const uint64_t *sub, long n, cudaStream_t s) {
    sub_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(inout, sub, n);
    return cudaGetLastError();
}
__global__ void add_body_kernel(uint64_t *lwe, int words, int count, uint64_t add) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < count) lwe[(size_t)i * words + words - 1] += add;
}
cudaError_t launch_add_body(uint64_t *lwe, int words, int count, uint64_t add, cudaStream_t s) {
    add_body_kernel<<<(count + 255) / 256, 256, 0, s>>>(lwe, words, count, add);
    return cudaGetLastError();
}
// XOR of encrypted bits with clear bits: bit j of byte `by` of the data adds (bit << 63) to the body of LWE (by, j)
__global__ void xor_clear_kernel(uint64_t *states, const uint8_t *data, int lw, long nbits) {
    const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nbits) return;
    const uint64_t bit = (data[i >> 3] >> (i & 7)) & 1;
    states[(size_t)i * lw + lw - 1] += bit << 63;
}
cudaError_t launch_xor_clear(uint64_t *states, const uint8_t *data, int lw, long nbits, cudaStream_t s) {
    xor_clear_kernel<<<(unsigned)((nbits + 255) / 256), 256, 0, s>>>(states, data, lw, nbits);
    return cudaGetLastError();
}
__global__ void fill_kernel(uint64_t *dst, long n, uint64_t v) {
    long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) dst[i] = v;
}
cudaError_t launch_fill_u64(uint64_t *dst, long n, uint64_t v, cudaStream_t s) {
    fill_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(dst, n, v);
    return cudaGetLastError();
}
__global__ void tree_leaves_kernel(const uint64_t *lut, size_t js, size_t os, int nouts, int nleaf, int kp1, uint64_t *out) {
    // grid: x over words of one GLWE, y = leaf, z = job*nouts + out
    const int job = blockIdx.z / nouts, o = blockIdx.z % nouts, leaf = blockIdx.y;
    const int gsz = kp1 * 512;
    uint64_t *dst = out + ((size_t)blockIdx.z * nleaf + leaf) * gsz;
    for (int w = blockIdx.x * blockDim.x + threadIdx.x; w < gsz; w += gridDim.x * blockDim.x)
        dst[w] = (w >= (kp1 - 1) * 512) ? lut[job * js + o * os + (size_t)leaf * 512 + (w - (kp1 - 1) * 512)] : 0;
}
cudaError_t launch_tree_leaves(const uint64_t *lut, size_t js, size_t os, int njobs, int nouts, int nleaf, int glwe_dim,
                               uint64_t *out, cudaStream_t s) {
    dim3 grid(((glwe_dim + 1) * 512 + 255) / 256, nleaf, njobs * nouts);
    tree_leaves_kernel<<<grid, 256, 0, s>>>(lut, js, os, nouts, nleaf, glwe_dim + 1, out);
    return cudaGetLastError();
}

// ---- add_scalar LUTs (server.rs:181-196 for the low byte, :225-248 for the others) ------------------
// luts: [nblk][nbits+1 polys][512]: polys 0..7 = bits of the sum, poly 8 = carry (bit 0 of the carry LUT);
// for nbits == 8 (low byte) the layout is the same with 8-bit inputs repeated over 512 entries.
__global__ void add_scalar_luts_kernel(const uint64_t *ctr, int byte_index, int nbits, uint64_t *luts) {
    const int blk = blockIdx.x;
    const uint64_t lo = ctr[2 * blk], hi = ctr[2 * blk + 1];
    const int sh = 8 * (15 - byte_index);
    const uint32_t ib = (uint32_t)((sh >= 64 ? hi >> (sh - 64) : lo >> sh) & 0xFF);
    for (int idx = threadIdx.x; idx < 512; idx += blockDim.x) {
        const uint32_t x = (nbits == 8) ? (idx & 0xFF) : idx;
        const uint32_t sum = (x & 0xFF) + ((nbits == 9) ? ((x >> 8) & 1) : 0) + ib;
        for (int b = 0; b < 8; b++) luts[((size_t)blk * 9 + b) * 512 + idx] = (uint64_t)((sum >> b) & 1) << 63;
        luts[((size_t)blk * 9 + 8) * 512 + idx] = (uint64_t)(sum > 255 ? 1 : 0) << 63;
    }
}
cudaError_t launch_add_scalar_luts(const uint64_t *ctr, int nblk, int byte_index, int nbits, uint64_t *luts, cudaStream_t s) {
    add_scalar_luts_kernel<<<nblk, 256, 0, s>>>(ctr, byte_index, nbits, luts);
    return cudaGetLastError();
}
