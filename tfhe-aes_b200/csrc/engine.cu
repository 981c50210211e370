// engine.cu — context, key preparation and the device-level stages of one WoPBS pass
// (keyswitch -> PBS -> PFKS -> Fourier GGSW -> vertical packing), i.e. the GPU restatement of
// many_wopbs_without_padding (many_wopbs.rs:31-116) batched over many encrypted bytes.
#include <algorithm>
#include <cstdlib>
#include <cstring>
#include "engine.h"
#include "twiddle_host.h"

static thread_local std::string g_create_error;

// ------------------------------------------------------------------------------------------------
// workspace
// ------------------------------------------------------------------------------------------------
int ws_reserve(tfa_ctx *ctx, size_t bytes) {
    bytes += 1 << 20;
    if (bytes > ctx->ws_cap) {
        CU(cudaStreamSynchronize(ctx->stream));
        if (ctx->ws) CU(cudaFree(ctx->ws));
        ctx->ws = nullptr; ctx->ws_cap = 0;
        size_t cap = bytes + bytes / 8;
        CU(cudaMalloc(&ctx->ws, cap));
        ctx->ws_cap = cap;
    }
    ctx->ws_off = 0;
    return TFA_OK;
}
void *ws_alloc(tfa_ctx *ctx, size_t bytes) {
    size_t off = (ctx->ws_off + 255) & ~(size_t)255;
    if (off + bytes > ctx->ws_cap) { ctx->err = "internal: workspace exhausted"; return nullptr; }
    ctx->ws_off = off + bytes;
    return ctx->ws + off;
}
#define WS(ptr, T, count)                                         \
    T *ptr = ws_get<T>(ctx, (count));                             \
    if (!ptr) return TFA_ERR_STATE

int require_keys(tfa_ctx *ctx) {
    if (!ctx->keys_ready) return ctx->fail(TFA_ERR_STATE, "keys not loaded (tfa_ctx_load_keys / tfa_client_keygen)");
    return TFA_OK;
}

// ------------------------------------------------------------------------------------------------
// context
// ------------------------------------------------------------------------------------------------
static int ilog2u(uint64_t v) { int r = 0; while (v > 1) { v >>= 1; r++; } return r; }

extern "C" void tfa_param_opt(tfa_params *o) {
    // client.rs:31-57
    *o = tfa_params{669, 4, 512, 8, 5, 2, 6, 12, 3, 15, 1, 2, 1, 0, 3.0517578125e-05, 3.162026630747649e-16, 3.162026630747649e-16};
}

extern "C" int tfa_ctx_create(const tfa_params *p, int device, void *stream, tfa_ctx **out) {
    if (!out) { g_create_error = "null output pointer"; return TFA_ERR_PARAM; }
    *out = nullptr;
    if (!p) { g_create_error = "null params"; return TFA_ERR_PARAM; }
    if (p->poly_size != 512) { g_create_error = "only polynomial_size 512 is implemented (client.rs:35)"; return TFA_ERR_PARAM; }
    if (p->glwe_dim != 4 && p->glwe_dim != 1) { g_create_error = "glwe_dimension must be 4 (PARAM_OPT) or 1 (test set)"; return TFA_ERR_PARAM; }
    if (p->pbs_base_log != 8 || p->pbs_level != 5 || p->cbs_base_log != 15 || p->cbs_level != 1) {
        g_create_error = "PBS (2^8, 5) and CBS (2^15, 1) decompositions are the compiled kernel variants (client.rs:42-43,51-52)";
        return TFA_ERR_PARAM;
    }
    if (p->ks_base_log * p->ks_level > 63 || p->pfks_base_log * p->pfks_level > 63 || p->ks_base_log > 14 || p->pfks_base_log > 14) {
        g_create_error = "keyswitch decomposition out of range"; return TFA_ERR_PARAM;
    }
    if (p->lwe_dim < 1 || p->lwe_dim > 2048) { g_create_error = "lwe_dimension out of range"; return TFA_ERR_PARAM; }
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0) {
        g_create_error = std::string("no CUDA device (there is no CPU fallback): ") + cudaGetErrorString(e);
        return TFA_ERR_CUDA;
    }
    if (device < 0 || device >= ndev) { g_create_error = "bad device index"; return TFA_ERR_PARAM; }
    e = cudaSetDevice(device);
    if (e != cudaSuccess) { g_create_error = cudaGetErrorString(e); return TFA_ERR_CUDA; }
    tfa_ctx *ctx = new tfa_ctx();
    ctx->p = *p;
    ctx->n = p->lwe_dim; ctx->k = p->glwe_dim; ctx->N = p->poly_size;
    ctx->big = ctx->k * ctx->N; ctx->lw = ctx->big + 1; ctx->gsz = (ctx->k + 1) * ctx->N;
    ctx->device = device;
    ctx->sm_count = 148;
    cudaDeviceGetAttribute(&ctx->sm_count, cudaDevAttrMultiProcessorCount, device);
    ctx->launches = 0;
    ctx->pbs_count = 0;
    ctx->profiling = false;
    ctx->pbs_schedule = 0;
    ctx->own_stream = (stream == nullptr);
    ctx->stream = (cudaStream_t)stream;
    ctx->bsk_f = nullptr; ctx->ksk = nullptr; ctx->pfpksk = nullptr; ctx->kp_ksk = nullptr; ctx->kp_pfpksk = nullptr;
    ctx->tw = nullptr; ctx->keys_allocated = ctx->keys_ready = false;
    ctx->d_lwe_sk = ctx->d_glwe_sk = nullptr;
    for (auto &l : ctx->lut_cache) l = nullptr;
    ctx->ws = nullptr; ctx->ws_cap = ctx->ws_off = 0;
    ctx->pin = nullptr; ctx->pin_cap = ctx->pin_off = 0; ctx->pin_ev_valid[0] = ctx->pin_ev_valid[1] = false;
    ctx->ks_cols_pad = (ctx->n + 2) & ~1;
    // which integer-keyswitch kernels this context will use (decided once: it fixes which key layouts exist)
    ctx->imma_ks = getenv("TFA_KS_IMMA") != nullptr || p->ks_base_log > 6 || !tc5_ks_supported(ctx->n + 1, ctx->ks_cols_pad, ctx->ks_kchunks() * 32);
    ctx->imma_pfks = getenv("TFA_PFKS_IMMA") != nullptr || p->pfks_base_log <= 6 || !tc5_pfks_supported(ctx->gsz, ctx->pf_kchunks() * 32);
    if (ctx->own_stream) {
        e = cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking);
        if (e != cudaSuccess) { g_create_error = cudaGetErrorString(e); delete ctx; return TFA_ERR_CUDA; }
    }
    cd tw[256];
    make_twiddle_table(tw);
    e = cudaMalloc(&ctx->tw, sizeof(tw));
    if (e == cudaSuccess) e = cudaMemcpyAsync(ctx->tw, tw, sizeof(tw), cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    if (e != cudaSuccess) { g_create_error = cudaGetErrorString(e); delete ctx; return TFA_ERR_CUDA; }
    *out = ctx;
    return TFA_OK;
}
extern "C" void tfa_ctx_destroy(tfa_ctx *ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    cudaFree(ctx->bsk_f); cudaFree(ctx->ksk); cudaFree(ctx->pfpksk); cudaFree(ctx->kp_ksk); cudaFree(ctx->kp_pfpksk);
    cudaFree(ctx->tw); cudaFree(ctx->d_lwe_sk); cudaFree(ctx->d_glwe_sk); cudaFree(ctx->ws);
    if (ctx->pin) { cudaFreeHost(ctx->pin); cudaEventDestroy(ctx->pin_ev[0]); cudaEventDestroy(ctx->pin_ev[1]); }
    for (auto l : ctx->lut_cache) cudaFree(l);
    if (ctx->own_stream) cudaStreamDestroy(ctx->stream);
    delete ctx;
}
extern "C" const char *tfa_last_error(const tfa_ctx *ctx) { return ctx ? ctx->err.c_str() : g_create_error.c_str(); }
extern "C" int tfa_ctx_synchronize(tfa_ctx *ctx) { CU(cudaStreamSynchronize(ctx->stream)); return TFA_OK; }
extern "C" int tfa_ctx_set_pbs_schedule(tfa_ctx *ctx, int schedule) {
    if (schedule != 0 && (schedule < 2 || schedule > 4))
        return ctx->fail(TFA_ERR_PARAM, "pbs schedule must be 0 (auto), 2 (warp-specialised), 3 (one PBS per two-CTA cluster) or 4 (two sets per CTA)");
    std::lock_guard<std::mutex> lk(ctx->mu);
    ctx->pbs_schedule = schedule;
    return TFA_OK;
}
extern "C" uint64_t tfa_ctx_launch_count(const tfa_ctx *ctx) { return ctx->launches; }
extern "C" uint64_t tfa_ctx_pbs_count(const tfa_ctx *ctx) { return ctx->pbs_count; }

// ------------------------------------------------------------------------------------------------
// key preparation
// ------------------------------------------------------------------------------------------------
extern "C" int tfa_ctx_alloc_keys(tfa_ctx *ctx) {
    std::lock_guard<std::mutex> lk(ctx->mu);
    CU(cudaSetDevice(ctx->device));
    if (ctx->keys_allocated) return TFA_OK;
    // idempotent per buffer: a call that failed half way can be repeated
    if (!ctx->bsk_f) CU(cudaMalloc(&ctx->bsk_f, ctx->bsk_f_bytes()));
    if (ctx->imma_ks && !ctx->kp_ksk) CU(cudaMalloc(&ctx->kp_ksk, ctx->kp_ksk_bytes()));
    if (ctx->imma_pfks && !ctx->kp_pfpksk) CU(cudaMalloc(&ctx->kp_pfpksk, ctx->kp_pfpksk_bytes()));
    if (!ctx->pfpksk) CU(cudaMalloc(&ctx->pfpksk, ctx->pfpksk_bytes()));
    if (!ctx->ksk) CU(cudaMalloc(&ctx->ksk, ctx->ksk_bytes()));
    ctx->keys_allocated = true;
    return TFA_OK;
}
// Device buffers that make up the prepared keys, for replication to other GPUs (one broadcast each): the Fourier BSK, the
// PFPKSK and the KSK in their standard layouts, then the mma.sync fallback layouts when this context uses them.
extern "C" int tfa_ctx_key_buffers(tfa_ctx *ctx, void **ptrs, size_t *bytes, int *count) {
    std::lock_guard<std::mutex> lk(ctx->mu);
    if (!ctx->keys_allocated) return ctx->fail(TFA_ERR_STATE, "key buffers not allocated");
    int c = 0;
    ptrs[c] = ctx->bsk_f; bytes[c++] = ctx->bsk_f_bytes();
    ptrs[c] = ctx->pfpksk; bytes[c++] = ctx->pfpksk_bytes();
    ptrs[c] = ctx->ksk; bytes[c++] = ctx->ksk_bytes();
    if (ctx->imma_ks) { ptrs[c] = ctx->kp_ksk; bytes[c++] = ctx->kp_ksk_bytes(); }
    if (ctx->imma_pfks) { ptrs[c] = ctx->kp_pfpksk; bytes[c++] = ctx->kp_pfpksk_bytes(); }
    *count = c;
    return TFA_OK;
}
extern "C" int tfa_ctx_keys_ready(tfa_ctx *ctx) {
    std::lock_guard<std::mutex> lk(ctx->mu);
    if (!ctx->keys_allocated) return ctx->fail(TFA_ERR_STATE, "key buffers not allocated");
    ctx->keys_ready = true;
    return TFA_OK;
}

// standard-domain buffers of the two integer keys (KSK with rows padded to ks_cols_pad words): they stay, they are the
// B operands of the tcgen05 keyswitch kernels exactly as they lie
int alloc_key_staging(tfa_ctx *ctx) {
    if (!ctx->ksk) CU(cudaMalloc(&ctx->ksk, ctx->ksk_bytes()));
    if (!ctx->pfpksk) CU(cudaMalloc(&ctx->pfpksk, ctx->pfpksk_bytes()));
    return TFA_OK;
}
// finishes key preparation from standard-domain device buffers: bsk_std [n*l*(k+1)*(k+1) polys] -> Fourier; ctx->ksk (padded
// rows) and ctx->pfpksk stay as they are (tcgen05 operands) and are re-laid out for the mma.sync kernels only if those will run
int prepare_keys_from_device(tfa_ctx *ctx, const u64 *bsk_std_dev) {
    const long npoly = (long)ctx->n * ctx->p.pbs_level * (ctx->k + 1) * (ctx->k + 1);
    RC(dev_fourier(ctx, bsk_std_dev, npoly, ctx->p.pbs_level, ctx->bsk_f));
    if (ctx->imma_ks) {
        CU(launch_imma_prepare_key(ctx->ksk, 0, 1, ctx->ks_rows(), ctx->n + 1, ctx->ks_cols_pad, ctx->kp_ksk, ctx->stream));
        ctx->launches++;
    }
    if (ctx->imma_pfks) {
        CU(launch_imma_prepare_key(ctx->pfpksk, (size_t)ctx->pf_rows() * ctx->gsz, ctx->k + 1, ctx->pf_rows(), ctx->gsz, ctx->gsz, ctx->kp_pfpksk,
                                   ctx->stream));
        ctx->launches++;
    }
    CU(cudaStreamSynchronize(ctx->stream));
    ctx->keys_ready = true;
    return TFA_OK;
}

extern "C" int tfa_ctx_load_keys(tfa_ctx *ctx, const uint64_t *bsk, const uint64_t *ksk, const uint64_t *pfpksk) {
    if (!bsk || !ksk || !pfpksk) return ctx->fail(TFA_ERR_PARAM, "null key pointer");
    RC(tfa_ctx_alloc_keys(ctx));
    std::lock_guard<std::mutex> lk(ctx->mu);
    CU(cudaSetDevice(ctx->device));
    RC(alloc_key_staging(ctx));
    const size_t bsk_bytes = (size_t)ctx->n * ctx->p.pbs_level * (ctx->k + 1) * ctx->gsz * 8;
    struct DevBuf {   // the 343 MB staging copy of the standard-domain BSK is freed on every path out of this function
        u64 *p = nullptr;
        ~DevBuf() { cudaFree(p); }
    } tmp;
    CU(cudaMalloc(&tmp.p, bsk_bytes));
    CU(cudaMemcpyAsync(tmp.p, bsk, bsk_bytes, cudaMemcpyHostToDevice, ctx->stream));
    CU(cudaMemsetAsync(ctx->ksk, 0, ctx->ksk_bytes(), ctx->stream));
    CU(cudaMemcpy2DAsync(ctx->ksk, (size_t)ctx->ks_cols_pad * 8, ksk, (size_t)(ctx->n + 1) * 8, (size_t)(ctx->n + 1) * 8,
                         (size_t)ctx->big * ctx->p.ks_level, cudaMemcpyHostToDevice, ctx->stream));
    CU(cudaMemcpyAsync(ctx->pfpksk, pfpksk, ctx->pfpksk_bytes(), cudaMemcpyHostToDevice, ctx->stream));
    return prepare_keys_from_device(ctx, tmp.p);
}

// ------------------------------------------------------------------------------------------------
// stages
// ------------------------------------------------------------------------------------------------
static int pick_G(int K, int count) {
    if (K == 4) return count > 296 ? 3 : (count > 148 ? 2 : 1);
    return count >= 16 ? 8 : (count >= 4 ? 4 : 1);
}

int dev_fourier(tfa_ctx *ctx, const u64 *polys, long npoly, int levels, double2 *out) {
    StageTimer t(ctx, ST_FOURIER);
    ConvertArgs a{polys, out, ctx->tw, npoly, ctx->k, levels};
    CU(launch_fourier_convert(a, ctx->stream));
    ctx->launches++;
    return TFA_OK;
}

// SURVEY §9.4(1): out = (0,..,0,b) - sum_i sum_l d_{i,l} KSK[i][l]
int dev_keyswitch(tfa_ctx *ctx, const u64 *in, int count, u64 *out) {
    const int np = ctx->n + 1, rows_pad = ctx->ks_kchunks() * 32;
    const int limbs = ctx->p.ks_base_log > 6 ? 2 : 1;  // digits in [-beta/2, beta/2]: one s8 limb holds [-64, 63]
    WS(dl, int8_t, (size_t)count * rows_pad);
    int8_t *dh = nullptr;
    if (limbs == 2) { dh = ws_get<int8_t>(ctx, (size_t)count * rows_pad); if (!dh) return TFA_ERR_STATE; }
    {
        StageTimer t(ctx, ST_KS_DECOMP);
        if (rows_pad != ctx->ks_rows()) {
            CU(cudaMemsetAsync(dl, 0, (size_t)count * rows_pad, ctx->stream));
            if (dh) CU(cudaMemsetAsync(dh, 0, (size_t)count * rows_pad, ctx->stream));
        }
        CU(launch_imma_decompose(in, ctx->lw, ctx->big, count, ctx->p.ks_base_log, ctx->p.ks_level, rows_pad, dl, dh, ctx->stream));
    }
    StageTimer t(ctx, ST_KS_GEMV);
    if (!ctx->imma_ks) {
        // 5th-generation tensor cores, key consumed in its standard layout (tc5_kernels.cu)
        CU(launch_tc5_keyswitch(dl, rows_pad, ctx->ksk, ctx->ks_rows(), np, ctx->ks_cols_pad, count, in, ctx->lw, ctx->big, out, np, ctx->stream));
        ctx->launches += 1;
        return TFA_OK;
    }
    CU(launch_gemv_init(out, np, np, count, nullptr, 0, in, ctx->lw, ctx->big, ctx->n, ctx->stream));
    ImmaGemvArgs g{};
    g.dl = dl; g.dh = dh; g.kp = ctx->kp_ksk; g.out = out; g.out_stride = np; g.rows_pad = rows_pad;
    g.kchunks = ctx->ks_kchunks(); g.ntiles = ctx->ks_ntiles(); g.ncols = np; g.nkeys = 1; g.count = count;
    CU(launch_imma_gemv(g, limbs, ctx->stream));
    ctx->launches += 3;
    return TFA_OK;
}

// SURVEY §9.4(5): for keys r = key0 .. key0 + nkeys - 1: glwe_r = - sum_j sum_l d_{j,l} PFPKSK_r[j][l]; out[b][r - key0][gsz] with
// stride.  The circuit bootstrap uses all k + 1 keys, GLWE packing key k alone.
int dev_pfks(tfa_ctx *ctx, const u64 *in, int count, u64 *out, int out_stride, int key0, int nkeys) {
    const int rows_pad = ctx->pf_kchunks() * 32;
    const int limbs = ctx->p.pfks_base_log > 6 ? 2 : 1;
    WS(dl, int8_t, (size_t)count * rows_pad);
    int8_t *dh = nullptr;
    if (limbs == 2) { dh = ws_get<int8_t>(ctx, (size_t)count * rows_pad); if (!dh) return TFA_ERR_STATE; }
    {
        StageTimer t(ctx, ST_PFKS_DECOMP);
        if (rows_pad != ctx->pf_rows()) {
            CU(cudaMemsetAsync(dl, 0, (size_t)count * rows_pad, ctx->stream));
            if (dh) CU(cudaMemsetAsync(dh, 0, (size_t)count * rows_pad, ctx->stream));
        }
        CU(launch_imma_decompose(in, ctx->lw, ctx->big + 1, count, ctx->p.pfks_base_log, ctx->p.pfks_level, rows_pad, dl, dh, ctx->stream));
    }
    StageTimer t(ctx, ST_PFKS_GEMV);
    if (!ctx->imma_pfks) {
        // 5th-generation tensor cores, key consumed in its standard layout (tc5_kernels.cu).  Launched in slices of at
        // most 6 144 bits: every column tile re-reads the digit planes of its launch (12.4 KB per bit), and 6 144 bits
        // of them (76 MB) stay in L2 next to the streamed key while 18 944 (234 MB) would be re-read from HBM 400 times.
        const int nslices = (count + 6143) / 6144;
        const int slice = (((count + nslices - 1) / nslices) + 127) & ~127;
        for (int b0 = 0; b0 < count; b0 += slice) {
            const int nb = count - b0 < slice ? count - b0 : slice;
            CU(launch_tc5_pfks(dl + (size_t)b0 * rows_pad, dh + (size_t)b0 * rows_pad, rows_pad, ctx->pfpksk + (size_t)key0 * ctx->pf_rows() * ctx->gsz,
                               nkeys, ctx->pf_rows(), ctx->gsz, nb, out + (size_t)b0 * out_stride, out_stride, ctx->stream));
            ctx->launches += 1;
        }
        return TFA_OK;
    }
    CU(launch_gemv_init(out, out_stride, nkeys * ctx->gsz, count, nullptr, 0, nullptr, 0, 0, 0, ctx->stream));
    ImmaGemvArgs g{};
    g.dl = dl; g.dh = dh; g.kp = ctx->kp_pfpksk + (size_t)key0 * ctx->pf_ntiles() * ctx->pf_kchunks() * 2048; g.out = out; g.out_stride = out_stride;
    g.rows_pad = rows_pad; g.kchunks = ctx->pf_kchunks(); g.ntiles = ctx->pf_ntiles(); g.ncols = ctx->gsz; g.nkeys = nkeys; g.count = count;
    CU(launch_imma_gemv(g, limbs, ctx->stream));
    ctx->launches += 3;
    return TFA_OK;
}

// SURVEY §9.4(3).  Three kernels of the same arithmetic (measured on B200, PARAM_OPT, 669 steps):
//   pbs_ws2_kernel.cu  two sets of three ciphertexts per CTA taking turns: 18.9 ms per wave of 888 against 2 x 10.1 ms.  Whole
//                      waves go to it, and so does a remainder of more than half a wave (pbs_ws_kernel would need two rounds of
//                      148 CTAs for it: 20.2 ms).
//   pbs_cl2_kernel.cu  one PBS per two-CTA cluster, levels transformed in parallel: at most one wave of clusters (74 ciphertexts)
//                      -- key expansion stages, carry chain of few blocks, a single CTR block.
//   pbs_ws_kernel.cu   warp-specialised, G ciphertexts per CTA (pick_G): a partial wave in 5-10 ms (10.6 ms per wave of 148 CTAs
//                      at G = 3, 9.9 ms at G = 2, 7.5 ms at G = 1); every other batch, and every batch at K = 1.
// Schedules 2, 3 and 4 force one of them (tfa_ctx_set_pbs_schedule); 3 and 4 exist at K = 4 only and fall back to pbs_ws_kernel.
int dev_pbs(tfa_ctx *ctx, const u64 *in, int count, const u64 *lut, u64 in_scale, u64 pre_add, u64 post_add, u64 *out) {
    StageTimer t(ctx, ST_PBS);
    ctx->pbs_count += (u64)count;
    PbsArgs a{};
    a.lwe_in = in; a.bsk = ctx->bsk_f; a.tw = ctx->tw; a.lut = lut; a.out = out;
    a.in_scale = in_scale; a.pre_add_body = pre_add; a.post_add = post_add; a.lwe_dim = ctx->n; a.count = count;
    const int sched = ctx->pbs_schedule;
    if (ctx->k == 4 && (sched == 0 || sched == 4)) {
        const int wave = 6 * ctx->sm_count;
        int n2 = sched == 4 ? count : (count / wave) * wave;
        if (count - n2 > wave / 2) n2 = count;
        if (n2 > 0) {
            PbsArgs b = a;
            b.count = n2;
            CU(launch_pbs_ws2(ctx->k, 3, ctx->p.pbs_base_log, ctx->p.pbs_level, b, ctx->stream));
            ctx->launches++;
            if (n2 == count) return TFA_OK;
            a.lwe_in += (size_t)n2 * (ctx->n + 1);
            a.out += (size_t)n2 * (ctx->k * ctx->N + 1);
            a.count = count -= n2;
        }
    }
    if (ctx->k == 4 && ((sched == 0 && count <= 74) || sched == 3)) CU(launch_pbs_cl2(a, ctx->stream));
    else CU(launch_pbs_ws(ctx->k, pick_G(ctx->k, count), ctx->p.pbs_base_log, ctx->p.pbs_level, a, ctx->stream));
    ctx->launches++;
    return TFA_OK;
}

// SURVEY §9.4(1), general form.  out [count][nbits][n+1] with bit 0 = least significant extracted bit
// (the reference's list stores the same ciphertexts in reverse order, many_wopbs.rs:179).
int dev_extract_bits(tfa_ctx *ctx, const u64 *in, int count, int delta_log, int nbits, u64 *out) {
    const int np = ctx->n + 1, lw = ctx->lw;
    if (nbits == 1 && 64 - delta_log - 1 == 0) return dev_keyswitch(ctx, in, count, out);  // the reference's case: KS only
    WS(buf, u64, (size_t)count * lw);
    WS(shifted, u64, (size_t)count * lw);
    WS(ks, u64, (size_t)count * np);
    WS(pbs, u64, (size_t)count * lw);
    WS(lut, u64, ctx->N);
    CU(cudaMemcpyAsync(buf, in, (size_t)count * lw * 8, cudaMemcpyDeviceToDevice, ctx->stream));
    for (int bit = 0; bit < nbits; bit++) {
        CU(launch_scale_lwe(buf, shifted, (long)count * lw, 1ull << (64 - delta_log - bit - 1), ctx->stream));
        RC(dev_keyswitch(ctx, shifted, count, ks));
        CU(cudaMemcpy2DAsync(out + (size_t)bit * np, (size_t)nbits * np * 8, ks, (size_t)np * 8, (size_t)np * 8, count,
                             cudaMemcpyDeviceToDevice, ctx->stream));
        ctx->launches += 1;
        if (bit == nbits - 1) break;
        CU(launch_fill_u64(lut, ctx->N, (u64)0 - (1ull << (delta_log - 1 + bit)), ctx->stream));
        RC(dev_pbs(ctx, ks, count, lut, 1, 1ull << 62, 1ull << (delta_log + bit - 1), pbs));
        CU(launch_sub_lwe(buf, pbs, (long)count * lw, ctx->stream));
        ctx->launches += 2;
    }
    return TFA_OK;
}

// SURVEY §9.4(2): ggsw_std [count][cbs_level][k+1][gsz]
int dev_circuit_bootstrap(tfa_ctx *ctx, const u64 *lwe_small, int count, u64 *ggsw_std) {
    const int kp1 = ctx->k + 1, L = ctx->p.cbs_level;
    WS(bs, u64, (size_t)count * ctx->lw);
    WS(lut, u64, (size_t)ctx->N * L);
    for (int lvl = 1; lvl <= L; lvl++) {
        const u64 alpha = 1ull << (63 - ctx->p.cbs_base_log * lvl);
        u64 *l = lut + (size_t)(lvl - 1) * ctx->N;
        CU(launch_fill_u64(l, ctx->N, (u64)0 - alpha, ctx->stream));
        ctx->launches++;
        // homomorphic_shift_boolean with DeltaLog(63): multiply by 2^(64-63-1) = 1, add q/4, PBS, add alpha
        RC(dev_pbs(ctx, lwe_small, count, l, 1, 1ull << 62, alpha, bs));
        RC(dev_pfks(ctx, bs, count, ggsw_std + (size_t)(lvl - 1) * kp1 * ctx->gsz, L * kp1 * ctx->gsz, 0, kp1));
    }
    return TFA_OK;
}

// SURVEY §9.4(7).  ggsw_f [njobs][nbits][...] with bit 0 = LSB.  LUT polynomials per output:
// lut[job*lut_job_stride + o*lut_out_stride + poly*N + j], lut_size/N polynomials each.
// Bits 0..nshared-1 of every job come from ggsw_shared instead, offset by shared_set[job] * shared_set_stride (double2) when
// shared_set (device, [njobs]) is given.
int dev_vertical_packing(tfa_ctx *ctx, const double2 *ggsw_f, int njobs, int nbits, const u64 *lut, size_t lut_job_stride,
                         size_t lut_out_stride, int nouts, int lut_size, u64 *out, const double2 *ggsw_shared, int nshared,
                         const int32_t *shared_set, size_t shared_set_stride) {
    const int npoly = lut_size / ctx->N;
    int tree = ilog2u(npoly);
    if (tree > nbits) tree = 0;
    if (nshared > 0 && tree > 0) return ctx->fail(TFA_ERR_UNSUPPORTED, "shared GGSWs are only wired into the blind-rotation half of vertical packing");
    const u64 *glwe_init = nullptr;
    const int K = ctx->k;
    if (tree > 0) {
        // CMux tree over the `tree` most significant bits: layer by layer, least significant tree bit first
        const int nleaf = 1 << tree;
        WS(bufa, u64, (size_t)njobs * nouts * nleaf * ctx->gsz);
        WS(bufb, u64, (size_t)njobs * nouts * (nleaf / 2) * ctx->gsz);
        CU(launch_tree_leaves(lut, lut_job_stride, lut_out_stride, njobs, nouts, nleaf, K, bufa, ctx->stream));
        ctx->launches++;
        u64 *src = bufa, *dst = bufb;
        int cnt = nleaf;
        for (int layer = 0; layer < tree; layer++, cnt >>= 1) {
            StageTimer tm(ctx, ST_TREE);
            TreeArgs t{};
            t.ggsw_f = ggsw_f; t.tw = ctx->tw; t.in = src; t.out = dst; t.nbits = nbits; t.bit_index = nbits - tree + layer;
            t.npairs = nouts * cnt / 2; t.njobs = njobs;
            int G = (K == 4) ? (t.npairs >= 3 ? 3 : 1) : (t.npairs >= 8 ? 8 : 1);
            CU(launch_cmux_tree(K, G, ctx->p.cbs_base_log, ctx->p.cbs_level, t, ctx->stream));
            ctx->launches++;
            u64 *tmp = src; src = dst; dst = tmp;
        }
        glwe_init = src;
    }
    StageTimer tm(ctx, ST_VP);
    VpArgs v{};
    v.ggsw_f = ggsw_f; v.tw = ctx->tw; v.lut = lut; v.glwe_init = glwe_init; v.out = out;
    v.lut_job_stride = lut_job_stride; v.lut_out_stride = lut_out_stride;
    v.nbits = nbits; v.nrot = nbits - tree; v.nouts = nouts; v.njobs = njobs;
    v.ggsw_shared = ggsw_shared; v.nshared = nshared; v.shared_set = shared_set; v.shared_set_stride = shared_set_stride;
    int G;
    if (K == 4) G = nouts >= 3 ? 3 : (nouts == 2 ? 2 : 1);
    else G = nouts >= 8 ? 8 : (nouts >= 4 ? 4 : 1);
    CU(launch_vp(K, G, ctx->p.cbs_base_log, ctx->p.cbs_level, v, ctx->stream));
    ctx->launches++;
    return TFA_OK;
}

size_t many_wopbs_scratch(const tfa_ctx *ctx, int nct, int nblocks, int nouts, int lut_size) {
    const int bpb = ilog2u((u64)ctx->p.message_modulus * ctx->p.carry_modulus);
    const size_t nb = (size_t)nct * nblocks * bpb;  // bits
    const size_t ggsw = (size_t)ctx->p.cbs_level * (ctx->k + 1) * ctx->gsz * 8;
    size_t s = 0;
    s += nb * (ctx->n + 1) * 8;                                 // extracted bits
    s += nb * ggsw * 2;                                          // ggsw std + fourier
    s += nb * ctx->lw * 8 * 4;                                   // pbs out, extract_bits buffers
    s += nb * (size_t)(ctx->big + 1) * ctx->p.pfks_level * 2;    // pfks digits
    s += nb * (size_t)ctx->big * ctx->p.ks_level * 2;            // ks digits
    const int npoly = lut_size / ctx->N;
    if (npoly > 1) s += (size_t)nct * nouts * npoly * ctx->gsz * 8 * 3 / 2;
    return s + (64 << 10) * 16;
}

// many_wopbs_without_padding (many_wopbs.rs:31-116) for nct radix ciphertexts of nblocks blocks.
// out [nct][nouts][lw].
int dev_many_wopbs(tfa_ctx *ctx, const u64 *ct_in, int nct, int nblocks, const u64 *lut, size_t lut_job_stride,
                   size_t lut_out_stride, int nouts, int lut_size, u64 *out) {
    const int block_mod = ctx->p.message_modulus * ctx->p.carry_modulus;
    const int bpb = ilog2u(block_mod);
    const int delta_log = ilog2u((1ull << 63) / (block_mod / 2));
    const int nbits = nblocks * bpb;               // selector bits per ciphertext
    const int nb = nct * nbits;
    // (1) custom_extract_bits (many_wopbs.rs:161-202): every block independently
    WS(bits, u64, (size_t)nb * (ctx->n + 1));
    RC(dev_extract_bits(ctx, ct_in, nct * nblocks, delta_log, bpb, bits));
    // (2) circuit bootstrap every bit (many_wopbs.rs:252-264) and move the GGSWs to the Fourier domain
    const size_t ggsw_words = (size_t)ctx->p.cbs_level * (ctx->k + 1) * ctx->gsz;
    WS(ggsw_std, u64, (size_t)nb * ggsw_words);
    WS(ggsw_f, double2, (size_t)nb * ggsw_words / 2);
    RC(dev_circuit_bootstrap(ctx, bits, nb, ggsw_std));
    RC(dev_fourier(ctx, ggsw_std, (long)nb * ctx->p.cbs_level * (ctx->k + 1) * (ctx->k + 1), ctx->p.cbs_level, ggsw_f));
    // (3) one vertical packing per LUT output (many_wopbs.rs:267-279)
    return dev_vertical_packing(ctx, ggsw_f, nct, nbits, lut, lut_job_stride, lut_out_stride, nouts, lut_size, out);
}

// GLWE packing (DESIGN §3): PFKS with key k of the inputs of PACK_SLICE_GLWES GLWEs at a time (6 144 bits: one tcgen05 PFKS
// launch, 126 MB of PFKS output at PARAM_OPT), then the rotation-sum and 16-bit rounding of glwe_pack_kernel.
static const int PACK_SLICE_GLWES = 12;
size_t pack_lwe_scratch(const tfa_ctx *ctx, int count) {
    const size_t nb = (size_t)std::min(count, PACK_SLICE_GLWES * ctx->N);
    return nb * ctx->gsz * 8 + nb * ctx->pf_kchunks() * 32 * 2 + 4096;   // PFKS output, two digit-limb planes
}
int dev_pack_lwe(tfa_ctx *ctx, const u64 *lwe, int count, uint16_t *packed) {
    const int slice = PACK_SLICE_GLWES * ctx->N;
    WS(pf, u64, (size_t)std::min(count, slice) * ctx->gsz);
    const size_t mark = ctx->ws_off;
    for (long b0 = 0; b0 < count; b0 += slice) {
        const int nb = (int)std::min((long)count - b0, (long)slice);
        ctx->ws_off = mark;
        RC(dev_pfks(ctx, lwe + (size_t)b0 * ctx->lw, nb, pf, ctx->gsz, ctx->k, 1));
        StageTimer t(ctx, ST_MISC);   // the PFKS above is timed in its own stages; the rotation-sum kernel is "misc"
        CU(launch_glwe_pack(pf, nb, ctx->k, packed + (size_t)(b0 / ctx->N) * ctx->gsz, ctx->stream));
        ctx->launches++;
    }
    return TFA_OK;
}
int dev_unpack_lwe(tfa_ctx *ctx, const uint16_t *packed, int count, u64 *lwe_out) {
    StageTimer t(ctx, ST_MISC);
    CU(launch_glwe_unpack(packed, count, ctx->k, lwe_out, ctx->stream));
    ctx->launches++;
    return TFA_OK;
}

// pinned staging for `bytes` of host data that an asynchronous copy on ctx->stream will read
static int pin_stage(tfa_ctx *ctx, size_t bytes, char **out) {
    const size_t cap = (size_t)16 << 20, half = cap / 2;
    if (bytes > half) return ctx->fail(TFA_ERR_PARAM, "gather table too large for the staging ring");
    if (!ctx->pin) {
        CU(cudaHostAlloc((void **)&ctx->pin, cap, cudaHostAllocDefault));
        CU(cudaEventCreateWithFlags(&ctx->pin_ev[0], cudaEventDisableTiming));
        CU(cudaEventCreateWithFlags(&ctx->pin_ev[1], cudaEventDisableTiming));
        ctx->pin_cap = cap; ctx->pin_off = 0;
    }
    bytes = (bytes + 255) & ~(size_t)255;
    const int h = ctx->pin_off < half ? 0 : 1;
    if (ctx->pin_off + bytes > (size_t)(h + 1) * half) {   // leave half h: everything staged in it has been queued before this event
        CU(cudaEventRecord(ctx->pin_ev[h], ctx->stream));
        ctx->pin_ev_valid[h] = true;
        const int nh = h ^ 1;
        if (ctx->pin_ev_valid[nh]) {                       // enter the other half once its previous contents have been copied
            CU(cudaEventSynchronize(ctx->pin_ev[nh]));
            ctx->pin_ev_valid[nh] = false;
        }
        ctx->pin_off = (size_t)nh * half;
    }
    *out = ctx->pin + ctx->pin_off;
    ctx->pin_off += bytes;
    return TFA_OK;
}

// the gather list goes through the context's pinned ring: the copy is asynchronous (a pageable source of this size would
// make the driver synchronise the stream) and does not depend on the lifetime of the host table
template <typename E>
static int upload_table(tfa_ctx *ctx, const std::vector<E> &entries, E **out) {
    WS(d, E, entries.size());
    char *stage = nullptr;
    RC(pin_stage(ctx, entries.size() * sizeof(E), &stage));
    memcpy(stage, entries.data(), entries.size() * sizeof(E));
    CU(cudaMemcpyAsync(d, stage, entries.size() * sizeof(E), cudaMemcpyHostToDevice, ctx->stream));
    *out = d;
    return TFA_OK;
}
int dev_lwe_sum(tfa_ctx *ctx, const std::vector<SumEntry> &entries, int unit_words) {
    StageTimer t(ctx, ST_LINEAR);
    SumEntry *d = nullptr;
    RC(upload_table(ctx, entries, &d));
    CU(launch_lwe_sum(d, (int)entries.size(), unit_words, ctx->stream));
    ctx->launches++;
    return TFA_OK;
}
int dev_lwe_sum_xor(tfa_ctx *ctx, const std::vector<SumXorEntry> &entries) {
    StageTimer t(ctx, ST_LINEAR);
    SumXorEntry *d = nullptr;
    RC(upload_table(ctx, entries, &d));
    CU(launch_lwe_sum_xor(d, (int)entries.size(), ctx->lw, ctx->stream));
    ctx->launches++;
    return TFA_OK;
}

// ------------------------------------------------------------------------------------------------
// per-stage GPU timing
// ------------------------------------------------------------------------------------------------
extern "C" int tfa_ctx_profile(tfa_ctx *ctx, int enable) {
    std::lock_guard<std::mutex> lk(ctx->mu);
    for (auto &r : ctx->prof) { cudaEventDestroy(r.a); cudaEventDestroy(r.b); }
    ctx->prof.clear();
    ctx->profiling = enable != 0;
    return TFA_OK;
}
extern "C" int tfa_ctx_profile_report(tfa_ctx *ctx, double *ms_per_stage /* [10] */, int *launch_groups /* [10] */) {
    std::lock_guard<std::mutex> lk(ctx->mu);
    CU(cudaStreamSynchronize(ctx->stream));
    for (int i = 0; i < ST_COUNT; i++) { ms_per_stage[i] = 0; launch_groups[i] = 0; }
    for (auto &r : ctx->prof) {
        float ms = 0;
        CU(cudaEventElapsedTime(&ms, r.a, r.b));
        ms_per_stage[r.stage] += ms; launch_groups[r.stage]++;
    }
    return TFA_OK;
}

// ------------------------------------------------------------------------------------------------
// measured FP64 pipe peak (SURVEY §8d asks for a DFMA microbenchmark: B200's FP64 peak is not in
// MEASURED_PEAKS.json).  16 independent FMA chains per thread, 2 CTAs of 512 threads per SM.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(512) dfma_peak_kernel(double *out, int iters, double a, double b) {
    double x[16];
#pragma unroll
    for (int i = 0; i < 16; i++) x[i] = threadIdx.x * 1e-3 + i;
    for (int it = 0; it < iters; it++) {
#pragma unroll
        for (int i = 0; i < 16; i++) x[i] = fma(x[i], a, b);
    }
    double s = 0;
#pragma unroll
    for (int i = 0; i < 16; i++) s += x[i];
    if (s == 123.456) out[0] = s;
}
// the same pipe driven by mma.sync.m8n8k4.f64 (256 FMAs per warp instruction): it reaches a little more of the nominal 64 FMA/clk/SM
// than plain DFMAs, whose three register operands cost a third issue cycle unless one comes from the reuse cache
__global__ void __launch_bounds__(256) dmma_peak_kernel(double *out, int iters, double seed) {
    double d[8][2];
#pragma unroll
    for (int i = 0; i < 8; i++) d[i][0] = d[i][1] = seed * i;
    const double ma = seed, mb = seed * 0.25;
    for (int it = 0; it < iters; it++) {
#pragma unroll
        for (int i = 0; i < 8; i++)
            asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n" : "+d"(d[i][0]), "+d"(d[i][1]) : "d"(ma), "d"(mb));
    }
    double s = 0;
#pragma unroll
    for (int i = 0; i < 8; i++) s += d[i][0] + d[i][1];
    if (s == 123.456) out[0] = s;
}
// both microbenchmarks; the roofline denominator is the larger of the two
extern "C" int tfa_measure_fp64_peaks(tfa_ctx *ctx, double *dfma_tflops, double *dmma_tflops) {
    std::lock_guard<std::mutex> lk(ctx->mu);
    CU(cudaSetDevice(ctx->device));
    int sms = 0;
    CU(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, ctx->device));
    double *d = nullptr;
    CU(cudaMalloc(&d, 8));
    cudaEvent_t e0, e1;
    CU(cudaEventCreate(&e0)); CU(cudaEventCreate(&e1));
    double best[2] = {0, 0};
    for (int which = 0; which < 2; which++)
        for (int rep = 0; rep < 5; rep++) {
            const int iters = which == 0 ? 20000 : 8000, grid = sms * 2;
            CU(cudaEventRecord(e0, ctx->stream));
            if (which == 0) dfma_peak_kernel<<<grid, 512, 0, ctx->stream>>>(d, iters, 1.0000001, 1e-9);
            else dmma_peak_kernel<<<grid, 256, 0, ctx->stream>>>(d, iters, 1e-9);
            CU(cudaEventRecord(e1, ctx->stream));
            CU(cudaEventSynchronize(e1));
            float ms = 0;
            CU(cudaEventElapsedTime(&ms, e0, e1));
            const double fl = which == 0 ? 2.0 * 16 * iters * 512.0 * grid : 2.0 * 8 * 256.0 * iters * 8.0 * grid;   // dmma: 8 instr x 256 FMA per warp, 8 warps
            if (rep > 0 && fl / (ms * 1e-3) * 1e-12 > best[which]) best[which] = fl / (ms * 1e-3) * 1e-12;
        }
    ctx->launches += 10;
    cudaEventDestroy(e0); cudaEventDestroy(e1); cudaFree(d);
    *dfma_tflops = best[0]; *dmma_tflops = best[1];
    return TFA_OK;
}
extern "C" int tfa_measure_fp64_peak(tfa_ctx *ctx, double *tflops) {
    double a = 0, b = 0;
    RC(tfa_measure_fp64_peaks(ctx, &a, &b));
    *tflops = a > b ? a : b;
    return TFA_OK;
}
