// engine.h — internal context of the library (not part of the C ABI).
#pragma once
#include <cuda_runtime.h>
#include <condition_variable>
#include <mutex>
#include <string>
#include <vector>
#include "../../include/tfhe_aes_b200.h"
#include "kernels.h"

typedef uint64_t u64;

struct tfa_ctx {
    tfa_params p;
    int n, k, N, big, lw, gsz;  // lw = k*N+1 words per big LWE, gsz = (k+1)*N words per GLWE
    int device, sm_count;
    cudaStream_t stream;
    bool own_stream;
    std::string err;
    std::mutex mu;
    u64 launches;
    u64 pbs_count;         // LWE ciphertexts blind-rotated since creation (tfa_ctx_pbs_count)

    // prepared keys (device)
    double2 *bsk_f;        // [n][pbs_level][k+1][k+1][256]
    u64 *ksk;              // keyswitch key, standard domain [big*ks_level][ks_cols_pad]: the B operand of the tcgen05 keyswitch as it lies
    u64 *pfpksk;           // PFPKSK list, standard domain [k+1][(big+1)*pfks_level][gsz]: the B operand of the tcgen05 PFKS
    // mma.sync fallback layouts: allocated, prepared and broadcast only when the fallback kernels will run (a shape the tcgen05
    // kernels do not take, or TFA_KS_IMMA / TFA_PFKS_IMMA set): +0.70 GB at PARAM_OPT otherwise
    uint8_t *kp_ksk;       // int8-limb fragment layout [ntiles][kchunks][2048]   (imma_kernels.cu)
    uint8_t *kp_pfpksk;    // same, [k+1][ntiles][kchunks][2048]
    bool imma_ks, imma_pfks;
    double2 *tw;           // 256 mid twiddles (twiddle_host.h)
    int ks_cols_pad;
    bool keys_allocated, keys_ready;

    // client-side secrets (tfa_client_keygen only)
    u64 *d_lwe_sk, *d_glwe_sk;
    std::vector<u64> h_lwe_sk, h_glwe_sk;

    // cached device LUT sets (sbox module): [0]=S [1]={S,2S,3S} [2]=invS [3]={9,11,13,14}x [4]=identity
    u64 *lut_cache[5];

    // optional per-stage GPU timing (tfa_ctx_profile): events around every launch group
    bool profiling;
    int pbs_schedule;      // 0 auto, 1 phase-synchronous, 2 warp-specialised, 3 cluster pair per ciphertext, 4 two sets per CTA (tfa_ctx_set_pbs_schedule)
    struct ProfRec { int stage; cudaEvent_t a, b; };
    std::vector<ProfRec> prof;

    // request coalescing of the per-block host entry points (api.cu): callers queue here, one of them runs the batch
    std::mutex qmu;
    std::condition_variable qcv;
    std::vector<struct CoalesceReq *> queue;
    bool leader = false;

    // bump workspace
    char *ws;
    size_t ws_cap, ws_off;
    // pinned staging ring for the small host-built tables of the linear layers (gather lists): the copy to the device is
    // asynchronous, and a half of the ring is only reused after the stream has passed the event recorded when it was last left
    char *pin;
    size_t pin_cap, pin_off;
    cudaEvent_t pin_ev[2];
    bool pin_ev_valid[2];

    size_t bsk_f_bytes() const { return (size_t)n * p.pbs_level * (k + 1) * 256 * (k + 1) * sizeof(double2); }
    size_t ksk_bytes() const { return (size_t)big * p.ks_level * ks_cols_pad * 8; }
    int ks_rows() const { return big * (int)p.ks_level; }
    int pf_rows() const { return (big + 1) * (int)p.pfks_level; }
    int ks_kchunks() const { return (ks_rows() + 31) / 32; }
    int pf_kchunks() const { return (pf_rows() + 31) / 32; }
    int ks_ntiles() const { return (n + 1 + 7) / 8; }
    int pf_ntiles() const { return (gsz + 7) / 8; }
    size_t kp_ksk_bytes() const { return (size_t)ks_ntiles() * ks_kchunks() * 2048; }
    size_t kp_pfpksk_bytes() const { return (size_t)(k + 1) * pf_ntiles() * pf_kchunks() * 2048; }
    size_t pfpksk_bytes() const { return (size_t)(k + 1) * (big + 1) * p.pfks_level * gsz * 8; }
    size_t byte_words() const { return (size_t)8 * lw; }

    int fail(int code, const std::string &what) { err = what; return code; }
    int fail_cuda(const char *what, cudaError_t e) {
        err = std::string(what) + ": " + cudaGetErrorString(e);
        return TFA_ERR_CUDA;
    }
};

#define CU(call)                                                       \
    do {                                                               \
        cudaError_t e__ = (call);                                      \
        if (e__ != cudaSuccess) return ctx->fail_cuda(#call, e__);     \
    } while (0)
#define RC(call)                  \
    do {                          \
        int r__ = (call);         \
        if (r__ != TFA_OK) return r__; \
    } while (0)

enum { ST_KS_DECOMP = 0, ST_KS_GEMV, ST_PBS, ST_PFKS_DECOMP, ST_PFKS_GEMV, ST_FOURIER, ST_VP, ST_TREE, ST_LINEAR, ST_MISC, ST_COUNT };
struct StageTimer {  // RAII: records two events on the context stream when profiling is on
    tfa_ctx *ctx; int idx;
    StageTimer(tfa_ctx *c, int stage) : ctx(c), idx(-1) {
        if (!c->profiling) return;
        tfa_ctx::ProfRec r; r.stage = stage;
        cudaEventCreate(&r.a); cudaEventCreate(&r.b);
        cudaEventRecord(r.a, c->stream);
        idx = (int)c->prof.size(); c->prof.push_back(r);
    }
    ~StageTimer() { if (idx >= 0) cudaEventRecord(ctx->prof[idx].b, ctx->stream); }
};

// workspace helpers
int ws_reserve(tfa_ctx *ctx, size_t bytes);      // make sure `bytes` of scratch are available, reset the bump pointer
void *ws_alloc(tfa_ctx *ctx, size_t bytes);      // bump allocation (256 B aligned); nullptr if exhausted
template <typename T>
static inline T *ws_get(tfa_ctx *ctx, size_t count) { return reinterpret_cast<T *>(ws_alloc(ctx, count * sizeof(T))); }

// device-level stages (all asynchronous on ctx->stream, scratch from the workspace)
int dev_keyswitch(tfa_ctx *ctx, const u64 *in, int count, u64 *out);
int dev_pbs(tfa_ctx *ctx, const u64 *in, int count, const u64 *lut, u64 in_scale, u64 pre_add, u64 post_add, u64 *out);
int dev_pfks(tfa_ctx *ctx, const u64 *in, int count, u64 *out, int out_stride);
int dev_fourier(tfa_ctx *ctx, const u64 *polys, long npoly, int levels, double2 *out);
int dev_extract_bits(tfa_ctx *ctx, const u64 *in, int count, int delta_log, int nbits, u64 *out /* [count][nbits][n+1], 0 = LSB */);
int dev_circuit_bootstrap(tfa_ctx *ctx, const u64 *lwe_small, int count, u64 *ggsw_std);
int dev_vertical_packing(tfa_ctx *ctx, const double2 *ggsw_f, int njobs, int nbits, const u64 *lut, size_t lut_job_stride,
                         size_t lut_out_stride, int nouts, int lut_size, u64 *out,
                         const double2 *ggsw_shared = nullptr, int nshared = 0);
int dev_many_wopbs(tfa_ctx *ctx, const u64 *ct_in, int nct, int nblocks, const u64 *lut, size_t lut_job_stride,
                   size_t lut_out_stride, int nouts, int lut_size, u64 *out);
size_t many_wopbs_scratch(const tfa_ctx *ctx, int nct, int nblocks, int nouts, int lut_size);
int dev_lwe_sum(tfa_ctx *ctx, const std::vector<SumEntry> &entries, int unit_words);
int dev_lwe_sum_xor(tfa_ctx *ctx, const std::vector<SumXorEntry> &entries);  // one encrypted byte per entry
int require_keys(tfa_ctx *ctx);
const u64 *cached_lut(tfa_ctx *ctx, int which);  // device pointer, see lut_cache
