// api.cu — the C ABI (include/tfhe_aes_b200.h): sbox module and Server entry points on top of the
// device stages of engine.cu.  Orchestration follows server.rs / sbox.rs line by line; the per-byte
// loops of the reference (server.rs:47-50, 59-61, 76-78, 88-91, 100-102) become one batched pass
// over all bytes of all resident blocks.
#include <algorithm>
#include <chrono>
#include <climits>
#include <condition_variable>
#include <cstring>
#include <mutex>
#include "engine.h"

static int ilog2u(uint64_t v) { int r = 0; while (v > 1) { v >>= 1; r++; } return r; }

// ------------------------------------------------------------------------------------------------
// tables (table.rs:2-37 = FIPS-197 S-box, generated from the field arithmetic) and sbox.rs:20-42
// ------------------------------------------------------------------------------------------------
static uint8_t SBOX[256], INV_SBOX[256];
static std::once_flag tables_once;   // process-wide tables, contexts on several threads may race to build them
static uint8_t xtime(uint8_t x) { return (uint8_t)((x << 1) ^ ((x & 0x80) ? 0x1B : 0)); }
static uint8_t gf_mul(uint8_t a, uint8_t b) { uint8_t r = 0; while (b) { if (b & 1) r ^= a; a = xtime(a); b >>= 1; } return r; }
static void build_tables() {
    for (int x = 0; x < 256; x++) {
        uint8_t inv = 0;
        if (x) for (int y = 1; y < 256; y++) if (gf_mul((uint8_t)x, (uint8_t)y) == 1) { inv = (uint8_t)y; break; }
        uint8_t s = inv, r = inv;
        for (int i = 0; i < 4; i++) { r = (uint8_t)((r << 1) | (r >> 7)); s ^= r; }
        s ^= 0x63;
        SBOX[x] = s; INV_SBOX[s] = (uint8_t)x;
    }
}
static void init_tables() { std::call_once(tables_once, build_tables); }

// ------------------------------------------------------------------------------------------------
// gen_lut (gen_lut.rs:9-42)
// ------------------------------------------------------------------------------------------------
extern "C" int tfa_lut_size(const tfa_params *p, int nb_block) {
    const int log_basis = ilog2u(p->message_modulus) + ilog2u(p->carry_modulus);
    if (nb_block < 1 || nb_block * log_basis > 24) return -1;
    const int sz = 1 << (nb_block * log_basis);
    return sz < (int)p->poly_size ? (int)p->poly_size : sz;
}
extern "C" int tfa_gen_lut(const tfa_params *p, int nb_block, const uint64_t *table, uint64_t *lut) {
    const uint64_t log_msg = ilog2u(p->message_modulus), log_carry = ilog2u(p->carry_modulus);
    const uint64_t log_basis = log_msg + log_carry, delta = 64 - log_basis;
    const int lut_size = tfa_lut_size(p, nb_block);
    if (lut_size < 0 || !table || !lut) return TFA_ERR_PARAM;
    const uint64_t nvals = 1ull << (nb_block * log_basis);
    for (int index = 0; index < lut_size; index++) {
        uint64_t value = 0, tmp_index = index;
        for (int i = 0; i < nb_block; i++) {
            const uint64_t tmp = tmp_index % (1ull << log_basis);
            tmp_index >>= log_basis;
            value += tmp << (log_msg * i);
        }
        const uint64_t fv = table[value % nvals];
        for (int b = 0; b < nb_block; b++) lut[(size_t)b * lut_size + index] = ((fv >> (log_msg * b)) % (1ull << log_msg)) << delta;
    }
    return TFA_OK;
}

// device-resident LUT sets of the sbox module, built once per context
const u64 *cached_lut(tfa_ctx *ctx, int which) {
    if (ctx->lut_cache[which]) return ctx->lut_cache[which];
    init_tables();
    static const int nl[5] = {1, 3, 1, 4, 1};
    const int L = nl[which];
    const int lsz = tfa_lut_size(&ctx->p, 8 / ilog2u((u64)ctx->p.message_modulus * ctx->p.carry_modulus));
    const int nblocks = 8 / ilog2u((u64)ctx->p.message_modulus * ctx->p.carry_modulus);
    std::vector<u64> host((size_t)L * nblocks * lsz), tab(256);
    static const int enc_m[3] = {1, 2, 3}, dec_m[4] = {9, 11, 13, 14};
    for (int i = 0; i < L; i++) {
        for (int x = 0; x < 256; x++) {
            switch (which) {
                case 0: tab[x] = SBOX[x]; break;                                   // sbox.rs:52
                case 1: tab[x] = gf_mul(SBOX[x], (uint8_t)enc_m[i]); break;        // sbox.rs:79-81
                case 2: tab[x] = INV_SBOX[x]; break;                               // sbox.rs:49
                case 3: tab[x] = gf_mul((uint8_t)x, (uint8_t)dec_m[i]); break;     // sbox.rs:74-77
                default: tab[x] = x; break;                                        // server.rs:118-119
            }
        }
        tfa_gen_lut(&ctx->p, nblocks, tab.data(), &host[(size_t)i * nblocks * lsz]);
    }
    u64 *d = nullptr;
    if (cudaMalloc(&d, host.size() * 8) != cudaSuccess) return nullptr;
    if (cudaMemcpyAsync(d, host.data(), host.size() * 8, cudaMemcpyHostToDevice, ctx->stream) != cudaSuccess) { cudaFree(d); return nullptr; }
    cudaStreamSynchronize(ctx->stream);
    ctx->lut_cache[which] = d;
    return d;
}

// ------------------------------------------------------------------------------------------------
// helpers for host-pointer entry points
// ------------------------------------------------------------------------------------------------
struct Guard {
    tfa_ctx *ctx;
    std::unique_lock<std::mutex> lk;
    explicit Guard(tfa_ctx *c) : ctx(c), lk(c->mu) { cudaSetDevice(c->device); }
};
#define H2D(dst, src, words) CU(cudaMemcpyAsync((dst), (src), (size_t)(words) * 8, cudaMemcpyHostToDevice, ctx->stream))
#define D2H(dst, src, words) CU(cudaMemcpyAsync((dst), (src), (size_t)(words) * 8, cudaMemcpyDeviceToHost, ctx->stream))
#define SYNC() CU(cudaStreamSynchronize(ctx->stream))
#define WSB(ptr, T, count)                    \
    T *ptr = ws_get<T>(ctx, (count));         \
    if (!ptr) return TFA_ERR_STATE

static int nblocks_per_byte(const tfa_ctx *ctx) { return 8 / ilog2u((u64)ctx->p.message_modulus * ctx->p.carry_modulus); }

// ------------------------------------------------------------------------------------------------
// many_wopbs / sbox / many_sbox
// ------------------------------------------------------------------------------------------------
static int many_wopbs_dev_nolock(tfa_ctx *ctx, const u64 *ct_in, int nct, int nblocks, const u64 *luts_dev, int L, u64 *out, bool reserve) {
    RC(require_keys(ctx));
    const int lsz = tfa_lut_size(&ctx->p, nblocks);
    if (lsz < 0 || nct < 1 || L < 1) return ctx->fail(TFA_ERR_PARAM, "many_wopbs: bad shape");
    if (reserve) RC(ws_reserve(ctx, many_wopbs_scratch(ctx, nct, nblocks, L * nblocks, lsz)));
    return dev_many_wopbs(ctx, ct_in, nct, nblocks, luts_dev, 0, (size_t)lsz, L * nblocks, lsz, out);
}
extern "C" int tfa_many_wopbs_dev(tfa_ctx *ctx, const uint64_t *ct_in, int nct, int nblocks, const uint64_t *luts_dev, int L, uint64_t *out) {
    Guard g(ctx);
    return many_wopbs_dev_nolock(ctx, ct_in, nct, nblocks, luts_dev, L, out, true);
}
extern "C" int tfa_many_wopbs(tfa_ctx *ctx, const uint64_t *ct_in, int nct, int nblocks, const uint64_t *luts, int L, uint64_t *out) {
    Guard g(ctx);
    RC(require_keys(ctx));
    const int lsz = tfa_lut_size(&ctx->p, nblocks);
    if (lsz < 0 || nct < 1 || L < 1) return ctx->fail(TFA_ERR_PARAM, "many_wopbs: bad shape");
    const size_t in_w = (size_t)nct * nblocks * ctx->lw, lut_w = (size_t)L * nblocks * lsz, out_w = (size_t)nct * L * nblocks * ctx->lw;
    RC(ws_reserve(ctx, many_wopbs_scratch(ctx, nct, nblocks, L * nblocks, lsz) + (in_w + lut_w + out_w) * 8));
    WSB(d_in, u64, in_w); WSB(d_lut, u64, lut_w); WSB(d_out, u64, out_w);
    H2D(d_in, ct_in, in_w); H2D(d_lut, luts, lut_w);
    RC(many_wopbs_dev_nolock(ctx, d_in, nct, nblocks, d_lut, L, d_out, false));
    D2H(out, d_out, out_w);
    SYNC();
    return TFA_OK;
}
static int sbox_like_dev(tfa_ctx *ctx, const u64 *in, int nct, int which, u64 *out) {
    static const int nl[5] = {1, 3, 1, 4, 1};
    const u64 *lut = cached_lut(ctx, which);
    if (!lut) return ctx->fail(TFA_ERR_CUDA, "LUT upload failed");
    return many_wopbs_dev_nolock(ctx, in, nct, nblocks_per_byte(ctx), lut, nl[which], out, false);
}
extern "C" int tfa_sbox(tfa_ctx *ctx, uint64_t *bytes, int nct, int inv) {
    Guard g(ctx);
    if (nct < 1) return ctx->fail(TFA_ERR_PARAM, "nct must be >= 1");
    RC(require_keys(ctx));
    const size_t w = (size_t)nct * ctx->byte_words();
    const int nb = nblocks_per_byte(ctx);
    RC(ws_reserve(ctx, many_wopbs_scratch(ctx, nct, nb, nb, tfa_lut_size(&ctx->p, nb)) + 2 * w * 8));
    WSB(d_in, u64, w); WSB(d_out, u64, w);
    H2D(d_in, bytes, w);
    RC(sbox_like_dev(ctx, d_in, nct, inv ? 2 : 0, d_out));
    D2H(bytes, d_out, w);
    SYNC();
    return TFA_OK;
}
extern "C" int tfa_many_sbox(tfa_ctx *ctx, const uint64_t *bytes_in, int nct, int inv, uint64_t *out) {
    Guard g(ctx);
    if (nct < 1) return ctx->fail(TFA_ERR_PARAM, "nct must be >= 1");
    RC(require_keys(ctx));
    const int L = inv ? 4 : 3, nb = nblocks_per_byte(ctx);
    const size_t w = (size_t)nct * ctx->byte_words();
    RC(ws_reserve(ctx, many_wopbs_scratch(ctx, nct, nb, L * nb, tfa_lut_size(&ctx->p, nb)) + (1 + L) * w * 8));
    WSB(d_in, u64, w); WSB(d_out, u64, w * L);
    H2D(d_in, bytes_in, w);
    RC(sbox_like_dev(ctx, d_in, nct, inv ? 3 : 1, d_out));
    D2H(out, d_out, w * L);
    SYNC();
    return TFA_OK;
}

// ------------------------------------------------------------------------------------------------
// linear layers as gather-sum tables (K7).  ShiftRows: new[r+4c] = old[r+4((c+r)%4)] (shift_rows.rs:9-20);
// inverse: new[r+4c] = old[r+4((c-r)%4)] (inv_shift_rows.rs:9-20).
// ------------------------------------------------------------------------------------------------
static inline int sr(int i) { int r = i & 3, c = i >> 2; return r + 4 * ((c + r) & 3); }
static inline int isr(int i) { int r = i & 3, c = i >> 2; return r + 4 * ((c - r) & 3); }

static SumEntry entry(u64 *dst, std::initializer_list<const u64 *> srcs) {
    SumEntry e{};
    e.dst = dst; e.nsrc = 0;
    for (auto s : srcs) e.src[e.nsrc++] = s;
    return e;
}
// the same round key for each of nblk blocks
static std::vector<const u64 *> same_rk(const u64 *rk, int nblk) { return std::vector<const u64 *>((size_t)nblk, rk); }
// state[b][i] += rk[b][i]                                                     (server.rs:278-282)
static int lin_add_round_key(tfa_ctx *ctx, u64 *state, const u64 *const *rk, int nblk) {
    const size_t bw = ctx->byte_words();
    std::vector<SumEntry> v;
    for (int b = 0; b < nblk; b++) for (int i = 0; i < 16; i++) {
        u64 *s = state + ((size_t)b * 16 + i) * bw;
        v.push_back(entry(s, {s, rk[b] + (size_t)i * bw}));
    }
    return dev_lwe_sum(ctx, v, (int)bw);
}
// state[b][4c+row] = MixColumns(ShiftRows(mul))[..] (+ rk[b])                 (mix_columns.rs:4-78)
// MIX_PICK[row][j] = which of {S,2S,3S} of shifted byte j of the column (mix_columns.rs:36-75)
static const int MIX_PICK[4][4] = {{1, 2, 0, 0}, {0, 1, 2, 0}, {0, 0, 1, 2}, {2, 0, 0, 1}};
static int lin_mix_columns(tfa_ctx *ctx, const u64 *mul, u64 *state, const u64 *const *rk, int nblk) {
    const size_t bw = ctx->byte_words();
    std::vector<SumEntry> v;
    for (int b = 0; b < nblk; b++) for (int col = 0; col < 4; col++) for (int row = 0; row < 4; row++) {
        SumEntry e{};
        e.dst = state + ((size_t)b * 16 + 4 * col + row) * bw;
        for (int j = 0; j < 4; j++) e.src[e.nsrc++] = mul + (((size_t)b * 16 + sr(4 * col + j)) * 3 + MIX_PICK[row][j]) * bw;
        if (rk) e.src[e.nsrc++] = rk[b] + (size_t)(4 * col + row) * bw;
        v.push_back(e);
    }
    return dev_lwe_sum(ctx, v, (int)bw);
}
// inv_mix_columns.rs:4-58 ([0]=9x [1]=11x [2]=13x [3]=14x)
static int lin_inv_mix_columns(tfa_ctx *ctx, const u64 *mul, u64 *state, int nblk) {
    const size_t bw = ctx->byte_words();
    std::vector<SumEntry> v;
    static const int pick[4][4] = {{3, 1, 2, 0}, {0, 3, 1, 2}, {2, 0, 3, 1}, {1, 2, 0, 3}};
    for (int b = 0; b < nblk; b++) for (int col = 0; col < 4; col++) for (int row = 0; row < 4; row++) {
        SumEntry e{};
        e.dst = state + ((size_t)b * 16 + 4 * col + row) * bw;
        for (int j = 0; j < 4; j++) e.src[e.nsrc++] = mul + (((size_t)b * 16 + 4 * col + j) * 4 + pick[row][j]) * bw;
        v.push_back(e);
    }
    return dev_lwe_sum(ctx, v, (int)bw);
}
// dst[b][i] = src[b][perm(i)] (+ rk[i]); src != dst
static int lin_permute_add(tfa_ctx *ctx, const u64 *src, u64 *dst, const u64 *rk, int nblk, int inverse) {
    const size_t bw = ctx->byte_words();
    std::vector<SumEntry> v;
    for (int b = 0; b < nblk; b++) for (int i = 0; i < 16; i++) {
        SumEntry e{};
        e.dst = dst + ((size_t)b * 16 + i) * bw;
        e.src[e.nsrc++] = src + ((size_t)b * 16 + (inverse ? isr(i) : sr(i))) * bw;
        if (rk) e.src[e.nsrc++] = rk + (size_t)i * bw;
        v.push_back(e);
    }
    return dev_lwe_sum(ctx, v, (int)bw);
}
// final ShiftRows + AddRoundKey + XOR with clear data in one pass: out[b][i] = mul[b][sr(i)] + rk[b][i], plus the clear byte
// data[b][i] when data[b] is non-null; mul != out
static int lin_final_round_xor(tfa_ctx *ctx, const u64 *mul, u64 *out, const u64 *const *rk, const uint8_t *const *data, int nblk) {
    const size_t bw = ctx->byte_words();
    std::vector<SumXorEntry> v;
    v.reserve((size_t)16 * nblk);
    for (int b = 0; b < nblk; b++) for (int i = 0; i < 16; i++) {
        SumXorEntry e{};
        e.dst = out + ((size_t)b * 16 + i) * bw;
        e.src[e.nsrc++] = mul + ((size_t)b * 16 + sr(i)) * bw;
        e.src[e.nsrc++] = rk[b] + (size_t)i * bw;
        e.clear_src = data[b] ? data[b] + i : nullptr;
        v.push_back(e);
    }
    return dev_lwe_sum_xor(ctx, v);
}

// ------------------------------------------------------------------------------------------------
// Server::aes_encrypt (server.rs:39-64), nblk states at once
// ------------------------------------------------------------------------------------------------
static size_t aes_scratch(const tfa_ctx *ctx, int nblk, int L) {
    const int nb = nblocks_per_byte(ctx);
    const size_t w = (size_t)nblk * 16 * ctx->byte_words() * 8;
    return many_wopbs_scratch(ctx, nblk * 16, nb, L * nb, tfa_lut_size(&ctx->p, nb)) * 2 + w * (L + 2) + (size_t)nblk * 16 * sizeof(SumEntry) * 4;
}
// rk_round[b]: round key of block b
static int aes_round_nolock(tfa_ctx *ctx, const u64 *const *rk_round, u64 *state, int nblk, u64 *mul) {
    RC(sbox_like_dev(ctx, state, nblk * 16, 1, mul));                      // server.rs:47-50 (many_sbox)
    return lin_mix_columns(ctx, mul, state, rk_round, nblk);               // server.rs:53-55
}
// nr = number of rounds: 10 (AES-128, the reference), 12 (AES-192), 14 (AES-256); rk holds nr + 1 round keys
static int aes_encrypt_nolock(tfa_ctx *ctx, const u64 *rk, u64 *state, int nblk, int nr = 10) {
    const size_t bw = ctx->byte_words(), rkw = 16 * bw;
    WSB(mul, u64, (size_t)nblk * 16 * 3 * bw);
    const size_t mark = ctx->ws_off;
    RC(lin_add_round_key(ctx, state, same_rk(rk, nblk).data(), nblk));     // server.rs:42
    for (int round = 1; round < nr; round++) {
        ctx->ws_off = mark;
        RC(aes_round_nolock(ctx, same_rk(rk + (size_t)round * rkw, nblk).data(), state, nblk, mul));
    }
    ctx->ws_off = mark;
    RC(sbox_like_dev(ctx, state, nblk * 16, 0, mul));                      // server.rs:59-61
    return lin_permute_add(ctx, mul, state, rk + (size_t)nr * rkw, nblk, 0);  // server.rs:62-63
}
// Server::aes_decrypt (server.rs:67-105)
static int aes_decrypt_nolock(tfa_ctx *ctx, const u64 *rk, u64 *state, int nblk, int nr = 10) {
    const size_t bw = ctx->byte_words(), rkw = 16 * bw;
    WSB(mul, u64, (size_t)nblk * 16 * 4 * bw);
    WSB(tmp, u64, (size_t)nblk * 16 * bw);
    const size_t mark = ctx->ws_off;
    RC(lin_add_round_key(ctx, state, same_rk(rk + (size_t)nr * rkw, nblk).data(), nblk));  // server.rs:70
    for (int round = nr; round >= 2; round--) {
        ctx->ws_off = mark;
        // inv_shift_rows commutes with the byte-wise S-box: S-box first, permutation fused with AddRoundKey
        RC(sbox_like_dev(ctx, state, nblk * 16, 2, mul));                  // server.rs:73-78
        RC(lin_permute_add(ctx, mul, tmp, rk + (size_t)(round - 1) * rkw, nblk, 1));  // server.rs:73,81
        ctx->ws_off = mark;
        RC(sbox_like_dev(ctx, tmp, nblk * 16, 3, mul));                    // server.rs:88-91
        RC(lin_inv_mix_columns(ctx, mul, state, nblk));                    // server.rs:94
    }
    ctx->ws_off = mark;
    RC(sbox_like_dev(ctx, state, nblk * 16, 2, mul));                      // server.rs:98-102
    return lin_permute_add(ctx, mul, state, rk, nblk, 1);                  // server.rs:98,104
}
// Server::aes_key_expansion (server.rs:107-167)
// nk = key words: 4 (AES-128, the reference), 6, 8 (FIPS-197 §5.2); every generated word is refreshed to noise level 1 as
// server.rs:149-150 does, and the extra SubWord of AES-256 (i mod 8 = 4) goes through the same S-box evaluation
static int key_expansion_nolock(tfa_ctx *ctx, const u64 *key_ct, const u64 *rcon_ct, u64 *rk, int nk = 4) {
    static const uint8_t RCON[10] = {0x01, 0x02, 0x04, 0x08, 0x10, 0x20, 0x40, 0x80, 0x1B, 0x36};  // key_expansion_utils.rs:10-12
    const size_t bw = ctx->byte_words();
    const int lw = ctx->lw;
    const int nwords = 4 * (nk + 6 + 1);
    CU(cudaMemcpyAsync(rk, key_ct, (size_t)4 * nk * bw * 8, cudaMemcpyDeviceToDevice, ctx->stream));  // server.rs:122-128
    WSB(rcon, u64, 10 * bw);
    if (rcon_ct) CU(cudaMemcpyAsync(rcon, rcon_ct, 10 * bw * 8, cudaMemcpyDeviceToDevice, ctx->stream));
    else {
        // trivial encryption of RCON (decrypts identically to server.rs:139-140's public-key encryption)
        std::vector<u64> h(10 * bw, 0);
        for (int r = 0; r < 10; r++) for (int j = 0; j < 8; j++) h[((size_t)r * 8 + j) * lw + lw - 1] = (u64)((RCON[r] >> j) & 1) << 63;
        CU(cudaMemcpyAsync(rcon, h.data(), h.size() * 8, cudaMemcpyHostToDevice, ctx->stream));
    }
    WSB(temp, u64, 4 * bw); WSB(sub, u64, 4 * bw); WSB(sum, u64, 4 * bw);
    const size_t mark = ctx->ws_off;
    auto W = [&](int i, int j) { return rk + ((size_t)i * 4 + j) * bw; };  // word i, byte j (flat = round-key layout)
    for (int i = nk; i < nwords; i++) {
        ctx->ws_off = mark;
        const u64 *t[4];
        if (nk > 6 && i % nk == 4) {
            std::vector<SumEntry> v;  // AES-256 only: temp = SubWord(w[i-1])
            for (int j = 0; j < 4; j++) v.push_back(entry(temp + (size_t)j * bw, {W(i - 1, j)}));
            RC(dev_lwe_sum(ctx, v, (int)bw));
            RC(sbox_like_dev(ctx, temp, 4, 0, sub));
            for (int j = 0; j < 4; j++) t[j] = sub + (size_t)j * bw;
        } else if (i % nk == 0) {
            std::vector<SumEntry> v;  // fhe_rot_word: temp[j] = w[i-1][(j+1)%4]
            for (int j = 0; j < 4; j++) v.push_back(entry(temp + (size_t)j * bw, {W(i - 1, (j + 1) % 4)}));
            RC(dev_lwe_sum(ctx, v, (int)bw));
            RC(sbox_like_dev(ctx, temp, 4, 0, sub));                        // fhe_sub_word
            std::vector<SumEntry> a{entry(sub, {sub, rcon + (size_t)(i / nk - 1) * bw})};  // server.rs:143
            RC(dev_lwe_sum(ctx, a, (int)bw));
            for (int j = 0; j < 4; j++) t[j] = sub + (size_t)j * bw;
        } else {
            for (int j = 0; j < 4; j++) t[j] = W(i - 1, j);
        }
        std::vector<SumEntry> v;
        for (int j = 0; j < 4; j++) v.push_back(entry(sum + (size_t)j * bw, {W(i - nk, j), t[j]}));  // server.rs:148
        RC(dev_lwe_sum(ctx, v, (int)bw));
        RC(sbox_like_dev(ctx, sum, 4, 4, W(i, 0)));                         // refresh, server.rs:150
    }
    return TFA_OK;
}
// Server::add_scalar (server.rs:172-275), all blocks stage by stage.  counters: device [nblk][2] (lo, hi)
static int add_scalar_nolock(tfa_ctx *ctx, u64 *state, const u64 *ctr_dev, int nblk) {
    if (nblocks_per_byte(ctx) != 8) return ctx->fail(TFA_ERR_UNSUPPORTED, "add_scalar needs 1-bit blocks (client.rs:53-54)");
    const size_t bw = ctx->byte_words();
    const int lw = ctx->lw;
    WSB(ns, u64, (size_t)nblk * 16 * bw);
    WSB(in9, u64, (size_t)nblk * 9 * lw);
    WSB(out9, u64, (size_t)nblk * 9 * lw);
    WSB(luts, u64, (size_t)nblk * 9 * 512);
    const size_t mark = ctx->ws_off;
    for (int stage = 0; stage < 16; stage++) {
        ctx->ws_off = mark;
        const int index = 15 - stage, nbits = stage == 0 ? 8 : 9;
        CU(launch_add_scalar_luts(ctr_dev, nblk, index, nbits, luts, ctx->stream));
        ctx->launches++;
        std::vector<SumEntry> v;
        for (int b = 0; b < nblk; b++) {  // gather the input radix: 8 bits of the byte (+ previous carry as block 8)
            for (int j = 0; j < 8; j++) v.push_back(entry(in9 + ((size_t)b * nbits + j) * lw, {state + ((size_t)b * 16 + index) * bw + (size_t)j * lw}));
            if (nbits == 9) v.push_back(entry(in9 + ((size_t)b * 9 + 8) * lw, {out9 + ((size_t)b * 9 + 8) * lw}));
        }
        RC(dev_lwe_sum(ctx, v, lw));
        // two LUTs per byte (sum, carry) for one circuit bootstrap; only the 8 sum bits and the carry
        // bit the reference reads back (server.rs:255-263) are evaluated
        RC(dev_many_wopbs(ctx, in9, nblk, nbits, luts, (size_t)9 * 512, 512, 9, 512, out9));
        v.clear();
        for (int b = 0; b < nblk; b++) for (int j = 0; j < 8; j++)
            v.push_back(entry(ns + ((size_t)b * 16 + index) * bw + (size_t)j * lw, {out9 + ((size_t)b * 9 + j) * lw}));
        RC(dev_lwe_sum(ctx, v, lw));
    }
    CU(cudaMemcpyAsync(state, ns, (size_t)nblk * 16 * bw * 8, cudaMemcpyDeviceToDevice, ctx->stream));
    return TFA_OK;
}
// Counter add of the CTR loop (main.rs:59-60: state = encrypted_iv.clone(); add_scalar(&mut state, i)) for nblk counters
// at once.  Every block starts from the SAME encrypted IV, so the 8 state bits of each stage are the same ciphertexts for
// all blocks: they are circuit-bootstrapped once (128 bits for the whole call) and their GGSWs are shared by the
// vertical packings of all blocks; per block and stage only the carry bit (block 8 of the 9-block radix of
// server.rs:216-222) goes through its own circuit bootstrap.  Per block 15 instead of 143 bootstraps; the outputs are the
// same functions of the same inputs (the LUTs, the selector order and the carry chain are those of add_scalar_nolock).
// Several IVs: iv_ct holds niv encrypted IVs side by side, all 128 * niv bits go through one circuit-bootstrap batch, and block b
// starts from IV blk_iv[b] (device [nblk]; nullptr when niv = 1): its vertical packings read that IV's GGSWs.
static int add_scalar_from_iv_nolock(tfa_ctx *ctx, const u64 *iv_ct, int niv, const int32_t *blk_iv, const u64 *ctr_dev, int nblk,
                                     u64 *states) {
    if (nblocks_per_byte(ctx) != 8) return ctx->fail(TFA_ERR_UNSUPPORTED, "add_scalar needs 1-bit blocks (client.rs:53-54)");
    const size_t bw = ctx->byte_words();
    const int lw = ctx->lw, np = ctx->n + 1, nbits_iv = 128 * niv;
    const size_t ggsw_words = (size_t)ctx->p.cbs_level * (ctx->k + 1) * ctx->gsz;
    // (1) the IV bits: extract (keyswitch), circuit bootstrap, Fourier — bit t of byte b of IV i at index 128*i + 8*b + t
    WSB(iv_bits, u64, (size_t)nbits_iv * np);
    WSB(iv_ggsw_std, u64, (size_t)nbits_iv * ggsw_words);
    WSB(iv_ggsw_f, double2, (size_t)nbits_iv * ggsw_words / 2);
    const int delta_log = 63;
    {
        const size_t mark0 = ctx->ws_off;
        RC(dev_extract_bits(ctx, iv_ct, nbits_iv, delta_log, 1, iv_bits));
        RC(dev_circuit_bootstrap(ctx, iv_bits, nbits_iv, iv_ggsw_std));
        RC(dev_fourier(ctx, iv_ggsw_std, (long)nbits_iv * ctx->p.cbs_level * (ctx->k + 1) * (ctx->k + 1), ctx->p.cbs_level, iv_ggsw_f));
        ctx->ws_off = mark0;
    }
    WSB(out9, u64, (size_t)nblk * 9 * lw);
    WSB(carry, u64, (size_t)nblk * lw);
    WSB(carry_bits, u64, (size_t)nblk * np);
    WSB(carry_ggsw_std, u64, (size_t)nblk * ggsw_words);
    WSB(carry_ggsw_f, double2, (size_t)nblk * ggsw_words / 2);
    WSB(luts, u64, (size_t)nblk * 9 * 512);
    const size_t mark = ctx->ws_off;
    for (int stage = 0; stage < 16; stage++) {
        ctx->ws_off = mark;
        const int index = 15 - stage, nbits = stage == 0 ? 8 : 9;
        CU(launch_add_scalar_luts(ctr_dev, nblk, index, nbits, luts, ctx->stream));
        ctx->launches++;
        if (stage > 0) {
            // the carry of the previous stage (output 8) is the 9th selector bit of this one
            std::vector<SumEntry> v;
            for (int b = 0; b < nblk; b++) v.push_back(entry(carry + (size_t)b * lw, {out9 + ((size_t)b * 9 + 8) * lw}));
            RC(dev_lwe_sum(ctx, v, lw));
            RC(dev_extract_bits(ctx, carry, nblk, delta_log, 1, carry_bits));
            RC(dev_circuit_bootstrap(ctx, carry_bits, nblk, carry_ggsw_std));
            RC(dev_fourier(ctx, carry_ggsw_std, (long)nblk * ctx->p.cbs_level * (ctx->k + 1) * (ctx->k + 1), ctx->p.cbs_level, carry_ggsw_f));
        }
        // the 8 sum bits and the carry bit the reference reads back (server.rs:255-263)
        RC(dev_vertical_packing(ctx, carry_ggsw_f, nblk, nbits, luts, (size_t)9 * 512, 512, 9, 512, out9,
                                iv_ggsw_f + (size_t)index * 8 * ggsw_words / 2, 8, blk_iv, (size_t)128 * ggsw_words / 2));
        std::vector<SumEntry> v;
        for (int b = 0; b < nblk; b++) for (int j = 0; j < 8; j++)
            v.push_back(entry(states + ((size_t)b * 16 + index) * bw + (size_t)j * lw, {out9 + ((size_t)b * 9 + j) * lw}));
        RC(dev_lwe_sum(ctx, v, lw));
    }
    return TFA_OK;
}
static size_t add_scalar_scratch(const tfa_ctx *ctx, int nblk, int niv = 1) {
    return many_wopbs_scratch(ctx, nblk, 9, 9, 512) + many_wopbs_scratch(ctx, 16 * niv, 8, 8, 512) +
           (size_t)nblk * (16 * ctx->byte_words() + 20 * ctx->lw + 9 * 512) * 8 + (size_t)nblk * 32 * sizeof(SumEntry) + (1 << 20);
}

// ---- device-pointer entry points -----------------------------------------------------------------
extern "C" int tfa_aes_encrypt_dev(tfa_ctx *ctx, const uint64_t *rk, uint64_t *states, int nblk) {
    Guard g(ctx);
    if (nblk < 1) return ctx->fail(TFA_ERR_PARAM, "nblk must be >= 1");
    RC(require_keys(ctx));
    RC(ws_reserve(ctx, aes_scratch(ctx, nblk, 3)));
    return aes_encrypt_nolock(ctx, rk, states, nblk);
}
extern "C" int tfa_aes_decrypt_dev(tfa_ctx *ctx, const uint64_t *rk, uint64_t *states, int nblk) {
    Guard g(ctx);
    if (nblk < 1) return ctx->fail(TFA_ERR_PARAM, "nblk must be >= 1");
    RC(require_keys(ctx));
    RC(ws_reserve(ctx, aes_scratch(ctx, nblk, 5)));
    return aes_decrypt_nolock(ctx, rk, states, nblk);
}
extern "C" int tfa_aes_round_dev(tfa_ctx *ctx, const uint64_t *rk_round, uint64_t *states, int nblk) {
    Guard g(ctx);
    if (nblk < 1) return ctx->fail(TFA_ERR_PARAM, "nblk must be >= 1");
    RC(require_keys(ctx));
    RC(ws_reserve(ctx, aes_scratch(ctx, nblk, 3)));
    WSB(mul, u64, (size_t)nblk * 16 * 3 * ctx->byte_words());
    return aes_round_nolock(ctx, same_rk(rk_round, nblk).data(), states, nblk, mul);
}
extern "C" int tfa_add_scalar_dev(tfa_ctx *ctx, uint64_t *states, const uint64_t *ctr_dev, int nblk) {
    Guard g(ctx);
    if (nblk < 1) return ctx->fail(TFA_ERR_PARAM, "nblk must be >= 1");
    RC(require_keys(ctx));
    RC(ws_reserve(ctx, add_scalar_scratch(ctx, nblk)));
    return add_scalar_nolock(ctx, states, ctr_dev, nblk);
}
extern "C" int tfa_aes_key_expansion_dev(tfa_ctx *ctx, const uint64_t *key_ct, const uint64_t *rcon_ct, uint64_t *rk) {
    Guard g(ctx);
    RC(require_keys(ctx));
    RC(ws_reserve(ctx, aes_scratch(ctx, 1, 1) + 32 * ctx->byte_words() * 8));
    return key_expansion_nolock(ctx, key_ct, rcon_ct, rk);
}
static int aes_ctr_nolock(tfa_ctx *ctx, const u64 *rk, const u64 *iv_ct, u64 first_lo, u64 first_hi, int nblk, u64 *out) {
    // main.rs:55-64: state = encrypted_iv.clone(); add_scalar(i); aes_encrypt
    const size_t sw = 16 * ctx->byte_words();
    std::vector<u64> ctr((size_t)nblk * 2);
    for (int b = 0; b < nblk; b++) {
        u64 lo = first_lo + (u64)b;
        ctr[2 * b] = lo; ctr[2 * b + 1] = first_hi + (lo < first_lo ? 1 : 0);
    }
    WSB(d_ctr, u64, ctr.size());
    CU(cudaMemcpyAsync(d_ctr, ctr.data(), ctr.size() * 8, cudaMemcpyHostToDevice, ctx->stream));
    const size_t mark = ctx->ws_off;
    static const bool per_block = getenv("TFA_CTR_PER_BLOCK_ADD") != nullptr;   // the reference's schedule, for comparison
    if (per_block) {
        for (int b = 0; b < nblk; b++) CU(cudaMemcpyAsync(out + (size_t)b * sw, iv_ct, sw * 8, cudaMemcpyDeviceToDevice, ctx->stream));
        RC(add_scalar_nolock(ctx, out, d_ctr, nblk));
    } else {
        RC(add_scalar_from_iv_nolock(ctx, iv_ct, 1, nullptr, d_ctr, nblk, out));
    }
    ctx->ws_off = mark;
    return aes_encrypt_nolock(ctx, rk, out, nblk);
}
extern "C" int tfa_aes_ctr_dev(tfa_ctx *ctx, const uint64_t *rk, const uint64_t *iv_ct, uint64_t first_lo, uint64_t first_hi, int nblk, uint64_t *out) {
    Guard g(ctx);
    if (nblk < 1) return ctx->fail(TFA_ERR_PARAM, "nblk must be >= 1");
    RC(require_keys(ctx));
    size_t a = aes_scratch(ctx, nblk, 3), b = add_scalar_scratch(ctx, nblk);
    RC(ws_reserve(ctx, (a > b ? a : b) + (size_t)nblk * 16));
    return aes_ctr_nolock(ctx, rk, iv_ct, first_lo, first_hi, nblk, out);
}

// ---- AES-CTR with a public IV ------------------------------------------------------------------------------------
// The counter blocks are known in the clear, so no counter add is evaluated: round 0 is the round key XOR a clear block (body
// words only, lwe_sum_xor).  Consecutive counters that agree on bytes 0..14 (a run, at most 256 blocks) differ in byte 15 alone:
//   round 1: only S-box input 15 differs per block; ShiftRows moves it to column 0, so after MixColumns + AddRoundKey bytes 0..3
//            differ per block and bytes 4..15 are the same ciphertexts for the whole run;
//   round 2: S-boxes 0..3 per block, 4..15 per run; every output column mixes exactly one per-block product with three per-run
//            ones, so from round 3 on all 16 bytes are per block.
// S-box evaluations: 15 + 12 = 27 per run and 1 + 4 + 16 (Nr - 2) per block (133 for AES-128 instead of 160 + the counter add).
struct CtrPlan {
    int G = 0, B = 0;                  // runs, blocks
    std::vector<int> blk_run, blk_stream, blk_pos;   // run, stream and position in its stream of each block
    std::vector<uint8_t> blk_low;      // byte 15 of the counter block of each block
    std::vector<int> run_stream;
    std::vector<uint8_t> run_high;     // [G][15]: bytes 0..14 of the counter blocks of each run
};
static int plan_public_ctr(tfa_ctx *ctx, const tfa_ctr_stream *streams, int nstreams, int rounds, CtrPlan &p) {
    if (!streams || nstreams < 1) return ctx->fail(TFA_ERR_PARAM, "aes_ctr_public_iv: nstreams must be >= 1");
    if (rounds != 10 && rounds != 12 && rounds != 14) return ctx->fail(TFA_ERR_PARAM, "rounds must be 10, 12 or 14");
    long long total = 0;
    for (int s = 0; s < nstreams; s++) {
        if (streams[s].nblk < 1 || !streams[s].round_keys) return ctx->fail(TFA_ERR_PARAM, "aes_ctr_public_iv: every stream needs nblk >= 1 and round keys");
        total += streams[s].nblk;
    }
    // 16 encrypted bytes per block are indexed with int in the S-box batches
    if (total > INT_MAX / 16) return ctx->fail(TFA_ERR_PARAM, "aes_ctr_public_iv: too many blocks in one call");
    typedef unsigned __int128 u128;
    p.B = (int)total;
    for (int s = 0; s < nstreams; s++) {
        u128 c = 0;
        for (int i = 0; i < 16; i++) c = (c << 8) | streams[s].iv[i];
        c += ((u128)streams[s].first_hi << 64) | streams[s].first_lo;          // wraps mod 2^128
        for (int b = 0; b < streams[s].nblk; b++) {
            const u128 ctr = c + (u128)b;
            const uint8_t low = (uint8_t)ctr;
            if (b == 0 || low == 0) {                                          // a new run, also at the wrap to 0
                p.run_stream.push_back(s);
                for (int i = 0; i < 15; i++) p.run_high.push_back((uint8_t)(ctr >> (8 * (15 - i))));
                p.G++;
            }
            p.blk_run.push_back(p.G - 1); p.blk_stream.push_back(s); p.blk_pos.push_back(b); p.blk_low.push_back(low);
        }
    }
    return TFA_OK;
}
static size_t ctr_public_scratch(const tfa_ctx *ctx, int G, int B) {
    const int nb = nblocks_per_byte(ctx);
    const size_t n1 = (size_t)15 * G + B, n2 = (size_t)12 * G + (size_t)4 * B, n3 = (size_t)16 * B, bw8 = ctx->byte_words() * 8;
    const size_t nmax = std::max(n1, std::max(n2, n3));
    return many_wopbs_scratch(ctx, (int)nmax, nb, 3 * nb, tfa_lut_size(&ctx->p, nb)) * 2 + (n1 + n2) * 4 * bw8 + n3 * 3 * bw8 +
           nmax * sizeof(SumXorEntry) * 2;
}
// streams[s].round_keys / data: device pointers; out [B][16][8][lw] device, also the state of rounds 2 .. nr-1
static int aes_ctr_public_nolock(tfa_ctx *ctx, const tfa_ctr_stream *streams, const CtrPlan &p, int nr, u64 *out) {
    const size_t bw = ctx->byte_words(), rkw = 16 * bw;
    const int G = p.G, B = p.B, n1 = 15 * G + B, n2 = 12 * G + 4 * B;
    WSB(x1, u64, (size_t)n1 * bw);                // round-1 S-box inputs: [G][15] per run, then [B] (byte 15)
    WSB(m1, u64, (size_t)n1 * 3 * bw);
    WSB(x2, u64, (size_t)n2 * bw);                // round-2 S-box inputs: [G][12] per run (bytes 4..15), then [B][4] (bytes 0..3)
    WSB(m2, u64, (size_t)n2 * 3 * bw);
    WSB(mul, u64, (size_t)B * 16 * 3 * bw);
    const size_t mark = ctx->ws_off;
    auto rk_of = [&](int stream, int round, int byte) { return streams[stream].round_keys + (size_t)round * rkw + (size_t)byte * bw; };
    // (1) AddRoundKey with the clear counter block, then the round-1 S-boxes of all runs and blocks in one batch
    {
        std::vector<SumXorEntry> v;
        v.reserve(n1);
        for (int g = 0; g < G; g++) for (int i = 0; i < 15; i++) {
            SumXorEntry e{};
            e.dst = x1 + ((size_t)15 * g + i) * bw; e.src[e.nsrc++] = rk_of(p.run_stream[g], 0, i); e.clear = p.run_high[(size_t)15 * g + i];
            v.push_back(e);
        }
        for (int b = 0; b < B; b++) {
            SumXorEntry e{};
            e.dst = x1 + ((size_t)15 * G + b) * bw; e.src[e.nsrc++] = rk_of(p.blk_stream[b], 0, 15); e.clear = p.blk_low[b];
            v.push_back(e);
        }
        RC(dev_lwe_sum_xor(ctx, v));
        RC(sbox_like_dev(ctx, x1, n1, 1, m1));
    }
    // (2) round-1 MixColumns + AddRoundKey: columns 1..3 once per run, column 0 per block; then the round-2 S-boxes
    ctx->ws_off = mark;
    {
        // {S,2S,3S} of round-1 state byte i: per block for i = 15, per run otherwise
        auto s1 = [&](int g, int b, int i, int k) { return m1 + ((i == 15 ? (size_t)15 * G + b : (size_t)15 * g + i) * 3 + k) * bw; };
        std::vector<SumEntry> v;
        v.reserve(n2);
        for (int g = 0; g < G; g++) for (int col = 1; col < 4; col++) for (int row = 0; row < 4; row++) {
            SumEntry e{};
            e.dst = x2 + ((size_t)12 * g + 4 * col + row - 4) * bw;
            for (int j = 0; j < 4; j++) e.src[e.nsrc++] = s1(g, -1, sr(4 * col + j), MIX_PICK[row][j]);   // sr(4 col + j) != 15 for col > 0
            e.src[e.nsrc++] = rk_of(p.run_stream[g], 1, 4 * col + row);
            v.push_back(e);
        }
        for (int b = 0; b < B; b++) for (int row = 0; row < 4; row++) {
            SumEntry e{};
            e.dst = x2 + ((size_t)12 * G + (size_t)4 * b + row) * bw;
            for (int j = 0; j < 4; j++) e.src[e.nsrc++] = s1(p.blk_run[b], b, sr(j), MIX_PICK[row][j]);
            e.src[e.nsrc++] = rk_of(p.blk_stream[b], 1, row);
            v.push_back(e);
        }
        RC(dev_lwe_sum(ctx, v, (int)bw));
        RC(sbox_like_dev(ctx, x2, n2, 1, m2));
    }
    // (3) round-2 MixColumns + AddRoundKey: the full per-block state
    ctx->ws_off = mark;
    {
        auto s2 = [&](int g, int b, int i, int k) { return m2 + ((i < 4 ? (size_t)12 * G + (size_t)4 * b + i : (size_t)12 * g + i - 4) * 3 + k) * bw; };
        std::vector<SumEntry> v;
        v.reserve((size_t)16 * B);
        for (int b = 0; b < B; b++) for (int col = 0; col < 4; col++) for (int row = 0; row < 4; row++) {
            SumEntry e{};
            e.dst = out + ((size_t)b * 16 + 4 * col + row) * bw;
            for (int j = 0; j < 4; j++) e.src[e.nsrc++] = s2(p.blk_run[b], b, sr(4 * col + j), MIX_PICK[row][j]);
            e.src[e.nsrc++] = rk_of(p.blk_stream[b], 2, 4 * col + row);
            v.push_back(e);
        }
        RC(dev_lwe_sum(ctx, v, (int)bw));
    }
    // (4) rounds 3 .. nr-1 as aes_encrypt_nolock, with the round key of each block's stream
    std::vector<const u64 *> rkb((size_t)B);
    for (int round = 3; round < nr; round++) {
        ctx->ws_off = mark;
        for (int b = 0; b < B; b++) rkb[b] = rk_of(p.blk_stream[b], round, 0);
        RC(aes_round_nolock(ctx, rkb.data(), out, B, mul));
    }
    // (5) final round: S-box, then ShiftRows + AddRoundKey + XOR with the clear data in one pass
    ctx->ws_off = mark;
    RC(sbox_like_dev(ctx, out, B * 16, 0, mul));
    std::vector<const uint8_t *> data((size_t)B);
    for (int b = 0; b < B; b++) {
        const tfa_ctr_stream &st = streams[p.blk_stream[b]];
        rkb[b] = rk_of(p.blk_stream[b], nr, 0);
        data[b] = st.data ? st.data + (size_t)p.blk_pos[b] * 16 : nullptr;
    }
    return lin_final_round_xor(ctx, mul, out, rkb.data(), data.data(), B);
}
extern "C" int tfa_aes_ctr_public_iv_dev(tfa_ctx *ctx, const tfa_ctr_stream *streams, int nstreams, int rounds, uint64_t *out) {
    Guard g(ctx);
    CtrPlan p;
    RC(plan_public_ctr(ctx, streams, nstreams, rounds, p));
    if (!out) return ctx->fail(TFA_ERR_PARAM, "aes_ctr_public_iv: null output");
    RC(require_keys(ctx));
    if (nblocks_per_byte(ctx) != 8) return ctx->fail(TFA_ERR_UNSUPPORTED, "aes_ctr_public_iv needs 1-bit blocks (client.rs:53-54)");
    RC(ws_reserve(ctx, ctr_public_scratch(ctx, p.G, p.B)));
    return aes_ctr_public_nolock(ctx, streams, p, rounds, out);
}

// ---- AES-CTR with encrypted IVs, many streams in one call ---------------------------------------------------------
// aes_ctr_nolock for all blocks of all streams at once: the bits of every distinct IV are circuit-bootstrapped in one batch, each
// stage of the counter add runs over all blocks (one vertical packing per stage, each block reading the GGSWs of its own stream's
// IV), and the rounds take the round keys of each block's stream.  128 * (distinct IVs) + (128 * Nr + 15) * B PBS.
struct CtrEncPlan {
    int B = 0;                          // blocks
    std::vector<const u64 *> ivs;       // distinct iv_ct pointers, in order of first use
    std::vector<int32_t> blk_iv;        // index into ivs of each block
    std::vector<int> blk_stream, blk_pos;
    std::vector<u64> ctr;               // [B][2]: first + position of each block as (lo, hi), mod 2^128
};
static int plan_enc_ctr(tfa_ctx *ctx, const tfa_ctr_enc_stream *streams, int nstreams, int rounds, CtrEncPlan &p) {
    if (!streams || nstreams < 1) return ctx->fail(TFA_ERR_PARAM, "aes_ctr_streams: nstreams must be >= 1");
    if (rounds != 10 && rounds != 12 && rounds != 14) return ctx->fail(TFA_ERR_PARAM, "rounds must be 10, 12 or 14");
    long long total = 0;
    for (int s = 0; s < nstreams; s++) {
        if (streams[s].nblk < 1 || !streams[s].round_keys || !streams[s].iv_ct)
            return ctx->fail(TFA_ERR_PARAM, "aes_ctr_streams: every stream needs nblk >= 1, round keys and an encrypted IV");
        total += streams[s].nblk;
    }
    if (total > INT_MAX / 16) return ctx->fail(TFA_ERR_PARAM, "aes_ctr_streams: too many blocks in one call");
    p.B = (int)total;
    p.blk_iv.reserve(p.B); p.blk_stream.reserve(p.B); p.blk_pos.reserve(p.B); p.ctr.reserve((size_t)2 * p.B);
    for (int s = 0; s < nstreams; s++) {
        const tfa_ctr_enc_stream &st = streams[s];
        const int iv = (int)(std::find(p.ivs.begin(), p.ivs.end(), st.iv_ct) - p.ivs.begin());
        if (iv == (int)p.ivs.size()) p.ivs.push_back(st.iv_ct);
        for (int b = 0; b < st.nblk; b++) {
            const u64 lo = st.first_lo + (u64)b;
            p.blk_iv.push_back(iv); p.blk_stream.push_back(s); p.blk_pos.push_back(b);
            p.ctr.push_back(lo); p.ctr.push_back(st.first_hi + (lo < st.first_lo ? 1 : 0));
        }
    }
    return TFA_OK;
}
static size_t ctr_streams_scratch(const tfa_ctx *ctx, int niv, int B) {
    const size_t a = aes_scratch(ctx, B, 3), c = add_scalar_scratch(ctx, B, niv) + (size_t)niv * 16 * ctx->byte_words() * 8;
    return std::max(a, c) + (size_t)B * (16 + 4) + 1024;
}
// streams[s].round_keys / data: device pointers; p.ivs: host or device pointers (copied side by side first); out [B][16][8][lw] device
static int aes_ctr_streams_nolock(tfa_ctx *ctx, const tfa_ctr_enc_stream *streams, const CtrEncPlan &p, int nr, u64 *out) {
    const size_t bw = ctx->byte_words(), sw = 16 * bw, rkw = 16 * bw;
    const int B = p.B, niv = (int)p.ivs.size();
    WSB(d_ctr, u64, p.ctr.size());
    WSB(d_blk_iv, int32_t, (size_t)B);
    CU(cudaMemcpyAsync(d_ctr, p.ctr.data(), p.ctr.size() * 8, cudaMemcpyHostToDevice, ctx->stream));
    CU(cudaMemcpyAsync(d_blk_iv, p.blk_iv.data(), (size_t)B * sizeof(int32_t), cudaMemcpyHostToDevice, ctx->stream));
    const size_t mark = ctx->ws_off;
    {
        WSB(ivs, u64, (size_t)niv * sw);
        for (int i = 0; i < niv; i++) CU(cudaMemcpyAsync(ivs + (size_t)i * sw, p.ivs[i], sw * 8, cudaMemcpyDefault, ctx->stream));
        RC(add_scalar_from_iv_nolock(ctx, ivs, niv, d_blk_iv, d_ctr, B, out));
    }
    ctx->ws_off = mark;
    WSB(mul, u64, (size_t)B * 16 * 3 * bw);
    const size_t mark2 = ctx->ws_off;
    std::vector<const u64 *> rkb((size_t)B);
    auto round_keys = [&](int round) {
        for (int b = 0; b < B; b++) rkb[b] = streams[p.blk_stream[b]].round_keys + (size_t)round * rkw;
        return rkb.data();
    };
    RC(lin_add_round_key(ctx, out, round_keys(0), B));
    for (int round = 1; round < nr; round++) {
        ctx->ws_off = mark2;
        RC(aes_round_nolock(ctx, round_keys(round), out, B, mul));
    }
    ctx->ws_off = mark2;
    RC(sbox_like_dev(ctx, out, B * 16, 0, mul));
    std::vector<const uint8_t *> data((size_t)B);
    for (int b = 0; b < B; b++) {
        const tfa_ctr_enc_stream &st = streams[p.blk_stream[b]];
        data[b] = st.data ? st.data + (size_t)p.blk_pos[b] * 16 : nullptr;
    }
    return lin_final_round_xor(ctx, mul, out, round_keys(nr), data.data(), B);
}
extern "C" int tfa_aes_ctr_streams_dev(tfa_ctx *ctx, const tfa_ctr_enc_stream *streams, int nstreams, int rounds, uint64_t *out) {
    Guard g(ctx);
    CtrEncPlan p;
    RC(plan_enc_ctr(ctx, streams, nstreams, rounds, p));
    if (!out) return ctx->fail(TFA_ERR_PARAM, "aes_ctr_streams: null output");
    RC(require_keys(ctx));
    if (nblocks_per_byte(ctx) != 8) return ctx->fail(TFA_ERR_UNSUPPORTED, "aes_ctr_streams needs 1-bit blocks (client.rs:53-54)");
    RC(ws_reserve(ctx, ctr_streams_scratch(ctx, (int)p.ivs.size(), p.B)));
    return aes_ctr_streams_nolock(ctx, streams, p, rounds, out);
}

// ---- host-pointer entry points ---------------------------------------------------------------------
// ---- request coalescing ------------------------------------------------------------------------------
// The reference calls add_scalar + aes_encrypt once per block from rayon workers that share one &Server (main.rs:55-64).
// One block exposes 128 bootstraps per round, a B200 wants 444 per wave of the PBS kernel, so concurrent per-block calls
// are merged: every caller queues its request; the first one becomes the leader, lingers a fraction of a millisecond while
// further callers arrive, runs all compatible requests (same operation, same round keys) as ONE batch and wakes the others.
// Blocks are independent, so each caller gets exactly what its own call would have produced.
enum { OP_ENCRYPT = 0, OP_DECRYPT = 1, OP_ADD_SCALAR = 2 };
struct CoalesceReq {
    int op;
    const u64 *rk;
    u64 *states;
    const u64 *counters;
    int nblk;
    int rc;
    bool done;
};
// round keys of two callers: the same buffer, or equal on 1 024 words sampled across the 23 MB (every caller of the Rust shim
// flattens its own copy; honest ciphertexts that agree on 1 024 random-looking words are the same ciphertexts)
static bool same_round_keys(const tfa_ctx *ctx, const u64 *a, const u64 *b) {
    if (a == b) return true;
    const size_t rkw = (size_t)11 * 16 * ctx->byte_words(), stride = rkw / 1024;
    for (size_t i = 0; i < 1024; i++)
        if (a[i * stride + (i & 7)] != b[i * stride + (i & 7)]) return false;
    return true;
}
static int run_batch(tfa_ctx *ctx, const std::vector<CoalesceReq *> &batch) {
    Guard g(ctx);
    RC(require_keys(ctx));
    int nblk = 0;
    for (auto r : batch) nblk += r->nblk;
    const int op = batch[0]->op;
    const size_t bw = ctx->byte_words(), sw = (size_t)nblk * 16 * bw, rkw = (size_t)11 * 16 * bw;
    const size_t scratch = op == OP_ADD_SCALAR ? add_scalar_scratch(ctx, nblk) + (size_t)nblk * 16 : aes_scratch(ctx, nblk, op == OP_ENCRYPT ? 3 : 5) + rkw * 8;
    RC(ws_reserve(ctx, scratch + sw * 8));
    WSB(d_st, u64, sw);
    size_t off = 0;
    for (auto r : batch) { H2D(d_st + off, r->states, (size_t)r->nblk * 16 * bw); off += (size_t)r->nblk * 16 * bw; }
    if (op == OP_ADD_SCALAR) {
        WSB(d_ctr, u64, (size_t)nblk * 2);
        size_t c = 0;
        for (auto r : batch) { H2D(d_ctr + c, r->counters, (size_t)r->nblk * 2); c += (size_t)r->nblk * 2; }
        RC(add_scalar_nolock(ctx, d_st, d_ctr, nblk));
    } else {
        WSB(d_rk, u64, rkw);
        H2D(d_rk, batch[0]->rk, rkw);
        if (op == OP_ENCRYPT) RC(aes_encrypt_nolock(ctx, d_rk, d_st, nblk));
        else RC(aes_decrypt_nolock(ctx, d_rk, d_st, nblk));
    }
    off = 0;
    for (auto r : batch) { D2H(r->states, d_st + off, (size_t)r->nblk * 16 * bw); off += (size_t)r->nblk * 16 * bw; }
    SYNC();
    return TFA_OK;
}
static int coalesced_call(tfa_ctx *ctx, int op, const u64 *rk, u64 *states, const u64 *counters, int nblk) {
    if (nblk < 1 || !states || (op == OP_ADD_SCALAR ? !counters : !rk)) return ctx->fail(TFA_ERR_PARAM, "nblk must be >= 1 and the pointers non-null");
    CoalesceReq me{op, rk, states, counters, nblk, TFA_OK, false};
    std::unique_lock<std::mutex> ql(ctx->qmu);
    ctx->queue.push_back(&me);
    ctx->qcv.notify_all();                                  // a lingering leader sees the arrival
    while (!me.done && ctx->leader) ctx->qcv.wait(ql);
    if (me.done) return me.rc;
    ctx->leader = true;
    while (!me.done) {
        // linger until no caller has arrived for 1 ms (at most 16 ms; the shortest AES call takes 200 ms at PARAM_OPT): threads
        // released together by the previous batch come back within a fraction of a millisecond of each other
        size_t seen = ctx->queue.size();
        for (int spin = 0; spin < 16; spin++) {
            ctx->qcv.wait_for(ql, std::chrono::microseconds(1000));
            if (ctx->queue.size() == seen) break;
            seen = ctx->queue.size();
        }
        // the batch: every queued request compatible with the oldest one, up to 1 024 blocks
        std::vector<CoalesceReq *> batch, rest;
        CoalesceReq *head = ctx->queue.front();
        int blocks = 0;
        for (auto r : ctx->queue) {
            const bool ok = r == head || (r->op == head->op && blocks + r->nblk <= 1024 && (head->op == OP_ADD_SCALAR || same_round_keys(ctx, head->rk, r->rk)));
            if (ok) { batch.push_back(r); blocks += r->nblk; } else rest.push_back(r);
        }
        ctx->queue.swap(rest);
        ql.unlock();
        const int rc = run_batch(ctx, batch);
        ql.lock();
        for (auto r : batch) { r->rc = rc; r->done = true; }
        ctx->qcv.notify_all();
    }
    ctx->leader = false;                                    // whoever is still queued elects the next leader
    ctx->qcv.notify_all();
    return me.rc;
}

extern "C" int tfa_aes_encrypt(tfa_ctx *ctx, const uint64_t *round_keys, uint64_t *states, int nblk) {
    return coalesced_call(ctx, OP_ENCRYPT, round_keys, states, nullptr, nblk);
}
extern "C" int tfa_aes_decrypt(tfa_ctx *ctx, const uint64_t *round_keys, uint64_t *states, int nblk) {
    return coalesced_call(ctx, OP_DECRYPT, round_keys, states, nullptr, nblk);
}
extern "C" int tfa_aes_encryption(tfa_ctx *ctx, const uint64_t *rk, uint64_t *st, int nblk) { return tfa_aes_encrypt(ctx, rk, st, nblk); }
extern "C" int tfa_aes_decryption(tfa_ctx *ctx, const uint64_t *rk, uint64_t *st, int nblk) { return tfa_aes_decrypt(ctx, rk, st, nblk); }

extern "C" int tfa_aes_round(tfa_ctx *ctx, const uint64_t *round_key, uint64_t *states, int nblk) {
    Guard g(ctx);
    if (nblk < 1) return ctx->fail(TFA_ERR_PARAM, "nblk must be >= 1");
    RC(require_keys(ctx));
    const size_t bw = ctx->byte_words(), sw = (size_t)nblk * 16 * bw;
    RC(ws_reserve(ctx, aes_scratch(ctx, nblk, 3) + (sw + 16 * bw) * 8));
    WSB(d_rk, u64, 16 * bw); WSB(d_st, u64, sw); WSB(mul, u64, sw * 3);
    H2D(d_rk, round_key, 16 * bw); H2D(d_st, states, sw);
    RC(aes_round_nolock(ctx, same_rk(d_rk, nblk).data(), d_st, nblk, mul));
    D2H(states, d_st, sw);
    SYNC();
    return TFA_OK;
}
// AES-128 / 192 / 256 (SURVEY §8f.4): key_bytes = 16, 24 or 32; rk_out holds key_bytes / 4 + 7 round keys
extern "C" int tfa_aes_key_expansion_ex(tfa_ctx *ctx, const uint64_t *key_ct, int key_bytes, const uint64_t *rcon_ct, uint64_t *rk_out) {
    Guard g(ctx);
    RC(require_keys(ctx));
    if (key_bytes != 16 && key_bytes != 24 && key_bytes != 32) return ctx->fail(TFA_ERR_PARAM, "key_bytes must be 16, 24 or 32");
    const int nk = key_bytes / 4, nrk = nk + 7;
    const size_t bw = ctx->byte_words();
    RC(ws_reserve(ctx, aes_scratch(ctx, 1, 1) + ((size_t)key_bytes + 10 + 16 * nrk + 32) * bw * 8));
    WSB(d_key, u64, (size_t)key_bytes * bw); WSB(d_rk, u64, (size_t)16 * nrk * bw);
    u64 *d_rcon = nullptr;
    H2D(d_key, key_ct, (size_t)key_bytes * bw);
    if (rcon_ct) { d_rcon = ws_get<u64>(ctx, 10 * bw); if (!d_rcon) return TFA_ERR_STATE; H2D(d_rcon, rcon_ct, 10 * bw); }
    RC(key_expansion_nolock(ctx, d_key, d_rcon, d_rk, nk));
    D2H(rk_out, d_rk, (size_t)16 * nrk * bw);
    SYNC();
    return TFA_OK;
}
extern "C" int tfa_aes_key_expansion(tfa_ctx *ctx, const uint64_t *key_ct, const uint64_t *rcon_ct, uint64_t *rk_out) {
    return tfa_aes_key_expansion_ex(ctx, key_ct, 16, rcon_ct, rk_out);
}
// rounds = 10, 12 or 14; round_keys [rounds + 1][16][8][lw]; states in place
static int aes_crypt_ex(tfa_ctx *ctx, const uint64_t *round_keys, uint64_t *states, int nblk, int rounds, bool decrypt) {
    Guard g(ctx);
    if (nblk < 1 || !round_keys || !states) return ctx->fail(TFA_ERR_PARAM, "nblk must be >= 1 and the pointers non-null");
    if (rounds != 10 && rounds != 12 && rounds != 14) return ctx->fail(TFA_ERR_PARAM, "rounds must be 10, 12 or 14");
    RC(require_keys(ctx));
    const size_t sw = (size_t)nblk * 16 * ctx->byte_words(), rkw = (size_t)(rounds + 1) * 16 * ctx->byte_words();
    RC(ws_reserve(ctx, aes_scratch(ctx, nblk, decrypt ? 5 : 3) + (sw + rkw) * 8));
    WSB(d_rk, u64, rkw); WSB(d_st, u64, sw);
    H2D(d_rk, round_keys, rkw); H2D(d_st, states, sw);
    if (decrypt) RC(aes_decrypt_nolock(ctx, d_rk, d_st, nblk, rounds));
    else RC(aes_encrypt_nolock(ctx, d_rk, d_st, nblk, rounds));
    D2H(states, d_st, sw);
    SYNC();
    return TFA_OK;
}
extern "C" int tfa_aes_encrypt_ex(tfa_ctx *ctx, const uint64_t *round_keys, uint64_t *states, int nblk, int rounds) {
    return aes_crypt_ex(ctx, round_keys, states, nblk, rounds, false);
}
extern "C" int tfa_aes_decrypt_ex(tfa_ctx *ctx, const uint64_t *round_keys, uint64_t *states, int nblk, int rounds) {
    return aes_crypt_ex(ctx, round_keys, states, nblk, rounds, true);
}
extern "C" int tfa_add_scalar(tfa_ctx *ctx, uint64_t *states, const uint64_t *counters, int nblk) {
    return coalesced_call(ctx, OP_ADD_SCALAR, nullptr, states, counters, nblk);
}
extern "C" int tfa_aes_ctr(tfa_ctx *ctx, const uint64_t *round_keys, const uint64_t *iv_ct, uint64_t first_lo, uint64_t first_hi, int nblk, uint64_t *out) {
    Guard g(ctx);
    if (nblk < 1) return ctx->fail(TFA_ERR_PARAM, "nblk must be >= 1");
    RC(require_keys(ctx));
    const size_t bw = ctx->byte_words(), sw = (size_t)nblk * 16 * bw, rkw = 176 * bw;
    size_t a = aes_scratch(ctx, nblk, 3), b = add_scalar_scratch(ctx, nblk);
    RC(ws_reserve(ctx, (a > b ? a : b) + (sw + rkw + 16 * bw) * 8 + (size_t)nblk * 16));
    WSB(d_rk, u64, rkw); WSB(d_iv, u64, 16 * bw); WSB(d_out, u64, sw);
    H2D(d_rk, round_keys, rkw); H2D(d_iv, iv_ct, 16 * bw);
    RC(aes_ctr_nolock(ctx, d_rk, d_iv, first_lo, first_hi, nblk, d_out));
    D2H(out, d_out, sw);
    SYNC();
    return TFA_OK;
}
extern "C" int tfa_aes_ctr_public_iv(tfa_ctx *ctx, const tfa_ctr_stream *streams, int nstreams, int rounds, uint64_t *out) {
    Guard g(ctx);
    CtrPlan p;
    RC(plan_public_ctr(ctx, streams, nstreams, rounds, p));
    if (!out) return ctx->fail(TFA_ERR_PARAM, "aes_ctr_public_iv: null output");
    RC(require_keys(ctx));
    if (nblocks_per_byte(ctx) != 8) return ctx->fail(TFA_ERR_UNSUPPORTED, "aes_ctr_public_iv needs 1-bit blocks (client.rs:53-54)");
    const size_t bw = ctx->byte_words(), rkw = (size_t)(rounds + 1) * 16 * bw, sw = (size_t)p.B * 16 * bw;
    std::vector<const u64 *> keys;                       // distinct round-key buffers: streams under one AES key upload it once
    for (int s = 0; s < nstreams; s++)
        if (std::find(keys.begin(), keys.end(), streams[s].round_keys) == keys.end()) keys.push_back(streams[s].round_keys);
    RC(ws_reserve(ctx, ctr_public_scratch(ctx, p.G, p.B) + (keys.size() * rkw + sw) * 8 + (size_t)p.B * 16 + 256 * (keys.size() + 2)));
    WSB(d_out, u64, sw);
    WSB(d_data, uint8_t, (size_t)p.B * 16);
    std::vector<u64 *> d_keys;
    for (auto k : keys) {
        WSB(d, u64, rkw);
        H2D(d, k, rkw);
        d_keys.push_back(d);
    }
    std::vector<tfa_ctr_stream> dev(streams, streams + nstreams);
    size_t off = 0;
    for (int s = 0; s < nstreams; s++) {
        dev[s].round_keys = d_keys[std::find(keys.begin(), keys.end(), streams[s].round_keys) - keys.begin()];
        if (streams[s].data) {
            CU(cudaMemcpyAsync(d_data + off, streams[s].data, (size_t)streams[s].nblk * 16, cudaMemcpyHostToDevice, ctx->stream));
            dev[s].data = d_data + off;
        }
        off += (size_t)streams[s].nblk * 16;
    }
    RC(aes_ctr_public_nolock(ctx, dev.data(), p, rounds, d_out));
    D2H(out, d_out, sw);
    SYNC();
    return TFA_OK;
}
extern "C" int tfa_aes_ctr_streams(tfa_ctx *ctx, const tfa_ctr_enc_stream *streams, int nstreams, int rounds, uint64_t *out) {
    Guard g(ctx);
    CtrEncPlan p;
    RC(plan_enc_ctr(ctx, streams, nstreams, rounds, p));
    if (!out) return ctx->fail(TFA_ERR_PARAM, "aes_ctr_streams: null output");
    RC(require_keys(ctx));
    if (nblocks_per_byte(ctx) != 8) return ctx->fail(TFA_ERR_UNSUPPORTED, "aes_ctr_streams needs 1-bit blocks (client.rs:53-54)");
    const size_t bw = ctx->byte_words(), rkw = (size_t)(rounds + 1) * 16 * bw, sw = (size_t)p.B * 16 * bw;
    std::vector<const u64 *> keys;                       // distinct round-key buffers: streams under one AES key upload it once
    for (int s = 0; s < nstreams; s++)
        if (std::find(keys.begin(), keys.end(), streams[s].round_keys) == keys.end()) keys.push_back(streams[s].round_keys);
    RC(ws_reserve(ctx, ctr_streams_scratch(ctx, (int)p.ivs.size(), p.B) + (keys.size() * rkw + sw) * 8 + (size_t)p.B * 16 +
                           256 * (keys.size() + 2)));
    WSB(d_out, u64, sw);
    WSB(d_data, uint8_t, (size_t)p.B * 16);
    std::vector<u64 *> d_keys;
    for (auto k : keys) {
        WSB(d, u64, rkw);
        H2D(d, k, rkw);
        d_keys.push_back(d);
    }
    std::vector<tfa_ctr_enc_stream> dev(streams, streams + nstreams);
    size_t off = 0;
    for (int s = 0; s < nstreams; s++) {
        dev[s].round_keys = d_keys[std::find(keys.begin(), keys.end(), streams[s].round_keys) - keys.begin()];
        if (streams[s].data) {
            CU(cudaMemcpyAsync(d_data + off, streams[s].data, (size_t)streams[s].nblk * 16, cudaMemcpyHostToDevice, ctx->stream));
            dev[s].data = d_data + off;
        }
        off += (size_t)streams[s].nblk * 16;
    }
    // the distinct IVs (host pointers in p.ivs) are copied to the device once each by aes_ctr_streams_nolock
    RC(aes_ctr_streams_nolock(ctx, dev.data(), p, rounds, d_out));
    D2H(out, d_out, sw);
    SYNC();
    return TFA_OK;
}
// ---- GLWE packing of LWE ciphertexts (see the header) ---------------------------------------------------------------
static int pack_args(tfa_ctx *ctx, const void *in, int count, const void *out, const char *what) {
    if (!in || !out) return ctx->fail(TFA_ERR_PARAM, std::string(what) + ": null pointer");
    // the packed batch holds ceil(count / N) * N coefficient slots, counted in int
    if (count < 1 || count > INT_MAX - (ctx->N - 1)) return ctx->fail(TFA_ERR_PARAM, std::string(what) + ": count must be in [1, INT_MAX - N + 1]");
    return TFA_OK;
}
static size_t packed_words(const tfa_ctx *ctx, int count) { return (size_t)((count + ctx->N - 1) / ctx->N) * ctx->gsz; }
extern "C" int tfa_pack_lwe_dev(tfa_ctx *ctx, const uint64_t *lwe, int count, uint16_t *packed) {
    Guard g(ctx);
    RC(pack_args(ctx, lwe, count, packed, "pack_lwe"));
    RC(require_keys(ctx));
    RC(ws_reserve(ctx, pack_lwe_scratch(ctx, count)));
    return dev_pack_lwe(ctx, lwe, count, packed);
}
extern "C" int tfa_pack_lwe(tfa_ctx *ctx, const uint64_t *lwe, int count, uint16_t *packed) {
    Guard g(ctx);
    RC(pack_args(ctx, lwe, count, packed, "pack_lwe"));
    RC(require_keys(ctx));
    const size_t iw = (size_t)count * ctx->lw, pw = packed_words(ctx, count);
    RC(ws_reserve(ctx, pack_lwe_scratch(ctx, count) + iw * 8 + pw * 2 + 512));
    WSB(d_in, u64, iw); WSB(d_packed, uint16_t, pw);
    H2D(d_in, lwe, iw);
    RC(dev_pack_lwe(ctx, d_in, count, d_packed));
    CU(cudaMemcpyAsync(packed, d_packed, pw * 2, cudaMemcpyDeviceToHost, ctx->stream));
    SYNC();
    return TFA_OK;
}
extern "C" int tfa_unpack_lwe_dev(tfa_ctx *ctx, const uint16_t *packed, int count, uint64_t *lwe_out) {
    Guard g(ctx);
    RC(pack_args(ctx, packed, count, lwe_out, "unpack_lwe"));
    return dev_unpack_lwe(ctx, packed, count, lwe_out);
}
extern "C" int tfa_unpack_lwe(tfa_ctx *ctx, const uint16_t *packed, int count, uint64_t *lwe_out) {
    Guard g(ctx);
    RC(pack_args(ctx, packed, count, lwe_out, "unpack_lwe"));
    const size_t ow = (size_t)count * ctx->lw, pw = packed_words(ctx, count);
    RC(ws_reserve(ctx, ow * 8 + pw * 2 + 512));
    WSB(d_packed, uint16_t, pw); WSB(d_out, u64, ow);
    CU(cudaMemcpyAsync(d_packed, packed, pw * 2, cudaMemcpyHostToDevice, ctx->stream));
    RC(dev_unpack_lwe(ctx, d_packed, count, d_out));
    D2H(lwe_out, d_out, ow);
    SYNC();
    return TFA_OK;
}

// transciphering step: states ^= clear data (see the header)
extern "C" int tfa_xor_clear_dev(tfa_ctx *ctx, uint64_t *states, const uint8_t *data_dev, int nblk) {
    Guard g(ctx);
    if (nblk < 1 || !states || !data_dev) return ctx->fail(TFA_ERR_PARAM, "xor_clear: bad arguments");
    if (nblocks_per_byte(ctx) != 8) return ctx->fail(TFA_ERR_UNSUPPORTED, "xor_clear needs 1-bit blocks (client.rs:53-54)");
    CU(launch_xor_clear(states, data_dev, ctx->lw, (long)nblk * 128, ctx->stream));
    ctx->launches++;
    return TFA_OK;
}
extern "C" int tfa_xor_clear(tfa_ctx *ctx, uint64_t *states, const uint8_t *data, int nblk) {
    Guard g(ctx);
    if (nblk < 1 || !states || !data) return ctx->fail(TFA_ERR_PARAM, "xor_clear: bad arguments");
    if (nblocks_per_byte(ctx) != 8) return ctx->fail(TFA_ERR_UNSUPPORTED, "xor_clear needs 1-bit blocks (client.rs:53-54)");
    const size_t sw = (size_t)nblk * 16 * ctx->byte_words();
    RC(ws_reserve(ctx, sw * 8 + (size_t)nblk * 16 + 512));
    WSB(d_st, u64, sw); WSB(d_data, uint8_t, (size_t)nblk * 16);
    H2D(d_st, states, sw);
    CU(cudaMemcpyAsync(d_data, data, (size_t)nblk * 16, cudaMemcpyHostToDevice, ctx->stream));
    CU(launch_xor_clear(d_st, d_data, ctx->lw, (long)nblk * 128, ctx->stream));
    ctx->launches++;
    D2H(states, d_st, sw);
    SYNC();
    return TFA_OK;
}
// linear layers alone
extern "C" int tfa_add_round_key(tfa_ctx *ctx, uint64_t *states, const uint64_t *round_key, int nblk) {
    Guard g(ctx);
    if (nblk < 1) return ctx->fail(TFA_ERR_PARAM, "nblk must be >= 1");
    const size_t bw = ctx->byte_words(), sw = (size_t)nblk * 16 * bw;
    RC(ws_reserve(ctx, (sw + 16 * bw) * 8 + (size_t)nblk * 16 * sizeof(SumEntry)));
    WSB(d_st, u64, sw); WSB(d_rk, u64, 16 * bw);
    H2D(d_st, states, sw); H2D(d_rk, round_key, 16 * bw);
    RC(lin_add_round_key(ctx, d_st, same_rk(d_rk, nblk).data(), nblk));
    D2H(states, d_st, sw);
    SYNC();
    return TFA_OK;
}
extern "C" int tfa_mix_columns(tfa_ctx *ctx, const uint64_t *mul, uint64_t *states_out, int nblk) {
    Guard g(ctx);
    if (nblk < 1) return ctx->fail(TFA_ERR_PARAM, "nblk must be >= 1");
    const size_t bw = ctx->byte_words(), sw = (size_t)nblk * 16 * bw;
    RC(ws_reserve(ctx, sw * 4 * 8 + (size_t)nblk * 16 * sizeof(SumEntry)));
    WSB(d_mul, u64, sw * 3); WSB(d_st, u64, sw);
    H2D(d_mul, mul, sw * 3);
    RC(lin_mix_columns(ctx, d_mul, d_st, nullptr, nblk));
    D2H(states_out, d_st, sw);
    SYNC();
    return TFA_OK;
}
extern "C" int tfa_inv_mix_columns(tfa_ctx *ctx, const uint64_t *mul, uint64_t *states_out, int nblk) {
    Guard g(ctx);
    if (nblk < 1) return ctx->fail(TFA_ERR_PARAM, "nblk must be >= 1");
    const size_t bw = ctx->byte_words(), sw = (size_t)nblk * 16 * bw;
    RC(ws_reserve(ctx, sw * 5 * 8 + (size_t)nblk * 16 * sizeof(SumEntry)));
    WSB(d_mul, u64, sw * 4); WSB(d_st, u64, sw);
    H2D(d_mul, mul, sw * 4);
    RC(lin_inv_mix_columns(ctx, d_mul, d_st, nblk));
    D2H(states_out, d_st, sw);
    SYNC();
    return TFA_OK;
}
extern "C" int tfa_shift_rows(tfa_ctx *ctx, uint64_t *states, int nblk, int inverse) {
    Guard g(ctx);
    if (nblk < 1) return ctx->fail(TFA_ERR_PARAM, "nblk must be >= 1");
    const size_t bw = ctx->byte_words(), sw = (size_t)nblk * 16 * bw;
    RC(ws_reserve(ctx, sw * 2 * 8 + (size_t)nblk * 16 * sizeof(SumEntry)));
    WSB(d_in, u64, sw); WSB(d_out, u64, sw);
    H2D(d_in, states, sw);
    RC(lin_permute_add(ctx, d_in, d_out, nullptr, nblk, inverse));
    D2H(states, d_out, sw);
    SYNC();
    return TFA_OK;
}

// ---- primitives for parity tests ---------------------------------------------------------------------
extern "C" int tfa_keyswitch(tfa_ctx *ctx, const uint64_t *in, int count, uint64_t *out) {
    Guard g(ctx);
    if (count < 1) return ctx->fail(TFA_ERR_PARAM, "count must be >= 1");
    RC(require_keys(ctx));
    const size_t iw = (size_t)count * ctx->lw, ow = (size_t)count * (ctx->n + 1);
    RC(ws_reserve(ctx, (iw + ow) * 8 + (size_t)count * ctx->big * ctx->p.ks_level * 2));
    WSB(d_in, u64, iw); WSB(d_out, u64, ow);
    H2D(d_in, in, iw);
    RC(dev_keyswitch(ctx, d_in, count, d_out));
    D2H(out, d_out, ow);
    SYNC();
    return TFA_OK;
}
extern "C" int tfa_bootstrap(tfa_ctx *ctx, const uint64_t *in, int count, const uint64_t *lut, uint64_t *out) {
    Guard g(ctx);
    if (count < 1) return ctx->fail(TFA_ERR_PARAM, "count must be >= 1");
    RC(require_keys(ctx));
    const size_t iw = (size_t)count * (ctx->n + 1), ow = (size_t)count * ctx->lw;
    RC(ws_reserve(ctx, (iw + ow + ctx->N) * 8));
    WSB(d_in, u64, iw); WSB(d_out, u64, ow); WSB(d_lut, u64, ctx->N);
    H2D(d_in, in, iw); H2D(d_lut, lut, ctx->N);
    RC(dev_pbs(ctx, d_in, count, d_lut, 1, 0, 0, d_out));
    D2H(out, d_out, ow);
    SYNC();
    return TFA_OK;
}
extern "C" int tfa_bootstrap_dev(tfa_ctx *ctx, const uint64_t *in, int count, const uint64_t *lut, uint64_t pre_add_body,
                                 uint64_t post_add_body, uint64_t *out) {
    Guard g(ctx);
    if (count < 1) return ctx->fail(TFA_ERR_PARAM, "count must be >= 1");
    RC(require_keys(ctx));
    return dev_pbs(ctx, in, count, lut, 1, pre_add_body, post_add_body, out);
}
extern "C" int tfa_extract_bits(tfa_ctx *ctx, const uint64_t *in, int count, int delta_log, int nbits, uint64_t *out) {
    Guard g(ctx);
    if (count < 1) return ctx->fail(TFA_ERR_PARAM, "count must be >= 1");
    RC(require_keys(ctx));
    if (nbits < 1 || delta_log < 1 || delta_log + nbits > 64) return ctx->fail(TFA_ERR_PARAM, "extract_bits: bad delta_log / nbits");
    const int np = ctx->n + 1;
    const size_t iw = (size_t)count * ctx->lw, ow = (size_t)count * nbits * np;
    RC(ws_reserve(ctx, iw * 8 * 5 + ow * 8 * 2 + (size_t)count * ctx->big * ctx->p.ks_level * 2 * 2 + (1 << 20)));
    WSB(d_in, u64, iw); WSB(d_out, u64, ow);
    H2D(d_in, in, iw);
    RC(dev_extract_bits(ctx, d_in, count, delta_log, nbits, d_out));
    std::vector<u64> h(ow);
    D2H(h.data(), d_out, ow);
    SYNC();
    for (int c = 0; c < count; c++)  // reference order: index 0 = most significant extracted bit
        for (int b = 0; b < nbits; b++) memcpy(out + ((size_t)c * nbits + b) * np, &h[((size_t)c * nbits + (nbits - 1 - b)) * np], (size_t)np * 8);
    return TFA_OK;
}
extern "C" int tfa_pfks(tfa_ctx *ctx, int key_index, const uint64_t *in, int count, uint64_t *out) {
    Guard g(ctx);
    if (count < 1) return ctx->fail(TFA_ERR_PARAM, "count must be >= 1");
    RC(require_keys(ctx));
    if (key_index < 0 || key_index > ctx->k) return ctx->fail(TFA_ERR_PARAM, "pfks: bad key index");
    const int kp1 = ctx->k + 1;
    const size_t iw = (size_t)count * ctx->lw, ow = (size_t)count * kp1 * ctx->gsz;
    RC(ws_reserve(ctx, (iw + ow) * 8 + (size_t)count * (ctx->big + 1) * ctx->p.pfks_level * 2));
    WSB(d_in, u64, iw); WSB(d_out, u64, ow);
    H2D(d_in, in, iw);
    RC(dev_pfks(ctx, d_in, count, d_out, kp1 * ctx->gsz, 0, kp1));
    CU(cudaMemcpy2DAsync(out, (size_t)ctx->gsz * 8, d_out + (size_t)key_index * ctx->gsz, (size_t)kp1 * ctx->gsz * 8, (size_t)ctx->gsz * 8,
                         count, cudaMemcpyDeviceToHost, ctx->stream));
    SYNC();
    return TFA_OK;
}
extern "C" int tfa_circuit_bootstrap(tfa_ctx *ctx, const uint64_t *in, int count, uint64_t *ggsw_out) {
    Guard g(ctx);
    if (count < 1) return ctx->fail(TFA_ERR_PARAM, "count must be >= 1");
    RC(require_keys(ctx));
    const size_t iw = (size_t)count * (ctx->n + 1), ow = (size_t)count * ctx->p.cbs_level * (ctx->k + 1) * ctx->gsz;
    RC(ws_reserve(ctx, (iw + ow + (size_t)count * ctx->lw) * 8 + (size_t)count * (ctx->big + 1) * ctx->p.pfks_level * 2 + (1 << 20)));
    WSB(d_in, u64, iw); WSB(d_out, u64, ow);
    H2D(d_in, in, iw);
    RC(dev_circuit_bootstrap(ctx, d_in, count, d_out));
    D2H(ggsw_out, d_out, ow);
    SYNC();
    return TFA_OK;
}
extern "C" int tfa_vertical_packing(tfa_ctx *ctx, const uint64_t *lut, int nouts, int npoly, const uint64_t *ggsw_std, int nggsw, uint64_t *out) {
    Guard g(ctx);
    if (npoly < 1 || (npoly & (npoly - 1))) return ctx->fail(TFA_ERR_PARAM, "vertical_packing: polynomial count must be a power of two");
    const size_t gw = (size_t)ctx->p.cbs_level * (ctx->k + 1) * ctx->gsz;
    const size_t lw_ = (size_t)nouts * npoly * ctx->N, ow = (size_t)nouts * ctx->lw;
    RC(ws_reserve(ctx, (lw_ + ow + 2 * gw * nggsw) * 8 + (size_t)nouts * npoly * ctx->gsz * 8 * 2 + (1 << 20)));
    WSB(d_lut, u64, lw_); WSB(d_out, u64, ow); WSB(d_g, u64, gw * nggsw); WSB(d_gf, double2, gw * nggsw / 2);
    H2D(d_lut, lut, lw_);
    for (int i = 0; i < nggsw; i++) H2D(d_g + (size_t)i * gw, ggsw_std + (size_t)(nggsw - 1 - i) * gw, gw);  // to LSB-first
    RC(dev_fourier(ctx, d_g, (long)nggsw * ctx->p.cbs_level * (ctx->k + 1) * (ctx->k + 1), ctx->p.cbs_level, d_gf));
    RC(dev_vertical_packing(ctx, d_gf, 1, nggsw, d_lut, 0, (size_t)npoly * ctx->N, nouts, npoly * ctx->N, d_out));
    D2H(out, d_out, ow);
    SYNC();
    return TFA_OK;
}
extern "C" int tfa_fourier_forward(tfa_ctx *ctx, const uint64_t *polys, int count, double *out) {
    Guard g(ctx);
    if (count < 1) return ctx->fail(TFA_ERR_PARAM, "count must be >= 1");
    RC(ws_reserve(ctx, (size_t)count * ctx->N * 8 * 2 + (1 << 20)));
    WSB(d_in, u64, (size_t)count * ctx->N); WSB(d_out, double2, (size_t)count * 256);
    H2D(d_in, polys, (size_t)count * ctx->N);
    RC(dev_fourier(ctx, d_in, count, 1, d_out));
    CU(cudaMemcpyAsync(out, d_out, (size_t)count * 256 * sizeof(double2), cudaMemcpyDeviceToHost, ctx->stream));
    SYNC();
    return TFA_OK;
}
