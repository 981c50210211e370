/*
 * tfhe_aes_b200.h — C ABI of the B200-native WoPBS S-box engine.
 *
 * Drop-in boundary for the hot path of rostin79s/TFHE-AES (SURVEY.md §8b).  The reference has no FFI:
 * its surface is the Rust `Server` (src/server/server.rs) and the `sbox` module
 * (src/server/sbox/{gen_lut,many_wopbs,sbox}.rs).  Each entry point below names the reference
 * function it replaces; INTEGRATION.md shows the Rust shim that binds them.
 *
 * Conventions
 *   - Every ciphertext is a flat little-endian u64 array, exactly tfhe-rs's container layout:
 *       LWE(big)   = mask[k*N] || body                  -> lw = k*N+1 words (2049 at PARAM_OPT)
 *       byte       = 8 LWEs, block j = bit j (LSB first; gen_lut.rs:35-36, many_wopbs.rs:100)
 *       state      = 16 bytes, index = 4*column + row, byte 0 = most significant byte of the u128
 *                    (client.rs:126-138)
 *       round keys = [11][16] bytes
 *   - Keys are handed over in the STANDARD domain with the level order defined here (level 1, the
 *     coarsest q/beta term, first); the engine converts the bootstrap key to its own Fourier layout:
 *       bsk    [n][pbs_level][k+1 rows][(k+1)*N]      row r<k encrypts -S_r*s_i*q/beta^l, row k: s_i*q/beta^l
 *       ksk    [k*N][ks_level][n+1]                   encrypts z_i*q/beta^l under the small key
 *       pfpksk [k+1][k*N+1][pfks_level][(k+1)*N]      tfhe-rs circuit-bootstrap PFPKSK list (f(x) = -x)
 *   - Host entry points borrow host pointers for the duration of the call (copy in, run, copy out,
 *     synchronise).  `_dev` entry points take device pointers and are asynchronous on the context's
 *     stream.
 *   - Every function returns 0 on success; tfa_last_error() describes the last failure.  There is no
 *     CPU fallback: without a CUDA device every compute entry point fails with TFA_ERR_CUDA.
 *   - Polynomial size is fixed to N = 512 (the reference's PARAM_OPT, client.rs:35).
 */
#ifndef TFHE_AES_B200_H
#define TFHE_AES_B200_H
#include <stddef.h>
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

enum {
    TFA_OK = 0,
    TFA_ERR_PARAM = 1,    /* unsupported / inconsistent parameters or arguments */
    TFA_ERR_CUDA = 2,     /* CUDA runtime error (including "no device") */
    TFA_ERR_STATE = 3,    /* keys not loaded, etc. */
    TFA_ERR_UNSUPPORTED = 4 /* e.g. MultiBit bootstrap keys (many_wopbs.rs:83-84 silently returns zeros; we refuse) */
};

/* WopbsParameters — client.rs:31-57 (PARAM_OPT) */
typedef struct tfa_params {
    uint32_t lwe_dim, glwe_dim, poly_size;
    uint32_t pbs_base_log, pbs_level;
    uint32_t ks_base_log, ks_level;
    uint32_t pfks_base_log, pfks_level;
    uint32_t cbs_base_log, cbs_level;
    uint32_t message_modulus, carry_modulus;
    uint32_t _pad;
    double lwe_std, glwe_std, pfks_std;
} tfa_params;

typedef struct tfa_ctx tfa_ctx;

/* ---- context: replaces Server::new (server.rs:32-35) -------------------------------------------- */
int tfa_ctx_create(const tfa_params *params, int device, void *cuda_stream /* cudaStream_t or NULL */, tfa_ctx **out);
void tfa_ctx_destroy(tfa_ctx *ctx);
const char *tfa_last_error(const tfa_ctx *ctx /* NULL: last error of a failed tfa_ctx_create */);
void tfa_param_opt(tfa_params *out); /* client.rs:31-57 */
/* keys borrowed from HOST memory, standard domain (layouts above) */
int tfa_ctx_load_keys(tfa_ctx *ctx, const uint64_t *bsk, const uint64_t *ksk, const uint64_t *pfpksk);
/* multi-GPU replication (SURVEY §8e): prepared device key buffers, to be filled by an NCCL broadcast
 * from the rank that called tfa_ctx_load_keys / tfa_client_keygen.  tfa_ctx_alloc_keys allocates them
 * on a receiving rank; tfa_ctx_keys_ready marks them valid after the broadcast. */
int tfa_ctx_alloc_keys(tfa_ctx *ctx);
/* at most 8 buffers; at PARAM_OPT three: Fourier BSK (342.5 MB), PFPKSK (629.5 MB) and KSK (65.9 MB) in the standard u64 layouts
 * the tcgen05 kernels consume = 1.04 GB.  The mma.sync fallback layouts follow only when the context uses those kernels
 * (a shape the tcgen05 kernels do not take, or TFA_KS_IMMA / TFA_PFKS_IMMA set in the environment at tfa_ctx_create). */
int tfa_ctx_key_buffers(tfa_ctx *ctx, void **dev_ptrs /* [8] */, size_t *bytes /* [8] */, int *count);
int tfa_ctx_keys_ready(tfa_ctx *ctx);
int tfa_ctx_synchronize(tfa_ctx *ctx);
/* per-stage GPU time of everything launched since tfa_ctx_profile(ctx, 1): stages are
 * 0 ks_decompose 1 ks_gemv 2 pbs 3 pfks_decompose 4 pfks_gemv 5 fourier 6 vp 7 cmux_tree 8 linear 9 misc (the GLWE pack / unpack kernels) */
int tfa_ctx_profile(tfa_ctx *ctx, int enable);
int tfa_ctx_profile_report(tfa_ctx *ctx, double *ms_per_stage /* [10] */, int *launch_groups /* [10] */);
/* PBS kernel schedule (same arithmetic, SURVEY §9.4(3)): 0 = automatic (default), 2 = warp-specialised kernel, 3 = one
 * ciphertext per two-CTA cluster (small batches), 4 = two ciphertext sets per CTA taking turns (large batches).  3 and 4 exist
 * for glwe_dimension 4 only; at glwe_dimension 1 they run the warp-specialised kernel.  For tests and measurements.  Any other
 * value returns TFA_ERR_PARAM and leaves the schedule unchanged. */
int tfa_ctx_set_pbs_schedule(tfa_ctx *ctx, int schedule);
/* DFMA microbenchmark: measured FP64 pipe peak of the device in TFLOP/s (roofline denominator) */
int tfa_measure_fp64_peak(tfa_ctx *ctx, double *tflops);   /* max of the two below */
int tfa_measure_fp64_peaks(tfa_ctx *ctx, double *dfma_tflops, double *dmma_tflops); /* FP64 pipe: DFMA and mma.sync.m8n8k4.f64 microbenchmarks */
/* number of kernels this library launched on the context since creation (bench.py's gpu_launches) */
uint64_t tfa_ctx_launch_count(const tfa_ctx *ctx);
/* LWE ciphertexts blind-rotated (programmable bootstraps, circuit-bootstrap ones included) on the context since creation */
uint64_t tfa_ctx_pbs_count(const tfa_ctx *ctx);

/* ---- sbox module --------------------------------------------------------------------------------- */
/* gen_lut (gen_lut.rs:9-42): table[v] = f(v) for v < 2^(nb_block*log2(msg*carry));
 * lut_out: [nb_block][tfa_lut_size()] */
int tfa_lut_size(const tfa_params *params, int nb_block);
int tfa_gen_lut(const tfa_params *params, int nb_block, const uint64_t *table, uint64_t *lut_out);
/* many_wopbs_without_padding (many_wopbs.rs:31-116), batched over nct independent radix ciphertexts
 * that share the same LUTs.  ct_in [nct][nblocks][lw]; luts [L][nblocks][lut_size];
 * out [nct][L][nblocks][lw].  L = 1 is wopbs_without_padding (sbox.rs:61, server.rs:150). */
int tfa_many_wopbs(tfa_ctx *ctx, const uint64_t *ct_in, int nct, int nblocks, const uint64_t *luts, int L, uint64_t *out);
int tfa_many_wopbs_dev(tfa_ctx *ctx, const uint64_t *ct_in, int nct, int nblocks, const uint64_t *luts_dev, int L, uint64_t *out);
/* sbox (sbox.rs:46-63): in place on nct bytes; many_sbox (sbox.rs:68-97): out [nct][3 or 4][8][lw] */
int tfa_sbox(tfa_ctx *ctx, uint64_t *bytes_inout, int nct, int inv);
int tfa_many_sbox(tfa_ctx *ctx, const uint64_t *bytes_in, int nct, int inv, uint64_t *out);

/* ---- Server (server.rs) ---------------------------------------------------------------------------- */
/* aes_key_expansion (server.rs:107-167).  rcon_ct: [10][8][lw] encryptions of RCON (server.rs:139-140)
 * or NULL for trivial (noise-free) encryptions, which decrypt identically. */
int tfa_aes_key_expansion(tfa_ctx *ctx, const uint64_t *key_ct, const uint64_t *rcon_ct, uint64_t *round_keys_out);
/* AES-192 / AES-256 on the same stages (SURVEY §8f.4; the reference is AES-128 only): key_ct [key_bytes][8][lw] with key_bytes =
 * 16, 24 or 32, rk_out [key_bytes/4 + 7][16][8][lw]; rounds = 10, 12 or 14.  Every round-key byte is refreshed to noise level 1 as
 * server.rs:149-150 does for AES-128. */
int tfa_aes_key_expansion_ex(tfa_ctx *ctx, const uint64_t *key_ct, int key_bytes, const uint64_t *rcon_ct_or_null, uint64_t *rk_out);
int tfa_aes_encrypt_ex(tfa_ctx *ctx, const uint64_t *round_keys, uint64_t *states_inout, int nblk, int rounds);
int tfa_aes_decrypt_ex(tfa_ctx *ctx, const uint64_t *round_keys, uint64_t *states_inout, int nblk, int rounds);
/* aes_encrypt (server.rs:39-64) / aes_decrypt (server.rs:67-105), batched over nblk states in place */
int tfa_aes_encrypt(tfa_ctx *ctx, const uint64_t *round_keys, uint64_t *states, int nblk);
int tfa_aes_decrypt(tfa_ctx *ctx, const uint64_t *round_keys, uint64_t *states, int nblk);
/* README.md:58-59 / BASELINE.json spellings */
int tfa_aes_encryption(tfa_ctx *ctx, const uint64_t *round_keys, uint64_t *states, int nblk);
int tfa_aes_decryption(tfa_ctx *ctx, const uint64_t *round_keys, uint64_t *states, int nblk);
/* add_scalar (server.rs:172-275), batched: states[b] += counters[b] (u128 as lo,hi pairs).
 * Deliberate divergence: the low-byte LUTs use counter & 0xFF, so counters >= 256 are correct
 * (the reference uses the whole counter, server.rs:181-182, and fails its own check client.rs:171). */
int tfa_add_scalar(tfa_ctx *ctx, uint64_t *states, const uint64_t *counters_lo_hi, int nblk);
/* the CTR loop of main.rs:55-64: out[b] = AES(iv + first + b), b < nblk */
int tfa_aes_ctr(tfa_ctx *ctx, const uint64_t *round_keys, const uint64_t *iv_ct, uint64_t first_lo, uint64_t first_hi,
                int nblk, uint64_t *out);
/* The step after the path (SURVEY §8f, transciphering): the reference stops at the encrypted keystream of main.rs:55-64;
 * XOR with clear data blocks (16 bytes each, AES byte order, e.g. the AES-CTR ciphertext a client uploaded) turns it into
 * encryptions of the data.  With one message bit per LWE at 2^63 a clear bit adds bit * 2^63 to the body: no bootstrap. */
int tfa_xor_clear(tfa_ctx *ctx, uint64_t *states, const uint8_t *data, int nblk);
int tfa_xor_clear_dev(tfa_ctx *ctx, uint64_t *states, const uint8_t *data_dev, int nblk);
/* AES-CTR with a PUBLIC initial counter block (only the AES key is encrypted, as in AES-CTR transciphering, where the IV travels in
 * the clear), for nstreams independent streams that share the context's FHE keys.  Output block b of stream s =
 * Enc( AES_K_s(iv_s + first_s + b mod 2^128) XOR data_s[b] ), in stream order: out [sum of nblk][16][8][lw].  rounds = 10 / 12 / 14
 * (AES-128 / 192 / 256); round_keys of each stream [rounds + 1][16][8][lw] (tfa_aes_key_expansion[_ex] output).  data NULL: the bare
 * keystream.  No counter add is evaluated; the first two rounds are evaluated once per run of counters that agree on bytes 0..14
 * (at most 256 blocks): 8 * (27 * runs + (16 * (rounds - 2) + 5) * blocks) PBS in all, 133 byte-WoPBS per AES-128 block instead of 160.
 * Errors: TFA_ERR_PARAM for nstreams < 1, an nblk < 1, a NULL round_keys, more than INT_MAX / 16 blocks in all or another rounds;
 * TFA_ERR_STATE without keys; TFA_ERR_UNSUPPORTED unless blocks carry one bit (message_modulus * carry_modulus = 2). */
typedef struct tfa_ctr_stream {
    const uint64_t *round_keys;
    const uint8_t *data;          /* [nblk][16] or NULL */
    uint64_t first_lo, first_hi;
    uint8_t iv[16];               /* AES byte order, byte 0 = most significant */
    int32_t nblk;
    int32_t _pad;
} tfa_ctr_stream;                 /* 56 bytes, no implicit padding */
/* host pointers; every distinct round-key buffer is copied once; synchronises before returning */
int tfa_aes_ctr_public_iv(tfa_ctx *ctx, const tfa_ctr_stream *streams, int nstreams, int rounds, uint64_t *out);
/* streams: host array whose round_keys and data are device pointers; out: device; asynchronous on the context stream */
int tfa_aes_ctr_public_iv_dev(tfa_ctx *ctx, const tfa_ctr_stream *streams, int nstreams, int rounds, uint64_t *out);
/* AES-CTR with ENCRYPTED initial counter blocks (the CTR loop of main.rs:55-64) for nstreams independent streams in one call, each with
 * its own AES key, encrypted IV and counter range; the streams share the context's FHE keys.  Output block b of stream s =
 * Enc( AES_K_s(IV_s + first_s + b mod 2^128) XOR data_s[b] ), in stream order: out [sum of nblk][16][8][lw].  rounds = 10 / 12 / 14
 * (AES-128 / 192 / 256), shared by all streams; round_keys of each stream [rounds + 1][16][8][lw]; iv_ct [16][8][lw]; data NULL: the
 * bare keystream.  Streams whose iv_ct is the same pointer share one IV: its 128 bits are circuit-bootstrapped once.  Every stage of
 * the counter add and every round runs over all blocks of the call at once: 128 * (distinct iv_ct) + (128 * rounds + 15) * (sum of
 * nblk) PBS, which for one stream equals tfa_aes_ctr.
 * Errors: TFA_ERR_PARAM for nstreams < 1, an nblk < 1, a NULL round_keys or iv_ct, a NULL out, more than INT_MAX / 16 blocks in all
 * or another rounds; TFA_ERR_STATE without keys; TFA_ERR_UNSUPPORTED unless blocks carry one bit.  The context stays usable. */
typedef struct tfa_ctr_enc_stream {
    const uint64_t *round_keys;   /* [rounds + 1][16][8][lw] */
    const uint64_t *iv_ct;        /* [16][8][lw] encrypted initial counter block */
    const uint8_t *data;          /* [nblk][16] clear bytes XORed into the output, or NULL */
    uint64_t first_lo, first_hi;  /* block b encrypts iv + first + b (mod 2^128) */
    int32_t nblk;
    int32_t _pad;
} tfa_ctr_enc_stream;             /* 48 bytes, no implicit padding */
/* host pointers; every distinct round-key and iv_ct buffer is copied once; synchronises before returning */
int tfa_aes_ctr_streams(tfa_ctx *ctx, const tfa_ctr_enc_stream *streams, int nstreams, int rounds, uint64_t *out);
/* streams: host array whose round_keys, iv_ct and data are device pointers; out: device; asynchronous on the context stream */
int tfa_aes_ctr_streams_dev(tfa_ctx *ctx, const tfa_ctr_enc_stream *streams, int nstreams, int rounds, uint64_t *out);
/* GLWE packing: `count` LWEs under the big key (lwe [count][lw], e.g. the [nblk][16][8][lw] output of the CTR entry points, i.e.
 * 128 * nblk LWEs) in ceil(count / N) GLWEs of 16-bit words, 1 639 times smaller at PARAM_OPT (1 280 bytes per AES block instead of
 * 2 098 176).  Format: packed [ceil(count / N)][k+1][N] uint16_t, i.e. ceil(count / N) * (k+1) * N * 2 bytes; each GLWE is its k
 * mask polynomials, then the body (tfhe-rs GlweCiphertext order).  LWE j is coefficient j % N of GLWE j / N; coefficients past
 * `count` in the last GLWE hold keyswitch noise only.  A word is round(x / 2^48) mod 2^16 of the native-modulus word x; widened as
 * (uint64_t)v << 48 it gives a native-modulus GLWE under the GLWE secret key, which a tfhe-rs client decrypts with
 * decrypt_glwe_ciphertext (coefficient j = message of LWE j).  Packing is sum_j X^(j % N) . PFKS_k(lwe_j) with pfpksk key k, the
 * last circuit-bootstrap key, whose output has the phase of its input at coefficient 0: no key beyond the context's.  Unpacking is sample extraction of every
 * coefficient, with no key and no bootstrap: the LWEs are again under the big key and can go into every entry point.  The
 * arithmetic does not depend on the message encoding.  Noise (DESIGN §3): the rounding adds a standard deviation of about 2^51.2
 * to each unpacked LWE, far below the 2^56.4 of the rounding every PBS applies.
 * Errors: TFA_ERR_PARAM for a NULL pointer or count outside [1, INT_MAX - N + 1]; TFA_ERR_STATE for tfa_pack_lwe[_dev] without
 * keys (unpacking needs none).  The context stays usable. */
int tfa_pack_lwe(tfa_ctx *ctx, const uint64_t *lwe /* [count][lw] */, int count, uint16_t *packed /* [ceil(count/N)][k+1][N] */);
int tfa_unpack_lwe(tfa_ctx *ctx, const uint16_t *packed /* [ceil(count/N)][k+1][N] */, int count, uint64_t *lwe_out /* [count][lw] */);
/* device pointers, asynchronous on the context stream (e.g. tfa_aes_ctr_streams_dev -> tfa_pack_lwe_dev without a host round trip) */
int tfa_pack_lwe_dev(tfa_ctx *ctx, const uint64_t *lwe_dev, int count, uint16_t *packed_dev);
int tfa_unpack_lwe_dev(tfa_ctx *ctx, const uint16_t *packed_dev, int count, uint64_t *lwe_out_dev);
/* one AES round on nblk states (BASELINE config 2): 16*nblk many_sbox + ShiftRows/MixColumns + AddRoundKey */
int tfa_aes_round(tfa_ctx *ctx, const uint64_t *round_key, uint64_t *states, int nblk);
/* linear layers alone (server.rs:278-282, mix_columns.rs:4, inv_mix_columns.rs:4, shift_rows.rs:5, inv_shift_rows.rs:5) */
int tfa_add_round_key(tfa_ctx *ctx, uint64_t *states, const uint64_t *round_key, int nblk);
int tfa_mix_columns(tfa_ctx *ctx, const uint64_t *mul_sbox_states /* [nblk][16][3][8][lw] */, uint64_t *states_out, int nblk);
int tfa_inv_mix_columns(tfa_ctx *ctx, const uint64_t *mul_states /* [nblk][16][4][8][lw] */, uint64_t *states_out, int nblk);
int tfa_shift_rows(tfa_ctx *ctx, uint64_t *states, int nblk, int inverse);

/* device-resident variants (device pointers, asynchronous on the context stream) */
int tfa_aes_encrypt_dev(tfa_ctx *ctx, const uint64_t *round_keys, uint64_t *states, int nblk);
int tfa_aes_decrypt_dev(tfa_ctx *ctx, const uint64_t *round_keys, uint64_t *states, int nblk);
int tfa_aes_round_dev(tfa_ctx *ctx, const uint64_t *round_key, uint64_t *states, int nblk);
int tfa_add_scalar_dev(tfa_ctx *ctx, uint64_t *states, const uint64_t *counters_lo_hi_dev, int nblk);
int tfa_aes_ctr_dev(tfa_ctx *ctx, const uint64_t *round_keys, const uint64_t *iv_ct, uint64_t first_lo, uint64_t first_hi,
                    int nblk, uint64_t *out);
int tfa_aes_key_expansion_dev(tfa_ctx *ctx, const uint64_t *key_ct, const uint64_t *rcon_ct, uint64_t *round_keys_out);

/* ---- primitives of the chain, exposed for parity tests (tfhe-rs core_crypto call sites) -------------- */
/* keyswitch big->small (inside extract_bits_assign, many_wopbs.rs:194): in [count][lw] -> out [count][n+1] */
int tfa_keyswitch(tfa_ctx *ctx, const uint64_t *in, int count, uint64_t *out);
/* programmable bootstrap with accumulator body `lut` [N]: in [count][n+1] -> out [count][lw] */
int tfa_bootstrap(tfa_ctx *ctx, const uint64_t *in, int count, const uint64_t *lut, uint64_t *out);
int tfa_bootstrap_dev(tfa_ctx *ctx, const uint64_t *in, int count, const uint64_t *lut, uint64_t pre_add_body,
                      uint64_t post_add_body, uint64_t *out);
/* extract_bits (many_wopbs.rs:194-199): in [count][lw] -> out [count][nbits][n+1], index 0 = MSB */
int tfa_extract_bits(tfa_ctx *ctx, const uint64_t *in, int count, int delta_log, int nbits, uint64_t *out);
/* PFKS with key `key_index` (inside circuit_bootstrap_boolean): in [count][lw] -> out [count][(k+1)N] */
int tfa_pfks(tfa_ctx *ctx, int key_index, const uint64_t *in, int count, uint64_t *out);
/* circuit_bootstrap_boolean (many_wopbs.rs:253): in [count][n+1] -> standard GGSW [count][cbs_level][k+1][(k+1)N] */
int tfa_circuit_bootstrap(tfa_ctx *ctx, const uint64_t *in, int count, uint64_t *ggsw_out);
/* vertical_packing (many_wopbs.rs:277): lut [nouts][npoly][N], ggsw_std [nggsw][cbs_level][k+1][(k+1)N]
 * (index 0 = MSB) -> out [nouts][lw] */
int tfa_vertical_packing(tfa_ctx *ctx, const uint64_t *lut, int nouts, int npoly, const uint64_t *ggsw_std, int nggsw, uint64_t *out);
/* forward negacyclic FFT of torus polynomials: in [count][N] -> out [count][N/2][2] doubles, natural order */
int tfa_fourier_forward(tfa_ctx *ctx, const uint64_t *polys, int count, double *out);

/* ---- client side (client.rs:70-175): key generation, encryption, decryption on the GPU.
 * Trusted-side harness so that benchmarks and examples are self-contained; not part of the server path.
 * Randomness is the ChaCha20 key stream under a 256-bit key.  seed = 0: the key comes from the operating system
 * (getrandom), fresh for every call, as tfhe-rs seeds its generator.  seed != 0: the key is a function of the seed only
 * -- reproducible material for tests and benchmarks, INSECURE: whoever knows the seed regenerates the secret keys, and two
 * encryption calls with the same non-zero seed reuse masks and noise.  Production users load tfhe-rs keys with
 * tfa_ctx_load_keys instead. */
int tfa_client_keygen(tfa_ctx *ctx, uint64_t seed); /* generates secret keys + BSK/KSK/PFPKSK and loads them */
void tfa_rng_block(const uint32_t key[8], uint64_t nonce, uint64_t counter, uint64_t out[8]); /* ChaCha20 block (64-bit counter / nonce), host; for tests */
int tfa_client_encrypt_bytes(tfa_ctx *ctx, const uint8_t *bytes, int count, uint64_t seed, uint64_t *out /* [count][8][lw] */);
int tfa_client_decrypt_bytes(tfa_ctx *ctx, const uint64_t *ct, int count, uint8_t *bytes_out);
int tfa_client_encrypt_bytes_dev(tfa_ctx *ctx, const uint8_t *bytes_host, int count, uint64_t seed, uint64_t *out_dev);
int tfa_client_decrypt_bytes_dev(tfa_ctx *ctx, const uint64_t *ct_dev, int count, uint8_t *bytes_out_host);
int tfa_client_set_secret_keys(tfa_ctx *ctx, const uint64_t *lwe_sk, const uint64_t *glwe_sk);
/* secret keys (host copies) so a test can cross-check generated keys with an independent implementation */
int tfa_client_secret_keys(tfa_ctx *ctx, uint64_t *lwe_sk /* [n] */, uint64_t *glwe_sk /* [k*N] */);

#ifdef __cplusplus
}
#endif
#endif
