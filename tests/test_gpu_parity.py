"""GPU parity tests: the CUDA path, called through the C ABI, against the CPU oracle on identical
keys and inputs.  Integer stages (keyswitch, PFKS, linear layers) must be bit-exact.  FP64 stages
(PBS, circuit bootstrap, vertical packing) are compared on the PHASE (b - <a, s>, i.e. message +
noise) with the tolerance written in each test, and always on the decrypted plaintext (exact).
Raw ciphertext words of a multi-step FP64 stage are not comparable: an FFT rounding difference of
one unit in the last decomposition digit replaces the mask by a different, equally valid one."""
import numpy as np
import pytest

from conftest import torus_absdiff

pytestmark = pytest.mark.gpu

KEY = bytes.fromhex("2b7e151628aed2a6abf7158809cf4f3c")
PT = [bytes.fromhex(h) for h in ("6bc1bee22e409f96e93d7e117393172a", "ae2d8a571e03ac9c9eb76fac45af8e51",
                                 "30c81c46a35ce411e5fbc1191a0a52ef", "f69f2445df4f9b17ad2b417be66c3710")]
CT = [bytes.fromhex(h) for h in ("3ad77bb40d7a3660a89ecaf32466ef97", "f5d3d58503b9699de785895a96fdbaaf",
                                 "43b1cd7f598ece23881b00e3ed030688", "7b0c785e27e8ad3f8223207104725dd4")]


# ---- FFT ------------------------------------------------------------------------------------------
def test_fourier_forward_matches_oracle(engine_test, oracle_test):
    rng = np.random.default_rng(10)
    polys = rng.integers(0, 2 ** 64, (7, 512), dtype=np.uint64)
    got = engine_test.fourier_forward(polys)
    for q in range(len(polys)):
        ref = oracle_test.fft_forward_torus(polys[q])
        # tolerance: a few ulp of the largest output (|X| <= 512 * 2^63)
        assert np.abs(got[q] - ref).max() <= 2e-15 * np.abs(ref).max()


# ---- integer stages: bit exact ----------------------------------------------------------------------
@pytest.mark.parametrize("count", [1, 8, 19])
def test_keyswitch_bit_exact(engine_test, oracle_test, count):
    rng = np.random.default_rng(count)
    ct = rng.integers(0, 2 ** 64, (count, oracle_test.lw), dtype=np.uint64)
    assert np.array_equal(engine_test.keyswitch(ct), oracle_test.keyswitch(ct))


def test_pfks_bit_exact(engine_test, oracle_test):
    rng = np.random.default_rng(3)
    ct = rng.integers(0, 2 ** 64, (5, oracle_test.lw), dtype=np.uint64)
    for key in range(oracle_test.k + 1):
        got = engine_test.pfks(key, ct)
        for i in range(len(ct)):
            assert np.array_equal(got[i], oracle_test.pfks(key, ct[i]))


def test_linear_layers_bit_exact(engine_test, oracle_test):
    rng = np.random.default_rng(4)
    lw = oracle_test.lw
    st = rng.integers(0, 2 ** 64, (3, 16, 8, lw), dtype=np.uint64)
    rk = rng.integers(0, 2 ** 64, (16, 8, lw), dtype=np.uint64)
    got = engine_test.add_round_key(st, rk)
    for b in range(3):
        assert np.array_equal(got[b], oracle_test.add_round_key(st[b], rk))
    mul = rng.integers(0, 2 ** 64, (2, 16, 3, 8, lw), dtype=np.uint64)
    got = engine_test.mix_columns(mul)
    for b in range(2):
        assert np.array_equal(got[b], oracle_test.mix_columns(mul[b]))
    mul4 = rng.integers(0, 2 ** 64, (2, 16, 4, 8, lw), dtype=np.uint64)
    got = engine_test.inv_mix_columns(mul4)
    for b in range(2):
        assert np.array_equal(got[b], oracle_test.inv_mix_columns(mul4[b]))
    for inverse in (False, True):
        got = engine_test.shift_rows(st, inverse)
        for b in range(3):
            assert np.array_equal(got[b], oracle_test.shift_rows(st[b], inverse))


# ---- FP64 stages --------------------------------------------------------------------------------------
def test_bootstrap_matches_oracle(engine_test, oracle_test):
    rng = np.random.default_rng(5)
    o = oracle_test
    msgs = rng.integers(0, 2, 9).astype(np.uint64)
    lwe = o.encrypt_lwe_small((msgs << np.uint64(63)) + np.uint64(1 << 62))
    lut = np.full(512, (1 << 64) - (1 << 48), dtype=np.uint64)  # the CBS accumulator (-2^48 everywhere)
    got, ref = engine_test.bootstrap(lwe, lut), o.bootstrap(lwe, lut)
    # tolerance 2^36 on the phase: both sides carry the PBS noise (decomposition rounding 2^24 * sqrt(kN/2)
    # per step plus FFT rounding ~2^26, SURVEY §9.7), payload is 2^48
    assert torus_absdiff(o.phase_big(got), o.phase_big(ref)) < 2 ** 36
    ph = o.phase_big(got) + np.uint64(1 << 48)
    assert np.array_equal(((ph + np.uint64(1 << 48)) >> np.uint64(49)) & np.uint64(1), msgs)


@pytest.mark.parametrize("schedule", [2])
@pytest.mark.parametrize("count", [3, 9, 20])
def test_bootstrap_both_kernel_schedules(engine_test, oracle_test, schedule, count):
    """The warp-specialised PBS kernel, forced with schedule 2, against the oracle; count 3 / 9 / 20 selects 1 / 4 / 8
    ciphertexts per CTA at the test parameters.  Schedule 1, the phase-synchronous kernel, no longer exists: the same counts
    run in test_bootstrap_after_rejected_pbs_schedules."""
    rng = np.random.default_rng(50 + count)
    o = oracle_test
    lut = rng.integers(0, 2 ** 64, 512, dtype=np.uint64)
    lwe = o.encrypt_lwe_small(rng.integers(0, 2 ** 64, count, dtype=np.uint64))
    engine_test.set_pbs_schedule(schedule)
    try:
        got = engine_test.bootstrap(lwe, lut)
    finally:
        engine_test.set_pbs_schedule(0)
    assert torus_absdiff(o.phase_big(got), o.phase_big(o.bootstrap(lwe, lut))) < 2 ** 36


@pytest.mark.parametrize("count", [3, 9, 20])
def test_bootstrap_after_rejected_pbs_schedules(pkg, engine_test, oracle_test, count):
    """Schedules other than 0, 2, 3 and 4 (1 included) are refused with TFA_ERR_PARAM and leave the automatic schedule in
    place: the bootstrap that follows still matches the oracle with 1 / 4 / 8 ciphertexts per CTA."""
    for schedule in (1, 5, -1):
        with pytest.raises(pkg.TfaError) as ei:
            engine_test.set_pbs_schedule(schedule)
        assert ei.value.code == 1, schedule   # TFA_ERR_PARAM
    rng = np.random.default_rng(50 + count)
    o = oracle_test
    lut = rng.integers(0, 2 ** 64, 512, dtype=np.uint64)
    lwe = o.encrypt_lwe_small(rng.integers(0, 2 ** 64, count, dtype=np.uint64))
    assert torus_absdiff(o.phase_big(engine_test.bootstrap(lwe, lut)), o.phase_big(o.bootstrap(lwe, lut))) < 2 ** 36


def test_bootstrap_general_lut(engine_test, oracle_test):
    rng = np.random.default_rng(6)
    o = oracle_test
    lut = rng.integers(0, 2 ** 64, 512, dtype=np.uint64)
    lwe = o.encrypt_lwe_small(rng.integers(0, 2 ** 64, 13, dtype=np.uint64))
    assert torus_absdiff(o.phase_big(engine_test.bootstrap(lwe, lut)), o.phase_big(o.bootstrap(lwe, lut))) < 2 ** 36


def test_extract_bits_reference_case_is_keyswitch(engine_test, oracle_test):
    o = oracle_test
    ct = o.encrypt_bits([1, 0, 1])
    got = engine_test.extract_bits(ct, 63, 1)
    for i in range(3):
        assert np.array_equal(got[i], o.extract_bits(ct[i], 63, 1))


def test_extract_bits_general_pbs_loop(engine_test2, oracle_test2):
    """message_modulus 4: two bits per block, the PBS loop of extract_bits runs (SURVEY §9.4(1))."""
    o = oracle_test2
    rng = np.random.default_rng(7)
    vals = rng.integers(0, 4, 6)
    ct = np.zeros((6, o.lw), dtype=np.uint64)
    for i, v in enumerate(vals):  # encode v * 2^62 under the big key
        bits = o.encrypt_bits([0])
        ct[i] = bits[0]
        ct[i, -1] += np.uint64(int(v) << 62)
    got = engine_test2.extract_bits(ct, 62, 2)
    for i, v in enumerate(vals):
        ref = o.extract_bits(ct[i], 62, 2)
        assert np.array_equal(got[i, 1], ref[1])            # first extracted (LSB): keyswitch only, bit exact
        # second bit goes through a PBS (FP64) and a keyswitch (rounds below 2^52): compare phases
        assert torus_absdiff(o.phase_small(got[i, 0]), o.phase_small(ref[0])) < 2 ** 58
        ph = o.phase_small(got[i])
        dec = ((ph + np.uint64(1 << 62)) >> np.uint64(63)) & np.uint64(1)
        assert int(dec[0]) == (int(v) >> 1) and int(dec[1]) == (int(v) & 1)


def test_circuit_bootstrap_matches_oracle(engine_test, oracle_test):
    o = oracle_test
    lwe = o.encrypt_lwe_small(np.array([0, 1 << 63, 1 << 63], dtype=np.uint64))
    got = engine_test.circuit_bootstrap(lwe)
    for i in range(3):
        ref = o.circuit_bootstrap_boolean(lwe[i])
        # every GGSW row is a GLWE of (-S_r or 1) * m * 2^49: compare the phases, tolerance 2^40
        # (PBS noise ~2^31 plus PFKS rounding below 2^28 over kN+1 terms)
        assert torus_absdiff(o.glwe_phase(got[i]), o.glwe_phase(ref)) < 2 ** 40


def test_vertical_packing_matches_oracle(engine_test, oracle_test):
    o = oracle_test
    rng = np.random.default_rng(8)
    bits = [1, 0, 1, 1, 0, 0, 1, 0]  # MSB first -> value 0xB2
    lwe = o.encrypt_lwe_small(np.array(bits, dtype=np.uint64) << np.uint64(63))
    ggsw = np.stack([o.circuit_bootstrap_boolean(l) for l in lwe])
    lut = rng.integers(0, 2, (5, 1, 512)).astype(np.uint64) << np.uint64(63)
    got = engine_test.vertical_packing(lut, ggsw)
    for j in range(5):
        ref = o.vertical_packing(lut[j], ggsw)
        assert torus_absdiff(o.phase_big(got[j]), o.phase_big(ref)) < 2 ** 54  # level-1 product: noise ~2^51 per step
    dec = o.decrypt_bits(got)
    assert np.array_equal(dec, (lut[:, 0, 0xB2] >> np.uint64(63)).astype(np.uint8))


def test_vertical_packing_cmux_tree(engine_test, oracle_test):
    """10 selector bits, N = 512: each LUT spans 2 polynomials, so the CMux tree has depth 1."""
    o = oracle_test
    rng = np.random.default_rng(9)
    value = 0x2B7
    bits = [(value >> (9 - i)) & 1 for i in range(10)]
    lwe = o.encrypt_lwe_small(np.array(bits, dtype=np.uint64) << np.uint64(63))
    ggsw = np.stack([o.circuit_bootstrap_boolean(l) for l in lwe])
    lut = rng.integers(0, 2, (3, 2, 512)).astype(np.uint64) << np.uint64(63)
    got = engine_test.vertical_packing(lut, ggsw)
    for j in range(3):
        assert torus_absdiff(o.phase_big(got[j]), o.phase_big(o.vertical_packing(lut[j], ggsw))) < 2 ** 54
    dec = o.decrypt_bits(got)
    assert np.array_equal(dec, (lut.reshape(3, 1024)[:, value] >> np.uint64(63)).astype(np.uint8))
    # 11 bits -> 4 polynomials -> depth 2
    value = 0x5A3
    bits = [(value >> (10 - i)) & 1 for i in range(11)]
    lwe = o.encrypt_lwe_small(np.array(bits, dtype=np.uint64) << np.uint64(63))
    ggsw = np.stack([o.circuit_bootstrap_boolean(l) for l in lwe])
    lut = rng.integers(0, 2, (2, 4, 512)).astype(np.uint64) << np.uint64(63)
    got = engine_test.vertical_packing(lut, ggsw)
    assert np.array_equal(o.decrypt_bits(got), (lut.reshape(2, 2048)[:, value] >> np.uint64(63)).astype(np.uint8))
    for j in range(2):
        assert torus_absdiff(o.phase_big(got[j]), o.phase_big(o.vertical_packing(lut[j], ggsw))) < 2 ** 54


# ---- sbox module ------------------------------------------------------------------------------------------
def test_many_wopbs_matches_oracle(pkg, engine_test, oracle_test):
    o = oracle_test
    data = bytes([0x00, 0x53, 0xFF, 0xA7, 0x10])
    ct = o.encrypt_bytes(data)
    luts = np.stack([pkg.gen_lut(engine_test.params, 8, f) for f in
                     (lambda x: pkg.SBOX[x], lambda x: pkg.mul2(pkg.SBOX[x]), lambda x: pkg.mul3(pkg.SBOX[x]))])
    assert np.array_equal(luts[0], o.gen_lut(8, np.frombuffer(pkg.SBOX, dtype=np.uint8).astype(np.uint64)))
    got = engine_test.many_wopbs(ct, luts)
    for i, b in enumerate(data):
        ref = o.many_wopbs(ct[i], luts)
        assert torus_absdiff(o.phase_big(got[i]), o.phase_big(ref)) < 2 ** 58  # decision threshold 2^62; noise ~2^53
        s = pkg.SBOX[b]
        assert o.decrypt_bytes(got[i]) == bytes([s, pkg.mul2(s), pkg.mul3(s)])


def test_sbox_and_many_sbox(pkg, engine_test, oracle_test):
    o = oracle_test
    data = bytes(range(0, 256, 37))
    ct = o.encrypt_bytes(data)
    assert o.decrypt_bytes(engine_test.sbox(ct, False)) == bytes(pkg.SBOX[b] for b in data)
    assert o.decrypt_bytes(engine_test.sbox(ct, True)) == bytes(pkg.INV_SBOX[b] for b in data)
    m = engine_test.many_sbox(ct, True)
    for i, b in enumerate(data):
        assert o.decrypt_bytes(m[i]) == bytes([pkg.mul9(b), pkg.mul11(b), pkg.mul13(b), pkg.mul14(b)])


def test_many_wopbs_two_bit_blocks(pkg, engine_test2, oracle_test2):
    """General path end to end: 2-bit blocks (extract_bits PBS loop) with an 8-bit LUT."""
    o, e = oracle_test2, engine_test2
    rng = np.random.default_rng(11)
    vals = [0x00, 0xC9, 0x7E]
    ct = np.zeros((len(vals), 4, o.lw), dtype=np.uint64)
    for i, v in enumerate(vals):
        for blk in range(4):
            ct[i, blk] = o.encrypt_bits([0])[0]
            ct[i, blk, -1] += np.uint64(((v >> (2 * blk)) & 3) << 62)
    luts = pkg.gen_lut(e.params, 4, lambda x: pkg.SBOX[x])[None]
    assert np.array_equal(luts[0], o.gen_lut(4, np.frombuffer(pkg.SBOX, dtype=np.uint8).astype(np.uint64)))
    got = e.many_wopbs(ct, luts)
    for i, v in enumerate(vals):
        ref = o.many_wopbs(ct[i], luts)
        ph_g, ph_r = o.phase_big(got[i, 0]), o.phase_big(ref[0])
        dec = lambda ph: sum(int(((p + np.uint64(1 << 61)) >> np.uint64(62)) & np.uint64(3)) << (2 * b) for b, p in enumerate(ph))
        assert dec(ph_g) == dec(ph_r) == pkg.SBOX[v]


# ---- Server -------------------------------------------------------------------------------------------------
def test_aes_round(pkg, engine_test, oracle_test, orc):
    o = oracle_test
    rng = np.random.default_rng(12)
    st = bytes(rng.integers(0, 256, 32, dtype=np.uint8))
    rk = bytes(rng.integers(0, 256, 16, dtype=np.uint8))
    got = engine_test.aes_round(o.encrypt_bytes(rk), o.encrypt_bytes(st).reshape(2, 16, 8, o.lw))
    for b in range(2):
        s = [pkg.SBOX[x] for x in st[16 * b:16 * b + 16]]
        t = [s[(i % 4) + 4 * (((i // 4) + (i % 4)) % 4)] for i in range(16)]
        exp = []
        for c in range(4):
            a = t[4 * c:4 * c + 4]
            exp += [pkg.mul2(a[0]) ^ pkg.mul3(a[1]) ^ a[2] ^ a[3], a[0] ^ pkg.mul2(a[1]) ^ pkg.mul3(a[2]) ^ a[3],
                    a[0] ^ a[1] ^ pkg.mul2(a[2]) ^ pkg.mul3(a[3]), pkg.mul3(a[0]) ^ a[1] ^ a[2] ^ pkg.mul2(a[3])]
        assert o.decrypt_bytes(got[b]) == bytes(x ^ y for x, y in zip(exp, rk))


def test_key_expansion_encrypt_decrypt_kat(pkg, engine_test, oracle_test, orc):
    """The reference's test() (main.rs:76-118): SP 800-38A F.1.1 vectors through key expansion,
    encryption and decryption; expected values from FIPS-197 (the `aes` crate in the reference)."""
    o = oracle_test
    srv = pkg.Server(engine_test)
    rk = srv.aes_key_expansion(o.encrypt_bytes(KEY))
    assert b"".join(o.decrypt_bytes(rk[r]) for r in range(11)) == orc.clear_round_keys(KEY)
    states = np.stack([o.encrypt_bytes(p) for p in PT])
    enc = srv.aes_encrypt(rk, states)
    for i in range(4):
        assert o.decrypt_bytes(enc[i]) == CT[i]
    dec = srv.aes_decrypt(rk, enc)
    for i in range(4):
        assert o.decrypt_bytes(dec[i]) == PT[i]
    # ciphertext-level agreement with the oracle on one block (tolerance as in test_many_wopbs)
    ref = o.aes_encrypt(rk, states[0])
    assert torus_absdiff(o.phase_big(enc[0]), o.phase_big(ref)) < 2 ** 59


def test_add_scalar_and_ctr(pkg, engine_test, oracle_test, orc):
    o = oracle_test
    srv = pkg.Server(engine_test)
    iv = (2 ** 128 - 300).to_bytes(16, "big")
    ctrs = [0, 1, 255, 256, 299, 300, 1023, 2 ** 64 + 5]
    st = np.stack([o.encrypt_bytes(iv)] * len(ctrs))
    got = srv.add_scalar(st, ctrs)
    for i, c in enumerate(ctrs):
        assert o.decrypt_bytes(got[i]) == ((int.from_bytes(iv, "big") + c) % 2 ** 128).to_bytes(16, "big"), c
    key = bytes(16)
    rk = srv.aes_key_expansion(o.encrypt_bytes(key))
    out = srv.aes_ctr(rk, o.encrypt_bytes(bytes(16)), 3, first=254)
    for b in range(3):
        assert o.decrypt_bytes(out[b]) == orc.clear_aes_encrypt(key, (254 + b).to_bytes(16, "big"))


def test_ctr_transciphering_xor(pkg, engine_test, oracle_test, orc):
    """The step after the keystream (SURVEY §8f): Enc(keystream) XOR clear AES-CTR ciphertext = Enc(message), and the
    CTR entry point with its shared IV bootstrap agrees block by block with add_scalar + aes_encrypt."""
    o = oracle_test
    srv = pkg.Server(engine_test)
    key = bytes.fromhex("000102030405060708090a0b0c0d0e0f")
    iv = int.from_bytes(bytes.fromhex("f0f1f2f3f4f5f6f7f8f9fafbfcfdfeff"), "big")
    rk = srv.aes_key_expansion(o.encrypt_bytes(key))
    iv_ct = o.encrypt_bytes(iv.to_bytes(16, "big"))
    nblk = 4
    ks = srv.aes_ctr(rk, iv_ct, nblk, first=0)
    message = bytes(range(64))
    stream = b"".join(orc.clear_aes_encrypt(key, ((iv + b) % 2 ** 128).to_bytes(16, "big")) for b in range(nblk))
    uploaded = bytes(m ^ k for m, k in zip(message, stream))            # what an AES-CTR client sends
    got = engine_test.xor_clear(ks, uploaded)
    assert b"".join(o.decrypt_bytes(got[b]) for b in range(nblk)) == message
    # reference schedule: clone the IV, add_scalar(i), aes_encrypt (main.rs:59-61)
    st = srv.add_scalar(np.stack([iv_ct] * nblk), list(range(nblk)))
    enc = engine_test.aes_encrypt(rk, st)
    for b in range(nblk):
        assert o.decrypt_bytes(enc[b]) == stream[16 * b:16 * b + 16] == o.decrypt_bytes(ks[b])


@pytest.mark.parametrize("iv,first", [(2 ** 128 - 2, 0), (2 ** 64 - 3, 1), (0x00FF_FFFF_FFFF_FFFF_FFFF_FFFF_FFFF_FF00, 254)])
def test_ctr_carry_chain_with_shared_iv_bootstrap(pkg, engine_test, oracle_test, orc, iv, first):
    """tfa_aes_ctr bootstraps the IV bits once and only the carries per block: carries must ripple through every byte,
    across the 64-bit boundary and wrap at 2^128 exactly as add_scalar (server.rs:172-275) block by block."""
    o = oracle_test
    srv = pkg.Server(engine_test)
    key = bytes.fromhex("2b7e151628aed2a6abf7158809cf4f3c")
    rk = srv.aes_key_expansion(o.encrypt_bytes(key))
    out = srv.aes_ctr(rk, o.encrypt_bytes(iv.to_bytes(16, "big")), 5, first=first)
    for b in range(5):
        assert o.decrypt_bytes(out[b]) == orc.clear_aes_encrypt(key, ((iv + first + b) % 2 ** 128).to_bytes(16, "big")), (hex(iv), first, b)


def test_client_keygen_roundtrip(pkg, orc):
    """Keys generated by the GPU client harness: engine-side encrypt/decrypt round trip, a full S-box,
    and a cross-check of an engine ciphertext with the oracle's decryption under the exported key."""
    e = pkg.Engine(pkg.param_test())
    e.client_keygen(1234)
    data = bytes([0x53, 0x00, 0xFF, 0x3C])
    ct = e.client_encrypt_bytes(data, seed=9)
    assert e.client_decrypt_bytes(ct) == data
    assert e.client_decrypt_bytes(e.sbox(ct)) == bytes(pkg.SBOX[b] for b in data)
    lwe_sk, glwe_sk = e.client_secret_keys()
    ph = (ct.reshape(-1, e.lw)[:, -1] - (ct.reshape(-1, e.lw)[:, :-1] * glwe_sk).sum(axis=1, dtype=np.uint64))
    bits = ((ph + np.uint64(1 << 62)) >> np.uint64(63)) & np.uint64(1)
    assert np.array_equal(bits.reshape(-1, 8), np.array([[(b >> j) & 1 for j in range(8)] for b in data], dtype=np.uint64))
    e.close()


# ---- PARAM_OPT (client.rs:31-57) ------------------------------------------------------------------------------
def test_opt_integer_stages_bit_exact(engine_opt, oracle_opt):
    rng = np.random.default_rng(20)
    ct = rng.integers(0, 2 ** 64, (9, oracle_opt.lw), dtype=np.uint64)
    assert np.array_equal(engine_opt.keyswitch(ct), oracle_opt.keyswitch(ct))
    got = engine_opt.pfks(2, ct[:2])
    for i in range(2):
        assert np.array_equal(got[i], oracle_opt.pfks(2, ct[i]))
    got = engine_opt.pfks(4, ct[:1])
    assert np.array_equal(got[0], oracle_opt.pfks(4, ct[0]))


def test_opt_keyswitches_across_tensor_tiles(engine_opt, oracle_opt):
    """The tcgen05 keyswitch kernels tile the bits by 128: 300 inputs = two full tiles and a ragged one; extreme words
    exercise the digit limbs (d = d_lo + 128 d_hi) and the 64-bit recombination.  Bit-exact against the oracle on a
    sample of rows of every tile and every PFKS key."""
    rng = np.random.default_rng(21)
    ct = rng.integers(0, 2 ** 64, (300, oracle_opt.lw), dtype=np.uint64)
    ct[0, :] = np.uint64(0xFFFFFFFFFFFFFFFF)
    ct[127, :] = np.uint64(0x8000000000000000)
    ct[128, :] = np.uint64(0x7FF7FF7FF7FF7FF7)
    ct[299, ::2] = np.uint64(0)
    sample = [0, 1, 127, 128, 255, 256, 299]
    ks = engine_opt.keyswitch(ct)
    for i in sample:
        assert np.array_equal(ks[i], oracle_opt.keyswitch(ct[i:i + 1])[0]), f"keyswitch row {i}"
    for key in range(oracle_opt.k + 1):
        got = engine_opt.pfks(key, ct)
        for i in sample:
            assert np.array_equal(got[i], oracle_opt.pfks(key, ct[i])), f"pfks key {key} row {i}"


def test_opt_bootstrap_matches_oracle(engine_opt, oracle_opt):
    o = oracle_opt
    msgs = np.array([0, 1, 1, 0, 1], dtype=np.uint64)
    ks = o.keyswitch(o.encrypt_bits(msgs))
    ks[:, -1] += np.uint64(1 << 62)
    lut = np.full(512, (1 << 64) - (1 << 48), dtype=np.uint64)
    got, ref = engine_opt.bootstrap(ks, lut), o.bootstrap(ks, lut)
    # 669 CMux steps, FFT rounding ~2^26 each (SURVEY §9.7) -> random walk ~2^31; bound 2^36
    assert torus_absdiff(o.phase_big(got), o.phase_big(ref)) < 2 ** 36
    ph = o.phase_big(got) + np.uint64(1 << 48)
    assert np.array_equal(((ph + np.uint64(1 << 48)) >> np.uint64(49)) & np.uint64(1), msgs)


@pytest.mark.parametrize("count", [150, 300])
def test_opt_bootstrap_wave_ws_kernel(engine_opt, oracle_opt, count):
    """PARAM_OPT with 2 (count 150) and 3 (count 300) ciphertexts per CTA of the warp-specialised kernel (forced schedule 2):
    the outputs decrypt to the encrypted bits, and a sample agrees with the oracle."""
    o = oracle_opt
    rng = np.random.default_rng(count)
    msgs = rng.integers(0, 2, count).astype(np.uint64)
    ks = o.keyswitch(o.encrypt_bits(msgs))
    ks[:, -1] += np.uint64(1 << 62)
    lut = np.full(512, (1 << 64) - (1 << 48), dtype=np.uint64)
    engine_opt.set_pbs_schedule(2)
    try:
        got = engine_opt.bootstrap(ks, lut)
    finally:
        engine_opt.set_pbs_schedule(0)
    ph = o.phase_big(got) + np.uint64(1 << 48)
    assert np.array_equal(((ph + np.uint64(1 << 48)) >> np.uint64(49)) & np.uint64(1), msgs)
    sample = [0, count // 2, count - 1]
    ref = o.bootstrap(ks[sample], lut)
    assert torus_absdiff(o.phase_big(got[sample]), o.phase_big(ref)) < 2 ** 36


@pytest.mark.parametrize("count,schedule", [(7, 4), (900, 0), (1400, 0)])
def test_opt_bootstrap_two_sets_per_cta(engine_opt, oracle_opt, count, schedule):
    """pbs_ws2_kernel (two sets of three ciphertexts per CTA, accumulators in tensor memory): same arithmetic as the
    warp-specialised kernel, so the outputs are bit-identical.  7 forced: ragged last CTA; 900 automatic: one wave of 888 + 12 through
    the cluster kernel; 1400 automatic: 888 + a remainder above half a wave, all through pbs_ws2_kernel."""
    o = oracle_opt
    rng = np.random.default_rng(count)
    base = 60
    msgs0 = rng.integers(0, 2, base).astype(np.uint64)
    ks0 = o.keyswitch(o.encrypt_bits(msgs0))
    ks0[:, -1] += np.uint64(1 << 62)
    pick = rng.integers(0, base, count)
    ks, msgs = ks0[pick], msgs0[pick]
    lut = np.full(512, (1 << 64) - (1 << 48), dtype=np.uint64)
    res = {}
    for sched in (2, schedule):
        engine_opt.set_pbs_schedule(sched)
        try:
            res[sched] = engine_opt.bootstrap(ks, lut)
        finally:
            engine_opt.set_pbs_schedule(0)
    ph = o.phase_big(res[schedule]) + np.uint64(1 << 48)
    assert np.array_equal(((ph + np.uint64(1 << 48)) >> np.uint64(49)) & np.uint64(1), msgs)
    n2 = 888 if count == 900 else count      # ciphertexts that went through pbs_ws2_kernel
    assert np.array_equal(res[2][:n2], res[schedule][:n2])
    if n2 < count:                            # the cluster kernel adds the two halves of a row in a different order
        assert torus_absdiff(o.phase_big(res[2][n2:]), o.phase_big(res[schedule][n2:])) < 2 ** 36


def test_opt_many_sbox_noise_within_tolerance(pkg, engine_opt, oracle_opt):
    """north_star: ciphertext noise variance within a stated tolerance of the reference path's.
    Tolerance: variance ratio GPU / oracle in [0.5, 2] over >= 1000 output LWEs (SURVEY §8c)."""
    o = oracle_opt
    rng = np.random.default_rng(21)
    data = bytes(rng.integers(0, 256, 44, dtype=np.uint8))
    ct = o.encrypt_bytes(data)
    got = engine_opt.many_sbox(ct, False)
    errs_g, errs_o = [], []
    for i, b in enumerate(data):
        s = pkg.SBOX[b]
        assert o.decrypt_bytes(got[i]) == bytes([s, pkg.mul2(s), pkg.mul3(s)])
        errs_g.append(o.decrypt_bits(got[i], with_err=True)[1])
    for i in range(0, len(data)):
        ref = o.many_sbox(ct[i], False)
        errs_o.append(o.decrypt_bits(ref, with_err=True)[1])
        if i < 4:
            assert torus_absdiff(o.phase_big(got[i]), o.phase_big(ref)) < 2 ** 58
    vg = np.var(np.concatenate(errs_g).astype(np.float64))
    vo = np.var(np.concatenate(errs_o).astype(np.float64))
    assert len(np.concatenate(errs_g)) >= 1000
    assert 0.5 < vg / vo < 2.0, (vg, vo)
    assert np.sqrt(vg) * np.sqrt(5) < 2 ** 62 / 8  # level-5 sum stays far below the decision boundary


@pytest.mark.slow
def test_opt_config1_ctr_block(pkg, engine_opt, oracle_opt):
    """BASELINE config 1: --number-of-outputs 1 --iv 0 --key 0 -> 66e94bd4ef8a2c3b884cfa59ca342b2e,
    plus counters that exercise the add_scalar carry fix (SURVEY §4 table)."""
    o = oracle_opt
    srv = pkg.Server(engine_opt)
    rk = srv.aes_key_expansion(o.encrypt_bytes(bytes(16)))
    out = srv.aes_ctr(rk, o.encrypt_bytes(bytes(16)), 2, first=0)
    assert o.decrypt_bytes(out[0]).hex() == "66e94bd4ef8a2c3b884cfa59ca342b2e"
    assert o.decrypt_bytes(out[1]).hex() == "58e2fccefa7e3061367f1d57a4e7455a"
    out = srv.aes_ctr(rk, o.encrypt_bytes(bytes(16)), 2, first=255)
    assert o.decrypt_bytes(out[0]).hex() == "f70ddef93ba62588242a0e67d0d645e0"
    assert o.decrypt_bytes(out[1]).hex() == "fb56cc09b680b1d07c5a52149e29f07c"
    dec = srv.aes_decrypt(rk, out)
    assert o.decrypt_bytes(dec[0]) == (255).to_bytes(16, "big")
    assert o.decrypt_bytes(dec[1]) == (256).to_bytes(16, "big")


# ---- boundary behaviour ---------------------------------------------------------------------------------------
def test_error_behaviour(pkg, engine_test):
    """The reference panics on misuse; the C ABI returns a status and a message (SURVEY §8b)."""
    e = pkg.Engine(pkg.param_test())
    with pytest.raises(pkg.TfaError) as ei:        # keys not loaded
        e.sbox(np.zeros((1, 8, e.lw), dtype=np.uint64))
    assert ei.value.code == 3
    e.close()
    with pytest.raises(pkg.TfaError) as ei:        # empty batch
        engine_test.many_wopbs(np.zeros((0, 8, engine_test.lw), dtype=np.uint64), np.zeros((1, 8, 512), dtype=np.uint64))
    assert ei.value.code == 1


def test_config4_decrypt_16_blocks(pkg, engine_test, oracle_test, orc):
    """BASELINE config 4 shape on the small parameter set: aes_decrypt on 16 CTR blocks."""
    o = oracle_test
    srv = pkg.Server(engine_test)
    key = bytes(range(16, 32))
    rk = srv.aes_key_expansion(o.encrypt_bytes(key))
    iv = 2 ** 64 - 3
    blocks = [orc.clear_aes_encrypt(key, ((iv + i) % 2 ** 128).to_bytes(16, "big")) for i in range(16)]
    states = np.stack([o.encrypt_bytes(b) for b in blocks])
    dec = srv.aes_decrypt(rk, states)
    for i in range(16):
        assert o.decrypt_bytes(dec[i]) == ((iv + i) % 2 ** 128).to_bytes(16, "big")


def test_ragged_batches(pkg, engine_test, oracle_test):
    """Batch sizes that are not multiples of any tile (ciphertexts per CTA, 16-bit MMA rows, 128-bit tiles)."""
    o = oracle_test
    for nct in (1, 3, 17):
        data = bytes((37 * i + nct) % 256 for i in range(nct))
        got = engine_test.sbox(o.encrypt_bytes(data), False)
        assert o.decrypt_bytes(got) == bytes(pkg.SBOX[b] for b in data)


@pytest.mark.slow
def test_cli_mirrors_reference_driver(pkg):
    """tfhe_aes_cli = src/main.rs on the engine (PARAM_OPT): keygen, key expansion, CTR, decrypt + verify."""
    import os
    import subprocess
    cli = os.path.join(os.path.dirname(pkg.lib_path()), "tfhe_aes_cli")
    if not os.path.exists(cli):
        pytest.skip("CLI not built")
    r = subprocess.run([cli, "--number-of-outputs", "3", "--iv", "254", "--key", "12345678901234567890"], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr
    assert "Passed" in r.stdout and "AES key expansion took" in r.stdout


# ---- AES-192 / AES-256 (SURVEY §8f.4): FIPS-197 Appendix C.2 / C.3 --------------------------------------------------
@pytest.mark.parametrize("nbytes,want", [(16, "69c4e0d86a7b0430d8cdb78070b4c55a"), (24, "dda97ca4864cdfe06eaf70a0ec0d7191"),
                                         (32, "8ea2b7ca516745bfeafc49904b496089")])
def test_aes_192_256_kat(pkg, engine_test, oracle_test, nbytes, want):
    import aes_clear
    o = oracle_test
    key, pt = bytes(range(nbytes)), bytes.fromhex("00112233445566778899aabbccddeeff")
    rk = engine_test.aes_key_expansion_ex(o.encrypt_bytes(key))
    assert len(rk) == nbytes // 4 + 7
    want_rk = aes_clear.round_keys(key)
    for r in range(len(rk)):
        assert o.decrypt_bytes(rk[r]) == want_rk[r], f"round key {r}"
    enc = engine_test.aes_crypt_ex(rk, o.encrypt_bytes(pt)[None])
    assert o.decrypt_bytes(enc[0]).hex() == want
    dec = engine_test.aes_crypt_ex(rk, enc, decrypt=True)
    assert o.decrypt_bytes(dec[0]) == pt
