"""GLWE packing of LWE ciphertexts (tfa_pack_lwe / tfa_unpack_lwe): N LWEs per GLWE of 16-bit words, and back by sample
extraction.  The pack is checked bit for bit against numpy over the oracle's PFKS (sum_i X^i PFKS_k(lwe_i), then
round(x / 2^48) mod 2^16), the unpack against numpy sample extraction; ciphertexts are encrypted and decrypted with the
oracle's keys, and clear AES comes from aes_clear (FIPS-197)."""
import ctypes as C

import numpy as np
import pytest

import aes_clear

COUNTS = [1, 7, 511, 512, 513, 1100]
INT_MAX = 2 ** 31 - 1


def ref_pack(o, lwes):
    """numpy: GLWE g = sum_i X^i . oracle.pfks(k, lwe[g N + i]), each word rounded to round(x / 2^48) mod 2^16"""
    N, k = o.N, o.k
    lwes = np.asarray(lwes, dtype=np.uint64).reshape(-1, o.lw)
    acc = np.zeros((-(-len(lwes) // N), k + 1, N), dtype=np.uint64)
    for j, lwe in enumerate(lwes):
        p = o.pfks(k, lwe).reshape(k + 1, N)
        i = j % N
        acc[j // N] += np.concatenate([np.uint64(0) - p[:, N - i:], p[:, :N - i]], axis=1)   # X^i . p (negacyclic)
    return (((acc >> np.uint64(47)) + np.uint64(1)) >> np.uint64(1)).astype(np.uint16)


def ref_unpack(packed, count, k, N):
    """numpy sample extraction of coefficient i % N of GLWE i // N, words widened as v << 48"""
    w = packed.astype(np.uint64) << np.uint64(48)
    out = np.zeros((count, k * N + 1), dtype=np.uint64)
    t = np.arange(N)
    for g in range(-(-count // N)):
        j = np.arange(min(N, count - g * N))[:, None]
        idx = (j - t[None, :]) % N
        for r in range(k):
            a = w[g, r][idx]
            out[g * N:g * N + len(j), r * N:(r + 1) * N] = np.where(t[None, :] <= j, a, np.uint64(0) - a)
        out[g * N:g * N + len(j), k * N] = w[g, k, :len(j)]
    return out


def widened(packed):
    return packed.astype(np.uint64) << np.uint64(48)


def glwe_bits(o, packed, count):
    """bits of the first `count` coefficients of the widened GLWEs, decoded as decrypt_bits does"""
    ph = o.glwe_phase(widened(packed)).ravel()[:count]
    return (((ph + np.uint64(2 ** 62)) >> np.uint64(63)) & np.uint64(1)).astype(np.uint8)


def random_bits(rng, count):
    return rng.integers(0, 2, count, dtype=np.uint8)


@pytest.mark.gpu
@pytest.mark.parametrize("count", COUNTS)
def test_pack_bit_exact(engine_test, oracle_test, count):
    """random u64 words and real encryptions: the packed words equal the numpy reference bit for bit"""
    o = oracle_test
    rng = np.random.default_rng(count)
    for lwes in (rng.integers(0, 2 ** 64, (count, o.lw), dtype=np.uint64), o.encrypt_bits(random_bits(rng, count))):
        got = engine_test.pack_lwe(lwes)
        assert got.dtype == np.uint16 and got.shape == (-(-count // o.N), o.k + 1, o.N)
        assert np.array_equal(got, ref_pack(o, lwes))


@pytest.mark.gpu
def test_pack_bit_exact_mma_sync_fallback(pkg, oracle_test, monkeypatch):
    """a context created with TFA_PFKS_IMMA set runs the PFKS on the mma.sync kernel, whose key k lies at its own offset in the
    fragment layout: the packed words are the same"""
    monkeypatch.setenv("TFA_PFKS_IMMA", "1")
    eng = pkg.Engine(pkg.param_test())
    monkeypatch.delenv("TFA_PFKS_IMMA")
    o = oracle_test
    eng.load_keys(o.bsk(), o.ksk(), o.pfpksk())
    p = o.params
    kp_pfpksk = (o.k + 1) * (o.gsz // 8) * (-(-o.lw * p.pfks_level // 32)) * 2048   # [k+1][column tiles][row chunks][2 KB]
    assert eng.key_buffers()[-1][1] == kp_pfpksk                               # the fragment layout of the PFPKSK exists
    lwes = np.random.default_rng(21).integers(0, 2 ** 64, (513, o.lw), dtype=np.uint64)
    assert np.array_equal(eng.pack_lwe(lwes), ref_pack(o, lwes))
    eng.close()


@pytest.mark.gpu
@pytest.mark.parametrize("count", COUNTS)
def test_unpack_bit_exact(engine_test, oracle_test, count):
    """unpacking a packed batch and random uint16 words both equal numpy sample extraction"""
    o = oracle_test
    rng = np.random.default_rng(100 + count)
    G = -(-count // o.N)
    packed = engine_test.pack_lwe(o.encrypt_bits(random_bits(rng, count)))
    for p in (packed, rng.integers(0, 2 ** 16, (G, o.k + 1, o.N), dtype=np.uint16)):
        assert np.array_equal(engine_test.unpack_lwe(p, count), ref_unpack(p, count, o.k, o.N))


@pytest.mark.gpu
@pytest.mark.parametrize("count", [7, 513, 1100])
def test_round_trip_decrypts(engine_test, oracle_test, count):
    """unpacked LWEs decrypt to the packed bits, and so do the widened GLWEs under the GLWE key"""
    o = oracle_test
    bits = random_bits(np.random.default_rng(200 + count), count)
    packed = engine_test.pack_lwe(o.encrypt_bits(bits))
    assert np.array_equal(o.decrypt_bits(engine_test.unpack_lwe(packed, count)), bits)
    assert np.array_equal(glwe_bits(o, packed, count), bits)


@pytest.mark.gpu
def test_round_trip_two_bit_blocks(engine_test2, oracle_test2):
    """2-bit messages at 2^62 (message_modulus 4): the format does not depend on the encoding"""
    o = oracle_test2
    count = 600
    vals = np.random.default_rng(7).integers(0, 4, count, dtype=np.uint64)
    lwes = o.encrypt_bits(np.zeros(count, dtype=np.uint8))
    lwes[:, -1] += vals << np.uint64(62)
    packed = engine_test2.pack_lwe(lwes)
    assert np.array_equal(packed, ref_pack(o, lwes))

    def decode(ph):
        return ((ph + np.uint64(2 ** 61)) >> np.uint64(62)) & np.uint64(3)

    assert np.array_equal(decode(o.phase_big(engine_test2.unpack_lwe(packed, count))), vals)
    assert np.array_equal(decode(o.glwe_phase(widened(packed)).ravel()[:count]), vals)


def _to_device(a, dev):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a).view(np.int64 if a.dtype == np.uint64 else np.int16).ravel().copy()).to(dev)


@pytest.mark.gpu
def test_device_variants_match_host_variants(engine_test, oracle_test):
    """pack_dev and unpack_dev on torch CUDA tensors give the host results, also chained on the device without a copy back"""
    import torch
    o, eng = oracle_test, engine_test
    count = 1100
    G = eng.packed_glwes(count)
    lwes = o.encrypt_bits(random_bits(np.random.default_rng(11), count))
    packed = eng.pack_lwe(lwes)
    dev = torch.device("cuda", 0)
    t_in = _to_device(lwes, dev)
    t_packed = torch.zeros(G * eng.gsz, dtype=torch.int16, device=dev)
    t_out = torch.zeros(count * eng.lw, dtype=torch.int64, device=dev)
    torch.cuda.synchronize()                                                   # the library runs on its own stream
    eng.pack_lwe_dev(t_in.data_ptr(), count, t_packed.data_ptr())
    eng.unpack_lwe_dev(t_packed.data_ptr(), count, t_out.data_ptr())
    eng.synchronize()
    assert np.array_equal(t_packed.cpu().numpy().view(np.uint16).reshape(packed.shape), packed)
    assert np.array_equal(t_out.cpu().numpy().view(np.uint64).reshape(count, eng.lw), eng.unpack_lwe(packed, count))
    # unpack_dev of host-packed words
    t_host_packed = _to_device(packed, dev)
    t_out.zero_()
    torch.cuda.synchronize()
    eng.unpack_lwe_dev(t_host_packed.data_ptr(), count, t_out.data_ptr())
    eng.synchronize()
    assert np.array_equal(t_out.cpu().numpy().view(np.uint64).reshape(count, eng.lw), ref_unpack(packed, count, eng.k, eng.N))


@pytest.mark.gpu
def test_errors_leave_the_context_usable(pkg, engine_test, oracle_test):
    o, eng = oracle_test, engine_test
    lib = eng.lib
    bits = random_bits(np.random.default_rng(12), 9)
    lwes = o.encrypt_bits(bits)
    want = eng.pack_lwe(lwes)
    small_lwe = np.zeros((2, eng.lw), dtype=np.uint64)
    small_packed = np.zeros((1, eng.k + 1, eng.N), dtype=np.uint16)

    def p(a):
        return a.ctypes.data_as(C.c_void_p)

    def still_works():
        packed = eng.pack_lwe(lwes)
        assert np.array_equal(packed, want)
        assert np.array_equal(o.decrypt_bits(eng.unpack_lwe(packed, 9)), bits)

    # TFA_ERR_PARAM: count < 1, a count whose ceil(count / N) * N overflows int, a NULL pointer; host and device entry points
    for fn in (lib.tfa_pack_lwe, lib.tfa_pack_lwe_dev):
        for args in ((p(small_lwe), 0, p(small_packed)), (p(small_lwe), -3, p(small_packed)),
                     (p(small_lwe), INT_MAX - eng.N + 2, p(small_packed)), (p(small_lwe), INT_MAX, p(small_packed)),
                     (None, 2, p(small_packed)), (p(small_lwe), 2, None)):
            assert fn(eng.h, *args) == 1, (fn, args)
            still_works()
    for fn in (lib.tfa_unpack_lwe, lib.tfa_unpack_lwe_dev):
        for args in ((p(small_packed), 0, p(small_lwe)), (p(small_packed), -1, p(small_lwe)),
                     (p(small_packed), INT_MAX - eng.N + 2, p(small_lwe)), (None, 2, p(small_lwe)), (p(small_packed), 2, None)):
            assert fn(eng.h, *args) == 1, (fn, args)
            still_works()
    with pytest.raises(pkg.TfaError) as ei:
        eng.pack_lwe(np.zeros((0, eng.lw), dtype=np.uint64))
    assert ei.value.code == 1
    with pytest.raises(ValueError):                                            # more LWEs than the GLWEs hold
        eng.unpack_lwe(want, eng.N + 1)
    still_works()
    # TFA_ERR_STATE: packing needs the PFPKSK; unpacking needs no key
    e = pkg.Engine(pkg.param_test())
    with pytest.raises(pkg.TfaError) as ei:
        e.pack_lwe(lwes)
    assert ei.value.code == 3
    assert np.array_equal(e.unpack_lwe(want, 9), eng.unpack_lwe(want, 9))
    e.close()
    still_works()


# ---- PARAM_OPT (client.rs:31-57) ------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.slow
def test_opt_transciphered_blocks_pack_and_stay_computable(pkg, engine_opt, oracle_opt):
    """8 blocks transciphered with aes_ctr_public_iv from the client's AES-CTR ciphertext pack into 2 GLWEs whose widened words
    decrypt to the FIPS-197 message; the unpacked bytes go through tfa_sbox and decrypt to SBOX[m]."""
    o = oracle_opt
    key = bytes.fromhex("2b7e151628aed2a6abf7158809cf4f3c")
    iv = 0xF0F1F2F3_F4F5F6F7_F8F9FAFB_FCFDFEFF
    nblk = 8
    msg = bytes((37 * i + 11) % 256 for i in range(16 * nblk))
    data = b"".join(aes_clear.xor(aes_clear.ctr_block(key, iv, b), msg[16 * b:16 * b + 16]) for b in range(nblk))
    rk = o.encrypt_bytes(b"".join(aes_clear.round_keys(key)))
    ct = engine_opt.aes_ctr_public_iv([(rk, iv, 0, nblk, data)])
    count = 128 * nblk
    packed = engine_opt.pack_lwe(ct)
    assert packed.shape == (2, 5, 512)
    assert packed.nbytes // nblk == 1280
    bits = glwe_bits(o, packed, count).reshape(-1, 8)
    assert bytes(int(sum(int(b) << j for j, b in enumerate(byte))) for byte in bits) == msg
    unpacked = engine_opt.unpack_lwe(packed, count)
    assert o.decrypt_bytes(unpacked) == msg
    out = engine_opt.sbox(unpacked.reshape(-1, 8, engine_opt.lw))
    assert o.decrypt_bytes(out) == bytes(aes_clear.SBOX[m] for m in msg)


@pytest.mark.gpu
@pytest.mark.slow
def test_opt_noise_of_the_16_bit_rounding(engine_opt, oracle_opt):
    """phase_big(unpacked) - phase_big(original) over 16 384 fresh encryptions: its variance is (h + 1) / 12 * 2^96 (h = Hamming
    weight of the GLWE key; the rounding error of every word is uniform on 2^48 and has mean 0) within [0.8, 1.25], and every
    error lies below 2^55.  The N errors of one GLWE are one error vector convolved with the key, so they are strongly correlated:
    32 GLWEs are needed for a relative spread of the estimate of about 6 % (4 096 LWEs would give 14 %)."""
    o = oracle_opt
    count = 32 * 512
    lwes = o.encrypt_bits(random_bits(np.random.default_rng(13), count))
    unpacked = engine_opt.unpack_lwe(engine_opt.pack_lwe(lwes), count)
    d = (o.phase_big(unpacked) - o.phase_big(lwes)).view(np.int64).astype(np.float64)
    h = int(o.glwe_sk().sum())
    ratio = np.mean(d ** 2) / ((h + 1) / 12 * 2.0 ** 96)
    assert 0.8 <= ratio <= 1.25, (ratio, h)
    assert np.abs(d).max() < 2.0 ** 55, np.log2(np.abs(d).max())
