"""AES-CTR with a public IV (tfa_aes_ctr_public_iv): only the AES key is encrypted, the counter blocks are known in the clear.
Expected values come from aes_clear (FIPS-197); ciphertexts are encrypted and decrypted with the oracle's keys."""
import numpy as np
import pytest

import aes_clear

pytestmark = pytest.mark.gpu

KEY = bytes.fromhex("2b7e151628aed2a6abf7158809cf4f3c")
RK_CACHE = {}


def round_keys(engine, oracle, key):
    """encrypted round keys of `key` ([Nr + 1][16][8][lw]), expanded once per engine and key"""
    k = (id(engine), key)
    if k not in RK_CACHE:
        RK_CACHE[k] = engine.aes_key_expansion_ex(oracle.encrypt_bytes(key))
    return RK_CACHE[k]


def keystream(key, iv, first, nblk):
    return [aes_clear.ctr_block(key, iv, first + b) for b in range(nblk)]


def pbs_expected(runs, blocks, rounds=10):
    """8 bit-level PBS per byte-WoPBS: 27 S-boxes per run, 5 + 16 (Nr - 2) per block"""
    return 8 * (27 * runs + (16 * (rounds - 2) + 5) * blocks)


def test_one_stream_across_a_run_boundary(pkg, engine_test, oracle_test):
    """IV low byte 0xFA, 12 blocks: two runs (6 + 6).  With data the output decrypts to the message, without data it is the
    keystream, and the encrypted-IV entry point produces the same keystream."""
    o = oracle_test
    srv = pkg.Server(engine_test)
    iv = int.from_bytes(bytes.fromhex("f0f1f2f3f4f5f6f7f8f9fafbfcfdfefa"), "big")
    nblk = 12
    rk = round_keys(engine_test, o, KEY)
    stream = keystream(KEY, iv, 0, nblk)
    message = bytes((7 * i + 3) % 256 for i in range(16 * nblk))
    uploaded = aes_clear.xor(message, b"".join(stream))                 # what an AES-CTR client sends with the IV
    got = srv.aes_ctr_public_iv(rk, iv, nblk, data=uploaded)
    assert got.shape == (nblk, 16, 8, engine_test.lw)
    assert b"".join(o.decrypt_bytes(got[b]) for b in range(nblk)) == message
    ks = srv.aes_ctr_public_iv(rk, iv.to_bytes(16, "big"), nblk)
    for b in range(nblk):
        assert o.decrypt_bytes(ks[b]) == stream[b], b
    ref = srv.aes_ctr(rk, o.encrypt_bytes(iv.to_bytes(16, "big")), nblk)
    for b in range(nblk):
        assert o.decrypt_bytes(ref[b]) == o.decrypt_bytes(ks[b]), b


@pytest.mark.parametrize("iv,first,nblk", [(2 ** 128 - 3, 0, 5), (2 ** 64 - 2, 0, 5),
                                           (0x00FF_FFFF_FFFF_FFFF_FFFF_FFFF_FFFF_FF00, 254, 5), (0x0123_4567_89AB_CDEF_0011_2233_4455_6637, 0, 300)])
def test_counter_carries_and_long_streams(pkg, engine_test, oracle_test, iv, first, nblk):
    """Counter blocks computed on the host: the wrap at 2^128, the carry across the 64-bit halves, a carry through 15 bytes,
    and a stream longer than 256 blocks (three runs)."""
    o = oracle_test
    rk = round_keys(engine_test, o, KEY)
    got = pkg.Server(engine_test).aes_ctr_public_iv(rk, iv, nblk, first=first)
    stream = keystream(KEY, iv, first, nblk)
    for b in range(nblk):
        assert o.decrypt_bytes(got[b]) == stream[b], (hex(iv), first, b)


def test_several_streams_in_one_call(engine_test, oracle_test):
    """Three AES keys and IVs, lengths 1, 1 and 7, data on the middle stream only: outputs in stream order."""
    o = oracle_test
    keys = [KEY, bytes(range(16)), bytes(range(200, 216))]
    ivs = [5, 2 ** 128 - 1, 0xABCDEF_0000_0000_0000_0000_0000_00FC]
    firsts = [0, 0, 1]
    lens = [1, 1, 7]
    data = bytes(range(100, 116))
    streams = [(round_keys(engine_test, o, k), iv, f, n, data if i == 1 else None)
               for i, (k, iv, f, n) in enumerate(zip(keys, ivs, firsts, lens))]
    got = engine_test.aes_ctr_public_iv(streams)
    assert len(got) == sum(lens)
    row = 0
    for i, (k, iv, f, n) in enumerate(zip(keys, ivs, firsts, lens)):
        for b, want in enumerate(keystream(k, iv, f, n)):
            if i == 1:
                want = aes_clear.xor(want, data)
            assert o.decrypt_bytes(got[row]) == want, (i, b)
            row += 1


@pytest.mark.parametrize("nbytes,rounds", [(24, 12), (32, 14)])
def test_aes_192_256(engine_test, oracle_test, nbytes, rounds):
    """FIPS-197 Appendix C.2 / C.3 keys, counters across a run boundary"""
    o = oracle_test
    key = bytes(range(nbytes))
    rk = round_keys(engine_test, o, key)
    assert len(rk) == rounds + 1
    iv = int.from_bytes(bytes.fromhex("00112233445566778899aabbccddeeff"), "big")   # block 0 is the Appendix C plaintext
    got = engine_test.aes_ctr_public_iv([(rk, iv, 0, 4, None)], rounds=rounds)
    assert o.decrypt_bytes(got[0]) == aes_clear.aes_encrypt_block(key, iv.to_bytes(16, "big"))
    for b, want in enumerate(keystream(key, iv, 0, 4)):
        assert o.decrypt_bytes(got[b]) == want, b


def test_exact_pbs_schedule(engine_test, oracle_test):
    """The PBS count of a call is 8 (27 G + 133 B) for AES-128: the first two rounds once per run, no counter add."""
    o = oracle_test
    rk = round_keys(engine_test, o, KEY)
    c0 = engine_test.pbs_count
    engine_test.aes_ctr_public_iv([(rk, 0x10, 0, 5, None)])                    # one run of 5 blocks
    assert engine_test.pbs_count - c0 == pbs_expected(1, 5)
    rk2 = round_keys(engine_test, o, bytes(range(16)))
    streams = [(rk, 0xFE, 0, 4, None),                                         # 2 runs (FE FF | 00 01)
               (rk2, 5, 0, 1, bytes(16)),                                      # 1 run
               (rk, 2 ** 128 - 1, 0, 2, None)]                                 # 2 runs (wrap to 0)
    c0 = engine_test.pbs_count
    engine_test.aes_ctr_public_iv(streams)
    assert engine_test.pbs_count - c0 == pbs_expected(5, 7)
    rk256 = round_keys(engine_test, o, bytes(range(32)))
    c0 = engine_test.pbs_count
    engine_test.aes_ctr_public_iv([(rk256, 0, 0, 3, None)], rounds=14)
    assert engine_test.pbs_count - c0 == pbs_expected(1, 3, rounds=14)


def test_device_variant_matches_host_variant(pkg, engine_test, oracle_test):
    """tfa_aes_ctr_public_iv_dev on torch CUDA tensors: the same decrypted bytes as the host entry point."""
    import torch
    o = oracle_test
    rk = round_keys(engine_test, o, KEY)
    rk2 = round_keys(engine_test, o, bytes(range(16)))
    data = bytes(range(48))
    host = engine_test.aes_ctr_public_iv([(rk, 0xFF, 0, 3, data), (rk2, 77, 2, 2, None)])
    dev = torch.device("cuda", 0)
    t_rk = torch.from_numpy(rk.view(np.int64).ravel().copy()).to(dev)
    t_rk2 = torch.from_numpy(rk2.view(np.int64).ravel().copy()).to(dev)
    t_data = torch.tensor(list(data), dtype=torch.uint8, device=dev)
    t_out = torch.zeros(5 * 16 * 8 * engine_test.lw, dtype=torch.int64, device=dev)
    torch.cuda.synchronize()                                                   # the library runs on its own stream
    engine_test.aes_ctr_public_iv_dev([(t_rk.data_ptr(), 0xFF, 0, 3, t_data.data_ptr()), (t_rk2.data_ptr(), 77, 2, 2, None)],
                                      t_out.data_ptr())
    engine_test.synchronize()
    got = t_out.cpu().numpy().view(np.uint64).reshape(5, 16, 8, engine_test.lw)
    for b in range(5):
        assert o.decrypt_bytes(got[b]) == o.decrypt_bytes(host[b]), b
    assert o.decrypt_bytes(got[0]) == aes_clear.xor(aes_clear.ctr_block(KEY, 0xFF, 0), data[:16])
    assert o.decrypt_bytes(got[4]) == aes_clear.ctr_block(bytes(range(16)), 77, 3)


def test_errors_leave_the_context_usable(pkg, engine_test, engine_test2, oracle_test):
    o = oracle_test
    rk = round_keys(engine_test, o, KEY)
    bad = [([], 10),                                                           # no stream
           ([(rk, 0, 0, 0, None)], 10),                                        # empty stream
           ([(rk, 0, 0, 2, None), (rk, 0, 0, -1, None)], 10),                  # negative length
           ([(None, 0, 0, 2, None)], 10),                                      # no round keys
           ([(rk, 0, 0, 2 ** 30, None), (rk, 0, 0, 2 ** 30, None)], 10),       # total block count overflows int
           ([(rk, 0, 0, 2, None)], 11)]                                        # not AES-128/192/256
    for streams, rounds in bad:
        with pytest.raises(pkg.TfaError) as ei:
            engine_test.aes_ctr_public_iv(streams, rounds=rounds)
        assert ei.value.code == 1, (streams, rounds)
    e = pkg.Engine(pkg.param_test())
    with pytest.raises(pkg.TfaError) as ei:                                    # keys not loaded
        e.aes_ctr_public_iv([(rk, 0, 0, 1, None)])
    assert ei.value.code == 3
    e.close()
    with pytest.raises(pkg.TfaError) as ei:                                    # 2-bit blocks
        engine_test2.aes_ctr_public_iv([(np.zeros((11, 16, 4, engine_test2.lw), dtype=np.uint64), 0, 0, 1, None)])
    assert ei.value.code == 4
    got = engine_test.aes_ctr_public_iv([(rk, 9, 0, 2, None)])
    assert [o.decrypt_bytes(got[b]) for b in range(2)] == keystream(KEY, 9, 0, 2)


# ---- PARAM_OPT (client.rs:31-57) ------------------------------------------------------------------------------
@pytest.mark.slow
def test_opt_148_blocks_and_noise(pkg, engine_opt, oracle_opt):
    """148 blocks in one stream with data decrypt to the message.  Noise: both this path and tfa_aes_ctr end on S-box output +
    round key (level 2), so the variance of the output bit errors over 18 944 LWEs each agrees within [0.9, 1.11] (about 7
    standard deviations of the ratio estimate)."""
    o = oracle_opt
    srv = pkg.Server(engine_opt)
    iv = 0x0F0E0D0C_0B0A0908_07060504_030201A0
    nblk = 148
    rk = round_keys(engine_opt, o, bytes(16))
    stream = keystream(bytes(16), iv, 0, nblk)
    message = bytes((31 * i + 5) % 256 for i in range(16 * nblk))
    got = srv.aes_ctr_public_iv(rk, iv, nblk, data=aes_clear.xor(message, b"".join(stream)))
    assert o.decrypt_bytes(got) == message
    ref = srv.aes_ctr(rk, o.encrypt_bytes(iv.to_bytes(16, "big")), nblk)
    assert o.decrypt_bytes(ref) == b"".join(stream)
    _, err_new = o.decrypt_bits(got, with_err=True)
    _, err_ref = o.decrypt_bits(ref, with_err=True)
    assert len(err_new) == len(err_ref) == nblk * 128
    ratio = np.var(err_new.astype(np.float64)) / np.var(err_ref.astype(np.float64))
    assert 0.9 <= ratio <= 1.11, ratio
