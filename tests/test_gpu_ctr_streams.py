"""AES-CTR with encrypted IVs, many streams in one call (tfa_aes_ctr_streams): every stream has its own AES key, encrypted IV and
counter range.  Expected values come from aes_clear (FIPS-197) and from one tfa_aes_ctr call per stream; ciphertexts are encrypted
and decrypted with the oracle's keys."""
import ctypes as C
import os
import shutil
import subprocess

import numpy as np
import pytest

import aes_clear

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
KEY = bytes.fromhex("2b7e151628aed2a6abf7158809cf4f3c")
RK_CACHE = {}


def round_keys(engine, oracle, key):
    """encrypted round keys of `key` ([Nr + 1][16][8][lw]), expanded once per engine and key"""
    k = (id(engine), key)
    if k not in RK_CACHE:
        RK_CACHE[k] = engine.aes_key_expansion_ex(oracle.encrypt_bytes(key))
    return RK_CACHE[k]


def enc_iv(oracle, iv):
    return oracle.encrypt_bytes(iv.to_bytes(16, "big"))


def keystream(key, iv, first, nblk):
    return [aes_clear.ctr_block(key, iv, first + b) for b in range(nblk)]


def pbs_expected(distinct_ivs, blocks, rounds=10):
    """128 IV-bit bootstraps per distinct IV; per block 15 carry bootstraps and 128 S-box bit bootstraps per round"""
    return 128 * distinct_ivs + (128 * rounds + 15) * blocks


def check_streams(o, got, streams_clear):
    """streams_clear: list of (key, iv, first, nblk, data or None); got in stream order"""
    assert len(got) == sum(s[3] for s in streams_clear)
    row = 0
    for i, (key, iv, first, nblk, data) in enumerate(streams_clear):
        for b, want in enumerate(keystream(key, iv, first, nblk)):
            if data is not None:
                want = aes_clear.xor(want, data[16 * b:16 * b + 16])
            assert o.decrypt_bytes(got[row]) == want, (i, b)
            row += 1


def test_struct_layout_matches_header(pkg, tmp_path):
    """TfaCtrEncStream has the size and field offsets of tfa_ctr_enc_stream as the C compiler lays it out from the header."""
    cc = shutil.which("cc") or shutil.which("gcc")
    if cc is None:
        pytest.skip("no C compiler")
    fields = [f for f, _ in pkg.TfaCtrEncStream._fields_]
    src = tmp_path / "layout.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "tfhe_aes_b200.h"\nint main(void) {\n'
                   '    printf("%zu", sizeof(tfa_ctr_enc_stream));\n' +
                   "".join(f'    printf(" %zu", offsetof(tfa_ctr_enc_stream, {f}));\n' for f in fields) + "    return 0;\n}\n")
    exe = tmp_path / "layout"
    subprocess.check_call([cc, "-I", os.path.join(ROOT, "include"), "-o", str(exe), str(src)])
    got = [int(x) for x in subprocess.check_output([str(exe)], text=True).split()]
    assert got[0] == C.sizeof(pkg.TfaCtrEncStream) == 48
    assert got[1:] == [getattr(pkg.TfaCtrEncStream, f).offset for f in fields]


@pytest.mark.gpu
def test_several_streams_in_one_call(pkg, engine_test, oracle_test):
    """Three AES keys and encrypted IVs, lengths 1, 1 and 7, data on the last stream only: outputs in stream order, and each
    stream decrypts as a separate aes_ctr call for it."""
    o = oracle_test
    srv = pkg.Server(engine_test)
    keys = [KEY, bytes(range(16)), bytes(range(200, 216))]
    ivs = [5, 2 ** 128 - 1, 0xABCDEF_0000_0000_0000_0000_0000_00FC]
    firsts = [0, 3, 1]
    lens = [1, 1, 7]
    data = bytes((13 * i + 1) % 256 for i in range(16 * 7))
    clear = [(k, iv, f, n, data if i == 2 else None) for i, (k, iv, f, n) in enumerate(zip(keys, ivs, firsts, lens))]
    rks = [round_keys(engine_test, o, k) for k in keys]
    cts = [enc_iv(o, iv) for iv in ivs]
    got = srv.aes_ctr_streams([(rk, ct, f, n, d) for rk, ct, (_, _, f, n, d) in zip(rks, cts, clear)])
    assert got.shape == (9, 16, 8, engine_test.lw)
    check_streams(o, got, clear)
    row = 0
    for rk, ct, (_, _, f, n, d) in zip(rks, cts, clear):
        ref = srv.aes_ctr(rk, ct, n, first=f)
        for b in range(n):
            want = o.decrypt_bytes(ref[b])
            if d is not None:
                want = aes_clear.xor(want, d[16 * b:16 * b + 16])
            assert o.decrypt_bytes(got[row]) == want, (row, b)
            row += 1


@pytest.mark.gpu
@pytest.mark.parametrize("iv,first,nblk", [(2 ** 128 - 3, 0, 5),                                   # counters wrap at 2^128
                                           (0x0102_0304_0506_0708_0000_0000_0000_FFFF, 2 ** 64 - 2, 4),  # first_lo carries into first_hi
                                           (0, 1022, 2),                                            # the values add_scalar.rs gets wrong
                                           (0x0123_4567_89AB_CDEF_0011_2233_4455_6637, 0, 300)])    # longer than 256 blocks
def test_counters(pkg, engine_test, oracle_test, iv, first, nblk):
    o = oracle_test
    rk = round_keys(engine_test, o, KEY)
    got = pkg.Server(engine_test).aes_ctr_streams([(rk, enc_iv(o, iv), first, nblk, None)])
    stream = keystream(KEY, iv, first, nblk)
    for b in range(nblk):
        assert o.decrypt_bytes(got[b]) == stream[b], (hex(iv), first, b)


@pytest.mark.gpu
def test_shared_ivs_and_exact_pbs_count(pkg, engine_test, oracle_test):
    """Streams that pass the same encrypted-IV array share its 128 bit bootstraps: the PBS count of a call is
    128 * distinct IVs + (128 Nr + 15) * blocks, and for one stream it equals tfa_aes_ctr's."""
    o = oracle_test
    eng = engine_test
    rk, rk2 = round_keys(eng, o, KEY), round_keys(eng, o, bytes(range(16)))
    iv_a, iv_b, iv_c = 0x77, 2 ** 100 + 3, 0xFFFF_FFFF
    ct_a, ct_b, ct_c = enc_iv(o, iv_a), enc_iv(o, iv_b), enc_iv(o, iv_c)
    # two streams on one IV array, different first (and keys)
    c0 = eng.pbs_count
    got = eng.aes_ctr_streams([(rk, ct_a, 0, 2, None), (rk2, ct_a, 40, 3, None)])
    assert eng.pbs_count - c0 == pbs_expected(1, 5)
    check_streams(o, got, [(KEY, iv_a, 0, 2, None), (bytes(range(16)), iv_a, 40, 3, None)])
    # three IVs, one of them used twice
    c0 = eng.pbs_count
    got = eng.aes_ctr_streams([(rk, ct_b, 0, 1, None), (rk, ct_c, 7, 2, None), (rk2, ct_b, 9, 1, None)])
    assert eng.pbs_count - c0 == pbs_expected(2, 4)
    check_streams(o, got, [(KEY, iv_b, 0, 1, None), (KEY, iv_c, 7, 2, None), (bytes(range(16)), iv_b, 9, 1, None)])
    # one stream: the same count as tfa_aes_ctr
    c0 = eng.pbs_count
    eng.aes_ctr_streams([(rk, ct_c, 0, 3, None)])
    one = eng.pbs_count - c0
    c0 = eng.pbs_count
    pkg.Server(eng).aes_ctr(rk, ct_c, 3)
    assert one == eng.pbs_count - c0 == pbs_expected(1, 3)


@pytest.mark.gpu
@pytest.mark.parametrize("nbytes,rounds", [(24, 12), (32, 14)])
def test_aes_192_256(pkg, engine_test, oracle_test, nbytes, rounds):
    """FIPS-197 Appendix C.2 / C.3 keys: block 0 of the first stream is the Appendix C ciphertext; PBS count with Nr = 12 / 14."""
    o = oracle_test
    key = bytes(range(nbytes))
    rk = round_keys(engine_test, o, key)
    assert len(rk) == rounds + 1
    iv = int.from_bytes(bytes.fromhex("00112233445566778899aabbccddeeff"), "big")
    c0 = engine_test.pbs_count
    got = pkg.Server(engine_test).aes_ctr_streams([(rk, enc_iv(o, iv), 0, 2, None), (rk, enc_iv(o, 12345), 6, 1, None)])
    assert engine_test.pbs_count - c0 == pbs_expected(2, 3, rounds)
    assert o.decrypt_bytes(got[0]) == aes_clear.aes_encrypt_block(key, iv.to_bytes(16, "big"))
    check_streams(o, got, [(key, iv, 0, 2, None), (key, 12345, 6, 1, None)])


def _to_device(a, dev):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.uint64).view(np.int64).ravel().copy()).to(dev)


@pytest.mark.gpu
def test_device_variant_matches_host_variant(engine_test, oracle_test):
    """tfa_aes_ctr_streams_dev on torch CUDA tensors: the same decrypted bytes as the host entry point."""
    import torch
    o = oracle_test
    rk, rk2 = round_keys(engine_test, o, KEY), round_keys(engine_test, o, bytes(range(16)))
    ct1, ct2 = enc_iv(o, 0xFF), enc_iv(o, 77)
    data = bytes(range(48))
    host = engine_test.aes_ctr_streams([(rk, ct1, 0, 3, data), (rk2, ct2, 2, 2, None), (rk2, ct1, 5, 1, None)])
    dev = torch.device("cuda", 0)
    t_rk, t_rk2, t_ct1, t_ct2 = (_to_device(a, dev) for a in (rk, rk2, ct1, ct2))
    t_data = torch.tensor(list(data), dtype=torch.uint8, device=dev)
    t_out = torch.zeros(6 * 16 * 8 * engine_test.lw, dtype=torch.int64, device=dev)
    torch.cuda.synchronize()                                                   # the library runs on its own stream
    engine_test.aes_ctr_streams_dev([(t_rk.data_ptr(), t_ct1.data_ptr(), 0, 3, t_data.data_ptr()),
                                     (t_rk2.data_ptr(), t_ct2.data_ptr(), 2, 2, None),
                                     (t_rk2.data_ptr(), t_ct1.data_ptr(), 5, 1, None)], t_out.data_ptr())
    engine_test.synchronize()
    got = t_out.cpu().numpy().view(np.uint64).reshape(6, 16, 8, engine_test.lw)
    for b in range(6):
        assert o.decrypt_bytes(got[b]) == o.decrypt_bytes(host[b]), b
    check_streams(o, got, [(KEY, 0xFF, 0, 3, data), (bytes(range(16)), 77, 2, 2, None), (bytes(range(16)), 0xFF, 5, 1, None)])


@pytest.mark.gpu
def test_errors_leave_the_context_usable(pkg, engine_test, engine_test2, oracle_test):
    import torch
    o = oracle_test
    eng = engine_test
    rk, ct = round_keys(eng, o, KEY), enc_iv(o, 9)

    def still_works():
        got = eng.aes_ctr_streams([(rk, ct, 0, 2, None)])
        assert [o.decrypt_bytes(got[b]) for b in range(2)] == keystream(KEY, 9, 0, 2)

    bad = [([], 10),                                                           # no stream
           ([(rk, ct, 0, 0, None)], 10),                                       # empty stream
           ([(rk, ct, 0, 2, None), (rk, ct, 0, -1, None)], 10),                # negative length
           ([(None, ct, 0, 2, None)], 10),                                     # no round keys
           ([(rk, None, 0, 2, None)], 10),                                     # no encrypted IV
           ([(rk, ct, 0, 2 ** 30, None), (rk, ct, 0, 2 ** 30, None)], 10),     # total block count overflows int
           ([(rk, ct, 0, 2, None)], 11)]                                       # not AES-128/192/256
    for streams, rounds in bad:
        with pytest.raises(pkg.TfaError) as ei:
            eng.aes_ctr_streams(streams, rounds=rounds)
        assert ei.value.code == 1, (streams, rounds)
        still_works()
    dev = torch.device("cuda", 0)
    t_rk, t_ct = _to_device(rk, dev), _to_device(ct, dev)
    torch.cuda.synchronize()
    with pytest.raises(pkg.TfaError) as ei:                                    # no output buffer
        eng.aes_ctr_streams_dev([(t_rk.data_ptr(), t_ct.data_ptr(), 0, 1, None)], 0)
    assert ei.value.code == 1
    still_works()
    e = pkg.Engine(pkg.param_test())
    with pytest.raises(pkg.TfaError) as ei:                                    # keys not loaded
        e.aes_ctr_streams([(rk, ct, 0, 1, None)])
    assert ei.value.code == 3
    e.close()
    still_works()
    e2 = engine_test2
    zeros_rk = np.zeros((11, 16, 4, e2.lw), dtype=np.uint64)
    with pytest.raises(pkg.TfaError) as ei:                                    # 2-bit blocks
        e2.aes_ctr_streams([(zeros_rk, np.zeros((16, 4, e2.lw), dtype=np.uint64), 0, 1, None)])
    assert ei.value.code == 4
    still_works()


# ---- PARAM_OPT (client.rs:31-57) ------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.slow
def test_opt_three_streams_and_noise(pkg, engine_opt, oracle_opt):
    """Three streams with their own keys and encrypted IVs, 5 blocks in all, match FIPS-197.  Noise: every output LWE is an S-box
    output plus a round-key bit; its phase must lie at least 9 sigma inside the decision boundary 2^62, with sigma the standard
    deviation of one S-box output measured here as test_opt_noise_level5_state does (1 024 LWEs)."""
    o = oracle_opt
    srv = pkg.Server(engine_opt)
    keys = [bytes(16), KEY, bytes(range(100, 116))]
    ivs = [0, 0x0F0E0D0C_0B0A0908_07060504_030201FF, 2 ** 128 - 2]
    firsts = [1023, 0, 1]
    lens = [1, 2, 2]
    data = bytes((31 * i + 5) % 256 for i in range(32))
    clear = [(k, iv, f, n, data if i == 1 else None) for i, (k, iv, f, n) in enumerate(zip(keys, ivs, firsts, lens))]
    reqs = [(srv.aes_key_expansion(o.encrypt_bytes(k)), enc_iv(o, iv), f, n, d) for k, iv, f, n, d in clear]
    got = srv.aes_ctr_streams(reqs)
    check_streams(o, got, clear)
    assert o.decrypt_bytes(got[0]).hex() == "09836c44648b1f262e7b8bb6310e3c73"   # SURVEY §4: key 0, iv 0, counter 1023
    _, err = o.decrypt_bits(got, with_err=True)
    assert len(err) == 5 * 128
    rng = np.random.default_rng(204)
    one = engine_opt.sbox(o.encrypt_bytes(bytes(rng.integers(0, 256, 128, dtype=np.uint8))), False)
    sigma = o.decrypt_bits(one, with_err=True)[1].astype(np.float64).std()
    margin = 2.0 ** 62 - np.abs(err.astype(np.float64))
    assert margin.min() >= 9 * sigma, (margin.min() / sigma)
