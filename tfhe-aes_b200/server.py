"""Host-side mirror of the reference's `Server` (src/server/server.rs) and `sbox` module
(src/server/sbox/{sbox,many_wopbs,gen_lut}.rs) on top of the C ABI — same method names, argument
order and meaning, so parity tests read like the reference's own driver (main.rs:33-72, :76-142).

Ciphertext containers are numpy uint64 arrays in tfhe-rs's flat layout:
  radix byte  = [8][lw]          (BaseRadixCiphertext<Ciphertext>, block j = bit j)
  state       = [16][8][lw]      (Vec<BaseRadixCiphertext>)
  round keys  = [11][16][8][lw]  (Vec<Vec<BaseRadixCiphertext>>)
Errors surface as exceptions (the reference panics).
"""
import numpy as np
from . import binding as _b


def many_wopbs_without_padding(engine, ct_in, luts):
    """many_wopbs.rs:31 — one radix ciphertext [nblocks][lw], list of LUTs -> list of radix ciphertexts."""
    ct = np.ascontiguousarray(ct_in, dtype=np.uint64)[None]
    out = engine.many_wopbs(ct, np.stack([np.asarray(l) for l in luts]))
    return [out[0, i] for i in range(out.shape[1])]


def sbox(engine, ct_in, inv):
    """sbox.rs:46 — returns the new byte (the reference assigns in place)."""
    return engine.sbox(ct_in, inv)[0]


def many_sbox(engine, ct_in, inv):
    """sbox.rs:68 — [S, 2S, 3S] or [9x, 11x, 13x, 14x]."""
    out = engine.many_sbox(ct_in, inv)
    return [out[0, i] for i in range(out.shape[1])]


class Server:
    """server.rs:24-35.  `engine` plays the role of (public_key, sks, wopbs_key): it owns the
    bootstrap / keyswitch / PFKS keys on the GPU."""

    def __init__(self, engine: _b.Engine):
        self.engine = engine

    def aes_key_expansion(self, key):
        """server.rs:107 — key: [16][8][lw] -> [11][16][8][lw]"""
        return self.engine.aes_key_expansion(key)

    def aes_encrypt(self, encrypted_round_keys, state):
        """server.rs:39 — returns the new state(s); accepts one state or a batch [nblk][16][8][lw]."""
        st = np.asarray(state)
        out = self.engine.aes_encrypt(encrypted_round_keys, st)
        return out[0] if st.ndim == 3 else out

    def aes_decrypt(self, encrypted_round_keys, state):
        """server.rs:67"""
        st = np.asarray(state)
        out = self.engine.aes_decrypt(encrypted_round_keys, st)
        return out[0] if st.ndim == 3 else out

    # README.md:58-59 spellings
    aes_encryption = aes_encrypt
    aes_decryption = aes_decrypt

    def add_scalar(self, state, i):
        """server.rs:172 — state + i (u128).  Uses i & 0xFF in the low byte (correct for i >= 256)."""
        st = np.asarray(state)
        if st.ndim == 3:
            return self.engine.add_scalar(st, [i])[0]
        return self.engine.add_scalar(st, list(i))

    def aes_ctr(self, encrypted_round_keys, encrypted_iv, number_of_outputs, first=0):
        """main.rs:55-64 — the CTR loop, all blocks in one batched call."""
        return self.engine.aes_ctr(encrypted_round_keys, encrypted_iv, first, number_of_outputs)

    def aes_ctr_public_iv(self, encrypted_round_keys, iv, number_of_outputs, first=0, data=None):
        """AES-CTR with the IV in the clear (only the AES key is encrypted): Enc(AES(iv + first + b) XOR data[b]) for
        b < number_of_outputs; data None gives the bare keystream.  AES-128/192/256 follow from the number of round keys."""
        rk = np.asarray(encrypted_round_keys)
        rounds = rk.size // (16 * 8 * self.engine.lw) - 1
        return self.engine.aes_ctr_public_iv([(rk, iv, first, number_of_outputs, data)], rounds)
