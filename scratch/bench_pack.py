#!/usr/bin/env python
"""GLWE packing of transciphered data at PARAM_OPT on one GPU: 148 AES-128-CTR blocks (18 944 LWEs) from one
tfa_aes_ctr_public_iv_dev call, packed into 37 GLWEs of 16-bit words with tfa_pack_lwe_dev and unpacked with tfa_unpack_lwe_dev.

Measured in one run, with CUDA events on the library's stream:
  * the transciphering call itself (best of --ctr-reps), the denominator of the pack-time fraction;
  * pack_dev and unpack_dev, best of --reps after two warm-up calls (the 310 MB input does not fit the 126 MB L2);
  * a device-to-host copy into pinned memory of the unpacked batch (310 MB) and of the packed batch (189 KB), best of --reps.
FHE keys come from the client harness; the round keys are the FIPS-197 expansion of the AES key encrypted by the client harness,
and the clear data is the client's AES-CTR ciphertext of a known message, so every output decrypts to that message.  Every
packed output is decrypted twice: as GLWEs with the client's GLWE secret key in numpy (the widened words v << 48 are multiples of
2^48, so the phase is exact modulo 2^16), and after unpacking with the client harness.  Prints one JSON line; --out also writes it.

  python scratch/bench_pack.py [--reps 10] [--ctr-reps 2] [--out FILE]
"""
import argparse
import importlib.util
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests"))
import aes_clear  # noqa: E402

NBLK = 148


def load_pkg():
    d = os.path.join(ROOT, "tfhe-aes_b200")
    spec = importlib.util.spec_from_file_location("tfhe_aes_b200", os.path.join(d, "__init__.py"), submodule_search_locations=[d])
    m = importlib.util.module_from_spec(spec)
    sys.modules["tfhe_aes_b200"] = m
    spec.loader.exec_module(m)
    return m


def gpu_info():
    """name, power limit and maximum SM clock (query only)"""
    try:
        r = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        name, power, clock = [x.strip() for x in r.stdout.strip().split(",")]
        return {"gpu": name, "power_limit": power, "sm_clock_max": clock}
    except Exception as e:  # noqa: BLE001
        return {"gpu": None, "nvidia_smi_error": str(e)}


def glwe_decrypt_bytes(packed, glwe_sk, k, N, count):
    """bytes of the first `count` bits of packed [G][k+1][N] uint16, under the GLWE key [k][N] (bits LSB first per byte)"""
    a = packed.astype(np.int64)
    ph = a[:, k, :].copy()
    for r in range(k):
        s = glwe_sk[r * N:(r + 1) * N].astype(np.int64)
        # negacyclic matrix: (A . S)[c] = sum_t A[t] * M[t][c], M[t][c] = s[c - t] for c >= t, -s[N + c - t] otherwise
        t, c = np.meshgrid(np.arange(N), np.arange(N), indexing="ij")
        m = np.where(c >= t, s[(c - t) % N], -s[(c - t) % N])
        ph -= a[:, r, :] @ m
    ph &= 0xFFFF
    bits = (((ph + (1 << 14)) >> 15) & 1).ravel()[:count].reshape(-1, 8)
    return bytes(int(sum(int(b) << j for j, b in enumerate(byte))) for byte in bits)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--ctr-reps", type=int, default=2)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    pkg = load_pkg()
    dev = torch.device("cuda", 0)
    stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(stream)
    eng = pkg.Engine(pkg.param_opt(), device=0, stream=stream.cuda_stream)
    lw, k, N = eng.lw, eng.k, eng.N
    count = 128 * NBLK
    G = eng.packed_glwes(count)
    eng.client_keygen(7)
    _, glwe_sk = eng.client_secret_keys()
    rng = np.random.default_rng(3)
    key = bytes(rng.integers(0, 256, 16, dtype=np.uint8))
    iv = int.from_bytes(bytes(rng.integers(0, 256, 16, dtype=np.uint8)), "big")
    msg = bytes(rng.integers(0, 256, 16 * NBLK, dtype=np.uint8))
    data = b"".join(aes_clear.xor(aes_clear.ctr_block(key, iv, b), msg[16 * b:16 * b + 16]) for b in range(NBLK))
    rk = torch.zeros(11 * 16 * 8 * lw, dtype=torch.int64, device=dev)
    eng.client_encrypt_bytes_dev(b"".join(aes_clear.round_keys(key)), rk.data_ptr(), seed=11)
    t_data = torch.tensor(list(data), dtype=torch.uint8, device=dev)
    ct = torch.zeros(count * lw, dtype=torch.int64, device=dev)
    packed = torch.zeros(G * (k + 1) * N, dtype=torch.int16, device=dev)
    unpacked = torch.zeros(count * lw, dtype=torch.int64, device=dev)
    h_unpacked = torch.empty(count * lw, dtype=torch.int64, pin_memory=True)
    h_packed = torch.empty(G * (k + 1) * N, dtype=torch.int16, pin_memory=True)
    torch.cuda.synchronize()

    def timed(fn):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream)
        fn()
        b.record(stream)
        b.synchronize()
        return a.elapsed_time(b) / 1e3

    t0 = time.perf_counter()
    ctr = lambda: eng.aes_ctr_public_iv_dev([(rk.data_ptr(), iv, 0, NBLK, t_data.data_ptr())], ct.data_ptr())  # noqa: E731
    ctr_s = [timed(ctr) for _ in range(args.ctr_reps)]
    assert eng.client_decrypt_bytes_dev(ct.data_ptr(), 16 * NBLK) == msg, "transciphered blocks differ from the message"

    pack = lambda: eng.pack_lwe_dev(ct.data_ptr(), count, packed.data_ptr())  # noqa: E731
    unpack = lambda: eng.unpack_lwe_dev(packed.data_ptr(), count, unpacked.data_ptr())  # noqa: E731
    for _ in range(2):
        timed(pack)
        timed(unpack)
    pack_s, unpack_s = [], []
    for _ in range(args.reps):                   # alternated
        pack_s.append(timed(pack))
        unpack_s.append(timed(unpack))
    d2h_unpacked_s = [timed(lambda: h_unpacked.copy_(unpacked, non_blocking=True)) for _ in range(args.reps)]
    d2h_packed_s = [timed(lambda: h_packed.copy_(packed, non_blocking=True)) for _ in range(args.reps)]

    p = h_packed.numpy().view(np.uint16).reshape(G, k + 1, N)
    assert glwe_decrypt_bytes(p, glwe_sk, k, N, count) == msg, "packed GLWEs do not decrypt to the message"
    assert eng.client_decrypt_bytes_dev(unpacked.data_ptr(), 16 * NBLK) == msg, "unpacked LWEs do not decrypt to the message"
    assert np.array_equal(h_unpacked.numpy().view(np.uint64).reshape(count, lw), eng.unpack_lwe(p, count))

    packed_bytes, unpacked_bytes = G * (k + 1) * N * 2, count * lw * 8
    line = {
        "workload": f"GLWE packing of {NBLK} transciphered AES-128-CTR blocks ({count} LWEs, {G} GLWEs), PARAM_OPT n=669 k=4 N=512, "
                    "client-harness keys",
        **gpu_info(), "torch_device": torch.cuda.get_device_name(0),
        "reps": args.reps,
        "timing": "CUDA events on the library stream around each call; best of reps after 2 warm-up calls (all reps listed); pack and "
                  "unpack alternate; the 310 MB pack input and unpack output exceed the 126 MB L2",
        "verified": "transciphered blocks, packed GLWEs (numpy decryption with the GLWE secret key) and unpacked LWEs all decrypt to the "
                    "message; the device unpack equals the host unpack of the same words",
        "aes_ctr_public_iv_s": [round(x, 4) for x in ctr_s],
        "pack_dev_ms": round(min(pack_s) * 1e3, 3), "pack_dev_ms_all": [round(x * 1e3, 3) for x in pack_s],
        "pack_ms_per_6144_bits": round(min(pack_s) * 1e3 * 6144 / count, 3),
        "unpack_dev_ms": round(min(unpack_s) * 1e3, 3), "unpack_dev_ms_all": [round(x * 1e3, 3) for x in unpack_s],
        "unpack_write_gb_s": round(unpacked_bytes / min(unpack_s) / 1e9, 1),
        "pack_fraction_of_ctr_call": round(min(pack_s) / min(ctr_s), 5),
        "d2h_pinned_unpacked_ms": round(min(d2h_unpacked_s) * 1e3, 3), "d2h_pinned_packed_ms": round(min(d2h_packed_s) * 1e3, 4),
        "unpacked_bytes": unpacked_bytes, "packed_bytes": packed_bytes,
        "bytes_per_block_unpacked": unpacked_bytes // NBLK, "bytes_per_block_packed": packed_bytes // NBLK,
        "size_ratio": round(unpacked_bytes / packed_bytes, 1),
        "wall_s": round(time.perf_counter() - t0, 1),
    }
    s = json.dumps(line)
    print(s)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(s + "\n")
    eng.close()


if __name__ == "__main__":
    main()
