#!/usr/bin/env python
"""AES-128-CTR at PARAM_OPT on one GPU: the encrypted-IV path (tfa_aes_ctr_dev: counter add + 10 rounds) against the public-IV
path (tfa_aes_ctr_public_iv_dev: no counter add, the first two rounds once per run of <= 256 counters).

Both paths run on the same keys (client harness), the same AES key and IV, 148 blocks per call (one run), alternated after a
warm-up; CUDA events on the library's stream.  PBS per block are counted with tfa_ctx_pbs_count.  Every output block of every
call is decrypted and compared with FIPS-197 (tests/aes_clear.py).  Also: single-block latency of both paths and the per-stage
split of one un-timed call of each (tfa_ctx_profile_report).  Prints one JSON line; --out also writes it to a file.

  python scratch/bench_ctr_public_iv.py [--blocks 148] [--reps 3] [--out FILE]
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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--blocks", type=int, default=148)
    ap.add_argument("--reps", type=int, default=3)
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
    lw, B = eng.lw, args.blocks
    sw = 16 * 8 * lw
    eng.client_keygen(7)
    key = bytes(range(16))
    iv = int.from_bytes(bytes.fromhex("f0e1d2c3b4a5968778695a4b3c2d1e0f"), "big")   # low byte 0x0F: 148 blocks stay in one run
    key_ct = torch.zeros(sw, dtype=torch.int64, device=dev)
    iv_ct = torch.zeros(sw, dtype=torch.int64, device=dev)
    rk = torch.zeros(11 * sw, dtype=torch.int64, device=dev)
    eng.client_encrypt_bytes_dev(key, key_ct.data_ptr(), seed=11)
    eng.client_encrypt_bytes_dev(iv.to_bytes(16, "big"), iv_ct.data_ptr(), seed=12)
    eng.aes_key_expansion_dev(key_ct.data_ptr(), rk.data_ptr())
    rng = np.random.default_rng(5)
    msg = bytes(rng.integers(0, 256, 16 * B, dtype=np.uint8))
    ks = b"".join(aes_clear.ctr_block(key, iv, b) for b in range(B))
    data = torch.tensor(list(aes_clear.xor(msg, ks)), dtype=torch.uint8, device=dev)
    out = torch.zeros(B * sw, dtype=torch.int64, device=dev)
    torch.cuda.synchronize()

    def enc_iv(n):
        eng.aes_ctr_dev(rk.data_ptr(), iv_ct.data_ptr(), 0, n, out.data_ptr())

    def pub_iv(n):
        eng.aes_ctr_public_iv_dev([(rk.data_ptr(), iv, 0, n, data.data_ptr())], out.data_ptr())

    def check(name, n):
        got = eng.client_decrypt_bytes_dev(out.data_ptr(), 16 * n)
        want = msg[:16 * n] if name == "public_iv" else ks[:16 * n]
        assert got == want, f"{name}: output differs from FIPS-197"

    def timed(name, fn, n):
        c0 = eng.pbs_count
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream)
        fn(n)
        b.record(stream)
        torch.cuda.synchronize()
        pbs = eng.pbs_count - c0
        check(name, n)
        return a.elapsed_time(b) / 1e3, pbs

    paths = {"encrypted_iv": enc_iv, "public_iv": pub_iv}
    t0 = time.perf_counter()
    for name, fn in paths.items():          # warm-up of both shapes
        timed(name, fn, B)
        timed(name, fn, 1)
    res = {name: {"s": [], "pbs": None, "latency_1blk_s": []} for name in paths}
    for _ in range(args.reps):              # alternated
        for name, fn in paths.items():
            s, pbs = timed(name, fn, B)
            res[name]["s"].append(s)
            res[name]["pbs"] = pbs
    for _ in range(args.reps):
        for name, fn in paths.items():
            s, pbs1 = timed(name, fn, 1)
            res[name]["latency_1blk_s"].append(s)
            res[name]["pbs_1blk"] = pbs1
    split = {}
    for name, fn in paths.items():          # one profiled call each, not part of the timings above
        eng.profile(True)
        fn(B)
        split[name] = {k: round(v[0], 2) for k, v in eng.profile_report().items()}
        eng.profile(False)
        torch.cuda.synchronize()
        check(name, B)
    summary = {}
    for name, r in res.items():
        best = min(r["s"])
        summary[name] = {"blocks_per_s": round(B / best, 2), "blocks_per_s_median": round(B / float(np.median(r["s"])), 2),
                         "call_s": [round(x, 4) for x in r["s"]], "pbs_per_block": round(r["pbs"] / B, 2),
                         "latency_1blk_s": round(min(r["latency_1blk_s"]), 4), "pbs_1blk": r["pbs_1blk"],
                         "stage_ms": split[name]}
    line = {
        "workload": f"AES-128-CTR, {B} blocks per call in one run of counters, PARAM_OPT n=669 k=4 N=512, keys from the client harness",
        **gpu_info(), "torch_device": torch.cuda.get_device_name(0),
        "reps": args.reps, "timing": "CUDA events on the library stream around one call; best of reps (median also given)",
        "verified": "every output block of every call decrypted and compared with FIPS-197",
        **summary,
        "speedup_blocks_per_s": round(summary["public_iv"]["blocks_per_s"] / summary["encrypted_iv"]["blocks_per_s"], 3),
        "time_ratio": round(1 / (summary["public_iv"]["blocks_per_s"] / summary["encrypted_iv"]["blocks_per_s"]), 3),
        "pbs_ratio": round(summary["public_iv"]["pbs_per_block"] / summary["encrypted_iv"]["pbs_per_block"], 3),
        "latency_ratio_1blk": round(summary["public_iv"]["latency_1blk_s"] / summary["encrypted_iv"]["latency_1blk_s"], 3),
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
