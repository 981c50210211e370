#!/usr/bin/env python
"""AES-128-CTR with encrypted IVs at PARAM_OPT on one GPU: many streams in ONE tfa_aes_ctr_streams_dev call against the same
streams as one tfa_aes_ctr_dev call each (what a server without the batched entry point issues per request).

Configurations (streams x blocks per stream): 148 x 1, 37 x 4, 16 x 9 and 1 x 148.  Every stream has its own AES key and its own
encrypted IV and counter start.  FHE keys come from the client harness; the round keys are the FIPS-197 expansion of each AES key
encrypted by the client harness (how the round keys were made does not change what the server evaluates).  Both arms write the
bare keystream into the same output buffer, so they do the same work and the same PBS count: 128 per stream for its IV plus
(128 * 10 + 15) per block.  The two arms alternate after one warm-up round of every configuration; each arm is timed with CUDA
events on the library's stream.  PBS are counted with tfa_ctx_pbs_count and checked against that formula, and every output block
of every call is decrypted and compared with FIPS-197 (tests/aes_clear.py).  Prints one JSON line; --out also writes it to a file.

  python scratch/bench_ctr_streams.py [--reps 2] [--out FILE]
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

CONFIGS = [(148, 1), (37, 4), (16, 9), (1, 148)]


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


def pbs_formula(distinct_ivs, blocks, rounds=10):
    return 128 * distinct_ivs + (128 * rounds + 15) * blocks


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=2)
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
    lw = eng.lw
    sw = 16 * 8 * lw
    eng.client_keygen(7)
    nmax = max(s for s, _ in CONFIGS)
    bmax = max(s * n for s, n in CONFIGS)
    rng = np.random.default_rng(9)
    keys = [bytes(rng.integers(0, 256, 16, dtype=np.uint8)) for _ in range(nmax)]
    ivs = [int.from_bytes(bytes(rng.integers(0, 256, 16, dtype=np.uint8)), "big") for _ in range(nmax)]
    firsts = [int(rng.integers(0, 2 ** 40)) for _ in range(nmax)]
    rk = torch.zeros(nmax * 11 * sw, dtype=torch.int64, device=dev)
    iv_ct = torch.zeros(nmax * sw, dtype=torch.int64, device=dev)
    for s in range(nmax):
        eng.client_encrypt_bytes_dev(b"".join(aes_clear.round_keys(keys[s])), rk.data_ptr() + s * 11 * sw * 8, seed=1000 + s)
        eng.client_encrypt_bytes_dev(ivs[s].to_bytes(16, "big"), iv_ct.data_ptr() + s * sw * 8, seed=2000 + s)
    out = torch.zeros(bmax * sw, dtype=torch.int64, device=dev)
    torch.cuda.synchronize()

    def streams_of(S, n):
        return [(rk.data_ptr() + s * 11 * sw * 8, iv_ct.data_ptr() + s * sw * 8, firsts[s], n, None) for s in range(S)]

    def batched(S, n):
        eng.aes_ctr_streams_dev(streams_of(S, n), out.data_ptr())

    def separate(S, n):
        for s, (r, iv, first, nb, _) in enumerate(streams_of(S, n)):
            eng.aes_ctr_dev(r, iv, first, nb, out.data_ptr() + s * n * sw * 8)

    def check(name, S, n):
        got = eng.client_decrypt_bytes_dev(out.data_ptr(), 16 * S * n)
        want = b"".join(aes_clear.ctr_block(keys[s], ivs[s], firsts[s] + b) for s in range(S) for b in range(n))
        assert got == want, f"{name} {S}x{n}: output differs from FIPS-197"

    def timed(name, fn, S, n):
        out.zero_()
        c0 = eng.pbs_count
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream)
        fn(S, n)
        b.record(stream)
        torch.cuda.synchronize()
        pbs = eng.pbs_count - c0
        assert pbs == pbs_formula(S, S * n), f"{name} {S}x{n}: {pbs} PBS, formula {pbs_formula(S, S * n)}"
        check(name, S, n)
        return a.elapsed_time(b) / 1e3

    arms = {"batched": batched, "separate": separate}
    t0 = time.perf_counter()
    for S, n in CONFIGS:                    # warm-up of every shape
        for name, fn in arms.items():
            timed(name, fn, S, n)
    res = {f"{S}x{n}": {name: [] for name in arms} for S, n in CONFIGS}
    for _ in range(args.reps):              # alternated
        for S, n in CONFIGS:
            for name, fn in arms.items():
                res[f"{S}x{n}"][name].append(timed(name, fn, S, n))
    configs = {}
    for S, n in CONFIGS:
        r = res[f"{S}x{n}"]
        c = {"streams": S, "blocks_per_stream": n, "pbs": pbs_formula(S, S * n)}
        for name in arms:
            best = min(r[name])
            c[name] = {"call_s": [round(x, 4) for x in r[name]], "blocks_per_s": round(S * n / best, 2)}
        c["speedup"] = round(min(r["separate"]) / min(r["batched"]), 3)
        configs[f"{S}x{n}"] = c
    line = {
        "workload": "AES-128-CTR keystream with encrypted IVs, PARAM_OPT n=669 k=4 N=512, client-harness keys; every stream its own "
                    "AES key, encrypted IV and counter start; batched = one tfa_aes_ctr_streams_dev call, separate = one "
                    "tfa_aes_ctr_dev call per stream",
        **gpu_info(), "torch_device": torch.cuda.get_device_name(0),
        "reps": args.reps, "timing": "CUDA events on the library stream around each arm; best of reps (all reps listed)",
        "verified": "every output block of every call decrypted and compared with FIPS-197; PBS count of every call equal to "
                    "128 * streams + 1295 * blocks",
        "configs": configs,
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
