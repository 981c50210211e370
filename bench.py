#!/usr/bin/env python
"""bench.py — FHE AES-128-CTR blocks/s (and WoPBS S-box evaluations/s) on N B200s.

One "step" = one batched pass of the hot path: `blocks_per_gpu` CTR blocks per GPU, each
add_scalar (server.rs:172) + aes_encrypt (server.rs:39) = 176 byte-WoPBS at PARAM_OPT (client.rs:31-57).
Run block by block as the reference does that is 1 423 PBS per block; the batched CTR entry point circuit-
bootstraps the 128 bits of the encrypted IV once per call (all blocks start from the same IV, main.rs:59), so a
block costs 1 280 (aes_encrypt) + 15 (carry bits of add_scalar) + 128 / blocks PBS.  Blocks are sharded across ranks by counter (main.rs:55-64); keys are generated on
rank 0 and replicated with one NCCL broadcast; there is no collective on the per-step path.

  python bench.py --gpus N --steps K --warmup W            (N>1: launched with torchrun)
  python bench.py ... --dump-outputs DIR                    also writes the output states of the last timed step
                                                            as .npy files, to compare two builds output for output
  python bench.py --impl reference ...                      CPU arm: the oracle port of the reference's
                                                            CPU path on all host threads (rank 0 only)
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

PBS_FLOP = 407_608_320           # SURVEY §8d: FP64 flops of one PBS at PARAM_OPT
SBOX_FLOP_L3 = 3_295_662_080     # one S-box evaluation with 3 LUTs
WOPBS_PER_BLOCK = 176            # 160 (aes_encrypt) + 16 (add_scalar) byte-WoPBS per CTR block
PBS_PER_BLOCK_REFERENCE = 1423   # block-by-block schedule of the reference (1 280 + 143)


def pbs_per_block(blocks):       # batched tfa_aes_ctr: IV bits bootstrapped once per call
    return 1280 + 15 + 128.0 / blocks


BSK_BYTES = 342_528_000
NCU_DRAM_BYTES_PER_WAVE = 354_475_264   # ncu --set full, pbs_ws2_kernel<4,3,2,8,5>, 148 CTAs x 6 ciphertexts (profiles/r2_pbs_ws2_kernel_ncu.txt: 348.85 MB read + 5.62 MB written)
PBS_WAVE = 6 * 148                      # ciphertexts per wave of the dominant kernel
METRIC = "aes128_ctr_blocks_per_s"
UNIT = "blocks/s"


def load_pkg():
    from __graft_entry__ import load_package
    return load_package()


class ClockSampler(threading.Thread):
    """nvidia-smi clocks + throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.stop_flag = index, [], False

    def run(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}", "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            time.sleep(0.2)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        sm = sorted(float(r[0]) for r in self.rows if r[0].replace(".", "").isdigit())
        reasons = []
        for i, name in enumerate(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")):
            if any(len(r) > 3 + i and r[3 + i].lower().startswith("active") for r in self.rows):
                reasons.append(name)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": float(self.rows[0][1]) if self.rows[0][1].replace(".", "").isdigit() else None,
                "power_w_max": max((float(r[2]) for r in self.rows if r[2].replace(".", "").isdigit()), default=None),
                "samples": len(self.rows), "reasons": reasons}


# ----------------------------------------------------------------------------------------------------
# CPU arm: the oracle port of the reference's CPU path (the reference itself is Rust over tfhe-rs and
# cannot be built here — no cargo, crate not vendored).  Structure of main.rs:55-64: one worker per
# block, each single-threaded; a bounded sample (one many_sbox per worker per step) scaled by counts.
# ----------------------------------------------------------------------------------------------------
_CPU = {}


def cpu_sample(evals_per_thread=1, threads=None):
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import orc
    from concurrent.futures import ThreadPoolExecutor
    threads = threads or os.cpu_count()
    if "o" not in _CPU:
        _CPU["o"] = orc.Oracle(orc.param_opt(), seed=11)   # keygen uses OpenMP internally (untimed)
        orc.lib().orc_set_threads(1)                        # each worker single-threaded, as the reference (main.rs:32)
    o = _CPU["o"]
    cts = o.encrypt_bytes(bytes(i % 256 for i in range(threads)))

    def work(i):
        orc.lib().orc_set_threads(1)                        # OpenMP ICVs are per thread: pin every worker to one
        for _ in range(evals_per_thread):
            out = o.many_sbox(cts[i], False)        # ctypes releases the GIL during the call
        return out
    t0 = time.perf_counter()
    with ThreadPoolExecutor(threads) as ex:
        outs = list(ex.map(work, range(threads)))
    dt = time.perf_counter() - t0
    sb = orc.sbox_table()
    assert o.decrypt_bytes(outs[0])[0] == sb[0]
    evals_per_s = threads * evals_per_thread / dt
    return {"evals_per_s": evals_per_s, "blocks_per_s": evals_per_s / WOPBS_PER_BLOCK, "seconds": dt, "threads": threads,
            "sample": f"{threads} workers x {evals_per_thread} many_sbox (L=3, PARAM_OPT) in parallel, 1 thread each; blocks/s = evals/s / {WOPBS_PER_BLOCK}"}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    vals = []
    nwarm = max(args.warmup_ref, min(args.warmup, 3))   # a CPU sample is ~2 s: honour --warmup up to 3 samples
    for _ in range(nwarm):
        cpu_sample(1)
    t_all = time.perf_counter()
    for _ in range(args.steps):
        r = cpu_sample(1)
        vals.append(r)
    per_step = (time.perf_counter() - t_all) / max(1, args.steps)
    v = float(np.mean([r["blocks_per_s"] for r in vals]))
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": nwarm,
            "ms_per_step": per_step * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u64+f64", "data": "synthetic",
            "config": {"workload": f"aes128_ctr (add_scalar + aes_encrypt = {WOPBS_PER_BLOCK} byte-WoPBS = {PBS_PER_BLOCK_REFERENCE} PBS per block), PARAM_OPT n=669 k=4 N=512; CPU port of the reference path (oracle), bounded sample scaled by the WoPBS count",
                       "note": "the Rust reference (tfhe-rs 0.11.2) cannot be built in this image; README.md:186 quotes 84 s/block/core"},
            "sbox_evals_per_s": float(np.mean([r["evals_per_s"] for r in vals])),
            "cpu_baseline": {"value": v, "unit": UNIT, "cores": vals[0]["threads"], "kind": "port", "sample": vals[0]["sample"]},
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


# ----------------------------------------------------------------------------------------------------
# Expected values: tests/aes_clear.py = FIPS-197 with a hard-coded S-box, cross-checked against the `cryptography` package
# when it is importable.  Nothing of the product (its S-box tables, its decryption kernel) takes part in the check:
# ciphertexts are copied to the host and decrypted here with numpy from the secret key (client.rs:147-175).
sys.path.insert(0, os.path.join(ROOT, "tests"))
import aes_clear  # noqa: E402


def numpy_phases(ct, glwe_sk):
    """b - <a, s> (message + noise) of every LWE of ct [..][lw] uint64, as uint64"""
    ct = ct.reshape(-1, ct.shape[-1])
    with np.errstate(over="ignore"):
        return ct[:, -1] - (ct[:, :-1] * glwe_sk).sum(axis=1, dtype=np.uint64)


def numpy_decrypt_bytes(ct, glwe_sk):
    """decrypt_without_padding on the host: ct [..][8][lw] uint64, bit j of a byte in LWE j (client.rs:154)"""
    with np.errstate(over="ignore"):
        bits = ((numpy_phases(ct, glwe_sk) + np.uint64(1 << 62)) >> np.uint64(63)).astype(np.uint8) & 1
    return bytes(np.packbits(bits.reshape(-1, 8), axis=1, bitorder="little").ravel())


DUMP_LWE_ROWS = 1024          # whole output LWEs written by --dump-outputs: 1024 x 2049 words = 16.8 MB in float64
DUMP_PHASES_MAX = 1 << 22     # phases written (32 MB in float64); a larger step writes a seeded sample of this many


def torus_f64(x):
    """uint64 torus elements -> float64 in [-0.5, 0.5): x / 2^64 read as signed (the low ~11 bits of a word are rounded)"""
    return np.asarray(x, dtype=np.uint64).view(np.int64).astype(np.float64) * 2.0 ** -64


def dump_outputs(path, ct, glwe_sk):
    """Write the output states of one step, ct [blocks][16][8][lw] uint64, as float64 .npy files under path:
    ciphertexts.npy  [rows][lw]   a sample of the output LWEs, rows drawn with np.random.default_rng(0), sorted;
    phases.npy       [blocks][16][8] the phase (message + noise) of every output LWE; past DUMP_PHASES_MAX LWEs,
                     a flat sample drawn with np.random.default_rng(1), sorted.
    Both are torus values in [-0.5, 0.5).  The samples depend only on the shape, so runs with the same arguments
    write the same elements."""
    os.makedirs(path, exist_ok=True)
    lwes = ct.reshape(-1, ct.shape[-1])
    n = lwes.shape[0]
    rows = np.arange(n) if n <= DUMP_LWE_ROWS else np.sort(np.random.default_rng(0).choice(n, DUMP_LWE_ROWS, replace=False))
    np.save(os.path.join(path, "ciphertexts.npy"), torus_f64(lwes[rows]))
    ph = numpy_phases(lwes, glwe_sk)
    if n <= DUMP_PHASES_MAX:
        ph = ph.reshape(ct.shape[:-1])
    else:
        ph = ph[np.sort(np.random.default_rng(1).choice(n, DUMP_PHASES_MAX, replace=False))]
    np.save(os.path.join(path, "phases.npy"), torus_f64(ph))


class DevPtrArray:
    """numpy-free view of a raw device allocation for torch.as_tensor (CUDA array interface)."""

    def __init__(self, ptr, nbytes):
        self.__cuda_array_interface__ = {"shape": (nbytes,), "typestr": "|u1", "data": (ptr, False), "version": 2}


def run_gpu(args):
    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world > 1:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product has no CPU path (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    pkg = load_pkg()
    # every kernel of the library runs on this (non-default) stream; the timing events are recorded on it too
    stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(stream)
    eng = pkg.Engine(pkg.param_opt(), device=local, stream=stream.cuda_stream)
    lw, B = eng.lw, args.blocks_per_gpu
    strong = args.total_blocks > 0          # BASELINE config 5: a fixed number of blocks split over the GPUs (main.rs:55-64 with --number-of-outputs)
    shard_start = 0
    if strong:
        shard_start, B = pkg.sharding.shard_range(args.total_blocks, rank, world)
        if B == 0:
            raise SystemExit("--total-blocks smaller than the number of GPUs")
    blocks_per_step = args.total_blocks if strong else B * world
    state_words = 16 * 8 * lw

    # ---- keys: generated on rank 0 (client harness), replicated by ONE NCCL broadcast -------------------
    t0 = time.perf_counter()
    if rank == 0:
        eng.client_keygen(args.seed)
    else:
        eng.alloc_keys()
    key_bytes = 0
    if world > 1:
        key_bytes = pkg.sharding.replicate_keys(eng, dist, rank, src=0, device=dev)   # ONE NCCL broadcast per key buffer
        sk = [torch.zeros(eng.n, dtype=torch.int64, device=dev), torch.zeros(eng.big, dtype=torch.int64, device=dev)]
        if rank == 0:
            a, b = eng.client_secret_keys()
            sk[0].copy_(torch.from_numpy(a.view(np.int64)))
            sk[1].copy_(torch.from_numpy(b.view(np.int64)))
        for t in sk:
            dist.broadcast(t, src=0)   # harness only: lets every rank verify its own blocks
        torch.cuda.synchronize()
        if rank != 0:
            eng.client_set_secret_keys(sk[0].cpu().numpy().view(np.uint64), sk[1].cpu().numpy().view(np.uint64))
    torch.cuda.synchronize()
    keygen_s = time.perf_counter() - t0

    # ---- AES key + IV: encrypted by the client, round keys expanded once on rank 0, broadcast -------------
    aes_key = bytes(range(16)) if args.key is None else args.key.to_bytes(16, "big")
    iv = args.iv.to_bytes(16, "big")
    rk = torch.zeros(11 * state_words, dtype=torch.int64, device=dev)
    iv_ct = torch.zeros(state_words, dtype=torch.int64, device=dev)
    t0 = time.perf_counter()
    if rank == 0:
        key_ct = torch.zeros(state_words, dtype=torch.int64, device=dev)
        eng.client_encrypt_bytes_dev(aes_key, key_ct.data_ptr(), seed=101)
        eng.client_encrypt_bytes_dev(iv, iv_ct.data_ptr(), seed=102)
        eng.aes_key_expansion_dev(key_ct.data_ptr(), rk.data_ptr())
        torch.cuda.synchronize()
    keyexp_s = time.perf_counter() - t0
    if world > 1:
        dist.broadcast(rk, src=0)
        dist.broadcast(iv_ct, src=0)
    out = torch.zeros(B * state_words, dtype=torch.int64, device=dev)

    glwe_sk = eng.client_secret_keys()[1]

    def expected(counter):
        # FIPS-197 AES-128 in the clear (what client.rs:163-171 gets from the `aes` crate)
        return aes_clear.ctr_block(aes_key, args.iv, counter)

    def decrypt_states(t):
        """device tensor of states -> bytes, through a host copy and numpy (not the product's decryption kernel)"""
        return numpy_decrypt_bytes(t.cpu().numpy().view(np.uint64).reshape(-1, lw), glwe_sk)

    def step(i):
        first = i * args.total_blocks + shard_start if strong else pkg.sharding.shard_counters(0, B, i, rank, world)[0]
        eng.aes_ctr_dev(rk.data_ptr(), iv_ct.data_ptr(), first, B, out.data_ptr())
        return first

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident timing ------------------------------------------------------------------------------
    for w in range(args.warmup):
        first = step(w)
    torch.cuda.synchronize()
    if args.warmup:
        got = decrypt_states(out)     # every block of the last warm-up step is verified (client.rs:147-175)
        for b in range(B):
            assert got[16 * b:16 * b + 16] == expected(first + b), f"rank {rank}: block {first + b} differs from FIPS-197"
    sampler = ClockSampler(local)
    launches0 = eng.launch_count
    barrier()
    sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for i in range(args.steps):
        first = step(args.warmup + i)
    e1.record(stream)
    barrier()
    sampler.stop_flag = True
    ms = e0.elapsed_time(e1)
    launches = eng.launch_count - launches0
    out_host = out.cpu().numpy().view(np.uint64).reshape(B, 16, 8, lw)
    got = numpy_decrypt_bytes(out_host, glwe_sk)
    for b in range(B):
        assert got[16 * b:16 * b + 16] == expected(first + b), f"rank {rank}: block {first + b} differs from FIPS-197"
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, out_host, glwe_sk)
    del out_host
    first_device = first
    t = torch.tensor([ms, float(launches)], dtype=torch.float64, device=dev)
    if world > 1:
        tmax = t.clone()
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        tsum = t.clone()
        dist.all_reduce(tsum, op=dist.ReduceOp.SUM)
        ms, launches = float(tmax[0]), int(tsum[1])
    blocks_total = blocks_per_step * args.steps
    value = blocks_total / (ms * 1e-3)

    # ---- end to end through the host C ABI: pinned host buffers, H2D of round keys + IV and D2H of every
    # output state inside the timed region (tfa_aes_ctr is the call a user of the reference's Server makes) --
    rk_h = torch.empty(11 * state_words, dtype=torch.int64).pin_memory()
    iv_h = torch.empty(state_words, dtype=torch.int64).pin_memory()
    out_h = torch.empty(B * state_words, dtype=torch.int64).pin_memory()
    rk_h.copy_(rk)
    iv_h.copy_(iv_ct)
    torch.cuda.synchronize()
    rk_np, iv_np, out_np = rk_h.numpy().view(np.uint64), iv_h.numpy().view(np.uint64), out_h.numpy().view(np.uint64)
    e2e_steps = max(1, args.e2e_steps)

    def e2e_step(i):
        first = (i * args.total_blocks + shard_start if strong else (i * world + rank) * B) + 100000
        res = eng.lib.tfa_aes_ctr(eng.h, rk_np.ctypes.data, iv_np.ctypes.data, first, 0, B, out_np.ctypes.data)
        assert res == 0, eng.lib.tfa_last_error(eng.h)
        return first
    e2e_step(0)
    barrier()
    t0 = time.perf_counter()
    for i in range(e2e_steps):
        first = e2e_step(1 + i)
    barrier()
    e2e_s = time.perf_counter() - t0
    # device time of the same region, max over ranks
    t = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_s = float(t[0])
    dec = numpy_decrypt_bytes(out_np.reshape(-1, lw), glwe_sk)
    for b in range(B):
        assert dec[16 * b:16 * b + 16] == expected(first + b), "e2e output differs from FIPS-197"
    e2e_value = blocks_per_step * e2e_steps / e2e_s

    # ---- the other configurations BASELINE.json names, device-resident, CUDA events on the library's stream (rank 0, one GPU) ----
    configs = None
    if rank == 0 and not args.no_configs:
        def timed(fn, reps=1):
            fn()                                   # warm-up (LUT caches, workspace growth)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(stream)
            for _ in range(reps):
                fn()
            b.record(stream)
            torch.cuda.synchronize()
            return a.elapsed_time(b) / reps * 1e-3
        one = torch.zeros(state_words, dtype=torch.int64, device=dev)
        # config 1: --number-of-outputs 1: add_scalar + aes_encrypt of one block (key expansion is config 3)
        t_single = timed(lambda: eng.aes_ctr_dev(rk.data_ptr(), iv_ct.data_ptr(), 7, 1, one.data_ptr()), reps=2)
        assert decrypt_states(one) == expected(7), "config 1 output differs from FIPS-197"
        # config 2: one AES round = 16 many_sbox (L = 3) + ShiftRows/MixColumns/AddRoundKey, on one block and on a full batch
        st1 = torch.zeros(state_words, dtype=torch.int64, device=dev)
        rng = np.random.default_rng(5)
        clear_states = bytes(rng.integers(0, 256, 16 * B, dtype=np.uint8))
        clear_rk = bytes(rng.integers(0, 256, 16, dtype=np.uint8))
        rk1 = torch.zeros(state_words, dtype=torch.int64, device=dev)
        stB = torch.zeros(B * state_words, dtype=torch.int64, device=dev)
        eng.client_encrypt_bytes_dev(clear_rk, rk1.data_ptr(), seed=103)
        eng.client_encrypt_bytes_dev(clear_states, stB.data_ptr(), seed=104)
        st1.copy_(stB[:state_words])
        t_round1 = timed(lambda: eng.aes_round_dev(rk1.data_ptr(), st1.data_ptr(), 1), reps=3)
        stB_in = stB.clone()
        def round_batch():
            stB.copy_(stB_in)
            eng.aes_round_dev(rk1.data_ptr(), stB.data_ptr(), B)
        t_roundB = timed(round_batch, reps=2)
        got = decrypt_states(stB)
        for b in range(B):
            assert got[16 * b:16 * b + 16] == aes_clear.aes_round(clear_states[16 * b:16 * b + 16], clear_rk), "config 2 output differs from the clear AES round"
        # config 3: aes_key_expansion (40 SubWord S-boxes + 160 refreshes, 50 dependent stages)
        key_ct2 = torch.zeros(state_words, dtype=torch.int64, device=dev)
        rk2 = torch.zeros(11 * state_words, dtype=torch.int64, device=dev)
        eng.client_encrypt_bytes_dev(aes_key, key_ct2.data_ptr(), seed=105)
        t_keyexp = timed(lambda: eng.aes_key_expansion_dev(key_ct2.data_ptr(), rk2.data_ptr()))
        assert decrypt_states(rk2) == b"".join(aes_clear.round_keys(aes_key)), "config 3 round keys differ from FIPS-197"
        # config 4: aes_decrypt on 16 CTR blocks (the first 16 outputs of the last timed step)
        n4 = min(16, B)
        dec4_in = out[:n4 * state_words].clone()
        dec4 = dec4_in.clone()
        def decrypt16():
            dec4.copy_(dec4_in)
            eng.aes_decrypt_dev(rk.data_ptr(), dec4.data_ptr(), n4)
        t_dec = timed(decrypt16)
        got = decrypt_states(dec4)
        for b in range(n4):
            assert got[16 * b:16 * b + 16] == ((args.iv + first_device + b) % 2 ** 128).to_bytes(16, "big"), "config 4 output differs from the counter block"
        configs = {"single_block_latency_s": round(t_single, 4), "aes_round_ms": round(t_round1 * 1e3, 3),
                   "aes_round_batch_ms": round(t_roundB * 1e3, 3), "aes_round_batch_blocks": B,
                   "sbox_evals_per_s_measured": 16 * B / t_roundB,
                   "key_expansion_s": round(t_keyexp, 4), "decrypt_16_blocks_s": round(t_dec, 4), "decrypt_blocks": n4,
                   "note": "config 1: add_scalar + aes_encrypt of one block (tfa_aes_ctr_dev, nblk = 1); config 2: tfa_aes_round_dev on 1 block and on a batch, "
                           "sbox_evals_per_s_measured = 16 x batch / time of that batch (many_sbox L = 3 + linear layer); config 3: tfa_aes_key_expansion_dev; "
                           "config 4: tfa_aes_decrypt_dev on 16 blocks; every output checked against FIPS-197 (tests/aes_clear.py)"}

    line = None
    if rank == 0:
        # ---- roofline of the dominant kernel (pbs_kernel): one launch of the step's per-round shape ----------
        count = 128 * B
        lwe_small = torch.randint(-2 ** 62, 2 ** 62, (count * (eng.n + 1),), dtype=torch.int64, device=dev)
        lut = torch.full((512,), -(1 << 48), dtype=torch.int64, device=dev)
        pbs_out = torch.zeros(count * lw, dtype=torch.int64, device=dev)
        for _ in range(2):
            eng.bootstrap_dev(lwe_small.data_ptr(), count, lut.data_ptr(), 1 << 62, 1 << 48, pbs_out.data_ptr())
        k0, k1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        reps = 3
        k0.record(stream)
        for _ in range(reps):
            eng.bootstrap_dev(lwe_small.data_ptr(), count, lut.data_ptr(), 1 << 62, 1 << 48, pbs_out.data_ptr())
        k1.record(stream)
        torch.cuda.synchronize()
        pbs_ms = k0.elapsed_time(k1) / reps
        peak_dfma, peak_dmma = eng.measure_fp64_peaks()
        fp64_peak = max(peak_dfma, peak_dmma)
        achieved = count * PBS_FLOP / (pbs_ms * 1e-3) * 1e-12
        # per-stage share of one step (CUDA events around every launch group)
        eng.profile(True)
        step(args.warmup + args.steps)
        prof = eng.profile_report()
        eng.profile(False)
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        hbm = peaks.get("hbm_gbs", 6650.0)
        cpu = None
        if not args.no_cpu_baseline:
            r = cpu_sample(1)
            cpu = {"value": r["blocks_per_s"], "unit": UNIT, "cores": r["threads"], "kind": "port", "sample": r["sample"],
                   "sbox_evals_per_s": r["evals_per_s"], "note": "CPU restatement of the reference path (oracle), not tfhe-rs; README.md:186 quotes 84 s/block/core"}
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "strong" if strong else "weak", "vs_baseline": None,
            "dtype": "u64+f64", "data": "synthetic",
            "config": {"workload": (f"aes128_ctr: {args.total_blocks} CTR blocks per step split over {world} GPU(s) ({B} on rank 0)" if strong else f"aes128_ctr: {B} CTR blocks per GPU per step") + f" (add_scalar + aes_encrypt = {WOPBS_PER_BLOCK} byte-WoPBS; {pbs_per_block(B):.1f} PBS per block with the IV bits bootstrapped once per call, {PBS_PER_BLOCK_REFERENCE} block by block), PARAM_OPT n=669 k=4 N=512",
                       "blocks_per_gpu": B, "global_blocks_per_step": blocks_per_step, "parallelism": f"blocks sharded over {world} GPU(s), keys replicated by NCCL broadcast",
                       "l2": "inputs larger than L2 (1.04 GB of keys streamed per pass and 2 MiB of state per block)", "verified": "every output block decrypted and compared with FIPS-197"},
            "sbox_evals_per_s": value * WOPBS_PER_BLOCK,
            "pbs_per_s": value * pbs_per_block(B),
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int((11 + 1) * state_words * 8 + 16 * B),
                    "d2h_bytes_per_step": int(B * state_words * 8), "steps": e2e_steps, "api": "tfa_aes_ctr (host buffers, pinned)"},
            "gpu_launches": launches,
            "clocks": sampler.summary(),
            "roofline": {"bound": "fp64", "kernel": "pbs_ws2_kernel<4,3,2,8,5>", "achieved": achieved, "peak": fp64_peak, "unit": "TFLOP/s", "frac": achieved / fp64_peak if fp64_peak else None,
                         "peak_source": "max of the DFMA and the mma.sync.m8n8k4.f64 microbenchmarks of the FP64 pipe in this run (MEASURED_PEAKS.json has no FP64 figure)",
                         "peak_dfma": peak_dfma, "peak_dmma": peak_dmma, "traffic": NCU_DRAM_BYTES_PER_WAVE * -(-count // PBS_WAVE),
                         "traffic_note": "dram__bytes_read.sum + dram__bytes_write.sum of one 888-PBS wave (profiles/r2_pbs_ws2_kernel_ncu.txt: 348.9 + 5.6 MB) x waves in this launch (the last 296 of 18 944 run as a wave of pbs_ws_kernel<4,2,8,5>); algorithmic = 342.5 MB of key per wave",
                         "launch_ms": pbs_ms, "pbs_per_launch": count, "flop_per_pbs": PBS_FLOP,
                         "bsk_hbm_gbs": BSK_BYTES * -(-count // PBS_WAVE) / (pbs_ms * 1e-3) * 1e-9, "hbm_peak_gbs": hbm,
                         "note": "the key (342.5 MB) is read from HBM once per wave of 888 PBS and served from L2 to the other CTAs"},
            "stage_ms_one_step": {k: round(v[0], 3) for k, v in prof.items()},
            "setup": {"keygen_s": round(keygen_s, 3), "key_expansion_s": round(keyexp_s, 3), "key_bytes_broadcast": key_bytes},
        }
        if cpu:
            line["cpu_baseline"] = cpu
        if configs:
            line["baseline_configs"] = configs
            line["sbox_evals_per_s_measured"] = configs["sbox_evals_per_s_measured"]
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--blocks-per-gpu", type=int, default=148)
    ap.add_argument("--e2e-steps", type=int, default=5)
    ap.add_argument("--seed", type=int, default=2024)
    ap.add_argument("--iv", type=int, default=0)
    ap.add_argument("--key", type=int, default=None)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="skip the BASELINE config 1-4 measurements (rank 0)")
    ap.add_argument("--total-blocks", type=int, default=0, help="strong scaling (BASELINE config 5): this many blocks per step split over the GPUs")
    ap.add_argument("--warmup-ref", type=int, default=0)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the output states of the last one (rank 0's blocks) as float64 .npy files "
                         "under DIR: ciphertexts.npy (a fixed sample of the output LWEs) and phases.npy (message + noise of each)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
