"""Every FP64 kernel instance, bit for bit against the exact integer reference of tests/exact_ref.py.

Why exact agreement is guaranteed here.  The kernels accept any u64 key and GGSW words; nothing in them depends on those
words being encryptions.  The synthetic contexts of this file load bootstrap keys and GGSWs with words |w| <= 2^16, while
the accumulators and LUTs stay full 64-bit random (so the digits cover their whole range).  Every exact sum that the
double-precision FFT product approximates is then bounded:
  * PBS, (2^8, 5), digits |d| <= 2^7:  |coef| <= (K+1) L N 2^7 2^16 = 5 * 5 * 512 * 2^23 ~ 2^36.6 at K = 4;
  * vertical packing / CMux, (2^15, 1), digits |d| <= 2^14:  |coef| <= (K+1) N 2^14 2^16 ~ 2^41.3 at K = 4.
The forward transforms of the digits and of the key words are exact inputs (integers below 2^53), and a length-512
negacyclic FFT product of such operands errs by well under bound * 2^-53 * 2 log2(512) < 2^-6.  f64_to_torus therefore rounds
every product to the exact integer, and the GPU output must equal the reference on every word (mask included) after every
one of the n blind-rotation steps.  A mismatch is a kernel or dispatch bug, never a tolerance question.  The one
decomposition detail the reference must copy is the kernels' tie rule at (2^8, 5) (exact_ref.signed_digits_85).

The keyswitching keys are zero (no test here uses them); their sizes are computed from the C ABI's layouts because
tfa_ctx_load_keys does not check them:  KSK K N ks_level (n + 1) words, PFPKSK (K+1) (K N + 1) pfks_level (K+1) N words.

Inputs come from a pool of LWEs per context (random words, the edge words 0, 2^64 - 1, 2^63 and modulus-switch ties
k 2^54 + 2^53, alone and mixed); a batch of `count` ciphertexts is a random pick from the pool, so the reference is computed
once per pool row and every output word of every ciphertext is compared.  One torch.profiler pass per context records the
kernels each case launched, and the sequence must be the one the dispatch comment of dev_pbs (engine.cu) and the G choice of
dev_vertical_packing promise.  W below is a wave of the two-set kernel, 6 x the device's SM count (888 on a B200).

Coverage: each instantiation and the tests that reach it (n = 25 unless marked slow, n = 669)
  LAUNCH_WS       pbs_ws_kernel<4,1,8,5>   auto 75, 148, W+75; schedule 2 at 1, 148; bootstrap_dev 75, W+75; slow 100, W+75
                  pbs_ws_kernel<4,2,8,5>   auto 149, 296; schedule 2 at 149, 296; slow 200
                  pbs_ws_kernel<4,3,8,5>   auto 297, W/2, W+W/2; schedule 2 at 297, 445; bootstrap_dev 297; slow 400
                  pbs_ws_kernel<1,1,8,5>   auto 1, 3; schedule 2 at 3; schedules 3 and 4 at 3 (fall back); slow 3
                  pbs_ws_kernel<1,4,8,5>   auto 4, 15; schedule 4 at 9 (falls back)
                  pbs_ws_kernel<1,8,8,5>   auto 16, 300; schedule 2 at 16; schedule 3 at 20 (falls back); bootstrap_dev 20; slow 20
  launch_pbs_ws2  pbs_ws2_kernel<4,3,2,8,5>  auto W/2+1, W-1, W, W+74, W+75, W+W/2, W+W/2+1, 2W; schedule 4 at 1, 5, 6, 7;
                                             bootstrap_dev W+75; slow W+75, schedule 4 at 7
  launch_pbs_cl2  pbs_cl2_kernel           auto 1, 74, W+74; schedule 3 at 1, 74, 75, 300; bootstrap_dev 1; slow 1, schedule 3
                                           at 100; real keys (slow) schedule 3 at 100
  LAUNCH_VP       vp_kernel<4,1,15,1>      nouts 1 (npoly 1, 2, 4); the full-range CMux step
                  vp_kernel<4,2,15,1>      nouts 2 (npoly 1, 4)
                  vp_kernel<4,3,15,1>      nouts 3, 4, 5, 7 (ragged last chunk at 4, 5, 7); npoly 2 with 3 outputs, npoly 4 with 5
                  vp_kernel<1,1,15,1>      nouts 1, 3
                  vp_kernel<1,4,15,1>      nouts 4, 7 (ragged), npoly 4 with 5 outputs
                  vp_kernel<1,8,15,1>      nouts 8, 11 (ragged), npoly 2 with 8 outputs
  LAUNCH_TREE     cmux_tree_kernel<4,3,15,1>  npoly 2 x 3 outputs, npoly 4 x 2 outputs (4 pairs: ragged), npoly 4 x 5 outputs
                  cmux_tree_kernel<4,1,15,1>  npoly 2 x 1 output, npoly 4 x 1 and x 2 outputs (second layer)
                  cmux_tree_kernel<1,8,15,1>  npoly 2 x 8 outputs, npoly 4 x 5 outputs (10 pairs: ragged)
                  cmux_tree_kernel<1,1,15,1>  npoly 2 x 1 output, npoly 4 x 1 output, npoly 4 x 5 outputs (second layer)
  fourier_convert_kernel   5 levels: every PBS case (bootstrap-key conversion); 1 level: every vertical-packing case
"""
import re

import numpy as np
import pytest

import exact_ref as X

pytestmark = pytest.mark.gpu
N = 512
WMAX = 2 ** 16        # small-norm key and GGSW words: |w| <= WMAX


def _params(pkg, n, K):
    return pkg.Params(n, K, 512, 8, 5, 2, 6, 12, 3, 15, 1, 2, 1, 0, 2.0 ** -24, 2.0 ** -50, 2.0 ** -50)


def _sm_count():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def _edge_pool(rng, P, n):
    """P LWEs of n + 1 words: rows of one edge word each, rows mixing edge words into random ones, random rows"""
    ties = (rng.integers(0, 1024, 64, dtype=np.uint64) << np.uint64(54)) + np.uint64(1 << 53)
    edges = np.concatenate([np.array([0, (1 << 64) - 1, 1 << 63], dtype=np.uint64), ties])
    pool = rng.integers(0, 2 ** 64, (P, n + 1), dtype=np.uint64)
    pool[0], pool[1], pool[2] = 0, (1 << 64) - 1, 1 << 63
    pool[3] = rng.choice(ties, n + 1)
    mix = rng.random((P, n + 1)) < 0.3
    mix[: P // 2] = False
    pool[mix] = rng.choice(edges, int(mix.sum()))
    pool[4:8, n] = [0, (1 << 64) - 1, 1 << 63, int(ties[0])]     # edge bodies under random masks
    return pool


class Synth:
    """An engine with a seeded small-norm bootstrap key and zero keyswitching keys, plus its input pool and references."""

    def __init__(self, pkg, n, K, seed, P):
        self.n, self.K = n, K
        rng = np.random.default_rng(seed)
        self.bsk = rng.integers(-WMAX, WMAX + 1, (n, 5, K + 1, K + 1, N)).astype(np.int64)
        self.eng = pkg.Engine(_params(pkg, n, K))
        ksk = np.zeros(K * N * 6 * (n + 1), dtype=np.uint64)
        pfpksk = np.zeros((K + 1) * (K * N + 1) * 3 * (K + 1) * N, dtype=np.uint64)
        self.eng.load_keys(self.bsk.view(np.uint64), ksk, pfpksk)
        self.lut = rng.integers(0, 2 ** 64, N, dtype=np.uint64)
        self.pool = _edge_pool(rng, P, n)
        self.rng = rng
        self._ref = {}

    def ref(self, pre_add=0, post_add=0):
        if (pre_add, post_add) not in self._ref:
            self._ref[pre_add, post_add] = X.blind_rotate(self.pool, self.lut, self.bsk, pre_add, post_add)
        return self._ref[pre_add, post_add]

    def run(self, count, schedule=0, pre_add=None, post_add=0):
        """count ciphertexts picked from the pool through tfa_bootstrap, or through tfa_bootstrap_dev when pre_add is given"""
        pick = self.rng.integers(0, len(self.pool), count)
        lwe = self.pool[pick]
        self.eng.set_pbs_schedule(schedule)
        try:
            if pre_add is None:
                out = self.eng.bootstrap(lwe, self.lut)
            else:
                out = _bootstrap_dev(self.eng, lwe, self.lut, pre_add, post_add)
        finally:
            self.eng.set_pbs_schedule(0)
        return pick, out


def _bootstrap_dev(eng, lwe, lut, pre_add, post_add):
    import torch
    d_in = torch.from_numpy(np.ascontiguousarray(lwe).view(np.int64)).cuda()
    d_lut = torch.from_numpy(lut.view(np.int64)).cuda()
    d_out = torch.empty(len(lwe) * eng.lw, dtype=torch.int64, device="cuda")
    torch.cuda.synchronize()                      # the engine's stream does not wait for torch's copies
    eng.bootstrap_dev(d_in.data_ptr(), len(lwe), d_lut.data_ptr(), pre_add, post_add, d_out.data_ptr())
    eng.synchronize()
    return d_out.cpu().numpy().view(np.uint64).reshape(len(lwe), eng.lw)


_KERNEL = re.compile(r"(pbs_ws_kernel|pbs_ws2_kernel|pbs_cl2_kernel|vp_kernel|cmux_tree_kernel)(<[0-9, ]*>)?")


def _profiled(run_cases):
    """Run run_cases() under one torch.profiler pass; return its result and the FP64 kernels launched, in start order, as
    'name<template args>' strings without spaces."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.init()
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        result = run_cases()
        torch.cuda.synchronize()
    kernels = []
    for e in prof.events():
        if e.device_type == torch.autograd.DeviceType.CUDA:
            m = _KERNEL.search(e.name)
            if m:
                kernels.append((e.time_range.start, (m.group(1) + (m.group(2) or "")).replace(" ", "")))
    return result, [k for _, k in sorted(kernels)]


def WS(K, G):
    return f"pbs_ws_kernel<{K},{G},8,5>"


WS2, CL2 = "pbs_ws2_kernel<4,3,2,8,5>", "pbs_cl2_kernel"


def _pbs_cases_k4(W):
    """(case id, count, schedule, pre_add or None for tfa_bootstrap, post_add, expected kernels) at K = 4"""
    auto = [(1, [CL2]), (74, [CL2]), (75, [WS(4, 1)]), (148, [WS(4, 1)]), (149, [WS(4, 2)]), (296, [WS(4, 2)]),
            (297, [WS(4, 3)]), (W // 2, [WS(4, 3)]), (W // 2 + 1, [WS2]), (W - 1, [WS2]), (W, [WS2]),
            (W + 74, [WS2, CL2]), (W + 75, [WS2, WS(4, 1)]), (W + W // 2, [WS2, WS(4, 3)]), (W + W // 2 + 1, [WS2]),
            (2 * W, [WS2])]
    cases = [(f"k4-auto-{c}", c, 0, None, 0, k) for c, k in auto]
    cases += [(f"k4-sched2-{c}", c, 2, None, 0, k) for c, k in
              [(1, [WS(4, 1)]), (148, [WS(4, 1)]), (149, [WS(4, 2)]), (296, [WS(4, 2)]), (297, [WS(4, 3)]), (445, [WS(4, 3)])]]
    cases += [(f"k4-sched3-{c}", c, 3, None, 0, [CL2]) for c in (1, 74, 75, 300)]
    cases += [(f"k4-sched4-{c}", c, 4, None, 0, [WS2]) for c in (1, 5, 6, 7)]
    pre, post = (1 << 62) + 0x123456789, 0xFEDCBA9876543210
    cases += [(f"k4-dev-{c}", c, 0, pre, post, k) for c, k in
              [(1, [CL2]), (75, [WS(4, 1)]), (297, [WS(4, 3)]), (W + 75, [WS2, WS(4, 1)])]]
    return cases


def _pbs_cases_k1():
    cases = [(f"k1-auto-{c}", c, 0, None, 0, [WS(1, g)]) for c, g in [(1, 1), (3, 1), (4, 4), (15, 4), (16, 8), (300, 8)]]
    cases += [(f"k1-sched2-{c}", c, 2, None, 0, [WS(1, g)]) for c, g in [(3, 1), (16, 8)]]
    cases += [(f"k1-sched3-{c}", c, 3, None, 0, [WS(1, g)]) for c, g in [(3, 1), (20, 8)]]    # schedules 3 and 4 exist at K = 4
    cases += [(f"k1-sched4-{c}", c, 4, None, 0, [WS(1, g)]) for c, g in [(3, 1), (9, 4)]]     # only: pbs_ws_kernel runs
    cases += [("k1-dev-20", 20, 0, (1 << 62) + 77, 0x0123456789ABCDEF, [WS(1, 8)])]
    return cases


def _run_pbs(synth, cases):
    def go():
        return {cid: synth.run(count, sched, pre, post) for cid, count, sched, pre, post, _ in cases}
    return _profiled(go)


def _check_pbs(synth, cases, results, cid):
    _, count, _, pre, post, _ = next(c for c in cases if c[0] == cid)
    pick, got = results[cid]
    want = synth.ref(pre or 0, post)[pick]
    bad = np.nonzero((got != want).any(axis=1))[0]
    assert bad.size == 0, f"{cid}: {bad.size} of {count} ciphertexts differ, first at {bad[:8]} (pool rows {pick[bad[:8]]})"


def _check_kernels(cases, kernels):
    want = [k for c in cases for k in c[5]]
    assert kernels == want, "kernels launched, per case in order: " + "; ".join(f"{c[0]}: {c[5]}" for c in cases) + f"\ngot {kernels}"


# ---- PBS, n = 25 -----------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def k4(pkg):
    s = Synth(pkg, 25, 4, seed=41, P=97)
    cases = _pbs_cases_k4(6 * _sm_count())
    results, kernels = _run_pbs(s, cases)
    yield s, cases, results, kernels
    s.eng.close()


@pytest.fixture(scope="module")
def k1(pkg):
    s = Synth(pkg, 25, 1, seed=11, P=97)
    cases = _pbs_cases_k1()
    results, kernels = _run_pbs(s, cases)
    yield s, cases, results, kernels
    s.eng.close()


def _ids(cases):
    return [c[0] for c in cases]


@pytest.mark.parametrize("i", range(len(_pbs_cases_k4(888))), ids=_ids(_pbs_cases_k4(888)))   # ids spelled for W = 888
def test_pbs_k4_bit_exact(k4, i):
    s, cases, results, _ = k4
    _check_pbs(s, cases, results, cases[i][0])


def test_pbs_k4_dispatch(k4):
    _check_kernels(k4[1], k4[3])


@pytest.mark.parametrize("cid", _ids(_pbs_cases_k1()))
def test_pbs_k1_bit_exact(k1, cid):
    s, cases, results, _ = k1
    _check_pbs(s, cases, results, cid)


def test_pbs_k1_dispatch(k1):
    _check_kernels(k1[1], k1[3])


# ---- PBS, n = 669 (slow) ---------------------------------------------------------------------------------------------------
def _pbs_cases_slow(W):
    pre, post = (1 << 62) + 5, 1 << 49
    return [("k4-auto-1", 4, 1, 0, None, 0, [CL2]), ("k4-auto-100", 4, 100, 0, None, 0, [WS(4, 1)]),
            ("k4-auto-200", 4, 200, 0, None, 0, [WS(4, 2)]), ("k4-auto-400", 4, 400, 0, None, 0, [WS(4, 3)]),
            ("k4-dev-W+75", 4, W + 75, 0, pre, post, [WS2, WS(4, 1)]), ("k4-sched3-100", 4, 100, 3, None, 0, [CL2]),
            ("k4-sched4-7", 4, 7, 4, None, 0, [WS2]), ("k1-auto-3", 1, 3, 0, None, 0, [WS(1, 1)]),
            ("k1-auto-20", 1, 20, 0, None, 0, [WS(1, 8)])]


@pytest.fixture(scope="module")
def slow669(pkg):
    ctx = {4: Synth(pkg, 669, 4, seed=669, P=61), 1: Synth(pkg, 669, 1, seed=670, P=31)}
    cases = _pbs_cases_slow(6 * _sm_count())

    def go():
        return {cid: ctx[K].run(count, sched, pre, post) for cid, K, count, sched, pre, post, _ in cases}
    results, kernels = _profiled(go)
    yield ctx, cases, results, kernels
    for s in ctx.values():
        s.eng.close()


@pytest.mark.slow
@pytest.mark.parametrize("cid", [c[0] for c in _pbs_cases_slow(888)])
def test_pbs_n669_bit_exact(slow669, cid):
    """All 669 steps: every word of every ciphertext (the pool makes the reference cheap, so nothing is sampled)."""
    ctx, cases, results, _ = slow669
    _, K, count, _, pre, post, _ = next(c for c in cases if c[0] == cid)
    pick, got = results[cid]
    want = ctx[K].ref(pre or 0, post)[pick]
    bad = np.nonzero((got != want).any(axis=1))[0]
    assert bad.size == 0, f"{cid}: {bad.size} of {count} ciphertexts differ, first at {bad[:8]}"


@pytest.mark.slow
def test_pbs_n669_dispatch(slow669):
    _check_kernels([c[:1] + c[2:] for c in slow669[1]], slow669[3])


# ---- vertical packing and CMux tree --------------------------------------------------------------------------------------
def VP(K, G):
    return f"vp_kernel<{K},{G},15,1>"


def TREE(K, G):
    return f"cmux_tree_kernel<{K},{G},15,1>"


# (K, npoly, nouts, nbits values, kernels per call)
_VP_CONFIGS = [
    (4, 1, 1, (1, 5, 9), [VP(4, 1)]), (4, 1, 2, (3, 8), [VP(4, 2)]), (4, 1, 3, (2, 9), [VP(4, 3)]),
    (4, 1, 4, (4,), [VP(4, 3)]), (4, 1, 5, (7,), [VP(4, 3)]), (4, 1, 7, (6, 10), [VP(4, 3)]),
    (4, 2, 1, (1, 2, 10), [TREE(4, 1), VP(4, 1)]), (4, 2, 3, (5,), [TREE(4, 3), VP(4, 3)]),
    (4, 4, 1, (2, 6), [TREE(4, 1), TREE(4, 1), VP(4, 1)]), (4, 4, 2, (3, 11), [TREE(4, 3), TREE(4, 1), VP(4, 2)]),
    (4, 4, 5, (4,), [TREE(4, 3), TREE(4, 3), VP(4, 3)]), (4, 4, 1, (1,), [VP(4, 1)]),     # 2 tree bits > 1 selector bit: no tree
    (1, 1, 1, (1, 9), [VP(1, 1)]), (1, 1, 3, (4,), [VP(1, 1)]), (1, 1, 4, (5,), [VP(1, 4)]), (1, 1, 7, (3,), [VP(1, 4)]),
    (1, 1, 8, (8,), [VP(1, 8)]), (1, 1, 11, (6,), [VP(1, 8)]),
    (1, 2, 8, (2, 9), [TREE(1, 8), VP(1, 8)]), (1, 2, 1, (4,), [TREE(1, 1), VP(1, 1)]),
    (1, 4, 5, (3, 10), [TREE(1, 8), TREE(1, 1), VP(1, 4)]), (1, 4, 1, (2,), [TREE(1, 1), TREE(1, 1), VP(1, 1)]),
]
_VP_CASES = [(f"k{K}-npoly{p}-nouts{o}-nbits{b}", K, p, o, b, k) for K, p, o, bs, k in _VP_CONFIGS for b in bs]


@pytest.fixture(scope="module")
def vp_runs(k4, k1):
    engines = {4: k4[0].eng, 1: k1[0].eng}
    rng = np.random.default_rng(7)

    def go():
        out = {}
        for cid, K, npoly, nouts, nbits, _ in _VP_CASES:
            ggsw = rng.integers(-WMAX, WMAX + 1, (nbits, 1, K + 1, K + 1, N)).astype(np.int64)
            lut = rng.integers(0, 2 ** 64, (nouts, npoly, N), dtype=np.uint64)
            got = engines[K].vertical_packing(lut, ggsw.view(np.uint64).reshape(nbits, 1, K + 1, (K + 1) * N))
            out[cid] = (lut, ggsw, got)
        return out
    return _profiled(go)


@pytest.mark.parametrize("cid", [c[0] for c in _VP_CASES])
def test_vertical_packing_bit_exact(vp_runs, cid):
    _, K, _, _, _, _ = next(c for c in _VP_CASES if c[0] == cid)
    lut, ggsw, got = vp_runs[0][cid]
    want = X.vertical_packing(lut, ggsw, K + 1)
    bad = np.nonzero((got != want).any(axis=1))[0]
    assert bad.size == 0, f"{cid}: outputs {bad} differ"


def test_vertical_packing_dispatch(vp_runs):
    _check_kernels([(c[0], None, None, None, None, c[5]) for c in _VP_CASES], vp_runs[1])


# ---- full-range GGSW words, real keys -----------------------------------------------------------------------------------
def test_cmux_step_full_range_ggsw(k4):
    """One CMux step (one selector bit, vp_kernel<4,1>) with uniformly random 64-bit GGSW words, like those of a real
    circuit-bootstrapped GGSW: the digits are computed from identical inputs on both sides, so only the FFT rounding of the
    product separates the GPU from exact_ref.  Bound: the exact sum has |coef| <= N 2^14 2^63 = 2^86 (one non-zero row, the
    body's difference, at base 2^15), and the double-precision product errs by at most ~ 2^86 * 2^-53 * 2 log2(512) ~ 2^37.2
    per coefficient (the GGSW words themselves are rounded to 53 bits, a relative 2^-53 as well), under 2^38.  Measured on a
    B200 (1000 W limit): 2^30.5, the typical rather than the worst-case rounding."""
    s = k4[0]
    rng = np.random.default_rng(99)
    ggsw = rng.integers(0, 2 ** 64, (1, 1, 5, 5, N), dtype=np.uint64)
    lut = rng.integers(0, 2 ** 64, (4, 1, N), dtype=np.uint64)
    got = s.eng.vertical_packing(lut[:1], ggsw.reshape(1, 1, 5, 5 * N))
    want = X.vertical_packing(lut[:1], ggsw, 5)
    with np.errstate(over="ignore"):
        d = np.abs((got - want).view(np.int64).astype(np.float64)).max()
    print(f"one CMux step, full-range GGSW words, K = 4: max |GPU - exact| = 2^{np.log2(d + 1):.2f}")
    assert d < 2 ** 38


def _random_lut_bootstrap(engine_opt, oracle_opt, schedule, seed):
    o = oracle_opt
    rng = np.random.default_rng(seed)
    lut = rng.integers(0, 2 ** 64, N, dtype=np.uint64)
    lwe = o.encrypt_lwe_small(rng.integers(0, 2 ** 64, 100, dtype=np.uint64))
    engine_opt.set_pbs_schedule(schedule)
    try:
        got = engine_opt.bootstrap(lwe, lut)
    finally:
        engine_opt.set_pbs_schedule(0)
    sample = [0, 1, 57, 99]
    ref = o.bootstrap(lwe[sample], lut)
    # tolerance 2^36 on the phase, as in test_gpu_parity: both sides carry FFT rounding (~2^26 per step, a random walk of
    # ~2^31 over 669 steps) and the kernels' tie rule differs from the oracle's; a wrong LUT coefficient is ~2^63 away
    with np.errstate(over="ignore"):
        d = np.abs((o.phase_big(got[sample]) - o.phase_big(ref)).view(np.int64).astype(np.float64)).max()
    assert d < 2 ** 36, f"phase difference 2^{np.log2(d + 1):.1f}"


@pytest.mark.slow
def test_opt_ws_kernel_g1_random_lut(engine_opt, oracle_opt):
    """pbs_ws_kernel<4,1> (automatic schedule, 100 ciphertexts) with the oracle's PARAM_OPT keys and a random LUT"""
    _random_lut_bootstrap(engine_opt, oracle_opt, 0, 100)


@pytest.mark.slow
def test_opt_cluster_kernel_random_lut(engine_opt, oracle_opt):
    """pbs_cl2_kernel forced (schedule 3) on 100 ciphertexts: more than one wave of clusters, random LUT, real keys"""
    _random_lut_bootstrap(engine_opt, oracle_opt, 3, 101)
