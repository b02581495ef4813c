"""The shapes bench.py times, compared with the C oracle byte for byte over the whole output (on seeded inputs):
transforms of 2^21 to 2^25 points through every entry point the prover uses (whole-domain, padded, the resident 2-D
transform with and without the valid-column hint, the wire path of short rows, W row / column blocks), the permutation
product across several iterations of its block-offset scan, the quotient on its table and no-table paths, the MSM
shards of a 2^22+32-point SRS, and the tuning knobs dp_create reads from the environment.

Every plan switches on at these sizes only: the three-pass single-worker transform picks its digit split per domain
from 2^20 up, the block-offset scan of the permutation product carries its running product across 256-block steps
from 2^18 elements up, each MSM shard picks its own window count.  Forward transforms are compared with the oracle's
output; an inverse is compared by feeding it that output and asking for the input back (a bijection: a full check).

DP_TEST_FULL=1 adds 2^24 at W = 4, 2^26 at W = 1 and W = 8, the 2^22 permutation product and the 2^25 quotient in
full against the oracle.  On a B200 host (16 CPU threads) the default run took 4 minutes with a peak host RSS of
11 GiB, DP_TEST_FULL=1 took 9 minutes and 64 GiB (the 2^25 quotient's 25 inputs and the oracle's own arrays).
DP_TEST_DRY_RUN_ON_EMULATOR=1 runs the same code at small sizes on the kernel-logic emulator, with the three-pass plan
forced down to 2^9 points."""
import contextlib
import ctypes as C
import functools
import os

import numpy as np
import pytest
import torch

from distributed_plonk_b200 import dispatcher as disp
from distributed_plonk_b200 import parallel
from distributed_plonk_b200._binding import Context
from tests import common

pytestmark = pytest.mark.gpu
DRY = os.environ.get("DP_TEST_DRY_RUN_ON_EMULATOR", "0") == "1"     # tests/conftest.py: the test code itself, on the emulator
FULL = os.environ.get("DP_TEST_FULL", "0") == "1" and not DRY

# the benchmark's 2^22-gate proof: iNTT(n) on 2^22 points, the coset transforms on the 2^25-point quotient domain
LOG_N, LOG_M = (9, 12) if DRY else (22, 25)
# every transform test runs at every size, so that each size's oracle references are made once (2^26: DP_TEST_FULL)
NTT_LOGS = [9, 10, 11, 12] if DRY else [21, 22, 23, 24, 25] + ([26] if FULL else [])
# the block-offset scan steps over 256 blocks of 1024 elements: 2^19 + 1029 is 514 blocks (three steps, the last partial)
PERM_N = (1 << 18) + 1029 if DRY else (1 << 19) + 1029
PERM_BIG = (1 << 18) + 1029 if DRY else 1 << 22
NB = (1 << 12) + 32 if DRY else (1 << 22) + 32                      # the benchmark's SRS: n + 32 bases
MSM_SMALL = (1 << 10) + 32 if DRY else (1 << 16) + 32
GEN_SEED = 0xD15791B07E5EED


def _dims(log):
    r = 1 << (log >> 1)
    return r, (1 << log) // r


class Buf:
    """a device array: CUDA memory on the GPU, host memory under the emulator (where device pointers are host pointers)"""

    def __init__(self, a=None, n_u64=None):
        if DRY:
            self.a = np.ascontiguousarray(a).view(np.uint64).copy() if a is not None else np.zeros(n_u64, dtype=np.uint64)
            self.ptr = self.a.ctypes.data
        else:
            self.t = (torch.from_numpy(np.ascontiguousarray(a).view(np.int64)).cuda() if a is not None
                      else torch.zeros(n_u64, dtype=torch.int64, device="cuda"))
            self.ptr = self.t.data_ptr()

    @classmethod
    def fr(cls, n):
        return cls(n_u64=4 * n)

    def read(self) -> np.ndarray:
        if DRY:
            return self.a.copy()
        torch.cuda.synchronize()
        return self.t.cpu().numpy().view(np.uint64)


def dcopy(dst, src, nbytes):
    if DRY:
        C.memmove(dst, src, nbytes)
    else:
        parallel.as_tensor(dst, nbytes, True).copy_(parallel.as_tensor(src, nbytes, True))
        torch.cuda.synchronize()


def make_ctx(gpu_lib, log_n, log_m, bases=None, me=0, W=1):
    c = Context(gpu_lib, 0, me, W)
    if DRY and os.environ.get("DP_NTT_NO_3PASS", "0") == "0":
        c.debug_set_three_pass(9)                          # the emulator's sizes are below the plan's 2^20
    c.init(np.zeros(0, dtype=np.uint8) if bases is None else bases, 1 << log_n, 1 << log_m)
    return c


@contextlib.contextmanager
def contexts(gpu_lib, log_n, log_m, W=1, bases=None):
    cs = []
    try:
        for p in range(W):
            cs.append(make_ctx(gpu_lib, log_n, log_m, bases, p, W))
        yield cs
    finally:
        for c in cs:
            c.close()


def domains_for(log):
    """(log n, log m, is_quot) of a context whose domain `log` is the one the benchmark transforms at that size"""
    return (LOG_N, LOG_M, False) if log == LOG_N else (log - 3, log, True)


class Refs:
    """seeded inputs of one transform size and their forward transforms, by the oracle on first use (its parallel
    distributed_fft; the serial fft takes several times longer above 2^20)"""

    def __init__(self, orc, log):
        self.orc, self.log, self.N = orc, log, 1 << log

    @functools.cached_property
    def x(self):                                           # dense
        return self.orc.gen_fr(0x7000 + self.log, self.N)

    @functools.cached_property
    def xp(self):                                          # n coefficients on the 8n-point domain: rows[:, c/8:] == 0
        a = np.zeros((self.N, 4), dtype=np.uint64)
        a[: self.N // 8] = self.orc.gen_fr(0x7100 + self.log, self.N // 8)
        return a

    def _fwd(self, a, coset):
        return self.orc.distributed_fft(a, self.N, False, coset, n_workers=1)

    @functools.cached_property
    def y(self):
        return self._fwd(self.x, False)

    @functools.cached_property
    def yc(self):
        return self._fwd(self.x, True)

    @functools.cached_property
    def ypc(self):
        return self._fwd(self.xp, True)


@pytest.fixture(scope="module")
def refs(request, orc):
    """one size at a time: tests taking this fixture by (indirect) parameter are grouped by size, and a size's arrays
    (five of 2^25 points are 5 GiB) are dropped before the next size's are made"""
    r = Refs(orc, request.param)
    yield r
    r.__dict__.clear()


@pytest.fixture(scope="module")
def bench_ctx(gpu_lib):
    c = make_ctx(gpu_lib, LOG_N, LOG_M)
    yield c
    c.close()


def fft_dev(ctx, a, log, is_quot, inv, cos):
    """dp_fft_dev (W = 1): rows [r][c] in, columns [c][r] out, as the benchmark calls it"""
    r, c = _dims(log)
    src, dst = Buf(disp.dispatcher_rows(a, log)), Buf.fr(1 << log)
    ctx.fft_dev(src.ptr, dst.ptr, is_quot, inv, cos)
    del src
    return disp.assemble(dst.read().reshape(c, r, 4))


def fft_dev_blocks(ctxs, a, log, is_quot, inv, cos):
    """dp_fft_dev_rows on every rank's row block, the all-to-all as device copies, dp_fft_dev_cols on every rank"""
    W = len(ctxs)
    r, c = _dims(log)
    rows = disp.dispatcher_rows(a, log)
    srcs = [Buf(rows[p * r // W:(p + 1) * r // W]) for p in range(W)]
    del rows
    bufs = [ctx.fft_dev_rows(srcs[p].ptr, is_quot, inv, cos) for p, ctx in enumerate(ctxs)]
    for p in range(W):                                     # block q of rank p's send buffer -> block p of rank q's receive buffer
        for q in range(W):
            nb = bufs[p][2] * 32
            dcopy(bufs[q][1] + p * nb, bufs[p][0] + q * nb, nb)
    del srcs
    outs = [Buf.fr((c // W) * r) for _ in range(W)]
    for ctx, o in zip(ctxs, outs):
        ctx.fft_dev_cols(o.ptr)
    return disp.assemble(np.concatenate([o.read().reshape(c // W, r, 4) for o in outs]))


def check_bench_transforms(ref, run, what, hinted=True):
    """the transforms the benchmark times at this size through run(a, is_inv, is_coset, hint) -> natural-order output:
    iNTT(n) on the n-point domain; on the quotient domain the coset NTT of n coefficients (with the valid-column hint
    when `hinted`), the coset iNTT of its output, and the coset NTT of a dense input"""
    log = ref.log
    if log == LOG_N:
        assert np.array_equal(run(ref.y, True, False, False), ref.x), f"{what} 2^{log} iNTT"
        assert np.array_equal(run(ref.x, False, False, False), ref.y), f"{what} 2^{log} NTT"
        return
    assert np.array_equal(run(ref.xp, False, True, hinted), ref.ypc), f"{what} 2^{log} coset NTT of 2^{log - 3} coefficients hint={hinted}"
    assert np.array_equal(run(ref.ypc, True, True, hinted), ref.xp), f"{what} 2^{log} coset iNTT back to 2^{log - 3} coefficients"
    assert np.array_equal(run(ref.x, False, True, False), ref.yc), f"{what} 2^{log} coset NTT, dense input"


def with_hint(ctxs, log, is_quot, hint, fn):
    c = _dims(log)[1]
    for ctx in ctxs:
        ctx.fft_dev_hint_valid_cols(is_quot, c // 8 if hint else 0)
    try:
        return fn()
    finally:
        for ctx in ctxs:
            ctx.fft_dev_hint_valid_cols(is_quot, 0)


# ---------------------------------------------------------------------------------------------------- transforms
@pytest.mark.timeout(1200)
@pytest.mark.parametrize("refs", NTT_LOGS, indirect=True)
def test_whole_ntt_dev(refs, bench_ctx):
    """dp_ntt_dev in place, every flag combination (the twiddles of the smallest resident domain that covers the size)"""
    for inv, cos in common.FLAG_COMBOS:
        fwd = refs.yc if cos else refs.y
        b = Buf(fwd if inv else refs.x)
        bench_ctx.ntt_dev(b.ptr, refs.log, inv, cos)
        assert np.array_equal(b.read(), refs.x if inv else fwd), f"dp_ntt_dev 2^{refs.log} inv={inv} coset={cos}"


@pytest.mark.timeout(1200)
@pytest.mark.parametrize("refs", NTT_LOGS, indirect=True)
def test_fft_dev_single_worker(refs, gpu_lib):
    """dp_fft_dev at W = 1 as the benchmark times it (bench.py fft_resident), hinted or not"""
    log_n, log_m, q = domains_for(refs.log)
    with contexts(gpu_lib, log_n, log_m) as cs:
        check_bench_transforms(refs, lambda a, inv, cos, hint: with_hint(cs, refs.log, q, hint, lambda: fft_dev(cs[0], a, refs.log, q, inv, cos)),
                               "dp_fft_dev W=1")


@pytest.mark.timeout(1200)
@pytest.mark.parametrize("refs", NTT_LOGS, indirect=True)
def test_fft_dev_three_pass_and_four_pass_plans(refs, gpu_lib, monkeypatch):
    """each size's three-pass digit split (single_worker_split) and the 2-D four-pass plan (DP_NTT_NO_3PASS=1) against
    the oracle: coset NTT of a dense input and its inverse on the quotient domain of that size"""
    for no3 in ("0", "1"):
        monkeypatch.setenv("DP_NTT_NO_3PASS", no3)
        with contexts(gpu_lib, refs.log - 3, refs.log) as cs:
            what = f"dp_fft_dev 2^{refs.log} DP_NTT_NO_3PASS={no3}"
            assert np.array_equal(fft_dev(cs[0], refs.x, refs.log, True, False, True), refs.yc), f"{what} coset NTT"
            assert np.array_equal(fft_dev(cs[0], refs.yc, refs.log, True, True, True), refs.x), f"{what} coset iNTT"


@pytest.mark.timeout(1200)
@pytest.mark.parametrize("refs", NTT_LOGS, indirect=True)
def test_ntt_dev_padded_and_wire_path(refs, gpu_lib):
    """the resident prover's dp_ntt_dev_padded(n_valid = N/8), and the wire path: dp_fft1_rows_short with rows cut after
    c/8 entries, dp_fft2_prepare, dp_fft2 (the quotient domain of a context at 2^(log - 3), 2^log)"""
    log, N = refs.log, refs.N
    r, c = _dims(log)
    with contexts(gpu_lib, log - 3, log) as (ctx,):
        b = Buf(refs.xp)
        ctx.ntt_dev_padded(b.ptr, N // 8, log, False, True)
        assert np.array_equal(b.read(), refs.ypc), f"dp_ntt_dev_padded 2^{log} n_valid=2^{log - 3} coset NTT"
        ctx.ntt_dev_padded(b.ptr, N, log, True, True)
        assert np.array_equal(b.read(), refs.xp), f"dp_ntt_dev_padded 2^{log} coset iNTT"
        del b
        short = np.ascontiguousarray(disp.dispatcher_rows(refs.xp, log)[:, : c // 8])
        tid = 0x7125
        ctx.fft_init(tid, disp.fft_workloads(log, 1), True, False, True)
        ctx.fft1_rows_short(tid, 0, short, r, c // 8)
        ctx.fft2_prepare(tid)
        got = disp.assemble(ctx.fft2(tid, c, r))
        assert np.array_equal(got, refs.ypc), f"dp_fft1_rows_short (row_len c/8 = {c // 8}) + dp_fft2 2^{log} coset NTT"


# all three at the benchmark's two sizes; one each elsewhere (2^24 at W = 4 is config 4's per-rank size)
W_FOR = {LOG_N - 1: (2,), LOG_N: (2, 4, 8), LOG_N + 1: (8,), LOG_N + 2: (4,), LOG_M: (2, 4, 8), LOG_M + 1: (8,)}


@pytest.mark.timeout(1800)
@pytest.mark.parametrize("refs", NTT_LOGS, indirect=True)
def test_row_and_column_blocks(refs, gpu_lib):
    """W ranks as W contexts on one GPU: dp_fft_dev_rows, the all-to-all as device copies, dp_fft_dev_cols.  (The
    fused peer-store exchange needs CUDA IPC, which a process cannot open on its own export: tests/test_gpu_multi.py.)"""
    log_n, log_m, q = domains_for(refs.log)
    for W in W_FOR[refs.log]:
        with contexts(gpu_lib, log_n, log_m, W) as cs:
            check_bench_transforms(refs, lambda a, inv, cos, hint: with_hint(cs, refs.log, q, hint, lambda: fft_dev_blocks(cs, a, refs.log, q, inv, cos)),
                                   f"dp_fft_dev_rows/cols W={W}")


NTT_KNOBS = [("DP_NTT_BLOCKS", "2"), ("DP_NTT_PREFETCH", "1"), ("DP_NTT_NO_3PASS", "1")]


@pytest.mark.timeout(1200)
@pytest.mark.parametrize("refs", NTT_LOGS, indirect=True)
def test_ntt_knobs(refs, gpu_lib, monkeypatch):
    """every kernel instantiation / schedule an NTT knob selects gives the same bytes: the benchmark's iNTT(n), and its
    hinted coset NTT and coset iNTT on the quotient domain"""
    log_n, log_m, q = domains_for(refs.log)
    for knob in NTT_KNOBS:
        with monkeypatch.context() as mp:
            mp.setenv(*knob)
            with contexts(gpu_lib, log_n, log_m) as cs:
                check_bench_transforms(refs, lambda a, inv, cos, hint: with_hint(cs, refs.log, q, hint, lambda: fft_dev(cs[0], a, refs.log, q, inv, cos)),
                                       f"dp_fft_dev {knob[0]}={knob[1]}")


# ------------------------------------------------------------------------------------------ permutation product
def perm_inputs(orc, n, seed, valid=False):
    """wires, identity and sigma values [5][n] and beta, gamma.  valid: sigma re-orders the identity values and the wires
    agree on every copied cell (cells paired at random across the whole array), so the grand product closes to 1"""
    T = 5
    if not valid:
        w, idp, sg = (np.stack([orc.gen_fr(seed + 20 * k + t, n) for t in range(T)]) for k in range(3))
    else:
        cells = T * n
        order = np.random.default_rng(seed).permutation(cells)
        h = cells // 2
        partner = np.arange(cells)
        partner[order[0:2 * h:2]], partner[order[1:2 * h:2]] = order[1:2 * h:2], order[0:2 * h:2]
        w = orc.gen_fr(seed, cells)[np.minimum(np.arange(cells), partner)].reshape(T, n, 4)
        ids = orc.gen_fr(seed + 1, cells)
        idp, sg = ids.reshape(T, n, 4), ids[partner].reshape(T, n, 4)
    beta, gamma = orc.gen_fr(seed + 60, 1)[0], orc.gen_fr(seed + 61, 1)[0]
    return w, idp, sg, beta, gamma


def perm_product_dev(ctx, w, idp, sg, beta, gamma):
    n = w.shape[1]
    dw, di, ds, out = Buf(w), Buf(idp), Buf(sg), Buf.fr(n)
    ctx.perm_product_dev(dw.ptr, di.ptr, ds.ptr, w.shape[0], n, beta, gamma, out.ptr)
    return out.read().reshape(n, 4)


@pytest.mark.timeout(900)
def test_perm_product_across_scan_steps(orc, bench_ctx):
    """more than 256 blocks: the block-offset scan carries its running product from one step to the next"""
    n = PERM_N
    blocks = -(-n // 1024)
    w, idp, sg, beta, gamma = perm_inputs(orc, n, 0x7200)
    ref = orc.perm_product(w, idp, sg, beta, gamma)
    assert np.array_equal(bench_ctx.perm_product(w, idp, sg, beta, gamma), ref), f"dp_perm_product n={n} ({blocks} blocks)"
    assert np.array_equal(perm_product_dev(bench_ctx, w, idp, sg, beta, gamma), ref), f"dp_perm_product_dev n={n} ({blocks} blocks)"


@pytest.mark.timeout(1800 if FULL else 900)
def test_perm_product_cycle_closes_at_bench_size(orc, bench_ctx):
    """n = 2^22 (4096 blocks, 16 scan steps) on a valid permutation: z[n-1] * A[n-1] / B[n-1] = 1, A and B the row's
    numerator and denominator products, by the oracle's scalar arithmetic; the device entry gives the same bytes.
    DP_TEST_FULL=1 compares with the serial oracle in full."""
    n = PERM_BIG
    w, idp, sg, beta, gamma = perm_inputs(orc, n, 0x7300, valid=True)
    z = bench_ctx.perm_product(w, idp, sg, beta, gamma)
    V = orc.vec_op
    one = common._fr_one(orc)[None]
    be, ga = beta[None], gamma[None]
    num, den = one, one
    for t in range(w.shape[0]):
        base = V("add", w[t, n - 1][None], ga)
        num = V("mul", num, V("add", base, V("mul", be, idp[t, n - 1][None])))
        den = V("mul", den, V("add", base, V("mul", be, sg[t, n - 1][None])))
    closing = V("mul", V("mul", z[n - 1][None], num), V("inv", den))
    assert np.array_equal(z[0][None], one), f"dp_perm_product n={n}: z[0] != 1"
    assert np.array_equal(closing, one), f"dp_perm_product n={n} ({n // 1024} blocks): the cycle does not close"
    assert np.array_equal(perm_product_dev(bench_ctx, w, idp, sg, beta, gamma), z), f"dp_perm_product_dev n={n} != dp_perm_product"
    if FULL:
        assert np.array_equal(z, orc.perm_product(w, idp, sg, beta, gamma)), f"dp_perm_product n={n} vs oracle"


# ---------------------------------------------------------------------------------------------------- quotient
QUOT_TABLE = [None, "0", "1"]          # auto (table when it fits in 1/8 of free memory), never (no-table path), always


def quotient_inputs(orc, m, seed):
    sel = [orc.gen_fr(seed + i, m) for i in range(13)]
    sig = [orc.gen_fr(seed + 20 + i, m) for i in range(5)]
    w = [orc.gen_fr(seed + 30 + i, m) for i in range(5)]
    z, pi = orc.gen_fr(seed + 40, m), orc.gen_fr(seed + 41, m)
    k = orc.gen_fr(seed + 42, 5)
    al, be, ga = (orc.gen_fr(seed + 43 + i, 1)[0] for i in range(3))
    return sel, sig, w, z, pi, k, al, be, ga


def device_quotient_inputs(m, seed):
    """25 uniform Fr arrays of m entries made on the device (the host oracle would need all of them at once)"""
    if DRY:
        from oracle import loader as orc
        return [Buf(orc.gen_fr(seed + i, m)) for i in range(25)]
    g = torch.Generator(device="cuda")
    g.manual_seed(seed)
    out = []
    for _ in range(25):
        b = Buf.fr(m)
        b.t.view(m, 4).copy_(torch.randint(-(1 << 63), (1 << 63) - 1, (m, 4), dtype=torch.int64, device="cuda", generator=g))
        b.t.view(m, 4)[:, 3] &= (1 << 62) - 1                 # < 2^254: a valid Montgomery representative
        out.append(b)
    return out


def quotient_dev(ctx, bufs, k, al, be, ga, m):
    out = Buf.fr(m)
    p = [b.ptr for b in bufs]
    ctx.quotient_evals_dev(p[0:13], p[13:18], p[18:23], p[23], p[24], k, al, be, ga, out.ptr)
    return out.read().reshape(m, 4)


def set_quot_table(monkeypatch, v):
    if v is None:
        monkeypatch.delenv("DP_QUOT_TABLE", raising=False)
    else:
        monkeypatch.setenv("DP_QUOT_TABLE", v)


@pytest.mark.timeout(1200)
def test_quotient_both_paths_vs_oracle(orc, gpu_lib, monkeypatch):
    """n = 2^19 on m = 2^22, host and device entries, DP_QUOT_TABLE unset, 0 (1/(x_i - 1) by block products and one
    inversion per block, in the kernel) and 1 (the resident table)"""
    log_n, log_m = LOG_N - 3, LOG_N
    m = 1 << log_m
    sel, sig, w, z, pi, k, al, be, ga = quotient_inputs(orc, m, 0x7400)
    ref = orc.quotient_evals(np.stack(sel), np.stack(sig), np.stack(w), z, pi, k, al, be, ga, 1 << log_n)
    for table in QUOT_TABLE:
        set_quot_table(monkeypatch, table)
        with contexts(gpu_lib, log_n, log_m) as (c,):
            what = f"quotient n=2^{log_n} m=2^{log_m} DP_QUOT_TABLE={table}"
            for rep in range(2):                           # the table, when kept, is reused by the second call
                assert np.array_equal(c.quotient_evals(sel, sig, w, z, pi, k, al, be, ga), ref), f"dp_quotient_evals {what} call {rep}"
            bufs = [Buf(a) for a in sel + sig + w + [z, pi]]
            assert np.array_equal(quotient_dev(c, bufs, k, al, be, ga, m), ref), f"dp_quotient_evals_dev {what}"


@pytest.mark.timeout(2400 if FULL else 1200)
def test_quotient_reinit_sequence(orc, gpu_lib, monkeypatch):
    """one context re-initialised (2^22, 2^25) -> (2^19, 2^22) -> (2^22, 2^25), a quotient after each: the 2^22 step
    against the oracle, the two 2^25 steps against each other and against the other DP_QUOT_TABLE settings (the
    table and no-table paths share no code for 1/(x_i - 1)).  DP_TEST_FULL=1: the 2^25 quotient against the oracle."""
    big_m, small_n, small_m = 1 << LOG_M, 1 << (LOG_N - 3), 1 << LOG_N
    bufs = device_quotient_inputs(big_m, 0x7500)
    k = orc.gen_fr(0x7542, 5)
    al, be, ga = (orc.gen_fr(0x7543 + i, 1)[0] for i in range(3))
    sel, sig, w, z, pi, _, _, _, _ = quotient_inputs(orc, small_m, 0x7600)
    ref_small = orc.quotient_evals(np.stack(sel), np.stack(sig), np.stack(w), z, pi, k, al, be, ga, small_n)
    first = None
    for table in QUOT_TABLE:
        set_quot_table(monkeypatch, table)
        with contexts(gpu_lib, LOG_N, LOG_M) as (c,):
            what = f"DP_QUOT_TABLE={table}"
            q1 = quotient_dev(c, bufs, k, al, be, ga, big_m)
            first = q1 if first is None else first
            assert np.array_equal(q1, first), f"quotient m=2^{LOG_M} {what} != DP_QUOT_TABLE={QUOT_TABLE[0]}"
            c.init(np.zeros(0, dtype=np.uint8), small_n, small_m)
            assert np.array_equal(c.quotient_evals(sel, sig, w, z, pi, k, al, be, ga), ref_small), \
                f"quotient n=2^{LOG_N - 3} m=2^{LOG_N} after re-init from m=2^{LOG_M} {what}"
            c.init(np.zeros(0, dtype=np.uint8), 1 << LOG_N, big_m)
            assert np.array_equal(quotient_dev(c, bufs, k, al, be, ga, big_m), first), \
                f"quotient m=2^{LOG_M} after re-init from m=2^{LOG_N} {what}"
    if FULL or DRY:
        host = [b.read().reshape(big_m, 4) for b in bufs]
        del bufs
        ref = orc.quotient_evals(np.stack(host[0:13]), np.stack(host[13:18]), np.stack(host[18:23]), host[23], host[24],
                                 k, al, be, ga, 1 << LOG_N)
        assert np.array_equal(first, ref), f"quotient n=2^{LOG_N} m=2^{LOG_M} vs oracle"


# ---------------------------------------------------------------------------------------------------------- MSM
@pytest.fixture(scope="module")
def srs(gpu_lib):
    """the benchmark's synthetic SRS: n distinct device-generated points, index 3 and the 32 padding entries at infinity"""
    c = Context(gpu_lib, 0, 0, 1)
    b = c.gen_bases(GEN_SEED, NB)
    c.close()
    b[3, :] = 0
    b[3, 96] = 1
    b[NB - 32:, :] = 0
    b[NB - 32:, 96] = 1
    return b


@pytest.fixture(scope="module")
def msm_scalars(orc):
    sets = common.scalar_sets(orc, NB, 0x7700)
    return {name: sets[name] for name in ("uniform", "witness-like")}


@pytest.mark.timeout(1800)
def test_msm_shards_as_benchmarked(orc, gpu_lib, srs, msm_scalars):
    """every rank's shard at N = 2, 4, 8 (parallel.msm_shard: starts not aligned, each shard its own window count and
    tree levels) against the oracle's MSM over the same bases, one at a time and then all as one dp_msm_dev_batch"""
    with contexts(gpu_lib, LOG_N, LOG_M, bases=srs) as (c,):
        jobs = [(W, rank, *parallel.msm_shard(NB, rank, W)) for W in (2, 4, 8) for rank in range(W)]
        for name, sc in msm_scalars.items():
            refs = {}
            for W, rank, lo, hi in jobs:
                refs[lo, hi] = orc.msm(srs[lo:hi], sc[lo:hi])
                common.assert_point_eq(orc, c.msm(lo, hi, sc[lo:hi]), refs[lo, hi], f"dp_msm shard {rank}/{W} [{lo}, {hi}) {name}")
            dev = [Buf(sc[lo:hi]) for _, _, lo, hi in jobs]
            outs = [Buf(n_u64=18) for _ in jobs]
            c.msm_dev_batch([(lo, hi, d.ptr, hi - lo, o.ptr) for (_, _, lo, hi), d, o in zip(jobs, dev, outs)])
            for (W, rank, lo, hi), o in zip(jobs, outs):
                common.assert_point_eq(orc, o.read().view(np.uint8), refs[lo, hi], f"dp_msm_dev_batch shard {rank}/{W} [{lo}, {hi}) {name}")


MSM_KNOBS = [("DP_MSM_BLOCKS", "4"), ("DP_MSM_BLOCKS", "5"), ("DP_MSM_CHUNK", "32"), ("DP_MSM_SORT_STREAM", "1")]


@pytest.mark.timeout(1200)
@pytest.mark.parametrize("knob", MSM_KNOBS, ids=[f"{k}={v}" for k, v in MSM_KNOBS])
def test_msm_knobs(orc, gpu_lib, srs, msm_scalars, monkeypatch, knob):
    """every kernel instantiation / schedule an MSM knob selects gives the oracle's point: 2^16+32 points from the start
    of the SRS, and rank 5's shard at N = 8"""
    monkeypatch.setenv(*knob)
    lo, hi = parallel.msm_shard(NB, 5, 8)
    with contexts(gpu_lib, LOG_N, LOG_M, bases=srs) as (c,):
        for name, sc in msm_scalars.items():
            what = f"{knob[0]}={knob[1]} {name}"
            common.assert_point_eq(orc, c.msm(0, MSM_SMALL, sc[:MSM_SMALL]), orc.msm(srs[:MSM_SMALL], sc[:MSM_SMALL]), f"dp_msm n={MSM_SMALL} {what}")
            common.assert_point_eq(orc, c.msm(lo, hi, sc[lo:hi]), orc.msm(srs[lo:hi], sc[lo:hi]), f"dp_msm shard 5/8 [{lo}, {hi}) {what}")
