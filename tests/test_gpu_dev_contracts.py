"""The C ABI around the kernels: stream order, capacities, accumulation, optional outputs, degenerate batches and error
reports of the entry points, against the CPU oracle.

include/tokengeex_b200.h promises more than the kernels compute: work queued on the legacy default stream before a
`_dev` call is ordered before the library's kernels; no call writes past a capacity it was given, and a too small one
is reported with the size that is needed; the `_dev` frequency and E-step passes add into what their buffer held;
status / proc_len / first_bad / bad_len may be NULL; an empty batch is a valid batch; NoPath and BAD_Z name the lowest
failing sample with its processed length or its z.  Every output buffer here is the head of a larger host array or
device tensor whose tail holds a canary, so that an overrun lands in the test's own memory and is seen.
"""
import ctypes as C
import random

import numpy as np
import pytest

from oracle import oracle as O
from tests.test_gpu_exact_counts import KERNEL_SETS, configure, limbs_to_ints, nearest
from tests.util import rand_samples, rand_vocab

pytestmark = pytest.mark.gpu

ALPHA = b"abcd"
TAIL = 64  # canary elements behind every output buffer
C32 = 0xA5A5A5A5
C64 = 0xA5A5A5A5A5A5A5A5
SENT = -0x5A5A5A5A5A5A5A5B  # device sentinel (int64; as int32 it is 0xA5A5A5A5)
SLEEP_CYCLES = 40_000_000  # torch.cuda._sleep: ~20 ms at B200 clocks
EM_HOT = 4096  # ids below this are counted in shared memory by the frequency pass (tgx_kernels.cuh)


@pytest.fixture(scope="module")
def N():
    from tokengeex_b200 import _native
    return _native


def torch_mod():
    import torch
    return torch


def big_vocab(seed=0x5EED):
    """Complete over 'abcd' with 6000 tokens of up to 7 bytes: ids on both sides of EM_HOT are used."""
    return rand_vocab(random.Random(seed), alphabet=ALPHA, n_tok=6000, max_len=7)


def dev(blob):
    return torch_mod().from_numpy(np.ascontiguousarray(blob)).cuda()


def dev_off(off):
    return torch_mod().from_numpy(np.asarray(off, np.uint64).view(np.int64).copy()).cuda()


def guarded(n, dtype, fill=SENT):
    """A device buffer of n elements followed by TAIL canary elements."""
    torch = torch_mod()
    if dtype == torch.int32:
        fill = fill & 0xFFFFFFFF
        fill = fill - (1 << 32) if fill >= 1 << 31 else fill
    return torch.full((n + TAIL,), fill, dtype=dtype, device="cuda")


def assert_tail(t, n, ctx=None):
    ref = t[-1].item()
    assert bool((t[n:] == ref).all()), ("canary overwritten", ctx)
    assert ref == guarded(0, t.dtype)[0].item(), ("canary overwritten", ctx)


def u64(t):
    return t.cpu().numpy().view(np.uint64)


def packed_pairs(ab):
    return (ab[:, 0].astype(np.uint64) << np.uint64(32)) | ab[:, 1].astype(np.uint64)


def host_buf(n, dtype, fill):
    return np.full(n + TAIL, fill, dtype)


def host_tail_ok(a, n, fill):
    return bool(np.all(a[n:] == np.array(fill, a.dtype)))


def want_first(wbad):
    return wbad - 1  # the oracle returns the lowest failing index + 1, or 0


# ----------------------------------------------------------------------------- a. stream order
@pytest.fixture(scope="module")
def stream_case():
    """Texts A and B with the same offsets, both with a path under a complete vocabulary, and the oracle's results
    for B."""
    rng = random.Random(77)
    toks, scores = big_vocab()
    sa = rand_samples(rng, ALPHA, 300, 1, 400)
    sb = [bytes(rng.choice(ALPHA) for _ in range(len(s))) for s in sa]
    blob_a, off = O.pack_samples(sa)
    blob_b, off_b = O.pack_samples(sb)
    assert np.array_equal(off, off_b)
    om = O.OracleModel(toks, scores)
    want = {
        "encode": om.encode_batch(blob_b, off, threads=8),
        "freq": om.token_frequencies(blob_b, off, threads=8),
        "pairs": om.pair_frequencies(blob_b, off, threads=8),
        "limbs": om.run_e_step_fixed(blob_b, off, threads=8)[0],
    }
    return toks, scores, blob_a, blob_b, off, want


STREAM_ENTRY_POINTS = ["encode_batch_dev", "token_frequencies_dev", "pair_frequencies_dev", "expected_counts_dev",
                       "expected_counts_fixed_dev", "counts_from_limbs_dev"]


@pytest.mark.parametrize("entry", STREAM_ENTRY_POINTS)
def test_dev_calls_order_after_the_default_stream(N, stream_case, entry):
    """The inputs and outputs of a `_dev` call are produced on the default stream behind a ~20 ms sleep kernel, and the
    call is made at once.  Its results must be the oracle's for the text written last (B), and nothing the default
    stream wrote after the sleep may overwrite them.  The handle is warmed with the identical call first, so that no
    buffer grows (cudaFree synchronises the device) in the measured call."""
    torch = torch_mod()
    toks, scores, blob_a, blob_b, off, want = stream_case
    gm = N.Model(toks, scores, device=0)
    V, S, n = len(toks), len(off) - 1, int(off[-1])
    d_text, d_a, d_b, d_off = dev(blob_a), dev(blob_a), dev(blob_b), dev_off(off)
    p = (d_text.data_ptr(), d_off.data_ptr(), S, n)
    if entry == "encode_batch_dev":
        ids = torch.zeros(n + 1, dtype=torch.int32, device="cuda")
        id_off = torch.zeros(S + 1, dtype=torch.int64, device="cuda")
        st = torch.zeros(S, dtype=torch.int32, device="cuda")
        pl = torch.zeros(S, dtype=torch.int64, device="cuda")
        outs = [ids, id_off, st, pl]
        call = lambda: gm.encode_batch_dev(*p, False, ids.data_ptr(), n + 1, id_off.data_ptr(), st.data_ptr(),
                                           pl.data_ptr())
        accs = []
    elif entry == "token_frequencies_dev":
        fr = torch.zeros(V, dtype=torch.int64, device="cuda")
        outs, accs = [], [fr]
        call = lambda: gm.token_frequencies_dev(*p, False, fr.data_ptr())
    elif entry == "pair_frequencies_dev":
        cap = n
        pairs = torch.zeros(cap, dtype=torch.int64, device="cuda")
        counts = torch.zeros(cap, dtype=torch.int64, device="cuda")
        outs, accs = [pairs, counts], []
        call = lambda: gm.pair_frequencies_dev(*p, False, pairs.data_ptr(), counts.data_ptr(), cap)
    elif entry == "expected_counts_dev":
        ex = torch.zeros(V, dtype=torch.float64, device="cuda")
        outs, accs = [], [ex]
        call = lambda: gm.expected_counts_dev(*p, ex.data_ptr())
    elif entry == "expected_counts_fixed_dev":
        limbs = torch.zeros(5 * V, dtype=torch.int64, device="cuda")
        outs, accs = [], [limbs]
        call = lambda: gm.expected_counts_fixed_dev(*p, limbs.data_ptr())
    else:
        lb = torch.zeros(5 * V, dtype=torch.int64, device="cuda")
        gm.expected_counts_fixed_dev(d_b.data_ptr(), d_off.data_ptr(), S, n, lb.data_ptr())
        limbs = torch.zeros_like(lb)
        ex = torch.zeros(V, dtype=torch.float64, device="cuda")
        outs, accs = [ex], []
        call = lambda: gm.counts_from_limbs_dev(limbs.data_ptr(), V, ex.data_ptr())
    call()  # warm: every buffer of the handle has its size
    d_text.copy_(d_a)
    torch.cuda.synchronize()
    torch.cuda._sleep(SLEEP_CYCLES)
    d_text.copy_(d_b)
    if entry == "counts_from_limbs_dev":
        limbs.copy_(lb)
    for t in outs:
        t.fill_(float("nan") if t.dtype == torch.float64 else -1)
    for t in accs:
        t.fill_(float("nan") if t.dtype == torch.float64 else SENT)
        t.zero_()
    r = call()
    torch.cuda.synchronize()
    if entry == "encode_batch_dev":
        tot, rc, bad = r
        wids, wid_off, wst, wpl, wbad = want["encode"]
        assert rc == 0 and bad == -1 and tot == wids.size
        assert np.array_equal(u64(id_off), wid_off)
        assert np.array_equal(ids.cpu().numpy().view(np.uint32)[:tot], wids)
        assert np.array_equal(st.cpu().numpy(), wst) and np.array_equal(u64(pl), wpl)
    elif entry == "token_frequencies_dev":
        assert r[0] == 0 and np.array_equal(u64(fr), want["freq"])
    elif entry == "pair_frequencies_dev":
        k, rc, bad, blen = r
        wp, wc = want["pairs"]
        assert rc == 0 and k == len(wc)
        assert np.array_equal(u64(pairs)[:k], packed_pairs(wp)) and np.array_equal(u64(counts)[:k], wc)
    elif entry == "expected_counts_dev" or entry == "counts_from_limbs_dev":
        if entry == "expected_counts_dev":
            assert r[0] == 0
        got = ex.cpu().numpy()
        assert np.array_equal(got.view(np.uint64), nearest(want["limbs"]).view(np.uint64))
    else:
        assert r[0] == 0 and limbs_to_ints(limbs, V) == want["limbs"]


# ----------------------------------------------------------------------------- b. capacities and output bounds
@pytest.fixture(scope="module")
def cap_case():
    """The big vocabulary, ~60 KB of samples (empty ones included) and a sample without a path ('z')."""
    rng = random.Random(1234)
    toks, scores = big_vocab()
    samples = rand_samples(rng, ALPHA, 300, 0, 400)
    nopath = samples[:150] + [b"abz" + b"c" * 30] + samples[150:] + [b"zz"]
    return toks, scores, samples, nopath


def host_encode(N, gm, blob, off, ids_cap, crlf=False, optional=True):
    """tgx_encode_batch into canary-guarded host buffers; asserts the canaries."""
    S = len(off) - 1
    ids = host_buf(ids_cap, np.uint32, C32)
    id_off = host_buf(S + 1, np.uint64, C64)
    status = host_buf(S, np.uint32, C32).view(np.int32)
    plen = host_buf(S, np.uint64, C64)
    bad = C.c_int64(12345)
    rc = N.lib().tgx_encode_batch(gm._h, N._p(blob, N.u8p), N._p(off, N.u64p), S, N.TGX_FLAG_CRLF if crlf else 0,
                                  N._p(ids, N.u32p), ids_cap, N._p(id_off, N.u64p),
                                  N._p(status, N.i32p) if optional else None, N._p(plen, N.u64p) if optional else None,
                                  C.byref(bad) if optional else None)
    assert host_tail_ok(ids, ids_cap, C32) and host_tail_ok(id_off, S + 1, C64)
    k = S if optional else 0
    assert host_tail_ok(status.view(np.uint32), k, C32) and host_tail_ok(plen, k, C64)
    return rc, ids[:ids_cap], id_off[:S + 1], status[:S], plen[:S], bad.value


@pytest.mark.parametrize("chunk", [1 << 28, 4096])
def test_encode_batch_host_capacity(N, cap_case, chunk):
    """ids_cap below the total fails with TGX_ERR_CAPACITY and id_off[S] = the total, wherever the overflow falls
    (first, a middle, the last of ~15 chunks); id offsets, status, processed lengths and first_bad are still complete;
    nothing is written past ids_cap; a retry with exactly the reported size gives the oracle's result.  With a NoPath
    sample in the batch as well, CAPACITY is returned (first_bad still names the sample)."""
    toks, scores, samples, nopath = cap_case
    gm, om = N.Model(toks, scores, device=0), O.OracleModel(toks, scores)
    gm.set_option(7, chunk)
    for batch in (samples, nopath):
        blob, off = N.pack(batch)
        wids, wid_off, wst, wpl, wbad = om.encode_batch(blob, off, threads=8)
        total = wids.size
        first = want_first(wbad)
        wstatus = np.where(wst != 0, N.TGX_ERR_NO_PATH, 0)
        for cap in sorted({0, 1, total // 3, total // 2, total - 1}):
            rc, ids, id_off, st, pl, bad = host_encode(N, gm, blob, off, cap)
            assert rc == N.TGX_ERR_CAPACITY and int(id_off[-1]) == total, (chunk, cap)
            assert np.array_equal(id_off, wid_off) and np.array_equal(st, wstatus) and np.array_equal(pl, wpl)
            assert bad == first
        rc, ids, id_off, st, pl, bad = host_encode(N, gm, blob, off, total)
        assert rc == (N.TGX_ERR_NO_PATH if first >= 0 else N.TGX_OK) and bad == first
        assert np.array_equal(ids, wids) and np.array_equal(id_off, wid_off)
        assert np.array_equal(st, wstatus) and np.array_equal(pl, wpl)


def test_encode_batch_dev_sizing_and_capacity(N, cap_case):
    """The sizing call (d_ids = NULL, ids_cap = 0) reports the total; ids_cap = total - 1 writes exactly the first
    total - 1 ids (the emit kernel's bound) and reports CAPACITY, also with a NoPath sample in the batch; ids_cap =
    total gives the oracle's ids."""
    torch = torch_mod()
    toks, scores, samples, nopath = cap_case
    gm, om = N.Model(toks, scores, device=0), O.OracleModel(toks, scores)
    L = N.lib()
    for batch in (samples, nopath):
        blob, off = N.pack(batch)
        wids, wid_off, wst, wpl, wbad = om.encode_batch(blob, off, threads=8)
        total, first = wids.size, want_first(wbad)
        S, n = len(off) - 1, int(off[-1])
        d_text, d_off = dev(blob), dev_off(off)
        id_off = guarded(S + 1, torch.int64)
        tot, bad = C.c_uint64(0), C.c_int64(7)
        rc = L.tgx_encode_batch_dev(gm._h, d_text.data_ptr(), d_off.data_ptr(), S, n, 0, None, 0, id_off.data_ptr(),
                                    None, None, C.byref(tot), C.byref(bad))
        torch.cuda.synchronize()
        assert rc == N.TGX_ERR_CAPACITY and tot.value == total and bad.value == first
        assert np.array_equal(u64(id_off)[:S + 1], wid_off)
        assert_tail(id_off, S + 1)
        for cap in (total - 1, total):
            ids = guarded(cap, torch.int32)
            id_off = guarded(S + 1, torch.int64)
            st = guarded(S, torch.int32)
            pl = guarded(S, torch.int64)
            rc = L.tgx_encode_batch_dev(gm._h, d_text.data_ptr(), d_off.data_ptr(), S, n, 0, ids.data_ptr(), cap,
                                        id_off.data_ptr(), st.data_ptr(), pl.data_ptr(), C.byref(tot), C.byref(bad))
            torch.cuda.synchronize()
            for t, k in ((ids, cap), (id_off, S + 1), (st, S), (pl, S)):
                assert_tail(t, k, cap)
            want_rc = N.TGX_ERR_CAPACITY if cap < total else (N.TGX_ERR_NO_PATH if first >= 0 else N.TGX_OK)
            assert rc == want_rc and tot.value == total and bad.value == first, cap
            assert np.array_equal(ids.cpu().numpy().view(np.uint32)[:cap], wids[:cap])
            assert np.array_equal(u64(id_off)[:S + 1], wid_off) and np.array_equal(u64(pl)[:S], wpl)
            assert np.array_equal(st.cpu().numpy()[:S], np.where(wst != 0, N.TGX_ERR_NO_PATH, 0))


def corpus_data(rng):
    """NUL-separated 'abcd' samples with empty ones, a leading and a trailing NUL: ~60 KB."""
    parts = rand_samples(rng, ALPHA, 300, 0, 400)
    return b"\x00" + b"\x00".join(parts) + b"\x00\x00"


def corpus_ref(om, data, sep):
    ids, off = [], [0]
    for s in data.split(b"\x00"):
        if s:
            ids += om.encode(s) + ([sep] if sep >= 0 else [])
            off.append(len(ids))
    return ids, off


def host_corpus(N, gm, data, id_bytes, sep, ids_cap, off_cap):
    a = np.frombuffer(data, np.uint8) if data else np.zeros(1, np.uint8)
    dt = np.uint16 if id_bytes == 2 else np.uint32
    cid = 0xA5A5 if id_bytes == 2 else C32
    ids = host_buf(ids_cap, dt, cid)
    off = host_buf(off_cap, np.uint64, C64)
    ns, ni, bad, pos = C.c_uint64(99), C.c_uint64(99), C.c_int64(99), C.c_uint64(99)
    rc = N.lib().tgx_encode_corpus(gm._h, a.ctypes.data, len(data), 0, 0, sep, id_bytes, ids.ctypes.data, ids_cap,
                                   N._p(off, N.u64p), off_cap, C.byref(ns), C.byref(ni), C.byref(bad), C.byref(pos))
    assert host_tail_ok(ids, ids_cap, cid) and host_tail_ok(off, off_cap, C64), (ids_cap, off_cap)
    return rc, ids[:ids_cap], off[:off_cap], ns.value, ni.value, bad.value, pos.value


@pytest.mark.parametrize("chunk", [1 << 28, 4096])
def test_encode_corpus_capacity(N, chunk):
    """ids_cap and off_cap each at need - 1 and at need, for u16 and u32 ids, with and without a separator, in one and
    in ~15 chunks: CAPACITY reports n_samples and n_ids, nothing is written past a capacity, and the exact sizes give
    the oracle's ids and offsets."""
    rng = random.Random(chunk)
    toks, scores = big_vocab()
    gm, om = N.Model(toks, scores, device=0), O.OracleModel(toks, scores)
    gm.set_option(7, chunk)
    data = corpus_data(rng)
    for id_bytes, sep in ((4, -1), (4, 70000), (2, -1), (2, len(toks) - 1)):
        wids, woff = corpus_ref(om, data, sep)
        need_ids, need_off = len(wids), len(woff)
        for ids_cap, off_cap in ((need_ids - 1, need_off), (need_ids, need_off - 1), (need_ids, need_off)):
            rc, ids, off, ns, ni, bad, pos = host_corpus(N, gm, data, id_bytes, sep, ids_cap, off_cap)
            ctx = (chunk, id_bytes, sep, ids_cap, off_cap)
            assert ns == need_off - 1 and ni == need_ids, ctx
            if ids_cap == need_ids and off_cap == need_off:
                assert rc == N.TGX_OK and bad == -1, ctx
                assert ids.astype(np.int64).tolist() == wids and off.tolist() == woff, ctx
            else:
                assert rc == N.TGX_ERR_CAPACITY, ctx


def host_pairs(N, gm, blob, off, cap, optional=True, crlf=False):
    S = len(off) - 1
    pairs = host_buf(cap, np.uint64, C64)
    counts = host_buf(cap, np.uint64, C64)
    n, bad, blen = C.c_uint64(0), C.c_int64(99), C.c_uint64(99)
    rc = N.lib().tgx_pair_frequencies(gm._h, N._p(blob, N.u8p), N._p(off, N.u64p), S, N.TGX_FLAG_CRLF if crlf else 0,
                                      N._p(pairs, N.u64p), N._p(counts, N.u64p), cap, C.byref(n),
                                      C.byref(bad) if optional else None, C.byref(blen) if optional else None)
    assert host_tail_ok(pairs, cap, C64) and host_tail_ok(counts, cap, C64)
    return rc, pairs[:cap], counts[:cap], n.value, bad.value, blen.value


def test_pair_frequencies_capacity(N, cap_case):
    """cap = n - 1: CAPACITY with *n_pairs = n and nothing written; cap = n: the oracle's pairs and counts in order,
    nothing past them.  Host entry point and Model.pair_frequencies_dev."""
    torch = torch_mod()
    toks, scores, samples, _ = cap_case
    gm, om = N.Model(toks, scores, device=0), O.OracleModel(toks, scores)
    blob, off = N.pack(samples)
    wp, wc = om.pair_frequencies(blob, off, threads=8)
    want = packed_pairs(wp)
    k = len(wc)
    assert k > 100
    rc, pairs, counts, n, bad, blen = host_pairs(N, gm, blob, off, k - 1)
    assert rc == N.TGX_ERR_CAPACITY and n == k
    assert np.all(pairs == np.uint64(C64)) and np.all(counts == np.uint64(C64))
    rc, pairs, counts, n, bad, blen = host_pairs(N, gm, blob, off, k)
    assert rc == N.TGX_OK and n == k and np.array_equal(pairs, want) and np.array_equal(counts, wc)
    d_text, d_off = dev(blob), dev_off(off)
    S, nb = len(off) - 1, int(off[-1])
    for cap in (k - 1, k):
        dp, dc = guarded(cap, torch.int64), guarded(cap, torch.int64)
        n, rc, bad, blen = gm.pair_frequencies_dev(d_text.data_ptr(), d_off.data_ptr(), S, nb, False, dp.data_ptr(),
                                                   dc.data_ptr(), cap)
        torch.cuda.synchronize()
        assert n == k and rc == (N.TGX_ERR_CAPACITY if cap < k else N.TGX_OK)
        assert_tail(dp, cap)
        assert_tail(dc, cap)
        if cap < k:
            assert bool((dp == SENT).all()) and bool((dc == SENT).all())
        else:
            assert np.array_equal(u64(dp)[:k], want) and np.array_equal(u64(dc)[:k], wc)


# ----------------------------------------------------------------------------- c. accumulation, NULLs, degenerate
def test_token_frequencies_dev_accumulates(N, cap_case):
    """freq[id] += counts: a prefilled buffer ends at prefill + the oracle's counts, a second call adds them again.
    Ids below EM_HOT (counted in shared memory first) and above it are both counted."""
    torch = torch_mod()
    toks, scores, samples, _ = cap_case
    gm, om = N.Model(toks, scores, device=0), O.OracleModel(toks, scores)
    blob, off = N.pack(samples)
    want = om.token_frequencies(blob, off, threads=8).astype(np.int64)
    V = len(toks)
    assert want[:EM_HOT].any() and want[EM_HOT:].any()
    prefill = np.random.default_rng(5).integers(0, 1 << 40, V, dtype=np.int64)
    fr = guarded(V, torch.int64)
    fr[:V] = torch.from_numpy(prefill).cuda()
    d_text, d_off = dev(blob), dev_off(off)
    for k in (1, 2):
        rc, bad, blen = gm.token_frequencies_dev(d_text.data_ptr(), d_off.data_ptr(), len(off) - 1, int(off[-1]),
                                                 False, fr.data_ptr())
        torch.cuda.synchronize()
        assert rc == 0 and bad == -1
        assert np.array_equal(fr[:V].cpu().numpy(), prefill + k * want), k
        assert_tail(fr, V, k)


def test_null_optional_outputs(N, cap_case):
    """status / proc_len / first_bad / bad_len NULL on the host and `_dev` encode and frequency entry points: the same
    return code and results, on a batch with a NoPath sample."""
    torch = torch_mod()
    toks, scores, _, nopath = cap_case
    gm, om = N.Model(toks, scores, device=0), O.OracleModel(toks, scores)
    L = N.lib()
    blob, off = N.pack(nopath)
    S, n = len(off) - 1, int(off[-1])
    wids, wid_off, *_ = om.encode_batch(blob, off, threads=8)
    rc, ids, id_off, *_ = host_encode(N, gm, blob, off, n + 1, optional=False)
    assert rc == N.TGX_ERR_NO_PATH and np.array_equal(ids[:wids.size], wids) and np.array_equal(id_off, wid_off)
    d_text, d_off = dev(blob), dev_off(off)
    d_ids, d_id_off = guarded(n + 1, torch.int32), guarded(S + 1, torch.int64)
    tot = C.c_uint64(0)
    rc = L.tgx_encode_batch_dev(gm._h, d_text.data_ptr(), d_off.data_ptr(), S, n, 0, d_ids.data_ptr(), n + 1,
                                d_id_off.data_ptr(), None, None, C.byref(tot), None)
    torch.cuda.synchronize()
    assert rc == N.TGX_ERR_NO_PATH and tot.value == wids.size
    assert np.array_equal(d_ids.cpu().numpy().view(np.uint32)[:wids.size], wids)
    assert np.array_equal(u64(d_id_off)[:S + 1], wid_off)
    fr = np.zeros(len(toks), np.uint64)
    rc = L.tgx_token_frequencies(gm._h, N._p(blob, N.u8p), N._p(off, N.u64p), S, 0, N._p(fr, N.u64p), None, None)
    assert rc == N.TGX_ERR_NO_PATH
    d_fr = torch.zeros(len(toks), dtype=torch.int64, device="cuda")
    rc = L.tgx_token_frequencies_dev(gm._h, d_text.data_ptr(), d_off.data_ptr(), S, n, 0, d_fr.data_ptr(), None, None)
    assert rc == N.TGX_ERR_NO_PATH
    rc, *_ = host_pairs(N, gm, blob, off, n, optional=False)
    assert rc == N.TGX_ERR_NO_PATH
    dp, dc = guarded(n, torch.int64), guarded(n, torch.int64)
    k = C.c_uint64(0)
    rc = L.tgx_pair_frequencies_dev(gm._h, d_text.data_ptr(), d_off.data_ptr(), S, n, 0, dp.data_ptr(), dc.data_ptr(),
                                    n, C.byref(k), None, None)
    assert rc == N.TGX_ERR_NO_PATH


DEGENERATE = {
    "no_samples": [],
    "all_empty": [b"", b"", b""],
    "one_byte": [b"a"],
    "all_nopath": [b"abz", b"z", b"cdz"],  # (each ends in 'z': nothing ends at eos, so z = 0.0 in the E-step too)
}


@pytest.mark.parametrize("case", list(DEGENERATE))
def test_degenerate_batches(N, case):
    """S = 0, S > 0 with only empty samples, one 1-byte sample, every sample NoPath: every entry point, host and
    `_dev`, matches the oracle; an empty batch returns TGX_OK and leaves the `_dev` accumulators untouched."""
    torch = torch_mod()
    samples = DEGENERATE[case]
    toks, scores = rand_vocab(random.Random(8), alphabet=ALPHA, n_tok=40, max_len=4)
    gm, om = N.Model(toks, scores, device=0), O.OracleModel(toks, scores)
    V, S = len(toks), len(samples)
    blob, off = N.pack(samples)
    n = int(off[-1])
    d_text, d_off = dev(blob), dev_off(off)
    wids, wid_off, wst, wpl, wbad = om.encode_batch(blob, off)
    first = want_first(wbad)
    want_rc = N.TGX_ERR_NO_PATH if first >= 0 else N.TGX_OK
    # encode, host and device
    rc, ids, id_off, st, pl, bad = host_encode(N, gm, blob, off, n + 1)
    assert rc == want_rc and bad == first and np.array_equal(id_off, wid_off) and np.array_equal(ids[:wids.size], wids)
    assert np.array_equal(pl, wpl) and np.array_equal(st != 0, wst != 0)
    d_ids, d_id_off = guarded(n + 1, torch.int32), guarded(S + 1, torch.int64)
    d_st, d_pl = guarded(S, torch.int32), guarded(S, torch.int64)
    tot, rc, bad = gm.encode_batch_dev(d_text.data_ptr(), d_off.data_ptr(), S, n, False, d_ids.data_ptr(), n + 1,
                                       d_id_off.data_ptr(), d_st.data_ptr(), d_pl.data_ptr())
    torch.cuda.synchronize()
    assert rc == want_rc and bad == first and tot == wids.size
    assert np.array_equal(u64(d_id_off)[:S + 1], wid_off) and np.array_equal(u64(d_pl)[:S], wpl)
    assert np.array_equal(d_ids.cpu().numpy().view(np.uint32)[:tot], wids)
    for t, k in ((d_ids, n + 1), (d_id_off, S + 1), (d_st, S), (d_pl, S)):
        assert_tail(t, k)
    # token frequencies
    fr, rc, bad, blen = gm.token_frequencies(blob, off)
    assert rc == want_rc and bad == first and (first < 0 or blen == wpl[first])
    if first < 0:
        assert np.array_equal(fr, om.token_frequencies(blob, off))
    prefill = np.arange(V, dtype=np.int64) * 3 + 1
    d_fr = guarded(V, torch.int64)
    d_fr[:V] = torch.from_numpy(prefill).cuda()
    rc, bad, blen = gm.token_frequencies_dev(d_text.data_ptr(), d_off.data_ptr(), S, n, False, d_fr.data_ptr())
    torch.cuda.synchronize()
    assert rc == want_rc and bad == first and (first < 0 or blen == wpl[first])
    if first < 0:
        assert np.array_equal(d_fr[:V].cpu().numpy(), prefill + om.token_frequencies(blob, off).astype(np.int64))
    assert_tail(d_fr, V)
    # pair frequencies
    cap = max(n, 1)
    rc, pairs, counts, k, bad, blen = host_pairs(N, gm, blob, off, cap)
    assert rc == want_rc and bad == first and (first < 0 or blen == wpl[first])
    dp, dc = guarded(cap, torch.int64), guarded(cap, torch.int64)
    k2, rc2, bad2, blen2 = gm.pair_frequencies_dev(d_text.data_ptr(), d_off.data_ptr(), S, n, False, dp.data_ptr(),
                                                   dc.data_ptr(), cap)
    torch.cuda.synchronize()
    assert rc2 == want_rc and bad2 == first and (first < 0 or blen2 == wpl[first])
    assert_tail(dp, cap)
    assert_tail(dc, cap)
    if first < 0:
        wp, wc = om.pair_frequencies(blob, off)
        assert k == k2 == len(wc) and np.array_equal(pairs[:k], packed_pairs(wp)) and np.array_equal(counts[:k], wc)
        assert np.array_equal(u64(dp)[:k], packed_pairs(wp)) and np.array_equal(u64(dc)[:k], wc)
    # E-step: host, f64 accumulate, limbs accumulate
    wex, wrc, wbz_s, wbz = om.run_e_step(blob, off)
    ex, rc, bs, bz = gm.expected_counts(blob, off)
    assert rc == (N.TGX_ERR_BAD_Z if wrc else N.TGX_OK) and bs == wbz_s and bz == wbz
    if not wrc:
        want_fx = om.run_e_step_fixed(blob, off)[0]
        assert np.array_equal(ex.view(np.uint64), nearest(want_fx).view(np.uint64))
    d_ex = guarded(V, torch.float64, 0.0)
    d_ex[:V] = torch.from_numpy(prefill.astype(np.float64)).cuda()
    rc, bs, bz = gm.expected_counts_dev(d_text.data_ptr(), d_off.data_ptr(), S, n, d_ex.data_ptr())
    torch.cuda.synchronize()
    assert rc == (N.TGX_ERR_BAD_Z if wrc else N.TGX_OK) and bs == wbz_s and bz == wbz
    if not wrc:
        assert np.array_equal(d_ex[:V].cpu().numpy(), prefill + nearest(want_fx))
    assert bool((d_ex[V:] == 0.0).all())
    d_l = guarded(5 * V, torch.int64)
    d_l[:5 * V] = 7
    rc, bs, bz = gm.expected_counts_fixed_dev(d_text.data_ptr(), d_off.data_ptr(), S, n, d_l.data_ptr())
    torch.cuda.synchronize()
    assert rc == (N.TGX_ERR_BAD_Z if wrc else N.TGX_OK) and bs == wbz_s and bz == wbz
    assert_tail(d_l, 5 * V)
    if not wrc:
        got = limbs_to_ints(d_l[:5 * V] - 7, V)
        assert got == want_fx
    if S == 0 or n == 0:  # empty batches leave the accumulators untouched
        assert np.array_equal(d_fr[:V].cpu().numpy(), prefill)
        assert np.array_equal(d_ex[:V].cpu().numpy(), prefill.astype(np.float64))
        assert bool((d_l[:5 * V] == 7).all())


CORPUS_DEGENERATE = [(b"", 0, []), (b"\x00\x00\x00", 0, []), (b"a", 1, None), (b"z\x00\x00zz\x00", 2, None)]


@pytest.mark.parametrize("i", range(len(CORPUS_DEGENERATE)))
def test_encode_corpus_degenerate(N, i):
    """tgx_encode_corpus on no bytes, only NUL bytes, one byte, and only NoPath samples."""
    data, n_samples, _ = CORPUS_DEGENERATE[i]
    toks, scores = rand_vocab(random.Random(8), alphabet=ALPHA, n_tok=40, max_len=4)
    gm, om = N.Model(toks, scores, device=0), O.OracleModel(toks, scores)
    rc, ids, off, ns, ni, bad, pos = host_corpus(N, gm, data, 4, -1, len(data) + 1, len(data) + 2)
    assert ns == n_samples
    if b"z" in data:
        assert rc == N.TGX_ERR_NO_PATH and bad == 0 and pos == 1 and ni == 0 and off[:3].tolist() == [0, 0, 0]
    else:
        wids, woff = corpus_ref(om, data, -1)
        assert rc == N.TGX_OK and bad == -1 and ni == len(wids)
        assert ids[:ni].tolist() == wids and off[:ns + 1].tolist() == woff


def test_crlf_through_dev_entry_points(N):
    """TGX_FLAG_CRLF through encode_batch_dev (with proc_len), token_frequencies_dev and pair_frequencies_dev on lone
    and doubled CR, CR LF pairs and random CR / LF text, with tokens that hold CR and LF."""
    torch = torch_mod()
    rng = random.Random(31)
    alpha = b"ab\r\n"
    toks, scores = rand_vocab(rng, alphabet=alpha, n_tok=120, max_len=5)
    gm, om = N.Model(toks, scores, device=0), O.OracleModel(toks, scores)
    samples = [b"\r\n", b"\r", b"\r\r\n", b"\n\r", b"\r\n\r\n", b"a\r", b"\r\na", b""]
    samples += rand_samples(rng, alpha, 150, 0, 200) + rand_samples(rng, b"\r\n", 30, 1, 40)
    blob, off = N.pack(samples)
    S, n = len(off) - 1, int(off[-1])
    pblob, poff = N.pack([O.crlf(s) for s in samples])
    wids, wid_off, wst, wpl, wbad = om.encode_batch(blob, off, crlf=True)
    assert wbad == 0 and wpl.tolist() == [len(O.crlf(s)) for s in samples]
    d_text, d_off = dev(blob), dev_off(off)
    d_ids, d_id_off = guarded(n + 1, torch.int32), guarded(S + 1, torch.int64)
    d_st, d_pl = guarded(S, torch.int32), guarded(S, torch.int64)
    tot, rc, bad = gm.encode_batch_dev(d_text.data_ptr(), d_off.data_ptr(), S, n, True, d_ids.data_ptr(), n + 1,
                                       d_id_off.data_ptr(), d_st.data_ptr(), d_pl.data_ptr())
    torch.cuda.synchronize()
    assert rc == 0 and bad == -1 and tot == wids.size
    assert np.array_equal(d_ids.cpu().numpy().view(np.uint32)[:tot], wids)
    assert np.array_equal(u64(d_id_off)[:S + 1], wid_off) and np.array_equal(u64(d_pl)[:S], wpl)
    assert not d_st[:S].any()
    d_fr = torch.zeros(len(toks), dtype=torch.int64, device="cuda")
    rc, bad, blen = gm.token_frequencies_dev(d_text.data_ptr(), d_off.data_ptr(), S, n, True, d_fr.data_ptr())
    assert rc == 0 and np.array_equal(u64(d_fr), om.token_frequencies(pblob, poff))
    wp, wc = om.pair_frequencies(pblob, poff)
    dp, dc = guarded(n, torch.int64), guarded(n, torch.int64)
    k, rc, bad, blen = gm.pair_frequencies_dev(d_text.data_ptr(), d_off.data_ptr(), S, n, True, dp.data_ptr(),
                                               dc.data_ptr(), n)
    torch.cuda.synchronize()
    assert rc == 0 and k == len(wc)
    assert np.array_equal(u64(dp)[:k], packed_pairs(wp)) and np.array_equal(u64(dc)[:k], wc)
    assert_tail(dp, n)
    assert_tail(dc, n)


# ----------------------------------------------------------------------------- d. error reports
@pytest.mark.parametrize("crlf", [False, True])
def test_nopath_reports_on_dev_paths(N, crlf):
    """first_bad / bad_len of the `_dev` frequency passes and of encode_batch_dev (and their host forms) are the
    oracle's lowest failing sample and its processed length (after crlf: shorter than the raw sample)."""
    torch = torch_mod()
    rng = random.Random(41)
    alpha = b"ab\r\n"
    toks, scores = rand_vocab(rng, alphabet=alpha, n_tok=120, max_len=5)
    gm, om = N.Model(toks, scores, device=0), O.OracleModel(toks, scores)
    samples = rand_samples(rng, alpha, 100, 0, 200)
    samples[37] = b"a\r\nb\r\nz\r\n\r\nab"
    samples[60] = b"z"
    samples[81] = b"\r\n\r\nz"
    blob, off = N.pack(samples)
    S, n = len(off) - 1, int(off[-1])
    wids, wid_off, wst, wpl, wbad = om.encode_batch(blob, off, crlf=crlf)
    first = want_first(wbad)
    assert first == 37 and wpl[first] == (len(samples[37]) - (4 if crlf else 0))
    d_text, d_off = dev(blob), dev_off(off)
    d_ids, d_id_off = guarded(n + 1, torch.int32), guarded(S + 1, torch.int64)
    d_st, d_pl = guarded(S, torch.int32), guarded(S, torch.int64)
    tot, rc, bad = gm.encode_batch_dev(d_text.data_ptr(), d_off.data_ptr(), S, n, crlf, d_ids.data_ptr(), n + 1,
                                       d_id_off.data_ptr(), d_st.data_ptr(), d_pl.data_ptr())
    torch.cuda.synchronize()
    assert rc == N.TGX_ERR_NO_PATH and bad == first and u64(d_pl)[first] == wpl[first]
    assert np.array_equal(d_st[:S].cpu().numpy() != 0, wst != 0)
    d_fr = torch.zeros(len(toks), dtype=torch.int64, device="cuda")
    rc, bad, blen = gm.token_frequencies_dev(d_text.data_ptr(), d_off.data_ptr(), S, n, crlf, d_fr.data_ptr())
    assert rc == N.TGX_ERR_NO_PATH and bad == first and blen == wpl[first]
    fr, rc, bad, blen = gm.token_frequencies(blob, off, crlf=crlf)
    assert rc == N.TGX_ERR_NO_PATH and bad == first and blen == wpl[first]
    dp, dc = guarded(n, torch.int64), guarded(n, torch.int64)
    k, rc, bad, blen = gm.pair_frequencies_dev(d_text.data_ptr(), d_off.data_ptr(), S, n, crlf, dp.data_ptr(),
                                               dc.data_ptr(), n)
    assert rc == N.TGX_ERR_NO_PATH and bad == first and blen == wpl[first]
    rc, pairs, counts, k, bad, blen = host_pairs(N, gm, blob, off, n, crlf=crlf)
    assert rc == N.TGX_ERR_NO_PATH and bad == first and blen == wpl[first]
    # the pair passes check NoPath before they count pairs: it wins over a capacity of 0
    rc, pairs, counts, k, bad, blen = host_pairs(N, gm, blob, off, 0, crlf=crlf)
    assert rc == N.TGX_ERR_NO_PATH and bad == first and blen == wpl[first]
    k, rc, bad, blen = gm.pair_frequencies_dev(d_text.data_ptr(), d_off.data_ptr(), S, n, crlf, 0, 0, 0)
    assert rc == N.TGX_ERR_NO_PATH and bad == first and blen == wpl[first]


# BAD_Z: single-path snippets whose z is not normal.  'q' (score 0.0): z = 0.0; 's' / 't' (tiny negative scores): z is
# subnormal; a snippet whose last byte ('z') no token covers: nothing ends at eos, z = 0.0.
def bad_z_vocab():
    toks, scores = rand_vocab(random.Random(99), alphabet=ALPHA, n_tok=300, max_len=8)
    return toks + [b"q", b"s", b"t"], scores + [0.0, -1e-310, -1e-320]


def bad_snippet(rng, kind, length):
    if kind == "nopath":
        return bytes(rng.choice(ALPHA) for _ in range(length - 1)) + b"z"
    if kind == "zero":
        return b"q" * length
    return (b"s" if length <= 20 else b"t") * length


# E-step placement: snippets of at least 4000 bytes on a warp each (option 5), below 1000 bytes one lane each
# (option 17), lane-group kernels (option 2 = 4 lanes) in between; the lane snippets, longest first, in three groups
# cut at 30 % and 60 % (options 30 / 31).
PLACEMENT = {19: 1, 5: 4000, 17: 1000, 2: 4, 30: 300, 31: 600}
LANE_LENS = list(range(990, 40, -50))  # 20 lane snippets: groups [0, 6), [6, 12), [12, 20) by sorted position
TARGETS = {"warp": 4500, "lane_group": 2500, "lane_g0": LANE_LENS[2], "lane_g1": LANE_LENS[8],
           "lane_g2": LANE_LENS[15]}


def bad_z_batch(rng, target, kind, other):
    """Good snippets of every placement in shuffled order; the sample of length TARGETS[target] is bad (`kind`), and
    when `other` is set so is a later sample of another placement."""
    lens = [6000, 4500, 3000, 2500, 1500] + LANE_LENS
    rng.shuffle(lens)
    samples = [bytes(rng.choice(ALPHA) for _ in range(L)) for L in lens]
    i = lens.index(TARGETS[target])
    samples[i] = bad_snippet(rng, kind, lens[i])
    if other:
        later = [j for j in range(i + 1, len(lens))]
        if later:
            j = rng.choice(later)
            samples[j] = bad_snippet(rng, rng.choice(["nopath", "zero", "sub"]), lens[j])
    return samples


def configs():
    return [(g, None) for g in KERNEL_SETS] + [("placement", PLACEMENT)]


@pytest.fixture(scope="module")
def bad_z_batches():
    rng = random.Random(2024)
    return [((target, kind, other), bad_z_batch(rng, target, kind, other))
            for target in TARGETS for kind in ("nopath", "zero", "sub") for other in (False, True)]


def run_bad_z(N, gm, om, samples, snip, dropout=0.0, seed=0, ctx=None):
    blob, off = N.pack(samples)
    if dropout > 0.0:
        _, wrc, wbad, wz = om.run_e_step_dropout(blob, off, dropout, seed, keyed=True, max_sample_length=snip)
    else:
        _, wrc, wbad, wz = om.run_e_step(blob, off, max_sample_length=snip)
    assert wrc == 1 and wbad >= 0, ctx
    torch = torch_mod()
    d_text, d_off = dev(blob), dev_off(off)
    limbs = torch.zeros(5 * gm.V, dtype=torch.int64, device="cuda")
    rc, bad, bz = gm.expected_counts_fixed_dev(d_text.data_ptr(), d_off.data_ptr(), len(off) - 1, int(off[-1]),
                                               limbs.data_ptr(), snippet_len=snip)
    assert rc == N.TGX_ERR_BAD_Z and bad == wbad, (ctx, bad, wbad)
    assert np.float64(bz).view(np.uint64) == np.float64(wz).view(np.uint64), (ctx, bz, wz)
    return wz


@pytest.mark.parametrize("dropout", [0.0, 0.3])
@pytest.mark.parametrize("cfg", configs(), ids=lambda c: str(c[0]))
def test_bad_z_every_kernel_set_and_placement(N, bad_z_batches, cfg, dropout):
    """bad_sample is the oracle's lowest sample with a non-normal z and bad_z its z, bit for bit, for z = 0 from
    NoPath, z = 0 from zero scores and subnormal z, wherever the snippet runs: warp, lane-group kernel, each of the
    three lane groups.  (The host reads z back from the alpha array at alpha[eos] of the snippet.)"""
    g, opts = cfg
    toks, scores = bad_z_vocab()
    om = O.OracleModel(toks, scores)
    gm = N.Model(toks, scores, device=0)
    if opts is None:
        configure(gm, g)
    else:
        for k, v in opts.items():
            gm.set_option(k, v)
    if dropout:
        gm.set_dropout(dropout, 17)
    zs = set()
    for ctx, samples in bad_z_batches:
        zs.add(run_bad_z(N, gm, om, samples, 81920, dropout, 17, (g, dropout) + ctx))
    assert 0.0 in zs and any(z != 0.0 and abs(z) < 2.2250738585072014e-308 for z in zs)


@pytest.mark.parametrize("g", KERNEL_SETS)
def test_bad_z_later_snippets(N, g):
    """Snippets of 300 bytes: a bad second snippet behind a good first one, and two bad snippets of one sample (the
    first one's z is reported), behind good samples and before other bad ones."""
    toks, scores = bad_z_vocab()
    om = O.OracleModel(toks, scores)
    gm = N.Model(toks, scores, device=0)
    configure(gm, g)
    rng = random.Random(303)
    snip = 300
    good = lambda L: bytes(rng.choice(ALPHA) for _ in range(L))
    cases = [
        [good(700), good(300) + bad_snippet(rng, "nopath", 300), good(50)],
        [good(100), good(300) + good(300) + b"q" * 120, b"q" * 10],
        [good(900), b"t" * 300 + b"q" * 300 + good(30), bad_snippet(rng, "nopath", 20)],
        [good(20), good(300) + bad_snippet(rng, "nopath", 300) + b"t" * 300, b"s" * 3],
        [b"s" * 2 + b"q" * 3],  # one short bad snippet; z = -2e-310 + 0.0 * 3
    ]
    for i, samples in enumerate(cases):
        run_bad_z(N, gm, om, samples, snip, ctx=(g, i))
