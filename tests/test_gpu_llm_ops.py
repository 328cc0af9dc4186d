"""Operator-level tests of the LLM endpoint's attention and sampling kernels (csrc/llm_attention.cu, csrc/llm.cu) through
b2s_op_llm_attn_decode / b2s_op_llm_attn_prefill / b2s_op_llm_argmax, each against a plain fp64 numpy reference.

The reference sees the operands the kernel sees: q after fp32 RoPE rounded to bf16, K and V as stored in the bf16 page
pool, gathered through the page table, and an exact softmax.

Error bar of an attention output row: |got - ref| <= 2^-7 * max|V| over the keys the row sees.  The kernels round P to
bf16 for the PV product while l is summed from the unrounded fp32 P (at most 2^-9 of max|V|), and round the output to
bf16 (2^-9 of |out| <= max|V|); scores are fp32 sums of exact bf16 products.  2^-7 is twice the sum of the two.
The cache has its own bars: appended and prefilled V rows equal their inputs bit for bit, K rows and rotated q are
within one bf16 ulp of the fp64 RoPE (plus the fp32 rounding of the two products where they cancel), and every pool
row, page, accumulator element and output row the call must not touch keeps its bits.

Input families, built in the rotated space (dims 0..63 carry needles, 64..126 noise, 127 a direction every query shares)
so that a mistake about a single key costs O(max|V|), not O(1/n):
  random   scores with a standard deviation of about 3;
  needle   per (sequence, q head) one key about 12 above the rest, at key 0, the appended row, 63 / 64 / 127 / 128 and
           the first and last block of every part of the stream partition; every q head of a group has its own;
  negative every real score <= -8, so a phantom key (a zero row past the context) would dominate;
  future   (prefill) query i scores about 30 on key i + 1.
Every pool row no sequence owns -- rows past the context, the row about to be appended, pages the table does not name --
holds a sentinel: K scoring about 32 against every query and large distinct V.  Unused page-table entries name a valid
sentinel page, so a wrong read shows up as a wrong number, not a fault."""
import math

import numpy as np
import pytest

from clearml_serving_b200 import llm as L
from tests.test_llm_attn_partition import owner, partition, segments_of

HD = 128
MAX_CTX = 4096
PPS = MAX_CTX // 64                   # page-table entries per slot
THETA = 500000.0
SCALE = 1.0 / math.sqrt(HD)
C0 = 8.0                              # every query's component along dim 127
SENT_K = 45.0                         # sentinel K along dim 127: score 45 * 8 / sqrt(128) ~ 32
BAR = 2.0 ** -7

_worst = {}                           # largest observed error / bar of each check, printed at the end of the module


def _note(what, ratio):
    _worst[what] = max(_worst.get(what, 0.0), float(ratio))


@pytest.fixture(scope="module", autouse=True)
def _report_worst_errors():
    yield
    if _worst:
        print("\nlargest observed error, as a fraction of its bar:")
        for k in sorted(_worst):
            print("  {:<40s} {:.4f}".format(k, _worst[k]))


# ------------------------------------------------------------------------------------------------ numerics
def bf16(x):
    """round to bf16 (nearest even), returned as float32 values"""
    return L.from_bf16_bits(L.to_bf16_bits(np.asarray(x, np.float32)))


def rope_tables(max_ctx=MAX_CTX, theta=THETA):
    """as llm_create builds them: fp32 inv_freq and angle, cos / sin in double rounded to fp32"""
    i = np.arange(64, dtype=np.float32)
    inv_freq = np.float32(1.0) / np.power(np.float32(theta), (2 * i) / np.float32(HD))
    ang = np.arange(max_ctx, dtype=np.float32)[:, None] * inv_freq[None, :]
    return np.cos(ang.astype(np.float64)).astype(np.float32), np.sin(ang.astype(np.float64)).astype(np.float32)


COS, SIN = rope_tables()


def rope64(x, pos):
    """rotate-half RoPE in fp64 of x [..., 128] at positions pos [...]: (value, |x1 c| + |x2 s| of each output)"""
    x = np.asarray(x, np.float64)
    c, s = COS[pos].astype(np.float64), SIN[pos].astype(np.float64)
    x1, x2 = x[..., :64], x[..., 64:]
    val = np.concatenate([x1 * c - x2 * s, x2 * c + x1 * s], -1)
    mag = np.concatenate([np.abs(x1 * c) + np.abs(x2 * s), np.abs(x2 * c) + np.abs(x1 * s)], -1)
    return val, mag


def rope32(x, pos):
    """the kernels' fp32 RoPE"""
    x = np.asarray(x, np.float32)
    c, s = COS[pos], SIN[pos]
    x1, x2 = x[..., :64], x[..., 64:]
    return np.concatenate([x1 * c - x2 * s, x2 * c + x1 * s], -1)


def unrope(y, pos):
    """inverse rotation: the fp32 input whose RoPE at pos is (about) y"""
    y = np.asarray(y, np.float64)
    c, s = COS[pos].astype(np.float64), SIN[pos].astype(np.float64)
    y1, y2 = y[..., :64], y[..., 64:]
    return np.concatenate([y1 * c + y2 * s, y2 * c - y1 * s], -1).astype(np.float32)


def assert_within_ulp(got, x, pos, what):
    """got (bf16 values) within one bf16 ulp of the fp64 RoPE of x at pos"""
    ref, mag = rope64(x, pos)
    ulp = np.exp2(np.floor(np.log2(np.maximum(np.abs(ref), 1e-30))) - 7)
    tol = ulp + 2.0 ** -22 * mag
    err = np.abs(got.astype(np.float64) - ref)
    assert np.all(err <= tol), "{}: {} elements off by more than one bf16 ulp (worst {:.3e})".format(
        what, int((err > tol).sum()), float((err - tol).max()))
    _note(what + " (ulp)", (err / tol).max() if err.size else 0.0)


def paged_attention_ref(kpool, vpool, pages, q, q_pos, heads=None):
    """fp64 attention of queries q [nq, hq, 128] at positions q_pos [nq] over keys 0 .. q_pos of ONE sequence whose
    key j lives in pool page pages[j // 64], row j % 64 (kpool / vpool [n_pages, kvh, 64, 128]).  Returns
    (out [nq, hq, 128], vmax [nq, hq]: max |V| over the keys each row sees); heads: the q heads to compute (others NaN)."""
    nq, hq, _ = q.shape
    kvh = kpool.shape[1]
    G = hq // kvh
    n = int(np.max(q_pos)) + 1
    j = np.arange(n)
    pg = np.asarray(pages)[j // 64]
    K = kpool[pg, :, j % 64, :].astype(np.float64)          # [n, kvh, 128]
    V = vpool[pg, :, j % 64, :].astype(np.float64)
    visible = j[None, :] <= np.asarray(q_pos)[:, None]      # [nq, n]
    out = np.full((nq, hq, HD), np.nan)
    vmax = np.zeros((nq, hq))
    vabs = np.maximum.accumulate(np.abs(V).max(-1), axis=0)  # [n, kvh]: max |V| over keys 0 .. j
    for hh in (range(hq) if heads is None else heads):
        kh = hh // G
        s = (q[:, hh, :].astype(np.float64) @ K[:, kh, :].T) * SCALE
        s = np.where(visible, s, -np.inf)
        s -= s.max(-1, keepdims=True)
        p = np.exp(s)
        p /= p.sum(-1, keepdims=True)
        out[:, hh, :] = p @ V[:, kh, :]
        vmax[:, hh] = vabs[np.asarray(q_pos), kh]
    return out, vmax


def assert_attention_close(got, ref, vmax, what):
    """got / ref [rows, heads, 128]: |got - ref| <= 2^-7 max|V| of each (row, head); NaN rows of ref are not checked"""
    ok = ~np.isnan(ref[..., 0])
    err = np.abs(got.astype(np.float64) - ref).max(-1)
    bar = BAR * vmax
    bad = ok & ~(err <= bar)
    assert not bad.any(), "{}: {} (row, head) pairs past the bar, e.g. row/head {} err {:.4g} bar {:.4g}".format(
        what, int(bad.sum()), tuple(int(v) for v in np.argwhere(bad)[0]), float(err[bad][0]), float(bar[bad][0]))
    _note(what.split(",")[0], (err[ok] / bar[ok]).max())


# ------------------------------------------------------------------------------------------------ inputs
def _noise(rng, shape, lo, hi, std):
    x = np.zeros(tuple(shape) + (HD,), np.float32)
    x[..., lo:hi] = rng.standard_normal(tuple(shape) + (hi - lo,), dtype=np.float32) * std
    return x


def family_vectors(rng, family, n_keys, G, kvh, q_pos, needles=None):
    """rotated-space targets of one sequence: q [nq, G * kvh, 128] for query positions q_pos, K / V [kvh, n_keys, 128].
    needles[(h, r)] = key of the needle of q head h * G + r (needle family)."""
    nq = len(q_pos)
    hq = G * kvh
    q = np.zeros((nq, hq, HD), np.float32)
    q[..., 127] = C0
    V = rng.standard_normal((kvh, n_keys, HD), dtype=np.float32)
    if family == "random":
        q += _noise(rng, (nq, hq), 0, 127, 3.0)
        K = rng.standard_normal((kvh, n_keys, HD), dtype=np.float32)
    elif family == "needle":
        q += _noise(rng, (nq, hq), 64, 127, 0.5)
        K = _noise(rng, (kvh, n_keys), 64, 127, 0.3)
        for (h, r), key in needles.items():
            q[:, h * G + r, r] += 4.0                       # dim r: this head's own needle direction
            K[h, key, r] += 34.0                            # 4 * 34 / sqrt(128) ~ 12
    elif family == "negative":
        q += _noise(rng, (nq, hq), 0, 127, 1.0)
        K = _noise(rng, (kvh, n_keys), 0, 127, 0.1)
        K[..., 127] = -rng.uniform(12.5, 20.0, (kvh, n_keys))   # scores -8.8 .. -14.1
    elif family == "future":
        d = np.asarray(q_pos) % 64
        q += _noise(rng, (nq, hq), 64, 127, 0.3)
        q[np.arange(nq), :, d] += 4.0
        K = _noise(rng, (kvh, n_keys), 64, 127, 0.3)
        K[:, np.arange(1, n_keys), (np.arange(1, n_keys) - 1) % 64] += 85.0     # key j answers query j - 1: ~30
    else:
        raise ValueError(family)
    return q, K, V


def sentinel_pools(rng, n_pages, kvh):
    """every row: K scoring ~32 against any query, V = +-(64 + distinct integer) -- bf16-exact"""
    K = np.zeros((n_pages, kvh, 64, HD), np.float32)
    K[..., 127] = SENT_K
    gid = np.arange(n_pages * kvh * 64).reshape(n_pages, kvh, 64, 1)
    sign = np.where(np.arange(HD) % 2 == 0, 1.0, -1.0).astype(np.float32)
    V = ((64 + gid % 97) * sign).astype(np.float32)
    return K, V


def page_layout(rng, n_blocks, n_slots, extra=3):
    """scrambled pages for sequences of n_blocks[b] pages in one shared pool; unused table entries name a sentinel page"""
    n_pages = int(sum(n_blocks)) + extra
    perm = rng.permutation(n_pages)
    sentinel_page = int(perm[-1])
    pages, at = [], 0
    for nb in n_blocks:
        pages.append(perm[at:at + nb].astype(np.int32))
        at += nb
    slots = rng.permutation(n_slots)[:len(n_blocks)].astype(np.int32)
    table = np.full((n_slots, PPS), sentinel_page, np.int32)
    for b, pg in enumerate(pages):
        table[slots[b], :len(pg)] = pg
    return n_pages, pages, slots, table


def interesting_keys(pos, extra=()):
    keys = {0, pos, 63, 64, 127, 128} | set(int(k) for k in extra)
    return sorted(k for k in keys if 0 <= k <= pos)


class DecodeCase(object):
    """one decode step of one layer: every sequence appends its row at position ctx[b] and attends to keys 0 .. ctx[b]"""

    def __init__(self, seed, ctx, hq, kvh, family, needle_keys=None, n_slots=None):
        rng = np.random.default_rng(seed)
        self.hq, self.kvh, self.G = hq, kvh, hq // kvh
        self.ctx = np.asarray(ctx, np.int32)
        self.n_seq = n_seq = len(ctx)
        self.pos = np.minimum(self.ctx, MAX_CTX - 1)
        nbk = [int(p) // 64 + 1 for p in self.pos]
        self.n_pages, self.pages, self.slots, self.table = page_layout(rng, nbk, n_slots or n_seq + 2)
        kp, vp = sentinel_pools(rng, self.n_pages, kvh)
        QKV = (hq + 2 * kvh) * HD
        self.ws = np.full((n_seq + 2, QKV), 7.0, np.float32)        # rows >= n_seq: must keep their value
        self.q_ref = np.zeros((n_seq, hq, HD), np.float32)
        self.k_in = np.zeros((n_seq, kvh, HD), np.float32)
        self.v_in = np.zeros((n_seq, kvh, HD), np.float32)
        for b in range(n_seq):
            pos = int(self.pos[b])
            needles = None
            if family == "needle":
                needles = {}
                for h in range(kvh):
                    ks = interesting_keys(pos, needle_keys(b, h) if needle_keys else ())
                    for r in range(self.G):
                        needles[(h, r)] = ks[(r + 3 * b + h) % len(ks)]
            q, K, V = family_vectors(rng, family, pos + 1, self.G, kvh, [pos], needles)
            x_q = unrope(q[0], pos)                                 # what the QKV projection hands over
            self.q_ref[b] = bf16(rope32(x_q, pos))
            self.k_in[b] = unrope(K[:, pos], pos)
            self.v_in[b] = V[:, pos] + rng.standard_normal((kvh, HD), dtype=np.float32) * 1e-3   # not bf16-exact
            self.ws[b, :hq * HD] = x_q.reshape(-1)
            self.ws[b, hq * HD:(hq + kvh) * HD] = self.k_in[b].reshape(-1)
            self.ws[b, (hq + kvh) * HD:] = self.v_in[b].reshape(-1)
            j = np.arange(pos)
            pg = self.pages[b][j // 64]
            kp[pg, :, j % 64, :] = bf16(K[:, :pos]).transpose(1, 0, 2)
            vp[pg, :, j % 64, :] = bf16(V[:, :pos]).transpose(1, 0, 2)
        self.kpool = L.to_bf16_bits(kp)
        self.vpool = L.to_bf16_bits(vp)

    def app_rows(self, b):
        """pool page / row of sequence b's appended row"""
        pos = int(self.pos[b])
        return int(self.pages[b][pos // 64]), pos % 64

    def expected_pools(self):
        """the pools after the step as the fp64 reference computes them (appended K = bf16 of the fp64 RoPE)"""
        kp, vp = L.from_bf16_bits(self.kpool).copy(), L.from_bf16_bits(self.vpool).copy()
        for b in range(self.n_seq):
            page, row = self.app_rows(b)
            kp[page, :, row, :] = bf16(rope64(self.k_in[b], int(self.pos[b]))[0])
            vp[page, :, row, :] = bf16(self.v_in[b])
        return kp, vp

    def reference(self):
        kp, vp = self.expected_pools()
        out = np.zeros((self.n_seq, self.hq, HD))
        vmax = np.zeros((self.n_seq, self.hq))
        for b in range(self.n_seq):
            o, vm = paged_attention_ref(kp, vp, self.table[self.slots[b]], self.q_ref[b][None], [int(self.pos[b])])
            out[b], vmax[b] = o[0], vm[0]
        return out, vmax


# ------------------------------------------------------------------------------------------------ CPU: the reference itself
@pytest.mark.parametrize("hq,kvh", [(4, 2), (7, 1), (8, 8)])
def test_paged_reference_is_dense_softmax_attention(hq, kvh):
    """the paged fp64 reference over a scrambled page table equals dense torch.softmax attention over the K / V it was
    built from, for causal prefill rows and for decode rows"""
    import torch
    rng = np.random.default_rng(hq * 10 + kvh)
    lens = [1, 64, 65, 200, 130]
    G = hq // kvh
    n_pages, pages, slots, table = page_layout(rng, [(n - 1) // 64 + 1 for n in lens], len(lens) + 3)
    kp, vp = sentinel_pools(rng, n_pages, kvh)
    dense = []
    for b, n in enumerate(lens):
        K = rng.standard_normal((kvh, n, HD)).astype(np.float32)
        V = rng.standard_normal((kvh, n, HD)).astype(np.float32)
        j = np.arange(n)
        kp[pages[b][j // 64], :, j % 64, :] = K.transpose(1, 0, 2)
        vp[pages[b][j // 64], :, j % 64, :] = V.transpose(1, 0, 2)
        dense.append((K, V))
    for b, n in enumerate(lens):
        K, V = (torch.from_numpy(a.astype(np.float64)).repeat_interleave(G, 0) for a in dense[b])   # [hq, n, 128]
        q = rng.standard_normal((n, hq, HD)) * 2
        qt = torch.from_numpy(q).transpose(0, 1)                                                      # [hq, n, 128]
        mask = torch.ones(n, n, dtype=torch.bool).tril()
        s = (qt @ K.transpose(1, 2) * SCALE).masked_fill(~mask, float("-inf"))
        want = (torch.softmax(s, -1) @ V).transpose(0, 1).numpy()
        got, vmax = paged_attention_ref(kp, vp, table[slots[b]], q, np.arange(n))
        np.testing.assert_allclose(got, want, rtol=1e-12, atol=1e-12)
        assert np.allclose(vmax[-1], np.abs(dense[b][1]).max((1, 2)).repeat(G))
        got1, _ = paged_attention_ref(kp, vp, table[slots[b]], q[-1:], [n - 1], heads=[0, hq - 1])   # one decode row
        np.testing.assert_allclose(got1[0, [0, hq - 1]], want[-1, [0, hq - 1]], rtol=1e-12, atol=1e-12)
        assert np.isnan(got1[0, 1:hq - 1]).all()


def test_rope_helpers_invert_and_match_the_tables():
    rng = np.random.default_rng(1)
    y = rng.standard_normal((5, HD)).astype(np.float32)
    pos = np.array([0, 1, 63, 700, MAX_CTX - 1])
    back, _ = rope64(unrope(y, pos), pos)
    np.testing.assert_allclose(back, y, rtol=1e-5, atol=1e-5)
    assert COS[0].min() == 1.0 and not SIN[0].any()


# ------------------------------------------------------------------------------------------------ stream partition coverage
STREAM_LENS = [1, 2000, 63, 64, 65, 127, 128, 129] + [int(x) for x in np.random.default_rng(2024).integers(1, 2001, 24)]
STREAM_SHAPES = [(32, 8), (8, 1)]                                # G = 4: two CTAs per SM; G = 8: one
STREAM_NCTA = [1, 3, 7, 64, 148, "T"]


def _stream_grid(hq, kvh, n_cta):
    return 2 * n_cta if hq // kvh <= 4 else n_cta


def _stream_n_cta(ctx, kvh, n_cta):
    if n_cta == "T":
        return partition(ctx, kvh, 1, MAX_CTX)[2]
    return n_cta


def stream_parts(ctx, hq, kvh, n_cta):
    """{(b, h): [(part, first block, last block), ...]} of the partition the kernel computes, from the CPU twin"""
    grid = _stream_grid(hq, kvh, n_cta)
    nb, prefix, T, n_eff, ranges = partition(ctx, kvh, grid, MAX_CTX)
    out = {}
    for c, rg in enumerate(ranges):
        for (b, h, j0, j1, nbb, seg0) in segments_of(rg, prefix, kvh, len(ctx)):
            part = 0 if (j0 == 0 and j1 == nbb) else c - owner(seg0, T, n_eff)
            out.setdefault((b, h), []).append((part, j0, j1 - 1))
    return out


def test_stream_cases_cover_whole_segments_and_every_split_size():
    sizes = set()
    for hq, kvh in STREAM_SHAPES:
        for n_cta in STREAM_NCTA:
            for parts in stream_parts(STREAM_LENS, hq, kvh, _stream_n_cta(STREAM_LENS, kvh, n_cta)).values():
                sizes.add(min(len(parts), 5))
    assert sizes == {1, 2, 3, 4, 5}, sizes


# ------------------------------------------------------------------------------------------------ GPU runners
def _dev(native, arr, nbytes=None):
    arr = np.ascontiguousarray(arr)
    b = native.DeviceBuffer(max(nbytes or arr.nbytes, 16))
    b.upload(arr)
    return b


class DecodeRun(object):
    """device buffers of a DecodeCase; launch() may be repeated after reset()"""

    def __init__(self, native, case, part=None):
        self.native, self.case = native, case
        c = case
        self.bufs = {
            "ws": _dev(native, c.ws), "k": _dev(native, c.kpool), "v": _dev(native, c.vpool),
            "ctx": _dev(native, c.ctx), "slots": _dev(native, c.slots), "table": _dev(native, c.table),
            "cos": _dev(native, COS), "sin": _dev(native, SIN),
            "out": _dev(native, np.full((c.n_seq + 1, c.hq * HD), 0x7fc1, np.uint16)),
        }
        self.part = part

    def reset(self):
        c = self.case
        self.bufs["ws"].upload(c.ws)
        self.bufs["k"].upload(c.kpool)
        self.bufs["v"].upload(c.vpool)

    def launch(self, stream_form, n_cta=148):
        c, d = self.case, self.bufs
        ws_part = cnt = None
        if stream_form:
            ws_part, cnt = self.part
        self.native.check(self.native.lib().b2s_op_llm_attn_decode(
            0, None, d["ws"].ptr, d["k"].ptr, d["v"].ptr, c.n_pages, d["ctx"].ptr, d["slots"].ptr, d["table"].ptr, PPS,
            d["cos"].ptr, d["sin"].ptr, MAX_CTX, d["out"].ptr, c.n_seq, c.hq, c.kvh, int(stream_form), int(n_cta),
            ws_part.ptr if ws_part else None, cnt.ptr if cnt else None))

    def out_bits(self):
        c = self.case
        return self.bufs["out"].download(np.uint16, (c.n_seq + 1) * c.hq * HD).reshape(c.n_seq + 1, c.hq, HD)

    def check(self, what):
        """every output against the fp64 reference, and everything the call must (not) have changed"""
        c, d = self.case, self.bufs
        bits = self.out_bits()
        assert (bits[c.n_seq] == 0x7fc1).all(), what + ": output row past n_seq written"
        ref, vmax = c.reference()
        assert_attention_close(L.from_bf16_bits(bits[:c.n_seq]), ref, vmax, "decode output, " + what)
        ws = d["ws"].download(np.float32, c.ws.size).reshape(c.ws.shape)
        assert not ws[:c.n_seq].any(), what + ": QKV accumulator rows not cleared"
        assert np.array_equal(ws[c.n_seq:], c.ws[c.n_seq:]), what + ": accumulator rows past n_seq changed"
        if self.part is not None:
            assert not self.part[1].download(np.int32, c.n_seq * c.kvh).any(), what + ": arrival counters not left at zero"
        kp = d["k"].download(np.uint16, c.kpool.size).reshape(c.kpool.shape)
        vp = d["v"].download(np.uint16, c.vpool.size).reshape(c.vpool.shape)
        touched = np.zeros(c.kpool.shape[:3], bool)
        for b in range(c.n_seq):
            page, row = c.app_rows(b)
            touched[page, :, row] = True
            assert np.array_equal(vp[page, :, row], L.to_bf16_bits(c.v_in[b])), what + ": appended V row of seq %d" % b
            assert_within_ulp(L.from_bf16_bits(kp[page, :, row]), c.k_in[b], int(c.pos[b]), "appended K row")
        assert np.array_equal(kp[~touched], c.kpool[~touched]), what + ": K pool rows outside the appended ones changed"
        assert np.array_equal(vp[~touched], c.vpool[~touched]), what + ": V pool rows outside the appended ones changed"
        return bits

    def free(self):
        for b in self.bufs.values():
            b.free()


def _part_buffers(native, n_cta, kvh):
    ws = _dev(native, np.full(2 * n_cta * 2 * 8 * 132, np.nan, np.float32))    # never read before written
    cnt = _dev(native, np.zeros(32 * kvh, np.int32))
    return ws, cnt


def _run_decode(native, case, stream_form, n_cta=148, what=""):
    part = _part_buffers(native, n_cta, case.kvh) if stream_form else None
    run = DecodeRun(native, case, part)
    try:
        run.launch(stream_form, n_cta)
        return run.check(what)
    finally:
        run.free()
        for b in part or ():
            b.free()


FAMILIES = ["random", "needle", "negative"]


# ------------------------------------------------------------------------------------------------ GPU: decode
gpu = pytest.mark.gpu


@gpu
@pytest.mark.parametrize("family", FAMILIES)
@pytest.mark.parametrize("stream_form", [0, 1])
@pytest.mark.parametrize("hq,kvh", [(32, 8), (16, 4)])
def test_decode_llama3_8b_shapes(gpu_native, hq, kvh, stream_form, family):
    """Llama-3-8B at TP 1 and TP 2 (G = 4): 32 sequences of 500 .. 640 cached tokens, one shared scrambled pool"""
    rng = np.random.default_rng(hq + kvh)
    ctx = [int(x) for x in rng.integers(500, 641, 32)]
    case = DecodeCase(hq * 100 + stream_form * 10 + FAMILIES.index(family), ctx, hq, kvh, family)
    _run_decode(gpu_native, case, stream_form, what="llama3 {} {} {}".format(hq, stream_form, family))


GROUP_SHAPES = [(1, 8), (2, 3), (3, 2), (4, 1), (5, 2), (7, 1), (8, 4)]     # (G, kv heads)
EDGE_CTX = [1, 2, 62, 63, 64, 65, 127, 128, 129, 700]


@gpu
@pytest.mark.parametrize("family", FAMILIES)
@pytest.mark.parametrize("stream_form", [0, 1])
@pytest.mark.parametrize("G,kvh", GROUP_SHAPES)
def test_decode_group_sizes_and_block_edges(gpu_native, G, kvh, stream_form, family):
    """every group size llm_create accepts around the G <= 4 / G > 4 switch of the stream form, contexts at block edges"""
    case = DecodeCase(G * 1000 + kvh * 10 + stream_form + 3 * FAMILIES.index(family), EDGE_CTX, G * kvh, kvh, family)
    _run_decode(gpu_native, case, stream_form, what="G{} kvh{} form{} {}".format(G, kvh, stream_form, family))


@gpu
@pytest.mark.parametrize("n_cta", STREAM_NCTA)
@pytest.mark.parametrize("hq,kvh", STREAM_SHAPES)
def test_decode_stream_partitions(gpu_native, hq, kvh, n_cta):
    """the stream form over 1 CTA .. one CTA per block: whole segments, splits of 2, 3, 4 and more parts (fast tail merge,
    arrival merge, merge_from_ws past four parts); needles on the first and last block of every part"""
    n = _stream_n_cta(STREAM_LENS, kvh, n_cta)
    parts = stream_parts(STREAM_LENS, hq, kvh, n)
    ends = {}
    for (b, h), lst in parts.items():
        ends[(b, h)] = [k for _, j0, j1 in lst for k in (64 * j0, 64 * j0 + 1, 64 * j1 + 63)]
    case = DecodeCase(7 + hq + STREAM_NCTA.index(n_cta), STREAM_LENS, hq, kvh, "needle",
                      needle_keys=lambda b, h: ends[(b, h)])
    _run_decode(gpu_native, case, 1, n_cta=n, what="stream {} {} n_cta {}".format(hq, kvh, n))


@gpu
@pytest.mark.parametrize("stream_form", [0, 1])
@pytest.mark.parametrize("family", ["needle", "random"])
def test_decode_at_the_last_position(gpu_native, stream_form, family):
    case = DecodeCase(41 + stream_form, [MAX_CTX - 1], 32, 8, family)
    _run_decode(gpu_native, case, stream_form, what="max_ctx - 1 form {} {}".format(stream_form, family))


@gpu
def test_decode_two_layers_share_the_stream_workspace(gpu_native):
    """two launches back to back (two layers: different pools and accumulators) on one part_ws / part_cnt"""
    ctx = [int(x) for x in np.random.default_rng(3).integers(1, 1500, 32)]
    cases = [DecodeCase(50 + i, ctx, 32, 8, fam) for i, fam in enumerate(("needle", "random"))]
    part = _part_buffers(gpu_native, 148, 8)
    runs = [DecodeRun(gpu_native, c, part) for c in cases]
    try:
        for r in runs:
            r.launch(1, 148)
        for i, r in enumerate(runs):
            r.check("layer {}".format(i))
    finally:
        for r in runs:
            r.free()
        for b in part:
            b.free()


@gpu
@pytest.mark.parametrize("hq,kvh", [(32, 8), (8, 1)])
def test_decode_stream_form_is_deterministic(gpu_native, hq, kvh):
    """three launches of the same inputs give the same bits: which CTA (fast path or arrival) finishes a row must not
    change it"""
    case = DecodeCase(60 + hq, STREAM_LENS, hq, kvh, "random")
    part = _part_buffers(gpu_native, 148, kvh)
    run = DecodeRun(gpu_native, case, part)
    try:
        first = None
        for i in range(3):
            run.reset()
            run.launch(1, 148)
            bits = run.check("repeat {}".format(i)) if i == 0 else run.out_bits()
            assert first is None or np.array_equal(bits, first), "launch {} differs from the first".format(i)
            first = bits
    finally:
        run.free()
        for b in part:
            b.free()


@gpu
def test_decode_per_sequence_form_is_batch_invariant(gpu_native):
    """stream_form 0: a sequence alone gives the bits it gets in a batch"""
    case = DecodeCase(70, EDGE_CTX, 16, 4, "random")
    batch = _run_decode(gpu_native, case, 0, what="batch")
    for b in (0, 5, 9):
        one = DecodeCase.__new__(DecodeCase)
        one.__dict__.update(case.__dict__)
        one.n_seq = 1
        for k in ("ctx", "pos", "slots", "q_ref", "k_in", "v_in"):
            setattr(one, k, getattr(case, k)[b:b + 1])
        one.pages = case.pages[b:b + 1]
        one.ws = np.concatenate([case.ws[b:b + 1], case.ws[case.n_seq:]])
        bits = _run_decode(gpu_native, one, 0, what="alone {}".format(b))
        assert np.array_equal(bits[0], batch[b]), "sequence {} alone differs from its batch row".format(b)


# ------------------------------------------------------------------------------------------------ prefill
class PrefillCase(object):
    def __init__(self, seed, lens, hq, kvh, family):
        rng = np.random.default_rng(seed)
        self.lens, self.hq, self.kvh, self.G = list(lens), hq, kvh, hq // kvh
        self.n_seq = len(lens)
        self.cu = np.concatenate([[0], np.cumsum(lens)]).astype(np.int32)
        self.T = T = int(self.cu[-1])
        self.tok_seq = np.repeat(np.arange(self.n_seq), lens).astype(np.int32)
        self.tok_pos = np.concatenate([np.arange(n) for n in lens]).astype(np.int32)
        self.n_pages, self.pages, self.slots, self.table = page_layout(rng, [(n - 1) // 64 + 1 for n in lens], self.n_seq + 2)
        kp, vp = sentinel_pools(rng, self.n_pages, kvh)
        self.kpool, self.vpool = L.to_bf16_bits(kp), L.to_bf16_bits(vp)
        QKV = (hq + 2 * kvh) * HD
        qkv = np.zeros((T, QKV), np.float32)
        for b, n in enumerate(lens):
            pos = np.arange(n)
            needles = None
            if family == "needle":
                ks = interesting_keys(n - 1, (n // 2, n - 2))
                needles = {(h, r): ks[(r + 3 * b + h) % len(ks)] for h in range(kvh) for r in range(self.G)}
            q, K, V = family_vectors(rng, family, n, self.G, kvh, pos, needles)
            s = slice(int(self.cu[b]), int(self.cu[b + 1]))
            qkv[s, :hq * HD] = unrope(q, pos[:, None]).reshape(n, -1)
            qkv[s, hq * HD:(hq + kvh) * HD] = unrope(K.transpose(1, 0, 2), pos[:, None]).reshape(n, -1)
            qkv[s, (hq + kvh) * HD:] = V.transpose(1, 0, 2).reshape(n, -1)
        self.qkv = L.to_bf16_bits(qkv)             # the QKV projection's bf16 output
        self.x = L.from_bf16_bits(self.qkv).reshape(T, hq + 2 * kvh, HD)

    def expected(self):
        """rotated q as the reference uses it (fp32 RoPE, bf16) and the pools after the call (fp64 RoPE, bf16)"""
        hq, kvh = self.hq, self.kvh
        q = bf16(rope32(self.x[:, :hq], self.tok_pos[:, None]))
        kp, vp = L.from_bf16_bits(self.kpool).copy(), L.from_bf16_bits(self.vpool).copy()
        k = bf16(rope64(self.x[:, hq:hq + kvh], self.tok_pos[:, None])[0])
        for t in range(self.T):
            b, p = int(self.tok_seq[t]), int(self.tok_pos[t])
            page = int(self.pages[b][p // 64])
            kp[page, :, p % 64] = k[t]
            vp[page, :, p % 64] = self.x[t, hq + kvh:]
        return q, kp, vp


def _run_prefill(native, case, heads_sample=None):
    c = case
    d = {"qkv": _dev(native, c.qkv), "k": _dev(native, c.kpool), "v": _dev(native, c.vpool), "cu": _dev(native, c.cu),
         "seq": _dev(native, c.tok_seq), "pos": _dev(native, c.tok_pos), "slots": _dev(native, c.slots),
         "table": _dev(native, c.table), "cos": _dev(native, COS), "sin": _dev(native, SIN),
         "out": _dev(native, np.full((c.T + 1, c.hq * HD), 0x7fc1, np.uint16))}
    try:
        native.check(native.lib().b2s_op_llm_attn_prefill(
            0, None, d["qkv"].ptr, d["k"].ptr, d["v"].ptr, d["cu"].ptr, d["seq"].ptr, d["pos"].ptr, d["slots"].ptr,
            d["table"].ptr, PPS, d["cos"].ptr, d["sin"].ptr, MAX_CTX, d["out"].ptr, c.n_seq, max(c.lens), c.hq, c.kvh))
        out = d["out"].download(np.uint16, (c.T + 1) * c.hq * HD).reshape(c.T + 1, c.hq, HD)
        qkv = d["qkv"].download(np.uint16, c.qkv.size).reshape(c.T, -1, HD)
        kp = d["k"].download(np.uint16, c.kpool.size).reshape(c.kpool.shape)
        vp = d["v"].download(np.uint16, c.vpool.size).reshape(c.vpool.shape)
    finally:
        for b in d.values():
            b.free()
    hq, kvh = c.hq, c.kvh
    assert (out[c.T] == 0x7fc1).all(), "output row past the last token written"
    # q rotated in place (one ulp of the fp64 RoPE); the k / v columns of qkv are read only
    assert_within_ulp(L.from_bf16_bits(qkv[:, :hq]), c.x[:, :hq], c.tok_pos[:, None], "prefill rotated q")
    assert np.array_equal(qkv[:, hq:], c.qkv.reshape(c.T, -1, HD)[:, hq:])
    # cache: written rows (V exact, K one ulp), every other row untouched
    touched = np.zeros(c.kpool.shape[:3], bool)
    for t in range(c.T):
        b, p = int(c.tok_seq[t]), int(c.tok_pos[t])
        page = int(c.pages[b][p // 64])
        touched[page, :, p % 64] = True
        assert np.array_equal(vp[page, :, p % 64], c.qkv.reshape(c.T, -1, HD)[t, hq + kvh:]), "prefilled V row, token %d" % t
    rows = np.argwhere(touched)
    tok_of = {}
    for t in range(c.T):
        b, p = int(c.tok_seq[t]), int(c.tok_pos[t])
        tok_of[(int(c.pages[b][p // 64]), p % 64)] = t
    ts = np.array([tok_of[(int(pg), int(r))] for pg, _, r in rows])
    assert_within_ulp(L.from_bf16_bits(kp[rows[:, 0], rows[:, 1], rows[:, 2]]),
                      c.x[ts, hq + rows[:, 1]], c.tok_pos[ts], "prefilled K row")
    assert np.array_equal(kp[~touched], c.kpool[~touched]) and np.array_equal(vp[~touched], c.vpool[~touched]), \
        "pool rows no token writes changed"
    # attention against the fp64 reference over the expected cache
    q, kpe, vpe = c.expected()
    got = L.from_bf16_bits(out[:c.T])
    for b, n in enumerate(c.lens):
        s = slice(int(c.cu[b]), int(c.cu[b + 1]))
        heads = None if heads_sample is None else heads_sample(b)
        ref, vmax = paged_attention_ref(kpe, vpe, c.table[c.slots[b]], q[s], np.arange(n), heads)
        assert_attention_close(got[s], ref, vmax, "prefill output")
    return kp, vp


PREFILL_LENS = [[1], [1, 2, 63, 64, 65], [127, 128, 129, 300], [1000, 5]]
PREFILL_SHAPES = [(4, 2), (32, 8), (8, 1), (7, 1)]


@gpu
@pytest.mark.parametrize("family", FAMILIES + ["future"])
@pytest.mark.parametrize("hq,kvh", PREFILL_SHAPES)
@pytest.mark.parametrize("lens", PREFILL_LENS, ids=["1", "1-65", "127-300", "1000-5"])
def test_prefill_matches_fp64_reference(gpu_native, lens, hq, kvh, family):
    case = PrefillCase(sum(lens) + hq * 7 + kvh + len(family), lens, hq, kvh, family)
    sample = None
    if hq * sum(n * n for n in lens) > 4e6:         # Llama-3-8B heads over 1000 tokens: a sample of (sequence, head) pairs
        rng = np.random.default_rng(hq)
        sample = lambda b: sorted({0, hq - 1} | set(int(h) for h in rng.choice(hq, 3, replace=False)))
    _run_prefill(gpu_native, case, sample)


@gpu
@pytest.mark.parametrize("stream_form", [0, 1])
def test_prefill_then_decode_matches_the_whole_sequence(gpu_native, stream_form):
    """the prefill op writes the cache, the decode op appends the next token and attends over all of it: the result is the
    fp64 attention of the extended sequence"""
    native = gpu_native
    hq, kvh = 32, 8
    lens = [130, 1, 64, 700, 63]
    pre = PrefillCase(80 + stream_form, lens, hq, kvh, "random")
    kp, vp = _run_prefill(native, pre, lambda b: [0, 5, 31])        # the cache as the prefill kernels wrote it
    # the decode step: sequence b at position lens[b] (its pages were laid out for lens[b] tokens: give it one more if needed)
    rng = np.random.default_rng(90)
    dec = DecodeCase.__new__(DecodeCase)
    dec.hq, dec.kvh, dec.G, dec.n_seq = hq, kvh, hq // kvh, len(lens)
    dec.ctx = np.array(lens, np.int32)
    dec.pos = dec.ctx.copy()
    table, pages = pre.table.copy(), [p.copy() for p in pre.pages]
    spare = list(range(pre.n_pages, pre.n_pages + len(lens)))
    extra_k, extra_v = sentinel_pools(rng, len(lens), kvh)
    kp = np.concatenate([kp, L.to_bf16_bits(extra_k)])
    vp = np.concatenate([vp, L.to_bf16_bits(extra_v)])
    for b, n in enumerate(lens):
        if n // 64 >= len(pages[b]):
            pages[b] = np.append(pages[b], spare[b]).astype(np.int32)
            table[pre.slots[b], n // 64] = spare[b]
    dec.n_pages, dec.pages, dec.slots, dec.table = pre.n_pages + len(lens), pages, pre.slots, table
    dec.kpool, dec.vpool = kp, vp
    QKV = (hq + 2 * kvh) * HD
    dec.ws = np.full((len(lens) + 2, QKV), 7.0, np.float32)
    x = rng.standard_normal((len(lens), QKV), dtype=np.float32)
    x[:, :hq * HD] *= 3
    dec.ws[:len(lens)] = x
    dec.q_ref = bf16(rope32(x[:, :hq * HD].reshape(-1, hq, HD), dec.pos[:, None]))
    dec.k_in = x[:, hq * HD:(hq + kvh) * HD].reshape(-1, kvh, HD)
    dec.v_in = x[:, (hq + kvh) * HD:].reshape(-1, kvh, HD)
    _run_decode(native, dec, stream_form, what="after prefill form {}".format(stream_form))


# ------------------------------------------------------------------------------------------------ argmax
def _argmax_row(rng, pattern, V, n_split):
    chunk = -(-V // n_split)
    x = rng.standard_normal(V).astype(np.float32)
    if pattern == 0:
        pass
    elif pattern == 1:
        x[0] = x.max() + 1
    elif pattern == 2:
        x[V - 1] = x.max() + 1
    elif pattern == 3:                              # equal maxima in one thread's strip (stride 256)
        i = min(5, V - 1)
        x[i] = x[min(i + 256, V - 1)] = x.max() + 1
    elif pattern == 4:                              # equal maxima on different threads, higher index on the lower thread
        x[[min(255, V - 1), min(257, V - 1)]] = x.max() + 1
    elif pattern == 5:                              # equal maxima across CTA chunks
        x[[min(chunk - 1, V - 1), min(chunk, V - 1), V - 1]] = x.max() + 1
    elif pattern == 6:                              # all negative
        x = -np.abs(x) - 1
    elif pattern == 7:                              # -inf entries, whole chunks of them
        x[rng.random(V) < 0.5] = -np.inf
        x[:min(chunk, V)] = -np.inf
    elif pattern == 8:                              # -0.0 before +0.0, in another chunk and in the same one
        x = -np.abs(x) - 1
        x[min(chunk - 1, V - 2)] = -0.0
        x[min(chunk, V - 1)] = 0.0
        x[V - 1] = 0.0
    elif pattern == 9:                              # nothing but -inf
        x[:] = -np.inf
    elif pattern == 10:                             # a constant row
        x[:] = 0.25
    elif pattern == 11:                             # -0.0 wins against earlier negatives, +0.0 later in the same chunk
        x = -np.abs(x) - 1
        x[V // 3] = -0.0
        x[V // 3 + 1] = 0.0
    return x


N_PATTERNS = 12


@gpu
@pytest.mark.parametrize("n_seq", [1, 32])
@pytest.mark.parametrize("n_split", [1, 7, 32, 64])
@pytest.mark.parametrize("vocab", [1000, 1024, 64128, 128256])
def test_argmax_is_the_first_maximum(gpu_native, vocab, n_split, n_seq):
    native = gpu_native
    rng = np.random.default_rng(vocab + n_split + n_seq)
    first = (vocab // 7 + n_split) % N_PATTERNS
    x = np.stack([_argmax_row(rng, (first + b) % N_PATTERNS, vocab, n_split) for b in range(n_seq)])
    d = {"x": _dev(native, x), "keep": _dev(native, np.full_like(x, np.nan)), "key": _dev(native, np.zeros(n_seq, np.uint64)),
         "cnt": _dev(native, np.zeros(n_seq, np.int32)), "tok": _dev(native, np.full(n_seq, -1, np.int32))}
    try:
        native.check(native.lib().b2s_op_llm_argmax(0, None, d["x"].ptr, d["keep"].ptr, n_seq, vocab, n_split,
                                                    d["key"].ptr, d["cnt"].ptr, d["tok"].ptr))
        tok = d["tok"].download(np.int32, n_seq)
        assert np.array_equal(tok, np.argmax(x, axis=1)), (tok, np.argmax(x, axis=1))
        assert not d["x"].download(np.float32, x.size).view(np.uint32).any(), "logits not cleared"
        assert np.array_equal(d["keep"].download(np.float32, x.size).view(np.uint32), x.reshape(-1).view(np.uint32))
        assert not d["key"].download(np.uint64, n_seq).any() and not d["cnt"].download(np.int32, n_seq).any()
    finally:
        for b in d.values():
            b.free()
