"""Operator-level GPU tests (-m gpu) for the DL building blocks, through the C ABI (b2s_op_*), each
against a plain fp32 reference of the same op (numpy / torch CPU).  Floating point: tolerance stated
per test (fp16 inputs, fp32 accumulation, fp16 or fp32 output)."""
import ctypes

import numpy as np
import pytest

from clearml_serving_b200 import llm as L

pytestmark = pytest.mark.gpu


def _gemm(native, A, B, bias=None, residual=None, act=0, out_f32=False, bf16=False):
    """A, B: fp16 arrays, or bf16 bit patterns (uint16) with bf16=True; returns C as float32 (fp32 or 16-bit output)"""
    M, K = A.shape
    N = B.shape[0]
    n_out = N // 2 if act == 4 else N          # SwiGLU: C is [M, N / 2]
    dA, dB = native.DeviceBuffer(A.nbytes), native.DeviceBuffer(B.nbytes)
    dC = native.DeviceBuffer(M * n_out * (4 if out_f32 else 2))
    dA.upload(A); dB.upload(B)
    dbias = dres = None
    if bias is not None:
        dbias = native.DeviceBuffer(bias.nbytes); dbias.upload(bias)
    if residual is not None:
        dres = native.DeviceBuffer(residual.nbytes); dres.upload(residual)
    try:
        native.check(native.lib().b2s_op_gemm(0, None, dA.ptr, dB.ptr, dC.ptr, M, N, K,
                                              dbias.ptr if dbias else None, dres.ptr if dres else None,
                                              act, 1 if bf16 else 0, 1 if out_f32 else 0))
        if out_f32:
            return dC.download(np.float32, M * n_out).reshape(M, n_out)
        if bf16:
            return L.from_bf16_bits(dC.download(np.uint16, M * n_out)).reshape(M, n_out)
        return dC.download(np.float16, M * n_out).reshape(M, n_out).astype(np.float32)
    finally:
        for b in (dA, dB, dC, dbias, dres):
            if b is not None:
                b.free()


def _operand(rng, shape, std, dtype):
    """random 16-bit GEMM operand: (what the kernel reads, its values as float32)"""
    if dtype == "bf16":
        bits = L.to_bf16_bits(rng.standard_normal(shape, dtype=np.float32) * np.float32(std))
        return bits, L.from_bf16_bits(bits)
    h = (rng.standard_normal(shape) * std).astype(np.float16)
    return h, h.astype(np.float32)


def _ref_act(x, act):
    if act == 1:
        from scipy.special import erf
        return 0.5 * x * (1.0 + erf(x / np.sqrt(2.0)))
    if act == 2:
        return np.maximum(x, 0)
    if act == 3:
        return np.tanh(x)
    return x


GEMM_SHAPES = [(128, 128, 64), (128, 128, 768), (256, 768, 768), (300, 2304, 768),
               (1000, 3072, 768), (77, 768, 3072), (5, 2, 768), (130, 200, 72), (260, 520, 136),
               (4000, 256, 64), (20000, 768, 768),
               # narrow, deep shapes (BERT FFN-down class): many k-blocks per tile, partly filled last wave
               (7424, 768, 3072), (2000, 1024, 4096), (640, 512, 8192),
               # 2-SM (cta_group::2) kernel: odd number of 128-row tiles (the last pair's second CTA is all
               # padding), last 256-column tile partial
               (4990, 1000, 2048),
               # 256 x 192 pair-tiles (fp32 output, width a multiple of 192)
               (4990, 960, 2048),
               # LLM prefill projections (bf16): Llama-3-8B QKV at TP 1 and O, a ragged wave, a narrow one
               (2048, 6144, 4096), (2000, 4096, 4096), (777, 1536, 512)]


@pytest.mark.parametrize("M,N,K,dtype", [pytest.param(M, N, K, dt, id="{}-{}-{}{}".format(M, N, K, "" if dt == "fp16" else "-bf16"))
                                         for dt in ("fp16", "bf16") for M, N, K in GEMM_SHAPES])
def test_gemm_fp16_matches_fp32_reference(gpu_native, M, N, K, dtype):
    rng = np.random.default_rng(M * 7 + N)
    A, A32 = _operand(rng, (M, K), 0.5, dtype)
    B, B32 = _operand(rng, (N, K), 0.05, dtype)
    bf = dtype == "bf16"
    ref = A32 @ B32.T
    got = _gemm(gpu_native, A, B, out_f32=True, bf16=bf)
    # fp32 accumulation of exact 16-bit products: only the summation order differs
    np.testing.assert_allclose(got, ref, rtol=1e-4, atol=1e-4 * np.abs(ref).max())
    got16 = _gemm(gpu_native, A, B, bf16=bf)
    tol = 8e-3 if bf else 2e-3                 # output rounding: 2^-9 (bf16) / 2^-11 (fp16) relative
    np.testing.assert_allclose(got16, ref, rtol=tol, atol=tol * np.abs(ref).max())


@pytest.mark.parametrize("M,N,dtype", [(M, N, "bf16") for N in (128, 192, 2048, 28672) for M in (1, 77, 300, 4096)]
                         + [(300, 2048, "fp16")])
def test_gemm_swiglu_epilogue(gpu_native, M, N, dtype):
    """act 4, the prefill gate/up projection: fused columns [64j, 64j+32) are gate, [64j+32, 64j+64) up, C[M, N/2] =
    silu(gate) * up.  Products above ~1e11 FLOP are checked on the first and last row of every 128-row tile plus
    random rows."""
    K = 4096 if N == 28672 else 512            # Llama-3-8B gate/up at TP 1: N = 2 * 14336, K = 4096
    rng = np.random.default_rng(M + N)
    A, A32 = _operand(rng, (M, K), 0.5, dtype)
    B, B32 = _operand(rng, (N, K), 0.05, dtype)
    got = _gemm(gpu_native, A, B, act=4, bf16=dtype == "bf16")
    assert got.shape == (M, N // 2)
    rows = np.arange(M)
    if 2.0 * M * N * K > 1e11:
        tiles = np.arange(0, M, 128)
        rows = np.unique(np.concatenate([tiles, np.minimum(tiles + 127, M - 1), rng.integers(0, M, 64)]))
    acc = (A32[rows] @ B32.T).astype(np.float64).reshape(len(rows), N // 64, 2, 32)
    gate, up = acc[:, :, 0, :], acc[:, :, 1, :]
    ref = (gate / (1.0 + np.exp(-gate)) * up).reshape(len(rows), N // 2)
    tol = 8e-3 if dtype == "bf16" else 2e-3
    np.testing.assert_allclose(got[rows], ref, rtol=tol, atol=tol * np.abs(ref).max())


@pytest.mark.parametrize("act", [0, 1, 2, 3])
def test_gemm_fused_epilogue(gpu_native, act):
    rng = np.random.default_rng(act)
    M, N, K = 200, 768, 768
    A = (rng.standard_normal((M, K)) * 0.5).astype(np.float16)
    B = (rng.standard_normal((N, K)) * 0.05).astype(np.float16)
    bias = rng.standard_normal(N).astype(np.float32)
    res = rng.standard_normal((M, N)).astype(np.float16)
    ref = _ref_act(A.astype(np.float32) @ B.astype(np.float32).T + bias, act) + res.astype(np.float32)
    got = _gemm(gpu_native, A, B, bias=bias, residual=res, act=act).astype(np.float32)
    np.testing.assert_allclose(got, ref, rtol=2e-3, atol=2e-3 * np.abs(ref).max())


def test_gemm_fp32_residual_stream_is_batch_invariant(gpu_native):
    """BERT's FFN-down shape (fp32 output + fp32 residual + bias): repeated launches are bit-identical and a row's
    result does not depend on the batch it is computed in (SURVEY.md 5.9 rule 4) -- the tile shape may change with M,
    the order in which a row's k-blocks are summed may not"""
    rng = np.random.default_rng(11)
    M, N, K = 7424, 768, 3072
    A = (rng.standard_normal((M, K)) * 0.5).astype(np.float16)
    B = (rng.standard_normal((N, K)) * 0.05).astype(np.float16)
    bias = rng.standard_normal(N).astype(np.float32)
    res = rng.standard_normal((M, N)).astype(np.float32)
    ref = A.astype(np.float32) @ B.astype(np.float32).T + bias + res
    first = None
    for _ in range(3):
        got = _gemm(gpu_native, A, B, bias=bias, residual=res, out_f32=True)
        np.testing.assert_allclose(got, ref, rtol=1e-4, atol=1e-4 * np.abs(ref).max())
        assert first is None or np.array_equal(got, first)
        first = got
    sub = _gemm(gpu_native, A[1000:1300], B, bias=bias, residual=res[1000:1300], out_f32=True)   # another batch composition
    assert np.array_equal(sub, first[1000:1300])


# ---------------------------------------------------------------- implicit-GEMM convolution
def _conv(native, x, w, bias, stride, pad, residual=None, act=0, act_after=0):
    n, H, W, C = x.shape
    Cout, KS = w.shape[0], w.shape[1]
    OH, OW = (H + 2 * pad - KS) // stride + 1, (W + 2 * pad - KS) // stride + 1
    bufs = [native.DeviceBuffer(a.nbytes) for a in (x, w, bias)]
    for b, a in zip(bufs, (x, w, bias)):
        b.upload(a)
    dy = native.DeviceBuffer(n * OH * OW * Cout * 2)
    dres = None
    if residual is not None:
        dres = native.DeviceBuffer(residual.nbytes); dres.upload(residual)
    try:
        native.check(native.lib().b2s_op_conv(0, None, bufs[0].ptr, n, H, W, C, bufs[1].ptr, Cout, KS, stride, pad,
                                              bufs[2].ptr, dres.ptr if dres else None, dy.ptr, act, act_after))
        return dy.download(np.float16, n * OH * OW * Cout).reshape(n, OH, OW, Cout)
    finally:
        for b in bufs + [dy, dres]:
            if b is not None:
                b.free()


@pytest.mark.parametrize("n,H,W,C,Cout,KS,stride,pad", [
    (2, 56, 56, 64, 64, 3, 1, 1),      # ResNet-50 layer1 conv2 (N = 64 tiles)
    (3, 28, 28, 128, 128, 3, 1, 1),    # layer2 conv2
    (2, 56, 56, 128, 128, 3, 2, 1),    # layer2.0 conv2: stride 2
    (5, 14, 14, 256, 256, 3, 1, 1),    # layer3 conv2: tiles straddle image rows and images
    (9, 7, 7, 512, 512, 3, 1, 1),      # layer4 conv2: 49-pixel images, 128-pixel tiles span 3 images
    (2, 56, 56, 256, 512, 1, 2, 0),    # layer2.0 downsample: 1x1 stride 2
    (1, 7, 7, 64, 64, 3, 1, 1),        # one small image: tensor < 128 KiB (descriptor workaround path)
    (4, 2, 2, 64, 128, 3, 1, 1),       # resnet18 on 64x64 images, layer4: the filter is larger than the image
    (2, 9, 11, 64, 72, 3, 2, 1),       # odd sizes, Cout not a multiple of the tile
    (40, 14, 14, 256, 1024, 1, 2, 0),  # wide output: 128 x 256 tiles / CTA pairs
    (64, 7, 7, 512, 512, 3, 1, 1),     # layer4 conv2 at batch 64: 26 pair-tiles x 72 k-blocks
])
def test_conv_implicit_gemm_matches_torch_fp32(gpu_native, n, H, W, C, Cout, KS, stride, pad):
    """the fp32 reference of the same op: torch conv2d on the fp16-rounded operands"""
    import torch
    rng = np.random.default_rng(H * 131 + C + KS)
    x = (rng.standard_normal((n, H, W, C)) * 0.5).astype(np.float16)
    w = (rng.standard_normal((Cout, KS, KS, C)) * (0.5 / np.sqrt(KS * KS * C))).astype(np.float16)
    bias = rng.standard_normal(Cout).astype(np.float32) * 0.1
    ref = torch.nn.functional.conv2d(torch.from_numpy(x.astype(np.float32)).permute(0, 3, 1, 2),
                                     torch.from_numpy(w.astype(np.float32)).permute(0, 3, 1, 2),
                                     torch.from_numpy(bias), stride=stride, padding=pad).permute(0, 2, 3, 1).numpy()
    got = _conv(gpu_native, x, w, bias, stride, pad).astype(np.float32)
    assert got.shape == ref.shape
    np.testing.assert_allclose(got, ref, rtol=2e-3, atol=2e-3 * np.abs(ref).max())
    # fused ResNet tail: relu(conv + bias + identity)
    res = rng.standard_normal(ref.shape).astype(np.float16)
    got2 = _conv(gpu_native, x, w, bias, stride, pad, residual=res, act=2, act_after=1).astype(np.float32)
    ref2 = np.maximum(ref + res.astype(np.float32), 0)
    np.testing.assert_allclose(got2, ref2, rtol=2e-3, atol=2e-3 * np.abs(ref2).max())


@pytest.mark.parametrize("n,C,H,W,Cout,dtype", [
    (2, 3, 224, 224, 64, np.float32),    # ResNet stem: 112-pixel output rows, one row per tile
    (3, 3, 64, 64, 64, np.float32),      # 32-pixel rows, four rows per tile
    (2, 3, 112, 96, 64, np.uint8),       # two 48-pixel rows per tile (96 of 128 rows live), uint8 pixels
    (1, 3, 50, 38, 128, np.float32),     # odd output size (25 x 19), N = 128 tiles
    (5, 1, 30, 30, 8, np.float32),       # one channel, 15-pixel rows (5 rows per tile), narrow output
])
def test_conv_stem_space_to_depth_matches_torch_fp32(gpu_native, n, C, H, W, Cout, dtype):
    """7x7 stride-2 pad-3 stem straight from NCHW request pixels; reference: torch conv2d on the fp16-rounded operands"""
    import torch
    from clearml_serving_b200 import formats
    native = gpu_native
    rng = np.random.default_rng(H * 7 + W + Cout)
    if dtype == np.uint8:
        x = rng.integers(0, 256, (n, C, H, W)).astype(np.uint8)
    else:
        x = (rng.standard_normal((n, C, H, W)) * 0.5).astype(np.float32)
    w = (rng.standard_normal((Cout, C, 7, 7)) * (0.5 / np.sqrt(49 * C))).astype(np.float16)
    bias = rng.standard_normal(Cout).astype(np.float32) * 0.1
    x16 = x.astype(np.float16).astype(np.float32)
    ref = torch.nn.functional.conv2d(torch.from_numpy(x16), torch.from_numpy(w.astype(np.float32)), torch.from_numpy(bias),
                                     stride=2, padding=3).relu().permute(0, 2, 3, 1).numpy()
    OH, OW = (H - 1) // 2 + 1, (W - 1) // 2 + 1
    w2 = formats.stem_s2d_weight(w.astype(np.float64)).astype(np.float16)
    dx, dw, db = _dev(native, x), _dev(native, w2), _dev(native, bias)
    dz = native.DeviceBuffer(n * (OH + 3) * (OW + 3) * 32)
    dy = native.DeviceBuffer(n * OH * OW * Cout * 2)
    try:
        native.check(native.lib().b2s_op_conv_stem(0, None, dx.ptr, 4 if dtype == np.uint8 else 0, n, C, H, W, dw.ptr, Cout,
                                                   db.ptr, dz.ptr, dy.ptr, 2))
        got = dy.download(np.float16, n * OH * OW * Cout).reshape(n, OH, OW, Cout).astype(np.float32)
    finally:
        for b in (dx, dw, db, dz, dy):
            b.free()
    assert got.shape == ref.shape
    np.testing.assert_allclose(got, ref, rtol=2e-3, atol=2e-3 * np.abs(ref).max())


# ---------------------------------------------------------------- LayerNorm / embedding / attention
def _dev(native, arr):
    b = native.DeviceBuffer(max(arr.nbytes, 16))
    b.upload(arr)
    return b


@pytest.mark.parametrize("rows,H", [(1, 768), (37, 768), (1000, 1024), (5, 256), (64, 3072)])
def test_layernorm_matches_torch(gpu_native, rows, H):
    import torch
    rng = np.random.default_rng(rows + H)
    x = (rng.standard_normal((rows, H)) * 2 + 0.3).astype(np.float32)
    gamma = rng.standard_normal(H).astype(np.float32)
    beta = rng.standard_normal(H).astype(np.float32)
    ref = torch.nn.functional.layer_norm(torch.from_numpy(x), (H,), torch.from_numpy(gamma), torch.from_numpy(beta), 1e-12).numpy()
    dx, dg, db = _dev(gpu_native, x), _dev(gpu_native, gamma), _dev(gpu_native, beta)
    d16, d32 = gpu_native.DeviceBuffer(rows * H * 2), gpu_native.DeviceBuffer(rows * H * 4)
    try:
        gpu_native.check(gpu_native.lib().b2s_op_layernorm(0, None, dx.ptr, rows, H, dg.ptr, db.ptr, 1e-12, d16.ptr, d32.ptr))
        o32 = d32.download(np.float32, rows * H).reshape(rows, H)
        o16 = d16.download(np.float16, rows * H).reshape(rows, H).astype(np.float32)
        np.testing.assert_allclose(o32, ref, rtol=1e-5, atol=1e-5)          # fp32 path: same formula as torch
        np.testing.assert_allclose(o16, ref, rtol=1e-3, atol=1e-3)          # fp16 rounding of the output
    finally:
        for b in (dx, dg, db, d16, d32):
            b.free()


def test_embedding_layernorm_matches_torch(gpu_native):
    import torch
    rng = np.random.default_rng(0)
    H, vocab, max_pos = 768, 1000, 512
    lens = [16, 1, 64, 200, 7]
    cu = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    T = int(cu[-1])
    ids = rng.integers(0, vocab, T).astype(np.int32)
    types = rng.integers(0, 2, T).astype(np.int32)
    word = (rng.standard_normal((vocab, H)) * 0.02).astype(np.float16)
    pos = (rng.standard_normal((max_pos, H)) * 0.02).astype(np.float16)
    typ = (rng.standard_normal((2, H)) * 0.02).astype(np.float16)
    gamma = (1 + 0.1 * rng.standard_normal(H)).astype(np.float32)
    beta = (0.1 * rng.standard_normal(H)).astype(np.float32)
    position = np.concatenate([np.arange(n) for n in lens])
    e = word[ids].astype(np.float32) + typ[types].astype(np.float32) + pos[position].astype(np.float32)
    ref = torch.nn.functional.layer_norm(torch.from_numpy(e), (H,), torch.from_numpy(gamma), torch.from_numpy(beta), 1e-12).numpy()
    bufs = [_dev(gpu_native, a) for a in (ids, types, cu, word, pos, typ, gamma, beta)]
    d16, d32 = gpu_native.DeviceBuffer(T * H * 2), gpu_native.DeviceBuffer(T * H * 4)
    try:
        gpu_native.check(gpu_native.lib().b2s_op_embed_layernorm(
            0, None, bufs[0].ptr, bufs[1].ptr, bufs[2].ptr, len(lens), T, H, bufs[3].ptr, bufs[4].ptr, bufs[5].ptr,
            vocab, max_pos, 2, bufs[6].ptr, bufs[7].ptr, 1e-12, d16.ptr, d32.ptr))
        o32 = d32.download(np.float32, T * H).reshape(T, H)
        np.testing.assert_allclose(o32, ref, rtol=1e-4, atol=1e-4)
        o16 = d16.download(np.float16, T * H).reshape(T, H).astype(np.float32)
        np.testing.assert_allclose(o16, ref, rtol=2e-3, atol=2e-3)
    finally:
        for b in bufs + [d16, d32]:
            b.free()


@pytest.mark.parametrize("lens,masked", [([16], False), ([64, 1, 256, 100, 33], False), ([128, 77], True), ([300, 512], False),
                                         ([384, 129, 5], True), ([257, 256, 383], False), ([1, 2, 127, 128], True)])
def test_attention_varlen_matches_torch(gpu_native, lens, masked):
    """per-sequence softmax(QK^T/8 + mask)V against torch fp32 on the fp16-rounded inputs; a request's
    output must not depend on its batch-mates (each sequence is also run alone and compared bit-wise)."""
    import torch
    heads, d = 12, 64
    H = heads * d
    rng = np.random.default_rng(len(lens) * 31 + lens[0])
    cu = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    T = int(cu[-1])
    qkv = (rng.standard_normal((T, 3 * H)) * 0.7).astype(np.float16)
    mask = np.ones(T, np.int32)
    if masked:
        mask[rng.random(T) < 0.2] = 0
        mask[cu[:-1]] = 1    # keep at least one visible key per sequence
    ref = np.zeros((T, H), np.float32)
    q32 = torch.from_numpy(qkv.astype(np.float32))
    for i, n in enumerate(lens):
        s = int(cu[i])
        blk = q32[s:s + n]
        q, k, v = [blk[:, j * H:(j + 1) * H].reshape(n, heads, d).transpose(0, 1) for j in range(3)]
        att = q @ k.transpose(1, 2) / 8.0
        att = att.masked_fill(torch.from_numpy(mask[s:s + n] == 0)[None, None, :], float("-inf"))
        ref[s:s + n] = (torch.softmax(att, -1) @ v).transpose(0, 1).reshape(n, H).numpy()
    dq, dcu, dm = _dev(gpu_native, qkv), _dev(gpu_native, cu), _dev(gpu_native, mask)
    dout = gpu_native.DeviceBuffer(T * H * 2)
    try:
        gpu_native.check(gpu_native.lib().b2s_op_attention(0, None, dq.ptr, dcu.ptr, dm.ptr if masked else None, dout.ptr,
                                                           len(lens), max(lens), heads, d, T))
        got = dout.download(np.float16, T * H).reshape(T, H)
        # fp16 P and fp16 output rounding: ~1e-3 relative to the value range of V
        np.testing.assert_allclose(got.astype(np.float32), ref, rtol=0, atol=4e-3 * np.abs(ref).max())
        # batch independence: sequence i alone gives the same bits
        for i, n in enumerate(lens[:2]):
            s = int(cu[i])
            one = _dev(gpu_native, np.ascontiguousarray(qkv[s:s + n]))
            cu1 = _dev(gpu_native, np.array([0, n], np.int64))
            m1 = _dev(gpu_native, np.ascontiguousarray(mask[s:s + n]))
            o1 = gpu_native.DeviceBuffer(n * H * 2)
            gpu_native.check(gpu_native.lib().b2s_op_attention(0, None, one.ptr, cu1.ptr, m1.ptr if masked else None, o1.ptr,
                                                               1, n, heads, d, 0))   # 0: T read back from the device
            assert np.array_equal(o1.download(np.float16, n * H).reshape(n, H), got[s:s + n])
            for b in (one, cu1, m1, o1):
                b.free()
    finally:
        for b in (dq, dcu, dm, dout):
            b.free()
