"""Per-op parity: every function of the kernel dispatch surface (reference voxtral_kernels.h) called
through the C ABI of libvoxtral_b200.so on host buffers, against the SAME function of the unmodified
reference (oracle/_ref/libvoxref.so) on the same seeded inputs, as recorded under tests/golden/reference/test_gpu_ops_parity.npz
(tests/conftest.py: `recorded`).

Tolerances: f32 elementwise ops -> a few ulp; dot-product ops (GEMV/GEMM/conv/attention/norm) -> relative
1e-5 of the output scale (the reference itself is -ffast-math + OpenBLAS, i.e. its summation order is
not canonical, SURVEY.md section 8c).
"""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
fp = C.POINTER(C.c_float)
u16p = C.POINTER(C.c_uint16)


def P(a):
    return a.ctypes.data_as(fp)


def bf16_weights(rng, n, k, scale):
    w = (rng.uniform(-1, 1, size=(n, k)) * scale).astype(np.float32)
    u = w.view(np.uint32)
    u = ((u + 0x7FFF + ((u >> 16) & 1)) >> 16).astype(np.uint16)          # RNE to bf16
    return np.ascontiguousarray(u)


def close(a, want, rtol):
    """`want`: the reference's output of the same call (tests/conftest.py: Recorded)."""
    scale = max(want.scale, 1e-6)
    err = want.max_abs_diff(a)
    assert err <= rtol * scale, f"max err {err:.3e} vs scale {scale:.3e} (rel {err / scale:.2e} > {rtol})"


@pytest.mark.parametrize("op", ["silu", "gelu"])
def test_activations(vb, ref, recorded, op):
    rng = np.random.default_rng(1)
    x = rng.normal(0, 3, size=5000).astype(np.float32)
    a = x.copy()
    getattr(vb.lib(), "vox_" + op)(P(a), a.size)

    def run_ref(b=x.copy()):
        getattr(ref.L, "vox_" + op)(P(b), b.size)
        return b
    close(a, recorded("out", run_ref), 2e-6)


def test_elementwise(vb, ref, recorded):
    rng = np.random.default_rng(2)
    x = rng.normal(size=4097).astype(np.float32)
    y = rng.normal(size=4097).astype(np.float32)

    def run_ref(name, *args):
        b = x.copy()
        getattr(ref.L, name)(P(b), *args, b.size)
        return b
    for name in ("vox_add_inplace", "vox_mul_inplace"):
        a = x.copy()
        getattr(vb.lib(), name)(P(a), P(y), a.size)
        b = recorded(name, lambda: run_ref(name, P(y)))
        assert np.array_equal(b.take(a), b.values), name
    a = x.copy()
    vb.lib().vox_axpy(P(a), 0.37, P(y), a.size)
    close(a, recorded("vox_axpy", lambda: run_ref("vox_axpy", 0.37, P(y))), 1e-6)
    a = x.copy()
    vb.lib().vox_scale(P(a), 1.7, a.size)
    b = recorded("vox_scale", lambda: run_ref("vox_scale", 1.7))
    assert np.array_equal(b.take(a), b.values)


@pytest.mark.parametrize("rows,hidden", [(1, 3072), (7, 1280), (3, 96)])
def test_rms_norm(vb, ref, recorded, rows, hidden):
    rng = np.random.default_rng(3)
    x = rng.normal(size=(rows, hidden)).astype(np.float32)
    w = rng.uniform(0.9, 1.1, size=hidden).astype(np.float32)
    a = np.empty_like(x)
    vb.lib().vox_rms_norm(P(a), P(x), P(w), rows, hidden, 1e-5)

    def run_ref(b=np.empty_like(x)):
        ref.L.vox_rms_norm(P(b), P(x), P(w), rows, hidden, 1e-5)
        return b
    close(a, recorded("out", run_ref), 2e-6)


# (M, K, N): decode GEMV shapes, prefill/encoder GEMM shapes, ragged sizes
@pytest.mark.parametrize("M,K,N,bias", [
    (1, 3072, 4096, False), (1, 3072, 1024, False), (1, 4096, 3072, False), (1, 9216, 3072, False),
    (1, 3072, 9216, False), (1, 1280, 2048, True), (1, 5120, 1280, True),
    (38, 3072, 1024, False), (5, 1280, 2048, True), (130, 2048, 1280, True), (3, 384, 70, True),
    # 2 <= M < 8: the live-stream encoder calls go through the multi-row streaming GEMV (vb_gemv_cols_dev)
    (2, 3072, 3072, False), (6, 2048, 1280, True), (7, 5120, 1280, True), (4, 3840, 1280, True), (8, 1280, 6144, True),
])
def test_linear_bf16(vb, ref, recorded, M, K, N, bias):
    rng = np.random.default_rng(4 + M + K + N)
    x = rng.normal(size=(M, K)).astype(np.float32)
    W = bf16_weights(rng, N, K, np.sqrt(3.0 / K))
    b = rng.normal(size=N).astype(np.float32) * 0.1 if bias else None
    ya, yb = np.empty((M, N), np.float32), np.empty((M, N), np.float32)
    bp = P(b) if bias else None
    vb.lib().vox_linear_bf16(P(ya), P(x), W.ctypes.data_as(u16p), bp, M, K, N)

    def run_ref():
        ref.L.vox_linear_bf16(P(yb), P(x), W.ctypes.data_as(u16p), bp, M, K, N)
        return yb
    # M == 1 runs the f32 FMA GEMV (decode path): 1e-5.  M > 1 runs on the tensor cores: products are exact (bf16 weight x
    # bf16 activation planes) but the tcgen05 accumulator does not round like an IEEE FMA chain -> ~1e-5 of the row scale
    # (measured 1.1e-5 at K=3072, identical with 2 or 3 planes), so 3e-5.
    close(ya, recorded("out", run_ref), 1e-5 if M == 1 else 3e-5)


def test_remaining_kernel_surface_symbols(vb, ref, recorded):
    """vox_copy, vox_matmul_t, vox_linear_nobias, vox_matmul_t_bf16 (voxtral_kernels.c:42-48,71-86,106-121,255-263): exported
    for header completeness, no pipeline caller; same host-pointer semantics as the reference."""
    rng = np.random.default_rng(55)
    L, R = vb.lib(), (ref.L if ref else None)
    for fn in ("vox_copy", "vox_matmul_t", "vox_linear_nobias", "vox_matmul_t_bf16"):
        getattr(L, fn).restype = None
    L.vox_copy.argtypes = [fp, fp, C.c_int]
    L.vox_matmul_t.argtypes = [fp, fp, fp, C.c_int, C.c_int, C.c_int]
    L.vox_linear_nobias.argtypes = [fp, fp, fp, C.c_int, C.c_int, C.c_int]
    L.vox_matmul_t_bf16.argtypes = [fp, fp, u16p, C.c_int, C.c_int, C.c_int]
    def run_ref(fn, out, *args):
        getattr(R, fn)(P(out), *args)
        return out
    src = rng.normal(size=1000).astype(np.float32); a = np.zeros_like(src)
    L.vox_copy(P(a), P(src), src.size)
    b = recorded("vox_copy", lambda: run_ref("vox_copy", np.zeros_like(src), P(src), src.size))
    assert np.array_equal(a, src) and np.array_equal(b.values, b.take(src))
    M, K, N = 7, 200, 33
    A = rng.normal(size=(M, K)).astype(np.float32); B = rng.normal(size=(N, K)).astype(np.float32)
    ya = np.empty((M, N), np.float32)
    L.vox_matmul_t(P(ya), P(A), P(B), M, K, N)
    close(ya, recorded("vox_matmul_t", lambda: run_ref("vox_matmul_t", np.empty_like(ya), P(A), P(B), M, K, N)), 1e-5)
    L.vox_linear_nobias(P(ya), P(A), P(B), M, K, N)
    close(ya, recorded("vox_linear_nobias", lambda: run_ref("vox_linear_nobias", np.empty_like(ya), P(A), P(B), M, K, N)), 1e-5)
    for M2, K2, N2 in ((1, 1280, 256), (9, 1280, 256), (5, 2048, 130)):
        A2 = rng.normal(size=(M2, K2)).astype(np.float32); W = bf16_weights(rng, N2, K2, np.sqrt(3.0 / K2))
        za = np.empty((M2, N2), np.float32)
        L.vox_matmul_t_bf16(P(za), P(A2), W.ctypes.data_as(u16p), M2, K2, N2)
        zb = recorded(f"vox_matmul_t_bf16_{M2}x{K2}x{N2}",
                      lambda: run_ref("vox_matmul_t_bf16", np.empty_like(za), P(A2), W.ctypes.data_as(u16p), M2, K2, N2))
        close(za, zb, 3e-5)


def test_linear_f32_and_matmul(vb, ref, recorded):
    rng = np.random.default_rng(5)
    M, K, N = 9, 200, 33
    x = rng.normal(size=(M, K)).astype(np.float32)
    W = rng.normal(size=(N, K)).astype(np.float32)
    b = rng.normal(size=N).astype(np.float32)
    ya, yb = np.empty((M, N), np.float32), np.empty((M, N), np.float32)
    vb.lib().vox_linear(P(ya), P(x), P(W), P(b), M, K, N)

    def run_linear():
        ref.L.vox_linear(P(yb), P(x), P(W), P(b), M, K, N)
        return yb
    close(ya, recorded("vox_linear", run_linear), 1e-5)
    B = rng.normal(size=(K, N)).astype(np.float32)
    vb.lib().vox_matmul(P(ya), P(x), P(B), M, K, N)

    def run_matmul():
        ref.L.vox_matmul(P(yb), P(x), P(B), M, K, N)
        return yb
    close(ya, recorded("vox_matmul", run_matmul), 1e-5)


def test_softmax(vb, ref, recorded):
    rng = np.random.default_rng(6)
    x = (rng.normal(size=(3, 1000)) * 4).astype(np.float32)
    a = x.copy()
    vb.lib().vox_softmax(P(a), 3, 1000)

    def run_ref(b=x.copy()):
        ref.L.vox_softmax(P(b), 3, 1000)
        return b
    close(a, recorded("out", run_ref), 1e-5)


@pytest.mark.parametrize("seq_q,seq_k,H,Hkv,hd,win,qoff", [
    (1, 300, 32, 8, 128, 8192, 299),        # decode step, GQA
    (38, 38, 32, 8, 128, 8192, 0),          # prefill
    (20, 820, 32, 32, 64, 750, 800),        # encoder chunk against a full window (mask on both sides)
    (150, 900, 32, 32, 64, 750, 750),       # several 64-query tiles, ragged last tile, window start inside a key tile
    (70, 70, 32, 32, 64, 750, 0),           # stream start: keys < window
    (9, 9, 4, 2, 32, 3, 0),                 # tiny window
    (5, 1755, 32, 32, 64, 750, 1750),       # live feed: 5 new positions against a full window (split-key kernel)
    (3, 70, 32, 32, 64, 750, 67),           # split-key kernel with fewer keys than 8 warps x 4 for some warps
    (2, 64, 32, 32, 64, 750, 10),           # split-key kernel, causal end before the end of the keys
    (300, 1500, 32, 32, 64, 750, 1200),     # tcgen05 kernel: three 128-query tiles, 14 key blocks each, full window, ragged last tile
    (128, 128, 32, 32, 64, 750, 0),         # tcgen05 kernel: exactly one tile, two key blocks, pure causal mask
    (129, 1000, 32, 32, 64, 750, 871),      # tcgen05 kernel: a second tile with a single row
    (33, 97, 32, 32, 64, 40, 64),           # tcgen05 kernel: small window that starts and ends inside key blocks
    (200, 200, 4, 4, 64, 100, 0),           # tcgen05 kernel: 4 heads, window shorter than the tile
])
def test_causal_attention(vb, ref, recorded, seq_q, seq_k, H, Hkv, hd, win, qoff):
    rng = np.random.default_rng(7 + seq_q)
    Q = rng.normal(size=(seq_q, H * hd)).astype(np.float32)
    K = rng.normal(size=(seq_k, Hkv * hd)).astype(np.float32)
    V = rng.normal(size=(seq_k, Hkv * hd)).astype(np.float32)
    a, b = np.empty_like(Q), np.empty_like(Q)
    scale = 1.0 / np.sqrt(hd)
    vb.lib().vox_causal_attention(P(a), P(Q), P(K), P(V), seq_q, seq_k, H, Hkv, hd, scale, win, qoff)

    def run_ref():
        ref.L.vox_causal_attention(P(b), P(Q), P(K), P(V), seq_q, seq_k, H, Hkv, hd, scale, win, qoff)
        return b
    close(a, recorded("out", run_ref), 2e-5)


@pytest.mark.parametrize("seq_q,seq_k,win,qoff", [(300, 1500, 750, 1200), (129, 1000, 750, 871), (33, 97, 40, 64)])
def test_causal_attention_p_in_tensor_memory(vb, ref, recorded, seq_q, seq_k, win, qoff):
    """k_attn_tc_t (VOX_CUDA_ATTN_P=tmem): P stored with tcgen05.st, P V with its A operand in TMEM.  Same plane products in the
    same order as the shared-memory kernel, so the two must agree to rounding noise; both against the reference."""
    import os
    rng = np.random.default_rng(70 + seq_q)
    H, hd = 32, 64
    Q = rng.normal(size=(seq_q, H * hd)).astype(np.float32)
    K = rng.normal(size=(seq_k, H * hd)).astype(np.float32)
    V = rng.normal(size=(seq_k, H * hd)).astype(np.float32)
    a, a_t, b = np.empty_like(Q), np.empty_like(Q), np.empty_like(Q)
    scale = 1.0 / np.sqrt(hd)
    vb.lib().vox_causal_attention(P(a), P(Q), P(K), P(V), seq_q, seq_k, H, H, hd, scale, win, qoff)
    old = os.environ.get("VOX_CUDA_ATTN_P")
    os.environ["VOX_CUDA_ATTN_P"] = "tmem"
    try:
        vb.lib().vox_causal_attention(P(a_t), P(Q), P(K), P(V), seq_q, seq_k, H, H, hd, scale, win, qoff)
    finally:
        if old is None:
            del os.environ["VOX_CUDA_ATTN_P"]
        else:
            os.environ["VOX_CUDA_ATTN_P"] = old
    def run_ref():
        ref.L.vox_causal_attention(P(b), P(Q), P(K), P(V), seq_q, seq_k, H, H, hd, scale, win, qoff)
        return b
    close(a_t, recorded("out", run_ref), 2e-5)
    assert np.abs(a_t - a).max() <= 1e-6 * max(float(np.abs(a).max()), 1e-6)


@pytest.mark.parametrize("hd,heads,pos0", [(128, 8, 0), (64, 32, 180000), (128, 32, 9000)])
def test_rope(vb, ref, recorded, hd, heads, pos0):
    rng = np.random.default_rng(8)
    seq = 5
    pos = (np.arange(seq) + pos0).astype(np.int32)
    fa = np.empty((seq, hd), np.float32)
    vb.lib().vox_compute_rope_freqs(P(fa), pos.ctypes.data_as(C.POINTER(C.c_int)), seq, hd, 1e6)

    def run_freqs(fb=np.empty((seq, hd), np.float32)):
        ref.L.vox_compute_rope_freqs(P(fb), pos.ctypes.data_as(C.POINTER(C.c_int)), seq, hd, 1e6)
        return fb
    fb = np.ascontiguousarray(recorded("freqs", run_freqs, whole=True).values, dtype=np.float32)     # the input of apply_rope
    # cos/sin of angle = (float)pos * freq: one ulp of the f32 ANGLE is pos*2^-23 rad, and the reference
    # build (-ffast-math, libmvec _ZGVdN8vv_powf/_ZGVdN8v_cosf) rounds freq differently from scalar libm, so
    # the tables agree to a few angle-ulps, not to 1e-6, at large positions (SURVEY.md section 7 hard part 6).
    tol = max(2e-6, 4.0 * (pos0 + seq) * 2.0 ** -23)
    assert float(np.abs(fa - fb).max()) <= tol
    x = rng.normal(size=(seq, heads * hd)).astype(np.float32)
    a = x.copy()
    vb.lib().vox_apply_rope(P(a), P(fb), seq, heads, hd)

    def run_apply(b=x.copy()):
        ref.L.vox_apply_rope(P(b), P(fb), seq, heads, hd)
        return b
    close(a, recorded("apply", run_apply), 2e-6)


@pytest.mark.parametrize("cin,cout,L,stride", [(128, 64, 50, 1), (64, 48, 50, 2), (64, 48, 51, 2)])
def test_causal_conv1d(vb, ref, recorded, cin, cout, L, stride):
    rng = np.random.default_rng(9)
    x = rng.normal(size=(cin, L)).astype(np.float32)
    w = (rng.normal(size=(cout, cin, 3)) * 0.05).astype(np.float32)
    b = rng.normal(size=cout).astype(np.float32)
    out_len = L if stride == 1 else (L + 1) // 2
    ya, yb = np.zeros((cout, out_len), np.float32), np.zeros((cout, out_len), np.float32)
    vb.lib().vox_causal_conv1d(P(ya), P(x), P(w), P(b), cin, cout, L, 3, stride)

    def run_causal():
        ref.L.vox_causal_conv1d(P(yb), P(x), P(w), P(b), cin, cout, L, 3, stride)
        return yb
    close(ya, recorded("causal", run_causal), 1e-5)
    # symmetric-padding variant
    out_len = (L + 2 - 3) // stride + 1
    ya, yb = np.zeros((cout, out_len), np.float32), np.zeros((cout, out_len), np.float32)
    vb.lib().vox_conv1d(P(ya), P(x), P(w), P(b), cin, cout, L, 3, stride, 1)

    def run_sym():
        ref.L.vox_conv1d(P(yb), P(x), P(w), P(b), cin, cout, L, 3, stride, 1)
        return yb
    close(ya, recorded("symmetric", run_sym), 1e-5)


def _mel_stream(L, pcm, chunks, free):
    ctx = L.vox_mel_ctx_init(32 * 1280)
    off = 0
    for c in chunks:
        seg = np.ascontiguousarray(pcm[off:off + c]); off += c
        if seg.size:
            L.vox_mel_feed(ctx, P(seg), seg.size)
    z = np.zeros(17 * 1280, np.float32)
    L.vox_mel_feed(ctx, P(z), z.size)
    L.vox_mel_finish(ctx, 0)
    n = C.c_int()
    p = L.vox_mel_data(ctx, C.byref(n))
    out = np.ctypeslib.as_array(p, shape=(n.value, 128)).copy()
    L.vox_mel_free(ctx)
    return out


def test_mel_batch_and_stream(vb, ref, recorded):
    from conftest import read_wav_f32, synth_wav
    pcm = read_wav_f32(synth_wav(2))
    n1 = C.c_int()
    pa = vb.lib().vox_mel_spectrogram(P(pcm), pcm.size, C.byref(n1))

    def run_batch(n2=C.c_int()):
        pb = ref.L.vox_mel_spectrogram(P(pcm), pcm.size, C.byref(n2))
        return np.ctypeslib.as_array(pb, shape=(n2.value, 128)).copy()
    b = recorded("batch", run_batch)
    assert n1.value == b.shape[0] == 200
    a = np.ctypeslib.as_array(pa, shape=(n1.value, 128)).copy()
    # log-mel values are O(1) and stored as (log10(p)+4)/4; bins whose power is a near-cancelling sum (1e-8 of the
    # frame energy) move by ~1e-3 relative under a different f32 summation order -> 5e-4 absolute after the log
    assert b.max_abs_diff(a) < 5e-4, b.max_abs_diff(a)
    # streaming: same frames regardless of how the audio is chunked; equals the reference stream mel
    sa = _mel_stream(vb.lib(), pcm, [pcm.size], None)
    sb = recorded("stream", lambda: _mel_stream(ref.L, pcm, [pcm.size], None))
    sc = _mel_stream(vb.lib(), pcm, [1000, 160, 1, 7777, pcm.size], None)
    assert sa.shape == sb.shape == sc.shape
    assert sb.max_abs_diff(sa) < 5e-4
    assert np.array_equal(sa, sc)
