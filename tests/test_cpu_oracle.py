"""Pins the CPU restatement (oracle/vox_oracle.c) against the UNMODIFIED reference compiled into
oracle/_ref/libvoxref.so, function by function, on seeded inputs: what the reference returned is recorded under
tests/golden/reference/test_cpu_oracle.npz (tests/conftest.py: `recorded`).  CPU only.

The reference build is -O3 -ffast-math (+ OpenBLAS for M>1), so "same arithmetic" means: bit-exact for the
purely elementwise f32 ops, ~1e-6 relative where the reference's summation order is not canonical.
"""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
fp = C.POINTER(C.c_float)
ip = C.POINTER(C.c_int)
u16p = C.POINTER(C.c_uint16)


def P(a):
    return a.ctypes.data_as(fp)


@pytest.fixture(scope="module")
def orc():
    so = os.path.join(ROOT, "oracle", "_build", "liboracle.so")
    src = os.path.join(ROOT, "oracle", "vox_oracle.c")
    if not os.path.exists(so) or os.path.getmtime(so) < os.path.getmtime(src):
        subprocess.check_call(["make", "-C", os.path.join(ROOT, "oracle"), "port"])
    L = C.CDLL(so)
    L.orc_stream_mel.restype = C.c_int
    L.orc_causal_conv1d_out_len.restype = C.c_int
    L.orc_argmax.restype = C.c_int
    return L


def bf16(rng, shape, scale):
    w = (rng.uniform(-1, 1, size=shape) * scale).astype(np.float32)
    u = w.view(np.uint32)
    return np.ascontiguousarray(((u + 0x7FFF + ((u >> 16) & 1)) >> 16).astype(np.uint16))


def rel(a, want):
    """`want`: the reference's output of the same call (tests/conftest.py: Recorded)."""
    return want.max_abs_diff(a) / max(want.scale, 1e-9)


def _ref_inplace(ref, fn, x, *args):
    b = x.copy()
    getattr(ref.L, fn)(P(b), *args)
    return b


def test_elementwise_and_activations(orc, ref, recorded):
    rng = np.random.default_rng(0)
    x = (rng.normal(size=4000) * 3).astype(np.float32)
    y = rng.normal(size=4000).astype(np.float32)
    for mine, theirs in (("orc_add", "vox_add_inplace"), ("orc_mul", "vox_mul_inplace")):
        a = x.copy()
        getattr(orc, mine)(P(a), P(y), C.c_int(a.size))
        b = recorded(theirs, lambda: _ref_inplace(ref, theirs, x, P(y), x.size))
        assert np.array_equal(b.take(a), b.values)
    for mine, theirs in (("orc_silu", "vox_silu"), ("orc_gelu", "vox_gelu")):
        a = x.copy()
        getattr(orc, mine)(P(a), C.c_int(a.size))
        assert rel(a, recorded(theirs, lambda: _ref_inplace(ref, theirs, x, x.size))) < 2e-6, mine
    a = x.reshape(4, 1000).copy()
    orc.orc_softmax(P(a), 4, 1000)
    assert rel(a, recorded("vox_softmax", lambda: _ref_inplace(ref, "vox_softmax", x.reshape(4, 1000), 4, 1000))) < 2e-6


@pytest.mark.parametrize("M,K,N,bias", [(1, 3072, 64, False), (1, 1280, 48, True), (7, 512, 40, True)])
def test_linear_bf16(orc, ref, recorded, M, K, N, bias):
    rng = np.random.default_rng(M * 100 + N)
    x = rng.normal(size=(M, K)).astype(np.float32)
    W = bf16(rng, (N, K), np.sqrt(3.0 / K))
    b = (rng.normal(size=N) * 0.1).astype(np.float32) if bias else None
    ya, yb = np.empty((M, N), np.float32), np.empty((M, N), np.float32)
    orc.orc_linear_bf16(P(ya), P(x), W.ctypes.data_as(u16p), P(b) if bias else None, M, K, N)

    def run_ref():
        ref.L.vox_linear_bf16(P(yb), P(x), W.ctypes.data_as(u16p), P(b) if bias else None, M, K, N)
        return yb
    assert rel(ya, recorded("out", run_ref)) < 3e-6


def test_rms_norm_rope_attention(orc, ref, recorded):
    rng = np.random.default_rng(5)
    x = rng.normal(size=(5, 3072)).astype(np.float32)
    w = rng.uniform(0.9, 1.1, size=3072).astype(np.float32)
    a = np.empty_like(x)
    orc.orc_rms_norm(P(a), P(x), P(w), 5, 3072, C.c_float(1e-5))
    assert rel(a, recorded("vox_rms_norm", lambda: _ref_inplace(ref, "vox_rms_norm", x, P(x), P(w), 5, 3072, 1e-5))) < 2e-6
    pos = np.array([0, 1, 37, 900, 8191], dtype=np.int32)
    fa = np.empty((5, 128), np.float32)
    orc.orc_rope_freqs(P(fa), pos.ctypes.data_as(ip), 5, 128, C.c_float(1e6))
    fb = recorded("vox_compute_rope_freqs", lambda: _ref_inplace(ref, "vox_compute_rope_freqs", fa, pos.ctypes.data_as(ip), 5, 128, 1e6),
                  whole=True)
    fb = np.ascontiguousarray(fb.values, dtype=np.float32)                # the input of apply_rope
    assert np.abs(fa - fb).max() < 4 * 8192 * 2.0 ** -23 + 2e-6          # a few ulps of the f32 ANGLE (fast-math libmvec in the ref)
    q = rng.normal(size=(5, 8 * 128)).astype(np.float32)
    a = q.copy()
    orc.orc_apply_rope(P(a), P(fb), 5, 8, 128)
    assert rel(a, recorded("vox_apply_rope", lambda: _ref_inplace(ref, "vox_apply_rope", q, P(fb), 5, 8, 128))) < 1e-6
    for (sq, sk, H, Hkv, hd, win, off) in [(3, 40, 8, 2, 32, 16, 37), (6, 6, 4, 4, 64, 750, 0), (1, 30, 32, 8, 128, 8192, 29)]:
        Q = rng.normal(size=(sq, H * hd)).astype(np.float32)
        K = rng.normal(size=(sk, Hkv * hd)).astype(np.float32)
        V = rng.normal(size=(sk, Hkv * hd)).astype(np.float32)
        a = np.empty_like(Q)
        sc = 1.0 / np.sqrt(hd)
        orc.orc_causal_attention(P(a), P(Q), P(K), P(V), sq, sk, H, Hkv, hd, C.c_float(sc), win, off)
        b = recorded(f"vox_causal_attention_{sq}x{sk}", lambda: _ref_inplace(ref, "vox_causal_attention", Q, P(Q), P(K), P(V), sq, sk, H,
                                                                            Hkv, hd, sc, win, off))
        assert rel(a, b) < 3e-6


@pytest.mark.parametrize("cin,cout,L,stride", [(16, 8, 21, 1), (16, 8, 21, 2), (16, 8, 22, 2)])
def test_causal_conv1d(orc, ref, recorded, cin, cout, L, stride):
    rng = np.random.default_rng(7)
    x = rng.normal(size=(cin, L)).astype(np.float32)
    w = (rng.normal(size=(cout, cin, 3)) * 0.1).astype(np.float32)
    b = rng.normal(size=cout).astype(np.float32)
    n = orc.orc_causal_conv1d_out_len(L, 3, stride)
    assert n == (L if stride == 1 else (L + 1) // 2)
    ya, yb = np.zeros((cout, n), np.float32), np.zeros((cout, n), np.float32)
    orc.orc_causal_conv1d(P(ya), P(x), P(w), P(b), cin, cout, L, 3, stride)
    want = recorded("out", lambda: _ref_inplace(ref, "vox_causal_conv1d", yb, P(x), P(w), P(b), cin, cout, L, 3, stride))
    assert rel(ya, want) < 3e-6


def _ref_stream_mel(ref, pcm, delay_tokens=6):
    ctx = ref.L.vox_mel_ctx_init(32 * 1280)
    ref.L.vox_mel_feed(ctx, P(pcm), pcm.size)
    align = (1280 - pcm.size % 1280) % 1280
    z = np.zeros(align + (delay_tokens + 1 + 10) * 1280, np.float32)
    ref.L.vox_mel_feed(ctx, P(z), z.size)
    ref.L.vox_mel_finish(ctx, 0)
    n = C.c_int()
    p = ref.L.vox_mel_data(ctx, C.byref(n))
    out = np.ctypeslib.as_array(p, shape=(n.value, 128)).copy()
    ref.L.vox_mel_free(ctx)
    return out


def test_stream_mel_matches_reference(orc, ref, recorded):
    rng = np.random.default_rng(9)
    for n in (1000, 16000, 20001):
        pcm = (rng.normal(size=n) * 0.1).astype(np.float32)
        want = recorded(f"mel_{n}", lambda: _ref_stream_mel(ref, pcm))
        frames = orc.orc_stream_mel(None, None, n, 6)
        assert frames == want.shape[0]
        got = np.empty((frames, 128), np.float32)
        orc.orc_stream_mel(P(got), P(pcm), n, 6)
        assert want.max_abs_diff(got) < 5e-4


def test_stream_mel_jfk_checksum(orc, ref, recorded):
    """Real speech: the first 1.5 s of the reference's samples/jfk.wav (tests/golden/jfk_1500ms.npy, 16 kHz s16).  The frame
    count, sum and minimum of the reference's streaming mel of it, and the mel itself, are recorded."""
    pcm = np.load(os.path.join(ROOT, "tests", "golden", "jfk_1500ms.npy")).astype(np.float32) / np.float32(32768.0)
    assert pcm.size == 24000
    frames = orc.orc_stream_mel(None, None, pcm.size, 6)
    want = recorded("mel", lambda: _ref_stream_mel(ref, np.ascontiguousarray(pcm)))
    assert frames == want.shape[0]
    got = np.empty((frames, 128), np.float32)
    orc.orc_stream_mel(P(got), P(np.ascontiguousarray(pcm)), pcm.size, 6)
    ref_sum, ref_min = recorded("sum_min", lambda: (lambda m: np.array([m.sum(dtype=np.float64), m.min()]))(_ref_stream_mel(ref, pcm))).values
    assert abs(float(got.sum(dtype=np.float64)) - ref_sum) < 0.5
    assert abs(float(got.min()) - ref_min) < 1e-6
    # real speech has bins whose power is pure rounding residue (1e-9 of the frame energy); their log moves by a few
    # percent with the summation order (-ffast-math reference), so: tight on average, loose on the worst bin
    d = np.abs(want.take(got) - want.values)
    assert d.mean() < 2e-5 and d.max() < 1e-2


def test_counts_and_time_conditioning(orc):
    for n, want in ((176000, (1496, 748, 187, 149)), (480000, (3392, 1696, 424, 386)), (9600000, (60392, 30196, 7549, 7511)),
                    (57600000, (360392, 180196, 45049, 45011)), (32000, (592, 296, 74, 36))):
        a, b, c, d = C.c_int(), C.c_int(), C.c_int(), C.c_int()
        orc.orc_stream_counts(n, 6, C.byref(a), C.byref(b), C.byref(c), C.byref(d))
        assert (a.value, b.value, c.value, d.value) == want       # SURVEY.md section 8 table + golden synth_s2
    x = np.array([0.5, 3.0, 3.0, -1.0], np.float32)
    assert orc.orc_argmax(P(x), 4) == 1                            # first maximum wins


def _run_pin(name, ref, tmp_path):
    """Build tests/c/<name>.c against the restatement (and, while recording, the reference) and run it; outputs land in tmp_path."""
    exe = str(tmp_path / name)
    odir = os.path.join(ROOT, "oracle", "_build")
    cmd = ["gcc", "-O2", "-I" + os.path.join(ROOT, "include"), "-I" + os.path.join(ROOT, "oracle"),
           os.path.join(ROOT, "tests", "c", name + ".c"), "-o", exe, "-L" + odir, "-loracle", "-Wl,-rpath," + odir, "-lm"]
    if ref is not None:
        rdir = os.path.dirname(ref.L._name)
        cmd[1:1] = ["-DPIN_REFERENCE"]
        cmd[-1:-1] = ["-L" + rdir, "-lvoxref", "-Wl,-rpath," + rdir]
    subprocess.check_call(cmd)
    r = subprocess.run([exe, str(tmp_path)], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr[-500:]


def test_decoder_step_restatement_matches_reference_forward(orc, ref, recorded, tmp_path):
    """orc_decoder_layer_step x 26 + final norm + tied-embedding logits + argmax vs the reference's own vox_decoder_forward at
    the real dimensions, three consecutive positions (tests/c/pin_decoder_step.c fills a public vox_ctx_t by hand).  This is
    the restatement tests/test_gpu_kv_ring_wrap.py uses as its checker."""
    _run_pin("pin_decoder_step", ref, tmp_path)
    for s in range(3):
        got = np.fromfile(tmp_path / f"orc_{s}.f32", np.float32)
        want = recorded(f"logits_{s}", lambda: np.fromfile(tmp_path / f"ref_{s}.f32", np.float32))
        tok_ref, kv_len = recorded(f"argmax_kv_len_{s}", lambda: np.fromfile(tmp_path / f"ref_{s}.i32", np.int32)).values
        diff = want.max_abs_diff(got)
        print(f"step {s} max_abs_diff {diff:.3e} logit_scale {want.scale:.3f} kv_len {kv_len}")
        assert int(np.argmax(got)) == tok_ref and kv_len == s + 1
        assert diff < 5e-6 * want.scale * 2          # measured 2.3e-5 on logits of scale 8: -ffast-math summation order


def test_encoder_layer_and_adapter_restatements_match_reference(orc, ref, recorded, tmp_path):
    """orc_encoder_layer x 32 + final norm vs vox_encoder_forward_incremental over two calls (7 then 5 rows: K/V cache carry,
    logical RoPE positions), and orc_adapter vs vox_adapter_forward, at the real dimensions (tests/c/pin_encoder_adapter.c)."""
    _run_pin("pin_encoder_adapter", ref, tmp_path)
    for name in ("encoder_full", "encoder_call_1", "encoder_call_2", "adapter"):
        width = 3072 if name == "adapter" else 1280
        got = np.fromfile(tmp_path / f"orc_{name}.f32", np.float32).reshape(-1, width)
        want = recorded(name, lambda: np.fromfile(tmp_path / f"ref_{name}.f32", np.float32).reshape(-1, width))
        diff = want.max_abs_diff(got)
        print(f"{name} max_abs_diff {diff:.3e} scale {want.scale:.3f}")
        assert diff < 2e-5 * max(want.scale, 1.0), name     # measured 5e-6..6e-6: OpenBLAS / -ffast-math summation order
    assert recorded("enc_cache_len", lambda: np.fromfile(tmp_path / "ref_enc_cache_len.i32", np.int32)).values.tolist() == [12]
