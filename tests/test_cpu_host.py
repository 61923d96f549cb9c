"""CPU-only checks of the boundary and of the host-side C code in libvoxtral_b200.so:
  - the library loads and exports every symbol include/voxtral_b200.h declares (no compute without a GPU);
  - the public structs are laid out exactly like the reference's (sizeof/offsetof via gcc);
  - the reference's UNCHANGED main.c compiles and links against the library (built by build() where its sources are);
  - vox_load refuses to run without a CUDA device (no CPU fallback);
  - tokenizer / safetensors / WAV host code behave like the reference's (oracle/_ref) on the same files;
  - golden fixtures are present and self-consistent with the stream bookkeeping.
The reference's side of each comparison is recorded under tests/golden/reference/test_cpu_host.npz (tests/conftest.py: `recorded`).
"""
import ctypes as C
import json
import os
import struct
import subprocess
import tempfile
import wave

import numpy as np
import pytest

from conftest import ROOT, golden

fp = C.POINTER(C.c_float)
REF = os.environ.get("VOX_REFERENCE_DIR", "")       # the reference's headers, read only while recording (tests/conftest.py)


def test_library_exports_every_declared_symbol(vb):
    L = vb.lib()
    names = vb.declared_symbols()
    assert len(names) >= 90
    missing = [n for n in names if not hasattr(L, n)]
    assert not missing, missing
    assert b"sm_100a" in L.vox_cuda_version()


def test_kernels_are_built_for_sm100a(vb):
    """The shipped objects must contain sm_100a SASS with the Blackwell-native instructions (B200_PROFILING.md)."""
    out = subprocess.run(["cuobjdump", "-sass", vb.LIB_PATH], capture_output=True, text=True).stdout
    if not out:
        pytest.skip("cuobjdump unavailable")
    assert "sm_100a" in out
    for mnemonic in ("UTCHMMA", "UTMALDG", "LDTM", "UBLKCP"):     # tcgen05.mma, TMA tensor load, tcgen05.ld, bulk copy
        assert mnemonic in out, mnemonic
    # per kernel: the tensor-core attention issues 6 + 6 plane products x 4 k-steps per key block, the persistent GEMM 4 k-steps
    # per plane and stage (the plane loop is not unrolled); both read their accumulators back with tcgen05.ld
    per = {}
    name = None
    for line in out.splitlines():
        if "Function :" in line:
            name = line.split("Function :")[1].strip()
            per[name] = {"UTCHMMA": 0, "UTMALDG": 0, "LDTM": 0}
        elif name:
            for m in per[name]:
                if m in line:
                    per[name][m] += 1
    attn = [v for k, v in per.items() if "k_attn_tc" in k]
    assert attn and attn[0]["UTCHMMA"] == 48 and attn[0]["UTMALDG"] >= 3 and attn[0]["LDTM"] >= 3, attn
    gemm2 = [v for k, v in per.items() if "k_gemm_tc2" in k]
    assert len(gemm2) == 5 and all(v["UTCHMMA"] >= 4 and v["UTMALDG"] >= 2 and v["LDTM"] >= 1 for v in gemm2), gemm2


def test_struct_layout_matches_reference_headers(tmp_path, recorded):
    fields = ["encoder", "adapter", "decoder", "safetensors", "model_dir", "kv_cache_k", "kv_cache_fp16", "kv_cache_len",
              "kv_cache_max", "kv_pos_offset", "delay_tokens", "t_cond", "ada_scale", "use_bf16", "enc_kv_cache_k",
              "enc_kv_cache_len", "enc_kv_cache_max", "enc_kv_cache_is_shared", "enc_kv_pos_offset", "enc_inc_cap",
              "enc_inc_x_norm", "enc_inc_rope_freqs", "dec_x", "dec_rope_freqs"]
    body = "\n".join(f'    printf("%zu\\n", offsetof(vox_ctx_t, {f}));' for f in fields)
    prog = ('#include <stddef.h>\n#include <stdio.h>\n#include "%s"\nint main(void){\n'
            '    printf("%%zu\\n%%zu\\n%%zu\\n%%zu\\n%%zu\\n", sizeof(vox_ctx_t), sizeof(vox_enc_layer_t), sizeof(vox_dec_layer_t),'
            ' sizeof(vox_encoder_t), sizeof(vox_decoder_t));\n%s\n'
            '    printf("%%zu\\n", offsetof(vox_enc_layer_t, w2_bias)); printf("%%zu\\n", offsetof(vox_dec_layer_t, w3_weight_bf16));\n'
            '    return 0; }\n')

    def layout(tag, prog, inc):
        src = tmp_path / f"{tag}.c"
        src.write_text(prog)
        subprocess.check_call(["gcc", "-I", inc, str(src), "-o", str(tmp_path / tag)])
        return np.array(subprocess.check_output([str(tmp_path / tag)], text=True).split(), np.int64)

    ours = layout("ours", prog % ("voxtral_b200.h", body), os.path.join(ROOT, "include"))
    want = recorded("vox_ctx_t", lambda: layout("ref", prog % ("voxtral.h", body), REF))
    assert np.array_equal(ours, want.values)
    # safetensors structs are public too
    prog2 = ('#include <stddef.h>\n#include <stdio.h>\n#include "%s"\nint main(void){ printf("%%zu %%zu %%zu %%zu\\n", sizeof(safetensor_t),'
             ' sizeof(safetensors_file_t), offsetof(safetensor_t, data_offset), offsetof(safetensors_file_t, tensors)); return 0; }\n')
    ours = layout("o2", prog2 % "voxtral_b200.h", os.path.join(ROOT, "include"))
    want = recorded("safetensors", lambda: layout("r2", prog2 % "voxtral_safetensors.h", REF))
    assert np.array_equal(ours, want.values)


CLI = os.path.join(ROOT, "voxtral.c_b200", "_build", "voxtral")


@pytest.mark.skipif(not os.path.exists(CLI), reason="CLI not built: build() links the reference's main.c where its sources are")
def test_reference_main_c_links_unchanged(vb):
    """Drop-in boundary: the reference CLI, compiled from its own main.c and headers (`make -C voxtral.c_b200 voxtral`, run by
    __graft_entry__.build()), links against this library and runs."""
    r = subprocess.run([CLI, "-h"], capture_output=True, text=True)
    assert r.returncode == 0 and "Usage" in r.stderr


def test_no_cpu_fallback(vb, tmp_path):
    if vb.have_gpu():
        pytest.skip("a GPU is present")
    code = ("import sys; sys.path.insert(0, %r); import vbload; m = vbload.load(); "
            "ctx = m.lib().vox_load(b'/nonexistent'); print('CTX', ctx)") % ROOT
    r = subprocess.run([os.sys.executable, "-c", code], capture_output=True, text=True)
    assert "CTX None" in r.stdout
    assert "no CPU fallback" in r.stderr
    # host-pointer kernel wrappers abort loudly instead of computing on the CPU
    code2 = ("import sys, ctypes, numpy as np; sys.path.insert(0, %r); import vbload; m = vbload.load(); "
             "x = np.ones(8, np.float32); m.lib().vox_silu(x.ctypes.data_as(ctypes.POINTER(ctypes.c_float)), 8); print('COMPUTED')") % ROOT
    r2 = subprocess.run([os.sys.executable, "-c", code2], capture_output=True, text=True)
    assert r2.returncode != 0 and "COMPUTED" not in r2.stdout and "no CPU fallback" in r2.stderr


def test_tokenizer_matches_reference(vb, ref, recorded, tmp_path):
    subprocess.check_call([os.sys.executable, os.path.join(ROOT, "tools", "make_synth_tekken.py"), str(tmp_path)])
    path = str(tmp_path / "tekken.json").encode()
    a = vb.lib().vox_tokenizer_load(path)
    assert a
    ids = list(range(0, 40)) + [999, 1000, 1001, 1064, 1255, 1256, 1263, 5000, 77777, 131071, 131072, -1, 200000]

    def run_ref():
        b = ref.L.vox_tokenizer_load(path)
        assert b
        out = [ref.L.vox_tokenizer_decode(b, i) or b"" for i in ids]
        ref.L.vox_tokenizer_free(b)
        return np.array(out, dtype=bytes)
    want = recorded("pieces", run_ref).values
    for i, w in zip(ids, want):
        assert (vb.lib().vox_tokenizer_decode(a, i) or b"") == w, i
    assert vb.lib().vox_tokenizer_decode(a, 1000) == b""          # raw byte 0x00 -> empty C string (INVALID class)
    assert vb.lib().vox_tokenizer_decode(a, 2) == b"</s>"
    vb.lib().vox_tokenizer_free(a)
    assert vb.lib().vox_tokenizer_load(b"/nonexistent/tekken.json") is None


def _write_wav(path, rate, channels, data):
    with wave.open(str(path), "wb") as w:
        w.setnchannels(channels); w.setsampwidth(2); w.setframerate(rate)
        w.writeframes(data.astype("<i2").tobytes())


@pytest.mark.parametrize("rate,channels", [(16000, 1), (16000, 2), (44100, 1), (8000, 2), (48000, 1)])
def test_wav_loader_matches_reference(vb, ref, recorded, tmp_path, rate, channels):
    rng = np.random.default_rng(rate + channels)
    pcm = rng.integers(-20000, 20000, size=(3001, channels))
    p = tmp_path / "a.wav"
    _write_wav(p, rate, channels, pcm)
    na = C.c_int()
    vb.lib().vox_load_wav.restype = fp
    pa = vb.lib().vox_load_wav(str(p).encode(), C.byref(na))

    def run_ref(nb=C.c_int()):
        ref.L.vox_load_wav.restype = fp
        pb = ref.L.vox_load_wav(str(p).encode(), C.byref(nb))
        return np.ctypeslib.as_array(pb, shape=(nb.value,)).copy()
    b = recorded("pcm", run_ref)
    assert na.value == b.shape[0] > 0
    a = np.ctypeslib.as_array(pa, shape=(na.value,))
    # integer ratios (8k, 16k) interpolate at exact positions.  For 44.1k/48k the tap position is a float expression
    # ((float)i * rate / 16000, voxtral_audio.c:118) that the -ffast-math reference build evaluates as i * (rate/16000):
    # the fractional weight then differs by ~ulp(position) ~ 1e-3, times the sample-to-sample slope.
    tol = 2e-6 if rate in (8000, 16000) else 2e-3
    assert b.max_abs_diff(a) < tol
    assert vb.lib().vox_load_wav(b"/nonexistent.wav", C.byref(na)) is None or not vb.lib().vox_load_wav(b"/nonexistent.wav", C.byref(na))


def test_safetensors_reader(vb, tmp_path):
    L = vb.lib()
    L.safetensors_open.restype = C.c_void_p; L.safetensors_open.argtypes = [C.c_char_p]
    L.safetensors_find.restype = C.c_void_p; L.safetensors_find.argtypes = [C.c_void_p, C.c_char_p]
    L.safetensors_get_f32.restype = fp; L.safetensors_get_f32.argtypes = [C.c_void_p, C.c_void_p]
    L.safetensor_numel.restype = C.c_int64; L.safetensor_numel.argtypes = [C.c_void_p]
    L.safetensors_close.argtypes = [C.c_void_p]
    rng = np.random.default_rng(3)
    a = rng.normal(size=(3, 5)).astype(np.float32)
    b16 = (rng.normal(size=7).astype(np.float32).view(np.uint32) >> 16).astype(np.uint16)
    h16 = rng.normal(size=4).astype(np.float16)
    blobs = [("layers.0.a", "F32", a.shape, a.tobytes()), ('b"quoted', "BF16", b16.shape, b16.tobytes()),
             ("half", "F16", h16.shape, h16.tobytes())]
    hdr, off = {"__metadata__": {"format": "pt"}}, 0
    for name, dt, shape, raw in blobs:
        hdr[name] = {"dtype": dt, "shape": list(shape), "data_offsets": [off, off + len(raw)]}
        off += len(raw)
    js = json.dumps(hdr).encode()
    path = tmp_path / "t.safetensors"
    path.write_bytes(struct.pack("<Q", len(js)) + js + b"".join(r for *_, r in blobs))
    sf = L.safetensors_open(str(path).encode())
    assert sf
    t = L.safetensors_find(sf, b"layers.0.a")
    assert t and L.safetensor_numel(t) == 15
    got = np.ctypeslib.as_array(L.safetensors_get_f32(sf, t), shape=(15,))
    assert np.array_equal(got, a.ravel())
    t = L.safetensors_find(sf, b'b"quoted')
    got = np.ctypeslib.as_array(L.safetensors_get_f32(sf, t), shape=(7,))
    assert np.array_equal(got, (b16.astype(np.uint32) << 16).view(np.float32))
    t = L.safetensors_find(sf, b"half")
    got = np.ctypeslib.as_array(L.safetensors_get_f32(sf, t), shape=(4,))
    assert np.array_equal(got, h16.astype(np.float32))
    assert not L.safetensors_find(sf, b"missing")
    L.safetensors_close(sf)
    (tmp_path / "bad.safetensors").write_bytes(bytes([5, 0, 0, 0, 0, 0, 0, 0]) + b"{bad")
    assert not L.safetensors_open(str(tmp_path / "bad.safetensors").encode())
    assert not L.safetensors_open(b"/nonexistent")


def test_goldens_are_consistent():
    for name in ("synth_s2_oneshot", "synth_s2_chunk1s"):
        g = golden(name)
        assert int(g["samples"]) == 32000
        assert len(g["tokens"]) == 36 == g["top_idx"].shape[0]
        assert np.array_equal(g["tokens"], g["top_idx"][:, 0])     # greedy token == top-1 of the traced logits
        assert (np.diff(g["top_val"], axis=1) <= 0).all()
        n_adapter = sum(int(g[f"adapter_{k}_shape"][0]) for k in range(int(g["n_adapter_calls"])))
        assert n_adapter == 74 and n_adapter - 38 == 36
    assert np.array_equal(golden("synth_s2_oneshot")["tokens"], golden("synth_s2_chunk1s")["tokens"])


def test_tokenizer_sequence_and_specials_match_reference(vb, ref, recorded, tmp_path):
    """vox_tokenizer_decode_seq / _bos / _eos / _vocab_size (voxtral_tokenizer.c) against the compiled reference."""
    subprocess.check_call([os.sys.executable, os.path.join(ROOT, "tools", "make_synth_tekken.py"), str(tmp_path)])
    path = str(tmp_path / "tekken.json").encode()
    seq = np.array([1, 32, 1064, 1100, 1255, 33, 5000, 1000, 1256, 77777, 2, 1300], np.int32)

    def run(L):
        L.vox_tokenizer_load.restype = C.c_void_p; L.vox_tokenizer_load.argtypes = [C.c_char_p]
        L.vox_tokenizer_decode_seq.restype = C.c_void_p; L.vox_tokenizer_decode_seq.argtypes = [C.c_void_p, C.POINTER(C.c_int), C.c_int]
        for fn in ("vox_tokenizer_bos", "vox_tokenizer_eos", "vox_tokenizer_vocab_size"):
            getattr(L, fn).restype = C.c_int; getattr(L, fn).argtypes = [C.c_void_p]
        t = L.vox_tokenizer_load(path)
        assert t
        p = L.vox_tokenizer_decode_seq(t, seq.ctypes.data_as(C.POINTER(C.c_int)), seq.size)
        return np.array([C.string_at(p), b"%d" % L.vox_tokenizer_bos(t), b"%d" % L.vox_tokenizer_eos(t),
                         b"%d" % L.vox_tokenizer_vocab_size(t),
                         C.string_at(L.vox_tokenizer_decode_seq(t, seq.ctypes.data_as(C.POINTER(C.c_int)), 0))], dtype=bytes)
    got = run(vb.lib())
    assert got.tolist() == recorded("decode_seq_bos_eos_vocab", lambda: run(ref.L)).values.tolist()
    assert got.tolist()[1:3] == [b"1", b"2"]


def test_wav_buffer_parser_matches_reference(vb, ref, recorded, tmp_path):
    """vox_parse_wav_buffer (voxtral_audio.c): a good stereo 22.05 kHz file, a truncated one, and garbage."""
    rng = np.random.default_rng(5)
    p = tmp_path / "b.wav"
    _write_wav(p, 22050, 2, rng.integers(-15000, 15000, size=(2500, 2)))
    blob = p.read_bytes()
    u8p = C.POINTER(C.c_uint8)
    def parse(L, data):
        """The parsed samples, or an empty array where the parser returns NULL."""
        L.vox_parse_wav_buffer.restype = fp; L.vox_parse_wav_buffer.argtypes = [u8p, C.c_size_t, C.POINTER(C.c_int)]
        n = C.c_int(-7)
        buf = (C.c_uint8 * len(data)).from_buffer_copy(data)
        out = L.vox_parse_wav_buffer(buf, len(data), C.byref(n))
        return np.zeros(0, np.float32) if not out else np.ctypeslib.as_array(out, shape=(n.value,)).copy()

    for data in (blob, blob[:len(blob) // 2], blob[:30], b"RIFFxxxxWAVEjunk" + bytes(64), bytes(100)):
        got = parse(vb.lib(), data)
        want = recorded(f"bytes_{len(data)}", lambda: parse(ref.L, data))
        assert got.shape == want.shape, len(data)
        if got.size:
            assert want.max_abs_diff(got) < 2e-3     # 22.05 kHz taps, see test_wav_loader_matches_reference


@pytest.mark.parametrize("kind", ["raw", "wav"])
def test_read_pcm_stdin_matches_reference(vb, ref, recorded, tmp_path, kind):
    """vox_read_pcm_stdin (voxtral_audio.c): raw s16le 16 kHz mono, or a WAV container, detected from the first bytes."""
    rng = np.random.default_rng(9)
    pcm = rng.integers(-12000, 12000, size=4097).astype("<i2")
    src = tmp_path / "in.bin"
    if kind == "raw":
        src.write_bytes(pcm.tobytes())
    else:
        _write_wav(src, 16000, 1, pcm)
    def read(lib):
        code = ("import ctypes as C, numpy as np, sys; L = C.CDLL(%r); L.vox_read_pcm_stdin.restype = C.POINTER(C.c_float); "
                "n = C.c_int(); p = L.vox_read_pcm_stdin(C.byref(n)); "
                "sys.stdout.buffer.write(np.ctypeslib.as_array(p, shape=(n.value,)).tobytes() if p else b'')") % lib
        with open(src, "rb") as f:
            r = subprocess.run([os.sys.executable, "-c", code], stdin=f, capture_output=True)
        assert r.returncode == 0, r.stderr.decode()[-500:]
        return np.frombuffer(r.stdout, np.float32)
    got = read(vb.LIB_PATH)
    want = recorded("pcm", lambda: read(ref.L._name))
    assert got.size == want.shape[0] == 4097
    assert want.max_abs_diff(got) < 2e-6


def test_mic_stubs_behave_like_the_reference_off_macos(vb):
    """voxtral_mic_macos.c:124-142: on anything but macOS start fails with -1, reads return 0 samples."""
    L = vb.lib()
    buf = (C.c_float * 16)()
    assert L.vox_mic_start() == -1
    assert L.vox_mic_read(buf, 16) == 0 and L.vox_mic_read_available() == 0
    L.vox_mic_stop()


def test_scenario_goldens_are_consistent():
    """Every reference trace under tests/golden/: greedy id == top-1 of the traced logits, top-8 sorted, drain counts add up to
    the number of text tokens, and the scenario-specific facts the GPU tests rely on."""
    import glob
    names = sorted(os.path.basename(p)[:-4] for p in glob.glob(os.path.join(ROOT, "tests", "golden", "*.npz")))
    assert {"synth_s2_oneshot", "synth_s2_chunk1s", "synth_s2_delay240", "synth_s2_flush", "synth_s2_alt3", "synth_s2_interval05",
            "synth_s2p03_oneshot", "synth_s2p03_chunk7001", "synth_s172_continuous"} <= set(names)
    for name in names:
        g = golden(name)
        assert np.array_equal(g["tokens"], g["top_idx"][:, 0]), name
        assert (np.diff(g["top_val"], axis=1) <= 0).all(), name
        if "drain_n" in g.files:
            n_text = int(np.sum(g["tokens"] >= 1000))            # control ids (< 1000) never reach the queue
            assert int(g["drain_n"].sum()) <= n_text and int(g["drain_n"].sum()) >= n_text - 8, name   # invalid (empty) pieces are dropped too
    assert len(golden("synth_s2_flush")["tokens"]) == 53 and list(golden("synth_s2_flush")["drain_n"]) == [0, 6, 17, 0, 0, 30]
    assert int(golden("synth_s172_continuous")["n_prefills"]) == 2 and len(golden("synth_s172_continuous")["tokens"]) == 2154
    assert golden("synth_s2_alt3")["alt"].tobytes().count(b"\n") == 36
    assert int(golden("synth_s2p03_oneshot")["samples"]) % 1280 == 480
