import ctypes as C
import os
import subprocess
import sys
import tempfile
import wave
import zlib

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import vbload  # noqa: E402

GOLDEN = os.path.join(ROOT, "tests", "golden")
# the seeded checkpoint (8.9 GB) and PCM are generated on first use, outside the tree, in a directory of the current user
SYNTH_DIR = os.environ.get("VOX_SYNTH_DIR", os.path.join(tempfile.gettempdir(), f"voxsynth_b200_{os.getuid()}"))
MODEL_MD5_SEED = "b200"


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


def _tool(name, src, extra=()):
    exe = os.path.join(ROOT, "tools", "_build", name)
    if not os.path.exists(exe) or os.path.getmtime(exe) < os.path.getmtime(os.path.join(ROOT, "tools", src)):
        os.makedirs(os.path.dirname(exe), exist_ok=True)
        subprocess.check_call(["gcc", "-O2", *extra, "-o", exe, os.path.join(ROOT, "tools", src), "-lm"])
    return exe


def ensure_synth_model(path=SYNTH_DIR):
    """Seeded synthetic checkpoint + tokenizer (bit-identical wherever it is generated)."""
    st = os.path.join(path, "consolidated.safetensors")
    if not (os.path.exists(st) and os.path.getsize(st) > 8_000_000_000):
        os.makedirs(path, exist_ok=True)
        subprocess.check_call([_tool("make_synth_model", "make_synth_model.c", ["-fopenmp"]), path])
    if not os.path.exists(os.path.join(path, "tekken.json")):
        subprocess.check_call([sys.executable, os.path.join(ROOT, "tools", "make_synth_tekken.py"), path])
    return path


def synth_wav(seconds, path=SYNTH_DIR):
    os.makedirs(path, exist_ok=True)
    fn = os.path.join(path, f"synth_{seconds:g}s.wav")
    if not os.path.exists(fn):
        subprocess.check_call([_tool("make_synth_wav", "make_synth_wav.c"), fn, f"{seconds:g}"])
    return fn


def read_wav_f32(fn):
    with wave.open(fn) as w:
        pcm = np.frombuffer(w.readframes(w.getnframes()), dtype=np.int16)
    return (pcm.astype(np.float32) / np.float32(32768.0)).astype(np.float32)


@pytest.fixture(scope="session")
def vb(request):
    if RECORD:
        return ReferenceAsEngine(request.getfixturevalue("ref"))
    m = vbload.load()
    if not os.path.exists(m.LIB_PATH):
        m.build()
    return m


class RefLib:
    """The UNMODIFIED reference, compiled by oracle/Makefile into oracle/_ref/libvoxref.so."""

    def __init__(self, path):
        self.L = C.CDLL(path)          # RTLD_LOCAL: must not interpose the engine's identical symbol names
        fp, i, f, vp = C.POINTER(C.c_float), C.c_int, C.c_float, C.c_void_p
        u16p = C.POINTER(C.c_uint16)
        ip = C.POINTER(C.c_int)
        sig = {
            "vox_load": (vp, [C.c_char_p]), "vox_free": (None, [vp]),
            "vox_rms_norm": (None, [fp, fp, fp, i, i, f]),
            "vox_linear_bf16": (None, [fp, fp, u16p, fp, i, i, i]),
            "vox_linear_nobias_bf16": (None, [fp, fp, u16p, i, i, i]),
            "vox_linear": (None, [fp, fp, fp, fp, i, i, i]),
            "vox_matmul": (None, [fp, fp, fp, i, i, i]),
            "vox_silu": (None, [fp, i]), "vox_gelu": (None, [fp, i]), "vox_softmax": (None, [fp, i, i]),
            "vox_add_inplace": (None, [fp, fp, i]), "vox_mul_inplace": (None, [fp, fp, i]),
            "vox_axpy": (None, [fp, f, fp, i]), "vox_scale": (None, [fp, f, i]),
            "vox_causal_attention": (None, [fp, fp, fp, fp, i, i, i, i, i, f, i, i]),
            "vox_compute_rope_freqs": (None, [fp, ip, i, i, f]),
            "vox_apply_rope": (None, [fp, fp, i, i, i]),
            "vox_conv1d": (None, [fp, fp, fp, fp, i, i, i, i, i, i]),
            "vox_causal_conv1d": (None, [fp, fp, fp, fp, i, i, i, i, i]),
            "vox_mel_spectrogram": (fp, [fp, i, ip]),
            "vox_mel_ctx_init": (vp, [i]), "vox_mel_feed": (i, [vp, fp, i]), "vox_mel_finish": (i, [vp, i]),
            "vox_mel_data": (fp, [vp, ip]), "vox_mel_free": (None, [vp]),
            "vox_mel_frame_offset": (i, [vp]), "vox_mel_discard_before": (None, [vp, i]),
            "vox_load_wav": (fp, [C.c_char_p, ip]),
            "vox_tokenizer_load": (vp, [C.c_char_p]), "vox_tokenizer_decode": (C.c_char_p, [vp, i]),
            "vox_tokenizer_free": (None, [vp]),
            "vox_decoder_forward": (i, [vp, fp, fp]), "vox_decoder_prefill": (None, [vp, fp, i]),
            "vox_encoder_forward_incremental": (fp, [vp, fp, i, ip]),
            "vox_encoder_forward": (fp, [vp, fp, i, ip]),
            "vox_copy": (None, [fp, fp, i]), "vox_matmul_t": (None, [fp, fp, fp, i, i, i]),
            "vox_linear_nobias": (None, [fp, fp, fp, i, i, i]), "vox_matmul_t_bf16": (None, [fp, fp, u16p, i, i, i]),
            "vox_adapter_forward": (fp, [vp, fp, i, ip]),
        }
        for n, (r, a) in sig.items():
            fn = getattr(self.L, n)
            fn.restype, fn.argtypes = r, a
        self.free = C.CDLL(None).free
        self.free.argtypes = [C.c_void_p]


@pytest.fixture(scope="session")
def ref():
    """The compiled reference; only recording (VOX_RECORD_REFERENCE=1) runs it, the tests read what it recorded."""
    if not RECORD:
        return None
    p = os.path.join(ROOT, "oracle", "_ref", "libvoxref.so")
    if not os.path.exists(p):
        subprocess.check_call(["make", "-C", os.path.join(ROOT, "oracle"), "ref", "REF=" + os.environ["VOX_REFERENCE_DIR"]])
    os.environ.setdefault("OPENBLAS_NUM_THREADS", str(os.cpu_count() or 8))
    return RefLib(p)


@pytest.fixture(scope="session")
def model_dir():
    return ensure_synth_model()


@pytest.fixture(scope="session")
def engine(vb, model_dir):
    e = vb.Engine(model_dir)
    yield e
    e.close()


# ------------------------------------------------------------------------------------------------
# Outputs of the unmodified reference, stored under tests/golden/reference/<test module>.npz.
#
# A test asks `recorded(tag, compute)` for what the reference returned on its seeded inputs.  Normally that is read from
# the fixture file; `compute` (which calls the reference) runs only when the fixtures are made, from the reference's sources
# (oracle/Makefile `ref` builds them into oracle/_ref/):
#     VOX_RECORD_REFERENCE=1 VOX_REFERENCE_DIR=<reference sources> python -m pytest tests -m "" -p no:cacheprovider
# In that mode `vb` and `engine` are the reference itself, so every comparison runs reference against reference on the host
# cores and no GPU is needed; tests that need the engine itself fail then and record nothing.
# ------------------------------------------------------------------------------------------------
RECORD = os.environ.get("VOX_RECORD_REFERENCE") == "1"
FULL_MAX = 256             # outputs up to this many values are stored whole
SAMPLES = 128              # larger ones: a fixed sample of at least this many values, at least one in every row
_recording = {}            # fixture file -> {key: array}


def _sample_index(shape, key):
    rows = int(shape[0]) if len(shape) > 1 else 1
    cols = int(np.prod(shape)) // rows
    per_row = min(cols, max(1, -(-SAMPLES // rows)))
    rng = np.random.default_rng(zlib.crc32(key.encode()))
    return np.concatenate([r * cols + np.sort(rng.choice(cols, per_row, replace=False)) for r in range(rows)])


class Recorded:
    """One reference output: `values` (whole, or the sample at `idx` of the flattened output), `scale` = max |output| of the
    whole output, `shape`.  `take(x)` picks the same elements out of an output of the engine."""

    def __init__(self, values, idx, scale, shape):
        self.values, self.idx, self.scale, self.shape = values, idx, float(scale), tuple(int(s) for s in shape)

    def take(self, x):
        x = np.asarray(x)
        assert x.shape == self.shape, (x.shape, self.shape)
        return x if self.idx is None else x.reshape(-1)[self.idx]

    def max_abs_diff(self, x):
        return float(np.abs(self.take(x).astype(np.float64) - self.values).max())


def _fixture_file(request):
    return os.path.join(GOLDEN, "reference", request.module.__name__.rsplit(".", 1)[-1] + ".npz")


@pytest.fixture
def recorded(request, ref):
    path = _fixture_file(request)
    store = None if RECORD else (np.load(path) if os.path.exists(path) else {})

    def get(tag, compute, whole=False):
        """`whole`: store the output whatever its size (for an output a test feeds back in as an input)."""
        key = f"{request.node.name}|{tag}"
        if RECORD:
            out = np.asarray(compute())
            rec = _recording.setdefault(path, {})
            rec[key + "|shape"] = np.array(out.shape, np.int64)
            if out.dtype.kind == "f":
                rec[key + "|scale"] = np.array(float(np.abs(out).max()) if out.size else 0.0)
            sampled = out.size > FULL_MAX and not whole
            rec[key + "|values"] = out.reshape(-1)[_sample_index(out.shape, key)] if sampled else out
        elif key + "|values" not in store:
            pytest.fail(f"no recorded reference output {key!r} in {os.path.relpath(path, ROOT)} (VOX_RECORD_REFERENCE=1, see conftest.py)")
        src = _recording[path] if RECORD else store
        shape, values = src[key + "|shape"], src[key + "|values"]
        idx = _sample_index(shape, key) if values.size < np.prod(shape) else None
        scale = src[key + "|scale"] if key + "|scale" in src else 0.0
        return Recorded(values, idx, scale, shape)

    return get


def pytest_sessionfinish(session):
    for path, rec in _recording.items():
        old = dict(np.load(path)) if os.path.exists(path) else {}
        old.update(rec)
        np.savez_compressed(path, **old)


class ReferenceAsEngine:
    """Stands in for the engine package while recording: the same C API names, served by the reference build."""

    def __init__(self, ref):
        self.ref, self.LIB_PATH, self.PKG_DIR = ref, ref.L._name, os.path.dirname(ref.L._name)
        ref.L.free_ = ref.free

    def lib(self):
        return self.ref.L

    def have_gpu(self):
        return False

    def Engine(self, model_dir):
        return _ReferenceEngine(self.ref, model_dir)


class _ReferenceEngine:
    def __init__(self, ref, model_dir):
        self.ref, self.model_dir = ref, model_dir
        self.ctx = ref.L.vox_load(model_dir.encode())
        assert self.ctx

    def close(self):
        self.ref.L.vox_free(self.ctx)

    def reset_caches(self):                    # a fresh context: empty decoder and encoder caches
        self.close()
        self.ctx = self.ref.L.vox_load(self.model_dir.encode())

    def decoder_prefill(self, embeds):
        e = np.ascontiguousarray(embeds, dtype=np.float32)
        self.ref.L.vox_decoder_prefill(self.ctx, e.ctypes.data_as(C.POINTER(C.c_float)), e.shape[0])

    def decoder_forward(self, embed):
        e = np.ascontiguousarray(embed, dtype=np.float32)
        logits = np.empty(131072, np.float32)
        fp = C.POINTER(C.c_float)
        return self.ref.L.vox_decoder_forward(self.ctx, e.ctypes.data_as(fp), logits.ctypes.data_as(fp)), logits

    def _rows(self, fn, x, width):
        x = np.ascontiguousarray(x, dtype=np.float32)
        n = C.c_int()
        p = fn(self.ctx, x.ctypes.data_as(C.POINTER(C.c_float)), x.shape[0], C.byref(n))
        out = np.ctypeslib.as_array(p, shape=(n.value * width,)).copy().reshape(n.value, width)
        self.ref.free(C.cast(p, C.c_void_p))
        return out

    def encoder_forward_incremental(self, x_new):
        return self._rows(self.ref.L.vox_encoder_forward_incremental, x_new, 1280)

    def adapter_forward(self, enc_out):
        return self._rows(self.ref.L.vox_adapter_forward, enc_out, 3072)


def golden(name):
    path = os.path.join(GOLDEN, name + ".npz")
    if not os.path.exists(path):
        pytest.skip(f"fixture {name}.npz not generated (tools/make_goldens.py)")
    return np.load(path)
