#!/usr/bin/env python3
"""bench.py -- real-time factor (audio-s / wall-s) + decoder tok/s of the B200 engine.

A "step" = one complete pass of the hot path (mel -> conv stem -> 32-layer encoder -> adapter ->
prefill -> greedy decode) over one synthetic 16 kHz recording, through the reference's streaming API
(vox_stream_init / feed / finish).  Workload at N=1: BASELINE.json configs[2] -- 10 min of synthetic PCM
on one GPU (the configuration the north-star target is quoted on).  N>1: one independent stream per GPU,
replicated weights (configs[3]), no data-path collective; weak scaling.

  value  whole-job audio seconds / device-timed seconds, PCM already resident in HBM
  e2e    the same metric through the public C API with HOST PCM (H2D of the PCM and D2H of the token
         ids inside the timed region), one pass after the timed steps
  roofline  decode step (the dominant phase, >90% of the time): algorithmic bytes per step
         (6.858 GB bf16 weights + f32 KV rows read) / device time per step, vs MEASURED_PEAKS.json
  cpu_baseline  the UNMODIFIED reference (oracle/_ref, built from /root/reference by oracle/Makefile)
         timed on this box's host cores on a bounded sample of the same workload

  parity_prefix  the ids of the benchmarked recording are compared, inside this run, with the reference's own trace of its
         first 60 s (tests/golden/synth_s60_oneshot.npz, oracle/ref_trace on the unmodified reference; the synthetic PCM and
         both models are causal, so that trace is the reference prefix of the 10-minute run)
  multistream  8 copies of the same recording on forked contexts, decoded by ONE persistent kernel per launch
         (vox_cuda_streams_decode: one weight pass for all streams); aggregate audio-s / device-s, ids equal to the
         single-stream run
  sharded_encoder  (N > 1) one 1-hour recording, encoder sharded by sequence over the N GPUs in host C with NCCL
         (vox_cuda_encode_sharded: per-layer K/V halo ncclSend/ncclRecv + adapter ncclAllGather), vs the same call unsharded

`--steps K --warmup W` run max(W, 3) untimed and K timed passes; the e2e pass follows.  cpu_baseline, multistream, live and
sharded_encoder are the extra legs: they run with `--extra-legs` and are null otherwise.
`--impl reference` times only that CPU reference arm.  `--dump-outputs DIR` writes what the last timed step returned to its
caller (token ids, unit counts) as DIR/<name>.npy in float64, so that two builds can be compared output for output: the
synthetic checkpoint and PCM are seeded, so the inputs are identical from run to run.  The model is the seeded synthetic checkpoint
(tools/make_synth_model.c): there is no network for the real weights; throughput does not depend on them.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WEIGHT_BYTES_PER_STEP = 2 * (26 * 116_391_936 + 131072 * 3072)      # bf16 matrices streamed by one decode step
KV_BYTES_PER_SLOT = 26 * 1024 * 4 * 2                                 # f32 K and V rows, all layers


T_START = time.perf_counter()


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def phase(name):
    """Progress on stderr: a run that is stopped early still shows how far it got."""
    log(f"bench: {name} ({time.perf_counter() - T_START:.1f} s)")


def ensure_inputs(seconds):
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from conftest import ensure_synth_model, read_wav_f32, synth_wav
    model = ensure_synth_model()
    pcm = read_wav_f32(synth_wav(seconds))
    return model, pcm


def expected_counts(n):
    align = (1280 - n % 1280) % 1280
    frames = (200 + 40960 + n + align + 17 * 1280 + 200 - 400) // 160 + 1 - 1
    pos = frames // 2
    tokens = pos // 4
    return frames, pos, tokens, tokens - 38


class ClockSampler(threading.Thread):
    """nvidia-smi clocks + throttle reasons during the timed region (B200_PROFILING.md)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.stop = index, [], threading.Event()

    def run(self):
        while not self.stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                      "-i", str(self.index)], capture_output=True, text=True, timeout=5).stdout
                self.rows.append([c.strip() for c in out.strip().split(",")])
            except Exception:
                pass
            self.stop.wait(0.25)

    def summary(self):
        sm = [float(r[0]) for r in self.rows if len(r) >= 7 and r[0].replace(".", "").isdigit()]
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for k, n in enumerate(names) if any(r[3 + k].lower().startswith("active") for r in self.rows if len(r) >= 7)]
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(self.rows[0][1]), "reasons": reasons,
                "samples": len(sm)}


def tensor_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d.get("bf16_tflops_sustained", d.get("bf16_tflops", 0.0))), "measured (MEASURED_PEAKS.json bf16_tflops_sustained)"
    return 1500.0, "fallback (B200_PROFILING.md)"


# f32-equivalent flops per encoder position (SURVEY section 8d): 32 layers x (wq|wk|wv + wo + w1|w3 + w2) = 1.93 GFLOP of linears
# + 0.197 GFLOP of window-750 attention.  The tensor cores execute 3 bf16 plane products per linear MAC and 6 per attention MAC.
ENC_LINEAR_GFLOP, ENC_ATTN_GFLOP = 1.93, 0.197


def encoder_block(positions_per_s):
    peak, src = tensor_peak()
    useful = (ENC_LINEAR_GFLOP + ENC_ATTN_GFLOP) * positions_per_s / 1e3
    issued = (3 * ENC_LINEAR_GFLOP + 6 * ENC_ATTN_GFLOP) * positions_per_s / 1e3
    return {"positions_per_s": positions_per_s, "bound": "tensor", "useful_tflops_f32_equivalent": useful,
            "issued_bf16_tflops": issued, "peak": peak, "unit": "TFLOP/s", "frac_issued": issued / peak if peak else None,
            "peak_source": src,
            "note": "whole encoder pass (mel, conv stem, 32 layers, adapter) timed with CUDA events; issued = 3 bf16 plane products "
                    "per linear MAC (exact f32 activations x bf16 weights) and 6 per attention MAC (f32 x f32), all on tcgen05"}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


# ----------------------------------------------------------------------------------------------
# CPU reference arm: oracle/_ref (the reference's own sources compiled by oracle/Makefile)
# ----------------------------------------------------------------------------------------------
def reference_sample(model_dir, seconds, enc_positions=1024, dec_steps=16):
    """Bounded sample of the workload on the host cores: stream mel of 30 s, one incremental encoder call,
    the 38-token prefill and `dec_steps` single-token forwards; extrapolated to the full recording."""
    refp = os.path.join(ROOT, "oracle", "_ref", "libvoxref.so")
    if not os.path.exists(refp):
        return None
    cores = os.cpu_count() or 1
    os.environ["OPENBLAS_NUM_THREADS"] = str(cores)
    R = C.CDLL(refp)
    fp, vp, ip = C.POINTER(C.c_float), C.c_void_p, C.POINTER(C.c_int)
    R.vox_load.restype = vp; R.vox_load.argtypes = [C.c_char_p]
    R.vox_encoder_forward_incremental.restype = fp
    R.vox_encoder_forward_incremental.argtypes = [vp, fp, C.c_int, ip]
    R.vox_decoder_prefill.argtypes = [vp, fp, C.c_int]
    R.vox_decoder_forward.restype = C.c_int; R.vox_decoder_forward.argtypes = [vp, fp, fp]
    R.vox_adapter_forward.restype = fp; R.vox_adapter_forward.argtypes = [vp, fp, C.c_int, ip]
    R.vox_mel_ctx_init.restype = vp; R.vox_mel_feed.argtypes = [vp, fp, C.c_int]; R.vox_mel_free.argtypes = [vp]
    free = C.CDLL(None).free; free.argtypes = [vp]
    ctx = R.vox_load(model_dir.encode())
    rng = np.random.default_rng(0)
    P = lambda a: a.ctypes.data_as(fp)
    n = C.c_int()
    # mel: 30 s of PCM through the incremental front end
    pcm = (rng.normal(size=480000) * 0.1).astype(np.float32)
    t = time.perf_counter(); m = R.vox_mel_ctx_init(40960); R.vox_mel_feed(m, P(pcm), pcm.size); t_mel = (time.perf_counter() - t) / 30.0
    R.vox_mel_free(m)
    x = np.abs(rng.normal(size=(enc_positions, 1280))).astype(np.float32)
    t = time.perf_counter(); p = R.vox_encoder_forward_incremental(ctx, P(x), enc_positions, C.byref(n)); t_enc = time.perf_counter() - t
    t = time.perf_counter(); q = R.vox_adapter_forward(ctx, p, enc_positions, C.byref(n)); t_ad = time.perf_counter() - t
    free(C.cast(p, vp)); free(C.cast(q, vp))
    emb = (rng.normal(size=(38 + dec_steps, 3072)) * 1.3).astype(np.float32)
    t = time.perf_counter(); R.vox_decoder_prefill(ctx, P(emb[:38].copy()), 38); t_pre = time.perf_counter() - t
    lg = np.empty(131072, np.float32)
    t = time.perf_counter()
    for s in range(dec_steps):
        R.vox_decoder_forward(ctx, P(emb[38 + s].copy()), P(lg))
    t_step = (time.perf_counter() - t) / dec_steps
    R.vox_free.argtypes = [vp]; R.vox_free(ctx)
    frames, pos, toks, steps = expected_counts(int(seconds * 16000))
    total = seconds * t_mel + pos * (t_enc + t_ad) / enc_positions + t_pre + steps * t_step
    return {"rtf": seconds / total, "tok_s": 1.0 / t_step, "cores": cores, "extrapolated": True,
            "measured": {"decoder_ms_per_forward": t_step * 1e3, "prefill_38_s": t_pre, "encoder_s_per_position": (t_enc + t_ad) / enc_positions,
                         "mel_s_per_audio_s": t_mel},
            "wall_sample_s": 30 * t_mel + t_enc + t_ad + t_pre + dec_steps * t_step,
            "sample": (f"reference build timed on host: {dec_steps} decoder forwards ({t_step*1e3:.0f} ms/step, single-threaded "
                       f"by construction), 38-token prefill ({t_pre:.2f} s), one {enc_positions}-position incremental encoder "
                       f"call + adapter ({(t_enc+t_ad):.2f} s, OpenBLAS {cores} threads), 30 s of streaming mel; "
                       f"EXTRAPOLATED linearly to the {seconds:g} s recording ({steps} steps, {pos} positions)")}


def ncu_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum of the decode kernel per step, read from the committed raw export of one
    `ncu --set full` capture (profiles/r02_decode_ncu_raw.csv: one launch = `steps` decode steps of a 30 s clip).  Not measured
    by this script: ncu cannot run inside a timed bench."""
    path = os.path.join(ROOT, "profiles", "r02_decode_ncu_raw.csv")
    meta = os.path.join(ROOT, "profiles", "r02_decode_ncu_raw.json")
    try:
        steps = json.load(open(meta))["steps_in_launch"]
        import csv
        rows = list(csv.reader(open(path)))
        hdr = rows[0]
        unit = rows[1]
        data = rows[2]
        tot = 0.0
        for name in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
            k = hdr.index(name)
            mult = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9, "Tbyte": 1e12}[unit[k]]
            tot += float(data[k].replace(",", "")) * mult
        return tot / steps, "profiles/r02_decode_ncu_raw.csv (ncu --set full, one launch, per step)"
    except Exception:
        return None, "no committed ncu export"



def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--seconds", type=float, default=600.0)
    ap.add_argument("--live-seconds", type=float, default=15.0, help="length of the 0.1-s live-feeding leg (N=1 only; 0 = skip)")
    ap.add_argument("--streams", type=int, default=8, help="streams per GPU in the multistream leg (N=1 only; 1 = skip)")
    ap.add_argument("--sharded-seconds", type=float, default=3600.0, help="recording length of the sharded-encoder leg (N>1)")
    ap.add_argument("--extra-legs", action="store_true", help="also run cpu_baseline, multistream, live and sharded_encoder")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step as DIR/<name>.npy (float64)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    n_gpus = max(args.gpus, world)
    workload = f"{args.seconds:g}s synthetic 16 kHz PCM per stream, one-shot feed+finish, greedy decode, synthetic Voxtral-Mini-4B checkpoint"
    frames, pos, toks, steps_expected = expected_counts(int(args.seconds * 16000))

    if args.impl == "reference":
        if rank != 0:
            return
        model, _ = ensure_inputs(min(args.seconds, 2.0))
        vals, last = [], None
        for i in range(args.warmup + args.steps):
            last = reference_sample(model, args.seconds)
            if last is None:
                print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref/libvoxref.so not built"}))
                return
            if i >= args.warmup:
                vals.append(last["rtf"])
        v = float(np.mean(vals))
        print(json.dumps({
            "impl": "reference", "metric": "real-time factor (audio-s/wall-s)", "value": v, "unit": "x real-time",
            "n_gpus": n_gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * args.seconds / v,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32 activations x bf16 weights",
            "data": "synthetic", "config": {"workload": workload},
            "decoder_tok_s": last["tok_s"],
            "reference_extrapolated": True, "reference_measured": last["measured"],
            "cpu_baseline": {"value": v, "unit": "x real-time", "cores": last["cores"], "kind": "reference", "sample": last["sample"]},
            "e2e": {"value": v, "unit": "x real-time", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))
        return

    # ------------------------------------------------------------------ B200 arm
    dist = None
    if world > 1:
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    os.environ["VOX_CUDA_DEVICE"] = str(local)

    def barrier():
        if dist is not None:
            dist.barrier()

    if rank == 0:
        ensure_inputs(args.seconds)
    barrier()
    model, pcm = ensure_inputs(args.seconds)
    phase("inputs ready")
    import vbload
    vb = vbload.load()
    multi = vbload.load_submodule("multi")
    t_load = time.perf_counter()
    eng = vb.Engine(model)
    load_s = time.perf_counter() - t_load
    phase("engine loaded")
    d_pcm = eng.to_device(pcm)
    profiling = os.environ.get("VOX_BENCH_PROFILE") == "1"      # ncu runs: fewer warm-ups, no extra legs (never a bench value)
    extra = args.extra_legs and not profiling

    def one_pass(device_input):
        s = eng.stream()
        if device_input:
            s.feed_device(d_pcm, pcm.size)
        else:
            s.feed(pcm)
        s.finish()
        ids = s.token_ids()
        c = s.counts()
        s.close()
        return ids, c

    def timed(k, fn):
        barrier()
        eng.timer_start()
        t0 = time.perf_counter()
        for _ in range(k):
            out = fn()
        dev_ms = eng.timer_stop_ms()
        wall = time.perf_counter() - t0
        if dist is not None:
            import torch
            dev_ms, wall_ms = multi.reduce_max([dev_ms, wall * 1e3], dist, torch.device("cuda", local))
            wall = wall_ms / 1e3
        barrier()
        return dev_ms, wall, out

    n_warm = args.warmup if profiling else max(args.warmup, 3)
    for _ in range(n_warm):
        ids, counts = one_pass(True)
    phase("warm-up done")
    sampler = ClockSampler(local); sampler.start()
    i_before = eng.info()
    dev_ms, _, (ids, counts) = timed(args.steps, lambda: one_pass(True))
    i_after = eng.info()
    sampler.stop.set(); sampler.join(timeout=3)
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, ids, counts)
    phase("timed steps done")
    e2e_ms, e2e_wall, (ids2, _) = timed(1, lambda: one_pass(False))
    phase("host-PCM pass done")

    # the work that was timed is the work the reference would do on this recording (an early EOS would shrink it silently)
    assert (counts["mel_frames"], counts["adapter_tokens"], len(ids)) == (frames, toks, steps_expected), \
        (counts, len(ids), (frames, toks, steps_expected))

    audio_s = args.seconds * args.steps * world
    value = audio_s / (dev_ms / 1e3)
    e2e_value = args.seconds * world / max(e2e_ms / 1e3, e2e_wall)
    dsteps = i_after["total_decode_steps"] - i_before["total_decode_steps"]
    dms = i_after["total_decode_kernel_ms"] - i_before["total_decode_kernel_ms"]
    n_dec = len(ids)
    # KV rows read by step i (position 38+i): min(pos+1, 8192) slots
    kv_slots = np.minimum(np.arange(38, 38 + n_dec) + 1, 8192).astype(np.float64)
    kv_mean = KV_BYTES_PER_SLOT * float(kv_slots.mean()) if n_dec else 0.0
    bytes_per_step = WEIGHT_BYTES_PER_STEP + kv_mean
    step_ms = dms / max(dsteps, 1)
    achieved = bytes_per_step / (step_ms / 1e3) / 1e9 if dsteps else 0.0
    peak, peak_src = peaks()

    # ---- parity of the benchmarked recording against the reference's own trace: of the whole recording when that fixture exists
    # (tests/golden/synth_s600_oneshot.npz: the unmodified reference run on the same 10-minute PCM, ~3 h of host time), else of its
    # first 60 s (the synthetic PCM is a pure function of the sample index and both models are causal)
    parity = None
    gfull = os.path.join(ROOT, "tests", "golden", f"synth_s{args.seconds:g}_oneshot.npz")
    gpath = os.path.join(ROOT, "tests", "golden", "synth_s60_oneshot.npz")
    if os.path.exists(gfull) and args.seconds > 60:
        g = np.load(gfull)
        ref = g["tokens"]; margin = g["top_val"][:, 0] - g["top_val"][:, 1]
        n_cmp = min(len(ids), len(ref))
        bad = np.nonzero(ids[:n_cmp] != ref[:n_cmp])[0]
        # a differing id is a near-tie flip if the reference's own top-2 margin there is < 2e-3 (the tests' rule) AND the engine
        # chose the reference's runner-up; anything else is a parity failure
        runner_up = g["top_idx"][:, 1]
        flips = [{"step": int(i), "reference_margin": float(margin[i]), "engine_id_is_reference_runner_up": bool(ids[i] == runner_up[i])}
                 for i in bad[:16]]
        near = all(f["reference_margin"] < 2e-3 and f["engine_id_is_reference_runner_up"] for f in flips) and bad.size <= 16
        parity = {"compared_ids": int(n_cmp), "reference_ids": int(len(ref)),
                  "reference": os.path.relpath(gfull, ROOT) + " (unmodified reference on the whole recording, oracle/ref_trace)",
                  "first_mismatch": int(bad[0]) if bad.size else None, "mismatching_ids": int(bad.size),
                  "reference_margin_at_mismatch": float(margin[bad[0]]) if bad.size else None,
                  "near_tie_flips": flips, "all_mismatches_are_near_ties": bool(near), "ids_equal": bool(bad.size == 0),
                  "rule": "parity_prefix_ok = every id equals the reference's, except where the reference's own top-2 logit margin is "
                          "< 2e-3 and the engine chose its runner-up (listed in near_tie_flips)",
                  "note": "recorded on a B200 (profiles/r02_bench.md): with VOX_CUDA_GEMM=v1 (plane-major accumulation in every tcgen05 "
                          "GEMM, 0.6 x the encoder throughput) the same build reproduces all 7511 ids of this recording"}
    elif os.path.exists(gpath) and args.seconds >= 60:
        g = np.load(gpath)
        ref = g["tokens"]; margin = g["top_val"][:, 0] - g["top_val"][:, 1]
        n_cmp = min(len(ids), len(ref) - 40)              # the last positions of the 60 s trace see its right padding
        bad = np.nonzero(ids[:n_cmp] != ref[:n_cmp])[0]
        parity = {"compared_ids": int(n_cmp), "reference": "tests/golden/synth_s60_oneshot.npz (unmodified reference, oracle/ref_trace)",
                  "first_mismatch": int(bad[0]) if bad.size else None,
                  "reference_margin_at_mismatch": float(margin[bad[0]]) if bad.size else None}
    if rank == 0 and os.environ.get("VOX_BENCH_SAVE_IDS"):   # for an offline comparison with a reference trace made later
        os.makedirs(os.path.join(ROOT, "gpurun_out"), exist_ok=True)
        np.save(os.path.join(ROOT, "gpurun_out", f"bench_ids_{args.seconds:g}s.npy"), np.asarray(ids, dtype=np.int32))
    parity_ok = bool(parity is not None and (parity["first_mismatch"] is None or parity.get("all_mismatches_are_near_ties", False)))

    # ---- several streams per weight pass on this GPU (N = 1 only: the scaling run keeps one stream per GPU)
    ms_block = None
    if world == 1 and extra and args.streams > 1:
        B = args.streams
        forks = [eng.fork() for _ in range(B - 1)]
        engines = [eng] + forks

        def batched_pass():
            streams = [e.stream() for e in engines]
            for s in streams:
                s.set_deferred(1)
                s.feed_device(d_pcm, pcm.size)
            vb.streams_decode(streams)
            for s in streams:
                s.finish()
            vb.streams_decode(streams)
            out = [s.token_ids() for s in streams]
            for s in streams:
                s.close()
            return out

        batched_pass()                                         # warm-up (workspaces of the forks grow here)
        j0 = eng.info()
        b_ms, _, b_ids = timed(1, batched_pass)
        j1 = eng.info()
        b_steps = j1["total_decode_steps"] - j0["total_decode_steps"]
        b_dms = j1["total_decode_kernel_ms"] - j0["total_decode_kernel_ms"]
        b_step_ms = b_dms / max(b_steps, 1)
        b_bytes = WEIGHT_BYTES_PER_STEP + B * kv_mean
        ms_block = {"streams": B, "value": B * args.seconds / (b_ms / 1e3), "unit": "x real-time (aggregate over the streams of this GPU)",
                    "per_stream": args.seconds / (b_ms / 1e3), "ms_per_pass": b_ms,
                    "ids_equal_single_stream": bool(all(np.array_equal(x, ids) for x in b_ids)),
                    "decode_ms_per_step": b_step_ms, "decoder_tok_s": B * b_steps / (b_dms / 1e3) if b_dms else None,
                    "roofline": {"bound": "hbm", "achieved": b_bytes / (b_step_ms / 1e3) / 1e9 if b_steps else 0.0, "peak": peak, "unit": "GB/s",
                                 "frac": (b_bytes / (b_step_ms / 1e3) / 1e9 / peak) if b_steps else 0.0, "bytes_per_step": b_bytes,
                                 "note": "one weight pass (6.858 GB) + the f32 KV rows of every stream per step"},
                    "api": "vox_cuda_ctx_fork + vox_cuda_stream_set_deferred + vox_cuda_streams_decode"}
        for f in forks:
            f.close()

    # ---- live shape (main.c --stdin -I 0.1 / --from-mic): 0.1 s feeds, one small encoder call + 1-2 decode steps per feed
    phase("multistream leg done")
    live = None
    if world == 1 and extra and args.live_seconds > 0:
        n_live = min(pcm.size, int(args.live_seconds * 16000))
        for rep in range(2):                                   # first repetition warms the small-M workspaces
            st = eng.stream()
            st.set_interval(0.1)
            st.set_continuous(1)
            times, l0 = [], eng.info()["kernel_launches"]
            for off in range(0, n_live, 1600):
                t0 = time.perf_counter()
                st.feed(pcm[off:off + 1600])
                st.get()
                times.append((time.perf_counter() - t0) * 1e3)
            st.finish()
            live_ids = st.token_ids()
            st.close()
        t = np.array(times[20:])                               # steady state: after the prompt delay
        live = {"feed_s": 0.1, "feeds": len(times), "ms_per_feed_median": float(np.median(t)), "ms_per_feed_p90": float(np.percentile(t, 90)),
                "ms_per_feed_max": float(t.max()), "budget_ms": 100.0, "launches_per_feed": (eng.info()["kernel_launches"] - l0) / max(len(times), 1),
                "ids_equal_one_shot_prefix": bool(np.array_equal(live_ids[:max(len(live_ids) - 40, 0)], ids[:max(len(live_ids) - 40, 0)])),
                "note": "host wall time per vox_stream_feed + vox_stream_get of 1600 samples, continuous mode.  The id comparison with the "
                        "one-shot pass is informative only (the encoder runs through different kernels per call shape: f32 rounding); "
                        "parity of the live path is tests/test_gpu_stream_scenarios.py against the reference's own 0.1-s trace"}

    # ---- one long recording, encoder sharded over the ranks (N > 1)
    sharded = None
    if world > 1 and extra:
        sharded = sharded_encoder_leg(vb, eng, dist, rank, world, local, multi, args.sharded_seconds)

    if rank == 0:
        phase("live leg done")
        cpu = reference_sample(model, args.seconds) if (world == 1 and extra) else None
        phase("host reference sample done")
        traffic, traffic_src = ncu_traffic()
        line = {
            "metric": "real-time factor (audio-s/wall-s)", "value": value, "unit": "x real-time", "n_gpus": n_gpus,
            "steps": args.steps, "warmup": n_warm, "ms_per_step": dev_ms / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32 activations x bf16 weights, f32 accumulate", "data": "synthetic",
            "config": {"workload": workload, "streams": world, "mel_frames": counts["mel_frames"],
                       "adapter_tokens": counts["adapter_tokens"], "decoder_steps": int(n_dec),
                       "weights": "seeded synthetic checkpoint (no network for the real one; throughput is weight-agnostic)",
                       "l2_policy": "inputs larger than L2: every step streams 6.86 GB of weights (L2 = 126 MB)"},
            "decoder_tok_s": (dsteps / (dms / 1e3)) * world if dms else None,
            "decode_ms_per_step": step_ms,
            "encoder_positions_per_s": ((i_after["total_encoder_positions"] - i_before["total_encoder_positions"]) /
                                        max((i_after["total_encoder_ms"] - i_before["total_encoder_ms"]) / 1e3, 1e-9)),
            "encoder": encoder_block((i_after["total_encoder_positions"] - i_before["total_encoder_positions"]) /
                                     max((i_after["total_encoder_ms"] - i_before["total_encoder_ms"]) / 1e3, 1e-9)),
            "load_s": load_s, "load_s_library": eng.info()["load_ms"] / 1e3,
            "gpu_launches": int(i_after["kernel_launches"] - i_before["kernel_launches"]),
            "clocks": sampler.summary(),
            "e2e": {"value": e2e_value, "unit": "x real-time", "h2d_bytes_per_step": int(pcm.nbytes),
                    "d2h_bytes_per_step": int(4 * n_dec)},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic, "traffic_source": traffic_src,
                         "kernel": "k_dec_v2<1>: persistent decode kernel, one step = 26 layers of GEMV + attention + logits GEMV",
                         "bytes_per_step": bytes_per_step, "peak_source": peak_src},
            "cpu_baseline": ({"value": cpu["rtf"], "unit": "x real-time", "cores": cpu["cores"], "kind": "reference",
                              "sample": cpu["sample"], "decoder_tok_s": cpu["tok_s"], "extrapolated": True,
                              "measured": cpu["measured"]} if cpu else None),
            "tokens_equal_between_legs": bool(np.array_equal(ids, ids2)),
            "parity_prefix_ok": parity_ok, "parity_prefix": parity,
            "multistream": ms_block,
            "live": live,
            "sharded_encoder": sharded,
        }
        print(json.dumps(line))
    eng.dev_free(d_pcm)
    eng.close()
    if dist is not None:
        dist.destroy_process_group()


def dump_outputs(out_dir, ids, counts):
    """The arrays vox_stream_* hands its caller for the benchmarked recording: the greedy token ids and the unit counts
    (mel frames, adapter tokens, decoder steps).  Integers, stored as float64 (exact)."""
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "token_ids.npy"), np.asarray(ids, dtype=np.float64))
    np.save(os.path.join(out_dir, "counts.npy"),
            np.array([counts["mel_frames"], counts["adapter_tokens"], counts["decoder_steps"]], dtype=np.float64))


def sharded_encoder_leg(vb, eng, dist, rank, world, local, multi, seconds):
    """One `seconds`-long recording: every rank encodes its slice (vox_cuda_encode_sharded, host C + NCCL), rank 0 also runs the
    same call unsharded on a forked context and checks adapter rows + a decoded prefix.  Returns the JSON block (rank 0)."""
    import torch
    L = vb.lib()
    fp = C.POINTER(C.c_float)
    if rank == 0:
        ensure_inputs(seconds)
    dist.barrier()
    _, pcm = ensure_inputs(seconds)
    uid = torch.zeros(128, dtype=torch.uint8)
    if rank == 0:
        buf = (C.c_char * 128)()
        assert L.vox_cuda_dist_unique_id(buf) == 0
        uid = torch.frombuffer(bytearray(buf.raw), dtype=torch.uint8).clone()
    uid = uid.cuda(local)
    dist.broadcast(uid, 0)
    raw = bytes(uid.cpu().tolist())
    assert L.vox_cuda_dist_init(eng.ctx, rank, world, raw) == 0

    def encode(ctx):
        d_ad = C.c_void_p(); T = C.c_int(); P = C.c_int(); ms = C.c_double()
        rc = L.vox_cuda_encode_sharded(ctx, pcm.ctypes.data_as(fp), pcm.size, C.byref(d_ad), C.byref(T), C.byref(P), C.byref(ms))
        assert rc == 0
        return d_ad, T.value, P.value, ms.value

    encode(eng.ctx)                                            # warm-up
    dist.barrier()
    d_ad, T, P, ms = encode(eng.ctx)
    ms_max = multi.reduce_max([ms], dist, torch.device("cuda", local))[0]
    block = None
    if rank == 0:
        f = eng.fork()                                         # a context without a communicator: the same call, unsharded
        encode(f.ctx)
        d1, T1, P1, ms1 = encode(f.ctx)
        a = np.empty((T, 3072), np.float32); b = np.empty((T1, 3072), np.float32)
        L.vox_cuda_memcpy_d2h(eng.ctx, a.ctypes.data_as(C.c_void_p), d_ad, a.nbytes)
        L.vox_cuda_memcpy_d2h(f.ctx, b.ctypes.data_as(C.c_void_p), d1, b.nbytes)
        n_ids = 256
        ids_s = np.zeros(n_ids, np.int32); ids_1 = np.zeros(n_ids, np.int32)
        ip = C.POINTER(C.c_int)
        g_s = L.vox_cuda_decode_adapter(eng.ctx, d_ad, T, ids_s.ctypes.data_as(ip), n_ids)
        g_1 = L.vox_cuda_decode_adapter(f.ctx, d1, T1, ids_1.ctypes.data_as(ip), n_ids)
        block = {"seconds": seconds, "positions": P, "adapter_tokens": T, "ranks": world,
                 "encode_ms": ms_max, "encode_ms_1gpu": ms1, "speedup_vs_1": ms1 / ms_max, "efficiency": ms1 / ms_max / world,
                 "positions_per_s": P / (ms_max / 1e3),
                 "collective": "ncclSend/ncclRecv of the last 750 K and V rows to the right neighbour in every layer + one ncclAllGather of the adapter rows, on the engine's stream (host C, vb_dist.c)",
                 "adapter_max_abs_diff_vs_unsharded": float(np.abs(a - b).max()) if T == T1 else None,
                 "adapter_scale": float(np.abs(b).max()),
                 "ids_prefix_equal_unsharded": bool(g_s == g_1 and np.array_equal(ids_s[:g_s], ids_1[:g_1])), "ids_prefix_len": int(g_s)}
        f.close()
    dist.barrier()
    return block


if __name__ == "__main__":
    main()
