#!/usr/bin/env python
"""bench.py -- headline benchmark of the hot path (contract in the task brief / DESIGN.md §Measurement).

A "step" is one pass of the hot path over one batch of synthetic input: stage-1 synthesis of
`utts_per_gpu` utterances (BASELINE.json configs[1]: T=48 prompt, 750 new tokens = 5.0 s of audio,
top_p 0.95, guidance 3.0, temperature 1.0, bf16 weights + bf16 KV cache) on every GPU.

  value  : whole-job stage-1 tokens/s with inputs already resident in HBM (prefill + decode on device)
  e2e    : same metric through the reference-facing plugin call mvb_s1_generate with HOST buffers
           (prompt/speaker host->device, tokens device->host inside the timed region)
  roofline: the persistent fused decode kernel (one launch = a burst of decode positions incl. the on-device sampler),
            algorithmic bytes / CUDA-event time vs measured HBM peak
  cpu_baseline: the reference's own CPU code (oracle/_ref, vendored by oracle/build_ref.py) timed on this box's host
            cores on a bounded sample; falls back to the oracle port only when oracle/_ref is absent
  configs : the other BASELINE configurations on the same engine (batch 8 mixed-length, 6 x 10 s long-form batch)

`--impl reference` times the reference's CPU implementation on the same metric; under torchrun only rank 0 runs it.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "metavoice-src_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402
import torch  # noqa: E402

T_PROMPT, N_NEW = 48, 750
MIX_LENS = [24, 32, 48, 64, 80, 96, 112, 120]      # BASELINE configs[2]: batch 8, mixed-length prompts (SURVEY.md 8d)
LONG_UTTS, LONG_T, LONG_NEW = 6, 64, 1500          # BASELINE configs[3]: 60 s = 6 chunks x 10 s submitted as one batch
SAMPLING = dict(guidance_scale=3.0, temperature=1.0, top_p=0.95)
W_BYTES = 2_476_953_600            # stage-1 weight bytes streamed per decode step (SURVEY.md §8d)
KV_BYTES_PER_POS = 393_216         # K+V bytes per cached position per utterance (2 CFG rows, 24 layers, bf16)


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(path):
        try:
            j = json.load(open(path))
            return float(j["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def measured_tensor_peak():
    """Dense bf16 TFLOP/s: the sustained figure of MEASURED_PEAKS.json (kernels timed inside a long step), else the recipe's fallback."""
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(path):
        try:
            return float(json.load(open(path))["bf16_tflops_sustained"]), "measured (MEASURED_PEAKS.json bf16_tflops_sustained)"
        except Exception:
            pass
    return 1590.0, "fallback (B200_PROFILING.md 1.59 PFLOP/s bf16)"


class ClockSampler:
    """nvidia-smi clocks/throttle reasons sampled DURING the timed region."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None
        return self

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def __exit__(self, *a):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                pass

    def summary(self):
        sm, mx, reasons = [], 0.0, set()
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx = max(mx, float(r[1]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                continue
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx or None, "reasons": sorted(reasons),
                "samples": len(sm)}


def build_engine(device, utts, rank, world):
    from mvb200 import synth
    from mvb200.fast_model import ModelArgs, Transformer, pack_arena
    d = synth.FULL
    cfg = ModelArgs.from_name("metavoice-1B")
    t0 = time.time()
    arena = offsets = None
    if rank == 0:
        arena, offsets = pack_arena(synth.stage1_state_dict(d, 0), d.n_layer)
        arena = arena.to(device)
    bcast_ms = None
    if world > 1:
        from mvb200.distributed import broadcast_arena
        arena, offsets, bcast_ms = broadcast_arena(arena, offsets, device)   # the ONE collective of the path: NCCL over NVLink
    model = Transformer(cfg, arena, offsets, device=device)
    model.setup_spk_cond_mask()
    model.setup_caches(2 * utts, cfg.block_size, kv_dtype="bf16")
    return model, time.time() - t0, bcast_ms


def resident_pass(model, d_idx, d_spk, lens, n_new, seed):
    """Prefill + decode with inputs already in HBM; returns tokens generated (device time is measured by the caller)."""
    import ctypes as C
    from mvb200 import _lib
    lib, h, st = model._lib, model.handle, model._stream()
    utts = len(lens)
    for u in range(utts):
        sp = _lib.Sampling(SAMPLING["guidance_scale"], SAMPLING["temperature"], SAMPLING["top_p"], 0, 9999, seed + u)
        _lib.check(lib.mvb_s1_set_speaker(h, u, d_spk[u].data_ptr(), st))
        _lib.check(lib.mvb_s1_begin(h, u, -1, 0, C.byref(sp), None, None, st))
        _lib.check(lib.mvb_s1_forward(h, u, d_idx[u].data_ptr(), lens[u], 0, None, 0, st))
    # decode() = n_new x (body, sampler) in ONE persistent launch.  Its first body replays the last prefill position
    # (idempotent cache write) so that the first token is sampled from the prefill logits exactly as generate() does (utils:211).
    _lib.check(lib.mvb_s1_decode(h, utts, n_new, st))
    return utts * n_new


def tokens_generated(model, utts):
    """n_gen of every utterance as the device recorded it (checked once per leg, outside the timed region)."""
    import ctypes as C
    from mvb200 import _lib
    out = []
    for u in range(utts):
        n, d = C.c_int32(0), C.c_int32(0)
        _lib.check(model._lib.mvb_s1_fetch(model.handle, u, None, 0, C.byref(n), C.byref(d), model._stream()))
        out.append(int(n.value))
    return out


def generated_tokens(model, utts, n_new):
    """The token ids the last decode left in every utterance slot, as mvb_s1_fetch hands them to a caller: int32 [utts, n_new]."""
    import ctypes as C
    from mvb200 import _lib
    out = np.zeros((utts, n_new), np.int32)
    for u in range(utts):
        n, d = C.c_int32(0), C.c_int32(0)
        _lib.check(model._lib.mvb_s1_fetch(model.handle, u, out[u].ctypes.data_as(C.c_void_p), n_new, C.byref(n), C.byref(d),
                                           model._stream()))
    return out


def step_roofline(model, lens, n_new, reps, device):
    """One persistent launch of `reps` decode positions around the middle of the utterance (CUDA events on the launching
    stream): algorithmic bytes = reps x weights + K/V of every cached position read + the appended position written."""
    import ctypes as C
    from mvb200 import _lib
    utts = len(lens)
    lib, h, st = model._lib, model.handle, model._stream()
    starts = [T + n_new // 2 - reps // 2 for T in lens]
    for u in range(utts):
        sp = _lib.Sampling(3.0, 1.0, 0.95, 0, 9999, 5 + u)
        _lib.check(lib.mvb_s1_begin(h, u, 100 + u, starts[u], C.byref(sp), None, None, st))
    _lib.check(lib.mvb_s1_decode(h, utts, 8, st))                      # warm
    for u in range(utts):
        sp = _lib.Sampling(3.0, 1.0, 0.95, 0, 9999, 5 + u)
        _lib.check(lib.mvb_s1_begin(h, u, 100 + u, starts[u], C.byref(sp), None, None, st))
    torch.cuda.synchronize(device)
    r0, r1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    r0.record()
    _lib.check(lib.mvb_s1_decode(h, utts, reps, st))
    r1.record()
    torch.cuda.synchronize(device)
    ms = r0.elapsed_time(r1)
    nbytes = 0
    for i in range(reps):
        nbytes += W_BYTES + sum(KV_BYTES_PER_POS * (s0 + i) + KV_BYTES_PER_POS for s0 in starts)
    return ms, nbytes, [s0 + reps // 2 for s0 in starts]


def ncu_traffic_per_position():
    """dram__bytes_read.sum + dram__bytes_write.sum of the persistent kernel per decode position, from the committed
    `ncu --set full` capture of a short launch (profiles/r2_ncu_traffic.json written by tools/ncu_traffic.py)."""
    path = os.path.join(ROOT, "profiles", "r2_ncu_traffic.json")
    try:
        return json.load(open(path))
    except Exception:
        return None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="mvb200", choices=["mvb200", "reference"])
    ap.add_argument("--utts-per-gpu", type=int, default=1)
    ap.add_argument("--skip-cpu-baseline", action="store_true")
    ap.add_argument("--skip-pipeline", action="store_true")
    ap.add_argument("--skip-configs", action="store_true", help="skip the batch-8 / long-form legs (BASELINE configs[2], [3])")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the token ids of the last timed step to DIR/stage1_tokens.npy "
                                                          "(float32 [utts-per-gpu, 750]; one file per rank when --gpus > 1)")
    a = ap.parse_args()
    if a.steps < 1 or a.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))

    if a.impl == "reference":
        if rank == 0:
            print(json.dumps(reference_arm(a)))
        return

    assert torch.cuda.is_available(), "bench.py needs a GPU (there is no CPU fallback)"
    device = torch.device(f"cuda:{local}")
    torch.cuda.set_device(device)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=device)
    utts = a.utts_per_gpu
    slots = utts if a.skip_configs else max(utts, len(MIX_LENS))
    model, build_s, bcast_ms = build_engine(device, slots, rank, world)
    from mvb200 import synth, fast_inference_utils as U

    def inputs(lens, base):
        pr = [synth.synthetic_prompt(T, seed=base + rank * 64 + u) for u, T in enumerate(lens)]
        sp = torch.cat([synth.synthetic_speaker(seed=base + 4 + rank * 64 + u) for u in range(len(lens))])
        return pr, sp, [q.view(1, -1).repeat(2, 1).to(device).contiguous() for q in pr], [sp[u].to(device).contiguous() for u in range(len(lens))]

    lens = [T_PROMPT] * utts
    prompts, spk, d_idx, d_spk = inputs(lens, 7)
    h_spk_pinned = spk.pin_memory()

    def barrier():
        torch.cuda.synchronize(device)
        if world > 1:
            import torch.distributed as dist
            dist.barrier()
        torch.cuda.synchronize(device)

    def timed_resident(lens_, d_idx_, d_spk_, n_new, steps, warmup, seed0):
        for w in range(warmup):
            resident_pass(model, d_idx_, d_spk_, lens_, n_new, seed0 + w)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        toks = 0
        for k in range(steps):
            toks += resident_pass(model, d_idx_, d_spk_, lens_, n_new, seed0 + 100 + k)
        e1.record()
        barrier()
        assert tokens_generated(model, len(lens_)) == [n_new] * len(lens_)
        return toks, e0.elapsed_time(e1)

    # ---- HBM-resident value ------------------------------------------------------------------
    for w in range(a.warmup):
        resident_pass(model, d_idx, d_spk, lens, N_NEW, 1000 + w)
    barrier()
    lc0 = model._lib.mvb_s1_launch_count(model.handle)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local) as clk:
        e0.record()
        toks = 0
        for k in range(a.steps):
            toks += resident_pass(model, d_idx, d_spk, lens, N_NEW, 2000 + k)
        e1.record()
        barrier()
    launches = model._lib.mvb_s1_launch_count(model.handle) - lc0
    ms = e0.elapsed_time(e1)
    assert tokens_generated(model, utts) == [N_NEW] * utts
    if a.dump_outputs:
        os.makedirs(a.dump_outputs, exist_ok=True)
        name = "stage1_tokens" if world == 1 else f"stage1_tokens_rank{rank}"
        np.save(os.path.join(a.dump_outputs, name + ".npy"), generated_tokens(model, utts, N_NEW).astype(np.float32))

    # ---- decode roofline: one persistent launch of `reps` positions at mid-utterance context ----
    reps = 200
    launch_ms, launch_bytes, mids = step_roofline(model, lens, N_NEW, reps, device)
    peak, peak_src = measured_peaks()
    achieved = launch_bytes / (launch_ms * 1e-3) / 1e9
    ncu = ncu_traffic_per_position()

    # ---- e2e through the host-buffer plugin call ---------------------------------------------
    for w in range(max(1, a.warmup // 2)):
        U.generate_batch(model, prompts, h_spk_pinned, max_new_tokens=N_NEW, end_of_audio_token=9999, seed=3000 + w, **SAMPLING)
    barrier()
    t0 = time.perf_counter()
    e2e_toks = 0
    for k in range(a.steps):
        out = U.generate_batch(model, prompts, h_spk_pinned, max_new_tokens=N_NEW, end_of_audio_token=9999, seed=4000 + k,
                               **SAMPLING)
        e2e_toks += sum(len(o) for o in out)
    barrier()
    e2e_s = time.perf_counter() - t0

    # ---- the other BASELINE configurations on the same engine (device-timed, max over ranks) -----
    cfg_times, cfg_info = [], {}
    if not a.skip_configs:
        # configs[2] / configs[4]: 8 mixed-length prompts per GPU, 750 tokens each, top-p sampling
        pr8, sp8, di8, ds8 = inputs(MIX_LENS, 31)
        t8, ms8 = timed_resident(MIX_LENS, di8, ds8, N_NEW, 2, 1, 6000)
        l8_ms, l8_bytes, l8_mid = step_roofline(model, MIX_LENS, N_NEW, 100, device)
        cfg_times.append(ms8)
        cfg_info["batch8_mixed"] = {"workload": f"BASELINE configs[2]/[4]: {len(MIX_LENS)} utterances per GPU, prompts {MIX_LENS}, {N_NEW} tokens each, top_p 0.95",
                                    "tokens_per_rank": t8, "roofline_frac": round(l8_bytes / (l8_ms * 1e-3) / 1e9 / peak, 4),
                                    "ms_per_position": round(l8_ms / 100, 4), "context_len_mid": l8_mid}
        if world == 1:
            # configs[3]: 60 s of speech = 6 chunks x 10 s (T=64, 1500 tokens each) submitted as one batch
            ll = [LONG_T] * LONG_UTTS
            prl, spl, dil, dsl = inputs(ll, 51)
            tl, msl = timed_resident(ll, dil, dsl, LONG_NEW, 1, 1, 7000)
            cfg_info["longform_60s"] = {"workload": f"BASELINE configs[3]: {LONG_UTTS} chunks x {LONG_NEW} tokens (10 s each), T={LONG_T}, one batch on 1 GPU",
                                        "value": round(tl / (msl * 1e-3), 1), "unit": "tokens/s",
                                        "audio_sec_per_s_stage1": round(tl / (msl * 1e-3) / 150.0, 2), "ms_total": round(msl, 1)}

    # ---- whole implemented pipeline (host text-side inputs -> wav on host) ------------------------------------------
    pipe = None
    if not a.skip_pipeline:
        pipe = pipeline_leg(model, prompts, spk, h_spk_pinned, utts, a.steps, device, world, barrier)

    times = torch.tensor([ms, e2e_s * 1e3] + cfg_times, dtype=torch.float64, device=device)
    if world > 1:
        import torch.distributed as dist
        dist.all_reduce(times, op=dist.ReduceOp.MAX)
    tl_ = [float(x) for x in times.cpu()]
    ms_max, e2e_ms_max = tl_[0], tl_[1]
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if rank != 0:
        return
    if "batch8_mixed" in cfg_info:
        c = cfg_info["batch8_mixed"]
        c["value"] = round(c.pop("tokens_per_rank") * world / (tl_[2] * 1e-3), 1)
        c["unit"] = "tokens/s"
        c["audio_sec_per_s_stage1"] = round(c["value"] / 150.0, 2)
    total_toks = toks * world
    value = total_toks / (ms_max * 1e-3)
    line = {
        "metric": "stage1_tok_per_s", "value": round(value, 2), "unit": "tokens/s", "n_gpus": world, "steps": a.steps,
        "warmup": a.warmup, "ms_per_step": round(ms_max / a.steps, 3), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "bf16 weights+KV, fp32 accumulate", "data": "synthetic (seeded random-init checkpoint in the reference layout)",
        "audio_sec_per_s_stage1": round(value / 150.0, 3),
        "config": {"workload": "BASELINE configs[1] stage-1: 1.2B causal LM, T=48 prompt, 750 new tokens (5.0 s audio), "
                               "top_p=0.95 guidance=3.0 temperature=1.0, CFG pair per utterance",
                   "utts_per_gpu": utts, "parallelism": f"replicas x{world}, utterances sharded, weights NCCL-broadcast at init",
                   "l2": "not flushed: 2.48 GB of weights are streamed every token (>> 126 MB L2)",
                   "stage2_vocoder_in_timed_region": False},
        "e2e": {"value": round(e2e_toks * world / (e2e_ms_max * 1e-3), 2), "unit": "tokens/s",
                "h2d_bytes_per_step": int(utts * (T_PROMPT * 4 * 2 + 256 * 4 + 32)), "d2h_bytes_per_step": int(utts * (N_NEW * 4 + 8))},
        "gpu_launches": int(launches),
        "roofline": {"bound": "hbm",
                     "kernel": f"k_decode_persistent: ONE launch = {reps} decode positions (24 x {{qkv, attention, wo, w1|w3, w2}} + head + on-device sampler each)",
                     "achieved": round(achieved, 1), "peak": peak, "peak_source": peak_src, "unit": "GB/s",
                     "frac": round(achieved / peak, 4),
                     "traffic": (int(ncu["dram_bytes_per_position"] * reps) if ncu else None),
                     "traffic_source": (ncu.get("source") if ncu else None),
                     "bytes_per_launch": int(launch_bytes), "ms_per_launch": round(launch_ms, 3),
                     "positions_per_launch": reps, "ms_per_position": round(launch_ms / reps, 4), "context_len_mid": mids[0]},
        "clocks": clk.summary(),
        "init": {"build_s": round(build_s, 2), "nccl_broadcast_ms": bcast_ms},
        "configs": cfg_info or None,
        "pipeline": pipe,
    }
    if not a.skip_cpu_baseline and world == 1:   # reported at N=1 only (rank 0 would otherwise hold the other ranks' cores)
        line["cpu_baseline"] = cpu_baseline()
    print(json.dumps(line))


def pipeline_leg(model, prompts, spk, h_spk_pinned, utts, steps, device, world, barrier):
    """Host text-side inputs -> wav BYTES on the host: stage-1 -> adapters -> stage-2 -> EnCodec decoder -> multi-band
    diffusion (parametrised config, parity unpinned) -> on-device loudness normalisation / compressor / PCM16.  Reports
    audio-seconds per second with per-stage milliseconds; DeepFilterNet (fast_inference.py:158-163) is NOT implemented."""
    from mvb200 import audio_out as A, synth, fast_inference_utils as U
    from mvb200.mbd import MBDSettings, MultiBandDiffusionEngine
    from mvb200.second_stage import SecondStage, flattened_interleaved_decode
    from mvb200.vocoder import EncodecDecodeEngine
    s2 = SecondStage(synth.stage2_checkpoint(synth.S2_FULL, 1), device=device, max_batch=1)
    codec = EncodecDecodeEngine(synth.encodec_model_and_state_dict(0)[1], device=device, max_frames=1024)
    mbd_cfg = MBDSettings()                 # hidden 48, depth 4, growth 4, k 8 / s 4, 4 band models x 20 calls, 32-band re-EQ
    mbd = MultiBandDiffusionEngine(synth.mbd_checkpoint(mbd_cfg, 0), mbd_cfg, device=device, max_seconds=6.0)
    frames = N_NEW // 2
    text_ids = torch.randint(1025, 1537, (11,), generator=torch.Generator().manual_seed(5)).tolist() + [1537]

    def pipeline_pass(seed):
        t_a = time.perf_counter()
        toks = U.generate_batch(model, prompts, h_spk_pinned, max_new_tokens=N_NEW, end_of_audio_token=9999, seed=seed, **SAMPLING)
        t_b = time.perf_counter()
        secs, t_s2, t_voc, t_mbd, t_post, nbytes = 0.0, 0.0, 0.0, 0.0, 0.0, 0
        for u in range(utts):
            _, cb = flattened_interleaved_decode(toks[u].tolist())
            cb = [(c + [7] * frames)[:frames] for c in cb]   # random-init weights do not alternate codebooks: pad/cut to 375 frames
            t0 = time.perf_counter()
            idx = s2.build_input(text_ids, cb)[None]
            codes8 = torch.cat([idx[0, :, len(text_ids):len(text_ids) + frames].to(device),
                                s2.forward_tokens(idx, spk[u:u + 1], 1.0, 200, seed=seed)[0, :, len(text_ids):len(text_ids) + frames]])
            codes8 = codes8.clamp_(0, 1023)
            torch.cuda.synchronize(device); t1 = time.perf_counter()
            wav = codec.decode(codes8)
            cond = codec.decode_latent(codes8)
            torch.cuda.synchronize(device); t2 = time.perf_counter()
            wav = mbd.tokens_to_wav(cond, wav, seed=seed)
            torch.cuda.synchronize(device); t3 = time.perf_counter()
            blob = A.wav_bytes_on_device(wav, 24000)          # loudness -14 LUFS + tanh compressor + PCM16 on device, bytes to host
            t4 = time.perf_counter()
            secs += wav.numel() / 24000.0; t_s2 += t1 - t0; t_voc += t2 - t1; t_mbd += t3 - t2; t_post += t4 - t3; nbytes += len(blob)
        return secs, t_b - t_a, t_s2, t_voc, t_mbd, t_post

    pipeline_pass(1)
    barrier()
    t0 = time.perf_counter()
    acc = [0.0] * 6
    for k in range(steps):
        r = pipeline_pass(5000 + k)
        acc = [a + b for a, b in zip(acc, r)]
    barrier()
    pipe_s = time.perf_counter() - t0
    audio_s, s1_s, s2_s, voc_s, mbd_s, post_s = acc
    # rooflines of the downstream stages (one utterance): stage-2 streams its bf16 weights once per forward (HBM-bound);
    # the SEANet decoder is fp32 CUDA-core work; the diffusion UNets are tcgen05 GEMM work (bf16 taps, two-term activations)
    hbm_peak, tensor_peak = measured_peaks()[0], measured_tensor_peak()[0]
    n_u = steps * utts
    s2_bytes = sum(v.numel() for k, v in synth.stage2_checkpoint(synth.S2_FULL, 1)["model"].items() if v.ndim == 2) * 2
    s2_gbs = s2_bytes / (s2_s / n_u) / 1e9
    voc_tf = 2 * codec.flops(frames) / (voc_s / n_u) / 1e12      # decode() + decode_latent() per utterance ~ 1 decoder pass + lookup
    mbd_tf = mbd.flops(frames * 320, frames) / (mbd_s / n_u) / 1e12
    stage_rooflines = {
        "stage2": {"bound": "hbm", "achieved": round(s2_gbs, 1), "peak": hbm_peak, "unit": "GB/s", "frac": round(s2_gbs / hbm_peak, 4),
                   "note": "bf16 weight bytes of one non-causal forward / wall time of build_input + forward + sampling (launch-bound at T = 387)"},
        "encodec_decoder": {"bound": "fp32", "achieved": round(voc_tf / 2, 2), "unit": "TFLOP/s",
                            "note": "fp32 FMA FLOPs of the SEANet decoder / wall time of decode + decode_latent"},
        "multiband_diffusion": {"bound": "tensor", "achieved": round(mbd_tf, 1), "peak": tensor_peak, "unit": "TFLOP/s",
                                "frac": round(mbd_tf / tensor_peak, 4),
                                "note": "algorithmic conv FLOPs of 80 UNet passes / wall time of tokens_to_wav (the two-term activation split "
                                        "doubles the issued MMA work; GroupNorm, transposes, FIR banks and the level-0 CUDA-core convs are in the time)"}}
    mbd.close(); codec.close(); s2.close()
    u = mbd_cfg.unet
    return {"audio_sec_per_s": round(audio_s * world / pipe_s, 3),
            "audio_sec_per_s_without_mbd": round(audio_s * world / (pipe_s - mbd_s), 3),
            "audio_s_per_step": round(audio_s / steps, 3),
            "ms_per_step": {"total": round(pipe_s / steps * 1e3, 2), "stage1": round(s1_s / steps * 1e3, 2), "stage2": round(s2_s / steps * 1e3, 2),
                            "encodec_decoder": round(voc_s / steps * 1e3, 2), "multiband_diffusion": round(mbd_s / steps * 1e3, 2),
                            "audio_post_pcm16": round(post_s / steps * 1e3, 2)},
            "mbd_config": f"PARAMETRISED, parity unpinned: {mbd_cfg.n_models} band UNets (hidden {u.hidden}, depth {u.depth}, growth {u.growth}, "
                          f"k{u.kernel}/s{u.stride}, {u.res_blocks} res block) x {len(mbd_cfg.steps()) - 1} calls, {mbd_cfg.eq_bands}-band re-EQ; "
                          "convolutions with >= 32 input channels on tcgen05 (bf16 taps, two-term bf16 activations, fp32 accumulate), the 1-channel input conv and the 1x1 condition conv on fp32 CUDA cores",
            "stage_rooflines": stage_rooflines,
            "coverage": "stage-1 (750 tokens) + token adapters + stage-2 (6 codebooks) + EnCodec SEANet decoder + multi-band diffusion "
                        "+ loudness/compressor/PCM16 on device, wav bytes on the host; DeepFilterNet is NOT implemented"}


def _oracle_stage1(dtype):
    from mvb200 import synth
    from oracle import stage1_port as P
    d = synth.FULL
    m = P.Stage1Oracle(synth.stage1_state_dict(d, 0), d.n_head, d.norm_eps, dtype, faithful_full_cache=True)
    m.setup_caches()
    return m


def effective_cores() -> int:
    """Host threads this process may really use: min(affinity mask, cgroup CPU quota).  On the GPU box nproc says 128
    but the container quota is 16 CPUs; oversubscribing makes torch's CPU kernels ~500x slower."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            n = min(n, max(1, int(float(q) / float(per))))
    except Exception:
        pass
    return max(1, n)


def _reference_stage1():
    """The reference's OWN fast path (fam.llm.fast_model.Transformer + fam.llm.fast_inference_utils.generate, bf16 = its
    production dtype) from oracle/_ref (or /root/reference), or None when neither is present."""
    try:
        from oracle import ref_harness as R
        if not R.runnable():
            return None
        from mvb200 import synth
        fiu = R.reference_functions()
        model = R.build_reference_model(synth.stage1_state_dict(synth.FULL, 0), synth.FULL, torch.bfloat16)
        return fiu, model
    except Exception as e:   # noqa: BLE001
        sys.stderr.write(f"reference stage-1 unavailable ({e}); using the oracle port\n")
        return None


def cpu_baseline(budget_s=20.0, model=None, ref=None):
    """The reference's CPU path on all usable host threads, on a bounded sample of the same workload: its own
    generate() (prefill of the T=48 prompt + k decode steps, k sized to the time budget from a short calibration call).
    Metric = the reference's own (utils:437-438): generated tokens / wall time including the prefill."""
    from mvb200 import synth
    cores = effective_cores()
    torch.set_num_threads(cores)
    prompt, spk = synth.synthetic_prompt(T_PROMPT), synth.synthetic_speaker().to(torch.bfloat16)
    if ref is None and model is None:
        ref = _reference_stage1()
    if ref is not None:
        fiu, rmodel = ref
        kw = dict(temperature=torch.tensor(1.0, dtype=torch.bfloat16), top_p=torch.tensor(0.95, dtype=torch.bfloat16),
                  guidance_scale=torch.tensor(3.0, dtype=torch.bfloat16), top_k=None)
        with torch.no_grad():
            torch.manual_seed(1337)
            t0 = time.perf_counter()
            fiu.generate(rmodel, prompt, spk, max_new_tokens=6, end_of_audio_token=9999, **kw)     # calibration (untimed)
            per_tok = (time.perf_counter() - t0) / 6
            k = int(max(8, min(N_NEW, budget_s / max(per_tok, 1e-3))))
            t0 = time.perf_counter()
            y = fiu.generate(rmodel, prompt, spk, max_new_tokens=k, end_of_audio_token=9999, **kw)
            dt = time.perf_counter() - t0
        n = int(y.numel()) - T_PROMPT
        return {"value": round(n / dt, 3), "unit": "tokens/s", "cores": cores, "kind": "reference",
                "sample": f"the reference's own generate() (oracle/_ref, bf16, torch CPU eager): prefill T={T_PROMPT} + {n - 1} decode "
                          f"steps of the 750-token workload in {dt:.1f} s on {cores} threads (cgroup quota; nproc={os.cpu_count()})"}
    from oracle import stage1_port as P
    m = model or _oracle_stage1(torch.bfloat16)
    kw = dict(guidance_scale=torch.tensor(3.0, dtype=torch.bfloat16), temperature=torch.tensor(1.0, dtype=torch.bfloat16),
              top_p=torch.tensor(0.95, dtype=torch.bfloat16))
    torch.manual_seed(1337)
    t0 = time.perf_counter()
    with torch.no_grad():
        logits = m.forward(prompt.view(1, -1).repeat(2, 1), spk, torch.arange(T_PROMPT))
        tok, _ = P.sample(logits, **kw)
        n, pos = 1, T_PROMPT
        while time.perf_counter() - t0 < budget_s and n < N_NEW:
            logits = m.forward(tok.view(1, -1).repeat(2, 1), spk, torch.tensor([pos]))
            tok, _ = P.sample(logits, **kw)
            n += 1; pos += 1
    dt = time.perf_counter() - t0
    return {"value": round(n / dt, 3), "unit": "tokens/s", "cores": cores, "kind": "port",
            "sample": f"oracle port (oracle/_ref absent): prefill T={T_PROMPT} + {n - 1} decode steps of the 750-token workload in {dt:.1f} s, "
                      f"bf16, torch CPU ({cores} threads = cgroup quota; nproc={os.cpu_count()})"}


def reference_arm(a):
    ref = _reference_stage1()
    m = None if ref is not None else _oracle_stage1(torch.bfloat16)
    for _ in range(min(a.warmup, 1)):
        cpu_baseline(3.0, m, ref)
    t0 = time.perf_counter()
    vals = [cpu_baseline(max(4.0, 60.0 / max(a.steps, 1)), m, ref) for _ in range(a.steps)]
    dt = time.perf_counter() - t0
    v = sum(x["value"] for x in vals) / len(vals)
    cb = dict(vals[-1]); cb["value"] = round(v, 3)
    return {"impl": "reference", "metric": "stage1_tok_per_s", "value": round(v, 3), "unit": "tokens/s", "n_gpus": a.gpus,
            "steps": a.steps, "warmup": a.warmup, "ms_per_step": round(dt / a.steps * 1e3, 1), "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": "BASELINE configs[1] stage-1 (each step = a bounded sample of the 750-token utterance: prefill T=48 + decode steps sized to a fixed time budget)"},
            "cpu_baseline": cb, "e2e": {"value": round(v, 3), "unit": "tokens/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}


if __name__ == "__main__":
    main()
