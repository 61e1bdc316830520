#!/usr/bin/env python
"""Benchmark of the hot path: batched Moonshine transcription (frontend -> encoder -> greedy decoder) on B200,
with the float CPU implementation timed beside it.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--model tiny|base|..] [--batch B]
                    [--headline-only] [--dump-outputs DIR]

One "step" = one pass of the hot path over one batch of B synthetic 10 s @ 16 kHz utterances.

Headline (`value`, `e2e`, `roofline`): BASELINE.json configs[1] -- moonshine-tiny, batch 32 per GPU.
  value = whole-job utterances/s with the PCM already resident in HBM (moonshine_b200_transcribe_device);
  e2e   = the same through the reference-facing C-ABI call with HOST buffers
          (moonshine_transcribe_batch_without_streaming: segmentation, H2D, encoder, decode, D2H, detokenisation).
`configs`: the other BASELINE operating points measured the same way in the same run --
  tiny_b1 (the reference's only operating point: one utterance, latency), base_b256 (configs[2]),
  base_streaming_b64 (configs[3]); with --gpus 8 also base_b2048_8gpu (configs[4], 256 utterances per GPU).
N > 1: one process per GPU (torchrun), weights NCCL-broadcast once at init, utterances sharded, no per-step
collective; the headline stays tiny / 32 per GPU so the driver's scaling efficiency compares like with like.

--impl reference: the CPU arm -- the Hugging Face float implementation of the same model (the graphs the reference
ships were exported from it), same seeded weights and inputs, ALL host cores, the headline's batch of 32 as one
batch per step (plus the reference's own batch-1 serial operating point, reported inside `cpu_baseline`).

--dump-outputs DIR: after the timed steps, write the token ids the device-resident path returned in its last timed
step as DIR/<config>_tokens.npy (rank 0's utterances), so that two builds can be compared output for output: the
weights and the audio are seeded, so the inputs are the same in every run with the same arguments.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from moonshine_b200.arch import ARCHS, frontend_lengths  # noqa: E402
from moonshine_b200.weights import pack_msw, synth_audio, synth_tokenizer_bin, synth_weights  # noqa: E402

N_SAMPLES = 160000  # 10 s @ 16 kHz
PUBLISHED = {"value_ms_per_10s_clip": 161.0, "source": "reference docs/word-level-timestamps.md:201 (tiny, shipped int8 ORT "
             "graphs, unnamed machine) = 6.2 utt/s; quoted for context, not measured here"}


def decoder_step_bytes(d, B, T, t, e_w=4, e_cross=2, e_self=4):
    """Algorithmic HBM bytes of ONE decoder-step launch at decode position t (BASELINE.md section 3 formula with this
    build's element sizes: fp32-equivalent weights (bf16 hi + lo planes), fp16 cross K/V, fp32 self K/V)."""
    D, I, L, V = d.dim, d.ffn, d.dec_layers, d.vocab
    p_step = L * (3 * D * D + D * D + D * D + D * D + 2 * I * D + 2 * I + I * D + D + 3 * D) + V * D + D
    cross = 2 * L * T * D
    self_r = 2 * L * t * D
    self_w = 2 * L * D
    return e_w * p_step + B * (e_cross * cross + e_self * (self_r + self_w) + 4)


def clocks_sampler(stop_evt, out):
    q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    try:
        p = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "100"],
                             stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
    except Exception:
        return

    def reader():
        for line in p.stdout:
            out.append(line.strip())
    th = threading.Thread(target=reader, daemon=True)
    th.start()
    stop_evt.wait()
    p.terminate()
    th.join(timeout=2)


def summarise_clocks(lines, dev_index):
    sm, mx, reasons = [], [], set()
    for ln in lines:
        f = [x.strip() for x in ln.split(",")]
        if len(f) < 9 or not f[0].isdigit() or int(f[0]) != dev_index:
            continue
        try:
            sm.append(float(f[1])); mx.append(float(f[2]))
        except ValueError:
            continue
        for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], f[5:9]):
            if v.lower().startswith("active"):
                reasons.add(name)
    if not sm:
        return {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
    hi = [x for x in sm if x > 0.5 * max(sm)]  # under load = samples above idle clocks
    return {"sm_mhz": float(np.median(hi)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons), "samples": len(sm)}


def host_threads():
    return int(os.environ.get("MOONSHINE_CPU_THREADS", "0")) or (os.cpu_count() or 1)


# ---------------------------------------------------------------------------------------------------------------
# CPU arm
# ---------------------------------------------------------------------------------------------------------------
def hf_arm(model, audios_serial, audios_batch, threads):
    """HF float model on `threads` cores: batch-1 serial over audios_serial, then audios_batch as ONE batch."""
    from oracle import hf_reference as hf
    import torch
    torch.set_num_threads(threads)
    weights = synth_weights(model, 0, "hf")
    m = hf.hf_model(ARCHS[model], weights)
    # the thread count that is fastest on THIS host for each shape (all cores is not: see hf.pick_threads)
    t_serial, seen_s = hf.pick_threads(m, audios_serial, threads, 1)
    s_dt, s_tok = hf.time_serial(m, audios_serial, t_serial)
    t_batch, seen_b = hf.pick_threads(m, audios_batch, threads, len(audios_batch))
    b_dt, b_tok = hf.time_batched(m, audios_batch, t_batch)
    return {"serial_s_per_utt": s_dt / len(audios_serial), "serial_utt_s": len(audios_serial) / s_dt,
            "serial_n": len(audios_serial), "batched_utt_s": len(audios_batch) / b_dt, "batched_n": len(audios_batch),
            "batched_s": b_dt, "tokens_serial": s_tok, "tokens_batched": b_tok, "model": m,
            "threads_serial": t_serial, "threads_batched": t_batch,
            "threads_tried": {"serial": {str(k): round(v, 3) for k, v in seen_s.items()},
                              "batched": {str(k): round(v, 3) for k, v in seen_b.items()}}}


def numpy_port_utt_s(model, audio, threads):
    """Cross-check only: the numpy oracle on one utterance (BLAS threads capped: more makes it slower)."""
    from oracle.moonshine_oracle import Dims, Oracle
    try:
        from threadpoolctl import threadpool_limits
        ctx = threadpool_limits(limits=min(threads, 16))
    except Exception:  # pragma: no cover
        import contextlib
        ctx = contextlib.nullcontext()
    with ctx:
        o = Oracle(Dims.from_product(ARCHS[model]), synth_weights(model, 0, "hf"))
        t0 = time.perf_counter()
        toks = o.greedy(audio, keep_logits=False)[0]
        return 1.0 / (time.perf_counter() - t0), toks


def run_reference(args):
    """--impl reference.  The reference's own ORT graphs / weights are not in the tree (SURVEY.md section 0), so the
    CPU arm is the HF float implementation they were exported from: same seeded weights, same inputs, same metric,
    the headline's batch as one batch per step, all host cores."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    model, B, threads = args.model, args.batch, host_threads()
    audios = [synth_audio(i, N_SAMPLES) for i in range(B)]
    try:
        from oracle import hf_reference as hf
        import torch
        torch.set_num_threads(threads)
        m = hf.hf_model(ARCHS[model], synth_weights(model, 0, "hf"))
        kind_note = "Hugging Face transformers MoonshineForConditionalGeneration, fp32, eager attention, KV cache"
        cores = threads
        threads, seen_b = hf.pick_threads(m, audios, cores, len(audios))   # warm-up included
        for _ in range(max(0, min(args.warmup, 2) - 1)):
            hf.time_batched(m, audios[:4], threads)
        t0 = time.perf_counter()
        for _ in range(args.steps):
            hf.time_batched(m, audios, threads)
        dt = time.perf_counter() - t0
        t_serial, seen_s = hf.pick_threads(m, audios, cores, 1)
        serial_dt, _ = hf.time_serial(m, audios[:3], t_serial)
        serial = {"serial_batch1_s_per_utt": serial_dt / 3, "serial_batch1_utt_s": 3 / serial_dt, "serial_threads": t_serial,
                  "threads_tried_s_per_short_sample": {"batched": {str(k): round(v, 3) for k, v in seen_b.items()},
                                                       "serial": {str(k): round(v, 3) for k, v in seen_s.items()}}}
    except Exception as e:  # transformers missing on the box: fall back to the numpy port, say so
        kind_note = f"numpy oracle port (HF arm unavailable: {type(e).__name__})"
        B = 2
        t0 = time.perf_counter()
        for _ in range(args.steps):
            for a in audios[:B]:
                numpy_port_utt_s(model, a, threads)
        dt = time.perf_counter() - t0
        serial = {}
    ups = args.steps * B / dt
    line = {
        "impl": "reference", "metric": "utterances_per_sec", "value": ups, "unit": "utt/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1000.0 * dt / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "rtf": (dt / (args.steps * B)) / 10.0,
        "config": {"workload": f"moonshine-{model}, batch={B} synthetic 10s@16kHz utterances, encoder + greedy decoder "
                               f"(configs[1] inputs and weights), CPU float implementation, one batch per step",
                   "batch": B, "weights": "seeded synthetic (HF init), fp32", "implementation": kind_note},
        "cpu_baseline": dict({"value": ups, "unit": "utt/s", "cores": threads, "kind": "port",
                              "sample": f"{args.steps} steps x {B} utterances as one batch, {threads} threads "
                                        f"(host has {os.cpu_count()} cores); {kind_note}"}, **serial),
        "published_reference": PUBLISHED,
        "e2e": {"value": ups, "unit": "utt/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ---------------------------------------------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------------------------------------------
def measured_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum per decoder-step launch, per config, from the committed ncu
    captures (profiles/r2_decoder_traffic.json, written by scripts/ncu_traffic.py on the GPU box)."""
    try:
        return json.load(open(os.path.join(ROOT, "profiles", "r2_decoder_traffic.json")))
    except Exception:
        return {}


def measure_config(api, torch, dist, model, B, steps, warmup, rank, world, local, want_e2e=True):
    """One operating point: device-resident loop (CUDA events on the library stream) + e2e loop through the ABI."""
    from moonshine_b200.dist import broadcast_bytes
    d = ARCHS[model]
    arch_enum = {"tiny": api.ModelArch.TINY, "base": api.ModelArch.BASE,
                 "tiny_streaming": api.ModelArch.TINY_STREAMING, "base_streaming": api.ModelArch.BASE_STREAMING}[model]
    # weights: rank 0 builds the container, ONE NCCL broadcast replicates it
    blob = pack_msw(model, synth_weights(model, 0, "hf")) if rank == 0 else b""
    msw = broadcast_bytes(blob, 0, device=f"cuda:{local}")
    del blob
    tr = api.Transcriber(model_arch=arch_enum, options={"vad_threshold": "0", "device": str(local), "return_audio_data": "false"},
                         memory_files={"model.msw": msw, "tokenizer.bin": synth_tokenizer_bin(d.vocab)})
    tr.set_timing(True)
    audios = [synth_audio(rank * B + i, N_SAMPLES) for i in range(B)]
    dev = torch.from_numpy(np.stack(audios)).cuda()
    lengths = [N_SAMPLES] * B
    stream = torch.cuda.ExternalStream(tr.cuda_stream_ptr(), device=torch.device("cuda", local))
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")  # > 126 MB L2

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    for _ in range(max(warmup, 1)):
        toks = tr.transcribe_device(dev.data_ptr(), N_SAMPLES, lengths)
    tm = tr.last_timings()
    launches_per_step = int(tm["kernel_launches"])
    sync_all()
    ev_ms, dec_ms, enc_ms, fe_ms, xkv_ms = [], [], [], [], []
    for _ in range(steps):
        flush.fill_(1)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        toks = tr.transcribe_device(dev.data_ptr(), N_SAMPLES, lengths)
        e1.record(stream)
        e1.synchronize()
        ev_ms.append(e0.elapsed_time(e1))
        tm = tr.last_timings()
        dec_ms.append(tm["decode_ms"]); enc_ms.append(tm["encoder_ms"])
        fe_ms.append(tm["frontend_ms"]); xkv_ms.append(tm["cross_kv_ms"])
    sync_all()
    dev_total_ms = float(sum(ev_ms))
    e2e_total = 0.0
    if want_e2e:
        for _ in range(2):
            tr.transcribe_batch_without_streaming(audios)
        sync_all()
        for _ in range(steps):
            flush.fill_(1)
            torch.cuda.synchronize()
            w0 = time.perf_counter()  # the call is synchronous (it returns the transcripts): wall clock = end to end
            tr.transcribe_batch_without_streaming(audios)
            e2e_total += time.perf_counter() - w0
        sync_all()
    t = torch.tensor([dev_total_ms, e2e_total], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)  # max over ranks
    dev_total_ms, e2e_total = [float(x) for x in t.tolist()]
    steps_run = int(tm["decode_steps"])
    dec_kernel = "decoder_step%d_kernel" % int(tm.get("decoder_version", 3) or 3)
    tr.close()
    del dev, flush
    torch.cuda.empty_cache()

    _, _, T = frontend_lengths(N_SAMPLES)
    if d.streaming:
        T = N_SAMPLES // 1280 * 4   # encoder features of the whole 1280-sample chunks (20 ms each)
    bytes_per_launch = float(np.mean([decoder_step_bytes(d, B, T, s) for s in range(max(steps_run, 1))]))
    launch_ms = float(np.mean(dec_ms)) / max(steps_run, 1)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    achieved = bytes_per_launch / (launch_ms * 1e-3) / 1e9
    utts = world * B * steps
    key = f"{model}_b{B}"
    rec = {
        "model": model, "batch_per_gpu": B, "global_batch": B * world, "steps": steps, "warmup": warmup,
        "value": utts / (dev_total_ms / 1000.0), "unit": "utt/s", "ms_per_step": dev_total_ms / steps,
        "rtf": (dev_total_ms / 1000.0) / (utts * 10.0),
        "stage_ms": {"frontend": float(np.mean(fe_ms)), "encoder": float(np.mean(enc_ms)), "cross_kv": float(np.mean(xkv_ms)),
                     "decode": float(np.mean(dec_ms)), "decode_launch_us": 1000.0 * launch_ms, "decode_steps": steps_run},
        "roofline": {"kernel": dec_kernel, "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                     "frac": achieved / peak, "traffic": measured_traffic().get(key), "bytes_per_launch": bytes_per_launch,
                     "peak_source": "MEASURED_PEAKS.json hbm_gbs" if peaks else "fallback 6650 GB/s"},
        "gpu_launches": launches_per_step * steps,
        "tokens_per_utt": float(np.mean([len(x) - 1 for x in toks])),
    }
    if want_e2e:
        rec["e2e"] = {"value": utts / e2e_total, "unit": "utt/s", "h2d_bytes_per_step": B * N_SAMPLES * 4,
                      "d2h_bytes_per_step": int(sum(len(x) for x in toks) * 4 + 4 * B), "ms_per_step": 1000.0 * e2e_total / steps,
                      "api": "moonshine_transcribe_batch_without_streaming (host PCM -> transcript_t; options vad_threshold=0, "
                             "return_audio_data=false)"}
    if B == 1:
        rec["latency_ms"] = {"device_resident": dev_total_ms / steps, "e2e": 1000.0 * e2e_total / steps if want_e2e else None}
    return rec, toks, audios


def dump_outputs(out_dir, outputs):
    """Token ids per operating point as float64 [utterances, longest], padded with -1 (ids are exact in float64)."""
    os.makedirs(out_dir, exist_ok=True)
    for name, toks in outputs.items():
        a = np.full((len(toks), max(len(t) for t in toks)), -1.0)
        for i, t in enumerate(toks):
            a[i, :len(t)] = t
        np.save(os.path.join(out_dir, f"{name}_tokens.npy"), a)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--model", default="tiny")
    ap.add_argument("--batch", type=int, default=32)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--headline-only", action="store_true", help="skip the other BASELINE configs")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the token ids of each config's last timed step to DIR/<config>_tokens.npy")
    args = ap.parse_args()
    if args.impl == "reference" and args.dump_outputs:
        ap.error("--dump-outputs applies to the GPU path")
    if args.impl == "reference":
        run_reference(args)
        return

    import torch
    import torch.distributed as dist
    from moonshine_b200 import api

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    model, B = args.model, args.batch
    d = ARCHS[model]

    clock_lines, stop_evt = [], threading.Event()
    th = threading.Thread(target=clocks_sampler, args=(stop_evt, clock_lines), daemon=True)
    th.start()
    time.sleep(0.3)
    wall0 = time.perf_counter()
    head, toks, audios = measure_config(api, torch, dist, model, B, args.steps, args.warmup, rank, world, local)
    wall_head = time.perf_counter() - wall0
    outputs = {f"{model}_b{B}": toks}

    # ---- the other BASELINE operating points (same run, same box) ----
    configs = {}
    default_headline = (model == "tiny" and B == 32)
    if default_headline and not args.headline_only:
        extra = []
        if world == 1:
            extra = [("tiny_b1", "tiny", 1), ("base_b256", "base", 256), ("base_streaming_b64", "base_streaming", 64)]
        elif world == 8:
            extra = [("base_b2048_8gpu", "base", 256)]
        for key, m2, b2 in extra:
            try:
                rec, outputs[key], _ = measure_config(api, torch, dist, m2, b2, args.steps, args.warmup, rank, world, local)
                configs[key] = rec
            except Exception as e:  # an extra config must never take the headline down
                configs[key] = {"error": f"{type(e).__name__}: {e}"}
    stop_evt.set()
    th.join(timeout=3)

    if rank == 0:
        K = args.steps
        steps_run = head["stage_ms"]["decode_steps"]
        line = {
            "metric": "utterances_per_sec", "value": head["value"], "unit": "utt/s", "n_gpus": world, "steps": K,
            "warmup": args.warmup, "ms_per_step": head["ms_per_step"], "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "rtf": head["rtf"],
            "config": {
                "workload": f"moonshine-{model}, batch={B} synthetic 10s@16kHz utterances per GPU, "
                            + ("streaming frontend + sliding-window encoder + adapter" if d.streaming else "conv frontend + encoder")
                            + f" + greedy decoder ({steps_run} decode steps; seeded random weights never emit EOS)",
                "batch_per_gpu": B, "global_batch": B * world, "audio_seconds_per_utt": 10.0,
                "weights": "seeded synthetic (HF init std 0.02), fp32 storage (bf16 hi+lo planes for tensor-core operands); cross K/V cache fp16",
                "parallelism": f"dp{world} (utterance shards, one NCCL weight broadcast at init)",
                "timing": "CUDA events on the library stream per step; 256 MB L2 flush between steps (outside the events)",
            },
            "stage_ms": head["stage_ms"], "roofline": head["roofline"], "e2e": head["e2e"],
            "gpu_launches": head["gpu_launches"], "tokens_per_utt": head["tokens_per_utt"],
            "configs": configs, "published_reference": PUBLISHED,
            "clocks": summarise_clocks(clock_lines, local), "wall_s_headline": wall_head,
        }
        if not args.no_cpu_baseline and world == 1:  # the CPU arm is timed beside the N = 1 line only
            threads = host_threads()
            try:
                r = hf_arm(model, audios[:3], audios[:min(B, 16)], threads)
                n = r["serial_n"]
                line["cpu_baseline"] = {
                    "value": r["batched_utt_s"], "unit": "utt/s", "cores": r["threads_batched"], "kind": "port",
                    "sample": f"first {r['batched_n']} utterances of the batch as ONE batch ({r['batched_s']:.1f} s, {r['threads_batched']} threads) and "
                              f"first {n} one at a time ({r['threads_serial']} threads), Hugging Face float implementation (fp32, torch; thread "
                              f"counts are the fastest of those tried on this {os.cpu_count()}-core host)",
                    "threads_tried_s_per_short_sample": r["threads_tried"],
                    "serial_batch1_utt_s": r["serial_utt_s"], "serial_batch1_s_per_utt": r["serial_s_per_utt"],
                    "tokens_match_gpu": bool(all(r["tokens_serial"][i] == toks[i] for i in range(n))),
                }
                np_ups, np_toks = numpy_port_utt_s(model, audios[0], threads)
                line["cpu_baseline"]["numpy_port_cross_check_utt_s"] = np_ups
                line["cpu_baseline"]["numpy_port_tokens_match_gpu"] = bool(np_toks == toks[0])
            except Exception as e:
                np_ups, np_toks = numpy_port_utt_s(model, audios[0], threads)
                line["cpu_baseline"] = {"value": np_ups, "unit": "utt/s", "cores": min(threads, 16), "kind": "port",
                                        "sample": f"1 utterance, numpy oracle (HF arm failed: {type(e).__name__}: {e})",
                                        "tokens_match_gpu": bool(np_toks == toks[0])}
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, outputs)
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
