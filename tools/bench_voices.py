#!/usr/bin/env python
"""Mixed-voice batches on one GPU: what a voice per text costs.

Workload: the bench's batch (64 texts of 52 ids, 400 frames, EOS never ends an utterance: min_gen_frames=10**9, bf16
AR weight storage), with voices of Tr = 150 frames (12 s at 12.5 Hz), each prepared from its own random codes.  Timed,
interleaved within every repetition, median over the repetitions (host clock around work that ends in a device
synchronise; L2 flushed by a 256 MiB write before each timed call, outside the timing):

  prefill_ms        the batched CUDA prefill alone: one shared voice (PrefillEngine.run) and 1 / 8 / 64 distinct voices
                    (PrefillEngine.run_voices; voice i % n for text i)
  synth_ms          SoproTTS.synthesize_batch(64 texts) with ref= (shared) and refs= with 1 / 8 / 64 distinct voices
  per_voice_calls_ms  what a caller without refs= does for 64 distinct voices: 64 synthesize_batch calls of one text each
  attn_kernel_ms    device time of the reference cross-attention kernels inside one prefill (torch.profiler, separate pass)

  python tools/bench_voices.py [--reps 5] [--warmup 2] [--out FILE]     -> one JSON line on stdout (and in FILE)
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

VOICE_FRAMES = 150
VOICE_COUNTS = (1, 8, 64)


def gpu_facts():
    out = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm,clocks.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=20).stdout.strip()
        out["power_limit"], out["sm_max_clock"], out["sm_clock_at_start"] = [x.strip() for x in q.split(",")]
    except Exception as e:  # the numbers stay valid without it; say that it is missing
        out["nvidia_smi_error"] = repr(e)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", help="also write the JSON line to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_voices.py: no CUDA device (the engines have no CPU path)")
    import bench
    from sopro_b200 import SoproTTS
    from sopro_b200.config import SoproTTSConfig
    from sopro_b200.tokenizer import IdsTokenizer
    from sopro_b200.weights import synth_mimi_state_dict

    torch.set_grad_enabled(False)
    dev = torch.device("cuda", 0)
    cfg = SoproTTSConfig()
    tts = SoproTTS.from_state_dict(cfg, bench.bench_state_dict(cfg), IdsTokenizer(bench.TEXT_VOCAB), synth_mimi_state_dict(),
                                   device=str(dev), weight_dtype="bf16")
    B, F = bench.BATCH_PER_GPU, bench.FRAMES
    texts = bench.bench_texts(0, B)
    seeds = list(range(1234, 1234 + B))
    codes = [torch.randint(0, 2048, (VOICE_FRAMES, 32), generator=torch.Generator().manual_seed(100 + i)) for i in range(B)]
    voices = [tts.prepare_reference(ref_tokens_tq=c) for c in codes]
    assert all(int(v.ref_seq.shape[1]) == VOICE_FRAMES for v in voices)
    refs = {n: [voices[i % n] for i in range(B)] for n in VOICE_COUNTS}
    model, st = tts.model, float(cfg.style_strength)
    ids = [tts.encode_text(t) for t in texts]
    kv_bytes = sum(c[k].numel() * 4 for c in voices[0].ref_kv_caches for k in ("k", "v"))
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    kw = dict(max_frames=F, seeds=seeds, min_gen_frames=10 ** 9)

    prefill = {"shared": lambda: model.prefill.run(ids, voices[0], n_frames=F + 1, style_strength=st)}
    for n in VOICE_COUNTS:
        prefill[f"voices_{n}"] = lambda n=n: model.prefill.run_voices(ids, refs[n], n_frames=F + 1, style_strength=st)
    synth = {"shared": lambda: tts.synthesize_batch(texts, ref=voices[0], **kw)}
    for n in VOICE_COUNTS:
        synth[f"voices_{n}"] = lambda n=n: tts.synthesize_batch(texts, refs=refs[n], **kw)
    synth["per_voice_calls_64"] = lambda: [tts.synthesize_batch([texts[i]], ref=voices[i], seeds=[seeds[i]], max_frames=F,
                                                                min_gen_frames=10 ** 9)[0] for i in range(B)]

    def timed(fn):
        flush.fill_(1)
        torch.cuda.synchronize(dev)
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize(dev)
        return (time.perf_counter() - t0) * 1e3

    with torch.inference_mode():
        for _ in range(args.warmup):
            for fn in list(prefill.values()) + list(synth.values()):
                fn()
        times = {("prefill", k): [] for k in prefill}
        times.update({("synth", k): [] for k in synth})
        for _ in range(args.reps):
            for k, fn in prefill.items():
                times[("prefill", k)].append(timed(fn))
            for k, fn in synth.items():
                times[("synth", k)].append(timed(fn))
        # device time of the attention kernels, one prefill each, in a run of its own
        attn = {}
        from torch.profiler import ProfilerActivity, profile

        for k in ("shared", "voices_64"):
            flush.fill_(1)
            torch.cuda.synchronize(dev)
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                prefill[k]()
                torch.cuda.synchronize(dev)
            attn[k] = sum(e.device_time_total for e in prof.key_averages() if "ref_attn" in e.key) / 1e3
    med = {key: float(np.median(v)) for key, v in times.items()}
    spread = {key: [float(np.min(v)), float(np.max(v))] for key, v in times.items()}
    line = {
        "tool": "tools/bench_voices.py", "gpu": gpu_facts(), "reps": args.reps, "warmup": args.warmup,
        "workload": f"{B} texts x {bench.TEXT_LEN} ids, {F} frames (min_gen_frames=10**9), bf16 AR weight storage, voices of "
                    f"Tr={VOICE_FRAMES} frames, voice i % n for text i",
        "voice_kv_mb": kv_bytes / 1e6, "voices_kv_mb_64": 64 * kv_bytes / 1e6,
        "prefill_ms": {k: med[("prefill", k)] for k in prefill},
        "synth_ms": {k: med[("synth", k)] for k in synth if k != "per_voice_calls_64"},
        "per_voice_calls_ms": med[("synth", "per_voice_calls_64")],
        "attn_kernel_ms": attn,
        "min_max_ms": {f"{a}:{k}": v for (a, k), v in spread.items()},
        "ratios": {"prefill_64_over_shared": med[("prefill", "voices_64")] / med[("prefill", "shared")],
                   "synth_64_over_shared": med[("synth", "voices_64")] / med[("synth", "shared")],
                   "per_voice_calls_over_synth_64": med[("synth", "per_voice_calls_64")] / med[("synth", "voices_64")]},
        "timing": "host clock around calls ending in a device synchronise; median over reps, configurations interleaved per rep; "
                  "L2 flushed (256 MiB write) before each call, outside the timing; clocks as the machine gives them",
    }
    text = json.dumps(line)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
