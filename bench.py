#!/usr/bin/env python
"""bench.py — AR frames/s of the Sopro hot path on N B200s (one process per GPU).

Workload (BASELINE.json configs[2]; x N GPUs it is configs[3]): per GPU a batch of 64 independent 400-frame
utterances (401 AR steps: reference model.py:242), 52 text tokens each, one shared prepared reference voice (3 s = 38
frames), bf16 weight storage for the AR stack, fp32 arithmetic, default sampler, EOS never sampled (head bias -30: the
length is pinned, SURVEY.md §8d).  A bench "step" is one full pass of the hot path over that batch.

  value   device-resident: text-K/V build + ONE persistent AR kernel launch (64 x 401 frames), inputs already in HBM
  e2e     the same metric through the PUBLIC API: SoproTTS.synthesize_batch(64 texts) = tokenise -> batched CUDA prefill ->
          noise tapes drawn on the host and uploaded -> persistent AR kernel -> CUDA NAR refiner -> tcgen05 Mimi decode
          -> waveforms copied to pinned host memory.  Host->device: text ids + noise tapes; device->host: the waveforms.

Data parallel, no data-path collective ("weak" scaling); NCCL is used once, to broadcast the weights from rank 0.

  python bench.py --gpus 1 --steps 5 --warmup 3
  python bench.py --gpus 1 --steps 5 --warmup 3 --dump-outputs DIR   # + what the last timed step returned, as DIR/*.npy
  python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...
  python bench.py --impl reference ...      # the reference's own CPU path (baseline/_ref when present, else the oracle port)
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

BATCH_PER_GPU = 64
FRAMES = 400
STEPS_AR = FRAMES + 1
TEXT_LEN = 52
REF_FRAMES = 38
TEXT_VOCAB = 1000
S_UTT_BYTES = 3280  # SURVEY.md §8d: cond row + embedding row + noise + token per utterance-step
MIMI_FLOP_PER_FRAME = 431.2e6  # SURVEY.md §8a11
MIMI_ALG_BYTES_PER_FRAME = 7936  # 32 codes x 8 B + 1920 samples x 4 B (SURVEY.md §8d)
WORKLOAD = "batch=64/GPU non-streaming, 400-frame utterances (401 AR steps), L_text=52, bf16 weights, fp32 math"


def _peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            j = json.load(f)
        return float(j["hbm_gbs"]), float(j.get("bf16_tflops_sustained", 1456.6)), float(j.get("bf16_tflops", 1710.5)), \
            "measured (MEASURED_PEAKS.json)"
    return 6650.0, 1400.0, 1590.0, "fallback (B200_PROFILING.md 6.65 TB/s, 1.59 PFLOP/s burst / ~1.4 sustained)"


def _inputs(cfg, rank, B, steps, L):
    from sopro_b200.sampling import noise_tape
    from sopro_b200.weights import hash_uniform

    D = int(cfg.d_model)
    s3 = np.float32(np.sqrt(3.0))
    cond = torch.from_numpy(hash_uniform(B * steps * D, 7_000_000 + rank) * s3).view(B, steps, D)
    txt = torch.from_numpy(hash_uniform(B * L * D, 8_000_000 + rank) * s3).view(B, L, D)
    noise = torch.stack([noise_tape(steps, cfg.ar_vocab(), seed=1234 + rank * B + i, keep=50) for i in range(B)])
    return cond.contiguous(), txt.contiguous(), noise.contiguous()


def bench_state_dict(cfg):
    """The synthetic checkpoint of the bench: seeded (hash-based, identical on every host), AR stack rounded through
    bf16 (the storage format of configs[2]), EOS logit bias -30 so no utterance ends early."""
    from sopro_b200.weights import round_through_bf16, synth_state_dict

    sd = round_through_bf16(synth_state_dict(cfg, TEXT_VOCAB, 0), ("ar.", "cb_embed."))
    sd["ar.head.bias"] = sd["ar.head.bias"].clone()
    sd["ar.head.bias"][int(cfg.codebook_size)] = -30.0
    return sd


def bench_texts(rank, B):
    return [" ".join(str((17 * i + 5 + 31 * (rank * B + j)) % TEXT_VOCAB) for i in range(TEXT_LEN - 2)) for j in range(B)]


def bench_ref_tokens():
    return torch.randint(0, 2048, (REF_FRAMES, 32), generator=torch.Generator().manual_seed(7))


def dump_outputs(out_dir, toks, n_tok, wav_host, wav_len):
    """Writes what the last timed step of each leg handed to its caller as DIR/<name>.npy, so that two builds can be
    compared output for output: the resident leg's AR tokens and frame counts (exact in float32), and the API leg's
    waveforms at one fixed, seeded set of sample positions shared by every utterance (zero past an utterance's end).
    The sample keeps the waveforms to 32 MiB; the full ones are about 3 MB per utterance."""
    os.makedirs(out_dir, exist_ok=True)
    B, cols = wav_host.shape
    k = min(cols, max(1, (32 << 20) // (4 * B)))
    idx = np.sort(np.random.default_rng(0).choice(cols, k, replace=False))
    lens = np.asarray(wav_len, dtype=np.int64)
    wav = wav_host.numpy()[:, idx]
    wav[idx[None, :] >= lens[:, None]] = 0.0
    arrays = {"ar_tokens": toks.astype(np.float32), "ar_frames": n_tok.astype(np.float32),
              "wav_samples": wav.astype(np.float32), "wav_sample_index": idx.astype(np.float64),
              "wav_lengths": lens.astype(np.float64)}
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


class ClockSampler(threading.Thread):
    """nvidia-smi style clock / throttle-reason samples during the timed region (NVML)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.stop_flag, self.sm, self.reasons, self.max_mhz = index, False, [], set(), None
        try:
            import pynvml

            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = int(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        names = {
            nv.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown",
            nv.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown",
            nv.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown",
            nv.nvmlClocksThrottleReasonSwPowerCap: "sw_power_cap",
        }
        while not self.stop_flag:
            try:
                self.sm.append(int(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                r = int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
                for bit, nm in names.items():
                    if r & bit:
                        self.reasons.add(nm)
            except Exception:
                pass
            time.sleep(0.05)

    def summary(self):
        return {"sm_mhz": int(np.median(self.sm)) if self.sm else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.sm)}


def usable_cpus() -> int:
    """Host threads this process may really use: affinity mask and cgroup quota, not the box's core count."""
    n = os.cpu_count() or 1
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except Exception:
        pass
    try:
        with open("/sys/fs/cgroup/cpu.max") as f:
            q, per = f.read().split()
            if q != "max":
                n = min(n, max(1, int(float(q) / float(per))))
    except Exception:
        pass
    return max(1, n)


# ------------------------------------------------------------------------------------------------------------------
# The CPU arm: the reference's own path.  `baseline/_ref` holds the UNMODIFIED reference (pip --target install made in
# the build container, recorded in DESIGN.md); it travels to the GPU box.  When it cannot be imported the oracle port
# (bit-equal to the reference, tests/test_oracle_golden.py) stands in and `kind` says "port".
# ------------------------------------------------------------------------------------------------------------------
class CpuReference:
    def __init__(self, cfg, sd):
        self.cfg, self.sd = cfg, sd
        self.kind, self.tts = "port", None
        ref_dir = os.path.join(ROOT, "baseline", "_ref")
        if os.path.isdir(os.path.join(ref_dir, "sopro")):
            try:
                sys.path.insert(0, ref_dir)
                import transformers as tr
                from sopro.codec.mimi import MimiCodec
                from sopro.config import SoproTTSConfig as RefCfg
                from sopro.model import SoproTTS as RefTTS
                from sopro.model import SoproTTSModel

                from sopro_b200.tokenizer import IdsTokenizer
                from sopro_b200.weights import synth_mimi_state_dict

                tok = IdsTokenizer(TEXT_VOCAB)
                model = SoproTTSModel(RefCfg(), tok).eval()
                missing, unexpected = model.load_state_dict(sd, strict=False)
                assert not unexpected and not missing, (missing[:3], unexpected[:3])
                hf = tr.MimiModel(tr.MimiConfig(num_quantizers=32)).eval()
                hf.load_state_dict(synth_mimi_state_dict(), strict=False)
                codec = object.__new__(MimiCodec)  # bypasses the hub download (reference codec/mimi.py:28-31)
                codec.device, codec.model = torch.device("cpu"), hf
                self.tts = RefTTS(model, RefCfg(), tok, codec, "cpu")
                self.kind = "reference"
            except Exception as ex:  # fall back to the port, and say why
                self.err = repr(ex)
                if ref_dir in sys.path:
                    sys.path.remove(ref_dir)

    def pick_threads(self):
        """The reference's AR step is ~1,240 tiny ATen calls (SURVEY.md §3.2): more intra-op threads than a handful
        only add fork/join cost.  Try a few counts on a 24-frame probe and keep the fastest."""
        top = usable_cpus()
        cands = sorted({c for c in (1, 4, 8, 16, 32, top) if c <= top})
        best, best_t = 1, float("inf")
        for c in cands:
            torch.set_num_threads(c)
            t0 = time.perf_counter()
            self.ar_utterance(0, frames=24)
            dt = time.perf_counter() - t0
            if dt < best_t:
                best, best_t = c, dt
            if dt > 20.0:
                break
        torch.set_num_threads(best)
        return best, top

    def ar_utterance(self, i, frames=FRAMES):
        """One utterance of the bench's AR workload (synthetic cond / text rows, seed 1234 + i) -> frames produced."""
        cond, txt, _ = _inputs(self.cfg, 0, 1, frames + 1, TEXT_LEN) if frames != FRAMES else self._full_inputs(i)
        if self.tts is not None:
            prep = {"cond_ar": cond, "txt_seq": txt, "text_mask": torch.ones(1, TEXT_LEN, dtype=torch.bool)}
            torch.manual_seed(1234 + i)
            n = 0
            for _t, _tok, _e in self.tts.model.ar_stream(prep, max_frames=frames, min_gen_frames=10 ** 9):
                n += 1
            return n
        from oracle import ar_oracle as O

        tape = O.noise_tape(1234 + i, frames + 1, self.cfg.ar_vocab())
        return len(O.ar_generate(self.sd, self.cfg, cond, txt, torch.ones(1, TEXT_LEN, dtype=torch.bool), max_frames=frames,
                                 sampling=O.ArSampling(min_gen_frames=10 ** 9), noise_tv=tape))

    def _full_inputs(self, i):
        if not hasattr(self, "_cache"):
            self._cache = _inputs(self.cfg, 0, 16, STEPS_AR, TEXT_LEN)
        c, t, _ = self._cache
        j = i % 16
        return c[j:j + 1], t[j:j + 1], None

    def ar_rate(self, n_utts):
        t0 = time.perf_counter()
        frames = sum(self.ar_utterance(i) for i in range(n_utts))
        dt = time.perf_counter() - t0
        return frames / dt, dt

    def stages(self, ttfa_runs=20):
        """The reference CLI's timing points (cli.py:120,141,159-165) on ONE utterance of the workload, and stream() TTFA
        p50 (streaming.py:133-152) with a prepared reference.  Reference only (the port has no public API)."""
        if self.tts is None:
            return None
        tts = self.tts
        text = bench_texts(0, 1)[0]
        ref = tts.prepare_reference(ref_tokens_tq=bench_ref_tokens())
        ids = tts.encode_text(text)
        st = float(tts.cfg.style_strength)
        out = {}
        t0 = time.perf_counter()
        prep = tts.model.prepare_conditioning(ids, ref, max_frames=FRAMES, device="cpu", style_strength=st)
        t1 = time.perf_counter()
        torch.manual_seed(1)
        hist = [tok for _t, tok, _e in tts.model.ar_stream(prep, max_frames=FRAMES, min_gen_frames=10 ** 9)]
        t2 = time.perf_counter()
        T = len(hist)
        codes = tts.model.nar_refine(prep["cond_ar"][:, :T], torch.tensor(hist).unsqueeze(0)).squeeze(0)
        t3 = time.perf_counter()
        wav = tts.codec.decode_full(codes.clamp(0, 2047))
        t4 = time.perf_counter()
        audio_s = wav.shape[-1] / 24000.0
        out.update(prefill_s=t1 - t0, ar_s=t2 - t1, ar_frames_per_sec=T / (t2 - t1), nar_s=t3 - t2, mimi_s=t4 - t3,
                   mimi_frames_per_sec=T / (t4 - t3), total_s=t4 - t0, frames=T, rtf=(t4 - t0) / audio_s)
        ts = []
        for i in range(ttfa_runs + 1):
            torch.manual_seed(1)
            a = time.perf_counter()
            it = tts.stream(text, ref=ref, max_frames=FRAMES, min_gen_frames=10 ** 9)
            next(it)
            b = time.perf_counter()
            it.close()
            if i:
                ts.append(b - a)
        out["ttfa_ms_p50"] = float(np.median(ts)) * 1e3
        return out


def cpu_baseline_block(cpu, n_utts, with_stages=True):
    threads, avail = cpu.pick_threads()
    v, dt = cpu.ar_rate(n_utts)
    what = ("the UNMODIFIED reference (baseline/_ref, SoproTTSModel.ar_stream on CPU)" if cpu.kind == "reference"
            else "oracle/ar_oracle.py (torch CPU eager restatement, bit-equal to the reference)")
    blk = {"value": v, "unit": "frames/s", "cores": threads, "cores_available": avail, "kind": cpu.kind,
           "sample": f"{n_utts} utterance(s) x 401 AR frames of the same workload, sequential, {dt:.1f} s; {what}; the reference "
                     "has no batch path, so batch-64 throughput on CPU is its batch-1 rate"}
    if with_stages:
        st = cpu.stages()
        if st is not None:
            blk["stages"] = st
            blk["stages_note"] = ("one utterance of the workload through the reference's public pieces at the CLI's timing points "
                                  "(cli.py:120,141,159-165): prefill / AR / NAR / Mimi decode / total -> RTF; stream() TTFA p50 over 20 "
                                  "runs with a prepared reference (streaming.py:133-152)")
    return blk


# ------------------------------------------------------------------------------------------------------------------
def extras(tts, ref, cfg, dev, peaks):
    """Side measurements of the other BASELINE.json configs on one GPU (not the headline `value`): batch-1 AR rate
    (fp32, configs[1]), stream() time-to-first-audio p50 measured AFTER complete streams (configs[1]), whole-stream time,
    synthesize() RTF at batch 1, Mimi decode of 10k frames with its roofline (configs[4])."""
    from sopro_b200.engine import Sampling

    out = {}
    text = bench_texts(0, 1)[0]

    def timed(fn, n, warm=2):
        ts = []
        for i in range(n + warm):
            torch.cuda.synchronize(dev)
            t0 = time.perf_counter()
            r = fn()
            torch.cuda.synchronize(dev)
            if i >= warm:
                ts.append(time.perf_counter() - t0)
        return float(np.median(ts)), r

    # batch-1 AR rate, device resident (bf16 weight storage like the headline; fp32 math)
    eng = tts.model.engine
    cond, txt, noise = _inputs(cfg, 0, 1, STEPS_AR, TEXT_LEN)
    cond, txt, noise = cond.to(dev), txt.to(dev), noise.to(dev)
    ses = eng.session(1, STEPS_AR, TEXT_LEN)
    sp = Sampling(min_gen_frames=2 ** 31 - 1)

    def ar1():
        ses.begin(cond, txt, [TEXT_LEN], noise, sp)
        ses.run()

    t, _ = timed(ar1, 5)
    out["batch1_ar_frames_per_sec"] = STEPS_AR / t
    out["batch1_us_per_ar_step"] = t / STEPS_AR * 1e6
    ses.close()
    # complete streams first (ADVICE r1: a first-chunk-only loop hides per-window costs), then TTFA p50 over 20 runs
    t_stream, nchunks = timed(lambda: sum(1 for _ in tts.stream(text, ref=ref, max_frames=FRAMES, seed=1, min_gen_frames=10 ** 9)), 2, warm=1)
    out["stream_400_frames_ms"] = t_stream * 1e3
    out["stream_chunks"] = int(nchunks)
    ts = []
    for i in range(22):
        torch.cuda.synchronize(dev)
        t0 = time.perf_counter()
        it = tts.stream(text, ref=ref, max_frames=FRAMES, seed=1, min_gen_frames=10 ** 9)
        c = next(it)
        c = c.cpu()  # the first audio in host memory
        t1 = time.perf_counter()
        it.close()
        torch.cuda.synchronize(dev)
        if i >= 2:
            ts.append(t1 - t0)
    out["ttfa_ms_p50"] = float(np.median(ts)) * 1e3
    out["ttfa_ms_min"] = float(np.min(ts)) * 1e3  # p50 moves with the box's power state (sw_power_cap boxes: +1.5 ms); the floor does not
    out["ttfa_ms_p90"] = float(np.percentile(ts, 90)) * 1e3
    out["ttfa_first_chunk_samples"] = int(c.numel())
    # RTF: whole synthesize() (tokenize + prefill + AR + NAR + Mimi) / audio seconds
    t, wav = timed(lambda: tts.synthesize(text, ref=ref, max_frames=FRAMES, seed=1, min_gen_frames=10 ** 9), 3, warm=1)
    out["rtf_batch1"] = t / (wav.shape[-1] / 24000.0)
    out["synthesize_batch1_ms"] = t * 1e3
    # reference-voice ingestion (once per voice, SURVEY.md §8f-4): Mimi ENCODE of a 10 s recording, then prepare_reference
    try:
        from sopro_b200.codec import MimiEncoderEngine
        from sopro_b200.weights import synth_mimi_encoder_state_dict, synth_mimi_state_dict

        esd = dict(synth_mimi_state_dict())
        esd.update(synth_mimi_encoder_state_dict())
        enc = MimiEncoderEngine(esd, dev, 32)
        voice = ((torch.rand(24000 * 10, generator=torch.Generator().manual_seed(9)) - 0.5) * 0.6).to(dev)
        t, vcodes = timed(lambda: enc.encode(voice), 3, warm=1)
        out["voice_encode_ms_10s"] = t * 1e3
        t, _ = timed(lambda: tts.model.prepare_reference(vcodes.permute(1, 0).contiguous()), 5, warm=2)
        out["prepare_reference_ms"] = t * 1e3
        enc.close()
        del enc, esd
    except Exception as e:  # a side measurement must never cost the bench line
        out["voice_encode_error"] = repr(e)
    # Mimi standalone: 25 x 400 = 10k frames
    codes = torch.randint(0, 2048, (25, 32, 400), generator=torch.Generator().manual_seed(5)).to(dev)
    t, _ = timed(lambda: tts.codec.engine.decode(codes), 3, warm=1)
    tts.codec.engine.set_precision("fp32")
    t32, _ = timed(lambda: tts.codec.engine.decode(codes), 1, warm=1)
    tts.codec.engine.set_precision("bf16_tc")
    out["mimi_fp32_mode_ms_per_10k_frames"] = t32 * 1e3
    hbm, tf_sus, tf_burst, src = peaks
    tfl = 10000 * MIMI_FLOP_PER_FRAME / t / 1e12
    mimi = {"bound": "tensor", "achieved": tfl, "peak": tf_sus, "unit": "TFLOP/s", "frac": tfl / tf_sus, "peak_burst": tf_burst,
            "frac_of_burst": tfl / tf_burst, "ms_per_10k_frames": t * 1e3, "frames_per_sec": 10000 / t,
            "precision": tts.codec.engine.precision, "alg_bytes_per_frame": MIMI_ALG_BYTES_PER_FRAME,
            "alg_gb_per_s": 10000 * MIMI_ALG_BYTES_PER_FRAME / t / 1e9, "alg_frac_of_hbm": 10000 * MIMI_ALG_BYTES_PER_FRAME / t / 1e9 / hbm,
            "peak_source": src, "traffic": None,
            "note": "whole decode (about 85 launches), 431.2 MFLOP of contractions per frame (SURVEY.md §8a11); peak = sustained cuBLAS bf16; "
                    "per-kernel tensor-pipe and DRAM figures: profiles/"}
    tp = os.path.join(ROOT, "profiles", "mimi_traffic.json")
    if os.path.exists(tp):
        with open(tp) as f:
            tj = json.load(f)
        mimi["traffic"] = tj.get("dram_bytes_per_frame")
        mimi["ncu_capture"] = tj.get("ncu")
    return out, mimi


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=BATCH_PER_GPU, help="utterances per GPU")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip batch-1 / TTFA / RTF / Mimi side measurements")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed to DIR/<name>.npy (rank 0, B200 arm)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the B200 arm's outputs; it does not apply to --impl reference")
    torch.set_grad_enabled(False)
    # Libraries (NCCL's version banner, ...) write to fd 1; the contract is ONE JSON line on stdout.
    # Everything else goes to stderr, the JSON is written to the real stdout at the end.
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)

    def emit(obj):
        os.write(real_stdout, (json.dumps(obj) + "\n").encode())

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    from sopro_b200.config import SoproTTSConfig

    cfg = SoproTTSConfig()
    config = {"workload": WORKLOAD, "batch_per_gpu": args.batch, "global_batch": args.batch * max(world, 1),
              "frames": FRAMES, "text_len": TEXT_LEN, "ref_frames": REF_FRAMES, "parallelism": f"dp{max(world, 1)}",
              "weights": "synthetic seeded (sopro_b200.weights.synth_state_dict), ar.* and cb_embed rounded through bf16, EOS head "
                         "bias -30 (length pinned to 401 frames)",
              "l2": "L2 flushed (256 MiB write) between timed steps, outside the event pairs"}

    # ------------------------------------------------------------------ reference arm
    if args.impl == "reference":
        if rank != 0:
            return
        cpu = CpuReference(cfg, bench_state_dict(cfg))
        threads, avail = cpu.pick_threads()
        for _ in range(max(args.warmup, 0)):
            cpu.ar_utterance(0)  # warm-up: one utterance
        secs, frames = 0.0, 0
        for i in range(max(args.steps, 1)):
            t0 = time.perf_counter()
            frames += cpu.ar_utterance(i)
            secs += time.perf_counter() - t0
        fps = frames / secs
        what = ("the UNMODIFIED reference from baseline/_ref (SoproTTSModel.ar_stream, torch CPU eager)" if cpu.kind == "reference"
                else "oracle/ar_oracle.py (torch CPU eager restatement of the reference, bit-equal to it)")
        blk = {"value": fps, "unit": "frames/s", "cores": threads, "cores_available": avail, "kind": cpu.kind,
               "sample": f"each step = 1 utterance x 401 AR frames of the bench workload, {what}; the reference has no batch path, so "
                         "batch-64 throughput on CPU is this rate"}
        try:
            st = cpu.stages()
            if st is not None:
                blk["stages"] = st
        except Exception as ex:
            blk["stages_error"] = repr(ex)
        line = {"impl": "reference", "metric": "ar_frames_per_sec", "value": fps, "unit": "frames/s", "n_gpus": args.gpus,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": secs / max(args.steps, 1) * 1e3,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": config, "cpu_baseline": blk,
                "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        emit(line)
        return

    # ------------------------------------------------------------------ B200 arm
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the B200 arm has no CPU fallback (use --impl reference for the CPU baseline)")
    import torch.distributed as dist

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    from sopro_b200.dp import DataParallelTTS
    from sopro_b200.engine import Sampling
    from sopro_b200.tokenizer import IdsTokenizer
    from sopro_b200.weights import synth_mimi_state_dict

    # weights: built on rank 0, broadcast once over NCCL/NVLink (the only collective of the path)
    sd = bench_state_dict(cfg) if rank == 0 else None
    dp = DataParallelTTS(cfg, sd, IdsTokenizer(TEXT_VOCAB), synth_mimi_state_dict(), device=dev, weight_dtype="bf16",
                         text_vocab=TEXT_VOCAB)
    tts = dp.tts
    eng = tts.model.engine
    B = args.batch
    ref = tts.prepare_reference(ref_tokens_tq=bench_ref_tokens())
    cond_h, txt_h, noise_h = _inputs(cfg, rank, B, STEPS_AR, TEXT_LEN)
    cond_d, txt_d, noise_d = cond_h.to(dev), txt_h.to(dev), noise_h.to(dev)
    samp = Sampling(min_gen_frames=2 ** 31 - 1)
    ses = eng.session(B, STEPS_AR, TEXT_LEN)
    lens = [TEXT_LEN] * B
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    # the API leg: this rank's shard of the global batch of texts (dp.shard_range), one seed per utterance
    all_texts = [t for r in range(max(world, 1)) for t in bench_texts(r, B)]
    all_seeds = list(range(1234, 1234 + len(all_texts)))
    wav_host = torch.empty((B, STEPS_AR * 1920), dtype=torch.float32).pin_memory()
    wav_len = [0] * B  # samples of each utterance in wav_host after the last API pass

    def one_pass_resident():
        ses.begin(cond_d, txt_d, lens, noise_d, samp)
        ses.run()

    def one_pass_api():
        wavs, (lo, hi) = dp.synthesize_batch(all_texts, ref=ref, seeds=all_seeds, max_frames=FRAMES, min_gen_frames=10 ** 9)
        frames = 0
        for j, w in enumerate(wavs):  # the result in host memory
            n = int(w.shape[-1])
            wav_host[j, :n].copy_(w.reshape(-1), non_blocking=True)
            wav_len[j] = n
            frames += n // 1920
        torch.cuda.current_stream(dev).synchronize()
        return frames

    def sync_all():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize(dev)

    for _ in range(max(args.warmup, 3)):
        one_pass_resident()
    for _ in range(2):
        one_pass_api()
    sync_all()
    clocks = ClockSampler(local_rank)
    clocks.start()
    # ---- device-resident throughput: K passes, each bracketed by its own event pair
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
          for _ in range(args.steps)]
    sync_all()
    for a, m, b in ev:
        flush.fill_(1)
        a.record()
        ses.begin(cond_d, txt_d, lens, noise_d, samp)
        m.record()
        ses.run()
        b.record()
    sync_all()
    t_total_ms = sum(a.elapsed_time(b) for a, _, b in ev)
    t_kernel_ms = sum(m.elapsed_time(b) for _, m, b in ev) / args.steps  # the persistent AR kernel alone
    toks, n_tok, _ = ses.read()
    frames_per_pass = int(n_tok.sum())
    # ---- end to end through the public API: texts in, waveforms in pinned host memory out
    e2e_ms, e2e_frames = 0.0, 0
    for i in range(args.steps):
        flush.fill_(1)
        torch.cuda.synchronize(dev)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        e2e_frames += one_pass_api()
        b.record()
        torch.cuda.synchronize(dev)
        e2e_ms += a.elapsed_time(b)
    clocks.stop_flag = True
    clocks.join(timeout=2)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, toks, n_tok, wav_host, wav_len)
    t = torch.tensor([t_total_ms, e2e_ms, t_kernel_ms], dtype=torch.float64, device=dev)
    fr = torch.tensor([float(frames_per_pass), float(e2e_frames)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(fr, op=dist.ReduceOp.SUM)
    t_total_ms, e2e_ms, t_kernel_ms = [float(x) for x in t.tolist()]
    frames_all, e2e_frames_all = [float(x) for x in fr.tolist()]
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    value = frames_all * args.steps / (t_total_ms / 1e3)
    e2e_value = e2e_frames_all / (e2e_ms / 1e3)
    peaks = _peaks()
    peak, peak_src = peaks[0], peaks[3]
    w_step = eng.step_weight_bytes
    alg_bytes_launch = (w_step + B * S_UTT_BYTES) * STEPS_AR
    achieved = alg_bytes_launch / (t_kernel_ms / 1e3) / 1e9
    traffic = None
    ncu_note = None
    tp = os.path.join(ROOT, "profiles", "ar_kernel_traffic.json")
    if os.path.exists(tp):
        with open(tp) as f:
            tj = json.load(f)
        traffic = tj.get("dram_bytes_per_launch")
        ncu_note = tj.get("ncu")
    W = max(world, 1)
    # launches of OUR kernels inside the timed regions, per rank: resident leg = kv_build + persistent AR per step; API leg per
    # step = prefill 24 + kv_build 1 + AR 6 (the launch resumes once per noise-tape block) + NAR on the tensor cores (1 + 4
    # stages x 54) + Mimi (about 85 per decode call x 3 calls at 12,800 frames)
    api_launches = 24 + 7 + 217 + 85 * 3
    line = {
        "metric": "ar_frames_per_sec", "value": value, "unit": "frames/s", "n_gpus": W, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": t_total_ms / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32 math / bf16 weight storage", "data": "synthetic", "config": config,
        "e2e": {"value": e2e_value, "unit": "frames/s",
                "api": "SoproTTS.synthesize_batch via sopro_b200.dp.DataParallelTTS (text -> prefill -> AR -> NAR -> Mimi -> host wav)",
                "ms_per_step": e2e_ms / args.steps, "rtf": (e2e_ms / 1e3) / (e2e_frames_all / W * 0.08),
                # whole job: every rank uploads its shard's text ids + noise tapes and downloads its waveforms
                "h2d_bytes_per_step": int(B * TEXT_LEN * 4 + B * STEPS_AR * 50 * 4) * W,
                "d2h_bytes_per_step": int(e2e_frames_all / args.steps) * 1920 * 4 + B * STEPS_AR * 4 * W},
        "gpu_launches": (2 * args.steps + api_launches * args.steps) * W,
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": traffic, "kernel": "ar_persistent_kernel<bf16>", "ms_per_launch": t_kernel_ms,
                     "alg_bytes_per_launch": alg_bytes_launch, "peak_source": peak_src,
                     "note": "algorithmic bytes = (W_step + B*3280) per AR step x 401 steps (SURVEY.md §8d); W_step is L2-resident "
                             "after the first step, so DRAM traffic is far below this",
                     # last committed ncu --set full capture of this kernel (not measured in this run)
                     "ncu_capture": ncu_note},
        "clocks": clocks.summary(),
        "extra": {"us_per_ar_step": t_kernel_ms / STEPS_AR * 1e3, "frames_per_pass_per_gpu": frames_per_pass,
                  "synthesize_batch_ms": e2e_ms / args.steps, "rtf_batch": (e2e_ms / 1e3) / (e2e_frames_all / W * 0.08),
                  "global_batch_rtf_note": "rtf = wall time of one synthesize_batch pass / seconds of audio ONE rank produced "
                                           "(ranks run in parallel; divide by n_gpus for the whole-job RTF)"},
    }
    if world == 1 and not args.no_extras:
        try:
            ex, mimi = extras(tts, ref, cfg, dev, peaks)
            line["extra"].update(ex)
            line["roofline_mimi"] = mimi
        except Exception as ex:  # the headline number must survive a failure in the side measurements
            line["extra"]["extras_error"] = repr(ex)
    if world > 1:  # the CPU baseline is measured at N=1 only (it does not depend on N)
        line["cpu_baseline"] = {"value": None, "unit": "frames/s", "cores": None, "kind": "reference",
                                "sample": "measured on rank 0 at N=1 only"}
    elif not args.no_cpu_baseline:
        line["cpu_baseline"] = cpu_baseline_block(CpuReference(cfg, sd), 12)
    emit(line)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
