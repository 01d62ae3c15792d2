"""Public API: ``SoproTTS`` with the reference's signatures (reference model.py:404-583) over the B200 engine.

``SoproTTS.model`` is a ``SoproModel``: it stands where the reference's ``SoproTTSModel`` stands
(model.py:53-401) and keeps its method names, but ``ar_stream`` drives the persistent CUDA kernel and the
codec decodes with the CUDA Mimi engine.  Prefill and the NAR refiner are torch ops on the same device
(sopro_b200/prefill.py).  There is no CPU path: constructing the model without a CUDA device raises.

Randomness: like the reference, sampling consumes the GLOBAL torch CPU generator (the reference has no seed
argument; its CLI calls torch.manual_seed, cli.py:72-75), one [V]-sized Exp(1) draw per generated frame, so
``torch.manual_seed(s); tts.synthesize(...)`` reproduces the reference's token ids.  Every generating method
additionally accepts ``seed=`` / ``generator=`` (an extension) to leave the global generator untouched.
"""
from __future__ import annotations

import os
import threading
from typing import Dict, Iterator, List, Optional, Sequence, Tuple

import torch

from . import prefill as P
from .codec import MimiCodec
from .config import TARGET_SR, SoproTTSConfig
from .engine import ArEngine, ArSession, Sampling
from .nar import NarEngine
from .prefill_cuda import PrefillEngine, RefPrepEngine
from .prefill import PreparedReference
from .weights import load_safetensors, read_safetensors_cfg


def center_crop_tokens(ref_tq: torch.Tensor, win_frames: int) -> torch.Tensor:
    """reference sampling.py:8-13"""
    T = int(ref_tq.size(0))
    if T <= win_frames:
        return ref_tq
    s = (T - win_frames) // 2
    return ref_tq[s: s + win_frames]


def _complete_state_dict(cfg: SoproTTSConfig, sd: Dict[str, torch.Tensor]) -> Dict[str, torch.Tensor]:
    """The reference loads with load_state_dict(strict=False) (model.py:443-446): tensors a checkpoint omits keep their
    module-init values.  The known omittable ones get those defaults here; anything else missing is ONE explicit error
    at construction instead of a KeyError deep inside the first synthesize call."""
    from .weights import param_specs

    Q = int(cfg.num_codebooks)
    tv = int(sd["text_enc.embed.emb.weight"].shape[0]) if "text_enc.embed.emb.weight" in sd else 0
    specs = param_specs(cfg, tv)
    out = dict(sd)
    missing = []
    for name, (shape, _kind, _fan) in specs.items():
        if name in out:
            continue
        if name in ("ref_cb_weights", "token2sv.cb_weights"):  # model.py:113-117, nn/speaker.py:22-23
            out[name] = torch.linspace(1.0, 0.1, Q)
        elif name == "nar_prev_cb_weights" or name.startswith("nar.head_id_emb."):  # model.py:70-72, nn/nar.py:79 (zeros)
            out[name] = torch.zeros(shape)
        else:
            missing.append(name)
    if missing:
        raise KeyError(f"checkpoint is missing {len(missing)} tensor(s) the engine needs: {missing[:12]}"
                       + (" ..." if len(missing) > 12 else ""))
    return out


_TAPE_POOL = None


def _tape_pool():
    """Host threads that draw noise tapes (the Exp(1) draws release the GIL)."""
    global _TAPE_POOL
    if _TAPE_POOL is None:
        from concurrent.futures import ThreadPoolExecutor

        _TAPE_POOL = ThreadPoolExecutor(max_workers=max(1, len(os.sched_getaffinity(0))))
    return _TAPE_POOL


_NATIVE_NOISE = None


def _native_noise_ok() -> bool:
    """The host-side mt19937 tape generator of the library (csrc/noise_host.cu) is used for private generators when it
    reproduces THIS torch build's CPU exponential_ bit for bit (checked once per process; a torch built with another
    sampling kernel falls back to torch itself)."""
    global _NATIVE_NOISE
    if _NATIVE_NOISE is None:
        try:
            import ctypes as C

            from . import _lib

            lib = _lib.load()
            h = C.c_void_p()
            _lib.check(lib.sopro_noise_create(C.c_uint64(987654321), C.byref(h)))
            got = torch.empty(3, 7)
            _lib.check(lib.sopro_noise_rows(h, 3, 97, 7, got.data_ptr()))
            lib.sopro_noise_destroy(h)
            want = torch.empty(3, 97).exponential_(1.0, generator=torch.Generator().manual_seed(987654321))[:, :7]
            _NATIVE_NOISE = bool(torch.equal(got, want))
        except Exception:
            _NATIVE_NOISE = False
    return _NATIVE_NOISE


class _Noise:
    """The Exp(1) draws `steps` successive torch.multinomial calls would consume (see sopro_b200/sampling.py),
    produced block by block as the kernel launches need them (a [n, V] draw equals n successive [V] draws), with
    the bookkeeping needed to leave the generator exactly where the reference would leave it."""

    def __init__(self, steps: int, vocab: int, seed: Optional[int], generator: Optional[torch.Generator]):
        self.steps, self.vocab = int(steps), int(vocab)
        self.private = seed is not None
        self.gen = torch.Generator().manual_seed(int(seed)) if seed is not None else (generator or torch.default_generator)
        self.marks: List[Tuple[int, torch.Tensor]] = []  # (first row of a block, generator state before it)
        self.drawn = 0
        self._native = None  # private generators: the library's host-side mt19937 (bit-equal to torch, skips unread draws)
        if seed is not None and int(seed) >= 0 and _native_noise_ok():  # (negative seeds: torch's own remapping, torch's path)
            import ctypes as C

            from . import _lib

            self._lib = _lib.load()
            h = C.c_void_p()
            _lib.check(self._lib.sopro_noise_create(C.c_uint64(int(seed) & 0xFFFFFFFFFFFFFFFF), C.byref(h)))
            self._native = h

    def __del__(self):
        if getattr(self, "_native", None) is not None:
            self._lib.sopro_noise_destroy(self._native)
            self._native = None

    def rows_keep(self, upto: int, keep: int) -> torch.Tensor:
        """Rows [drawn, upto), first `keep` columns -> [n, keep] (empty when already drawn)."""
        upto = min(int(upto), self.steps)
        n = upto - self.drawn
        if n <= 0:
            return torch.empty(0, int(keep))
        if self._native is not None:
            out = torch.empty(n, int(keep))
            self.rows_into(upto, keep, out.numpy())
            return out
        return self.rows(upto)[:, : int(keep)]

    def rows_into(self, upto: int, keep: int, out) -> None:
        """Rows [drawn, upto), first `keep` columns, written into the float32 numpy array `out` [n, keep] (C-contiguous)."""
        upto = min(int(upto), self.steps)
        n = upto - self.drawn
        if n <= 0:
            return
        if self._native is not None:
            assert out.flags["C_CONTIGUOUS"] and out.shape == (n, keep)
            from . import _lib

            _lib.check(self._lib.sopro_noise_rows(self._native, n, self.vocab, int(keep), out.ctypes.data))
            self.drawn = upto
        else:
            out[...] = self.rows(upto)[:, :keep].numpy()

    def rows(self, upto: int) -> torch.Tensor:
        """Draw rows [drawn, upto) -> [n, V] (empty when already drawn)."""
        upto = min(int(upto), self.steps)
        n = upto - self.drawn
        if n <= 0:
            return torch.empty(0, self.vocab)
        if not self.private:
            self.marks.append((self.drawn, self.gen.get_state()))
        if self._native is not None:
            out = torch.empty(n, self.vocab)
            self.rows_into(upto, self.vocab, out.numpy())
            return out
        self.drawn = upto
        return torch.empty(n, self.vocab).exponential_(1.0, generator=self.gen)

    @property
    def tape(self) -> torch.Tensor:
        """All rows at once (only valid before any block has been drawn)."""
        assert self.drawn == 0
        return self.rows(self.steps)

    def settle(self, steps_used: int) -> None:
        """Rewind to the state after exactly `steps_used` draws (the reference stops drawing when it stops stepping)."""
        if self.private or steps_used >= self.drawn:
            return
        start, state = [m for m in self.marks if m[0] <= steps_used][-1]
        self.gen.set_state(state)
        if steps_used > start:
            torch.empty(int(steps_used - start), self.vocab).exponential_(1.0, generator=self.gen)
        self.drawn = int(steps_used)


class SoproModel:
    def __init__(self, cfg: SoproTTSConfig, state_dict: Dict[str, torch.Tensor], device, weight_dtype: str = "fp32"):
        dev = torch.device(device)
        if dev.type != "cuda":
            raise RuntimeError("sopro_b200 runs on CUDA devices only (sm_100a); there is no CPU fallback")
        self.cfg = cfg
        state_dict = _complete_state_dict(cfg, state_dict)
        self.device = torch.device("cuda", dev.index if dev.index is not None else torch.cuda.current_device())
        self.eos_id = int(cfg.codebook_size)
        self.weight_dtype = weight_dtype
        self.engine = ArEngine(cfg, state_dict, self.device, weight_dtype)
        # (every stage owns its device copy of the weights it needs inside its CUDA engine; no torch-side copy is kept)
        self.text_pos = P.sinusoid_table(int(cfg.max_text_len) + 8, int(cfg.d_model), self.device)
        self.frame_pos = P.sinusoid_table(int(cfg.pos_emb_max) + 8, int(cfg.d_model), self.device)
        # AR sessions are CHECKED OUT per generator / call and returned when it ends (ar_stream is a suspended
        # generator: two interleaved streams must never share a session's device state)
        self._sessions: Dict[Tuple[int, int, int], List[ArSession]] = {}
        self._sessions_busy: set = set()
        self._sessions_lock = threading.Lock()
        self.prefill = PrefillEngine(cfg, state_dict, self.device, self.text_pos, self.frame_pos)
        self.refprep = RefPrepEngine(cfg, state_dict, self.device)
        self.nar = NarEngine(cfg, state_dict, self.device)

    # ---- geometry helpers (reference model.py:119-131)
    def rf_ar(self) -> int:
        return self.cfg.rf_ar()

    def rf_nar(self) -> int:
        return self.cfg.rf_nar()

    def eval(self):
        return self

    def _checkout(self, batch: int, steps: int, text_len: int) -> ArSession:
        """An idle session of this geometry (a fresh one when every cached one is in use); pair with _release."""
        key = (int(batch), int(steps), (int(text_len) + 63) // 64 * 64)
        with self._sessions_lock:
            for ses in self._sessions.get(key, []):
                if id(ses) not in self._sessions_busy:
                    self._sessions_busy.add(id(ses))
                    return ses
            # evict idle sessions of other geometries beyond 8 cached (never one a live generator holds)
            idle = [(k, x) for k, v in self._sessions.items() for x in v if id(x) not in self._sessions_busy and k != key]
            total = sum(len(v) for v in self._sessions.values())
            while total >= 8 and idle:
                k, x = idle.pop(0)
                self._sessions[k].remove(x)
                x.close()
                total -= 1
            ses = self.engine.session(*key)
            self._sessions.setdefault(key, []).append(ses)
            self._sessions_busy.add(id(ses))
            return ses

    def _release(self, ses: ArSession) -> None:
        with self._sessions_lock:
            self._sessions_busy.discard(id(ses))

    # ---- prefill
    @torch.no_grad()
    def prepare_reference(self, ref_tokens_tq: torch.Tensor, *, device=None) -> PreparedReference:
        """reference model.py:152-170 on the CUDA reference-preparation engine (Token2SV, reference encoder, cached K/V)."""
        ref_btq = ref_tokens_tq.unsqueeze(0).to(device=self.device, dtype=torch.long)
        sv, seq, caches = self.refprep.run(ref_btq[0])
        return PreparedReference(ref_tokens_btq=ref_btq, sv_ref=sv, ref_seq=seq, ref_kv_caches=caches)

    @torch.no_grad()
    def speaker_vector(self, ref_tokens_tq: torch.Tensor) -> torch.Tensor:
        """Token2SV alone (SoproTTS.encode_speaker, reference model.py:458-475) -> [sv_dim]"""
        return self.refprep.run(ref_tokens_tq.to(self.device))[0].squeeze(0)

    @torch.no_grad()
    def prepare_conditioning(self, text_ids_1d: torch.Tensor, ref: PreparedReference, *, max_frames: int, device=None,
                             style_strength: float = 1.2) -> Dict[str, torch.Tensor]:
        """reference model.py:174-216 on the CUDA prefill engine (sopro_b200/csrc/nar_engine.cu: ~25 fused fp32 kernels)."""
        return self.prepare_conditioning_batch([text_ids_1d], ref, max_frames=max_frames, style_strength=style_strength)[0]

    @torch.no_grad()
    def prepare_conditioning_batch(self, text_ids: Sequence[torch.Tensor], ref: Optional[PreparedReference] = None, *,
                                   refs: Optional[Sequence[PreparedReference]] = None, max_frames: int,
                                   style_strength: float = 1.2) -> List[Dict[str, torch.Tensor]]:
        """NEW (the reference is batch-1): the prefill of B texts in ONE pass, all with the prepared reference `ref`, or
        text i with its own `refs[i]` (exactly one of the two); element i is the `prep` dict of model.py:210-216 for
        text i (views into the batch tensors)."""
        txt_seq, lens, txt_pool, cond = self.prefill_batch(text_ids, ref, refs, n_frames=int(max_frames) + 1,
                                                           style_strength=float(style_strength))
        svs: Dict[int, torch.Tensor] = {}
        out = []
        for i, L in enumerate(lens):
            r = ref if refs is None else refs[i]
            if id(r) not in svs:
                sv = r.sv_ref.to(self.device)
                svs[id(r)] = sv.unsqueeze(0) if sv.dim() == 1 else sv
            out.append({"txt_seq": txt_seq[i: i + 1, :L], "text_mask": torch.ones((1, L), dtype=torch.bool, device=self.device),
                        "txt_pool": txt_pool[i: i + 1], "sv_ref": svs[id(r)], "cond_ar": cond[i: i + 1]})
        return out

    def prefill_batch(self, text_ids: Sequence[torch.Tensor], ref: Optional[PreparedReference],
                      refs: Optional[Sequence[PreparedReference]], *, n_frames: int, style_strength: float):
        """The batched CUDA prefill with one voice for every text (`ref`) or a voice per text (`refs`, told apart by
        object identity); exactly one of the two.  -> txt_seq [B, Lmax, D], lens, txt_pool [B, D], cond_ar [B, n_frames, D]."""
        if (ref is None) == (refs is None):
            raise ValueError("pass exactly one of ref= (one voice for every text) or refs= (one voice per text)")
        if refs is None:
            return self.prefill.run(text_ids, ref, n_frames=n_frames, style_strength=style_strength)
        if len(refs) != len(text_ids):
            raise ValueError(f"refs has {len(refs)} entries for {len(text_ids)} texts")
        return self.prefill.run_voices(text_ids, list(refs), n_frames=n_frames, style_strength=style_strength)

    @torch.no_grad()
    def nar_refine(self, cond_seq: torch.Tensor, rvq1_1xT: torch.Tensor, lens: Optional[torch.Tensor] = None) -> torch.Tensor:
        """reference model.py:307-347 on the CUDA NAR engine (sopro_b200/csrc/nar_engine.cu): 4 stage passes of fused fp32
        kernels, ids equal to the reference's.  cond [B, T, D], rvq1 [B, T] -> [B, T, Q] int64.  `lens` (extension):
        valid frames per utterance of a ragged batch (the refiner is not causal)."""
        if int(cond_seq.size(1)) == 0:
            return torch.zeros((int(cond_seq.size(0)), 0, int(self.cfg.num_codebooks)), dtype=torch.long, device=self.device)
        return self.nar.refine(cond_seq, rvq1_1xT, lens)

    # ---- the hot path
    def _sampling(self, top_p, temperature, anti_loop, loop_streak, recovery_top_p, recovery_temp, min_gen_frames,
                  stop_on_first_eos) -> Sampling:
        mg = int(min_gen_frames if min_gen_frames is not None else self.cfg.min_gen_frames)
        # top_p=None is legal in the reference (sampling.py:69: `top_p is not None and top_p < 1.0`) == no top-p
        top_p = 1.0 if top_p is None else top_p
        recovery_top_p = 1.0 if recovery_top_p is None else recovery_top_p
        return Sampling(top_p=float(top_p), temperature=float(temperature), recovery_top_p=float(recovery_top_p),
                        recovery_temp=float(recovery_temp), repetition_penalty=1.1, top_k=50, anti_loop=bool(anti_loop),
                        loop_streak=int(loop_streak), min_gen_frames=min(mg, 2 ** 31 - 1), stop_on_first_eos=stop_on_first_eos)

    def _noise_cols(self, samp: Sampling) -> int:
        """Exp(1) draws per step the kernel reads: the top_k sorted ranks with top-p (sampling.py:83-84), every
        vocabulary id on the unsorted multinomial branch taken when top_p >= 1 (sampling.py:88-93)."""
        return int(samp.top_k) if (samp.top_p < 1.0 and samp.recovery_top_p < 1.0) else int(self.cfg.ar_vocab())

    @torch.no_grad()
    def ar_chunks(self, prep: Dict[str, torch.Tensor], *, max_frames: int, chunk_frames: int = 0, top_p: float = 0.9,
                  temperature: float = 1.05, anti_loop: bool = True, loop_streak: int = 8, recovery_top_p: float = 0.85,
                  recovery_temp: float = 1.2, min_gen_frames: Optional[int] = None, seed: Optional[int] = None,
                  generator: Optional[torch.Generator] = None, progress: Optional[dict] = None):
        """The persistent kernel driven `chunk_frames` frames per launch (0 = the whole utterance in one launch).
        Yields ``(tokens, finished, prefetch)`` per launch: the frames it produced (ints), whether the utterance is over
        (EOS past min_gen_frames, or max_frames reached), and a callable that enqueues the NEXT launch right away on the
        current CUDA stream -- a streaming consumer queues it behind its own NAR + Mimi work so it runs while the audio is
        handed out; without the call the next launch is enqueued when the generator is resumed.  Frames computed ahead
        of a consumer that stops early are abandoned: on exit the RNG is settled to ``progress["consumed"]`` frames
        (default: every frame yielded), i.e. exactly the draws the reference would have made."""
        cond, txt = prep["cond_ar"], prep["txt_seq"]
        steps = int(max_frames) + 1
        if cond.size(1) < steps:
            raise ValueError(f"cond_ar has {cond.size(1)} rows, need max_frames+1 = {steps}")
        L = int(txt.size(1))
        noise = _Noise(steps, self.cfg.ar_vocab(), seed, generator)
        samp = self._sampling(top_p, temperature, anti_loop, loop_streak, recovery_top_p, recovery_temp, min_gen_frames, False)
        nk = self._noise_cols(samp)
        ses = self._checkout(1, steps, L)
        per = steps if chunk_frames <= 0 else int(chunk_frames)
        st = {"launched": 0, "read": 0, "yielded": 0}

        def launch():
            """Draw + upload the noise rows of the next launch and enqueue it (no-op while one is in flight)."""
            if st["launched"] >= steps or st["launched"] > st["read"]:
                return
            lo = noise.drawn
            blk = noise.rows_keep(st["launched"] + per, nk)
            if blk.size(0):
                n_new = int(blk.size(0))
                if stage is not None:  # pinned staging rows: the upload is asynchronous, ordered before the launch on this stream
                    stage[lo: lo + n_new].copy_(blk)
                    tape[0, lo: lo + n_new].copy_(stage[lo: lo + n_new], non_blocking=True)
                else:
                    tape[0, lo: lo + n_new].copy_(blk)
            ses.run(per)
            st["launched"] = min(steps, st["launched"] + per)

        try:
            # the session keeps a pointer to this device tape; each launch's rows are drawn and uploaded just before it
            tape = torch.zeros(1, steps, nk, device=self.device)
            stage = torch.empty(steps, nk, pin_memory=True) if self.device.type == "cuda" else None
            ses.begin(cond[:, :steps], txt, [L], tape, samp)
            t = 0
            while t < steps:
                launch()
                toks, n, done = ses.read()  # synchronises the stream the launch ran on
                upto = int(n[0])
                st["read"] = st["launched"]
                chunk = [int(x) for x in toks[0, t:upto]]
                finished = bool(done[0]) or upto >= steps or upto < st["launched"]
                t = upto
                st["yielded"] = upto
                yield chunk, finished, (launch if not finished else (lambda: None))
                if finished:
                    break
        finally:
            self._release(ses)
            noise.settle(int(progress["consumed"]) if progress is not None and "consumed" in progress else st["yielded"])

    @torch.no_grad()
    def ar_stream(self, prep: Dict[str, torch.Tensor], *, max_frames: int, top_p: float = 0.9, temperature: float = 1.05,
                  anti_loop: bool = True, loop_streak: int = 8, recovery_top_p: float = 0.85, recovery_temp: float = 1.2,
                  min_gen_frames: Optional[int] = None, launch_frames: int = 0, seed: Optional[int] = None,
                  generator: Optional[torch.Generator] = None) -> Iterator[Tuple[int, int, bool]]:
        """Yields (t, token, is_eos) like the reference generator (model.py:218-305).  The persistent kernel runs
        `launch_frames` frames per launch (0 = the whole utterance in one launch); a consumer that stops iterating
        early simply abandons the frames computed ahead, and the RNG is settled to the frames actually consumed."""
        progress = {"consumed": 0}
        gen = self.ar_chunks(prep, max_frames=max_frames, chunk_frames=launch_frames, top_p=top_p, temperature=temperature,
                             anti_loop=anti_loop, loop_streak=loop_streak, recovery_top_p=recovery_top_p,
                             recovery_temp=recovery_temp, min_gen_frames=min_gen_frames, seed=seed, generator=generator,
                             progress=progress)
        t = 0
        try:
            for chunk, _finished, _prefetch in gen:
                for tok in chunk:
                    progress["consumed"] = t + 1
                    yield t, tok, tok == self.eos_id
                    t += 1
        finally:
            gen.close()

    def _draw_tapes(self, B: int, steps: int, nk: int, seeds: Optional[Sequence[int]]) -> torch.Tensor:
        """[B, steps, nk] Exp(1) draws: utterance i's rows are what `steps` multinomial calls consume after
        torch.manual_seed(seeds[i]) (private generators, drawn on host threads -- the draws release the GIL); without
        seeds the global generator is consumed utterance after utterance, full length each."""
        V = self.cfg.ar_vocab()
        out = torch.empty((B, steps, nk), dtype=torch.float32, pin_memory=torch.cuda.is_available())
        if seeds is None:
            for i in range(B):
                out[i] = _Noise(steps, V, None, None).tape[:, :nk]
            return out
        from concurrent.futures import ThreadPoolExecutor

        view = out.numpy()  # worker threads are outside the caller's inference_mode: write through numpy

        def one(i):
            _Noise(steps, V, int(seeds[i]), None).rows_into(steps, nk, view[i])

        with ThreadPoolExecutor(max_workers=min(B, max(1, len(os.sched_getaffinity(0))))) as ex:
            list(ex.map(one, range(B)))
        return out

    @torch.no_grad()
    def ar_generate_tensors(self, cond: torch.Tensor, txt: torch.Tensor, lens: Sequence[int], *, max_frames: int, top_p: float = 0.9,
                            temperature: float = 1.05, anti_loop: bool = True, min_gen_frames: Optional[int] = None,
                            seeds: Optional[Sequence[int]] = None, stop_on_first_eos: bool = True):
        """B utterances in ONE persistent launch from batch tensors (cond [B, >=steps, D], txt [B, Lmax, D], lens).
        -> (tokens [B, steps] int32 numpy, n_tokens [B])."""
        B, steps = int(cond.shape[0]), int(max_frames) + 1
        samp = self._sampling(top_p, temperature, anti_loop, 8, 0.85, 1.2, min_gen_frames, stop_on_first_eos)
        nk = self._noise_cols(samp)
        ses = self._checkout(B, steps, max(int(x) for x in lens))
        try:
            if seeds is None or steps < 64:
                tapes = self._draw_tapes(B, steps, nk, seeds)  # host threads; the prefill kernels queued before run meanwhile
                ses.begin(cond[:, :steps], txt, [int(x) for x in lens], tapes.to(self.device, non_blocking=True), samp)
                ses.run()
            else:
                # Private generators: the tape is drawn in growing blocks of steps and the persistent kernel is launched
                # block by block (it resumes from its device state), so the host draws block k+1 while the device
                # generates block k; only the first, short block is exposed (and that one overlaps the prefill).
                V = self.cfg.ar_vocab()
                gens = [_Noise(steps, V, int(seeds[i]), None) for i in range(B)]
                host = torch.empty((B, steps, nk), dtype=torch.float32, pin_memory=torch.cuda.is_available())
                view = host.numpy()
                dev = torch.empty((B, steps, nk), dtype=torch.float32, device=self.device)
                pool = _tape_pool()

                def draw(a: int, b: int) -> None:
                    def one(i):
                        gens[i].rows_into(b, nk, view[i, a:b])
                    list(pool.map(one, range(B)))
                    dev[:, a:b].copy_(host[:, a:b], non_blocking=True)

                # block k+1 must be drawn faster than the device generates block k: the host draws ~10 steps per ms
                # (64 utterances, 16 threads), the kernel runs ~6 steps per ms -> blocks grow by 1.5x
                edges, a, step = [], 0, 24
                while a < steps:
                    b = min(steps, a + step)
                    if steps - b < 24:
                        b = steps
                    edges.append((a, b))
                    a, step = b, (step * 3) // 2
                draw(*edges[0])
                ses.begin(cond[:, :steps], txt, [int(x) for x in lens], dev, samp)
                ses.run(edges[0][1])
                for a, b in edges[1:]:
                    draw(a, b)
                    ses.run(b - a)
            toks, n, _ = ses.read()
        finally:
            self._release(ses)
        return toks, n

    @torch.no_grad()
    def ar_generate_batch(self, preps: Sequence[Dict[str, torch.Tensor]], *, max_frames: int, top_p: float = 0.9,
                          temperature: float = 1.05, anti_loop: bool = True, min_gen_frames: Optional[int] = None,
                          seeds: Optional[Sequence[int]] = None, stop_on_first_eos: bool = True) -> List[List[int]]:
        """NEW capability (the reference is batch-1): B independent utterances in ONE persistent launch.  Utterance i
        equals the reference run alone with seed seeds[i] (SURVEY.md §0.3).  Without seeds the global generator is
        consumed utterance after utterance, full length each."""
        B, steps = len(preps), int(max_frames) + 1
        D = int(self.cfg.d_model)
        lens = [int(p["txt_seq"].size(1)) for p in preps]
        cond = torch.stack([p["cond_ar"][0, :steps] for p in preps])
        txt = torch.zeros(B, max(lens), D, device=self.device)
        for i, p in enumerate(preps):
            txt[i, : lens[i]] = p["txt_seq"][0]
        toks, n = self.ar_generate_tensors(cond, txt, lens, max_frames=max_frames, top_p=top_p, temperature=temperature,
                                           anti_loop=anti_loop, min_gen_frames=min_gen_frames, seeds=seeds,
                                           stop_on_first_eos=stop_on_first_eos)
        return [toks[i, : n[i]].tolist() for i in range(B)]

    @torch.no_grad()
    def generate_tokens(self, text_ids_1d: torch.Tensor, ref: PreparedReference, *, max_frames: int, device=None,
                        top_p: float = 0.9, temperature: float = 1.05, anti_loop: bool = True, style_strength: float = 1.2,
                        min_gen_frames: Optional[int] = None, seed: Optional[int] = None,
                        generator: Optional[torch.Generator] = None) -> torch.Tensor:
        """reference model.py:349-401: prefill, AR until the first EOS, cut there, NAR refine -> [T, Q] int64."""
        prep = self.prepare_conditioning(text_ids_1d, ref, max_frames=max_frames, style_strength=style_strength)
        hist: List[int] = []
        for _t, tok, is_eos in self.ar_stream(prep, max_frames=max_frames, top_p=top_p, temperature=temperature,
                                              anti_loop=anti_loop, min_gen_frames=min_gen_frames, seed=seed, generator=generator):
            hist.append(tok)
            if is_eos:
                break
        T = hist.index(self.eos_id) if self.eos_id in hist else len(hist)
        if T <= 0:
            return torch.zeros((0, int(self.cfg.num_codebooks)), dtype=torch.long, device=self.device)
        rvq1 = torch.tensor(hist[:T], device=self.device, dtype=torch.long).unsqueeze(0)
        return self.nar_refine(prep["cond_ar"][:, :T, :], rvq1).squeeze(0)


class SoproTTS:
    def __init__(self, model: SoproModel, cfg: SoproTTSConfig, tokenizer, codec: MimiCodec, device: str):
        self.model = model
        self.cfg = cfg
        self.tokenizer = tokenizer
        self.codec = codec
        self.device = torch.device(device)

    # ---- construction
    @classmethod
    def from_pretrained(cls, repo_id: str, *, revision: Optional[str] = None, cache_dir: Optional[str] = None,
                        token: Optional[str] = None, device: Optional[str] = None, weight_dtype: str = "fp32",
                        mimi_precision: str = "bf16_tc") -> "SoproTTS":
        """reference model.py:419-451: HF snapshot -> cfg from the safetensors header -> tokenizer -> weights -> Mimi."""
        from huggingface_hub import snapshot_download

        from .tokenizer import TextTokenizer

        device = device or "cuda"
        local_dir = repo_id if os.path.isdir(repo_id) else snapshot_download(repo_id=repo_id, revision=revision,
                                                                             cache_dir=cache_dir, token=token)
        model_path = os.path.join(local_dir, "model.safetensors")
        if not os.path.exists(model_path):
            raise FileNotFoundError(f"Expected {model_path} in repo snapshot.")
        cfg = read_safetensors_cfg(model_path)
        tokenizer = TextTokenizer(model_name=local_dir)
        model = SoproModel(cfg, load_safetensors(model_path), device, weight_dtype)
        codec = MimiCodec(num_quantizers=cfg.num_codebooks, device=device, precision=mimi_precision)
        return cls(model=model, cfg=cfg, tokenizer=tokenizer, codec=codec, device=device)

    @classmethod
    def from_state_dict(cls, cfg: SoproTTSConfig, state_dict: Dict[str, torch.Tensor], tokenizer,
                        mimi_state_dict: Dict[str, torch.Tensor], *, device: str = "cuda", weight_dtype: str = "fp32",
                        mimi_hf_model=None, mimi_precision: str = "bf16_tc") -> "SoproTTS":
        """Offline constructor (synthetic or locally stored checkpoints): no hub access."""
        model = SoproModel(cfg, state_dict, device, weight_dtype)
        codec = MimiCodec(int(cfg.num_codebooks), device=device, state_dict=mimi_state_dict, hf_model=mimi_hf_model,
                          precision=mimi_precision)
        return cls(model=model, cfg=cfg, tokenizer=tokenizer, codec=codec, device=device)

    # ---- reference plumbing (model.py:453-529)
    def encode_text(self, text: str) -> torch.Tensor:
        return torch.tensor(self.tokenizer.encode(text), dtype=torch.long, device=self.device)

    def encode_reference(self, *, ref_audio_path: Optional[str] = None, ref_tokens_tq: Optional[torch.Tensor] = None,
                         ref_seconds: Optional[float] = None) -> torch.Tensor:
        if ref_tokens_tq is None and ref_audio_path is None:
            raise RuntimeError("SoproTTS requires a reference. Provide ref_audio_path=... or ref_tokens_tq=...")
        if ref_tokens_tq is not None and ref_audio_path is not None:
            raise RuntimeError("Provide only one of ref_audio_path or ref_tokens_tq (not both).")
        if ref_seconds is None:
            ref_seconds = 12.0
        if ref_tokens_tq is not None:
            ref = ref_tokens_tq.to(self.device).long()
            if ref_seconds and ref_seconds > 0:
                ref = center_crop_tokens(ref, max(1, int(round(ref_seconds * float(self.cfg.mimi_fps)))))
            return ref
        crop = ref_seconds if ref_seconds is not None and ref_seconds > 0 else None
        return self.codec.encode_file(ref_audio_path, crop_seconds=crop).to(self.device).long()

    @torch.inference_mode()
    def encode_speaker(self, **kw) -> torch.Tensor:
        return self.model.speaker_vector(self.encode_reference(**kw)).detach()

    @torch.inference_mode()
    def prepare_reference(self, *, ref_audio_path: Optional[str] = None, ref_tokens_tq: Optional[torch.Tensor] = None,
                          ref_seconds: Optional[float] = None) -> PreparedReference:
        tokens_tq = self.encode_reference(ref_audio_path=ref_audio_path, ref_tokens_tq=ref_tokens_tq, ref_seconds=ref_seconds)
        return self.model.prepare_reference(tokens_tq, device=self.device)

    # ---- synthesis (model.py:531-580)
    @torch.inference_mode()
    def synthesize(self, text: str, *, ref: Optional[PreparedReference] = None, ref_audio_path: Optional[str] = None,
                   ref_tokens_tq: Optional[torch.Tensor] = None, max_frames: int = 400, top_p: float = 0.9,
                   temperature: float = 1.05, anti_loop: bool = True, style_strength: Optional[float] = None,
                   ref_seconds: Optional[float] = None, min_gen_frames: Optional[int] = None, seed: Optional[int] = None,
                   generator: Optional[torch.Generator] = None) -> torch.Tensor:
        text_ids = self.encode_text(text)
        if ref is None:
            ref = self.prepare_reference(ref_audio_path=ref_audio_path, ref_tokens_tq=ref_tokens_tq, ref_seconds=ref_seconds)
        tokens_tq = self.model.generate_tokens(
            text_ids, ref=ref, max_frames=max_frames, top_p=top_p, temperature=temperature, anti_loop=anti_loop,
            style_strength=float(style_strength if style_strength is not None else self.cfg.style_strength),
            min_gen_frames=min_gen_frames, seed=seed, generator=generator)
        return self.codec.decode_full(tokens_tq)

    @torch.inference_mode()
    def synthesize_batch(self, texts: Sequence[str], *, ref: Optional[PreparedReference] = None,
                         refs: Optional[Sequence[PreparedReference]] = None, max_frames: int = 400, top_p: float = 0.9,
                         temperature: float = 1.05, anti_loop: bool = True, style_strength: Optional[float] = None,
                         min_gen_frames: Optional[int] = None, seeds: Optional[Sequence[int]] = None) -> List[torch.Tensor]:
        """NEW: B texts -> B waveforms [1, 1, N_i], all in the voice of one prepared reference `ref`, or text i in the
        voice of its own `refs[i]` (exactly one of the two; a server caching one PreparedReference per user passes the
        cached objects, repeated ones are recognised by identity).  One batched prefill, one persistent AR launch, one
        ragged NAR pass, padded Mimi decodes; utterance i equals synthesize(texts[i], ref=(ref or refs[i]), seed=seeds[i])."""
        st = float(style_strength if style_strength is not None else self.cfg.style_strength)
        model = self.model
        ids = [self.encode_text(t) for t in texts]
        txt_seq, lens, _pool, cond = model.prefill_batch(ids, ref, refs, n_frames=int(max_frames) + 1, style_strength=st)
        toks, n = model.ar_generate_tensors(cond, txt_seq, lens, max_frames=max_frames, top_p=top_p, temperature=temperature,
                                            anti_loop=anti_loop, min_gen_frames=min_gen_frames, seeds=seeds)
        eos, B = model.eos_id, len(texts)
        Ts = []
        for i in range(B):
            row = toks[i, : n[i]]
            hit = (row == eos).nonzero()[0]
            Ts.append(int(hit[0]) if hit.size else int(n[i]))
        out: List[torch.Tensor] = [torch.zeros(1, 1, 0, device=self.device) for _ in texts]
        Tmax = max(Ts)
        if Tmax == 0:
            return out
        # NAR refiner over the ragged batch (not causal: `lens` makes the padding act as each utterance's zero padding)
        rvq1 = torch.from_numpy(toks[:, :Tmax].copy()).to(self.device)
        codes = model.nar_refine(cond[:, :Tmax], rvq1.clamp_(0, eos - 1), lens=torch.tensor(Ts, dtype=torch.int32))  # [B, Tmax, Q]
        # Mimi decode is causal and per-utterance: right-pad to the longest of a chunk, decode together, cut
        live = sorted((i for i in range(B) if Ts[i] > 0), key=lambda i: -Ts[i])
        hop = self.codec.engine.hop
        cap = 12800  # frames per decode call (workspace bound)
        while live:
            chunk, frames = [], 0
            while live and (not chunk or (len(chunk) + 1) * max(frames, Ts[live[0]]) <= cap):
                frames = max(frames, Ts[live[0]])
                chunk.append(live.pop(0))
            idx = torch.tensor(chunk, device=self.device)
            batch = codes[idx, :frames].permute(0, 2, 1).to(torch.int32)
            keep = torch.arange(frames, device=self.device)[None, :] < torch.tensor([Ts[i] for i in chunk], device=self.device)[:, None]
            batch = (batch * keep[:, None, :]).contiguous()  # padding frames decode code 0; their samples are cut below
            wav = self.codec.engine.decode(batch)
            for j, i in enumerate(chunk):
                out[i] = wav[j: j + 1, :, : Ts[i] * hop].clone()
        return out

    def stream(self, text: str, **kwargs) -> Iterator[torch.Tensor]:
        from .streaming import stream as _stream

        return _stream(self, text, **kwargs)

    def save_wav(self, path: str, wav_1xT: torch.Tensor) -> None:
        from .audio import save_audio

        save_audio(path, wav_1xT, sr=TARGET_SR)
