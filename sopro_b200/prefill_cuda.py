"""Host side of the CUDA prefill (libsopro_b200.so: sopro_prefill_*; reference model.py:172-216): text encoder,
FiLM, cached reference cross-attention and cond_norm for B texts that share one prepared reference voice (`run`) or
each bring their own (`run_voices`) -- and of the once-per-voice reference preparation in front of it (sopro_refprep_*;
reference model.py:152-170)."""
from __future__ import annotations

import ctypes as C
from typing import Dict, List, Sequence

import torch

from . import _lib
from .config import SoproTTSConfig
from .nar import _f32, fill_ssm_block


class PrefillEngine:
    def __init__(self, cfg: SoproTTSConfig, state_dict: Dict[str, torch.Tensor], device, text_pos: torch.Tensor,
                 frame_pos: torch.Tensor):
        self.lib = _lib.load()
        dev = torch.device(device if not isinstance(device, int) else f"cuda:{device}")
        if dev.type != "cuda":
            raise _lib.SoproError("PrefillEngine needs a CUDA device; there is no CPU path")
        self.device = torch.device("cuda", dev.index if dev.index is not None else 0)
        self.cfg = cfg
        sd = state_dict
        c = _lib.PrefillConfig()
        c.d_model, c.n_layers_text = int(cfg.d_model), int(cfg.n_layers_text)
        c.text_kernel = int(sd["text_enc.layers.0.dw.dw.weight"].shape[-1]) if c.n_layers_text > 0 else 7
        c.text_vocab = int(sd["text_enc.embed.emb.weight"].shape[0])
        c.sv_dim = int(sd["spk_film.mlp.0.weight"].shape[1])
        c.ref_layers, c.ref_heads, c.ref_gmax = int(cfg.ref_xattn_layers), int(cfg.ref_xattn_heads), float(cfg.ref_xattn_gmax)
        c.max_text_len, c.max_frames_pos = int(text_pos.shape[0]), int(frame_pos.shape[0])
        keep: list = []

        def ptr(t: torch.Tensor):
            t = _f32(t)
            keep.append(t)
            return C.cast(t.data_ptr(), C.POINTER(C.c_float))

        w = _lib.PrefillWeights()
        w.text_emb, w.text_pos, w.frame_pos = ptr(sd["text_enc.embed.emb.weight"]), ptr(text_pos), ptr(frame_pos)
        for i in range(c.n_layers_text):
            fill_ssm_block(w.text_block[i], sd, f"text_enc.layers.{i}.", keep)
        w.text_norm_w = ptr(sd["text_enc.norm.weight"])
        w.film_w0, w.film_b0 = ptr(sd["spk_film.mlp.0.weight"]), ptr(sd["spk_film.mlp.0.bias"])
        w.film_w2, w.film_b2 = ptr(sd["spk_film.mlp.2.weight"]), ptr(sd["spk_film.mlp.2.bias"])
        w.film_norm_w, w.film_norm_b = ptr(sd["spk_film.norm.weight"]), ptr(sd["spk_film.norm.bias"])
        for i in range(c.ref_layers):
            p = f"ref_xattn.blocks.{i}."
            w.ref_layer[i].nq_w, w.ref_layer[i].q_w = ptr(sd[p + "nq.weight"]), ptr(sd[p + "q_proj.weight"])
            w.ref_layer[i].o_w, w.ref_layer[i].gate = ptr(sd[p + "out_proj.weight"]), float(sd[p + "gate"])
        w.cond_norm_w = ptr(sd["cond_norm.weight"])
        h = C.c_void_p()
        _lib.check(self.lib.sopro_prefill_create(C.byref(c), C.byref(w), self.device.index, C.byref(h)))
        self._h = h
        self.D, self.n_ref = int(cfg.d_model), int(c.ref_layers)
        self.max_text_len, self.sv_dim = int(c.max_text_len), int(c.sv_dim)
        del keep

    def run(self, text_ids: Sequence[torch.Tensor], ref, *, n_frames: int, style_strength: float):
        """text_ids: B 1-D id tensors; ref: PreparedReference (shared).  -> txt_seq [B, Lmax, D], lens (list),
        txt_pool [B, D], cond_ar [B, n_frames, D] on the device."""
        B = len(text_ids)
        ids, ln, lens, Lmax = self._texts(text_ids)
        sv = ref.sv_ref.to(self.device, torch.float32).reshape(-1, ref.sv_ref.shape[-1]).contiguous()
        ks, vs, Tr = self._ref_kv(ref)
        kp = (C.c_void_p * max(1, self.n_ref))(*[int(k.data_ptr()) for k in ks])
        vp = (C.c_void_p * max(1, self.n_ref))(*[int(v.data_ptr()) for v in vs])
        txt_seq = torch.empty((B, Lmax, self.D), dtype=torch.float32, device=self.device)
        txt_pool = torch.empty((B, self.D), dtype=torch.float32, device=self.device)
        cond = torch.empty((B, int(n_frames), self.D), dtype=torch.float32, device=self.device)
        _lib.check(self.lib.sopro_prefill_run(self._h, ids.data_ptr(), ln.data_ptr(), B, Lmax, sv.data_ptr(), 1 if sv.shape[0] == 1 else 0,
                                              kp, vp, Tr, float(style_strength), int(n_frames), txt_seq.data_ptr(), txt_pool.data_ptr(),
                                              cond.data_ptr(), int(torch.cuda.current_stream(self.device).cuda_stream)))
        self._keep = (ids, ln, sv, ks, vs)  # alive until the stream has consumed them
        return txt_seq, lens, txt_pool, cond

    def run_voices(self, text_ids: Sequence[torch.Tensor], refs: Sequence, *, n_frames: int, style_strength: float):
        """text_ids: B 1-D id tensors; refs: B PreparedReference, text i conditioned on refs[i] (the same object may
        appear several times: voices are told apart by identity).  -> as `run`.  Utterance i is bit-equal to `run` on
        the same texts with refs[i] shared by all of them."""
        B = len(text_ids)
        if len(refs) != B:
            raise ValueError(f"{len(refs)} references for {B} texts")
        slot: Dict[int, int] = {}
        voices: list = []
        voice = []
        for r in refs:
            if id(r) not in slot:
                slot[id(r)] = len(voices)
                voices.append(r)
            voice.append(slot[id(r)])
        ids, ln, lens, Lmax = self._texts(text_ids)
        nv = len(voices)
        sv = torch.stack([r.sv_ref.to(self.device, torch.float32).reshape(-1) for r in voices])
        if sv.shape[1] != self.sv_dim:
            raise ValueError(f"a prepared reference holds ONE speaker vector of {self.sv_dim} values")
        kv = [self._ref_kv(r) for r in voices]  # per voice: ([K of each layer], [V of each layer], Tr)
        # entry l * n_voices + v: voice v's K / V of layer l (each voice's own tensors, no packing copy)
        kp = (C.c_void_p * max(1, self.n_ref * nv))(*[int(kv[v][0][l].data_ptr()) for l in range(self.n_ref) for v in range(nv)])
        vp = (C.c_void_p * max(1, self.n_ref * nv))(*[int(kv[v][1][l].data_ptr()) for l in range(self.n_ref) for v in range(nv)])
        voice_c = (C.c_int32 * B)(*voice)
        tr_c = (C.c_int32 * nv)(*[t for _k, _v, t in kv])
        txt_seq = torch.empty((B, Lmax, self.D), dtype=torch.float32, device=self.device)
        txt_pool = torch.empty((B, self.D), dtype=torch.float32, device=self.device)
        cond = torch.empty((B, int(n_frames), self.D), dtype=torch.float32, device=self.device)
        _lib.check(self.lib.sopro_prefill_run_voices(self._h, ids.data_ptr(), ln.data_ptr(), B, Lmax, voice_c, nv, sv.data_ptr(), tr_c,
                                                     kp, vp, float(style_strength), int(n_frames), txt_seq.data_ptr(),
                                                     txt_pool.data_ptr(), cond.data_ptr(),
                                                     int(torch.cuda.current_stream(self.device).cuda_stream)))
        self._keep = (ids, ln, sv, kv)  # alive until the stream has consumed them
        return txt_seq, lens, txt_pool, cond

    def _texts(self, text_ids: Sequence[torch.Tensor]):
        """B 1-D id tensors -> padded ids [B, Lmax] and lengths [B] on the device, lens, Lmax"""
        B = len(text_ids)
        lens = [int(t.numel()) for t in text_ids]
        if min(lens) < 1:
            raise ValueError("empty text")
        Lmax = max(lens)
        if Lmax > self.max_text_len:
            raise ValueError(f"text of {Lmax} tokens exceeds max_text_len {self.max_text_len}")
        ids = torch.zeros((B, Lmax), dtype=torch.int32)
        for i, t in enumerate(text_ids):
            ids[i, : lens[i]] = t.to("cpu", torch.int32)
        ids = ids.to(self.device, non_blocking=True)
        ln = torch.tensor(lens, dtype=torch.int32).to(self.device, non_blocking=True)
        return ids, ln, lens, Lmax

    def _ref_kv(self, ref):
        """One prepared voice's cached K / V per layer as contiguous fp32 [H, Tr, D/H] device tensors, and Tr."""
        ks: List[torch.Tensor] = []
        vs: List[torch.Tensor] = []
        Tr = 1
        for c in ref.ref_kv_caches[: self.n_ref]:
            if c.get("key_padding_mask") is not None:
                raise NotImplementedError("prepared references with a key padding mask are not produced by prepare_reference")
            k = c["k"].to(self.device, torch.float32)
            v = c["v"].to(self.device, torch.float32)
            if k.dim() == 4:
                if k.size(0) != 1:
                    raise ValueError("the prefill batches texts over ONE shared prepared reference")
                k, v = k[0], v[0]
            ks.append(k.contiguous())
            vs.append(v.contiguous())
            Tr = int(k.shape[1])
        return ks, vs, Tr

    def close(self) -> None:
        if getattr(self, "_h", None):
            self.lib.sopro_prefill_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class RefPrepEngine:
    """``SoproTTSModel.prepare_reference`` (reference model.py:152-170) on the device: Token2SV, the reference encoder
    and the cached K / V of the reference cross-attention layers, from one voice's codes [Tr, Q]."""

    def __init__(self, cfg: SoproTTSConfig, state_dict: Dict[str, torch.Tensor], device):
        self.lib = _lib.load()
        dev = torch.device(device if not isinstance(device, int) else f"cuda:{device}")
        if dev.type != "cuda":
            raise _lib.SoproError("RefPrepEngine needs a CUDA device; there is no CPU path")
        self.device = torch.device("cuda", dev.index if dev.index is not None else 0)
        sd = state_dict
        c = _lib.RefPrepConfig()
        c.d_model, c.n_codebooks, c.codebook_size = int(cfg.d_model), int(cfg.num_codebooks), int(cfg.codebook_size)
        c.sv_embed_dim, c.sv_dim = int(sd["token2sv.emb.weight"].shape[1]), int(sd["token2sv.proj.weight"].shape[0])
        c.sv_kernel = int(sd["token2sv.enc.0.dw.weight"].shape[-1])
        c.ref_enc_layers = int(cfg.ref_enc_layers)
        c.ref_enc_kernel = int(sd["ref_enc_blocks.0.dw.dw.weight"].shape[-1]) if c.ref_enc_layers > 0 else 7
        c.ref_layers, c.ref_heads = int(cfg.ref_xattn_layers), int(cfg.ref_xattn_heads)
        keep: list = []

        def ptr(t: torch.Tensor):
            t = _f32(t)
            keep.append(t)
            return C.cast(t.data_ptr(), C.POINTER(C.c_float))

        w = _lib.RefPrepWeights()
        w.sv_emb, w.sv_cb_weights = ptr(sd["token2sv.emb.weight"]), ptr(sd["token2sv.cb_weights"])
        w.sv_dw0_w, w.sv_dw0_b = ptr(sd["token2sv.enc.0.dw.weight"]), ptr(sd["token2sv.enc.0.dw.bias"])
        w.sv_dw1_w, w.sv_dw1_b = ptr(sd["token2sv.enc.3.dw.weight"]), ptr(sd["token2sv.enc.3.dw.bias"])
        w.pool_w0, w.pool_b0 = ptr(sd["token2sv.pool.attn.0.weight"]), ptr(sd["token2sv.pool.attn.0.bias"])
        w.pool_w2, w.pool_b2 = ptr(sd["token2sv.pool.attn.2.weight"]), float(sd["token2sv.pool.attn.2.bias"].reshape(-1)[0])
        w.proj_w, w.proj_b = ptr(sd["token2sv.proj.weight"]), ptr(sd["token2sv.proj.bias"])
        w.cb_embed, w.ref_cb_weights = ptr(sd["cb_embed.emb.weight"]), ptr(sd["ref_cb_weights"])
        for i in range(c.ref_enc_layers):
            fill_ssm_block(w.ref_block[i], sd, f"ref_enc_blocks.{i}.", keep)
        w.ref_norm_w = ptr(sd["ref_enc_norm.weight"])
        for i in range(c.ref_layers):
            p = f"ref_xattn.blocks.{i}."
            w.layer[i].nkv_w, w.layer[i].k_w, w.layer[i].v_w = ptr(sd[p + "nkv.weight"]), ptr(sd[p + "k_proj.weight"]), ptr(sd[p + "v_proj.weight"])
        h = C.c_void_p()
        _lib.check(self.lib.sopro_refprep_create(C.byref(c), C.byref(w), self.device.index, C.byref(h)))
        self._h = h
        self.D, self.H, self.n_ref, self.sv_dim, self.Q, self.V = int(c.d_model), int(c.ref_heads), int(c.ref_layers), int(c.sv_dim), int(c.n_codebooks), int(c.codebook_size)
        del keep

    def run(self, ref_tokens_tq: torch.Tensor):
        """codes [Tr, Q] -> (sv_ref [1, sv], ref_seq [1, Tr, D], [{"k": [1, H, Tr, D/H], "v": ..., "key_padding_mask": None}])"""
        if ref_tokens_tq.dim() != 2 or int(ref_tokens_tq.shape[1]) != self.Q or int(ref_tokens_tq.shape[0]) < 1:
            raise ValueError(f"reference codes must be [Tr >= 1, {self.Q}], got {tuple(ref_tokens_tq.shape)}")
        tok = ref_tokens_tq.to(self.device, torch.int32).contiguous()
        Tr = int(tok.shape[0])
        sv = torch.empty((1, self.sv_dim), dtype=torch.float32, device=self.device)
        seq = torch.empty((1, Tr, self.D), dtype=torch.float32, device=self.device)
        ks = [torch.empty((1, self.H, Tr, self.D // self.H), dtype=torch.float32, device=self.device) for _ in range(self.n_ref)]
        vs = [torch.empty_like(k) for k in ks]
        kp = (C.c_void_p * max(1, self.n_ref))(*[int(k.data_ptr()) for k in ks])
        vp = (C.c_void_p * max(1, self.n_ref))(*[int(v.data_ptr()) for v in vs])
        st = int(torch.cuda.current_stream(self.device).cuda_stream)
        _lib.check(self.lib.sopro_refprep_run(self._h, tok.data_ptr(), Tr, sv.data_ptr(), seq.data_ptr(), kp, vp, st))
        try:
            _lib.check(self.lib.sopro_refprep_check(self._h, st))  # also keeps `tok` alive until the kernels have read it
        except _lib.SoproError as e:
            raise IndexError(str(e)) from None  # the reference's embedding lookup raises IndexError
        return sv, seq, [{"k": k, "v": v, "key_padding_mask": None} for k, v in zip(ks, vs)]

    def close(self) -> None:
        if getattr(self, "_h", None):
            self.lib.sopro_refprep_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
