"""Mixed-voice batches (a prepared reference per text) WITHOUT a GPU: the host side of PrefillEngine.run_voices
(voices told apart by identity, the tables handed to sopro_prefill_run_voices) and the public API around it
(SoproTTS.synthesize_batch / SoproModel.prepare_conditioning_batch with refs=, DataParallelTTS slicing refs with the
texts).  The CUDA engines are replaced by the oracle-backed fakes of tests/test_host_pipeline_cpu.py; the fake
run_voices answers through the torch restatement of the prefill, text by text with its own voice."""
import os
import types

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from oracle import mimi_oracle as M
from sopro_b200 import prefill as P
from sopro_b200.config import SoproTTSConfig
from sopro_b200.model import SoproModel, SoproTTS
from sopro_b200.prefill_cuda import PrefillEngine
from sopro_b200.tokenizer import IdsTokenizer
from sopro_b200.weights import synth_state_dict
from tests.test_dp_gloo import _free_port
from tests.test_host_pipeline_cpu import _FakeArEngine, _FakeCodec, _FakeNar, _FakePrefill, _FakeRefPrep

torch.set_grad_enabled(False)


class _FakeVoicesPrefill(_FakePrefill):
    """PrefillEngine.run / run_voices through the restatement; run_voices records the voices it was handed."""

    def __init__(self, m):
        super().__init__(m)
        self.voice_calls = []

    def run_voices(self, text_ids, refs, *, n_frames, style_strength):
        self.voice_calls.append([id(r) for r in refs])
        parts = [self.run([ids], r, n_frames=n_frames, style_strength=style_strength) for ids, r in zip(text_ids, refs)]
        lens = [p[1][0] for p in parts]
        txt = torch.zeros(len(parts), max(lens), int(self.m.cfg.d_model))
        for i, p in enumerate(parts):
            txt[i, : lens[i]] = p[0][0]
        return txt, lens, torch.cat([p[2] for p in parts]), torch.cat([p[3] for p in parts])


@pytest.fixture(scope="module")
def tts():
    cfg = SoproTTSConfig()
    sd = synth_state_dict(cfg, text_vocab=1000, seed=0)
    sd["ar.head.bias"] = sd["ar.head.bias"].clone()
    sd["ar.head.bias"][int(cfg.codebook_size)] += 2.5  # EOS a few times more likely than a code: ragged lengths
    m = object.__new__(SoproModel)  # the real constructor insists on a CUDA device and builds the CUDA engines
    m.cfg, m.device, m.eos_id, m.weight_dtype = cfg, torch.device("cpu"), int(cfg.codebook_size), "fp32"
    m.engine = _FakeArEngine(cfg, sd)
    skip = ("ar.blocks.", "ar.head.", "ar.norm.")
    m.sd = {k: v.float() for k, v in sd.items() if not k.startswith(skip) and v.is_floating_point()}
    m.text_pos = P.sinusoid_table(int(cfg.max_text_len) + 8, int(cfg.d_model), "cpu")
    m.frame_pos = P.sinusoid_table(int(cfg.pos_emb_max) + 8, int(cfg.d_model), "cpu")
    import threading

    m._sessions, m._sessions_busy, m._sessions_lock = {}, set(), threading.Lock()
    m.prefill, m.nar, m.refprep = _FakeVoicesPrefill(m), _FakeNar(m), _FakeRefPrep(m)
    t = SoproTTS(model=m, cfg=cfg, tokenizer=IdsTokenizer(1000), codec=_FakeCodec(M.synth_mimi_state_dict()), device="cpu")
    g = torch.Generator().manual_seed(21)
    t.voices = [t.prepare_reference(ref_tokens_tq=torch.randint(0, 2048, (n, 32), generator=g)) for n in (12, 5, 20)]
    return t


TEXTS = ["3 14 15 92 65 35", " ".join(str(7 * i + 1) for i in range(15)), "8 9", "27 18 28 18"]
SEEDS = [1, 2, 3, 4]
KW = dict(max_frames=20, min_gen_frames=3)


def test_mixed_voice_batch_equals_each_text_alone_with_its_voice(tts):
    a, b, c = tts.voices
    refs = [a, b, a, c]
    tts.model.prefill.voice_calls.clear()
    wavs = tts.synthesize_batch(TEXTS, refs=refs, seeds=SEEDS, **KW)
    assert tts.model.prefill.voice_calls == [[id(r) for r in refs]]  # one prefill, the voices in text order
    assert len(wavs) == len(TEXTS)
    for text, r, seed, w in zip(TEXTS, refs, SEEDS, wavs):
        single = tts.synthesize_batch([text], ref=r, seeds=[seed], **KW)[0]
        assert single.shape == w.shape, (single.shape, w.shape)
        np.testing.assert_allclose(w.numpy(), single.numpy(), rtol=0, atol=1e-5)
    # the voices matter: the same text and seed in another voice is another waveform
    other = tts.synthesize_batch([TEXTS[1]], ref=a, seeds=[SEEDS[1]], **KW)[0]
    assert other.shape != wavs[1].shape or not torch.equal(other, wavs[1])


def test_prepare_conditioning_batch_with_a_voice_per_text(tts):
    a, b, c = tts.voices
    ids = [tts.encode_text(t) for t in TEXTS[:3]]
    preps = tts.model.prepare_conditioning_batch(ids, refs=[c, a, c], max_frames=8, style_strength=1.2)
    for p, i, r in zip(preps, ids, [c, a, c]):
        alone = tts.model.prepare_conditioning(i, r, max_frames=8, style_strength=1.2)
        assert set(p) == set(alone)
        for k in p:
            assert torch.equal(p[k], alone[k]), k
    assert preps[0]["sv_ref"] is preps[2]["sv_ref"] and torch.equal(preps[1]["sv_ref"], a.sv_ref)


def test_exactly_one_of_ref_and_refs(tts):
    a, b, _ = tts.voices
    with pytest.raises(ValueError):
        tts.synthesize_batch(TEXTS[:2], ref=a, refs=[a, b], **KW)
    with pytest.raises(ValueError):
        tts.synthesize_batch(TEXTS[:2], **KW)
    with pytest.raises(ValueError):
        tts.synthesize_batch(TEXTS[:2], refs=[a], **KW)
    ids = [tts.encode_text(t) for t in TEXTS[:2]]
    with pytest.raises(ValueError):
        tts.model.prepare_conditioning_batch(ids, a, refs=[a, b], max_frames=4)
    with pytest.raises(ValueError):
        tts.model.prepare_conditioning_batch(ids, max_frames=4)
    with pytest.raises(ValueError):
        tts.model.prepare_conditioning_batch(ids, refs=[a, b, a], max_frames=4)


# ---------------------------------------------------------------------------------------------------------------
# PrefillEngine.run_voices: what reaches sopro_prefill_run_voices (a recording stand-in for the library)
# ---------------------------------------------------------------------------------------------------------------
def _voice(Tr, seed, H=2, dh=192, layers=3):
    g = torch.Generator().manual_seed(seed)
    caches = [{"k": torch.randn(1, H, Tr, dh, generator=g), "v": torch.randn(1, H, Tr, dh, generator=g), "key_padding_mask": None}
              for _ in range(layers)]
    return P.PreparedReference(ref_tokens_btq=torch.zeros(1, Tr, 32, dtype=torch.long), sv_ref=torch.randn(1, 192, generator=g),
                               ref_seq=torch.zeros(1, Tr, 384), ref_kv_caches=caches)


class _RecordingLib:
    def __init__(self):
        self.calls = []

    def sopro_prefill_run_voices(self, h, ids, ln, B, Lmax, voice, n_voices, sv, ref_len, ref_k, ref_v, style, n_frames, txt, pool,
                                 cond, stream):
        n = 3 * n_voices
        self.calls.append(dict(B=B, Lmax=Lmax, voice=list(voice), n_voices=n_voices, sv=sv, ref_len=list(ref_len),
                               k=[ref_k[i] for i in range(n)], v=[ref_v[i] for i in range(n)], n_frames=n_frames))
        return 0


@pytest.fixture()
def engine(monkeypatch):
    eng = object.__new__(PrefillEngine)  # the real constructor loads the library and uploads weights to a CUDA device
    eng.lib, eng._h, eng.device = _RecordingLib(), None, torch.device("cpu")
    eng.D, eng.n_ref, eng.max_text_len, eng.sv_dim = 384, 3, 512, 192
    monkeypatch.setattr(torch.cuda, "current_stream", lambda device=None: types.SimpleNamespace(cuda_stream=0))
    return eng


def test_run_voices_hands_each_voice_once_by_identity(engine):
    a, b, c = _voice(7, 1), _voice(150, 2), _voice(1, 3)
    a_again = _voice(7, 1)  # equal contents, another object: another voice
    refs = [b, a, b, c, a_again, a]
    texts = [torch.arange(n) for n in (5, 1, 9, 3, 4, 2)]
    engine.run_voices(texts, refs, n_frames=11, style_strength=1.2)
    call = engine.lib.calls[-1]
    order = [b, a, c, a_again]  # first-seen order
    assert call["B"] == 6 and call["Lmax"] == 9 and call["n_frames"] == 11
    assert call["n_voices"] == 4 and call["voice"] == [0, 1, 0, 2, 3, 1]
    assert call["ref_len"] == [150, 7, 1, 7]
    nv = call["n_voices"]
    for l in range(3):
        for v, r in enumerate(order):  # entry l * n_voices + v, the voice's own tensors (no packing copy)
            assert call["k"][l * nv + v] == r.ref_kv_caches[l]["k"].data_ptr()
            assert call["v"][l * nv + v] == r.ref_kv_caches[l]["v"].data_ptr()
    sv = engine._keep[2]
    assert call["sv"] == sv.data_ptr() and sv.shape == (4, 192) and sv.is_contiguous()
    assert torch.equal(sv, torch.cat([r.sv_ref for r in order]))


def test_run_voices_rejects_mismatched_inputs(engine):
    a = _voice(7, 1)
    with pytest.raises(ValueError):
        engine.run_voices([torch.arange(3), torch.arange(2)], [a], n_frames=5, style_strength=1.0)
    batched = _voice(7, 2)
    batched.ref_kv_caches[0]["k"] = batched.ref_kv_caches[0]["k"].repeat(2, 1, 1, 1)
    with pytest.raises(ValueError):
        engine.run_voices([torch.arange(3)], [batched], n_frames=5, style_strength=1.0)
    wide = _voice(7, 3)
    wide.sv_ref = torch.randn(2, 192)
    with pytest.raises(ValueError):
        engine.run_voices([torch.arange(3)], [wide], n_frames=5, style_strength=1.0)
    assert engine.lib.calls == []


# ---------------------------------------------------------------------------------------------------------------
# DataParallelTTS: each rank gets the refs of its own texts (world 2 over gloo, like tests/test_dp_gloo.py)
# ---------------------------------------------------------------------------------------------------------------
def _dp_worker(rank, world, port, out):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    import sopro_b200.model as model_mod
    from sopro_b200.dp import DataParallelTTS
    from tests.cases import SMALL_CFG

    class _StubTTS:  # stands where SoproTTS.from_state_dict builds the CUDA engines
        def __init__(self):
            self.calls = []

        def synthesize_batch(self, texts, *, ref=None, refs=None, seeds=None, **kw):
            self.calls.append((list(texts), ref, refs, seeds))
            return [f"wav:{t}:{r}" for t, r in zip(texts, refs)]

    orig = model_mod.SoproTTS.from_state_dict
    model_mod.SoproTTS.from_state_dict = classmethod(lambda cls, cfg, sd, tok, msd, **kw: _StubTTS())
    try:
        cfg = SoproTTSConfig(**SMALL_CFG)
        sd0 = synth_state_dict(cfg, 64, 0) if rank == 0 else None
        dp = DataParallelTTS(cfg, sd0, None, None, device="cpu", text_vocab=64)
        texts = [f"t{i}" for i in range(5)]
        refs = ["vA", "vB", "vA", "vC", "vB"]
        wavs, span = dp.synthesize_batch(texts, refs=refs, seeds=[10, 11, 12, 13, 14], max_frames=3)
        try:
            dp.synthesize_batch(texts, refs=refs[:4])
            mismatch = None
        except ValueError as e:
            mismatch = str(e)
        out[rank] = (span, wavs, dp.tts.calls[0], mismatch)
    finally:
        model_mod.SoproTTS.from_state_dict = orig
        dist.destroy_process_group()


def test_data_parallel_slices_refs_with_the_texts():
    world, port = 2, _free_port()
    with mp.Manager() as m:
        out = m.dict()
        mp.spawn(_dp_worker, args=(world, port, out), nprocs=world, join=True)
        res = dict(out)
    assert res[0][0] == (0, 2) and res[1][0] == (2, 5)
    assert res[0][1] == ["wav:t0:vA", "wav:t1:vB"] and res[1][1] == ["wav:t2:vA", "wav:t3:vC", "wav:t4:vB"]
    assert res[0][2] == (["t0", "t1"], None, ["vA", "vB"], [10, 11])
    assert res[1][2] == (["t2", "t3", "t4"], None, ["vA", "vC", "vB"], [12, 13, 14])
    assert res[0][3] and res[1][3]  # every rank rejects a refs list that does not match the texts
