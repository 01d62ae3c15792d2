"""GPU: mixed-voice prefill (sopro_prefill_run_voices, PrefillEngine.run_voices) and synthesize_batch(refs=...).

Utterance i of a mixed-voice batch must equal the batch-1 reference run on text i with voice refs[i].  That is carried
by bit-equality with the shared-voice prefill (sopro_prefill_run with refs[i] shared by the same text list), which
tests/test_prefill_gpu.py pins to the reference, and by the CPU restatement per text at the suite's 2e-5."""
import ctypes as C

import pytest
import torch

from tests.cases import e2e_inputs

pytestmark = pytest.mark.gpu
torch.set_grad_enabled(False)
_S = {}


def _setup():
    from sopro_b200 import prefill as P
    from sopro_b200.prefill_cuda import PrefillEngine, RefPrepEngine

    if "e" not in _S:
        cfg, sd, _ = e2e_inputs()
        tpos = P.sinusoid_table(int(cfg.max_text_len) + 8, int(cfg.d_model), "cpu")
        fpos = P.sinusoid_table(int(cfg.pos_emb_max) + 8, int(cfg.d_model), "cpu")
        _S["e"] = PrefillEngine(cfg, sd, 0, tpos, fpos)
        _S["rp"] = RefPrepEngine(cfg, sd, 0)
        _S["pos"] = (tpos, fpos)
    return _S["e"], _S["pos"]


def _voice(Tr, seed):
    """A voice prepared on the device from random codes [Tr, 32]."""
    from sopro_b200.prefill import PreparedReference

    _setup()
    tok = torch.randint(0, 2048, (Tr, 32), generator=torch.Generator().manual_seed(seed))
    sv, seq, caches = _S["rp"].run(tok)
    return PreparedReference(ref_tokens_btq=tok.unsqueeze(0), sv_ref=sv, ref_seq=seq, ref_kv_caches=caches)


def _texts(lens, seed):
    g = torch.Generator().manual_seed(seed)
    return [torch.randint(0, 1000, (n,), generator=g) for n in lens]


def _assert_rows_equal_shared(eng, texts, refs, n_frames, style=1.2):
    """Every utterance of run_voices(texts, refs) equals its rows of run(texts, refs[i]), bit for bit."""
    txt, lens, pool, cond = eng.run_voices(texts, refs, n_frames=n_frames, style_strength=style)
    shared = {}
    for i, r in enumerate(refs):
        if id(r) not in shared:
            shared[id(r)] = eng.run(texts, r, n_frames=n_frames, style_strength=style)
        t1, l1, p1, c1 = shared[id(r)]
        assert l1 == lens
        L = lens[i]
        assert torch.equal(txt[i, :L], t1[i, :L]), i
        assert torch.equal(pool[i], p1[i]), i
        assert torch.equal(cond[i], c1[i]), (i, float((cond[i] - c1[i]).abs().max()))
    return txt, lens, pool, cond


def test_mixed_voices_equal_the_shared_voice_prefill_and_the_restatement():
    from sopro_b200 import prefill as P

    eng, (tpos, fpos) = _setup()
    cfg, sd, _ = e2e_inputs()
    voices = [_voice(Tr, 30 + Tr) for Tr in (1, 38, 150)]
    texts = _texts((52, 1, 7, 300, 52, 33), 8)
    refs = [voices[v] for v in (0, 1, 2, 1, 0, 2)]
    F = 60
    txt, lens, pool, cond = _assert_rows_equal_shared(eng, texts, refs, F + 1)
    worst = 0.0
    for i, (ids, r) in enumerate(zip(texts, refs)):
        cpu_ref = P.PreparedReference(ref_tokens_btq=r.ref_tokens_btq, sv_ref=r.sv_ref.cpu(), ref_seq=r.ref_seq.cpu(),
                                      ref_kv_caches=[{k: (v.cpu() if v is not None else None) for k, v in c.items()} for c in r.ref_kv_caches])
        want = P.prepare_conditioning(sd, cfg, ids, cpu_ref, max_frames=F, device="cpu", style_strength=1.2, text_pos=tpos, frame_pos=fpos)
        for got, w in ((txt[i, : lens[i]], want["txt_seq"][0]), (pool[i], want["txt_pool"][0]), (cond[i], want["cond_ar"][0])):
            err = float((got.cpu() - w).abs().max())
            worst = max(worst, err)
            assert err <= 2e-5, (i, err)
    print(f"mixed-voice prefill vs CPU restatement: max abs err {worst:.2e}")


def test_more_than_sixteen_voices():
    """20 voices: the per-voice FiLM rows run in launches of at most 16 rows on the skinny kernel (one launch of 20
    rows would take the tile kernel, whose summation order differs from the shared voice's M = 1 launch)."""
    eng, _ = _setup()
    voices = [_voice(Tr, 100 + i) for i, Tr in enumerate(torch.randint(1, 160, (20,), generator=torch.Generator().manual_seed(2)).tolist())]
    texts = _texts(torch.randint(1, 80, (20,), generator=torch.Generator().manual_seed(3)).tolist(), 9)
    refs = [voices[(7 * i) % 20] for i in range(20)]
    _assert_rows_equal_shared(eng, texts, refs, 33)


def test_long_voice_takes_the_large_shared_memory_path():
    """Tr = 1200: 8 warps x (2 x 384 + 1200) floats = 63 KB of dynamic shared memory (above the 48 KB default)."""
    eng, _ = _setup()
    big, small = _voice(1200, 5), _voice(1, 6)
    texts = _texts((40, 9, 17), 10)
    _assert_rows_equal_shared(eng, texts, [big, small, big], 25)
    _assert_rows_equal_shared(eng, texts, [small, big, small], 25)


def test_synthesize_batch_with_a_voice_per_text_equals_single_synthesis():
    from oracle import mimi_oracle as M
    from sopro_b200 import SoproTTS
    from sopro_b200.tokenizer import IdsTokenizer

    cfg, sd, inp = e2e_inputs()
    if "tts" not in _S:
        _S["tts"] = SoproTTS.from_state_dict(cfg, sd, IdsTokenizer(1000), M.synth_mimi_state_dict(), device="cuda:0")
    tts = _S["tts"]
    g = torch.Generator().manual_seed(4)
    rA = tts.prepare_reference(ref_tokens_tq=inp["ref_tokens_tq"])
    rB = tts.prepare_reference(ref_tokens_tq=torch.randint(0, 2048, (150, 32), generator=g))
    rC = tts.prepare_reference(ref_tokens_tq=torch.randint(0, 2048, (12, 32), generator=g))
    texts = [" ".join(str(7 * i + 3) for i in range(20)), " ".join(str(i) for i in range(3, 40, 3)), "5 9",
             " ".join(str(11 * i + 1) for i in range(30))]
    refs, seeds = [rA, rB, rA, rC], [1, 2, 3, 4]
    kw = dict(max_frames=16, min_gen_frames=10 ** 9)
    wavs = tts.synthesize_batch(texts, refs=refs, seeds=seeds, **kw)
    for t, r, s, w in zip(texts, refs, seeds, wavs):
        assert torch.equal(tts.synthesize(t, ref=r, seed=s, **kw), w)
    shared = tts.synthesize_batch(texts, ref=rA, seeds=seeds, **kw)
    assert torch.equal(shared[0], wavs[0]) and torch.equal(shared[2], wavs[2])
    assert not torch.equal(shared[1], wavs[1])  # another voice, another waveform


def test_rejected_inputs_launch_nothing():
    from sopro_b200 import _lib

    eng, _ = _setup()
    voices = [_voice(Tr, 200 + Tr) for Tr in (4, 9)]
    B, L, F, nv, RL = 3, 6, 5, 2, eng.n_ref
    ids = torch.randint(0, 1000, (B, L), dtype=torch.int32, device="cuda")
    ln = torch.full((B,), L, dtype=torch.int32, device="cuda")
    sv = torch.cat([v.sv_ref for v in voices]).contiguous()
    k = [voices[v].ref_kv_caches[l]["k"] for l in range(RL) for v in range(nv)]
    vv = [voices[v].ref_kv_caches[l]["v"] for l in range(RL) for v in range(nv)]
    txt = torch.empty(B, L, eng.D, device="cuda")
    pool = torch.empty(B, eng.D, device="cuda")
    cond = torch.empty(B, F, eng.D, device="cuda")

    def call(voice=(0, 1, 0), tr=(4, 9), kp=None):
        kp = kp if kp is not None else [t.data_ptr() for t in k]
        for o in (txt, pool, cond):
            o.fill_(float("nan"))
        return eng.lib.sopro_prefill_run_voices(
            eng._h, ids.data_ptr(), ln.data_ptr(), B, L, (C.c_int32 * B)(*voice), nv, sv.data_ptr(), (C.c_int32 * nv)(*tr),
            (C.c_void_p * (RL * nv))(*kp), (C.c_void_p * (RL * nv))(*[t.data_ptr() for t in vv]), 1.2, F, txt.data_ptr(),
            pool.data_ptr(), cond.data_ptr(), int(torch.cuda.current_stream().cuda_stream))

    bad = {"voice index out of range": dict(voice=(0, 2, 0)), "negative voice index": dict(voice=(0, -1, 0)),
           "Tr = 0": dict(tr=(4, 0)), "Tr = 4097": dict(tr=(4097, 9)), "null K pointer": dict(kp=[k[0].data_ptr(), None] + [t.data_ptr() for t in k[2:]])}
    for what, args in bad.items():
        with pytest.raises(_lib.SoproError):
            _lib.check(call(**args))
        torch.cuda.synchronize()
        assert all(bool(torch.isnan(o).all()) for o in (txt, pool, cond)), f"{what}: a kernel ran"
    _lib.check(call())
    torch.cuda.synchronize()
    assert all(bool(torch.isfinite(o).all()) for o in (pool, cond))
    want = eng.run([ids[b].cpu() for b in range(B)], voices[0], n_frames=F, style_strength=1.2)
    assert torch.equal(cond[0], want[3][0]) and torch.equal(cond[2], want[3][2])
