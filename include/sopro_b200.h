/*
 * sopro_b200 — C-ABI of the B200-native Sopro hot path.
 *
 * The reference (samuel-vitorino/sopro) is pure Python/PyTorch and has no FFI;
 * every entry point below names the reference interface it replaces
 * (paths relative to the reference's src/sopro/).  Plain pointers and sizes
 * only, no torch types.  Unless a parameter says "host", pointers are CUDA
 * device pointers owned by the caller; `stream` is a cudaStream_t passed as
 * void* (NULL = legacy default stream).  Every function returns 0 on success
 * or a negative sopro_status; sopro_last_error() gives the message for the
 * calling thread.  There is no CPU fallback: creating an engine on a device
 * that is not sm_100 fails.
 */
#ifndef SOPRO_B200_H_
#define SOPRO_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SOPRO_MAX_AR_LAYERS 16

enum sopro_status {
  SOPRO_OK = 0,
  SOPRO_ERR_INVALID = -1,     /* bad argument / unsupported geometry */
  SOPRO_ERR_CUDA = -2,        /* a CUDA runtime call failed */
  SOPRO_ERR_UNSUPPORTED = -3, /* device is not sm_100, or feature not built */
  SOPRO_ERR_STATE = -4        /* call out of order */
};

enum sopro_wdtype { SOPRO_W_F32 = 0, SOPRO_W_BF16 = 1 };

/* Geometry of the AR generator.  Replaces the fields of SoproTTSConfig the AR
 * path reads (config.py:14-27) + the literals in nn/generator.py:12-42. */
typedef struct sopro_ar_config {
  int32_t d_model;                          /* cfg.d_model (384) */
  int32_t n_layers;                         /* cfg.n_layers_ar (6) */
  int32_t kernel;                           /* cfg.ar_kernel (13) */
  int32_t n_heads;                          /* 4, nn/generator.py:36 */
  int32_t vocab;                            /* codebook_size + 1 (2049), model.py:83 */
  int32_t eos_id;                           /* codebook_size, model.py:59 */
  int32_t dilation[SOPRO_MAX_AR_LAYERS];    /* nn/generator.py:16-20 */
  int32_t has_attn[SOPRO_MAX_AR_LAYERS];    /* 1 if a TextXAttnBlock follows block i */
  int32_t weight_dtype;                     /* sopro_wdtype: storage of the matrices */
} sopro_ar_config_t;

/* HOST pointers to fp32 tensors in the reference's state_dict layout. */
typedef struct sopro_ar_layer_weights {
  const float* norm_w;    /* ar.blocks.i.norm.weight      [D]        nn/blocks.py:123 */
  const float* glu_w;     /* ar.blocks.i.glu.pro.weight   [2D, D]    nn/blocks.py:19 */
  const float* glu_b;     /* ar.blocks.i.glu.pro.bias     [2D] */
  const float* dw_w;      /* ar.blocks.i.dw.dw.weight     [D, 1, k]  nn/blocks.py:48 */
  const float* dw_b;      /* ar.blocks.i.dw.dw.bias       [D] */
  const float* ffn_norm_w;/* ar.blocks.i.ff.0.weight      [D]        nn/blocks.py:129 */
  const float* ffn_w1;    /* ar.blocks.i.ff.1.weight      [4D, D] */
  const float* ffn_b1;    /* ar.blocks.i.ff.1.bias        [4D] */
  const float* ffn_w2;    /* ar.blocks.i.ff.3.weight      [D, 4D] */
  const float* ffn_b2;    /* ar.blocks.i.ff.3.bias        [D] */
  /* cross-attention after block i (NULL when has_attn[i] == 0)  nn/text.py:57-65 */
  const float* nq_w;      /* ar.x_attns.i.nq.weight       [D] */
  const float* nkv_w;     /* ar.x_attns.i.nkv.weight      [D] */
  const float* q_w;       /* ar.x_attns.i.q_proj.weight   [D, D] */
  const float* k_w;       /* ar.x_attns.i.k_proj.weight   [D, D] */
  const float* v_w;       /* ar.x_attns.i.v_proj.weight   [D, D] */
  const float* o_w;       /* ar.x_attns.i.out_proj.weight [D, D] */
  float gate_tanh;        /* tanh(ar.x_attns.i.gate), evaluated by the caller in fp32 (nn/text.py:131) */
} sopro_ar_layer_weights_t;

typedef struct sopro_ar_weights {
  sopro_ar_layer_weights_t layer[SOPRO_MAX_AR_LAYERS];
  const float* final_norm_w; /* ar.norm.weight  [D]      nn/generator.py:41 */
  const float* head_w;       /* ar.head.weight  [V, D]   nn/generator.py:42 */
  const float* head_b;       /* ar.head.bias    [V] */
  const float* cb_embed;     /* cb_embed.emb.weight [Q*V'+1, D]  nn/embeddings.py:47-49 */
  int64_t cb_embed_rows;     /* Q*codebook_size + 1 */
  int64_t bos_row;           /* Q*codebook_size, nn/embeddings.py:49 */
} sopro_ar_weights_t;

/* Per-utterance sampling knobs: kwargs of SoproTTSModel.ar_stream (model.py:218-231)
 * plus the literals it passes to sample_token (model.py:284-291). */
typedef struct sopro_ar_sampling {
  float top_p;               /* 0.9 */
  float temperature;         /* 1.05 */
  float recovery_top_p;      /* 0.85 */
  float recovery_temp;       /* 1.2 */
  float repetition_penalty;  /* 1.1 */
  int32_t top_k;             /* 50; must be in [1, 64] */
  int32_t anti_loop;         /* 1 */
  int32_t loop_streak;       /* 8 */
  int32_t min_gen_frames;    /* cfg.min_gen_frames (12) */
  int32_t stop_on_first_eos; /* 1 = what generate_tokens/stream consumers do (model.py:382-383,
                                streaming.py:114-115); 0 = ar_stream's own rule (model.py:304) */
} sopro_ar_sampling_t;

typedef struct sopro_engine sopro_engine_t;
typedef struct sopro_ar_session sopro_ar_session_t;

const char* sopro_last_error(void);
const char* sopro_version(void);

/* Engine = device-resident copy of the AR step weights (converted to
 * cfg->weight_dtype).  Replaces SoproTTSModel.ar + cb_embed residency after
 * SoproTTS.from_pretrained (model.py:443-446). */
int sopro_engine_create(const sopro_ar_config_t* cfg, const sopro_ar_weights_t* host_weights,
                        int device, sopro_engine_t** out);
int sopro_engine_destroy(sopro_engine_t* e);
/* bytes of step-resident weights as stored on the device (W_step of SURVEY.md §8d) */
int64_t sopro_engine_step_weight_bytes(const sopro_engine_t* e);
int sopro_engine_num_sms(const sopro_engine_t* e);

/* Session = state of a batch of independent utterances: conv ring buffers, text
 * K/V, history, outputs.  Replaces ARRVQ1Generator.init_stream_state
 * (nn/generator.py:44-68) and the locals of ar_stream (model.py:242-255). */
int sopro_ar_session_create(sopro_engine_t* e, int max_batch, int max_steps, int max_text_len,
                            sopro_ar_session_t** out);
int sopro_ar_session_destroy(sopro_ar_session_t* s);

/* Launch geometry override (0 = automatic): utterances per CTA team. */
int sopro_ar_session_set_team(sopro_ar_session_t* s, int utts_per_team);

/* Arithmetic unit of the step's contractions: 0 or -1 = packed fp32 FMA (FFMA2) tiles -- the default and the faster one at
 * the 22..86 weight rows a CTA owns per stage; 1 = tensor cores (tcgen05, every fp32 activation split into three exact bf16
 * terms against bf16 weights, fp32 accumulation) or fail when the launch cannot use them (needs bf16 weight storage,
 * d_model % 64 == 0, teams of 5..8 utterances).  -1 also honours the environment variable SOPRO_AR_TC=1.  Both produce the
 * reference's token ids (tests/test_ar_gpu.py). */
int sopro_ar_session_set_contraction(sopro_ar_session_t* s, int mode);

/* Start `batch` utterances.  Zeroes the rings, builds the text K/V caches on the
 * device (TextXAttnBlock.build_kv_cache, nn/text.py:75-83), resets history.
 *   cond_ar   [batch, steps, D] f32   prep["cond_ar"] rows 0..steps-1 (model.py:272)
 *   txt_seq   [batch, text_stride, D] f32   prep["txt_seq"], padded to text_stride rows
 *   text_len  [batch] i32 HOST        valid rows per utterance (text_mask, model.py:186)
 *   noise     [batch, steps, noise_k] f32   Exp(1) draws: what torch.multinomial would
 *             consume at each step, q of argmax(p/q); noise_k >= top_k when top_p < 1
 *             (rank-aligned, sampling.py:83-84), noise_k >= vocab otherwise (sampling.py:93)
 *   sampling  [batch] HOST
 */
int sopro_ar_begin(sopro_ar_session_t* s, int batch, int steps, const float* cond_ar,
                   const float* txt_seq, int text_stride, const int32_t* text_len,
                   const float* noise, int noise_k, const sopro_ar_sampling_t* sampling,
                   void* stream);

/* Advance every live utterance by up to n_steps frames (the body of the
 * `for t in range(max_steps)` loop, model.py:265-305) in ONE persistent kernel.
 * Asynchronous on `stream`. Returns after enqueueing. */
int sopro_ar_run(sopro_ar_session_t* s, int n_steps, void* stream);

/* Device views of the outputs (valid until the session is destroyed):
 *   tokens   [batch, steps] i32   token per step: what ar_stream yields (model.py:302)
 *   n_tokens [batch] i32          steps taken so far;   done [batch] i32 */
int sopro_ar_outputs(sopro_ar_session_t* s, const int32_t** tokens, const int32_t** n_tokens,
                     const int32_t** done);
/* Synchronous copy to HOST buffers (tokens row stride = steps given to begin). */
int sopro_ar_read(sopro_ar_session_t* s, int32_t* tokens_host, int32_t* n_tokens_host,
                  int32_t* done_host, void* stream);
/* steps the slowest live utterance has reached (host value, after the last run completes) */
int sopro_ar_position(sopro_ar_session_t* s);

/* One-call host-buffer path (what a ctypes/cgo caller with numpy-like buffers uses;
 * bench.py's e2e leg): H2D of cond/text/noise, begin, run to completion, D2H of
 * tokens, synchronises `stream`.  All pointers HOST. */
int sopro_ar_generate_host(sopro_ar_session_t* s, int batch, int steps, const float* cond_ar,
                           const float* txt_seq, int text_stride, const int32_t* text_len,
                           const float* noise, int noise_k, const sopro_ar_sampling_t* sampling,
                           int32_t* tokens_out, int32_t* n_tokens_out, void* stream);

/* ---- host-side noise tapes --------------------------------------------------------------------------------------
 * The Exp(1) draws torch.multinomial consumes on the CPU (reference sampling.py:83-93: multinomial == argmax(p / q),
 * q ~ Exp(1) from torch's CPU generator, `vocab` draws per step), reproduced bit for bit by a host-side mt19937 for a
 * PRIVATE generator seeded like torch.manual_seed(seed).  Only the first `keep` columns of each [vocab] row are
 * materialised (the sampler reads top_k of them); the generator still advances by the whole row.  Pure host code. */
typedef struct sopro_noise sopro_noise_t;
int sopro_noise_create(uint64_t seed, sopro_noise_t** out);
/* next n_rows rows of the tape -> out [n_rows, keep] f32 (host) */
int sopro_noise_rows(sopro_noise_t* g, int n_rows, int vocab, int keep, float* out);
int sopro_noise_destroy(sopro_noise_t* g);

/* ---- test / debug hooks (used by tests/, not by the product path) ---- */
/* teacher forcing: token fed back at step t is forced[b, t]; the sampled one goes to
 * `sampled` (sopro_ar_debug_sampled).  NULL disables. [batch, steps] i32 device. */
int sopro_ar_set_forced_tokens(sopro_ar_session_t* s, const int32_t* forced);
/* trace_blocks [steps, n_layers, batch, D] f32 (residual stream after block i incl. its
 * cross-attention), trace_logits [steps, batch, V] f32; NULL disables. device. */
int sopro_ar_set_trace(sopro_ar_session_t* s, float* trace_blocks, float* trace_logits);
/* clock64 stamps of one step: buf [grid, 224] i64 device (grid = SM count): one stamp at step
 * start, then five per stage (activations staged, weight tiles done, whole CTA done, barrier
 * arrival posted, barrier released). NULL = off */
int sopro_ar_set_timing(sopro_ar_session_t* s, int64_t* buf, int step);
/* copy the sampled (pre-forcing) tokens into dst [batch, steps] i32 (device) */
int sopro_ar_debug_sampled(sopro_ar_session_t* s, int32_t* dst, void* stream);
/* copy the text K/V built by sopro_ar_begin into k_dst / v_dst, each
 * [n_attn_layers, batch, H, Lpad, Dh] f32 (device), Lpad = max_text_len rounded up to 4 */
int sopro_ar_debug_kv(sopro_ar_session_t* s, float* k_dst, float* v_dst, void* stream);
/* Host-only views of the operand images the engines build (no device needed): the tensor-core image of an AR step matrix
 * W [N][K] ([K / D slices][groups of 8 rows][D / 64 chunks][8 x 128 B, 16-byte units XOR row]; glu: group = 4 channels, value
 * rows then gate rows) and the NAR refiner's W6 [N][6K] (bf16 terms of the six product pairs mm, lh, hl, mh, hm, hh). */
int sopro_debug_pack_umma(const float* W, int N, int K, int d_model, int glu, uint8_t* out, int64_t bytes);
int sopro_debug_pack_w6(const float* W, int N, int K, uint16_t* out);
/* The kernel's sampler (sample_token, sampling.py:24-93) on ONE logits row, outside the step: HOST buffers; `hist` = the
 * n_hist tokens generated so far (repetition penalty looks at the last 50), `noise` = the Exp(1) draws of this step (first
 * noise_k columns of the tape row: >= top_k when top_p < 1, vocab otherwise), `recovery` != 0 samples with the recovery
 * (top_p, temperature).  -> token_out.  Needs a device but no engine. */
int sopro_debug_sample(const float* logits, int vocab, const int32_t* hist, int n_hist, const float* noise, int noise_k,
                       const sopro_ar_sampling_t* sampling, int recovery, int device, int32_t* token_out);


/* ======================= Mimi codec decode (codes -> waveform) =======================
 * Replaces transformers.MimiModel.decode as the reference calls it: MimiCodec.decode_full
 * (codec/mimi.py:65-72) and, through it, MimiStreamDecoder.decode_step (codec/mimi.py:115-181).
 * Citations below are transformers/models/mimi/modeling_mimi.py (5.5.0). */
#define SOPRO_MIMI_MAX_LAYERS 16
#define SOPRO_MIMI_MAX_RATIOS 8

typedef struct sopro_mimi_config {
  int32_t hidden;        /* 512  MimiConfig.hidden_size */
  int32_t codebook_dim;  /* 256  (hidden == 2*codebook_dim: the two 1x1 output projections are fused) */
  int32_t n_q;           /* 32   num_quantizers */
  int32_t n_sem;         /* 1    num_semantic_quantizers */
  int32_t vocab;         /* 2048 codebook_size */
  int32_t n_layers;      /* 8 */
  int32_t n_heads;       /* 8 */
  int32_t ffn;           /* 2048 intermediate_size */
  int32_t window;        /* 250  sliding_window */
  int32_t num_filters;   /* 64 */
  int32_t kernel;        /* 7 */
  int32_t last_kernel;   /* 3 */
  int32_t res_kernel;    /* 3 */
  int32_t compress;      /* 2 */
  int32_t n_ratios;      /* 4 */
  int32_t ratios[SOPRO_MIMI_MAX_RATIOS]; /* 8,6,5,4 */
  float norm_eps;        /* 1e-5 */
  float rope_theta;      /* 10000 */
} sopro_mimi_config_t;

/* HOST fp32 pointers, state_dict layouts. */
typedef struct sopro_mimi_layer_weights {
  const float *ln1_w, *ln1_b;            /* input_layernorm                 :933 */
  const float *q_w, *k_w, *v_w, *o_w;    /* self_attn.*_proj.weight [C,C]    :676-679 */
  const float* ls1;                      /* self_attn_layer_scale.scale     :935 */
  const float *ln2_w, *ln2_b;            /* post_attention_layernorm        :934 */
  const float *fc1_w, *fc2_w;            /* mlp.fc1 [F,C], mlp.fc2 [C,F] */
  const float* ls2;                      /* mlp_layer_scale.scale */
} sopro_mimi_layer_weights_t;

typedef struct sopro_mimi_stage_weights {
  const float *convt_w, *convt_b;        /* decoder.layers.{i}.conv: ConvTranspose1d [Cin, Cout, 2r], [Cout] */
  const float *res1_w, *res1_b;          /* ...block.1.conv [Cout/2, Cout, 3] */
  const float *res2_w, *res2_b;          /* ...block.3.conv [Cout, Cout/2, 1] */
} sopro_mimi_stage_weights_t;

typedef struct sopro_mimi_weights {
  const float* embed;         /* [n_q, vocab, codebook_dim]: embed_sum / clamp(cluster_usage, 1e-5)  (:1192-1196),
                                 semantic codebooks first, then acoustic */
  const float* sem_out_proj;  /* quantizer.semantic_residual_vector_quantizer.output_proj.weight [C, Dc] */
  const float* ac_out_proj;   /* quantizer.acoustic_...output_proj.weight [C, Dc] */
  const float* upsample_w;    /* upsample.conv.weight [C, 1, 4] */
  sopro_mimi_layer_weights_t layer[SOPRO_MIMI_MAX_LAYERS];
  const float *conv0_w, *conv0_b; /* decoder.layers.0.conv [16F, C, 7] */
  sopro_mimi_stage_weights_t stage[SOPRO_MIMI_MAX_RATIOS];
  const float *last_w, *last_b;   /* decoder.layers.14.conv [1, F, 3] */
} sopro_mimi_weights_t;

typedef struct sopro_mimi sopro_mimi_t;

int sopro_mimi_create(const sopro_mimi_config_t* cfg, const sopro_mimi_weights_t* host_weights, int device,
                      sopro_mimi_t** out);
int sopro_mimi_destroy(sopro_mimi_t* m);
int64_t sopro_mimi_samples_per_frame(const sopro_mimi_t* m); /* 1920 */
/* codes [B, n_q, T] i32 (device) -> wav [B, T*1920] f32 (device).  MimiModel.decode (:1633-1680). */
int sopro_mimi_decode(sopro_mimi_t* m, const int32_t* codes, int B, int T, float* wav, void* stream);
/* same with HOST buffers; synchronises the stream */
int sopro_mimi_decode_host(sopro_mimi_t* m, const int32_t* codes_host, int B, int T, float* wav_host, void* stream);

/* Arithmetic of the dense blocks (transformer linears, SEANet Conv1d / ConvTranspose1d).
 *   SOPRO_MIMI_BF16_TC (default): bf16 operands on the tcgen05 tensor cores, fp32 accumulation in tensor
 *     memory, fp32 residual streams / LayerNorm / softmax; within 2e-2 * max|wav| of the fp32 reference.
 *   SOPRO_MIMI_FP32: every contraction in fp32 on the FMA pipe; within 1e-4 of the reference
 *     (what transformers computes on CPU, modeling_mimi.py). */
#define SOPRO_MIMI_FP32 0
#define SOPRO_MIMI_BF16_TC 1
int sopro_mimi_set_precision(sopro_mimi_t* m, int precision);
/* Decodes of at most 64 frames (B*T: streaming chunks, time-to-first-audio) are launch-bound (~100 kernels); they
 * are captured once per (B, T, precision) into a CUDA graph over internal static buffers and replayed (default on).
 * Results are identical to the plain path. */
int sopro_mimi_set_graphs(sopro_mimi_t* m, int enabled);

/* A decode that meets a code outside [0, vocab) (e.g. an uncut EOS id) clamps it and sets a sticky flag instead of
 * reading outside the codebook (the reference's embedding lookup raises IndexError, modeling_mimi.py:1192-1196).
 * sopro_mimi_check synchronises `stream`, returns SOPRO_ERR_INVALID if the flag was set since the last check, and
 * clears it.  The *_host entry points validate their host buffers up front instead. */
int sopro_mimi_check(sopro_mimi_t* m, void* stream);

/* ---- streaming decode with persistent state: MimiStreamDecoder.decode_step / MimiDecodeState (reference
 * codec/mimi.py:75-181).  A stream carries one K/V ring per transformer layer (the last `window` positions), the
 * previous RVQ frame of the upsampler and the (taps-1) left-context rows of every causal conv (what transformers'
 * MimiConv1dPaddingCache holds, modeling_mimi.py:77-170), so a chunk costs O(chunk) and, decoder being causal, the
 * chunks concatenate to exactly what sopro_mimi_decode gives for the whole sequence (bit-identical in SOPRO_MIMI_FP32
 * mode; within the tensor-core mode's stated tolerance otherwise).  The reference instead re-decodes 2 overlap frames
 * on top of a transformers KV cache with no conv context and documents its stream as not bit-exact (README.md:151).
 * One stream = one utterance; streams of one decoder are independent; the arithmetic mode is the decoder's at
 * create / reset time. */
typedef struct sopro_mimi_stream sopro_mimi_stream_t;
int sopro_mimi_stream_create(sopro_mimi_t* m, int max_chunk_frames, sopro_mimi_stream_t** out);
int sopro_mimi_stream_destroy(sopro_mimi_stream_t* s);
int sopro_mimi_stream_reset(sopro_mimi_stream_t* s, void* stream);     /* back to frame 0 (MimiDecodeState()) */
int64_t sopro_mimi_stream_frames(const sopro_mimi_stream_t* s);        /* MimiDecodeState.frames_seen */
/* the next n frames: codes [n_q, n] i32 (device) -> wav [n*1920] f32 (device); any n >= 1 (longer than
 * max_chunk_frames is processed in pieces) */
int sopro_mimi_decode_step(sopro_mimi_stream_t* s, const int32_t* codes, int n, float* wav, void* stream);
int sopro_mimi_decode_step_host(sopro_mimi_stream_t* s, const int32_t* codes_host, int n, float* wav_host, void* stream);

/* ---- Mimi ENCODE (waveform -> codes): MimiCodec.encode_file's model call (reference codec/mimi.py:41-63 ->
 * MimiModel.encode, modeling_mimi.py:1455-1488, 1522-1611), once per reference voice.  SEANet encoder (:454-497:
 * conv k7, 4 x [ResnetBlock, ELU, strided conv kernel 2r stride r] with r = reversed(ratios), ELU, conv k3), the
 * encoder transformer (same layer as the decoder's), the 25 -> 12.5 Hz conv (kernel 4, stride 2, replicate padding,
 * :1419-1429) and the split residual vector quantizer's nearest-neighbour search (:1262-1280, :1311-1338).  fp32
 * throughout (the codes are an argmin): batch 1, any sample count >= 1; every strided conv pads its input on the right
 * to a full window (MimiConv1d._get_extra_padding_for_conv1d, :273-285), so T = ceil(ceil(..ceil(n/4)../8)/2).
 * HOST fp32 pointers in state_dict layouts; `cfg` is the decoder's sopro_mimi_config_t. */
typedef struct sopro_mimi_enc_stage_weights {
  const float *res1_w, *res1_b;   /* encoder.layers.{1+3s}.block.1.conv [C/2, C, 3], [C/2]   (C = 64 << s) */
  const float *res2_w, *res2_b;   /* encoder.layers.{1+3s}.block.3.conv [C, C/2, 1], [C] */
  const float *down_w, *down_b;   /* encoder.layers.{3+3s}.conv [2C, C, 2r], [2C],  r = ratios[n_ratios-1-s] */
} sopro_mimi_enc_stage_weights_t;

typedef struct sopro_mimi_encoder_weights {
  const float *conv0_w, *conv0_b;                    /* encoder.layers.0.conv [F, 1, 7], [F] */
  sopro_mimi_enc_stage_weights_t stage[SOPRO_MIMI_MAX_RATIOS];
  const float *last_w, *last_b;                      /* encoder.layers.14.conv [hidden, 16F, 3], [hidden] */
  sopro_mimi_layer_weights_t layer[SOPRO_MIMI_MAX_LAYERS]; /* encoder_transformer.layers.* */
  const float* downsample_w;                         /* downsample.conv.weight [hidden, hidden, 4], no bias */
  const float* sem_in_proj;                          /* quantizer.semantic_...input_proj.weight [Dc, hidden] */
  const float* ac_in_proj;                           /* quantizer.acoustic_...input_proj.weight [Dc, hidden] */
  const float* embed;                                /* [n_q, vocab, Dc] as in sopro_mimi_weights_t */
} sopro_mimi_encoder_weights_t;

typedef struct sopro_mimi_encoder sopro_mimi_encoder_t;
int sopro_mimi_encoder_create(const sopro_mimi_config_t* cfg, const sopro_mimi_encoder_weights_t* host_weights, int device,
                              sopro_mimi_encoder_t** out);
int sopro_mimi_encoder_destroy(sopro_mimi_encoder_t* e);
/* MimiModel.get_encoded_length (:1490-1503): frames produced for n_samples input samples; < 0 on bad arguments */
int64_t sopro_mimi_encoded_frames(const sopro_mimi_encoder_t* e, int64_t n_samples);
/* wav [n_samples] f32 @24 kHz (device) -> codes [n_q, T] i32 (device), T = sopro_mimi_encoded_frames(n_samples).
 * `latent` (optional, device [T, hidden] f32) receives the pre-quantizer embeddings (tests compare them with the
 * oracle's; the codes are their nearest neighbours). */
int sopro_mimi_encode(sopro_mimi_encoder_t* e, const float* wav, int64_t n_samples, int32_t* codes, float* latent, void* stream);
/* same with HOST buffers; synchronises the stream */
int sopro_mimi_encode_host(sopro_mimi_encoder_t* e, const float* wav_host, int64_t n_samples, int32_t* codes_host,
                           float* latent_host, void* stream);

/* ------------------------------------------------------------------------------------------------
 * NAR refiner: SoproTTSModel.nar_refine (reference model.py:307-347) over NARSinglePass.forward_stage
 * (nn/nar.py:89-116), NARStageAdapter (nn/nar.py:13-32), SSMLiteBlock.forward (nn/blocks.py:143-148) and
 * CodebookEmbedding.sum_embed_subset (nn/embeddings.py:77-112).  Given the AR tokens (codebook 0) and the
 * conditioning rows it fills codebooks 1..Q-1 stage by stage (argmax).  fp32 throughout: the ids equal the
 * reference's.  HOST fp32 pointers in state_dict layouts; the engine uploads its own copy.
 * ------------------------------------------------------------------------------------------------ */
#define SOPRO_MAX_SSM_LAYERS 16
#define SOPRO_NAR_MAX_STAGES 8
#define SOPRO_NAR_MAX_CODEBOOKS 64

typedef struct sopro_ssm_block_weights { /* SSMLiteBlock (nn/blocks.py:113-133) */
  const float* norm_w;              /* norm.weight [D] */
  const float *glu_w, *glu_b;       /* glu.pro [2D, D], [2D] */
  const float *dw_w, *dw_b;         /* dw.dw [D, 1, k], [D] */
  const float* ffn_norm_w;          /* ff.0.weight [D] */
  const float *ffn_w1, *ffn_b1;     /* ff.1 [4D, D], [4D] */
  const float *ffn_w2, *ffn_b2;     /* ff.3 [D, 4D], [D] */
} sopro_ssm_block_weights_t;

typedef struct sopro_nar_config {
  int32_t d_model;        /* 384 */
  int32_t n_layers;       /* cfg.n_layers_nar (6) */
  int32_t kernel;         /* cfg.nar_kernel_size (11) */
  int32_t dilation[SOPRO_MAX_SSM_LAYERS]; /* nn/nar.py:47-52 */
  int32_t n_codebooks;    /* Q = 32 */
  int32_t codebook_size;  /* V = 2048 */
  int32_t head_dim;       /* cfg.nar_head_dim (256) */
  int32_t adapter_hidden; /* 256 (nn/nar.py:14) */
  int32_t n_stages;       /* non-empty stages of B, C, D, E (nn/nar.py:41-44) */
  int32_t stage_first[SOPRO_NAR_MAX_STAGES]; /* first codebook of the stage; stages cover 1..Q-1 consecutively */
  int32_t stage_count[SOPRO_NAR_MAX_STAGES];
} sopro_nar_config_t;

typedef struct sopro_nar_weights {
  sopro_ssm_block_weights_t block[SOPRO_MAX_SSM_LAYERS];  /* nar.blocks.{i} */
  const float* norm_w;                     /* nar.norm.weight [D] */
  const float *pre_w, *pre_b;              /* nar.pre [Hn, D], [Hn] */
  const float* stage_emb;                  /* nar.stage_emb.weight [n_stages, D] */
  const float* adapter_norm_w;             /* nar.adapter.norm.weight [D] */
  const float *adapter_w0, *adapter_b0;    /* nar.adapter.mlp.0 [256, D], [256] */
  const float *adapter_w2, *adapter_b2;    /* nar.adapter.mlp.2 [2D, 256], [2D] */
  const float* head_w[SOPRO_NAR_MAX_CODEBOOKS]; /* nar.heads.{stage}.{j}.weight [V, Hn], indexed by CODEBOOK (1..Q-1) */
  const float* head_b[SOPRO_NAR_MAX_CODEBOOKS];
  const float* head_id_emb[SOPRO_NAR_MAX_STAGES]; /* nar.head_id_emb.{stage}.weight [count, Hn] */
  const float* mix[SOPRO_NAR_MAX_STAGES];         /* nar.mix.{stage} [2] (softmaxed, model.py:335-337) */
  const float* prev_cb_weights;            /* nar_prev_cb_weights [Q] (model.py:70-72) */
  const float* cb_embed;                   /* cb_embed.emb.weight [Q*V + 1, D] */
} sopro_nar_weights_t;

typedef struct sopro_nar sopro_nar_t;
int sopro_nar_create(const sopro_nar_config_t* cfg, const sopro_nar_weights_t* host_weights, int device, sopro_nar_t** out);
int sopro_nar_destroy(sopro_nar_t* n);
/* cond: rows [b][t][d_model] f32 (device), utterance b starting at cond + b*cond_batch_stride (floats) -- cond_ar[:, :T]
 * of the prefill; rvq1 [B, Tmax] i32 (device): the AR tokens; lens [B] i32 (device) or NULL: valid frames per
 * utterance (the refiner is not causal: rows >= lens[b] are padding and act as the zero padding of the convs);
 * codes [B, Tmax, Q] i32 (device) out: codebook 0 = rvq1, 1..Q-1 refined (rows >= lens[b] are undefined). */
int sopro_nar_refine(sopro_nar_t* n, const float* cond, int64_t cond_batch_stride, const int32_t* rvq1, const int32_t* lens,
                     int B, int Tmax, int32_t* codes, void* stream);
/* test hook (teacher forcing): when non-NULL, every stage conditions on the previous codebooks of forced_codes
 * [B, Tmax, Q] i32 (device) instead of on its own argmax results, so one near-tie flip cannot cascade. */
int sopro_nar_set_forced(sopro_nar_t* n, const int32_t* forced_codes);
/* Arithmetic unit of the refiner's contractions: -1 = automatic (tensor cores -- tcgen05, every fp32 operand split into
 * three exact bf16 terms, the six products that reach fp32's last bit, fp32 accumulation -- whenever more than 16 rows are
 * refined; the fp32 FMA skinny kernel below that), 0 = fp32 FMA kernels only (also: environment SOPRO_NAR_TC=0), 1 = as -1
 * but fails if the geometry has no tensor-core images. */
int sopro_nar_set_contraction(sopro_nar_t* n, int mode);
/* One utterance's streaming windows (B == 1, <= 256 frames, no lens / forced codes) are replayed from CUDA graphs captured
 * over internal static buffers (a window is 113..217 launches): identical results, launch overhead removed.  Default on. */
int sopro_nar_set_graphs(sopro_nar_t* n, int enabled);

/* ------------------------------------------------------------------------------------------------
 * Prefill: SoproTTSModel.prepare_conditioning (reference model.py:172-216) for B texts that share one prepared
 * reference voice (sopro_prefill_run) or each bring their own (sopro_prefill_run_voices): TextEncoder (nn/text.py:16-44) -> txt_seq, txt_pool; base = txt_pool + frame sinusoid;
 * SpeakerFiLM (nn/speaker.py:64-85); RefXAttnStack with cached K/V (nn/ref.py:57-108, 111-160); cond_norm -> cond_ar.
 * fp32 (cond_ar / txt_seq feed the id-exact AR kernel).  HOST fp32 weight pointers, state_dict layouts.
 * prepare_reference (once per voice: Token2SV, reference encoder, K/V projections) is sopro_refprep_* below.
 * ------------------------------------------------------------------------------------------------ */
#define SOPRO_PREFILL_MAX_REF_LAYERS 8

typedef struct sopro_prefill_config {
  int32_t d_model;        /* 384 */
  int32_t n_layers_text;  /* cfg.n_layers_text (2) */
  int32_t text_kernel;    /* 7 (nn/text.py:24) */
  int32_t text_vocab;     /* rows of text_enc.embed.emb.weight */
  int32_t sv_dim;         /* cfg.sv_student_dim (192) */
  int32_t ref_layers;     /* cfg.ref_xattn_layers (3) */
  int32_t ref_heads;      /* cfg.ref_xattn_heads (2) */
  float ref_gmax;         /* cfg.ref_xattn_gmax */
  int32_t max_text_len;   /* rows of text_pos */
  int32_t max_frames_pos; /* rows of frame_pos */
} sopro_prefill_config_t;

typedef struct sopro_prefill_ref_layer {
  const float* nq_w;      /* ref_xattn.blocks.{i}.nq.weight [D] */
  const float* q_w;       /* ...q_proj.weight [D, D] */
  const float* o_w;       /* ...out_proj.weight [D, D] */
  float gate;             /* ...gate (scalar; gmax * tanh(gate) is applied, nn/ref.py:105) */
} sopro_prefill_ref_layer_t;

typedef struct sopro_prefill_weights {
  const float* text_emb;   /* text_enc.embed.emb.weight [vocab, D] */
  const float* text_pos;   /* sinusoid table [max_text_len, D] (nn/embeddings.py:11-25; a non-persistent buffer) */
  const float* frame_pos;  /* sinusoid table [max_frames_pos, D] */
  sopro_ssm_block_weights_t text_block[SOPRO_MAX_SSM_LAYERS]; /* text_enc.layers.{i} */
  const float* text_norm_w;             /* text_enc.norm.weight */
  const float *film_w0, *film_b0;       /* spk_film.mlp.0 [D, sv], [D] */
  const float *film_w2, *film_b2;       /* spk_film.mlp.2 [2D, D], [2D] */
  const float *film_norm_w, *film_norm_b; /* spk_film.norm (LayerNorm) */
  sopro_prefill_ref_layer_t ref_layer[SOPRO_PREFILL_MAX_REF_LAYERS];
  const float* cond_norm_w;             /* cond_norm.weight */
} sopro_prefill_weights_t;

typedef struct sopro_prefill sopro_prefill_t;
int sopro_prefill_create(const sopro_prefill_config_t* cfg, const sopro_prefill_weights_t* host_weights, int device,
                         sopro_prefill_t** out);
int sopro_prefill_destroy(sopro_prefill_t* p);
/* All pointers below are DEVICE pointers.  text_ids [B, Lmax] i32 (padded), text_len [B] i32; sv [B or 1, sv_dim]
 * (sv_shared != 0: one speaker vector for the batch); ref_k / ref_v: HOST arrays of ref_layers device pointers to the
 * prepared reference's cached K / V [H, Tr, D/H] (PreparedReference.ref_kv_caches, model.py:45-50);
 * n_frames = max_frames + 1.  Outputs: txt_seq [B, Lmax, D] (rows >= text_len[b] undefined), txt_pool [B, D],
 * cond_ar [B, n_frames, D] -- the `prep` dict of model.py:210-216. */
int sopro_prefill_run(sopro_prefill_t* p, const int32_t* text_ids, const int32_t* text_len, int B, int Lmax, const float* sv,
                      int sv_shared, const float* const* ref_k, const float* const* ref_v, int Tr, float style_strength,
                      int n_frames, float* txt_seq, float* txt_pool, float* cond_ar, void* stream);
/* The same prefill for B texts that each bring their own prepared voice (n_voices distinct voices in the call).
 * DEVICE: text_ids [B, Lmax] i32, text_len [B] i32, sv [n_voices, sv_dim] (row v: voice v's speaker vector); outputs
 * as sopro_prefill_run.  HOST (reusable as soon as the call returns; the tables are staged into the engine's workspace
 * on `stream`): voice [B] i32, text b's voice in [0, n_voices); ref_len [n_voices] i32, Tr of each voice in [1, 4096];
 * ref_k / ref_v [ref_layers * n_voices] device pointers, entry l * n_voices + v = voice v's cached K / V of layer l,
 * [H, Tr_v, D/H] (PreparedReference.ref_kv_caches[l]).  Utterance b's txt_seq / txt_pool / cond_ar rows are bit-equal
 * to what sopro_prefill_run computes for the same texts with voice[b]'s reference shared by all of them (sv_shared = 1).
 * A null pointer, n_voices < 1, a voice index or a Tr out of range return SOPRO_ERR_INVALID before any launch. */
int sopro_prefill_run_voices(sopro_prefill_t* p, const int32_t* text_ids, const int32_t* text_len, int B, int Lmax,
                             const int32_t* voice, int n_voices, const float* sv, const int32_t* ref_len,
                             const float* const* ref_k, const float* const* ref_v, float style_strength, int n_frames,
                             float* txt_seq, float* txt_pool, float* cond_ar, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Reference preparation: SoproTTSModel.prepare_reference (reference model.py:152-170), once per voice, from the
 * voice's codes: Token2SV (nn/speaker.py:12-61, AttentiveStatsPool nn/blocks.py:165-188) -> sv_ref;
 * _encode_reference_seq (model.py:136-150) -> ref_seq; RefXAttnStack.build_kv_caches (nn/ref.py) -> the K / V the
 * prefill engine reads.  fp32.  HOST fp32 weight pointers, state_dict layouts.
 * ------------------------------------------------------------------------------------------------ */
typedef struct sopro_refprep_config {
  int32_t d_model;        /* 384 */
  int32_t sv_embed_dim;   /* 192: Token2SV's d */
  int32_t sv_dim;         /* cfg.sv_student_dim (192) */
  int32_t n_codebooks;    /* 32 */
  int32_t codebook_size;  /* 2048 */
  int32_t sv_kernel;      /* 7 (nn/speaker.py:24,27) */
  int32_t ref_enc_layers; /* cfg.ref_enc_layers (2) */
  int32_t ref_enc_kernel; /* 7 */
  int32_t ref_layers;     /* cfg.ref_xattn_layers (3) */
  int32_t ref_heads;      /* cfg.ref_xattn_heads (2) */
} sopro_refprep_config_t;

typedef struct sopro_refprep_kv_layer {
  const float* nkv_w;     /* ref_xattn.blocks.{i}.nkv.weight [D] */
  const float* k_w;       /* ...k_proj.weight [D, D] */
  const float* v_w;       /* ...v_proj.weight [D, D] */
} sopro_refprep_kv_layer_t;

typedef struct sopro_refprep_weights {
  const float* sv_emb;          /* token2sv.emb.weight [Q*V, d] */
  const float* sv_cb_weights;   /* token2sv.cb_weights [Q] (softmax taken by the engine) */
  const float *sv_dw0_w, *sv_dw0_b; /* token2sv.enc.0.dw [d, 1, k], [d] */
  const float *sv_dw1_w, *sv_dw1_b; /* token2sv.enc.3.dw */
  const float *pool_w0, *pool_b0;   /* token2sv.pool.attn.0 [d, d], [d] */
  const float* pool_w2;             /* token2sv.pool.attn.2.weight [1, d] */
  float pool_b2;                    /* token2sv.pool.attn.2.bias */
  const float *proj_w, *proj_b;     /* token2sv.proj [sv, 2d], [sv] */
  const float* cb_embed;            /* cb_embed.emb.weight [>= Q*V, D] (the first Q*V rows are read) */
  const float* ref_cb_weights;      /* ref_cb_weights [Q] */
  sopro_ssm_block_weights_t ref_block[SOPRO_MAX_SSM_LAYERS]; /* ref_enc_blocks.{i} */
  const float* ref_norm_w;          /* ref_enc_norm.weight */
  sopro_refprep_kv_layer_t layer[SOPRO_PREFILL_MAX_REF_LAYERS];
} sopro_refprep_weights_t;

typedef struct sopro_refprep sopro_refprep_t;
int sopro_refprep_create(const sopro_refprep_config_t* cfg, const sopro_refprep_weights_t* host_weights, int device,
                         sopro_refprep_t** out);
int sopro_refprep_destroy(sopro_refprep_t* p);
/* DEVICE pointers: tokens [Tr, Q] i32 -> sv [sv_dim], ref_seq [Tr, D]; ref_k / ref_v: HOST arrays of ref_layers device
 * pointers, each [H, Tr, D/H] (PreparedReference.ref_kv_caches[i]["k"/"v"], model.py:45-50). */
int sopro_refprep_run(sopro_refprep_t* p, const int32_t* tokens, int Tr, float* sv, float* ref_seq, float* const* ref_k,
                      float* const* ref_v, void* stream);
/* synchronises `stream`; SOPRO_ERR_INVALID if a run since the last check met a code outside [0, codebook_size) (the
 * reference's embedding lookup raises IndexError); clears the flag */
int sopro_refprep_check(sopro_refprep_t* p, void* stream);

/* test hook: one tensor-core implicit GEMM (no reference counterpart).  X bf16 [B][rows][cin] (device),
 * W bf16 [N][taps*cin] (device); out[b][m][n] = epi(sum_j sum_ci X[b][m + j*dil - pad][ci] * W[n][j*cin+ci] +
 * bias[n % bias_mod]); epi: 0 none, 1 GELU(erf), 2 R + scale*acc, 3 R + acc; out_f32 / out_bf16 may be null;
 * out_elu applies ELU to the bf16 copy only. */
int sopro_debug_tc_gemm(const void* X, int B, int64_t rows, int cin, int taps, int dil, int pad, const void* W, int N,
                        const float* bias, int bias_mod, int epi, const float* R, const float* scale, float* out_f32,
                        void* out_bf16, int out_elu, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* SOPRO_B200_H_ */
