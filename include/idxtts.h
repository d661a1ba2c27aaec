/*
 * idxtts.h — C-ABI of libidxtts.so, the B200 (sm_100a) compute library behind the
 * IndexTTS / IndexTTS2 `.infer()` entry points.
 *
 * Every entry point replaces one "module-level seam" of the reference pipeline
 * (SURVEY.md §8b).  The reference file:line each one stands in for is cited on the
 * declaration.  Rules that hold for every call:
 *
 *   - plain C types only: opaque handle, raw pointers, sizes; no torch/C++ types.
 *   - data pointers may be HOST or DEVICE pointers; the library inspects them with
 *     cudaPointerGetAttributes and stages host buffers through pinned memory on its
 *     own stream (the copies are therefore inside any timing of the call).
 *   - the caller owns every input and output buffer; the engine owns only its packed
 *     weights, KV cache and work arenas.
 *   - return value: 0 on success, non-zero error code otherwise; the message is
 *     available from idx_last_error().  The Python shim turns it into RuntimeError,
 *     like the reference's AT_ERROR in anti_alias_activation_cuda.cu:214-225.
 *   - one handle = one CUDA device = one caller thread at a time (the reference is
 *     not re-entrant either: infer_v2_5.py:268-275, gpt/model_v2.py:88).
 *   - calls are synchronous with respect to the host unless stated otherwise.
 *   - STREAM CONTRACT: the engine launches on its own non-blocking stream.  Device buffers handed
 *     to a call must be complete with respect to that stream: a caller that produced them with
 *     asynchronous work on another stream (e.g. torch's current stream) calls
 *     idx_wait_stream(e, that_stream) first — the engine stream then waits (on the device, no host
 *     block) for everything queued on that stream so far.  The Python shim does this before every
 *     call.  Outputs need nothing: every call drains the engine stream before it returns.
 */
#ifndef IDXTTS_H
#define IDXTTS_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct idx_engine idx_engine;

typedef enum {
  IDX_F32 = 0,
  IDX_BF16 = 1,
  IDX_F16 = 2,
  IDX_I32 = 3,
  IDX_I64 = 4
} idx_dtype;

enum {
  IDX_OK = 0,
  IDX_ERR_CUDA = 1,     /* a CUDA runtime call or kernel failed                    */
  IDX_ERR_ARG = 2,      /* bad argument / shape / missing weight                    */
  IDX_ERR_STATE = 3,    /* call order violated (e.g. generate before finalize)      */
  IDX_ERR_NOGPU = 4     /* no sm_100 device: there is NO CPU fallback, by design    */
};

/* ------------------------------------------------------------------ lifecycle -- */

/* Create an engine bound to CUDA device `device`.  Fails with IDX_ERR_NOGPU when no
 * CUDA device is visible — the product path never falls back to the CPU.           */
int idx_create(int device, idx_engine** out);
void idx_destroy(idx_engine* e);
/* Last error message of this engine (or of the failed idx_create when e == NULL).   */
const char* idx_last_error(const idx_engine* e);
/* Library/ABI version and build flags ("sm_100a;...").                              */
const char* idx_version(void);
/* Number of kernel launches issued by this engine since creation (bench.py reports
 * the delta over the timed region as `gpu_launches`).                               */
int64_t idx_launch_count(const idx_engine* e);
/* Block until all work queued by this engine has finished.                          */
int idx_sync(idx_engine* e);
/* Order the engine stream after all work queued so far on `cuda_stream` (a cudaStream_t passed as
 * void*; NULL = the legacy default stream): event record + cudaStreamWaitEvent, no host block.  */
int idx_wait_stream(idx_engine* e, void* cuda_stream);
/* CUDA events on the engine's own stream (slots 0..15) — what bench.py times with, since the
 * engine does not launch on torch's current stream.                                   */
int idx_event_record(idx_engine* e, int slot);
int idx_event_elapsed_ms(idx_engine* e, int slot_a, int slot_b, double* ms);

/* Engine options.  "gemm_backend": 0 = automatic (tcgen05 implicit GEMM wherever the shape
 * allows — the default), 1 = SIMT fp32 everywhere (strict-fp32 parity runs).  "tail_f16" (with gemm_backend 0): 1 = the
 * DiT / WaveNet / BigVGAN-resblock GEMMs read fp16 operands (kind::f16; activations written as fp16 by the kernel that
 * produces them, fp32 accumulate and fp32 residual streams — the default), 0 = tf32 over fp32 storage (round 1).
 * Options belong to the handle: another engine (another GPU, another thread) keeps its own.        */
int idx_set_option(idx_engine* e, const char* name, int value);

/* -------------------------------------------------------------------- weights -- */

/* Register one tensor of a checkpoint under its reference state-dict name, prefixed
 * by the module it belongs to ("gpt.", "bigvgan.", "s2mel.", "codec." ...).
 * Replaces `load_checkpoint` (indextts/utils/checkpoint.py:22-35) + `.to(device)`
 * (infer_v2_5.py:141-146): the Python loader walks the state dict and calls this
 * once per tensor.  The engine keeps its own copy (repacked at finalize time), so
 * the caller may free `data` as soon as the call returns.                           */
int idx_load_weight(idx_engine* e, const char* name, const void* data, int dtype,
                    int ndim, const int64_t* shape);

/* ------------------------------------------------------------------------ GPT -- */

/* Geometry of UnifiedVoice (indextts/gpt/model_v2.py:305-420).                      */
typedef struct {
  int32_t layers;            /* cfg.gpt.layers                                      */
  int32_t model_dim;         /* cfg.gpt.model_dim (1280)                            */
  int32_t heads;             /* cfg.gpt.heads (head_dim must be 64)                 */
  int32_t number_mel_codes;  /* 8194                                                */
  int32_t start_mel_token;   /* 8192                                                */
  int32_t stop_mel_token;    /* 8193                                                */
  int32_t max_mel_positions; /* rows of mel_pos_embedding.emb.weight                */
  int32_t max_prompt;        /* longest [cond][text] prompt the KV cache must hold  */
  int32_t max_batch;         /* concurrent sequences (beams count as sequences)     */
  int32_t weights_bf16;      /* 1: bf16 weights + autocast rounding points (use_bf16
                                path, infer_v2_5.py:143-146,758); 0: fp32           */
} idx_gpt_config;

/* Pack the registered "gpt.*" tensors into the per-SM weight streams of the fused
 * decode kernel and allocate the KV cache.  Replaces post_init_gpt2_config
 * (gpt/model_v2.py:422-493).                                                         */
int idx_gpt_init(idx_engine* e, const idx_gpt_config* cfg);

/* Sampling parameters = the hf_generate_kwargs consumed by
 * GenerationMixin.generate (gpt/transformers_generation_utils.py:1869-2385), in the
 * processor order fixed at :900-905,1019-1047.                                      */
typedef struct {
  int32_t do_sample;            /* 0: greedy argmax                                  */
  int32_t num_beams;            /* 1, or 2..4: beam search (do_sample = 1: beam-sample,
                                   the reference default num_beams = 3); each request
                                   then occupies num_beams rows: nreq * num_beams <= 8 */
  int32_t top_k;                /* 0 = off                                           */
  float top_p;                  /* 1.0 = off                                         */
  float temperature;            /* 1.0 = off                                         */
  float repetition_penalty;     /* 1.0 = off; reference default 10.0                 */
  float length_penalty;         /* beams only                                        */
  int32_t max_new_tokens;       /* max_generate_length                               */
  uint64_t seed;                /* Philox seed of the device sampler                 */
  int32_t forbid_stop_before;   /* mask stop_mel_token for the first n steps (bench:
                                   length-deterministic runs, SURVEY §8d); 0 = off   */
  int32_t mel_pos_mode;         /* 0: KV-cache rule — step k >= 1 sits at mel position k+1
                                   (trap P1, gpt/model_v2.py:158-161); 1: the rule of decoding
                                   WITHOUT a cache, the v1 CPU default (infer.py:101,
                                   gpt/model.py:139-156): position k                      */
} idx_sampling;

/* One utterance (= one text segment) of a generate call.                            */
typedef struct {
  const void* prompt_emb;   /* [prompt_len, model_dim] f32: the [cond][text] embeddings
                               produced by prepare_gpt_inputs (model_v2.py:648-714),
                               without left padding                                   */
  int32_t prompt_len;
  int32_t* codes_out;       /* [max_new_tokens] generated codes, stop token included  */
  int32_t* n_codes_out;     /* number of codes written                                */
  float* logits_out;        /* optional [max_new_tokens, number_mel_codes] f32 of the
                               raw step logits (tests); NULL to skip.  With
                               num_beams > 1: [max_new_tokens, num_beams, codes]      */
  const int32_t* forced_codes; /* optional teacher forcing: feed these codes instead of
                               the sampled ones (tests); NULL for free running        */
} idx_gpt_request;

/* Autoregressive speech-token generation for `nreq` utterances decoded as one batch.
 * Replaces UnifiedVoice.inference_speech → GPT2InferenceModel.generate
 * (gpt/model_v2.py:716-825, :121-198) and the HF _sample loop
 * (transformers_generation_utils.py:3123-3297).                                      */
int idx_gpt_generate(idx_engine* e, const idx_gpt_request* reqs, int nreq,
                     const idx_sampling* sp);

/* Build the [cond(3)][start_text, text.., stop_text] prompt embeddings of
 * prepare_gpt_inputs (gpt/model_v2.py:648-714,754-768) on the device.
 *   style      [192] f32   campplus embedding (infer_v2_5.py:644-649)
 *   emo_vec    [model_dim] f32 merged emotion vector (model_v2.py:833-838)
 *   text_ids   [n_text] i32 (without start/stop), lang id
 *   out        [3 + n_text + 2, model_dim] f32                                       */
int idx_gpt_prepare_inputs(idx_engine* e, const float* style, const float* emo_vec,
                           const int32_t* text_ids, int n_text, int lang, float* out);

/* Emotion-vector path (SURVEY §8a row a7): ConformerEncoder(conv2d2, rel-pos) + PerceiverResampler(1 latent)
 * + emovec_layer + emo_layer of UnifiedVoice (gpt/model_v2.py:375-392).                              */
typedef struct {
  int32_t idim;          /* 1024 (w2v-BERT features)                                            */
  int32_t odim;          /* emo_condition_module.output_size (512)                              */
  int32_t linear_units;  /* 1024                                                                */
  int32_t heads;         /* attention_heads (4)                                                 */
  int32_t blocks;        /* num_blocks (4)                                                      */
  int32_t cnn_kernel;    /* 15                                                                  */
  int32_t p_dim;         /* perceiver dim (1024)                                                */
  int32_t p_heads;       /* 4                                                                   */
  int32_t p_dim_head;    /* 64                                                                  */
  int32_t p_depth;       /* 2                                                                   */
  int32_t p_ff_mult;     /* perceiver_mult (2)                                                  */
  int32_t model_dim;     /* 1280                                                                */
} idx_emo_config;
int idx_emo_init(idx_engine* e, const idx_emo_config* cfg);

/* base + alpha * (emo - base), each = emo_layer(emovec_layer(perceiver(conformer(feats)))).
 * spk_feats [Ts, idim], emo_feats [Te, idim] (NULL or the same pointer = same audio) → emo_vec [model_dim].
 * Replaces UnifiedVoice.merge_emovec (gpt/model_v2.py:833-838), call site infer_v2_5.py:759-765; callers
 * cache the result per (speaker, emotion, alpha) — the reference recomputes it per segment (trap P11).   */
int idx_merge_emovec(idx_engine* e, const float* spk_feats, int Ts, const float* emo_feats, int Te,
                     float alpha, float* emo_vec_out);

/* ---- IndexTTS v1 / v1.5 GPT side (SURVEY section 8 row a13, indextts/gpt/model.py) ------------------------------
 * Prompt encoder: ConformerEncoder(100-bin mel, conv2d2) + PerceiverResampler(n_latents = 32) -> conds
 * (get_conditioning, model.py:493-503); tensors "gpt.conditioning_encoder.*", "gpt.perceiver_encoder.*".           */
int idx_v1_cond_init(idx_engine* e, const idx_emo_config* cfg, int n_latents);
/* mel [T, idim] f32 -> conds [n_latents, model_dim] f32                                                           */
int idx_v1_get_conditioning(idx_engine* e, const float* mel, int T, float* conds_out);
/* prepare_gpt_inputs of v1 (model.py:597-660): [conds][text_embedding(start, text.., stop) + text_pos(0..)]
 *   out [n_latents + n_text + 2, model_dim] f32 — the prompt rows for idx_gpt_generate                             */
int idx_gpt_prepare_inputs_v1(idx_engine* e, const float* conds, int n_latents, const int32_t* text_ids, int n_text,
                              float* out);
/* UnifiedVoice.forward(..., return_latent=True) (model.py:526-589) for one utterance: one teacher-forced pass over
 * [conds][start_text, text, stop_text][start_mel, codes.., stop_mel]; final_norm(ln_f(hidden)) at the mel
 * positions without the last two -> latents [n_codes, model_dim] f32, the input of idx_v1_vocode.                  */
int idx_gpt_latents_v1(idx_engine* e, const float* conds, int n_latents, const int32_t* text_ids, int n_text,
                       const int32_t* codes, int n_codes, float* latents_out);


/* Beam search trace of the last idx_gpt_generate call with num_beams > 1 (tests, debugging): for every step and
 * beam slot the (parent beam, token) chosen by BeamSearchScorer.process
 * (gpt/transformers_beam_search.py:215-320) and the running beam score; the score of the returned hypothesis
 * (BeamSearchScorer.finalize :322-420).
 *   parents_tokens [max_steps][num_beams][2] i32, scores [max_steps][num_beams] f32 (either may be NULL)    */
int idx_gpt_beam_trace(const idx_engine* e, int utterance, int32_t* parents_tokens, float* scores,
                       int max_steps, int32_t* steps_out, double* final_score);

/* Timing of the last generate call, measured with CUDA events on the engine stream:
 * out[0] = prefill ms, out[1] = decode ms, out[2] = decode steps,
 * out[3] = fused-step kernel launches.                                               */
int idx_gpt_last_timing(const idx_engine* e, double* out4);

/* Diagnostic: when `enable` is non-zero the fused kernel records %globaltimer (ns) of CTA 0 at
 * every phase boundary of the last step of each launch (2 stamps per grid barrier: before and
 * after).  Copies up to n (<= 256) stamps of the most recent launch into stamps_out.          */
int idx_gpt_profile(idx_engine* e, int enable, int64_t* stamps_out, int n);
/* Diagnostic (profiling enabled as above): %globaltimer stamps of EVERY CTA at the sub-phase boundaries of the middle
 * layer of the last decode step: stamps_out [num_SMs][64] (0 where a slot is unused).                          */
int idx_gpt_profile_fine(idx_engine* e, int64_t* stamps_out, int n);

/* ------------------------------------------------------------------- BigVGAN -- */

/* Geometry of the BigVGAN-v2 generator (s2mel/modules/bigvgan/config.json:11-21).    */
typedef struct {
  int32_t num_mels;                 /* 80                                            */
  int32_t upsample_initial_channel; /* 1536                                          */
  int32_t num_upsamples;            /* 6                                             */
  int32_t upsample_rates[8];        /* 4,4,2,2,2,2                                   */
  int32_t upsample_kernel_sizes[8]; /* 8,8,4,4,4,4                                   */
  int32_t num_kernels;              /* 3                                             */
  int32_t resblock_kernel_sizes[4]; /* 3,7,11                                        */
  int32_t resblock_dilations[4][3]; /* 1,3,5 each                                    */
  int32_t use_tanh_at_final;        /* 0 → clamp(-1,1)                               */
  int32_t use_bias_at_final;        /* 0                                             */
  int32_t snake_logscale;           /* 1                                             */
} idx_bigvgan_config;

/* Fold/pack "bigvgan.*" (weight-norm already removed, as after
 * bigvgan.remove_weight_norm(), infer_v2_5.py:229-232).                              */
int idx_bigvgan_init(idx_engine* e, const idx_bigvgan_config* cfg);

/* mel [B, num_mels, F] f32 (reference NCT layout) → wav [B, 1, F*prod(rates)] f32.
 * Replaces BigVGAN.forward (s2mel/modules/bigvgan/bigvgan.py:360-386), call site
 * infer_v2_5.py:850.                                                                 */
int idx_bigvgan_forward(idx_engine* e, const float* mel, int B, int F, float* wav);

/* Standalone anti-aliased SnakeBeta activation: x[B,C,T] f32 → y[B,C,T] f32.
 * Drop-in for the reference's only native FFI, `fwd_cuda`
 * (alias_free_activation/cuda/anti_alias_activation_cuda.cu:214-225), with the
 * torch-path semantics of alias_free_activation/torch/act.py:8-30.
 * alpha/beta are the log-scale per-channel parameters [C].                           */
int idx_antialias_snake(idx_engine* e, const float* x, const float* alpha,
                        const float* beta, int B, int C, int T, int logscale, float* y);

/* ---- IndexTTS v1 / v1.5 vocoder (SURVEY section 8 row a13) -------------------------------------------------------
 * Latent-conditioned BigVGAN with its ECAPA-TDNN speaker encoder (indextts/BigVGAN/models.py:129-249,
 * indextts/BigVGAN/ECAPA_TDNN.py:429-582), tensors registered under "bigvgan_v1." (weight norm removed as after
 * BigVGAN.remove_weight_norm(), models.py:251-262).  gen_cfg->num_mels = gpt_dim (the latent width).              */
int idx_v1_vocoder_init(idx_engine* e, const idx_bigvgan_config* gen_cfg, int n_mels, int speaker_embedding_dim,
                        int cond_in_each_up_layer);
/* ECAPA_TDNN.forward for one full-length utterance: mel_ref [Tm, n_mels] f32 -> emb [speaker_embedding_dim].      */
int idx_v1_speaker_embedding(idx_engine* e, const float* mel_ref, int Tm, float* emb_out);
/* BigVGAN.forward(x, mel_ref) (models.py:201-249; call site infer.py:~660): latent [T, gpt_dim] f32 and the
 * reference mel [Tm, n_mels] f32 -> wav [T * prod(rates)] f32 in [-1, 1] (tanh).                                   */
int idx_v1_vocode(idx_engine* e, const float* latent, int T, const float* mel_ref, int Tm, float* wav_out);

/* Device time of the last idx_bigvgan_forward in ms (CUDA events).                   */
int idx_bigvgan_last_ms(const idx_engine* e, double* ms);

/* Diagnostic (tests): one multi-tap channels-last GEMM — the building block of every Conv1d /
 * ConvTranspose1d / Linear of the vocoder and s2mel paths — through a chosen back end
 * (backend 1 = SIMT fp32, 2 = tcgen05 tf32, 0 = automatic).  wk is K-major [N][taps*K];
 * D[b][m][n] = scale*(act(sum + bias) + res + (accum ? out : 0)) stored at
 * out[b*out_elems_per_batch + out_off + m*ldo + n] where 0 <= flat < out_valid.            */
int idx_debug_conv_gemm(idx_engine* e, const float* A, int B, int Tin, int K, const float* wk,
                        int taps, int dil, int pad, int M, int N, const float* bias, int biasN,
                        int act, const float* res, int accum, float scale, long long out_off,
                        int ldo, long long out_valid, long long out_elems_per_batch, int backend,
                        float* out);

/* Diagnostic (tests): the fp16 tensor-core GEMM of idx_debug_conv_gemm with a fused pair epilogue, its operands
 * prepared as the DiT / WaveNet prepare them (fp16 images of A and wk; SwiGLU / gate weight rows and bias interleaved).
 * wk [N][taps*K] and bias [N] (or null) in the module's row order; fp16 results as raw bits:
 *   epi 1 (SwiGLU): rows w1 | w3  -> out16 [B][M][N/2] = silu(w1 x + b1) * (w3 x + b3)
 *   epi 2 (gate):   rows a | c    -> out16 [B][M][N/2] = tanh(a + g[b][j]) * sigmoid(c + g[b][N/2 + j]),
 *                   g = aux [B][aux_stride] (aux_stride 0: one [N] vector for every batch entry)
 *   epi 3 (RoPE):   rows q | k | v of H = aux_stride heads of 64 (N = 192 H), RoPE table over T = M rows (aux unused)
 *                   -> out16 = Qr | Kr | Vb, each [B*H][M][64]: q rotated and multiplied by scale, k rotated, v as is.
 * N % 32 != 0 or a missing gate vector returns IDX_ERR_ARG.                                                    */
int idx_debug_gemm_pair_epilogue(idx_engine* e, const float* A, int B, int Tin, int K, const float* wk,
                                 int taps, int dil, int pad, int M, int N, const float* bias, int epi,
                                 const float* aux, int aux_stride, float scale, uint16_t* out16);

/* Diagnostic (tests): flash attention over fp16 qkv16 = Qr | Kr | Vb, each [B*H][T][64] (what epi 3 above writes),
 * through kernel 1 (mma.sync; q pre-scaled by 1/8, softmax in base e) or 2 (tcgen05; q pre-scaled by log2(e)/8,
 * softmax in base 2).  out [B][T][H*64] f32 and / or out16 (fp16 bits, same shape); either may be null.          */
int idx_debug_flash_attention(idx_engine* e, const uint16_t* qkv16, int B, int T, int H, int kernel,
                              float* out, uint16_t* out16);

/* Diagnostic (tests): the DiT attention with interleaved-pair RoPE (base 1e4) on fp32 qkv [B][T][3*H*64] (q | k | v)
 * -> out [B][T][H*64] through backend 1 (SIMT fp32) or 0 (fp16 rotate / split + mma.sync flash kernel).           */
int idx_debug_attention_rope(idx_engine* e, const float* qkv, int B, int T, int H, int backend, float* out);

/* ---------------------------------------------------------------- s2mel + codec -- */

/* Geometry of the s2mel section of config.yaml as MyModel reads it
 * (s2mel/modules/commons.py:390-414, diffusion_transformer.py:103-184).              */
typedef struct {
  int32_t hidden;        /* DiT.hidden_dim (512)                                        */
  int32_t heads;         /* DiT.num_heads (8; head_dim must be 64)                      */
  int32_t depth;         /* DiT.depth (13)                                              */
  int32_t wn_hidden;     /* wavenet.hidden_dim (512, must equal hidden)                 */
  int32_t wn_layers;     /* wavenet.num_layers (8)                                      */
  int32_t wn_kernel;     /* wavenet.kernel_size (5)                                     */
  int32_t in_channels;   /* DiT.in_channels (80 mel bins)                               */
  int32_t content_dim;   /* DiT.content_dim = length_regulator.channels (512)           */
  int32_t style_dim;     /* style_encoder.dim (192)                                     */
  int32_t lr_in;         /* length_regulator.in_channels (1024)                         */
  int32_t lr_convs;      /* len(length_regulator.sampling_ratios) (4)                   */
} idx_s2mel_config;

/* Pack "s2mel.cfm.*" and "s2mel.length_regulator.*" (weight norm folded by the loader, the
 * same tensors load_checkpoint2 reads: s2mel/modules/commons.py:579-635).              */
int idx_s2mel_init(idx_engine* e, const idx_s2mel_config* cfg);

/* EnhancedCodec geometry (codec/models.py:23-39).                                      */
typedef struct {
  int32_t codebook_size, hidden_size, codebook_dim, vocos_dim, vocos_intermediate_dim,
      vocos_num_layers;
} idx_codec_config;
int idx_codec_init(idx_engine* e, const idx_codec_config* cfg);

/* codes [n] i32 → S_infer [2n, hidden_size] f32.  Replaces EnhancedCodec.decode
 * (codec/models.py:205-231), call site infer_v2_5.py:832.                              */
int idx_codec_decode(idx_engine* e, const int32_t* codes, int n, float* S_out);

/* S [n_in, lr_in] → cond [ylen, content_dim].  Replaces InterpolateRegulator.forward
 * (s2mel/modules/length_regulator.py:90-141), call site infer_v2_5.py:835-838
 * (ylen = int(n_in * 1.72 * duration_factor), computed by the caller).                 */
int idx_length_regulate(idx_engine* e, const float* S, int n_in, int ylen, float* cond_out);

/* One evaluation of the CFM estimator: x, prompt_x [B,80,T], t [B], style [B,style_dim],
 * cond [B,T,content_dim] → out [B,80,T].  Replaces DiT.forward
 * (s2mel/modules/diffusion_transformer.py:186-257); full-length sequences (x_lens = T).  */
int idx_dit_forward(idx_engine* e, const float* x, const float* prompt_x, const float* t,
                    const float* style, const float* cond, int B, int T, float* out);

/* Euler solve of the flow-matching ODE with classifier-free guidance:
 *   mu [T, content_dim], prompt [80, P] (reference mel), style [style_dim], z [80, T] (the
 *   torch.randn noise the caller drew — trap P6), n_steps (25), cfg_rate (0.7) → mel [80, T]
 *   with the first P frames zeroed.  Replaces BASECFM.inference / solve_euler
 *   (s2mel/modules/flow_matching.py:30-115), call site infer_v2_5.py:841-845.           */
int idx_cfm_solve(idx_engine* e, const float* mu, int T, const float* prompt, int P,
                  const float* style, const float* z, int n_steps, float cfg_rate, float* mel_out);

/* The per-segment tail of IndexTTS2.infer (infer_v2_5.py:827-856) as one call.            */
typedef struct {
  const int32_t* codes;           /* [n_codes] generated codes, cut before stop_mel_token (:809-821) */
  int32_t n_codes;
  const float* prompt_condition;  /* [P, content_dim] length-regulated reference features (:651-656)  */
  const float* ref_mel;           /* [80, P] reference mel (:640)                                     */
  int32_t P;
  const float* style;             /* [style_dim] campplus style vector, 192 in IndexTTS-2.5 (:644-649)   */
  const float* z;                 /* [80, P + F] the torch.randn noise of cfm.inference (trap P6)     */
  int32_t F;                      /* int(2 * n_codes * 1.72 * duration_factor) (:833)                 */
  float* wav_out;                 /* optional [F * 256] f32 in [-1, 1]                                */
  int16_t* pcm16_out;             /* optional [F * 256] clamp(32767*wav) as int16 (:855)              */
  float* mel_out;                 /* optional [80, F] generated mel (tests)                           */
} idx_vocode_request;

/* codes → codec decode → length regulator → CFM (n_steps, cfg_rate) → BigVGAN → waveform.     */
int idx_codes_to_wav(idx_engine* e, const idx_vocode_request* r, int n_steps, float cfg_rate);

/* Device ms of the last codec decode / length regulator / CFM solve (CUDA events).       */
int idx_s2mel_last_ms(const idx_engine* e, double* ms3);

#ifdef __cplusplus
}
#endif
#endif /* IDXTTS_H */
