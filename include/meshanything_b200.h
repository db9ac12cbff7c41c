/*
 * meshanything_b200.h -- C ABI of libmeshanything_b200.so (sm_100a).
 *
 * The reference (buaacyw/MeshAnything) exposes no FFI: its boundary is the Python surface
 * (SURVEY.md section 8b).  These entry points are the seams inside `MeshAnything.forward`
 * (/root/reference/MeshAnything/models/meshanything.py:134-176) that the drop-in Python facade
 * (MeshAnything/models/meshanything.py in this repo) binds with ctypes; INTEGRATION.md shows the
 * binding.  Plain pointers and sizes only; all pointers are DEVICE pointers unless noted; the
 * caller (PyTorch) owns every allocation; no entry point allocates device memory or synchronises
 * the device unless stated.  Every function returns 0 on success, non-zero on error
 * (ma_last_error() gives the message).  `stream` is a cudaStream_t passed as void*.
 *
 * Numerics: fp16 weights/activations at the reference's autocast rounding points, fp32
 * accumulation in the canonical order of DESIGN.md section 3 (bit-exact against oracle/).
 */
#ifndef MESHANYTHING_B200_H
#define MESHANYTHING_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MA_ABI_VERSION 1
#define MA_MAX_LAYERS 32

/* epilogues of ma_linear_f16 */
#define MA_EPI_NONE 0
#define MA_EPI_RELU 1 /* OPTDecoderLayer activation_fn (opt-350m: relu) */
#define MA_EPI_GELU 2 /* nn.GELU() exact erf: transformer_blocks.py:239, BERT intermediate */
/* OR-ed into `epilogue`: the segmented accumulation order of the decoder's split-K layers (DESIGN.md section 3):
 * 16 segment dots (64-wide: out_proj, K = 1024; 256-wide: fc2, K = 4096) added with a balanced tree. */
#define MA_LIN_SEG64 0x10
#define MA_LIN_SEG256 0x20

int ma_abi_version(void);
const char* ma_last_error(void);

/* ---- canonical building blocks (also the unit-test surface) ------------------------------- */

/* y[m][n] = fp16( dot(W[n][:], x[m][:]) + bias[n] ) then epilogue.  Replaces nn.Linear under fp16
 * autocast (every q/k/v/out_proj/fc1/fc2/lm_head/input_layer call of shape_opt.py:243,155 and HF
 * OPTDecoderLayer).  W [N][K] fp16 row-major, bias [N] fp16 or NULL, x [M][ldx] fp16, y [M][ldy]
 * fp16.  K % 256 == 0. */
int ma_linear_f16(const void* W, const void* bias, const void* x, int ldx, void* y, int ldy, int M, int N, int K,
                  int epilogue, void* stream);

/* h = x (+ float(res16)); out = LayerNorm(h) * gamma + beta  (fp32 statistics).  Replaces the
 * residual add + nn.LayerNorm pairs of OPTDecoderLayer (post-LN) and the miche/BERT LayerNorms.
 * x fp32 [M][W] or NULL (then h = float(res16)), res16 fp16 [M][W] or NULL; out32 / out16 optional.
 * W in {768, 1024}. */
int ma_layernorm(const float* x, const void* res16, const float* gamma, const float* beta, float eps, int M, int W,
                 float* out32, void* out16, void* stream);

/* Row m attends keys [0, nkeys[m]) of cache slot slots[m] (NULL: slot 0): softmax(q k^T * scale) v,
 * fp32 accumulate, fp16 out.  Replaces flash_attn_func (OptFlashAttention2) and the eager einsum
 * attention of transformer_blocks.py:57-74,166-185.
 * q [M][ldq] fp16 (head h at columns h*64..); K,V: [slot][head][T][64] fp16; out [M][ldo] fp16;
 * scratch: ma_attention_scratch_bytes(M, H, max_keys) bytes, zero-initialised once by the caller. */
size_t ma_attention_scratch_bytes(int M, int H, int max_keys);
int ma_attention_f16(const void* q, int ldq, const void* K, const void* V, long T, int H, const int* slots,
                     const int* nkeys, int max_keys, int M, float scale, void* out, int ldo, void* scratch,
                     void* stream);
/* One decode step of a batch: row m = cache slot m, 16 heads.  qkv [M][ldq] fp16 holds q | k | v of the current token
 * (columns 0.., 1024.., 2048..); the k / v rows are appended to the cache at position nkeys[m]-1 and row m attends keys
 * [0, nkeys[m]) -- the same arithmetic as ma_attention_f16, bit for bit, as one persistent pipelined kernel
 * (attention_stream.cu).  This is the flash_attn_func call of OptFlashAttention2 on the decode path plus the cache
 * update of transformers' OPT attention (past_key_value concat).  scratch as for ma_attention_f16 with H = 16. */
int ma_attention_decode_f16(const void* qkv, int ldq, void* K, void* V, long T, const int* nkeys, int max_keys, int M,
                            float scale, void* out, int ldo, void* scratch, void* stream);

/* ---- ShapeOPT decoder (shape_opt.py:188-460 + HF generate) --------------------------------- */

typedef struct {
  int n_layers, vocab, codebook, npos;
  const void* wqkv[MA_MAX_LAYERS]; /* fp16 [3072][1024]: q_proj, k_proj, v_proj rows stacked */
  const void* bqkv[MA_MAX_LAYERS]; /* fp16 [3072] */
  const void* wo[MA_MAX_LAYERS];   /* fp16 [1024][1024] out_proj */
  const void* bo[MA_MAX_LAYERS];
  const void* w1[MA_MAX_LAYERS];   /* fp16 [4096][1024] fc1 */
  const void* b1[MA_MAX_LAYERS];
  const void* w2[MA_MAX_LAYERS];   /* fp16 [1024][4096] fc2 */
  const void* b2[MA_MAX_LAYERS];
  const float* ln1g[MA_MAX_LAYERS]; /* self_attn_layer_norm */
  const float* ln1b[MA_MAX_LAYERS];
  const float* ln2g[MA_MAX_LAYERS]; /* final_layer_norm (per layer) */
  const float* ln2b[MA_MAX_LAYERS];
  const void* lm_head;    /* fp16 [vocab][1024], no bias (shape_opt.py:22) */
  const void* tok_table;  /* fp16 [codebook][1024] = input_layer(quantize_codebooks[0]) (shape_opt.py:243),
                             folded once at load time with ma_linear_f16 */
  const float* extra;     /* fp32 [3][1024]    extra_embeds */
  const float* tok_pos;   /* fp32 [12][1024]   token_embed_positions */
  const float* cond;      /* fp32 [2][1024]    cond_embed */
  const float* pos;       /* fp32 [npos][1024] embed_positions incl. the 2 offset rows */
} ma_decoder_weights;

typedef struct {
  int do_sample;   /* 0: greedy argmax on fp16 logits, lowest index on ties */
  int top_k;       /* 50 in the reference (meshanything.py:156) */
  float top_p;     /* 0.95 (meshanything.py:157) */
  uint64_t seed;
} ma_sampling;

/* One pick of HF's sampling chain on its own (test surface; ma_decode_generate runs the same kernel per step):
 * logits fp16 [B][vocab] -> out_tokens int32 [B].  do_sample = 0: argmax.  Otherwise TopKLogitsWarper(top_k)
 * (every logit >= the k-th largest value survives, ties included) then TopPLogitsWarper(top_p), then one
 * Philox(seed, row, step) uniform through the inverse CDF.  out_support int32 [B][256] (optional): the ids that
 * survived both warpers, by descending logit, -1 padded.  1 <= top_k <= 128. */
int ma_sample_tokens(const void* logits, int B, int vocab, const ma_sampling* sampling, int32_t* out_tokens,
                     int32_t* out_support, void* stream);

size_t ma_kv_cache_bytes(int n_layers, int B, int tmax);
size_t ma_decoder_workspace_bytes(int B, int tmax);

/* transformer.generate(inputs_embeds=prefix, max_new_tokens=..., bos/eos/pad) of
 * meshanything.py:144-162.  prefix fp32 [B][257][1024]; out_ids int32 [B][max_new] (rows that
 * finished are padded with pad_id, HF semantics); out_lens int32 [B] = tokens generated up to and
 * including eos.  kv: ma_kv_cache_bytes, ws: ma_decoder_workspace_bytes (contents undefined on
 * entry).  Optional test hooks: forced_ids int32 [B][max_new] (teacher forcing: fed instead of the
 * pick), logits_out fp16 [max_new][B][vocab].  Enqueues everything on `stream`; polls a pinned flag
 * for early exit but never blocks on the device. */
int ma_decode_generate(const ma_decoder_weights* w, const float* prefix, int B, int tmax, int max_new,
                       const ma_sampling* sampling, int eos_id, int pad_id, void* kv, void* ws, int32_t* out_ids,
                       int32_t* out_lens, const int32_t* forced_ids, void* logits_out, int flags, void* stream);

/* ---- continuous batching over B cache slots (SURVEY.md section 8(f)2; replaces HF generate's "pad finished rows
 * until the longest sequence ends", transformers generation/utils.py _greedy_search/_sample, for a queue of shapes).
 * Same kv / ws buffers and sizes as ma_decode_generate; out_ids int32 [B][max_new] is indexed by slot.
 *   ma_decode_slots_init    every slot free (finished = 1).
 *   ma_decode_slot_prefill  loads `prefix` (fp32 [257][1024]) into `slot`, clears its out_ids row, picks its first
 *                           token; the slot is live from the next step on.
 *   ma_decode_slots_step    n_steps decode steps of all slots; finished slots are frozen (no output, no state change);
 *                           a slot finishes on eos or after max_new tokens.  max_ctx = the largest number of keys any
 *                           live slot attends to at the first of these steps (257 + tokens generated so far), an upper
 *                           bound is fine: it only sizes the attention grid.
 *   ma_decode_slots_poll    copies finished[B] / lens[B] to host memory and waits for the stream (the one
 *                           synchronising call; the scheduler calls it every few dozen steps).
 * Every sequence gets the ids a solo ma_decode_generate would give it (batch-invariant arithmetic). */
int ma_decode_slots_init(int B, int tmax, int pad_id, void* ws, void* stream);
/* Sampling only: the Philox stream of the sequence about to be prefilled into `slot` (e.g. its index in the queue).
 * Draws are keyed by (seed, stream, token index), so shapes that pass through the same slot are independent and a
 * shape's samples do not depend on the slot it lands in.  Call before ma_decode_slot_prefill; default stream 0. */
int ma_decode_slot_stream(int slot, int B, int tmax, int stream_id, void* ws, void* stream);
/* Measurement hook (bench.py, tools/): declares every slot live at cached position `pos` having generated `gen` tokens,
 * last token `tok`, WITHOUT running the steps that lead there -- the KV cache keeps whatever it holds (the caller
 * zero-fills it).  Lets a bounded number of ma_decode_slots_step calls be timed at a chosen context length. */
int ma_decode_slots_seek(int B, int tmax, int pos, int gen, int tok, void* ws, void* stream);
int ma_decode_slot_prefill(const ma_decoder_weights* w, const float* prefix, int slot, int B, int tmax, int max_new,
                           const ma_sampling* sampling, int eos_id, int pad_id, void* kv, void* ws, int32_t* out_ids,
                           void* stream);
int ma_decode_slots_step(const ma_decoder_weights* w, int B, int tmax, int max_new, int n_steps, int max_ctx,
                         const ma_sampling* sampling, int eos_id, int pad_id, void* kv, void* ws, int32_t* out_ids,
                         int flags, void* stream);
int ma_decode_slots_poll(int B, int tmax, void* ws, int32_t* finished_host, int32_t* lens_host, void* stream);

/* flags of ma_decode_generate */
#define MA_GEN_NO_GRAPH 1   /* plain launches instead of a CUDA graph per step */
#define MA_GEN_NO_FAST 2    /* batch-1: use the general batched kernels instead of the fused GEMV path */
#define MA_GEN_NO_PDL 4     /* batch-1 fast path without programmatic dependent launch */
#define MA_GEN_NO_EARLY_EXIT 8
#define MA_GEN_NO_MEGA 16    /* batch-1 greedy: per-phase kernels (decode_fast.cu) instead of the persistent kernel */
#define MA_GEN_TC 64         /* batches: decoder GEMMs on the tensor cores (tcgen05) -- logits within a tolerance of the
                                canonical kernels instead of bit-exact ids; implied by sampling */
#define MA_GEN_TRACE 32      /* persistent kernel records globaltimer stamps of CTA 0 at every phase boundary */

/* Debug read-back (synchronises the device): what = 0 -> int error word of the persistent kernel (non-zero: a
 * hand-off between SMs timed out; value = 1 + the CTA that gave up first), what = 1 -> its uint64 trace stamps,
 * what = 2 -> the per-CTA stamps.  A time-out also makes the kernel stop emitting tokens and set out_lens[0] = -1. */
int ma_decoder_debug(void* ws, int B, int tmax, int what, void* host_out, int nbytes);
/* Test hook of the persistent kernel: bound of every in-kernel wait in ns (0 = keep; default: seconds) and fault
 * injection (fault = c + 1: CTA c withholds its out_proj rows from the third token on, so the hand-off times out). */
void ma_mega_set_debug(unsigned long long timeout_ns, int fault);


/* Same contract as ma_linear_f16 on the tcgen05 tensor cores (TMA-fed, accumulator in TMEM): fp16 in, fp32
 * accumulate in the hardware's order (NOT the canonical order: results agree with ma_linear_f16 to fp32 rounding,
 * not bit for bit).  M >= 64, N % 128 == 0, K % 64 == 0.  Used by ma_encoder_forward / ma_detokenize. */
int ma_linear_tc_f16(const void* W, const void* bias, const void* x, int ldx, void* y, int ldy, int M, int N, int K,
                     int epilogue, void* stream);
/* The same contract for FEW rows (1 <= M <= 128; any N; K % 64 == 0): swap-AB weight-streaming tcgen05 GEMM with the K
 * dimension split across CTAs and a deterministic last-CTA reduction (gemm_ws.cu).  Replaces the cuBLAS GEMMs of HF's
 * OPTDecoderLayer for a decode step of a batch (shape_opt.py:403-410).  scratch: ma_linear_ws_scratch_bytes() bytes,
 * zero-filled once by the caller.  Hardware accumulation order: compared under a tolerance. */
size_t ma_linear_ws_scratch_bytes(void);
/* 1 (default): the K slices of a row block are a thread-block cluster and are added over distributed shared memory;
 * 0: partial tiles through L2 and an atomic ticket (kept for A/B timing).  Both add the slices in slice order. */
void ma_linear_ws_set_mode(int cluster);
int ma_linear_ws_f16(const void* W, const void* bias, const void* x, int ldx, void* y, int ldy, int M, int N, int K,
                     int epilogue, void* scratch, void* stream);
/* 0: canonical CUDA-core kernels everywhere; 1: encoder / detokenizer GEMMs on the tensor cores; 2: their attention
 * too (ma_attention_tc_f16).  Returns the previous setting. */
int ma_set_tensor_cores(int enable);
/* Linear calls of ma_encoder_forward / ma_detokenize since load: how many ran on tcgen05 and how many fell back to the
 * canonical CUDA-core kernel because their shape cannot be tiled (M < 64, N % 128 != 0). */
void ma_tensor_core_linear_counts(unsigned long long* on_tcgen05, unsigned long long* canonical_fallback);

/* Dense non-causal attention on the tensor cores (tcgen05 flash attention; replaces F.scaled_dot_product_attention of
 * transformer_blocks.py:57-74,166-185 and BERT's attention in meshanything.py:62-64).  q fp16 [n_slots*rows_per_slot][ldq]
 * (head h at columns 64h..64h+63), K fp16 [n_slots][H][T][64], Vt fp16 [n_slots][H][64][Tpad] = V transposed, zero for
 * keys >= nkeys, Tpad a multiple of 64 and >= nkeys rounded up to 128; every query of a slot sees the first nkeys
 * keys of that slot.  out fp16 [rows][ldo].  Hardware accumulation order: compared under a tolerance. */
int ma_attention_tc_f16(const void* q, int ldq, const void* K, const void* Vt, long T, long Tpad, int H,
                        int rows_per_slot, int n_slots, int nkeys, float scale, void* out, int ldo, void* stream);
/* Vt[((slot*H + h)*64 + d)*Tpad + t] = src[(slot*n + t)*ld + col0 + h*head_stride + d] for t < n, 0 for n <= t < Tpad */
int ma_transpose_heads_f16(const void* src, int ld, int col0, int head_stride, int H, int n, long Tpad, int n_slots,
                           void* dst, void* stream);

/* ---- Michelangelo point-cloud encoder (a1-a8) ----------------------------------------------- */

typedef struct { /* ResidualAttentionBlock, transformer_blocks.py:77-115 (qkv_bias: false) */
  const void* c_qkv_w;            /* fp16 [2304][768] */
  const void *c_proj_w, *c_proj_b; /* fp16 [768][768], [768] */
  const float *ln1_g, *ln1_b, *ln2_g, *ln2_b;
  const void *fc_w, *fc_b;        /* fp16 [3072][768], [3072] */
  const void *proj_w, *proj_b;    /* fp16 [768][3072], [768] */
} ma_miche_block;

typedef struct {
  const void *input_proj_w, *input_proj_b; /* fp16 [768][256] (54 input columns, zero padded), [768] */
  const float* query;                      /* fp32 [257][768]  sal_perceiver.py:42 */
  const void *cq_w, *ckv_w;                /* fp16 [768][768], [1536][768]  (no bias) */
  const void *cproj_w, *cproj_b;
  const float *ln1_g, *ln1_b, *ln2_g, *ln2_b, *ln3_g, *ln3_b;
  const void *fc_w, *fc_b, *proj_w, *proj_b;
  ma_miche_block enc[8];                   /* encoder.self_attn.resblocks */
  const float *lnpost_g, *lnpost_b;
  const void *pre_kl_w, *pre_kl_b;         /* fp16 [128][768] */
  const void *post_kl_w, *post_kl_b;       /* fp16 [768][256] (64 input columns, zero padded) */
  ma_miche_block dec[16];                  /* transformer.resblocks */
  const void *cond_head_w, *cond_head_b;   /* fp16 [1024][768]   meshanything.py:120 */
  const void *cond_w, *cond_b;             /* fp16 [1024][1536]  meshanything.py:121 */
} ma_encoder_weights;

size_t ma_encoder_workspace_bytes(int B);

/* point_encoder.encode_latents + MeshAnything.process_point_feature (meshanything.py:137-138):
 * pc_normal fp16 [B][4096][6] -> point_feature fp32 [B][257][768], prefix fp32 [B][257][1024]. */
int ma_encoder_forward(const ma_encoder_weights* w, const void* pc_normal, int B, float* point_feature, float* prefix,
                       void* ws, void* stream);

/* ---- VQ detokenizer (a17-a18) ------------------------------------------------------------------ */

typedef struct { /* BERT layer in optimum-BetterTransformer spelling */
  const void *in_w, *in_b;     /* fp16 [2304][768], [2304] */
  const void *out_w, *out_b;   /* fp16 [768][768], [768] */
  const void *l1_w, *l1_b;     /* fp16 [3072][768], [3072] */
  const void *l2_w, *l2_b;     /* fp16 [768][3072], [768] */
  const float *n1_g, *n1_b, *n2_g, *n2_b;
} ma_bert_layer;

typedef struct {
  int n_layers;
  ma_bert_layer layer[8];
  const float* pos_embedding;  /* fp32 [18000][768] */
  const float* point_pe;       /* fp32 [257][768] */
  const float *ln_g, *ln_b, *pln_g, *pln_b;
  const void *cond_w, *cond_b, *cond_head_w, *cond_head_b; /* fp16 [768][768] */
  const void *down_w, *down_b; /* fp16 [768][3072] project_down_codebook */
  const void *coor_w, *coor_b; /* fp16 [1152][768] to_coor_logits.0 */
  const float* codebook;       /* fp32 [8192][1024] quantize_codebooks[0] */
} ma_tokenizer_weights;

size_t ma_detokenize_workspace_bytes(int B, int F);

/* ids post-processing + get_codes + NoiseResistantDecoder (meshanything.py:163-174): gen_ids int32
 * [B][max_new] = raw generate() output, max_new = 9F+2; -> out_xyz fp32 [B][F][3][3] (NaN rows = absent
 * faces); ids_out optional int32 [B][9F] = the post-processed ids (-1 = absent). */
int ma_detokenize(const ma_tokenizer_weights* w, const int32_t* gen_ids, int max_new, int B, int F,
                  const float* point_feature, float* out_xyz, int32_t* ids_out, void* ws, void* stream);

/* ---- mesh -> point cloud (SURVEY.md section 8(f)3) ------------------------------------------------------------
 * Area-weighted surface sampling with face normals: trimesh.Trimesh.sample(count, return_index=True) +
 * mesh.face_normals[idx] of /root/reference/mesh_to_pc.py:49-53.  vertices fp32 [V][3], faces int32 [F][3] ->
 * out_pc_normal fp16 [n_samples][6] (point | unit face normal), out_face_idx int32 [n_samples] (optional).  Philox
 * stream keyed by (seed, sample).  ws: ma_sample_surface_workspace_bytes(F) bytes. */
size_t ma_sample_surface_workspace_bytes(int n_faces);
int ma_sample_surface(const float* vertices, const int32_t* faces, int n_faces, int n_samples, unsigned long long seed,
                      void* out_pc_normal, int32_t* out_face_idx, void* ws, void* stream);

/* ---- watertight remesh (`--mc`): unsigned distance field + marching cubes -------------------------------------
 * Grid of size^3 nodes (size in 32..256; the reference uses 2^7), spacing h = 2 / size, node (i, j, k) at
 * (-1 + i h, -1 + j h, -1 + k h); fields are fp32 [size][size][size] indexed [i][j][k], k fastest.
 *
 * ma_mesh_udf: vertices fp32 [V][3] (normalised to +-0.9), faces int32 [F][3] (indices in [0, V), not checked here) ->
 * out_field[n] = min(d(n), 2h), d the exact distance from node n to the nearest triangle; zero-area triangles count by
 * their edges and points.  Bit-identical for any order of the faces.  Needs no workspace. */
int ma_mesh_udf(const float* vertices, const int32_t* faces, int n_faces, int size, float* out_field, void* stream);

/* Marching cubes of `field` at `level` (inside: field < level), one vertex per crossing grid edge, triangles oriented
 * with (v1 - v0) x (v2 - v0) towards increasing field; closed wherever the level set stays inside the grid.
 * ma_marching_cubes_count writes out_counts (device int32 [2]) = (vertices, triangles) and the per-node offsets into ws
 * (ma_marching_cubes_workspace_bytes(size) bytes); ma_marching_cubes_emit, given the same field, level and ws, writes
 * out_vertices fp32 [V][3] = ((index * h) - 1) * inv_scale + (cx, cy, cz) and out_faces int32 [F][3], vertices in
 * order of owning node then axis, triangles in cell order then table order. */
size_t ma_marching_cubes_workspace_bytes(int size);
int ma_marching_cubes_count(const float* field, int size, float level, int32_t* out_counts, void* ws, void* stream);
int ma_marching_cubes_emit(const float* field, int size, float level, float inv_scale, float cx, float cy, float cz,
                           float* out_vertices, int32_t* out_faces, void* ws, void* stream);

/* number of kernels launched by the library since load (bench.py's gpu_launches) */
unsigned long long ma_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif
