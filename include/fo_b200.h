/*
 * fo_b200.h -- C ABI of the B200-native streaming speech encoder + adapter path.
 *
 * The reference (TheDoctor-JI/Freeze-Omni) has no FFI: its boundary for this path is the Python
 * nn.Module surface that models/audioLLM.py and models/utils.py touch (SURVEY.md 8b).  The Python
 * drop-ins in freeze_omni_b200/ keep that surface and bind the entry points below with ctypes.
 * Each entry names the reference interface it replaces (paths relative to the reference root).
 *
 * Conventions
 *   - every function returns 0 on success, <0 on error; fo_last_error() returns the thread-local
 *     message of the last failure.  There is no CPU fallback: without a CUDA device fo_create fails.
 *   - data pointers may be HOST or DEVICE pointers (detected with cudaPointerGetAttributes); host
 *     buffers are copied on `stream` inside the call (pinned host memory keeps this asynchronous).
 *   - all work is enqueued on the caller's stream (cudaStream_t passed as void*); calls on one
 *     context must be serialised by the caller (the reference serialises per pipeline object,
 *     bin/dialog_state_pred.py:279-283).
 *   - floating-point tensors cross the boundary as fp32, row-major, innermost dimension last.
 *   - the session ids of one call must be distinct (a duplicate is FO_ERR_ARG: two rows would advance one session's state).
 */
#ifndef FO_B200_H
#define FO_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FO_ABI_VERSION 6

enum { FO_F32 = 0, FO_BF16 = 1, FO_I16 = 2 };     /* compute dtype / PCM sample type */
enum { FO_OK = 0, FO_ERR_ARG = -1, FO_ERR_CUDA = -2, FO_ERR_STATE = -3, FO_ERR_NOMEM = -4 };

typedef struct fo_ctx fo_ctx;

/* Shipped values in comments (SURVEY.md 2.3).  Mirrors the yaml the reference feeds to
 * speechEncoder.__init__ (models/encoder/encoder.py:46-99) and CNNSubsampling.__init__
 * (models/adapter.py:73-110). */
typedef struct fo_config {
    int32_t feat_dim;          /* 80    encoder-input-dim */
    int32_t d_model;           /* 1024  subsampling-output-dim == transformer-attention-dim */
    int32_t n_heads;           /* 16 */
    int32_t ffn_dim;           /* 4096  transformer-linear-units */
    int32_t n_layers;          /* 24    transformer-num-blocks */
    int32_t chunk_size;        /* 4     transformer-chunk_size (encoder frames) */
    int32_t left_chunks;       /* 16    transformer-left_chunks */
    int32_t input_layer_linear;/* 1     transformer-input-layer == "linear" (0: "none") */
    int32_t pos_max_len;       /* 5000  RelPositionalEncoding max_len (attention.py:78) */
    int32_t llm_dim;           /* 3584  llm_embed_dim */
    int32_t adapter_kernel;    /* 5 */
    int32_t adapter_gelu;      /* 1     activation_func == "gelu" (0: relu) */
    int32_t has_encoder;       /* build the encoder part */
    int32_t has_adapter;       /* build the adapter part */
    /* streaming frontend (bin/inference.py:43-56 / models/AudioFeatureGating.py:19-41) */
    int32_t sample_rate;       /* 16000 */
    int32_t frame_len;         /* 400 samples */
    int32_t frame_shift;       /* 160 samples */
    int32_t frames_per_chunk;  /* 16 */
    int32_t context_frames;    /* 3 */
    /* capacity */
    int32_t max_sessions;      /* session slots resident in HBM */
    int32_t max_stream_frames; /* largest fbank-frame count of one streaming call (>= context+frames_per_chunk); the encoder
                                * frames per chunk it gives are capped at 8 (35 feature frames), what the streaming attention takes */
    /* positionwise layer: 0 or 1 = PositionwiseFeedForward (models/encoder/attention.py:122-143);
     * k >= 2 = Conv1dLinear with kernel_size k (models/encoder/attention.py:198-266): causal depthwise conv over
     * time (left context carried per session and layer) + 1x1 conv + ReLU + Linear */
    int32_t ffn_conv_kernel;
    /* adapter norm (models/adapter.py:100-103): 0 = LayerNorm(2C, eps 1e-3); 1 = BatchNorm1d(2C, eps 1e-3) in eval mode
     * (running statistics; tensors adapter.bn2.{weight,bias,running_mean,running_var}) */
    int32_t adapter_batchnorm;
    /* adapter module (models/audioLLM.py:159-166): 0 = CNNSubsampling (adapter.py:72-157, the shipped 'subsampling'; when
     * 4 * d_model < llm_dim it has TWO convolutions and two caches, adapter.py:84-96,123-143: tensors adapter.conv1d1 / bn1 /
     * conv1d2 / bn2 (BatchNorm1d + ReLU by construction) / project);
     * 1 = LinearAdapter (adapter.py:59-70): y = Linear(d_model -> llm_dim)(x), no cache, no subsampling (t_out = t),
     * tensors adapter.adpter.{weight,bias};
     * 2 = CNNAdapter (adapter.py:10-57): two causal stride-1 convolutions with BatchNorm1d + ReLU, Linear(4 * d_model -> llm_dim),
     * no cache (zero left context every call), t_out = t */
    int32_t adapter_type;
    /* TransformerLayer options (models/encoder/transformer.py:56-70): post_norm = 1 is transformer-normalize-before: false
     * (LayerNorms after the residual adds, :89-90,97-98,117-118,127-128, and no after_norm, :232-233); concat_after = 1 replaces
     * x + att by x + concat_linear(cat(layer input, att)) (:85-87,108-113; tensor enc.1.encoders.N.concat_linear.{weight,bias}) */
    int32_t post_norm;
    int32_t concat_after;
    /* 1: the positionwise layer is MultiLayeredConv1d (models/encoder/attention.py:145-196, transformer-positionwise-layer-type
     * "conv1d"): Conv1d(d_model -> ffn_dim, k, padding (k-1)/2) -> ReLU -> Conv1d(ffn_dim -> d_model, k, padding (k-1)/2) over
     * time with k = ffn_conv_kernel (odd, 3..9); tensors feed_forward.w_1.weight (ffn_dim, d_model, k), w_2.weight (d_model,
     * ffn_dim, k).  Full-utterance encode only: the reference module has no infer(), the streaming entries refuse such a context. */
    int32_t ffn_multi_conv;
} fo_config;

typedef struct fo_stats_t {
    int64_t stream_steps;      /* fo_encode_stream / fo_encode_stream_chunks[_v] / fo_stream_step[s_v] calls */
    int64_t session_chunks;    /* sum over steps of sessions x chunks advanced */
    int64_t offline_calls;
    int64_t offline_frames;    /* encoder frames produced offline */
    int64_t kernel_launches;   /* kernels of this library enqueued so far (graph replays count their nodes) */
    int64_t sessions_in_use;
    int64_t device_bytes;      /* HBM held by the context */
    int64_t graph_replays;
    /* 16-bit contexts stage GEMM outputs that feed the tensor cores as IEEE fp16 (weights are bf16-rounded); a value beyond
     * +-65504 is clamped AND counted here.  Non-zero means the model's activations left the fp16 range: results are no longer
     * within the parity bound; run the context in FO_F32.  (The reference's autocast bf16 has fp32 range.) */
    int64_t act_saturations;
} fo_stats_t;

int         fo_abi_version(void);
const char* fo_last_error(void);

/* ---- lifetime: replaces speechEncoder(...) / CNNSubsampling(...) construction + .to(device) ---- */
int fo_create(const fo_config* cfg, int device, int dtype, fo_ctx** out);
/* fo_create on one group of the device's SMs, so that several contexts share a GPU without waiting on each other's grids
 * (a user and a system encoder, an LLM beside them).  The device's SMs are split into sm_split equal groups of a multiple of
 * 8 SMs (the granularity of CUDA green contexts: at least 8, in multiples of 8; 148 SMs split 2 ways give 2 x 72); the context
 * runs on group sm_group.  The split is made once per process and device: contexts created with the same sm_split and
 * different groups run on disjoint SMs.  Every grid, GEMM plan and the layer stack are sized to the group's SMs
 * (fo_get_option "sm_count").  Entry points keep their stream contract: the work of a call runs on a stream of the group,
 * after what the caller enqueued on `stream` before the call and before what it enqueues there after it.  Refused, with
 * nothing allocated: sm_split < 1, sm_group outside [0, sm_split), groups below 8 SMs, a driver without green contexts
 * (CUDA 12.4+).  There is no fall-back to the whole device.
 * Shared by every context of the process: the fbank twiddle table (contexts whose frame lengths need different FFT sizes
 * must not run their frontends at the same time) and the counters of fo_stats.kernel_launches / options "tc_launches",
 * "tc_persist_launches" (totals over all contexts and threads). */
int fo_create_on_sms(const fo_config* cfg, int device, int dtype, int sm_split, int sm_group, fo_ctx** out);
int fo_destroy(fo_ctx* ctx);

/* ---- weights: replaces load_state_dict (models/utils.py:11-20).  `name` is the reference's
 * state-dict key ("enc.1.encoders.0.self_attn.linear_q.weight", "conv1d2.weight", ...; adapter keys
 * are prefixed "adapter."), plus the host-built constants "fbank.window" (frame_len),
 * "fbank.mel" (feat_dim x fft/2+1) and "pos.table" (pos_max_len x d_model).  data is fp32. */
int fo_load_tensor(fo_ctx* ctx, const char* name, const void* data, const int64_t* shape, int ndim);
int fo_finalize_weights(fo_ctx* ctx);   /* checks completeness, repacks into kernel layouts */

/* ---- sessions: replace the per-identity cache objects the service keeps
 * (bin/dialog_state_pred.py:221-232): encoder KV list, adapter cnn cache, pe_index, fbank carry. */
int fo_session_alloc(fo_ctx* ctx, int n, int32_t* ids_out);     /* fresh == buffer [None]*L, cache None, pe_index 0 */
int fo_session_reset(fo_ctx* ctx, int n, const int32_t* ids);
int fo_session_free(fo_ctx* ctx, int n, const int32_t* ids);
/* scalar state: frames appended so far (cache_len = min(n_frames, chunk*left)) and pe_index */
int fo_session_get_state(fo_ctx* ctx, int32_t id, int64_t* n_frames, int64_t* pe_index);
int fo_session_set_pe_index(fo_ctx* ctx, int n, const int32_t* ids, const int64_t* pe_index);
/* reference layout of one layer's cache (models/encoder/attention.py:415-428): K,V (H, cache_len, d_k) */
int fo_session_export_kv(fo_ctx* ctx, int32_t id, int layer, float* K, float* V, int32_t* cache_len);
int fo_session_import_kv(fo_ctx* ctx, int32_t id, int layer, const float* K, const float* V, int32_t cache_len);
int fo_session_set_frames(fo_ctx* ctx, int32_t id, int64_t n_frames);
/* adapter cache in the reference layout (models/adapter.py:141-143): (d_model, kernel-1); valid=0 means None */
int fo_session_export_adapter_cache(fo_ctx* ctx, int32_t id, float* cache, int32_t* valid);
int fo_session_import_adapter_cache(fo_ctx* ctx, int32_t id, const float* cache, int32_t valid);

/* entry `which` of the reference's cache list for the two-conv CNNSubsampling (adapter.py:123-143): which = 0 is the second
 * conv's left context (2 * d_model, kernel-1), which = 1 the first conv's (d_model, kernel-1).  Single-conv: which = 0 only. */
int fo_session_export_adapter_cache_n(fo_ctx* ctx, int32_t id, int which, float* cache, int32_t* valid);
int fo_session_import_adapter_cache_n(fo_ctx* ctx, int32_t id, int which, const float* cache, int32_t valid);

/* Conv1dLinear left context of one layer in the reference layout (models/encoder/attention.py:221,258): (d_model, k-1) */
int fo_session_export_ffn_cache(fo_ctx* ctx, int32_t id, int layer, float* cache);

/* ---- session snapshots: the whole state of n sessions -- KV window of every layer, pe_index, adapter caches, Conv1dLinear
 * context, fbank sample carry, feature ring -- as n consecutive records of `bytes` each (one record can be sliced out), so that
 * a conversation moves to another slot, context or GPU and continues bit for bit as if it had never moved.  The format
 * (versioned; layout in fo_api.cu) carries a fingerprint of every setting that fixes the state's shape and meaning; capacities
 * (max_sessions, max_stream_frames) and options are not in it, so a record moves between contexts that differ in them.
 * Restoring into a context with other weights of the same shapes is not detected: the caller pairs records with their model.
 * buf is host or device memory (a device buffer must be on the context's device).  Both calls are ordered on `stream` after
 * every step enqueued there before (fo_stream_step_async included) and never synchronise the device; host buffers go through
 * a staging buffer of their own, a few records at a time (a pinned host buffer is complete once `stream` reaches the call).
 * Neither grows a step workspace: a snapshot between two graph-replayed steps does not force a re-capture. */
int fo_session_snapshot_bytes(fo_ctx* ctx, int64_t* bytes);
/* records of sessions ids[0..n) into buf (n x bytes) */
int fo_session_save(fo_ctx* ctx, const int32_t* ids, int n, void* buf, void* stream);
/* records of buf into the allocated slots ids[0..n) (fo_session_alloc; restoring into a second slot forks a session).  Every
 * header is checked first -- for a device buf one small read-back and a sync of `stream`: a bad magic, version, record size or
 * fingerprint field in any record is FO_ERR_ARG naming the first mismatching field, and none of the n slots is touched. */
int fo_session_restore(fo_ctx* ctx, const int32_t* ids, int n, const void* buf, void* stream);

/* ---- frontend: replaces audioEncoderProcessor.process (bin/inference.py:71-80) /
 * AudioFeatureGating._extract_fbank (models/AudioFeatureGating.py:54-75).
 * pcm: (n, frame_shift*frames_per_chunk) samples, FO_F32 or FO_I16; value used = sample * scale.
 * feats_out (n, context+frames_per_chunk, feat_dim) may be NULL (the block stays in the session). */
int fo_fbank_stream(fo_ctx* ctx, const int32_t* ids, int n, const void* pcm, int pcm_dtype, float scale,
                    float* feats_out, void* stream);
/* replaces torchaudio.compliance.kaldi.fbank on whole signals (call sites as above).
 * pcm (B, n_samples); out (B, 1 + (n_samples-frame_len)/frame_shift, feat_dim). */
int fo_fbank_offline(fo_ctx* ctx, const void* pcm, int pcm_dtype, int B, int64_t n_samples, float scale,
                     float* out, void* stream);
/* torchaudio.compliance.kaldi.fbank on B signals of different lengths packed end to end (a corpus without padding).
 * pcm: sum n_samples[i] samples, FO_F32 or FO_I16, host or device; value used = sample * scale.  n_samples: HOST, B int64.
 * Utterance i gets m_i = 1 + (n_samples[i] - frame_len) / frame_shift frames (snip_edges: trailing samples that fill no frame
 * are dropped); out (sum m_i, feat_dim) in utterance order, every row bit-identical to fo_fbank_offline of that utterance
 * alone.  FO_ERR_ARG, with nothing enqueued, for B <= 0, an n_samples[i] < frame_len (naming i) or a bad pcm_dtype. */
int fo_fbank_offline_packed(fo_ctx* ctx, const void* pcm, int pcm_dtype, const int64_t* n_samples, int B, float scale,
                            float* out, void* stream);

/* ---- streaming chunk: replaces speechEncoder.infer (models/encoder/encoder.py:149-155) followed by
 * CNNSubsampling.forward(cache=..., return_cache=True) (models/adapter.py:112-157), i.e. the two
 * starred calls of AudioLLM.recognize (models/audioLLM.py:380-387), for n sessions at once.
 * feats (n, t_in, feat_dim) or NULL = the block left in the sessions by fo_fbank_stream.
 * enc_out (n, t, d_model), adapter_out (n, t_out, llm_dim): either may be NULL.
 * t = ((t_in-1)/2-1)/2; t_out = (t + kernel-1 - kernel)/2 + 1.
 * Every streaming entry refuses (FO_ERR_ARG, nothing enqueued, no session advanced) a context with chunk_size <= 0 (full
 * attention: fo_encode_offline only), t beyond the context's max_t (<= 8), and window + t > 128 keys (e.g. left_chunks 32). */
int fo_encode_stream(fo_ctx* ctx, const int32_t* ids, int n, const float* feats, int t_in,
                     float* enc_out, float* adapter_out, void* stream);
/* k consecutive chunks per session in one call, equal to k successive fo_encode_stream calls of one chunk each
 * (speechEncoder.infer + CNNSubsampling.forward(cache) k times, models/audioLLM.py:380-387): speech-onset replay and
 * catch-up encoding stream the weights once for n*k*t token rows instead of k times.
 * feats (n, k, t_in, feat_dim), required: every chunk block carries its own context frames, as fo_fbank_stream returns them.
 * enc_out (n, k, t, d_model), adapter_out (n, k, t_out, llm_dim): either may be NULL.  A session's state advances by k chunks.
 * window + k*t keys must fit the multi-chunk attention (128: k <= 16 with the shipped chunking); beyond that FO_ERR_ARG
 * names the largest k.  An armed hand-off (fo_handoff_arm) applies when armed for n*k blocks: block i*k + j is chunk j of
 * session i (onset flag, embedding rows, mask row and row_start per block).  Counts as one stream step and n*k session chunks. */
int fo_encode_stream_chunks(fo_ctx* ctx, const int32_t* ids, int n, int k, const float* feats, int t_in,
                            float* enc_out, float* adapter_out, void* stream);
/* fo_encode_stream_chunks with a chunk count per session: session ids[i] advances by chunks[i] >= 1 consecutive chunks.
 * feats (B, t_in, feat_dim) with B = sum(chunks), blocks in (session, chunk) order: session i's blocks are
 * [off_i, off_i + chunks[i]), off_i = chunks[0] + ... + chunks[i-1].  enc_out (B, t, d_model), adapter_out (B, t_out, llm_dim),
 * same block order; either may be NULL.  Equal to chunks[i] successive single-chunk calls per session.
 * An armed hand-off applies when armed for B blocks (block off_i + j is chunk j of session i).
 * FO_ERR_ARG, with nothing enqueued, when a count is < 1 or window + chunks[i] * t exceeds the 128 keys of the streaming
 * attention.  One stream step, sum(chunks) session chunks. */
int fo_encode_stream_chunks_v(fo_ctx* ctx, const int32_t* ids, const int32_t* chunks, int n, const float* feats, int t_in,
                              float* enc_out, float* adapter_out, void* stream);
/* fbank + encode in one call (one captured graph): PCM in, embeddings out */
int fo_stream_step(fo_ctx* ctx, const int32_t* ids, int n, const void* pcm, int pcm_dtype, float scale,
                   float* enc_out, float* adapter_out, void* stream);
/* recorded audio of any length: session ids[i] takes chunks[i] >= 1 consecutive chunks of PCM, with the results and the session
 * state afterwards (KV ring, n_frames, pe_index, adapter caches, Conv1dLinear context, fbank sample carry, feature ring) of
 * chunks[i] successive fo_stream_step calls.  pcm (B, frame_shift * frames_per_chunk) samples, B = sum(chunks), blocks in
 * (session, chunk) order as in fo_encode_stream_chunks_v; FO_F32 or FO_I16, value used = sample * scale.  enc_out (B, t, d_model),
 * adapter_out (B, t_out, llm_dim), same block order; either may be NULL.  No cap on the counts: the call runs in passes of a
 * bounded number of blocks (option "steps_pass_blocks"), so the device memory it adds does not grow with the recording.
 * An armed hand-off (fo_handoff_arm) applies when armed for B blocks: block off_i + j is chunk j of session i, as in
 * fo_encode_stream_chunks_v, and gets its onset flag, its fp16 rows [prefix_len, prefix_len + t_out) -- bit for bit the fp32
 * adapter rows the call returns without the arm, rounded to fp16 (clamped to +-65504 and counted in act_saturations) --, its
 * mask row and its row_start; adapter_out must then be NULL, enc_out still works.
 * FO_ERR_ARG, with nothing enqueued and no session touched: the geometry rules of every streaming entry, a count < 1, a
 * duplicate or unallocated id, a MultiLayeredConv1d context, and, while a hand-off is armed, an arm for another block count,
 * adapter_out given or too few rows per block.  Every refusal leaves an armed hand-off armed for the next call.
 * Ordered after outstanding fo_stream_step_async steps.  One stream step, sum(chunks) session chunks. */
int fo_stream_steps_v(fo_ctx* ctx, const int32_t* ids, const int32_t* chunks, int n, const void* pcm, int pcm_dtype,
                      float scale, float* enc_out, float* adapter_out, void* stream);
/* the two halves of fo_stream_steps_v, for callers that choose which blocks reach the encoder (a VAD-gated service replaying
 * a recorded conversation: StreamScheduler.replay).  fo_fbank_stream_v: session ids[i] takes chunks[i] >= 1 consecutive chunks of
 * PCM, laid out as in fo_stream_steps_v; feats_out (B, context + frames_per_chunk, feat_dim), B = sum(chunks), same block order,
 * every block with its context frames; host or device, or NULL.  Features, sample carry and feature ring afterwards are
 * bit-identical to chunks[i] successive fo_fbank_stream calls.  Needs a frontend only; no session's encoder state moves.  It runs
 * no adapter, so an armed hand-off is neither applied nor consumed.
 * FO_ERR_ARG, with nothing enqueued: a count < 1, a duplicate or unallocated id, a bad pcm_dtype. */
int fo_fbank_stream_v(fo_ctx* ctx, const int32_t* ids, const int32_t* chunks, int n, const void* pcm, int pcm_dtype, float scale,
                      float* feats_out, void* stream);
/* fo_stream_steps_v from features: feats (B, t_in, feat_dim), B = sum(chunks), in (session, chunk) order, every block with its
 * own context frames (as fo_fbank_stream_v returns them); no cap on the counts, the same passes, results, armed hand-off and
 * refusals as fo_stream_steps_v.  On the features fo_fbank_stream_v produced it is bit-identical to fo_stream_steps_v of that
 * PCM.  One stream step, sum(chunks) session chunks. */
int fo_encode_stream_steps_v(fo_ctx* ctx, const int32_t* ids, const int32_t* chunks, int n, const float* feats, int t_in,
                             float* enc_out, float* adapter_out, void* stream);
/* pipelined form for HOST buffers (a server loop that already holds the next chunk; the reference runs this loop one chunk
 * and one session at a time, bin/dialog_state_pred.py:793-814 -> models/audioLLM.py:380-387): returns once the step is enqueued.
 * The PCM upload and the read-back of enc_out / adapter_out run on two internal copy streams with double-buffered staging,
 * so the copies of step i overlap the kernels of step i+1; the outputs of a step are valid after fo_stream_wait(ticket).
 * At most two steps may be outstanding; the host buffers of a step must stay untouched until its wait returns. */
int fo_stream_step_async(fo_ctx* ctx, const int32_t* ids, int n, const void* pcm, int pcm_dtype, float scale,
                         float* enc_out, float* adapter_out, void* stream, int64_t* ticket);
int fo_stream_wait(fo_ctx* ctx, int64_t ticket);
/* the same with the LLM hand-off fused into the adapter projection: replaces
 *   inputs_embeds = torch.cat((chat_prefix_embeds, inputs_embeds), 1) ... inputs_embeds.half()   (models/audioLLM.py:404-411).
 * embeds_f16 is a DEVICE buffer (n, rows_per_session, llm_dim) of IEEE fp16 that the caller pre-fills (chat prefix);
 * the t_out adapter rows of session i are written to rows [row_offset, row_offset + t_out) of its block, nothing else
 * is touched.  bf16 contexts only.  enc_out may be NULL. */
int fo_stream_step_embeds(fo_ctx* ctx, const int32_t* ids, int n, const void* pcm, int pcm_dtype, float scale,
                          float* enc_out, void* embeds_f16, int64_t rows_per_session, int64_t row_offset, void* stream);

/* The hand-off with the status-dependent chat prefix and the attention mask, i.e. all of
 *   if status == 'ipu_sl': inputs_embeds = cat(chat_prefix_embeds, inputs_embeds); attention_mask = cat(chat_prefix_mask, attention_mask)
 *   inputs_embeds.half()                                                                          (models/audioLLM.py:383-411)
 * Arms the NEXT streaming call of n blocks (its adapter_out must be NULL): fo_encode_stream / fo_stream_step (one block per
 * session), fo_encode_stream_chunks[_v], or the recording entries fo_stream_steps_v / fo_encode_stream_steps_v (any n: a block
 * per session chunk, however long the recording).  The t_out adapter rows of block i are written as fp16 to rows
 * [prefix_len, prefix_len + t_out) of block i of embeds_f16 (n, rows_per_session, llm_dim), whose rows [0, prefix_len) the caller
 * filled once with the chat-prefix embeddings.  onset (HOST, n bytes): 1 where the
 * block's status is 'ipu_sl'.  attn_mask (DEVICE, n x rows_per_session bytes) row i becomes [prefix_mask | 1 x t_out | 0 ..] for an
 * onset block and [0 x prefix_len | 1 x t_out | 0 ..] otherwise (prefix_mask: DEVICE, prefix_len bytes, NULL = all ones);
 * row_start (DEVICE, n) = 0 / prefix_len.  The LLM input of block i is rows [row_start[i], prefix_len + t_out) of its block,
 * with the same slice of attn_mask (the caller prepends the past-KV mask, audioLLM.py:418-420).  bf16 contexts only.
 * fo_encode_stream & co. consume the arm whatever their outcome; the recording entries refuse a call whose block count differs,
 * or that passes adapter_out, and leave the arm in place (fo_fbank_stream_v ignores it). */
int fo_handoff_arm(fo_ctx* ctx, int n, void* embeds_f16, int64_t rows_per_session, int64_t prefix_len, const uint8_t* onset,
                   const uint8_t* prefix_mask, uint8_t* attn_mask, int32_t* row_start);

/* ---- full utterance: replaces speechEncoder.forward (models/encoder/encoder.py:104-147) and
 * CNNSubsampling.forward(cache=None).  feats (B, T, feat_dim), ilens (B) int32 valid lengths.
 * chunk<=0 means full attention; left<0 means unlimited left context (models/masks.py:50-56,110-122).
 * enc_out (B, T', d_model), mask_out (B, T') uint8, adapter_out (B, T'', llm_dim),
 * adapter_mask_out (B, T'') uint8; any output may be NULL. */
int fo_encode_offline(fo_ctx* ctx, const float* feats, const int32_t* ilens, int B, int T, int chunk, int left,
                      float* enc_out, uint8_t* mask_out, float* adapter_out, uint8_t* adapter_mask_out,
                      void* stream);

/* ---- full utterances of different lengths packed end to end, no padding rows: utterance i (T_i >= 7 feature frames) gets
 * exactly the rows speechEncoder.forward + CNNSubsampling.forward(cache=None) (or the configured adapter) return for it alone.
 * feats (sum T_i, feat_dim), lens (B) int32 T_i; enc_out (sum T'_i, d_model) with T'_i = ((T_i - 1)/2 - 1)/2, adapter_out
 * (sum T''_i, llm_dim) with T''_i = (T'_i - 1)/2 + 1 for CNNSubsampling and T'_i for CNNAdapter / LinearAdapter, both in
 * utterance order, every row valid; either may be NULL.  chunk / left as for fo_encode_offline.  FO_ERR_ARG, with nothing
 * enqueued, for B <= 0, a T_i < 7 or a T'_i past pos_max_len. */
int fo_encode_offline_packed(fo_ctx* ctx, const float* feats, const int32_t* lens, int B, int chunk, int left,
                             float* enc_out, float* adapter_out, void* stream);
/* PCM -> embeddings for utterances of different lengths packed end to end: torchaudio.compliance.kaldi.fbank +
 * speechEncoder.forward (models/encoder/encoder.py:104-147) + the configured adapter per utterance, in one call.  pcm and
 * n_samples as in fo_fbank_offline_packed; enc_out / adapter_out / chunk / left as in fo_encode_offline_packed for the frame
 * counts m_i; feats_out (sum m_i, feat_dim) receives the features of fo_fbank_offline_packed.  Any output may be NULL; host or
 * device.  The fbank writes each utterance's frames straight onto the packed encoder's feature grid.
 * Passes: utterance i takes ceil(m_i / 4) * 4 grid frames, and the call runs over consecutive utterances in call order, a pass
 * taking them while their grid frames fit the option "packed_pass_frames" (default: a 10 GiB workspace budget; never more than
 * the conv2 GEMM of one pass takes; fo_get_option returns the frames in force); an utterance larger than that runs in a pass
 * of its own.  So the device memory the call adds
 * follows the budget, not the corpus.  Host PCM is uploaded one pass at a time, host outputs copied back per pass.  Each pass's
 * rows are bit-identical to fo_fbank_offline per utterance followed by fo_encode_offline_packed over that pass's utterances.
 * FO_ERR_ARG, with nothing enqueued, for a context without a finalized encoder, adapter_out without an adapter, B <= 0, a bad
 * pcm_dtype, an m_i < 7 or a T'_i past pos_max_len (naming the utterance; all are checked before the first pass).
 * Counts as one offline call. */
int fo_encode_offline_packed_pcm(fo_ctx* ctx, const void* pcm, int pcm_dtype, const int64_t* n_samples, int B, float scale,
                                 int chunk, int left, float* enc_out, float* adapter_out, float* feats_out, void* stream);

/* ---- stateless adapter: replaces CNNSubsampling.forward (models/adapter.py:112-157) when the
 * caller owns the cache tensor.  x (B, T, d_model); mask (B, T) uint8 or NULL (all valid);
 * cache_in (B, d_model, kernel-1) or NULL (left zero pad); cache_out same shape or NULL;
 * y (B, (T-1)/2+1, llm_dim). */
int fo_adapter_forward(fo_ctx* ctx, const float* x, const uint8_t* mask, int B, int T,
                       const float* cache_in, float* cache_out, float* y, void* stream);
/* the same for adapters with two cache entries (two-conv CNNSubsampling): cache0 (B, 2 * d_model, kernel-1), cache1
 * (B, d_model, kernel-1) in the order of the reference's list; CNNAdapter / LinearAdapter take no caches (all NULL);
 * y (B, t_out, llm_dim) with t_out = T for CNNAdapter / LinearAdapter. */
int fo_adapter_forward2(fo_ctx* ctx, const float* x, const uint8_t* mask, int B, int T, const float* cache0_in,
                        const float* cache1_in, float* cache0_out, float* cache1_out, float* y, void* stream);

/* ---- introspection / tuning ---- */
int fo_stats(fo_ctx* ctx, fo_stats_t* out);
/* options (value = default):
 *   "gemm_backend" 0 = SIMT FFMA, 1 = tcgen05 (bf16 contexts; their default)      "use_graph" 1: CUDA-graph replay of the streaming step
 *   "pdl" 1: programmatic dependent launch along the kernel chain                   "l2_prefetch" 0: next-kernel L2 prefetch, bit0 weights, bit1 KV rings
 *   "defer_reduce" 1: split-K GEMMs of the residual stream leave the reduction to the LayerNorm that follows
 *   "tc_persist" 1: persistent tile loop for fat short-K GEMMs (offline path)       "fuse_ln" 0: LayerNorm inside the residual GEMM's epilogue
 *   "session_groups" 1 (..4): layer kernels of session groups on parallel streams
 *   "stack_rows" 8 (0..16): streaming steps of up to this many token rows (sessions x encoder frames per call) run all
 *       transformer layers in ONE cooperative launch (csrc/fo_stack.cu; bf16 contexts, pre-norm linear-FFN layers) instead of
 *       the per-kernel chain; the first such step builds the kernel's row-padded copy of the layer matrices (+ 2 x 12 D^2 bytes
 *       per layer, 604 MB for the shipped model).  0 = always the chain.
 *   "steps_pass_blocks" 0: blocks (session chunks) per pass of fo_stream_steps_v, fo_fbank_stream_v and
 *       fo_encode_stream_steps_v; 0 = as many as 1 GiB of workspace holds (720 blocks of the shipped model in bf16)
 *   "profile_gemm" 0/1, "debug_skip" (timing attribution), "tc_swap"/"tc_bn"/"tc_split" (-1 = cost model): development
 * get-only: "tc_launches", "tc_persist_launches", "stack_launches", "ring_cap", "max_t", "profile_gemm_us", "profile_gemm_count",
 *   "steps_pass_blocks_in_use" (the blocks per pass "steps_pass_blocks" gives at the context's chunking), "sm_count" (the SMs
 *   of the context's group, fo_create_on_sms, or of the device).
 * Development environment variables read once per process: FO_TC_OCC, FO_TC_KB, FO_TC_KBD, FO_TC_SMAX, FO_TC_CAP, FO_TC_SKINNY (tile
 * plan of the skinny GEMMs), FO_PDL_MIN, FO_PERSIST_DBG, FO_TC_TRACE. */
int fo_set_option(fo_ctx* ctx, const char* name, int64_t value);
int fo_get_option(fo_ctx* ctx, const char* name, int64_t* value);
/* per-shape totals of the GEMM launches timed while option "profile_gemm" was 1: text lines "M N K launches microseconds"
 * (M = GEMM rows incl. the padding rows of the implicit-GEMM convolutions). */
int fo_profile_dump(fo_ctx* ctx, char* buf, int cap);
/* development builds only (FO_TRACE_BUILD=1): after fo_set_option("trace", n) every CTA of the step's main kernels appends one
 * record of 8 uint64 {kernel id | smid << 8 | aux << 16 | linear block id << 32, grid dims, 6 x %globaltimer ns}; this copies up to
 * cap_records of them out and restarts the log.  A regular build records nothing (n_records = 0). */
int fo_debug_trace_read(fo_ctx* ctx, uint64_t* out, int64_t cap_records, int64_t* n_records);
/* n_ctas CTAs launched as the context launches its kernels (on `stream`, in its SM group if it has one) write the id of the
 * SM they ran on to out (n_ctas int32, device or host memory; a host buffer is filled when the call returns).  graph = 0: a
 * direct launch; graph = 1: the launch captured into a CUDA graph on the context's capture stream and replayed, as a streaming
 * step is.  Each CTA stays ~20 us, so that a launch spreads over every SM the context can reach. */
int fo_debug_sm_ids(fo_ctx* ctx, int n_ctas, int graph, int32_t* out, void* stream);
/* host-only: the tile plan of the tcgen05 GEMM for (activation rows, output columns, K) -- swap = weights on the UMMA-M side,
 * bn = UMMA N, split = K splits; can_defer = a consumer kernel finishes the split-K sum.  Needs no GPU (CPU tests of the plan). */
int fo_debug_plan(int64_t act_rows, int n_out, int K, int can_defer, int* swap, int* bn, int* split);
/* host-only: whether a streaming step of n_sessions x frames token rows takes the one-launch layer stack (csrc/fo_stack.cu,
 * option "stack_rows") on a device of `sms` SMs with smem_max bytes of opt-in shared memory per CTA, and its plan: dynamic
 * shared memory, K chunk of the FFN2 activations, weight rows per CTA of the QKV / FFN1 / out-proj (= FFN2) slices.
 * Returns 0 and the plan, or 1 when the step does not qualify.  Needs no GPU (CPU tests). */
int fo_debug_stack_plan(int d_model, int ffn_dim, int heads, int n_sessions, int frames, int window, int layers, int sms,
                        int smem_max, int* smem_bytes, int* ffn2_chunk, int* rows_qkv, int* rows_ffn1, int* rows_out);
/* one GEMM of the library, exposed for kernel-level parity tests and roofline measurement:
 * C[M,N] = A[M,K] * W[N,K]^T (+bias) in the context's dtype, fp32 in/out on device pointers. */
int fo_debug_gemm(fo_ctx* ctx, const float* A, const float* W, const float* bias, float* C,
                  int M, int N, int K, int backend, int relu, int iters, float* ms_out, void* stream);
/* one attention launcher of the library on caller-given tensors, exposed for kernel-level parity tests.  Runs on `stream` and
 * returns when it is done.  All tensors are fp32 device pointers, all tables host arrays:
 *   qkv (rows, 3D) Q | K | V as the QKV GEMM writes them: bf16 contexts convert K | V to fp16 (round to nearest, as the
 *       activations are), Q is read as fp32 from the same array;  ptab (ptab_rows, D) the rel-pos table P_l, at least the
 *       context's pos_rows rows (head-major copy built as fo_finalize_weights builds it);  pos_u, pos_v (D);
 *   out (rows, D): the attention output converted to fp32; rows no query writes (packed gaps) are 0.
 * mode FO_ATT_OFFLINE: n utterances padded to T rows (rows = n*T), seq = ilens (n) -- fo_encode_offline's attention.
 *      FO_ATT_PACKED: n utterances of seq[b] rows back to back with `gap` unused rows between them -- fo_encode_offline_packed's.
 *      chunk, left: the band of both offline modes.
 *      FO_ATT_STREAM: sessions seq (n), t frames each (rows = n*t) against `layer`'s KV ring at each slot's n_frames / pe_index;
 *      nsplit > 0 (bf16 contexts): q / k / v summed from split-K partials part [nsplit][rows][3D] + part_bias (3D), qkv unused.
 *      FO_ATT_CHUNKS: sessions seq bring cnt[b] chunks of t frames, rows from (off[b] - off[0]) * t (off = off[0] + running sum
 *      of cnt), `group` chunks per CTA.
 * The streaming modes append the new K/V rows to the ring as a step does, and advance no session.  FO_ERR_ARG, nothing
 * launched: t > max_t, window + t > ring capacity or 128, window + group * t > 128, T or a length past pos_rows, ptab_rows < pos_rows. */
enum { FO_ATT_OFFLINE = 0, FO_ATT_PACKED = 1, FO_ATT_STREAM = 2, FO_ATT_CHUNKS = 3 };
int fo_debug_attention(fo_ctx* ctx, int mode, int n, const int32_t* seq, const int32_t* cnt, const int32_t* off, int T, int gap,
                       int chunk, int left, int t, int layer, int group, const float* qkv, const float* part, int nsplit,
                       const float* part_bias, const float* ptab, int ptab_rows, const float* pos_u, const float* pos_v,
                       float* out, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* FO_B200_H */
