// C ABI (include/fo_b200.h) over the sm_100a kernels: context, weight packing, session slots resident in
// HBM, and the three step programs (streaming chunk, full utterance, stateless adapter).
//
// HBM layout per context
//   weights     compute dtype (fp32 | bf16), [N][K] row-major (K-major operands for the GEMMs):
//               conv2 as [C][(kh*3+kw)*C + ci], sub-Linear with K permuted to f*C + c so the conv2 output
//               (b, t, f, c) feeds it without a transpose, Wq|Wk|Wv stacked to [3D][D], adapter conv as
//               [2D][tau*D + ci]; biases / LayerNorm / pos_bias in fp32.
//   pos tables  per layer P_l = pe[0:pos_max_len] * Wpos_l^T (weights-only, SURVEY 0-iv), [L][pos][D].
//   sessions    KV ring [L][slot][K|V][H][cap][64] (cap = window + max frames per call, rounded to 8),
//               n_frames / pe_index / adapter-cache flag int32 [slot], adapter cache fp32 [slot][2][k-1][D]
//               (double buffered), fbank sample buffer fp32 [slot][carry+chunk], feature ring [slot][ctx+m][F].
//   workspace   activations of one step, grown on demand, reused.
#include <stdarg.h>
#include <string.h>
#include <math.h>

#include <algorithm>
#include <map>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/fo_b200.h"
#include "fo_common.cuh"

namespace fo {

std::atomic<long long> g_launches{0};
thread_local long long t_launches = 0;
thread_local int g_use_pdl = 1;   // launch attribute actually applied (set per step, by the thread that enqueues it)
int g_want_pdl = 1;       // option "pdl"
static thread_local char g_err[1024] = "";

void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

namespace {

struct DevBuf {
    void* p = nullptr;
    size_t cap = 0;
};

struct HostTensor {          // staged fp32 weight on device until finalize
    float* d = nullptr;
    std::vector<int64_t> shape;
    long long numel = 0;
};

struct LayerW {
    void *wqkv = nullptr, *wo = nullptr, *w1 = nullptr, *w2 = nullptr;
    void* wcat = nullptr;                     // concat_linear [D][2D] (transformer-concat-after)
    float* bcat = nullptr;
    float* ptab = nullptr;                    // P_l = pe * Wpos_l^T, fp32 [pos_rows][D] (offline attention)
    void* ptab_h = nullptr;                   // the same, [H][pos_rows][64] in the activation type (streaming attention)
    float *bqkv = nullptr, *bo = nullptr, *b1 = nullptr, *b2 = nullptr;
    float *dw_w = nullptr, *dw_b = nullptr;   // Conv1dLinear depthwise taps [C][k] and bias (fp32); w1 is then the 1x1 conv
    float *pos_u = nullptr, *pos_v = nullptr, *ln1g = nullptr, *ln1b = nullptr, *ln2g = nullptr, *ln2b = nullptr;
};

}  // namespace
}  // namespace fo

using namespace fo;

struct fo_ctx {
    fo_config cfg;
    int device = 0, dtype = FO_F32;
    size_t esz = 4;                           // bytes per activation / weight element
    bool finalized = false;
    long long device_bytes = 0;
    std::map<std::string, HostTensor> staged;
    std::vector<void*> owned;                 // every cudaMalloc of this context

    // derived dims
    int F = 0, F1 = 0, F2 = 0, D = 0, H = 0, FF = 0, L = 0, E = 0, KA = 0;
    int KF = 0;                               // Conv1dLinear kernel size (0: plain feed-forward)
    int KM = 0;                               // MultiLayeredConv1d kernel size (0: off); full-utterance encode only
    float* ffn_cache = nullptr;               // [slot][L][KF-1][D] fp32: left context of the depthwise conv
    int window = 0, full_chunk = 0, pe_wrap = 0, pos_rows = 0, ring_cap = 0, max_t = 0;
    int carry = 0, chunk_samples = 0, fft = 0;

    // packed weights
    float *cmvn_mean = nullptr, *cmvn_istd = nullptr, *conv1_w = nullptr, *conv1_b = nullptr;
    void *conv2_w = nullptr, *sub_w = nullptr, *emb_w = nullptr;
    float *conv2_b = nullptr, *sub_b = nullptr, *emb_b = nullptr, *emb_g = nullptr, *emb_beta = nullptr;
    std::vector<LayerW> layers;
    float *after_g = nullptr, *after_b = nullptr;
    // adapter: ad_nst causal convolutions (0 LinearAdapter, 1 CNNSubsampling, 2 CNNAdapter and CNNSubsampling with
    // 4 * enc_out_dim < llm_embed_dim, adapter.py:10-57,83-96), then a norm of the last conv's rows (ad_ln_*: LayerNorm
    // or folded BatchNorm, then ReLU or GELU) and the projection to llm_dim
    struct AdStage {
        void* w = nullptr;                    // [cout][KA * cin] (implicit GEMM over the staged rows)
        float* b = nullptr;
        int cin = 0, cout = 0, stride = 1;
        float *in_scale = nullptr, *in_shift = nullptr;   // folded BatchNorm of the previous conv: conv_stage feeds
                                                          // ReLU(x * scale + shift) to this one
        float* cache = nullptr;               // [slot][2][k-1][cin] fp32, double buffered by ad_valid (carried caches only)
    } ad_st[2];
    int ad_nst = 0;
    bool ad_carry = false;                    // CNNSubsampling carries the caches; CNNAdapter starts from zeros every call
    float ad_ln_eps = 1e-3f;                  // < 0: folded BatchNorm (affine only)
    int ad_ln_act = 1;                        // 1 ReLU, 2 GELU
    void* ad_proj_w = nullptr;
    float *ad_ln_g = nullptr, *ad_ln_b = nullptr, *ad_proj_b = nullptr;
    float *fb_window = nullptr, *fb_mel = nullptr;
    int *fb_lo = nullptr, *fb_hi = nullptr;

    // sessions
    void* ring = nullptr;                     // [L][S][2][H][cap][64]
    int32_t *n_frames = nullptr, *pe_index = nullptr, *ad_valid = nullptr;
    float *samples = nullptr, *feat_ring = nullptr;
    std::vector<uint8_t> slot_used;
    std::vector<int32_t> free_slots;
    long long sessions_in_use = 0;

    // step plumbing
    static const int NSTAGE = 8;
    int32_t* ids_host[NSTAGE] = {nullptr};
    cudaEvent_t ids_event[NSTAGE] = {nullptr};
    int ids_cursor = 0;
    int32_t* ids_dev = nullptr;               // [3][max_sessions]: session ids, then cnt_dev and off_dev
    int32_t* cnt_dev = nullptr;               // chunks per session of a multi-chunk call (fo_encode_stream_chunks[_v])
    int32_t* off_dev = nullptr;               // first block of each session in that call (prefix sums of cnt)
    DevBuf ws[48];                            // named workspaces, see enum below
    // options
    int gemm_backend = 0, use_graph = 0, split_k = 1;
    int tc_npa = 0, tc_npb = 0;
    TcTune tc_tune{-1, -1, -1};               // debugging: force the tile plan of the tcgen05 GEMM
    static const int MAX_GROUPS = 4;
    TcWorkspace tc_wsg[MAX_GROUPS];           // split-K partials + tile counters of the tcgen05 GEMM, one per session group
    TcWorkspace* tc_cur = &tc_wsg[0];
    int debug_skip = 0;                       // timing attribution only (results invalid): bit0 attention, bit1 LayerNorm,
                                              // bit2 QKV/out GEMMs, bit3 FFN GEMMs, bit4 subsampling/adapter GEMMs, bit5 EVERY GEMM launch (nothing else)
    int use_prefetch = 0;                     // next-kernel L2 prefetch (L2Prefetch): bit0 weights, bit1 this layer's KV rings.
                                              // Off: it paid 2 % with one GEMM CTA per SM; with two co-resident CTAs hiding
                                              // each other's cold loads it costs 1-2 % at 16-128 sessions (r75/r76)
    int pf_slot_lo = 0, pf_slot_hi = 0;       // slot range of the sessions of the current step
    int step_part = 0;                        // development (timing attribution, results invalid): 1 = front only (fbank .. embed), 2 = layers + adapter only
    int defer_reduce = 1;                     // split-K GEMMs of the residual stream leave the reduction to the LayerNorm that follows
    int fuse_ln = 0;                          // LayerNorm inside the epilogue of the GEMM that completes the residual rows
                                              // (measured slower than the stand-alone kernel at 64-256 sessions: off)
    // fo_stream_step_async: host <-> device copies on an internal stream, staging buffers double-buffered by ticket parity
    cudaStream_t copy_stream = nullptr;       // read-backs (device -> host) of the pipelined steps
    cudaStream_t upload_stream = nullptr;     // their PCM uploads: a stream of their own, so that the upload of step i+1 does not queue
                                              // behind the read-back of step i (which waits for step i's kernels)
    cudaEvent_t ev_in[2] = {nullptr, nullptr}, ev_compute[2] = {nullptr, nullptr}, ev_out[2] = {nullptr, nullptr};
    long long async_ticket = 0;
    unsigned long long* trace_buf = nullptr;  // development (FO_TRACE_BUILD): CTA timeline records, 8 x u64 each
    unsigned int* trace_cnt = nullptr;
    unsigned int trace_cap = 0;
    unsigned long long* sat_counter = nullptr; // device: fp16-range saturations counted by the GEMM epilogues (Epilogue::sat)
    cudaEvent_t ev_sync = nullptr;            // recorded after every synchronous step: the copy stream of a later async step
                                              // must not overwrite the staging buffers that step still reads
    std::vector<int32_t> ids_last;            // session ids currently in ids_dev (uploaded on ids_last_stream)
    std::vector<int32_t> cnt_last;            // chunk counts currently in cnt_dev (empty: none uploaded with ids_last)
    cudaStream_t ids_last_stream = nullptr;
    std::vector<long long> id_stamp;          // check_ids: call number that last named each slot (duplicate detection)
    long long id_call = 0;
    void* handoff = nullptr;                  // fo_stream_step_embeds: fp16 destination of the adapter rows for this call
    long long handoff_rows = 0, handoff_off = 0;
    // fo_handoff_arm: the NEXT streaming call writes its adapter rows into `embeds` and the mask / start rows beside them
    struct Armed {
        bool on = false;
        void* embeds = nullptr;
        long long rows = 0, prefix = 0;
        int n = 0;
        std::vector<uint8_t> onset;
        const uint8_t* prefix_mask = nullptr;     // device (or null)
        uint8_t* attn_mask = nullptr;
        int32_t* row_start = nullptr;
    } armed;
    uint8_t* onset_dev = nullptr;
    // an armed recording call: {caller block, onset flag} of every pass block, pass after pass (pinned, uploaded one pass at a
    // time into WS_HOTAB); reused once ho_tab_event (the previous armed call's last upload) has completed
    int2* ho_tab_host = nullptr;
    long long ho_tab_cap = 0;
    cudaEvent_t ho_tab_event = nullptr;
    int groups = 1;                           // session groups whose layer kernels run on parallel streams
    cudaStream_t grp_stream[MAX_GROUPS] = {nullptr};
    cudaEvent_t ev_fork = nullptr, ev_join[MAX_GROUPS] = {nullptr};
    cudaStream_t mix_stream[MAX_GROUPS] = {nullptr};   // per group: the multi-chunk attention of a call that mixes counts
    cudaEvent_t ev_mix_fork[MAX_GROUPS] = {nullptr}, ev_mix_join[MAX_GROUPS] = {nullptr};
    int profile_gemm = 0;                     // time every GEMM launch with a CUDA event pair (bench roofline)
    // weight-streaming layer stack (fo_stack.cu): all layers of a step of <= stack_rows token rows in one cooperative launch
    int stack_rows = 8;                       // option "stack_rows": steps of up to this many token rows take the stack kernel (<= STACK_MAX_ROWS; 0 = never)
    StackLayer* stack_layers = nullptr;       // device table, built at the first use
    unsigned int* stack_bar = nullptr;        // grid-barrier words of the kernel
    unsigned long long* stack_trace = nullptr;
    long long stack_launches = 0;
    int steps_pass_blocks = 0;                // option: blocks per pass of fo_stream_steps_v (0: from STEPS_PASS_BYTES)
    int packed_pass_frames = 0;               // option: grid feature frames per pass of fo_encode_offline_packed_pcm (0: from PACKED_PASS_BYTES)
    struct ProfRec { cudaEvent_t e0, e1; int M, N, K; };
    std::vector<ProfRec> prof_events;
    // captured step graphs, keyed by the shape of the call; invalidated when a workspace moves
    struct StepGraph {
        cudaGraphExec_t exec = nullptr;
        long long epoch = -1;        // ws_epoch the graph was captured at
        long long warm_epoch = -1;   // ws_epoch after the last eager run of this key
        long long launches = 0;      // kernels inside the graph
        long long stacks = 0;        // stack-kernel launches inside the graph
    };
    std::map<std::string, StepGraph> graphs;
    long long ws_epoch = 0;
    // session snapshots (fo_session_save / fo_session_restore): buffers of their own, allocated at the first use, so that a
    // snapshot between two graph-replayed steps neither grows a step workspace nor invalidates the captured graphs
    int32_t* snap_ids_dev = nullptr;
    int32_t* snap_ids_host = nullptr;         // pinned; reused once snap_ids_event (its last upload) has completed
    cudaEvent_t snap_ids_event = nullptr;
    int32_t* snap_hdr_host = nullptr;         // pinned [max_sessions][SNAP_HDR_WORDS]: headers of a device buffer, read back
    char* snap_stage = nullptr;               // device staging of host buffers, snap_stage_n records
    int snap_stage_n = 0;
    cudaStream_t cap_stream = nullptr;        // capture happens here (the caller's stream may be the legacy
                                              // default stream, which cannot be captured); replay on the caller's
    // SMs the context's grids are sized to: its SM group (fo_create_on_sms), else the device
    int sms = 148;
    int smem_optin = 0, coop = 0;             // the device's opt-in shared memory per CTA, cooperative-launch support
    void* green = nullptr;                    // the group's green context (fo_partition.cu); null: the whole device
    cudaStream_t exec_stream = nullptr;       // with a group: the stream of the group every entry point enqueues on (OnGroup)
    cudaEvent_t ev_enter = nullptr, ev_leave = nullptr;
    std::string leave_err;                    // a call whose caller's stream could not be ordered after its work (OnGroup):
                                              // the next call through OnGroup returns this as its error
    // stats
    fo_stats_t stats;
    std::mutex mu;
};

namespace {

enum { WS_FEATS = 0, WS_C1, WS_C2, WS_XSUB, WS_EMB, WS_X, WS_H, WS_QKV, WS_ATT, WS_FFH, WS_ENC, WS_XIN, WS_ACONV, WS_AH,
       WS_Y, WS_MASK2, WS_ILENS, WS_ILENS2, WS_AMASK, WS_PCM, WS_TMP0, WS_TMP1, WS_TMP2, WS_TMP3, WS_Q32, WS_HC, WS_PART, WS_PCM2, WS_ENC2, WS_Y2, WS_AC1, WS_XIN2, WS_TMP4, WS_TMP5, WS_HP, WS_FP, WS_PACK, WS_SROWS,
       WS_PKTAB, WS_FGRID, WS_XP, WS_FBTAB, WS_HOTAB, WS_COUNT };
static_assert(WS_COUNT <= (int)(sizeof(fo_ctx::ws) / sizeof(DevBuf)), "fo_ctx::ws holds every named workspace");

int dev_alloc(fo_ctx* c, void** p, size_t bytes) {
    *p = nullptr;
    if (bytes == 0) bytes = 16;
    cudaError_t e = cudaMalloc(p, bytes);
    if (e != cudaSuccess) {
        set_error("cudaMalloc(%zu bytes) failed: %s", bytes, cudaGetErrorString(e));
        return FO_ERR_NOMEM;
    }
    c->owned.push_back(*p);
    c->device_bytes += (long long)bytes;
    return 0;
}

int ctx_sync(fo_ctx* c);

int ws_ensure(fo_ctx* c, int which, size_t bytes, void** out) {
    DevBuf& b = c->ws[which];
    if (b.cap < bytes) {
        if (b.p) {
            // grown buffers are rare (first call at a new size); wait for users of the old one
            FO_TRY(ctx_sync(c));
            for (auto& q : c->owned)
                if (q == b.p) { q = nullptr; break; }
            cudaFree(b.p);
            c->device_bytes -= (long long)b.cap;
        }
        size_t cap = bytes + bytes / 8 + 256;
        FO_TRY(dev_alloc(c, &b.p, cap));
        b.cap = cap;
        c->ws_epoch += 1;                       // captured graphs hold the old pointers
    }
    *out = b.p;
    return 0;
}

bool is_device_ptr(const void* p) {
    cudaPointerAttributes a;
    cudaError_t e = cudaPointerGetAttributes(&a, p);
    if (e != cudaSuccess) { cudaGetLastError(); return false; }
    return a.type == cudaMemoryTypeDevice || a.type == cudaMemoryTypeManaged;
}

// input: returns a device pointer holding `bytes` of p (copying through workspace `which` when p is host memory)
int in_dev(fo_ctx* c, const void* p, size_t bytes, int which, cudaStream_t st, const void** out) {
    if (is_device_ptr(p)) { *out = p; return 0; }
    void* d;
    FO_TRY(ws_ensure(c, which, bytes, &d));
    FO_CUDA(cudaMemcpyAsync(d, p, bytes, cudaMemcpyHostToDevice, st));
    *out = d;
    return 0;
}
// output: device pointer to write (user's if device memory, else workspace); finish with out_done
int out_dev(fo_ctx* c, void* p, size_t bytes, int which, void** out) {
    if (p && is_device_ptr(p)) { *out = p; return 0; }
    return ws_ensure(c, which, bytes, out);
}
int out_done(void* user, void* dev, size_t bytes, cudaStream_t st) {
    if (user && user != dev) FO_CUDA(cudaMemcpyAsync(user, dev, bytes, cudaMemcpyDeviceToHost, st));
    return 0;
}

// every internal stream of the context: in its SM group when it has one
int make_stream(fo_ctx* c, cudaStream_t* st) {
    if (c->green) return sm_group_stream(c->green, st);
    FO_CUDA(cudaStreamCreateWithFlags(st, cudaStreamNonBlocking));
    return 0;
}

// cudaDeviceSynchronize, and the context's own streams when they live in its SM group's green context
int ctx_sync(fo_ctx* c) {
    FO_CUDA(cudaDeviceSynchronize());
    if (!c->green) return 0;
    for (cudaStream_t s : {c->exec_stream, c->cap_stream, c->copy_stream, c->upload_stream})
        if (s) FO_CUDA(cudaStreamSynchronize(s));
    for (int g = 0; g < fo_ctx::MAX_GROUPS; ++g) {
        if (c->grp_stream[g]) FO_CUDA(cudaStreamSynchronize(c->grp_stream[g]));
        if (c->mix_stream[g]) FO_CUDA(cudaStreamSynchronize(c->mix_stream[g]));
    }
    return 0;
}

// The stream an entry point enqueues on.  A whole-device context works on the caller's stream itself.  A context on an SM
// group works on its execution stream in that group, ordered after what the caller enqueued on its stream before the call
// and before what the caller enqueues after it: caller -> record -> wait -> the call's work -> record -> caller waits.
struct OnGroup {
    fo_ctx* c;
    cudaStream_t user, st;
    int err = 0;
    OnGroup(fo_ctx* c_, void* stream) : c(c_), user((cudaStream_t)stream), st((cudaStream_t)stream) {
        if (!c || !c->green) return;
        if (!c->leave_err.empty()) {
            set_error("%s", c->leave_err.c_str());
            c->leave_err.clear();
            err = FO_ERR_CUDA;
            return;
        }
        cudaError_t e = cudaEventRecord(c->ev_enter, user);
        if (e == cudaSuccess) e = cudaStreamWaitEvent(c->exec_stream, c->ev_enter, 0);
        if (e != cudaSuccess) { set_error("entering the context's SM group: %s", cudaGetErrorString(e)); err = FO_ERR_CUDA; return; }
        st = c->exec_stream;
    }
    ~OnGroup() {
        if (st == user) return;
        cudaError_t e = cudaEventRecord(c->ev_leave, st);
        if (e == cudaSuccess) e = cudaStreamWaitEvent(user, c->ev_leave, 0);
        if (e != cudaSuccess)
            c->leave_err = std::string("a previous call could not order the caller's stream after its work in the context's SM group: ") +
                           cudaGetErrorString(e);
    }
};
// at the top of an entry point taking `void* stream`: from here on `stream` is the stream the call enqueues on
#define FO_ON_GROUP(c, stream)                       \
    OnGroup on_group_(c, stream);                    \
    FO_TRY(on_group_.err);                           \
    stream = (void*)on_group_.st

int check_ids(fo_ctx* c, const int32_t* ids, int n) {
    FO_CHECK(ids != nullptr && n > 0, "ids must be a host array of n > 0 session ids");
    FO_CHECK(n <= c->cfg.max_sessions, "n (%d) exceeds max_sessions (%d)", n, c->cfg.max_sessions);
    if ((int)c->id_stamp.size() != c->cfg.max_sessions) c->id_stamp.assign(c->cfg.max_sessions, 0);
    const long long call = ++c->id_call;
    for (int i = 0; i < n; ++i) {
        FO_CHECK(ids[i] >= 0 && ids[i] < c->cfg.max_sessions && c->slot_used[ids[i]], "session id %d is not allocated", ids[i]);
        // two rows of one batch would append to the same KV ring / adapter cache / fbank carry concurrently
        FO_CHECK(c->id_stamp[ids[i]] != call, "session id %d appears twice in one batch (ids must be distinct)", ids[i]);
        c->id_stamp[ids[i]] = call;
    }
    return 0;
}

// chunks (multi-chunk calls): the per-session counts, uploaded with their block offsets to cnt_dev / off_dev
int upload_ids(fo_ctx* c, const int32_t* ids, int n, cudaStream_t st, const uint8_t* onset = nullptr, int n_onset = 0,
               const int32_t* chunks = nullptr) {
    // the same sessions (and counts) as in the previous step (the steady state of a server loop): the device copy is still valid
    if (!onset && st == c->ids_last_stream && (int)c->ids_last.size() == n && memcmp(c->ids_last.data(), ids, sizeof(int32_t) * n) == 0 &&
        (!chunks || ((int)c->cnt_last.size() == n && memcmp(c->cnt_last.data(), chunks, sizeof(int32_t) * n) == 0)))
        return 0;
    c->ids_last.assign(ids, ids + n);
    if (chunks) c->cnt_last.assign(chunks, chunks + n);
    else c->cnt_last.clear();
    c->ids_last_stream = st;
    const int k = c->ids_cursor, S = c->cfg.max_sessions;
    c->ids_cursor = (k + 1) % fo_ctx::NSTAGE;
    FO_CUDA(cudaEventSynchronize(c->ids_event[k]));
    memcpy(c->ids_host[k], ids, sizeof(int32_t) * n);
    FO_CUDA(cudaMemcpyAsync(c->ids_dev, c->ids_host[k], sizeof(int32_t) * n, cudaMemcpyHostToDevice, st));
    if (chunks) {
        int32_t* ch = c->ids_host[k] + S;
        memcpy(ch, chunks, sizeof(int32_t) * n);
        for (int i = 0, o = 0; i < n; o += chunks[i++]) ch[S + i] = o;
        FO_CUDA(cudaMemcpyAsync(c->cnt_dev, ch, sizeof(int32_t) * n, cudaMemcpyHostToDevice, st));
        FO_CUDA(cudaMemcpyAsync(c->off_dev, ch + S, sizeof(int32_t) * n, cudaMemcpyHostToDevice, st));
    }
    if (onset) {                                 // behind the ids and the count table: the hand-off's per-block onset flags
        uint8_t* oh = reinterpret_cast<uint8_t*>(c->ids_host[k] + 3 * S);
        memcpy(oh, onset, n_onset);
        FO_CUDA(cudaMemcpyAsync(c->onset_dev, oh, n_onset, cudaMemcpyHostToDevice, st));
    }
    FO_CUDA(cudaEventRecord(c->ids_event[k], st));
    return 0;
}

// ---- GEMM dispatch ----------------------------------------------------------------------------
// M = GEMM rows over the (possibly padded) row grid of `ga`; rm maps them to rows of C.  `fused_ln` reports whether
// the kernel that ran also did the LayerNorm requested in ep.ln_* (only the tcgen05 kernel does).
template <typename TA>
int gemm_raw(fo_ctx* c, const TA* A, const AGather& ga, const void* W, int M, int N, int K, const Epilogue& ep,
             const RowMap& rm, cudaStream_t st, bool* fused_ln, int* deferred);
template <>
int gemm_raw<float>(fo_ctx* c, const float* A, const AGather& ga, const void* W, int M, int N, int K, const Epilogue& ep,
                    const RowMap& rm, cudaStream_t st, bool* fused_ln, int* deferred) {
    *fused_ln = false;
    *deferred = 0;
    return gemm_simt<float, float>(A, ga, reinterpret_cast<const float*>(W), M, N, K, ep, rm, st);
}
template <>
int gemm_raw<act16>(fo_ctx* c, const act16* A, const AGather& ga, const void* W, int M, int N, int K, const Epilogue& ep,
                    const RowMap& rm, cudaStream_t st, bool* fused_ln, int* deferred) {
    *fused_ln = false;
    *deferred = 0;
    Epilogue eps = ep;
    eps.sat = c->sat_counter;
    if (c->gemm_backend == 1) {
        Epilogue e = eps;
        if (!c->fuse_ln) e.ln_gamma = nullptr;
        // the split-K reduction can ride on the LayerNorm that follows (residual stream in place, rows normalised next)
        e.defer_reduce = c->defer_reduce && ep.ln_gamma && !c->fuse_ln && ep.residual == ep.c_f32 && ep.c_f32 && !ep.c_act &&
                         !ep.relu && ep.scale == 1.0f && N <= 1024 && N % 256 == 0;
        // ... or on a consumer kernel that asked for it (QKV -> streaming attention): bias only, no residual / activation
        if (ep.defer_reduce == 2 && c->defer_reduce && !ep.relu && ep.scale == 1.0f && !ep.residual && !ep.ln_gamma) e.defer_reduce = 2;
        int r = gemm_tc(A, 1, ga, W, M, N, K, e, rm, *c->tc_cur, st, deferred);
        if (r == 0) *fused_ln = e.ln_gamma != nullptr;
        if (r <= 0) return r;
    }
    return gemm_simt<act16, act16>(A, ga, reinterpret_cast<const act16*>(W), M, N, K, eps, rm, st);
}
template <typename TA>
int gemm(fo_ctx* c, const TA* A, const AGather& ga, const void* W, int M, int N, int K, const Epilogue& ep,
         const RowMap& rm, cudaStream_t st, int* deferred_out = nullptr) {
    bool fused = false;
    int deferred = 0;
    int r;
    if (c->debug_skip & 32) {
        r = 0;                                    // timing attribution: every GEMM launch dropped, the rest of the step kept
    } else if (!c->profile_gemm) {
        r = gemm_raw<TA>(c, A, ga, W, M, N, K, ep, rm, st, &fused, &deferred);
    } else {
        cudaEvent_t e0, e1;
        FO_CUDA(cudaEventCreate(&e0));
        FO_CUDA(cudaEventCreate(&e1));
        FO_CUDA(cudaEventRecord(e0, st));
        r = gemm_raw<TA>(c, A, ga, W, M, N, K, ep, rm, st, &fused, &deferred);
        FO_CUDA(cudaEventRecord(e1, st));
        c->prof_events.push_back(fo_ctx::ProfRec{e0, e1, M, N, K});
    }
    if (deferred_out) { *deferred_out = deferred; return r; }      // the caller's next kernel finishes the sum
    if (r == 0 && deferred > 0)                   // the GEMM left raw split-K partials: the LayerNorm finishes the sum
        return layer_norm_reduce<TA>(ep.c_f32, c->tc_cur->partial, deferred, ep.bias, M, N, ep.ln_gamma, ep.ln_beta, ep.ln_eps,
                                     reinterpret_cast<TA*>(ep.ln_act), ep.ln_f32, st);
    // rows of C: the GEMM rows of an implicit-GEMM convolution run over a padded grid that the row map compacts
    const int out_rows = rm.p1 ? (M / rm.p1) * rm.q1 : M;
    if (r == 0 && ep.ln_gamma && !fused)          // LayerNorm of the finished rows as its own kernel (fp32 / FFMA paths)
        r = layer_norm<TA>(ep.c_f32, out_rows, N, ep.ln_gamma, ep.ln_beta, ep.ln_eps, 0, 1.0f, reinterpret_cast<TA*>(ep.ln_act),
                           ep.ln_f32, st);
    return r;
}
// plain row-major A (M, K)
template <typename TA>
int gemm(fo_ctx* c, const TA* A, const void* W, int M, int N, int K, const Epilogue& ep, cudaStream_t st) {
    return gemm<TA>(c, A, plain_rows(K, M), W, M, N, K, ep, RowMap(), st);
}

const HostTensor* staged(fo_ctx* c, const std::string& name) {
    auto it = c->staged.find(name);
    return it == c->staged.end() ? nullptr : &it->second;
}

int need(fo_ctx* c, const std::string& name, std::initializer_list<int64_t> shape, const HostTensor** out) {
    const HostTensor* t = staged(c, name);
    FO_CHECK(t != nullptr, "finalize: tensor '%s' was never loaded", name.c_str());
    bool ok = t->shape.size() == shape.size();
    size_t i = 0;
    for (int64_t s : shape) { if (ok && t->shape[i] != s) ok = false; ++i; }
    FO_CHECK(ok, "finalize: tensor '%s' has the wrong shape", name.c_str());
    *out = t;
    return 0;
}

int keep_f32(fo_ctx* c, const std::string& name, std::initializer_list<int64_t> shape, float** out) {
    const HostTensor* t;
    FO_TRY(need(c, name, shape, &t));
    void* d;
    FO_TRY(dev_alloc(c, &d, t->numel * sizeof(float)));
    FO_CUDA(cudaMemcpy(d, t->d, t->numel * sizeof(float), cudaMemcpyDeviceToDevice));
    *out = reinterpret_cast<float*>(d);
    return 0;
}

template <typename TW>
int keep_w(fo_ctx* c, const std::string& name, std::initializer_list<int64_t> shape, void** out) {
    const HostTensor* t;
    FO_TRY(need(c, name, shape, &t));
    void* d;
    FO_TRY(dev_alloc(c, &d, t->numel * sizeof(TW)));
    FO_TRY(convert_weight<TW>(t->d, t->numel, reinterpret_cast<TW*>(d), 0));
    *out = d;
    return 0;
}

template <typename TW>
int finalize_t(fo_ctx* c) {
    const int D = c->D, F = c->F, FF = c->FF, L = c->L, E = c->E, KA = c->KA, F2 = c->F2, H = c->H;
    const fo_config& g = c->cfg;
    if (g.has_encoder) {
        if (staged(c, "global_cmvn.mean")) {
            FO_TRY(keep_f32(c, "global_cmvn.mean", {F}, &c->cmvn_mean));
            FO_TRY(keep_f32(c, "global_cmvn.istd", {F}, &c->cmvn_istd));
        }
        FO_TRY(keep_f32(c, "enc.0.core.conv.0.weight", {D, 1, 3, 3}, &c->conv1_w));
        FO_TRY(keep_f32(c, "enc.0.core.conv.0.bias", {D}, &c->conv1_b));
        const HostTensor* t;
        FO_TRY(need(c, "enc.0.core.conv.2.weight", {D, D, 3, 3}, &t));
        FO_TRY(dev_alloc(c, &c->conv2_w, (size_t)D * D * 9 * sizeof(TW)));
        FO_TRY(repack_conv2<TW>(t->d, D, reinterpret_cast<TW*>(c->conv2_w), 0));
        FO_TRY(keep_f32(c, "enc.0.core.conv.2.bias", {D}, &c->conv2_b));
        FO_TRY(need(c, "enc.0.core.out.0.weight", {D, (int64_t)D * F2}, &t));
        FO_TRY(dev_alloc(c, &c->sub_w, (size_t)D * D * F2 * sizeof(TW)));
        FO_TRY(repack_sublinear<TW>(t->d, D, F2, reinterpret_cast<TW*>(c->sub_w), 0));
        FO_TRY(keep_f32(c, "enc.0.core.out.0.bias", {D}, &c->sub_b));
        if (g.input_layer_linear) {
            FO_TRY(keep_w<TW>(c, "enc.1.embed.0.weight", {D, D}, &c->emb_w));
            FO_TRY(keep_f32(c, "enc.1.embed.0.bias", {D}, &c->emb_b));
            FO_TRY(keep_f32(c, "enc.1.embed.1.weight", {D}, &c->emb_g));
            FO_TRY(keep_f32(c, "enc.1.embed.1.bias", {D}, &c->emb_beta));
        }
        // positional table (fp32 sin/cos built on the host exactly as attention.py:13-30 does)
        const HostTensor* pe;
        FO_TRY(need(c, "pos.table", {g.pos_max_len, D}, &pe));
        // rows past pos_max_len (streaming positions of left_chunks <= 0 contexts, fo_create): the same fp32 operations as the
        // table, pos * exp(2i * -(ln 10000 / D)) then sin / cos.  The host's expf may differ from torch's by one ulp in a few
        // columns, i.e. ~1e-4 in the argument at position 5000 -- the size of the fp32 rounding of the argument itself.
        const float* pe_rows = pe->d;
        struct TmpBuf { void* p = nullptr; ~TmpBuf() { if (p) cudaFree(p); } } pe_ext;
        if (c->pos_rows > g.pos_max_len) {
            const int extra = c->pos_rows - g.pos_max_len;
            std::vector<float> hx((size_t)extra * D);
            const float s = (float)(-(log(10000.0) / D));
            for (int i = 0; i < D / 2; ++i) {
                const float dt = expf((float)(2 * i) * s);
                for (int r = 0; r < extra; ++r) {
                    const float a = (float)(g.pos_max_len + r) * dt;
                    hx[(size_t)r * D + 2 * i] = sinf(a);
                    hx[(size_t)r * D + 2 * i + 1] = cosf(a);
                }
            }
            FO_CUDA(cudaMalloc(&pe_ext.p, (size_t)c->pos_rows * D * sizeof(float)));
            FO_CUDA(cudaMemcpy(pe_ext.p, pe->d, (size_t)g.pos_max_len * D * sizeof(float), cudaMemcpyDeviceToDevice));
            FO_CUDA(cudaMemcpy((float*)pe_ext.p + (size_t)g.pos_max_len * D, hx.data(), hx.size() * sizeof(float), cudaMemcpyHostToDevice));
            pe_rows = (const float*)pe_ext.p;
        }
        c->layers.resize(L);
        for (int l = 0; l < L; ++l) {
            LayerW& w = c->layers[l];
            const std::string p = "enc.1.encoders." + std::to_string(l) + ".";
            const HostTensor *q, *k, *v, *bq, *bk, *bv;
            FO_TRY(need(c, p + "self_attn.linear_q.weight", {D, D}, &q));
            FO_TRY(need(c, p + "self_attn.linear_k.weight", {D, D}, &k));
            FO_TRY(need(c, p + "self_attn.linear_v.weight", {D, D}, &v));
            FO_TRY(need(c, p + "self_attn.linear_q.bias", {D}, &bq));
            FO_TRY(need(c, p + "self_attn.linear_k.bias", {D}, &bk));
            FO_TRY(need(c, p + "self_attn.linear_v.bias", {D}, &bv));
            FO_TRY(dev_alloc(c, &w.wqkv, (size_t)3 * D * D * sizeof(TW)));
            TW* wq = reinterpret_cast<TW*>(w.wqkv);
            FO_TRY(convert_weight<TW>(q->d, (long long)D * D, wq, 0));
            FO_TRY(convert_weight<TW>(k->d, (long long)D * D, wq + (size_t)D * D, 0));
            FO_TRY(convert_weight<TW>(v->d, (long long)D * D, wq + (size_t)2 * D * D, 0));
            void* bq3;
            FO_TRY(dev_alloc(c, &bq3, (size_t)3 * D * sizeof(float)));
            w.bqkv = reinterpret_cast<float*>(bq3);
            FO_CUDA(cudaMemcpy(w.bqkv, bq->d, D * sizeof(float), cudaMemcpyDeviceToDevice));
            FO_CUDA(cudaMemcpy(w.bqkv + D, bk->d, D * sizeof(float), cudaMemcpyDeviceToDevice));
            FO_CUDA(cudaMemcpy(w.bqkv + 2 * D, bv->d, D * sizeof(float), cudaMemcpyDeviceToDevice));
            FO_TRY(keep_w<TW>(c, p + "self_attn.linear_out.weight", {D, D}, &w.wo));
            FO_TRY(keep_f32(c, p + "self_attn.linear_out.bias", {D}, &w.bo));
            FO_TRY(keep_f32(c, p + "self_attn.pos_bias_u", {H, 64}, &w.pos_u));
            FO_TRY(keep_f32(c, p + "self_attn.pos_bias_v", {H, 64}, &w.pos_v));
            if (c->KF >= 2) {                         // Conv1dLinear (attention.py:217-233)
                FO_TRY(keep_f32(c, p + "feed_forward.w_1.0.weight", {D, 1, c->KF}, &w.dw_w));
                FO_TRY(keep_f32(c, p + "feed_forward.w_1.0.bias", {D}, &w.dw_b));
                FO_TRY(keep_w<TW>(c, p + "feed_forward.w_1.1.weight", {FF, D, 1}, &w.w1));
                FO_TRY(keep_f32(c, p + "feed_forward.w_1.1.bias", {FF}, &w.b1));
            } else if (c->KM) {                        // MultiLayeredConv1d: both convolutions as implicit GEMMs, [co][tau * Cin + ci]
                const HostTensor* t;
                FO_TRY(need(c, p + "feed_forward.w_1.weight", {FF, D, c->KM}, &t));
                FO_TRY(dev_alloc(c, &w.w1, (size_t)FF * D * c->KM * sizeof(TW)));
                FO_TRY(repack_adapter_conv<TW>(t->d, FF, D, c->KM, reinterpret_cast<TW*>(w.w1), 0));
                FO_TRY(keep_f32(c, p + "feed_forward.w_1.bias", {FF}, &w.b1));
                FO_TRY(need(c, p + "feed_forward.w_2.weight", {D, FF, c->KM}, &t));
                FO_TRY(dev_alloc(c, &w.w2, (size_t)FF * D * c->KM * sizeof(TW)));
                FO_TRY(repack_adapter_conv<TW>(t->d, D, FF, c->KM, reinterpret_cast<TW*>(w.w2), 0));
            } else {
                FO_TRY(keep_w<TW>(c, p + "feed_forward.w_1.weight", {FF, D}, &w.w1));
                FO_TRY(keep_f32(c, p + "feed_forward.w_1.bias", {FF}, &w.b1));
            }
            if (!c->KM) FO_TRY(keep_w<TW>(c, p + "feed_forward.w_2.weight", {D, FF}, &w.w2));
            FO_TRY(keep_f32(c, p + "feed_forward.w_2.bias", {D}, &w.b2));
            FO_TRY(keep_f32(c, p + "norm1.weight", {D}, &w.ln1g));
            FO_TRY(keep_f32(c, p + "norm1.bias", {D}, &w.ln1b));
            FO_TRY(keep_f32(c, p + "norm2.weight", {D}, &w.ln2g));
            FO_TRY(keep_f32(c, p + "norm2.bias", {D}, &w.ln2b));
            if (g.concat_after) {
                FO_TRY(keep_w<TW>(c, p + "concat_linear.weight", {D, 2 * D}, &w.wcat));
                FO_TRY(keep_f32(c, p + "concat_linear.bias", {D}, &w.bcat));
            }
            // P_l = pe * Wpos^T  (attention.py:433): a function of the weights only, so it is tabulated once
            // instead of per layer per chunk.  fp32 FFMA GEMM over the fp32 sin/cos table and the weights as
            // the context holds them (rounded to bf16 in a bf16 context); the table stays fp32.
            const HostTensor* wp;
            FO_TRY(need(c, p + "self_attn.linear_pos.weight", {D, D}, &wp));
            float* wpos;
            FO_CUDA(cudaMalloc((void**)&wpos, (size_t)D * D * sizeof(float)));
            int r = 0;
            if (sizeof(TW) == 2) {
                bf16* w16;
                if (cudaMalloc((void**)&w16, (size_t)D * D * sizeof(bf16)) != cudaSuccess) r = FO_ERR_NOMEM;
                if (r == 0) r = f32_to_bf16(wp->d, w16, (long long)D * D, 0);
                if (r == 0) r = bf16_to_f32(w16, wpos, (long long)D * D, 0);
                cudaDeviceSynchronize();
                cudaFree(w16);
            } else {
                if (cudaMemcpy(wpos, wp->d, (size_t)D * D * sizeof(float), cudaMemcpyDeviceToDevice) != cudaSuccess) r = FO_ERR_CUDA;
            }
            void* pt = nullptr;
            if (r == 0) r = dev_alloc(c, &pt, (size_t)c->pos_rows * D * sizeof(float));
            w.ptab = reinterpret_cast<float*>(pt);
            if (r == 0) {
                Epilogue ep;
                ep.c_f32 = w.ptab;
                ep.ldc = D;
                r = gemm_simt<float, float>(pe_rows, plain_rows(D, c->pos_rows), wpos, c->pos_rows, D, D, ep, RowMap(), 0);
            }
            if (r == 0) r = dev_alloc(c, &w.ptab_h, (size_t)c->pos_rows * D * (sizeof(TW) == 2 ? 2 : 4));
            if (r == 0) {
                if (sizeof(TW) == 2) r = ptab_head_major<act16>(w.ptab, c->pos_rows, H, reinterpret_cast<act16*>(w.ptab_h), 0);
                else r = ptab_head_major<float>(w.ptab, c->pos_rows, H, reinterpret_cast<float*>(w.ptab_h), 0);
            }
            cudaDeviceSynchronize();
            cudaFree(wpos);
            FO_TRY(r);
        }
        if (!g.post_norm) {                   // transformer.py:232-233: after_norm exists only with normalize_before
            FO_TRY(keep_f32(c, "enc.1.after_norm.weight", {D}, &c->after_g));
            FO_TRY(keep_f32(c, "enc.1.after_norm.bias", {D}, &c->after_b));
        }
        // frontend constants
        if (staged(c, "fbank.window")) {
            FO_TRY(keep_f32(c, "fbank.window", {g.frame_len}, &c->fb_window));
            FO_TRY(keep_f32(c, "fbank.mel", {F, c->fft / 2 + 1}, &c->fb_mel));
            std::vector<float> mel((size_t)F * (c->fft / 2 + 1));
            FO_CUDA(cudaMemcpy(mel.data(), c->fb_mel, mel.size() * sizeof(float), cudaMemcpyDeviceToHost));
            std::vector<int> lo(F), hi(F);
            const int nb = c->fft / 2 + 1;
            for (int m = 0; m < F; ++m) {
                int a = nb, b = 0;
                for (int k = 0; k < nb; ++k)
                    if (mel[(size_t)m * nb + k] != 0.f) { if (k < a) a = k; b = k + 1; }
                if (a > b) a = b = 0;
                lo[m] = a;
                hi[m] = b;
            }
            void *dlo, *dhi;
            FO_TRY(dev_alloc(c, &dlo, F * sizeof(int)));
            FO_TRY(dev_alloc(c, &dhi, F * sizeof(int)));
            FO_CUDA(cudaMemcpy(dlo, lo.data(), F * sizeof(int), cudaMemcpyHostToDevice));
            FO_CUDA(cudaMemcpy(dhi, hi.data(), F * sizeof(int), cudaMemcpyHostToDevice));
            c->fb_lo = reinterpret_cast<int*>(dlo);
            c->fb_hi = reinterpret_cast<int*>(dhi);
        }
    }
    if (g.has_adapter) {
        // eval-mode BatchNorm1d(eps 1e-3) as a per-channel affine map of the running statistics (adapter.py:25-26,87,92,100-101):
        // y = (x - mean) / sqrt(var + 1e-3) * gamma + beta = x * s + (beta - mean * s); folded once, in double
        auto keep_bn = [&](const std::string& name, int n, float** gam_d, float** bet_d, bool fold) -> int {
            FO_TRY(keep_f32(c, "adapter." + name + ".weight", {n}, gam_d));
            FO_TRY(keep_f32(c, "adapter." + name + ".bias", {n}, bet_d));
            if (!fold) return 0;
            const HostTensor *rm, *rv;
            FO_TRY(need(c, "adapter." + name + ".running_mean", {n}, &rm));
            FO_TRY(need(c, "adapter." + name + ".running_var", {n}, &rv));
            std::vector<float> gam(n), bet(n), mean(n), var(n);
            FO_CUDA(cudaMemcpy(gam.data(), *gam_d, n * sizeof(float), cudaMemcpyDeviceToHost));
            FO_CUDA(cudaMemcpy(bet.data(), *bet_d, n * sizeof(float), cudaMemcpyDeviceToHost));
            FO_CUDA(cudaMemcpy(mean.data(), rm->d, n * sizeof(float), cudaMemcpyDeviceToHost));
            FO_CUDA(cudaMemcpy(var.data(), rv->d, n * sizeof(float), cudaMemcpyDeviceToHost));
            for (int i = 0; i < n; ++i) {
                const double sc = (double)gam[i] / sqrt((double)var[i] + 1e-3);
                gam[i] = (float)sc;
                bet[i] = (float)((double)bet[i] - (double)mean[i] * sc);
            }
            FO_CUDA(cudaMemcpy(*gam_d, gam.data(), n * sizeof(float), cudaMemcpyHostToDevice));
            FO_CUDA(cudaMemcpy(*bet_d, bet.data(), n * sizeof(float), cudaMemcpyHostToDevice));
            return 0;
        };
        auto keep_conv = [&](const std::string& name, fo_ctx::AdStage& s) -> int {
            const HostTensor* t;
            FO_TRY(need(c, "adapter." + name + ".weight", {s.cout, s.cin, KA}, &t));
            FO_TRY(dev_alloc(c, &s.w, (size_t)s.cout * s.cin * KA * sizeof(TW)));
            FO_TRY(repack_adapter_conv<TW>(t->d, s.cout, s.cin, KA, reinterpret_cast<TW*>(s.w), 0));
            return keep_f32(c, "adapter." + name + ".bias", {s.cout}, &s.b);
        };
        // two convs: conv1d1 + bn1 + ReLU, then conv1d2 + bn2 + ReLU; one conv: conv1d2 + bn2 (LayerNorm or BatchNorm)
        const int ns = c->ad_nst;
        if (ns == 2) {
            FO_TRY(keep_conv("conv1d1", c->ad_st[0]));
            FO_TRY(keep_bn("bn1", c->ad_st[1].cin, &c->ad_st[1].in_scale, &c->ad_st[1].in_shift, true));
        }
        if (ns > 0) {
            FO_TRY(keep_conv("conv1d2", c->ad_st[ns - 1]));
            FO_TRY(keep_bn("bn2", c->ad_st[ns - 1].cout, &c->ad_ln_g, &c->ad_ln_b, c->ad_ln_eps < 0.f));
        }
        const std::string proj = ns > 0 ? "adapter.project" : "adapter.adpter";    // LinearAdapter's module name, spelt as such
        FO_TRY(keep_w<TW>(c, proj + ".weight", {E, ns > 0 ? c->ad_st[ns - 1].cout : D}, &c->ad_proj_w));
        FO_TRY(keep_f32(c, proj + ".bias", {E}, &c->ad_proj_b));
    }
    FO_CUDA(cudaDeviceSynchronize());
    for (auto& kv : c->staged) cudaFree(kv.second.d);
    c->staged.clear();
    c->finalized = true;
    return 0;
}

FbankParams fbank_params(fo_ctx* c) {
    FbankParams p;
    p.frame_len = c->cfg.frame_len;
    p.frame_shift = c->cfg.frame_shift;
    p.fft_size = c->fft;
    p.n_mel = c->F;
    p.window = c->fb_window;
    p.mel = c->fb_mel;
    p.mel_lo = c->fb_lo;
    p.sms = c->sms;
    p.mel_hi = c->fb_hi;
    return p;
}

// frames out of the first n adapter convolutions (default: all) for T encoder frames.  A causal conv over k-1 cached / padded
// frames maps T frames to (T - 1) / stride + 1 (adapter.py:137-144); LinearAdapter keeps the frame rate (adapter.py:69-70).
inline int ad_frames(const fo_ctx* c, int T, int n = -1) {
    for (int i = 0; i < (n < 0 ? c->ad_nst : n); ++i) T = (T - 1) / c->ad_st[i].stride + 1;
    return T;
}

// Where the adapter's projection writes: fp32 rows of y, or fp16 rows of an LLM hand-off buffer (audioLLM.py:404-411), base
// past the prefix.  The rows are (session, k chunks, t_out frames); row r of chunk j of session b goes to row r of output
// block b * k + j, blocks `pitch` rows apart.  Into y they are plain row-major.
struct AdOut {
    float* y = nullptr;
    void* h16 = nullptr;      // instead of y
    long long pitch = 0;      // rows per output block
    int k = 1;
};

// RowMap of the projection onto o's blocks, t_out rows per chunk
inline void chunk_rowmap(const AdOut& o, int t_out, RowMap* rm) {
    rm->p1 = o.k * t_out; rm->p0 = t_out; rm->v1 = o.k; rm->v0 = t_out; rm->q1 = (int)(o.k * o.pitch); rm->q0 = (int)o.pitch;
}

// ---- adapter program on device buffers -----------------------------------------------------------
// enc (B, T, D) fp32 -> B * t_out rows of E at `out`.  Each conv: conv_stage builds its A operand from [left context | input
// rows] (the mask on the first conv's input, the previous conv's folded BatchNorm + ReLU on a later one), then an implicit
// GEMM into fp32; the last conv's rows are normalised and projected.  LinearAdapter projects the encoder rows as they are
// (the reference does not even apply the pad mask).  Left context: the slot caches of ids_dev when the adapter carries them,
// else per stage cache_in[i] (reference layout (B, C, k-1); null = zeros), the new one to cache_out[i] if given.
// mix (carried caches, chunks of sessions with different counts or odd t): enc holds the call's blocks packed, session b's
// cnt[b] chunks of `unit` frames from block off[b].  The convolutions run over B sessions x T = kmax * unit rows, padded at
// the end of each session's run (the conv is causal, so the real rows' outputs are those of the sequential calls); the
// real output rows are packed to (block, frame) order before the norm and the projection.  pick (odd t): every conv at
// stride 1, then the rows of the stride-2 outputs picked per chunk.
struct AdMix {
    const int32_t* cnt;
    const int32_t* off;
    int kmax, unit, blocks;
    bool pick;
};
// pack (fo_encode_offline_packed): enc holds B utterances packed end to end, utterance b's rows from enc_off[b]; cnt[i * B + b]
// = its rows into conv i, cnt[ns * B + b] its output rows, which go to out.y packed from off[b] (`rows` in all).  The convs run
// over a grid of B x T rows (T = the longest utterance): each utterance from the first row of its run, with zero left context
// (so the stride-2 phase starts at its first frame) and zeros behind it.
struct AdPack {
    const int32_t* cnt;
    const int32_t* enc_off;
    const int32_t* off;
    int rows;
};
template <typename TA>
int adapter_program(fo_ctx* c, const float* enc, const uint8_t* mask, int B, int T, const int32_t* ids_dev,
                    const float* const* cache_in, float* const* cache_out, const AdOut& out, cudaStream_t st,
                    const AdMix* mix = nullptr, const AdPack* pack = nullptr) {
    const int D = c->D, E = c->E, KA = c->KA, ns = c->ad_nst;
    const bool grid = mix != nullptr;                                          // per-session padded grid
    const int t_out = grid ? ad_frames(c, mix->unit) : ad_frames(c, T);       // grid: frames out of one chunk
    const int M = pack ? pack->rows : grid ? mix->blocks * t_out : B * t_out;
    const bool run_gemm = !(c->debug_skip & 16);
    const float* x = enc;
    const bool pick = grid && mix->pick;
    for (int i = 0; i < ns; ++i) {
        const fo_ctx::AdStage& s = c->ad_st[i];
        const int stride = pick ? 1 : s.stride;
        const int Ti = pick ? T : ad_frames(c, T, i);
        AGather ga;
        RowMap rm;
        if (stride == 1) conv1d_gather(B, Ti, s.cin, KA, &ga, &rm);
        else adapter_gather(B, Ti, s.cin, KA, &ga, &rm);
        void *xin, *conv;
        FO_TRY(ws_ensure(c, i == 0 ? WS_XIN : WS_XIN2, (size_t)ga.planes * ga.rows * s.cin * sizeof(TA), &xin));
        FO_TRY(ws_ensure(c, i + 1 == ns ? WS_ACONV : WS_AC1, (size_t)B * (pick ? T : ad_frames(c, T, i + 1)) * s.cout * sizeof(float), &conv));
        SessionRows sr;
        if (grid) {
            sr.cnt = mix->cnt;
            sr.off = i == 0 ? mix->off : nullptr;          // the first conv reads the packed encoder rows
            sr.unit = pick ? mix->unit : ad_frames(c, mix->unit, i);
        } else if (pack) {
            sr.cnt = pack->cnt + (long long)i * B;
            sr.off = i == 0 ? pack->enc_off : nullptr;
            sr.unit = 1;
        }
        FO_TRY(conv_stage<TA>(x, i == 0 ? mask : nullptr, B, Ti, s.cin, KA - 1, stride, s.in_scale, s.in_shift,
                              c->ad_carry ? ids_dev : nullptr, s.cache, c->ad_valid, cache_in ? cache_in[i] : nullptr,
                              cache_out ? cache_out[i] : nullptr, reinterpret_cast<TA*>(xin), st, sr));
        Epilogue e;
        e.bias = s.b;
        e.c_f32 = reinterpret_cast<float*>(conv);
        e.ldc = s.cout;
        if (run_gemm) FO_TRY(gemm<TA>(c, reinterpret_cast<const TA*>(xin), ga, s.w, (int)ga.rows, s.cout, KA * s.cin, e, rm, st));
        x = reinterpret_cast<const float*>(conv);
    }
    const int K = ns > 0 ? c->ad_st[ns - 1].cout : D;
    if (grid && ns > 0) {
        void* pk;
        FO_TRY(ws_ensure(c, WS_PACK, (size_t)M * K * sizeof(float), &pk));
        if (pick) FO_TRY(pick_chunk_rows(x, B, mix->kmax, mix->unit, t_out, K, mix->cnt, mix->off, reinterpret_cast<float*>(pk), st));
        else FO_TRY(pack_session_blocks(x, reinterpret_cast<float*>(pk), (long long)t_out * K * sizeof(float), B, mix->kmax, mix->cnt,
                                        mix->off, st));
        x = reinterpret_cast<const float*>(pk);
    } else if (pack && ns > 0) {
        void* pk;
        FO_TRY(ws_ensure(c, WS_PACK, (size_t)M * K * sizeof(float), &pk));
        FO_TRY(pack_session_blocks(x, reinterpret_cast<float*>(pk), (long long)K * sizeof(float), B, ad_frames(c, T),
                                   pack->cnt + (long long)ns * B, pack->off, st));
        x = reinterpret_cast<const float*>(pk);
    }
    const TA* a = reinterpret_cast<const TA*>(enc);
    if (ns > 0 || sizeof(TA) == 2) {                 // the projection's operand in the activation type
        void* ah;
        FO_TRY(ws_ensure(c, ns > 0 ? WS_AH : WS_XIN, (size_t)M * K * sizeof(TA), &ah));
        if (ns > 0) FO_TRY(layer_norm<TA>(x, M, K, c->ad_ln_g, c->ad_ln_b, c->ad_ln_eps, c->ad_ln_act, 1.0f, reinterpret_cast<TA*>(ah), nullptr, st));
        else FO_TRY(f32_to_act16(enc, reinterpret_cast<act16*>(ah), (long long)M * D, st));
        a = reinterpret_cast<const TA*>(ah);
    }
    Epilogue e;
    e.bias = c->ad_proj_b;
    e.ldc = E;
    RowMap rm;
    if (out.h16) chunk_rowmap(out, grid ? t_out : t_out / out.k, &rm);
    if (out.h16) e.c_act = reinterpret_cast<TA*>(out.h16);     // straight from the epilogue: no fp32 copy, no .half()
    else e.c_f32 = out.y;
    if (run_gemm) FO_TRY(gemm<TA>(c, a, plain_rows(K, M), c->ad_proj_w, M, E, K, e, rm, st));
    return 0;
}

// ---- encoder trunk shared by streaming and offline ------------------------------------------------
// feats (B, T, F) fp32 device.  Produces the residual stream x (M, D) after `embed` and pos scaling.
template <typename TA>
int subsample_program(fo_ctx* c, const float* feats, int B, int T, float** x_out, cudaStream_t st) {
    const int D = c->D, F = c->F, F1 = c->F1, F2 = c->F2;
    const int T1 = (T - 1) / 2, T2 = (T1 - 1) / 2, M = B * T2;
    void *c1, *c2, *xsub, *emb, *x;
    AGather ga;
    RowMap rm;
    conv2_gather(B, T2, F2, D, &ga, &rm);
    FO_TRY(ws_ensure(c, WS_C1, (size_t)ga.planes * ga.rows * D * sizeof(TA), &c1));
    FO_TRY(ws_ensure(c, WS_C2, (size_t)M * F2 * D * sizeof(TA), &c2));
    FO_TRY(ws_ensure(c, WS_X, (size_t)M * D * sizeof(float), &x));
    FO_TRY(cmvn_conv1<TA>(feats, B, T, F, c->cmvn_mean, c->cmvn_istd, c->conv1_w, c->conv1_b, D,
                          reinterpret_cast<TA*>(c1), st));
    Epilogue e;
    e.bias = c->conv2_b;
    e.relu = 1;
    e.c_act = c2;
    e.ldc = D;
    if (!(c->debug_skip & 16)) FO_TRY(gemm<TA>(c, reinterpret_cast<const TA*>(c1), ga, c->conv2_w, (int)ga.rows, D, 9 * D, e, rm, st));
    const float xscale = sqrtf((float)D);
    if (c->cfg.input_layer_linear) {
        FO_TRY(ws_ensure(c, WS_XSUB, (size_t)M * D * sizeof(TA), &xsub));
        FO_TRY(ws_ensure(c, WS_EMB, (size_t)M * D * sizeof(float), &emb));
        Epilogue e2;
        e2.bias = c->sub_b;
        e2.c_act = xsub;
        e2.ldc = D;
        if (!(c->debug_skip & 16)) FO_TRY(gemm<TA>(c, reinterpret_cast<const TA*>(c2), c->sub_w, M, D, F2 * D, e2, st));
        Epilogue e3;
        e3.bias = c->emb_b;
        e3.c_f32 = reinterpret_cast<float*>(emb);
        e3.ldc = D;
        if (!(c->debug_skip & 16)) FO_TRY(gemm<TA>(c, reinterpret_cast<const TA*>(xsub), c->emb_w, M, D, D, e3, st));
        FO_TRY(layer_norm<TA>(reinterpret_cast<const float*>(emb), M, D, c->emb_g, c->emb_beta, 1e-5f, 1, xscale, nullptr,
                              reinterpret_cast<float*>(x), st));
    } else {
        Epilogue e2;
        e2.bias = c->sub_b;
        e2.c_f32 = reinterpret_cast<float*>(x);
        e2.ldc = D;
        e2.scale = xscale;
        FO_TRY(gemm<TA>(c, reinterpret_cast<const TA*>(c2), c->sub_w, M, D, F2 * D, e2, st));
    }
    *x_out = reinterpret_cast<float*>(x);
    return 0;
}

// One transformer layer minus the attention core.  LayerNorms ride on the GEMM that completes the residual stream:
// out-proj (+residual) -> norm2 -> h;  FFN2 (+residual) -> next layer's norm1 -> h, or after_norm -> encoder output.
struct NextNorm {
    const float* gamma;
    const float* beta;
    float* out_f32;          // after_norm of the last layer: fp32 encoder output rows (else null -> h)
};
// fp32 rows -> the activation type of the context (post-norm layers feed the un-normalised layer input to the GEMMs)
template <typename TA> int to_act(const float* x, TA* y, long long n, cudaStream_t st);
template <> int to_act<float>(const float* x, float* y, long long n, cudaStream_t st) { return scale_rows(x, y, n, 1.0f, st); }
template <> int to_act<act16>(const float* x, act16* y, long long n, cudaStream_t st) { return f32_to_act16(x, y, n, st); }
inline L2Prefetch pf1(const void* p, long long bytes) {
    L2Prefetch f;
    f.ptr[0] = p; f.bytes[0] = bytes;
    return f;
}
template <typename TA>
int layer_pre(fo_ctx* c, const LayerW& w, int M, TA* h, TA* qkv, float* q32, const L2Prefetch& pf, cudaStream_t st,
              int* deferred = nullptr) {
    const int D = c->D;
    if (deferred) *deferred = 0;
    if (c->debug_skip & 4) return 0;
    Epilogue e;
    e.prefetch = pf;
    e.bias = w.bqkv;
    e.c_act = qkv;
    e.ldc = 3 * D;
    if (sizeof(TA) == 2) {            // bf16 context: Q stays fp32 (columns < D), K|V are written as bf16
        e.c_f32 = q32;
        e.split_col = D;
    }
    static int qkv_defer_max_rows = -1;
    if (qkv_defer_max_rows < 0) { const char* e0 = getenv("FO_QKV_DEFER_MAXM"); qkv_defer_max_rows = e0 ? atoi(e0) : 128; }
    // streaming, few rows: the attention kernel finishes a split-K sum of the QKV GEMM while it loads its rows (r102: -7 % of
    // the step at 1 session, -1 % at 32; at 64 sessions the fp32 partial traffic costs more than the finer K split gains: +4 %)
    if (deferred && sizeof(TA) == 2 && M <= qkv_defer_max_rows) {
        e.defer_reduce = 2;
        return gemm<TA>(c, h, plain_rows(D, M), w.wqkv, M, 3 * D, D, e, RowMap(), st, deferred);
    }
    return gemm<TA>(c, h, w.wqkv, M, 3 * D, D, e, st);
}
struct FfnConv {                  // Conv1dLinear only: where the rows come from
    int B = 0, T = 0;             // rows = B * T (per-session counts: T = the largest session's rows)
    const int32_t* cnt = nullptr; // streaming with per-session chunk counts (depthwise_conv)
    const int32_t* off = nullptr;
    int t = 0;
    const int32_t* ids = nullptr; // streaming: session slots (left context carried); offline: null (zero padding)
    int layer = 0;
    void* hc = nullptr;           // depthwise output buffer (M, D), activation type
    void* hp = nullptr;           // MultiLayeredConv1d: zero-padded layer input (B, T + k - 1, D) and hidden rows (B, T + k - 1, FF)
    void* fp = nullptr;
    // MultiLayeredConv1d over packed utterances (B = 1, T = all rows): k - 1 rows between two utterances, from row gap_at[i],
    // are zeroed in both padded buffers, so each utterance sees (k-1)/2 zero rows on either side
    const int32_t* gap_at = nullptr;
    int n_gaps = 0;
};
template <typename TA>
int layer_post(fo_ctx* c, const LayerW& w, float* x, int M, TA* att, TA* h, TA* ffh, const NextNorm& nn,
               const void* next_wqkv, const FfnConv& fc, cudaStream_t st) {
    const int D = c->D, FF = c->FF;
    const long long wsz = (long long)c->esz;
    // transformer-normalize-before: false -> the LayerNorms follow the residual adds (norm1 after attention, norm2 after the
    // feed-forward, transformer.py:89-90,97-98,117-118,127-128): the normalised rows replace the residual stream AND feed the
    // next GEMM.  transformer-concat-after -> x + concat_linear(cat(layer input, att)) (transformer.py:85-87,108-113): linear_out
    // writes its rows behind the layer input (`h` is then a [2][M][D] pair of planes) and concat_linear reads both as ONE K = 2D operand.
    const bool post = c->cfg.post_norm != 0, cat = c->cfg.concat_after != 0;
    Epilogue e;
    if (c->use_prefetch & 1) e.prefetch = pf1(w.w2, (long long)D * FF * wsz);       // out-proj runs: FFN2's weights
    e.bias = cat ? w.bcat : w.bo;
    e.residual = x;
    e.c_f32 = x;
    e.ldc = D;
    e.ln_gamma = post ? w.ln1g : w.ln2g;
    e.ln_beta = post ? w.ln1b : w.ln2b;
    e.ln_act = h;
    if (post) e.ln_f32 = x;
    if (!(c->debug_skip & 4)) {
        if (cat) {
            Epilogue eo;
            eo.bias = w.bo;
            eo.c_act = h + (long long)M * D;                      // plane 1 of the concat operand
            eo.ldc = D;
            FO_TRY(gemm<TA>(c, att, w.wo, M, D, D, eo, st));
            AGather ga = plain_rows(D, M);
            ga.n_seg = 2; ga.planes = 2; ga.plane[1] = 1;
            FO_TRY(gemm<TA>(c, h, ga, w.wcat, M, D, 2 * D, e, RowMap(), st));
        } else {
            FO_TRY(gemm<TA>(c, att, w.wo, M, D, D, e, st));
        }
    }
    if (c->debug_skip & 8) return 0;
    const TA* ffn_in = h;
    if (c->KF >= 2) {
        // Conv1dLinear: causal depthwise conv over time on norm2's output, then the 1x1 conv is the FFN1 GEMM
        const long long slot_stride = (long long)c->L * (c->KF - 1) * D;
        FO_TRY(depthwise_conv<TA>(h, fc.B, fc.T, D, c->KF, w.dw_w, w.dw_b, fc.ids,
                                  c->ffn_cache + (long long)fc.layer * (c->KF - 1) * D, slot_stride,
                                  reinterpret_cast<TA*>(fc.hc), st, fc.cnt, fc.off, fc.t));
        ffn_in = reinterpret_cast<const TA*>(fc.hc);
    }
    Epilogue e1;
    if ((c->use_prefetch & 1) && next_wqkv) e1.prefetch = pf1(next_wqkv, 3LL * D * D * wsz);   // FFN1 runs: next layer's QKV weights
    e1.bias = w.b1;
    e1.relu = 1;
    e1.c_act = ffh;
    e1.ldc = FF;
    AGather ga2 = plain_rows(FF, M);
    RowMap rm2;
    const TA* ffn2_in = ffh;
    int M2 = M, K2 = FF;
    if (c->KM) {
        // MultiLayeredConv1d (attention.py:158-196): both Conv1d(k, padding (k-1)/2) as implicit GEMMs over zero-padded rows;
        // the first writes its ReLU rows at offset (k-1)/2 of the (pre-zeroed) padded hidden buffer, i.e. already padded for the second
        const int k = c->KM, lead = (k - 1) / 2, R1 = fc.T + k - 1;
        TA* hp = reinterpret_cast<TA*>(fc.hp);
        TA* fp = reinterpret_cast<TA*>(fc.fp);
        FO_TRY(pad_rows<TA>(h, fc.B, fc.T, D, lead, k - 1 - lead, hp, st));
        FO_TRY(zero_row_runs<TA>(hp + (long long)lead * D, fc.gap_at, fc.n_gaps, k - 1, D, st));
        AGather ga1;
        RowMap rm1;
        conv1d_gather(fc.B, fc.T, D, k, &ga1, &rm1);
        rm1.q1 = R1;                                           // output rows stay on the padded grid ...
        e1.c_act = fp + (long long)lead * FF;                  // ... shifted past the leading zero rows
        FO_TRY(gemm<TA>(c, hp, ga1, w.w1, (int)ga1.rows, FF, k * D, e1, rm1, st));
        FO_TRY(zero_row_runs<TA>(fp + (long long)lead * FF, fc.gap_at, fc.n_gaps, k - 1, FF, st));
        conv1d_gather(fc.B, fc.T, FF, k, &ga2, &rm2);
        ffn2_in = fp;
        M2 = (int)ga2.rows;
        K2 = k * FF;
    } else {
        FO_TRY(gemm<TA>(c, ffn_in, w.w1, M, FF, D, e1, st));
    }
    Epilogue e2;
    e2.bias = w.b2;
    e2.residual = x;
    e2.c_f32 = x;
    e2.ldc = D;
    e2.ln_gamma = post ? w.ln2g : nn.gamma;
    e2.ln_beta = post ? w.ln2b : nn.beta;
    if (nn.out_f32) e2.ln_f32 = nn.out_f32;               // last layer: the encoder output rows
    else { e2.ln_act = h; if (post) e2.ln_f32 = x; }
    return gemm<TA>(c, ffn2_in, ga2, w.w2, M2, D, K2, e2, rm2, st);
}

// All layers of a small streaming step in one cooperative launch (fo_stack.cu).  Returns 1 when the step does not qualify
// (rows, layer options, dimensions) and the per-kernel chain has to run.
int stack_program(fo_ctx* c, int n, int t, float* x, void* qkv, float* q32, void* att, void* ffh, float* enc_out_dev,
                  cudaStream_t st) {
    const int D = c->D, H = c->H;
    if (c->dtype != FO_BF16 || c->stack_rows <= 0 || n * t > std::min(c->stack_rows, (int)STACK_MAX_ROWS)) return 1;
    if (c->cfg.post_norm || c->cfg.concat_after || c->KF >= 2 || c->KM || c->debug_skip || c->profile_gemm) return 1;
    const long long layer_stride = (long long)c->cfg.max_sessions * 2LL * H * c->ring_cap * 64;
    if (!c->stack_layers) {
        // the kernel reads its own copy of the four layer matrices with every row padded by 16 bytes (one bulk copy per
        // weight slice, bank-conflict-free fragments, fo_stack.cu:load_rows): +604 MB for the shipped model, built at the
        // first step that qualifies
        auto padded = [&](const void* src, int rows, int K, const __half** out) -> int {
            void* d;
            FO_TRY(dev_alloc(c, &d, (size_t)rows * (K * 2 + 16)));
            FO_CUDA(cudaMemcpy2D(d, (size_t)K * 2 + 16, src, (size_t)K * 2, (size_t)K * 2, rows, cudaMemcpyDeviceToDevice));
            *out = reinterpret_cast<const __half*>(d);
            return 0;
        };
        std::vector<StackLayer> tab(c->L);
        for (int l = 0; l < c->L; ++l) {
            const LayerW& w = c->layers[l];
            StackLayer& s = tab[l];
            FO_TRY(padded(w.wqkv, 3 * D, D, &s.wqkv));
            FO_TRY(padded(w.wo, D, D, &s.wo));
            FO_TRY(padded(w.w1, c->FF, D, &s.w1));
            FO_TRY(padded(w.w2, D, c->FF, &s.w2));
            s.bqkv = w.bqkv; s.bo = w.bo; s.b1 = w.b1; s.b2 = w.b2;
            s.ln1g = w.ln1g; s.ln1b = w.ln1b; s.ln2g = w.ln2g; s.ln2b = w.ln2b; s.pos_u = w.pos_u; s.pos_v = w.pos_v;
            s.ptab_h = reinterpret_cast<const __half*>(w.ptab_h);
            s.ring = reinterpret_cast<__half*>(c->ring) + l * layer_stride;
        }
        void *pt, *pb, *ptr;
        FO_TRY(dev_alloc(c, &pt, tab.size() * sizeof(StackLayer)));
        FO_TRY(dev_alloc(c, &pb, 4096));
        FO_TRY(dev_alloc(c, &ptr, (size_t)(35 * c->L + 8 + 16384) * sizeof(unsigned long long)));
        FO_CUDA(cudaMemcpy(pt, tab.data(), tab.size() * sizeof(StackLayer), cudaMemcpyHostToDevice));
        FO_CUDA(cudaMemset(pb, 0, 4096));
        FO_CUDA(cudaMemset(ptr, 0, (size_t)(35 * c->L + 8 + 16384) * sizeof(unsigned long long)));
        FO_CUDA(cudaDeviceSynchronize());               // the copies above ran on the default stream
        c->stack_bar = reinterpret_cast<unsigned int*>(pb);
        c->stack_trace = reinterpret_cast<unsigned long long*>(ptr);
        c->stack_layers = reinterpret_cast<StackLayer*>(pt);
    }
    StackArgs s;
    s.layers = c->stack_layers;
    s.L = c->L; s.D = D; s.FF = c->FF;
    s.a.ids = c->ids_dev;
    s.a.n_frames = c->n_frames;
    s.a.pe_index = c->pe_index;
    s.a.n = n; s.a.t = t; s.a.H = H; s.a.ring_cap = c->ring_cap; s.a.window = c->window; s.a.full_chunk = c->full_chunk;
    s.a.pe_wrap = c->pe_wrap; s.a.pos_rows = c->pos_rows;
    s.a.ring_slot_stride = 2LL * H * c->ring_cap * 64;
    s.x = x;
    s.q32 = q32;
    s.kv = reinterpret_cast<__half*>(qkv);
    s.att = reinterpret_cast<__half*>(att);
    s.ffh = reinterpret_cast<__half*>(ffh);
    s.after_g = c->after_g; s.after_b = c->after_b;
    s.enc_out = enc_out_dev;
    s.bar = c->stack_bar;
    s.sat = c->sat_counter;
    static int want_trace = -1;
    if (want_trace < 0) want_trace = getenv("FO_STACK_TRACE") ? 1 : 0;
    s.trace = want_trace ? c->stack_trace : nullptr;
    if (!c->coop) return 1;
    const int r = stream_stack(s, c->sms, c->smem_optin, st);
    if (r != 0) return r;
    c->stack_launches += 1;
    if (want_trace) {
        cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
        cudaStreamIsCapturing(st, &cs);
        if (cs == cudaStreamCaptureStatusNone) {
            std::vector<unsigned long long> hb(35 * c->L + 8 + 16384);
            FO_CUDA(cudaStreamSynchronize(st));
            FO_CUDA(cudaMemcpy(hb.data(), c->stack_trace, hb.size() * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
            const int lm = c->L / 2;
            fprintf(stderr, "stack_trace n=%d total=%.2f us; layer %d (qkv attn out ffn1 ffn2) ns:", n, (hb[5 * c->L + 1] - hb[0]) * 1e-3, lm);
            for (int q = 0; q < 5; ++q) fprintf(stderr, " %lld", (long long)(hb[5 * lm + q + 1] - hb[5 * lm + q]));
            fprintf(stderr, "; first barrier at %lld ns\n  inside (activations ready, weights landed, own MMAs done, all warps done, stored; from the phase start):", (long long)(hb[1] - hb[0]));
            for (int q = 0; q < 5; ++q) {
                if (q == 1) continue;
                const int ph = 5 * lm + q;
                fprintf(stderr, " [");
                for (int k : {0, 1, 4, 2, 3}) fprintf(stderr, "%lld ", (long long)(hb[5 * c->L + 2 + 6 * ph + k] - hb[ph]));
                fprintf(stderr, "]");
            }
            fprintf(stderr, "\n  barriers of that layer, over the CTAs (ns from the phase start): ");
            {
                const int G = c->sms;
                for (int q = 0; q < 5; ++q) {
                    const unsigned long long* a = hb.data() + 35 * c->L + 8 + 2 * G * q;
                    unsigned long long amin = ~0ULL, amax = 0, rmin = ~0ULL, rmax = 0;
                    int slow = 0;
                    for (int g = 0; g < G; ++g) {
                        if (a[2 * g] > amax) { amax = a[2 * g]; slow = g; }
                        amin = std::min(amin, a[2 * g]);
                        rmin = std::min(rmin, a[2 * g + 1]); rmax = std::max(rmax, a[2 * g + 1]);
                    }
                    const unsigned long long t0 = hb[5 * lm + q];
                    fprintf(stderr, "[arrive %lld..%lld (last: cta %d) leave %lld..%lld] ", (long long)(amin - t0), (long long)(amax - t0), slow,
                            (long long)(rmin - t0), (long long)(rmax - t0));
                }
            }
            fprintf(stderr, "\n");
        }
    }
    return 0;
}

// Chunk counts of a streaming call: `blocks` = sum of the per-session counts (in cnt_dev / off_dev when kmax > 1), `kmax` the
// largest, `n1` the length of the leading run of sessions with one chunk; off = host prefix sums of the counts (n + 1
// entries), null when every session brings kmax chunks.
struct Mix {
    int blocks = 0, kmax = 1, n1 = 0;
    const int32_t* off = nullptr;
    int group = 0;               // > 0: a pass of fo_stream_steps_v (`group` chunks per attention CTA; counts uncapped)
    bool uniform(int n) const { return blocks == n * kmax; }
    int block(int i) const { return off ? off[i] : i * kmax; }
};

// The adapter of a multi-chunk call (rows (session, chunk, frame) in enc), equal to cnt[b] sequential single-chunk calls per
// session.  `out` names one output block per (session, chunk); this function sets its chunk mapping.
template <typename TA>
int adapter_chunks(fo_ctx* c, const float* enc, int n, const Mix& m, int t, AdOut out, cudaStream_t st) {
    // LinearAdapter works per row and CNNAdapter starts from zero left context on every call (adapter.py:41-52):
    // independent blocks of t frames
    if (!c->ad_carry) return adapter_program<TA>(c, enc, nullptr, m.blocks, t, c->ids_dev, nullptr, nullptr, out, st);
    const int k = m.kmax;
    if (t % 2 == 0 && m.uniform(n)) {
        // CNNSubsampling with even t: every chunk brings an even number of frames to the stride-2 conv, so one pass over a
        // session's k*t frames with the carried cache gives the k sequential outputs and leaves the same cache
        out.k = k;
        return adapter_program<TA>(c, enc, nullptr, n, k * t, c->ids_dev, nullptr, nullptr, out, st);
    }
    // The same pass over a per-session grid of kmax*t rows, each session's padding at its end.  With odd t the output phase of
    // the stride-2 conv shifts between chunks (a joint stride-2 pass yields other frames, and fewer), but in the session's
    // continuous stream S = [cache | x_0 | x_1 ..] output m of chunk j is the conv at S position j * t + 2 m: stride-1 convs over
    // the grid and a row pick give every chunk at once.
    const AdMix mix{c->cnt_dev, c->off_dev, k, t, m.blocks, t % 2 != 0};
    return adapter_program<TA>(c, enc, nullptr, n, k * t, c->ids_dev, nullptr, nullptr, out, st, &mix);
}

// Session groups of a streaming step of n sessions (see stream_program)
int step_groups(const fo_ctx* c, int n) {
    int G = c->profile_gemm ? 1 : c->groups;
    if (G > fo_ctx::MAX_GROUPS) G = fo_ctx::MAX_GROUPS;
    while (G > 1 && n < 8 * G) --G;
    if (c->cfg.concat_after) G = 1;                         // the concat operand is a [2][M][D] pair of planes over ALL rows
    return G;
}

// m.kmax > 1: several consecutive chunks per session (fo_encode_stream_chunks[_v]); rows are ordered (session, chunk, frame),
// so every per-session kernel sees a session's cnt[b]*t new rows as one run
template <typename TA>
int stream_program(fo_ctx* c, int n, const Mix& m, const float* feats, int t_in, float* enc_out_dev, float* y_dev, cudaStream_t st) {
    const int D = c->D, FF = c->FF, H = c->H;
    const int T1 = (t_in - 1) / 2, t = (T1 - 1) / 2, M = m.blocks * t;
    float* x;
    if (c->step_part == 2) {
        void* xp;
        FO_TRY(ws_ensure(c, WS_X, (size_t)M * D * sizeof(float), &xp));
        x = reinterpret_cast<float*>(xp);
    } else {
        FO_TRY(subsample_program<TA>(c, feats, m.blocks, t_in, &x, st));   // every block brings its own context frames
        if (c->step_part == 1) return 0;
    }
    void *h, *qkv, *att, *ffh;
    FO_TRY(ws_ensure(c, WS_H, (size_t)(c->cfg.concat_after ? 2 : 1) * M * D * sizeof(TA), &h));   // concat_after: [layer input | linear_out rows]
    FO_TRY(ws_ensure(c, WS_QKV, (size_t)M * 3 * D * sizeof(TA), &qkv));
    FO_TRY(ws_ensure(c, WS_ATT, (size_t)M * D * sizeof(TA), &att));
    FO_TRY(ws_ensure(c, WS_FFH, (size_t)M * FF * sizeof(TA), &ffh));
    float* q32 = reinterpret_cast<float*>(qkv);
    if (sizeof(TA) == 2) { void* q; FO_TRY(ws_ensure(c, WS_Q32, (size_t)M * 3 * D * sizeof(float), &q)); q32 = reinterpret_cast<float*>(q); }
    void* hc = nullptr;
    if (c->KF >= 2) FO_TRY(ws_ensure(c, WS_HC, (size_t)M * D * sizeof(TA), &hc));
    // The 24 layers run per SESSION GROUP on parallel streams (fork/join with events, also under graph capture):
    // sessions are independent, every layer kernel of a 64-session step is latency bound (<= 148 CTAs, 8-16 us), so
    // two groups' kernels overlap each other's pipeline fill, epilogue and launch gaps.  Rows of one group are
    // contiguous, so the groups just take slices of the same workspaces.
    int stacked = 1;
    if (sizeof(TA) == 2 && m.kmax == 1 && !m.group) {       // the stack kernel's attention is single-chunk
        stacked = stack_program(c, n, t, x, qkv, q32, att, ffh, enc_out_dev, st);
        if (stacked < 0) return stacked;
    }
    const int G = stacked == 0 ? 1 : step_groups(c, n);
    // a call mixing one-chunk sessions (the leading n1) with multi-chunk ones: the multi-chunk attention sizes its shared
    // memory by the largest count, so the one-chunk sessions keep the single-chunk kernel, and the two run side by side
    const long long layer_stride = (long long)c->cfg.max_sessions * 2LL * H * c->ring_cap * 64;
    if (G > 1) {
        FO_CUDA(cudaEventRecord(c->ev_fork, st));
        for (int g = 1; g < G; ++g) FO_CUDA(cudaStreamWaitEvent(c->grp_stream[g], c->ev_fork, 0));
    }
    const int per = (n + G - 1) / G;
    for (int l = 0; l < c->L && stacked != 0; ++l) {
        const LayerW& w = c->layers[l];
        const bool last = l + 1 == c->L;
        for (int g = 0; g < G; ++g) {
            const int s0 = g * per, ng = std::min(per, n - s0);
            if (ng <= 0) continue;
            cudaStream_t sg = g == 0 ? st : c->grp_stream[g];
            c->tc_cur = &c->tc_wsg[g];
            const long long r0 = (long long)m.block(s0) * t;   // the group's rows: its sessions' blocks (host prefix sums)
            const int Mg = (m.block(s0 + ng) - m.block(s0)) * t;
            AttnStream a;
            a.ids = c->ids_dev + s0;
            a.n_frames = c->n_frames;
            a.pe_index = c->pe_index;
            a.n = ng; a.t = t; a.H = H; a.ring_cap = c->ring_cap; a.window = c->window; a.full_chunk = c->full_chunk;
            a.pe_wrap = c->pe_wrap; a.pos_rows = c->pos_rows;
            a.ring_slot_stride = 2LL * H * c->ring_cap * 64;
            a.chunk_size = c->cfg.chunk_size;
            a.cnt = c->cnt_dev + s0;
            a.off = c->off_dev + s0;
            TA* hg = reinterpret_cast<TA*>(h) + r0 * D;
            TA* qkvg = reinterpret_cast<TA*>(qkv) + r0 * 3 * D;
            TA* attg = reinterpret_cast<TA*>(att) + r0 * D;
            TA* ffhg = reinterpret_cast<TA*>(ffh) + r0 * FF;
            float* q32g = q32 + r0 * 3 * D;
            float* xg = x + r0 * D;
            int r = 0;
            if (l == 0) r = c->cfg.post_norm ? to_act<TA>(xg, hg, (long long)Mg * D, sg)          // post-norm: the layer input as it is
                                             : layer_norm<TA>(xg, Mg, D, w.ln1g, w.ln1b, 1e-5f, 0, 1.0f, hg, nullptr, sg);
            L2Prefetch pfq;                                   // QKV runs: this layer's KV rings (attention) + out-proj weights
            if (c->use_prefetch & 2) {
                const long long slot_bytes = a.ring_slot_stride * (long long)sizeof(TA);
                pfq.ptr[0] = reinterpret_cast<const char*>(c->ring) + ((long long)l * layer_stride) * sizeof(TA) + (long long)c->pf_slot_lo * slot_bytes;
                pfq.bytes[0] = (long long)(c->pf_slot_hi - c->pf_slot_lo + 1) * slot_bytes;
            }
            if (c->use_prefetch & 1) {
                pfq.ptr[1] = w.wo;
                pfq.bytes[1] = (long long)D * D * c->esz;
                a.prefetch = pf1(w.w1, (long long)D * FF * c->esz);                       // attention runs: FFN1's weights
            }
            int qkv_splits = 0;
            // the multi-chunk attention reads finished QKV rows: no split-K reduction deferred to it
            if (r == 0) r = layer_pre<TA>(c, w, Mg, hg, qkvg, q32g, pfq, sg, m.kmax == 1 && !m.group ? &qkv_splits : nullptr);
            if (qkv_splits > 0) {
                a.part = c->tc_cur->partial;
                a.part_bias = w.bqkv;
                a.nsplit = qkv_splits;
                a.part_stride = (long long)Mg * 3 * D;
            }
            TA* ring_l = reinterpret_cast<TA*>(c->ring) + l * layer_stride;
            const int n1g = std::min(std::max(m.n1 - s0, 0), ng);  // the group's share of the leading one-chunk run
            if (r == 0 && !(c->debug_skip & 1) && n1g < ng) {
                // multi-chunk sessions (rows from the end of the one-chunk run): on a forked stream when both kernels run.  A pass
                // of fo_stream_steps_v (n1 = 0, never forked) spreads a session's chunks over groups of m.group per CTA.
                AttnStream am = a;
                am.ids += n1g; am.cnt += n1g; am.off += n1g; am.n = ng - n1g;
                am.chunks = m.group ? m.group : m.kmax;
                const long long ro = (long long)n1g * t;
                const bool fork = n1g > 0;
                cudaStream_t sm = fork ? c->mix_stream[g] : sg;
                if (fork) {
                    FO_CUDA(cudaEventRecord(c->ev_mix_fork[g], sg));
                    FO_CUDA(cudaStreamWaitEvent(sm, c->ev_mix_fork[g], 0));
                }
                r = attention_chunks<TA>(am, cdiv(m.kmax, am.chunks), qkvg + ro * 3 * D, q32g + ro * 3 * D, ring_l,
                                         reinterpret_cast<const TA*>(w.ptab_h), w.pos_u, w.pos_v, attg + ro * D, sm);
                if (r == 0 && n1g > 0) {
                    AttnStream a1 = a;
                    a1.n = n1g;
                    r = attention_stream<TA>(a1, qkvg, q32g, ring_l, reinterpret_cast<const TA*>(w.ptab_h), w.pos_u, w.pos_v, attg, sg);
                }
                if (fork) {
                    FO_CUDA(cudaEventRecord(c->ev_mix_join[g], sm));
                    FO_CUDA(cudaStreamWaitEvent(sg, c->ev_mix_join[g], 0));
                }
            } else if (r == 0 && !(c->debug_skip & 1)) {        // every session of the group brings one chunk
                r = attention_stream<TA>(a, qkvg, q32g, ring_l, reinterpret_cast<const TA*>(w.ptab_h), w.pos_u, w.pos_v, attg, sg);
            }
            NextNorm nn{last ? c->after_g : c->layers[l + 1].ln1g, last ? c->after_b : c->layers[l + 1].ln1b,
                        last ? enc_out_dev + r0 * D : nullptr};
            FfnConv fc;
            fc.B = ng; fc.T = m.kmax * t; fc.ids = c->ids_dev + s0; fc.layer = l;   // Conv1dLinear: one pass over each session's rows with the carry
            if (m.kmax > 1) { fc.cnt = a.cnt; fc.off = a.off; fc.t = t; }
            fc.hc = hc ? reinterpret_cast<TA*>(hc) + r0 * D : nullptr;
            if (r == 0) r = layer_post<TA>(c, w, xg, Mg, attg, hg, ffhg, nn, last ? nullptr : c->layers[l + 1].wqkv, fc, sg);
            if (r != 0) { c->tc_cur = &c->tc_wsg[0]; return r; }
        }
    }
    c->tc_cur = &c->tc_wsg[0];
    if (G > 1) {
        for (int g = 1; g < G; ++g) {
            FO_CUDA(cudaEventRecord(c->ev_join[g], c->grp_stream[g]));
            FO_CUDA(cudaStreamWaitEvent(st, c->ev_join[g], 0));
        }
    }
    const bool run_adapter = c->cfg.has_adapter && (y_dev || c->handoff);
    if (run_adapter) {
        AdOut out;
        if (c->handoff) {
            out.h16 = reinterpret_cast<TA*>(c->handoff) + c->handoff_off * c->E;
            out.pitch = c->handoff_rows;
        } else {
            out.y = y_dev;
            out.pitch = ad_frames(c, t);
        }
        if (m.kmax == 1) FO_TRY(adapter_program<TA>(c, enc_out_dev, nullptr, n, t, c->ids_dev, nullptr, nullptr, out, st));
        else FO_TRY(adapter_chunks<TA>(c, enc_out_dev, n, m, t, out, st));
    }
    FO_TRY(advance_sessions(c->ids_dev, n, t, c->cfg.chunk_size, c->pe_wrap, c->n_frames, c->pe_index,
                            (run_adapter && c->ad_carry) ? c->ad_valid : nullptr, st, m.kmax, m.kmax > 1 ? c->cnt_dev : nullptr));
    return 0;
}

template <typename TA>
int offline_program(fo_ctx* c, const float* feats, const int32_t* ilens_dev, int B, int T, int chunk, int left,
                    float* enc_out_dev, uint8_t* mask2, int32_t* ilens2, float* y_dev, cudaStream_t st) {
    const int D = c->D, FF = c->FF, H = c->H;
    const int T1 = (T - 1) / 2, T2 = (T1 - 1) / 2, M = B * T2;
    FO_TRY(subsample_mask(ilens_dev, B, T, T2, mask2, ilens2, st));
    float* x;
    FO_TRY(subsample_program<TA>(c, feats, B, T, &x, st));
    void *h, *qkv, *att, *ffh;
    FO_TRY(ws_ensure(c, WS_H, (size_t)(c->cfg.concat_after ? 2 : 1) * M * D * sizeof(TA), &h));   // concat_after: [layer input | linear_out rows]
    FO_TRY(ws_ensure(c, WS_QKV, (size_t)M * 3 * D * sizeof(TA), &qkv));
    FO_TRY(ws_ensure(c, WS_ATT, (size_t)M * D * sizeof(TA), &att));
    FO_TRY(ws_ensure(c, WS_FFH, (size_t)M * FF * sizeof(TA), &ffh));
    float* q32 = reinterpret_cast<float*>(qkv);
    if (sizeof(TA) == 2) { void* q; FO_TRY(ws_ensure(c, WS_Q32, (size_t)M * 3 * D * sizeof(float), &q)); q32 = reinterpret_cast<float*>(q); }
    void* hc = nullptr;
    if (c->KF >= 2) FO_TRY(ws_ensure(c, WS_HC, (size_t)M * D * sizeof(TA), &hc));
    void *hp = nullptr, *fp = nullptr;
    if (c->KM) {
        const size_t rows = (size_t)B * (T2 + c->KM - 1);
        FO_TRY(ws_ensure(c, WS_HP, rows * D * sizeof(TA), &hp));
        FO_TRY(ws_ensure(c, WS_FP, rows * FF * sizeof(TA), &fp));
        FO_CUDA(cudaMemsetAsync(fp, 0, rows * FF * sizeof(TA), st));      // the padding rows stay zero: the GEMM only writes the T2 inner rows
    }
    if (c->cfg.post_norm) FO_TRY(to_act<TA>(x, reinterpret_cast<TA*>(h), (long long)M * D, st));
    else FO_TRY(layer_norm<TA>(x, M, D, c->layers[0].ln1g, c->layers[0].ln1b, 1e-5f, 0, 1.0f, reinterpret_cast<TA*>(h), nullptr, st));
    for (int l = 0; l < c->L; ++l) {
        const LayerW& w = c->layers[l];
        const bool last = l + 1 == c->L;
        FO_TRY(layer_pre<TA>(c, w, M, reinterpret_cast<TA*>(h), reinterpret_cast<TA*>(qkv), q32, L2Prefetch(), st));
        if (!(c->debug_skip & 1))
        FO_TRY(attention_offline<TA>(reinterpret_cast<const TA*>(qkv), q32, B, T2, H, ilens2, chunk, left,
                                     w.ptab, reinterpret_cast<const TA*>(w.ptab_h), c->pos_rows, w.pos_u, w.pos_v,
                                     reinterpret_cast<TA*>(att), st));
        NextNorm nn{last ? c->after_g : c->layers[l + 1].ln1g, last ? c->after_b : c->layers[l + 1].ln1b,
                    last ? enc_out_dev : nullptr};
        FfnConv fc;
        fc.B = B; fc.T = T2; fc.ids = nullptr; fc.layer = l; fc.hc = hc; fc.hp = hp; fc.fp = fp;
        FO_TRY(layer_post<TA>(c, w, x, M, reinterpret_cast<TA*>(att), reinterpret_cast<TA*>(h), reinterpret_cast<TA*>(ffh), nn, nullptr, fc, st));
    }
    if (c->cfg.has_adapter && y_dev) {
        AdOut out;
        out.y = y_dev;
        FO_TRY(adapter_program<TA>(c, enc_out_dev, mask2, B, T2, nullptr, nullptr, nullptr, out, st));
    }
    return 0;
}

// Device tables of a packed call (fo_encode_offline_packed), one int32 upload; each field is an offset into it.
struct PackTab {
    int B = 0, tmax = 0, fmax = 0;    // utterances, longest in encoder rows, longest in feature frames
    int rows = 0, trunk = 0, ad_rows = 0, gap = 0, tiles = 0, grid_frames = 0;
    int o_tiles = 0, o_lens = 0, o_eoff = 0, o_xrow = 0, o_grow = 0, o_flen = 0, o_foff = 0, o_frow = 0, o_gaps = 0, o_adcnt = 0,
        o_aoff = 0;
    int o_soff = 0;                   // PCM entry only: int64 sample offsets (two words each, 8-byte aligned), else 0
    std::vector<int32_t> h;
};
// Packed twin of offline_program: B utterances back to back, every kernel on their rows only.
//  - front: the features go onto one grid where every utterance starts at a multiple of 4 frames (the subsampling's stride),
//    so each conv2 output row sees the frames of one utterance; its rows (at most 2 extra per utterance) are gathered out.
//  - layers: row-generic GEMMs / LayerNorms over all rows; attention per (utterance, query tile) from a tile table; the
//    depthwise conv restarts at each utterance.  MultiLayeredConv1d (two-sided conv) keeps k - 1 zeroed rows between
//    utterances in the residual stream (`gap`), and the encoder rows are gathered out of it at the end.
//  - adapter: adapter_program's packed mode.
// The features reach the grid (WS_FGRID, spare frames zeroed) either from packed features (offline_packed_program) or straight
// from the fbank of packed PCM (fo_encode_offline_packed_pcm); offline_packed_trunk runs everything from the grid on.
template <typename TA>
int offline_packed_trunk(fo_ctx* c, const float* fg, const PackTab& p, const int32_t* tab, int chunk, int left, float* enc_out_dev,
                         float* y_dev, cudaStream_t st) {
    const int D = c->D, FF = c->FF, H = c->H, B = p.B, M = p.trunk;
    void* xp;
    float* xg;
    FO_TRY(subsample_program<TA>(c, fg, 1, p.grid_frames, &xg, st));
    FO_TRY(ws_ensure(c, WS_XP, (size_t)M * D * sizeof(float), &xp));
    float* x = reinterpret_cast<float*>(xp);
    if (p.gap) FO_CUDA(cudaMemsetAsync(x, 0, (size_t)M * D * sizeof(float), st));
    FO_TRY(copy_utt_rows(xg, tab + p.o_grow, x, tab + p.o_xrow, tab + p.o_lens, B, p.tmax, D, st));
    void *h, *qkv, *att, *ffh;
    FO_TRY(ws_ensure(c, WS_H, (size_t)(c->cfg.concat_after ? 2 : 1) * M * D * sizeof(TA), &h));
    FO_TRY(ws_ensure(c, WS_QKV, (size_t)M * 3 * D * sizeof(TA), &qkv));
    FO_TRY(ws_ensure(c, WS_ATT, (size_t)M * D * sizeof(TA), &att));
    FO_TRY(ws_ensure(c, WS_FFH, (size_t)M * FF * sizeof(TA), &ffh));
    float* q32 = reinterpret_cast<float*>(qkv);
    if (sizeof(TA) == 2) { void* q; FO_TRY(ws_ensure(c, WS_Q32, (size_t)M * 3 * D * sizeof(float), &q)); q32 = reinterpret_cast<float*>(q); }
    void* hc = nullptr;
    if (c->KF >= 2) FO_TRY(ws_ensure(c, WS_HC, (size_t)M * D * sizeof(TA), &hc));
    void *hp = nullptr, *fp = nullptr;
    if (c->KM) {
        const size_t rows = (size_t)M + c->KM - 1;
        FO_TRY(ws_ensure(c, WS_HP, rows * D * sizeof(TA), &hp));
        FO_TRY(ws_ensure(c, WS_FP, rows * FF * sizeof(TA), &fp));
        FO_CUDA(cudaMemsetAsync(fp, 0, rows * FF * sizeof(TA), st));
    }
    float* enc_rows = enc_out_dev;                  // the last layer's output rows: straight to enc_out unless there are gaps
    if (p.gap) { void* e; FO_TRY(ws_ensure(c, WS_ENC2, (size_t)M * D * sizeof(float), &e)); enc_rows = reinterpret_cast<float*>(e); }
    AttnVarlen vl;
    vl.tiles = reinterpret_cast<const int2*>(tab + p.o_tiles);
    vl.lens = tab + p.o_lens;
    vl.rows = tab + p.o_xrow;
    vl.n = p.tiles;
    if (c->cfg.post_norm) FO_TRY(to_act<TA>(x, reinterpret_cast<TA*>(h), (long long)M * D, st));
    else FO_TRY(layer_norm<TA>(x, M, D, c->layers[0].ln1g, c->layers[0].ln1b, 1e-5f, 0, 1.0f, reinterpret_cast<TA*>(h), nullptr, st));
    for (int l = 0; l < c->L; ++l) {
        const LayerW& w = c->layers[l];
        const bool last = l + 1 == c->L;
        FO_TRY(layer_pre<TA>(c, w, M, reinterpret_cast<TA*>(h), reinterpret_cast<TA*>(qkv), q32, L2Prefetch(), st));
        if (!(c->debug_skip & 1))
        FO_TRY(attention_offline_packed<TA>(reinterpret_cast<const TA*>(qkv), q32, vl, B, p.tmax, H, chunk, left, w.ptab,
                                            reinterpret_cast<const TA*>(w.ptab_h), c->pos_rows, w.pos_u, w.pos_v,
                                            reinterpret_cast<TA*>(att), st));
        NextNorm nn{last ? c->after_g : c->layers[l + 1].ln1g, last ? c->after_b : c->layers[l + 1].ln1b, last ? enc_rows : nullptr};
        FfnConv fc;
        fc.ids = nullptr; fc.layer = l; fc.hc = hc; fc.hp = hp; fc.fp = fp;
        if (c->KM) { fc.B = 1; fc.T = M; fc.gap_at = tab + p.o_gaps; fc.n_gaps = B - 1; }
        else { fc.B = B; fc.T = p.tmax; fc.cnt = tab + p.o_lens; fc.off = tab + p.o_eoff; fc.t = 1; }
        FO_TRY(layer_post<TA>(c, w, x, M, reinterpret_cast<TA*>(att), reinterpret_cast<TA*>(h), reinterpret_cast<TA*>(ffh), nn, nullptr, fc, st));
    }
    if (p.gap) FO_TRY(copy_utt_rows(enc_rows, tab + p.o_xrow, enc_out_dev, tab + p.o_eoff, tab + p.o_lens, B, p.tmax, D, st));
    if (c->cfg.has_adapter && y_dev) {
        AdOut out;
        out.y = y_dev;
        const AdPack pk{tab + p.o_adcnt, tab + p.o_eoff, tab + p.o_aoff, p.ad_rows};
        FO_TRY(adapter_program<TA>(c, enc_out_dev, nullptr, B, p.tmax, nullptr, nullptr, nullptr, out, st, nullptr, &pk));
    }
    return 0;
}

// feature grid of a packed call: grid_frames fp32 rows, zeroed (the spare frames behind each utterance stay zero)
int packed_grid(fo_ctx* c, const PackTab& p, float** fg, cudaStream_t st) {
    void* g;
    FO_TRY(ws_ensure(c, WS_FGRID, (size_t)p.grid_frames * c->F * sizeof(float), &g));
    FO_CUDA(cudaMemsetAsync(g, 0, (size_t)p.grid_frames * c->F * sizeof(float), st));
    *fg = reinterpret_cast<float*>(g);
    return 0;
}

template <typename TA>
int offline_packed_program(fo_ctx* c, const float* feats, const PackTab& p, const int32_t* tab, int chunk, int left,
                           float* enc_out_dev, float* y_dev, cudaStream_t st) {
    float* fg;
    FO_TRY(packed_grid(c, p, &fg, st));
    FO_TRY(copy_utt_rows(feats, tab + p.o_foff, fg, tab + p.o_frow, tab + p.o_flen, p.B, p.fmax, c->F, st));
    return offline_packed_trunk<TA>(c, fg, p, tab, chunk, left, enc_out_dev, y_dev, st);
}

// Arguments of fo_debug_attention once checked: the device tables (`tab`, uploaded to the entry's own scratch), the rows of
// qkv / out, and the launch geometry of the mode.
struct DebugAttn {
    int mode = 0, n = 0, T = 0, chunk = 0, left = 0, t = 0, layer = 0, group = 1, groups = 1, tmax = 0, ntiles = 0, nsplit = 0;
    long long rows = 0;
    std::vector<int32_t> tab;          // offline: ilens | packed: tiles {b, q}, lens, rows | streaming: ids, cnt, off
    const float *qkv = nullptr, *part = nullptr, *part_bias = nullptr, *ptab = nullptr, *pos_u = nullptr, *pos_v = nullptr;
    float* out = nullptr;
};

// fo_debug_attention in the context's element type: K|V and the rel-pos table converted as the step programs hold them, one
// launcher call, the output converted back to fp32.  Nothing here advances a session or touches the step's id tables.
template <typename TA>
int debug_attention_run(fo_ctx* c, const DebugAttn& d, cudaStream_t st) {
    const int D = c->D, H = c->H;
    constexpr bool F16 = sizeof(TA) == 2;
    const bool need_qkv = F16 && d.nsplit == 0;
    const size_t tab_b = (d.tab.size() * sizeof(int32_t) + 255) & ~(size_t)255;
    const size_t qkv_b = need_qkv ? (((size_t)d.rows * 3 * D * sizeof(TA) + 255) & ~(size_t)255) : 0;
    const size_t ptab_b = ((size_t)H * c->pos_rows * 64 * sizeof(TA) + 255) & ~(size_t)255;
    const size_t out_b = F16 ? (size_t)d.rows * D * sizeof(TA) : 0;
    char* scratch = nullptr;
    FO_CUDA(cudaMalloc(&scratch, tab_b + qkv_b + ptab_b + out_b));
    int32_t* tab = reinterpret_cast<int32_t*>(scratch);
    TA* qkv = need_qkv ? reinterpret_cast<TA*>(scratch + tab_b) : F16 ? nullptr : reinterpret_cast<TA*>(const_cast<float*>(d.qkv));
    TA* ptab_h = reinterpret_cast<TA*>(scratch + tab_b + qkv_b);
    TA* out = F16 ? reinterpret_cast<TA*>(scratch + tab_b + qkv_b + ptab_b) : reinterpret_cast<TA*>(d.out);
    int r = 0;
    auto run = [&]() -> int {
        FO_CUDA(cudaMemcpyAsync(tab, d.tab.data(), d.tab.size() * sizeof(int32_t), cudaMemcpyHostToDevice, st));
        if (need_qkv) FO_TRY(f32_to_act16(d.qkv, reinterpret_cast<act16*>(qkv), d.rows * 3 * D, st));
        FO_TRY(ptab_head_major<TA>(d.ptab, c->pos_rows, H, ptab_h, st));
        FO_CUDA(cudaMemsetAsync(out, 0, (size_t)d.rows * D * sizeof(TA), st));      // rows no query writes (packed gaps) read 0
        if (d.mode == FO_ATT_OFFLINE)
            return attention_offline<TA>(qkv, d.qkv, d.n, d.T, H, tab, d.chunk, d.left, d.ptab, ptab_h, c->pos_rows, d.pos_u,
                                         d.pos_v, out, st);
        if (d.mode == FO_ATT_PACKED) {
            AttnVarlen vl;
            vl.tiles = reinterpret_cast<const int2*>(tab);
            vl.lens = tab + 2 * d.ntiles;
            vl.rows = vl.lens + d.n;
            vl.n = d.ntiles;
            return attention_offline_packed<TA>(qkv, d.qkv, vl, d.n, d.tmax, H, d.chunk, d.left, d.ptab, ptab_h, c->pos_rows,
                                                d.pos_u, d.pos_v, out, st);
        }
        AttnStream a;                     // as stream_program fills it
        a.ids = tab;
        a.n_frames = c->n_frames;
        a.pe_index = c->pe_index;
        a.n = d.n; a.t = d.t; a.H = H; a.ring_cap = c->ring_cap; a.window = c->window; a.full_chunk = c->full_chunk;
        a.pe_wrap = c->pe_wrap; a.pos_rows = c->pos_rows;
        a.ring_slot_stride = 2LL * H * c->ring_cap * 64;
        a.chunk_size = c->cfg.chunk_size;
        TA* ring_l = reinterpret_cast<TA*>(c->ring) + (long long)d.layer * c->cfg.max_sessions * a.ring_slot_stride;
        if (d.mode == FO_ATT_STREAM) {
            if (d.nsplit > 0) {
                a.part = d.part;
                a.part_bias = d.part_bias;
                a.nsplit = d.nsplit;
                a.part_stride = d.rows * 3 * D;
            }
            return attention_stream<TA>(a, qkv, d.qkv, ring_l, ptab_h, d.pos_u, d.pos_v, out, st);
        }
        a.cnt = tab + d.n;
        a.off = tab + 2 * d.n;
        a.chunks = d.group;
        return attention_chunks<TA>(a, d.groups, qkv, d.qkv, ring_l, ptab_h, d.pos_u, d.pos_v, out, st);
    };
    r = run();
    if (r == 0 && F16) r = act16_to_f32(reinterpret_cast<const act16*>(out), d.out, d.rows * D, st);
    const cudaError_t e = cudaStreamSynchronize(st);
    cudaFree(scratch);
    if (r == 0 && e != cudaSuccess) { set_error("fo_debug_attention: %s", cudaGetErrorString(e)); r = FO_ERR_CUDA; }
    return r;
}

}  // namespace

// =================================================================================================
extern "C" {

int fo_abi_version(void) { return FO_ABI_VERSION; }
const char* fo_last_error(void) { return g_err; }

}  // extern "C"

// fo_create (sm_split 0: the whole device) and fo_create_on_sms
static int create_ctx(const fo_config* cfg, int device, int dtype, int sm_split, int sm_group, fo_ctx** out) {
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0) {
        set_error("fo_create: no CUDA device (%s); this library has no CPU path", cudaGetErrorString(e));
        return FO_ERR_CUDA;
    }
    FO_CHECK(device >= 0 && device < ndev, "fo_create: device %d out of range", device);
    FO_CUDA(cudaSetDevice(device));
    cudaDeviceProp prop;
    FO_CUDA(cudaGetDeviceProperties(&prop, device));
    FO_CHECK(prop.major == 10, "fo_create: kernels are built for sm_100a only; device is sm_%d%d", prop.major, prop.minor);
    FO_CHECK(cfg->d_model % 128 == 0 && cfg->d_model / cfg->n_heads == 64 && cfg->d_model % cfg->n_heads == 0,
             "fo_create: d_model must be a multiple of 128 with d_k == 64");
    FO_CHECK(cfg->ffn_dim % 64 == 0 && cfg->llm_dim % 64 == 0, "fo_create: ffn_dim and llm_dim must be multiples of 64");
    FO_CHECK(cfg->feat_dim >= 11 && cfg->n_layers > 0 && cfg->max_sessions > 0, "fo_create: bad sizes");
    FO_CHECK(cfg->adapter_kernel >= 2 && cfg->adapter_kernel <= AGather::MAX_SEG, "fo_create: adapter kernel must be in 2..9");
    FO_CHECK(cfg->has_encoder || cfg->has_adapter, "fo_create: nothing to build");
    FO_CHECK(!cfg->ffn_multi_conv || (cfg->ffn_conv_kernel % 2 == 1 && cfg->ffn_conv_kernel >= 3 && cfg->ffn_conv_kernel <= AGather::MAX_SEG),
             "fo_create: MultiLayeredConv1d needs an odd ffn_conv_kernel in 3..9");
    FO_CHECK(cfg->adapter_type >= 0 && cfg->adapter_type <= 2, "fo_create: adapter_type must be 0 (subsampling), 1 (linear) or 2 (cnn)");
    FO_CHECK(!(cfg->has_adapter && (cfg->adapter_type == 2 || (cfg->adapter_type == 0 && 4 * cfg->d_model < cfg->llm_dim))) || 4 * cfg->d_model <= 4096,
             "fo_create: the two-conv adapters normalise 4 * d_model channels; d_model must be <= 1024");

    void* green = nullptr;
    int sms = prop.multiProcessorCount;
    if (sm_split > 0) FO_TRY(sm_group_acquire(device, sm_split, sm_group, &green, &sms));

    fo_ctx* c = new fo_ctx();
    c->cfg = *cfg;
    c->device = device;
    c->dtype = dtype;
    c->esz = dtype == FO_BF16 ? 2 : 4;
    c->sms = sms;
    c->green = green;
    c->smem_optin = (int)prop.sharedMemPerBlockOptin;
    c->coop = prop.cooperativeLaunch;
    memset(&c->stats, 0, sizeof(c->stats));
    c->F = cfg->feat_dim; c->F1 = (c->F - 1) / 2; c->F2 = (c->F1 - 1) / 2;
    c->D = cfg->d_model; c->H = cfg->n_heads; c->FF = cfg->ffn_dim; c->L = cfg->n_layers; c->E = cfg->llm_dim;
    c->KA = cfg->adapter_kernel;
    // adapter module: 0 CNNSubsampling, conv(C -> 2C, stride 2), or with 4 * enc_out_dim < llm_embed_dim (adapter.py:83)
    // conv(C -> 2C) then conv(2C -> 4C, stride 2); 1 LinearAdapter, no conv; 2 CNNAdapter, the two convs at stride 1, no cache
    if (cfg->has_adapter && cfg->adapter_type != 1) {
        const bool two = cfg->adapter_type == 2 || 4 * cfg->d_model < cfg->llm_dim;
        c->ad_nst = two ? 2 : 1;
        c->ad_st[0].cin = c->D;
        c->ad_st[0].cout = 2 * c->D;
        c->ad_st[0].stride = two ? 1 : 2;
        if (two) {
            c->ad_st[1].cin = 2 * c->D;
            c->ad_st[1].cout = 4 * c->D;
            c->ad_st[1].stride = cfg->adapter_type == 2 ? 1 : 2;
        }
        c->ad_carry = cfg->adapter_type == 0;
        // the two-conv modules are BatchNorm1d and ReLU by construction, whatever activation_func / norm say (adapter.py:20-29,84-95)
        c->ad_ln_eps = two || cfg->adapter_batchnorm ? -1.0f : 1e-3f;
        c->ad_ln_act = !two && cfg->adapter_gelu ? 2 : 1;
    }
    c->KF = (cfg->ffn_conv_kernel >= 2 && !cfg->ffn_multi_conv) ? cfg->ffn_conv_kernel : 0;
    c->KM = cfg->ffn_multi_conv ? cfg->ffn_conv_kernel : 0;
    const bool streaming = cfg->chunk_size > 0 && cfg->left_chunks > 0;
    c->window = streaming ? cfg->chunk_size * cfg->left_chunks : 1;                  // attention.py:290-295
    c->full_chunk = (cfg->left_chunks + 1) * cfg->chunk_size;                         // attention.py:83
    c->pe_wrap = cfg->chunk_size > 0 ? cfg->chunk_size * (cfg->pos_max_len / cfg->chunk_size) - c->full_chunk : cfg->pos_max_len;
    const int msf = cfg->max_stream_frames > 0 ? cfg->max_stream_frames : cfg->frames_per_chunk + cfg->context_frames;
    c->max_t = (((msf - 1) / 2) - 1) / 2;
    if (c->max_t < 1) c->max_t = 1;
    if (c->max_t > STREAM_MAX_T) c->max_t = STREAM_MAX_T;      // the streaming attention takes at most 8 frames per chunk
    c->ring_cap = ((c->window + c->max_t + 7) / 8) * 8;
    // Rel-pos rows the streaming kernels may read: a call at pe_index % pe_wrap = pe sees positions
    // max(0, pe - full_chunk) + [0, window + t).  With left_chunks <= 0 (full_chunk 0, pe_wrap = pos_max_len) that runs up to
    // pe_wrap + t - 1, past the reference's max_len rows; its RelPositionalEncoding.infer evaluates the sinusoid there
    // (attention.py:111-117), so the tables get real rows up to the last reachable position (fo_finalize_weights).
    c->pos_rows = cfg->pos_max_len;
    if (cfg->chunk_size > 0)
        c->pos_rows = std::max(c->pos_rows, std::max(0, c->pe_wrap - 1 - c->full_chunk) + c->window + c->max_t);
    c->carry = cfg->frame_len - cfg->frame_shift;
    c->chunk_samples = cfg->frame_shift * cfg->frames_per_chunk;
    c->fft = 1;
    while (c->fft < cfg->frame_len) c->fft <<= 1;
    c->gemm_backend = dtype == FO_BF16 ? 1 : 0;
    c->use_graph = 1;

    int r = 0;
    const int S = cfg->max_sessions;
    if (cfg->has_encoder) {
        const size_t ring_bytes = (size_t)c->L * S * 2 * c->H * c->ring_cap * 64 * c->esz;
        if (!r) r = dev_alloc(c, &c->ring, ring_bytes);
        void* p = nullptr;
        if (!r) { r = dev_alloc(c, &p, S * sizeof(int32_t)); c->n_frames = (int32_t*)p; }
        if (!r) { r = dev_alloc(c, &p, S * sizeof(int32_t)); c->pe_index = (int32_t*)p; }
        if (!r) { r = dev_alloc(c, &p, (size_t)S * (c->carry + c->chunk_samples) * sizeof(float)); c->samples = (float*)p; }
        if (!r) { r = dev_alloc(c, &p, (size_t)S * (cfg->context_frames + cfg->frames_per_chunk) * c->F * sizeof(float)); c->feat_ring = (float*)p; }
        if (!r && cudaMemset(c->ring, 0, ring_bytes) != cudaSuccess) r = FO_ERR_CUDA;
        if (!r && c->KF >= 2) {
            if (c->KF > 16) { set_error("fo_create: ffn_conv_kernel must be <= 16"); r = FO_ERR_ARG; }
            const size_t fb = (size_t)S * c->L * (c->KF - 1) * c->D * sizeof(float);
            if (!r) { r = dev_alloc(c, &p, fb); c->ffn_cache = (float*)p; }
            if (!r && cudaMemset(c->ffn_cache, 0, fb) != cudaSuccess) r = FO_ERR_CUDA;
        }
    }
    {
        void* p = nullptr;
        if (!r) { r = dev_alloc(c, &p, S * sizeof(int32_t)); c->ad_valid = (int32_t*)p; }
        for (int i = 0; i < c->ad_nst && c->ad_carry && !r; ++i) {
            r = dev_alloc(c, &p, (size_t)S * 2 * (c->KA - 1) * c->ad_st[i].cin * sizeof(float));
            c->ad_st[i].cache = (float*)p;
        }
        if (!r) { r = dev_alloc(c, &p, 3 * S * sizeof(int32_t)); c->ids_dev = (int32_t*)p; c->cnt_dev = c->ids_dev + S; c->off_dev = c->ids_dev + 2 * S; }
        if (!r) { r = dev_alloc(c, &p, (size_t)S * STREAM_CHUNKS_MAX_KEYS); c->onset_dev = (uint8_t*)p; }   // one flag per block, <= 128 blocks per session
        if (!r) { r = dev_alloc(c, &p, sizeof(unsigned long long)); c->sat_counter = (unsigned long long*)p; }
        if (!r && cudaMemset(c->sat_counter, 0, sizeof(unsigned long long)) != cudaSuccess) r = FO_ERR_CUDA;
    }
    for (int k = 0; k < fo_ctx::NSTAGE && !r; ++k) {
        if (cudaMallocHost((void**)&c->ids_host[k], 3 * S * sizeof(int32_t) + (size_t)S * STREAM_CHUNKS_MAX_KEYS) != cudaSuccess ||
            cudaEventCreateWithFlags(&c->ids_event[k], cudaEventDisableTiming) != cudaSuccess) {
            set_error("fo_create: pinned staging allocation failed");
            r = FO_ERR_NOMEM;
        }
    }
    if (!r) r = make_stream(c, &c->cap_stream);
    if (!r && c->green) r = make_stream(c, &c->exec_stream);
    if (!r && c->green && (cudaEventCreateWithFlags(&c->ev_enter, cudaEventDisableTiming) != cudaSuccess ||
                           cudaEventCreateWithFlags(&c->ev_leave, cudaEventDisableTiming) != cudaSuccess)) r = FO_ERR_CUDA;
    for (int g = 1; g < fo_ctx::MAX_GROUPS && !r; ++g) {
        r = make_stream(c, &c->grp_stream[g]);
        if (!r && cudaEventCreateWithFlags(&c->ev_join[g], cudaEventDisableTiming) != cudaSuccess) {
            set_error("fo_create: group stream creation failed");
            r = FO_ERR_CUDA;
        }
    }
    if (!r && cudaEventCreateWithFlags(&c->ev_fork, cudaEventDisableTiming) != cudaSuccess) r = FO_ERR_CUDA;
    for (int g = 0; g < fo_ctx::MAX_GROUPS && !r; ++g) {
        r = make_stream(c, &c->mix_stream[g]);
        if (!r && (cudaEventCreateWithFlags(&c->ev_mix_fork[g], cudaEventDisableTiming) != cudaSuccess ||
            cudaEventCreateWithFlags(&c->ev_mix_join[g], cudaEventDisableTiming) != cudaSuccess)) {
            set_error("fo_create: stream creation failed");
            r = FO_ERR_CUDA;
        }
    }
    if (r) { fo_destroy(c); return r; }
    c->slot_used.assign(S, 0);
    c->free_slots.reserve(S);
    for (int s = S - 1; s >= 0; --s) c->free_slots.push_back(s);
    *out = c;
    return 0;
}

extern "C" {

int fo_create(const fo_config* cfg, int device, int dtype, fo_ctx** out) {
    FO_CHECK(cfg && out, "fo_create: null argument");
    *out = nullptr;
    FO_CHECK(dtype == FO_F32 || dtype == FO_BF16, "fo_create: dtype must be FO_F32 or FO_BF16");
    return create_ctx(cfg, device, dtype, 0, 0, out);
}

int fo_create_on_sms(const fo_config* cfg, int device, int dtype, int sm_split, int sm_group, fo_ctx** out) {
    FO_CHECK(cfg && out, "fo_create_on_sms: null argument");
    *out = nullptr;
    FO_CHECK(dtype == FO_F32 || dtype == FO_BF16, "fo_create_on_sms: dtype must be FO_F32 or FO_BF16");
    FO_CHECK(sm_split >= 1, "fo_create_on_sms: sm_split must be >= 1 (got %d)", sm_split);
    FO_CHECK(sm_group >= 0 && sm_group < sm_split, "fo_create_on_sms: sm_group %d is outside [0, sm_split = %d)", sm_group, sm_split);
    return create_ctx(cfg, device, dtype, sm_split, sm_group, out);
}

int fo_destroy(fo_ctx* c) {
    if (!c) return 0;
    cudaSetDevice(c->device);
    ctx_sync(c);
    for (auto& kv : c->staged) cudaFree(kv.second.d);
    for (auto& kv : c->graphs) if (kv.second.exec) cudaGraphExecDestroy(kv.second.exec);
    if (c->cap_stream) cudaStreamDestroy(c->cap_stream);
    if (c->exec_stream) cudaStreamDestroy(c->exec_stream);
    if (c->ev_enter) cudaEventDestroy(c->ev_enter);
    if (c->ev_leave) cudaEventDestroy(c->ev_leave);
    if (c->copy_stream) cudaStreamDestroy(c->copy_stream);
    if (c->upload_stream) cudaStreamDestroy(c->upload_stream);
    for (int i = 0; i < 2; ++i) {
        if (c->ev_in[i]) cudaEventDestroy(c->ev_in[i]);
        if (c->ev_compute[i]) cudaEventDestroy(c->ev_compute[i]);
        if (c->ev_out[i]) cudaEventDestroy(c->ev_out[i]);
    }
    for (int g = 1; g < fo_ctx::MAX_GROUPS; ++g) {
        if (c->grp_stream[g]) cudaStreamDestroy(c->grp_stream[g]);
        if (c->ev_join[g]) cudaEventDestroy(c->ev_join[g]);
    }
    for (int g = 0; g < fo_ctx::MAX_GROUPS; ++g) {
        if (c->mix_stream[g]) cudaStreamDestroy(c->mix_stream[g]);
        if (c->ev_mix_fork[g]) cudaEventDestroy(c->ev_mix_fork[g]);
        if (c->ev_mix_join[g]) cudaEventDestroy(c->ev_mix_join[g]);
    }
    if (c->ev_fork) cudaEventDestroy(c->ev_fork);
    if (c->ev_sync) cudaEventDestroy(c->ev_sync);
    if (c->snap_ids_event) cudaEventDestroy(c->snap_ids_event);
    if (c->snap_ids_host) cudaFreeHost(c->snap_ids_host);
    if (c->snap_hdr_host) cudaFreeHost(c->snap_hdr_host);
    if (c->ho_tab_event) cudaEventDestroy(c->ho_tab_event);
    if (c->ho_tab_host) cudaFreeHost(c->ho_tab_host);
    for (void* p : c->owned) if (p) cudaFree(p);
    for (int k = 0; k < fo_ctx::NSTAGE; ++k) {
        if (c->ids_host[k]) cudaFreeHost(c->ids_host[k]);
        if (c->ids_event[k]) cudaEventDestroy(c->ids_event[k]);
    }
    delete c;
    return 0;
}

int fo_load_tensor(fo_ctx* c, const char* name, const void* data, const int64_t* shape, int ndim) {
    FO_CHECK(c && name && data && shape && ndim > 0 && ndim <= 4, "fo_load_tensor: bad argument");
    FO_CHECK(!c->finalized, "fo_load_tensor: weights already finalized");
    FO_CUDA(cudaSetDevice(c->device));
    HostTensor t;
    t.numel = 1;
    for (int i = 0; i < ndim; ++i) { FO_CHECK(shape[i] > 0, "fo_load_tensor: bad shape"); t.shape.push_back(shape[i]); t.numel *= shape[i]; }
    FO_CUDA(cudaMalloc((void**)&t.d, t.numel * sizeof(float)));
    cudaError_t e = cudaMemcpy(t.d, data, t.numel * sizeof(float), cudaMemcpyDefault);
    if (e != cudaSuccess) { cudaFree(t.d); set_error("fo_load_tensor(%s): %s", name, cudaGetErrorString(e)); return FO_ERR_CUDA; }
    auto it = c->staged.find(name);
    if (it != c->staged.end()) { cudaFree(it->second.d); c->staged.erase(it); }
    c->staged[name] = t;
    return 0;
}

int fo_finalize_weights(fo_ctx* c) {
    FO_CHECK(c && !c->finalized, "fo_finalize_weights: bad state");
    FO_CUDA(cudaSetDevice(c->device));
    if (c->dtype == FO_BF16) {
        FO_TRY(gemm_tc_init());
        for (int g = 0; g < fo_ctx::MAX_GROUPS; ++g) {
            FO_TRY(gemm_tc_workspace(&c->tc_wsg[g]));
            c->tc_wsg[g].sms = c->sms;
            c->owned.push_back(c->tc_wsg[g].partial);
            c->owned.push_back(c->tc_wsg[g].counters);
            c->device_bytes += (long long)c->tc_wsg[g].partial_bytes;
        }
    }
    return c->dtype == FO_BF16 ? finalize_t<act16>(c) : finalize_t<float>(c);
}

// ---- sessions ------------------------------------------------------------------------------------
static int reset_slot(fo_ctx* c, int s) {
    const int32_t z = 0;
    if (c->n_frames) {
        FO_CUDA(cudaMemcpy(c->n_frames + s, &z, 4, cudaMemcpyHostToDevice));
        FO_CUDA(cudaMemcpy(c->pe_index + s, &z, 4, cudaMemcpyHostToDevice));
        FO_CUDA(cudaMemset(c->samples + (size_t)s * (c->carry + c->chunk_samples), 0, (size_t)(c->carry + c->chunk_samples) * 4));
        FO_CUDA(cudaMemset(c->feat_ring + (size_t)s * (c->cfg.context_frames + c->cfg.frames_per_chunk) * c->F, 0,
                           (size_t)(c->cfg.context_frames + c->cfg.frames_per_chunk) * c->F * 4));
    }
    FO_CUDA(cudaMemcpy(c->ad_valid + s, &z, 4, cudaMemcpyHostToDevice));
    if (c->ffn_cache) {
        const size_t per = (size_t)c->L * (c->KF - 1) * c->D;
        FO_CUDA(cudaMemset(c->ffn_cache + (size_t)s * per, 0, per * sizeof(float)));     // left_padding zeros (attention.py:215,251)
    }
    return 0;
}

int fo_session_alloc(fo_ctx* c, int n, int32_t* ids_out) {
    FO_CHECK(c && ids_out && n > 0, "fo_session_alloc: bad argument");
    std::lock_guard<std::mutex> lk(c->mu);
    FO_CHECK((int)c->free_slots.size() >= n, "fo_session_alloc: %d sessions requested, %zu slots free", n, c->free_slots.size());
    FO_CUDA(cudaSetDevice(c->device));
    FO_TRY(ctx_sync(c));
    for (int i = 0; i < n; ++i) {
        int s = c->free_slots.back();
        c->free_slots.pop_back();
        c->slot_used[s] = 1;
        ids_out[i] = s;
        FO_TRY(reset_slot(c, s));
    }
    c->sessions_in_use += n;
    return 0;
}

int fo_session_reset(fo_ctx* c, int n, const int32_t* ids) {
    FO_CHECK(c, "null context");
    FO_TRY(check_ids(c, ids, n));
    FO_CUDA(cudaSetDevice(c->device));
    FO_TRY(ctx_sync(c));
    for (int i = 0; i < n; ++i) FO_TRY(reset_slot(c, ids[i]));
    return 0;
}

int fo_session_free(fo_ctx* c, int n, const int32_t* ids) {
    FO_CHECK(c, "null context");
    std::lock_guard<std::mutex> lk(c->mu);
    FO_TRY(check_ids(c, ids, n));
    for (int i = 0; i < n; ++i) {
        if (!c->slot_used[ids[i]]) continue;
        c->slot_used[ids[i]] = 0;
        c->free_slots.push_back(ids[i]);
        c->sessions_in_use -= 1;
    }
    return 0;
}

int fo_session_get_state(fo_ctx* c, int32_t id, int64_t* n_frames, int64_t* pe_index) {
    FO_CHECK(c && c->n_frames, "fo_session_get_state: context has no encoder");
    FO_TRY(check_ids(c, &id, 1));
    FO_CUDA(cudaSetDevice(c->device));
    int32_t a = 0, b = 0;
    FO_CUDA(cudaMemcpy(&a, c->n_frames + id, 4, cudaMemcpyDeviceToHost));
    FO_CUDA(cudaMemcpy(&b, c->pe_index + id, 4, cudaMemcpyDeviceToHost));
    if (n_frames) *n_frames = a;
    if (pe_index) *pe_index = b;
    return 0;
}

int fo_session_set_pe_index(fo_ctx* c, int n, const int32_t* ids, const int64_t* pe_index) {
    FO_CHECK(c && c->pe_index && pe_index, "fo_session_set_pe_index: bad argument");
    FO_TRY(check_ids(c, ids, n));
    FO_CUDA(cudaSetDevice(c->device));
    for (int i = 0; i < n; ++i) {
        int32_t v = (int32_t)pe_index[i];
        FO_CUDA(cudaMemcpy(c->pe_index + ids[i], &v, 4, cudaMemcpyHostToDevice));
    }
    return 0;
}

int fo_session_set_frames(fo_ctx* c, int32_t id, int64_t n_frames) {
    FO_CHECK(c && c->n_frames && n_frames >= 0, "fo_session_set_frames: bad argument");
    FO_TRY(check_ids(c, &id, 1));
    FO_CUDA(cudaSetDevice(c->device));
    int32_t v = (int32_t)n_frames;
    FO_CUDA(cudaMemcpy(c->n_frames + id, &v, 4, cudaMemcpyHostToDevice));
    return 0;
}

static int kv_ptrs(fo_ctx* c, int32_t id, int layer, void** k, void** v, int32_t* nf) {
    FO_CHECK(c && c->ring, "context has no encoder");
    FO_TRY(check_ids(c, &id, 1));
    FO_CHECK(layer >= 0 && layer < c->L, "layer %d out of range", layer);
    FO_CUDA(cudaSetDevice(c->device));
    FO_TRY(ctx_sync(c));
    FO_CUDA(cudaMemcpy(nf, c->n_frames + id, 4, cudaMemcpyDeviceToHost));
    const size_t per_kv = (size_t)c->H * c->ring_cap * 64;
    char* base = reinterpret_cast<char*>(c->ring) + (((size_t)layer * c->cfg.max_sessions + id) * 2) * per_kv * c->esz;
    *k = base;
    *v = base + per_kv * c->esz;
    return 0;
}

int fo_session_export_kv(fo_ctx* c, int32_t id, int layer, float* K, float* V, int32_t* cache_len) {
    void *k, *v;
    int32_t nf;
    FO_TRY(kv_ptrs(c, id, layer, &k, &v, &nf));
    const int cl = nf < c->window ? nf : c->window;
    if (cache_len) *cache_len = cl;
    if (cl == 0 || (!K && !V)) return 0;
    const size_t bytes = (size_t)c->H * cl * 64 * sizeof(float);
    void *dk, *dv;
    FO_TRY(out_dev(c, K, bytes, WS_TMP0, &dk));
    FO_TRY(out_dev(c, V, bytes, WS_TMP1, &dv));
    if (c->dtype == FO_BF16) {
        FO_TRY(ring_export<act16>((act16*)k, c->H, c->ring_cap, nf - cl, cl, (float*)dk, 0));
        FO_TRY(ring_export<act16>((act16*)v, c->H, c->ring_cap, nf - cl, cl, (float*)dv, 0));
    } else {
        FO_TRY(ring_export<float>((float*)k, c->H, c->ring_cap, nf - cl, cl, (float*)dk, 0));
        FO_TRY(ring_export<float>((float*)v, c->H, c->ring_cap, nf - cl, cl, (float*)dv, 0));
    }
    if (K) FO_TRY(out_done(K, dk, bytes, 0));
    if (V) FO_TRY(out_done(V, dv, bytes, 0));
    FO_TRY(ctx_sync(c));
    return 0;
}

int fo_session_import_kv(fo_ctx* c, int32_t id, int layer, const float* K, const float* V, int32_t cache_len) {
    void *k, *v;
    int32_t nf;
    FO_TRY(kv_ptrs(c, id, layer, &k, &v, &nf));
    FO_CHECK(K && V && cache_len >= 0 && cache_len <= c->window, "fo_session_import_kv: bad argument");
    FO_CHECK(nf >= cache_len, "fo_session_import_kv: set n_frames (fo_session_set_frames) >= cache_len first");
    if (cache_len == 0) return 0;
    const size_t bytes = (size_t)c->H * cache_len * 64 * sizeof(float);
    const void *dk, *dv;
    FO_TRY(in_dev(c, K, bytes, WS_TMP0, 0, &dk));
    FO_TRY(in_dev(c, V, bytes, WS_TMP1, 0, &dv));
    if (c->dtype == FO_BF16) {
        FO_TRY(ring_import<act16>((act16*)k, c->H, c->ring_cap, nf - cache_len, cache_len, (const float*)dk, 0));
        FO_TRY(ring_import<act16>((act16*)v, c->H, c->ring_cap, nf - cache_len, cache_len, (const float*)dv, 0));
    } else {
        FO_TRY(ring_import<float>((float*)k, c->H, c->ring_cap, nf - cache_len, cache_len, (const float*)dk, 0));
        FO_TRY(ring_import<float>((float*)v, c->H, c->ring_cap, nf - cache_len, cache_len, (const float*)dv, 0));
    }
    FO_TRY(ctx_sync(c));
    return 0;
}

// Entry `which` of the reference's cache list (adapter.py:123-143) is the left context of conv ad_nst - 1 - which: single-conv
// CNNSubsampling has one entry (d_model channels); the two-conv branch has cache[0] = second conv's input (2 * d_model channels)
// and cache[1] = first conv's input (d_model)
inline int ad_stage_of_entry(const fo_ctx* c, int which) { return c->ad_nst - 1 - which; }

static int ad_cache_of(fo_ctx* c, int which, float** base, int* C) {
    FO_CHECK(c && c->ad_carry, "context's adapter carries no cache");
    if (c->ad_nst == 1) FO_CHECK(which == 0, "single-conv CNNSubsampling has one cache entry (which = 0)");
    else FO_CHECK(which == 0 || which == 1, "two-conv CNNSubsampling has cache entries 0 and 1");
    const fo_ctx::AdStage& s = c->ad_st[ad_stage_of_entry(c, which)];
    *base = s.cache;
    *C = s.cin;
    return 0;
}

int fo_session_export_adapter_cache_n(fo_ctx* c, int32_t id, int which, float* cache, int32_t* valid) {
    float* base;
    int C;
    FO_TRY(ad_cache_of(c, which, &base, &C));
    FO_TRY(check_ids(c, &id, 1));
    FO_CUDA(cudaSetDevice(c->device));
    FO_TRY(ctx_sync(c));
    int32_t live = 0;
    FO_CUDA(cudaMemcpy(&live, c->ad_valid + id, 4, cudaMemcpyDeviceToHost));
    if (valid) *valid = live != 0;
    if (!live || !cache) return 0;
    const int km1 = c->KA - 1;
    std::vector<float> tm((size_t)km1 * C), out((size_t)km1 * C);
    FO_CUDA(cudaMemcpy(tm.data(), base + ((size_t)id * 2 + (live == 2 ? 1 : 0)) * km1 * C, tm.size() * 4, cudaMemcpyDeviceToHost));
    for (int r = 0; r < km1; ++r)
        for (int ch = 0; ch < C; ++ch) out[(size_t)ch * km1 + r] = tm[(size_t)r * C + ch];    // (C, k-1) as adapter.py:141
    FO_CUDA(cudaMemcpy(cache, out.data(), out.size() * 4, cudaMemcpyDefault));
    return 0;
}

int fo_session_import_adapter_cache_n(fo_ctx* c, int32_t id, int which, const float* cache, int32_t valid) {
    float* base;
    int C;
    FO_TRY(ad_cache_of(c, which, &base, &C));
    FO_TRY(check_ids(c, &id, 1));
    FO_CUDA(cudaSetDevice(c->device));
    FO_TRY(ctx_sync(c));
    int32_t live = 0;
    FO_CUDA(cudaMemcpy(&live, c->ad_valid + id, 4, cudaMemcpyDeviceToHost));
    if (valid) {
        FO_CHECK(cache, "fo_session_import_adapter_cache: null cache");
        const int km1 = c->KA - 1;
        std::vector<float> in((size_t)km1 * C), tm((size_t)km1 * C);
        FO_CUDA(cudaMemcpy(in.data(), cache, in.size() * 4, cudaMemcpyDefault));
        for (int r = 0; r < km1; ++r)
            for (int ch = 0; ch < C; ++ch) tm[(size_t)r * C + ch] = in[(size_t)ch * km1 + r];
        // the entries of one session share the live-half flag: write into the half that is (or becomes) live
        const int half = live == 2 ? 1 : 0;
        FO_CUDA(cudaMemcpy(base + ((size_t)id * 2 + half) * km1 * C, tm.data(), tm.size() * 4, cudaMemcpyHostToDevice));
        if (!live) live = 1;
    } else {
        live = 0;
    }
    FO_CUDA(cudaMemcpy(c->ad_valid + id, &live, 4, cudaMemcpyHostToDevice));
    return 0;
}

int fo_session_export_adapter_cache(fo_ctx* c, int32_t id, float* cache, int32_t* valid) {
    return fo_session_export_adapter_cache_n(c, id, 0, cache, valid);
}
int fo_session_import_adapter_cache(fo_ctx* c, int32_t id, const float* cache, int32_t valid) {
    return fo_session_import_adapter_cache_n(c, id, 0, cache, valid);
}

int fo_session_export_ffn_cache(fo_ctx* c, int32_t id, int layer, float* cache) {
    FO_CHECK(c && c->ffn_cache && cache, "fo_session_export_ffn_cache: context has no Conv1dLinear cache");
    FO_TRY(check_ids(c, &id, 1));
    FO_CHECK(layer >= 0 && layer < c->L, "layer %d out of range", layer);
    FO_CUDA(cudaSetDevice(c->device));
    FO_TRY(ctx_sync(c));
    const int km1 = c->KF - 1, D = c->D;
    std::vector<float> tm((size_t)km1 * D), out((size_t)km1 * D);
    FO_CUDA(cudaMemcpy(tm.data(), c->ffn_cache + ((size_t)id * c->L + layer) * km1 * D, tm.size() * 4, cudaMemcpyDeviceToHost));
    for (int r = 0; r < km1; ++r)
        for (int ch = 0; ch < D; ++ch) out[(size_t)ch * km1 + r] = tm[(size_t)r * D + ch];    // (D, k-1) as attention.py:258
    FO_CUDA(cudaMemcpy(cache, out.data(), out.size() * 4, cudaMemcpyDefault));
    return 0;
}

// ---- session snapshots ------------------------------------------------------------------------------
// Record of one session (fo_session_save), `bytes` per context, sections at multiples of 256 bytes:
//   header   256 B of int32 words: [0] magic "FOSS", [1] format version, [2..3] record bytes (int64), [4..] the fingerprint
//            below (one word per field, in that order), [56] n_frames, [57] pe_index, [58] adapter-cache valid flag (0 / 1)
//   KV       encoder only: [L][K|V][H][window][64] in the ring's element type (fp16 for bf16 contexts, fp32 for fp32): the last
//            min(n_frames, window) frames, oldest first, unswizzled; rows past them zero.  The window is all the streaming
//            attention reads (single-, multi-chunk and stack kernels alike), so the record does not depend on ring_cap;
//            restored, frame f goes to ring row f % ring_cap with the chunk swizzle c ^ (f & 7) (as ring_import_kernel)
//   fp32     each only when the context has the part: Conv1dLinear left context [L][KF-1][D]; the live half of each carried
//            adapter stage cache [k-1][cin] (stage order; zeros while the cache is None); fbank sample buffer [carry+chunk];
//            feature ring [ctx+m][F]
// The fingerprint is every setting that fixes the state's shape and meaning.  Capacities (max_sessions, max_stream_frames, hence
// max_t and ring_cap) and run-time options are not in it: a record moves between contexts that differ in them.  Weights are not
// in it either: restoring into a context with other weights of the same shapes is the caller's responsibility.
namespace {

constexpr int32_t SNAP_MAGIC = 0x53534F46;       // "FOSS" little-endian
constexpr int32_t SNAP_VERSION = 1;
constexpr int SNAP_W_FP = 4;                     // first fingerprint word
constexpr long long SNAP_STAGE_BYTES = 64LL << 20;   // device staging of host buffers: whole records up to this size

struct SnapField { const char* name; int32_t value; };

std::vector<SnapField> snap_fingerprint(const fo_ctx* c) {
    const fo_config& g = c->cfg;
    return {{"dtype", c->dtype}, {"feat_dim", g.feat_dim}, {"d_model", g.d_model}, {"n_heads", g.n_heads}, {"ffn_dim", g.ffn_dim},
            {"n_layers", g.n_layers}, {"chunk_size", g.chunk_size}, {"left_chunks", g.left_chunks}, {"window", c->window},
            {"pe_wrap", c->pe_wrap}, {"ffn_conv_kernel", c->KF}, {"has_encoder", g.has_encoder != 0},
            {"has_adapter", g.has_adapter != 0}, {"adapter_type", g.adapter_type}, {"adapter_kernel", g.adapter_kernel},
            {"adapter_stages", c->ad_nst}, {"adapter_cin0", c->ad_st[0].cin}, {"adapter_cin1", c->ad_st[1].cin},
            {"sample_rate", g.sample_rate}, {"frame_len", g.frame_len}, {"frame_shift", g.frame_shift},
            {"frames_per_chunk", g.frames_per_chunk}, {"context_frames", g.context_frames}};
}

inline long long round256(long long x) { return (x + 255) & ~255LL; }

// geometry of the record and of the context's state arrays; returns the record size
long long snap_layout(fo_ctx* c, SnapArgs* a) {
    const int S = c->cfg.max_sessions;
    long long off = SNAP_HDR_WORDS * 4;
    if (c->ring) {
        a->ring = reinterpret_cast<char*>(c->ring);
        a->L = c->L; a->S = S; a->H = c->H; a->cap = c->ring_cap; a->window = c->window; a->esz = (int)c->esz;
        a->kv_off = off;
        off = round256(off + (long long)c->L * 2 * c->H * c->window * 64 * c->esz);
    }
    a->n_frames = c->n_frames;
    a->pe_index = c->pe_index;
    a->ad_valid = c->ad_valid;
    a->nseg = 0;
    auto add = [&](void* base, long long bytes, long long stride, int half) {
        SnapSeg& s = a->seg[a->nseg++];
        s.base = reinterpret_cast<char*>(base); s.bytes = bytes; s.slot_stride = stride; s.rec_off = off; s.adapter_half = half;
        off = round256(off + bytes);
    };
    if (c->ffn_cache) {
        const long long b = (long long)c->L * (c->KF - 1) * c->D * 4;
        add(c->ffn_cache, b, b, 0);
    }
    for (int i = 0; i < c->ad_nst && c->ad_carry; ++i) {
        const long long b = (long long)(c->KA - 1) * c->ad_st[i].cin * 4;
        add(c->ad_st[i].cache, b, 2 * b, 1);
    }
    if (c->samples) {
        const long long b = (long long)(c->carry + c->chunk_samples) * 4;
        add(c->samples, b, b, 0);
        const long long f = (long long)(c->cfg.context_frames + c->cfg.frames_per_chunk) * c->F * 4;
        add(c->feat_ring, f, f, 0);
    }
    memset(a->hdr, 0, sizeof(a->hdr));
    a->hdr[0] = SNAP_MAGIC;
    a->hdr[1] = SNAP_VERSION;
    const long long bytes = round256(off);
    memcpy(&a->hdr[2], &bytes, 8);
    const std::vector<SnapField> fp = snap_fingerprint(c);
    for (size_t i = 0; i < fp.size(); ++i) a->hdr[SNAP_W_FP + i] = fp[i].value;
    a->rec_bytes = bytes;
    return bytes;
}

// shared checks of save and restore and the record geometry; *on_device = buf is device memory (of this context's device: a
// buffer of another GPU is refused, copy it over first)
int snap_begin(fo_ctx* c, const char* fn, const int32_t* ids, int n, const void* buf, SnapArgs* a, bool* on_device) {
    FO_CHECK(c && buf, "%s: null context or buffer", fn);
    FO_TRY(check_ids(c, ids, n));
    FO_CUDA(cudaSetDevice(c->device));
    cudaPointerAttributes pa;
    if (cudaPointerGetAttributes(&pa, buf) != cudaSuccess) { cudaGetLastError(); pa.type = cudaMemoryTypeUnregistered; }
    *on_device = pa.type == cudaMemoryTypeDevice || pa.type == cudaMemoryTypeManaged;
    FO_CHECK(!*on_device || pa.device == c->device, "%s: buf is memory of device %d, the context is on device %d", fn, pa.device,
             c->device);
    const int S = c->cfg.max_sessions;
    if (!c->snap_ids_dev) {
        void* p;
        FO_TRY(dev_alloc(c, &p, (size_t)S * sizeof(int32_t)));
        c->snap_ids_dev = (int32_t*)p;
        FO_CUDA(cudaMallocHost((void**)&c->snap_ids_host, (size_t)S * sizeof(int32_t)));
        FO_CUDA(cudaMallocHost((void**)&c->snap_hdr_host, (size_t)S * SNAP_HDR_WORDS * 4));
        FO_CUDA(cudaEventCreateWithFlags(&c->snap_ids_event, cudaEventDisableTiming));
    }
    snap_layout(c, a);
    a->n = n;
    return 0;
}

// the ids of the call into the snapshot path's own device array (not the steps' ids_dev, which a step may reuse as it is)
int snap_upload_ids(fo_ctx* c, const int32_t* ids, int n, cudaStream_t st, SnapArgs* a) {
    FO_CUDA(cudaEventSynchronize(c->snap_ids_event));      // the previous call's upload has left the pinned array
    memcpy(c->snap_ids_host, ids, sizeof(int32_t) * n);
    FO_CUDA(cudaMemcpyAsync(c->snap_ids_dev, c->snap_ids_host, sizeof(int32_t) * n, cudaMemcpyHostToDevice, st));
    FO_CUDA(cudaEventRecord(c->snap_ids_event, st));
    a->ids = c->snap_ids_dev;
    return 0;
}

// device staging for host buffers: a bounded number of whole records, reused batch after batch in stream order
int snap_staging(fo_ctx* c, long long bytes) {
    if (c->snap_stage) return 0;
    c->snap_stage_n = (int)std::max(1LL, std::min((long long)c->cfg.max_sessions, SNAP_STAGE_BYTES / bytes));
    void* p;
    FO_TRY(dev_alloc(c, &p, (size_t)c->snap_stage_n * bytes));
    c->snap_stage = (char*)p;
    return 0;
}

// record i's header: 0, or FO_ERR_ARG naming the first field that does not match this context
int snap_check_header(const fo_ctx* c, const SnapArgs& a, int i, const int32_t* h) {
    FO_CHECK(h[0] == SNAP_MAGIC, "fo_session_restore: record %d: bad magic 0x%08x (not a session snapshot)", i, (unsigned)h[0]);
    FO_CHECK(h[1] == SNAP_VERSION, "fo_session_restore: record %d: format version %d, this library reads version %d", i, h[1],
             SNAP_VERSION);
    // the fingerprint before the size, which follows from it: a record of another model names the setting that differs
    const std::vector<SnapField> fp = snap_fingerprint(c);
    for (size_t f = 0; f < fp.size(); ++f)
        FO_CHECK(h[SNAP_W_FP + f] == fp[f].value, "fo_session_restore: record %d: %s is %d, this context has %d", i, fp[f].name,
                 h[SNAP_W_FP + f], fp[f].value);
    long long bytes;
    memcpy(&bytes, &h[2], 8);
    FO_CHECK(bytes == a.rec_bytes, "fo_session_restore: record %d: record size %lld bytes, this context's is %lld", i, bytes,
             a.rec_bytes);
    FO_CHECK(h[SNAP_W_NFRAMES] >= 0 && h[SNAP_W_PE] >= 0 && (h[SNAP_W_ADVALID] == 0 || h[SNAP_W_ADVALID] == 1),
             "fo_session_restore: record %d: bad session state (n_frames %d, pe_index %d, adapter flag %d)", i, h[SNAP_W_NFRAMES],
             h[SNAP_W_PE], h[SNAP_W_ADVALID]);
    return 0;
}

}  // namespace

int fo_session_snapshot_bytes(fo_ctx* c, int64_t* bytes) {
    FO_CHECK(c && bytes, "fo_session_snapshot_bytes: bad argument");
    SnapArgs a;
    *bytes = snap_layout(c, &a);
    return 0;
}

int fo_session_save(fo_ctx* c, const int32_t* ids, int n, void* buf, void* stream) {
    FO_ON_GROUP(c, stream);
    const cudaStream_t st = (cudaStream_t)stream;
    SnapArgs a;
    bool on_device;
    FO_TRY(snap_begin(c, "fo_session_save", ids, n, buf, &a, &on_device));
    FO_TRY(snap_upload_ids(c, ids, n, st, &a));
    if (on_device) {
        a.rec = (char*)buf;
        return session_pack(a, st);
    }
    FO_TRY(snap_staging(c, a.rec_bytes));
    for (int i0 = 0; i0 < n; i0 += c->snap_stage_n) {
        SnapArgs b = a;
        b.ids = a.ids + i0;
        b.n = std::min(c->snap_stage_n, n - i0);
        b.rec = c->snap_stage;
        FO_TRY(session_pack(b, st));
        FO_CUDA(cudaMemcpyAsync((char*)buf + (size_t)i0 * a.rec_bytes, c->snap_stage, (size_t)b.n * a.rec_bytes,
                                cudaMemcpyDeviceToHost, st));
    }
    return 0;
}

int fo_session_restore(fo_ctx* c, const int32_t* ids, int n, const void* buf, void* stream) {
    FO_ON_GROUP(c, stream);
    const cudaStream_t st = (cudaStream_t)stream;
    SnapArgs a;
    bool on_device;
    FO_TRY(snap_begin(c, "fo_session_restore", ids, n, buf, &a, &on_device));
    // every header is checked before anything else is enqueued: a refused call leaves all n slots as they were.  The buffer may
    // be the output of a save still in flight on `stream` (a host buffer included), hence the sync before the headers are read
    const int32_t* hdr = (const int32_t*)buf;
    long long hstride = a.rec_bytes / 4;
    if (on_device) {
        FO_CUDA(cudaMemcpy2DAsync(c->snap_hdr_host, SNAP_HDR_WORDS * 4, buf, (size_t)a.rec_bytes, SNAP_HDR_WORDS * 4, n,
                                  cudaMemcpyDeviceToHost, st));
        hdr = c->snap_hdr_host;
        hstride = SNAP_HDR_WORDS;
    }
    FO_CUDA(cudaStreamSynchronize(st));
    for (int i = 0; i < n; ++i) FO_TRY(snap_check_header(c, a, i, hdr + i * hstride));
    FO_TRY(snap_upload_ids(c, ids, n, st, &a));
    if (on_device) {
        a.rec = (char*)buf;
        return session_unpack(a, st);
    }
    FO_TRY(snap_staging(c, a.rec_bytes));
    for (int i0 = 0; i0 < n; i0 += c->snap_stage_n) {
        SnapArgs b = a;
        b.ids = a.ids + i0;
        b.n = std::min(c->snap_stage_n, n - i0);
        b.rec = c->snap_stage;
        FO_CUDA(cudaMemcpyAsync(c->snap_stage, (const char*)buf + (size_t)i0 * a.rec_bytes, (size_t)b.n * a.rec_bytes,
                                cudaMemcpyHostToDevice, st));
        FO_TRY(session_unpack(b, st));
    }
    return 0;
}

// ---- frontend ------------------------------------------------------------------------------------
int fo_fbank_stream(fo_ctx* c, const int32_t* ids, int n, const void* pcm, int pcm_dtype, float scale,
                    float* feats_out, void* stream) {
    FO_CHECK(c && c->finalized && c->fb_window, "fo_fbank_stream: context has no finalized frontend");
    FO_CHECK(pcm && (pcm_dtype == FO_F32 || pcm_dtype == FO_I16), "fo_fbank_stream: pcm must be FO_F32 or FO_I16");
    FO_TRY(check_ids(c, ids, n));
    FO_CUDA(cudaSetDevice(c->device));
    FO_ON_GROUP(c, stream);
    cudaStream_t st = (cudaStream_t)stream;
    FO_TRY(upload_ids(c, ids, n, st));
    const size_t in_bytes = (size_t)n * c->chunk_samples * (pcm_dtype == FO_I16 ? 2 : 4);
    const void* dp;
    FO_TRY(in_dev(c, pcm, in_bytes, WS_PCM, st, &dp));
    const int rows = c->cfg.context_frames + c->cfg.frames_per_chunk;
    const size_t out_bytes = (size_t)n * rows * c->F * sizeof(float);
    void* dout = nullptr;
    if (feats_out) FO_TRY(out_dev(c, feats_out, out_bytes, WS_FEATS, &dout));
    FO_TRY(fbank_stream(fbank_params(c), c->ids_dev, n, dp, pcm_dtype == FO_I16, scale, c->cfg.frames_per_chunk,
                        c->cfg.context_frames, c->samples, c->feat_ring, (float*)dout, st));
    if (feats_out) FO_TRY(out_done(feats_out, dout, out_bytes, st));
    return 0;
}

int fo_fbank_offline(fo_ctx* c, const void* pcm, int pcm_dtype, int B, int64_t n_samples, float scale, float* out,
                     void* stream) {
    FO_CHECK(c && c->finalized && c->fb_window, "fo_fbank_offline: context has no finalized frontend");
    FO_CHECK(pcm && out && B > 0 && (pcm_dtype == FO_F32 || pcm_dtype == FO_I16), "fo_fbank_offline: bad argument");
    FO_CHECK(n_samples >= c->cfg.frame_len, "fo_fbank_offline: signal shorter than one frame");
    FO_CUDA(cudaSetDevice(c->device));
    FO_ON_GROUP(c, stream);
    cudaStream_t st = (cudaStream_t)stream;
    const size_t in_bytes = (size_t)B * n_samples * (pcm_dtype == FO_I16 ? 2 : 4);
    const void* dp;
    FO_TRY(in_dev(c, pcm, in_bytes, WS_PCM, st, &dp));
    const int m = (int)(1 + (n_samples - c->cfg.frame_len) / c->cfg.frame_shift);
    const size_t out_bytes = (size_t)B * m * c->F * sizeof(float);
    void* dout;
    FO_TRY(out_dev(c, out, out_bytes, WS_FEATS, &dout));
    FO_TRY(fbank_offline(fbank_params(c), dp, pcm_dtype == FO_I16, B, n_samples, scale, (float*)dout, st));
    FO_TRY(out_done(out, dout, out_bytes, st));
    return 0;
}

// ---- streaming chunk --------------------------------------------------------------------------------
// One step = [fbank of the new PCM ->] subsampling -> 24 layers -> after_norm -> adapter -> session advance,
// ~180 kernels that only touch context-owned buffers (staged input, workspaces, session state).  That body is
// captured once per call shape into a CUDA graph and replayed; the user's buffers are reached by one copy on
// either side of the graph.  The first call of a shape runs eagerly (it sizes the workspaces), the second
// captures.  A workspace that moves (ws_epoch) invalidates the graphs.
struct StepArgs {
    int n, t_in;
    Mix m;                     // chunks per session (fo_encode_stream_chunks[_v]; one each otherwise)
    bool with_fbank, want_y;
    int pcm_is_i16;
    float scale;
    int buf;                   // which set of PCM / encoder-output / adapter-output staging buffers (fo_stream_step_async alternates)
};
inline int ws_pcm(int buf) { return buf ? WS_PCM2 : WS_PCM; }
inline int ws_enc(int buf) { return buf ? WS_ENC2 : WS_ENC; }
inline int ws_y(int buf) { return buf ? WS_Y2 : WS_Y; }

static int step_body(fo_ctx* c, const StepArgs& a, cudaStream_t st) {
    void *dfeats, *denc, *dy = nullptr;
    const int T1 = (a.t_in - 1) / 2, t = (T1 - 1) / 2;
    const int t_out = ad_frames(c, t);
    const size_t blocks = (size_t)a.m.blocks;
    FO_TRY(ws_ensure(c, WS_FEATS, blocks * a.t_in * c->F * sizeof(float), &dfeats));
    FO_TRY(ws_ensure(c, ws_enc(a.buf), blocks * t * c->D * sizeof(float), &denc));
    if (a.want_y) FO_TRY(ws_ensure(c, ws_y(a.buf), blocks * t_out * c->E * sizeof(float), &dy));
    if (a.with_fbank && c->step_part != 2) {
        void* dp;
        FO_TRY(ws_ensure(c, ws_pcm(a.buf), (size_t)a.n * c->chunk_samples * 4, &dp));
        FO_TRY(fbank_stream(fbank_params(c), c->ids_dev, a.n, dp, a.pcm_is_i16, a.scale, c->cfg.frames_per_chunk,
                            c->cfg.context_frames, c->samples, c->feat_ring, (float*)dfeats, st));
    }
    return c->dtype == FO_BF16 ? stream_program<act16>(c, a.n, a.m, (const float*)dfeats, a.t_in, (float*)denc, (float*)dy, st)
                               : stream_program<float>(c, a.n, a.m, (const float*)dfeats, a.t_in, (float*)denc, (float*)dy, st);
}

static int run_step(fo_ctx* c, const StepArgs& a, cudaStream_t st) {
    // programmatic dependent launch along the chain: a kernel's prologue (barrier / TMEM set-up, weight stages, the attention
    // kernel's ring copies) runs while its predecessor drains.  Pays at every batch size since the prologues carry real work
    // (r85: -7 % at 1-4 sessions, -6 % at 8, -2.6 % at 64); FO_PDL_MIN raises the threshold for experiments.
    static int pdl_min = -1;
    if (pdl_min < 0) { const char* e = getenv("FO_PDL_MIN"); pdl_min = e ? atoi(e) : 1; }
    g_use_pdl = g_want_pdl && a.n >= pdl_min;
    if (!c->use_graph || c->profile_gemm) return step_body(c, a, st);
    char key[256];
    uint32_t sbits;
    memcpy(&sbits, &a.scale, 4);
    // the chunk counts enter as totals only (they are device data); the rows of session groups other than the first are
    // baked into the graph as the block where each group starts
    int len = snprintf(key, sizeof(key), "%d/%p/%lld/%lld/%d/%d.%d.%d/%d/%d/%d/%d/%08x/%d/%d/%d/%d-%d", a.buf, c->handoff, c->handoff_rows, c->handoff_off, a.n,
             a.m.blocks, a.m.kmax, a.m.n1, a.t_in, (int)a.with_fbank, (int)a.want_y, a.pcm_is_i16, sbits,
             c->gemm_backend, c->groups, (((c->debug_skip * 2 + c->defer_reduce) * 2 + c->fuse_ln) * 4 + c->use_prefetch) * 64 + c->stack_rows,
             ((c->use_prefetch & 2) ? c->pf_slot_lo * 2 + g_use_pdl : g_use_pdl), (c->use_prefetch & 2) ? c->pf_slot_hi : 0);   // the prefetch range is baked into the graph
    if (a.m.off) {
        const int G = step_groups(c, a.n), per = (a.n + G - 1) / G;
        for (int g = 1; g < G && g * per < a.n && len < (int)sizeof(key) - 16; ++g) len += snprintf(key + len, sizeof(key) - len, "/%d", a.m.off[g * per]);
    }
    if (c->graphs.size() > 256 && c->graphs.find(key) == c->graphs.end()) {
        for (auto& kv : c->graphs) if (kv.second.exec) cudaGraphExecDestroy(kv.second.exec);
        c->graphs.clear();
    }
    fo_ctx::StepGraph& g = c->graphs[key];
    if (g.exec && g.epoch == c->ws_epoch) {
        FO_CUDA(cudaGraphLaunch(g.exec, st));
        g_launches += g.launches;
        c->stack_launches += g.stacks;
        c->stats.graph_replays += 1;
        return 0;
    }
    if (g.exec) { cudaGraphExecDestroy(g.exec); g.exec = nullptr; }
    if (g.warm_epoch != c->ws_epoch) {             // first call of this shape (or buffers moved): eager
        FO_TRY(step_body(c, a, st));
        g.warm_epoch = c->ws_epoch;
        return 0;
    }
    const long long l0 = t_launches, e0 = c->ws_epoch, s0 = c->stack_launches;
    FO_CUDA(cudaStreamBeginCapture(c->cap_stream, cudaStreamCaptureModeRelaxed));
    int r = step_body(c, a, c->cap_stream);
    cudaGraph_t graph = nullptr;
    cudaError_t ce = cudaStreamEndCapture(c->cap_stream, &graph);
    if (r != 0) { if (graph) cudaGraphDestroy(graph); return r; }
    if (ce != cudaSuccess || !graph) {
        set_error("graph capture of the streaming step failed: %s", cudaGetErrorString(ce));
        return FO_ERR_CUDA;
    }
    FO_CHECK(c->ws_epoch == e0, "a workspace moved during graph capture");
    ce = cudaGraphInstantiate(&g.exec, graph, 0);
    cudaGraphDestroy(graph);
    if (ce != cudaSuccess) { g.exec = nullptr; set_error("cudaGraphInstantiate: %s", cudaGetErrorString(ce)); return FO_ERR_CUDA; }
    g.epoch = c->ws_epoch;
    g.launches = t_launches - l0;                  // counted (by this thread) while capturing, not yet run
    g_launches -= g.launches;
    g.stacks = c->stack_launches - s0;
    FO_CUDA(cudaGraphLaunch(g.exec, st));
    g_launches += g.launches;
    c->stats.graph_replays += 1;
    return 0;
}

// What every streaming entry checks before it enqueues anything, so that a refused call leaves the sessions as they were:
// chunk_size > 0 (with chunk_size <= 0 pe_index would step backwards into negative values, attention.py:107,120), at most
// max_t (<= STREAM_MAX_T) encoder frames per chunk, and window + t keys within the 128 the streaming attention stages.
static int stream_geometry(const fo_ctx* c, int t_in) {
    const int t = ((t_in - 1) / 2 - 1) / 2;
    FO_CHECK(c->cfg.chunk_size > 0, "streaming needs transformer-chunk_size > 0 (got %d); chunk_size <= 0 is full attention, "
                                    "use fo_encode_offline", c->cfg.chunk_size);
    FO_CHECK(t >= 1 && t <= c->max_t, "streaming call of %d feature frames gives %d encoder frames; context allows 1..%d",
             t_in, t, c->max_t);
    FO_CHECK(c->window + t <= STREAM_CHUNKS_MAX_KEYS,
             "streaming call: the attention window (%d frames) + %d new frames exceeds the %d keys of the streaming attention",
             c->window, t, STREAM_CHUNKS_MAX_KEYS);
    return 0;
}

// copies between the caller's buffers and the context's staging buffers, then the step
// chunks (fo_encode_stream_chunks[_v], feats only; m.kmax > 1): chunks[i] consecutive chunk blocks of session i, feats
// (m.blocks, t_in, F) in (session, chunk) order
static int stream_common(fo_ctx* c, const int32_t* ids, int n, const int32_t* chunks, const Mix& m, const void* pcm, int pcm_dtype,
                         float scale, const float* feats, int t_in, float* enc_out, float* adapter_out, cudaStream_t st) {
    const int T1 = (t_in - 1) / 2, t = (T1 - 1) / 2;
    FO_TRY(stream_geometry(c, t_in));
    if (adapter_out) FO_CHECK(c->cfg.has_adapter, "adapter_out requested but the context has no adapter");
    FO_CHECK(!c->KM, "this context's positionwise layer is MultiLayeredConv1d, which has no streaming form (the reference module has no infer(), "
                     "models/encoder/attention.py:145-196); use fo_encode_offline");
    const int t_out = ad_frames(c, t);
    const size_t enc_bytes = (size_t)m.blocks * t * c->D * sizeof(float);
    const size_t y_bytes = (size_t)m.blocks * t_out * c->E * sizeof(float);
    if (c->copy_stream && c->async_ticket > 0) {
        // a synchronous call after pipelined ones reuses staging set 0 (and the shared intermediates): let the read-backs of
        // the steps still in flight on the copy stream finish first
        FO_CUDA(cudaStreamWaitEvent(st, c->ev_out[0], 0));
        if (c->async_ticket > 1) FO_CUDA(cudaStreamWaitEvent(st, c->ev_out[1], 0));
    }
    fo_ctx::Armed armed = c->armed;              // consumed by this call, whatever its outcome
    c->armed.on = false;
    if (armed.on) {
        FO_CHECK(armed.n == m.blocks, "fo_handoff_arm was armed for %d blocks, this call advances %d sessions by %d chunks in all", armed.n, n, m.blocks);
        FO_CHECK(armed.rows * m.kmax < (1LL << 31), "hand-off: %d chunks of %lld rows per session are too many rows", m.kmax, armed.rows);
        FO_CHECK(!adapter_out && !c->handoff, "an armed hand-off replaces adapter_out: pass NULL");
        FO_CHECK(armed.rows >= armed.prefix + t_out, "hand-off: %d adapter rows behind a %lld-row prefix do not fit %lld rows per session",
                 t_out, armed.prefix, armed.rows);
        c->handoff = armed.embeds;
        c->handoff_rows = armed.rows;
        c->handoff_off = armed.prefix;
    }
    struct HandoffReset { fo_ctx* c; bool on; ~HandoffReset() { if (on) { c->handoff = nullptr; c->handoff_rows = c->handoff_off = 0; } } } hreset{c, armed.on};
    FO_TRY(upload_ids(c, ids, n, st, armed.on ? armed.onset.data() : nullptr, m.blocks, chunks));
    c->pf_slot_lo = c->pf_slot_hi = ids[0];
    for (int i = 1; i < n; ++i) { c->pf_slot_lo = std::min(c->pf_slot_lo, (int)ids[i]); c->pf_slot_hi = std::max(c->pf_slot_hi, (int)ids[i]); }
    StepArgs a{n, t_in, m, pcm != nullptr, adapter_out != nullptr, pcm_dtype == FO_I16, scale, 0};
    void* stage;
    if (pcm) {
        const size_t in_bytes = (size_t)n * c->chunk_samples * (pcm_dtype == FO_I16 ? 2 : 4);
        FO_TRY(ws_ensure(c, WS_PCM, (size_t)n * c->chunk_samples * 4, &stage));
        FO_CUDA(cudaMemcpyAsync(stage, pcm, in_bytes, cudaMemcpyDefault, st));
    } else if (feats) {
        const size_t in_bytes = (size_t)m.blocks * t_in * c->F * sizeof(float);
        FO_TRY(ws_ensure(c, WS_FEATS, in_bytes, &stage));
        FO_CUDA(cudaMemcpyAsync(stage, feats, in_bytes, cudaMemcpyDefault, st));
    } else {
        // the block fo_fbank_stream left in the sessions' feature rings
        FO_TRY(ws_ensure(c, WS_FEATS, (size_t)n * t_in * c->F * sizeof(float), &stage));
        for (int i = 0; i < n; ++i)
            FO_CUDA(cudaMemcpyAsync((float*)stage + (size_t)i * t_in * c->F, c->feat_ring + (size_t)ids[i] * t_in * c->F,
                                    (size_t)t_in * c->F * sizeof(float), cudaMemcpyDeviceToDevice, st));
    }
    FO_TRY(run_step(c, a, st));
    if (armed.on && armed.attn_mask)
        FO_TRY(handoff_mask(c->onset_dev, armed.prefix_mask, m.blocks, (int)armed.prefix, t_out, (int)armed.rows, armed.attn_mask, armed.row_start, st));
    if (enc_out) FO_CUDA(cudaMemcpyAsync(enc_out, c->ws[WS_ENC].p, enc_bytes, cudaMemcpyDefault, st));
    if (adapter_out) FO_CUDA(cudaMemcpyAsync(adapter_out, c->ws[WS_Y].p, y_bytes, cudaMemcpyDefault, st));
    if (!c->ev_sync) FO_CUDA(cudaEventCreateWithFlags(&c->ev_sync, cudaEventDisableTiming));
    FO_CUDA(cudaEventRecord(c->ev_sync, st));
    c->stats.stream_steps += 1;
    c->stats.session_chunks += m.blocks;
    return 0;
}

int fo_encode_stream(fo_ctx* c, const int32_t* ids, int n, const float* feats, int t_in, float* enc_out,
                     float* adapter_out, void* stream) {
    FO_CHECK(c && c->finalized && c->cfg.has_encoder, "fo_encode_stream: context has no finalized encoder");
    FO_TRY(check_ids(c, ids, n));
    FO_CUDA(cudaSetDevice(c->device));
    FO_ON_GROUP(c, stream);
    if (feats) FO_CHECK(t_in >= 7, "fo_encode_stream: need at least 7 feature frames");
    else t_in = c->cfg.context_frames + c->cfg.frames_per_chunk;
    Mix m;
    m.blocks = m.n1 = n;
    return stream_common(c, ids, n, nullptr, m, nullptr, FO_F32, 1.0f, feats, t_in, enc_out, adapter_out, (cudaStream_t)stream);
}

int fo_encode_stream_chunks(fo_ctx* c, const int32_t* ids, int n, int k, const float* feats, int t_in, float* enc_out,
                            float* adapter_out, void* stream) {
    FO_CHECK(c && c->finalized && c->cfg.has_encoder, "fo_encode_stream_chunks: context has no finalized encoder");
    FO_CHECK(feats, "fo_encode_stream_chunks: feats must not be NULL (the feature ring holds one block per session)");
    FO_CHECK(k >= 1, "fo_encode_stream_chunks: k must be >= 1");
    FO_CHECK(t_in >= 7, "fo_encode_stream_chunks: need at least 7 feature frames per chunk");
    FO_TRY(check_ids(c, ids, n));
    FO_TRY(stream_geometry(c, t_in));
    const int t = ((t_in - 1) / 2 - 1) / 2;
    if (k > 1) {
        const int kmax = std::max(1, (STREAM_CHUNKS_MAX_KEYS - c->window) / t);
        FO_CHECK(c->window + k * t <= STREAM_CHUNKS_MAX_KEYS,
                 "fo_encode_stream_chunks: the attention window (%d frames) + %d chunks x %d frames exceeds %d keys; the largest k is %d",
                 c->window, k, t, STREAM_CHUNKS_MAX_KEYS, kmax);
    }
    FO_CUDA(cudaSetDevice(c->device));
    FO_ON_GROUP(c, stream);
    // the uniform case of fo_encode_stream_chunks_v: every session brings k chunks
    const std::vector<int32_t> chunks(n, k);
    Mix m;
    m.blocks = n * k;
    m.kmax = k;
    m.n1 = k == 1 ? n : 0;
    return stream_common(c, ids, n, k > 1 ? chunks.data() : nullptr, m, nullptr, FO_F32, 1.0f, feats, t_in, enc_out, adapter_out,
                         (cudaStream_t)stream);
}

int fo_encode_stream_chunks_v(fo_ctx* c, const int32_t* ids, const int32_t* chunks, int n, const float* feats, int t_in,
                              float* enc_out, float* adapter_out, void* stream) {
    FO_CHECK(c && c->finalized && c->cfg.has_encoder, "fo_encode_stream_chunks_v: context has no finalized encoder");
    FO_CHECK(feats, "fo_encode_stream_chunks_v: feats must not be NULL (the feature ring holds one block per session)");
    FO_CHECK(chunks, "fo_encode_stream_chunks_v: chunks must be a host array of n counts");
    FO_CHECK(t_in >= 7, "fo_encode_stream_chunks_v: need at least 7 feature frames per chunk");
    FO_TRY(check_ids(c, ids, n));
    FO_TRY(stream_geometry(c, t_in));
    const int t = ((t_in - 1) / 2 - 1) / 2;
    const int kcap = std::max(1, (STREAM_CHUNKS_MAX_KEYS - c->window) / t);
    std::vector<int32_t> off(n + 1, 0);
    Mix m;
    for (int i = 0; i < n; ++i) {
        FO_CHECK(chunks[i] >= 1, "fo_encode_stream_chunks_v: session %d (id %d) has chunk count %d; counts must be >= 1", i, ids[i], chunks[i]);
        FO_CHECK(c->window + (long long)chunks[i] * t <= STREAM_CHUNKS_MAX_KEYS,
                 "fo_encode_stream_chunks_v: session %d (id %d): the attention window (%d frames) + %d chunks x %d frames exceeds %d keys; "
                 "the largest count is %d", i, ids[i], c->window, chunks[i], t, STREAM_CHUNKS_MAX_KEYS, kcap);
        off[i + 1] = off[i] + chunks[i];
        m.kmax = std::max(m.kmax, (int)chunks[i]);
        if (m.n1 == i && chunks[i] == 1) m.n1 = i + 1;
    }
    m.blocks = off[n];
    if (!m.uniform(n)) m.off = off.data();
    FO_CUDA(cudaSetDevice(c->device));
    FO_ON_GROUP(c, stream);
    return stream_common(c, ids, n, m.kmax > 1 ? chunks : nullptr, m, nullptr, FO_F32, 1.0f, feats, t_in, enc_out, adapter_out,
                         (cudaStream_t)stream);
}

int fo_handoff_arm(fo_ctx* c, int n, void* embeds_f16, int64_t rows_per_session, int64_t prefix_len, const uint8_t* onset,
                   const uint8_t* prefix_mask, uint8_t* attn_mask, int32_t* row_start) {
    FO_CHECK(c && c->finalized && c->cfg.has_encoder && c->cfg.has_adapter, "fo_handoff_arm: context needs a finalized encoder + adapter");
    FO_CHECK(c->dtype == FO_BF16, "fo_handoff_arm: the fp16 hand-off is built for bf16 contexts");
    // n blocks: one per session, or per (session, chunk) of a multi-chunk or recording call -- the latter has no cap on the
    // counts, so neither has n; a call of another block count refuses the arm
    FO_CHECK(n > 0 && embeds_f16 && onset, "fo_handoff_arm: bad argument");
    FO_CHECK(prefix_len >= 0 && rows_per_session > prefix_len && rows_per_session < (1LL << 31), "fo_handoff_arm: bad row counts");
    cudaPointerAttributes pa;
    FO_CHECK(cudaPointerGetAttributes(&pa, embeds_f16) == cudaSuccess && pa.type == cudaMemoryTypeDevice && pa.device == c->device,
             "fo_handoff_arm: embeds must be device memory of this context's GPU");
    if (attn_mask) FO_CHECK(is_device_ptr(attn_mask) && (!row_start || is_device_ptr(row_start)) && (!prefix_mask || is_device_ptr(prefix_mask)),
                            "fo_handoff_arm: attn_mask, row_start and prefix_mask are device pointers");
    c->armed.on = true;
    c->armed.embeds = embeds_f16;
    c->armed.rows = rows_per_session;
    c->armed.prefix = prefix_len;
    c->armed.n = n;
    c->armed.onset.assign(onset, onset + n);
    c->armed.prefix_mask = prefix_mask;
    c->armed.attn_mask = attn_mask;
    c->armed.row_start = row_start;
    return 0;
}

int fo_stream_step_embeds(fo_ctx* c, const int32_t* ids, int n, const void* pcm, int pcm_dtype, float scale, float* enc_out,
                          void* embeds_f16, int64_t rows_per_session, int64_t row_offset, void* stream) {
    FO_CHECK(c && c->finalized && c->cfg.has_encoder && c->cfg.has_adapter && c->fb_window,
             "fo_stream_step_embeds: context needs a finalized frontend + encoder + adapter");
    FO_CHECK(c->dtype == FO_BF16, "fo_stream_step_embeds: the fp16 hand-off is built for bf16 contexts");
    FO_CHECK(pcm && (pcm_dtype == FO_F32 || pcm_dtype == FO_I16), "fo_stream_step_embeds: pcm must be FO_F32 or FO_I16");
    FO_TRY(check_ids(c, ids, n));
    FO_CUDA(cudaSetDevice(c->device));
    FO_ON_GROUP(c, stream);
    const int t_in = c->cfg.context_frames + c->cfg.frames_per_chunk;
    const int t = ((t_in - 1) / 2 - 1) / 2, t_out = ad_frames(c, t);
    FO_CHECK(embeds_f16 && row_offset >= 0 && rows_per_session >= row_offset + t_out && rows_per_session < (1LL << 31),
             "fo_stream_step_embeds: a session's %d rows at offset %lld do not fit %lld rows per session", t_out,
             (long long)row_offset, (long long)rows_per_session);
    cudaPointerAttributes pa;
    FO_CHECK(cudaPointerGetAttributes(&pa, embeds_f16) == cudaSuccess && pa.type == cudaMemoryTypeDevice && pa.device == c->device,
             "fo_stream_step_embeds: embeds must be device memory of this context's GPU");
    c->handoff = embeds_f16;
    c->handoff_rows = rows_per_session;
    c->handoff_off = row_offset;
    Mix m;
    m.blocks = m.n1 = n;
    const int r = stream_common(c, ids, n, nullptr, m, pcm, pcm_dtype, scale, nullptr, t_in, enc_out, nullptr, (cudaStream_t)stream);
    c->handoff = nullptr;
    c->handoff_rows = c->handoff_off = 0;
    return r;
}

int fo_stream_step_async(fo_ctx* c, const int32_t* ids, int n, const void* pcm, int pcm_dtype, float scale, float* enc_out,
                         float* adapter_out, void* stream, int64_t* ticket) {
    FO_CHECK(c && c->finalized && c->cfg.has_encoder && c->fb_window, "fo_stream_step_async: context has no finalized encoder + frontend");
    FO_CHECK(pcm && (pcm_dtype == FO_F32 || pcm_dtype == FO_I16) && ticket, "fo_stream_step_async: bad argument");
    FO_CHECK(!c->KM, "fo_stream_step_async: MultiLayeredConv1d has no streaming form; use fo_encode_offline");
    if (adapter_out) FO_CHECK(c->cfg.has_adapter, "adapter_out requested but the context has no adapter");
    FO_TRY(check_ids(c, ids, n));
    FO_TRY(stream_geometry(c, c->cfg.context_frames + c->cfg.frames_per_chunk));
    FO_CUDA(cudaSetDevice(c->device));
    FO_ON_GROUP(c, stream);
    cudaStream_t st = (cudaStream_t)stream;
    if (!c->copy_stream) {
        FO_TRY(make_stream(c, &c->copy_stream));
        FO_TRY(make_stream(c, &c->upload_stream));
        for (int i = 0; i < 2; ++i) {
            FO_CUDA(cudaEventCreateWithFlags(&c->ev_in[i], cudaEventDisableTiming));
            FO_CUDA(cudaEventCreateWithFlags(&c->ev_compute[i], cudaEventDisableTiming));
            FO_CUDA(cudaEventCreateWithFlags(&c->ev_out[i], cudaEventDisableTiming));
        }
    }
    const int buf = (int)(c->async_ticket & 1);
    const int t_in = c->cfg.context_frames + c->cfg.frames_per_chunk;
    const int t = ((t_in - 1) / 2 - 1) / 2, t_out = ad_frames(c, t);
    FO_TRY(upload_ids(c, ids, n, st));
    c->pf_slot_lo = c->pf_slot_hi = ids[0];
    for (int i = 1; i < n; ++i) { c->pf_slot_lo = std::min(c->pf_slot_lo, (int)ids[i]); c->pf_slot_hi = std::max(c->pf_slot_hi, (int)ids[i]); }
    Mix m;
    m.blocks = m.n1 = n;
    StepArgs a{n, t_in, m, true, adapter_out != nullptr, pcm_dtype == FO_I16, scale, buf};
    // inputs: copy stream, once the step that last read this PCM buffer (two tickets ago) is done
    void* stage;
    FO_TRY(ws_ensure(c, ws_pcm(buf), (size_t)n * c->chunk_samples * 4, &stage));
    if (c->async_ticket >= 2) FO_CUDA(cudaStreamWaitEvent(c->upload_stream, c->ev_compute[buf], 0));
    // a synchronous step still queued on `st` stages its PCM in WS_PCM as well and reads the shared intermediates
    if (c->ev_sync) FO_CUDA(cudaStreamWaitEvent(c->upload_stream, c->ev_sync, 0));
    FO_CUDA(cudaMemcpyAsync(stage, pcm, (size_t)n * c->chunk_samples * (pcm_dtype == FO_I16 ? 2 : 4), cudaMemcpyDefault, c->upload_stream));
    FO_CUDA(cudaEventRecord(c->ev_in[buf], c->upload_stream));
    FO_CUDA(cudaStreamWaitEvent(st, c->ev_in[buf], 0));
    // outputs of two tickets ago must have left this buffer set before the step overwrites it
    if (c->async_ticket >= 2) FO_CUDA(cudaStreamWaitEvent(st, c->ev_out[buf], 0));
    FO_TRY(run_step(c, a, st));
    FO_CUDA(cudaEventRecord(c->ev_compute[buf], st));
    FO_CUDA(cudaStreamWaitEvent(c->copy_stream, c->ev_compute[buf], 0));
    if (enc_out) FO_CUDA(cudaMemcpyAsync(enc_out, c->ws[ws_enc(buf)].p, (size_t)n * t * c->D * sizeof(float), cudaMemcpyDefault, c->copy_stream));
    if (adapter_out) FO_CUDA(cudaMemcpyAsync(adapter_out, c->ws[ws_y(buf)].p, (size_t)n * t_out * c->E * sizeof(float), cudaMemcpyDefault, c->copy_stream));
    FO_CUDA(cudaEventRecord(c->ev_out[buf], c->copy_stream));
    *ticket = c->async_ticket++;
    c->stats.stream_steps += 1;
    c->stats.session_chunks += n;
    return 0;
}

int fo_stream_wait(fo_ctx* c, int64_t ticket) {
    FO_CHECK(c && c->copy_stream && ticket >= 0 && ticket < c->async_ticket, "fo_stream_wait: unknown ticket");
    FO_CHECK(c->async_ticket - ticket <= 2, "fo_stream_wait: ticket %lld is older than the two steps in flight", (long long)ticket);
    FO_CUDA(cudaSetDevice(c->device));
    FO_CUDA(cudaEventSynchronize(c->ev_out[ticket & 1]));
    return 0;
}

int fo_stream_step(fo_ctx* c, const int32_t* ids, int n, const void* pcm, int pcm_dtype, float scale, float* enc_out,
                   float* adapter_out, void* stream) {
    FO_CHECK(c && c->finalized && c->cfg.has_encoder && c->fb_window, "fo_stream_step: context has no finalized encoder + frontend");
    FO_CHECK(pcm && (pcm_dtype == FO_F32 || pcm_dtype == FO_I16), "fo_stream_step: pcm must be FO_F32 or FO_I16");
    FO_TRY(check_ids(c, ids, n));
    FO_CUDA(cudaSetDevice(c->device));
    FO_ON_GROUP(c, stream);
    Mix m;
    m.blocks = m.n1 = n;
    return stream_common(c, ids, n, nullptr, m, pcm, pcm_dtype, scale, nullptr, c->cfg.context_frames + c->cfg.frames_per_chunk, enc_out,
                         adapter_out, (cudaStream_t)stream);
}

// ---- recorded audio: many chunks per session, exact-streaming ----------------------------------------
// The recording entries (fo_stream_steps_v, fo_fbank_stream_v, fo_encode_stream_steps_v) run in passes of at most P blocks
// (option "steps_pass_blocks", else STEPS_PASS_BYTES over the workspace bytes of one block): each pass gives every session that
// still has chunks its next min(remaining, q) chunks, q = the longest remaining count spread evenly over the passes that
// max(1, P / sessions left) chunks per pass would take.  A pass takes its blocks' features from PCM (fbank_stream_blocks) or
// from the caller, then runs the streaming program, whose attention spreads a session's chunks over groups of CTAs (Mix::group).
// Every workspace is sized by the pass, so the device memory a call adds does not grow with the recording.
// Passes run eagerly: a captured graph per pass shape would multiply with recording lengths.
constexpr long long STEPS_PASS_BYTES = 1LL << 30;

// workspace bytes one block of a pass adds: PCM and sample rows, features, conv1 planes (the six-plane implicit-GEMM operand
// of conv2) and conv2 rows, residual / LayerNorm / attention rows, QKV (+ fp32 Q), FFN hidden rows, encoder and adapter rows
static long long steps_block_bytes(const fo_ctx* c, int t_in) {
    const int t = ((t_in - 1) / 2 - 1) / 2, t_out = ad_frames(c, t);
    const long long esz = (long long)c->esz, D = c->D;
    long long b = (long long)(2 * c->chunk_samples + c->carry) * 4 + (long long)t_in * c->F * 4;
    b += 6LL * t * (c->F2 + 1) * D * esz + (long long)t * c->F2 * D * esz;
    b += (long long)t * D * (4 + 4 + 4 + 5 * esz) + (long long)t * 3 * D * (esz + 4) + (long long)t * c->FF * esz;
    if (c->cfg.has_adapter) b += (long long)t * 4 * D * (esz + 4) + (long long)t_out * c->E * 4;
    return b;
}

static int steps_pass_blocks(const fo_ctx* c, int t_in) {
    return c->steps_pass_blocks > 0 ? c->steps_pass_blocks
                                    : (int)std::max(1LL, std::min(1LL << 20, STEPS_PASS_BYTES / steps_block_bytes(c, t_in)));
}

static int check_steps_counts(const char* fn, const int32_t* ids, const int32_t* chunks, int n) {
    for (int i = 0; i < n; ++i)
        FO_CHECK(chunks[i] >= 1, "%s: session %d (id %d) has chunk count %d; counts must be >= 1", fn, i, ids[i], chunks[i]);
    return 0;
}

// What one recording call reads and writes.  Blocks come from PCM (pcm != null) or from the caller's features (feats);
// feats_out receives the features of PCM blocks; with `encode` the blocks run through the encoder into enc_out / adapter_out.
struct StepsIo {
    const void* pcm = nullptr;
    int pcm_dtype = FO_F32;
    float scale = 1.0f;
    const float* feats = nullptr;
    float* feats_out = nullptr;
    bool encode = false;
    float* enc_out = nullptr;
    float* adapter_out = nullptr;
    const fo_ctx::Armed* armed = nullptr;   // the hand-off this call took (fo_handoff_arm), in place of adapter_out
};

// The pass loop shared by the recording entries; arguments are checked by the caller, so nothing here refuses a call.
static int steps_passes(fo_ctx* c, const int32_t* ids, const int32_t* chunks, int n, int t_in, const StepsIo& io, cudaStream_t st) {
    std::vector<long long> off(n + 1, 0);
    for (int i = 0; i < n; ++i) off[i + 1] = off[i] + chunks[i];
    if (c->copy_stream && c->async_ticket > 0) {       // as in stream_common: pipelined steps still read the shared buffers
        FO_CUDA(cudaStreamWaitEvent(st, c->ev_out[0], 0));
        if (c->async_ticket > 1) FO_CUDA(cudaStreamWaitEvent(st, c->ev_out[1], 0));
    }
    const int T1 = (t_in - 1) / 2, t = (T1 - 1) / 2, t_out = c->cfg.has_encoder ? ad_frames(c, t) : 0;
    const int P = steps_pass_blocks(c, t_in);
    const long long pcm_row = (long long)c->chunk_samples * (io.pcm_dtype == FO_I16 ? 2 : 4);
    const long long feat_row = (long long)t_in * c->F, enc_row = (long long)t * c->D, y_row = (long long)t_out * c->E;
    const fo_ctx::Armed* ho = io.armed;
    const bool want_y = io.adapter_out != nullptr || ho;
    long long tab_pos = 0;
    if (ho) {
        // the pass tables of the whole call, in pinned memory: wait until the previous armed call has uploaded its own
        if (c->ho_tab_event) FO_CUDA(cudaEventSynchronize(c->ho_tab_event));
        else FO_CUDA(cudaEventCreateWithFlags(&c->ho_tab_event, cudaEventDisableTiming));
        if (c->ho_tab_cap < off[n]) {
            if (c->ho_tab_host) FO_CUDA(cudaFreeHost(c->ho_tab_host));
            c->ho_tab_host = nullptr;
            c->ho_tab_cap = 0;
            FO_CUDA(cudaMallocHost((void**)&c->ho_tab_host, (size_t)off[n] * sizeof(int2)));
            c->ho_tab_cap = off[n];
        }
    }
    const int sms = c->sms;
    const int gmax = std::max(1, (STREAM_CHUNKS_MAX_KEYS - c->window) / std::max(1, t));
    g_use_pdl = g_want_pdl;
    std::vector<int32_t> done(n, 0), pids, pcnt, poff, psrc;
    for (;;) {
        pids.clear(); pcnt.clear(); psrc.clear();
        for (int i = 0; i < n; ++i) if (done[i] < chunks[i]) psrc.push_back(i);
        const int na = (int)psrc.size();
        if (na == 0) break;
        // at most P / na chunks per session, spread evenly over the passes the longest session still needs
        int q = std::max(1, P / na), rmax = 0;
        for (int i : psrc) rmax = std::max(rmax, chunks[i] - done[i]);
        q = (rmax + (rmax + q - 1) / q - 1) / ((rmax + q - 1) / q);
        poff.assign(1, 0);
        Mix m;
        for (int i : psrc) {
            pids.push_back(ids[i]);
            pcnt.push_back(std::min(q, chunks[i] - done[i]));
            poff.push_back(poff.back() + pcnt.back());
            m.kmax = std::max(m.kmax, (int)pcnt.back());
        }
        m.blocks = poff.back();
        m.off = poff.data();
        FO_TRY(upload_ids(c, pids.data(), na, st, nullptr, 0, pcnt.data()));
        c->pf_slot_lo = *std::min_element(pids.begin(), pids.end());
        c->pf_slot_hi = *std::max_element(pids.begin(), pids.end());
        void *dpcm = nullptr, *drows = nullptr, *dfeats, *denc = nullptr, *dy = nullptr;
        if (io.pcm) {
            FO_TRY(ws_ensure(c, WS_PCM, (size_t)m.blocks * c->chunk_samples * 4, &dpcm));
            FO_TRY(ws_ensure(c, WS_SROWS, (size_t)m.blocks * (c->carry + c->chunk_samples) * sizeof(float), &drows));
        }
        FO_TRY(ws_ensure(c, WS_FEATS, (size_t)m.blocks * feat_row * sizeof(float), &dfeats));
        if (io.encode) {
            FO_TRY(ws_ensure(c, WS_ENC, (size_t)m.blocks * enc_row * sizeof(float), &denc));
            if (want_y) FO_TRY(ws_ensure(c, WS_Y, (size_t)m.blocks * y_row * sizeof(float), &dy));
        }
        if (io.pcm) {
            for (int a = 0; a < na; ++a) {
                const int i = psrc[a];
                FO_CUDA(cudaMemcpyAsync((char*)dpcm + poff[a] * pcm_row, (const char*)io.pcm + (off[i] + done[i]) * pcm_row,
                                        pcnt[a] * pcm_row, cudaMemcpyDefault, st));
            }
            FO_TRY(fbank_stream_blocks(fbank_params(c), c->ids_dev, c->cnt_dev, c->off_dev, na, m.kmax, m.blocks, dpcm,
                                       io.pcm_dtype == FO_I16, io.scale, c->cfg.frames_per_chunk, c->cfg.context_frames, c->samples,
                                       c->feat_ring, (float*)drows, (float*)dfeats, st));
        } else {
            for (int a = 0; a < na; ++a) {
                const int i = psrc[a];
                FO_CUDA(cudaMemcpyAsync((float*)dfeats + poff[a] * feat_row, io.feats + (off[i] + done[i]) * feat_row,
                                        pcnt[a] * feat_row * sizeof(float), cudaMemcpyDefault, st));
            }
        }
        if (io.feats_out)
            for (int a = 0; a < na; ++a) {
                const int i = psrc[a];
                FO_CUDA(cudaMemcpyAsync(io.feats_out + (off[i] + done[i]) * feat_row, (float*)dfeats + poff[a] * feat_row,
                                        pcnt[a] * feat_row * sizeof(float), cudaMemcpyDefault, st));
            }
        if (io.encode) {
            // chunks per attention CTA: enough (session, head, group) CTAs to fill the SMs, each staging at most 128 keys
            const int want = std::max(1, (sms + na * c->H - 1) / (na * c->H));
            m.group = std::min(gmax, std::max(1, (m.kmax + want - 1) / want));
            FO_TRY(c->dtype == FO_BF16 ? stream_program<act16>(c, na, m, (const float*)dfeats, t_in, (float*)denc, (float*)dy, st)
                                       : stream_program<float>(c, na, m, (const float*)dfeats, t_in, (float*)denc, (float*)dy, st));
            for (int a = 0; a < na; ++a) {
                const int i = psrc[a];
                const long long b0 = off[i] + done[i];
                if (io.enc_out) FO_CUDA(cudaMemcpyAsync(io.enc_out + b0 * enc_row, (float*)denc + poff[a] * enc_row,
                                                        pcnt[a] * enc_row * sizeof(float), cudaMemcpyDefault, st));
                if (io.adapter_out) FO_CUDA(cudaMemcpyAsync(io.adapter_out + b0 * y_row, (float*)dy + poff[a] * y_row,
                                                            pcnt[a] * y_row * sizeof(float), cudaMemcpyDefault, st));
            }
            if (ho) {
                // pass block poff[a] + j is chunk done_i + j of session i, the caller's block off_i + done_i + j
                int2* tab = c->ho_tab_host + tab_pos;
                for (int a = 0; a < na; ++a) {
                    const int i = psrc[a];
                    for (int j = 0; j < pcnt[a]; ++j) {
                        const long long d = off[i] + done[i] + j;
                        tab[poff[a] + j] = make_int2((int)d, ho->onset[d]);
                    }
                }
                void* dtab;
                FO_TRY(ws_ensure(c, WS_HOTAB, (size_t)m.blocks * sizeof(int2), &dtab));
                FO_CUDA(cudaMemcpyAsync(dtab, tab, (size_t)m.blocks * sizeof(int2), cudaMemcpyHostToDevice, st));
                FO_TRY(handoff_rows((const float*)dy, (const int2*)dtab, m.blocks, t_out, c->E, ho->embeds, (int)ho->rows, (int)ho->prefix,
                                    ho->prefix_mask, ho->attn_mask, ho->row_start, c->sat_counter, st));
                tab_pos += m.blocks;
            }
        }
        for (int a = 0; a < na; ++a) done[psrc[a]] += pcnt[a];
    }
    if (ho) FO_CUDA(cudaEventRecord(c->ho_tab_event, st));
    if (!c->ev_sync) FO_CUDA(cudaEventCreateWithFlags(&c->ev_sync, cudaEventDisableTiming));
    FO_CUDA(cudaEventRecord(c->ev_sync, st));
    if (io.encode) {
        c->stats.stream_steps += 1;
        c->stats.session_chunks += off[n];
    }
    return 0;
}

// the refusals of the encoding recording entries (fo_stream_steps_v, fo_encode_stream_steps_v).  Unlike stream_common, a refused
// call leaves an armed hand-off armed: nothing here consumes it.
static int check_steps_encode(fo_ctx* c, const char* fn, const int32_t* ids, const int32_t* chunks, int n, int t_in,
                              const float* adapter_out) {
    FO_CHECK(chunks, "%s: chunks must be a host array of n counts", fn);
    FO_TRY(check_ids(c, ids, n));
    FO_TRY(stream_geometry(c, t_in));
    FO_CHECK(!c->KM, "%s: MultiLayeredConv1d has no streaming form (models/encoder/attention.py:145-196); use fo_encode_offline", fn);
    if (adapter_out) FO_CHECK(c->cfg.has_adapter, "adapter_out requested but the context has no adapter");
    FO_TRY(check_steps_counts(fn, ids, chunks, n));
    if (c->armed.on) {
        long long blocks = 0;
        for (int i = 0; i < n; ++i) blocks += chunks[i];
        const int t_out = ad_frames(c, ((t_in - 1) / 2 - 1) / 2);
        FO_CHECK(c->armed.n == blocks, "%s: the LLM hand-off is armed for %d blocks (fo_handoff_arm), this call brings %lld; "
                                       "it stays armed", fn, c->armed.n, blocks);
        FO_CHECK(!adapter_out, "%s: an armed LLM hand-off replaces adapter_out: pass NULL (the hand-off stays armed)", fn);
        FO_CHECK(c->armed.rows >= c->armed.prefix + t_out, "%s: the armed hand-off's %lld rows per block do not hold %d adapter rows "
                 "behind a %lld-row prefix; it stays armed", fn, c->armed.rows, t_out, c->armed.prefix);
    }
    return 0;
}

// after check_steps_encode: the call takes the armed hand-off, if any, into `armed` (io.armed points at it)
static void take_arm(fo_ctx* c, fo_ctx::Armed* armed, StepsIo* io) {
    if (!c->armed.on) return;
    *armed = c->armed;
    c->armed.on = false;
    io->armed = armed;
}

int fo_stream_steps_v(fo_ctx* c, const int32_t* ids, const int32_t* chunks, int n, const void* pcm, int pcm_dtype, float scale,
                      float* enc_out, float* adapter_out, void* stream) {
    FO_CHECK(c && c->finalized && c->cfg.has_encoder && c->fb_window, "fo_stream_steps_v: context has no finalized encoder + frontend");
    FO_CHECK(pcm && (pcm_dtype == FO_F32 || pcm_dtype == FO_I16), "fo_stream_steps_v: pcm must be FO_F32 or FO_I16");
    const int t_in = c->cfg.context_frames + c->cfg.frames_per_chunk;
    FO_TRY(check_steps_encode(c, "fo_stream_steps_v", ids, chunks, n, t_in, adapter_out));
    FO_CUDA(cudaSetDevice(c->device));
    FO_ON_GROUP(c, stream);
    StepsIo io;
    io.pcm = pcm;
    io.pcm_dtype = pcm_dtype;
    io.scale = scale;
    io.encode = true;
    io.enc_out = enc_out;
    io.adapter_out = adapter_out;
    fo_ctx::Armed armed;
    take_arm(c, &armed, &io);
    return steps_passes(c, ids, chunks, n, t_in, io, (cudaStream_t)stream);
}

int fo_encode_stream_steps_v(fo_ctx* c, const int32_t* ids, const int32_t* chunks, int n, const float* feats, int t_in,
                             float* enc_out, float* adapter_out, void* stream) {
    FO_CHECK(c && c->finalized && c->cfg.has_encoder, "fo_encode_stream_steps_v: context has no finalized encoder");
    FO_CHECK(feats, "fo_encode_stream_steps_v: feats must not be NULL");
    FO_CHECK(t_in >= 7, "fo_encode_stream_steps_v: need at least 7 feature frames per chunk");
    FO_TRY(check_steps_encode(c, "fo_encode_stream_steps_v", ids, chunks, n, t_in, adapter_out));
    FO_CUDA(cudaSetDevice(c->device));
    FO_ON_GROUP(c, stream);
    StepsIo io;
    io.feats = feats;
    io.encode = true;
    io.enc_out = enc_out;
    io.adapter_out = adapter_out;
    fo_ctx::Armed armed;
    take_arm(c, &armed, &io);
    return steps_passes(c, ids, chunks, n, t_in, io, (cudaStream_t)stream);
}

int fo_fbank_stream_v(fo_ctx* c, const int32_t* ids, const int32_t* chunks, int n, const void* pcm, int pcm_dtype, float scale,
                      float* feats_out, void* stream) {
    FO_CHECK(c && c->finalized && c->fb_window, "fo_fbank_stream_v: context has no finalized frontend");
    FO_CHECK(pcm && (pcm_dtype == FO_F32 || pcm_dtype == FO_I16), "fo_fbank_stream_v: pcm must be FO_F32 or FO_I16");
    FO_CHECK(chunks, "fo_fbank_stream_v: chunks must be a host array of n counts");
    FO_TRY(check_ids(c, ids, n));
    FO_TRY(check_steps_counts("fo_fbank_stream_v", ids, chunks, n));
    FO_CUDA(cudaSetDevice(c->device));
    FO_ON_GROUP(c, stream);
    StepsIo io;
    io.pcm = pcm;
    io.pcm_dtype = pcm_dtype;
    io.scale = scale;
    io.feats_out = feats_out;
    return steps_passes(c, ids, chunks, n, c->cfg.context_frames + c->cfg.frames_per_chunk, io, (cudaStream_t)stream);
}

// ---- full utterance -----------------------------------------------------------------------------------
int fo_encode_offline(fo_ctx* c, const float* feats, const int32_t* ilens, int B, int T, int chunk, int left,
                      float* enc_out, uint8_t* mask_out, float* adapter_out, uint8_t* adapter_mask_out, void* stream) {
    FO_CHECK(c && c->finalized && c->cfg.has_encoder, "fo_encode_offline: context has no finalized encoder");
    FO_CHECK(feats && ilens && B > 0 && T >= 7, "fo_encode_offline: need feats, ilens and T >= 7");
    const int T1 = (T - 1) / 2, T2 = (T1 - 1) / 2;
    FO_CHECK(T2 <= c->cfg.pos_max_len, "fo_encode_offline: %d encoder frames exceed the positional table (%d)", T2, c->cfg.pos_max_len);
    FO_CUDA(cudaSetDevice(c->device));
    FO_ON_GROUP(c, stream);
    cudaStream_t st = (cudaStream_t)stream;
    const void *dfeats, *dil;
    FO_TRY(in_dev(c, feats, (size_t)B * T * c->F * sizeof(float), WS_FEATS, st, &dfeats));
    FO_TRY(in_dev(c, ilens, (size_t)B * sizeof(int32_t), WS_ILENS, st, &dil));
    const int t_out = ad_frames(c, T2);
    const size_t enc_bytes = (size_t)B * T2 * c->D * sizeof(float), y_bytes = (size_t)B * t_out * c->E * sizeof(float);
    void *denc, *dy = nullptr, *dmask, *dil2, *damask = nullptr;
    FO_TRY(out_dev(c, enc_out, enc_bytes, WS_ENC, &denc));
    FO_TRY(out_dev(c, mask_out, (size_t)B * T2, WS_MASK2, &dmask));
    FO_TRY(ws_ensure(c, WS_ILENS2, (size_t)B * sizeof(int32_t), &dil2));
    if (adapter_out || adapter_mask_out) FO_CHECK(c->cfg.has_adapter, "adapter outputs requested but the context has no adapter");
    if (adapter_out) FO_TRY(out_dev(c, adapter_out, y_bytes, WS_Y, &dy));
    int r = c->dtype == FO_BF16
                ? offline_program<act16>(c, (const float*)dfeats, (const int32_t*)dil, B, T, chunk, left, (float*)denc,
                                        (uint8_t*)dmask, (int32_t*)dil2, (float*)dy, st)
                : offline_program<float>(c, (const float*)dfeats, (const int32_t*)dil, B, T, chunk, left, (float*)denc,
                                         (uint8_t*)dmask, (int32_t*)dil2, (float*)dy, st);
    FO_TRY(r);
    if (adapter_mask_out) {
        FO_TRY(out_dev(c, adapter_mask_out, (size_t)B * t_out, WS_AMASK, &damask));
        if (c->cfg.adapter_type != 0) FO_CUDA(cudaMemcpyAsync(damask, dmask, (size_t)B * T2, cudaMemcpyDeviceToDevice, st));   // mask unchanged
        else FO_TRY(stride2_mask((const uint8_t*)dmask, B, T2, t_out, (uint8_t*)damask, st));
        FO_TRY(out_done(adapter_mask_out, damask, (size_t)B * t_out, st));
    }
    if (enc_out) FO_TRY(out_done(enc_out, denc, enc_bytes, st));
    if (mask_out) FO_TRY(out_done(mask_out, dmask, (size_t)B * T2, st));
    if (adapter_out) FO_TRY(out_done(adapter_out, dy, y_bytes, st));
    c->stats.offline_calls += 1;
    c->stats.offline_frames += (long long)B * T2;
    return 0;
}

// ---- full utterances packed end to end ---------------------------------------------------------------------
// PackTab of B utterances of T[b] feature frames (refusals name utterance b0 + b of the caller's call).  soff (optional, the
// PCM entry): each utterance's first sample, appended to the table as int64.
static int pack_tab(fo_ctx* c, const int32_t* T, int B, const char* who, int b0, const long long* soff, PackTab* pt) {
    PackTab& p = *pt;
    p.B = B;
    const int ns = c->cfg.has_adapter ? c->ad_nst : 0, tq = attention_offline_tile_rows(c->dtype == FO_BF16);
    p.gap = c->KM ? c->KM - 1 : 0;
    long long frames = 0, rows = 0, ad_rows = 0, grid = 0, tiles = 0;
    for (int b = 0; b < B; ++b) {
        FO_CHECK(T[b] >= 7, "%s: utterance %d has %d feature frames; each needs >= 7", who, b0 + b, T[b]);
        const int t2 = ((T[b] - 1) / 2 - 1) / 2;
        FO_CHECK(t2 <= c->cfg.pos_max_len, "%s: utterance %d has %d encoder frames, past the positional table (%d)",
                 who, b0 + b, t2, c->cfg.pos_max_len);
        frames += T[b];
        rows += t2;
        ad_rows += ad_frames(c, t2);
        grid += b + 1 < B ? (T[b] + 3) / 4 * 4 : T[b];
        tiles += cdiv(t2, tq);
        p.tmax = std::max(p.tmax, t2);
        p.fmax = std::max(p.fmax, T[b]);
    }
    FO_CHECK(grid < (1LL << 28), "%s: %lld feature frames in one call; pass fewer utterances", who, frames);
    p.rows = (int)rows; p.ad_rows = (int)ad_rows; p.grid_frames = (int)grid; p.tiles = (int)tiles;
    p.trunk = (int)(rows + (long long)(B - 1) * p.gap);
    // table: tiles {b, q} | lens | eoff | xrow | grow | flen | foff | frow | gaps | adcnt | aoff [| soff (int64)]
    p.o_tiles = 0; p.o_lens = 2 * p.tiles; p.o_eoff = p.o_lens + B; p.o_xrow = p.o_eoff + B + 1; p.o_grow = p.o_xrow + B;
    p.o_flen = p.o_grow + B; p.o_foff = p.o_flen + B; p.o_frow = p.o_foff + B + 1; p.o_gaps = p.o_frow + B;
    p.o_adcnt = p.o_gaps + B; p.o_aoff = p.o_adcnt + (ns + 1) * B;
    std::vector<int32_t>& h = p.h;
    p.o_soff = soff ? (p.o_aoff + B + 1 + 1) / 2 * 2 : 0;
    h.assign(soff ? p.o_soff + 2 * B : p.o_aoff + B + 1, 0);
    if (soff) memcpy(h.data() + p.o_soff, soff, (size_t)B * sizeof(long long));
    int32_t* tl = h.data();
    for (int b = 0, g = 0; b < B; ++b) {
        const int t2 = ((T[b] - 1) / 2 - 1) / 2;
        h[p.o_lens + b] = t2;
        h[p.o_eoff + b + 1] = h[p.o_eoff + b] + t2;
        h[p.o_xrow + b] = h[p.o_eoff + b] + b * p.gap;
        h[p.o_gaps + b] = h[p.o_xrow + b] + t2;
        h[p.o_frow + b] = g;
        h[p.o_grow + b] = g / 4;                           // encoder row of frame g on the grid: rows 4 r .. 4 r + 6 feed row r
        h[p.o_flen + b] = T[b];
        h[p.o_foff + b + 1] = h[p.o_foff + b] + T[b];
        g += (T[b] + 3) / 4 * 4;
        for (int i = 0; i <= ns; ++i) h[p.o_adcnt + i * B + b] = ad_frames(c, t2, i);
        h[p.o_aoff + b + 1] = h[p.o_aoff + b] + ad_frames(c, t2);
        for (int q = 0; q < cdiv(t2, tq); ++q) { *tl++ = b; *tl++ = q; }
    }
    return 0;
}

int fo_encode_offline_packed(fo_ctx* c, const float* feats, const int32_t* lens, int B, int chunk, int left, float* enc_out,
                             float* adapter_out, void* stream) {
    FO_CHECK(c && c->finalized && c->cfg.has_encoder, "fo_encode_offline_packed: context has no finalized encoder");
    FO_CHECK(feats && lens && B > 0 && B <= 65535, "fo_encode_offline_packed: need feats, lens and 1 <= B <= 65535");
    if (adapter_out) FO_CHECK(c->cfg.has_adapter, "adapter_out requested but the context has no adapter");
    FO_CUDA(cudaSetDevice(c->device));
    FO_ON_GROUP(c, stream);
    cudaStream_t st = (cudaStream_t)stream;
    PackTab p;
    std::vector<int32_t> T(B);
    if (is_device_ptr(lens)) {
        FO_CUDA(cudaMemcpyAsync(T.data(), lens, (size_t)B * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
        FO_CUDA(cudaStreamSynchronize(st));
    } else {
        std::copy(lens, lens + B, T.begin());
    }
    FO_TRY(pack_tab(c, T.data(), B, "fo_encode_offline_packed", 0, nullptr, &p));
    const long long frames = p.h[p.o_foff + B], rows = p.rows, ad_rows = p.ad_rows;
    void *dtab, *dfeats, *denc, *dy = nullptr;
    FO_TRY(ws_ensure(c, WS_PKTAB, p.h.size() * sizeof(int32_t), &dtab));
    FO_CUDA(cudaMemcpyAsync(dtab, p.h.data(), p.h.size() * sizeof(int32_t), cudaMemcpyHostToDevice, st));
    FO_TRY(in_dev(c, feats, (size_t)frames * c->F * sizeof(float), WS_FEATS, st, (const void**)&dfeats));
    const size_t enc_bytes = (size_t)rows * c->D * sizeof(float), y_bytes = (size_t)ad_rows * c->E * sizeof(float);
    FO_TRY(out_dev(c, enc_out, enc_bytes, WS_ENC, &denc));
    if (adapter_out) FO_TRY(out_dev(c, adapter_out, y_bytes, WS_Y, &dy));
    const int32_t* tab = reinterpret_cast<const int32_t*>(dtab);
    FO_TRY(c->dtype == FO_BF16
               ? offline_packed_program<act16>(c, (const float*)dfeats, p, tab, chunk, left, (float*)denc, (float*)dy, st)
               : offline_packed_program<float>(c, (const float*)dfeats, p, tab, chunk, left, (float*)denc, (float*)dy, st));
    if (enc_out) FO_TRY(out_done(enc_out, denc, enc_bytes, st));
    if (adapter_out) FO_TRY(out_done(adapter_out, dy, y_bytes, st));
    c->stats.offline_calls += 1;
    c->stats.offline_frames += rows;
    return 0;
}

// ---- packed PCM: fbank of utterances of different lengths, and PCM -> embeddings in passes ------------------------------
// frames of an utterance of n samples (kaldi snip_edges: the trailing samples that fill no frame are dropped); 0 below one frame
static long long utt_frames(const fo_ctx* c, long long n) {
    return n >= c->cfg.frame_len ? 1 + (n - c->cfg.frame_len) / c->cfg.frame_shift : 0;
}

int fo_fbank_offline_packed(fo_ctx* c, const void* pcm, int pcm_dtype, const int64_t* n_samples, int B, float scale, float* out,
                            void* stream) {
    FO_CHECK(c && c->finalized && c->fb_window, "fo_fbank_offline_packed: context has no finalized frontend");
    FO_CHECK(pcm && n_samples && out && B > 0, "fo_fbank_offline_packed: need pcm, n_samples, out and B >= 1");
    FO_CHECK(pcm_dtype == FO_F32 || pcm_dtype == FO_I16, "fo_fbank_offline_packed: pcm must be FO_F32 or FO_I16");
    // table: sample offsets (int64) | frame offsets (B + 1, int32); the frame offsets are also the output rows
    std::vector<int32_t> h(2 * (size_t)B + B + 1, 0);
    long long* soff = reinterpret_cast<long long*>(h.data());
    int32_t* foff = h.data() + 2 * (size_t)B;
    long long samples = 0, frames = 0;
    for (int b = 0; b < B; ++b) {
        FO_CHECK(n_samples[b] >= c->cfg.frame_len, "fo_fbank_offline_packed: utterance %d has %lld samples, shorter than one frame (%d)",
                 b, (long long)n_samples[b], c->cfg.frame_len);
        soff[b] = samples;
        samples += n_samples[b];
        frames += utt_frames(c, n_samples[b]);
        FO_CHECK(frames < (1LL << 31), "fo_fbank_offline_packed: more than 2^31 - 1 frames in one call; pass fewer utterances");
        foff[b + 1] = (int32_t)frames;
    }
    FO_CUDA(cudaSetDevice(c->device));
    FO_ON_GROUP(c, stream);
    cudaStream_t st = (cudaStream_t)stream;
    void* dtab;
    FO_TRY(ws_ensure(c, WS_FBTAB, h.size() * sizeof(int32_t), &dtab));
    FO_CUDA(cudaMemcpyAsync(dtab, h.data(), h.size() * sizeof(int32_t), cudaMemcpyHostToDevice, st));
    const void* dp;
    FO_TRY(in_dev(c, pcm, (size_t)samples * (pcm_dtype == FO_I16 ? 2 : 4), WS_PCM, st, &dp));
    const size_t out_bytes = (size_t)frames * c->F * sizeof(float);
    void* dout;
    FO_TRY(out_dev(c, out, out_bytes, WS_FEATS, &dout));
    FbankVarlen vl;
    vl.sample_off = reinterpret_cast<const long long*>(dtab);
    vl.frame_off = reinterpret_cast<const int32_t*>(dtab) + 2 * (size_t)B;
    vl.out_row = vl.frame_off;
    vl.n = B;
    vl.frames = frames;
    FO_TRY(fbank_offline_packed(fbank_params(c), dp, pcm_dtype == FO_I16, scale, vl, (float*)dout, nullptr, st));
    FO_TRY(out_done(out, dout, out_bytes, st));
    return 0;
}

// fo_encode_offline_packed_pcm runs in passes over consecutive utterances: utterance i takes ceil(m_i / 4) * 4 frames of the
// feature grid, and a pass takes utterances in call order while their grid frames fit P (option "packed_pass_frames", else
// PACKED_PASS_BYTES over the workspace bytes of one encoder row); an utterance larger than P runs in a pass of its own.  Every
// workspace is sized by the pass, so the device memory a call adds follows P, not the corpus.  Passes run eagerly (no graphs).
constexpr long long PACKED_PASS_BYTES = 10LL << 30;

// workspace bytes of one encoder row of a pass (4 grid frames): PCM staging and the feature grid (+ feats_out staging), conv1
// planes and conv2 rows, sub-Linear / residual / LayerNorm / attention rows, QKV (+ fp32 Q), FFN hidden rows, encoder and
// adapter rows -- the terms of steps_block_bytes per encoder frame
static long long packed_row_bytes(const fo_ctx* c) {
    const long long esz = (long long)c->esz, D = c->D;
    long long b = 4LL * c->cfg.frame_shift * 4 + 2 * 4LL * c->F * 4;
    b += 6LL * (c->F2 + 1) * D * esz + (long long)c->F2 * D * esz;
    b += D * (4 + 4 + 4 + 5 * esz) + 3 * D * (esz + 4) + (long long)c->FF * esz;
    if (c->cfg.has_adapter) b += 4 * D * (esz + 4) + (long long)c->E * 4;
    return b;
}
// ... and never more grid frames than the conv2 implicit GEMM of one pass (T' (F2 + 1) rows, d_model columns) can take
static int packed_pass_frames(const fo_ctx* c) {
    const long long cap = std::max(4LL, gemm_tc_max_rows(c->D) / (c->F2 + 1) * 4);
    const long long P = c->packed_pass_frames > 0 ? c->packed_pass_frames : PACKED_PASS_BYTES / packed_row_bytes(c) * 4;
    return (int)std::max(4LL, std::min({1LL << 26, cap, P}));
}

int fo_encode_offline_packed_pcm(fo_ctx* c, const void* pcm, int pcm_dtype, const int64_t* n_samples, int B, float scale, int chunk,
                                 int left, float* enc_out, float* adapter_out, float* feats_out, void* stream) {
    const char* who = "fo_encode_offline_packed_pcm";
    FO_CHECK(c && c->finalized && c->cfg.has_encoder && c->fb_window, "%s: context has no finalized encoder + frontend", who);
    FO_CHECK(pcm && n_samples && B > 0 && B <= 65535, "%s: need pcm, n_samples and 1 <= B <= 65535", who);
    FO_CHECK(pcm_dtype == FO_F32 || pcm_dtype == FO_I16, "%s: pcm must be FO_F32 or FO_I16", who);
    if (adapter_out) FO_CHECK(c->cfg.has_adapter, "adapter_out requested but the context has no adapter");
    // every utterance is checked before the first pass: m_i frames, T'_i encoder rows; offsets of the whole call
    std::vector<int32_t> T(B);
    std::vector<long long> soff(B + 1, 0), foff(B + 1, 0), eoff(B + 1, 0), aoff(B + 1, 0);
    for (int b = 0; b < B; ++b) {
        const long long m = utt_frames(c, n_samples[b]);
        FO_CHECK(m >= 7, "%s: utterance %d has %lld samples, %lld feature frames; each needs >= 7", who, b, (long long)n_samples[b], m);
        const long long t2 = ((m - 1) / 2 - 1) / 2;
        FO_CHECK(t2 <= c->cfg.pos_max_len, "%s: utterance %d has %lld encoder frames, past the positional table (%d)", who, b, t2,
                 c->cfg.pos_max_len);
        T[b] = (int32_t)m;
        soff[b + 1] = soff[b] + n_samples[b];
        foff[b + 1] = foff[b] + m;
        eoff[b + 1] = eoff[b] + t2;
        aoff[b + 1] = aoff[b] + ad_frames(c, (int)t2);
    }
    FO_CUDA(cudaSetDevice(c->device));
    FO_ON_GROUP(c, stream);
    cudaStream_t st = (cudaStream_t)stream;
    const int P = packed_pass_frames(c), F = c->F, D = c->D, E = c->E;
    const size_t esz_pcm = pcm_dtype == FO_I16 ? 2 : 4;
    const bool pcm_dev = is_device_ptr(pcm), enc_dev = enc_out && is_device_ptr(enc_out);
    const bool y_dev = adapter_out && is_device_ptr(adapter_out), f_dev = feats_out && is_device_ptr(feats_out);
    std::vector<long long> ps(B);
    for (int b0 = 0, b1; b0 < B; b0 = b1) {
        long long g = (T[b0] + 3) / 4 * 4;
        for (b1 = b0 + 1; b1 < B && g + (T[b1] + 3) / 4 * 4 <= P; ++b1) g += (T[b1] + 3) / 4 * 4;
        const int n = b1 - b0;
        for (int b = b0; b < b1; ++b) ps[b - b0] = soff[b] - soff[b0];
        PackTab p;
        FO_TRY(pack_tab(c, T.data() + b0, n, who, b0, ps.data(), &p));
        void *dtab, *dpcm, *denc, *dy = nullptr, *dfeats = nullptr;
        FO_TRY(ws_ensure(c, WS_PKTAB, p.h.size() * sizeof(int32_t), &dtab));
        FO_CUDA(cudaMemcpyAsync(dtab, p.h.data(), p.h.size() * sizeof(int32_t), cudaMemcpyHostToDevice, st));
        const size_t pcm_bytes = (size_t)(soff[b1] - soff[b0]) * esz_pcm;
        const char* src = (const char*)pcm + (size_t)soff[b0] * esz_pcm;
        if (pcm_dev) {
            dpcm = const_cast<char*>(src);
        } else {
            FO_TRY(ws_ensure(c, WS_PCM, pcm_bytes, &dpcm));
            FO_CUDA(cudaMemcpyAsync(dpcm, src, pcm_bytes, cudaMemcpyHostToDevice, st));
        }
        const size_t enc_bytes = (size_t)p.rows * D * sizeof(float), y_bytes = (size_t)p.ad_rows * E * sizeof(float);
        const size_t f_bytes = (size_t)(foff[b1] - foff[b0]) * F * sizeof(float);
        if (enc_dev) denc = enc_out + eoff[b0] * D;
        else FO_TRY(ws_ensure(c, WS_ENC, enc_bytes, &denc));
        if (y_dev) dy = adapter_out + aoff[b0] * E;
        else if (adapter_out) FO_TRY(ws_ensure(c, WS_Y, y_bytes, &dy));
        if (f_dev) dfeats = feats_out + foff[b0] * F;
        else if (feats_out) FO_TRY(ws_ensure(c, WS_FEATS, f_bytes, &dfeats));
        const int32_t* tab = reinterpret_cast<const int32_t*>(dtab);
        float* fg;
        FO_TRY(packed_grid(c, p, &fg, st));
        FbankVarlen vl;
        vl.frame_off = tab + p.o_foff;
        vl.sample_off = reinterpret_cast<const long long*>(tab + p.o_soff);
        vl.out_row = tab + p.o_frow;
        vl.n = n;
        vl.frames = foff[b1] - foff[b0];
        FO_TRY(fbank_offline_packed(fbank_params(c), dpcm, pcm_dtype == FO_I16, scale, vl, fg, (float*)dfeats, st));
        FO_TRY(c->dtype == FO_BF16 ? offline_packed_trunk<act16>(c, fg, p, tab, chunk, left, (float*)denc, (float*)dy, st)
                                   : offline_packed_trunk<float>(c, fg, p, tab, chunk, left, (float*)denc, (float*)dy, st));
        if (enc_out && !enc_dev) FO_CUDA(cudaMemcpyAsync(enc_out + eoff[b0] * D, denc, enc_bytes, cudaMemcpyDeviceToHost, st));
        if (adapter_out && !y_dev) FO_CUDA(cudaMemcpyAsync(adapter_out + aoff[b0] * E, dy, y_bytes, cudaMemcpyDeviceToHost, st));
        if (feats_out && !f_dev) FO_CUDA(cudaMemcpyAsync(feats_out + foff[b0] * F, dfeats, f_bytes, cudaMemcpyDeviceToHost, st));
    }
    c->stats.offline_calls += 1;
    c->stats.offline_frames += eoff[B];
    return 0;
}

int fo_adapter_forward2(fo_ctx* c, const float* x, const uint8_t* mask, int B, int T, const float* cache0_in, const float* cache1_in,
                        float* cache0_out, float* cache1_out, float* y, void* stream) {
    FO_CHECK(c && c->finalized && c->cfg.has_adapter, "fo_adapter_forward: context has no finalized adapter");
    FO_CHECK(x && y && B > 0 && T > 0, "fo_adapter_forward: bad argument");
    FO_CUDA(cudaSetDevice(c->device));
    FO_ON_GROUP(c, stream);
    cudaStream_t st = (cudaStream_t)stream;
    const int km1 = c->KA - 1, t_out = ad_frames(c, T);
    FO_CHECK(t_out >= 1, "fo_adapter_forward: input too short");
    if (!c->ad_carry) FO_CHECK(!cache0_in && !cache0_out && !cache1_in && !cache1_out, "fo_adapter_forward: this adapter carries no cache");
    if (c->ad_nst < 2) FO_CHECK(!cache1_in && !cache1_out, "fo_adapter_forward: single-conv CNNSubsampling has one cache entry");
    const void *dx, *dm = nullptr;
    FO_TRY(in_dev(c, x, (size_t)B * T * c->D * sizeof(float), WS_ENC, st, &dx));
    if (mask) FO_TRY(in_dev(c, mask, (size_t)B * T, WS_MASK2, st, &dm));
    // user_*[which]: the reference's cache list order; stage_*[i]: conv i's left context
    const float* user_in[2] = {cache0_in, cache1_in};
    float* user_out[2] = {cache0_out, cache1_out};
    const float* stage_in[2] = {nullptr, nullptr};
    float* stage_out[2] = {nullptr, nullptr};
    void* dev_out[2] = {nullptr, nullptr};
    size_t bytes[2] = {0, 0};
    for (int w = 0; w < c->ad_nst; ++w) {
        const int i = ad_stage_of_entry(c, w);
        bytes[w] = (size_t)B * c->ad_st[i].cin * km1 * sizeof(float);
        const void* din = nullptr;
        if (user_in[w]) FO_TRY(in_dev(c, user_in[w], bytes[w], w ? WS_TMP4 : WS_TMP0, st, &din));
        if (user_out[w]) FO_TRY(out_dev(c, user_out[w], bytes[w], w ? WS_TMP5 : WS_TMP1, &dev_out[w]));
        stage_in[i] = (const float*)din;
        stage_out[i] = (float*)dev_out[w];
    }
    void* dy;
    const size_t y_bytes = (size_t)B * t_out * c->E * sizeof(float);
    FO_TRY(out_dev(c, y, y_bytes, WS_Y, &dy));
    AdOut out;
    out.y = (float*)dy;
    int r = c->dtype == FO_BF16 ? adapter_program<act16>(c, (const float*)dx, (const uint8_t*)dm, B, T, nullptr, stage_in, stage_out, out, st)
                                : adapter_program<float>(c, (const float*)dx, (const uint8_t*)dm, B, T, nullptr, stage_in, stage_out, out, st);
    FO_TRY(r);
    for (int w = 0; w < 2; ++w)
        if (user_out[w]) FO_TRY(out_done(user_out[w], dev_out[w], bytes[w], st));
    FO_TRY(out_done(y, dy, y_bytes, st));
    return 0;
}

int fo_adapter_forward(fo_ctx* c, const float* x, const uint8_t* mask, int B, int T, const float* cache_in,
                       float* cache_out, float* y, void* stream) {
    FO_CHECK(c && !(c->ad_carry && c->ad_nst == 2 && (cache_in || cache_out)),
             "fo_adapter_forward: the two-conv CNNSubsampling carries two caches; use fo_adapter_forward2");
    return fo_adapter_forward2(c, x, mask, B, T, cache_in, nullptr, cache_out, nullptr, y, stream);
}

// ---- introspection --------------------------------------------------------------------------------------
int fo_stats(fo_ctx* c, fo_stats_t* out) {
    FO_CHECK(c && out, "fo_stats: null argument");
    *out = c->stats;
    out->kernel_launches = g_launches.load();
    out->sessions_in_use = c->sessions_in_use;
    out->device_bytes = c->device_bytes;
    out->act_saturations = 0;
    if (c->sat_counter) {
        // counted by kernels that may still be in flight on the caller's streams: a blocking copy orders after them
        unsigned long long v = 0;
        FO_CUDA(cudaSetDevice(c->device));
        FO_CUDA(cudaMemcpy(&v, c->sat_counter, sizeof(v), cudaMemcpyDeviceToHost));
        out->act_saturations = (int64_t)v;
    }
    return 0;
}

int fo_set_option(fo_ctx* c, const char* name, int64_t value) {
    FO_CHECK(c && name, "fo_set_option: null argument");
    if (!strcmp(name, "gemm_backend")) {
        FO_CHECK(value == 0 || (value == 1 && c->dtype == FO_BF16), "gemm_backend 1 (tcgen05) needs a bf16 context");
        c->gemm_backend = (int)value;
    } else if (!strcmp(name, "use_graph")) c->use_graph = value != 0;
    else if (!strcmp(name, "split_k")) c->split_k = (int)value;
    else if (!strcmp(name, "debug_skip")) c->debug_skip = (int)value;
    else if (!strcmp(name, "step_part")) { c->step_part = (int)value; c->ws_epoch += 1; }
    else if (!strcmp(name, "trace")) {
        // development builds (FO_TRACE_BUILD): value > 0 allocates room for `value` CTA records and binds the kernels to it,
        // 0 unbinds.  fo_debug_trace_read copies the records out.
        FO_CUDA(cudaSetDevice(c->device));
        FO_TRY(ctx_sync(c));
        if (value > 0 && (unsigned int)value > c->trace_cap) {
            void* p = nullptr;
            FO_TRY(dev_alloc(c, &p, (size_t)value * 8 * sizeof(unsigned long long)));
            c->trace_buf = (unsigned long long*)p;
            c->trace_cap = (unsigned int)value;
            if (!c->trace_cnt) { FO_TRY(dev_alloc(c, &p, sizeof(unsigned int))); c->trace_cnt = (unsigned int*)p; }
        }
        if (c->trace_cnt) FO_CUDA(cudaMemset(c->trace_cnt, 0, sizeof(unsigned int)));
        unsigned long long* b = value > 0 ? c->trace_buf : nullptr;
        trace_bind_gemm(b, c->trace_cnt, c->trace_cap);
        trace_bind_attention(b, c->trace_cnt, c->trace_cap);
        trace_bind_elementwise(b, c->trace_cnt, c->trace_cap);
        trace_bind_fbank(b, c->trace_cnt, c->trace_cap);
    }
    else if (!strcmp(name, "tc_plan")) {
        // development: plan of the skinny GEMM with (N, K): N | K << 16 | swap << 32 | bn << 33 | split << 42 | cap_kb << 48; 0 clears
        const uint64_t v = (uint64_t)value;
        gemm_tc_plan_override((int)(v & 0xFFFF), (int)((v >> 16) & 0xFFFF), (int)((v >> 32) & 1), (int)((v >> 33) & 0x1FF),
                              (int)((v >> 42) & 0x3F), (int)((v >> 48) & 0xFF));
        c->ws_epoch += 1;                       // captured graphs hold the old plans
    }
    else if (!strcmp(name, "fuse_ln")) c->fuse_ln = value != 0;
    else if (!strcmp(name, "stack_rows")) c->stack_rows = (int)value;
    else if (!strcmp(name, "steps_pass_blocks")) {
        FO_CHECK(value >= 0 && value <= (1 << 20), "steps_pass_blocks must be 0 (byte budget) or 1..%d blocks", 1 << 20);
        c->steps_pass_blocks = (int)value;
    }
    else if (!strcmp(name, "packed_pass_frames")) {
        FO_CHECK(value == 0 || (value >= 4 && value <= (1 << 26)), "packed_pass_frames must be 0 (byte budget) or 4..%d grid frames",
                 1 << 26);
        c->packed_pass_frames = (int)value;
    }
    else if (!strcmp(name, "defer_reduce")) c->defer_reduce = value != 0;
    else if (!strcmp(name, "tc_persist")) gemm_tc_set_persist(value != 0);
    else if (!strcmp(name, "l2_prefetch")) c->use_prefetch = (int)(value & 3);
    else if (!strcmp(name, "pdl")) g_want_pdl = value != 0;
    else if (!strcmp(name, "session_groups")) {
        FO_CHECK(value >= 1 && value <= fo_ctx::MAX_GROUPS, "session_groups must be 1..%d", fo_ctx::MAX_GROUPS);
        c->groups = (int)value;
    }
    else if (!strcmp(name, "tc_npa")) { c->tc_npa = (int)value; gemm_tc_force_producers(c->tc_npa, c->tc_npb); }
    else if (!strcmp(name, "tc_npb")) { c->tc_npb = (int)value; gemm_tc_force_producers(c->tc_npa, c->tc_npb); }
    else if (!strcmp(name, "tc_swap")) { c->tc_tune.swap = (int)value; gemm_tc_force(c->tc_tune); }
    else if (!strcmp(name, "tc_bn")) { c->tc_tune.bn = (int)value; gemm_tc_force(c->tc_tune); }
    else if (!strcmp(name, "tc_split")) { c->tc_tune.split = (int)value; gemm_tc_force(c->tc_tune); }
    else if (!strcmp(name, "profile_gemm")) {
        c->profile_gemm = value != 0;
        if (value) {
            for (auto& pr : c->prof_events) { cudaEventDestroy(pr.e0); cudaEventDestroy(pr.e1); }
            c->prof_events.clear();
        }
    }
    else { set_error("fo_set_option: unknown option '%s'", name); return FO_ERR_ARG; }
    return 0;
}

int fo_get_option(fo_ctx* c, const char* name, int64_t* value) {
    FO_CHECK(c && name && value, "fo_get_option: null argument");
    if (!strcmp(name, "gemm_backend")) *value = c->gemm_backend;
    else if (!strcmp(name, "use_graph")) *value = c->use_graph;
    else if (!strcmp(name, "split_k")) *value = c->split_k;
    else if (!strcmp(name, "session_groups")) *value = c->groups;
    else if (!strcmp(name, "fuse_ln")) *value = c->fuse_ln;
    else if (!strcmp(name, "stack_rows")) *value = c->stack_rows;
    else if (!strcmp(name, "steps_pass_blocks")) *value = c->steps_pass_blocks;
    else if (!strcmp(name, "steps_pass_blocks_in_use")) {             // P of a recording call at the context's chunking
        FO_CHECK(c->finalized, "fo_get_option: steps_pass_blocks_in_use needs a finalized context");
        *value = steps_pass_blocks(c, c->cfg.context_frames + c->cfg.frames_per_chunk);
    }
    else if (!strcmp(name, "packed_pass_frames")) *value = packed_pass_frames(c);    // the budget's frames when not set
    else if (!strcmp(name, "stack_launches")) *value = c->stack_launches;
    else if (!strcmp(name, "defer_reduce")) *value = c->defer_reduce;
    else if (!strcmp(name, "tc_persist_launches")) *value = gemm_tc_persist_launches();
    else if (!strcmp(name, "l2_prefetch")) *value = c->use_prefetch;
    else if (!strcmp(name, "pdl")) *value = g_want_pdl;
    else if (!strcmp(name, "profile_gemm_count")) *value = (int64_t)c->prof_events.size();
    else if (!strcmp(name, "profile_gemm_us")) {
        double us = 0.0;
        for (auto& pr : c->prof_events) {
            FO_CUDA(cudaEventSynchronize(pr.e1));
            float ms = 0.f;
            FO_CUDA(cudaEventElapsedTime(&ms, pr.e0, pr.e1));
            us += 1e3 * ms;
        }
        *value = (int64_t)us;
    }
    else if (!strcmp(name, "tc_launches")) *value = gemm_tc_launches();
    else if (!strcmp(name, "ring_cap")) *value = c->ring_cap;
    else if (!strcmp(name, "max_t")) *value = c->max_t;
    else if (!strcmp(name, "sm_count")) *value = c->sms;
    else { set_error("fo_get_option: unknown option '%s'", name); return FO_ERR_ARG; }
    return 0;
}

int fo_profile_dump(fo_ctx* c, char* buf, int cap) {
    FO_CHECK(c && buf && cap > 0, "fo_profile_dump: bad argument");
    std::map<std::string, std::pair<long long, double>> agg;       // "M N K" -> (launches, microseconds)
    for (auto& pr : c->prof_events) {
        FO_CUDA(cudaEventSynchronize(pr.e1));
        float ms = 0.f;
        FO_CUDA(cudaEventElapsedTime(&ms, pr.e0, pr.e1));
        char key[64];
        snprintf(key, sizeof(key), "%d %d %d", pr.M, pr.N, pr.K);
        auto& a = agg[key];
        a.first += 1;
        a.second += 1e3 * ms;
    }
    int off = 0;
    for (auto& kv : agg) {
        int w = snprintf(buf + off, cap - off, "%s %lld %.3f\n", kv.first.c_str(), kv.second.first, kv.second.second);
        if (w < 0 || w >= cap - off) break;
        off += w;
    }
    buf[off < cap ? off : cap - 1] = 0;
    return 0;
}

int fo_debug_trace_read(fo_ctx* c, uint64_t* out, int64_t cap_records, int64_t* n_records) {
    FO_CHECK(c && out && n_records, "fo_debug_trace_read: null argument");
    *n_records = 0;
    if (!c->trace_cnt) return 0;
    FO_CUDA(cudaSetDevice(c->device));
    FO_TRY(ctx_sync(c));
    unsigned int n = 0;
    FO_CUDA(cudaMemcpy(&n, c->trace_cnt, sizeof(n), cudaMemcpyDeviceToHost));
    if (n > c->trace_cap) n = c->trace_cap;
    if ((int64_t)n > cap_records) n = (unsigned int)cap_records;
    FO_CUDA(cudaMemcpy(out, c->trace_buf, (size_t)n * 8 * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
    FO_CUDA(cudaMemset(c->trace_cnt, 0, sizeof(unsigned int)));
    *n_records = n;
    return 0;
}

int fo_debug_stack_plan(int d_model, int ffn_dim, int heads, int n_sessions, int frames, int window, int layers, int sms,
                        int smem_max, int* smem_bytes, int* ffn2_chunk, int* rows_qkv, int* rows_ffn1, int* rows_out) {
    FO_CHECK(smem_bytes && ffn2_chunk && rows_qkv && rows_ffn1 && rows_out, "fo_debug_stack_plan: null argument");
    return stack_plan(d_model, ffn_dim, heads, n_sessions, frames, window, layers, sms, smem_max, smem_bytes, ffn2_chunk, rows_qkv,
                      rows_ffn1, rows_out);
}

int fo_debug_sm_ids(fo_ctx* c, int n_ctas, int graph, int32_t* out, void* stream) {
    FO_CHECK(c && out && n_ctas > 0 && n_ctas <= 65535, "fo_debug_sm_ids: bad argument");
    FO_CUDA(cudaSetDevice(c->device));
    FO_ON_GROUP(c, stream);
    const cudaStream_t st = (cudaStream_t)stream;
    void* d;
    FO_TRY(out_dev(c, out, (size_t)n_ctas * sizeof(int32_t), WS_TMP0, &d));
    if (!graph) {
        FO_TRY(sm_ids((int32_t*)d, n_ctas, st));
    } else {
        // as run_step does with a step: captured on the capture stream, instantiated, replayed on the stream of the call
        FO_CUDA(cudaStreamBeginCapture(c->cap_stream, cudaStreamCaptureModeRelaxed));
        const int r = sm_ids((int32_t*)d, n_ctas, c->cap_stream);
        cudaGraph_t g = nullptr;
        const cudaError_t ce = cudaStreamEndCapture(c->cap_stream, &g);
        if (r != 0) { if (g) cudaGraphDestroy(g); return r; }
        FO_CUDA(ce);
        cudaGraphExec_t ge = nullptr;
        const cudaError_t ie = cudaGraphInstantiate(&ge, g, 0);
        cudaGraphDestroy(g);
        FO_CUDA(ie);
        const cudaError_t le = cudaGraphLaunch(ge, st);
        const cudaError_t se = le == cudaSuccess ? cudaStreamSynchronize(st) : le;
        cudaGraphExecDestroy(ge);
        FO_CUDA(se);
    }
    return out_done(out, d, (size_t)n_ctas * sizeof(int32_t), st);
}

int fo_debug_plan(int64_t act_rows, int n_out, int K, int can_defer, int* swap, int* bn, int* split) {
    FO_CHECK(act_rows > 0 && n_out > 0 && K > 0 && K % 64 == 0 && swap && bn && split, "fo_debug_plan: bad argument");
    gemm_tc_plan(act_rows, n_out, K, can_defer, swap, bn, split);
    return 0;
}

int fo_debug_gemm(fo_ctx* c, const float* A, const float* W, const float* bias, float* C, int M, int N, int K,
                  int backend, int relu, int iters, float* ms_out, void* stream) {
    FO_CHECK(c && A && W && C && M > 0 && N > 0 && K > 0, "fo_debug_gemm: bad argument");
    FO_CUDA(cudaSetDevice(c->device));
    FO_ON_GROUP(c, stream);
    cudaStream_t st = (cudaStream_t)stream;
    Epilogue ep;
    ep.bias = bias;
    ep.c_f32 = C;
    ep.ldc = N;
    ep.relu = relu;
    const int saved = c->gemm_backend;
    cudaEvent_t e0, e1;
    FO_CUDA(cudaEventCreate(&e0));
    FO_CUDA(cudaEventCreate(&e1));
    int r = 0;
    // one eager launch (result + lazy initialisation), then `iters` launches captured into a graph and timed as
    // one graph launch, so the number is device time without host launch overhead
    const void *pa = A, *pw = W;
    if (c->dtype == FO_BF16) {
        void *a16, *w16;
        FO_TRY(ws_ensure(c, WS_TMP2, (size_t)M * K * 2, &a16));
        FO_TRY(ws_ensure(c, WS_TMP3, (size_t)N * K * 2, &w16));
        FO_TRY(f32_to_act16(A, (act16*)a16, (long long)M * K, st));
        FO_TRY(f32_to_weight16(W, (act16*)w16, (long long)N * K, st));
        pa = a16;
        pw = w16;
    }
    c->gemm_backend = backend;
    auto one = [&](cudaStream_t s) {
        return c->dtype == FO_BF16 ? gemm<act16>(c, (const act16*)pa, pw, M, N, K, ep, s) : gemm<float>(c, (const float*)pa, pw, M, N, K, ep, s);
    };
    r = one(st);
    if (r == 0 && iters > 0) {
        cudaGraph_t graph = nullptr;
        cudaGraphExec_t exec = nullptr;
        FO_CUDA(cudaStreamSynchronize(st));
        FO_CUDA(cudaStreamBeginCapture(c->cap_stream, cudaStreamCaptureModeRelaxed));
        for (int i = 0; i < iters && r == 0; ++i) r = one(c->cap_stream);
        cudaError_t ce = cudaStreamEndCapture(c->cap_stream, &graph);
        if (r == 0 && ce == cudaSuccess) ce = cudaGraphInstantiate(&exec, graph, 0);
        if (graph) cudaGraphDestroy(graph);
        if (r == 0 && ce == cudaSuccess) {
            cudaGraphLaunch(exec, st);
            cudaEventRecord(e0, st);
            cudaGraphLaunch(exec, st);
            cudaEventRecord(e1, st);
        } else {
            cudaEventRecord(e0, st);
            cudaEventRecord(e1, st);
            if (r == 0) { set_error("fo_debug_gemm: graph capture failed: %s", cudaGetErrorString(ce)); r = FO_ERR_CUDA; }
        }
        cudaEventSynchronize(e1);
        if (exec) cudaGraphExecDestroy(exec);
    } else {
        cudaEventRecord(e0, st);
        cudaEventRecord(e1, st);
    }
    c->gemm_backend = saved;
    cudaError_t e = cudaEventSynchronize(e1);
    float ms = 0.f;
    cudaEventElapsedTime(&ms, e0, e1);
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    FO_TRY(r);
    FO_CUDA(e);
    if (ms_out) *ms_out = iters > 0 ? ms / iters : 0.f;
    return 0;
}

int fo_debug_attention(fo_ctx* c, int mode, int n, const int32_t* seq, const int32_t* cnt, const int32_t* off, int T, int gap,
                       int chunk, int left, int t, int layer, int group, const float* qkv, const float* part, int nsplit,
                       const float* part_bias, const float* ptab, int ptab_rows, const float* pos_u, const float* pos_v,
                       float* out, void* stream) {
    FO_CHECK(c && c->finalized && c->cfg.has_encoder, "fo_debug_attention: context has no finalized encoder");
    FO_CHECK(mode >= FO_ATT_OFFLINE && mode <= FO_ATT_CHUNKS && n > 0 && seq && ptab && pos_u && pos_v && out,
             "fo_debug_attention: bad argument");
    FO_CHECK(ptab_rows >= c->pos_rows, "fo_debug_attention: the rel-pos table has %d rows; this context reads %d", ptab_rows,
             c->pos_rows);
    FO_CHECK(nsplit >= 0 && (nsplit == 0 || (mode == FO_ATT_STREAM && c->dtype == FO_BF16 && part && part_bias)),
             "fo_debug_attention: split-K partials (with their bias) go with the stream mode of a bf16 context");
    FO_CHECK(qkv || nsplit > 0, "fo_debug_attention: qkv is null");
    DebugAttn d;
    d.mode = mode; d.n = n; d.chunk = chunk; d.left = left; d.nsplit = nsplit;
    d.qkv = qkv; d.part = part; d.part_bias = part_bias; d.ptab = ptab; d.pos_u = pos_u; d.pos_v = pos_v; d.out = out;
    if (mode == FO_ATT_OFFLINE) {
        FO_CHECK(T > 0 && T <= c->pos_rows, "fo_debug_attention: T = %d outside 1..%d (rel-pos rows)", T, c->pos_rows);
        for (int b = 0; b < n; ++b) FO_CHECK(seq[b] >= 0, "fo_debug_attention: ilens[%d] < 0", b);
        d.T = T;
        d.rows = (long long)n * T;
        d.tab.assign(seq, seq + n);
    } else if (mode == FO_ATT_PACKED) {
        FO_CHECK(gap >= 0, "fo_debug_attention: gap < 0");
        const int tq = attention_offline_tile_rows(c->dtype == FO_BF16);
        std::vector<int32_t> lens(n), rows(n);
        for (int b = 0; b < n; ++b) {
            FO_CHECK(seq[b] >= 1 && seq[b] <= c->pos_rows, "fo_debug_attention: lens[%d] = %d outside 1..%d", b, seq[b], c->pos_rows);
            lens[b] = seq[b];
            rows[b] = (int32_t)d.rows;
            d.rows += seq[b] + (b + 1 < n ? gap : 0);
            d.tmax = std::max(d.tmax, seq[b]);
            for (int q = 0; q < cdiv(seq[b], tq); ++q) { d.tab.push_back(b); d.tab.push_back(q); }   // as fo_encode_offline_packed
        }
        d.ntiles = (int)d.tab.size() / 2;
        d.tab.insert(d.tab.end(), lens.begin(), lens.end());
        d.tab.insert(d.tab.end(), rows.begin(), rows.end());
    } else {
        FO_CHECK(c->ring, "fo_debug_attention: context has no streaming sessions");
        FO_CHECK(layer >= 0 && layer < c->L, "fo_debug_attention: layer %d out of range", layer);
        FO_CHECK(t >= 1 && t <= c->max_t && t <= STREAM_MAX_T, "fo_debug_attention: t = %d outside 1..%d (max_t)", t, c->max_t);
        FO_CHECK(c->window + t <= c->ring_cap && c->window + t <= STREAM_CHUNKS_MAX_KEYS,
                 "fo_debug_attention: window %d + t %d exceeds ring capacity %d or %d keys", c->window, t, c->ring_cap,
                 STREAM_CHUNKS_MAX_KEYS);
        FO_TRY(check_ids(c, seq, n));
        d.t = t; d.layer = layer;
        d.tab.assign(seq, seq + n);
        if (mode == FO_ATT_STREAM) {
            d.rows = (long long)n * t;
        } else {
            FO_CHECK(cnt && off && group >= 1, "fo_debug_attention: the chunks mode needs cnt, off and group >= 1");
            FO_CHECK(c->window + group * t <= STREAM_CHUNKS_MAX_KEYS, "fo_debug_attention: window %d + %d chunks x %d frames exceeds %d keys",
                     c->window, group, t, STREAM_CHUNKS_MAX_KEYS);
            FO_CHECK(off[0] >= 0, "fo_debug_attention: off[0] < 0");
            int kmax = 0;
            for (int b = 0; b < n; ++b) {
                FO_CHECK(cnt[b] >= 1 && (b == 0 || off[b] == off[b - 1] + cnt[b - 1]),
                         "fo_debug_attention: cnt[%d] < 1 or off is not the running sum of cnt", b);
                kmax = std::max(kmax, cnt[b]);
                d.rows += (long long)cnt[b] * t;
            }
            d.group = group;
            d.groups = cdiv(kmax, group);      // as stream_program
            d.tab.insert(d.tab.end(), cnt, cnt + n);
            d.tab.insert(d.tab.end(), off, off + n);
        }
    }
    FO_CUDA(cudaSetDevice(c->device));
    FO_ON_GROUP(c, stream);
    cudaStream_t st = (cudaStream_t)stream;
    return c->dtype == FO_BF16 ? debug_attention_run<act16>(c, d, st) : debug_attention_run<float>(c, d, st);
}

}  // extern "C"
