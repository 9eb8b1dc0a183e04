// Shared declarations of the sm_100a kernels behind include/fo_b200.h.
#pragma once
#include <atomic>
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <stdint.h>
#include <stdio.h>
#include <string>

typedef __nv_bfloat16 bf16;
// 16-bit storage type of a "bf16" context.  The WEIGHTS are rounded to bf16 (what the reference's autocast computes
// with) and then held in IEEE fp16 containers -- exact for |w| >= 6.1e-5 (8 significand bits fit in 11), below that the
// absolute error is < 3e-8 -- because tcgen05.mma kind::f16 needs both operands in ONE format (a bf16 x fp16 mix
// raises an illegal-instruction fault on B200), and the ACTIVATIONS that feed the tensor cores are staged as fp16:
// same 2 bytes and MMA rate, fp32 accumulation, but 11 instead of 8 significand bits, which is what brings 24 layers of
// re-rounded GEMM inputs under the 2e-2 parity bar (bf16 activations measured 2.2e-2).  Every staged activation is a
// LayerNorm / ReLU / softmax-weighted output, far inside fp16 range; conversions saturate instead of overflowing.
typedef __half act16;

namespace fo {

// ---- error plumbing --------------------------------------------------------------------------
void set_error(const char* fmt, ...);
#define FO_CUDA(expr)                                                                             \
    do {                                                                                          \
        cudaError_t _e = (expr);                                                                  \
        if (_e != cudaSuccess) {                                                                  \
            fo::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
            (void)cudaGetLastError();   /* a refused launch must not fail the next call's checks */ \
            return -2;                                                                            \
        }                                                                                         \
    } while (0)
#define FO_CHECK(cond, ...)                                                                       \
    do {                                                                                          \
        if (!(cond)) { fo::set_error(__VA_ARGS__); return -1; }                                   \
    } while (0)
#define FO_TRY(expr) do { int _r = (expr); if (_r != 0) return _r; } while (0)

extern std::atomic<long long> g_launches;      // kernels enqueued by this library, every thread (fo_stats.kernel_launches)
extern thread_local long long t_launches;       // the same, by this thread (kernels counted while a graph is captured)
#define FO_LAUNCHED() (fo::g_launches.fetch_add(1), ++fo::t_launches)

__host__ __device__ inline int cdiv(int a, int b) { return (a + b - 1) / b; }
// pe_index after j streaming steps of pe = pe % wrap + chunk_size (attention.py:107,120), in closed form since j may run into
// the thousands: pe itself for j = 0, else (pe % wrap + (j - 1) * chunk_size) % wrap + chunk_size.  Equal to the loop for every
// int pe, negative ones included; its value mod wrap is (pe % wrap + j * chunk_size) % wrap.
__host__ __device__ inline int pe_after(int pe, int j, int chunk_size, int wrap) {
    return j == 0 ? pe : (int)(((long long)(pe % wrap) + (long long)(j - 1) * chunk_size) % wrap) + chunk_size;
}

// ---- programmatic dependent launch ------------------------------------------------------------------
// The kernels of the streaming chain are launched with programmaticStreamSerialization: a kernel may start (launch
// latency, barrier/TMEM set-up, and in the GEMM the first WEIGHT stages, which do not depend on the previous kernel)
// while its predecessor is still draining.  FO_PDL_TRIGGER lets the successor launch as soon as every CTA of this
// grid has started; FO_PDL_WAIT returns once the predecessor grid has completed and its memory is visible.  Every
// thread executes FO_PDL_WAIT before it touches global memory that another kernel of the chain writes or reads.
extern thread_local int g_use_pdl;   // set per step by the host thread that enqueues it
#define FO_PDL_TRIGGER() asm volatile("griddepcontrol.launch_dependents;" ::: "memory")
#define FO_PDL_WAIT() asm volatile("griddepcontrol.wait;" ::: "memory")
template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args&&... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = g_use_pdl ? 1 : 0;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

// ---- whole-step CTA timeline (development builds: FO_TRACE_BUILD=1 python -m freeze_omni_b200.build) ----------------
// Every CTA of the traced kernels appends one record {id word, 6 x %globaltimer} to a device buffer; tools/step_timeline.py
// replays ONE captured step and reconstructs the in-chain timeline (kernel spans, gaps, overlap under PDL).  Each
// translation unit owns its copy of the three device symbols (no relocatable device code); fo_set_option("trace", n) binds them.
#ifdef FO_TRACE_BUILD
#ifdef __CUDACC__
static __device__ unsigned long long* g_tr_buf = nullptr;
static __device__ unsigned int* g_tr_cnt = nullptr;
static __device__ unsigned int g_tr_cap = 0;
__device__ __forceinline__ unsigned long long fo_gtime() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}
#define FO_TR_DECL() __shared__ unsigned long long s_tr[6]
#define FO_TR_STAMP(i) do { s_tr[i] = fo_gtime(); } while (0)
// one thread, after the CTA's work is done; kid = kernel id, aux = free 16 bits (e.g. split / tile info)
#define FO_TR_FLUSH(kid, aux)                                                                                     \
    do {                                                                                                          \
        if (g_tr_buf) {                                                                                           \
            s_tr[5] = fo_gtime();                                                                                 \
            const unsigned int slot_ = atomicAdd(g_tr_cnt, 1u);                                                   \
            if (slot_ < g_tr_cap) {                                                                               \
                unsigned int smid_;                                                                               \
                asm volatile("mov.u32 %0, %%smid;" : "=r"(smid_));                                                \
                unsigned long long* r_ = g_tr_buf + (unsigned long long)slot_ * 8;                                \
                const unsigned long long lin_ = ((unsigned long long)blockIdx.z * gridDim.y + blockIdx.y) * gridDim.x + blockIdx.x; \
                r_[0] = (unsigned long long)(kid) | ((unsigned long long)smid_ << 8) | ((unsigned long long)((aux) & 0xFFFF) << 16) | (lin_ << 32); \
                r_[1] = (unsigned long long)gridDim.x | ((unsigned long long)gridDim.y << 20) | ((unsigned long long)gridDim.z << 40); \
                for (int i_ = 0; i_ < 6; ++i_) r_[2 + i_] = s_tr[i_];                                             \
            }                                                                                                     \
        }                                                                                                         \
    } while (0)
// raw record of six caller-supplied stamps (e.g. per-k-block arrival times of one CTA's MMA thread)
#define FO_TR_RAW(kid, aux, arr)                                                                                  \
    do {                                                                                                          \
        if (g_tr_buf) {                                                                                           \
            const unsigned int slot_ = atomicAdd(g_tr_cnt, 1u);                                                   \
            if (slot_ < g_tr_cap) {                                                                               \
                unsigned long long* r_ = g_tr_buf + (unsigned long long)slot_ * 8;                                \
                r_[0] = (unsigned long long)(kid) | ((unsigned long long)((aux) & 0xFFFF) << 16);                 \
                r_[1] = (unsigned long long)gridDim.x | ((unsigned long long)gridDim.y << 20) | ((unsigned long long)gridDim.z << 40); \
                for (int i_ = 0; i_ < 6; ++i_) r_[2 + i_] = (arr)[i_];                                            \
            }                                                                                                     \
        }                                                                                                         \
    } while (0)
#define FO_TR_BIND_DEF(fn)                                                                                        \
    void fn(unsigned long long* buf, unsigned int* cnt, unsigned int cap) {                                       \
        cudaMemcpyToSymbol(g_tr_buf, &buf, sizeof(buf));                                                          \
        cudaMemcpyToSymbol(g_tr_cnt, &cnt, sizeof(cnt));                                                          \
        cudaMemcpyToSymbol(g_tr_cap, &cap, sizeof(cap));                                                          \
    }
#endif
#else
#define FO_TR_DECL() do { } while (0)
#define FO_TR_STAMP(i) do { } while (0)
#define FO_TR_FLUSH(kid, aux) do { } while (0)
#define FO_TR_RAW(kid, aux, arr) do { } while (0)
#define FO_TR_BIND_DEF(fn) void fn(unsigned long long*, unsigned int*, unsigned int) {}
#endif
void trace_bind_gemm(unsigned long long* buf, unsigned int* cnt, unsigned int cap);
void trace_bind_attention(unsigned long long* buf, unsigned int* cnt, unsigned int cap);
void trace_bind_elementwise(unsigned long long* buf, unsigned int* cnt, unsigned int cap);
void trace_bind_fbank(unsigned long long* buf, unsigned int* cnt, unsigned int cap);
// ---- dtype helpers ---------------------------------------------------------------------------
__device__ __forceinline__ float to_f(float v) { return v; }
__device__ __forceinline__ float to_f(bf16 v) { return __bfloat162float(v); }
__device__ __forceinline__ float to_f(__half v) { return __half2float(v); }
template <typename T> __device__ __forceinline__ T from_f(float v);
template <> __device__ __forceinline__ float from_f<float>(float v) { return v; }
template <> __device__ __forceinline__ bf16 from_f<bf16>(float v) { return __float2bfloat16_rn(v); }
template <> __device__ __forceinline__ __half from_f<__half>(float v) { return __float2half_rn(fminf(fmaxf(v, -65504.f), 65504.f)); }
// weight rounding of a 16-bit context: to bf16 precision, stored in the container type
template <typename TW> __device__ __forceinline__ TW weight_cast(float v) { return from_f<TW>(v); }
template <> __device__ __forceinline__ __half weight_cast<__half>(float v) {
    return __float2half_rn(fminf(fmaxf(__bfloat162float(__float2bfloat16_rn(v)), -65504.f), 65504.f));
}
// two floats -> one packed 32-bit pair of the 16-bit type
template <typename T> __device__ __forceinline__ uint32_t pack2(float a, float b);
template <> __device__ __forceinline__ uint32_t pack2<bf16>(float a, float b) {
    __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
    return *reinterpret_cast<uint32_t*>(&h);
}
template <> __device__ __forceinline__ uint32_t pack2<__half>(float a, float b) {
    __half2 h = __floats2half2_rn(fminf(fmaxf(a, -65504.f), 65504.f), fminf(fmaxf(b, -65504.f), 65504.f));
    return *reinterpret_cast<uint32_t*>(&h);
}
template <typename T> __device__ __forceinline__ float2 unpack2(uint32_t v);
template <> __device__ __forceinline__ float2 unpack2<bf16>(uint32_t v) { return __bfloat1622float2(*reinterpret_cast<__nv_bfloat162*>(&v)); }
template <> __device__ __forceinline__ float2 unpack2<__half>(uint32_t v) { return __half22float2(*reinterpret_cast<__half2*>(&v)); }

// ---- implicit-GEMM operand addressing (conv2 of the subsampling, adapter conv) --------------------
// The activation operand of a GEMM is stored as [planes][rows][seg_len] (seg_len = channels, innermost).
// Column k of GEMM row r lives in segment s = k / seg_len at
//     A[(plane[s] * rows + r + rowoff[s]) * seg_len + k % seg_len]
// i.e. every k-segment is a plain 2-D box of one plane shifted by a row offset -- exactly what one TMA
// box load fetches.  The producers write their outputs in this layout (cmvn_conv1: 6 planes indexed by
// (kernel row, column parity); conv_stage at stride 2: 2 planes indexed by time parity), so neither convolution
// ever materialises im2col.  GEMM rows then run over a PADDED row grid; RowMap drops the padding rows
// and compacts the rest on the way out.  Plain row-major A is the case n_seg = 1.
struct AGather {
    static constexpr int MAX_SEG = 9;
    int seg_len;          // contiguous run along k (channels); K = n_seg * seg_len
    int n_seg;
    long long rows;       // rows per plane
    int planes;
    int plane[MAX_SEG];
    int rowoff[MAX_SEG];
};
inline AGather plain_rows(int K, long long rows) {
    AGather g;
    g.seg_len = K; g.n_seg = 1; g.rows = rows; g.planes = 1;
    for (int i = 0; i < AGather::MAX_SEG; ++i) { g.plane[i] = 0; g.rowoff[i] = 0; }
    return g;
}
// GEMM row r -> output row:  a = r / p1, b = (r % p1) / p0, c = r % p0;  kept iff b < v1 && c < v0;
// output row = a * q1 + b * q0 + c.  p1 == 0 is the identity.
struct RowMap {
    int p0 = 0, p1 = 0, v0 = 0, v1 = 0, q0 = 0, q1 = 0;
};
__host__ __device__ inline bool row_map(const RowMap& rm, int r, long long& dst) {
    if (rm.p1 == 0) { dst = r; return true; }
    const int a = r / rm.p1, rem = r - a * rm.p1;
    const int b = rem / rm.p0, c = rem - b * rm.p0;
    dst = (long long)a * rm.q1 + (long long)b * rm.q0 + c;
    return b < rm.v1 && c < rm.v0;
}

// ---- next-kernel L2 prefetch ------------------------------------------------------------------------
// A streaming step is a chain of short kernels, each of which starts by pulling data nobody has touched since the
// previous step (this GEMM's weights, this layer's KV rings) from HBM.  Those addresses do not depend on the
// activations, so every kernel asks L2 for the NEXT kernel's cold inputs while it runs (cp.async.bulk.prefetch.L2),
// taking the HBM latency off the critical path of the chain.
struct L2Prefetch {
    const void* ptr[2] = {nullptr, nullptr};
    long long bytes[2] = {0, 0};
};
#ifdef __CUDACC__
__device__ __forceinline__ void l2_prefetch_slice(const L2Prefetch& pf, int cta, int nctas, int tid, int nthreads) {
#pragma unroll
    for (int k = 0; k < 2; ++k) {
        if (pf.ptr[k] == nullptr) continue;
        const long long per = ((pf.bytes[k] + nctas - 1) / nctas + 2047) & ~2047LL;
        const long long start = (long long)cta * per, end = min(pf.bytes[k], start + per);
        const char* base = reinterpret_cast<const char*>(pf.ptr[k]);
        for (long long off = start + (long long)tid * 2048; off < end; off += (long long)nthreads * 2048) {
            const unsigned sz = (unsigned)min(2048LL, end - off) & ~15u;
            if (sz) asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(base + off), "r"(sz) : "memory");
        }
    }
}
#endif

// ---- GEMM epilogue ---------------------------------------------------------------------------
// C[m][n] = act((acc + bias[n]) * scale) (+ residual[m][n]);  written as fp32 (c_f32) and/or as the
// activation type (c_act).  residual may alias c_f32 (in-place residual stream).
struct Epilogue {
    const float* bias = nullptr;
    const float* residual = nullptr;  // fp32, leading dimension ldc
    float* c_f32 = nullptr;
    void* c_act = nullptr;            // float* or bf16* depending on the context dtype
    int ldc = 0;
    int relu = 0;
    float scale = 1.0f;
    int split_col = 0;                // > 0: columns < split_col go to c_f32 only, columns >= split_col to c_act only
    // Fused LayerNorm of the finished rows of c_f32 (the residual stream; requires N == ldc): the CTA that completes a
    // block of rows (last of the column tiles to arrive on the block's counter) normalises those rows and writes them
    // as the activation type (ln_act) and/or fp32 (ln_f32).  tcgen05 kernel only; gemm_ln() in fo_api.cu launches the
    // stand-alone kernel on the other paths.
    const float* ln_gamma = nullptr;
    const float* ln_beta = nullptr;
    float ln_eps = 1e-5f;
    void* ln_act = nullptr;
    float* ln_f32 = nullptr;
    int* ln_counters = nullptr;
    L2Prefetch prefetch;              // cold inputs of the kernels that follow (tcgen05 kernel only)
    // The caller runs a LayerNorm over the finished rows right after this GEMM and lets IT finish a split-K reduction:
    // every split CTA then just writes its raw accumulators as [split][M][N] fp32 and exits (no tile counters, no
    // last-CTA pass, no bias / residual here); layer_norm_reduce() folds  x += bias + sum_s partial_s  into its row pass.
    int defer_reduce = 0;
    // fp16-range guard of a 16-bit context (DESIGN 4a): every value the epilogue stages as fp16 for the tensor cores is
    // clamped to +-65504; when that clamp actually changes a value the kernel counts it here (fo_stats.act_saturations).
    // Only GEMM outputs are unbounded (FFN1 ReLU, K|V, conv outputs); LayerNorm / softmax-weighted outputs are bounded by
    // construction.  nullptr = not counted.
    unsigned long long* sat = nullptr;
};
#ifdef __CUDACC__
__device__ __forceinline__ void count_sat4(unsigned long long* sat, float a, float b, float c, float d) {
    if (sat && fmaxf(fmaxf(fabsf(a), fabsf(b)), fmaxf(fabsf(c), fabsf(d))) > 65504.f)
        atomicAdd(sat, (unsigned long long)((fabsf(a) > 65504.f) + (fabsf(b) > 65504.f) + (fabsf(c) > 65504.f) + (fabsf(d) > 65504.f)));
}
#endif

// C[rowmap(m), n] = A[m, :] . W[n, :]  for m < M (padded GEMM rows), n < N.  A/W are TIn (float or bf16),
// accumulate fp32.
template <typename TA, typename TW>
int gemm_simt(const TA* A, const AGather& ga, const TW* W, int M, int N, int K, const Epilogue& ep,
              const RowMap& rmap, cudaStream_t st);

// tcgen05 + TMA path (bf16 only).  Returns 1 if the shape is not supported (caller uses gemm_simt),
// <0 on error.  The workspace (split-K partials + tile counters) belongs to one context / one stream.
struct TcWorkspace {
    float* partial = nullptr;
    size_t partial_bytes = 0;
    int* counters = nullptr;       // split-K arrivals per output tile
    int* ln_counters = nullptr;    // fused-LayerNorm arrivals per row block
    int sms = 148;                 // SMs the context's grids spread over (its SM group, or the device)
};
struct TcTune { int swap, bn, split; };      // -1 / 0 = let the cost model decide
int gemm_tc_init();
int gemm_tc_workspace(TcWorkspace* ws);       // allocates; the caller frees the two device pointers
// the tile plan the host would pick for a context on the whole device (pure host logic; fo_debug_plan exposes it to the CPU tests)
void gemm_tc_plan(long long act_rows, int n_out, int K, int can_defer, int* swap, int* bn, int* split);
void gemm_tc_force(const TcTune& t);
void gemm_tc_plan_override(int N, int K, int swap, int bn, int split, int cap_kb);   // N <= 0 clears (development)
void gemm_tc_set_persist(int on);          // persistent tile loop for fat short-K GEMMs (default on)
long long gemm_tc_persist_launches();
void gemm_tc_force_producers(int npa, int npb);   // 0 = default
long long gemm_tc_launches();                // tcgen05 kernel launches so far (tests check the path taken)
long long gemm_tc_max_rows(int N);           // the most activation rows one GEMM of N output columns takes (its tile table)
// A and W: 16-bit operands of ONE format (fp16 when is_fp16, else bf16); c_act / ln_act are written in the same type.
int gemm_tc(const void* A, int is_fp16, const AGather& ga, const void* W, int M, int N, int K, const Epilogue& ep,
            const RowMap& rmap, const TcWorkspace& ws, cudaStream_t st, int* deferred_splits = nullptr);

// ---- frontend --------------------------------------------------------------------------------
struct FbankParams {
    int frame_len, frame_shift, fft_size, n_mel;
    const float* window;   // frame_len
    const float* mel;      // n_mel x (fft_size/2+1), zero outside each triangle
    const int* mel_lo;     // first non-zero fft bin per mel filter
    const int* mel_hi;     // one past the last non-zero bin
    int sms;               // SMs of the context: the grid-stride kernels launch 16 CTAs per SM
};
// Streaming: per session s = ids[b]: samples = [carry[s] (frame_len-frame_shift) | new chunk], m = frames_per_chunk
// frames; ring[s] <- [last ctx frames | new frames]; optional copy of the ring block to feats_out.
int fbank_stream(const FbankParams& p, const int32_t* ids, int n, const void* pcm, int pcm_is_i16, float scale,
                 int frames_per_chunk, int ctx_frames, float* carry, float* ring, float* feats_out,
                 cudaStream_t st);
// The same for cnt[b] consecutive chunks of session ids[b] (blocks (session, chunk) from off[b]; kmax the largest count):
// pcm (blocks, chunk samples); feats_out (blocks, ctx+m, n_mel) gets every block as fbank_stream would return it after the
// blocks before it, and each session ends holding its last block's carry and ring.  rows: (blocks, carry + chunk) fp32 scratch.
int fbank_stream_blocks(const FbankParams& p, const int32_t* ids, const int32_t* cnt, const int32_t* off, int n, int kmax,
                        int blocks, const void* pcm, int pcm_is_i16, float scale, int frames_per_chunk, int ctx_frames,
                        float* carry, float* ring, float* rows, float* feats_out, cudaStream_t st);
int fbank_offline(const FbankParams& p, const void* pcm, int pcm_is_i16, int B, long long n_samples, float scale,
                  float* out, cudaStream_t st);
// Utterances of different lengths back to back (fo_fbank_offline_packed, fo_encode_offline_packed_pcm): utterance b of n has
// frame_off[b + 1] - frame_off[b] frames (kaldi snip_edges: 1 + (n_samples - frame_len) / frame_shift), its samples from
// sample_off[b] of pcm; its frames go to rows out_row[b].. of out, and to rows frame_off[b].. of out2 (optional).  Every frame
// is computed as fbank_offline computes it.  Device tables; frames = frame_off[n].
struct FbankVarlen {
    const int32_t* frame_off = nullptr;   // n + 1 prefix sums of the frame counts
    const long long* sample_off = nullptr;
    const int32_t* out_row = nullptr;
    int n = 0;
    long long frames = 0;
};
int fbank_offline_packed(const FbankParams& p, const void* pcm, int pcm_is_i16, float scale, const FbankVarlen& vl, float* out,
                         float* out2, cudaStream_t st);

// ---- elementwise / normalisation ----------------------------------------------------------------
// CMVN + Conv2d(1->C,3,2) + ReLU, written as the A operand of the conv2 implicit GEMM:
// c1[kh*2 + (f1&1)][(b*T2 + t2)*(F2+1) + f1/2][c] = relu(conv1)[b][c][2*t2 + kh][f1]   (see conv2_gather)
template <typename TA>
int cmvn_conv1(const float* feats, int B, int T, int F, const float* mean, const float* istd, const float* w1,
               const float* b1, int C, TA* c1, cudaStream_t st);
// A-operand description and row map of conv2 (3x3, stride 2) over that layout; GEMM rows = B*T2*(F2+1)
void conv2_gather(int B, int T2, int F2, int C, AGather* ga, RowMap* rm);
// same for the adapter conv (kernel k, stride 2) over xin[time&1][b*RP + time/2][D], RP = (k-1+T+1)/2
void adapter_gather(int B, int T, int D, int k, AGather* ga, RowMap* rm);
// LayerNorm over the last dim of x (M, D) fp32.  y_act (activation type) and/or y_f32 outputs.
// act: 0 none, 1 relu, 2 gelu(erf); result multiplied by out_scale after the activation.
template <typename TA>
int layer_norm(const float* x, int M, int D, const float* gamma, const float* beta, float eps, int act,
               float out_scale, TA* y_act, float* y_f32, cudaStream_t st);
// x (M, D) += bias + sum_{s < nsplit} partial[s] (fixed order), then the row norm of the updated x (D <= 1024)
template <typename TA>
int layer_norm_reduce(float* x, const float* partial, int nsplit, const float* bias, int M, int D, const float* gamma,
                      const float* beta, float eps, TA* y_act, float* y_f32, cudaStream_t st);
// scale-copy (input-layer "none"): y = x * s
int scale_rows(const float* x, float* y, long long n, float s, cudaStream_t st);
// staging of an adapter conv (see conv_stage_kernel): virtual rows x[b][0..k-2] = left context (cache or 0),
// x[b][k-1+i] = in[b][i] (zeroed where mask == 0, or ReLU(in * scale + shift) when scale != null), C channels, stride 1
// (conv1d_gather layout) or 2 (adapter_gather layout); new cache = last k-1 rows (fp32), slot-resident (ids != null,
// (slot, 2, k-1, C) time-major) or explicit (B, C, k-1)
// Per-session rows of a call whose sessions bring different chunk counts (fo_encode_stream_chunks_v); cnt == null: every
// session has the T rows of the uniform layout.  Session b's real input is its first cnt[b] * unit of T padded rows; with
// `off` non-null, `in` is packed instead, session b's rows starting at row off[b] * unit.  The new cache comes from the real rows.
struct SessionRows {
    const int32_t* cnt = nullptr;
    const int32_t* off = nullptr;
    int unit = 0;
};
template <typename TA>
int conv_stage(const float* in, const uint8_t* mask, int B, int T, int C, int km1, int stride, const float* scale,
               const float* shift, const int32_t* ids, float* slot_cache, int32_t* slot_valid, const float* cache_in,
               float* cache_out, TA* xin, cudaStream_t st, const SessionRows& sr = SessionRows());
// Packs fp32 blocks of `bytes` from a per-session grid of kmax blocks to block order: src block b * kmax + j (j < cnt[b]) ->
// dst block off[b] + j.
int pack_session_blocks(const float* src, float* dst, long long bytes, int n, int kmax, const int32_t* cnt, const int32_t* off,
                        cudaStream_t st);
// The carried stride-2 adapter conv over chunks of odd t, run at stride 1 over each session's kmax * t grid rows: output m of
// chunk j is grid row j * t + 2 m.  src (n, kmax * t, C) -> dst (blocks, t_out, C), session b's chunks j < cnt[b] from block off[b].
int pick_chunk_rows(const float* src, int n, int kmax, int t, int t_out, int C, const int32_t* cnt, const int32_t* off, float* dst,
                    cudaStream_t st);
void conv1d_gather(int B, int T, int C, int k, AGather* ga, RowMap* rm);
// (B, T, C) -> zero-padded (B, lead + T + trail, C) in the activation type
template <typename TA>
int pad_rows(const TA* in, int B, int T, int C, int lead, int trail, TA* out, cudaStream_t st);
// runs of `gap` rows starting at rows at[0..n) of buf (device table) set to zero
template <typename TA>
int zero_row_runs(TA* buf, const int32_t* at, int n, int gap, int C, cudaStream_t st);
// fp32 rows of n utterances moved between layouts: utterance b's lens[b] (<= rows_max) rows from src row srow[b] to dst
// row drow[b] (device tables)
int copy_utt_rows(const float* src, const int32_t* srow, float* dst, const int32_t* drow, const int32_t* lens, int n, int rows_max,
                  int C, cudaStream_t st);
// Conv1dLinear's causal depthwise Conv1d over time (attention.py:217-224,251): y[r][c] = b[c] + sum_tau w[c][tau] *
// xin[r + tau][c], xin = [left context (k-1 rows) | x].  Streaming (ids != null): x is (n, t, C), the left context of
// session ids[b] lives in slot_cache (fp32, (k-1, C) per slot, stride slot_stride) and is replaced by the last k-1 rows
// of xin.  Offline (ids == null): x is (B, T, C) with zero left padding per utterance.  cnt / off (streaming, per-session
// chunk counts): session b's rows are the cnt[b] * t rows from row (off[b] - off[0]) * t; T is then the largest of them.
// With ids == null the same tables describe utterances packed end to end (t = 1), each with zero left context.
template <typename TA>
int depthwise_conv(const TA* x, int B, int T, int C, int k, const float* w, const float* bias, const int32_t* ids,
                   float* slot_cache, long long slot_stride, TA* y, cudaStream_t st, const int32_t* cnt = nullptr,
                   const int32_t* off = nullptr, int t = 0);
int subsample_mask(const int32_t* ilens, int B, int T, int T2, uint8_t* mask2, int32_t* ilens2, cudaStream_t st);
// attention-mask rows + input start rows of the LLM hand-off (audioLLM.py:404-411); device pointers
int handoff_mask(const uint8_t* onset, const uint8_t* prefix_mask, int n, int P, int t_out, int rows, uint8_t* attn_mask,
                 int32_t* row_start, cudaStream_t st);
// the hand-off of one pass of the recording entries: pass block b's fp32 adapter rows (y) as fp16 into caller block tab[b].x,
// its mask row and row_start from onset flag tab[b].y (tab: device, nblk entries)
int handoff_rows(const float* y, const int2* tab, int nblk, int t_out, int E, void* embeds_f16, int rows, int P,
                 const uint8_t* prefix_mask, uint8_t* attn_mask, int32_t* row_start, unsigned long long* sat, cudaStream_t st);
int stride2_mask(const uint8_t* mask, int B, int T, int To, uint8_t* out, cudaStream_t st);

// ---- attention -----------------------------------------------------------------------------------
struct AttnStream {
    const int32_t* ids;       // (n) session slots
    const int32_t* n_frames;  // per slot: encoder frames appended before this step
    const int32_t* pe_index;  // per slot
    int n, t, H, ring_cap, window, full_chunk, pe_wrap, pos_rows;
    long long ring_slot_stride;   // elements between sessions of one layer: 2*H*ring_cap*64
    L2Prefetch prefetch;          // cold inputs of the kernels that follow
    // the QKV GEMM may have left raw split-K partials [nsplit][n*t][3D] fp32 (Epilogue::defer_reduce): the kernel then forms
    // q / k / v = sum_s partial_s + bias itself instead of reading the finished qkv / q32 rows
    const float* part = nullptr;
    const float* part_bias = nullptr;
    int nsplit = 0;
    long long part_stride = 0;
    // consecutive chunks per session (attention_chunks: fo_encode_stream_chunks[_v], passes of fo_stream_steps_v): rows are
    // (session, chunk, frame); session b brings cnt[b] chunks and its rows start at row (off[b] - off[0]) * t; chunk j of a
    // session is attended exactly as the j-th of cnt[b] sequential calls (chunk_size: pe_index step).  `chunks` is the number
    // of chunks one CTA attends (it sizes shared memory).  attention_stream reads rows b * t and no table.
    int chunks = 1;
    int chunk_size = 0;
    const int32_t* cnt = nullptr;
    const int32_t* off = nullptr;
};
// staged keys of the multi-chunk attention (window + chunks * t at most): bounds the chunks of one call
constexpr int STREAM_CHUNKS_MAX_KEYS = 128;
// encoder frames of one streaming chunk (query rows of an attention CTA, the MMA's N); fo_create caps the context's max_t here
constexpr int STREAM_MAX_T = 8;
// qkv (n*t, 3*D) activation type (K and V columns are read from it); q32 (n*t, 3*D) fp32 whose first D
// columns hold Q (the QKV GEMM keeps Q in fp32, Epilogue::split_col); ring = this layer's
// (slot, 2, H, ring_cap, 64); ptab (pos_rows, D) fp32; out (n*t, D).  One chunk per session; appends the new K/V rows to
// the ring.
template <typename TA>
int attention_stream(const AttnStream& a, const TA* qkv, const float* q32, TA* ring, const TA* ptab_h,
                     const float* pos_u, const float* pos_v, TA* out, cudaStream_t st);
// Session b's cnt[b] consecutive chunks (cnt[b] <= groups * a.chunks), with the same tensors.  One CTA per (session, head,
// group of a.chunks chunks), grid z = `groups`; each chunk sees window + t keys, staged from the ring (frames before the
// call) and from the call's own K|V rows in qkv.  The last min(cnt[b] * t, ring_cap) new frames go to the ring after every
// read of it: appended by the CTA itself when groups == 1 (the only reader of its ring), else by a second kernel.
template <typename TA>
int attention_chunks(const AttnStream& a, int groups, const TA* qkv, const float* q32, TA* ring, const TA* ptab_h,
                     const float* pos_u, const float* pos_v, TA* out, cudaStream_t st);
// ptab_h: the same table as [H][pos_rows][64] in the activation type (rows of one head contiguous -> one bulk copy)
template <typename TA>
int ptab_head_major(const float* in, int pos_rows, int H, TA* out, cudaStream_t st);
// offline: qkv (B*T, 3*D); valid lengths ilens (B); window from (chunk, left); positions 0..T-1.
template <typename TA>
int attention_offline(const TA* qkv, const float* q32, int B, int T, int H, const int32_t* ilens, int chunk, int left,
                      const float* ptab, const TA* ptab_h, int pos_rows, const float* pos_u, const float* pos_v, TA* out,
                      cudaStream_t st);
// offline, utterances of different lengths packed end to end (fo_encode_offline_packed): utterance b has lens[b] rows from
// row rows[b] of qkv / q32 / out, all valid, positions 0..lens[b]-1.  One CTA per tile table entry {b, query tile} and head;
// the host lists ceil(lens[b] / attention_offline_tile_rows()) tiles per utterance.  Device pointers.
struct AttnVarlen {
    const int2* tiles = nullptr;
    const int32_t* lens = nullptr;
    const int32_t* rows = nullptr;
    int n = 0;                    // tile table entries
};
int attention_offline_tile_rows(int is16);
// tmax: the longest utterance (bounds pos_rows as T does for the padded form)
template <typename TA>
int attention_offline_packed(const TA* qkv, const float* q32, const AttnVarlen& vl, int B, int tmax, int H, int chunk, int left,
                             const float* ptab, const TA* ptab_h, int pos_rows, const float* pos_u, const float* pos_v, TA* out,
                             cudaStream_t st);
// end of a streaming step: n_frames += t, pe_index = pe_index % wrap + chunk_size (attention.py:107,120),
// and flip the live half of the double-buffered adapter cache.  Either group may be null.  chunks > 1: the session
// advanced by that many chunks of t frames (pe_index stepped `chunks` times; the adapter cache still flips once).  cnt
// non-null: session b's own count cnt[b] replaces `chunks`.
int advance_sessions(const int32_t* ids, int n, int t, int chunk_size, int pe_wrap, int32_t* n_frames,
                     int32_t* pe_index, int32_t* adapter_valid, cudaStream_t st, int chunks = 1,
                     const int32_t* cnt = nullptr);

// ---- weight-streaming layer stack for a handful of sessions (fo_stack.cu) ---------------------------
// All transformer layers of a streaming step in ONE cooperative launch when the step has at most 16 token rows (1-4
// sessions): at that size a layer is pure weight streaming, and the per-kernel chain spends ~5 us per kernel on
// dependency latency (181 kernels, 0.94 ms at one session against an HBM floor of 0.12 ms).  See fo_stack.cu.
struct StackLayer {                 // one entry per layer, device resident
    const __half *wqkv, *wo, *w1, *w2;            // [3D][D], [D][D], [FF][D], [D][FF], K-major, bf16-rounded in fp16 containers;
                                                  // the kernel's own copy with every row padded by 16 bytes (row pitch 2K + 16)
    const float *bqkv, *bo, *b1, *b2;
    const float *ln1g, *ln1b, *ln2g, *ln2b, *pos_u, *pos_v;
    const __half* ptab_h;                         // [H][pos_rows][64], chunk-swizzled by position
    __half* ring;                                 // this layer's (slot, 2, H, ring_cap, 64)
};
struct StackArgs {
    const StackLayer* layers = nullptr;
    int L = 0, D = 0, FF = 0;
    AttnStream a;                                 // ids / n_frames / pe_index / n / t / H / ring geometry
    float* x = nullptr;                           // residual stream (n*t, D) fp32, in place
    float* q32 = nullptr;                         // (n*t, D) fp32
    __half* kv = nullptr;                         // (n*t, 2D) the chunk's own K | V rows
    __half* att = nullptr;                        // (n*t, D)
    __half* ffh = nullptr;                        // (n*t, FF)
    const float* after_g = nullptr;               // after_norm -> enc_out (n*t, D) fp32
    const float* after_b = nullptr;
    float* enc_out = nullptr;
    unsigned int* bar = nullptr;                  // grid-barrier flags, one per CTA (<= 1024), all equal between launches
    unsigned long long* sat = nullptr;            // fp16-range guard counter (Epilogue::sat)
    unsigned long long* trace = nullptr;          // development: %globaltimer of CTA 0 after every grid barrier, [L*5 + 2]
};
constexpr int STACK_MAX_ROWS = 16;
// One cooperative launch of G CTAs, G = the SMs of the context (its SM group, or the device); smem_max = opt-in shared memory
// per CTA.  0 = launched; 1 = shape not supported or the grid not co-resident (the caller runs the per-kernel chain); < 0 error
int stream_stack(const StackArgs& a, int G, int smem_max, cudaStream_t st);
// host-only: does a step of n sessions x t frames qualify on a device of `sms` SMs with smem_max bytes of shared memory per CTA,
// and with which plan (dynamic shared memory, K chunk of the FFN2 activations, weight rows per CTA and phase); 1 = no
int stack_plan(int D, int FF, int H, int n, int t, int window, int L, int sms, int smem_max, int* smem_bytes, int* ffn2_chunk,
               int* rows_qkv, int* rows_ffn1, int* rows_out);

// ---- SM groups (fo_partition.cu): CUDA green contexts of fo_create_on_sms ---------------------------------------
constexpr int SM_GROUP_GRANULE = 8;           // smallest group and its multiple on sm_90 and later (cuda.h, green contexts)
// the green context of group `group` of `split` equal groups of `device`'s SMs (made at the first use, kept for the process)
int sm_group_acquire(int device, int split, int group, void** green, int* sms);
int sm_group_stream(void* green, cudaStream_t* st);          // a non-blocking stream whose work runs on the group's SMs
int sm_ids(int32_t* out, int n, cudaStream_t st);            // n CTAs write their %smid (fo_debug_sm_ids)

// ---- conversions -----------------------------------------------------------------------------------
int f32_to_bf16(const float* src, bf16* dst, long long n, cudaStream_t st);
int f32_to_act16(const float* src, act16* dst, long long n, cudaStream_t st);
int f32_to_weight16(const float* src, act16* dst, long long n, cudaStream_t st);   // bf16-rounded, fp16 container
int bf16_to_f32(const bf16* src, float* dst, long long n, cudaStream_t st);
int act16_to_f32(const act16* src, float* dst, long long n, cudaStream_t st);
// dst[n][perm(k)] = src[n][k] style weight repacks (done once at finalize)
template <typename TW>
int repack_conv2(const float* w, int C, TW* out, cudaStream_t st);          // (co,ci,3,3) -> [co][(kh*3+kw)*C+ci]
template <typename TW>
int repack_sublinear(const float* w, int C, int F2, TW* out, cudaStream_t st); // [n][c*F2+f] -> [n][f*C+c]
template <typename TW>
int repack_adapter_conv(const float* w, int C2, int C, int k, TW* out, cudaStream_t st); // (co,ci,k) -> [co][tau*C+ci]
template <typename TW>
int convert_weight(const float* w, long long n, TW* out, cudaStream_t st);
// ring <-> reference (H, n, 64) layout
template <typename TA>
int ring_export(const TA* ring_kv, int H, int ring_cap, long long first_frame, int n, float* out, cudaStream_t st);
template <typename TA>
int ring_import(TA* ring_kv, int H, int ring_cap, long long first_frame, int n, const float* in, cudaStream_t st);

// ---- session snapshots (fo_session.cu; the record format is fo_api.cu's, see fo_session_save there) ------------------
// One flat fp32 section of a record: `bytes` of each slot's state, copied as they are.
struct SnapSeg {
    char* base = nullptr;          // the context's array (slot 0)
    long long slot_stride = 0;     // bytes between slots
    long long rec_off = 0;         // byte offset inside a record
    long long bytes = 0;
    int adapter_half = 0;          // 1: double-buffered adapter cache, two halves of `bytes`; the live one is picked by ad_valid
};
constexpr int SNAP_HDR_WORDS = 64;             // header: 256 bytes of int32 words
constexpr int SNAP_W_NFRAMES = 56, SNAP_W_PE = 57, SNAP_W_ADVALID = 58;   // per-session words; the rest is the same in every record
constexpr int SNAP_MAX_SEGS = 5;
struct SnapArgs {
    const int32_t* ids = nullptr;  // (n) slots, device
    int n = 0;
    char* rec = nullptr;           // n records of rec_bytes
    long long rec_bytes = 0;
    // KV rings [L][S][K|V][H][cap][64] of esz-byte elements (16-bit rings chunk-swizzled by frame); null: no encoder
    char* ring = nullptr;
    int L = 0, S = 0, H = 0, cap = 0, window = 0, esz = 0;
    long long kv_off = 0;          // record section [L][K|V][H][window][64]
    int32_t *n_frames = nullptr, *pe_index = nullptr, *ad_valid = nullptr;
    SnapSeg seg[SNAP_MAX_SEGS];
    int nseg = 0;
    int32_t hdr[SNAP_HDR_WORDS];   // pack: the header words every record starts with
};
// pack: slots -> records (header included); unpack: records -> slots (n_frames, pe_index, adapter flag from the headers,
// which the caller has validated).  One launch each on `st`.
int session_pack(const SnapArgs& a, cudaStream_t st);
int session_unpack(const SnapArgs& a, cudaStream_t st);

}  // namespace fo
