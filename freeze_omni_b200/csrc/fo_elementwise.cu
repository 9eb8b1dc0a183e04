// HBM-bound kernels of the path: CMVN + first subsampling conv, LayerNorm variants, adapter cache
// staging, mask subsampling, weight repacks and KV-ring import/export.  All of them move each byte
// once, with the channel dimension innermost so warps read and write full 128-byte lines.
#include "fo_common.cuh"

namespace fo {

namespace {

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// ---- CMVN + Conv2d(1 -> C, 3x3, stride 2) + ReLU ------------------------------------------------
// reference: encoder/cmvn.py:32-34 then subsampling.py:28-29.  One CTA per (b, t1): the three input
// rows are normalised into shared memory once, each thread owns CPT consecutive output channels
// (weights in registers) and sweeps the F1 frequency positions; stores are channel-contiguous.
// Output layout = A operand of the conv2 implicit GEMM (conv2_gather): row t1 lands in the kernel-row
// plane(s) it serves (t1 odd: kh=1; t1 even: kh=0 at t2=t1/2 and kh=2 at t2=t1/2-1), column f1 in the
// parity plane f1&1 at f1/2, rows of F2+1 entries.
template <typename TA, int CPT>
__global__ void __launch_bounds__(256)
cmvn_conv1_kernel(const float* __restrict__ feats, int T, int F, const float* __restrict__ mean,
                  const float* __restrict__ istd, const float* __restrict__ w1, const float* __restrict__ b1,
                  int C, int T2, int F1, int F2P, long long NR, TA* __restrict__ c1) {
    extern __shared__ float rows[];     // 3 * F
    FO_PDL_TRIGGER();
    FO_PDL_WAIT();
    const int b = blockIdx.y, t1 = blockIdx.x;
    for (int i = threadIdx.x; i < 3 * F; i += blockDim.x) {
        int r = i / F, f = i - r * F;
        float v = feats[((long long)b * T + 2 * t1 + r) * F + f];
        rows[i] = mean ? (v - mean[f]) * istd[f] : v;
    }
    __syncthreads();
    for (int c0 = threadIdx.x * CPT; c0 < C; c0 += blockDim.x * CPT) {
        float w[CPT][9], bias[CPT];
#pragma unroll
        for (int j = 0; j < CPT; ++j) {
            bias[j] = b1[c0 + j];
#pragma unroll
            for (int q = 0; q < 9; ++q) w[j][q] = w1[(c0 + j) * 9 + q];
        }
        // destinations of this conv1 row: (kernel row kh, output row t2)
        int kh_a, t2_a, kh_b = -1, t2_b = 0;
        if (t1 & 1) { kh_a = 1; t2_a = t1 >> 1; }
        else {
            kh_a = 0; t2_a = t1 >> 1;
            if (t1 >= 2) { kh_b = 2; t2_b = (t1 >> 1) - 1; }
            if (t2_a >= T2) { kh_a = kh_b; t2_a = t2_b; kh_b = -1; }
        }
        TA* out_a = c1 + (((long long)kh_a * 2) * NR + ((long long)b * T2 + t2_a) * F2P) * C + c0;
        TA* out_b = kh_b >= 0 ? c1 + (((long long)kh_b * 2) * NR + ((long long)b * T2 + t2_b) * F2P) * C + c0 : nullptr;
        for (int f1 = 0; f1 < F1; ++f1) {
            float x[9];
#pragma unroll
            for (int r = 0; r < 3; ++r)
#pragma unroll
                for (int q = 0; q < 3; ++q) x[r * 3 + q] = rows[r * F + 2 * f1 + q];
            TA v[CPT];
#pragma unroll
            for (int j = 0; j < CPT; ++j) {
                float a = bias[j];
#pragma unroll
                for (int q = 0; q < 9; ++q) a = fmaf(w[j][q], x[q], a);
                v[j] = from_f<TA>(fmaxf(a, 0.f));
            }
            const long long off = ((long long)(f1 & 1) * NR + (f1 >> 1)) * C;
            if (sizeof(TA) == 2) {
                *reinterpret_cast<uint2*>(out_a + off) = *reinterpret_cast<uint2*>(v);
                if (out_b) *reinterpret_cast<uint2*>(out_b + off) = *reinterpret_cast<uint2*>(v);
            } else {
                *reinterpret_cast<uint4*>(out_a + off) = *reinterpret_cast<uint4*>(v);
                if (out_b) *reinterpret_cast<uint4*>(out_b + off) = *reinterpret_cast<uint4*>(v);
            }
        }
    }
}

// ---- LayerNorm ---------------------------------------------------------------------------------
// one warp per row, 4 rows per CTA (a 256-row streaming step spreads over 64 SMs); two-pass in registers (mean, then
// centred variance) like ATen's CPU kernel.  The row and gamma/beta are all requested before the first reduction so
// one memory latency covers them.
template <typename TA, int MAXV>
__global__ void __launch_bounds__(128)
layer_norm_kernel(const float* __restrict__ x, int M, int D, const float* __restrict__ gamma,
                  const float* __restrict__ beta, float eps, int act, float out_scale, TA* __restrict__ y_act,
                  float* __restrict__ y_f32) {
    FO_PDL_TRIGGER();
    const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    const int nv = D >> 7;                    // float4 per lane
    float4 g[MAXV], bt[MAXV];
    if (MAXV <= 8) {                          // weights do not depend on the previous kernel: fetch them before the wait
#pragma unroll
        for (int i = 0; i < MAXV; ++i)
            if (i < nv) {
                g[i] = *reinterpret_cast<const float4*>(gamma + (i * 32 + lane) * 4);
                bt[i] = *reinterpret_cast<const float4*>(beta + (i * 32 + lane) * 4);
            }
    }
    FO_PDL_WAIT();
    if (row >= M) return;
    const float4* xr = reinterpret_cast<const float4*>(x + (long long)row * D);
    float4 v[MAXV];
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < MAXV; ++i)
        if (i < nv) v[i] = xr[i * 32 + lane];
#pragma unroll
    for (int i = 0; i < MAXV; ++i)
        if (i < nv) s += v[i].x + v[i].y + v[i].z + v[i].w;
    // eps < 0: per-channel affine only (BatchNorm1d in eval mode with the running statistics folded into gamma / beta)
    const bool affine_only = eps < 0.f;
    const float mu = affine_only ? 0.f : warp_sum(s) / D;
    float q = 0.f;
#pragma unroll
    for (int i = 0; i < MAXV; ++i)
        if (i < nv) {
            float a = v[i].x - mu, b = v[i].y - mu, c = v[i].z - mu, d = v[i].w - mu;
            q += a * a + b * b + c * c + d * d;
        }
    const float rstd = affine_only ? 1.f : rsqrtf(warp_sum(q) / D + eps);
#pragma unroll
    for (int i = 0; i < MAXV; ++i)
        if (i < nv) {
            const int col = (i * 32 + lane) * 4;
            float4 gg, bb;
            if (MAXV <= 8) { gg = g[i]; bb = bt[i]; }
            else {
                gg = *reinterpret_cast<const float4*>(gamma + col);
                bb = *reinterpret_cast<const float4*>(beta + col);
            }
            float o[4] = {(v[i].x - mu) * rstd * gg.x + bb.x, (v[i].y - mu) * rstd * gg.y + bb.y,
                          (v[i].z - mu) * rstd * gg.z + bb.z, (v[i].w - mu) * rstd * gg.w + bb.w};
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                if (act == 1) o[j] = fmaxf(o[j], 0.f);
                else if (act == 2) o[j] = 0.5f * o[j] * (1.f + erff(o[j] * 0.70710678118654752440f));
                o[j] *= out_scale;
            }
            long long off = (long long)row * D + col;
            if (y_f32) *reinterpret_cast<float4*>(y_f32 + off) = make_float4(o[0], o[1], o[2], o[3]);
            if (y_act) {
                TA t[4];
#pragma unroll
                for (int j = 0; j < 4; ++j) t[j] = from_f<TA>(o[j]);
                if (sizeof(TA) == 2) *reinterpret_cast<uint2*>(y_act + off) = *reinterpret_cast<uint2*>(t);
                else *reinterpret_cast<uint4*>(y_act + off) = *reinterpret_cast<uint4*>(t);
            }
        }
}

// LayerNorm that also finishes a deferred split-K reduction (Epilogue::defer_reduce): x += bias + sum_s partial_s in
// split order (deterministic), x written back, then the row norm.  TWO warps per row (each lane holds D/256 float4 of the
// row), so that x and all NS partial rows are in flight together: with one warp per row the partial loads of the splits
// went out one after the other (5.1 us per launch in profiles/r01_j, 14 % of the step).  D <= 1024, D % 256 == 0.
template <typename TA, int NS>
__global__ void __launch_bounds__(128)
layer_norm_reduce_kernel(float* __restrict__ x, const float* __restrict__ partial, int nsplit, const float* __restrict__ bias,
                         int M, int D, const float* __restrict__ gamma, const float* __restrict__ beta, float eps,
                         TA* __restrict__ y_act, float* __restrict__ y_f32) {
    __shared__ float red[2][2][2];               // [row in CTA][half][sum | sq]
    FO_TR_DECL();
    if (threadIdx.x == 0) FO_TR_STAMP(0);
    FO_PDL_TRIGGER();
    const int wid = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int rr = wid >> 1, half = wid & 1;
    const int row = blockIdx.x * 2 + rr;
    const int nv = D >> 8;                       // float4 per lane
    const int f0 = half * (D >> 3) + lane;       // first float4 of this lane within the row (half a row = D/8 float4)
    float4 g[4], bt[4], bs[4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
        if (i < nv) {                            // constants: before the dependency wait
            g[i] = *(reinterpret_cast<const float4*>(gamma) + f0 + i * 32);
            bt[i] = *(reinterpret_cast<const float4*>(beta) + f0 + i * 32);
            bs[i] = bias ? *(reinterpret_cast<const float4*>(bias) + f0 + i * 32) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
    FO_PDL_WAIT();
    if (threadIdx.x == 0) FO_TR_STAMP(1);
    const bool live = row < M;
    float4* xr = reinterpret_cast<float4*>(x + (long long)(live ? row : 0) * D) + f0;
    const long long split_stride = ((long long)M * D) >> 2;
    const float4* pr = reinterpret_cast<const float4*>(partial + (long long)(live ? row : 0) * D) + f0;
    float4 xv[4], v[4];
    if (live) {
        float4 pv[NS > 0 ? NS : 1][4];
#pragma unroll
        for (int i = 0; i < 4; ++i)
            if (i < nv) xv[i] = xr[i * 32];
        if (NS > 0) {
#pragma unroll
            for (int s = 0; s < NS; ++s)
#pragma unroll
                for (int i = 0; i < 4; ++i)
                    if (i < nv) pv[s][i] = __ldcg(pr + s * split_stride + i * 32);
        }
#pragma unroll
        for (int i = 0; i < 4; ++i) v[i] = make_float4(0.f, 0.f, 0.f, 0.f);
        // same association as the GEMM's own split-K epilogue: ((sum_s partial_s) + bias) + residual -> bit-identical results
        if (NS > 0) {
#pragma unroll
            for (int s = 0; s < NS; ++s)
#pragma unroll
                for (int i = 0; i < 4; ++i)
                    if (i < nv) { v[i].x += pv[s][i].x; v[i].y += pv[s][i].y; v[i].z += pv[s][i].z; v[i].w += pv[s][i].w; }
        } else {
            for (int s = 0; s < nsplit; ++s)
#pragma unroll
                for (int i = 0; i < 4; ++i)
                    if (i < nv) {
                        const float4 a = __ldcg(pr + s * split_stride + i * 32);
                        v[i].x += a.x; v[i].y += a.y; v[i].z += a.z; v[i].w += a.w;
                    }
        }
    }
    float sum = 0.f;
#pragma unroll
    for (int i = 0; i < 4; ++i)
        if (i < nv && live) {
            v[i].x = (v[i].x + bs[i].x) + xv[i].x; v[i].y = (v[i].y + bs[i].y) + xv[i].y;
            v[i].z = (v[i].z + bs[i].z) + xv[i].z; v[i].w = (v[i].w + bs[i].w) + xv[i].w;
            xr[i * 32] = v[i];
            sum += v[i].x + v[i].y + v[i].z + v[i].w;
        }
    sum = warp_sum(sum);
    if (lane == 0) red[rr][half][0] = sum;
    __syncthreads();
    const float mu = (red[rr][0][0] + red[rr][1][0]) / D;
    float q = 0.f;
#pragma unroll
    for (int i = 0; i < 4; ++i)
        if (i < nv && live) {
            const float a = v[i].x - mu, b = v[i].y - mu, c = v[i].z - mu, d = v[i].w - mu;
            q += a * a + b * b + c * c + d * d;
        }
    q = warp_sum(q);
    if (lane == 0) red[rr][half][1] = q;
    __syncthreads();
    if (threadIdx.x == 0) { FO_TR_STAMP(2); FO_TR_STAMP(3); FO_TR_STAMP(4); FO_TR_FLUSH(3, 0); }
    if (!live) return;
    const float rstd = rsqrtf((red[rr][0][1] + red[rr][1][1]) / D + eps);
#pragma unroll
    for (int i = 0; i < 4; ++i)
        if (i < nv) {
            const int col = (f0 + i * 32) * 4;
            const float o0 = (v[i].x - mu) * rstd * g[i].x + bt[i].x, o1 = (v[i].y - mu) * rstd * g[i].y + bt[i].y;
            const float o2 = (v[i].z - mu) * rstd * g[i].z + bt[i].z, o3 = (v[i].w - mu) * rstd * g[i].w + bt[i].w;
            const long long off = (long long)row * D + col;
            if (y_f32) *reinterpret_cast<float4*>(y_f32 + off) = make_float4(o0, o1, o2, o3);
            if (y_act) {
                TA t[4] = {from_f<TA>(o0), from_f<TA>(o1), from_f<TA>(o2), from_f<TA>(o3)};
                if (sizeof(TA) == 2) *reinterpret_cast<uint2*>(y_act + off) = *reinterpret_cast<uint2*>(t);
                else *reinterpret_cast<uint4*>(y_act + off) = *reinterpret_cast<uint4*>(t);
            }
        }
}

__global__ void scale_rows_kernel(const float* __restrict__ x, float* __restrict__ y, long long n, float s) {
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) y[i] = x[i] * s;
}

// ---- causal-conv staging of the adapter (CNNSubsampling adapter.py:120-143; CNNAdapter adapter.py:33-52) ---------------
// grid (B, km1 + T); thread = channel.  Builds the A operand of a causal Conv1d(C -> *, k, stride) run as an implicit GEMM
// from fp32 rows `in` (B, T, C):
//   virtual rows [0, km1) = left context (old cache, or zeros), rows [km1, km1 + T) = f(in) with
//   f(v) = v (masked to 0 where mask == 0)                         when scale == nullptr  (first conv: the module's input)
//   f(v) = max(v * scale[c] + shift[c], 0)                         otherwise             (second conv: ReLU(BatchNorm_eval(conv1)))
// stride 1: one plane, xin[b * (km1 + T) + r][C] (conv1d_gather);  stride 2: two planes by row parity (adapter_gather).
// The new cache = the last km1 virtual rows, fp32: explicit caches in the reference layout (B, C, km1); slot-resident caches
// time-major and double-buffered per slot: slot_valid = 0 (None), 1 (half 0 live), 2 (half 1 live); the new rows go to the
// other half and advance_sessions() flips the flag after every block has read it.  SessionRows: rows of a session past its
// real length Tb are padding (0, no cache), and the cache comes from its last real rows.
template <typename TA>
__global__ void conv_stage_kernel(const float* __restrict__ in, const uint8_t* __restrict__ mask, int T, int C, int km1, int stride,
                                  const float* __restrict__ scale, const float* __restrict__ shift,
                                  const int32_t* __restrict__ ids, float* slot_cache, const int32_t* __restrict__ slot_valid,
                                  const float* __restrict__ cache_in, float* cache_out, TA* __restrict__ xin, SessionRows sr) {
    FO_PDL_TRIGGER();
    FO_PDL_WAIT();
    const int b = blockIdx.x, r = blockIdx.y;          // r in [0, km1 + T)
    int Tb = T;
    long long in0 = (long long)b * T;                  // input row of the session's first frame
    if (sr.cnt) {
        Tb = sr.cnt[b] * sr.unit;
        if (sr.off) in0 = (long long)sr.off[b] * sr.unit;
    }
    const int slot = ids ? ids[b] : -1;
    const int live = ids ? slot_valid[slot] : 0;
    const bool have_old = ids ? (live != 0) : (cache_in != nullptr);
    const float* old_half = ids ? slot_cache + ((long long)slot * 2 + (live == 2 ? 1 : 0)) * km1 * C : nullptr;
    float* new_half = ids ? slot_cache + ((long long)slot * 2 + (live == 1 ? 1 : 0)) * km1 * C : nullptr;
    const int R1 = km1 + T, RP = (km1 + T + 1) >> 1;
    for (int c = threadIdx.x; c < C; c += blockDim.x) {
        float v;
        if (r < km1) {
            if (!have_old) v = 0.f;
            else if (ids) v = old_half[(long long)r * C + c];
            else v = cache_in[((long long)b * C + c) * km1 + r];
        } else if (r - km1 < Tb) {
            const int t = r - km1;
            v = in[(in0 + t) * C + c];
            if (scale) v = fmaxf(v * scale[c] + shift[c], 0.f);
            else if (mask && !mask[(long long)b * T + t]) v = 0.f;
        } else {
            v = 0.f;                                     // padding behind a session's real rows (causal: no real output reads it)
        }
        if (stride == 1) xin[((long long)b * R1 + r) * C + c] = from_f<TA>(v);
        else xin[(((long long)(r & 1) * gridDim.x + b) * RP + (r >> 1)) * C + c] = from_f<TA>(v);
        const int cr = r - Tb;                           // row of the new cache this element becomes
        if (cr >= 0 && cr < km1) {
            if (ids) new_half[(long long)cr * C + c] = v;
            else if (cache_out) cache_out[((long long)b * C + c) * km1 + cr] = v;
        }
    }
}

// grid (ceil(T / DW_TB), B), block = channels (strided).  Each thread owns one channel of DW_TB consecutive output rows:
// it walks the k-1+DW_TB input rows once (sliding window in registers), so every input element is read once per CTA.
constexpr int DW_TB = 16;
constexpr int DW_KMAX = 16;
template <typename TA>
__global__ void __launch_bounds__(256)
depthwise_conv_kernel(const TA* __restrict__ x, int T, int C, int k, const float* __restrict__ w,
                      const float* __restrict__ bias, const int32_t* __restrict__ ids, float* slot_cache,
                      long long slot_stride, TA* __restrict__ y, int row0, const int32_t* __restrict__ cnt,
                      const int32_t* __restrict__ off, int t) {
    FO_PDL_TRIGGER();
    FO_PDL_WAIT();
    const int b = blockIdx.y, r0 = row0 + blockIdx.x * DW_TB;
    long long base = (long long)b * T;                 // the session's first row
    if (cnt) {                                         // per-session counts: cnt[b] * t rows from block off[b] - off[0]
        base = (long long)(off[b] - off[0]) * t;
        T = cnt[b] * t;
        if (r0 >= T) return;
    }
    const int nr = min(DW_TB, T - r0);
    const int km1 = k - 1;
    float* cache = ids ? slot_cache + (long long)ids[b] * slot_stride : nullptr;
    for (int c = threadIdx.x; c < C; c += blockDim.x) {
        float wv[DW_KMAX], win[DW_KMAX];
#pragma unroll
        for (int q = 0; q < DW_KMAX; ++q) wv[q] = q < k ? w[c * k + q] : 0.f;
        const float bv = bias[c];
        // left context of the first output row: rows r0-km1 .. r0-1 of the virtual [context | x]
#pragma unroll
        for (int q = 0; q < DW_KMAX - 1; ++q) {
            if (q < km1) {
                const int r = r0 - km1 + q;
                float v = 0.f;
                if (r >= 0) v = to_f(x[(base + r) * C + c]);
                else if (cache) v = cache[(long long)(km1 + r) * C + c];        // row r of the old context, r in [-km1, -1]
                win[q] = v;
            }
        }
        for (int i = 0; i < nr; ++i) {
            const float cur = to_f(x[(base + r0 + i) * C + c]);
            float acc = bv;
#pragma unroll
            for (int q = 0; q < DW_KMAX - 1; ++q)
                if (q < km1) acc = fmaf(wv[q], win[q], acc);
            acc = fmaf(wv[km1], cur, acc);
            y[(base + r0 + i) * C + c] = from_f<TA>(acc);
#pragma unroll
            for (int q = 0; q < DW_KMAX - 2; ++q)
                if (q < km1 - 1) win[q] = win[q + 1];
            win[km1 - 1] = cur;
        }
        // streaming: the CTA that owns the last rows writes the new context (single CTA per session when T <= DW_TB;
        // for longer calls the old context is only read by the first CTA and written by the last one, after a
        // kernel-wide ordering that a second launch provides: the host runs streaming calls with T > DW_TB as one launch
        // per DW_TB rows)
        if (cache && r0 + nr == T) {
            for (int q = 0; q < km1; ++q) cache[(long long)q * C + c] = win[q];
        }
    }
}

__global__ void subsample_mask_kernel(const int32_t* __restrict__ ilens, int T, int T2, uint8_t* __restrict__ mask2,
                                      int32_t* __restrict__ ilens2) {
    // subsampling.py:65: m'[j] = m[4j + 6]; ilens' = m'.sum  (subsampling.py:100)
    const int b = blockIdx.x;
    const int len = ilens[b];
    int cnt = 0;
    for (int j = threadIdx.x; j < T2; j += blockDim.x) {
        uint8_t v = (4 * j + 6) < len ? 1 : 0;
        mask2[(long long)b * T2 + j] = v;
    }
    if (threadIdx.x == 0) {
        for (int j = 0; j < T2; ++j) cnt += (4 * j + 6) < len ? 1 : 0;
        ilens2[b] = cnt;
    }
}

__global__ void stride2_mask_kernel(const uint8_t* __restrict__ mask, int T, int To, uint8_t* __restrict__ out) {
    const int b = blockIdx.x;
    for (int j = threadIdx.x; j < To; j += blockDim.x) out[(long long)b * To + j] = mask[(long long)b * T + 2 * j];
}

__global__ void f32_to_bf16_kernel(const float* __restrict__ s, bf16* __restrict__ d, long long n) {
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) d[i] = __float2bfloat16_rn(s[i]);
}
__global__ void f32_to_act16_kernel(const float* __restrict__ s, act16* __restrict__ d, long long n) {
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) d[i] = from_f<act16>(s[i]);
}
__global__ void bf16_to_f32_kernel(const bf16* __restrict__ s, float* __restrict__ d, long long n) {
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) d[i] = __bfloat162float(s[i]);
}
__global__ void act16_to_f32_kernel(const act16* __restrict__ s, float* __restrict__ d, long long n) {
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) d[i] = __half2float(s[i]);
}

template <typename TW>
__global__ void repack_conv2_kernel(const float* __restrict__ w, int C, TW* __restrict__ out) {
    // out[co][(kh*3+kw)*C + ci] = w[co][ci][kh][kw]
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    long long total = (long long)C * C * 9;
    if (i >= total) return;
    int ci = i % C;
    int q = (i / C) % 9;
    int co = i / (9LL * C);
    out[i] = weight_cast<TW>(w[((long long)co * C + ci) * 9 + q]);
}
template <typename TW>
__global__ void repack_sublinear_kernel(const float* __restrict__ w, int C, int F2, long long N, TW* __restrict__ out) {
    // out[n][f*C + c] = w[n][c*F2 + f]      (subsampling.py:63 flattens (c, f))
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    long long K = (long long)C * F2;
    if (i >= N * K) return;
    long long n = i / K;
    int k = i % K;
    int f = k / C, c = k % C;
    out[i] = weight_cast<TW>(w[n * K + (long long)c * F2 + f]);
}
template <typename TW>
__global__ void repack_adapter_conv_kernel(const float* __restrict__ w, int C2, int C, int k, TW* __restrict__ out) {
    // out[co][tau*C + ci] = w[co][ci][tau]
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    long long total = (long long)C2 * C * k;
    if (i >= total) return;
    int ci = i % C;
    int tau = (i / C) % k;
    long long co = i / ((long long)C * k);
    out[i] = weight_cast<TW>(w[(co * C + ci) * k + tau]);
}
template <typename TW>
__global__ void convert_weight_kernel(const float* __restrict__ w, long long n, TW* __restrict__ out) {
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = weight_cast<TW>(w[i]);
}

template <typename TA>
__global__ void ring_export_kernel(const TA* __restrict__ ring, int H, int cap, long long first, int n,
                                   float* __restrict__ out) {
    // out[h][j][d] = ring[h][(first + j) % cap][d]
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (long long)H * n * 64) return;
    int d = i & 63;
    int j = (i >> 6) % n;
    int h = i / (64LL * n);
    // 16-bit rings carry the chunk swizzle of the fp16 attention kernel: chunk c of frame f at c ^ (f & 7)
    const int dd = sizeof(TA) == 2 ? ((((d >> 3) ^ (int)((first + j) & 7)) << 3) + (d & 7)) : d;
    out[i] = to_f(ring[((long long)h * cap + (first + j) % cap) * 64 + dd]);
}
template <typename TA>
__global__ void ring_import_kernel(TA* __restrict__ ring, int H, int cap, long long first, int n,
                                   const float* __restrict__ in) {
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (long long)H * n * 64) return;
    int d = i & 63;
    int j = (i >> 6) % n;
    int h = i / (64LL * n);
    const int dd = sizeof(TA) == 2 ? ((((d >> 3) ^ (int)((first + j) & 7)) << 3) + (d & 7)) : d;
    ring[((long long)h * cap + (first + j) % cap) * 64 + dd] = from_f<TA>(in[i]);
}

inline int blocks_for(long long n, int t) { return (int)((n + t - 1) / t); }

}  // namespace

template <typename TA>
int cmvn_conv1(const float* feats, int B, int T, int F, const float* mean, const float* istd, const float* w1,
               const float* b1, int C, TA* c1, cudaStream_t st) {
    const int T1 = (T - 1) / 2, F1 = (F - 1) / 2, T2 = (T1 - 1) / 2, F2 = (F1 - 1) / 2;
    if (B <= 0 || T2 <= 0) return 0;
    FO_CHECK(C % 4 == 0, "cmvn_conv1: channel count must be a multiple of 4");
    dim3 grid(2 * T2 + 1, B);                          // conv1 rows that feed a conv2 output row
    const int threads = C / 4 >= 256 ? 256 : ((C / 4 + 31) / 32) * 32;
    FO_CUDA(launch_pdl(cmvn_conv1_kernel<TA, 4>, grid, dim3(threads), 3 * F * sizeof(float), st, feats, T, F, mean, istd, w1, b1, C,
                       T2, F1, F2 + 1, (long long)B * T2 * (F2 + 1), c1));
    FO_LAUNCHED();
    FO_CUDA(cudaGetLastError());
    return 0;
}
void conv2_gather(int B, int T2, int F2, int C, AGather* ga, RowMap* rm) {
    const int F2P = F2 + 1;
    ga->seg_len = C; ga->n_seg = 9; ga->rows = (long long)B * T2 * F2P; ga->planes = 6;
    for (int kh = 0; kh < 3; ++kh)
        for (int kw = 0; kw < 3; ++kw) {
            ga->plane[kh * 3 + kw] = kh * 2 + (kw & 1);
            ga->rowoff[kh * 3 + kw] = kw >> 1;
        }
    rm->p0 = F2P; rm->p1 = T2 * F2P; rm->v0 = F2; rm->v1 = T2; rm->q0 = F2; rm->q1 = T2 * F2;
}
void adapter_gather(int B, int T, int D, int k, AGather* ga, RowMap* rm) {
    const int RP = (k - 1 + T + 1) / 2, t_out = (T - 1) / 2 + 1;
    ga->seg_len = D; ga->n_seg = k; ga->rows = (long long)B * RP; ga->planes = 2;
    for (int i = 0; i < AGather::MAX_SEG; ++i) { ga->plane[i] = i & 1; ga->rowoff[i] = i >> 1; }
    rm->p0 = RP; rm->p1 = RP; rm->v0 = t_out; rm->v1 = 1; rm->q0 = 0; rm->q1 = t_out;
}

template int cmvn_conv1<float>(const float*, int, int, int, const float*, const float*, const float*, const float*, int, float*, cudaStream_t);
template int cmvn_conv1<bf16>(const float*, int, int, int, const float*, const float*, const float*, const float*, int, bf16*, cudaStream_t);
template int cmvn_conv1<__half>(const float*, int, int, int, const float*, const float*, const float*, const float*, int, __half*, cudaStream_t);

template <typename TA>
int layer_norm(const float* x, int M, int D, const float* gamma, const float* beta, float eps, int act,
               float out_scale, TA* y_act, float* y_f32, cudaStream_t st) {
    if (M <= 0) return 0;
    FO_CHECK(D % 128 == 0 && D <= 4096, "layer_norm: D (%d) must be a multiple of 128 and <= 4096", D);
    const int rows_per_cta = 4;
    dim3 grid(cdiv(M, rows_per_cta));
    if (D <= 1024)
        FO_CUDA(launch_pdl(layer_norm_kernel<TA, 8>, grid, dim3(128), 0, st, x, M, D, gamma, beta, eps, act, out_scale, y_act, y_f32));
    else if (D <= 2048)      // the adapter's norm over 2C: half the registers of the general variant
        FO_CUDA(launch_pdl(layer_norm_kernel<TA, 16>, grid, dim3(128), 0, st, x, M, D, gamma, beta, eps, act, out_scale, y_act, y_f32));
    else
        FO_CUDA(launch_pdl(layer_norm_kernel<TA, 32>, grid, dim3(128), 0, st, x, M, D, gamma, beta, eps, act, out_scale, y_act, y_f32));
    FO_LAUNCHED();
    FO_CUDA(cudaGetLastError());
    return 0;
}
template int layer_norm<float>(const float*, int, int, const float*, const float*, float, int, float, float*, float*, cudaStream_t);
template int layer_norm<bf16>(const float*, int, int, const float*, const float*, float, int, float, bf16*, float*, cudaStream_t);
template int layer_norm<__half>(const float*, int, int, const float*, const float*, float, int, float, __half*, float*, cudaStream_t);

template <typename TA>
int layer_norm_reduce(float* x, const float* partial, int nsplit, const float* bias, int M, int D, const float* gamma,
                      const float* beta, float eps, TA* y_act, float* y_f32, cudaStream_t st) {
    if (M <= 0) return 0;
    FO_CHECK(D % 256 == 0 && D <= 1024, "layer_norm_reduce: D=%d not supported", D);
    const dim3 grid(cdiv(M, 2));
    if (nsplit == 2)
        FO_CUDA(launch_pdl(layer_norm_reduce_kernel<TA, 2>, grid, dim3(128), 0, st, x, partial, nsplit, bias, M, D, gamma, beta, eps, y_act, y_f32));
    else if (nsplit == 4)
        FO_CUDA(launch_pdl(layer_norm_reduce_kernel<TA, 4>, grid, dim3(128), 0, st, x, partial, nsplit, bias, M, D, gamma, beta, eps, y_act, y_f32));
    else
        FO_CUDA(launch_pdl(layer_norm_reduce_kernel<TA, 0>, grid, dim3(128), 0, st, x, partial, nsplit, bias, M, D, gamma, beta, eps, y_act, y_f32));
    FO_LAUNCHED();
    FO_CUDA(cudaGetLastError());
    return 0;
}
template int layer_norm_reduce<float>(float*, const float*, int, const float*, int, int, const float*, const float*, float, float*, float*, cudaStream_t);
template int layer_norm_reduce<__half>(float*, const float*, int, const float*, int, int, const float*, const float*, float, __half*, float*, cudaStream_t);

int scale_rows(const float* x, float* y, long long n, float s, cudaStream_t st) {
    if (n <= 0) return 0;
    scale_rows_kernel<<<blocks_for(n, 256), 256, 0, st>>>(x, y, n, s);
    FO_LAUNCHED();
    FO_CUDA(cudaGetLastError());
    return 0;
}

// rows of B sequences (B, T, C) copied into zero-padded sequences (B, lead + T + trail, C): the A operand of a Conv1d with
// symmetric padding run as an implicit GEMM (MultiLayeredConv1d, attention.py:171-184); 16-byte chunks
template <typename TA>
__global__ void pad_rows_kernel(const TA* __restrict__ in, int T, int C, int lead, int trail, TA* __restrict__ out) {
    FO_PDL_TRIGGER();
    FO_PDL_WAIT();
    const int b = blockIdx.y, r = blockIdx.x;             // r in [0, lead + T + trail)
    const int R = lead + T + trail;
    constexpr int EPV = 16 / sizeof(TA);
    const uint4* src = (r >= lead && r < lead + T) ? reinterpret_cast<const uint4*>(in + ((long long)b * T + (r - lead)) * C) : nullptr;
    uint4* dst = reinterpret_cast<uint4*>(out + ((long long)b * R + r) * C);
    for (int i = threadIdx.x; i < C / EPV; i += blockDim.x) dst[i] = src ? src[i] : make_uint4(0, 0, 0, 0);
}
template <typename TA>
int pad_rows(const TA* in, int B, int T, int C, int lead, int trail, TA* out, cudaStream_t st) {
    if (B <= 0 || T <= 0) return 0;
    FO_CHECK(C % (16 / (int)sizeof(TA)) == 0, "pad_rows: C must be a multiple of %d", 16 / (int)sizeof(TA));
    FO_CUDA(launch_pdl(pad_rows_kernel<TA>, dim3(lead + T + trail, B), dim3(128), 0, st, in, T, C, lead, trail, out));
    FO_LAUNCHED();
    FO_CUDA(cudaGetLastError());
    return 0;
}
template int pad_rows<float>(const float*, int, int, int, int, int, float*, cudaStream_t);
template int pad_rows<__half>(const __half*, int, int, int, int, int, __half*, cudaStream_t);

// grid (gap, n): rows at[i] .. at[i] + gap - 1 of buf set to zero
template <typename TA>
__global__ void zero_row_runs_kernel(TA* __restrict__ buf, const int32_t* __restrict__ at, int C) {
    FO_PDL_TRIGGER();
    FO_PDL_WAIT();
    TA* d = buf + ((long long)at[blockIdx.y] + blockIdx.x) * C;
    for (int c = threadIdx.x; c < C; c += blockDim.x) d[c] = from_f<TA>(0.f);
}
template <typename TA>
int zero_row_runs(TA* buf, const int32_t* at, int n, int gap, int C, cudaStream_t st) {
    if (n <= 0 || gap <= 0) return 0;
    FO_CUDA(launch_pdl(zero_row_runs_kernel<TA>, dim3(gap, n), dim3(128), 0, st, buf, at, C));
    FO_LAUNCHED();
    FO_CUDA(cudaGetLastError());
    return 0;
}
template int zero_row_runs<float>(float*, const int32_t*, int, int, int, cudaStream_t);
template int zero_row_runs<__half>(__half*, const int32_t*, int, int, int, cudaStream_t);

// grid (rows_max, n): row r < lens[b] of utterance b, src row srow[b] + r -> dst row drow[b] + r
__global__ void copy_utt_rows_kernel(const float* __restrict__ src, const int32_t* __restrict__ srow, float* __restrict__ dst,
                                     const int32_t* __restrict__ drow, const int32_t* __restrict__ lens, int C) {
    FO_PDL_TRIGGER();
    FO_PDL_WAIT();
    const int b = blockIdx.y, r = blockIdx.x;
    if (r >= lens[b]) return;
    const float* s = src + ((long long)srow[b] + r) * C;
    float* d = dst + ((long long)drow[b] + r) * C;
    for (int c = threadIdx.x; c < C; c += blockDim.x) d[c] = s[c];
}
int copy_utt_rows(const float* src, const int32_t* srow, float* dst, const int32_t* drow, const int32_t* lens, int n, int rows_max,
                  int C, cudaStream_t st) {
    if (n <= 0 || rows_max <= 0) return 0;
    FO_CUDA(launch_pdl(copy_utt_rows_kernel, dim3(rows_max, n), dim3(C >= 256 ? 256 : 128), 0, st, src, srow, dst, drow, lens, C));
    FO_LAUNCHED();
    FO_CUDA(cudaGetLastError());
    return 0;
}

template <typename TA>
int conv_stage(const float* in, const uint8_t* mask, int B, int T, int C, int km1, int stride, const float* scale,
               const float* shift, const int32_t* ids, float* slot_cache, int32_t* slot_valid, const float* cache_in,
               float* cache_out, TA* xin, cudaStream_t st, const SessionRows& sr) {
    if (B <= 0) return 0;
    FO_CHECK(stride == 1 || stride == 2, "conv_stage: stride must be 1 or 2");
    dim3 grid(B, km1 + T);
    FO_CUDA(launch_pdl(conv_stage_kernel<TA>, grid, dim3(256), 0, st, in, mask, T, C, km1, stride, scale, shift, ids, slot_cache,
                       (const int32_t*)slot_valid, cache_in, cache_out, xin, sr));
    FO_LAUNCHED();
    FO_CUDA(cudaGetLastError());
    return 0;
}
template int conv_stage<float>(const float*, const uint8_t*, int, int, int, int, int, const float*, const float*, const int32_t*, float*, int32_t*, const float*, float*, float*, cudaStream_t, const SessionRows&);
template int conv_stage<__half>(const float*, const uint8_t*, int, int, int, int, int, const float*, const float*, const int32_t*, float*, int32_t*, const float*, float*, __half*, cudaStream_t, const SessionRows&);

// grid (n, kmax): block j < cnt[b] of session b
__global__ void pack_session_blocks_kernel(const char* __restrict__ src, char* __restrict__ dst, long long bytes, int kmax,
                                           const int32_t* __restrict__ cnt, const int32_t* __restrict__ off) {
    FO_PDL_TRIGGER();
    FO_PDL_WAIT();
    const int b = blockIdx.x, j = blockIdx.y;
    if (j >= cnt[b]) return;
    const char* s = src + ((long long)b * kmax + j) * bytes;
    char* d = dst + ((long long)off[b] + j) * bytes;
    if (((bytes | (long long)(size_t)src | (long long)(size_t)dst) & 15) == 0) {
        for (long long i = threadIdx.x * 16LL; i < bytes; i += blockDim.x * 16LL)
            *reinterpret_cast<uint4*>(d + i) = *reinterpret_cast<const uint4*>(s + i);
    } else {
        for (long long i = threadIdx.x * 4LL; i < bytes; i += blockDim.x * 4LL)
            *reinterpret_cast<float*>(d + i) = *reinterpret_cast<const float*>(s + i);
    }
}
// grid (kmax * t_out, n): row m of chunk j < cnt[b] of session b <- row j * t + 2 m of the session's T-row grid
__global__ void pick_chunk_rows_kernel(const float* __restrict__ src, int T, int C, int t, int t_out, const int32_t* __restrict__ cnt,
                                       const int32_t* __restrict__ off, float* __restrict__ dst) {
    FO_PDL_TRIGGER();
    FO_PDL_WAIT();
    const int b = blockIdx.y, j = blockIdx.x / t_out, m = blockIdx.x % t_out;
    if (j >= cnt[b]) return;
    const float* s = src + ((long long)b * T + (long long)j * t + 2 * m) * C;
    float* d = dst + ((long long)(off[b] + j) * t_out + m) * C;
    for (int c = threadIdx.x; c < C; c += blockDim.x) d[c] = s[c];
}
int pick_chunk_rows(const float* src, int n, int kmax, int t, int t_out, int C, const int32_t* cnt, const int32_t* off, float* dst,
                    cudaStream_t st) {
    if (n <= 0) return 0;
    FO_CUDA(launch_pdl(pick_chunk_rows_kernel, dim3(kmax * t_out, n), dim3(256), 0, st, src, kmax * t, C, t, t_out, cnt, off, dst));
    FO_LAUNCHED();
    FO_CUDA(cudaGetLastError());
    return 0;
}

int pack_session_blocks(const float* src, float* dst, long long bytes, int n, int kmax, const int32_t* cnt, const int32_t* off,
                        cudaStream_t st) {
    if (n <= 0) return 0;
    FO_CHECK(bytes % 4 == 0, "pack_session_blocks: blocks of fp32 elements");
    FO_CUDA(launch_pdl(pack_session_blocks_kernel, dim3(n, kmax), dim3(256), 0, st, (const char*)src, (char*)dst, bytes, kmax, cnt, off));
    FO_LAUNCHED();
    FO_CUDA(cudaGetLastError());
    return 0;
}

// stride-1 causal conv (kernel k) over xin[b * (k-1+T) + r][C]: tap tau of output row t reads row t + tau
void conv1d_gather(int B, int T, int C, int k, AGather* ga, RowMap* rm) {
    const int R1 = k - 1 + T;
    ga->seg_len = C; ga->n_seg = k; ga->rows = (long long)B * R1; ga->planes = 1;
    for (int i = 0; i < AGather::MAX_SEG; ++i) { ga->plane[i] = 0; ga->rowoff[i] = i; }
    rm->p0 = R1; rm->p1 = R1; rm->v0 = T; rm->v1 = 1; rm->q0 = 0; rm->q1 = T;
}

template <typename TA>
int depthwise_conv(const TA* x, int B, int T, int C, int k, const float* w, const float* bias, const int32_t* ids,
                   float* slot_cache, long long slot_stride, TA* y, cudaStream_t st, const int32_t* cnt, const int32_t* off, int t) {
    if (B <= 0 || T <= 0) return 0;
    FO_CHECK(k >= 2 && k <= DW_KMAX, "depthwise_conv: kernel size %d outside 2..%d", k, DW_KMAX);
    FO_CHECK(!cnt || (off && t > 0), "depthwise_conv: per-session counts need their row offsets");
    if (ids && (T > DW_TB || cnt)) {
        // streaming, several chunks per session (fo_encode_stream_chunks[_v]): the first rows read the carried context and the
        // last ones replace it, so the row blocks run in order, one launch each (up to the largest session's rows)
        for (int r0 = 0; r0 < T; r0 += DW_TB) {
            FO_CUDA(launch_pdl(depthwise_conv_kernel<TA>, dim3(1, B), dim3(256), 0, st, x, T, C, k, w, bias, ids, slot_cache, slot_stride, y, r0,
                               cnt, off, t));
            FO_LAUNCHED();
        }
        return 0;
    }
    // one launch: per-utterance rows with zero left context (offline; cnt / off: utterances packed end to end, T the longest),
    // or a streaming call whose sessions' rows fit one row block
    dim3 grid(cdiv(T, DW_TB), B);
    FO_CUDA(launch_pdl(depthwise_conv_kernel<TA>, grid, dim3(256), 0, st, x, T, C, k, w, bias, ids, slot_cache, slot_stride, y, 0,
                       cnt, off, t));
    FO_LAUNCHED();
    return 0;
}
template int depthwise_conv<float>(const float*, int, int, int, int, const float*, const float*, const int32_t*, float*, long long, float*, cudaStream_t, const int32_t*, const int32_t*, int);
template int depthwise_conv<__half>(const __half*, int, int, int, int, const float*, const float*, const int32_t*, float*, long long, __half*, cudaStream_t, const int32_t*, const int32_t*, int);

// LLM hand-off bookkeeping (models/audioLLM.py:404-411): per session the attention-mask row over its block of the inputs_embeds
// buffer, [prefix_mask | 1 x t_out | 0 ...] when the block opens an IPU (status 'ipu_sl': the chat prefix is part of the input) and
// [0 x P | 1 x t_out | 0 ...] otherwise, plus the row where the session's input starts (0 / P).  One CTA writes block b's row.
__device__ __forceinline__ void handoff_mask_row(bool on, const uint8_t* __restrict__ prefix_mask, int P, int t_out, int rows,
                                                 long long b, uint8_t* __restrict__ attn_mask, int32_t* __restrict__ row_start) {
    for (int r = threadIdx.x; r < rows; r += blockDim.x) {
        uint8_t v;
        if (r < P) v = on ? (prefix_mask ? (prefix_mask[r] != 0) : 1) : 0;
        else v = r < P + t_out ? 1 : 0;
        attn_mask[b * rows + r] = v;
    }
    if (threadIdx.x == 0 && row_start) row_start[b] = on ? 0 : P;
}
__global__ void handoff_mask_kernel(const uint8_t* __restrict__ onset, const uint8_t* __restrict__ prefix_mask, int P, int t_out,
                                    int rows, uint8_t* __restrict__ attn_mask, int32_t* __restrict__ row_start) {
    handoff_mask_row(onset[blockIdx.x] != 0, prefix_mask, P, t_out, rows, blockIdx.x, attn_mask, row_start);
}

// The hand-off of a pass of the recording entries: CTA b takes pass block b's t_out fp32 adapter rows (y, contiguous per block) to
// the caller's block tab[b].x -- rows [P, P + t_out) of embeds, as fp16 with the clamp and saturation count of the projection
// epilogue's hand-off write -- and writes that block's mask row and row_start from its onset flag tab[b].y.
__global__ void __launch_bounds__(256) handoff_rows_kernel(const float* __restrict__ y, const int2* __restrict__ tab, int t_out, int E,
                                                           __half* __restrict__ embeds, int rows, int P,
                                                           const uint8_t* __restrict__ prefix_mask, uint8_t* __restrict__ attn_mask,
                                                           int32_t* __restrict__ row_start, unsigned long long* sat) {
    const int2 e = tab[blockIdx.x];
    const long long n = (long long)t_out * E;
    const float* src = y + blockIdx.x * n;
    __half* dst = embeds + ((long long)e.x * rows + P) * E;
    if (n % 8 == 0 && (reinterpret_cast<uintptr_t>(dst) & 15) == 0) {
        // 8 values per step: two 16-byte loads, one 16-byte store (src is 32-byte aligned: blocks of t_out * E floats, E % 8 == 0)
        const float4* s4 = reinterpret_cast<const float4*>(src);
        uint4* d4 = reinterpret_cast<uint4*>(dst);
        for (long long i = threadIdx.x; i < n / 8; i += blockDim.x) {
            const float4 a = s4[2 * i], b = s4[2 * i + 1];
            count_sat4(sat, a.x, a.y, a.z, a.w);
            count_sat4(sat, b.x, b.y, b.z, b.w);
            d4[i] = make_uint4(pack2<__half>(a.x, a.y), pack2<__half>(a.z, a.w), pack2<__half>(b.x, b.y), pack2<__half>(b.z, b.w));
        }
    } else {
        for (long long i = threadIdx.x; i < n; i += blockDim.x) {
            const float v = src[i];
            count_sat4(sat, v, 0.f, 0.f, 0.f);
            dst[i] = from_f<__half>(v);
        }
    }
    if (attn_mask) handoff_mask_row(e.y != 0, prefix_mask, P, t_out, rows, e.x, attn_mask, row_start);
}
int handoff_mask(const uint8_t* onset, const uint8_t* prefix_mask, int n, int P, int t_out, int rows, uint8_t* attn_mask,
                 int32_t* row_start, cudaStream_t st) {
    if (n <= 0) return 0;
    handoff_mask_kernel<<<n, 128, 0, st>>>(onset, prefix_mask, P, t_out, rows, attn_mask, row_start);
    FO_LAUNCHED();
    FO_CUDA(cudaGetLastError());
    return 0;
}
int handoff_rows(const float* y, const int2* tab, int nblk, int t_out, int E, void* embeds_f16, int rows, int P,
                 const uint8_t* prefix_mask, uint8_t* attn_mask, int32_t* row_start, unsigned long long* sat, cudaStream_t st) {
    if (nblk <= 0) return 0;
    handoff_rows_kernel<<<nblk, 256, 0, st>>>(y, tab, t_out, E, reinterpret_cast<__half*>(embeds_f16), rows, P, prefix_mask, attn_mask,
                                              row_start, sat);
    FO_LAUNCHED();
    FO_CUDA(cudaGetLastError());
    return 0;
}

int subsample_mask(const int32_t* ilens, int B, int T, int T2, uint8_t* mask2, int32_t* ilens2, cudaStream_t st) {
    if (B <= 0) return 0;
    subsample_mask_kernel<<<B, 128, 0, st>>>(ilens, T, T2, mask2, ilens2);
    FO_LAUNCHED();
    FO_CUDA(cudaGetLastError());
    return 0;
}
int stride2_mask(const uint8_t* mask, int B, int T, int To, uint8_t* out, cudaStream_t st) {
    if (B <= 0) return 0;
    stride2_mask_kernel<<<B, 128, 0, st>>>(mask, T, To, out);
    FO_LAUNCHED();
    FO_CUDA(cudaGetLastError());
    return 0;
}

int f32_to_bf16(const float* src, bf16* dst, long long n, cudaStream_t st) {
    if (n <= 0) return 0;
    f32_to_bf16_kernel<<<blocks_for(n, 256), 256, 0, st>>>(src, dst, n);
    FO_LAUNCHED();
    FO_CUDA(cudaGetLastError());
    return 0;
}
int f32_to_act16(const float* src, act16* dst, long long n, cudaStream_t st) {
    if (n <= 0) return 0;
    f32_to_act16_kernel<<<blocks_for(n, 256), 256, 0, st>>>(src, dst, n);
    FO_LAUNCHED();
    FO_CUDA(cudaGetLastError());
    return 0;
}
int f32_to_weight16(const float* src, act16* dst, long long n, cudaStream_t st) { return convert_weight<act16>(src, n, dst, st); }
int bf16_to_f32(const bf16* src, float* dst, long long n, cudaStream_t st) {
    if (n <= 0) return 0;
    bf16_to_f32_kernel<<<blocks_for(n, 256), 256, 0, st>>>(src, dst, n);
    FO_LAUNCHED();
    FO_CUDA(cudaGetLastError());
    return 0;
}
int act16_to_f32(const act16* src, float* dst, long long n, cudaStream_t st) {
    if (n <= 0) return 0;
    act16_to_f32_kernel<<<blocks_for(n, 256), 256, 0, st>>>(src, dst, n);
    FO_LAUNCHED();
    FO_CUDA(cudaGetLastError());
    return 0;
}

template <typename TW>
int repack_conv2(const float* w, int C, TW* out, cudaStream_t st) {
    long long n = (long long)C * C * 9;
    repack_conv2_kernel<TW><<<blocks_for(n, 256), 256, 0, st>>>(w, C, out);
    FO_CUDA(cudaGetLastError());
    return 0;
}
template <typename TW>
int repack_sublinear(const float* w, int C, int F2, TW* out, cudaStream_t st) {
    long long n = (long long)C * C * F2;
    repack_sublinear_kernel<TW><<<blocks_for(n, 256), 256, 0, st>>>(w, C, F2, C, out);
    FO_CUDA(cudaGetLastError());
    return 0;
}
template <typename TW>
int repack_adapter_conv(const float* w, int C2, int C, int k, TW* out, cudaStream_t st) {
    long long n = (long long)C2 * C * k;
    repack_adapter_conv_kernel<TW><<<blocks_for(n, 256), 256, 0, st>>>(w, C2, C, k, out);
    FO_CUDA(cudaGetLastError());
    return 0;
}
template <typename TW>
int convert_weight(const float* w, long long n, TW* out, cudaStream_t st) {
    if (n <= 0) return 0;
    convert_weight_kernel<TW><<<blocks_for(n, 256), 256, 0, st>>>(w, n, out);
    FO_CUDA(cudaGetLastError());
    return 0;
}
template int repack_conv2<float>(const float*, int, float*, cudaStream_t);
template int repack_conv2<bf16>(const float*, int, bf16*, cudaStream_t);
template int repack_conv2<__half>(const float*, int, __half*, cudaStream_t);
template int repack_sublinear<__half>(const float*, int, int, __half*, cudaStream_t);
template int repack_adapter_conv<__half>(const float*, int, int, int, __half*, cudaStream_t);
template int convert_weight<__half>(const float*, long long, __half*, cudaStream_t);
template int repack_sublinear<float>(const float*, int, int, float*, cudaStream_t);
template int repack_sublinear<bf16>(const float*, int, int, bf16*, cudaStream_t);
template int repack_adapter_conv<float>(const float*, int, int, int, float*, cudaStream_t);
template int repack_adapter_conv<bf16>(const float*, int, int, int, bf16*, cudaStream_t);
template int convert_weight<float>(const float*, long long, float*, cudaStream_t);
template int convert_weight<bf16>(const float*, long long, bf16*, cudaStream_t);

template <typename TA>
int ring_export(const TA* ring_kv, int H, int ring_cap, long long first_frame, int n, float* out, cudaStream_t st) {
    if (n <= 0) return 0;
    long long tot = (long long)H * n * 64;
    ring_export_kernel<TA><<<blocks_for(tot, 256), 256, 0, st>>>(ring_kv, H, ring_cap, first_frame, n, out);
    FO_CUDA(cudaGetLastError());
    return 0;
}
template <typename TA>
int ring_import(TA* ring_kv, int H, int ring_cap, long long first_frame, int n, const float* in, cudaStream_t st) {
    if (n <= 0) return 0;
    long long tot = (long long)H * n * 64;
    ring_import_kernel<TA><<<blocks_for(tot, 256), 256, 0, st>>>(ring_kv, H, ring_cap, first_frame, n, in);
    FO_CUDA(cudaGetLastError());
    return 0;
}
template int ring_export<float>(const float*, int, int, long long, int, float*, cudaStream_t);
template int ring_export<bf16>(const bf16*, int, int, long long, int, float*, cudaStream_t);
template int ring_export<__half>(const __half*, int, int, long long, int, float*, cudaStream_t);
template int ring_import<float>(float*, int, int, long long, int, const float*, cudaStream_t);
template int ring_import<bf16>(bf16*, int, int, long long, int, const float*, cudaStream_t);
template int ring_import<__half>(__half*, int, int, long long, int, const float*, cudaStream_t);

FO_TR_BIND_DEF(trace_bind_elementwise)

}  // namespace fo
