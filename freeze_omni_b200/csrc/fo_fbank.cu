// Kaldi-compatible log-mel filterbank frontend (reference call sites bin/inference.py:77-78 and
// models/AudioFeatureGating.py:65-69 -> torchaudio.compliance.kaldi.fbank, kaldi.py:514-645) with the
// streaming state of audioEncoderProcessor (bin/inference.py:57-69): sample carry + feature-context ring.
//
// One warp per frame: coalesced sample load -> frame mean (shuffle reduction) -> pre-emphasis and Povey
// window in fp32 with the same operation order as torchaudio -> real FFT of size P computed as a P/2-point
// complex FFT on packed samples, butterflies in fp64 in shared memory (the fp32 radix-2 variant measured
// 1.5e-4 relative from exact arithmetic on assets/question.wav; fp64 makes the result exact to fp32
// rounding, and B200 has full-rate FP64 pipes) -> power spectrum -> sparse triangular mel sums ->
// log(max(., FLT_EPSILON)).  Bytes moved per frame: frame_shift samples in, n_mel floats out.
#include <algorithm>
#include <mutex>

#include "fo_common.cuh"

namespace fo {

namespace {

constexpr int FB_WARPS = 4;
constexpr int MAX_FFT = 1024;
__device__ double2 c_twiddle[MAX_FFT / 2];       // exp(-2 pi i k / P), k < P/2 (L1-resident table)
static int g_twiddle_fft = 0;

struct SampleSrc {
    const void* base;       // fp32 or int16 samples
    int is_i16;
    float scale;
    long long row_stride;   // samples between consecutive signals
    const int32_t* row_ids; // optional indirection: signal b reads row row_ids[b]
};

__device__ __forceinline__ float fetch(const SampleSrc& s, long long row, long long i) {
    const long long o = row * s.row_stride + i;
    return s.is_i16 ? (float)reinterpret_cast<const int16_t*>(s.base)[o] * s.scale
                    : reinterpret_cast<const float*>(s.base)[o] * s.scale;
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// Which signal and frame a warp takes, where its samples start and where its mel row goes.
//  Uniform (VL = false): B signals of frames_per_signal frames each, signal b at sample row src.row_ids[b] (or b) of
//    src.row_stride samples; out row = out + (out_ids ? out_ids[b] : b) * out_row_stride + (out_frame0 + f) * n_mel, and out2
//    (optional, dense (B, out2_frames, n_mel)) receives the same frame at row out2_frame0 + f.
//  Varlen (VL = true, fbank_offline_packed): frame fr of the call belongs to the utterance b with frame_off[b] <= fr <
//    frame_off[b + 1] (binary search of the device table), local frame f = fr - frame_off[b]; its samples start at
//    sample_off[b] + f * frame_shift of src.base; out row = out + (out_row[b] + f) * n_mel, out2 (optional) row frame_off[b] + f.
template <bool VL>
__device__ __forceinline__ void fbank_frame(const FbankVarlen& vl, const SampleSrc& src, int frames_per_signal, int frame_shift,
                                            long long fr, int& b, int& f, long long& srow, long long& s0) {
    if constexpr (VL) {
        int lo = 0, hi = vl.n;                             // frame_off[lo] <= fr < frame_off[hi]
        while (hi - lo > 1) {
            const int mid = (lo + hi) >> 1;
            if (vl.frame_off[mid] <= fr) lo = mid;
            else hi = mid;
        }
        b = lo;
        f = (int)(fr - vl.frame_off[b]);
        srow = 0;
        s0 = vl.sample_off[b] + (long long)f * frame_shift;
    } else {
        b = (int)(fr / frames_per_signal);
        f = (int)(fr % frames_per_signal);
        srow = src.row_ids ? src.row_ids[b] : b;
        s0 = (long long)f * frame_shift;
    }
}

template <bool VL>
__global__ void __launch_bounds__(FB_WARPS * 32)
fbank_kernel(FbankParams p, SampleSrc src, int B, int frames_per_signal, float* __restrict__ out,
             const int32_t* __restrict__ out_ids, long long out_row_stride, int out_frame0, float* __restrict__ out2,
             int out2_frames, int out2_frame0, FbankVarlen vl) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int P = p.fft_size, M = P >> 1;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    // per-warp scratch: M double2 (FFT), P floats (samples, then power spectrum)
    double2* z = reinterpret_cast<double2*>(smem_raw) + (size_t)warp * M;
    float* xs = reinterpret_cast<float*>(smem_raw + (size_t)FB_WARPS * M * sizeof(double2)) + (size_t)warp * (P + 32);
    int log2m = 0;
    while ((1 << log2m) < M) ++log2m;

    const long long total = VL ? vl.frames : (long long)B * frames_per_signal;
    for (long long fr = (long long)blockIdx.x * FB_WARPS + warp; fr < total; fr += (long long)gridDim.x * FB_WARPS) {
        int b, f;
        long long srow, s0;
        fbank_frame<VL>(vl, src, frames_per_signal, p.frame_shift, fr, b, f, srow, s0);
        // 1. samples + mean (kaldi.py:183-186)
        float part = 0.f;
        for (int i = lane; i < p.frame_len; i += 32) {
            const float v = fetch(src, srow, s0 + i);
            xs[i] = v;
            part += v;
        }
        const float mean = warp_sum(part) / (float)p.frame_len;
        __syncwarp();
        // 2. pre-emphasis with replicate pad, window (kaldi.py:193-205); pack pairs as complex
        for (int n = lane; n < M; n += 32) {
            double2 c;
            float y[2];
#pragma unroll
            for (int q = 0; q < 2; ++q) {
                const int i = 2 * n + q;
                if (i < p.frame_len) {
                    const float cur = __fsub_rn(xs[i], mean);
                    const float prev = __fsub_rn(xs[i > 0 ? i - 1 : 0], mean);
                    y[q] = __fmul_rn(__fsub_rn(cur, __fmul_rn(0.97f, prev)), p.window[i]);
                } else {
                    y[q] = 0.f;
                }
            }
            c.x = (double)y[0];
            c.y = (double)y[1];
            z[n] = c;
        }
        __syncwarp();
        // 3. M-point complex FFT, decimation in frequency, in place; result index bit-reversed
        for (int len = M; len >= 2; len >>= 1) {
            const int half = len >> 1;
            const int tw_step = P / len;                  // w_len^j = twiddle[j * P / len]
            for (int k = lane; k < (M >> 1); k += 32) {
                const int grp = k / half, j = k - grp * half;
                const int i0 = grp * len + j, i1 = i0 + half;
                const double2 a = z[i0], bb = z[i1];
                const double2 w = c_twiddle[j * tw_step];
                const double dx = a.x - bb.x, dy = a.y - bb.y;
                z[i0] = make_double2(a.x + bb.x, a.y + bb.y);
                z[i1] = make_double2(dx * w.x - dy * w.y, dx * w.y + dy * w.x);
            }
            __syncwarp();
        }
        // 4. unpack to the real-input spectrum, power (kaldi.py:616-618); bin M (Nyquist) has zero mel weight
        for (int k = lane; k < M; k += 32) {
            const int kr = __brev((unsigned)k) >> (32 - log2m);
            const int km = (M - k) & (M - 1);
            const int kmr = __brev((unsigned)km) >> (32 - log2m);
            const double2 zk = z[kr], zm = z[kmr];
            const double ex = 0.5 * (zk.x + zm.x), ey = 0.5 * (zk.y - zm.y);      // even part
            const double ox = 0.5 * (zk.y + zm.y), oy = -0.5 * (zk.x - zm.x);     // odd part = -i/2 (zk - conj zm)
            const double2 w = c_twiddle[k];
            const double re = ex + ox * w.x - oy * w.y;
            const double im = ey + ox * w.y + oy * w.x;
            xs[k] = (float)(re * re + im * im);
        }
        __syncwarp();
        // 5. mel + log (kaldi.py:630-633)
        float *o, *o2;
        if constexpr (VL) {
            o = out + ((long long)vl.out_row[b] + f) * p.n_mel;
            o2 = out2 ? out2 + ((long long)vl.frame_off[b] + f) * p.n_mel : nullptr;
        } else {
            const long long orow = out_ids ? out_ids[b] : b;
            o = out + orow * out_row_stride + (long long)(out_frame0 + f) * p.n_mel;
            o2 = out2 ? out2 + ((long long)b * out2_frames + out2_frame0 + f) * p.n_mel : nullptr;
        }
        for (int m = lane; m < p.n_mel; m += 32) {
            const int lo = p.mel_lo[m], hi = p.mel_hi[m];
            const float* wrow = p.mel + (long long)m * (M + 1);
            double e = 0.0;
            for (int k = lo; k < hi; ++k) e += (double)wrow[k] * (double)xs[k];
            const float v = logf(fmaxf((float)e, 1.1920928955078125e-07f));
            o[m] = v;
            if (o2) o2[m] = v;
        }
        __syncwarp();
    }
}

// Streaming ingest (bin/inference.py:61-69): per session, slide the sample buffer and the feature ring.
//   samples[s] = [samples[s][-carry:] | pcm[b] * scale]     ring[s][:ctx] = ring[s][-ctx:]
__global__ void __launch_bounds__(256)
frontend_ingest_kernel(const int32_t* __restrict__ ids, const void* __restrict__ pcm, int is_i16, float scale,
                       int carry, int chunk, int ctx, int m, int n_mel, float* __restrict__ samples,
                       float* __restrict__ ring, float* __restrict__ feats_out) {
    extern __shared__ float tmp[];        // carry + ctx*n_mel
    const int b = blockIdx.x, s = ids[b];
    float* sm = samples + (long long)s * (carry + chunk);
    float* rg = ring + (long long)s * (ctx + m) * n_mel;
    for (int i = threadIdx.x; i < carry; i += blockDim.x) tmp[i] = sm[chunk + i];
    for (int i = threadIdx.x; i < ctx * n_mel; i += blockDim.x) tmp[carry + i] = rg[m * n_mel + i];
    __syncthreads();
    for (int i = threadIdx.x; i < carry; i += blockDim.x) sm[i] = tmp[i];
    for (int i = threadIdx.x; i < chunk; i += blockDim.x) {
        const long long o = (long long)b * chunk + i;
        sm[carry + i] = is_i16 ? (float)reinterpret_cast<const int16_t*>(pcm)[o] * scale
                               : reinterpret_cast<const float*>(pcm)[o] * scale;
    }
    for (int i = threadIdx.x; i < ctx * n_mel; i += blockDim.x) {
        rg[i] = tmp[carry + i];
        if (feats_out) feats_out[(long long)b * (ctx + m) * n_mel + i] = tmp[carry + i];
    }
}

// Several consecutive chunks per session (fbank_stream_blocks), block = (session b, chunk j), packed from off[b]: the sample row
// of a block is [the carry samples before it | its chunk] -- block 0 takes them from the session's sample buffer, a later
// block from the tail of the previous block's PCM.  Values are formed as frontend_ingest_kernel forms them.
__global__ void __launch_bounds__(256)
frontend_blocks_kernel(const int32_t* __restrict__ ids, const int32_t* __restrict__ cnt, const int32_t* __restrict__ off,
                       const void* __restrict__ pcm, int is_i16, float scale, int carry, int chunk,
                       const float* __restrict__ samples, float* __restrict__ rows) {
    const int j = blockIdx.x, b = blockIdx.y;
    if (j >= cnt[b]) return;
    const long long blk = off[b] + j;
    float* r = rows + blk * (carry + chunk);
    const float* sm = samples + (long long)ids[b] * (carry + chunk) + chunk;
    for (int i = threadIdx.x; i < carry + chunk; i += blockDim.x) {
        if (i < carry && j == 0) { r[i] = sm[i]; continue; }
        const long long o = blk * chunk + i - carry;            // i < carry: the previous block's tail
        r[i] = is_i16 ? (float)reinterpret_cast<const int16_t*>(pcm)[o] * scale : reinterpret_cast<const float*>(pcm)[o] * scale;
    }
}

// One CTA per session, after the per-frame kernel: the context rows of every block (block 0: the last ctx frames of the
// session's feature ring; block j: the last ctx new frames of block j - 1, which frames_per_chunk >= ctx puts among that
// block's computed rows), then the session keeps its last block's sample row and features, as fo_fbank_stream leaves them.
__global__ void __launch_bounds__(256)
frontend_blocks_finish_kernel(const int32_t* __restrict__ ids, const int32_t* __restrict__ cnt, const int32_t* __restrict__ off,
                              int carry, int chunk, int ctx, int m, int n_mel, const float* __restrict__ rows,
                              float* __restrict__ feats, float* __restrict__ samples, float* __restrict__ ring) {
    const int b = blockIdx.x, s = ids[b], k = cnt[b];
    const long long blk_feats = (long long)(ctx + m) * n_mel;
    float* f0 = feats + off[b] * blk_feats;
    float* rg = ring + (long long)s * blk_feats;
    for (long long i = threadIdx.x; i < (long long)k * ctx * n_mel; i += blockDim.x) {
        const int j = (int)(i / (ctx * n_mel)), e = (int)(i % (ctx * n_mel));
        f0[j * blk_feats + e] = j == 0 ? rg[m * n_mel + e] : f0[(j - 1) * blk_feats + m * n_mel + e];
    }
    __syncthreads();
    const float* last = f0 + (k - 1) * blk_feats;
    for (int i = threadIdx.x; i < blk_feats; i += blockDim.x) rg[i] = last[i];
    const float* lr = rows + (off[b] + k - 1) * (long long)(carry + chunk);
    for (int i = threadIdx.x; i < carry + chunk; i += blockDim.x) samples[(long long)s * (carry + chunk) + i] = lr[i];
}

// The twiddle table is process-wide constant memory, uploaded under a lock: contexts of one process whose frame lengths need
// different FFT sizes must not run their frontends concurrently (include/fo_b200.h, fo_create_on_sms).
int upload_twiddles(int P) {
    static std::mutex mu;
    std::lock_guard<std::mutex> lk(mu);
    if (g_twiddle_fft == P) return 0;
    FO_CHECK(P >= 64 && P <= MAX_FFT && (P & (P - 1)) == 0, "fbank: FFT size %d unsupported", P);
    static double2 host[MAX_FFT / 2];
    const double PI = 3.14159265358979323846264338327950288;
    for (int k = 0; k < P / 2; ++k) {
        host[k].x = cos(-2.0 * PI * k / P);
        host[k].y = sin(-2.0 * PI * k / P);
    }
    FO_CUDA(cudaMemcpyToSymbol(c_twiddle, host, sizeof(double2) * (P / 2)));
    FO_CUDA(cudaFuncSetAttribute(fbank_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024));
    FO_CUDA(cudaFuncSetAttribute(fbank_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024));
    g_twiddle_fft = P;
    return 0;
}

size_t fbank_smem(int P) { return (size_t)FB_WARPS * (P / 2) * sizeof(double2) + (size_t)FB_WARPS * (P + 32) * sizeof(float); }

}  // namespace

int fbank_stream(const FbankParams& p, const int32_t* ids, int n, const void* pcm, int pcm_is_i16, float scale,
                 int frames_per_chunk, int ctx_frames, float* carry, float* ring, float* feats_out,
                 cudaStream_t st) {
    if (n <= 0) return 0;
    FO_TRY(upload_twiddles(p.fft_size));
    const int carry_n = p.frame_len - p.frame_shift, chunk = p.frame_shift * frames_per_chunk;
    FO_CHECK(frames_per_chunk >= ctx_frames && chunk >= carry_n, "fbank_stream: chunk shorter than its carry/context");
    const size_t sm1 = (size_t)(carry_n + ctx_frames * p.n_mel) * sizeof(float);
    frontend_ingest_kernel<<<n, 256, sm1, st>>>(ids, pcm, pcm_is_i16, scale, carry_n, chunk, ctx_frames,
                                               frames_per_chunk, p.n_mel, carry, ring, feats_out);
    FO_LAUNCHED();
    FO_CUDA(cudaGetLastError());
    SampleSrc src{carry, 0, 1.0f, (long long)(carry_n + chunk), ids};
    const long long frames = (long long)n * frames_per_chunk;
    const int grid = (int)((frames + FB_WARPS - 1) / FB_WARPS);
    fbank_kernel<false><<<grid, FB_WARPS * 32, fbank_smem(p.fft_size), st>>>(
        p, src, n, frames_per_chunk, ring, ids, (long long)(ctx_frames + frames_per_chunk) * p.n_mel, ctx_frames,
        feats_out, ctx_frames + frames_per_chunk, ctx_frames, FbankVarlen());
    FO_LAUNCHED();
    FO_CUDA(cudaGetLastError());
    return 0;
}

int fbank_stream_blocks(const FbankParams& p, const int32_t* ids, const int32_t* cnt, const int32_t* off, int n, int kmax,
                        int blocks, const void* pcm, int pcm_is_i16, float scale, int frames_per_chunk, int ctx_frames,
                        float* carry, float* ring, float* rows, float* feats_out, cudaStream_t st) {
    if (n <= 0) return 0;
    FO_TRY(upload_twiddles(p.fft_size));
    const int carry_n = p.frame_len - p.frame_shift, chunk = p.frame_shift * frames_per_chunk;
    FO_CHECK(frames_per_chunk >= ctx_frames && chunk >= carry_n, "fbank_stream_blocks: chunk shorter than its carry/context");
    frontend_blocks_kernel<<<dim3(kmax, n), 256, 0, st>>>(ids, cnt, off, pcm, pcm_is_i16, scale, carry_n, chunk, carry, rows);
    FO_LAUNCHED();
    FO_CUDA(cudaGetLastError());
    SampleSrc src{rows, 0, 1.0f, (long long)(carry_n + chunk), nullptr};
    const long long frames = (long long)blocks * frames_per_chunk;
    fbank_kernel<false><<<(int)((frames + FB_WARPS - 1) / FB_WARPS), FB_WARPS * 32, fbank_smem(p.fft_size), st>>>(
        p, src, blocks, frames_per_chunk, feats_out, nullptr, (long long)(ctx_frames + frames_per_chunk) * p.n_mel, ctx_frames,
        nullptr, 0, 0, FbankVarlen());
    FO_LAUNCHED();
    FO_CUDA(cudaGetLastError());
    frontend_blocks_finish_kernel<<<n, 256, 0, st>>>(ids, cnt, off, carry_n, chunk, ctx_frames, frames_per_chunk, p.n_mel, rows,
                                                     feats_out, carry, ring);
    FO_LAUNCHED();
    FO_CUDA(cudaGetLastError());
    return 0;
}

int fbank_offline(const FbankParams& p, const void* pcm, int pcm_is_i16, int B, long long n_samples, float scale,
                  float* out, cudaStream_t st) {
    if (B <= 0 || n_samples < p.frame_len) return 0;
    FO_TRY(upload_twiddles(p.fft_size));
    const int m = (int)(1 + (n_samples - p.frame_len) / p.frame_shift);
    SampleSrc src{pcm, pcm_is_i16, scale, n_samples, nullptr};
    const long long frames = (long long)B * m;
    long long want = (frames + FB_WARPS - 1) / FB_WARPS;
    const int grid = (int)std::min<long long>(want, 16LL * p.sms);  // persistent-ish: 16 CTAs per SM of the context, grid-stride
    fbank_kernel<false><<<grid, FB_WARPS * 32, fbank_smem(p.fft_size), st>>>(p, src, B, m, out, nullptr,
                                                                             (long long)m * p.n_mel, 0, nullptr, 0, 0, FbankVarlen());
    FO_LAUNCHED();
    FO_CUDA(cudaGetLastError());
    return 0;
}

int fbank_offline_packed(const FbankParams& p, const void* pcm, int pcm_is_i16, float scale, const FbankVarlen& vl, float* out,
                         float* out2, cudaStream_t st) {
    if (vl.n <= 0 || vl.frames <= 0) return 0;
    FO_TRY(upload_twiddles(p.fft_size));
    SampleSrc src{pcm, pcm_is_i16, scale, 0, nullptr};
    long long want = (vl.frames + FB_WARPS - 1) / FB_WARPS;
    const int grid = (int)std::min<long long>(want, 16LL * p.sms);  // as fbank_offline
    fbank_kernel<true><<<grid, FB_WARPS * 32, fbank_smem(p.fft_size), st>>>(p, src, 0, 0, out, nullptr, 0, 0, out2, 0, 0, vl);
    FO_LAUNCHED();
    FO_CUDA(cudaGetLastError());
    return 0;
}

FO_TR_BIND_DEF(trace_bind_fbank)

}  // namespace fo
