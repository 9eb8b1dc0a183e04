// Weight-streaming layer stack: every transformer layer of a streaming step in ONE cooperative launch, for steps of at
// most 16 token rows (1-4 sessions of 4 encoder frames; taken by default up to 8 rows).  Reference loop being replaced:
// Transformer.infer / TransformerLayer.infer (models/encoder/transformer.py:103-130, 273-285) with
// MultiHeadedAttention.infer (models/encoder/attention.py:407-459) and PositionwiseFeedForward (attention.py:137-143).
//
// Why a second execution form next to the per-kernel chain of fo_api.cu: with <= 16 rows a layer is pure weight
// streaming (25 MB of weights against 0.1 GFLOP), and the chain's 7 dependent kernels per layer each cost ~5 us of
// dependency latency (grid completion -> griddepcontrol.wait -> first load -> ... -> stores drained): 0.92 ms for one
// session against an HBM floor of 0.12 ms.  Here
//   * 148 CTAs (one per SM) stay resident for all layers; a phase boundary is a grid barrier (release add + acquire
//     poll, ~1 us), five per layer: QKV | attention | out-proj | FFN1 | FFN2;
//   * every CTA owns a fixed slice of the OUTPUT rows of each weight matrix (3D/G, D/G, FF/G, D/G rows over full K).  The
//     kernel reads its own copy of the four layer matrices whose rows are padded by 16 bytes in HBM, so a slice is ONE
//     contiguous cp.async.bulk that lands with the row stride that makes the MMA fragment loads bank-conflict free; it is
//     requested one to four phases AHEAD of its use -- weights never depend on activations, so HBM streaming runs straight
//     through the barriers; no split-K, no partial sums in global memory;
//   * the activations of a phase are tiny (<= 16 x 4096 fp16), every CTA re-reads them from L2 and the LayerNorm in
//     front of QKV / FFN1 is simply recomputed by every CTA (16 KB of fp32 rows) -- no LayerNorm phase;
//   * the contraction is mma.sync.m16n8k16 (up to 8 token rows: 16 weight rows on M, the tokens on N; the 8 warps split K
//     and reduce through shared memory): tcgen05 needs >= 64 rows per operand tile and its 128-lane TMEM epilogue; for
//     4-8 rows the warp-level MMA wastes nothing that matters (0.1 GFLOP per layer);
//   * attention units (session, head) run on the first n*H CTAs; their ring / rel-pos rows are requested a phase early
//     (they never depend on this step), the other CTAs prefetch the next layer's small parameters into L2 meanwhile.
// Arithmetic matches the chain: fp16-staged activations x bf16-rounded weights in fp16 containers, fp32 accumulation,
// residual stream / LayerNorm / softmax / Q in fp32 (DESIGN 4a); only the summation order inside a dot product differs.
//
// Measured (B200, shipped model, graph replay; tools/stack_check.py, FO_STACK_TRACE=1 prints the in-kernel stamps): one
// session 0.92 -> 0.69 ms per 160 ms chunk (kernel 0.55 ms = 24 x 22.7 us; front 0.07, adapter 0.06 stay on the chain), two
// sessions 0.95 -> 0.82 ms, four sessions 0.95 -> 1.04 ms (hence the default threshold of 8 rows).  A layer is 5 x
// (barrier ~1.3 us incl. skew + activation rows ready 1.1-1.6 us + MMAs 0.6-0.9 us + reduce / store 0.35 us) with the
// attention unit at ~3.4 us: latency of dependent L2 round trips, not bandwidth (25 MB per 22.7 us = 1.1 TB/s).
#include <stdlib.h>

#include <algorithm>
#include <map>
#include <mutex>

#include "fo_attn_core.cuh"

namespace fo {
namespace {

constexpr int ST_THREADS = 256;
constexpr int ST_WARPS = ST_THREADS / 32;
constexpr int BAR_COUNTER = 512;          // counter word of the barrier buffer (the words below it are the per-CTA records)
constexpr int MAXG = 4;                    // 8-row weight groups per CTA and phase (<= 32 rows)

#define ST_NOINLINE __device__ __noinline__

struct StackLayout {                       // byte offsets into the dynamic shared memory
    int s1, s2, s3, act, red, attn;
    int act_bytes;
    int kc;                                // K chunk of the FFN2 activations held in `act` at a time
    int dbg;                               // development (FO_STACK_DBG, results invalid): 1 = no epilogue stores
};

__device__ __forceinline__ uint32_t lds32s(uint32_t addr) {        // explicit shared-space load (inside non-inlined code the
    uint32_t v;                                                    // compiler only sees generic pointers)
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(addr));
    return v;
}
__device__ __forceinline__ unsigned long long gtime() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}

// Grid barrier.  Every CTA adds one to ONE counter (release: the CTA's writes of the phase, ordered before it by the CTA
// barrier, become visible with it) and polls it (acquire) until all G arrivals of this barrier are in.  Measured (per-CTA
// %globaltimer stamps, tools/stack_check.py): the first CTA leaves 0.9-1.0 us after the last one arrived.  Measured and lost:
//   * the arrivals spread over 8 counters polled by 8 lanes (relaxed loads + acquire fence): 1.2-2.6 us;
//   * per-CTA flags polled by a warp: ~5 us (148 warps re-reading the lines the flags are being stored to);
//   * a two-level counter tree (groups of 16, last arrival adds to a root): 3.3 us, three dependent L2 round trips;
//   * issuing the next weight slices' bulk copies just before / inside the barrier: 2.1-2.6 us -- 148 SMs x 40-58 KB arrive as
//     one burst through HBM -> L2 -> SM and the arrive / poll traffic queues behind it.  `issue` therefore runs AFTER the
//     barrier (last warp): the burst then overlaps the L2 latency of the phase's activation loads and its shared-memory work.
// The counter only grows, across launches too: flags[cta] records how many barriers the CTA has passed so far (every CTA
// passes the same number per launch), the targets continue from there and nothing is ever reset; compared through a
// signed difference.
template <typename F>
__device__ __forceinline__ void grid_barrier(unsigned int* flags, unsigned int target, int G, F&& issue, unsigned long long* arr = nullptr) {
    __syncthreads();
    if (threadIdx.x == 0) {
        if (arr) arr[0] = gtime();
        unsigned int* ctr = flags + BAR_COUNTER;
        asm volatile("red.release.gpu.global.add.u32 [%0], 1;" ::"l"(ctr) : "memory");
        const unsigned int want = target * (unsigned int)G;
        unsigned int v, spins = 0;
        do {
            asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(ctr) : "memory");
            if (++spins > (1u << 23)) __trap();                // seconds: a CTA is missing (never on a cooperative launch) -- fail loudly
        } while ((int)(v - want) < 0);
        if (arr) arr[1] = gtime();
    }
    __syncthreads();
    if (threadIdx.x >= ST_THREADS - 32) issue();
}

// one thread: rows [r0, r0 + nr) of a weight matrix -> shared memory, ONE bulk copy.  The stack kernel reads its own copy
// of the layer weights whose rows are padded by 16 bytes in HBM (StackLayer): the slice is then contiguous in HBM AND lands
// with the padded row stride that makes the B-fragment loads bank-conflict free (rows shift by 4 banks).  One copy per row
// from the unpadded matrices cost ~50 ns of issue time each, 3 us per layer on whichever warp issued them (measured).
__device__ __forceinline__ void load_rows(__half* dst, const __half* Wp, int r0, int nr, int K, uint64_t* bar) {
    if (nr <= 0) return;
    const uint32_t bytes = (uint32_t)nr * (uint32_t)(K * 2 + 16);
    mbar_expect_tx(bar, bytes);
    bulk_g2s(dst, reinterpret_cast<const char*>(Wp) + (long long)r0 * (K * 2 + 16), bytes, bar);
}

// LayerNorm of the M rows of x (fp32, read through L2: other CTAs wrote them in this launch) into fp16 rows of `act`.
// TWO warps per row (a lane holds D/256 float4 of it), so that with 4 rows all 8 warps work and x, gamma and beta are all
// requested before the first reduction (one L2 latency); two-pass (mean, centred variance) like layer_norm_reduce_kernel.
// Every warp runs the same number of iterations (CTA barriers inside).
ST_NOINLINE void ln_rows(const float* x, int M, int D, const float* __restrict__ gamma,
                                        const float* __restrict__ beta, __half* act, int astr, int warp, int lane, float* red) {
    const int hq = D >> 3;                          // float4 per half row; lane holds those at lane, lane + 32, ... (D <= 1024)
    const int pair = warp >> 1, half = warp & 1;
    const int f0 = half * (D >> 3) + lane;          // first float4 of this lane within the row
    for (int m0 = 0; m0 < M; m0 += ST_WARPS / 2) {
        const int m = m0 + pair;
        const bool live = m < M;
        const float4* xr = reinterpret_cast<const float4*>(x + (long long)(live ? m : 0) * D) + f0;
        float4 v[4], gg[4], bb[4];
#pragma unroll
        for (int i = 0; i < 4; ++i)
            if (lane + i * 32 < hq) {
                v[i] = __ldcg(xr + i * 32);
                gg[i] = __ldg(reinterpret_cast<const float4*>(gamma) + f0 + i * 32);
                bb[i] = __ldg(reinterpret_cast<const float4*>(beta) + f0 + i * 32);
            }
        float s = 0.f;
#pragma unroll
        for (int i = 0; i < 4; ++i)
            if (lane + i * 32 < hq) s += v[i].x + v[i].y + v[i].z + v[i].w;
        s = warp_sum(s);
        if (lane == 0) red[warp * 2] = s;
        __syncthreads();
        const float mu = (red[pair * 4] + red[pair * 4 + 2]) / D;
        float q = 0.f;
#pragma unroll
        for (int i = 0; i < 4; ++i)
            if (lane + i * 32 < hq) {
                const float a = v[i].x - mu, b = v[i].y - mu, c = v[i].z - mu, d = v[i].w - mu;
                q += a * a + b * b + c * c + d * d;
            }
        q = warp_sum(q);
        if (lane == 0) red[warp * 2 + 1] = q;
        __syncthreads();
        const float rstd = rsqrtf((red[pair * 4 + 1] + red[pair * 4 + 3]) / D + 1e-5f);
        if (live) {
#pragma unroll
            for (int i = 0; i < 4; ++i)
                if (lane + i * 32 < hq) {
                    const int col = (f0 + i * 32) * 4;
                    uint2 o;
                    o.x = pack2<__half>((v[i].x - mu) * rstd * gg[i].x + bb[i].x, (v[i].y - mu) * rstd * gg[i].y + bb[i].y);
                    o.y = pack2<__half>((v[i].z - mu) * rstd * gg[i].z + bb[i].z, (v[i].w - mu) * rstd * gg[i].w + bb[i].w);
                    *reinterpret_cast<uint2*>(act + (long long)m * astr + col) = o;
                }
        }
    }
}

// M rows x kc halves of a row-major fp16 matrix (leading dimension ld, column offset k0) -> padded rows of `act`
ST_NOINLINE void load_act(const __half* src, int M, int ld, int k0, int kc, __half* act, int astr, int tid) {
    const int per = kc >> 3, total = M * per;
#pragma unroll 8
    for (int i = tid; i < total; i += ST_THREADS) {
        const int r = i / per, c8 = i - r * per;
        const uint4 v = __ldcg(reinterpret_cast<const uint4*>(src + (long long)r * ld + k0) + c8);
        *reinterpret_cast<uint4*>(act + (long long)r * astr + c8 * 8) = v;
    }
}

// This warp's partial tiles of the slice: tile gi (16 tokens x 8 weight rows) = act[:, kk] . w[gi*8 + n, wk0 + kk] over the
// warp's eighth of the kc columns, stored to (or, for the later K chunks of FFN2, added to) red[warp][gi][lane][4].
// With a single weight group (out-proj, FFN2: 7 rows per CTA) consecutive k steps go to four accumulators in turn and are
// summed at the end (one dependent HMMA chain and one load round trip per k step otherwise).  Not inlined: the four GEMM
// phases share this code -- the fully inlined kernel was 210 KB of SASS and every phase started with instruction-cache misses.
ST_NOINLINE void slice_gemm(const __half* act, int astr, int M, const __half* w, int wstr, int wk0, int kc,
                                        int ng, float* red, int accumulate) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int g = lane >> 2, c = lane & 3;
    const int kw = kc / ST_WARPS;
    const bool lo = g < M, hi = g + 8 < M;
    const uint32_t a0p = smem_u32(act) + (uint32_t)(g * astr + c * 2) * 2u;          // byte addresses in shared memory
    const uint32_t a1p = a0p + (uint32_t)(8 * astr) * 2u;
    const uint32_t bp = smem_u32(w) + (uint32_t)(g * wstr + wk0 + c * 2) * 2u;
    const uint32_t gstep = (uint32_t)(8 * wstr) * 2u;
    const int kend = (warp + 1) * kw;
    float d[MAXG][4] = {};
    if (M <= 8) {
        // up to 8 token rows: the WEIGHT rows go on the MMA-M side (16 per tile) and the tokens on N = 8 -- half the HMMAs of
        // the other orientation for the QKV / FFN1 slices (21 / 28 rows: 2 tiles instead of 3 / 4 groups); the legacy
        // mma.sync pipe of sm_100 retires one m16n8k16 per ~40 clocks per SM sub-partition, and it is what bounds these loops
        const int nt = (ng + 1) >> 1;
        const uint32_t wp0 = smem_u32(w) + (uint32_t)(g * wstr + wk0 + c * 2) * 2u;       // weight row g (and g + 8) of a tile
        const uint32_t wp1 = wp0 + gstep;
        const uint32_t tp = smem_u32(act) + (uint32_t)(g * astr + c * 2) * 2u;            // token g
        if (nt == 1 && kw % (16 * MAXG) == 0) {
#pragma unroll 2
            for (int kk = warp * kw; kk < kend; kk += 16 * MAXG) {
                uint32_t a[MAXG][4], b[MAXG][2];
#pragma unroll
                for (int s = 0; s < MAXG; ++s) {
                    const uint32_t k = (uint32_t)(kk + 16 * s) * 2u;
                    a[s][0] = lds32s(wp0 + k);
                    a[s][1] = lds32s(wp1 + k);
                    a[s][2] = lds32s(wp0 + k + 16);
                    a[s][3] = lds32s(wp1 + k + 16);
                    b[s][0] = lo ? lds32s(tp + k) : 0u;
                    b[s][1] = lo ? lds32s(tp + k + 16) : 0u;
                }
#pragma unroll
                for (int s = 0; s < MAXG; ++s) mma16816(d[s], a[s], b[s]);
            }
#pragma unroll
            for (int r = 0; r < 4; ++r) d[0][r] = (d[0][r] + d[1][r]) + (d[2][r] + d[3][r]);
        } else {
#pragma unroll 2
            for (int kk = warp * kw; kk < kend; kk += 16) {
                const uint32_t k = (uint32_t)kk * 2u;
                uint32_t b[2];
                b[0] = lo ? lds32s(tp + k) : 0u;
                b[1] = lo ? lds32s(tp + k + 16) : 0u;
#pragma unroll
                for (int ti = 0; ti < MAXG / 2; ++ti)
                    if (ti < nt) {
                        uint32_t a[4];
                        a[0] = lds32s(wp0 + ti * 2 * gstep + k);
                        a[1] = lds32s(wp1 + ti * 2 * gstep + k);
                        a[2] = lds32s(wp0 + ti * 2 * gstep + k + 16);
                        a[3] = lds32s(wp1 + ti * 2 * gstep + k + 16);
                        mma16816(d[ti], a, b);
                    }
            }
        }
        ng = nt;                                               // tiles stored below
    } else if (ng == 1 && kw % (16 * MAXG) == 0) {
#pragma unroll 2
        for (int kk = warp * kw; kk < kend; kk += 16 * MAXG) {
            uint32_t a[MAXG][4], b[MAXG][2];
#pragma unroll
            for (int s = 0; s < MAXG; ++s) {
                const uint32_t k = (uint32_t)(kk + 16 * s) * 2u;
                a[s][0] = lo ? lds32s(a0p + k) : 0u;
                a[s][1] = hi ? lds32s(a1p + k) : 0u;
                a[s][2] = lo ? lds32s(a0p + k + 16) : 0u;
                a[s][3] = hi ? lds32s(a1p + k + 16) : 0u;
                b[s][0] = lds32s(bp + k);
                b[s][1] = lds32s(bp + k + 16);
            }
#pragma unroll
            for (int s = 0; s < MAXG; ++s) mma16816(d[s], a[s], b[s]);
        }
#pragma unroll
        for (int r = 0; r < 4; ++r) d[0][r] = (d[0][r] + d[1][r]) + (d[2][r] + d[3][r]);
    } else {
#pragma unroll 2
        for (int kk = warp * kw; kk < kend; kk += 16) {
            const uint32_t k = (uint32_t)kk * 2u;
            uint32_t a[4];
            a[0] = lo ? lds32s(a0p + k) : 0u;
            a[1] = hi ? lds32s(a1p + k) : 0u;
            a[2] = lo ? lds32s(a0p + k + 16) : 0u;
            a[3] = hi ? lds32s(a1p + k + 16) : 0u;
#pragma unroll
            for (int gi = 0; gi < MAXG; ++gi)
                if (gi < ng) {
                    uint32_t b[2];
                    b[0] = lds32s(bp + gi * gstep + k);
                    b[1] = lds32s(bp + gi * gstep + k + 16);
                    mma16816(d[gi], a, b);
                }
        }
    }
#pragma unroll
    for (int gi = 0; gi < MAXG; ++gi)
        if (gi < ng) {
            float4* rp = reinterpret_cast<float4*>(red + ((warp * MAXG + gi) * 32 + lane) * 4);
            float4 v = make_float4(d[gi][0], d[gi][1], d[gi][2], d[gi][3]);
            if (accumulate) { const float4 o = *rp; v.x += o.x; v.y += o.y; v.z += o.z; v.w += o.w; }
            *rp = v;
        }
}
// element (token m, weight row j of the slice): sum over the warps in warp order (deterministic)
// (wm: slice_gemm put the weight rows on the MMA-M side -- tile = 16 weight rows x 8 tokens)
__device__ __forceinline__ float red_sum(const float* red, int m, int j, bool wm) {
    const int gi = wm ? j >> 4 : j >> 3, n = j & 7;
    const int idx = wm ? (gi * 32 + n * 4 + (m >> 1)) * 4 + (m & 1) + 2 * ((j >> 3) & 1)
                       : (gi * 32 + (m & 7) * 4 + (n >> 1)) * 4 + (n & 1) + 2 * (m >> 3);
    float s = 0.f;
#pragma unroll
    for (int w = 0; w < ST_WARPS; ++w) s += red[w * MAXG * 128 + idx];
    return s;
}

__device__ __forceinline__ void prefetch_l2(const void* ptr, long long bytes, int tid) {
    if (!ptr || (reinterpret_cast<uintptr_t>(ptr) & 15)) return;
    const char* base = reinterpret_cast<const char*>(ptr);
    for (long long off = (long long)tid * 2048; off < bytes; off += (long long)ST_THREADS * 2048) {
        const unsigned sz = (unsigned)min(2048LL, bytes - off) & ~15u;
        if (sz) asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(base + off), "r"(sz) : "memory");
    }
}
// the small per-layer parameters (LayerNorm, biases, pos_bias_u/v) of a layer: idle CTA `idx` asks L2 for item `idx`
__device__ __forceinline__ void prefetch_small(const StackLayer& w, int D, int FF, int idx, int tid) {
    switch (idx) {
        case 0: prefetch_l2(w.ln1g, D * 4LL, tid); break;
        case 1: prefetch_l2(w.ln1b, D * 4LL, tid); break;
        case 2: prefetch_l2(w.ln2g, D * 4LL, tid); break;
        case 3: prefetch_l2(w.ln2b, D * 4LL, tid); break;
        case 4: prefetch_l2(w.bqkv, 3LL * D * 4, tid); break;
        case 5: prefetch_l2(w.bo, D * 4LL, tid); break;
        case 6: prefetch_l2(w.b1, FF * 4LL, tid); break;
        case 7: prefetch_l2(w.b2, D * 4LL, tid); break;
        case 8: prefetch_l2(w.pos_u, D * 4LL, tid); break;
        case 9: prefetch_l2(w.pos_v, D * 4LL, tid); break;
        default: break;
    }
}

// ---- attention unit (session b, head h): attention_stream_mma_kernel of fo_attention.cu as a phase of this kernel ----
struct AttnGeom {
    int slot, nf, cl, first, nk, start, np;
};
__device__ __forceinline__ AttnGeom attn_geom(const AttnStream& a, int b) {
    AttnGeom g;
    g.slot = a.ids[b];
    g.nf = a.n_frames[g.slot];
    g.cl = min(g.nf, a.window);
    g.first = g.nf - g.cl;
    g.nk = g.cl + a.t;
    const int pe = a.pe_index[g.slot] % a.pe_wrap;
    g.start = max(0, pe - a.full_chunk);                 // attention.py:112-114
    g.np = min(g.nk, a.pos_rows - g.start);
    return g;
}
// thread 0, one phase early: cached K / V rows of the ring and the rel-pos rows of this head -> the unit's shared memory
__device__ __forceinline__ void attn_issue(const AttnStream& a, const AttnGeom& g, const StackLayer& w, int h, unsigned char* region,
                                           uint64_t* bar) {
    const MmaUnitLayout lay = mma_unit_layout(a.window, a.t);
    const __half* ringK = w.ring + (long long)g.slot * a.ring_slot_stride + (long long)h * a.ring_cap * DK;
    const __half* ringV = ringK + (long long)a.H * a.ring_cap * DK;
    ring_window_copy(ringK, ringV, a.ring_cap, g.first, g.cl, reinterpret_cast<__half*>(region), reinterpret_cast<__half*>(region + lay.v),
                     w.ptab_h + ((long long)h * a.pos_rows + g.start) * DK, reinterpret_cast<__half*>(region + lay.p), g.np, bar);
}
// Staging of the stack kernel's attention phase: the chunk's own K / V rows from p.kv and Q from p.q32 (written by other CTAs in
// this launch, hence __ldcg), appended to the ring in the same pass; the ring window and rel-pos rows were issued a phase early
// (attn_issue).  The core is attn_chunk_mma over all ST_WARPS warps.
__device__ __forceinline__ void attn_unit(const StackArgs& p, const AttnGeom& ge, const StackLayer& w, int b, int h, unsigned char* region,
                                          uint64_t* bar, uint32_t parity, int tid) {
    const AttnStream& a = p.a;
    const int t = a.t, D = a.H * DK, cap = a.ring_cap;
    const MmaUnitLayout lay = mma_unit_layout(a.window, t);
    const int vrows = lay.vrows;
    __half* Ks = reinterpret_cast<__half*>(region);
    __half* Ps = reinterpret_cast<__half*>(region + lay.p);
    __half* Vs = reinterpret_cast<__half*>(region + lay.v);
    __half* quh = reinterpret_cast<__half*>(region + lay.qu);
    __half* qvh = reinterpret_cast<__half*>(region + lay.qv);
    const int nf = ge.nf, cl = ge.cl, nk = ge.nk, start = ge.start, np = ge.np;
    __half* ringK = w.ring + (long long)ge.slot * a.ring_slot_stride + (long long)h * cap * DK;
    __half* ringV = ringK + (long long)a.H * cap * DK;
    // the chunk's own K / V rows: into the tile and appended to the ring.  16-byte chunk c of the row of frame f lives at
    // chunk c ^ (f & 7) (bank-conflict-free fragment loads although the bulk copies land rows densely)
    for (int i = tid; i < t * 8 * 2; i += ST_THREADS) {
        const int which = i / (t * 8), r = (i >> 3) % t, c = i & 7;
        const uint4 val = __ldcg(reinterpret_cast<const uint4*>(p.kv + (long long)(b * t + r) * 2 * D + which * D + h * DK) + c);
        const int pc = c ^ ((nf + r) & 7);
        *reinterpret_cast<uint4*>((which ? Vs : Ks) + (cl + r) * DK + pc * 8) = val;
        *reinterpret_cast<uint4*>((which ? ringV : ringK) + (long long)((nf + r) % cap) * DK + pc * 8) = val;
    }
    for (int i = tid; i < (vrows - nk) * 8; i += ST_THREADS)          // zero V rows behind the last key (probability 0 x finite)
        *reinterpret_cast<uint4*>(Vs + (nk + (i >> 3)) * DK + (i & 7) * 8) = make_uint4(0, 0, 0, 0);
    for (int i = tid + np * 8; i < nk * 8; i += ST_THREADS) {          // in-bounds clamp only: pos_rows covers every reachable position
        const int j = i >> 3, c = i & 7;
        *reinterpret_cast<uint4*>(Ps + j * DK + (c ^ ((start + j) & 7)) * 8) =
            *reinterpret_cast<const uint4*>(w.ptab_h + ((long long)h * a.pos_rows + a.pos_rows - 1) * DK + (c ^ ((a.pos_rows - 1) & 7)) * 8);
    }
    for (int i = tid; i < t * DK; i += ST_THREADS) {
        const int r = i / DK, d = i % DK;
        const float q = __ldcg(p.q32 + (long long)(b * t + r) * D + h * DK + d);
        const int o = r * DK + (((d >> 3) ^ (r & 7)) << 3) + (d & 7);
        quh[o] = from_f<__half>(q + __ldg(w.pos_u + h * DK + d));
        qvh[o] = from_f<__half>(q + __ldg(w.pos_v + h * DK + d));
    }
    __syncthreads();
    mbar_wait(bar, parity);
    attn_chunk_mma<ST_WARPS>(Ks, Vs, ge.first, Ps, start, quh, qvh, reinterpret_cast<__half*>(region + lay.ph),
                             reinterpret_cast<float*>(region + lay.sc), vrows, nk, t, p.att + (long long)b * t * D + h * DK, D);
}

// development stamps inside a phase (CTA 0, thread 0): trace[5L + 2 + 6 * phase + k]
#define ST_STAMP(k)                                                                                  \
    do {                                                                                             \
        if (p.trace && cta == 0 && tid == 0) p.trace[5 * p.L + 2 + 6 * epoch + (k)] = gtime();       \
    } while (0)

__global__ void __launch_bounds__(ST_THREADS, 1)
stream_stack_kernel(const __grid_constant__ StackArgs p, const __grid_constant__ StackLayout lay) {
    extern __shared__ __align__(128) unsigned char smem[];
    __shared__ __align__(8) uint64_t bars[4];             // S1, S2, S3 filled; attention rows landed
    __shared__ float lnred[ST_WARPS * 2];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int G = gridDim.x, cta = blockIdx.x;
    const int D = p.D, FF = p.FF, H = p.a.H, t = p.a.t, M = p.a.n * t;
    const int wsD = D + 8, wsF = FF + 8;                  // padded row strides (halves): rows shift by 4 banks
    const bool wm = M <= 8;                               // orientation of the MMA tiles (slice_gemm)
    __half* S1 = reinterpret_cast<__half*>(smem + lay.s1);       // QKV slice, then this layer's FFN1 slice
    __half* S2 = reinterpret_cast<__half*>(smem + lay.s2);       // FFN2 slice
    __half* S3 = reinterpret_cast<__half*>(smem + lay.s3);       // out-proj slice
    __half* ACT = reinterpret_cast<__half*>(smem + lay.act);     // the phase's activation rows
    float* RED = reinterpret_cast<float*>(smem + lay.red);       // the warps' partial tiles
    unsigned char* ATT = smem + lay.attn;
    const int qr0 = (int)((long long)cta * 3 * D / G), qn = (int)((long long)(cta + 1) * 3 * D / G) - qr0;
    const int or0 = (int)((long long)cta * D / G), on = (int)((long long)(cta + 1) * D / G) - or0;
    const int fr0 = (int)((long long)cta * FF / G), fn = (int)((long long)(cta + 1) * FF / G) - fr0;
    const bool has_attn = cta < p.a.n * H;
    const int ab = cta / H, ah = cta % H;
    uint32_t par1 = 0, par2 = 0, par3 = 0, para = 0;
    unsigned int epoch = 0;
    const unsigned int base = p.bar[cta];                 // barriers this CTA has passed in earlier launches (see grid_barrier)
    AttnGeom ge = {};
    if (has_attn) ge = attn_geom(p.a, ab);                // session state is constant during the launch

    if (tid == 0) {
        for (int i = 0; i < 4; ++i) mbar_init(&bars[i], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    {
        const StackLayer w0 = p.layers[0];
        if (tid == ST_THREADS - 32) {
            load_rows(S1, w0.wqkv, qr0, qn, D, &bars[0]);
            load_rows(S3, w0.wo, or0, on, D, &bars[2]);
            load_rows(S2, w0.w2, or0, on, FF, &bars[1]);
            if (has_attn) attn_issue(p.a, ge, w0, ah, ATT, &bars[3]);
        }
        prefetch_small(w0, D, FF, cta, tid);
    }
    if (p.trace && cta == 0 && tid == 0) p.trace[0] = gtime();

    for (int l = 0; l < p.L; ++l) {
        const StackLayer w = p.layers[l];
        const bool more = l + 1 < p.L;
        unsigned long long* arr = (p.trace && l == p.L / 2) ? p.trace + 35 * p.L + 8 + 2 * cta : nullptr;   // + 2 * G * phase
        // bias (and residual) of the element this thread finishes: requested before the phase's work, off the critical path
        float pb = 0.f, px = 0.f;
        // ---------------- QKV: h = norm1(x) (every CTA), q / k / v columns [qr0, qr0 + qn) ----------------
        if (tid < M * qn) pb = __ldg(w.bqkv + qr0 + tid % qn);
        ln_rows(p.x, M, D, w.ln1g, w.ln1b, ACT, wsD, warp, lane, lnred);
        __syncthreads();
        ST_STAMP(0);
        if (qn > 0) {
            mbar_wait(&bars[0], par1);
            par1 ^= 1;
            ST_STAMP(1);
            slice_gemm(ACT, wsD, M, S1, wsD, 0, D, (qn + 7) >> 3, RED, 0);
            ST_STAMP(4);
        }
        __syncthreads();                                       // S1 is free, the partial tiles are in RED
        ST_STAMP(2);
        for (int e = tid; e < M * qn; e += ST_THREADS) {
            const int m = e / qn, j = e - m * qn, col = qr0 + j;
            const float v = red_sum(RED, m, j, wm) + (e == tid ? pb : __ldg(w.bqkv + col));
            if (lay.dbg & 1) continue;
            if (col < D) p.q32[(long long)m * D + col] = v;                       // Q stays fp32
            else {
                if (p.sat && fabsf(v) > 65504.f) atomicAdd(p.sat, 1ULL);
                p.kv[(long long)m * 2 * D + col - D] = from_f<__half>(v);
            }
        }
        ST_STAMP(3);
        grid_barrier(p.bar, base + ++epoch, G, [&] {
            if (lane != 0) return;
            load_rows(S1, w.w1, fr0, fn, D, &bars[0]);                  // this layer's FFN1 and FFN2 slices: they land while most
            if (l > 0) load_rows(S2, w.w2, or0, on, FF, &bars[1]);      // CTAs idle through the attention phase
        }, arr ? arr + 2 * G * 0 : nullptr);
        if (p.trace && cta == 0 && tid == 0) p.trace[epoch] = gtime();
        // ---------------- attention units on the first n*H CTAs ----------------
        if (has_attn) {
            attn_unit(p, ge, w, ab, ah, ATT, &bars[3], para, tid);
            para ^= 1;
        } else if (more) {
            prefetch_small(p.layers[l + 1], D, FF, cta - p.a.n * H, tid);
        }
        grid_barrier(p.bar, base + ++epoch, G, [] {}, arr ? arr + 2 * G * 1 : nullptr);
        if (p.trace && cta == 0 && tid == 0) p.trace[epoch] = gtime();
        // ---------------- out-proj: x[:, or0 .. ] += att . Wo^T + bo ----------------
        if (tid < M * on) {
            pb = __ldg(w.bo + or0 + tid % on);
            px = __ldcg(p.x + (long long)(tid / on) * D + or0 + tid % on);
        }
        load_act(p.att, M, D, 0, D, ACT, wsD, tid);
        __syncthreads();
        ST_STAMP(0);
        if (on > 0) {
            mbar_wait(&bars[2], par3);
            par3 ^= 1;
            ST_STAMP(1);
            slice_gemm(ACT, wsD, M, S3, wsD, 0, D, (on + 7) >> 3, RED, 0);
            ST_STAMP(4);
        }
        __syncthreads();
        ST_STAMP(2);
        for (int e = tid; e < M * on; e += ST_THREADS) {
            const int m = e / on, j = e - m * on, col = or0 + j;
            float* xp = p.x + (long long)m * D + col;
            const float xv = e == tid ? (red_sum(RED, m, j, wm) + pb) + px : (red_sum(RED, m, j, wm) + __ldg(w.bo + col)) + __ldcg(xp);
            if (!(lay.dbg & 1)) *xp = xv;
        }
        ST_STAMP(3);
        grid_barrier(p.bar, base + ++epoch, G, [&] { if (more && lane == 0) load_rows(S3, p.layers[l + 1].wo, or0, on, D, &bars[2]); }, arr ? arr + 2 * G * 2 : nullptr);
        if (p.trace && cta == 0 && tid == 0) p.trace[epoch] = gtime();
        // ---------------- FFN1: relu(norm2(x) . W1^T + b1), columns [fr0, fr0 + fn) ----------------
        if (tid < M * fn) pb = __ldg(w.b1 + fr0 + tid % fn);
        ln_rows(p.x, M, D, w.ln2g, w.ln2b, ACT, wsD, warp, lane, lnred);
        __syncthreads();
        ST_STAMP(0);
        if (fn > 0) {
            mbar_wait(&bars[0], par1);
            par1 ^= 1;
            ST_STAMP(1);
            slice_gemm(ACT, wsD, M, S1, wsD, 0, D, (fn + 7) >> 3, RED, 0);
            ST_STAMP(4);
        }
        __syncthreads();
        ST_STAMP(2);
        for (int e = tid; e < M * fn; e += ST_THREADS) {
            const int m = e / fn, j = e - m * fn, col = fr0 + j;
            const float v = fmaxf(red_sum(RED, m, j, wm) + (e == tid ? pb : __ldg(w.b1 + col)), 0.f);
            if (p.sat && v > 65504.f) atomicAdd(p.sat, 1ULL);
            if (!(lay.dbg & 1)) p.ffh[(long long)m * FF + col] = from_f<__half>(v);
        }
        ST_STAMP(3);
        grid_barrier(p.bar, base + ++epoch, G, [&] { if (more && lane == 0) load_rows(S1, p.layers[l + 1].wqkv, qr0, qn, D, &bars[0]); }, arr ? arr + 2 * G * 3 : nullptr);
        if (p.trace && cta == 0 && tid == 0) p.trace[epoch] = gtime();
        // ---------------- FFN2: x[:, or0 .. ] += ffh . W2^T + b2 (K = FF in chunks of lay.kc) ----------------
        {
            const int kc = lay.kc, astr = kc + 8;
            if (tid < M * on) {
                pb = __ldg(w.b2 + or0 + tid % on);
                px = __ldcg(p.x + (long long)(tid / on) * D + or0 + tid % on);
            }
            for (int k0 = 0; k0 < FF; k0 += kc) {
                if (k0) __syncthreads();                       // the previous chunk has been consumed
                load_act(p.ffh, M, FF, k0, kc, ACT, astr, tid);
                __syncthreads();
                if (k0 == 0) ST_STAMP(0);
                if (on > 0) {
                    if (k0 == 0) { mbar_wait(&bars[1], par2); par2 ^= 1; ST_STAMP(1); }
                    slice_gemm(ACT, astr, M, S2, wsF, k0, kc, (on + 7) >> 3, RED, k0 != 0);
                    ST_STAMP(4);
                }
            }
            __syncthreads();
            ST_STAMP(2);
            for (int e = tid; e < M * on; e += ST_THREADS) {
                const int m = e / on, j = e - m * on, col = or0 + j;
                float* xp = p.x + (long long)m * D + col;
                const float xv = e == tid ? (red_sum(RED, m, j, wm) + pb) + px : (red_sum(RED, m, j, wm) + __ldg(w.b2 + col)) + __ldcg(xp);
                if (!(lay.dbg & 1)) *xp = xv;
            }
            ST_STAMP(3);
        }
        grid_barrier(p.bar, base + ++epoch, G, [&] {
            if (!more || lane != 0) return;
            if (has_attn) attn_issue(p.a, ge, p.layers[l + 1], ah, ATT, &bars[3]);   // next layer's ring / rel-pos rows
        }, arr ? arr + 2 * G * 4 : nullptr);
        if (p.trace && cta == 0 && tid == 0) p.trace[epoch] = gtime();
    }
    // after_norm -> encoder output rows (fp32), one row per CTA
    if (cta < M && warp == 0) {
        const int nv = D >> 7;
        const float4* xr = reinterpret_cast<const float4*>(p.x + (long long)cta * D);
        float4 v[8];
        float s = 0.f;
#pragma unroll
        for (int i = 0; i < 8; ++i)
            if (i < nv) v[i] = __ldcg(xr + i * 32 + lane);
#pragma unroll
        for (int i = 0; i < 8; ++i)
            if (i < nv) s += v[i].x + v[i].y + v[i].z + v[i].w;
        const float mu = warp_sum(s) / D;
        float q = 0.f;
#pragma unroll
        for (int i = 0; i < 8; ++i)
            if (i < nv) {
                const float a = v[i].x - mu, b = v[i].y - mu, c = v[i].z - mu, d = v[i].w - mu;
                q += a * a + b * b + c * c + d * d;
            }
        const float rstd = rsqrtf(warp_sum(q) / D + 1e-5f);
#pragma unroll
        for (int i = 0; i < 8; ++i)
            if (i < nv) {
                const int col = (i * 32 + lane) * 4;
                const float4 gg = __ldg(reinterpret_cast<const float4*>(p.after_g + col));
                const float4 bb = __ldg(reinterpret_cast<const float4*>(p.after_b + col));
                *reinterpret_cast<float4*>(p.enc_out + (long long)cta * D + col) =
                    make_float4((v[i].x - mu) * rstd * gg.x + bb.x, (v[i].y - mu) * rstd * gg.y + bb.y,
                                (v[i].z - mu) * rstd * gg.z + bb.z, (v[i].w - mu) * rstd * gg.w + bb.w);
            }
    }
    if (tid == 0) p.bar[cta] = base + epoch;              // the next launch continues the barrier numbering from here
    if (p.trace && cta == 0 && tid == 0) p.trace[epoch + 1] = gtime();
}

}  // namespace

// Shared-memory plan of the kernel for a step shape on a device of G SMs with smem_max bytes per CTA; false = the step does
// not qualify (pure host logic: fo_debug_stack_plan exposes it to the CPU tests).
static bool stack_layout(int D, int FF, int H, int n, int t, int window, int L, int G, int smem_max, StackLayout* lay, int* smem) {
    const int M = n * t;
    if (G < 1 || M < 1 || M > STACK_MAX_ROWS || t > 8 || H * DK != D || D % 128 || D > 1024 || FF % 128 || FF > 4096 ||
        n * H > G || window + t > 128 || L < 1)
        return false;
    auto cdivi = [](int x, int y) { return (x + y - 1) / y; };
    const int rowD = D * 2 + 16, rowF = FF * 2 + 16;
    const int r1 = std::max(cdivi(3 * D, G), cdivi(FF, G)), r2 = cdivi(D, G);
    if (r1 > 8 * MAXG || r2 > 8 * MAXG) return false;
    int off = 0;
    auto take = [&](int bytes) { const int o = off; off += (bytes + 127) & ~127; return o; };
    lay->s1 = take(r1 * rowD);
    lay->s2 = take(r2 * rowF);
    lay->s3 = take(r2 * rowD);
    lay->act_bytes = M * rowD;
    // FFN2's activation rows (M x FF fp16) pass through the same buffer in K chunks (a multiple of 128 columns each)
    int kc = FF;
    while (kc > 128 && (M * (kc * 2 + 16) > std::max(lay->act_bytes, 33024) || FF % kc)) kc -= 128;
    lay->kc = kc;
    lay->dbg = 0;
    lay->act_bytes = std::max(lay->act_bytes, M * (kc * 2 + 16));
    lay->act = take(lay->act_bytes);
    lay->red = take(ST_WARPS * MAXG * 128 * 4);
    lay->attn = take(mma_unit_layout(window, t).bytes);
    *smem = off;
    return off <= smem_max;
}

int stack_plan(int D, int FF, int H, int n, int t, int window, int L, int sms, int smem_max, int* smem_bytes, int* ffn2_chunk,
               int* rows_qkv, int* rows_ffn1, int* rows_out) {
    StackLayout lay;
    int smem = 0;
    if (!stack_layout(D, FF, H, n, t, window, L, sms, smem_max, &lay, &smem)) return 1;
    *smem_bytes = smem;
    *ffn2_chunk = lay.kc;
    *rows_qkv = (3 * D + sms - 1) / sms;
    *rows_ffn1 = (FF + sms - 1) / sms;
    *rows_out = (D + sms - 1) / sms;
    return 0;
}

int stream_stack(const StackArgs& a, int G, int smem_max, cudaStream_t st) {
    StackLayout lay;
    int smem = 0;
    if (!stack_layout(a.D, a.FF, a.a.H, a.a.n, a.a.t, a.a.window, a.L, G, smem_max, &lay, &smem)) return 1;
    static int dbg = -1;
    if (dbg < 0) { const char* e = getenv("FO_STACK_DBG"); dbg = e ? atoi(e) : 0; }
    lay.dbg = dbg;
    // the kernel's shared-memory opt-in only grows, per device, under a lock: contexts of different SM counts (hence layouts)
    // may launch from several host threads
    {
        static std::mutex mu;
        static std::map<int, int> attr_smem;
        int dev = 0;
        FO_CUDA(cudaGetDevice(&dev));
        std::lock_guard<std::mutex> lk(mu);
        if (smem > attr_smem[dev]) {
            FO_CUDA(cudaFuncSetAttribute(stream_stack_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
            attr_smem[dev] = smem;
        }
    }
    // the G CTAs wait on each other at the grid barriers: one must fit every SM of the group
    int occ = 0;
    FO_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, stream_stack_kernel, ST_THREADS, smem));
    if (occ < 1) return 1;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(G);
    cfg.blockDim = dim3(ST_THREADS);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeCooperative;
    attr[0].val.cooperative = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    FO_CUDA(cudaLaunchKernelEx(&cfg, stream_stack_kernel, a, lay));
    FO_LAUNCHED();
    return 0;
}

}  // namespace fo
