// Chunk attention with key-position rel-pos bias (reference: MultiHeadedAttention.infer / .forward,
// models/encoder/attention.py:407-459 / 350-405; no rel_shift, SURVEY 2.4-3):
//     score[i][j] = ((q_i + u) . K_j + (q_i + v) . P[pos_j]) / sqrt(d_k),   softmax over j,   out = sum_j p_ij V_j
// d_k is 64.  Streaming: one CTA per (session, head); the cached K/V rows come from the session's ring in
// HBM with cp.async.bulk (TMA bulk copy, mbarrier completion) while the chunk's own rows arrive from the
// fused QKV GEMM output and are appended to the ring in the same pass.  Offline: one CTA per
// (utterance, head, 4 query rows); the band [start,end) of models/masks.py:50-56 and the pad mask are
// evaluated arithmetically, never materialised; key tiles + online softmax cover unbounded left context.
#include <stdlib.h>

#include <algorithm>

#include "fo_common.cuh"

namespace fo {


namespace {

constexpr int DK = 64;
constexpr int TQ_MAX = STREAM_MAX_T;   // query rows per CTA (streaming chunk: 4, fork: 7)
constexpr int ATT_THREADS = 128;

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "WAIT_LOOP:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra DONE;\n\t"
        "bra WAIT_LOOP;\n\t"
        "DONE:\n\t}" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(dst)),
                 "l"(src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}

template <typename TA> struct Chunk;        // one 16-byte slice of a 64-wide row
template <> struct Chunk<float> {
    static constexpr int EPC = 4, NCH = 16;
    static __device__ __forceinline__ void load(const float* p, float (&v)[4]) {
        float4 t = *reinterpret_cast<const float4*>(p);
        v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
    }
};
template <> struct Chunk<__half> {
    static constexpr int EPC = 8, NCH = 8;
    static __device__ __forceinline__ void load(const __half* p, float (&v)[8]) {
        uint4 t = *reinterpret_cast<const uint4*>(p);
        const __half2* h = reinterpret_cast<const __half2*>(&t);
#pragma unroll
        for (int i = 0; i < 4; ++i) { const float2 f = __half22float2(h[i]); v[2 * i] = f.x; v[2 * i + 1] = f.y; }
    }
};
template <> struct Chunk<bf16> {
    static constexpr int EPC = 8, NCH = 8;
    static __device__ __forceinline__ void load(const bf16* p, float (&v)[8]) {
        uint4 t = *reinterpret_cast<const uint4*>(p);
        const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&t);
#pragma unroll
        for (int i = 0; i < 4; ++i) { v[2 * i] = __low2float(h[i]); v[2 * i + 1] = __high2float(h[i]); }
    }
};

// scores of key row j (smem) against nq query rows; chunk order is rotated by j so that the 8 lanes of
// one shared-memory phase touch 8 different 16-byte bank groups (rows are 128 B / 256 B apart).
template <typename TA>
__device__ __forceinline__ void score_row(const TA* Krow, const TA* Prow, const float* qu, const float* qv, int nq,
                                          int rot, float (&acc)[TQ_MAX]) {
    constexpr int EPC = Chunk<TA>::EPC, NCH = Chunk<TA>::NCH;
#pragma unroll
    for (int i = 0; i < TQ_MAX; ++i) acc[i] = 0.f;
#pragma unroll 2
    for (int c = 0; c < NCH; ++c) {
        const int cc = (c + rot) & (NCH - 1);
        float kv[EPC], pv[EPC];
        Chunk<TA>::load(Krow + cc * EPC, kv);
        Chunk<TA>::load(Prow + cc * EPC, pv);
#pragma unroll
        for (int i = 0; i < TQ_MAX; ++i) {
            if (i < nq) {
                const float* a = qu + i * DK + cc * EPC;
                const float* b = qv + i * DK + cc * EPC;
                float s = acc[i];
#pragma unroll
                for (int e = 0; e < EPC; ++e) s = fmaf(a[e], kv[e], fmaf(b[e], pv[e], s));
                acc[i] = s;
            }
        }
    }
}

__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// ---------------------------------------------------------------------------------------------
// Streaming chunk attention (fp32 contexts; the fp16 variant below runs the contractions on mma.sync), one CTA per
// (session, head), 4 warps.  Steady state: 64 cached + 4 new keys, 4 queries.
//   load   thread 0 starts the bulk copies of the ring's K/V rows (HBM -> smem, mbarrier); meanwhile every thread
//          fetches its share of the chunk's own K/V rows (appended to the ring in the same pass), the rel-pos rows
//          P_l[start + j] and Q, all issued before the first use so that one memory latency covers them
//   score  warp = query row, lane = keys lane, lane+32, lane+64: ((q+u).K_j + (q+v).P_j)/8 with the 16-byte chunks
//          of a row visited in a lane-rotated order (conflict-free); scores stay in registers
//   soft   warp-shuffle max / sum in fp32, probabilities to a 1 KB smem strip
//   PV     lane = output dims (2*lane, 2*lane+1), loop over the keys
// smem rows are sized by window + t (68), not by the ring capacity, so 7 CTAs fit per SM and the 1024 CTAs of a
// 64-session layer are ONE wave.
template <typename TA>
__global__ void __launch_bounds__(ATT_THREADS, 7)
attention_stream_kernel(AttnStream a, const TA* __restrict__ qkv, const float* __restrict__ q32, TA* __restrict__ ring,
                        const TA* __restrict__ ptab_h, const float* __restrict__ pos_u, const float* __restrict__ pos_v,
                        TA* __restrict__ out) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    constexpr int EPC = Chunk<TA>::EPC, NCH = Chunk<TA>::NCH;
    FO_PDL_TRIGGER();
    FO_PDL_WAIT();
    const int cap = a.ring_cap;
    const int t = a.t, D = a.H * DK;
    const int rows = a.window + t;                  // most keys a call can see
    TA* Ks = reinterpret_cast<TA*>(smem_raw);
    TA* Vs = Ks + rows * DK;
    TA* Ps = Vs + rows * DK;                        // rel-pos rows, rounded from the fp32 table to the activation type
    float* qu = reinterpret_cast<float*>(Ps + rows * DK);
    float* qv = qu + t * DK;
    float* prob = qv + t * DK;                      // t x rows
    __shared__ __align__(8) uint64_t bar;

    const int b = blockIdx.x, h = blockIdx.y;
    const int slot = a.ids[b];
    const int nf = a.n_frames[slot];
    const int cl = min(nf, a.window);
    const int first = nf - cl;
    const int nk = cl + t;
    const int pe = a.pe_index[slot] % a.pe_wrap;
    const int start = max(0, pe - a.full_chunk);     // attention.py:112-114
    TA* ringK = ring + (long long)slot * a.ring_slot_stride + (long long)h * cap * DK;
    TA* ringV = ringK + (long long)a.H * cap * DK;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;

    // rel-pos rows P_l[start .. start+nk) of this head are contiguous in the head-major table: one bulk copy
    const int np = min(nk, a.pos_rows - start);
    if (tid == 0) {
        mbar_init(&bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        const int p0 = first % cap;
        const int len1 = min(cl, cap - p0), len2 = cl - len1;
        const uint32_t rowb = DK * sizeof(TA);
        mbar_expect_tx(&bar, (2u * cl + np) * rowb);
        bulk_g2s(Ps, ptab_h + ((long long)h * a.pos_rows + start) * DK, np * rowb, &bar);
        if (len1 > 0) {
            bulk_g2s(Ks, ringK + (long long)p0 * DK, len1 * rowb, &bar);
            bulk_g2s(Vs, ringV + (long long)p0 * DK, len1 * rowb, &bar);
        }
        if (len2 > 0) {
            bulk_g2s(Ks + len1 * DK, ringK, len2 * rowb, &bar);
            bulk_g2s(Vs + len1 * DK, ringV, len2 * rowb, &bar);
        }
    }
    // ---- loads into registers (no dependent use before they are all issued) ----
    // (a) chunk's own K/V rows: t rows x NCH chunks x {K,V}
    const int n_new = t * NCH * 2;
    uint4 newv = make_uint4(0, 0, 0, 0);
    int new_which = 0, new_r = 0, new_c = 0;
    const bool has_new = tid < n_new;                // t <= 8, NCH <= 16: n_new <= 256 -> second slot below
    if (has_new) {
        new_which = tid / (t * NCH);
        new_r = (tid / NCH) % t;
        new_c = tid % NCH;
        newv = *reinterpret_cast<const uint4*>(qkv + (long long)(b * t + new_r) * 3 * D + (new_which + 1) * D + h * DK + new_c * EPC);
    }
    // (c) Q + biases: t*64 floats, two per thread when t <= 4
    float qreg[4], ureg[4], vreg[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const int i = tid + k * ATT_THREADS;
        if (i < t * DK) {
            const int r = i / DK, d = i % DK;
            qreg[k] = q32[(long long)(b * t + r) * 3 * D + h * DK + d];
            ureg[k] = pos_u[h * DK + d];
            vreg[k] = pos_v[h * DK + d];
        }
    }
    l2_prefetch_slice(a.prefetch, blockIdx.y * gridDim.x + blockIdx.x, gridDim.x * gridDim.y, tid, ATT_THREADS);
    // ---- registers -> smem / ring ----
    if (has_new) {
        TA* sdst = (new_which ? Vs : Ks) + (cl + new_r) * DK + new_c * EPC;
        *reinterpret_cast<uint4*>(sdst) = newv;
        TA* gdst = (new_which ? ringV : ringK) + (long long)((nf + new_r) % cap) * DK + new_c * EPC;
        *reinterpret_cast<uint4*>(gdst) = newv;
    }
    for (int i = tid + ATT_THREADS; i < n_new; i += ATT_THREADS) {      // only when t*NCH*2 > 128 (fp32 context or t > 8)
        const int which = i / (t * NCH), r = (i / NCH) % t, c = i % NCH;
        const uint4 val = *reinterpret_cast<const uint4*>(qkv + (long long)(b * t + r) * 3 * D + (which + 1) * D + h * DK + c * EPC);
        *reinterpret_cast<uint4*>((which ? Vs : Ks) + (cl + r) * DK + c * EPC) = val;
        *reinterpret_cast<uint4*>((which ? ringV : ringK) + (long long)((nf + r) % cap) * DK + c * EPC) = val;
    }
    // the table holds every position a call can reach (fo_create sizes pos_rows): this clamp only keeps reads in bounds
    for (int i = tid + np * (DK / 8); i < nk * (DK / 8); i += ATT_THREADS) {
        const int j = i / (DK / 8), c = i % (DK / 8);
        const TA* src = ptab_h + ((long long)h * a.pos_rows + a.pos_rows - 1) * DK + c * 8;
#pragma unroll
        for (int e = 0; e < 8; ++e) Ps[j * DK + c * 8 + e] = src[e];
    }
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const int i = tid + k * ATT_THREADS;
        if (i < t * DK) { qu[i] = qreg[k] + ureg[k]; qv[i] = qreg[k] + vreg[k]; }
    }
    for (int i = tid + 4 * ATT_THREADS; i < t * DK; i += ATT_THREADS) {
        const int r = i / DK, d = i % DK;
        const float q = q32[(long long)(b * t + r) * 3 * D + h * DK + d];
        qu[i] = q + pos_u[h * DK + d];
        qv[i] = q + pos_v[h * DK + d];
    }
    __syncthreads();
    mbar_wait(&bar, 0);

    // ---- scores + softmax + PV: warp = query row ----
    constexpr int KPL = 4;                                // keys per lane (<= 128 keys per call)
    for (int i = warp; i < t; i += ATT_THREADS / 32) {
        const float* qui = qu + i * DK;
        const float* qvi = qv + i * DK;
        float sc[KPL];
#pragma unroll
        for (int k = 0; k < KPL; ++k) sc[k] = 0.f;
#pragma unroll 2
        for (int c = 0; c < NCH; ++c) {
            const int cc = (c + lane) & (NCH - 1);
            float au[EPC], av[EPC];
#pragma unroll
            for (int e = 0; e < EPC; e += 4) {
                const float4 x = *reinterpret_cast<const float4*>(qui + cc * EPC + e);
                const float4 y = *reinterpret_cast<const float4*>(qvi + cc * EPC + e);
                au[e] = x.x; au[e + 1] = x.y; au[e + 2] = x.z; au[e + 3] = x.w;
                av[e] = y.x; av[e + 1] = y.y; av[e + 2] = y.z; av[e + 3] = y.w;
            }
#pragma unroll
            for (int k = 0; k < KPL; ++k) {
                const int j = lane + 32 * k;
                if (j < nk) {
                    float kv[EPC], pp[EPC];
                    Chunk<TA>::load(Ks + j * DK + cc * EPC, kv);
                    Chunk<TA>::load(Ps + j * DK + cc * EPC, pp);
                    float s = sc[k];
#pragma unroll
                    for (int e = 0; e < EPC; ++e) s = fmaf(au[e], kv[e], fmaf(av[e], pp[e], s));
                    sc[k] = s;
                }
            }
        }
        float m = -INFINITY;
#pragma unroll
        for (int k = 0; k < KPL; ++k) {
            sc[k] = (lane + 32 * k < nk) ? sc[k] * 0.125f : -INFINITY;
            m = fmaxf(m, sc[k]);
        }
        m = warp_max(m);
        float ssum = 0.f;
        float* pr = prob + i * rows;
#pragma unroll
        for (int k = 0; k < KPL; ++k) {
            const int j = lane + 32 * k;
            if (j < nk) {
                const float e = __expf(sc[k] - m);
                pr[j] = e;
                ssum += e;
            }
        }
        for (int j = lane + 32 * KPL; j < nk; j += 32) pr[j] = 0.f;      // unreachable for nk <= 128 (checked on the host)
        ssum = warp_sum(ssum);
        __syncwarp();
        const float inv = 1.f / ssum;
        float o0 = 0.f, o1 = 0.f;
        if constexpr (sizeof(TA) == 2) {
            const uint32_t* vp = reinterpret_cast<const uint32_t*>(Vs) + lane;
#pragma unroll 4
            for (int j = 0; j < nk; ++j) {
                const float p = pr[j];
                const float2 vv = unpack2<TA>(vp[j * (DK / 2)]);
                o0 = fmaf(p, vv.x, o0);
                o1 = fmaf(p, vv.y, o1);
            }
        } else {
#pragma unroll 4
            for (int j = 0; j < nk; ++j) {
                const float p = pr[j];
                o0 = fmaf(p, to_f(Vs[j * DK + 2 * lane]), o0);
                o1 = fmaf(p, to_f(Vs[j * DK + 2 * lane + 1]), o1);
            }
        }
        TA* o = out + (long long)(b * t + i) * D + h * DK + 2 * lane;
        if constexpr (sizeof(TA) == 2) {
            *reinterpret_cast<uint32_t*>(o) = pack2<TA>(o0 * inv, o1 * inv);
        } else {
            o[0] = from_f<TA>(o0 * inv);
            o[1] = from_f<TA>(o1 * inv);
        }
    }
}

// ---------------------------------------------------------------------------------------------
// fp16 variant of the streaming kernel with the two small contractions on the legacy tensor-core path
// (mma.sync.m16n8k16, fp32 accumulate; the attention core is 1 % of the FLOPs, far too small for tcgen05):
//   S^T (keys x queries) = K (keys x 64) . (q+u)^T  +  P (keys x 64) . (q+v)^T     key tiles of 16 over the 4 warps
//   O^T (64 x queries)   = V^T (64 x keys) . prob^T                                   one 16-dim tile per warp
// With 4 query rows the scalar kernel spends ~13 k FMA/convert instructions per CTA on these; here they are ~60 MMAs.
// Loads, ring append, masking, fp32 softmax and the outputs are as in attention_stream_kernel.  (q+u), (q+v) and the
// normalised probabilities are rounded to fp16 for the MMAs.
__device__ __forceinline__ void mma16816(float (&d)[4], const uint32_t (&a)[4], const uint32_t (&b)[2]) {
    asm volatile(
        "mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
        : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
        : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b[0]), "r"(b[1]));
}
__device__ __forceinline__ uint32_t lds32(const __half* p) { return *reinterpret_cast<const uint32_t*>(p); }
#ifdef FO_TC_TRACE_BUILD
__device__ unsigned long long g_attn_trace[16];
#define AT_TRACE(slot)                                                                                   \
    do {                                                                                                 \
        if (threadIdx.x == 0 && blockIdx.x == gridDim.x / 2 && blockIdx.y == 0) {                        \
            unsigned long long t_;                                                                       \
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_));                                       \
            g_attn_trace[slot] = t_;                                                                     \
        }                                                                                                \
    } while (0)
#else
#define AT_TRACE(slot) do { } while (0)
#endif

template <bool DEFER>            // DEFER: q / k / v of the chunk are summed from the QKV GEMM's split-K partials (AttnStream::part)
__global__ void __launch_bounds__(ATT_THREADS, 7)
attention_stream_mma_kernel(AttnStream a, const __half* __restrict__ qkv, const float* __restrict__ q32,
                            __half* __restrict__ ring, const __half* __restrict__ ptab_h, const float* __restrict__ pos_u,
                            const float* __restrict__ pos_v, __half* __restrict__ out) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    typedef __half TA;
    constexpr int EPC = 8, NCH = 8;
    AT_TRACE(0);
    FO_TR_DECL();
    if (threadIdx.x == 0) FO_TR_STAMP(0);
    FO_PDL_TRIGGER();
    // Everything up to FO_PDL_WAIT below touches only data that no kernel of THIS step has written before this launch:
    // the session state (advance_sessions runs at the end of a step, and a step starts with stream copies, which order
    // it after the previous step completely), the ring rows of earlier frames (appended by this kernel, this layer, in
    // earlier steps) and constants.  So the ring / rel-pos bulk copies fly while the QKV GEMM is still draining.
    AT_TRACE(1);
    const int cap = a.ring_cap;
    const int t = a.t, D = a.H * DK;
    const int rows = a.window + t;                  // K / P rows held; a partial last key tile reads on into the next
    const int vrows = (rows + 15) & ~15;            // array (finite or masked); V is padded with zero rows instead
    TA* Ks = reinterpret_cast<TA*>(smem_raw);
    TA* Ps = Ks + rows * DK;
    TA* Vs = Ps + rows * DK;
    TA* quh = Vs + vrows * DK;                      // (q+u), (q+v) as fp16, t x 64 each
    TA* qvh = quh + t * DK;
    TA* ph = qvh + t * DK;                          // normalised probabilities, t x vrows
    float* sc = reinterpret_cast<float*>(ph + t * vrows);   // scores t x vrows (fp32); later the output tile t x 64
    __shared__ __align__(8) uint64_t bar;

    const int b = blockIdx.x, h = blockIdx.y;
    const int slot = a.ids[b];
    const int nf = a.n_frames[slot];
    const int cl = min(nf, a.window);
    const int first = nf - cl;
    const int nk = cl + t;
    const int pe = a.pe_index[slot] % a.pe_wrap;
    const int start = max(0, pe - a.full_chunk);     // attention.py:112-114
    TA* ringK = ring + (long long)slot * a.ring_slot_stride + (long long)h * cap * DK;
    TA* ringV = ringK + (long long)a.H * cap * DK;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;

    const int np = min(nk, a.pos_rows - start);
    AT_TRACE(2);
    if (tid == 0) {
        mbar_init(&bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        const int p0 = first % cap;
        const int len1 = min(cl, cap - p0), len2 = cl - len1;
        const uint32_t rowb = DK * sizeof(TA);
        mbar_expect_tx(&bar, (2u * cl + np) * rowb);
        bulk_g2s(Ps, ptab_h + ((long long)h * a.pos_rows + start) * DK, np * rowb, &bar);
        if (len1 > 0) {
            bulk_g2s(Ks, ringK + (long long)p0 * DK, len1 * rowb, &bar);
            bulk_g2s(Vs, ringV + (long long)p0 * DK, len1 * rowb, &bar);
        }
        if (len2 > 0) {
            bulk_g2s(Ks + len1 * DK, ringK, len2 * rowb, &bar);
            bulk_g2s(Vs + len1 * DK, ringV, len2 * rowb, &bar);
        }
    }
    AT_TRACE(3);
    float ureg[4], vreg[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const int i = tid + k * ATT_THREADS;
        if (i < t * DK) {
            ureg[k] = pos_u[h * DK + i % DK];
            vreg[k] = pos_v[h * DK + i % DK];
        }
    }
    FO_PDL_WAIT();                                  // from here on: the QKV GEMM's output
    if (threadIdx.x == 0) FO_TR_STAMP(1);
    // chunk's own K/V rows -> registers
    const int n_new = t * NCH * 2;
    uint4 newv = make_uint4(0, 0, 0, 0);
    int new_which = 0, new_r = 0, new_c = 0;
    const bool has_new = tid < n_new;
    // one 16-byte chunk (8 dims) of a new K / V row: from the finished fp16 rows, or summed from the QKV GEMM's split-K partials
    auto load_new = [&](int which, int r, int cc) -> uint4 {
        const long long off = (long long)(b * t + r) * 3 * D + (which + 1) * D + h * DK + cc * EPC;
        if constexpr (!DEFER) return *reinterpret_cast<const uint4*>(qkv + off);
        float4 lo = make_float4(0.f, 0.f, 0.f, 0.f), hi = lo;
        for (int sp = 0; sp < a.nsplit; ++sp) {
            const float4 p0 = __ldcg(reinterpret_cast<const float4*>(a.part + sp * a.part_stride + off));
            const float4 p1 = __ldcg(reinterpret_cast<const float4*>(a.part + sp * a.part_stride + off + 4));
            lo.x += p0.x; lo.y += p0.y; lo.z += p0.z; lo.w += p0.w;
            hi.x += p1.x; hi.y += p1.y; hi.z += p1.z; hi.w += p1.w;
        }
        const float* bp = a.part_bias + (which + 1) * D + h * DK + cc * EPC;
        uint4 o;
        o.x = pack2<TA>(lo.x + bp[0], lo.y + bp[1]); o.y = pack2<TA>(lo.z + bp[2], lo.w + bp[3]);
        o.z = pack2<TA>(hi.x + bp[4], hi.y + bp[5]); o.w = pack2<TA>(hi.z + bp[6], hi.w + bp[7]);
        return o;
    };
    auto load_q = [&](int r, int d) -> float {
        const long long off = (long long)(b * t + r) * 3 * D + h * DK + d;
        if constexpr (!DEFER) return q32[off];
        float acc = 0.f;
        for (int sp = 0; sp < a.nsplit; ++sp) acc += __ldcg(a.part + sp * a.part_stride + off);
        return acc + a.part_bias[h * DK + d];
    };
    if (has_new) {
        new_which = tid / (t * NCH);
        new_r = (tid / NCH) % t;
        new_c = tid % NCH;
        newv = load_new(new_which, new_r, new_c);
    }
    float qreg[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const int i = tid + k * ATT_THREADS;
        if (i < t * DK) {
            const int r = i / DK, d = i % DK;
            qreg[k] = load_q(r, d);
        }
    }
    l2_prefetch_slice(a.prefetch, blockIdx.y * gridDim.x + blockIdx.x, gridDim.x * gridDim.y, tid, ATT_THREADS);
    // 16-byte chunk c of the row of frame f lives at chunk c ^ (f & 7) (kv_swz): rows that the MMA fragment loads read
    // together then sit in different banks, although the bulk copies land the rows densely (128 B apart)
    if (has_new) {
        const int pc = new_c ^ ((nf + new_r) & 7);
        *reinterpret_cast<uint4*>((new_which ? Vs : Ks) + (cl + new_r) * DK + pc * EPC) = newv;
        *reinterpret_cast<uint4*>((new_which ? ringV : ringK) + (long long)((nf + new_r) % cap) * DK + pc * EPC) = newv;
    }
    for (int i = tid + ATT_THREADS; i < n_new; i += ATT_THREADS) {      // t > 8 only
        const int which = i / (t * NCH), r = (i / NCH) % t, c = i % NCH;
        const uint4 val = load_new(which, r, c);
        const int pc = c ^ ((nf + r) & 7);
        *reinterpret_cast<uint4*>((which ? Vs : Ks) + (cl + r) * DK + pc * EPC) = val;
        *reinterpret_cast<uint4*>((which ? ringV : ringK) + (long long)((nf + r) % cap) * DK + pc * EPC) = val;
    }
    // zero rows of V behind the last key (they enter the PV MMAs with probability 0: they must be finite)
    for (int i = tid; i < (vrows - nk) * NCH; i += ATT_THREADS)
        *reinterpret_cast<uint4*>(Vs + (nk + i / NCH) * DK + (i % NCH) * EPC) = make_uint4(0, 0, 0, 0);
    for (int i = tid + np * NCH; i < nk * NCH; i += ATT_THREADS) {       // in-bounds clamp only: pos_rows covers every reachable position
        const int j = i / NCH, c = i % NCH;
        *reinterpret_cast<uint4*>(Ps + j * DK + (c ^ ((start + j) & 7)) * EPC) =
            *reinterpret_cast<const uint4*>(ptab_h + ((long long)h * a.pos_rows + a.pos_rows - 1) * DK + (c ^ ((a.pos_rows - 1) & 7)) * EPC);
    }
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const int i = tid + k * ATT_THREADS;
        if (i < t * DK) {
            const int r = i / DK, d = i % DK;
            const int o = r * DK + (((d >> 3) ^ (r & 7)) << 3) + (d & 7);      // same chunk swizzle, keyed by the query row
            quh[o] = from_f<TA>(qreg[k] + ureg[k]);
            qvh[o] = from_f<TA>(qreg[k] + vreg[k]);
        }
    }
    for (int i = tid + 4 * ATT_THREADS; i < t * DK; i += ATT_THREADS) {
        const int r = i / DK, d = i % DK;
        const float q = load_q(r, d);
        const int o = r * DK + (((d >> 3) ^ (r & 7)) << 3) + (d & 7);
        quh[o] = from_f<TA>(q + pos_u[h * DK + d]);
        qvh[o] = from_f<TA>(q + pos_v[h * DK + d]);
    }
    AT_TRACE(4);
    __syncthreads();
    mbar_wait(&bar, 0);
    AT_TRACE(5);
    if (threadIdx.x == 0) FO_TR_STAMP(2);

    const int g = lane >> 2, c = lane & 3;
    // ---- scores: S^T tile (16 keys x 8 queries) per MMA chain ----
    for (int k0 = warp * 16; k0 < nk; k0 += 16 * (ATT_THREADS / 32)) {
        float d[4] = {0.f, 0.f, 0.f, 0.f};
        // swizzle keys of the rows this lane reads: K rows by frame number, P rows by position, q rows by query index
        const int kk0 = (first + k0 + g) & 7, kk1 = (first + k0 + g + 8) & 7;
        const int kp0 = (start + k0 + g) & 7, kp1 = (start + k0 + g + 8) & 7;
        const TA* kr0 = Ks + (k0 + g) * DK + c * 2;
        const TA* kr1 = Ks + (k0 + g + 8) * DK + c * 2;
        const TA* pr0 = Ps + (k0 + g) * DK + c * 2;
        const TA* pr1 = Ps + (k0 + g + 8) * DK + c * 2;
#pragma unroll
        for (int ks = 0; ks < DK / 16; ++ks) {
            const int c0 = ks * 2, c1 = ks * 2 + 1;                 // the two 16-byte chunks of this k step
            uint32_t af[4], bf[2];
            af[0] = lds32(kr0 + ((c0 ^ kk0) << 3));
            af[1] = lds32(kr1 + ((c0 ^ kk1) << 3));
            af[2] = lds32(kr0 + ((c1 ^ kk0) << 3));
            af[3] = lds32(kr1 + ((c1 ^ kk1) << 3));
            bf[0] = g < t ? lds32(quh + g * DK + ((c0 ^ g) << 3) + c * 2) : 0u;
            bf[1] = g < t ? lds32(quh + g * DK + ((c1 ^ g) << 3) + c * 2) : 0u;
            mma16816(d, af, bf);
            af[0] = lds32(pr0 + ((c0 ^ kp0) << 3));
            af[1] = lds32(pr1 + ((c0 ^ kp1) << 3));
            af[2] = lds32(pr0 + ((c1 ^ kp0) << 3));
            af[3] = lds32(pr1 + ((c1 ^ kp1) << 3));
            bf[0] = g < t ? lds32(qvh + g * DK + ((c0 ^ g) << 3) + c * 2) : 0u;
            bf[1] = g < t ? lds32(qvh + g * DK + ((c1 ^ g) << 3) + c * 2) : 0u;
            mma16816(d, af, bf);
        }
        const int q0 = c * 2;
        if (q0 < t) { sc[q0 * vrows + k0 + g] = d[0] * 0.125f; sc[q0 * vrows + k0 + g + 8] = d[2] * 0.125f; }
        if (q0 + 1 < t) { sc[(q0 + 1) * vrows + k0 + g] = d[1] * 0.125f; sc[(q0 + 1) * vrows + k0 + g + 8] = d[3] * 0.125f; }
    }
    __syncthreads();
    AT_TRACE(6);
    // ---- softmax (fp32), probabilities normalised and rounded to fp16 ----
    for (int i = warp; i < t; i += ATT_THREADS / 32) {
        float sv[4];
        float m = -INFINITY;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const int j = lane + 32 * k;
            sv[k] = j < nk ? sc[i * vrows + j] : -INFINITY;
            m = fmaxf(m, sv[k]);
        }
        m = warp_max(m);
        float ssum = 0.f;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            sv[k] = (lane + 32 * k < nk) ? __expf(sv[k] - m) : 0.f;
            ssum += sv[k];
        }
        ssum = warp_sum(ssum);
        const float inv = 1.f / ssum;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const int j = lane + 32 * k;
            if (j < vrows) ph[i * vrows + j] = __float2half_rn(sv[k] * inv);
        }
    }
    __syncthreads();
    AT_TRACE(7);
    // ---- PV: O^T tile (16 dims x 8 queries) per warp ----
    {
        float d[4] = {0.f, 0.f, 0.f, 0.f};
        const int dim0 = warp * 16;
        const int mi = lane >> 3, r = lane & 7;
        for (int key0 = 0; key0 < nk; key0 += 16) {
            uint32_t af[4], bf[2];
            const int vrow = key0 + r + ((mi & 2) ? 8 : 0);
            const TA* ap = Vs + vrow * DK + ((((dim0 >> 3) + (mi & 1)) ^ ((first + vrow) & 7)) << 3);
            const uint32_t saddr = smem_u32(ap);
            asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];"
                         : "=r"(af[0]), "=r"(af[1]), "=r"(af[2]), "=r"(af[3])
                         : "r"(saddr));
            bf[0] = g < t ? lds32(ph + g * vrows + key0 + c * 2) : 0u;
            bf[1] = g < t ? lds32(ph + g * vrows + key0 + 8 + c * 2) : 0u;
            mma16816(d, af, bf);
        }
        const int q0 = c * 2;
        if (q0 < t) { sc[q0 * DK + dim0 + g] = d[0]; sc[q0 * DK + dim0 + g + 8] = d[2]; }
        if (q0 + 1 < t) { sc[(q0 + 1) * DK + dim0 + g] = d[1]; sc[(q0 + 1) * DK + dim0 + g + 8] = d[3]; }
    }
    __syncthreads();
    AT_TRACE(8);
    for (int i = tid; i < t * (DK / 2); i += ATT_THREADS) {
        const int q = i / (DK / 2), pr = i % (DK / 2);
        *reinterpret_cast<uint32_t*>(out + (long long)(b * t + q) * D + h * DK + 2 * pr) =
            pack2<__half>(sc[q * DK + 2 * pr], sc[q * DK + 2 * pr + 1]);
    }
    AT_TRACE(9);
    if (threadIdx.x == 0) { FO_TR_STAMP(3); FO_TR_STAMP(4); FO_TR_FLUSH(2, 0); }
}

// ---------------------------------------------------------------------------------------------
// Several consecutive chunks of every session in one call (AttnStream::chunks = k, fo_encode_stream_chunks).  One CTA per
// (session, head) stages the keys once -- the ring window of frames [first, nf) (first = nf - min(nf, window)) by bulk
// copy, then the call's own k*t rows -- and walks the k query chunks in order.  Chunk j sees exactly what the j-th
// sequential single-chunk call would see:
//     nf_j = nf + j*t,  keys = frames [nf_j - min(nf_j, window), nf_j + t)   (a contiguous run of the staged rows)
//     pe_j = pe_index stepped j times by pe = pe % wrap + chunk_size,  rel-pos rows P[max(0, pe_j % wrap - full_chunk) + m]
// The rel-pos window moves (and may wrap) with pe_j, so it is re-staged per chunk.  The new rows go to the ring only after
// the staged copy of the old window has landed: the ring holds window + max_t rows, fewer than the call's keys, so a later
// chunk's rows would overwrite frames an earlier chunk still needs.  Layouts (fp16 chunk swizzle of K/V by frame and of P
// by position, q swizzled by query row) are those of the single-chunk kernels.
__device__ __forceinline__ int chunk_pe(int pe, int j, const AttnStream& a) {
    for (int i = 0; i < j; ++i) pe = pe % a.pe_wrap + a.chunk_size;
    return pe % a.pe_wrap;
}

// stage the call's new K/V rows (smem rows cl + r, frame nf + r) and, once the ring window has landed, append them to the
// ring (only the last `cap` of them when the call brings more frames than the ring holds)
template <typename TA, int NCH, bool SWZ>
__device__ __forceinline__ void chunks_stage_new(const AttnStream& a, const TA* qkv, TA* Ks, TA* Vs, int b, int h, int nf, int cl,
                                                 int kt) {
    constexpr int EPC = 16 / sizeof(TA);
    const int D = a.H * DK;
    for (int i = threadIdx.x; i < kt * NCH * 2; i += ATT_THREADS) {
        const int which = i / (kt * NCH), r = (i / NCH) % kt, c = i % NCH;
        const int pc = SWZ ? (c ^ ((nf + r) & 7)) : c;
        *reinterpret_cast<uint4*>((which ? Vs : Ks) + (cl + r) * DK + pc * EPC) =
            *reinterpret_cast<const uint4*>(qkv + (long long)(b * kt + r) * 3 * D + (which + 1) * D + h * DK + c * EPC);
    }
}
template <typename TA, int NCH>
__device__ __forceinline__ void chunks_append_ring(const AttnStream& a, const TA* Ks, const TA* Vs, TA* ringK, TA* ringV, int nf,
                                                   int cl, int kt) {
    constexpr int EPC = 16 / sizeof(TA);
    const int r0 = max(0, kt - a.ring_cap);
    for (int i = threadIdx.x; i < (kt - r0) * NCH * 2; i += ATT_THREADS) {
        const int which = i / ((kt - r0) * NCH), r = r0 + (i / NCH) % (kt - r0), c = i % NCH;
        *reinterpret_cast<uint4*>((which ? ringV : ringK) + (long long)((nf + r) % a.ring_cap) * DK + c * EPC) =
            *reinterpret_cast<const uint4*>((which ? Vs : Ks) + (cl + r) * DK + c * EPC);
    }
}
__device__ __forceinline__ void chunks_start_ring_copy(const void* ringK, const void* ringV, void* Ks, void* Vs, int first, int cl,
                                                       int cap, uint32_t rowb, uint64_t* bar) {
    mbar_init(bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    const int p0 = first % cap;
    const int len1 = min(cl, cap - p0), len2 = cl - len1;
    mbar_expect_tx(bar, 2u * cl * rowb);
    if (len1 > 0) {
        bulk_g2s(Ks, (const char*)ringK + (long long)p0 * rowb, len1 * rowb, bar);
        bulk_g2s(Vs, (const char*)ringV + (long long)p0 * rowb, len1 * rowb, bar);
    }
    if (len2 > 0) {
        bulk_g2s((char*)Ks + len1 * rowb, ringK, len2 * rowb, bar);
        bulk_g2s((char*)Vs + len1 * rowb, ringV, len2 * rowb, bar);
    }
}

// fp32 (parity) form: scalar FFMA contractions as in attention_stream_kernel
template <typename TA>
__global__ void __launch_bounds__(ATT_THREADS)
attention_chunks_kernel(AttnStream a, const TA* __restrict__ qkv, const float* __restrict__ q32, TA* __restrict__ ring,
                        const TA* __restrict__ ptab_h, const float* __restrict__ pos_u, const float* __restrict__ pos_v,
                        TA* __restrict__ out) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    constexpr int EPC = Chunk<TA>::EPC, NCH = Chunk<TA>::NCH;
    FO_PDL_TRIGGER();
    FO_PDL_WAIT();
    const int cap = a.ring_cap, t = a.t, kt = a.chunks * t, D = a.H * DK;
    const int rows = a.window + kt, prow = a.window + t;
    TA* Ks = reinterpret_cast<TA*>(smem_raw);
    TA* Vs = Ks + rows * DK;
    TA* Ps = Vs + rows * DK;
    float* qu = reinterpret_cast<float*>(Ps + prow * DK);
    float* qv = qu + t * DK;
    float* prob = qv + t * DK;                      // t x prow
    __shared__ __align__(8) uint64_t bar;

    const int b = blockIdx.x, h = blockIdx.y;
    const int slot = a.ids[b];
    const int nf = a.n_frames[slot];
    const int cl = min(nf, a.window), first = nf - cl;
    TA* ringK = ring + (long long)slot * a.ring_slot_stride + (long long)h * cap * DK;
    TA* ringV = ringK + (long long)a.H * cap * DK;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    if (tid == 0) chunks_start_ring_copy(ringK, ringV, Ks, Vs, first, cl, cap, DK * sizeof(TA), &bar);
    chunks_stage_new<TA, NCH, false>(a, qkv, Ks, Vs, b, h, nf, cl, kt);
    __syncthreads();
    mbar_wait(&bar, 0);
    chunks_append_ring<TA, NCH>(a, Ks, Vs, ringK, ringV, nf, cl, kt);

    const int pe0 = a.pe_index[slot];
    for (int j = 0; j < a.chunks; ++j) {
        const int nfj = nf + j * t, clj = min(nfj, a.window);
        const int o = nfj - clj - first;            // staged row of this chunk's first key
        const int nk = clj + t;
        const int start = max(0, chunk_pe(pe0, j, a) - a.full_chunk);
        for (int i = tid; i < nk * NCH; i += ATT_THREADS) {        // the min() keeps reads in bounds; pos_rows covers every reachable position
            const int r = i / NCH, c = i % NCH, pos = min(start + r, a.pos_rows - 1);
            *reinterpret_cast<uint4*>(Ps + r * DK + c * EPC) = *reinterpret_cast<const uint4*>(ptab_h + ((long long)h * a.pos_rows + pos) * DK + c * EPC);
        }
        for (int i = tid; i < t * DK; i += ATT_THREADS) {
            const int r = i / DK, d = i % DK;
            const float q = q32[(long long)(b * kt + j * t + r) * 3 * D + h * DK + d];
            qu[i] = q + pos_u[h * DK + d];
            qv[i] = q + pos_v[h * DK + d];
        }
        __syncthreads();
        constexpr int KPL = 4;                        // keys per lane: nk <= window + t <= STREAM_CHUNKS_MAX_KEYS
        for (int i = warp; i < t; i += ATT_THREADS / 32) {
            const float* qui = qu + i * DK;
            const float* qvi = qv + i * DK;
            float sc[KPL];
#pragma unroll
            for (int k = 0; k < KPL; ++k) sc[k] = 0.f;
            for (int c = 0; c < NCH; ++c) {
                const int cc = (c + lane) & (NCH - 1);
#pragma unroll
                for (int k = 0; k < KPL; ++k) {
                    const int jj = lane + 32 * k;
                    if (jj < nk) {
                        float kv[EPC], pp[EPC];
                        Chunk<TA>::load(Ks + (o + jj) * DK + cc * EPC, kv);
                        Chunk<TA>::load(Ps + jj * DK + cc * EPC, pp);
                        float s = sc[k];
#pragma unroll
                        for (int e = 0; e < EPC; ++e) s = fmaf(qui[cc * EPC + e], kv[e], fmaf(qvi[cc * EPC + e], pp[e], s));
                        sc[k] = s;
                    }
                }
            }
            float m = -INFINITY;
#pragma unroll
            for (int k = 0; k < KPL; ++k) {
                sc[k] = (lane + 32 * k < nk) ? sc[k] * 0.125f : -INFINITY;
                m = fmaxf(m, sc[k]);
            }
            m = warp_max(m);
            float ssum = 0.f;
            float* pr = prob + i * prow;
#pragma unroll
            for (int k = 0; k < KPL; ++k) {
                const int jj = lane + 32 * k;
                if (jj < nk) {
                    const float e = __expf(sc[k] - m);
                    pr[jj] = e;
                    ssum += e;
                }
            }
            ssum = warp_sum(ssum);
            __syncwarp();
            const float inv = 1.f / ssum;
            float o0 = 0.f, o1 = 0.f;
            for (int jj = 0; jj < nk; ++jj) {
                const float p = pr[jj];
                o0 = fmaf(p, to_f(Vs[(o + jj) * DK + 2 * lane]), o0);
                o1 = fmaf(p, to_f(Vs[(o + jj) * DK + 2 * lane + 1]), o1);
            }
            TA* op = out + (long long)(b * kt + j * t + i) * D + h * DK + 2 * lane;
            op[0] = from_f<TA>(o0 * inv);
            op[1] = from_f<TA>(o1 * inv);
        }
        __syncthreads();                              // Ps / qu / prob are restaged by the next chunk
    }
}

// fp16 form: the two contractions on mma.sync as in attention_stream_mma_kernel, per query chunk (t <= 8 = the MMA's N)
__global__ void __launch_bounds__(ATT_THREADS)
attention_chunks_mma_kernel(AttnStream a, const __half* __restrict__ qkv, const float* __restrict__ q32, __half* __restrict__ ring,
                            const __half* __restrict__ ptab_h, const float* __restrict__ pos_u, const float* __restrict__ pos_v,
                            __half* __restrict__ out) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    typedef __half TA;
    constexpr int EPC = 8, NCH = 8;
    FO_PDL_TRIGGER();
    FO_PDL_WAIT();
    const int cap = a.ring_cap, t = a.t, kt = a.chunks * t, D = a.H * DK;
    const int rows = a.window + kt;
    const int krows = ((rows + 15) & ~15) + 16;     // a chunk's last key tile may read up to 15 rows past the staged keys
    const int vrows = (a.window + t + 15) & ~15;    // rel-pos rows / probability columns of one chunk
    TA* Ks = reinterpret_cast<TA*>(smem_raw);
    TA* Vs = Ks + krows * DK;
    TA* Ps = Vs + krows * DK;
    TA* quh = Ps + vrows * DK;
    TA* qvh = quh + t * DK;
    TA* ph = qvh + t * DK;                          // t x vrows
    float* sc = reinterpret_cast<float*>(ph + t * vrows);   // t x max(vrows, 64)
    __shared__ __align__(8) uint64_t bar;

    const int b = blockIdx.x, h = blockIdx.y;
    const int slot = a.ids[b];
    const int nf = a.n_frames[slot];
    const int cl = min(nf, a.window), first = nf - cl;
    const int nk_all = cl + kt;
    TA* ringK = ring + (long long)slot * a.ring_slot_stride + (long long)h * cap * DK;
    TA* ringV = ringK + (long long)a.H * cap * DK;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    if (tid == 0) chunks_start_ring_copy(ringK, ringV, Ks, Vs, first, cl, cap, DK * sizeof(TA), &bar);
    chunks_stage_new<TA, NCH, true>(a, qkv, Ks, Vs, b, h, nf, cl, kt);
    // rows behind the last key: K is masked there, V enters the PV MMAs with probability 0 and must be finite
    for (int i = tid; i < (krows - nk_all) * NCH; i += ATT_THREADS) {
        *reinterpret_cast<uint4*>(Ks + (nk_all + i / NCH) * DK + (i % NCH) * EPC) = make_uint4(0, 0, 0, 0);
        *reinterpret_cast<uint4*>(Vs + (nk_all + i / NCH) * DK + (i % NCH) * EPC) = make_uint4(0, 0, 0, 0);
    }
    __syncthreads();
    mbar_wait(&bar, 0);
    chunks_append_ring<TA, NCH>(a, Ks, Vs, ringK, ringV, nf, cl, kt);

    const int g = lane >> 2, c = lane & 3;
    const int pe0 = a.pe_index[slot];
    for (int j = 0; j < a.chunks; ++j) {
        const int nfj = nf + j * t, clj = min(nfj, a.window);
        const int o = nfj - clj - first;
        const int nk = clj + t;
        const int start = max(0, chunk_pe(pe0, j, a) - a.full_chunk);
        for (int i = tid; i < nk * NCH; i += ATT_THREADS) {        // row r = position start + r, swizzled by that position
            const int r = i / NCH, cc = i % NCH, pos = min(start + r, a.pos_rows - 1);
            *reinterpret_cast<uint4*>(Ps + r * DK + ((cc ^ ((start + r) & 7)) * EPC)) =
                *reinterpret_cast<const uint4*>(ptab_h + ((long long)h * a.pos_rows + pos) * DK + ((cc ^ (pos & 7)) * EPC));
        }
        for (int i = tid; i < t * DK; i += ATT_THREADS) {
            const int r = i / DK, d = i % DK;
            const float q = q32[(long long)(b * kt + j * t + r) * 3 * D + h * DK + d];
            const int sw = r * DK + (((d >> 3) ^ (r & 7)) << 3) + (d & 7);
            quh[sw] = from_f<TA>(q + pos_u[h * DK + d]);
            qvh[sw] = from_f<TA>(q + pos_v[h * DK + d]);
        }
        __syncthreads();
        for (int k0 = warp * 16; k0 < nk; k0 += 16 * (ATT_THREADS / 32)) {
            float d[4] = {0.f, 0.f, 0.f, 0.f};
            const int kk0 = (first + o + k0 + g) & 7, kk1 = (first + o + k0 + g + 8) & 7;
            const int kp0 = (start + k0 + g) & 7, kp1 = (start + k0 + g + 8) & 7;
            const TA* kr0 = Ks + (o + k0 + g) * DK + c * 2;
            const TA* kr1 = Ks + (o + k0 + g + 8) * DK + c * 2;
            const TA* pr0 = Ps + (k0 + g) * DK + c * 2;
            const TA* pr1 = Ps + (k0 + g + 8) * DK + c * 2;
#pragma unroll
            for (int ks = 0; ks < DK / 16; ++ks) {
                const int c0 = ks * 2, c1 = ks * 2 + 1;
                uint32_t af[4], bf[2];
                af[0] = lds32(kr0 + ((c0 ^ kk0) << 3));
                af[1] = lds32(kr1 + ((c0 ^ kk1) << 3));
                af[2] = lds32(kr0 + ((c1 ^ kk0) << 3));
                af[3] = lds32(kr1 + ((c1 ^ kk1) << 3));
                bf[0] = g < t ? lds32(quh + g * DK + ((c0 ^ g) << 3) + c * 2) : 0u;
                bf[1] = g < t ? lds32(quh + g * DK + ((c1 ^ g) << 3) + c * 2) : 0u;
                mma16816(d, af, bf);
                af[0] = lds32(pr0 + ((c0 ^ kp0) << 3));
                af[1] = lds32(pr1 + ((c0 ^ kp1) << 3));
                af[2] = lds32(pr0 + ((c1 ^ kp0) << 3));
                af[3] = lds32(pr1 + ((c1 ^ kp1) << 3));
                bf[0] = g < t ? lds32(qvh + g * DK + ((c0 ^ g) << 3) + c * 2) : 0u;
                bf[1] = g < t ? lds32(qvh + g * DK + ((c1 ^ g) << 3) + c * 2) : 0u;
                mma16816(d, af, bf);
            }
            const int q0 = c * 2;
            if (q0 < t) { sc[q0 * vrows + k0 + g] = d[0] * 0.125f; sc[q0 * vrows + k0 + g + 8] = d[2] * 0.125f; }
            if (q0 + 1 < t) { sc[(q0 + 1) * vrows + k0 + g] = d[1] * 0.125f; sc[(q0 + 1) * vrows + k0 + g + 8] = d[3] * 0.125f; }
        }
        __syncthreads();
        for (int i = warp; i < t; i += ATT_THREADS / 32) {
            float sv[4];
            float m = -INFINITY;
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const int jj = lane + 32 * k;
                sv[k] = jj < nk ? sc[i * vrows + jj] : -INFINITY;
                m = fmaxf(m, sv[k]);
            }
            m = warp_max(m);
            float ssum = 0.f;
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                sv[k] = (lane + 32 * k < nk) ? __expf(sv[k] - m) : 0.f;
                ssum += sv[k];
            }
            ssum = warp_sum(ssum);
            const float inv = 1.f / ssum;
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const int jj = lane + 32 * k;
                if (jj < vrows) ph[i * vrows + jj] = __float2half_rn(sv[k] * inv);
            }
        }
        __syncthreads();
        {
            float d[4] = {0.f, 0.f, 0.f, 0.f};
            const int dim0 = warp * 16;
            const int mi = lane >> 3, r = lane & 7;
            for (int key0 = 0; key0 < nk; key0 += 16) {
                uint32_t af[4], bf[2];
                const int vrow = o + key0 + r + ((mi & 2) ? 8 : 0);
                const TA* ap = Vs + vrow * DK + ((((dim0 >> 3) + (mi & 1)) ^ ((first + vrow) & 7)) << 3);
                const uint32_t saddr = smem_u32(ap);
                asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];"
                             : "=r"(af[0]), "=r"(af[1]), "=r"(af[2]), "=r"(af[3])
                             : "r"(saddr));
                bf[0] = g < t ? lds32(ph + g * vrows + key0 + c * 2) : 0u;
                bf[1] = g < t ? lds32(ph + g * vrows + key0 + 8 + c * 2) : 0u;
                mma16816(d, af, bf);
            }
            const int q0 = c * 2;
            if (q0 < t) { sc[q0 * DK + dim0 + g] = d[0]; sc[q0 * DK + dim0 + g + 8] = d[2]; }
            if (q0 + 1 < t) { sc[(q0 + 1) * DK + dim0 + g] = d[1]; sc[(q0 + 1) * DK + dim0 + g + 8] = d[3]; }
        }
        __syncthreads();
        for (int i = tid; i < t * (DK / 2); i += ATT_THREADS) {
            const int q = i / (DK / 2), pr = i % (DK / 2);
            *reinterpret_cast<uint32_t*>(out + (long long)(b * kt + j * t + q) * D + h * DK + 2 * pr) =
                pack2<__half>(sc[q * DK + 2 * pr], sc[q * DK + 2 * pr + 1]);
        }
        __syncthreads();                              // Ps / quh / ph / sc are restaged by the next chunk
    }
}

// ---------------------------------------------------------------------------------------------
constexpr int KT = 96;          // key tile: the shipped band of a 32-query block (64 left + 32 own keys) in one pass
constexpr int QB = 32;          // query rows per CTA
constexpr int QPW = QB / (ATT_THREADS / 32);   // queries per warp

// Full-utterance attention.  CTA = (32-query block, head, utterance), 4 warps x 8 queries.  The union of the block's
// key windows is walked in tiles of 96 keys (K, V and the rel-pos rows staged once per tile and shared by the 32
// queries; rows padded by 16 B so that lanes reading different rows hit different banks).  Scores are register
// blocked: lane = keys lane, lane+32, lane+64 of the tile against FOUR queries at a time, so every K / P chunk read
// from shared memory feeds four dot products and the query chunks are warp-wide broadcasts.  Window [start,end) of
// masks.py:50-56 and the pad mask (masks.py:110-120) are applied arithmetically; online softmax across tiles
// (unbounded left context works); PV with lane = output dims.  A row whose whole window is masked yields zeros
// (attention.py:396-397).
template <typename TA>
__global__ void __launch_bounds__(ATT_THREADS)
attention_offline_kernel(const TA* __restrict__ qkv, const float* __restrict__ q32, int T, int H,
                         const int32_t* __restrict__ ilens, int chunk, int left, const float* __restrict__ ptab,
                         const float* __restrict__ pos_u, const float* __restrict__ pos_v, TA* __restrict__ out) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    constexpr int EPC = Chunk<TA>::EPC, NCH = Chunk<TA>::NCH;
    constexpr int DKP = DK + EPC;                          // padded row (16 B): conflict-free 16-byte row reads
    constexpr int QG = 4;                                  // queries per register block
    TA* Ks = reinterpret_cast<TA*>(smem_raw);
    TA* Vs = Ks + KT * DKP;
    TA* Ps = Vs + KT * DKP;
    float* qu = reinterpret_cast<float*>(Ps + KT * DKP);   // QB x 64
    float* qv = qu + QB * DK;
    float* prob = qv + QB * DK;                            // warps x KT
    __shared__ int win[QB][2];

    const int qb = blockIdx.x, h = blockIdx.y, b = blockIdx.z;
    const int D = H * DK;
    const int q0 = qb * QB;
    const int nq = min(QB, T - q0);
    const int klen = ilens ? min(ilens[b], T) : T;        // pad mask on keys (masks.py:110-120)
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;

    if (tid < QB) {
        int s = 0, e = 0;                                  // rows past the end: empty window
        if (tid < nq) {
            const int i = q0 + tid;
            s = 0; e = T;
            if (chunk > 0) {                               // masks.py:50-56
                s = left < 0 ? 0 : max((i / chunk - left) * chunk, 0);
                e = min((i / chunk + 1) * chunk, T);
            }
            e = min(e, klen);
        }
        win[tid][0] = s;
        win[tid][1] = e;
    }
    for (int i = tid; i < QB * (DK / 4); i += ATT_THREADS) {
        const int r = i / (DK / 4), c = (i % (DK / 4)) * 4;
        float4 q = make_float4(0.f, 0.f, 0.f, 0.f);
        if (r < nq) q = *reinterpret_cast<const float4*>(q32 + ((long long)b * T + q0 + r) * 3 * D + h * DK + c);
        const float4 u = *reinterpret_cast<const float4*>(pos_u + h * DK + c);
        const float4 v = *reinterpret_cast<const float4*>(pos_v + h * DK + c);
        *reinterpret_cast<float4*>(qu + r * DK + c) = make_float4(q.x + u.x, q.y + u.y, q.z + u.z, q.w + u.w);
        *reinterpret_cast<float4*>(qv + r * DK + c) = make_float4(q.x + v.x, q.y + v.y, q.z + v.z, q.w + v.w);
    }
    __syncthreads();
    int k_lo = T, k_hi = 0;
    for (int r = 0; r < nq; ++r)
        if (win[r][1] > win[r][0]) { k_lo = min(k_lo, win[r][0]); k_hi = max(k_hi, win[r][1]); }

    float m_run[QPW], l_run[QPW], o0[QPW], o1[QPW];
#pragma unroll
    for (int qi = 0; qi < QPW; ++qi) { m_run[qi] = -INFINITY; l_run[qi] = 0.f; o0[qi] = 0.f; o1[qi] = 0.f; }
    float* pr = prob + warp * KT;

    for (int kt = k_lo; kt < k_hi; kt += KT) {
        const int nk = min(KT, k_hi - kt);
        __syncthreads();                                   // previous tile fully consumed
        for (int i = tid; i < nk * NCH * 2; i += ATT_THREADS) {
            const int which = i / (nk * NCH);              // 0 K, 1 V
            const int j = (i / NCH) % nk, c = i % NCH;
            const TA* src = qkv + ((long long)b * T + kt + j) * 3 * D + (which + 1) * D + h * DK + c * EPC;
            TA* dst = (which == 0 ? Ks : Vs) + j * DKP + c * EPC;
            *reinterpret_cast<uint4*>(dst) = *reinterpret_cast<const uint4*>(src);
        }
        for (int i = tid; i < nk * (DK / 4); i += ATT_THREADS) {
            const int j = i / (DK / 4), c = i % (DK / 4);
            const float4 v4 = *reinterpret_cast<const float4*>(ptab + (long long)(kt + j) * D + h * DK + c * 4);
            TA* d = Ps + j * DKP + c * 4;
            if constexpr (sizeof(TA) == 2) {
                uint2 hh;
                hh.x = pack2<TA>(v4.x, v4.y);
                hh.y = pack2<TA>(v4.z, v4.w);
                *reinterpret_cast<uint2*>(d) = hh;
            } else {
                *reinterpret_cast<float4*>(d) = v4;
            }
        }
        __syncthreads();
#pragma unroll
        for (int g = 0; g < QPW / QG; ++g) {
            const int rb = warp * QPW + g * QG;            // first query of the register block
            bool any = false;
#pragma unroll
            for (int q = 0; q < QG; ++q) any = any || (win[rb + q][1] > kt && win[rb + q][0] < kt + nk && win[rb + q][1] > win[rb + q][0]);
            if (!any) continue;                            // warp-uniform
            float sc[QG][3];
#pragma unroll
            for (int q = 0; q < QG; ++q) { sc[q][0] = 0.f; sc[q][1] = 0.f; sc[q][2] = 0.f; }
#pragma unroll 1
            for (int c = 0; c < NCH; ++c) {
                float au[QG][EPC], av[QG][EPC];
#pragma unroll
                for (int q = 0; q < QG; ++q)
#pragma unroll
                    for (int e = 0; e < EPC; e += 4) {     // same address in every lane: broadcast
                        const float4 x = *reinterpret_cast<const float4*>(qu + (rb + q) * DK + c * EPC + e);
                        const float4 y = *reinterpret_cast<const float4*>(qv + (rb + q) * DK + c * EPC + e);
                        au[q][e] = x.x; au[q][e + 1] = x.y; au[q][e + 2] = x.z; au[q][e + 3] = x.w;
                        av[q][e] = y.x; av[q][e + 1] = y.y; av[q][e + 2] = y.z; av[q][e + 3] = y.w;
                    }
#pragma unroll
                for (int k = 0; k < 3; ++k) {
                    const int j = lane + 32 * k;
                    if (j < nk) {
                        float kv[EPC], pp[EPC];
                        Chunk<TA>::load(Ks + j * DKP + c * EPC, kv);
                        Chunk<TA>::load(Ps + j * DKP + c * EPC, pp);
#pragma unroll
                        for (int q = 0; q < QG; ++q) {
                            float s = sc[q][k];
#pragma unroll
                            for (int e = 0; e < EPC; ++e) s = fmaf(au[q][e], kv[e], fmaf(av[q][e], pp[e], s));
                            sc[q][k] = s;
                        }
                    }
                }
            }
#pragma unroll
            for (int q = 0; q < QG; ++q) {
                const int qi = g * QG + q;
                const int lo = win[rb + q][0], hi = win[rb + q][1];
                float m = -INFINITY;
                float sq[3];
#pragma unroll
                for (int k = 0; k < 3; ++k) {
                    const int key = kt + lane + 32 * k;
                    sq[k] = (lane + 32 * k < nk && key >= lo && key < hi) ? sc[q][k] * 0.125f : -INFINITY;
                    m = fmaxf(m, sq[k]);
                }
                m = warp_max(m);
                if (m == -INFINITY) continue;              // this query sees nothing in this tile (warp-uniform)
                const float m_new = fmaxf(m_run[qi], m);
                const float corr = __expf(m_run[qi] - m_new);  // m_run = -inf -> 0
                float ssum = 0.f;
                __syncwarp();                              // previous query's PV is done with the strip
#pragma unroll
                for (int k = 0; k < 3; ++k) {
                    const int j = lane + 32 * k;
                    if (j < nk) {
                        const float e = __expf(sq[k] - m_new); // masked keys: exp(-inf) = 0
                        pr[j] = e;
                        ssum += e;
                    }
                }
                ssum = warp_sum(ssum);
                __syncwarp();
                l_run[qi] = l_run[qi] * corr + ssum;
                float a0 = o0[qi] * corr, a1 = o1[qi] * corr;
                const int j0 = max(lo - kt, 0), j1 = min(hi - kt, nk);
                if constexpr (sizeof(TA) == 2) {
                    const uint32_t* vp = reinterpret_cast<const uint32_t*>(Vs) + lane;
#pragma unroll 4
                    for (int j = j0; j < j1; ++j) {
                        const float2 vv = unpack2<TA>(vp[j * (DKP / 2)]);
                        const float p = pr[j];
                        a0 = fmaf(p, vv.x, a0);
                        a1 = fmaf(p, vv.y, a1);
                    }
                } else {
#pragma unroll 4
                    for (int j = j0; j < j1; ++j) {
                        const float p = pr[j];
                        a0 = fmaf(p, to_f(Vs[j * DKP + 2 * lane]), a0);
                        a1 = fmaf(p, to_f(Vs[j * DKP + 2 * lane + 1]), a1);
                    }
                }
                o0[qi] = a0;
                o1[qi] = a1;
                m_run[qi] = m_new;
            }
        }
    }
#pragma unroll
    for (int qi = 0; qi < QPW; ++qi) {
        const int r = warp * QPW + qi;
        if (r < nq) {
            const float inv = l_run[qi] > 0.f ? 1.f / l_run[qi] : 0.f;
            TA* o = out + ((long long)b * T + q0 + r) * D + h * DK + 2 * lane;
            if constexpr (sizeof(TA) == 2) {
                *reinterpret_cast<uint32_t*>(o) = pack2<TA>(o0[qi] * inv, o1[qi] * inv);
            } else {
                o[0] = from_f<TA>(o0[qi] * inv);
                o[1] = from_f<TA>(o1[qi] * inv);
            }
        }
    }
}

__device__ __forceinline__ void cp_async16(void* dst_smem, const void* src) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_u32(dst_smem)), "l"(src) : "memory");
}

// ---- full-utterance attention, fp16 contexts ------------------------------------------------------------------------
// Flash-attention style on mma.sync.m16n8k16: CTA = (64-query block, head, utterance), four warps x 16 queries; queries on the
// MMA-M side, so a warp's (q+u) / (q+v) fragments live in registers for the whole CTA and its probabilities go from the
// score accumulators straight into the A fragments of the PV MMAs (no score / probability tile in shared memory).  K, V and
// the rel-pos rows of a 64-key tile are staged by cp.async into a DOUBLE-buffered, XOR-swizzled tile (tile t+1 flies while
// tile t is multiplied) and read with ldmatrix (K / P rows as B fragments, V transposed).  Arithmetic as in the fp32
// kernel above: s = ((q+u).k_j + (q+v).p_j) / 8 with p_j the rel-pos row of key POSITION j (attention.py:377-388 without the
// rel_shift), band [start_i, end_i) of masks.py:50-56 and the pad mask evaluated arithmetically, fp32 online softmax,
// fully masked rows -> zeros (attention.py:396-397).
// 16-key groups outside the band of all 16 rows of a warp are skipped (5 of 8 groups remain with the shipped band).  Measured
// on the 32 x 30 s slice of BASELINE config 4: 147 us per layer launch in the pipeline, against 200 us for the first mma.sync
// kernel (32-query CTAs, keys on the MMA-M side, score / probability tiles in shared memory), which it replaces.
constexpr int FQ = 64;           // queries per CTA
constexpr int FK = 64;           // keys per tile
__device__ __forceinline__ void ldsm_x4(uint32_t (&r)[4], const __half* p) {
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(smem_u32(p)));
}
__device__ __forceinline__ void ldsm_x4_t(uint32_t (&r)[4], const __half* p) {
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(smem_u32(p)));
}
__device__ __forceinline__ void mma16816_ab(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
    asm volatile(
        "mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
        : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
        : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ float fast_exp2(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ uint32_t pack2_nosat(float a, float b) {      // values in [0, 1]: no clamp needed
    __half2 h = __floats2half2_rn(a, b);
    return *reinterpret_cast<uint32_t*>(&h);
}
__global__ void __launch_bounds__(ATT_THREADS, 4)
attention_offline_fa_kernel(const __half* __restrict__ qkv, const float* __restrict__ q32, int T, int H,
                            const int32_t* __restrict__ ilens, int chunk, int left, const __half* __restrict__ ptab_h,
                            int pos_rows, const float* __restrict__ pos_u, const float* __restrict__ pos_v,
                            __half* __restrict__ out) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    typedef __half TA;
    constexpr int NCH = 8;                                   // 16-byte chunks per 64-element row
    TA* tiles = reinterpret_cast<TA*>(smem_raw);             // [2 stages][K | P | V][FK][64]
    const int qb = blockIdx.x, h = blockIdx.y, b = blockIdx.z;
    const int D = H * DK;
    const int q0 = qb * FQ;
    const int klen = ilens ? min(ilens[b], T) : T;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int g = lane >> 2, c = lane & 3;

    // band of a query row (masks.py:50-56 + pad mask): keys [s, e)
    auto win_lo = [&](int i) { return chunk > 0 ? (left < 0 ? 0 : max((i / chunk - left) * chunk, 0)) : 0; };
    auto win_hi = [&](int i) { return min(chunk > 0 ? min((i / chunk + 1) * chunk, T) : T, klen); };
    const int last_q = min(q0 + FQ, T) - 1;
    const int k_lo = win_lo(q0) & ~7;                        // tile rows keep (row & 7) == (position & 7): the rel-pos table is
    const int k_hi = win_hi(last_q);                         // pre-swizzled by position, so its rows are copied chunk for chunk
    const int ntiles = k_hi > k_lo ? (k_hi - k_lo + FK - 1) / FK : 0;
    // this warp's rows and their windows
    const int r0 = q0 + warp * 16 + g, r1 = r0 + 8;
    const int s0 = r0 < T ? win_lo(r0) : 0, e0 = r0 < T ? win_hi(r0) : 0;
    const int s1 = r1 < T ? win_lo(r1) : 0, e1 = r1 < T ? win_hi(r1) : 0;
    const int wq_first = q0 + warp * 16, wq_last = min(wq_first + 15, T - 1);
    const int w_lo = wq_first < T ? win_lo(wq_first) : 0, w_hi = wq_first < T ? win_hi(wq_last) : 0;

    auto load_tile = [&](int t, int stage) {
        const int kt = k_lo + t * FK;
        TA* Ks = tiles + (size_t)stage * 3 * FK * DK;
        TA* Ps = Ks + FK * DK;
        TA* Vs = Ps + FK * DK;
        for (int i = tid; i < FK * NCH * 3; i += ATT_THREADS) {
            const int which = i / (FK * NCH);                // 0 K, 1 P, 2 V
            const int j = (i / NCH) % FK, cc = i % NCH, key = kt + j;
            TA* dst = (which == 0 ? Ks : which == 1 ? Ps : Vs) + j * DK;
            if (which == 1) {
                if (key < pos_rows && key < k_hi) cp_async16(dst + (cc << 3), ptab_h + ((long long)h * pos_rows + key) * DK + (cc << 3));
                else *reinterpret_cast<uint4*>(dst + (cc << 3)) = make_uint4(0, 0, 0, 0);
            } else {
                TA* d2 = dst + ((cc ^ (j & 7)) << 3);
                if (key < k_hi) cp_async16(d2, qkv + ((long long)b * T + key) * 3 * D + (which == 0 ? 1 : 2) * D + h * DK + cc * 8);
                else *reinterpret_cast<uint4*>(d2) = make_uint4(0, 0, 0, 0);     // finite operands for the masked columns
            }
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
    };
    if (ntiles > 0) load_tile(0, 0);

    // (q+u), (q+v) A fragments of this warp's 16 queries: a0 (row g, k 2c..), a1 (row g+8), a2 (row g, k 2c+8..), a3 (row g+8)
    uint32_t qu[4][4], qv[4][4];
    {
        const float* qr0 = q32 + ((long long)b * T + min(r0, T - 1)) * 3 * D + h * DK;
        const float* qr1 = q32 + ((long long)b * T + min(r1, T - 1)) * 3 * D + h * DK;
#pragma unroll
        for (int ks = 0; ks < 4; ++ks) {
#pragma unroll
            for (int hf = 0; hf < 2; ++hf) {
                const int d = ks * 16 + hf * 8 + c * 2;
                const float2 u = *reinterpret_cast<const float2*>(pos_u + h * DK + d);
                const float2 v = *reinterpret_cast<const float2*>(pos_v + h * DK + d);
                const float2 a = *reinterpret_cast<const float2*>(qr0 + d);
                const float2 bq = *reinterpret_cast<const float2*>(qr1 + d);
                qu[ks][hf * 2] = pack2<__half>(a.x + u.x, a.y + u.y);
                qu[ks][hf * 2 + 1] = pack2<__half>(bq.x + u.x, bq.y + u.y);
                qv[ks][hf * 2] = pack2<__half>(a.x + v.x, a.y + v.y);
                qv[ks][hf * 2 + 1] = pack2<__half>(bq.x + v.x, bq.y + v.y);
            }
        }
    }
    float oacc[8][4];
#pragma unroll
    for (int n = 0; n < 8; ++n) { oacc[n][0] = 0.f; oacc[n][1] = 0.f; oacc[n][2] = 0.f; oacc[n][3] = 0.f; }
    float m0 = -INFINITY, m1 = -INFINITY, l0 = 0.f, l1 = 0.f;
    const int mi = lane >> 3, rr = lane & 7;                  // ldmatrix: this lane addresses row rr of matrix mi

    for (int t = 0; t < ntiles; ++t) {
        const int stage = t & 1;
        if (t + 1 < ntiles) {
            load_tile(t + 1, stage ^ 1);                     // (the stage was released by the barrier that ended tile t-1)
            asm volatile("cp.async.wait_group 1;" ::: "memory");
        } else {
            asm volatile("cp.async.wait_group 0;" ::: "memory");
        }
        __syncthreads();
        const int kt = k_lo + t * FK;
        if (kt < w_hi && kt + FK > w_lo) {                   // warp-uniform: some key of the tile is inside some row's band
            const TA* Ks = tiles + (size_t)stage * 3 * FK * DK;
            const TA* Ps = Ks + FK * DK;
            const TA* Vs = Ps + FK * DK;
            // 16-key groups of the tile that intersect the band of at least one of this warp's rows (warp-uniform): with the
            // shipped band (68 keys) a warp needs 5 of the 8 groups of its two tiles
            bool act[4];
#pragma unroll
            for (int np = 0; np < 4; ++np) act[np] = kt + np * 16 < w_hi && kt + np * 16 + 16 > w_lo;
            float sacc[8][4];
#pragma unroll
            for (int n = 0; n < 8; ++n) { sacc[n][0] = 0.f; sacc[n][1] = 0.f; sacc[n][2] = 0.f; sacc[n][3] = 0.f; }
            // ---- S = (q+u) K^T + (q+v) P^T : per k-step one ldmatrix.x4 feeds two 8-key n-tiles ----
#pragma unroll
            for (int np = 0; np < 4; ++np) {                 // n-tile pair (16 keys)
                if (!act[np]) continue;
#pragma unroll
                for (int ks = 0; ks < 4; ++ks) {
                    const int key = np * 16 + (mi >> 1) * 8 + rr;
                    const int chk = ks * 2 + (mi & 1);
                    uint32_t kf[4], pf[4];
                    ldsm_x4(kf, Ks + key * DK + ((chk ^ (key & 7)) << 3));
                    ldsm_x4(pf, Ps + key * DK + ((chk ^ (key & 7)) << 3));
                    mma16816_ab(sacc[np * 2], qu[ks], kf[0], kf[1]);
                    mma16816_ab(sacc[np * 2 + 1], qu[ks], kf[2], kf[3]);
                    mma16816_ab(sacc[np * 2], qv[ks], pf[0], pf[1]);
                    mma16816_ab(sacc[np * 2 + 1], qv[ks], pf[2], pf[3]);
                }
            }
            // ---- mask, scale, online softmax in the exp2 domain (rows g and g+8; a row lives in the 4 lanes that share g):
            //      s2 = s / 8 * log2(e), p = 2^(s2 - m) ----
            constexpr float SC = 0.125f * 1.4426950408889634f;
            const int ds0 = s0 - kt - c * 2, de0 = e0 - kt - c * 2, ds1 = s1 - kt - c * 2, de1 = e1 - kt - c * 2;
            float mx0 = -INFINITY, mx1 = -INFINITY;
#pragma unroll
            for (int n = 0; n < 8; ++n) {
                if (!act[n >> 1]) continue;
#pragma unroll
                for (int e = 0; e < 2; ++e) {
                    const int j = n * 8 + e;                 // key = kt + c * 2 + j
                    sacc[n][e] = (j >= ds0 && j < de0) ? sacc[n][e] * SC : -INFINITY;
                    sacc[n][2 + e] = (j >= ds1 && j < de1) ? sacc[n][2 + e] * SC : -INFINITY;
                    mx0 = fmaxf(mx0, sacc[n][e]);
                    mx1 = fmaxf(mx1, sacc[n][2 + e]);
                }
            }
            mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 1));
            mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 2));
            mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 1));
            mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 2));
            const float mn0 = fmaxf(m0, mx0), mn1 = fmaxf(m1, mx1);
            // a row with nothing unmasked so far keeps m = -inf; subtracting 0 instead makes every 2^(-inf - 0) an exact 0
            const float ms0 = mn0 == -INFINITY ? 0.f : mn0, ms1 = mn1 == -INFINITY ? 0.f : mn1;
            const float cf0 = fast_exp2(m0 - ms0), cf1 = fast_exp2(m1 - ms1);      // m = -inf -> 0 (and l, o are 0 then)
            m0 = mn0; m1 = mn1;
            l0 *= cf0; l1 *= cf1;
            uint32_t pa[4][4];                               // probabilities as A fragments: k-step kk = keys 16kk .. 16kk+15
#pragma unroll
            for (int n = 0; n < 8; ++n) {
                if (!act[n >> 1]) continue;
                const float p00 = fast_exp2(sacc[n][0] - ms0), p01 = fast_exp2(sacc[n][1] - ms0);
                const float p10 = fast_exp2(sacc[n][2] - ms1), p11 = fast_exp2(sacc[n][3] - ms1);
                l0 += p00 + p01;
                l1 += p10 + p11;
                pa[n >> 1][(n & 1) * 2] = pack2_nosat(p00, p01);
                pa[n >> 1][(n & 1) * 2 + 1] = pack2_nosat(p10, p11);
            }
#pragma unroll
            for (int n = 0; n < 8; ++n) { oacc[n][0] *= cf0; oacc[n][1] *= cf0; oacc[n][2] *= cf1; oacc[n][3] *= cf1; }
            // ---- O += P V : V transposed by ldmatrix, one x4 = 16 keys x two 8-dim n-tiles ----
#pragma unroll
            for (int kk = 0; kk < 4; ++kk) {
                if (!act[kk]) continue;
#pragma unroll
                for (int dp = 0; dp < 4; ++dp) {             // dim n-tile pair
                    const int key = kk * 16 + (mi & 1) * 8 + rr;
                    const int chk = dp * 2 + (mi >> 1);
                    uint32_t vf[4];
                    ldsm_x4_t(vf, Vs + key * DK + ((chk ^ (key & 7)) << 3));
                    mma16816_ab(oacc[dp * 2], pa[kk], vf[0], vf[1]);
                    mma16816_ab(oacc[dp * 2 + 1], pa[kk], vf[2], vf[3]);
                }
            }
        }
        __syncthreads();                                     // the stage may be refilled
    }
    // ---- normalise; a row's partial sums live in its 4 lanes ----
    l0 += __shfl_xor_sync(0xffffffffu, l0, 1); l0 += __shfl_xor_sync(0xffffffffu, l0, 2);
    l1 += __shfl_xor_sync(0xffffffffu, l1, 1); l1 += __shfl_xor_sync(0xffffffffu, l1, 2);
    const float i0 = l0 > 0.f ? 1.f / l0 : 0.f, i1 = l1 > 0.f ? 1.f / l1 : 0.f;      // fully masked row -> zeros
    // stage the warp's 16 x 64 tile (warp-private region of the tile buffer, all tiles consumed) and store 16-byte chunks
    TA* ot = tiles + warp * 16 * DK;
#pragma unroll
    for (int n = 0; n < 8; ++n) {
        *reinterpret_cast<uint32_t*>(ot + g * DK + n * 8 + c * 2) = pack2<__half>(oacc[n][0] * i0, oacc[n][1] * i0);
        *reinterpret_cast<uint32_t*>(ot + (g + 8) * DK + n * 8 + c * 2) = pack2<__half>(oacc[n][2] * i1, oacc[n][3] * i1);
    }
    __syncwarp();
#pragma unroll
    for (int i = lane; i < 16 * NCH; i += 32) {
        const int r = i >> 3, cc = i & 7, row = q0 + warp * 16 + r;
        if (row < T)
            *reinterpret_cast<uint4*>(out + ((long long)b * T + row) * D + h * DK + cc * 8) = *reinterpret_cast<const uint4*>(ot + r * DK + cc * 8);
    }
}

__global__ void advance_sessions_kernel(const int32_t* __restrict__ ids, int n, int t, int chunk_size, int pe_wrap,
                                        int32_t* n_frames, int32_t* pe_index, int32_t* adapter_valid, int chunks) {
    FO_PDL_TRIGGER();
    FO_PDL_WAIT();
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= n) return;
    const int s = ids[b];
    if (n_frames) {
        n_frames[s] += chunks * t;
        int pe = pe_index[s];
        for (int j = 0; j < chunks; ++j) pe = pe % pe_wrap + chunk_size;   // attention.py:107,120 (+chunk_size, not +t)
        pe_index[s] = pe;
    }
    if (adapter_valid) adapter_valid[s] = adapter_valid[s] == 1 ? 2 : 1;
}

// launcher of the multi-chunk kernels (AttnStream::chunks > 1)
template <typename TA>
int attention_stream_chunks(const AttnStream& a, const TA* qkv, const float* q32, TA* ring, const TA* ptab_h,
                            const float* pos_u, const float* pos_v, TA* out, cudaStream_t st) {
    const int kt = a.chunks * a.t, rows = a.window + kt, prow = a.window + a.t;
    FO_CHECK(a.t <= TQ_MAX, "attention_stream: %d frames per chunk exceeds %d", a.t, TQ_MAX);
    FO_CHECK(rows <= STREAM_CHUNKS_MAX_KEYS, "attention_stream: window %d + %d chunks x %d frames exceeds %d keys", a.window,
             a.chunks, a.t, STREAM_CHUNKS_MAX_KEYS);
    dim3 grid(a.n, a.H);
    static bool attr_set[2] = {false, false};
    size_t smem;
    if constexpr (sizeof(TA) == 2) {
        const int krows = ((rows + 15) & ~15) + 16, vrows = (prow + 15) & ~15;
        smem = (size_t)(2 * krows + vrows) * DK * 2 + (size_t)2 * a.t * DK * 2 + (size_t)a.t * vrows * 2 +
               (size_t)a.t * std::max(vrows, DK) * 4;
        if (!attr_set[1]) {
            FO_CUDA(cudaFuncSetAttribute(attention_chunks_mma_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024));
            attr_set[1] = true;
        }
        FO_CHECK(smem <= 160 * 1024, "attention_stream: multi-chunk call too large for shared memory");
        FO_CUDA(launch_pdl(attention_chunks_mma_kernel, grid, dim3(ATT_THREADS), smem, st, a, reinterpret_cast<const __half*>(qkv), q32,
                           reinterpret_cast<__half*>(ring), reinterpret_cast<const __half*>(ptab_h), pos_u, pos_v,
                           reinterpret_cast<__half*>(out)));
    } else {
        smem = (size_t)(2 * rows + prow) * DK * sizeof(TA) + (size_t)2 * a.t * DK * sizeof(float) + (size_t)a.t * prow * sizeof(float);
        if (!attr_set[0]) {
            FO_CUDA(cudaFuncSetAttribute(attention_chunks_kernel<TA>, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024));
            attr_set[0] = true;
        }
        FO_CHECK(smem <= 160 * 1024, "attention_stream: multi-chunk call too large for shared memory");
        FO_CUDA(launch_pdl(attention_chunks_kernel<TA>, grid, dim3(ATT_THREADS), smem, st, a, qkv, q32, ring, ptab_h, pos_u, pos_v, out));
    }
    FO_LAUNCHED();
    FO_CUDA(cudaGetLastError());
    return 0;
}

}  // namespace

template <typename TA>
int attention_stream(const AttnStream& a, const TA* qkv, const float* q32, TA* ring, const TA* ptab_h,
                     const float* pos_u, const float* pos_v, TA* out, cudaStream_t st) {
    if (a.n <= 0) return 0;
    if (a.chunks > 1) return attention_stream_chunks<TA>(a, qkv, q32, ring, ptab_h, pos_u, pos_v, out, st);
    FO_CHECK(a.t <= TQ_MAX, "attention_stream: %d frames per call exceeds %d", a.t, TQ_MAX);
    FO_CHECK(a.ring_cap >= a.window + a.t, "attention_stream: ring capacity %d < window %d + %d", a.ring_cap, a.window, a.t);
    const int rows = a.window + a.t;
    FO_CHECK(rows <= 128, "attention_stream: window + frames per call (%d) exceeds 128 keys", rows);
    const size_t smem = (size_t)3 * rows * DK * sizeof(TA) + (size_t)2 * a.t * DK * sizeof(float) +
                        (size_t)a.t * rows * sizeof(float);
    static bool attr_set[2] = {false, false};
    if (!attr_set[sizeof(TA) == 2]) {
        FO_CUDA(cudaFuncSetAttribute(attention_stream_kernel<TA>, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024));
        attr_set[sizeof(TA) == 2] = true;
    }
    FO_CHECK(smem <= 160 * 1024, "attention_stream: window too large for shared memory");
    dim3 grid(a.n, a.H);
    if constexpr (sizeof(TA) == 2) {
            const int vrows = (rows + 15) & ~15;
            const size_t sm = (size_t)(2 * rows + vrows) * DK * 2 + (size_t)2 * a.t * DK * 2 + (size_t)a.t * vrows * 2 +
                              (size_t)a.t * std::max(vrows, DK) * 4;
            // past 48 KB (window + t > ~115 keys, e.g. left_chunks 31) the launch needs the opt-in
            static bool mma_attr_set = false;
            if (!mma_attr_set) {
                FO_CUDA(cudaFuncSetAttribute(attention_stream_mma_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024));
                FO_CUDA(cudaFuncSetAttribute(attention_stream_mma_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024));
                mma_attr_set = true;
            }
            FO_CHECK(sm <= 160 * 1024, "attention_stream: window too large for shared memory");
            if (a.nsplit > 0)
                FO_CUDA(launch_pdl(attention_stream_mma_kernel<true>, grid, dim3(ATT_THREADS), sm, st, a, reinterpret_cast<const __half*>(qkv), q32,
                                   reinterpret_cast<__half*>(ring), reinterpret_cast<const __half*>(ptab_h), pos_u, pos_v,
                                   reinterpret_cast<__half*>(out)));
            else
                FO_CUDA(launch_pdl(attention_stream_mma_kernel<false>, grid, dim3(ATT_THREADS), sm, st, a, reinterpret_cast<const __half*>(qkv), q32,
                                   reinterpret_cast<__half*>(ring), reinterpret_cast<const __half*>(ptab_h), pos_u, pos_v,
                                   reinterpret_cast<__half*>(out)));
            FO_LAUNCHED();
#ifdef FO_TC_TRACE_BUILD
            if (getenv("FO_TC_TRACE") && st == nullptr) {
                cudaStreamSynchronize(st);
                unsigned long long hb[16];
                cudaMemcpyFromSymbol(hb, g_attn_trace, sizeof(hb));
                fprintf(stderr, "attn_trace n=%d:", a.n);
                for (int i = 1; i <= 9; ++i) fprintf(stderr, " t%d=%lld", i, (long long)(hb[i] - hb[0]));
                fprintf(stderr, " ns\n");
            }
#endif
    } else {
        FO_CUDA(launch_pdl(attention_stream_kernel<TA>, grid, dim3(ATT_THREADS), smem, st, a, qkv, q32, ring, ptab_h, pos_u, pos_v, out));
        FO_LAUNCHED();
    }
    FO_CUDA(cudaGetLastError());
    return 0;
}
template int attention_stream<float>(const AttnStream&, const float*, const float*, float*, const float*, const float*, const float*, float*, cudaStream_t);
// head-major copy of a rel-pos table in the activation type: out[h][pos][64] = (TA) in[pos][h*64 + d]
template <typename TA>
__global__ void ptab_head_major_kernel(const float* __restrict__ in, int pos_rows, int H, TA* __restrict__ out) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long total = (long long)pos_rows * H * DK;
    if (i >= total) return;
    const int d = (int)(i % DK);
    const long long r = i / DK;
    const int pos = (int)(r % pos_rows), h = (int)(r / pos_rows);
    // 16-bit tables carry the chunk swizzle of the fp16 attention kernel (chunk c of the row of position p at c ^ (p & 7))
    const int dd = sizeof(TA) == 2 ? ((((d >> 3) ^ (pos & 7)) << 3) + (d & 7)) : d;
    out[r * DK + dd] = from_f<TA>(in[((long long)pos * H + h) * DK + d]);
}
template <typename TA>
int ptab_head_major(const float* in, int pos_rows, int H, TA* out, cudaStream_t st) {
    const long long total = (long long)pos_rows * H * DK;
    ptab_head_major_kernel<TA><<<(unsigned)((total + 255) / 256), 256, 0, st>>>(in, pos_rows, H, out);
    FO_CUDA(cudaGetLastError());
    return 0;
}
template int ptab_head_major<float>(const float*, int, int, float*, cudaStream_t);
template int ptab_head_major<__half>(const float*, int, int, __half*, cudaStream_t);
template int attention_stream<__half>(const AttnStream&, const __half*, const float*, __half*, const __half*, const float*, const float*, __half*, cudaStream_t);

template <typename TA>
int attention_offline(const TA* qkv, const float* q32, int B, int T, int H, const int32_t* ilens, int chunk, int left,
                      const float* ptab, const TA* ptab_h, int pos_rows, const float* pos_u, const float* pos_v, TA* out,
                      cudaStream_t st) {
    if (B <= 0 || T <= 0) return 0;
    dim3 grid(cdiv(T, QB), H, B);
    const size_t smem = (size_t)3 * KT * (DK + 16 / sizeof(TA)) * sizeof(TA) + (size_t)2 * QB * DK * sizeof(float) +
                        (size_t)(ATT_THREADS / 32) * KT * sizeof(float);
    static bool attr_set[2] = {false, false};
    if (!attr_set[sizeof(TA) == 2]) {
        FO_CUDA(cudaFuncSetAttribute(attention_offline_kernel<TA>, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024));
        attr_set[sizeof(TA) == 2] = true;
    }
    if constexpr (sizeof(TA) == 2) {
        if (!ptab_h || T > pos_rows) return 1;
        {
            const size_t smf = (size_t)2 * 3 * FK * DK * 2;      // 48 KB: double-buffered K | P | V tiles
            static bool attr3 = false;
            if (!attr3) {
                FO_CUDA(cudaFuncSetAttribute(attention_offline_fa_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024));
                attr3 = true;
            }
            attention_offline_fa_kernel<<<dim3(cdiv(T, FQ), H, B), ATT_THREADS, smf, st>>>(
                reinterpret_cast<const __half*>(qkv), q32, T, H, ilens, chunk, left, reinterpret_cast<const __half*>(ptab_h), pos_rows,
                pos_u, pos_v, reinterpret_cast<__half*>(out));
            FO_LAUNCHED();
            FO_CUDA(cudaGetLastError());
            return 0;
        }
    } else {
        attention_offline_kernel<TA><<<grid, ATT_THREADS, smem, st>>>(qkv, q32, T, H, ilens, chunk, left, ptab, pos_u, pos_v, out);
    }
    FO_LAUNCHED();
    FO_CUDA(cudaGetLastError());
    return 0;
}
template int attention_offline<float>(const float*, const float*, int, int, int, const int32_t*, int, int, const float*, const float*, int, const float*, const float*, float*, cudaStream_t);
template int attention_offline<bf16>(const bf16*, const float*, int, int, int, const int32_t*, int, int, const float*, const bf16*, int, const float*, const float*, bf16*, cudaStream_t);
template int attention_offline<__half>(const __half*, const float*, int, int, int, const int32_t*, int, int, const float*, const __half*, int, const float*, const float*, __half*, cudaStream_t);

int advance_sessions(const int32_t* ids, int n, int t, int chunk_size, int pe_wrap, int32_t* n_frames,
                      int32_t* pe_index, int32_t* adapter_valid, cudaStream_t st, int chunks) {
    if (n <= 0) return 0;
    FO_CUDA(launch_pdl(advance_sessions_kernel, dim3(cdiv(n, 128)), dim3(128), 0, st, ids, n, t, chunk_size, pe_wrap, n_frames, pe_index, adapter_valid,
                       chunks));
    FO_LAUNCHED();
    FO_CUDA(cudaGetLastError());
    return 0;
}

FO_TR_BIND_DEF(trace_bind_attention)

}  // namespace fo
