// Chunk attention with key-position rel-pos bias (reference: MultiHeadedAttention.infer / .forward,
// models/encoder/attention.py:407-459 / 350-405; no rel_shift, SURVEY 2.4-3):
//     score[i][j] = ((q_i + u) . K_j + (q_i + v) . P[pos_j]) / sqrt(d_k),   softmax over j,   out = sum_j p_ij V_j
// d_k is 64.  Streaming: one CTA per (session, head[, group of chunks]); the cached K/V rows come from the session's ring in
// HBM with cp.async.bulk (TMA bulk copy, mbarrier completion) while the chunk's own rows arrive from the
// fused QKV GEMM output and are appended to the ring.  The four streaming kernels (one chunk or several, fp16 or fp32)
// differ in how they stage the rows; the per-chunk math is attn_chunk_mma / attn_chunk_ffma (fo_attn_core.cuh).
// Offline: one CTA per (utterance, head, query block); the band [start,end) of models/masks.py:50-56 and the pad mask
// are evaluated arithmetically, never materialised; key tiles + online softmax cover unbounded left context.
#include <stdlib.h>

#include <algorithm>
#include <array>

#include "fo_attn_core.cuh"

namespace fo {


namespace {

constexpr int ATT_THREADS = 128;

// ---------------------------------------------------------------------------------------------
// Single-chunk streaming attention of fp32 contexts (k = 1), one CTA per (session, head), 4 warps.  Steady state: 64 cached
// + 4 new keys, 4 queries.  Staging: thread 0 starts the bulk copies of the ring window and of the rel-pos rows
// P_l[start .. start+nk) (HBM -> smem, mbarrier); meanwhile every thread fetches its share of the chunk's own K/V rows
// (appended to the ring in the same pass) and Q, all issued before the first use so that one memory latency covers them.
// smem rows are sized by window + t (68), not by the ring capacity.
__global__ void __launch_bounds__(ATT_THREADS, 7)
attention_stream_kernel(AttnStream a, const float* __restrict__ qkv, const float* __restrict__ q32, float* __restrict__ ring,
                        const float* __restrict__ ptab_h, const float* __restrict__ pos_u, const float* __restrict__ pos_v,
                        float* __restrict__ out) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    constexpr int EPC = 4, NCH = DK / EPC;
    FO_PDL_TRIGGER();
    FO_PDL_WAIT();
    const int cap = a.ring_cap;
    const int t = a.t, D = a.H * DK;
    const int rows = a.window + t;                  // most keys a call can see
    float* Ks = reinterpret_cast<float*>(smem_raw);
    float* Vs = Ks + rows * DK;
    float* Ps = Vs + rows * DK;
    float* qu = Ps + rows * DK;
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
    float* ringK = ring + (long long)slot * a.ring_slot_stride + (long long)h * cap * DK;
    float* ringV = ringK + (long long)a.H * cap * DK;
    const int tid = threadIdx.x;

    // rel-pos rows P_l[start .. start+nk) of this head are contiguous in the head-major table: one bulk copy
    const int np = min(nk, a.pos_rows - start);
    if (tid == 0) {
        mbar_init(&bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        ring_window_copy(ringK, ringV, cap, first, cl, Ks, Vs, ptab_h + ((long long)h * a.pos_rows + start) * DK, Ps, np, &bar);
    }
    // ---- loads into registers (no dependent use before they are all issued) ----
    // (a) chunk's own K/V rows: t rows x NCH chunks x {K,V}
    const int n_new = t * NCH * 2;
    uint4 newv = make_uint4(0, 0, 0, 0);
    int new_which = 0, new_r = 0, new_c = 0;
    const bool has_new = tid < n_new;                // t <= 4: one slot per thread, more rows in the loop below
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
        float* sdst = (new_which ? Vs : Ks) + (cl + new_r) * DK + new_c * EPC;
        *reinterpret_cast<uint4*>(sdst) = newv;
        float* gdst = (new_which ? ringV : ringK) + (long long)((nf + new_r) % cap) * DK + new_c * EPC;
        *reinterpret_cast<uint4*>(gdst) = newv;
    }
    for (int i = tid + ATT_THREADS; i < n_new; i += ATT_THREADS) {      // only when t > 4
        const int which = i / (t * NCH), r = (i / NCH) % t, c = i % NCH;
        const uint4 val = *reinterpret_cast<const uint4*>(qkv + (long long)(b * t + r) * 3 * D + (which + 1) * D + h * DK + c * EPC);
        *reinterpret_cast<uint4*>((which ? Vs : Ks) + (cl + r) * DK + c * EPC) = val;
        *reinterpret_cast<uint4*>((which ? ringV : ringK) + (long long)((nf + r) % cap) * DK + c * EPC) = val;
    }
    // the table holds every position a call can reach (fo_create sizes pos_rows): this clamp only keeps reads in bounds
    for (int i = tid + np * (DK / 8); i < nk * (DK / 8); i += ATT_THREADS) {
        const int j = i / (DK / 8), c = i % (DK / 8);
        const float* src = ptab_h + ((long long)h * a.pos_rows + a.pos_rows - 1) * DK + c * 8;
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
    attn_chunk_ffma(Ks, Vs, Ps, qu, qv, prob, rows, nk, t, out + (long long)b * t * D + h * DK, D);
}

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

// ---------------------------------------------------------------------------------------------
// Single-chunk streaming attention of fp16 contexts (k = 1), the contractions on mma.sync (attn_chunk_mma).  With 4 query
// rows the scalar form spends ~13 k FMA/convert instructions per CTA on them; here they are ~60 MMAs.  Staging: the ring
// window and rel-pos bulk copies are issued BEFORE the dependency wait, the chunk's own K/V rows are appended to the ring
// in the same pass, and with DEFER q / k / v are summed from the QKV GEMM's split-K partials (AttnStream::part).  Shared
// memory is sized by window + t (mma_unit_layout: 30,592 B at 64 + 4 keys), so 7 CTAs fit per SM and the 1024 CTAs of a
// 64-session layer are ONE wave.  (q+u), (q+v) are rounded to fp16 for the MMAs.
template <bool DEFER>
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
    const MmaUnitLayout lay = mma_unit_layout(a.window, t);
    const int vrows = lay.vrows;
    TA* Ks = reinterpret_cast<TA*>(smem_raw);
    TA* Ps = reinterpret_cast<TA*>(smem_raw + lay.p);
    TA* Vs = reinterpret_cast<TA*>(smem_raw + lay.v);
    TA* quh = reinterpret_cast<TA*>(smem_raw + lay.qu);
    TA* qvh = reinterpret_cast<TA*>(smem_raw + lay.qv);
    TA* ph = reinterpret_cast<TA*>(smem_raw + lay.ph);
    float* sc = reinterpret_cast<float*>(smem_raw + lay.sc);
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
    const int tid = threadIdx.x;

    const int np = min(nk, a.pos_rows - start);
    AT_TRACE(2);
    if (tid == 0) {
        mbar_init(&bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        ring_window_copy(ringK, ringV, cap, first, cl, Ks, Vs, ptab_h + ((long long)h * a.pos_rows + start) * DK, Ps, np, &bar);
    }
    AT_TRACE(3);
    // bias of dimension tid % 64: the same for every Q element this thread stages below (ATT_THREADS is a multiple of 64)
    const float ub = pos_u[h * DK + tid % DK], vb = pos_v[h * DK + tid % DK];
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
    float qreg[2];                                  // Q of t <= 4 rows; more rows are loaded where they are stored
#pragma unroll
    for (int k = 0; k < 2; ++k) {
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
    for (int k = 0; k < 2; ++k) {
        const int i = tid + k * ATT_THREADS;
        if (i < t * DK) {
            const int r = i / DK, d = i % DK;
            const int o = r * DK + (((d >> 3) ^ (r & 7)) << 3) + (d & 7);      // same chunk swizzle, keyed by the query row
            quh[o] = from_f<TA>(qreg[k] + ub);
            qvh[o] = from_f<TA>(qreg[k] + vb);
        }
    }
    for (int i = tid + 2 * ATT_THREADS; i < t * DK; i += ATT_THREADS) {
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
    attn_chunk_mma<ATT_THREADS / 32>(Ks, Vs, first, Ps, start, quh, qvh, ph, sc, vrows, nk, t, out + (long long)b * t * D + h * DK, D);
    AT_TRACE(9);
    if (threadIdx.x == 0) { FO_TR_STAMP(3); FO_TR_STAMP(4); FO_TR_FLUSH(2, 0); }
}

// ---------------------------------------------------------------------------------------------
// Several consecutive chunks of every session in one call (fo_encode_stream_chunks[_v], passes of fo_stream_steps_v): session b
// brings k = cnt[b] chunks from row row0 = (off[b] - off[0]) * t.  CTA (b, h, z) takes chunks [j0, j1) = [z * G, min(k, (z + 1)
// * G)), G = a.chunks, and stages the keys of all of them once: frames [first, nf + j1 * t) with first = nf_j0 - min(nf_j0,
// window) -- those before the call (frame < nf) from the ring by bulk copy, the rest from the call's own K|V rows (qkv row =
// frame - nf) -- then walks its query chunks in order.  Shared memory is sized by G.  Chunk j sees exactly what the j-th
// sequential single-chunk call would see:
//     nf_j = nf + j*t,  keys = frames [nf_j - min(nf_j, window), nf_j + t)   (a contiguous run of the staged rows)
//     pe_j = pe_after(pe_index, j),  rel-pos rows P[max(0, pe_j % wrap - full_chunk) + m]
// The rel-pos window moves (and may wrap) with pe_j, so it is re-staged per chunk.  The new rows go to the ring only after
// every read of the old window: the ring holds window + max_t rows, fewer than the call's keys, so a later chunk's rows would
// overwrite frames an earlier chunk still needs.  With one group per session (gridDim.z == 1) the CTA is the only reader of
// its (slot, head) ring and appends them itself once its window copy has landed; with several, chunks_append_ring_kernel
// appends them after the grid.  Layouts (fp16 chunk swizzle of K/V by frame and of P by position, q swizzled by query row)
// are those of the single-chunk kernels.
struct StepsGroup {
    int j0, j1, nf, first, cr, kn;      // chunks; frames before the call; first staged frame; staged rows from ring / from qkv
};
__device__ __forceinline__ bool steps_group(const AttnStream& a, int b, StepsGroup* g) {
    g->j0 = blockIdx.z * a.chunks;
    const int k = a.cnt[b];
    if (g->j0 >= k) return false;
    g->j1 = min(k, g->j0 + a.chunks);
    g->nf = a.n_frames[a.ids[b]];
    const int nf0 = g->nf + g->j0 * a.t;
    g->first = nf0 - min(nf0, a.window);
    g->cr = max(0, g->nf - g->first);
    g->kn = g->nf + g->j1 * a.t - (g->first + g->cr);
    return true;
}

// stage the new K/V rows (qkv row r -> smem row cl + r, frame nf + r)
template <typename TA, int NCH, bool SWZ>
__device__ __forceinline__ void chunks_stage_new(const AttnStream& a, const TA* qkv, TA* Ks, TA* Vs, int h, int nf, int cl,
                                                 int kt) {
    constexpr int EPC = 16 / sizeof(TA);
    const int D = a.H * DK;
    for (int i = threadIdx.x; i < kt * NCH * 2; i += ATT_THREADS) {
        const int which = i / (kt * NCH), r = (i / NCH) % kt, c = i % NCH;
        const int pc = SWZ ? (c ^ ((nf + r) & 7)) : c;
        *reinterpret_cast<uint4*>((which ? Vs : Ks) + (cl + r) * DK + pc * EPC) =
            *reinterpret_cast<const uint4*>(qkv + (long long)r * 3 * D + (which + 1) * D + h * DK + c * EPC);
    }
}
// append the staged new rows (smem row cl + r = frame nf + r) to the ring: only the last `cap` of them when the call brings
// more frames than the ring holds
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

// Multi-chunk streaming attention of fp32 contexts.  The rel-pos rows and Q of every chunk are re-staged before its core
// (attn_chunk_ffma).
__global__ void __launch_bounds__(ATT_THREADS)
attention_chunks_kernel(AttnStream a, const float* __restrict__ qkv, const float* __restrict__ q32, float* __restrict__ ring,
                        const float* __restrict__ ptab_h, const float* __restrict__ pos_u, const float* __restrict__ pos_v,
                        float* __restrict__ out) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    constexpr int EPC = 4, NCH = DK / EPC;
    FO_PDL_TRIGGER();
    FO_PDL_WAIT();
    const int cap = a.ring_cap, t = a.t, D = a.H * DK;
    const int rows = a.window + a.chunks * t, prow = a.window + t;
    float* Ks = reinterpret_cast<float*>(smem_raw);
    float* Vs = Ks + rows * DK;
    float* Ps = Vs + rows * DK;
    float* qu = Ps + prow * DK;
    float* qv = qu + t * DK;
    float* prob = qv + t * DK;                      // t x prow
    __shared__ __align__(8) uint64_t bar;

    const int b = blockIdx.x, h = blockIdx.y;
    StepsGroup g;
    if (!steps_group(a, b, &g)) return;
    const int slot = a.ids[b];
    const long long row0 = (long long)(a.off[b] - a.off[0]) * t;     // the session's rows: the pointers start there
    qkv += row0 * 3 * D; q32 += row0 * 3 * D; out += row0 * D;
    float* ringK = ring + (long long)slot * a.ring_slot_stride + (long long)h * cap * DK;
    float* ringV = ringK + (long long)a.H * cap * DK;
    const int tid = threadIdx.x;
    if (tid == 0) {
        mbar_init(&bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        ring_window_copy<float>(ringK, ringV, cap, g.first, g.cr, Ks, Vs, nullptr, nullptr, 0, &bar);
    }
    const int fs = g.first + g.cr;
    chunks_stage_new<float, NCH, false>(a, qkv + (long long)(fs - g.nf) * 3 * D, Ks, Vs, h, fs, g.cr, g.kn);
    __syncthreads();
    mbar_wait(&bar, 0);
    if (gridDim.z == 1) chunks_append_ring<float, NCH>(a, Ks, Vs, ringK, ringV, g.nf, g.cr, g.kn);

    const int pe0 = a.pe_index[slot];
    for (int j = g.j0; j < g.j1; ++j) {
        const int nfj = g.nf + j * t, clj = min(nfj, a.window);
        const int o = nfj - clj - g.first;          // staged row of this chunk's first key
        const int nk = clj + t;
        const int start = max(0, pe_after(pe0, j, a.chunk_size, a.pe_wrap) % a.pe_wrap - a.full_chunk);
        for (int i = tid; i < nk * NCH; i += ATT_THREADS) {        // the min() keeps reads in bounds; pos_rows covers every reachable position
            const int r = i / NCH, c = i % NCH, pos = min(start + r, a.pos_rows - 1);
            *reinterpret_cast<uint4*>(Ps + r * DK + c * EPC) = *reinterpret_cast<const uint4*>(ptab_h + ((long long)h * a.pos_rows + pos) * DK + c * EPC);
        }
        for (int i = tid; i < t * DK; i += ATT_THREADS) {
            const int r = i / DK, d = i % DK;
            const float q = q32[(long long)(j * t + r) * 3 * D + h * DK + d];
            qu[i] = q + pos_u[h * DK + d];
            qv[i] = q + pos_v[h * DK + d];
        }
        __syncthreads();
        attn_chunk_ffma(Ks + o * DK, Vs + o * DK, Ps, qu, qv, prob, prow, nk, t, out + (long long)(j * t) * D + h * DK, D);
        __syncthreads();                              // Ps / qu / prob are restaged by the next chunk
    }
}

// Multi-chunk streaming attention of fp16 contexts (t <= 8 = the MMA's N).  Staging as in attention_chunks_kernel, with the
// K/V rows swizzled by frame and padded past the last staged key; each chunk's core is attn_chunk_mma.
__global__ void __launch_bounds__(ATT_THREADS)
attention_chunks_mma_kernel(AttnStream a, const __half* __restrict__ qkv, const float* __restrict__ q32, __half* __restrict__ ring,
                            const __half* __restrict__ ptab_h, const float* __restrict__ pos_u, const float* __restrict__ pos_v,
                            __half* __restrict__ out) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    typedef __half TA;
    constexpr int EPC = 8, NCH = 8;
    FO_PDL_TRIGGER();
    FO_PDL_WAIT();
    const int cap = a.ring_cap, t = a.t, D = a.H * DK;
    const int rows = a.window + a.chunks * t;
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
    StepsGroup g;
    if (!steps_group(a, b, &g)) return;
    const int slot = a.ids[b];
    const long long row0 = (long long)(a.off[b] - a.off[0]) * t;     // the session's rows: the pointers start there
    qkv += row0 * 3 * D; q32 += row0 * 3 * D; out += row0 * D;
    const int nk_all = g.cr + g.kn;
    TA* ringK = ring + (long long)slot * a.ring_slot_stride + (long long)h * cap * DK;
    TA* ringV = ringK + (long long)a.H * cap * DK;
    const int tid = threadIdx.x;
    if (tid == 0) {
        mbar_init(&bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        ring_window_copy<TA>(ringK, ringV, cap, g.first, g.cr, Ks, Vs, nullptr, nullptr, 0, &bar);
    }
    const int fs = g.first + g.cr;
    chunks_stage_new<TA, NCH, true>(a, qkv + (long long)(fs - g.nf) * 3 * D, Ks, Vs, h, fs, g.cr, g.kn);
    // rows behind the last key: K is masked there, V enters the PV MMAs with probability 0 and must be finite
    for (int i = tid; i < (krows - nk_all) * NCH; i += ATT_THREADS) {
        *reinterpret_cast<uint4*>(Ks + (nk_all + i / NCH) * DK + (i % NCH) * EPC) = make_uint4(0, 0, 0, 0);
        *reinterpret_cast<uint4*>(Vs + (nk_all + i / NCH) * DK + (i % NCH) * EPC) = make_uint4(0, 0, 0, 0);
    }
    __syncthreads();
    mbar_wait(&bar, 0);
    if (gridDim.z == 1) chunks_append_ring<TA, NCH>(a, Ks, Vs, ringK, ringV, g.nf, g.cr, g.kn);

    const int pe0 = a.pe_index[slot];
    for (int j = g.j0; j < g.j1; ++j) {
        const int nfj = g.nf + j * t, clj = min(nfj, a.window);
        const int o = nfj - clj - g.first;          // staged row of this chunk's first key
        const int nk = clj + t;
        const int start = max(0, pe_after(pe0, j, a.chunk_size, a.pe_wrap) % a.pe_wrap - a.full_chunk);
        for (int i = tid; i < nk * NCH; i += ATT_THREADS) {        // row r = position start + r, swizzled by that position
            const int r = i / NCH, cc = i % NCH, pos = min(start + r, a.pos_rows - 1);
            *reinterpret_cast<uint4*>(Ps + r * DK + ((cc ^ ((start + r) & 7)) * EPC)) =
                *reinterpret_cast<const uint4*>(ptab_h + ((long long)h * a.pos_rows + pos) * DK + ((cc ^ (pos & 7)) * EPC));
        }
        for (int i = tid; i < t * DK; i += ATT_THREADS) {
            const int r = i / DK, d = i % DK;
            const float q = q32[(long long)(j * t + r) * 3 * D + h * DK + d];
            const int sw = r * DK + (((d >> 3) ^ (r & 7)) << 3) + (d & 7);
            quh[sw] = from_f<TA>(q + pos_u[h * DK + d]);
            qvh[sw] = from_f<TA>(q + pos_v[h * DK + d]);
        }
        __syncthreads();
        attn_chunk_mma<ATT_THREADS / 32>(Ks + o * DK, Vs + o * DK, g.first + o, Ps, start, quh, qvh, ph, sc, vrows, nk, t,
                                         out + (long long)(j * t) * D + h * DK, D);
        __syncthreads();                              // Ps / quh / ph / sc are restaged by the next chunk
    }
}

// The ring after a multi-chunk call of several groups per session: the last min(cnt[b] * t, cap) new K|V rows of session b at
// row frame % cap (fp16: chunk-swizzled by frame), as the same frames appended by single steps leave it.  One CTA per
// (session, head).
template <typename TA, bool SWZ>
__global__ void __launch_bounds__(ATT_THREADS)
chunks_append_ring_kernel(AttnStream a, const TA* __restrict__ qkv, TA* __restrict__ ring) {
    constexpr int EPC = 16 / sizeof(TA), NCH = DK / EPC;
    FO_PDL_TRIGGER();
    FO_PDL_WAIT();
    const int b = blockIdx.x, h = blockIdx.y, D = a.H * DK;
    const int kt = a.cnt[b] * a.t, r0 = max(0, kt - a.ring_cap), nr = kt - r0;
    const int nf = a.n_frames[a.ids[b]];
    qkv += (long long)(a.off[b] - a.off[0]) * a.t * 3 * D;
    TA* ringK = ring + (long long)a.ids[b] * a.ring_slot_stride + (long long)h * a.ring_cap * DK;
    TA* ringV = ringK + (long long)a.H * a.ring_cap * DK;
    for (int i = threadIdx.x; i < nr * NCH * 2; i += ATT_THREADS) {
        const int which = i / (nr * NCH), r = r0 + (i / NCH) % nr, c = i % NCH;
        const int pc = SWZ ? (c ^ ((nf + r) & 7)) : c;
        *reinterpret_cast<uint4*>((which ? ringV : ringK) + (long long)((nf + r) % a.ring_cap) * DK + pc * EPC) =
            *reinterpret_cast<const uint4*>(qkv + (long long)r * 3 * D + (which + 1) * D + h * DK + c * EPC);
    }
}
// ---------------------------------------------------------------------------------------------
constexpr int KT = 96;         // key tile: the shipped band of a 32-query block (64 left + 32 own keys) in one pass
constexpr int QB = 32;          // query rows per CTA
constexpr int QPW = QB / (ATT_THREADS / 32);   // queries per warp

// Which query tile of which utterance a CTA of the offline kernels takes, and where that utterance's rows are.  Padded
// (VL = false): tile blockIdx.x of utterance blockIdx.z, rows b * T.., keys cut by the pad mask ilens.  Packed (VL = true,
// attention_offline_packed): entry blockIdx.x of the tile table; T becomes the utterance's own length, every key of it valid.
template <bool VL>
__device__ __forceinline__ void utterance_tile(const AttnVarlen& vl, const int32_t* ilens, int& T, int& qb, int& b, int& klen,
                                               long long& row0) {
    if constexpr (VL) {
        const int2 tl = vl.tiles[blockIdx.x];
        b = tl.x;
        qb = tl.y;
        T = vl.lens[b];
        klen = T;
        row0 = vl.rows[b];
    } else {
        qb = blockIdx.x;
        b = blockIdx.z;
        klen = ilens ? min(ilens[b], T) : T;               // pad mask on keys (masks.py:110-120)
        row0 = (long long)b * T;
    }
}

// Full-utterance attention.  CTA = (32-query block, head, utterance), 4 warps x 8 queries.  The union of the block's
// key windows is walked in tiles of 96 keys (K, V and the rel-pos rows staged once per tile and shared by the 32
// queries; rows padded by 16 B so that lanes reading different rows hit different banks).  Scores are register
// blocked: lane = keys lane, lane+32, lane+64 of the tile against FOUR queries at a time, so every K / P chunk read
// from shared memory feeds four dot products and the query chunks are warp-wide broadcasts.  Window [start,end) of
// masks.py:50-56 and the pad mask (masks.py:110-120) are applied arithmetically; online softmax across tiles
// (unbounded left context works); PV with lane = output dims.  A row whose whole window is masked yields zeros
// (attention.py:396-397).  fp32 contexts; fp16 contexts run attention_offline_fa_kernel below.
template <bool VL>
__global__ void __launch_bounds__(ATT_THREADS)
attention_offline_kernel(const float* __restrict__ qkv, const float* __restrict__ q32, int T, int H,
                         const int32_t* __restrict__ ilens, int chunk, int left, const float* __restrict__ ptab,
                         const float* __restrict__ pos_u, const float* __restrict__ pos_v, float* __restrict__ out,
                         AttnVarlen vl) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    constexpr int EPC = 4, NCH = DK / EPC;
    constexpr int DKP = DK + EPC;                          // padded row (16 B): conflict-free 16-byte row reads
    constexpr int QG = 4;                                  // queries per register block
    float* Ks = reinterpret_cast<float*>(smem_raw);
    float* Vs = Ks + KT * DKP;
    float* Ps = Vs + KT * DKP;
    float* qu = Ps + KT * DKP;                             // QB x 64
    float* qv = qu + QB * DK;
    float* prob = qv + QB * DK;                            // warps x KT
    __shared__ int win[QB][2];

    const int h = blockIdx.y;
    int qb, b, klen;
    long long row0;
    utterance_tile<VL>(vl, ilens, T, qb, b, klen, row0);
    const int D = H * DK;
    const int q0 = qb * QB;
    const int nq = min(QB, T - q0);
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
        if (r < nq) q = *reinterpret_cast<const float4*>(q32 + (row0 + q0 + r) * 3 * D + h * DK + c);
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
            const float* src = qkv + (row0 + kt + j) * 3 * D + (which + 1) * D + h * DK + c * EPC;
            float* dst = (which == 0 ? Ks : Vs) + j * DKP + c * EPC;
            *reinterpret_cast<uint4*>(dst) = *reinterpret_cast<const uint4*>(src);
        }
        for (int i = tid; i < nk * (DK / 4); i += ATT_THREADS) {
            const int j = i / (DK / 4), c = i % (DK / 4);
            const float4 v4 = *reinterpret_cast<const float4*>(ptab + (long long)(kt + j) * D + h * DK + c * 4);
            *reinterpret_cast<float4*>(Ps + j * DKP + c * 4) = v4;
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
                        ld4(Ks + j * DKP + c * EPC, kv);
                        ld4(Ps + j * DKP + c * EPC, pp);
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
#pragma unroll 4
                for (int j = j0; j < j1; ++j) {
                    const float p = pr[j];
                    a0 = fmaf(p, Vs[j * DKP + 2 * lane], a0);
                    a1 = fmaf(p, Vs[j * DKP + 2 * lane + 1], a1);
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
            float* o = out + (row0 + q0 + r) * D + h * DK + 2 * lane;
            o[0] = o0[qi] * inv;
            o[1] = o1[qi] * inv;
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
template <bool VL>
__global__ void __launch_bounds__(ATT_THREADS, 4)
attention_offline_fa_kernel(const __half* __restrict__ qkv, const float* __restrict__ q32, int T, int H,
                            const int32_t* __restrict__ ilens, int chunk, int left, const __half* __restrict__ ptab_h,
                            int pos_rows, const float* __restrict__ pos_u, const float* __restrict__ pos_v,
                            __half* __restrict__ out, AttnVarlen vl) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    typedef __half TA;
    constexpr int NCH = 8;                                   // 16-byte chunks per 64-element row
    TA* tiles = reinterpret_cast<TA*>(smem_raw);             // [2 stages][K | P | V][FK][64]
    const int h = blockIdx.y;
    int qb, b, klen;
    long long row0;
    utterance_tile<VL>(vl, ilens, T, qb, b, klen, row0);
    const int D = H * DK;
    const int q0 = qb * FQ;
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
                if (key < k_hi) cp_async16(d2, qkv + (row0 + key) * 3 * D + (which == 0 ? 1 : 2) * D + h * DK + cc * 8);
                else *reinterpret_cast<uint4*>(d2) = make_uint4(0, 0, 0, 0);     // finite operands for the masked columns
            }
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
    };
    if (ntiles > 0) load_tile(0, 0);

    // (q+u), (q+v) A fragments of this warp's 16 queries: a0 (row g, k 2c..), a1 (row g+8), a2 (row g, k 2c+8..), a3 (row g+8)
    uint32_t qu[4][4], qv[4][4];
    {
        const float* qr0 = q32 + (row0 + min(r0, T - 1)) * 3 * D + h * DK;
        const float* qr1 = q32 + (row0 + min(r1, T - 1)) * 3 * D + h * DK;
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
            *reinterpret_cast<uint4*>(out + (row0 + row) * D + h * DK + cc * 8) = *reinterpret_cast<const uint4*>(ot + r * DK + cc * 8);
    }
}

__global__ void advance_sessions_kernel(const int32_t* __restrict__ ids, int n, int t, int chunk_size, int pe_wrap,
                                        int32_t* n_frames, int32_t* pe_index, int32_t* adapter_valid, int chunks,
                                        const int32_t* __restrict__ cnt) {
    FO_PDL_TRIGGER();
    FO_PDL_WAIT();
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= n) return;
    if (cnt) chunks = cnt[b];
    const int s = ids[b];
    if (n_frames) {
        n_frames[s] += chunks * t;
        pe_index[s] = pe_after(pe_index[s], chunks, chunk_size, pe_wrap);   // attention.py:107,120 (+chunk_size, not +t)
    }
    if (adapter_valid) adapter_valid[s] = adapter_valid[s] == 1 ? 2 : 1;
}

}  // namespace

template <typename TA>
int attention_stream(const AttnStream& a, const TA* qkv, const float* q32, TA* ring, const TA* ptab_h,
                     const float* pos_u, const float* pos_v, TA* out, cudaStream_t st) {
    if (a.n <= 0) return 0;
    const int t = a.t, prow = a.window + t;
    FO_CHECK(t <= STREAM_MAX_T, "attention_stream: %d frames per chunk exceeds %d", t, STREAM_MAX_T);
    FO_CHECK(a.ring_cap >= prow, "attention_stream: ring capacity %d < window %d + %d", a.ring_cap, a.window, t);
    using Kernel = void (*)(AttnStream, const TA*, const float*, TA*, const TA*, const float*, const float*, TA*);
    // [0] one chunk, [1] one chunk summed from the QKV GEMM's split-K partials (fp16 only)
    std::array<Kernel, 2> kernels;
    size_t smem;
    if constexpr (sizeof(TA) == 2) {
        kernels = {attention_stream_mma_kernel<false>, attention_stream_mma_kernel<true>};
        smem = (size_t)mma_unit_layout(a.window, t).bytes;
    } else {
        kernels = {attention_stream_kernel, attention_stream_kernel};
        smem = (size_t)3 * prow * DK * 4 + (size_t)2 * t * DK * 4 + (size_t)t * prow * 4;
    }
    FO_CHECK(smem <= 160 * 1024, "attention_stream: window too large for shared memory");
    static std::atomic<bool> opted_in{false};      // past 48 KB (window + t > ~115 keys, e.g. left_chunks 31) a launch needs the opt-in
    if (!opted_in) {
        for (Kernel k : kernels) FO_CUDA(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024));
        opted_in = true;
    }
    const Kernel kern = kernels[a.nsplit > 0 ? 1 : 0];
    FO_CUDA(launch_pdl(kern, dim3(a.n, a.H), dim3(ATT_THREADS), smem, st, a, qkv, q32, ring, ptab_h, pos_u, pos_v, out));
    FO_LAUNCHED();
#ifdef FO_TC_TRACE_BUILD
    if (sizeof(TA) == 2 && getenv("FO_TC_TRACE") && st == nullptr) {
        cudaStreamSynchronize(st);
        unsigned long long hb[16];
        cudaMemcpyFromSymbol(hb, g_attn_trace, sizeof(hb));
        fprintf(stderr, "attn_trace n=%d:", a.n);
        for (int i : {1, 2, 3, 4, 5, 9}) fprintf(stderr, " t%d=%lld", i, (long long)(hb[i] - hb[0]));
        fprintf(stderr, " ns\n");
    }
#endif
    FO_CUDA(cudaGetLastError());
    return 0;
}
template int attention_stream<float>(const AttnStream&, const float*, const float*, float*, const float*, const float*, const float*, float*, cudaStream_t);

template <typename TA>
int attention_chunks(const AttnStream& a, int groups, const TA* qkv, const float* q32, TA* ring, const TA* ptab_h,
                     const float* pos_u, const float* pos_v, TA* out, cudaStream_t st) {
    if (a.n <= 0) return 0;
    const int t = a.t, rows = a.window + a.chunks * t, prow = a.window + t;     // staged keys, keys of one chunk
    FO_CHECK(t <= STREAM_MAX_T && a.ring_cap >= prow && a.cnt && a.off && groups >= 1, "attention_chunks: bad geometry");
    FO_CHECK(rows <= STREAM_CHUNKS_MAX_KEYS, "attention_chunks: window %d + %d chunks x %d frames exceeds %d keys", a.window,
             a.chunks, t, STREAM_CHUNKS_MAX_KEYS);
    size_t smem;
    void (*kern)(AttnStream, const TA*, const float*, TA*, const TA*, const float*, const float*, TA*);
    if constexpr (sizeof(TA) == 2) {
        kern = attention_chunks_mma_kernel;
        const int krows = ((rows + 15) & ~15) + 16, vrows = (prow + 15) & ~15;
        smem = (size_t)(2 * krows + vrows) * DK * 2 + (size_t)2 * t * DK * 2 + (size_t)t * vrows * 2 + (size_t)t * std::max(vrows, DK) * 4;
    } else {
        kern = attention_chunks_kernel;
        smem = (size_t)(2 * rows + prow) * DK * 4 + (size_t)2 * t * DK * 4 + (size_t)t * prow * 4;
    }
    static std::atomic<bool> opted_in{false};      // past 48 KB a launch needs the opt-in
    if (!opted_in) {
        FO_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024));
        opted_in = true;
    }
    FO_CUDA(launch_pdl(kern, dim3(a.n, a.H, groups), dim3(ATT_THREADS), smem, st, a, qkv, q32, ring, ptab_h, pos_u, pos_v, out));
    FO_LAUNCHED();
    FO_CUDA(cudaGetLastError());
    if (groups > 1) {                  // several CTAs read a session's ring: the append waits for the whole grid
        FO_CUDA(launch_pdl(chunks_append_ring_kernel<TA, sizeof(TA) == 2>, dim3(a.n, a.H), dim3(ATT_THREADS), 0, st, a, qkv, ring));
        FO_LAUNCHED();
        FO_CUDA(cudaGetLastError());
    }
    return 0;
}
template int attention_chunks<float>(const AttnStream&, int, const float*, const float*, float*, const float*, const float*, const float*, float*, cudaStream_t);
template int attention_chunks<__half>(const AttnStream&, int, const __half*, const float*, __half*, const __half*, const float*, const float*, __half*, cudaStream_t);
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

// One launcher for both forms: vl == null is the padded batch (grid x = query tiles, z = utterances), else the packed one
// (grid x = vl->n tile table entries).
template <typename TA>
int attention_offline_any(const TA* qkv, const float* q32, int B, int T, int H, const int32_t* ilens, int chunk, int left,
                          const float* ptab, const TA* ptab_h, int pos_rows, const float* pos_u, const float* pos_v, TA* out,
                          const AttnVarlen* vl, cudaStream_t st) {
    if (B <= 0 || T <= 0 || (vl && vl->n <= 0)) return 0;
    const AttnVarlen v = vl ? *vl : AttnVarlen();
    if constexpr (sizeof(TA) == 2) {
        if (!ptab_h || T > pos_rows) return 1;
        const size_t smem = (size_t)2 * 3 * FK * DK * 2;      // 48 KB: double-buffered K | P | V tiles
        static std::atomic<bool> attr_set{false};
        if (!attr_set) {
            FO_CUDA(cudaFuncSetAttribute(attention_offline_fa_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024));
            FO_CUDA(cudaFuncSetAttribute(attention_offline_fa_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024));
            attr_set = true;
        }
        if (vl)
            attention_offline_fa_kernel<true><<<dim3(v.n, H, 1), ATT_THREADS, smem, st>>>(qkv, q32, T, H, ilens, chunk, left, ptab_h,
                                                                                         pos_rows, pos_u, pos_v, out, v);
        else
            attention_offline_fa_kernel<false><<<dim3(cdiv(T, FQ), H, B), ATT_THREADS, smem, st>>>(qkv, q32, T, H, ilens, chunk, left,
                                                                                                  ptab_h, pos_rows, pos_u, pos_v, out, v);
    } else {
        const size_t smem = (size_t)3 * KT * (DK + 4) * 4 + (size_t)2 * QB * DK * 4 + (size_t)(ATT_THREADS / 32) * KT * 4;
        static std::atomic<bool> attr_set{false};
        if (!attr_set) {
            FO_CUDA(cudaFuncSetAttribute(attention_offline_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024));
            FO_CUDA(cudaFuncSetAttribute(attention_offline_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024));
            attr_set = true;
        }
        if (vl)
            attention_offline_kernel<true><<<dim3(v.n, H, 1), ATT_THREADS, smem, st>>>(qkv, q32, T, H, ilens, chunk, left, ptab, pos_u,
                                                                                      pos_v, out, v);
        else
            attention_offline_kernel<false><<<dim3(cdiv(T, QB), H, B), ATT_THREADS, smem, st>>>(qkv, q32, T, H, ilens, chunk, left, ptab,
                                                                                               pos_u, pos_v, out, v);
    }
    FO_LAUNCHED();
    FO_CUDA(cudaGetLastError());
    return 0;
}
template <typename TA>
int attention_offline(const TA* qkv, const float* q32, int B, int T, int H, const int32_t* ilens, int chunk, int left,
                      const float* ptab, const TA* ptab_h, int pos_rows, const float* pos_u, const float* pos_v, TA* out,
                      cudaStream_t st) {
    return attention_offline_any<TA>(qkv, q32, B, T, H, ilens, chunk, left, ptab, ptab_h, pos_rows, pos_u, pos_v, out, nullptr, st);
}
template <typename TA>
int attention_offline_packed(const TA* qkv, const float* q32, const AttnVarlen& vl, int B, int tmax, int H, int chunk, int left,
                             const float* ptab, const TA* ptab_h, int pos_rows, const float* pos_u, const float* pos_v, TA* out,
                             cudaStream_t st) {
    return attention_offline_any<TA>(qkv, q32, B, tmax, H, nullptr, chunk, left, ptab, ptab_h, pos_rows, pos_u, pos_v, out, &vl, st);
}
int attention_offline_tile_rows(int is16) { return is16 ? FQ : QB; }
template int attention_offline<float>(const float*, const float*, int, int, int, const int32_t*, int, int, const float*, const float*, int, const float*, const float*, float*, cudaStream_t);
template int attention_offline<__half>(const __half*, const float*, int, int, int, const int32_t*, int, int, const float*, const __half*, int, const float*, const float*, __half*, cudaStream_t);
template int attention_offline_packed<float>(const float*, const float*, const AttnVarlen&, int, int, int, int, int, const float*, const float*, int, const float*, const float*, float*, cudaStream_t);
template int attention_offline_packed<__half>(const __half*, const float*, const AttnVarlen&, int, int, int, int, int, const float*, const __half*, int, const float*, const float*, __half*, cudaStream_t);

int advance_sessions(const int32_t* ids, int n, int t, int chunk_size, int pe_wrap, int32_t* n_frames,
                      int32_t* pe_index, int32_t* adapter_valid, cudaStream_t st, int chunks, const int32_t* cnt) {
    if (n <= 0) return 0;
    FO_CUDA(launch_pdl(advance_sessions_kernel, dim3(cdiv(n, 128)), dim3(128), 0, st, ids, n, t, chunk_size, pe_wrap, n_frames, pe_index, adapter_valid,
                       chunks, cnt));
    FO_LAUNCHED();
    FO_CUDA(cudaGetLastError());
    return 0;
}

FO_TR_BIND_DEF(trace_bind_attention)

}  // namespace fo
