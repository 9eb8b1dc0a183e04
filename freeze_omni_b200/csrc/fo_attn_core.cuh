// Streaming chunk attention core, shared by the kernels of fo_attention.cu (single-chunk and multi-chunk, fp16 and fp32)
// and the attention phase of the layer-stack kernel (fo_stack.cu):
//     score[i][j] = ((q_i + u) . K_j + (q_i + v) . P_j) / 8,   fp32 softmax over the chunk's nk keys,   out_i = sum_j p_ij V_j
// The kernels differ only in how they stage K / V / P / Q in shared memory; everything from the staged rows to the stored
// output rows is here, so masking, swizzle and softmax exist once per precision.
#pragma once
#include "fo_common.cuh"

namespace fo {

constexpr int DK = 64;          // head dimension

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
__device__ __forceinline__ void mma16816(float (&d)[4], const uint32_t (&a)[4], const uint32_t (&b)[2]) {
    asm volatile(
        "mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
        : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
        : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b[0]), "r"(b[1]));
}
__device__ __forceinline__ uint32_t lds32(const __half* p) { return *reinterpret_cast<const uint32_t*>(p); }
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
__device__ __forceinline__ void ld4(const float* p, float (&v)[4]) {
    const float4 t = *reinterpret_cast<const float4*>(p);
    v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
}

// One thread: the cl cached rows of frames [first, first + cl) of one head's ring (K and V, cap rows each) -> rows 0..cl-1
// of Ks / Vs, in two runs when the window wraps past the ring's end, and np rel-pos rows from prow -> Ps, all completing on
// `bar` (initialised by the caller).
template <typename T>
__device__ __forceinline__ void ring_window_copy(const T* ringK, const T* ringV, int cap, int first, int cl, T* Ks, T* Vs,
                                                 const T* prow, T* Ps, int np, uint64_t* bar) {
    const uint32_t rowb = DK * sizeof(T);
    const int p0 = first % cap;
    const int len1 = min(cl, cap - p0), len2 = cl - len1;
    mbar_expect_tx(bar, (2u * cl + np) * rowb);
    if (np > 0) bulk_g2s(Ps, prow, np * rowb, bar);
    if (len1 > 0) {
        bulk_g2s(Ks, ringK + (long long)p0 * DK, len1 * rowb, bar);
        bulk_g2s(Vs, ringV + (long long)p0 * DK, len1 * rowb, bar);
    }
    if (len2 > 0) {
        bulk_g2s(Ks + len1 * DK, ringK, len2 * rowb, bar);
        bulk_g2s(Vs + len1 * DK, ringV, len2 * rowb, bar);
    }
}

// Shared-memory layout (byte offsets) of one fp16 single-chunk unit with rows = window + t staged keys
// (attention_stream_mma_kernel, the stack kernel's attention phase):
//   K, P    rows x 64 each; a partial last key tile reads on into the next array (those scores are masked)
//   V       vrows = round16(rows) x 64, zero rows behind the last key
//   qu, qv  (q+u), (q+v) as fp16, t x 64 each
//   ph      normalised probabilities, t x vrows (fp16)
//   sc      scores t x vrows (fp32), later the output tile t x 64
struct MmaUnitLayout {
    int vrows, p, v, qu, qv, ph, sc, bytes;
};
__host__ __device__ inline MmaUnitLayout mma_unit_layout(int window, int t) {
    const int rows = window + t;
    MmaUnitLayout l;
    l.vrows = (rows + 15) & ~15;
    l.p = rows * DK * 2;
    l.v = 2 * l.p;
    l.qu = l.v + l.vrows * DK * 2;
    l.qv = l.qu + t * DK * 2;
    l.ph = l.qv + t * DK * 2;
    l.sc = l.ph + t * l.vrows * 2;
    l.bytes = l.sc + t * (l.vrows > DK ? l.vrows : DK) * 4;
    return l;
}

// fp16 core of one chunk on mma.sync.m16n8k16 (fp32 accumulate; the attention core is 1 % of the FLOPs, far too small for
// tcgen05), run by all NWARPS warps of the CTA:
//   S^T (keys x queries) = K (keys x 64) . (q+u)^T  +  P (keys x 64) . (q+v)^T     key tiles of 16 over the warps
//   O^T (64 x queries)   = V^T (64 x keys) . prob^T                                   one 16-dim tile per warp, warps 0-3
// then fp32 softmax, probabilities normalised and rounded to fp16, and out[q * ostride + d] = O[q][d] as fp16.
// Ks / Vs point at the chunk's first key, of frame number f0; Ps at the rel-pos row of position `start`.  16-byte chunk c
// of a row lives at chunk c ^ (x & 7), x = the frame number (K, V), the position (P) or the query row (quh, qvh), so the
// fragment loads of rows read together hit different banks.  ph / sc are t rows of `vrows` >= round16(nk) (sc at least
// 64) columns.  Preconditions: the caller has synchronised the CTA after staging; K and P are readable up to
// round16(nk) rows, with any finite or masked values past nk; V is finite up to round16(nk) rows (probability 0 x V).
// Ends with the CTA synchronised after the scratch reads; the output stores are the last thing it does.
template <int NWARPS>
__device__ __forceinline__ void attn_chunk_mma(const __half* Ks, const __half* Vs, int f0, const __half* Ps, int start,
                                               const __half* quh, const __half* qvh, __half* ph, float* sc, int vrows, int nk,
                                               int t, __half* out, long long ostride) {
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int g = lane >> 2, c = lane & 3;
    // ---- scores: S^T tile (16 keys x 8 queries) per MMA chain ----
    for (int k0 = warp * 16; k0 < nk; k0 += 16 * NWARPS) {
        float d[4] = {0.f, 0.f, 0.f, 0.f};
        const int kk0 = (f0 + k0 + g) & 7, kk1 = (f0 + k0 + g + 8) & 7;
        const int kp0 = (start + k0 + g) & 7, kp1 = (start + k0 + g + 8) & 7;
        const __half* kr0 = Ks + (k0 + g) * DK + c * 2;
        const __half* kr1 = Ks + (k0 + g + 8) * DK + c * 2;
        const __half* pr0 = Ps + (k0 + g) * DK + c * 2;
        const __half* pr1 = Ps + (k0 + g + 8) * DK + c * 2;
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
    // ---- softmax (fp32), probabilities normalised and rounded to fp16 ----
    for (int i = warp; i < t; i += NWARPS) {
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
    // ---- PV: O^T tile (16 dims x 8 queries) per warp ----
    if (warp < DK / 16) {
        float d[4] = {0.f, 0.f, 0.f, 0.f};
        const int dim0 = warp * 16;
        const int mi = lane >> 3, r = lane & 7;
        for (int key0 = 0; key0 < nk; key0 += 16) {
            uint32_t af[4], bf[2];
            const int vrow = key0 + r + ((mi & 2) ? 8 : 0);
            const __half* ap = Vs + vrow * DK + ((((dim0 >> 3) + (mi & 1)) ^ ((f0 + vrow) & 7)) << 3);
            asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];"
                         : "=r"(af[0]), "=r"(af[1]), "=r"(af[2]), "=r"(af[3])
                         : "r"(smem_u32(ap)));
            bf[0] = g < t ? lds32(ph + g * vrows + key0 + c * 2) : 0u;
            bf[1] = g < t ? lds32(ph + g * vrows + key0 + 8 + c * 2) : 0u;
            mma16816(d, af, bf);
        }
        const int q0 = c * 2;
        if (q0 < t) { sc[q0 * DK + dim0 + g] = d[0]; sc[q0 * DK + dim0 + g + 8] = d[2]; }
        if (q0 + 1 < t) { sc[(q0 + 1) * DK + dim0 + g] = d[1]; sc[(q0 + 1) * DK + dim0 + g + 8] = d[3]; }
    }
    __syncthreads();
    for (int i = tid; i < t * (DK / 2); i += NWARPS * 32) {
        const int q = i / (DK / 2), pr = i % (DK / 2);
        *reinterpret_cast<uint32_t*>(out + q * ostride + 2 * pr) = pack2<__half>(sc[q * DK + 2 * pr], sc[q * DK + 2 * pr + 1]);
    }
}

// fp32 core of one chunk in scalar FFMA (the parity form of fp32 contexts), 4 warps, warp = query row:
//   score  lane = keys lane, lane+32, lane+64, lane+96: ((q+u).K_j + (q+v).P_j)/8, the 16-byte chunks of a row visited in a
//          lane-rotated order (the 8 lanes of a shared-memory phase touch 8 different bank groups); scores stay in registers
//   soft   warp-shuffle max / sum, exponentials to the query's row of `prob` (pstride >= nk columns)
//   PV     lane = output dims 2*lane, 2*lane+1, loop over the keys; out[i * ostride + d]
// Ks / Vs point at the chunk's first key, Ps at its rel-pos row; qu / qv hold (q+u), (q+v) as t x 64 fp32.  Precondition: the
// caller has synchronised the CTA after staging; nk <= 128.
__device__ __forceinline__ void attn_chunk_ffma(const float* Ks, const float* Vs, const float* Ps, const float* qu, const float* qv,
                                                float* prob, int pstride, int nk, int t, float* out, long long ostride) {
    constexpr int EPC = 4, NCH = DK / EPC, KPL = 4;          // floats per 16-byte chunk, chunks per row, keys per lane
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    for (int i = warp; i < t; i += 4) {
        const float* qui = qu + i * DK;
        const float* qvi = qv + i * DK;
        float sc[KPL];
#pragma unroll
        for (int k = 0; k < KPL; ++k) sc[k] = 0.f;
#pragma unroll 2
        for (int c = 0; c < NCH; ++c) {
            const int cc = (c + lane) & (NCH - 1);
            float au[EPC], av[EPC];
            ld4(qui + cc * EPC, au);
            ld4(qvi + cc * EPC, av);
#pragma unroll
            for (int k = 0; k < KPL; ++k) {
                const int j = lane + 32 * k;
                if (j < nk) {
                    float kv[EPC], pp[EPC];
                    ld4(Ks + j * DK + cc * EPC, kv);
                    ld4(Ps + j * DK + cc * EPC, pp);
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
        float* pr = prob + i * pstride;
#pragma unroll
        for (int k = 0; k < KPL; ++k) {
            const int j = lane + 32 * k;
            if (j < nk) {
                const float e = __expf(sc[k] - m);
                pr[j] = e;
                ssum += e;
            }
        }
        ssum = warp_sum(ssum);
        __syncwarp();
        const float inv = 1.f / ssum;
        float o0 = 0.f, o1 = 0.f;
#pragma unroll 4
        for (int j = 0; j < nk; ++j) {
            const float p = pr[j];
            o0 = fmaf(p, Vs[j * DK + 2 * lane], o0);
            o1 = fmaf(p, Vs[j * DK + 2 * lane + 1], o1);
        }
        float* op = out + i * ostride + 2 * lane;
        op[0] = o0 * inv;
        op[1] = o1 * inv;
    }
}

}  // namespace fo
