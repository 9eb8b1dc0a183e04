// Session snapshots: gather n session slots into n records (fo_session_save) and scatter n records into n slots
// (fo_session_restore), one launch each.  The record format is defined in fo_api.cu; this file only moves bytes.
//
// Grid: per session, one CTA per (layer, K|V, head) unit of the KV ring plus one CTA for the header and the flat fp32
// sections.  A unit is the last cl = min(n_frames, window) frames of one head's ring, rows of 64 elements: at most two
// contiguous runs of the ring (split where the ring wraps), copied in 16-byte chunks.  16-bit rings hold chunk c of the
// row of frame f at chunk c ^ (f & 7) (the attention kernels' swizzle), records hold it at c: the chunk index is
// (un)swizzled in flight.  Record rows past cl are zero.  A pure HBM copy: every thread keeps 4 chunks in flight.
#include "fo_common.cuh"

namespace fo {
namespace {

constexpr int SNAP_THREADS = 256;
constexpr int SNAP_ILP = 4;

template <bool PACK>
__device__ __forceinline__ void kv_unit(const SnapArgs& a, int b, int slot, int u, int nf) {
    const int h = u % a.H, kv = (u / a.H) & 1, l = u / (2 * a.H);
    const int nch = 4 * a.esz;                                         // 16-byte chunks per 64-element row
    const int cl = min(nf, a.window);
    const int r0 = (nf - cl) % a.cap;                                  // ring row of the oldest frame in the window
    uint4* ring = reinterpret_cast<uint4*>(a.ring) + ((((long long)l * a.S + slot) * 2 + kv) * a.H + h) * a.cap * nch;
    uint4* rec = reinterpret_cast<uint4*>(a.rec + (long long)b * a.rec_bytes + a.kv_off) +
                 (((long long)l * 2 + kv) * a.H + h) * a.window * nch;
    const int total = (PACK ? a.window : cl) * nch;
    const bool swz = a.esz == 2;
    for (int i0 = threadIdx.x; i0 < total; i0 += SNAP_THREADS * SNAP_ILP) {
        uint4 v[SNAP_ILP];
        int dst[SNAP_ILP];
#pragma unroll
        for (int k = 0; k < SNAP_ILP; ++k) {
            const int i = i0 + k * SNAP_THREADS;
            dst[k] = -1;
            if (i >= total) continue;
            const int j = i / nch, c = i % nch;                        // record row j = frame nf - cl + j
            int row = r0 + j;
            if (row >= a.cap) row -= a.cap;                            // second run: from the ring's start
            const int rc = row * nch + (swz ? c ^ ((nf - cl + j) & 7) : c);
            if (PACK) {
                v[k] = j < cl ? __ldg(ring + rc) : make_uint4(0, 0, 0, 0);
                dst[k] = i;
            } else {
                v[k] = __ldg(rec + i);
                dst[k] = rc;
            }
        }
#pragma unroll
        for (int k = 0; k < SNAP_ILP; ++k)
            if (dst[k] >= 0) (PACK ? rec : ring)[dst[k]] = v[k];
    }
}

// flat byte copy, 16-byte chunks when both ends and the size allow it (every section of the shipped model does), else words
__device__ __forceinline__ void flat_copy(char* dst, const char* src, long long bytes) {
    if ((((uintptr_t)dst | (uintptr_t)src | (uintptr_t)bytes) & 15) == 0) {
        for (long long i = threadIdx.x; i < bytes / 16; i += SNAP_THREADS)
            reinterpret_cast<uint4*>(dst)[i] = src ? __ldg(reinterpret_cast<const uint4*>(src) + i) : make_uint4(0, 0, 0, 0);
    } else {
        for (long long i = threadIdx.x; i < bytes / 4; i += SNAP_THREADS)
            reinterpret_cast<int32_t*>(dst)[i] = src ? reinterpret_cast<const int32_t*>(src)[i] : 0;
    }
}

template <bool PACK>
__device__ __forceinline__ void session_copy_cta(const SnapArgs& a) {
    const int units = a.ring ? a.L * 2 * a.H : 0;
    const int b = blockIdx.x / (units + 1), u = blockIdx.x % (units + 1);
    const int slot = a.ids[b];
    const int32_t* hdr = reinterpret_cast<const int32_t*>(a.rec + (long long)b * a.rec_bytes);
    if (u < units) {
        kv_unit<PACK>(a, b, slot, u, PACK ? a.n_frames[slot] : hdr[SNAP_W_NFRAMES]);
        return;
    }
    // header, scalar state and the flat sections of session b
    const int live = PACK ? a.ad_valid[slot] : 0;                      // adapter cache: 0 none, 1 / 2 half 0 / 1 live
    if (PACK) {
        int32_t* out = reinterpret_cast<int32_t*>(a.rec + (long long)b * a.rec_bytes);
        for (int w = threadIdx.x; w < SNAP_HDR_WORDS; w += SNAP_THREADS) {
            int32_t v = a.hdr[w];
            if (w == SNAP_W_NFRAMES) v = a.n_frames ? a.n_frames[slot] : 0;
            if (w == SNAP_W_PE) v = a.pe_index ? a.pe_index[slot] : 0;
            if (w == SNAP_W_ADVALID) v = live != 0;
            out[w] = v;
        }
    } else if (threadIdx.x == 0) {
        if (a.n_frames) a.n_frames[slot] = hdr[SNAP_W_NFRAMES];
        if (a.pe_index) a.pe_index[slot] = hdr[SNAP_W_PE];
        a.ad_valid[slot] = hdr[SNAP_W_ADVALID] ? 1 : 0;             // 1: half 0 is live, where the cache is written below
    }
    for (int s = 0; s < a.nseg; ++s) {
        const SnapSeg& g = a.seg[s];
        char* st = g.base + slot * g.slot_stride;
        char* rec = a.rec + (long long)b * a.rec_bytes + g.rec_off;
        if (PACK) {
            const char* src = st;
            if (g.adapter_half) src = live == 0 ? nullptr : st + (live == 2 ? g.bytes : 0);   // no cache yet: zeros
            flat_copy(rec, src, g.bytes);
            for (long long i = g.bytes / 4 + threadIdx.x; i < ((g.bytes + 255) & ~255LL) / 4; i += SNAP_THREADS)
                reinterpret_cast<int32_t*>(rec)[i] = 0;                // padding to the next section: records are deterministic
        } else {
            flat_copy(st, rec, g.bytes);
        }
    }
}

__global__ void __launch_bounds__(SNAP_THREADS) session_pack_kernel(const SnapArgs a) { session_copy_cta<true>(a); }
__global__ void __launch_bounds__(SNAP_THREADS) session_unpack_kernel(const SnapArgs a) { session_copy_cta<false>(a); }

int session_copy(void (*kernel)(SnapArgs), const SnapArgs& a, cudaStream_t st) {
    if (a.n <= 0) return 0;
    const int units = a.ring ? a.L * 2 * a.H : 0;
    kernel<<<(unsigned)a.n * (units + 1), SNAP_THREADS, 0, st>>>(a);
    FO_LAUNCHED();
    FO_CUDA(cudaGetLastError());
    return 0;
}

}  // namespace

int session_pack(const SnapArgs& a, cudaStream_t st) { return session_copy(session_pack_kernel, a, st); }
int session_unpack(const SnapArgs& a, cudaStream_t st) { return session_copy(session_unpack_kernel, a, st); }

}  // namespace fo
