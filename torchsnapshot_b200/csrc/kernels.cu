// sm_100a copy kernels of the checkpoint data plane.
//
//   tsnap_bulk_copy_kernel : dense 16B-aligned runs.  One warp per CTA, one elected lane drives a
//       ring of shared-memory stages with the bulk async-copy engine (TMA, 1-D form):
//       cp.async.bulk global->shared (mbarrier complete_tx) then cp.async.bulk shared->global
//       (bulk_group).  No register staging, ~10 instructions per 16 KiB.
//   tsnap_lsu_copy_kernel  : everything else — dense runs at odd alignment (slab members sit back
//       to back with no padding, T:batcher.py:307), strided views (narrow on dim != 0, transposes,
//       reshard-on-load overlap boxes, T:io_preparers/sharded_tensor.py:285-298) and fused dtype
//       casts.  Destination-aligned 16 B stores, widest naturally aligned loads.
//   (transposes and short-run column shards the TMA unit can address: transpose_tma.cu)
//
// Both are persistent: grid = SMs x resident CTAs, tiles taken round-robin from a host-built tile
// table (plan.h).  HBM-bound byte movement: algorithmic traffic = 2 x payload bytes.
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <stdint.h>
#include <stdlib.h>

#include "kernels.h"
#include "ptx.cuh"

namespace tsnap {

// ------------------------------------------------------------------------------------------------
// bulk (TMA) copy kernel
// ------------------------------------------------------------------------------------------------
// Piece = one <= kStageBytes slice of a tile.  A cursor walks this CTA's tiles and yields pieces in
// order; the same order is used for loads and stores, so stage = piece_ordinal % kStages.
struct PieceCursor {
    const Member* members;
    const Tile* tiles;
    uint32_t ntiles;
    uint32_t tile;       // current tile (global index)
    uint64_t pos, end;   // byte cursor inside the current member
    const char* src;
    char* dst;
    uint32_t stride;
    bool open;
};

__device__ __forceinline__ bool cursor_next(PieceCursor& c, uint32_t stage_bytes, const char** src, char** dst,
                                            uint32_t* bytes) {
    while (true) {
        if (c.open && c.pos < c.end) {
            uint64_t n = c.end - c.pos;
            if (n > stage_bytes) n = stage_bytes;
            *src = c.src + c.pos;
            *dst = c.dst + c.pos;
            *bytes = (uint32_t)n;
            c.pos += n;
            return true;
        }
        if (c.open) c.tile += c.stride;
        if (c.tile >= c.ntiles) return false;
        const Tile t = c.tiles[c.tile];
        const Member* m = c.members + t.member;
        const uint64_t mbytes = m->bytes;
        c.src = reinterpret_cast<const char*>(m->src);
        c.dst = reinterpret_cast<char*>(m->dst);
        c.pos = (uint64_t)t.index * kTileBulk;
        c.end = c.pos + kTileBulk;
        if (c.end > mbytes) c.end = mbytes;
        c.open = true;
    }
}

template <int kStages, int kStageBytes>
__global__ void __launch_bounds__(32) tsnap_bulk_copy_kernel(const Member* __restrict__ members,
                                                             const Tile* __restrict__ tiles, uint32_t ntiles) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    // [kStages * kStageBytes data][kStages mbarriers]
    unsigned char* data = smem_raw;
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem_raw + kStages * kStageBytes);
    if (threadIdx.x != 0) return;  // one elected lane drives the copy engine

    for (int s = 0; s < kStages; ++s) mbar_init(smem_u32(&bars[s]), 1);
    fence_mbar_init();
    fence_proxy_async_smem();
    const uint64_t policy = policy_evict_first();

    PieceCursor cur;
    cur.members = members;
    cur.tiles = tiles;
    cur.ntiles = ntiles;
    cur.tile = blockIdx.x;
    cur.stride = gridDim.x;
    cur.open = false;
    cur.pos = cur.end = 0;

    char* st_dst[kStages];
    uint32_t st_bytes[kStages];
    uint32_t issued = 0, stored = 0;

    const char* src;
    char* dst;
    uint32_t bytes;
    // prologue: fill the ring
#pragma unroll
    for (int s = 0; s < kStages; ++s) {
        if (issued == (uint32_t)s && cursor_next(cur, kStageBytes, &src, &dst, &bytes)) {
            const uint32_t bar = smem_u32(&bars[s]);
            mbar_expect_tx(bar, bytes);
            bulk_g2s(smem_u32(data + s * kStageBytes), src, bytes, bar, policy);
            st_dst[s] = dst;
            st_bytes[s] = bytes;
            ++issued;
        }
    }
    while (stored < issued) {
        const uint32_t s = stored % kStages;
        mbar_wait(smem_u32(&bars[s]), (stored / kStages) & 1);
        // bytes landed through the async proxy and are read back by it; the fence orders the
        // mbarrier observation before the store is issued.
        fence_proxy_async_smem();
        char* d = nullptr;
        uint32_t b = 0;
#pragma unroll
        for (int k = 0; k < kStages; ++k)
            if (k == (int)s) {
                d = st_dst[k];
                b = st_bytes[k];
            }
        bulk_s2g(d, smem_u32(data + s * kStageBytes), b);
        bulk_commit();
        ++stored;
        // the stage written out one iteration ago is free once all but the newest store group
        // have finished reading shared memory
        if (stored >= 2) {
            bulk_wait_read<1>();
            if (cursor_next(cur, kStageBytes, &src, &dst, &bytes)) {
                const uint32_t fs = (stored - 2) % kStages;
                const uint32_t bar = smem_u32(&bars[fs]);
                mbar_expect_tx(bar, bytes);
                bulk_g2s(smem_u32(data + fs * kStageBytes), src, bytes, bar, policy);
#pragma unroll
                for (int k = 0; k < kStages; ++k)
                    if (k == (int)fs) {
                        st_dst[k] = dst;
                        st_bytes[k] = bytes;
                    }
                ++issued;
            }
        }
    }
    bulk_wait_all<0>();
}

// ------------------------------------------------------------------------------------------------
// rows kernel: strided members with long 16 B-aligned runs, run by run through the copy engine
// ------------------------------------------------------------------------------------------------
// Same ring as the dense kernel (kStages x kStageBytes of shared memory, mbarrier per stage, bulk async-groups
// for the stores), but warp-collective: a stage holds up to kStageBytes of the member's LOGICAL bytes — a
// sequence of run segments — and the 32 lanes issue the per-run cp.async.bulk requests in parallel.  A side
// whose runs are adjacent (the wire image on save, the file image on restore) is moved with ONE request per
// stage.  No data passes through registers (SASS: UBLKCP.S.G / UBLKCP.G.S only).
struct RowsPiece {
    uint32_t member;  // index into the member table
    uint64_t pos;     // logical byte position inside the member
    uint32_t n;       // logical bytes
};

struct RowsCursor {
    const Member* members;
    const Tile* tiles;
    uint32_t ntiles, tile, stride;
    uint64_t pos, end;
    uint32_t member;
    bool open;
};

__device__ __forceinline__ bool rows_next(RowsCursor& c, uint32_t stage_bytes, RowsPiece* out) {
    while (true) {
        if (c.open && c.pos < c.end) {
            uint64_t n = c.end - c.pos;
            if (n > stage_bytes) n = stage_bytes;
            out->member = c.member;
            out->pos = c.pos;
            out->n = (uint32_t)n;
            c.pos += n;
            return true;
        }
        if (c.open) c.tile += c.stride;
        if (c.tile >= c.ntiles) return false;
        const Tile t = c.tiles[c.tile];
        c.member = t.member;
        const uint64_t mbytes = c.members[t.member].bytes;
        c.pos = (uint64_t)t.index * kTileBulk;
        c.end = c.pos + kTileBulk;
        if (c.end > mbytes) c.end = mbytes;
        c.open = true;
    }
}

__device__ __forceinline__ void rows_offsets(const Member& m, uint64_t row, int64_t* so, int64_t* dofs) {
    if (m.nouter == 1) {
        *so = (int64_t)row * m.sstride[0];
        *dofs = (int64_t)row * m.dstride[0];
        return;
    }
    int64_t s = 0, d = 0;
    for (int i = (int)m.nouter - 1; i >= 0; --i) {
        const uint64_t sz = (uint64_t)m.osize[i];
        const uint64_t idx = row % sz;
        row /= sz;
        s += (int64_t)idx * m.sstride[i];
        d += (int64_t)idx * m.dstride[i];
    }
    *so = s;
    *dofs = d;
}

// issues the copy-engine requests of one piece on one side.  kLoad: global -> stage (completion on `bar`),
// else stage -> global (bulk async-group of the issuing lane).
template <bool kLoad>
__device__ __forceinline__ void rows_issue(const Member& m, uint64_t pos, uint32_t n, uint32_t stage_smem, uint32_t bar,
                                           uint64_t policy, uint32_t lane) {
    const bool dense = (m.shift & (kLoad ? kRowsSrcDense : kRowsDstDense)) != 0;
    if (dense) {
        if (lane == 0) {
            if (kLoad) bulk_g2s(stage_smem, reinterpret_cast<const char*>(m.src) + pos, n, bar, policy);
            else bulk_s2g(reinterpret_cast<char*>(m.dst) + pos, stage_smem, n);
        }
        return;
    }
    const uint64_t inner = m.inner;
    const uint64_t row0 = pos / inner;
    const uint64_t col0 = pos - row0 * inner;
    uint64_t len0 = inner - col0;
    if (len0 > n) len0 = n;
    const uint32_t nseg = 1 + (uint32_t)((n - len0 + inner - 1) / inner);
    for (uint32_t k = lane; k < nseg; k += 32) {
        const uint64_t seg_off = k == 0 ? 0 : len0 + (uint64_t)(k - 1) * inner;  // inside the stage
        uint64_t len = k == 0 ? len0 : inner;
        if (seg_off + len > n) len = n - seg_off;
        int64_t so, dofs;
        rows_offsets(m, row0 + k, &so, &dofs);
        const uint64_t col = k == 0 ? col0 : 0;
        if (kLoad) bulk_g2s(stage_smem + (uint32_t)seg_off, reinterpret_cast<const char*>(m.src) + so + col, (uint32_t)len, bar, policy);
        else bulk_s2g(reinterpret_cast<char*>(m.dst) + dofs + col, stage_smem + (uint32_t)seg_off, (uint32_t)len);
    }
}

template <int kStages, int kStageBytes>
__global__ void __launch_bounds__(32) tsnap_rows_copy_kernel(const Member* __restrict__ members,
                                                             const Tile* __restrict__ tiles, uint32_t ntiles) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    // [kStages * kStageBytes data][kStages member records][kStages mbarriers]
    unsigned char* data = smem_raw;
    Member* st_m = reinterpret_cast<Member*>(smem_raw + kStages * kStageBytes);
    uint64_t* bars = reinterpret_cast<uint64_t*>(st_m + kStages);
    const uint32_t lane = threadIdx.x;
    if (lane == 0) {
        for (int s = 0; s < kStages; ++s) mbar_init(smem_u32(&bars[s]), 1);
        fence_mbar_init();
        fence_proxy_async_smem();
    }
    __syncwarp();
    const uint64_t policy = policy_evict_first();

    RowsCursor cur;
    cur.members = members;
    cur.tiles = tiles;
    cur.ntiles = ntiles;
    cur.tile = blockIdx.x;
    cur.stride = gridDim.x;
    cur.open = false;
    cur.pos = cur.end = 0;
    cur.member = 0;

    uint64_t st_pos[kStages];
    uint32_t st_n[kStages];
    uint32_t issued = 0, stored = 0;

    // stage `s` <- piece `p`: the member record travels with the stage (loads of the next member are in flight while
    // the previous member's stage is being stored)
    auto load_piece = [&](int s, const RowsPiece& p) {
        const uint32_t* g = reinterpret_cast<const uint32_t*>(members + p.member);
        uint32_t* d = reinterpret_cast<uint32_t*>(&st_m[s]);
        for (uint32_t i = lane; i < sizeof(Member) / 4; i += 32) d[i] = g[i];
        const uint32_t bar = smem_u32(&bars[s]);
        if (lane == 0) mbar_expect_tx(bar, p.n);
        __syncwarp();
        rows_issue<true>(st_m[s], p.pos, p.n, smem_u32(data + s * kStageBytes), bar, policy, lane);
    };

    RowsPiece p;
#pragma unroll
    for (int s = 0; s < kStages; ++s) {
        if (issued == (uint32_t)s && rows_next(cur, kStageBytes, &p)) {
            load_piece(s, p);
            st_pos[s] = p.pos;
            st_n[s] = p.n;
            ++issued;
        }
    }
    while (stored < issued) {
        const uint32_t s = stored % kStages;
        mbar_wait(smem_u32(&bars[s]), (stored / kStages) & 1);
        fence_proxy_async_smem();
        uint64_t pos = 0;
        uint32_t n = 0;
#pragma unroll
        for (int k = 0; k < kStages; ++k)
            if (k == (int)s) {
                pos = st_pos[k];
                n = st_n[k];
            }
        rows_issue<false>(st_m[s], pos, n, smem_u32(data + s * kStageBytes), 0, policy, lane);
        bulk_commit();
        ++stored;
        if (stored >= 2) {
            bulk_wait_read<1>();  // every lane: all but its newest store group have finished reading shared memory
            __syncwarp();
            if (rows_next(cur, kStageBytes, &p)) {
                const uint32_t fs = (stored - 2) % kStages;
                load_piece((int)fs, p);
#pragma unroll
                for (int k = 0; k < kStages; ++k)
                    if (k == (int)fs) {
                        st_pos[k] = p.pos;
                        st_n[k] = p.n;
                    }
                ++issued;
            }
        }
    }
    bulk_wait_all<0>();
}

// ------------------------------------------------------------------------------------------------
// LSU kernel
// ------------------------------------------------------------------------------------------------
constexpr int kLsuThreads = 256;
constexpr int kLsuUnroll = 4;

// 16 B destination vectors, 16 B aligned source: straight streaming copy
__device__ __forceinline__ void contig_body_aligned(const char* __restrict__ s, char* __restrict__ d, uint64_t nvec) {
    const uint64_t i = threadIdx.x;
    const uint64_t step = (uint64_t)kLsuThreads * kLsuUnroll;
    for (uint64_t base = 0; base < nvec; base += step) {
        uint4 v[kLsuUnroll];
#pragma unroll
        for (int k = 0; k < kLsuUnroll; ++k) {
            const uint64_t j = base + i + (uint64_t)k * kLsuThreads;
            if (j < nvec) v[k] = ld_stream16(s + j * 16);
        }
#pragma unroll
        for (int k = 0; k < kLsuUnroll; ++k) {
            const uint64_t j = base + i + (uint64_t)k * kLsuThreads;
            if (j < nvec) st_stream16(d + j * 16, v[k]);
        }
    }
}

__device__ __forceinline__ uint4 ld_cached16(const void* p) {
    uint4 v;
    asm volatile("ld.global.nc.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p));
    return v;
}

// bytes [sh, sh+16) of the 32-byte concatenation lo:hi  (sh = 4*W + r, r in 0..3)
template <int W>
__device__ __forceinline__ uint4 shift_window(const uint4& lo, const uint4& hi, uint32_t rbits) {
    const uint32_t w[8] = {lo.x, lo.y, lo.z, lo.w, hi.x, hi.y, hi.z, hi.w};
    uint4 o;
    o.x = __funnelshift_r(w[W + 0], w[W + 1], rbits);
    o.y = __funnelshift_r(w[W + 1], w[W + 2], rbits);
    o.z = __funnelshift_r(w[W + 2], w[W + 3], rbits);
    o.w = __funnelshift_r(w[W + 3], w[(W + 4) & 7], rbits);
    return o;
}

// Source and destination disagree on their position inside a 16 B line (slab members are unpadded, so
// one odd-sized tensor shifts everything after it).  All global accesses stay 16 B wide and aligned: each
// output vector is cut out of two neighbouring aligned source vectors with funnel shifts.  The second
// load of every pair is the first load of the next thread, so it is served by L1.  The aligned loads may
// touch up to 15 bytes before/after the run, but never leave the 16 B lines that hold its bytes.
template <int W>
__device__ __forceinline__ void contig_body_shift_w(const char* __restrict__ s, char* __restrict__ d, uint64_t nvec,
                                                    uint32_t sh) {
    const char* a = s - sh;  // 16 B aligned
    const uint32_t rbits = (sh & 3) * 8;
    const uint64_t i = threadIdx.x;
    constexpr int kUnroll = 2;
    const uint64_t step = (uint64_t)kLsuThreads * kUnroll;
    for (uint64_t base = 0; base < nvec; base += step) {
        uint4 lo[kUnroll], hi[kUnroll];
#pragma unroll
        for (int k = 0; k < kUnroll; ++k) {
            const uint64_t j = base + i + (uint64_t)k * kLsuThreads;
            if (j < nvec) {
                lo[k] = ld_cached16(a + j * 16);
                hi[k] = ld_cached16(a + j * 16 + 16);
            }
        }
#pragma unroll
        for (int k = 0; k < kUnroll; ++k) {
            const uint64_t j = base + i + (uint64_t)k * kLsuThreads;
            if (j < nvec) st_stream16(d + j * 16, shift_window<W>(lo[k], hi[k], rbits));
        }
    }
}

__device__ __noinline__ void contig_body_shift(const char* s, char* d, uint64_t nvec) {
    const uint32_t sh = (uint32_t)(reinterpret_cast<uint64_t>(s) & 15);
    switch (sh >> 2) {
        case 0: contig_body_shift_w<0>(s, d, nvec, sh); break;
        case 1: contig_body_shift_w<1>(s, d, nvec, sh); break;
        case 2: contig_body_shift_w<2>(s, d, nvec, sh); break;
        default: contig_body_shift_w<3>(s, d, nvec, sh); break;
    }
}

__device__ __forceinline__ void tile_contig(const Member& m, uint32_t index) {
    const uint64_t a = (uint64_t)index * kTileLsu;
    uint64_t lo = a > m.shift ? a - m.shift : 0;
    uint64_t hi = a + kTileLsu - m.shift;
    if (hi > m.bytes) hi = m.bytes;
    const char* s = reinterpret_cast<const char*>(m.src) + lo;
    char* d = reinterpret_cast<char*>(m.dst) + lo;
    const uint64_t n = hi - lo;
    uint64_t head = (16 - (reinterpret_cast<uint64_t>(d) & 15)) & 15;
    if (head > n) head = n;
    const uint64_t nvec = (n - head) >> 4;
    const uint64_t tail = n - head - (nvec << 4);
    // ragged edges: single bytes, warp 0 the head, warp 1 the tail
    if (threadIdx.x < head) d[threadIdx.x] = s[threadIdx.x];
    if (threadIdx.x >= 32 && threadIdx.x - 32 < tail) {
        const uint64_t o = head + (nvec << 4) + (threadIdx.x - 32);
        d[o] = s[o];
    }
    s += head;
    d += head;
    if ((reinterpret_cast<uint64_t>(s) & 15) == 0) contig_body_aligned(s, d, nvec);
    else contig_body_shift(s, d, nvec);
}

__device__ __forceinline__ void outer_offsets(const Member& m, uint64_t row, int64_t* so, int64_t* dofs) {
    int64_t s = 0, d = 0;
    if ((row >> 32) == 0) {
        uint32_t r = (uint32_t)row;
        for (int i = (int)m.nouter - 1; i >= 0; --i) {
            const uint64_t sz64 = (uint64_t)m.osize[i];
            uint32_t idx;
            if (sz64 >> 32) {
                idx = r;
                r = 0;
            } else {
                const uint32_t sz = (uint32_t)sz64;
                idx = r % sz;
                r = r / sz;
            }
            s += (int64_t)idx * m.sstride[i];
            d += (int64_t)idx * m.dstride[i];
        }
    } else {
        for (int i = (int)m.nouter - 1; i >= 0; --i) {
            const uint64_t sz = (uint64_t)m.osize[i];
            const uint64_t idx = row % sz;
            row /= sz;
            s += (int64_t)idx * m.sstride[i];
            d += (int64_t)idx * m.dstride[i];
        }
    }
    *so = s;
    *dofs = d;
}

// row index -> byte offsets on both sides; the single-outer-dim case (2-D narrow / column shard) needs no division
__device__ __forceinline__ void row_offsets(const Member& m, uint64_t row, int64_t* so, int64_t* dofs) {
    if (m.nouter == 1) {
        *so = (int64_t)row * m.sstride[0];
        *dofs = (int64_t)row * m.dstride[0];
    } else {
        outer_offsets(m, row, so, dofs);
    }
}

// One granule (sizeof(T) bytes) per thread and step; kU independent loads are issued before the stores so that
// several requests per thread are in flight.  (row, col) of a thread's granule is divided out once per tile and
// then advanced incrementally: consecutive granules of a thread are a constant number of bytes apart.
template <typename T>
__device__ __forceinline__ void tile_strided_t(const Member& m, uint64_t lo, uint64_t hi) {
    constexpr int kU = sizeof(T) >= 8 ? 4 : 8;  // bytes in flight per SM = 3 CTAs x 256 thr x kU x sizeof(T)
    const char* sb = reinterpret_cast<const char*>(m.src);
    char* db = reinterpret_cast<char*>(m.dst);
    const uint64_t inner = m.inner;
    const uint64_t stride = (uint64_t)kLsuThreads * sizeof(T);
    uint64_t pos = lo + (uint64_t)threadIdx.x * sizeof(T);
    if (pos >= hi) return;
    uint64_t row, col, drow, dcol;
    if ((m.bytes >> 32) == 0) {
        const uint32_t in = (uint32_t)inner;
        row = (uint32_t)pos / in;
        col = (uint32_t)pos - (uint32_t)row * in;
        drow = (uint32_t)stride / in;
        dcol = (uint32_t)stride - (uint32_t)drow * in;
    } else {
        row = pos / inner;
        col = pos - row * inner;
        drow = stride / inner;
        dcol = stride - drow * inner;
    }
    while (pos < hi) {
        T v[kU];
        int64_t dst_off[kU];
#pragma unroll
        for (int k = 0; k < kU; ++k) {
            dst_off[k] = -1;
            if (pos < hi) {
                int64_t so, dofs;
                row_offsets(m, row, &so, &dofs);
                v[k] = __ldg(reinterpret_cast<const T*>(sb + so + (int64_t)col));
                dst_off[k] = dofs + (int64_t)col;
            }
            pos += stride;
            row += drow;
            col += dcol;
            if (col >= inner) {
                col -= inner;
                ++row;
            }
        }
#pragma unroll
        for (int k = 0; k < kU; ++k)
            if (dst_off[k] >= 0) *reinterpret_cast<T*>(db + dst_off[k]) = v[k];
    }
}

__device__ __noinline__ void tile_strided(const Member& m, uint32_t index) {
    const uint64_t lo = (uint64_t)index * kTileLsu;
    uint64_t hi = lo + kTileLsu;
    if (hi > m.bytes) hi = m.bytes;
    switch (m.unit) {
        case 16: tile_strided_t<uint4>(m, lo, hi); break;
        case 8: tile_strided_t<uint2>(m, lo, hi); break;
        case 4: tile_strided_t<uint32_t>(m, lo, hi); break;
        case 2: tile_strided_t<uint16_t>(m, lo, hi); break;
        default: tile_strided_t<uint8_t>(m, lo, hi); break;
    }
}

// element i (compile-time constant after unrolling) of a 16 B vector, without taking the vector's address
template <typename T>
__device__ __forceinline__ T vec_get(const uint4& v, int i) {
    const uint32_t w[4] = {v.x, v.y, v.z, v.w};
    if (sizeof(T) == 8) return (T)(((uint64_t)w[2 * i + 1] << 32) | w[2 * i]);
    if (sizeof(T) == 4) return (T)w[i];
    if (sizeof(T) == 2) return (T)((w[i >> 1] >> (16 * (i & 1))) & 0xffffu);
    return (T)((w[i >> 2] >> (8 * (i & 3))) & 0xffu);
}
template <typename T>
__device__ __forceinline__ void vec_put(uint32_t (&w)[4], int i, T x) {
    if (sizeof(T) == 8) {
        w[2 * i] = (uint32_t)((uint64_t)x);
        w[2 * i + 1] = (uint32_t)((uint64_t)x >> 32);
    } else if (sizeof(T) == 4) {
        w[i] = (uint32_t)x;
    } else if (sizeof(T) == 2) {
        w[i >> 1] |= (uint32_t)x << (16 * (i & 1));
    } else {
        w[i >> 2] |= (uint32_t)x << (8 * (i & 3));
    }
}

// ---- tiled transpose ---------------------------------------------------------------------------
// kModeTranspose: dim A is unit-stride on the source, dim B on the destination.  One tile = side x side elements of
// (A, B) for one index of the remaining dims: read with consecutive threads along A, write with consecutive threads
// along B, through a padded shared-memory tile — both sides see full-line accesses instead of an element gather.
template <typename T, int kA, int kB>
__device__ __forceinline__ void tile_transpose_t(const Member& m, uint32_t index, unsigned char* tbuf) {
    const uint32_t A = m.shift & 255, B = (m.shift >> 8) & 255;
    const uint64_t sA = (uint64_t)m.osize[A], sB = (uint64_t)m.osize[B];
    const uint32_t tilesA = (uint32_t)((sA + kA - 1) / kA), tilesB = (uint32_t)((sB + kB - 1) / kB);
    const uint32_t ib = index % tilesB;
    uint32_t rest = index / tilesB;
    const uint32_t ia = rest % tilesA;
    rest /= tilesA;
    int64_t so = 0, dofs = 0;
    for (int i = (int)m.nouter - 1; i >= 0; --i) {
        if ((uint32_t)i == A || (uint32_t)i == B) continue;
        const uint32_t sz = (uint32_t)m.osize[i];
        const uint32_t idx = rest % sz;
        rest /= sz;
        so += (int64_t)idx * m.sstride[i];
        dofs += (int64_t)idx * m.dstride[i];
    }
    const uint64_t a0 = (uint64_t)ia * kA, b0 = (uint64_t)ib * kB;
    const uint32_t na = (uint32_t)(sA - a0 < (uint64_t)kA ? sA - a0 : kA);
    const uint32_t nb = (uint32_t)(sB - b0 < (uint64_t)kB ? sB - b0 : kB);
    const int64_t ssB = m.sstride[B], dsA = m.dstride[A];
    const char* sp = reinterpret_cast<const char*>(m.src) + so + (int64_t)a0 * m.sstride[A] + (int64_t)b0 * ssB;
    char* dp = reinterpret_cast<char*>(m.dst) + dofs + (int64_t)a0 * dsA + (int64_t)b0 * m.dstride[B];
    T(*tile)[kA + 1] = reinterpret_cast<T(*)[kA + 1]>(tbuf);  // tile[b][a], one element of padding per row
    constexpr int V = 16 / (int)sizeof(T);  // elements per 16 B vector
    constexpr int kVecIn = kA / V;          // vectors per source row (along A)
    constexpr int kVecOut = kB / V;         // vectors per destination row (along B)
    constexpr int kIter = kB * kVecIn / kLsuThreads;
    static_assert(kB * kVecIn == kA * kVecOut && kIter * kLsuThreads == kB * kVecIn, "tile geometry");
    const bool full = na == (uint32_t)kA && nb == (uint32_t)kB && ((reinterpret_cast<uint64_t>(sp) | (uint64_t)ssB) & 15) == 0 &&
                      ((reinterpret_cast<uint64_t>(dp) | (uint64_t)dsA) & 15) == 0;
    if (full) {
        // interior tile: 16 B vectors on both global sides, all loads in flight before the first shared-memory store
        uint4 r[kIter];
#pragma unroll
        for (int k = 0; k < kIter; ++k) {
            const uint32_t idx = threadIdx.x + (uint32_t)k * kLsuThreads;
            r[k] = ld_stream16(sp + (int64_t)(idx / kVecIn) * ssB + (idx % kVecIn) * 16);
        }
#pragma unroll
        for (int k = 0; k < kIter; ++k) {
            const uint32_t idx = threadIdx.x + (uint32_t)k * kLsuThreads;
            const uint32_t b = idx / kVecIn, v = idx % kVecIn;
#pragma unroll
            for (int i = 0; i < V; ++i) tile[b][v * V + i] = vec_get<T>(r[k], i);
        }
        __syncthreads();
#pragma unroll
        for (int k = 0; k < kIter; ++k) {
            const uint32_t idx = threadIdx.x + (uint32_t)k * kLsuThreads;
            const uint32_t a = idx / kVecOut, v = idx % kVecOut;
            uint32_t w[4] = {0, 0, 0, 0};
#pragma unroll
            for (int i = 0; i < V; ++i) vec_put<T>(w, i, tile[v * V + i][a]);
            st_stream16(dp + (int64_t)a * dsA + v * 16, make_uint4(w[0], w[1], w[2], w[3]));
        }
        return;  // the caller's loop synchronises before the tile buffer is reused
    }
    // edge tiles / unaligned bases: element accesses, still coalesced on both sides
    for (uint32_t e = threadIdx.x; e < nb * (uint32_t)kA; e += kLsuThreads) {
        const uint32_t b = e / kA, a = e % kA;
        if (a < na) tile[b][a] = __ldg(reinterpret_cast<const T*>(sp + (int64_t)b * ssB) + a);
    }
    __syncthreads();
    for (uint32_t e = threadIdx.x; e < na * (uint32_t)kB; e += kLsuThreads) {
        const uint32_t a = e / kB, b = e % kB;
        if (b < nb) reinterpret_cast<T*>(dp + (int64_t)a * dsA)[b] = tile[b][a];
    }
}

__device__ __noinline__ void tile_transpose(const Member& m, uint32_t index, unsigned char* tbuf) {
    switch (m.unit) {  // geometry = plan.h transpose_side_a / transpose_side_b
        case 8: tile_transpose_t<uint64_t, 64, 32>(m, index, tbuf); break;
        case 4: tile_transpose_t<uint32_t, 64, 64>(m, index, tbuf); break;
        case 2: tile_transpose_t<uint16_t, 128, 64>(m, index, tbuf); break;
        default: tile_transpose_t<uint8_t, 128, 128>(m, index, tbuf); break;
    }
}

// ---- fused cast -------------------------------------------------------------------------------
// raw element bits; a source that is not element aligned (a wire piece packed behind an odd-sized slab member) is
// assembled byte by byte, little-endian: the mirror of store_bytes
template <typename U>
__device__ __forceinline__ U load_bits(const char* p, bool aligned) {
    if (aligned) return *reinterpret_cast<const U*>(p);
    U v = 0;
    for (int i = 0; i < (int)sizeof(U); ++i) v |= (U)((U)(unsigned char)p[i] << (8 * i));
    return v;
}
__device__ __forceinline__ double load_elem(const char* p, uint32_t dt, bool aligned) {
    switch (dt) {
        case TSNAP_F16: return (double)__half2float(__ushort_as_half(load_bits<unsigned short>(p, aligned)));
        case TSNAP_BF16: return (double)__bfloat162float(__ushort_as_bfloat16(load_bits<unsigned short>(p, aligned)));
        case TSNAP_F32: return (double)__uint_as_float(load_bits<unsigned int>(p, aligned));
        default: return __longlong_as_double((long long)load_bits<unsigned long long>(p, aligned));
    }
}
__device__ __forceinline__ void store_bytes(char* p, const void* v, int n, bool aligned) {
    const char* c = reinterpret_cast<const char*>(v);
    if (aligned) {
        if (n == 2) *reinterpret_cast<uint16_t*>(p) = *reinterpret_cast<const uint16_t*>(c);
        else if (n == 4) *reinterpret_cast<uint32_t*>(p) = *reinterpret_cast<const uint32_t*>(c);
        else *reinterpret_cast<uint64_t*>(p) = *reinterpret_cast<const uint64_t*>(c);
    } else {
        for (int i = 0; i < n; ++i) p[i] = c[i];
    }
}
// affine quantisation as torch's CUDA quantize_per_tensor does it: nearbyint(x / scale) + zero_point in double
// precision, clamped to the integer range (ATen/native/quantized/cuda/AffineQuantizer.cu)
__device__ __forceinline__ uint8_t quantize_elem(float x, double scale, int64_t zp, bool is_signed) {
    long long q = (long long)(nearbyint((double)x / scale) + (double)zp);
    const long long lo = is_signed ? -128 : 0, hi = is_signed ? 127 : 255;
    q = q < lo ? lo : (q > hi ? hi : q);
    return (uint8_t)(int8_t)q;
}

__device__ __forceinline__ void convert_store(char* p, uint32_t ddt, const char* sp, uint32_t sdt, bool aligned, bool src_aligned) {
    // <=32-bit float sources convert through fp32 (exact widening).  fp64 sources narrow to fp32 directly and to
    // fp16 / bf16 through fp32 (two roundings): torch's copy kernel has no direct double -> half conversion either.
    if (sdt == TSNAP_F64) {
        const double x = __longlong_as_double((long long)load_bits<unsigned long long>(sp, src_aligned));
        if (ddt == TSNAP_F32) { const float f = (float)x; store_bytes(p, &f, 4, aligned); }
        else if (ddt == TSNAP_F16) { const __half h = __float2half_rn((float)x); store_bytes(p, &h, 2, aligned); }
        else if (ddt == TSNAP_BF16) { const __nv_bfloat16 b = __float2bfloat16_rn((float)x); store_bytes(p, &b, 2, aligned); }
        else store_bytes(p, &x, 8, aligned);
        return;
    }
    const float f = (float)load_elem(sp, sdt, src_aligned);
    if (ddt == TSNAP_F32) store_bytes(p, &f, 4, aligned);
    else if (ddt == TSNAP_F16) { const __half h = __float2half_rn(f); store_bytes(p, &h, 2, aligned); }
    else if (ddt == TSNAP_BF16) { const __nv_bfloat16 b = __float2bfloat16_rn(f); store_bytes(p, &b, 2, aligned); }
    else { const double x = (double)f; store_bytes(p, &x, 8, aligned); }
}

// dense, 16 B aligned, 2-byte <-> 4-byte float conversions: 8 elements per thread, 16 B accesses
template <bool kNarrow, bool kBf16>
__device__ __forceinline__ void cast_dense_vec(const char* __restrict__ s, char* __restrict__ d, uint64_t nelem) {
    const uint64_t ngroups = nelem >> 3;
    for (uint64_t g = threadIdx.x; g < ngroups; g += kLsuThreads) {
        if (kNarrow) {  // fp32 -> bf16 / fp16
            const uint4 a = ld_stream16(s + g * 32);
            const uint4 b = ld_stream16(s + g * 32 + 16);
            const float f[8] = {__uint_as_float(a.x), __uint_as_float(a.y), __uint_as_float(a.z), __uint_as_float(a.w),
                                __uint_as_float(b.x), __uint_as_float(b.y), __uint_as_float(b.z), __uint_as_float(b.w)};
            uint32_t o[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                if (kBf16) {
                    const __nv_bfloat162 p = __floats2bfloat162_rn(f[2 * i], f[2 * i + 1]);
                    o[i] = *reinterpret_cast<const uint32_t*>(&p);
                } else {
                    const __half2 p = __floats2half2_rn(f[2 * i], f[2 * i + 1]);
                    o[i] = *reinterpret_cast<const uint32_t*>(&p);
                }
            }
            st_stream16(d + g * 16, make_uint4(o[0], o[1], o[2], o[3]));
        } else {  // bf16 / fp16 -> fp32
            const uint4 a = ld_stream16(s + g * 16);
            const uint32_t w[4] = {a.x, a.y, a.z, a.w};
            float f[8];
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                if (kBf16) {
                    const float2 p = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&w[i]));
                    f[2 * i] = p.x;
                    f[2 * i + 1] = p.y;
                } else {
                    const float2 p = __half22float2(*reinterpret_cast<const __half2*>(&w[i]));
                    f[2 * i] = p.x;
                    f[2 * i + 1] = p.y;
                }
            }
            st_stream16(d + g * 32, make_uint4(__float_as_uint(f[0]), __float_as_uint(f[1]), __float_as_uint(f[2]), __float_as_uint(f[3])));
            st_stream16(d + g * 32 + 16, make_uint4(__float_as_uint(f[4]), __float_as_uint(f[5]), __float_as_uint(f[6]), __float_as_uint(f[7])));
        }
    }
}

__device__ __noinline__ void tile_cast(const Member& m, uint32_t index) {
    const uint64_t lo = (uint64_t)index * kTileLsu;
    uint64_t hi = lo + kTileLsu;
    if (hi > m.bytes) hi = m.bytes;
    uint64_t e0 = lo / m.dst_esz;
    const uint64_t e1 = hi / m.dst_esz;
    const char* sb = reinterpret_cast<const char*>(m.src);
    char* db = reinterpret_cast<char*>(m.dst);
    // fast path: one dense run on both sides, 16 B aligned, fp32 <-> {bf16, fp16}
    if (m.nouter == 0 && ((m.src | m.dst) & 15) == 0) {
        const bool narrow = m.src_dtype == TSNAP_F32 && (m.dst_dtype == TSNAP_BF16 || m.dst_dtype == TSNAP_F16);
        const bool widen = m.dst_dtype == TSNAP_F32 && (m.src_dtype == TSNAP_BF16 || m.src_dtype == TSNAP_F16);
        if (narrow || widen) {
            const uint64_t n = e1 - e0;
            const char* s = sb + e0 * m.src_esz;
            char* d = db + e0 * m.dst_esz;
            if (narrow) {
                if (m.dst_dtype == TSNAP_BF16) cast_dense_vec<true, true>(s, d, n);
                else cast_dense_vec<true, false>(s, d, n);
            } else {
                if (m.src_dtype == TSNAP_BF16) cast_dense_vec<false, true>(s, d, n);
                else cast_dense_vec<false, false>(s, d, n);
            }
            e0 += n & ~uint64_t(7);  // the ragged tail (< 8 elements) goes through the scalar loop below
        }
    }
    // the wire side of a load may sit at any byte offset (slab members are packed without padding)
    bool src_aligned = (m.src % m.src_esz) == 0;
    for (uint32_t i = 0; i < m.nouter; ++i) src_aligned = src_aligned && ((uint64_t)m.sstride[i] % m.src_esz) == 0;
    if (m.dst_dtype == TSNAP_QINT8 || m.dst_dtype == TSNAP_QUINT8) {
        // quantise-on-save: 1-byte destination elements, consecutive threads write consecutive bytes
        const bool is_signed = m.dst_dtype == TSNAP_QINT8;
        for (uint64_t e = e0 + threadIdx.x; e < e1; e += kLsuThreads) {
            const uint64_t row = e / m.inner, col = e - row * m.inner;
            int64_t so, dofs;
            outer_offsets(m, row, &so, &dofs);
            const float x = (float)load_elem(sb + so + col * m.src_esz, m.src_dtype, src_aligned);
            reinterpret_cast<uint8_t*>(db + dofs)[col] = quantize_elem(x, m.q_scale, m.q_zero_point, is_signed);
        }
        if ((m.shift & 1) && hi == m.bytes && threadIdx.x < 16) {
            // the per-tensor trailer of T:serialization.py:278-310, byte by byte (the payload length is arbitrary)
            const unsigned char* t = threadIdx.x < 8 ? reinterpret_cast<const unsigned char*>(&m.q_scale) : reinterpret_cast<const unsigned char*>(&m.q_zero_point);
            db[m.bytes + threadIdx.x] = (char)t[threadIdx.x & 7];
        }
        return;
    }
    bool aligned = (m.dst % m.dst_esz) == 0;
    for (uint32_t i = 0; i < m.nouter; ++i) aligned = aligned && ((uint64_t)m.dstride[i] % m.dst_esz) == 0;
    for (uint64_t e = e0 + threadIdx.x; e < e1; e += kLsuThreads) {
        const uint64_t row = e / m.inner, col = e - row * m.inner;
        int64_t so, dofs;
        outer_offsets(m, row, &so, &dofs);
        convert_store(db + dofs + col * m.dst_esz, m.dst_dtype, sb + so + col * m.src_esz, m.src_dtype, aligned, src_aligned);
    }
}

// kMinBlocks = CTAs per SM the register allocation is bounded for: 3 caps it at 80 registers (the strided path then
// spills), 2 at 128, 6 at 40.  Three builds: strided tiles run on <2>, transpose tiles on <6> (a latency-bound
// load -> shared -> store cycle: more resident CTAs in different phases keep the memory system busy), every other mode
// on <3> (kernels.h, A/B in profiles/r02_kernel_cases.md).
template <int kMinBlocks>
__global__ void __launch_bounds__(kLsuThreads, kMinBlocks) tsnap_lsu_copy_kernel(const Member* __restrict__ members,
                                                                            const Tile* __restrict__ tiles, uint32_t ntiles) {
    __shared__ Member sm;
    __shared__ __align__(16) unsigned char tbuf[64 * 65 * 4 + 64];  // transpose tile: 64 x 65 x 4 B >= 64 x 129 x 2 B, 32 x 65 x 8 B, 128 x 129 B
    uint32_t loaded = 0xffffffffu;
    Tile next = blockIdx.x < ntiles ? tiles[blockIdx.x] : Tile{0, 0};
    for (uint32_t t = blockIdx.x; t < ntiles; t += gridDim.x) {
        const Tile tl = next;
        if (t + gridDim.x < ntiles) next = tiles[t + gridDim.x];  // the descriptor of the next tile is in flight behind this tile's work
        // stage the member record in shared memory: every thread needs all of it (consecutive tiles of a CTA mostly
        // belong to the same member: reload only on change)
        __syncthreads();  // also fences the previous tile's use of sm / tbuf
        if (tl.member != loaded) {
            const uint32_t* g = reinterpret_cast<const uint32_t*>(members + tl.member);
            uint32_t* s = reinterpret_cast<uint32_t*>(&sm);
            for (uint32_t i = threadIdx.x; i < sizeof(Member) / 4; i += kLsuThreads) s[i] = g[i];
            loaded = tl.member;
            __syncthreads();
        }
        switch (sm.mode) {
            case kModeContig: tile_contig(sm, tl.index); break;
            case kModeStrided: tile_strided(sm, tl.index); break;
            case kModeCast: tile_cast(sm, tl.index); break;
            case kModeTranspose: tile_transpose(sm, tl.index, tbuf); break;
            default: {
                // a bulk-mode member routed here (never emitted by the planner when bulk is disabled,
                // kept for robustness): dense and 16B aligned on both sides
                const uint64_t a = (uint64_t)tl.index * kTileLsu;
                uint64_t hi = a + kTileLsu;
                if (hi > sm.bytes) hi = sm.bytes;
                contig_body_aligned(reinterpret_cast<const char*>(sm.src) + a, reinterpret_cast<char*>(sm.dst) + a,
                                    (hi - a) >> 4);
            }
        }
    }
}

// ------------------------------------------------------------------------------------------------
// launchers
// ------------------------------------------------------------------------------------------------
// Ring geometry of the copy-engine kernels, picked by a 10-point sweep on B200 (profiles/r01_ncu_summary.md): two
// 48 KiB stages per one-warp CTA, two CTAs per SM (0.98 of the measured copy peak).  TSNAP_B200_BULK_CFG=0 selects the
// first version's geometry (3 x 16 KiB, 4 CTAs per SM; 0.95) for A/B runs.
struct BulkCfg {
    int stages, stage_bytes, ctas_per_sm;
};
static const BulkCfg kBulkCfgs[] = {
    {3, 16384, 4},  // 0: fallback
    {2, 49152, 2},  // 1: default
};
static int bulk_cfg_index() {
    static const int idx = [] {
        const char* e = getenv("TSNAP_B200_BULK_CFG");
        return e && atoi(e) == 0 ? 0 : 1;
    }();
    return idx;
}

template <int S, int B>
static cudaError_t bulk_attr() {
    cudaError_t e = cudaFuncSetAttribute(tsnap_bulk_copy_kernel<S, B>, cudaFuncAttributeMaxDynamicSharedMemorySize, S * B + S * 8);
    if (e == cudaSuccess)
        e = cudaFuncSetAttribute(tsnap_rows_copy_kernel<S, B>, cudaFuncAttributeMaxDynamicSharedMemorySize, S * B + S * (int)sizeof(Member) + S * 8);
    return e;
}
template <int S, int B>
static void bulk_launch(const Member* m, const Tile* t, uint32_t n, uint32_t grid, cudaStream_t st) {
    tsnap_bulk_copy_kernel<S, B><<<grid, 32, S * B + S * 8, st>>>(m, t, n);
}
template <int S, int B>
static void rows_launch(const Member* m, const Tile* t, uint32_t n, uint32_t grid, cudaStream_t st) {
    tsnap_rows_copy_kernel<S, B><<<grid, 32, S * B + S * (int)sizeof(Member) + S * 8, st>>>(m, t, n);
}

// resident CTAs per SM of the two builds of the LSU kernel, from the occupancy calculator: each persistent grid is
// exactly one wave
static int g_lsu_ctas_per_sm[3] = {3, 2, 6};

cudaError_t init_kernels() {
    cudaError_t e = bulk_attr<3, 16384>();
    if (e == cudaSuccess) e = bulk_attr<2, 49152>();
    if (e == cudaSuccess) {
        int n = 0;
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, tsnap_lsu_copy_kernel<3>, kLsuThreads, 0) == cudaSuccess && n > 0) g_lsu_ctas_per_sm[0] = n;
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, tsnap_lsu_copy_kernel<2>, kLsuThreads, 0) == cudaSuccess && n > 0) g_lsu_ctas_per_sm[1] = n;
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, tsnap_lsu_copy_kernel<6>, kLsuThreads, 0) == cudaSuccess && n > 0) g_lsu_ctas_per_sm[2] = n;
    }
    return e;
}

cudaError_t launch_bulk(const Member* d_members, const Tile* d_tiles, uint32_t ntiles, int sm_count,
                        cudaStream_t stream) {
    if (ntiles == 0) return cudaSuccess;
    const int ci = bulk_cfg_index();
    uint32_t grid = (uint32_t)sm_count * kBulkCfgs[ci].ctas_per_sm;
    if (grid > ntiles) grid = ntiles;
    if (ci == 0) bulk_launch<3, 16384>(d_members, d_tiles, ntiles, grid, stream);
    else bulk_launch<2, 49152>(d_members, d_tiles, ntiles, grid, stream);
    return cudaGetLastError();
}

cudaError_t launch_rows(const Member* d_members, const Tile* d_tiles, uint32_t ntiles, int sm_count,
                        cudaStream_t stream) {
    if (ntiles == 0) return cudaSuccess;
    const int ci = bulk_cfg_index();
    uint32_t grid = (uint32_t)sm_count * kBulkCfgs[ci].ctas_per_sm;
    if (grid > ntiles) grid = ntiles;
    if (ci == 0) rows_launch<3, 16384>(d_members, d_tiles, ntiles, grid, stream);
    else rows_launch<2, 49152>(d_members, d_tiles, ntiles, grid, stream);
    return cudaGetLastError();
}

cudaError_t launch_lsu(const Member* d_members, const Tile* d_tiles, uint32_t ntiles, int sm_count,
                       cudaStream_t stream, int variant) {
    if (ntiles == 0) return cudaSuccess;
    uint32_t grid = (uint32_t)sm_count * (uint32_t)g_lsu_ctas_per_sm[variant];
    if (grid > ntiles) grid = ntiles;
    if (variant == kLsuStrided) tsnap_lsu_copy_kernel<2><<<grid, kLsuThreads, 0, stream>>>(d_members, d_tiles, ntiles);
    else if (variant == kLsuTranspose) tsnap_lsu_copy_kernel<6><<<grid, kLsuThreads, 0, stream>>>(d_members, d_tiles, ntiles);
    else tsnap_lsu_copy_kernel<3><<<grid, kLsuThreads, 0, stream>>>(d_members, d_tiles, ntiles);
    return cudaGetLastError();
}

}  // namespace tsnap
