// cov_radix.cuh — stable LSD radix sort of (uint32 key, int32 value) pairs and an exclusive prefix sum, written for this
// library (no CUB).  Used by the Morton ordering of a cloud (cov_spatial_sort) and by the voxel-grid filter.
//
// One pass sorts by 8 key bits with three launches:
//   upsweep    G blocks, block b counts the digits of its contiguous range of 4096-key tiles      4 B/key read
//   scan       one warp per digit turns the digit-major count matrix [256][G] into exclusive offsets (the digits' totals
//              come from the upsweep's atomics, so no warp waits for another)                        ~0.5 MB
//   downsweep  the same G blocks walk their ranges tile by tile: a warp ranks 32 consecutive keys at a time (eight
//              ballots, one per digit bit, give every lane the mask of the lanes with its digit — MATCH.ANY does the same
//              in one instruction but at a fraction of the rate; the group's first lane advances the warp's digit counter, a
//              lane's rank is that counter plus the number of group lanes below it), the warps' counters are scanned per digit,
//              the tile is reordered by digit in shared memory and written out in runs, so equal digits keep their input
//              order (tile, warp, round, lane = ascending index): the sort is STABLE.                 8 B read + 8 B written/key
// The passes ping-pong between two buffers; with an even number of passes the result is back in the first one.
// 2^31 > n: positions are 32-bit.  G = 3 blocks per SM (all resident, equal ranges) keeps the count matrix small enough for
// a single-block scan.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "cov_common.cuh"  // TMA bulk copies and their mbarriers

namespace covradix {

constexpr int kThreads = 256;
constexpr int kWarps = kThreads / 32;
constexpr int kIpt = 16;                       // keys per thread per tile
constexpr int kTile = kThreads * kIpt;         // 4096
constexpr int kBins = 256;
constexpr int kMaxGrid = 1024;                 // blocks; the scan kernel handles any G <= this
constexpr unsigned kFullMask = 0xffffffffu;

struct Plan {
    int grid;                 // G
    int64_t tiles_per_block;  // block b owns tiles [b * tpb, min((b + 1) * tpb, tiles))
    int64_t tiles;
};

inline Plan make_plan(int64_t n, int sm_count) {
    Plan p;
    p.tiles = (n + kTile - 1) / kTile;
    int64_t g = (int64_t)sm_count * 3;   // what is resident at once (80 registers, 42 KB of shared memory per block)
    if (g > kMaxGrid) g = kMaxGrid;
    if (g > p.tiles) g = p.tiles;
    if (g < 1) g = 1;
    p.tiles_per_block = (p.tiles + g - 1) / g;
    p.grid = (int)((p.tiles + p.tiles_per_block - 1) / p.tiles_per_block);
    if (p.grid < 1) p.grid = 1;
    return p;
}

// bytes of the count matrix (what the sort needs besides the two pairs of buffers)
inline size_t temp_bytes() { return ((size_t)kBins * kMaxGrid + 4 * kBins) * sizeof(unsigned); }

__global__ void __launch_bounds__(kThreads) upsweep_kernel(const unsigned* __restrict__ keys, int64_t n, int shift, unsigned dmask,
                                                           int64_t tiles_per_block, unsigned* __restrict__ counts,
                                                           unsigned* __restrict__ totals) {
    __shared__ unsigned whist[kWarps][kBins];
    const int t = threadIdx.x, warp = t >> 5;
#pragma unroll
    for (int w = 0; w < kWarps; ++w) whist[w][t] = 0u;
    __syncthreads();
    const int64_t begin = (int64_t)blockIdx.x * tiles_per_block * kTile;   // a multiple of 4096 keys: 16-byte aligned
    int64_t end = begin + tiles_per_block * kTile;
    if (end > n) end = n;
    unsigned* wh = whist[warp];
    // four 16-byte loads in flight per thread (the range is streamed once; a single 4-byte load per thread would leave
    // the memory system idle), then the 16 shared-memory atomics
    const int64_t end4 = begin + ((end - begin) & ~(int64_t)(4 * 4 * kThreads - 1));
    for (int64_t i = begin + (int64_t)t * 4; i < end4; i += 4 * 4 * kThreads) {
        uint4 v[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) v[u] = __ldg(reinterpret_cast<const uint4*>(keys + i + (int64_t)u * 4 * kThreads));
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            atomicAdd(&wh[(v[u].x >> shift) & dmask], 1u);
            atomicAdd(&wh[(v[u].y >> shift) & dmask], 1u);
            atomicAdd(&wh[(v[u].z >> shift) & dmask], 1u);
            atomicAdd(&wh[(v[u].w >> shift) & dmask], 1u);
        }
    }
    for (int64_t i = end4 + t; i < end; i += kThreads) atomicAdd(&wh[(__ldg(keys + i) >> shift) & dmask], 1u);
    __syncthreads();
    unsigned c = 0;
#pragma unroll
    for (int w = 0; w < kWarps; ++w) c += whist[w][t];
    counts[(size_t)t * gridDim.x + blockIdx.x] = c;   // digit-major: row t = digit t over the blocks
    if (c) atomicAdd(totals + t, c);                  // zero before the launch
}

// counts[d][b] -> number of keys that precede block b's first key of digit d in the sorted order: all keys of smaller
// digits (from `totals`) plus digit d's keys of earlier blocks.  One warp per digit, 8 blocks of 32 warps.
__global__ void __launch_bounds__(1024) scan_rows_kernel(unsigned* __restrict__ counts, const unsigned* __restrict__ totals, int G) {
    const int lane = threadIdx.x & 31;
    const int d = blockIdx.x * 32 + (threadIdx.x >> 5);
    unsigned base = 0u;
    for (int k = lane; k < d; k += 32) base += totals[k];
    base = __reduce_add_sync(kFullMask, base);
    unsigned* row = counts + (size_t)d * G;
    for (int c0 = 0; c0 < G; c0 += 32) {
        const int i = c0 + lane;
        const unsigned x = i < G ? row[i] : 0u;
        unsigned inc = x;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned u = __shfl_up_sync(kFullMask, inc, o);
            if (lane >= o) inc += u;
        }
        if (i < G) row[i] = base + inc - x;
        base += __shfl_sync(kFullMask, inc, 31);
    }
}

// exclusive prefix sum of m values (m <= 256 * kMaxGrid) by one block of 1024 threads: coalesced chunks of 4096 values
// (four consecutive ones per thread) with a running carry
__global__ void __launch_bounds__(1024) scan_small_kernel(unsigned* __restrict__ v, int m) {
    __shared__ unsigned wsum[32];
    const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
    unsigned carry = 0u;
    for (int c0 = 0; c0 < m; c0 += 4096) {
        const int i0 = c0 + t * 4;
        unsigned x[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) x[k] = (i0 + k < m) ? v[i0 + k] : 0u;
        const unsigned s = x[0] + x[1] + x[2] + x[3];
        unsigned inc = s;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned u = __shfl_up_sync(kFullMask, inc, o);
            if (lane >= o) inc += u;
        }
        if (lane == 31) wsum[warp] = inc;
        __syncthreads();
        unsigned wbase = 0u, total = 0u;
#pragma unroll
        for (int w = 0; w < 32; ++w) {
            const unsigned y = wsum[w];
            wbase += (w < warp) ? y : 0u;
            total += y;
        }
        unsigned run = carry + wbase + inc - s;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            if (i0 + k < m) v[i0 + k] = run;
            run += x[k];
        }
        carry += total;
        __syncthreads();   // wsum is rewritten by the next chunk
    }
}

// dynamic shared memory of the downsweep kernel: [stage keys][stage vals][tile keys][tile vals][warp counters][base][doff]
constexpr size_t kDownSmemBytes = 4 * (size_t)kTile * 4 + ((size_t)kWarps * kBins + 2 * kBins) * 4;

// The NEXT tile's keys and values arrive by TMA while the current tile is ranked and written (ncu on the first version,
// which loaded them with plain loads at the point of use: 13 of 25 stall cycles per issue were the wait for those
// loads).  Two single-buffered 16 KB stages, each refilled as soon as the block has consumed it: the keys right after
// they were read into registers, the values right after the reorder.  A ragged last tile is loaded by hand.
__global__ void __launch_bounds__(kThreads, 3) downsweep_kernel(const unsigned* __restrict__ keys_in, const int32_t* __restrict__ vals_in,
                                                             unsigned* __restrict__ keys_out, int32_t* __restrict__ vals_out, int64_t n,
                                                             int shift, unsigned dmask, int64_t tiles_per_block, int64_t tiles,
                                                             const unsigned* __restrict__ offsets) {
    extern __shared__ __align__(128) unsigned char rs_smem[];
    unsigned* st_keys = reinterpret_cast<unsigned*>(rs_smem);
    int32_t* st_vals = reinterpret_cast<int32_t*>(st_keys + kTile);
    unsigned* s_keys = reinterpret_cast<unsigned*>(st_vals + kTile);
    int32_t* s_vals = reinterpret_cast<int32_t*>(s_keys + kTile);
    unsigned (*s_whist)[kBins] = reinterpret_cast<unsigned (*)[kBins]>(s_vals + kTile);   // per warp: digit counts of the tile, then exclusive offsets over warps
    unsigned* s_base = &s_whist[kWarps][0];       // where the block's next key of each digit goes
    unsigned* s_doff = s_base + kBins;            // exclusive offsets of the digits inside the tile
    __shared__ unsigned s_wtot[kWarps];
    __shared__ __align__(8) unsigned long long bar_k, bar_v;

    const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
    const unsigned lt = (1u << lane) - 1u;
    s_base[t] = offsets[(size_t)t * gridDim.x + blockIdx.x];
    const int64_t tile0 = (int64_t)blockIdx.x * tiles_per_block;
    const int64_t tile1 = min(tile0 + tiles_per_block, tiles);
    // thread 0 stages whole tiles only; every thread derives the same predicate when it consumes them
    auto stage_keys = [&](int64_t tile) {
        if (tile < tile1 && (tile + 1) * kTile <= n) {
            mbar_expect_tx(&bar_k, kTile * 4u);
            tma_copy(st_keys, keys_in + tile * kTile, kTile * 4u, &bar_k);
        }
    };
    auto stage_vals = [&](int64_t tile) {
        if (tile < tile1 && (tile + 1) * kTile <= n) {
            mbar_expect_tx(&bar_v, kTile * 4u);
            tma_copy(st_vals, vals_in + tile * kTile, kTile * 4u, &bar_v);
        }
    };
    if (t == 0) {
        mbar_init(&bar_k, 1);
        mbar_init(&bar_v, 1);
        mbar_fence_init();
        stage_keys(tile0);
        stage_vals(tile0);
    }
    __syncthreads();
    unsigned par_k = 0u, par_v = 0u;
    for (int64_t tile = tile0; tile < tile1; ++tile) {
        const int64_t base_i = tile * kTile;
        const int ntile = (int)min((int64_t)kTile, n - base_i);
        const bool whole = ntile == kTile;
#pragma unroll
        for (int w = 0; w < kWarps; ++w) s_whist[w][t] = 0u;

        unsigned key[kIpt];
        unsigned rank[kIpt];
        if (whole) {
            mbar_wait(&bar_k, par_k);
            par_k ^= 1u;
#pragma unroll
            for (int r = 0; r < kIpt; ++r) key[r] = st_keys[warp * (32 * kIpt) + r * 32 + lane];
        } else {
#pragma unroll
            for (int r = 0; r < kIpt; ++r) {
                const int li = warp * (32 * kIpt) + r * 32 + lane;   // position inside the tile: (warp, round, lane)
                key[r] = li < ntile ? __ldg(keys_in + base_i + li) : 0xffffffffu;
            }
        }
        __syncthreads();   // counters cleared; s_base of the previous tile updated; the key stage has been read by everyone
        if (t == 0) {
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // the reads above before the refill below
            stage_keys(tile + 1);
        }
#pragma unroll
        for (int r = 0; r < kIpt; ++r) {
            const int li = warp * (32 * kIpt) + r * 32 + lane;
            const bool valid = li < ntile;
            const unsigned d = valid ? ((key[r] >> shift) & dmask) : (unsigned)kBins;   // past the end: a group of its own
            unsigned grp = __ballot_sync(kFullMask, valid);   // lanes with this lane's digit (validity is a ninth bit)
            grp = valid ? grp : ~grp;
#pragma unroll
            for (int bit = 0; bit < 8; ++bit) {
                const bool one = (d >> bit) & 1u;
                const unsigned bal = __ballot_sync(kFullMask, one);
                grp &= one ? bal : ~bal;
            }
            const int leader = __ffs(grp) - 1;
            unsigned old = 0u;
            if (lane == leader && valid) {
                old = s_whist[warp][d];
                s_whist[warp][d] = old + __popc(grp);
            }
            old = __shfl_sync(kFullMask, old, leader);
            rank[r] = old + __popc(grp & lt);
            __syncwarp();   // the counter update is visible to the next round's leaders
        }
        __syncthreads();

        // thread t owns digit t: exclusive scan over the warps, the tile's count, the digits' offsets inside the tile
        unsigned cnt = 0u;
#pragma unroll
        for (int w = 0; w < kWarps; ++w) {
            const unsigned c = s_whist[w][t];
            s_whist[w][t] = cnt;
            cnt += c;
        }
        unsigned inc = cnt;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned u = __shfl_up_sync(kFullMask, inc, o);
            if (lane >= o) inc += u;
        }
        if (lane == 31) s_wtot[warp] = inc;
        __syncthreads();
        unsigned wbase = 0u;
#pragma unroll
        for (int w = 0; w < kWarps; ++w) wbase += (w < warp) ? s_wtot[w] : 0u;
        s_doff[t] = wbase + inc - cnt;
        __syncthreads();

        // reorder the tile by digit in shared memory (stable)
        if (whole) {
            mbar_wait(&bar_v, par_v);
            par_v ^= 1u;
        }
#pragma unroll
        for (int r = 0; r < kIpt; ++r) {
            const int li = warp * (32 * kIpt) + r * 32 + lane;
            if (li < ntile) {
                const unsigned d = (key[r] >> shift) & dmask;
                const unsigned lp = s_doff[d] + s_whist[warp][d] + rank[r];
                s_keys[lp] = key[r];
                s_vals[lp] = whole ? st_vals[li] : __ldg(vals_in + base_i + li);
            }
        }
        __syncthreads();   // the tile is in place; the value stage has been read by everyone
        if (t == 0) {
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            stage_vals(tile + 1);
        }

        // write the digits' runs to their places
#pragma unroll
        for (int k = 0; k < kIpt; ++k) {
            const int i = k * kThreads + t;
            if (i < ntile) {
                const unsigned kk = s_keys[i];
                const unsigned d = (kk >> shift) & dmask;
                const unsigned pos = s_base[d] + ((unsigned)i - s_doff[d]);
                keys_out[pos] = kk;
                vals_out[pos] = s_vals[i];
            }
        }
        __syncthreads();   // every thread has read s_base / s_doff / the tile
        s_base[t] += cnt;
    }
}

// Sort n pairs by key bits [begin_bit, end_bit).  (keys_a, vals_a) hold the input; (keys_b, vals_b) are scratch of the
// same size; `temp` has temp_bytes().  Returns 0 when the sorted pairs end in the a buffers, 1 when in the b buffers.
inline int sort_pairs(unsigned* keys_a, int32_t* vals_a, unsigned* keys_b, int32_t* vals_b, int64_t n, int begin_bit, int end_bit,
                      void* temp, int sm_count, cudaStream_t s) {
    const Plan p = make_plan(n, sm_count);
    // 74 KB of dynamic shared memory per block, three blocks per SM; setting a constant attribute again is harmless, so
    // no once-flag (and no race between host threads) is needed
    cudaFuncSetAttribute(downsweep_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kDownSmemBytes);
    cudaFuncSetAttribute(downsweep_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, 100);
    unsigned* counts = reinterpret_cast<unsigned*>(temp);
    unsigned* totals = counts + (size_t)kBins * kMaxGrid;   // per pass: the digits' totals
    cudaMemsetAsync(totals, 0, 4 * kBins * sizeof(unsigned), s);
    int where = 0, pass = 0;
    for (int bit = begin_bit; bit < end_bit; bit += 8) {
        const int nb = end_bit - bit < 8 ? end_bit - bit : 8;
        const unsigned dmask = (1u << nb) - 1u;
        const unsigned* kin = where ? keys_b : keys_a;
        const int32_t* vin = where ? vals_b : vals_a;
        unsigned* kout = where ? keys_a : keys_b;
        int32_t* vout = where ? vals_a : vals_b;
        upsweep_kernel<<<p.grid, kThreads, 0, s>>>(kin, n, bit, dmask, p.tiles_per_block, counts, totals + pass * kBins);
        scan_rows_kernel<<<kBins / 32, 1024, 0, s>>>(counts, totals + pass * kBins, p.grid);
        ++pass;
        downsweep_kernel<<<p.grid, kThreads, kDownSmemBytes, s>>>(kin, vin, kout, vout, n, bit, dmask, p.tiles_per_block, p.tiles,
                                                                  counts);
        where ^= 1;
    }
    return where;
}

// ---- exclusive prefix sum of n ints (flags / counts; total < 2^31), three launches over contiguous ranges ----
constexpr int kScanChunk = 2048;   // ints per block-iteration: 256 threads x 8

__global__ void __launch_bounds__(kThreads) scan_reduce_kernel(const int* __restrict__ in, int64_t n, int64_t per_block,
                                                               unsigned* __restrict__ part) {
    __shared__ unsigned ws[kWarps];
    const int t = threadIdx.x;
    const int64_t begin = (int64_t)blockIdx.x * per_block;
    int64_t end = begin + per_block;
    if (end > n) end = n;
    unsigned s = 0;
    for (int64_t i = begin + t; i < end; i += kThreads) s += (unsigned)__ldg(in + i);
    s = __reduce_add_sync(kFullMask, s);
    if ((t & 31) == 0) ws[t >> 5] = s;
    __syncthreads();
    if (t == 0) {
        unsigned tot = 0;
#pragma unroll
        for (int w = 0; w < kWarps; ++w) tot += ws[w];
        part[blockIdx.x] = tot;
    }
}

__global__ void __launch_bounds__(kThreads) scan_apply_kernel(const int* __restrict__ in, int* __restrict__ out, int64_t n,
                                                              int64_t per_block, const unsigned* __restrict__ part_excl) {
    __shared__ unsigned ws[kWarps];
    const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
    const int64_t begin = (int64_t)blockIdx.x * per_block;
    int64_t end = begin + per_block;
    if (end > n) end = n;
    unsigned run = part_excl[blockIdx.x];
    for (int64_t c0 = begin; c0 < end; c0 += kScanChunk) {
        // thread t owns 8 consecutive values
        const int64_t i0 = c0 + (int64_t)t * 8;
        unsigned v[8];
        unsigned s = 0;
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            v[k] = (i0 + k < end) ? (unsigned)__ldg(in + i0 + k) : 0u;
            s += v[k];
        }
        unsigned inc = s;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned u = __shfl_up_sync(kFullMask, inc, o);
            if (lane >= o) inc += u;
        }
        if (lane == 31) ws[warp] = inc;
        __syncthreads();
        unsigned wbase = 0u, total = 0u;
#pragma unroll
        for (int w = 0; w < kWarps; ++w) {
            const unsigned x = ws[w];
            wbase += (w < warp) ? x : 0u;
            total += x;
        }
        unsigned ex = run + wbase + inc - s;
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            if (i0 + k < end) out[i0 + k] = (int)ex;
            ex += v[k];
        }
        run += total;
        __syncthreads();   // ws is rewritten by the next chunk
    }
}

// bytes of scratch for exclusive_sum
inline size_t scan_temp_bytes() { return (size_t)kMaxGrid * sizeof(unsigned); }

inline void exclusive_sum(const int* in, int* out, int64_t n, void* temp, int sm_count, cudaStream_t s) {
    int64_t g = (int64_t)sm_count * 4;
    if (g > kMaxGrid) g = kMaxGrid;
    const int64_t chunks = (n + kScanChunk - 1) / kScanChunk;
    if (g > chunks) g = chunks;
    if (g < 1) g = 1;
    const int64_t per_block = ((chunks + g - 1) / g) * kScanChunk;
    const int grid = (int)((n + per_block - 1) / per_block);
    unsigned* part = reinterpret_cast<unsigned*>(temp);
    scan_reduce_kernel<<<grid, kThreads, 0, s>>>(in, n, per_block, part);
    scan_small_kernel<<<1, 1024, 0, s>>>(part, grid);
    scan_apply_kernel<<<grid, kThreads, 0, s>>>(in, out, n, per_block, part);
}

}  // namespace covradix
