// rt_sort.cuh — hand-written stable LSD radix sort of (uint32 key, int32 value) pairs, 8-bit
// digits, no CUB: per-block histograms -> one-block exclusive scan -> stable scatter with
// warp __match_any ranking.  Used by the LBVH build (Morton codes).  The element count may
// live on the device (n_dev), so a sort can be enqueued before the host knows it.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace rt {

#define SORT_THREADS 256
#define SORT_WARPS (SORT_THREADS / 32)
#define SORT_MAX_BLOCKS 4096

__device__ __forceinline__ void sort_extent(int& n, int& chunk, int nblocks, const unsigned long long* n_dev) {
    if (n_dev) n = (int)*n_dev;
    chunk = (n + nblocks - 1) / nblocks;
    chunk = (chunk + SORT_THREADS - 1) / SORT_THREADS * SORT_THREADS;
}

static __global__ void k_sort_hist(const uint32_t* __restrict__ keys, int n, const unsigned long long* n_dev, int shift,
                                   int nblocks, int* __restrict__ hist /*[256][nblocks]*/) {
    __shared__ int sh[256];
    int chunk;
    sort_extent(n, chunk, nblocks, n_dev);
    sh[threadIdx.x] = 0;
    __syncthreads();
    int begin = blockIdx.x * chunk, end = min(begin + chunk, n);
    for (int i = begin + threadIdx.x; i < end; i += SORT_THREADS) atomicAdd(&sh[(keys[i] >> shift) & 255], 1);
    __syncthreads();
    hist[threadIdx.x * nblocks + blockIdx.x] = sh[threadIdx.x];
}

// Offsets from the per-block histograms hist[digit][block]: block `d` of k_sort_rowscan turns
// row d into its exclusive prefix over the blocks and records the row total; k_sort_digitscan
// turns the 256 totals into the digits' base offsets.  (A single-block scan over all
// 256 * nblocks counters took 0.58 ms per radix pass at 4096 blocks — most of the sort.)
static __global__ void k_sort_rowscan(int* __restrict__ hist, int nblocks, int* __restrict__ totals) {
    __shared__ int warp_sums[SORT_WARPS];
    int* row = hist + (size_t)blockIdx.x * nblocks;
    const int per = (nblocks + SORT_THREADS - 1) / SORT_THREADS;
    const int begin = min((int)threadIdx.x * per, nblocks), end = min(begin + per, nblocks);
    int sum = 0;
    for (int i = begin; i < end; i++) sum += row[i];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    int incl = sum;
    for (int o = 1; o < 32; o <<= 1) {
        int v = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += v;
    }
    if (lane == 31) warp_sums[w] = incl;
    __syncthreads();
    int wbase = 0, total = 0;
    for (int k = 0; k < SORT_WARPS; k++) {
        if (k < w) wbase += warp_sums[k];
        total += warp_sums[k];
    }
    int run = wbase + incl - sum;
    for (int i = begin; i < end; i++) {
        int v = row[i];
        row[i] = run;
        run += v;
    }
    if (threadIdx.x == 0) totals[blockIdx.x] = total;
}
// exclusive scan of the 256 digit totals, in place, by one block of 256 threads
static __global__ void k_sort_digitscan(int* __restrict__ totals) {
    __shared__ int sh[256];
    const int t = threadIdx.x;
    const int v = totals[t];
    sh[t] = v;
    __syncthreads();
    for (int o = 1; o < 256; o <<= 1) {
        int add = t >= o ? sh[t - o] : 0;
        __syncthreads();
        sh[t] += add;
        __syncthreads();
    }
    totals[t] = sh[t] - v;
}

static __global__ void k_sort_scatter(const uint32_t* __restrict__ keys_in, const int* __restrict__ vals_in,
                                      uint32_t* __restrict__ keys_out, int* __restrict__ vals_out, int n,
                                      const unsigned long long* n_dev, int shift, int nblocks,
                                      const int* __restrict__ offsets, const int* __restrict__ digit_base) {
    __shared__ int base[256];
    __shared__ int warp_cnt[SORT_WARPS][256];
    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
    int chunk;
    sort_extent(n, chunk, nblocks, n_dev);
    base[tid] = offsets[tid * nblocks + blockIdx.x] + digit_base[tid];
    for (int k = 0; k < SORT_WARPS; k++) warp_cnt[k][tid] = 0;
    __syncthreads();
    int begin = blockIdx.x * chunk, end = min(begin + chunk, n);
    for (int tile = begin; tile < end; tile += SORT_THREADS) {
        int i = tile + tid;
        bool valid = i < end;
        uint32_t key = valid ? keys_in[i] : 0u;
        int val = valid ? vals_in[i] : 0;
        uint32_t digit = valid ? ((key >> shift) & 255u) : (0x10000u + lane);
        unsigned peers = __match_any_sync(0xffffffffu, digit);
        int rank = __popc(peers & ((1u << lane) - 1u));
        if (valid && rank == 0) warp_cnt[w][digit] = __popc(peers);
        __syncthreads();
        if (valid) {
            int off = 0;
            for (int k = 0; k < w; k++) off += warp_cnt[k][digit];
            int pos = base[digit] + off + rank;
            keys_out[pos] = key;
            vals_out[pos] = val;
        }
        __syncthreads();
        int tot = 0;
        for (int k = 0; k < SORT_WARPS; k++) {
            tot += warp_cnt[k][tid];
            warp_cnt[k][tid] = 0;
        }
        base[tid] += tot;
        __syncthreads();
    }
}

// Sorts by all 32 key bits (four passes).  n_max sizes the grid; the real count is n_max, or
// *n_dev when n_dev != nullptr.  On return kin/vin point at the sorted data (the pointers are
// swapped once per pass).  hist: 256 * (SORT_MAX_BLOCKS + 1) ints of scratch.
static inline void sort_pairs(cudaStream_t stream, uint32_t*& kin, uint32_t*& kout, int*& vin, int*& vout, int* hist,
                              int n_max, const unsigned long long* n_dev, int* launches) {
    int sblocks = (n_max + 4095) / 4096;
    if (sblocks > SORT_MAX_BLOCKS) sblocks = SORT_MAX_BLOCKS;
    if (sblocks < 1) sblocks = 1;
    for (int shift = 0; shift < 32; shift += 8) {
        k_sort_hist<<<sblocks, SORT_THREADS, 0, stream>>>(kin, n_max, n_dev, shift, sblocks, hist);
        int* totals = hist + (size_t)256 * SORT_MAX_BLOCKS;
        k_sort_rowscan<<<256, SORT_THREADS, 0, stream>>>(hist, sblocks, totals);
        k_sort_digitscan<<<1, 256, 0, stream>>>(totals);
        k_sort_scatter<<<sblocks, SORT_THREADS, 0, stream>>>(kin, vin, kout, vout, n_max, n_dev, shift, sblocks, hist, totals);
        if (launches) (*launches) += 4;
        uint32_t* tk = kin; kin = kout; kout = tk;
        int* tv = vin; vin = vout; vout = tv;
    }
}

}  // namespace rt
