// spectral_b200/csrc/topk.cuh -- exact top-k selection over device-resident costs (spectral_topk_device, spectral_sweep_topk).
//
// Order: ascending on (key(cost), global index), key = an order-preserving 64-bit image of the double in which -0.0 equals
// +0.0 and every NaN lies above +inf.  The k-th smallest entry is found by an MSB-first radix select (TK_BITS-bit digits, a
// fixed number of passes, no host readback), the entries below it and the first ties at it are compacted into <= 1024
// candidates, and one block sorts those.  Scratch is O(k + grid), independent of the number of entries.
//
// Two index modes:
//   implicit  global index = index_offset + i.  The select runs on the 64-bit key only; the ties at the threshold key are taken
//             in position order (= index order), from per-block tie counts over contiguous block ranges.  6 + 2 launches.
//   explicit  index[i] (int64; < 0 marks an empty slot, ranked after everything and returned as (+inf, -1)).  Index order is
//             not position order, so the select runs on the 128-bit composite (key, index) instead.  12 + 2 launches.  Used by
//             the cross-rank merge, on nranks x k records.
#pragma once

#include <cub/block/block_reduce.cuh>
#include <cub/block/block_scan.cuh>

#include "common.cuh"

constexpr int TK_BITS = 11, TK_BINS = 1 << TK_BITS;   // 2048 bins: 8 KB of shared memory per block
constexpr int TK_THREADS = 256, TK_UNROLL = 4;        // TK_BINS / TK_THREADS = 8 bins per thread in the digit pick
constexpr int TK_FIN_THREADS = 1024;                   // k_topk_finish: one compare-exchange per thread per bitonic step
constexpr int TK_MAX = SPECTRAL_TOPK_MAX;              // 1024 candidates at most
constexpr int TK_GRID_MAX = 1024;                      // blocks per launch at most (block_ties[] capacity)
constexpr int TK_PASSES_MAX = (128 + TK_BITS - 1) / TK_BITS;  // 12: the explicit-index select
static_assert(TK_BINS % TK_THREADS == 0, "the digit pick gives every thread the same number of bins");

typedef unsigned long long tk_u64;

struct TopkState {
  tk_u64 pre_hi, pre_lo;  // the composite prefix selected so far (the threshold T once every pass has run)
  unsigned r;             // rank of the k-th entry among those that share the prefix (1-based); after the last pass: ties to take at T
  unsigned ticket;        // last-block election of the pass / finish kernels (reset by the last block)
  unsigned cand;          // candidates written below T by k_topk_compact (reset by k_topk_finish)
  unsigned pad;
};

struct TopkScratch {
  unsigned *hist;          // [TK_PASSES_MAX][TK_BINS], zero between calls (each pass' last block clears its own)
  TopkState *st;
  unsigned *block_ties;    // [TK_GRID_MAX] entries equal to T per block
  tk_u64 *ck, *ci;         // [TK_MAX] candidate keys and indices (index as unsigned: -1 -> all ones)
  double *cc;              // [TK_MAX] candidate costs, as stored
};

struct TopkArgs {
  const double *cost;       // entry i at cost[i * cost_stride]
  const long long *index;   // NULL: implicit index index_offset + i; else entry i's index at index[i * cost_stride]
  long long index_offset;
  int cost_stride;
  int n;                    // entries
  int keff;                 // min(k, n): entries that are selected
  int k;                    // output slots; [keff, k) are written as (+inf, -1)
  int total_bits;           // 64 (implicit) or 128 (explicit)
  double *out_cost;         // slot j at out_cost[j * out_stride]
  long long *out_index;     // slot j at out_index[j * out_stride]
  int out_stride;
  TopkScratch s;
};

// order-preserving image of a double: -0.0 -> +0.0, every NaN -> all ones (above +inf = 0xFFF0...)
__device__ __forceinline__ tk_u64 tk_key(double c) {
  if (c != c) return ~0ull;
  const tk_u64 u = c == 0.0 ? 0ull : (tk_u64)__double_as_longlong(c);
  return (u >> 63) ? ~u : (u | 0x8000000000000000ull);
}

// entry i: select composite (kh, kl), its global index (unsigned image) and stored cost
__device__ __forceinline__ void tk_entry(const TopkArgs &a, long long i, tk_u64 &kh, tk_u64 &kl, tk_u64 &idx, double &c) {
  c = a.cost[i * a.cost_stride];
  kh = tk_key(c);
  if (a.index) {
    const long long g = a.index[i * a.cost_stride];
    idx = (tk_u64)g;
    if (g < 0) { kh = ~0ull; idx = ~0ull; }
    kl = idx;
  } else {
    idx = (tk_u64)(a.index_offset + i);
    kl = 0;  // implicit mode: ties at the key are resolved by position, not by the select
  }
}

// bits [pos, pos + w) of the 128-bit value (hi:lo), w <= TK_BITS
__device__ __forceinline__ unsigned tk_digit(tk_u64 hi, tk_u64 lo, int pos, int w) {
  tk_u64 v;
  if (pos >= 64) v = hi >> (pos - 64);
  else if (pos == 0) v = lo;
  else v = (lo >> pos) | (hi << (64 - pos));
  return (unsigned)(v & ((1ull << w) - 1));
}
// (ah:al) and (bh:bl) agree on every bit >= top (0 < top <= 128)
__device__ __forceinline__ bool tk_same_above(tk_u64 ah, tk_u64 al, tk_u64 bh, tk_u64 bl, int top) {
  if (top >= 128) return true;
  if (top >= 64) return ((ah ^ bh) >> (top - 64)) == 0;
  return ah == bh && ((al ^ bl) >> top) == 0;
}
__device__ __forceinline__ bool tk_less(tk_u64 ah, tk_u64 al, tk_u64 bh, tk_u64 bl) { return ah < bh || (ah == bh && al < bl); }

// the contiguous range of entries owned by block b of g
__device__ __forceinline__ void tk_range(int n, int b, int g, long long &beg, long long &end) {
  const long long chunk = ((long long)n + g - 1) / g;
  beg = (long long)b * chunk;
  end = beg + chunk < n ? beg + chunk : n;
  if (beg > n) beg = n;
}

__device__ __forceinline__ void tk_pass_bits(const TopkArgs &a, int pass, int &pos, int &w) {
  const int top = 128 - TK_BITS * pass, floor_bit = 128 - a.total_bits;
  pos = top - TK_BITS > floor_bit ? top - TK_BITS : floor_bit;
  w = top - pos;
}

// One radix pass: histogram of digit `pass` over the entries that share the prefix, merged into hist[pass]; the last block
// picks the digit that holds the r-th entry, extends the prefix, updates r and clears hist[pass] for the next call.
__global__ void __launch_bounds__(TK_THREADS) k_topk_pass(const TopkArgs a, int pass) {
  __shared__ unsigned h[TK_BINS];
  __shared__ bool is_last;
  typedef cub::BlockScan<unsigned, TK_THREADS> Scan;
  __shared__ typename Scan::TempStorage scan_tmp;
  int pos, w;
  tk_pass_bits(a, pass, pos, w);
  const int top = pos + w;
  tk_u64 ph = 0, pl = 0;
  if (pass > 0) { ph = a.s.st->pre_hi; pl = a.s.st->pre_lo; }
  for (int j = threadIdx.x; j < TK_BINS; j += TK_THREADS) h[j] = 0;
  __syncthreads();
  const int lane = threadIdx.x & 31;
  long long beg, end;
  tk_range(a.n, blockIdx.x, gridDim.x, beg, end);
  for (long long i0 = beg; i0 < end; i0 += TK_THREADS * TK_UNROLL) {
    unsigned d[TK_UNROLL];
#pragma unroll
    for (int u = 0; u < TK_UNROLL; u++) {
      const long long i = i0 + u * TK_THREADS + threadIdx.x;
      d[u] = ~0u;
      if (i < end) {
        tk_u64 kh, kl, idx;
        double c;
        tk_entry(a, i, kh, kl, idx, c);
        if (tk_same_above(kh, kl, ph, pl, top)) d[u] = tk_digit(kh, kl, pos, w);
      }
    }
#pragma unroll
    for (int u = 0; u < TK_UNROLL; u++) {  // one shared atomic per distinct digit of the warp (runs of equal costs are common)
      const unsigned peers = __match_any_sync(0xffffffffu, d[u]);
      if (d[u] != ~0u && lane == __ffs(peers) - 1) atomicAdd(&h[d[u]], (unsigned)__popc(peers));
    }
  }
  __syncthreads();
  unsigned *gh = a.s.hist + (size_t)pass * TK_BINS;
  for (int j = threadIdx.x; j < TK_BINS; j += TK_THREADS)
    if (h[j]) atomicAdd(&gh[j], h[j]);
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) is_last = atomicAdd(&a.s.st->ticket, 1u) == gridDim.x - 1;
  __syncthreads();
  if (!is_last) return;
  __threadfence();
  // the digit pick: thread t owns bins [8 t, 8 t + 8)
  constexpr int PER = TK_BINS / TK_THREADS;
  unsigned cnt[PER], sum = 0;
#pragma unroll
  for (int j = 0; j < PER; j++) {
    cnt[j] = __ldcg(&gh[threadIdx.x * PER + j]);
    gh[threadIdx.x * PER + j] = 0;
    sum += cnt[j];
  }
  unsigned before;
  Scan(scan_tmp).ExclusiveSum(sum, before);
  const unsigned r = pass == 0 ? (unsigned)a.keff : a.s.st->r;
  if (before < r && before + sum >= r) {
    unsigned c = before;
    int dsel = 0;
#pragma unroll
    for (int j = 0; j < PER; j++) {
      if (c + cnt[j] >= r) { dsel = threadIdx.x * PER + j; break; }
      c += cnt[j];
    }
    const tk_u64 dd = (tk_u64)dsel;
    if (pos >= 64) ph |= dd << (pos - 64);
    else {
      pl |= dd << pos;
      if (pos + w > 64) ph |= dd >> (64 - pos);
    }
    a.s.st->pre_hi = ph; a.s.st->pre_lo = pl; a.s.st->r = r - c;
  }
  if (threadIdx.x == 0) a.s.st->ticket = 0;
}

// Every entry strictly below T becomes a candidate (fewer than keff of them, slot by atomic: the final sort orders them);
// the entries equal to T are counted per block.
__global__ void __launch_bounds__(TK_THREADS) k_topk_compact(const TopkArgs a) {
  typedef cub::BlockReduce<unsigned, TK_THREADS> Red;
  __shared__ typename Red::TempStorage red_tmp;
  const tk_u64 th = a.s.st->pre_hi, tl = a.s.st->pre_lo;
  const int lane = threadIdx.x & 31;
  long long beg, end;
  tk_range(a.n, blockIdx.x, gridDim.x, beg, end);
  unsigned ties = 0;
  for (long long i0 = beg; i0 < end; i0 += TK_THREADS) {
    const long long i = i0 + threadIdx.x;
    tk_u64 kh = ~0ull, kl = ~0ull, idx = 0;
    double c = 0.0;
    bool less = false;
    if (i < end) {
      tk_entry(a, i, kh, kl, idx, c);
      less = tk_less(kh, kl, th, tl);
      ties += (kh == th && kl == tl) ? 1u : 0u;
    }
    const unsigned m = __ballot_sync(0xffffffffu, less);
    if (m) {
      unsigned base = 0;
      if (lane == __ffs(m) - 1) base = atomicAdd(&a.s.st->cand, (unsigned)__popc(m));
      base = __shfl_sync(0xffffffffu, base, __ffs(m) - 1);
      if (less) {
        const unsigned slot = base + __popc(m & ((1u << lane) - 1));
        a.s.ck[slot] = kh; a.s.ci[slot] = idx; a.s.cc[slot] = c;
      }
    }
  }
  const unsigned tot = Red(red_tmp).Sum(ties);
  if (threadIdx.x == 0) a.s.block_ties[blockIdx.x] = tot;
}

// The first r entries equal to T in position order (exclusive scan of the per-block tie counts, then a block scan inside the
// range), placed after the candidates below T; the last block sorts the keff candidates by (key, index) and writes the k slots.
__global__ void __launch_bounds__(TK_FIN_THREADS) k_topk_finish(const TopkArgs a) {
  typedef cub::BlockScan<unsigned, TK_FIN_THREADS> Scan;
  typedef cub::BlockReduce<unsigned, TK_FIN_THREADS> Red;
  __shared__ union { typename Scan::TempStorage scan; typename Red::TempStorage red; } tmp;
  __shared__ tk_u64 sk[TK_MAX], si[TK_MAX];
  __shared__ double sc[TK_MAX];
  __shared__ bool is_last;
  const tk_u64 th = a.s.st->pre_hi, tl = a.s.st->pre_lo;
  const unsigned r = a.s.st->r, less = (unsigned)a.keff - r;
  const unsigned mine = a.s.block_ties[blockIdx.x];
  if (mine) {
    unsigned part = 0;
    for (int b = threadIdx.x; b < (int)blockIdx.x; b += TK_FIN_THREADS) part += a.s.block_ties[b];
    const unsigned before = Red(tmp.red).Sum(part);
    __shared__ unsigned s_before;
    if (threadIdx.x == 0) s_before = before;
    __syncthreads();
    unsigned rank0 = s_before;  // tie rank of the next tie of this block
    long long beg, end;
    tk_range(a.n, blockIdx.x, gridDim.x, beg, end);
    for (long long i0 = beg; i0 < end && rank0 < r; i0 += TK_FIN_THREADS) {
      const long long i = i0 + threadIdx.x;
      tk_u64 kh = 0, kl = 0, idx = 0;
      double c = 0.0;
      unsigned tie = 0;
      if (i < end) {
        tk_entry(a, i, kh, kl, idx, c);
        tie = (kh == th && kl == tl) ? 1u : 0u;
      }
      unsigned ex, agg;
      Scan(tmp.scan).ExclusiveSum(tie, ex, agg);
      if (tie && rank0 + ex < r) {
        const unsigned slot = less + rank0 + ex;
        a.s.ck[slot] = kh; a.s.ci[slot] = idx; a.s.cc[slot] = c;
      }
      rank0 += agg;
      __syncthreads();  // tmp.scan is reused by the next tile
    }
  }
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) is_last = atomicAdd(&a.s.st->ticket, 1u) == gridDim.x - 1;
  __syncthreads();
  if (!is_last) return;
  __threadfence();
  int n2 = 1;
  while (n2 < a.keff) n2 <<= 1;
  for (int j = threadIdx.x; j < n2; j += TK_FIN_THREADS) {
    if (j < a.keff) { sk[j] = __ldcg(&a.s.ck[j]); si[j] = __ldcg(&a.s.ci[j]); sc[j] = __ldcg(&a.s.cc[j]); }
    else { sk[j] = ~0ull; si[j] = ~0ull; sc[j] = 0.0; }
  }
  __syncthreads();
  // bitonic sort of n2 <= 1024 (key, index) pairs, ascending; the pairs are distinct except for empty slots (explicit mode)
  for (int size = 2; size <= n2; size <<= 1)
    for (int stride = size >> 1; stride > 0; stride >>= 1) {
      for (int t = threadIdx.x; t < (n2 >> 1); t += TK_FIN_THREADS) {
        const int lo = 2 * t - (t & (stride - 1)), hi = lo + stride;
        const bool up = (lo & size) == 0;
        const bool gt = tk_less(sk[hi], si[hi], sk[lo], si[lo]);
        if (gt == up) {
          const tk_u64 k0 = sk[lo], i0 = si[lo];
          const double c0 = sc[lo];
          sk[lo] = sk[hi]; si[lo] = si[hi]; sc[lo] = sc[hi];
          sk[hi] = k0; si[hi] = i0; sc[hi] = c0;
        }
      }
      __syncthreads();
    }
  for (int j = threadIdx.x; j < a.k; j += TK_FIN_THREADS) {
    const bool real = j < a.keff && si[j] != ~0ull;
    a.out_cost[(size_t)j * a.out_stride] = real ? sc[j] : __longlong_as_double(0x7FF0000000000000LL);
    a.out_index[(size_t)j * a.out_stride] = real ? (long long)si[j] : -1LL;
  }
  if (threadIdx.x == 0) { a.s.st->ticket = 0; a.s.st->cand = 0; }
}
