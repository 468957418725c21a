// Masked residual statistics of a predicted nDSM against the ground-truth DSM (the evaluation step of the inference CLI,
// evaluator.py:53-99): per class ("all" valid pixels + up to 8 masks) count, mean, MAE, RMSE, min, max, median,
// median of |r| and NMAD, with the order statistics exact.
//
// Order statistics come from an MSD radix select on the order-preserving uint64 code of each value (encode_f64),
// 8-bit digits, so one selection round is 8 histogram passes.  A "pair" is the two middle ranks (n-1)/2 and n/2 of
// one value stream of one class; while both ranks sit in the same bucket (always for odd n) they share one histogram.
//   pass 0          residual_stats_kernel: validity, r = pred - gt, per-class sums / min / max (thread partials in
//                   grid-stride order, fixed block tree, block partials in block order) and the digit-0 histograms
//                   of the round-1 streams r and |r|
//   reduce          stats_reduce_kernel: one block per class sums the block partials in a fixed order
//   passes 1..7     select_hist_kernel, round 1: digits 1..7 of r and |r|
//   passes 8..15    select_hist_kernel, round 2: digits 0..7 of |r - median(r)| (needs the round-1 median)
// After every histogram pass select_pick_kernel (one block) walks each selection's 256 bins, appends the digit to the
// selection's prefix, moves its remaining rank into the bucket and clears the histograms, so the passes chain on the
// stream without a host round trip.  Counts are integer atomics (shared memory, then global): bitwise deterministic.
// The grid depends on n only, so a class's result does not depend on the other classes of the call.
#include "t2h_common.cuh"

namespace t2h {

constexpr int kEvalThreads = 256;
constexpr int kEvalMaxBlocks = 8 * kSMs;
constexpr int kEvalMaxClasses = 9;  // "all" + 8 masks
constexpr int kBins = 256;
constexpr int kDigits = 8;
constexpr unsigned kNoSlot = 0xffffffffu;

struct EvalPartial {
  double sum, sum_abs, sum_sq;
  unsigned long long kmin, kmax;  // encode_f64 codes
  long long count;
};
struct EvalSelection {
  unsigned long long prefix[2];  // digits chosen so far of the ranks (n-1)/2 and n/2
  unsigned long long rank[2];    // remaining rank inside the current bucket
};
struct EvalClass {
  long long count;
  double median;  // median(r), the centre of the NMAD round
};
struct EvalWorkspace {
  unsigned long long* hist;  // [2 * 2C slots][256], slot = 2 * pair + side
  EvalSelection* sel;        // [3C]: round 1 pairs (2c: r, 2c + 1: |r|), then round 2 pairs (c: |r - median|)
  EvalClass* cls;            // [C]
  EvalPartial* part;         // [C][blocks]
};

static int eval_blocks(int64_t n_px) {
  const int64_t b = (n_px + kEvalThreads - 1) / kEvalThreads;
  return (int)(b < 1 ? 1 : (b > kEvalMaxBlocks ? kEvalMaxBlocks : b));
}

static size_t eval_layout(int64_t n_px, int nc, char* base, EvalWorkspace* ws) {
  size_t off = 0;
  auto take = [&](size_t bytes) {
    char* p = base ? base + off : nullptr;
    off += (bytes + 255) & ~(size_t)255;
    return p;
  };
  ws->hist = (unsigned long long*)take(sizeof(unsigned long long) * 4 * nc * kBins);
  ws->sel = (EvalSelection*)take(sizeof(EvalSelection) * 3 * nc);
  ws->cls = (EvalClass*)take(sizeof(EvalClass) * nc);
  ws->part = (EvalPartial*)take(sizeof(EvalPartial) * nc * eval_blocks(n_px));
  return off;
}

// class bits of pixel i (bit 0 = "all", bit c + 1 = mask c), 0 when i is past the end or the pixel is not valid
__device__ __forceinline__ unsigned load_residual(const double* __restrict__ pred, const double* __restrict__ gt,
                                                  const uint8_t* __restrict__ bits, int64_t i, int64_t n,
                                                  int use_nodata, double nodata, unsigned class_mask, double& r) {
  if (i >= n) return 0u;
  const double p = __ldg(pred + i), g = __ldg(gt + i);
  if (!isfinite(p) || !isfinite(g) || (use_nodata && g == nodata)) return 0u;
  r = __dsub_rn(p, g);
  return (1u | (bits ? (unsigned)__ldg(bits + i) << 1 : 0u)) & class_mask;
}

// warp-aggregated shared histogram increment; every lane of the warp calls it, kNoSlot = nothing to count
__device__ __forceinline__ void hist_add(unsigned* s_hist, unsigned slot) {
  if (!__any_sync(0xffffffffu, slot != kNoSlot)) return;  // the usual case once a bucket is narrow
  const unsigned peers = __match_any_sync(0xffffffffu, slot);
  if (slot != kNoSlot && (int)(threadIdx.x & 31) == __ffs(peers) - 1) atomicAdd(s_hist + slot, (unsigned)__popc(peers));
}

__device__ __forceinline__ void hist_flush(const unsigned* s_hist, int n_slots, unsigned long long* hist) {
  __syncthreads();
  for (int j = threadIdx.x; j < n_slots * kBins; j += kEvalThreads)
    if (s_hist[j]) atomicAdd(hist + j, (unsigned long long)s_hist[j]);
}

// fixed-order block reduction (xor butterfly in each warp, warps in order); the result is valid in thread 0
__device__ __forceinline__ void block_reduce(EvalPartial& p, EvalPartial* s_warp) {
#pragma unroll
  for (int off = 16; off; off >>= 1) {
    p.sum += __shfl_xor_sync(0xffffffffu, p.sum, off);
    p.sum_abs += __shfl_xor_sync(0xffffffffu, p.sum_abs, off);
    p.sum_sq += __shfl_xor_sync(0xffffffffu, p.sum_sq, off);
    p.kmin = min(p.kmin, __shfl_xor_sync(0xffffffffu, p.kmin, off));
    p.kmax = max(p.kmax, __shfl_xor_sync(0xffffffffu, p.kmax, off));
    p.count += __shfl_xor_sync(0xffffffffu, p.count, off);
  }
  __syncthreads();  // s_warp may still be read by thread 0 for the previous class
  if ((threadIdx.x & 31) == 0) s_warp[threadIdx.x >> 5] = p;
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int w = 1; w < kEvalThreads / 32; ++w) {
      const EvalPartial& q = s_warp[w];
      p.sum += q.sum; p.sum_abs += q.sum_abs; p.sum_sq += q.sum_sq;
      p.kmin = min(p.kmin, q.kmin); p.kmax = max(p.kmax, q.kmax); p.count += q.count;
    }
  }
}

template <int NC>
__global__ void __launch_bounds__(kEvalThreads)
residual_stats_kernel(const double* __restrict__ pred, const double* __restrict__ gt, const uint8_t* __restrict__ bits,
                      int64_t n, int use_nodata, double nodata, EvalWorkspace ws) {
  __shared__ unsigned s_hist[4 * NC * kBins];
  __shared__ EvalPartial s_warp[kEvalThreads / 32];
  for (int j = threadIdx.x; j < 4 * NC * kBins; j += kEvalThreads) s_hist[j] = 0;
  __syncthreads();
  double sum[NC], sum_abs[NC], sum_sq[NC];
  unsigned long long kmin[NC], kmax[NC];
  long long cnt[NC];
#pragma unroll
  for (int c = 0; c < NC; ++c) { sum[c] = sum_abs[c] = sum_sq[c] = 0.0; kmin[c] = ~0ull; kmax[c] = 0ull; cnt[c] = 0; }
  const int lane = threadIdx.x & 31;
  const int64_t stride = (int64_t)gridDim.x * kEvalThreads;
  for (int64_t i = (int64_t)blockIdx.x * kEvalThreads + threadIdx.x; i - lane < n; i += stride) {  // warp-uniform
    double r = 0.0;
    const unsigned cls = load_residual(pred, gt, bits, i, n, use_nodata, nodata, (1u << NC) - 1u, r);
    const double a = fabs(r);
    const unsigned long long kr = encode_f64(r), ka = encode_f64(a);
#pragma unroll
    for (int c = 0; c < NC; ++c) {
      const bool in = (cls >> c) & 1u;
      if (in) {
        sum[c] += r;
        sum_abs[c] += a;
        sum_sq[c] = fma(r, r, sum_sq[c]);
        kmin[c] = min(kmin[c], kr);
        kmax[c] = max(kmax[c], kr);
        ++cnt[c];
      }
      // digit 0: both ranks of a pair share side 0 of the pair's slots (pair 2c -> slot 4c, pair 2c + 1 -> 4c + 2)
      hist_add(s_hist, in ? (unsigned)(4 * c) * kBins + (unsigned)(kr >> 56) : kNoSlot);
      hist_add(s_hist, in ? (unsigned)(4 * c + 2) * kBins + (unsigned)(ka >> 56) : kNoSlot);
    }
  }
#pragma unroll
  for (int c = 0; c < NC; ++c) {
    EvalPartial p{sum[c], sum_abs[c], sum_sq[c], kmin[c], kmax[c], cnt[c]};
    block_reduce(p, s_warp);
    if (threadIdx.x == 0) ws.part[(int64_t)c * gridDim.x + blockIdx.x] = p;
  }
  hist_flush(s_hist, 4 * NC, ws.hist);
}

// one block per class: block partials in a fixed order; writes count, mean, mae, rmse, min, max
__global__ void __launch_bounds__(kEvalThreads)
stats_reduce_kernel(EvalWorkspace ws, int n_blocks, double* __restrict__ out_stats, int64_t* __restrict__ out_count) {
  __shared__ EvalPartial s_warp[kEvalThreads / 32];
  const int c = blockIdx.x;
  EvalPartial p{0.0, 0.0, 0.0, ~0ull, 0ull, 0};
  for (int b = threadIdx.x; b < n_blocks; b += kEvalThreads) {
    const EvalPartial& q = ws.part[(int64_t)c * n_blocks + b];
    p.sum += q.sum; p.sum_abs += q.sum_abs; p.sum_sq += q.sum_sq;
    p.kmin = min(p.kmin, q.kmin); p.kmax = max(p.kmax, q.kmax); p.count += q.count;
  }
  block_reduce(p, s_warp);
  if (threadIdx.x == 0) {
    const double nan = __longlong_as_double(0x7ff8000000000000ll), n = (double)p.count;
    double* o = out_stats + (int64_t)c * 8;
    ws.cls[c].count = p.count;
    out_count[c] = p.count;
    o[0] = p.count ? p.sum / n : nan;
    o[1] = p.count ? p.sum_abs / n : nan;
    o[2] = p.count ? sqrt(p.sum_sq / n) : nan;
    o[3] = p.count ? decode_f64(p.kmin) : nan;
    o[4] = p.count ? decode_f64(p.kmax) : nan;
  }
}

// one histogram pass: digit `digit` of the round-1 streams r, |r| (round 1, digit >= 1) or of |r - median(r)| (round 2)
__global__ void __launch_bounds__(kEvalThreads)
select_hist_kernel(const double* __restrict__ pred, const double* __restrict__ gt, const uint8_t* __restrict__ bits,
                   int64_t n, int nc, int use_nodata, double nodata, int round, int digit, EvalWorkspace ws) {
  extern __shared__ unsigned s_hist[];  // [2 * n_pairs][256]
  __shared__ unsigned long long s_prefix[2 * 2 * kEvalMaxClasses];
  __shared__ int s_shared[2 * kEvalMaxClasses];
  __shared__ double s_median[kEvalMaxClasses];
  const int n_pairs = round == 1 ? 2 * nc : nc;
  const EvalSelection* sel = ws.sel + (round == 1 ? 0 : 2 * nc);
  for (int j = threadIdx.x; j < 2 * n_pairs * kBins; j += kEvalThreads) s_hist[j] = 0;
  if (threadIdx.x < n_pairs) {
    const unsigned long long lo = digit ? sel[threadIdx.x].prefix[0] : 0ull;
    const unsigned long long hi = digit ? sel[threadIdx.x].prefix[1] : 0ull;
    s_prefix[2 * threadIdx.x] = lo;
    s_prefix[2 * threadIdx.x + 1] = hi;
    s_shared[threadIdx.x] = lo == hi;
  }
  if (round == 2 && threadIdx.x < nc) s_median[threadIdx.x] = ws.cls[threadIdx.x].median;
  __syncthreads();
  const int shift = 56 - 8 * digit;
  const unsigned long long high = digit ? ~0ull << (shift + 8) : 0ull;  // the digits already chosen
  const int lane = threadIdx.x & 31;
  const int64_t stride = (int64_t)gridDim.x * kEvalThreads;
  auto count = [&](int pair, unsigned long long key, bool in) {
    const unsigned d = (unsigned)(key >> shift) & (kBins - 1);
    hist_add(s_hist, in && !((key ^ s_prefix[2 * pair]) & high) ? (unsigned)(2 * pair) * kBins + d : kNoSlot);
    if (!s_shared[pair])
      hist_add(s_hist, in && !((key ^ s_prefix[2 * pair + 1]) & high) ? (unsigned)(2 * pair + 1) * kBins + d : kNoSlot);
  };
  for (int64_t i = (int64_t)blockIdx.x * kEvalThreads + threadIdx.x; i - lane < n; i += stride) {  // warp-uniform
    double r = 0.0;
    const unsigned cls = load_residual(pred, gt, bits, i, n, use_nodata, nodata, (1u << nc) - 1u, r);
    if (round == 1) {
      const unsigned long long kr = encode_f64(r), ka = encode_f64(fabs(r));
      for (int c = 0; c < nc; ++c) {
        const bool in = (cls >> c) & 1u;
        count(2 * c, kr, in);
        count(2 * c + 1, ka, in);
      }
    } else {
      for (int c = 0; c < nc; ++c) count(c, encode_f64(fabs(__dsub_rn(r, s_median[c]))), (cls >> c) & 1u);
    }
  }
  hist_flush(s_hist, 2 * n_pairs, ws.hist);
}

// move (prefix, rank) into the bucket of the next digit that holds the rank
__device__ __forceinline__ void descend(const unsigned long long* h, int shift, unsigned long long& prefix,
                                        unsigned long long& rank) {
  unsigned long long below = 0;
  for (int b = 0; b < kBins; ++b) {
    if (rank < below + h[b]) {
      prefix |= (unsigned long long)b << shift;
      rank -= below;
      return;
    }
    below += h[b];
  }
}

// one thread per pair: consume the histograms of digit `digit`, clear them; after the last digit decode the two middle
// values and write median (round 1, r), medae (round 1, |r|) or nmad (round 2)
__global__ void __launch_bounds__(kEvalThreads)
select_pick_kernel(int nc, int round, int digit, EvalWorkspace ws, double* __restrict__ out_stats) {
  const int n_pairs = round == 1 ? 2 * nc : nc;
  const int p = threadIdx.x;
  if (p < n_pairs) {
    EvalSelection& s = ws.sel[(round == 1 ? 0 : 2 * nc) + p];
    const int c = round == 1 ? p >> 1 : p;
    const int field = round == 1 ? 5 + (p & 1) : 7;
    const long long n = ws.cls[c].count;
    if (n > 0) {
      if (digit == 0) {
        s.prefix[0] = s.prefix[1] = 0ull;
        s.rank[0] = (unsigned long long)(n - 1) / 2;
        s.rank[1] = (unsigned long long)n / 2;
      }
      const bool shared = s.prefix[0] == s.prefix[1];  // as select_hist_kernel saw it
      const unsigned long long* h = ws.hist + (int64_t)2 * p * kBins;
      const int shift = 56 - 8 * digit;
      descend(h, shift, s.prefix[0], s.rank[0]);
      descend(shared ? h : h + kBins, shift, s.prefix[1], s.rank[1]);
      if (digit == kDigits - 1) {
        const double a = decode_f64(s.prefix[0]), b = decode_f64(s.prefix[1]);
        const double med = (n & 1) ? a : __dadd_rn(a, b) / 2.0;  // np.median: mean of the two middle values
        if (round == 1 && !(p & 1)) ws.cls[c].median = med;
        out_stats[(int64_t)c * 8 + field] = round == 1 ? med : __dmul_rn(1.4826, med);
      }
    } else if (digit == kDigits - 1) {
      out_stats[(int64_t)c * 8 + field] = __longlong_as_double(0x7ff8000000000000ll);
    }
  }
  __syncthreads();
  for (int j = threadIdx.x; j < 2 * n_pairs * kBins; j += kEvalThreads) ws.hist[j] = 0ull;
}

}  // namespace t2h

using namespace t2h;

extern "C" size_t t2h_residual_stats_workspace_bytes(int64_t n_px, int n_masks) {
  if (n_px < 0 || n_masks < 0 || n_masks > kEvalMaxClasses - 1) return 0;
  EvalWorkspace ws;
  return eval_layout(n_px, 1 + n_masks, nullptr, &ws);
}

extern "C" int t2h_residual_stats(const double* pred, const double* gt, int64_t n_px, const uint8_t* mask_bits,
                                  int n_masks, int use_nodata, double nodata, void* workspace, size_t workspace_bytes,
                                  double* out_stats, int64_t* out_count, t2h_stream_t stream) {
  if (n_px < 0 || n_masks < 0 || n_masks > kEvalMaxClasses - 1 || (n_px > 0 && (!pred || !gt)) ||
      (n_px > 0 && n_masks > 0 && !mask_bits) || !workspace || !out_stats || !out_count)
    return T2H_ERR_INVALID_ARGUMENT;
  const int nc = 1 + n_masks;
  EvalWorkspace ws;
  if (workspace_bytes < eval_layout(n_px, nc, (char*)workspace, &ws)) return T2H_ERR_WORKSPACE_TOO_SMALL;
  const cudaStream_t s = (cudaStream_t)stream;
  const uint8_t* bits = n_masks ? mask_bits : nullptr;
  const int blocks = eval_blocks(n_px);
  if (cudaMemsetAsync(ws.hist, 0, sizeof(unsigned long long) * 4 * nc * kBins, s) != cudaSuccess) {
    (void)cudaGetLastError();
    return T2H_ERR_CUDA;
  }
#define T2H_EVAL_STATS(NC_) \
  case NC_: residual_stats_kernel<NC_><<<blocks, kEvalThreads, 0, s>>>(pred, gt, bits, n_px, use_nodata, nodata, ws); break;
  switch (nc) {
    T2H_EVAL_STATS(1) T2H_EVAL_STATS(2) T2H_EVAL_STATS(3) T2H_EVAL_STATS(4) T2H_EVAL_STATS(5)
    T2H_EVAL_STATS(6) T2H_EVAL_STATS(7) T2H_EVAL_STATS(8) T2H_EVAL_STATS(9)
  }
#undef T2H_EVAL_STATS
  T2H_CHECK_LAUNCH();
  stats_reduce_kernel<<<nc, kEvalThreads, 0, s>>>(ws, blocks, out_stats, out_count);
  for (int round = 1; round <= 2; ++round) {
    const int n_pairs = round == 1 ? 2 * nc : nc;
    for (int digit = 0; digit < kDigits; ++digit) {
      if (round == 2 || digit > 0)  // digit 0 of round 1 was counted by residual_stats_kernel
        select_hist_kernel<<<blocks, kEvalThreads, sizeof(unsigned) * 2 * n_pairs * kBins, s>>>(
            pred, gt, bits, n_px, nc, use_nodata, nodata, round, digit, ws);
      select_pick_kernel<<<1, kEvalThreads, 0, s>>>(nc, round, digit, ws, out_stats);
    }
  }
  T2H_CHECK_LAUNCH();
  return T2H_OK;
}
