// Post-path reductions on device (SURVEY 8(f).3). The reference hands back raw draws only (mcmc.js:1029) and leaves the
// summary (mean / sd / quantiles, README.md:44-52 plots them) to the caller; with 2^20..2^22 chains the raw block is GBs, so the
// summary is formed where the draws are and only a few hundred bytes cross PCIe / NVLink.
//
// Input everywhere: a device-resident sample block in amwg_sample_device's layout, x[row][entry][chain] (chain fastest).
//   K_m1  amwg_chain_moments_kernel : one thread per (chain, entry): mean and M2 of the chain over its rows, two sequential passes
//                                     (coalesced over chains; HBM-bound: 2 reads of the block), Chan-merged per CTA in a fixed tree
//   K_m2  amwg_merge_moments_kernel : one CTA per entry merges the per-CTA records, again in a FIXED order, so the result does
//                                     not depend on scheduling
//   K_q   amwg_digit_hist_kernel    : one pass of an exact MSD radix select over the order-preserving 64-bit key of the draws:
//                                     counts of the next 8-bit digit among the values whose higher digits equal a given prefix
//                                     (integer counts: exact, order independent, summed across GPUs by the caller)
//   K_a1  amwg_split_autocov_kernel : one thread per (chain, live entry), both halves of the split chain: one pass for the two
//                                     half-chain means, one pass forming a tile of L lagged products from a sliding window of
//                                     centred values in registers (one DFMA per product, no load); per-CTA fixed trees
//   K_a2  amwg_merge_autocov_kernel : one CTA per live entry merges the per-CTA records and sums in a FIXED order
// Included at the end of amwg_kernels.cu (same translation unit: shares CUDA_TRY / fail()).
#pragma once

namespace summary {

constexpr int kMaxPrefixes = 32;      // distinct prefixes per entry and pass (order statistics being selected at once)
// lags per autocovariance tile: the window and the sums take 2 x 16 doubles per thread and fit 128 registers without spills
// (2 CTAs of 256 threads per SM); a 32-lag tile needs more than 255 and spills
constexpr int kLagTile = 16;

__device__ __forceinline__ unsigned long long ordered_key(double x) {
  unsigned long long u = (unsigned long long)__double_as_longlong(x);
  return (u >> 63) ? ~u : (u | 0x8000000000000000ull);      // ascending keys == ascending doubles (-0 < +0, NaN on top)
}

struct Moments { double n, mean, m2, sum_w; };     // n chain means merged so far; sum_w = sum of the within-chain M2

__device__ __forceinline__ Moments merge(const Moments& a, const Moments& b) {
  if (b.n == 0.0) return a;
  if (a.n == 0.0) return b;
  Moments r;
  r.n = a.n + b.n;
  const double d = b.mean - a.mean;
  r.mean = a.mean + d * (b.n / r.n);
  r.m2 = a.m2 + b.m2 + d * d * (a.n * b.n / r.n);
  r.sum_w = a.sum_w + b.sum_w;
  return r;
}

template <int THREADS>
__device__ __forceinline__ Moments cta_merge(Moments* sh, Moments mine) {      // fixed tree: the result does not depend on scheduling
  const int t = threadIdx.x;
  sh[t] = mine;
  __syncthreads();
  for (int w = THREADS >> 1; w > 0; w >>= 1) {
    if (t < w) sh[t] = merge(sh[t], sh[t + w]);
    __syncthreads();
  }
  return sh[0];
}

// K_m1: per chain, mean and M2 over its rows (two sequential passes over a coalesced column); the CTA's chains are merged in a
// fixed order into one record per (entry, CTA).
__global__ void __launch_bounds__(256) amwg_chain_moments_kernel(const double* __restrict__ x, long long rows, int entries, long long C,
                                                                 Moments* __restrict__ partial) {
  __shared__ Moments sh[256];
  const int e = blockIdx.y;
  const size_t stride = (size_t)entries * C;
  Moments acc{0.0, 0.0, 0.0, 0.0};
  for (long long c = (long long)blockIdx.x * blockDim.x + threadIdx.x; c < C; c += (long long)gridDim.x * blockDim.x) {
    const double* p = x + (size_t)e * C + c;
    double s = 0.0;
    long long r = 0;
    for (; r + 8 <= rows; r += 8) {                          // eight loads in flight per thread, the sum stays sequential
      double v[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) v[u] = p[(r + u) * stride];
#pragma unroll
      for (int u = 0; u < 8; ++u) s += v[u];
    }
    for (; r < rows; ++r) s += p[r * stride];
    const double m = s / (double)rows;
    double m2 = 0.0;
    r = 0;
    for (; r + 8 <= rows; r += 8) {
      double v[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) v[u] = p[(r + u) * stride];
#pragma unroll
      for (int u = 0; u < 8; ++u) { double d = v[u] - m; m2 = fma(d, d, m2); }
    }
    for (; r < rows; ++r) { double d = p[r * stride] - m; m2 = fma(d, d, m2); }
    acc = merge(acc, Moments{1.0, m, 0.0, m2});
  }
  const Moments tot = cta_merge<256>(sh, acc);
  if (threadIdx.x == 0) partial[(size_t)e * gridDim.x + blockIdx.x] = tot;
}

// K_m2: one CTA per entry merges the per-CTA records. out[entry][4] = {chains, mean of the chain means, M2 of the chain means,
// sum over chains of the within-chain M2}
__global__ void __launch_bounds__(1024) amwg_merge_moments_kernel(const Moments* __restrict__ partial, int n_partial, double* __restrict__ out) {
  __shared__ Moments sh[1024];
  const int e = blockIdx.x;
  Moments acc{0.0, 0.0, 0.0, 0.0};
  for (int i = threadIdx.x; i < n_partial; i += 1024) acc = merge(acc, partial[(size_t)e * n_partial + i]);
  const Moments tot = cta_merge<1024>(sh, acc);
  if (threadIdx.x == 0) { out[e * 4 + 0] = tot.n; out[e * 4 + 1] = tot.mean; out[e * 4 + 2] = tot.m2; out[e * 4 + 3] = tot.sum_w; }
}

// counts[entry][prefix][256] += number of values of `entry` whose key's top 8*pass bits equal prefix[entry][p] and whose next
// byte is the bin. Grid: (chain blocks, entries). Shared-memory histogram per CTA, flushed with 64-bit global atomics.
__global__ void __launch_bounds__(256) amwg_digit_hist_kernel(const double* __restrict__ x, long long rows, int entries, long long C, int pass,
                                                              const unsigned long long* __restrict__ prefix, int n_prefix,
                                                              unsigned long long* __restrict__ counts) {
  __shared__ unsigned int hist[kMaxPrefixes * 256];
  __shared__ unsigned long long pre[kMaxPrefixes];
  const int e = blockIdx.y;
  for (int i = threadIdx.x; i < n_prefix * 256; i += blockDim.x) hist[i] = 0u;
  if (threadIdx.x < n_prefix) pre[threadIdx.x] = prefix[(size_t)e * n_prefix + threadIdx.x];
  __syncthreads();
  unsigned long long pre_lo = pre[0], pre_hi = pre[0];        // most values lie outside [lowest, highest] prefix in the late passes
  for (int q = 1; q < n_prefix; ++q) { pre_lo = pre[q] < pre_lo ? pre[q] : pre_lo; pre_hi = pre[q] > pre_hi ? pre[q] : pre_hi; }
  const int shift = 56 - 8 * pass;
  const size_t stride = (size_t)entries * C;
  for (long long c = (long long)blockIdx.x * blockDim.x + threadIdx.x; c < C; c += (long long)gridDim.x * blockDim.x) {
    const double* p = x + (size_t)e * C + c;
    // consecutive rows of one chain mostly fall in the same bin (always, in the leading passes of a narrow posterior): count the
    // run in a register and touch the shared histogram once per run instead of once per value
    int last = -1;
    unsigned int run = 0;
    auto count = [&](double x) {
      const unsigned long long k = ordered_key(x);
      int idx = (int)((k >> shift) & 255ull);
      if (pass) {
        const unsigned long long hi = k >> (shift + 8);
        int q = n_prefix;
        if (hi >= pre_lo && hi <= pre_hi) { q = 0; while (q < n_prefix && pre[q] != hi) ++q; }   // the first match counts (padding repeats a prefix)
        idx = (q < n_prefix) ? q * 256 + idx : -1;
      }
      if (idx == last) { ++run; return; }
      if (last >= 0) atomicAdd(&hist[last], run);
      last = idx; run = 1;
    };
    long long r = 0;
    for (; r + 8 <= rows; r += 8) {                          // eight loads in flight per thread
      double v[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) v[u] = p[(r + u) * stride];
#pragma unroll
      for (int u = 0; u < 8; ++u) count(v[u]);
    }
    for (; r < rows; ++r) count(p[r * stride]);
    if (last >= 0) atomicAdd(&hist[last], run);
  }
  __syncthreads();
  for (int i = threadIdx.x; i < n_prefix * 256; i += blockDim.x)
    if (hist[i]) atomicAdd(&counts[(size_t)e * n_prefix * 256 + i], (unsigned long long)hist[i]);
}

template <int THREADS>
__device__ __forceinline__ double cta_sum(double* sh, double mine) {            // fixed tree, like cta_merge
  const int t = threadIdx.x;
  sh[t] = mine;
  __syncthreads();
  for (int w = THREADS >> 1; w > 0; w >>= 1) {
    if (t < w) sh[t] += sh[t + w];
    __syncthreads();
  }
  const double r = sh[0];
  __syncthreads();                                                               // sh is reused by the next call
  return r;
}

// K_a1: split-chain autocovariance sums for the lags [lag0, lag0 + L) of the live entries (grid: chain blocks x live entries).
// Per chain, h = rows / 2; the half-chains are rows [0, h) and [rows - h, rows) (the middle row of an odd `rows` is dropped).
// y = x, or y = (x <= thr[entry]) in indicator mode; c_n = y_n - (mean of y over the half). Per half:
//   S_t += sum_{n=0}^{h-1-t} c_n c_{n+t}.
// The window holds c_{n+lag0+j} at slot (n + j) % L; with the n-loop unrolled by L every slot index is static. Values past the
// half's end read as 0, so for a given lag t the sequence of nonzero additions (n ascending, chains in grid-stride order) does
// not depend on lag0 or L: a lag's sum is the same bits whichever tile holds it, and lags >= h sum to exactly 0.
template <int L, bool INDICATOR>
__global__ void __launch_bounds__(256, 2) amwg_split_autocov_kernel(const double* __restrict__ x, long long rows, int entries, long long C,
                                                                 const int* __restrict__ live, const double* __restrict__ thr, int lag0,
                                                                 Moments* __restrict__ part_m, double* __restrict__ part_s) {
  __shared__ Moments sh[256];
  __shared__ double shs[256];
  const int e = live[blockIdx.y];
  const double th = INDICATOR ? thr[e] : 0.0;
  const int h = (int)(rows / 2);                           // rows < 2^31 (checked by the caller): 32-bit row counters
  const size_t stride = (size_t)entries * C;
  double acc[L];
#pragma unroll
  for (int j = 0; j < L; ++j) acc[j] = 0.0;
  Moments mm{0.0, 0.0, 0.0, 0.0};
  for (long long c = (long long)blockIdx.x * blockDim.x + threadIdx.x; c < C; c += (long long)gridDim.x * blockDim.x) {
#pragma unroll 1
    for (int half = 0; half < 2; ++half) {
      const double* p = x + (size_t)e * C + c + (half ? (size_t)(rows - h) * stride : 0);
      auto y = [&](int r) -> double { const double v = p[r * stride]; return INDICATOR ? (v <= th ? 1.0 : 0.0) : v; };
      double s = 0.0;
      int r = 0;
      for (; r + 8 <= h; r += 8) {                           // eight loads in flight per thread, the sum stays sequential
        double v[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) v[u] = y(r + u);
#pragma unroll
        for (int u = 0; u < 8; ++u) s += v[u];
      }
      for (; r < h; ++r) s += y(r);
      const double m = s / (double)h;
      mm = merge(mm, Moments{1.0, m, 0.0, 0.0});
      if (lag0 >= h) continue;                               // every product of the tile is past the end: the sums stay 0
      const double c1 = 1.0 - m, c0 = 0.0 - m;             // an indicator's two centred values, the same bits as y - m
      auto cen = [&](const double* q, int r) -> double {
        if (r >= h) return 0.0;
        const double v = *q;
        return INDICATOR ? (v <= th ? c1 : c0) : v - m;
      };
      double w[L];
#pragma unroll
      for (int j = 0; j < L; ++j) w[j] = cen(p + (size_t)(lag0 + j) * stride, lag0 + j);
      const double* pn = p;                                  // row n, and row n + lag0 + L (the value entering the window)
      const double* pw = p + (size_t)(lag0 + L) * stride;
      for (int n = 0; n < h - lag0; n += L) {
#pragma unroll
        for (int u = 0; u < L; ++u) {
          const double cn = cen(pn, n + u);
#pragma unroll
          for (int j = 0; j < L; ++j) acc[j] = fma(cn, w[(u + j) % L], acc[j]);
          w[u] = cen(pw, n + u + lag0 + L);
          pn += stride;
          pw += stride;
        }
      }
    }
  }
  const Moments tot = cta_merge<256>(sh, mm);
  const size_t slot = (size_t)blockIdx.y * gridDim.x + blockIdx.x;
  if (threadIdx.x == 0) part_m[slot] = tot;
#pragma unroll
  for (int j = 0; j < L; ++j) {
    const double v = cta_sum<256>(shs, acc[j]);
    if (threadIdx.x == 0) part_s[slot * L + j] = v;
  }
}

// K_a2: one CTA per live entry. out[live][3 + n_out] = {half-chains, mean of the half-chain means, M2 of the half-chain means,
// S_lag0 .. S_{lag0+n_out-1}}
template <int L>
__global__ void __launch_bounds__(256) amwg_merge_autocov_kernel(const Moments* __restrict__ part_m, const double* __restrict__ part_s,
                                                                 int n_partial, int n_out, double* __restrict__ out) {
  __shared__ Moments sh[256];
  __shared__ double shs[256];
  const size_t e = blockIdx.x;
  Moments acc{0.0, 0.0, 0.0, 0.0};
  for (int i = threadIdx.x; i < n_partial; i += 256) acc = merge(acc, part_m[e * n_partial + i]);
  const Moments tot = cta_merge<256>(sh, acc);
  double* o = out + e * (3 + n_out);
  if (threadIdx.x == 0) { o[0] = tot.n; o[1] = tot.mean; o[2] = tot.m2; }
  for (int j = 0; j < n_out; ++j) {
    double s = 0.0;
    for (int i = threadIdx.x; i < n_partial; i += 256) s += part_s[(e * n_partial + i) * L + j];
    const double v = cta_sum<256>(shs, s);
    if (threadIdx.x == 0) o[3 + j] = v;
  }
}

}  // namespace summary

extern "C" int amwg_summary_moments(int device, const double* dev_samples, int64_t rows, int32_t entries, int64_t chains, double* host_stats) {
  if (rows <= 0 || entries <= 0 || chains <= 0) return fail("amwg_summary_moments: empty sample block");
  if (!dev_samples || !host_stats) return fail("amwg_summary_moments: null pointer");
  CUDA_TRY(cudaSetDevice(device));
  const unsigned bx = (unsigned)std::min<int64_t>((chains + 255) / 256, 148 * 8);     // depends on `chains` only: a fixed merge order
  // scratch that lives as long as the process (per device, grown on demand): no cudaMalloc / cudaFree on the path of a call
  struct Scratch { void* p = nullptr; size_t bytes = 0; };
  static Scratch scratch[64];
  static std::mutex scratch_mu;
  const size_t need_partial = (size_t)entries * bx * sizeof(summary::Moments), need_out = (size_t)entries * 4 * sizeof(double);
  const size_t need = ((need_partial + 255) / 256) * 256 + need_out;
  summary::Moments* partial = nullptr;
  double* d_out = nullptr;
  {
    std::lock_guard<std::mutex> lock(scratch_mu);
    if (device < 0 || device >= 64) return fail("amwg_summary_moments: device index out of range");
    Scratch& sc = scratch[device];
    if (sc.bytes < need) {
      if (sc.p) cudaFree(sc.p);
      sc.p = nullptr; sc.bytes = 0;
      CUDA_TRY(cudaMalloc(&sc.p, need));
      sc.bytes = need;
    }
    partial = reinterpret_cast<summary::Moments*>(sc.p);
    d_out = reinterpret_cast<double*>(reinterpret_cast<char*>(sc.p) + ((need_partial + 255) / 256) * 256);
  }
  summary::amwg_chain_moments_kernel<<<dim3(bx, (unsigned)entries), 256>>>(dev_samples, rows, entries, chains, partial);
  summary::amwg_merge_moments_kernel<<<(unsigned)entries, 1024>>>(partial, (int)bx, d_out);
  cudaError_t e = cudaGetLastError();
  if (e == cudaSuccess) e = cudaMemcpy(host_stats, d_out, need_out, cudaMemcpyDeviceToHost);
  if (e != cudaSuccess) return fail(std::string("amwg_summary_moments: ") + cudaGetErrorString(e));
  return 0;
}

extern "C" int amwg_summary_digit_hist(int device, const double* dev_samples, int64_t rows, int32_t entries, int64_t chains, int32_t pass,
                                       const uint64_t* dev_prefix, int32_t n_prefix, uint64_t* dev_counts) {
  if (rows <= 0 || entries <= 0 || chains <= 0) return fail("amwg_summary_digit_hist: empty sample block");
  if (pass < 0 || pass > 7) return fail("amwg_summary_digit_hist: pass must be 0..7");
  if (n_prefix < 1 || n_prefix > summary::kMaxPrefixes) return fail("amwg_summary_digit_hist: n_prefix must be 1.." + std::to_string(summary::kMaxPrefixes));
  if (rows >= (int64_t)1 << 32) return fail("amwg_summary_digit_hist: more than 2^32 rows");
  if (!dev_samples || !dev_prefix || !dev_counts) return fail("amwg_summary_digit_hist: null pointer");
  CUDA_TRY(cudaSetDevice(device));
  // a CTA's shared bins are 32-bit: bound the values one CTA sees by 2^32 (rows < 2^32 and the grid below keeps chains per CTA small)
  int64_t bx = std::min<int64_t>((chains + 255) / 256, 148 * 8);
  while (bx < (chains + 255) / 256 && ((chains + bx - 1) / bx) * rows >= ((int64_t)1 << 32)) bx *= 2;
  summary::amwg_digit_hist_kernel<<<dim3((unsigned)bx, (unsigned)entries), 256>>>(dev_samples, rows, entries, chains, pass,
                                                                                  reinterpret_cast<const unsigned long long*>(dev_prefix), n_prefix,
                                                                                  reinterpret_cast<unsigned long long*>(dev_counts));
  CUDA_TRY(cudaGetLastError());
  CUDA_TRY(cudaDeviceSynchronize());
  return 0;
}

extern "C" int amwg_summary_autocov(int device, const double* dev_samples, int64_t rows, int32_t entries, int64_t chains,
                                    const double* dev_threshold, const int32_t* host_live, int32_t n_live, int32_t lag0, int32_t n_lags,
                                    double* host_out) {
  if (entries <= 0 || chains <= 0) return fail("amwg_summary_autocov: empty sample block");
  if (rows < 8) return fail("amwg_summary_autocov: rows must be >= 8 (split chains of at least 4 draws)");
  if (rows >= ((int64_t)1 << 31) - 64) return fail("amwg_summary_autocov: rows must be < 2^31 - 64");
  if (lag0 < 0) return fail("amwg_summary_autocov: lag0 must be >= 0");
  if (n_lags < 1 || n_lags > summary::kLagTile) return fail("amwg_summary_autocov: n_lags must be 1.." + std::to_string(summary::kLagTile));
  if (!dev_samples || !host_out) return fail("amwg_summary_autocov: null pointer");
  if (host_live && (n_live < 1 || n_live > entries)) return fail("amwg_summary_autocov: n_live must be 1..entries");
  const int32_t live_n = host_live ? n_live : entries;
  std::vector<int32_t> live((size_t)live_n);
  for (int32_t i = 0; i < live_n; ++i) {
    live[i] = host_live ? host_live[i] : i;
    if (live[i] < 0 || live[i] >= entries) return fail("amwg_summary_autocov: live entry index out of range");
  }
  if (device < 0 || device >= 64) return fail("amwg_summary_autocov: device index out of range");
  CUDA_TRY(cudaSetDevice(device));
  constexpr int L = summary::kLagTile;
  const unsigned bx = (unsigned)std::min<int64_t>((chains + 255) / 256, 148 * 8);     // depends on `chains` only: a fixed merge order
  auto up = [](size_t b) { return ((b + 255) / 256) * 256; };
  const size_t need_m = up((size_t)live_n * bx * sizeof(summary::Moments)), need_s = up((size_t)live_n * bx * L * sizeof(double));
  const size_t need_out = (size_t)live_n * (3 + n_lags) * sizeof(double);
  const size_t need = need_m + need_s + up(need_out) + (size_t)live_n * sizeof(int32_t);
  struct Scratch { void* p = nullptr; size_t bytes = 0; };                             // per device, grown on demand (as above)
  static Scratch scratch[64];
  static std::mutex scratch_mu;
  std::lock_guard<std::mutex> lock(scratch_mu);                                        // held across the call: the scratch is shared
  Scratch& sc = scratch[device];
  if (sc.bytes < need) {
    if (sc.p) cudaFree(sc.p);
    sc.p = nullptr; sc.bytes = 0;
    CUDA_TRY(cudaMalloc(&sc.p, need));
    sc.bytes = need;
  }
  char* base = reinterpret_cast<char*>(sc.p);
  auto* part_m = reinterpret_cast<summary::Moments*>(base);
  auto* part_s = reinterpret_cast<double*>(base + need_m);
  auto* d_out = reinterpret_cast<double*>(base + need_m + need_s);
  auto* d_live = reinterpret_cast<int*>(base + need_m + need_s + up(need_out));
  CUDA_TRY(cudaMemcpy(d_live, live.data(), (size_t)live_n * sizeof(int32_t), cudaMemcpyHostToDevice));
  const dim3 grid(bx, (unsigned)live_n);
  if (dev_threshold)
    summary::amwg_split_autocov_kernel<L, true><<<grid, 256>>>(dev_samples, rows, entries, chains, d_live, dev_threshold, lag0, part_m, part_s);
  else
    summary::amwg_split_autocov_kernel<L, false><<<grid, 256>>>(dev_samples, rows, entries, chains, d_live, nullptr, lag0, part_m, part_s);
  summary::amwg_merge_autocov_kernel<L><<<(unsigned)live_n, 256>>>(part_m, part_s, (int)bx, n_lags, d_out);
  cudaError_t e = cudaGetLastError();
  if (e == cudaSuccess) e = cudaMemcpy(host_out, d_out, need_out, cudaMemcpyDeviceToHost);
  if (e != cudaSuccess) return fail(std::string("amwg_summary_autocov: ") + cudaGetErrorString(e));
  return 0;
}
