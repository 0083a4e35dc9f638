// Rank normalisation on device for sample_summary(rank=True): the exact pooled average rank of every split draw of one entry,
// and z = Phi^-1((r - 3/8) / (S + 1/4)) scattered into a z block in the sample block's layout.
//
//   K_r0  amwg_rank_keys_kernel     : the split draws of one entry (first and last h rows of each chain, optionally folded about a
//                                     centre) -> order-preserving 64-bit keys (-0 canonicalised to +0) and 32-bit positions r'*C + c
//   K_r1  amwg_rank_hist8_kernel    : one read of the keys -> all eight 8-bit digit histograms (warp-aggregated shared atomics);
//                                     the host skips every pass whose digit is the same for all keys
//   K_r2  amwg_rank_count_kernel    : per pass, the digit counts of every 4096-key tile, digit-major [256][tiles]
//   K_r3  exclusive scan            : (generic, three phases per level) the tile counts -> each tile's first slot per digit
//   K_r4  amwg_rank_scatter_pass_kernel : per pass, a stable scatter: each warp ranks its 512 keys row by row with __match_any_sync
//                                     and per-warp digit counters in shared memory; the warps of a tile are ordered by a per-digit
//                                     scan, the tiles by K_r3. LSD over the non-skipped digits, double-buffered (key, payload)
//   K_r5  amwg_rank_flags/heads/ends: run-length encoding of the sorted keys: run index per position (scan of the head flags), the
//                                     run's key and its count (or summed weight) from the positions of its head and its end
//   K_r6  amwg_rank_z_kernel        : z per run from the draws below it (a scan of the counts, plus the rank offset of this GPU's
//                                     key range) and its own count: average rank below + (count + 1) / 2
//   K_r7  amwg_rank_scatter_kernel  : z[run of sorted position i] -> out at the payload of i. One thread per draw: linear in the
//                                     number of draws whatever the tie multiplicity (no thread walks a run)
// Included at the end of amwg_kernels.cu after amwg_summary.cuh (shares ordered_key, CUDA_TRY / fail()).
#pragma once

namespace rank {

constexpr int kThreads = 256;
constexpr int kWarps = kThreads / 32;
constexpr int kItems = 16;                          // keys per thread and pass: 16 keys, payloads and ranks stay in registers
constexpr int kTile = kThreads * kItems;            // 4096 keys per CTA tile of a sort pass
constexpr int kScanItems = 8;
constexpr int kScanTile = kThreads * kScanItems;    // 2048 values per CTA of a scan level

__device__ __forceinline__ unsigned long long rank_key(double x) {
  return summary::ordered_key(x == 0.0 ? 0.0 : x);   // -0 and +0 tie
}

__device__ __forceinline__ unsigned lanemask_lt() {
  unsigned m;
  asm("mov.u32 %0, %%lanemask_lt;" : "=r"(m));
  return m;
}

// K_r0. Grid: (chain blocks, row blocks); rows r' of the split block: [0, h) are rows [0, h), [h, 2h) are rows [rows - h, rows).
__global__ void __launch_bounds__(kThreads) amwg_rank_keys_kernel(const double* __restrict__ x, long long rows, int entries, long long C,
                                                                   int e, int fold, double center, unsigned long long* __restrict__ keys,
                                                                   unsigned int* __restrict__ vals) {
  const long long h = rows / 2;
  for (long long rp = blockIdx.y; rp < 2 * h; rp += gridDim.y) {
    const long long r = rp < h ? rp : rp + (rows - 2 * h);
    const double* p = x + ((size_t)r * entries + e) * C;
    for (long long c = (long long)blockIdx.x * blockDim.x + threadIdx.x; c < C; c += (long long)gridDim.x * blockDim.x) {
      double v = p[c];
      if (fold) v = fabs(v - center);
      const size_t i = (size_t)rp * C + c;
      keys[i] = rank_key(v);
      vals[i] = (unsigned int)i;
    }
  }
}

// K_r1: hist[d][256] += counts of byte d (0 = least significant) over all keys.
__global__ void __launch_bounds__(kThreads) amwg_rank_hist8_kernel(const unsigned long long* __restrict__ keys, long long n,
                                                                    unsigned long long* __restrict__ hist) {
  __shared__ unsigned int sh[8 * 256];
  for (int i = threadIdx.x; i < 8 * 256; i += kThreads) sh[i] = 0u;
  __syncthreads();
  const long long step = (long long)gridDim.x * kThreads;
  for (long long base = (long long)blockIdx.x * kThreads; base < n; base += step) {   // uniform trip count per warp
    const long long i = base + threadIdx.x;
    const bool on = i < n;
    const unsigned long long k = on ? keys[i] : 0ull;
#pragma unroll
    for (int d = 0; d < 8; ++d) {
      const unsigned bin = on ? (unsigned)((k >> (8 * d)) & 255ull) : 256u;
      const unsigned peers = __match_any_sync(0xffffffffu, bin);       // posterior keys share their top bytes: one atomic per bin
      if (on && (peers & lanemask_lt()) == 0) atomicAdd(&sh[d * 256 + bin], (unsigned)__popc(peers));
    }
  }
  __syncthreads();
  for (int i = threadIdx.x; i < 8 * 256; i += kThreads)
    if (sh[i]) atomicAdd(&hist[i], (unsigned long long)sh[i]);
}

// K_r2: counts[d * n_tiles + tile] = keys of the tile whose digit (at `shift`) is d.
__global__ void __launch_bounds__(kThreads) amwg_rank_count_kernel(const unsigned long long* __restrict__ keys, long long n, int shift,
                                                                    unsigned int* __restrict__ counts, long long n_tiles) {
  __shared__ unsigned int sh[256];
  sh[threadIdx.x] = 0u;
  __syncthreads();
  const long long tile = blockIdx.x;
  const long long base = tile * kTile;
#pragma unroll 4
  for (int j = 0; j < kItems; ++j) {
    const long long i = base + (long long)j * kThreads + threadIdx.x;
    const bool on = i < n;
    const unsigned bin = on ? (unsigned)((keys[i] >> shift) & 255ull) : 256u;
    const unsigned peers = __match_any_sync(0xffffffffu, bin);
    if (on && (peers & lanemask_lt()) == 0) atomicAdd(&sh[bin], (unsigned)__popc(peers));
  }
  __syncthreads();
  counts[(size_t)threadIdx.x * n_tiles + tile] = sh[threadIdx.x];
}

// K_r4: one stable pass. Warp w of tile t owns positions [t*kTile + w*32*kItems, +32*kItems), read row by row (row j: 32
// consecutive keys). A key's slot = first slot of its digit in the tile (K_r3) + keys of that digit in earlier warps + keys of
// that digit earlier in its own warp (earlier rows, then lower lanes of its row): position order is kept.
__global__ void __launch_bounds__(kThreads) amwg_rank_scatter_pass_kernel(const unsigned long long* __restrict__ kin, const unsigned int* __restrict__ vin,
                                                                           unsigned long long* __restrict__ kout, unsigned int* __restrict__ vout,
                                                                           long long n, int shift, const unsigned int* __restrict__ offsets,
                                                                           long long n_tiles) {
  __shared__ unsigned int cnt[kWarps][256];
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const long long tile = blockIdx.x;
#pragma unroll
  for (int q = 0; q < kWarps; ++q) cnt[q][threadIdx.x] = 0u;
  __syncthreads();
  const long long start = tile * kTile + (long long)w * 32 * kItems;
  const unsigned lt = lanemask_lt();
  unsigned long long k[kItems];
  unsigned int v[kItems], rk[kItems];
#pragma unroll
  for (int j = 0; j < kItems; ++j) {
    const long long i = start + (long long)j * 32 + lane;
    const bool on = i < n;
    k[j] = on ? kin[i] : 0ull;
    v[j] = on ? vin[i] : 0u;
  }
#pragma unroll
  for (int j = 0; j < kItems; ++j) {
    const bool on = start + (long long)j * 32 + lane < n;
    const unsigned d = on ? (unsigned)((k[j] >> shift) & 255ull) : 256u;
    const unsigned peers = __match_any_sync(0xffffffffu, d);
    rk[j] = (on ? cnt[w][d] : 0u) + (unsigned)__popc(peers & lt);
    __syncwarp();
    if (on && (peers & lt) == 0) cnt[w][d] += (unsigned)__popc(peers);
    __syncwarp();
  }
  __syncthreads();
  {                                                            // per digit: exclusive over the warps, from the tile's first slot
    const int d = threadIdx.x;
    unsigned s = offsets[(size_t)d * n_tiles + tile];
#pragma unroll
    for (int q = 0; q < kWarps; ++q) { const unsigned c = cnt[q][d]; cnt[q][d] = s; s += c; }
  }
  __syncthreads();
#pragma unroll
  for (int j = 0; j < kItems; ++j) {
    if (start + (long long)j * 32 + lane < n) {
      const unsigned d = (unsigned)((k[j] >> shift) & 255ull);
      const unsigned pos = cnt[w][d] + rk[j];
      kout[pos] = k[j];
      vout[pos] = v[j];
    }
  }
}

// ---- exclusive scan (in place allowed): per level, tile sums -> scan of the sums (recursively) -> tiles scanned from their sum
template <typename T>
__device__ __forceinline__ T block_exclusive(T mine, T* sh_warp, T* total) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  T inc = mine;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const T y = __shfl_up_sync(0xffffffffu, inc, o);
    if (lane >= o) inc += y;
  }
  if (lane == 31) sh_warp[w] = inc;
  __syncthreads();
  T before = 0, all = 0;
#pragma unroll
  for (int q = 0; q < kWarps; ++q) { if (q < w) before += sh_warp[q]; all += sh_warp[q]; }
  __syncthreads();
  *total = all;
  return before + inc - mine;
}

template <typename T>
__global__ void __launch_bounds__(kThreads) amwg_scan_reduce_kernel(const T* __restrict__ in, long long n, T* __restrict__ sums) {
  __shared__ T sh[kWarps];
  const long long base = (long long)blockIdx.x * kScanTile + (long long)threadIdx.x * kScanItems;
  T s = 0;
#pragma unroll
  for (int u = 0; u < kScanItems; ++u) if (base + u < n) s += in[base + u];
  T total;
  block_exclusive<T>(s, sh, &total);
  if (threadIdx.x == 0) sums[blockIdx.x] = total;
}

template <typename T>
__global__ void __launch_bounds__(kThreads) amwg_scan_down_kernel(T* data, long long n, const T* __restrict__ tile_off) {
  __shared__ T sh[kWarps];
  const long long base = (long long)blockIdx.x * kScanTile + (long long)threadIdx.x * kScanItems;
  T v[kScanItems];
  T s = 0;
#pragma unroll
  for (int u = 0; u < kScanItems; ++u) { v[u] = base + u < n ? data[base + u] : (T)0; s += v[u]; }
  T total;
  T run = block_exclusive<T>(s, sh, &total) + (tile_off ? tile_off[blockIdx.x] : (T)0);
#pragma unroll
  for (int u = 0; u < kScanItems; ++u) if (base + u < n) { const T c = v[u]; data[base + u] = run; run += c; }
}

// ---- run-length encoding of sorted keys
__device__ __forceinline__ bool is_head(const unsigned long long* k, long long i) { return i == 0 || k[i] != k[i - 1]; }
__device__ __forceinline__ bool is_end(const unsigned long long* k, long long i, long long n) { return i == n - 1 || k[i + 1] != k[i]; }

__global__ void __launch_bounds__(kThreads) amwg_rank_flags_kernel(const unsigned long long* __restrict__ keys, long long n, unsigned int* __restrict__ flag) {
  for (long long i = (long long)blockIdx.x * kThreads + threadIdx.x; i < n; i += (long long)gridDim.x * kThreads)
    flag[i] = (i > 0 && keys[i] != keys[i - 1]) ? 1u : 0u;
}

// w_excl[i] = weights[vals[i]] (scanned afterwards): the summed weight before each sorted position
__global__ void __launch_bounds__(kThreads) amwg_rank_weights_kernel(const unsigned int* __restrict__ vals, const long long* __restrict__ weights,
                                                                      long long n, long long* __restrict__ w) {
  for (long long i = (long long)blockIdx.x * kThreads + threadIdx.x; i < n; i += (long long)gridDim.x * kThreads) w[i] = weights[vals[i]];
}

// run_id (exclusive scan of the flags) += own flag -> the run index; at a head: the run's key and the weight before it
__global__ void __launch_bounds__(kThreads) amwg_rank_heads_kernel(const unsigned long long* __restrict__ keys, long long n, unsigned int* __restrict__ run_id,
                                                                    const long long* __restrict__ w_excl, unsigned long long* __restrict__ run_keys,
                                                                    long long* __restrict__ run_counts) {
  for (long long i = (long long)blockIdx.x * kThreads + threadIdx.x; i < n; i += (long long)gridDim.x * kThreads) {
    const bool head = is_head(keys, i);
    const unsigned r = run_id[i] + ((head && i > 0) ? 1u : 0u);
    run_id[i] = r;
    if (head) {
      if (run_keys) run_keys[r] = keys[i];
      run_counts[r] = w_excl ? w_excl[i] : i;
    }
  }
}

// at a run's end: count = weight up to and including it - weight before the head (one thread per run touches run_counts[r])
__global__ void __launch_bounds__(kThreads) amwg_rank_ends_kernel(const unsigned long long* __restrict__ keys, long long n, const unsigned int* __restrict__ run_id,
                                                                   const long long* __restrict__ w_excl, const unsigned int* __restrict__ vals,
                                                                   const long long* __restrict__ weights, long long* __restrict__ run_counts) {
  for (long long i = (long long)blockIdx.x * kThreads + threadIdx.x; i < n; i += (long long)gridDim.x * kThreads) {
    if (!is_end(keys, i, n)) continue;
    const unsigned r = run_id[i];
    const long long incl = w_excl ? w_excl[i] + weights[vals[i]] : i + 1;
    run_counts[r] = incl - run_counts[r];
  }
}

// K_r6: below = exclusive scan of the counts; average rank (1-based) = offset + below + (count + 1) / 2, exact in doubles below 2^50.
// `below` is the z array itself (the scan runs in the output): each thread reads its slot, then overwrites it.
__global__ void __launch_bounds__(kThreads) amwg_rank_z_kernel(const long long* below, const long long* __restrict__ counts, long long n_runs,
                                                                long long offset, double total, double* z) {
  for (long long i = (long long)blockIdx.x * kThreads + threadIdx.x; i < n_runs; i += (long long)gridDim.x * kThreads) {
    const double r = (double)(offset + below[i]) + 0.5 * (double)(counts[i] + 1);
    z[i] = normcdfinv((r - 0.375) / (total + 0.25));
  }
}

// K_r7: out[(p / C * entries + e) * C + p % C] = run_z[run_id[i]], p = vals[i]
__global__ void __launch_bounds__(kThreads) amwg_rank_scatter_kernel(const unsigned int* __restrict__ vals, const unsigned int* __restrict__ run_id, long long n,
                                                                      const double* __restrict__ run_z, double* __restrict__ out, int entries,
                                                                      long long C, int e) {
  for (long long i = (long long)blockIdx.x * kThreads + threadIdx.x; i < n; i += (long long)gridDim.x * kThreads) {
    const unsigned long long p = vals[i];
    const unsigned long long rp = p / (unsigned long long)C, c = p - rp * (unsigned long long)C;
    out[(rp * (unsigned long long)entries + (unsigned long long)e) * (unsigned long long)C + c] = run_z[run_id[i]];
  }
}

// ---- host helpers
struct Scratch { void* p = nullptr; size_t bytes = 0; };

// per-device scratch, grown on demand; the caller holds scratch_mu (through a Lease). Up to kKeepBytes stays allocated between calls
// (no cudaMalloc on the path of a call for the scan partials and small sorts); a larger one (the tile counts of a big sort, n / 4
// bytes) is freed when the call ends, so no O(draws) memory outlives the call.
static std::mutex scratch_mu;
static Scratch scratch[64];
constexpr size_t kKeepBytes = (size_t)64 << 20;

struct Lease {
  std::lock_guard<std::mutex> lock{scratch_mu};
  int device;
  explicit Lease(int d) : device(d) {}
  ~Lease() {
    Scratch& sc = scratch[device];
    if (sc.bytes > kKeepBytes) { cudaDeviceSynchronize(); cudaFree(sc.p); sc.p = nullptr; sc.bytes = 0; }
  }
};

static cudaError_t scratch_get(int device, size_t need, void** out) {
  Scratch& sc = scratch[device];
  if (sc.bytes < need) {
    if (sc.p) cudaFree(sc.p);
    sc.p = nullptr; sc.bytes = 0;
    const cudaError_t e = cudaMalloc(&sc.p, need);
    if (e != cudaSuccess) return e;
    sc.bytes = need;
  }
  *out = sc.p;
  return cudaSuccess;
}

static size_t up256(size_t b) { return ((b + 255) / 256) * 256; }

template <typename T>
static size_t scan_scratch_bytes(long long n) {              // the tile sums of every level
  size_t b = 0;
  while (n > kScanTile) { n = (n + kScanTile - 1) / kScanTile; b += up256((size_t)n * sizeof(T)); }
  return b;
}

template <typename T>
static void exclusive_scan(T* data, long long n, char* tmp) {
  if (n <= kScanTile) { amwg_scan_down_kernel<T><<<1, kThreads>>>(data, n, nullptr); return; }
  const long long tiles = (n + kScanTile - 1) / kScanTile;
  T* sums = reinterpret_cast<T*>(tmp);
  amwg_scan_reduce_kernel<T><<<(unsigned)tiles, kThreads>>>(data, n, sums);
  exclusive_scan<T>(sums, tiles, tmp + up256((size_t)tiles * sizeof(T)));
  amwg_scan_down_kernel<T><<<(unsigned)tiles, kThreads>>>(data, n, sums);
}

static unsigned grid_for(long long n) { return (unsigned)std::max<long long>(1, std::min<long long>((n + kThreads - 1) / kThreads, 148 * 16)); }

}  // namespace rank

static int rank_device_check(const char* fn, int device) {
  if (device < 0 || device >= 64) return fail(std::string(fn) + ": device index out of range");
  return 0;
}

extern "C" int amwg_summary_rank_keys(int device, const double* dev_samples, int64_t rows, int32_t entries, int64_t chains, int32_t entry,
                                      const double* host_center, uint64_t* dev_keys, uint32_t* dev_vals) {
  if (rows <= 0 || entries <= 0 || chains <= 0) return fail("amwg_summary_rank_keys: empty sample block");
  if (rows < 2) return fail("amwg_summary_rank_keys: rows must be >= 2 (split chains of at least one draw)");
  if (entry < 0 || entry >= entries) return fail("amwg_summary_rank_keys: entry out of range");
  if ((rows / 2) * 2 > (((int64_t)1 << 32) - 1) / chains) return fail("amwg_summary_rank_keys: 2^32 or more split draws of one entry");
  if (!dev_samples || !dev_keys || !dev_vals) return fail("amwg_summary_rank_keys: null pointer");
  if (rank_device_check("amwg_summary_rank_keys", device)) return -1;
  CUDA_TRY(cudaSetDevice(device));
  const int64_t h2 = (rows / 2) * 2;
  const dim3 grid((unsigned)std::min<int64_t>((chains + 255) / 256, 148 * 8), (unsigned)std::min<int64_t>(h2, 65535));
  rank::amwg_rank_keys_kernel<<<grid, rank::kThreads>>>(dev_samples, rows, entries, chains, entry, host_center ? 1 : 0,
                                                        host_center ? *host_center : 0.0, reinterpret_cast<unsigned long long*>(dev_keys), dev_vals);
  CUDA_TRY(cudaGetLastError());
  CUDA_TRY(cudaDeviceSynchronize());
  return 0;
}

extern "C" int amwg_summary_rank_sort(int device, uint64_t* dev_keys, uint32_t* dev_vals, int64_t n, uint64_t* dev_keys_alt, uint32_t* dev_vals_alt,
                                      int32_t* host_passes) {
  if (n < 1) return fail("amwg_summary_rank_sort: n must be >= 1");
  if (n >= ((int64_t)1 << 32)) return fail("amwg_summary_rank_sort: 2^32 or more keys");
  if (!dev_keys || !dev_vals || !dev_keys_alt || !dev_vals_alt || !host_passes) return fail("amwg_summary_rank_sort: null pointer");
  if (rank_device_check("amwg_summary_rank_sort", device)) return -1;
  CUDA_TRY(cudaSetDevice(device));
  using u64 = unsigned long long;
  const long long n_tiles = (n + rank::kTile - 1) / rank::kTile;
  const size_t need_hist = rank::up256(8 * 256 * sizeof(u64)), need_cnt = rank::up256((size_t)256 * n_tiles * sizeof(unsigned));
  const size_t need = need_hist + need_cnt + rank::scan_scratch_bytes<unsigned>(256 * n_tiles);
  rank::Lease lease(device);
  void* sp = nullptr;
  CUDA_TRY(rank::scratch_get(device, need, &sp));
  char* base = reinterpret_cast<char*>(sp);
  u64* d_hist = reinterpret_cast<u64*>(base);
  unsigned* d_cnt = reinterpret_cast<unsigned*>(base + need_hist);
  char* d_tmp = base + need_hist + need_cnt;
  CUDA_TRY(cudaMemset(d_hist, 0, 8 * 256 * sizeof(u64)));
  rank::amwg_rank_hist8_kernel<<<rank::grid_for(n), rank::kThreads>>>(reinterpret_cast<const u64*>(dev_keys), n, d_hist);
  CUDA_TRY(cudaGetLastError());
  u64 hist[8 * 256];
  CUDA_TRY(cudaMemcpy(hist, d_hist, sizeof hist, cudaMemcpyDeviceToHost));
  u64 *k0 = reinterpret_cast<u64*>(dev_keys), *k1 = reinterpret_cast<u64*>(dev_keys_alt);
  unsigned *v0 = dev_vals, *v1 = dev_vals_alt;
  int run = 0, skipped = 0;
  for (int d = 0; d < 8; ++d) {
    bool one = false;
    for (int b = 0; b < 256; ++b) if (hist[d * 256 + b] == (u64)n) { one = true; break; }
    if (one) { ++skipped; continue; }                       // every key has the same byte d: the pass would not move a key
    const int shift = 8 * d;
    rank::amwg_rank_count_kernel<<<(unsigned)n_tiles, rank::kThreads>>>(k0, n, shift, d_cnt, n_tiles);
    rank::exclusive_scan<unsigned>(d_cnt, 256 * n_tiles, d_tmp);
    rank::amwg_rank_scatter_pass_kernel<<<(unsigned)n_tiles, rank::kThreads>>>(k0, v0, k1, v1, n, shift, d_cnt, n_tiles);
    std::swap(k0, k1);
    std::swap(v0, v1);
    ++run;
  }
  CUDA_TRY(cudaGetLastError());
  CUDA_TRY(cudaDeviceSynchronize());
  host_passes[0] = run;
  host_passes[1] = skipped;
  host_passes[2] = run & 1;                                   // 1: the sorted pairs are in the _alt buffers
  return 0;
}

extern "C" int amwg_summary_rank_runs(int device, const uint64_t* dev_sorted_keys, const uint32_t* dev_sorted_vals, const int64_t* dev_weights,
                                      int64_t* dev_weight_scan, int64_t n, uint32_t* dev_run_id, uint64_t* dev_run_keys, int64_t* dev_run_counts,
                                      int64_t* host_n_runs) {
  if (n < 1) return fail("amwg_summary_rank_runs: n must be >= 1");
  if (n >= ((int64_t)1 << 32)) return fail("amwg_summary_rank_runs: 2^32 or more keys");
  if (!dev_sorted_keys || !dev_run_id || !dev_run_counts || !host_n_runs) return fail("amwg_summary_rank_runs: null pointer");
  if (dev_weights && (!dev_sorted_vals || !dev_weight_scan)) return fail("amwg_summary_rank_runs: null pointer (weights need the sorted payloads and a scan buffer)");
  if (rank_device_check("amwg_summary_rank_runs", device)) return -1;
  CUDA_TRY(cudaSetDevice(device));
  using u64 = unsigned long long;
  const u64* keys = reinterpret_cast<const u64*>(dev_sorted_keys);
  const size_t need = std::max(rank::scan_scratch_bytes<unsigned>(n), rank::scan_scratch_bytes<long long>(n)) + 256;
  rank::Lease lease(device);
  void* sp = nullptr;
  CUDA_TRY(rank::scratch_get(device, need, &sp));
  long long* w_excl = dev_weights ? reinterpret_cast<long long*>(dev_weight_scan) : nullptr;
  char* tmp = reinterpret_cast<char*>(sp);
  const unsigned g = rank::grid_for(n);
  if (w_excl) {
    rank::amwg_rank_weights_kernel<<<g, rank::kThreads>>>(dev_sorted_vals, reinterpret_cast<const long long*>(dev_weights), n, w_excl);
    rank::exclusive_scan<long long>(w_excl, n, tmp);
  }
  rank::amwg_rank_flags_kernel<<<g, rank::kThreads>>>(keys, n, dev_run_id);
  rank::exclusive_scan<unsigned>(dev_run_id, n, tmp);
  rank::amwg_rank_heads_kernel<<<g, rank::kThreads>>>(keys, n, dev_run_id, w_excl, reinterpret_cast<u64*>(dev_run_keys),
                                                      reinterpret_cast<long long*>(dev_run_counts));
  rank::amwg_rank_ends_kernel<<<g, rank::kThreads>>>(keys, n, dev_run_id, w_excl, dev_sorted_vals, reinterpret_cast<const long long*>(dev_weights),
                                                     reinterpret_cast<long long*>(dev_run_counts));
  CUDA_TRY(cudaGetLastError());
  uint32_t last = 0;
  CUDA_TRY(cudaMemcpy(&last, dev_run_id + (n - 1), sizeof last, cudaMemcpyDeviceToHost));
  *host_n_runs = (int64_t)last + 1;
  return 0;
}

extern "C" int amwg_summary_rank_z(int device, const int64_t* dev_run_counts, int64_t n_runs, int64_t offset, int64_t total, double* dev_run_z) {
  if (n_runs < 1) return fail("amwg_summary_rank_z: n_runs must be >= 1");
  if (offset < 0 || total < 1 || total >= ((int64_t)1 << 50)) return fail("amwg_summary_rank_z: need 0 <= offset and 1 <= total < 2^50");
  if (!dev_run_counts || !dev_run_z) return fail("amwg_summary_rank_z: null pointer");
  if (rank_device_check("amwg_summary_rank_z", device)) return -1;
  CUDA_TRY(cudaSetDevice(device));
  const size_t need = rank::scan_scratch_bytes<long long>(n_runs) + 256;
  rank::Lease lease(device);
  void* sp = nullptr;
  CUDA_TRY(rank::scratch_get(device, need, &sp));
  long long* below = reinterpret_cast<long long*>(dev_run_z);           // the counts scanned in the output buffer
  CUDA_TRY(cudaMemcpyAsync(below, dev_run_counts, (size_t)n_runs * sizeof(long long), cudaMemcpyDeviceToDevice, 0));
  rank::exclusive_scan<long long>(below, n_runs, reinterpret_cast<char*>(sp));
  rank::amwg_rank_z_kernel<<<rank::grid_for(n_runs), rank::kThreads>>>(below, reinterpret_cast<const long long*>(dev_run_counts), n_runs, offset,
                                                                       (double)total, dev_run_z);
  CUDA_TRY(cudaGetLastError());
  CUDA_TRY(cudaDeviceSynchronize());
  return 0;
}

extern "C" int amwg_summary_rank_scatter(int device, const uint32_t* dev_sorted_vals, const uint32_t* dev_run_id, int64_t n, const double* dev_run_z,
                                         double* dev_out, int32_t entries, int64_t chains, int32_t entry) {
  if (n < 1) return fail("amwg_summary_rank_scatter: n must be >= 1");
  if (n >= ((int64_t)1 << 32)) return fail("amwg_summary_rank_scatter: 2^32 or more keys");
  if (entries <= 0 || chains <= 0) return fail("amwg_summary_rank_scatter: empty output block");
  if (entry < 0 || entry >= entries) return fail("amwg_summary_rank_scatter: entry out of range");
  if (!dev_sorted_vals || !dev_run_id || !dev_run_z || !dev_out) return fail("amwg_summary_rank_scatter: null pointer");
  if (rank_device_check("amwg_summary_rank_scatter", device)) return -1;
  CUDA_TRY(cudaSetDevice(device));
  rank::amwg_rank_scatter_kernel<<<rank::grid_for(n), rank::kThreads>>>(dev_sorted_vals, dev_run_id, n, dev_run_z, dev_out, entries, chains, entry);
  CUDA_TRY(cudaGetLastError());
  CUDA_TRY(cudaDeviceSynchronize());
  return 0;
}
