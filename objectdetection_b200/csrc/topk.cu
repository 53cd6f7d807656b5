// topk.cu — segmented radix select + in-segment sort: tf.nn.top_k(sorted=True) semantics
// (k largest per row, descending, ties -> lower index). Call sites replaced: proposals_tf.py:169,
// detection.py:221; also the score ordering inside tf.image.non_max_suppression.
//
// Every element gets a unique orderable key  c = (score_key << ib) | (2^ib - 1 - index),  ib = ceil(log2(cols)),
// so "k largest by (value desc, index asc)" is "k largest c". Selection is a most-significant-digit radix select
// (12-bit digits) in three launches: a histogram pass over the leading digit (per-CTA shared-memory histograms ->
// global atomics -> the last CTA of the row, found with a ticket counter, scans the 4096 buckets), a split pass
// (keys above the threshold bucket are winners, keys inside it become candidates) and a one-CTA-per-row tail
// that resolves the remaining digits over the candidates in shared memory. The k winners are then ordered by
// 1024-key tile sorts (register/shuffle bitonic) plus a merge-rank kernel (binary search of every key in every other
// sorted tile) for k <= 16384, or a global-memory bitonic sort above that.
#include "topk.cuh"

namespace od {

constexpr int kDigitBits = 12;
constexpr int kBins = 1 << kDigitBits;
constexpr int kSelThreads = 256;
constexpr int kSortThreads = 1024;
constexpr int64_t kSmemSortMax = 16384;

struct __align__(16) SelState {
  unsigned long long prefix;  // determined high bits of the k-th key (low `shift` bits are zero)
  int32_t shift;              // number of undetermined low bits
  int32_t k_rem;              // how many to take among the elements matching `prefix`
  int32_t done;               // every element matching `prefix` is selected
  uint32_t reserved;          // number of winners above the threshold bucket (region boundary for the rank sort)
  uint32_t out_count;         // slot counter of the winners buffer
  uint32_t cand_count;        // number of keys in the threshold bucket of the first digit (may exceed the buffer)
};

__device__ __forceinline__ unsigned long long topk_key(float s, uint32_t idx, int ib) {
  return ((unsigned long long)score_key(s) << ib) | (unsigned long long)((1u << ib) - 1u - idx);
}

struct RowChunk {
  int64_t begin, end;
};
__device__ __forceinline__ RowChunk row_chunk(int64_t cols) {
  const int64_t per = (cols + gridDim.x - 1) / gridDim.x;
  RowChunk c;
  c.begin = per * blockIdx.x;
  c.end = min(cols, c.begin + per);
  return c;
}

// Selected <=> (c >> shift) >= (prefix >> shift). Exactly k elements qualify.
__global__ void __launch_bounds__(kSelThreads)
topk_collect_kernel(const float* __restrict__ scores, int64_t cols, int64_t row_stride, int64_t col_stride, int ib,
                    int take_all, int64_t buf_stride, SelState* __restrict__ states,
                    unsigned long long* __restrict__ buf) {
  const int row = blockIdx.y;
  SelState* st = states + row;
  const int shift = take_all ? 0 : st->shift;
  const unsigned long long thr = take_all ? 0ull : (st->prefix >> shift);
  const float* srow = scores + (int64_t)row * row_stride;
  unsigned long long* out = buf + (int64_t)row * buf_stride;
  const RowChunk ch = row_chunk(cols);
  const int lane = threadIdx.x & 31;
  for (int64_t i0 = ch.begin; i0 < ch.end; i0 += kSelThreads) {
    const int64_t i = i0 + threadIdx.x;
    unsigned long long c = 0;
    bool sel = false;
    if (i < ch.end) {
      c = topk_key(srow[i * col_stride], (uint32_t)i, ib);
      sel = (c >> shift) >= thr;
    }
    const uint32_t ballot = __ballot_sync(0xffffffffu, sel);
    if (ballot) {
      uint32_t base = 0;
      if (lane == 0) base = atomicAdd(&st->out_count, (uint32_t)__popc(ballot));
      base = __shfl_sync(0xffffffffu, base, 0);
      if (sel) out[base + __popc(ballot & ((1u << lane) - 1u))] = c;
    }
  }
}

// First-digit histogram only: per-CTA shared-memory histogram of the leading `bits` bits -> global histogram.
// The consumers (split / tail) locate the threshold bucket themselves, so there is no last-CTA tail here.
__global__ void __launch_bounds__(kSelThreads)
topk_hist1_kernel(const float* __restrict__ scores, int64_t cols, int64_t row_stride, int64_t col_stride, int ib,
                  int shift, uint32_t* __restrict__ hist) {
  pdl_prologue();
  __shared__ uint32_t sh[kBins];
  const int row = blockIdx.y;
  for (int b = threadIdx.x; b < kBins; b += kSelThreads) sh[b] = 0;
  __syncthreads();
  const float* srow = scores + (int64_t)row * row_stride;
  const RowChunk ch = row_chunk(cols);
  for (int64_t i0 = ch.begin + threadIdx.x; i0 < ch.end; i0 += 4 * kSelThreads) {
    float v[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int64_t i = i0 + u * kSelThreads;
      v[u] = (i < ch.end) ? __ldg(&srow[i * col_stride]) : 0.0f;
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int64_t i = i0 + u * kSelThreads;
      if (i < ch.end) {
        OD_DBG_IDX((uint32_t)(topk_key(v[u], (uint32_t)i, ib) >> shift), kBins);
        atomicAdd(&sh[(uint32_t)(topk_key(v[u], (uint32_t)i, ib) >> shift)], 1u);
      }
    }
  }
  __syncthreads();
  uint32_t* hrow = hist + (int64_t)row * kBins;
  for (int b = threadIdx.x; b < kBins; b += kSelThreads) {
    const uint32_t v = sh[b];
    if (v) atomicAdd(&hrow[b], v);
  }
}

// Block-wide: bucket of a 4096-bin histogram (global or shared) that holds the k-th largest key, scanning from the
// top; returns through shared memory (bucket, keys to take inside it, whether that is the whole bucket).
struct BucketPick {
  int bucket, k_rem, done;
};
template <int THREADS, typename Load>
__device__ __forceinline__ BucketPick pick_bucket(Load load_bin, int k, uint32_t* warp_sums, BucketPick* s_pick) {
  constexpr int kPer = kBins / THREADS;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int top_bin = kBins - 1 - tid * kPer;   // thread 0 owns the highest buckets
  uint32_t local[kPer];
  uint32_t sum = 0;
#pragma unroll
  for (int q = 0; q < kPer; ++q) {
    local[q] = load_bin(top_bin - q);
    sum += local[q];
  }
  uint32_t incl = sum;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const uint32_t v = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += v;
  }
  if (lane == 31) warp_sums[warp] = incl;
  __syncthreads();
  uint32_t warp_off = 0;
  for (int w = 0; w < warp; ++w) warp_off += warp_sums[w];
  const uint32_t before = warp_off + incl - sum;
  if ((uint32_t)k > before && (uint32_t)k <= before + sum) {
    uint32_t cum = before;
#pragma unroll
    for (int q = 0; q < kPer; ++q) {
      if ((uint32_t)k > cum && (uint32_t)k <= cum + local[q]) {
        s_pick->bucket = top_bin - q;
        s_pick->k_rem = k - (int)cum;
        s_pick->done = ((int)local[q] == k - (int)cum);
      }
      cum += local[q];
    }
  }
  __syncthreads();
  const BucketPick r = *s_pick;
  __syncthreads();
  return r;
}

// Block-wide exclusive prefix sum of one int per thread; returns (offset of this thread, block total).
template <int THREADS>
__device__ __forceinline__ int2 block_exclusive_scan(int v, uint32_t* warp_sums) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  int incl = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int t = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += t;
  }
  if (lane == 31) warp_sums[warp] = (uint32_t)incl;
  __syncthreads();
  int off = 0, total = 0;
#pragma unroll
  for (int w = 0; w < THREADS / 32; ++w) {
    const int c = (int)warp_sums[w];
    if (w < warp) off += c;
    total += c;
  }
  __syncthreads();
  return make_int2(off + incl - v, total);
}

// ---- select = 3 launches: (1) topk_hist_kernel on the leading 12-bit digit -> the bucket b that holds the k-th key;
// (2) topk_split_kernel re-reads the row once: keys above b are winners (-> buf), keys in b are candidates
// (-> cand); (3) topk_tail_kernel, one CTA per row, resolves the remaining digits over the (few thousand)
// candidates with shared-memory histograms and appends the winners among them. If the candidates overflow their
// buffer (heavily clustered or tied scores), the tail falls back to scanning the original row: slow, still exact.
constexpr int kTailThreads = 1024;

constexpr int kSplitPer = 8;   // keys per thread and tile: one atomic per CTA, tile and list instead of one per warp
__global__ void __launch_bounds__(kSelThreads)
topk_split_kernel(const float* __restrict__ scores, int64_t cols, int64_t row_stride, int64_t col_stride, int ib, int k,
                  int shift, int64_t buf_stride, int64_t cand_cap, const uint32_t* __restrict__ hist,
                  SelState* __restrict__ states, unsigned long long* __restrict__ buf, unsigned long long* __restrict__ cand) {
  pdl_prologue();
  __shared__ uint32_t warp_sums[kSelThreads / 32];
  __shared__ BucketPick s_pick;
  __shared__ uint32_t s_base[2];
  const int row = blockIdx.y;
  SelState* st = states + row;
  const uint32_t* hrow = hist + (int64_t)row * kBins;
  const BucketPick pk = pick_bucket<kSelThreads>([&](int b) { return __ldg(&hrow[b]); }, k, warp_sums, &s_pick);
  const unsigned long long bucket = (unsigned long long)pk.bucket;
  const int take_bucket = pk.done;   // the whole bucket is selected: no candidates left to resolve
  if (blockIdx.x == 0 && threadIdx.x == 0) {   // for the tail kernel
    st->prefix = bucket << shift;
    st->shift = shift;
    st->k_rem = pk.k_rem;
    st->done = pk.done;
  }
  const float* srow = scores + (int64_t)row * row_stride;
  unsigned long long* out = buf + (int64_t)row * buf_stride;
  unsigned long long* cnd = cand + (int64_t)row * cand_cap;
  const RowChunk ch = row_chunk(cols);
  for (int64_t t0 = ch.begin; t0 < ch.end; t0 += (int64_t)kSplitPer * kSelThreads) {
    float v[kSplitPer];
#pragma unroll
    for (int u = 0; u < kSplitPer; ++u) {
      const int64_t i = t0 + u * kSelThreads + threadIdx.x;
      v[u] = (i < ch.end) ? __ldg(&srow[i * col_stride]) : 0.0f;
    }
    uint32_t wmask = 0, cmask = 0;
#pragma unroll
    for (int u = 0; u < kSplitPer; ++u) {
      const int64_t i = t0 + u * kSelThreads + threadIdx.x;
      if (i < ch.end) {
        const unsigned long long d = topk_key(v[u], (uint32_t)i, ib) >> shift;
        if ((d > bucket) || (take_bucket && d == bucket)) wmask |= 1u << u;
        else if (d == bucket) cmask |= 1u << u;
      }
    }
    const int2 ws = block_exclusive_scan<kSelThreads>(__popc(wmask), warp_sums);
    const int2 cs = block_exclusive_scan<kSelThreads>(__popc(cmask), warp_sums);
    if (threadIdx.x == 0) {
      s_base[0] = ws.y ? atomicAdd(&st->out_count, (uint32_t)ws.y) : 0u;
      s_base[1] = cs.y ? atomicAdd(&st->cand_count, (uint32_t)cs.y) : 0u;
    }
    __syncthreads();
    uint32_t wpos = s_base[0] + (uint32_t)ws.x, cpos = s_base[1] + (uint32_t)cs.x;
#pragma unroll
    for (int u = 0; u < kSplitPer; ++u) {
      const int64_t i = t0 + u * kSelThreads + threadIdx.x;
      if ((wmask >> u) & 1u) {
        OD_DBG_IDX(wpos, k);
        out[wpos++] = topk_key(v[u], (uint32_t)i, ib);
      }
      if ((cmask >> u) & 1u) {
        if (cpos < (uint32_t)cand_cap) cnd[cpos] = topk_key(v[u], (uint32_t)i, ib);   // beyond the capacity only the count grows
        ++cpos;
      }
    }
    __syncthreads();
  }
}

__global__ void __launch_bounds__(kTailThreads)
topk_tail_kernel(const float* __restrict__ scores, int64_t cols, int64_t row_stride, int64_t col_stride, int ib,
                 int64_t buf_stride, int64_t cand_cap, SelState* __restrict__ states, unsigned long long* __restrict__ buf,
                 const unsigned long long* __restrict__ cand) {
  pdl_prologue();
  __shared__ uint32_t sh[kBins];
  __shared__ uint32_t warp_sums[kTailThreads / 32];
  __shared__ BucketPick s_pick;
  const int row = blockIdx.x;
  SelState* st = states + row;
  // keys written so far (by the split pass) are all greater than the ones this kernel appends: the rank sort
  // uses that boundary to halve its compares
  if (threadIdx.x == 0) st->reserved = st->out_count;
  if (st->done) return;   // the split pass already emitted everything
  const int tid = threadIdx.x;
  const int shift1 = st->shift;
  unsigned long long prefix = st->prefix;
  int k_rem = st->k_rem, done = 0, shift = shift1;
  const uint32_t n_cand = st->cand_count;
  const bool overflow = n_cand > (uint32_t)cand_cap;
  const int64_t n_src = overflow ? cols : (int64_t)n_cand;
  const float* srow = scores + (int64_t)row * row_stride;
  const unsigned long long* cnd = cand + (int64_t)row * cand_cap;
  auto key_at = [&](int64_t i) -> unsigned long long {
    return overflow ? topk_key(srow[i * col_stride], (uint32_t)i, ib) : cnd[i];
  };
  while (shift > 0 && !done) {
    const int bits = shift >= kDigitBits ? kDigitBits : shift;
    const int new_shift = shift - bits;
    const uint32_t mask = (1u << bits) - 1u;
    for (int b = tid; b < kBins; b += kTailThreads) sh[b] = 0;
    __syncthreads();
    for (int64_t i = tid; i < n_src; i += kTailThreads) {
      const unsigned long long c = key_at(i);
      if ((c >> shift) == (prefix >> shift)) atomicAdd(&sh[(uint32_t)(c >> new_shift) & mask], 1u);
    }
    __syncthreads();
    const BucketPick pk = pick_bucket<kTailThreads>([&](int b) { return sh[b]; }, k_rem, warp_sums, &s_pick);
    prefix |= (unsigned long long)pk.bucket << new_shift;
    k_rem = pk.k_rem;
    done = pk.done;
    shift = new_shift;
  }
  // winners among the candidates: same leading digit, and (c >> shift) >= (prefix >> shift). This CTA is the only
  // writer of the row by now (the split kernel has finished), so the output offset is a plain running count.
  const unsigned long long thr = prefix >> shift;
  unsigned long long* out = buf + (int64_t)row * buf_stride;
  uint32_t base = st->out_count;
  for (int64_t i0 = 0; i0 < n_src; i0 += kTailThreads) {
    const int64_t i = i0 + tid;
    unsigned long long c = 0;
    bool sel = false;
    if (i < n_src) {
      c = key_at(i);
      sel = ((c >> shift1) == (prefix >> shift1)) && ((c >> shift) >= thr);
    }
    const int2 sc = block_exclusive_scan<kTailThreads>(sel ? 1 : 0, warp_sums);
    if (sel) {
      OD_DBG_IDX(base + (uint32_t)sc.x, buf_stride);
      out[base + (uint32_t)sc.x] = c;
    }
    base += (uint32_t)sc.y;
  }
}

// Tile sort + merge rank (k <= kMergeMaxK): (1) topk_tile_sort_kernel sorts every 1024-key tile of the winners in
// shared memory (bitonic, one CTA per tile); (2) topk_merge_emit_kernel stages all sorted tiles of a row in shared
// memory; the final position of a key is its position inside its own tile plus, for every other tile, the number of
// keys greater than it, found by binary search: ~60 compares per key instead of k.
constexpr int kTileKeys = 1024;
constexpr int kTileSortThreads = kTileKeys;   // one key per thread, held in a register
constexpr int kMergeThreads = 256;
constexpr int64_t kMergeMaxK = 16384;

// Bitonic network over 1024 keys, one per thread: partner distances below 32 are warp shuffles (40 of the 55 stages,
// no barrier), the rest go through shared memory.
__global__ void __launch_bounds__(kTileSortThreads)
topk_tile_sort_kernel(unsigned long long* __restrict__ buf, int64_t buf_stride, int k) {
  pdl_prologue();
  __shared__ unsigned long long skeys[kTileKeys];
  const int row = blockIdx.y, t0 = blockIdx.x * kTileKeys, t = threadIdx.x;
  unsigned long long* seg = buf + (int64_t)row * buf_stride + t0;
  unsigned long long key = (t0 + t < k) ? seg[t] : 0ull;   // padding zeros sort last and stay out of the buffer
  for (int kk = 2; kk <= kTileKeys; kk <<= 1) {
    const bool desc = ((t & kk) == 0);
    for (int j = kk >> 1; j > 0; j >>= 1) {
      unsigned long long other;
      if (j >= 32) {
        skeys[t] = key;
        __syncthreads();
        other = skeys[t ^ j];
        __syncthreads();
      } else {
        other = __shfl_xor_sync(0xffffffffu, key, j);
      }
      const bool keep_max = (((t & j) == 0) == desc);   // lower index of a descending pair keeps the larger key
      key = keep_max ? (key > other ? key : other) : (key < other ? key : other);
    }
  }
  if (t0 + t < k) seg[t] = key;
}

__global__ void __launch_bounds__(kMergeThreads)
topk_merge_emit_kernel(const unsigned long long* __restrict__ buf, int64_t buf_stride, int k, int ib,
                       const float* __restrict__ scores, int64_t row_stride, int64_t col_stride,
                       int32_t* __restrict__ idx_out, float* __restrict__ val_out) {
  pdl_prologue();
  extern __shared__ unsigned long long sk[];   // [k] the row's sorted tiles
  const int row = blockIdx.y;
  const unsigned long long* in = buf + (int64_t)row * buf_stride;
  for (int i = threadIdx.x; i < k; i += kMergeThreads) sk[i] = in[i];
  __syncthreads();
  const int me = blockIdx.x * kMergeThreads + threadIdx.x;
  if (me >= k) return;
  const unsigned long long mine = sk[me];
  const int my_tile = me / kTileKeys;
  int rank = me - my_tile * kTileKeys;   // keys ahead of me inside my (descending) tile
  const int ntiles = (k + kTileKeys - 1) / kTileKeys;
  for (int t = 0; t < ntiles; ++t) {
    if (t == my_tile) continue;
    const unsigned long long* tp = sk + t * kTileKeys;
    int lo = 0, hi = min(kTileKeys, k - t * kTileKeys);   // first position whose key is not greater than mine
    while (lo < hi) {
      const int mid = (lo + hi) >> 1;
      if (tp[mid] > mine) lo = mid + 1;
      else hi = mid;
    }
    rank += lo;
  }
  const uint32_t imask = (1u << ib) - 1u;
  const uint32_t idx = imask - (uint32_t)(mine & imask);
  OD_DBG_IDX(rank, k);
  idx_out[(int64_t)row * k + rank] = (int32_t)idx;
  if (val_out) val_out[(int64_t)row * k + rank] = scores[(int64_t)row * row_stride + (int64_t)idx * col_stride];
}

// ---- generic descending sort of uint64 segments (shared-memory when it fits, global bitonic otherwise)
__global__ void __launch_bounds__(kSortThreads)
sort_u64_smem_kernel(unsigned long long* __restrict__ keys, int n_pow2) {
  extern __shared__ unsigned long long skeys[];
  unsigned long long* seg = keys + (int64_t)blockIdx.x * n_pow2;
  for (int i = threadIdx.x; i < n_pow2; i += kSortThreads) skeys[i] = seg[i];
  __syncthreads();
  block_bitonic_sort_desc(skeys, n_pow2);
  for (int i = threadIdx.x; i < n_pow2; i += kSortThreads) seg[i] = skeys[i];
}

__global__ void bitonic_step_global_kernel(unsigned long long* __restrict__ keys, int64_t n_pow2, int64_t k, int64_t j) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (n_pow2 >> 1)) return;
  unsigned long long* seg = keys + (int64_t)blockIdx.y * n_pow2;
  const int64_t i = ((t & ~(j - 1)) << 1) | (t & (j - 1));
  const int64_t l = i | j;
  const bool desc = ((i & k) == 0);
  const unsigned long long a = seg[i], b = seg[l];
  if ((a < b) == desc) {
    seg[i] = b;
    seg[l] = a;
  }
}

__global__ void pad_emit_kernel(const unsigned long long* __restrict__ buf, int64_t k, int ib,
                                const float* __restrict__ scores, int64_t row_stride, int64_t col_stride,
                                int64_t buf_stride, int32_t* __restrict__ idx_out, float* __restrict__ val_out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int row = blockIdx.y;
  if (i >= k) return;
  const uint32_t imask = (1u << ib) - 1u;
  const uint32_t idx = imask - (uint32_t)(buf[(int64_t)row * buf_stride + i] & imask);
  idx_out[(int64_t)row * k + i] = (int32_t)idx;
  if (val_out) val_out[(int64_t)row * k + i] = scores[(int64_t)row * row_stride + (int64_t)idx * col_stride];
}

int sort_u64_desc_launch(unsigned long long* keys, int64_t rows, int64_t n_pow2, cudaStream_t st) {
  if (rows == 0 || n_pow2 <= 1) return OD_OK;
  if (n_pow2 <= kSmemSortMax) {
    const size_t smem = (size_t)n_pow2 * sizeof(unsigned long long);
    OD_CUDA(cudaFuncSetAttribute(sort_u64_smem_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    sort_u64_smem_kernel<<<(unsigned)rows, kSortThreads, smem, st>>>(keys, (int)n_pow2);
    OD_LAUNCH_CHECK("sort_u64_smem_kernel");
    return OD_OK;
  }
  const dim3 grid((unsigned)((n_pow2 / 2 + 255) / 256), (unsigned)rows);
  for (int64_t k = 2; k <= n_pow2; k <<= 1)
    for (int64_t j = k >> 1; j > 0; j >>= 1) {
      bitonic_step_global_kernel<<<grid, 256, 0, st>>>(keys, n_pow2, k, j);
      count_launches(1);
    }
  OD_LAUNCH_CHECK_NC("bitonic_step_global_kernel");
  return OD_OK;
}

static int blocks_per_row(int64_t rows, int64_t cols) {
  const int64_t by_work = (cols + 2047) / 2048;
  const int64_t by_fill = (2 * kNumSMsB200 + rows - 1) / rows;
  int64_t b = by_work < by_fill ? by_work : by_fill;
  return (int)(b < 1 ? 1 : b);
}

// Candidate buffer entries per row for the split/tail select.
static int64_t cand_capacity(int64_t cols, int64_t k) {
  int64_t cap = 4 * next_pow2(k > 0 ? k : 1);
  if (cap < 16384) cap = 16384;
  return cap < cols ? cap : cols;
}

size_t topk_workspace_bytes(int64_t rows, int64_t cols, int64_t k) {
  Workspace w(nullptr, 0);
  w.take<SelState>((size_t)rows);
  w.take<uint32_t>((size_t)rows * kBins);
  w.take<unsigned long long>((size_t)rows * (size_t)next_pow2(k > 0 ? k : 1));
  w.take<unsigned long long>((size_t)rows * (size_t)cand_capacity(cols, k));
  return w.off + 256;
}

int topk_launch(const float* scores, int64_t rows, int64_t cols, int64_t row_stride, int64_t col_stride, int64_t k,
                int32_t* idx_out, float* val_out, void* ws, size_t ws_bytes, cudaStream_t st) {
  if (k < 0 || k > cols) OD_FAIL(OD_ERR_PARAM, "k=%lld must be in [0, cols=%lld]", (long long)k, (long long)cols);
  if (rows == 0 || k == 0) return OD_OK;
  if (cols >= ((int64_t)1 << 31) || rows > 65535) OD_FAIL(OD_ERR_PARAM, "top-k supports cols < 2^31 and rows <= 65535");
  if (!ws) OD_FAIL(OD_ERR_WORKSPACE, "top-k workspace is NULL");
  Workspace w(ws, ws_bytes);
  const int64_t n_pow2 = next_pow2(k);
  SelState* states = w.take<SelState>((size_t)rows);
  uint32_t* hist = w.take<uint32_t>((size_t)rows * kBins);
  unsigned long long* buf = w.take<unsigned long long>((size_t)rows * (size_t)n_pow2);
  const int64_t cap = cand_capacity(cols, k);
  unsigned long long* cand = w.take<unsigned long long>((size_t)rows * (size_t)cap);
  if (!w.ok()) OD_FAIL(OD_ERR_WORKSPACE, "top-k workspace %zu < %zu bytes", ws_bytes, w.off);
  const int ib = index_bits(cols);
  const int total_bits = 32 + ib;
  const dim3 grid((unsigned)blocks_per_row(rows, cols), (unsigned)rows);
  // state + histogram are contiguous at the head of the workspace
  OD_CUDA(cudaMemsetAsync(states, 0, (size_t)((char*)buf - (char*)states), st));
  const int take_all = (k == cols);
  if (take_all) {
    topk_collect_kernel<<<grid, kSelThreads, 0, st>>>(scores, cols, row_stride, col_stride, ib, 1, n_pow2, states, buf);
    OD_LAUNCH_CHECK("topk_collect_kernel");
  } else {
    const int shift1 = total_bits - kDigitBits;   // total_bits >= 33
    OD_CUDA(launch_pdl(topk_hist1_kernel, grid, dim3(kSelThreads), 0, st, scores, cols, row_stride, col_stride, ib, shift1, hist));
    OD_LAUNCH_CHECK("topk_hist1_kernel");
    OD_CUDA(launch_pdl(topk_split_kernel, grid, dim3(kSelThreads), 0, st, scores, cols, row_stride, col_stride, ib, (int)k, shift1, n_pow2, cap, hist,
                                                    states, buf, cand));
    OD_LAUNCH_CHECK("topk_split_kernel");
    OD_CUDA(launch_pdl(topk_tail_kernel, dim3((unsigned)rows), dim3(kTailThreads), 0, st, scores, cols, row_stride, col_stride, ib, n_pow2, cap, states, buf, cand));
    OD_LAUNCH_CHECK("topk_tail_kernel");
  }
  if (k <= kMergeMaxK) {
    const int ntiles = (int)((k + kTileKeys - 1) / kTileKeys);
    OD_CUDA(launch_pdl(topk_tile_sort_kernel, dim3((unsigned)ntiles, (unsigned)rows), dim3(kTileSortThreads), 0, st, buf, n_pow2, (int)k));
    OD_LAUNCH_CHECK("topk_tile_sort_kernel");
    const size_t smem = (size_t)k * sizeof(unsigned long long);
    static const size_t merge_static = static_smem_bytes((const void*)topk_merge_emit_kernel);
    if (smem + merge_static > 48 * 1024)
      OD_CUDA(cudaFuncSetAttribute(topk_merge_emit_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    OD_CUDA(launch_pdl(topk_merge_emit_kernel, dim3((unsigned)((k + kMergeThreads - 1) / kMergeThreads), (unsigned)rows), dim3(kMergeThreads), smem, st, 
        buf, n_pow2, (int)k, ib, scores, row_stride, col_stride, idx_out, val_out));
    OD_LAUNCH_CHECK("topk_merge_emit_kernel");
  } else {
    // zero the padding, sort in global memory, then emit
    for (int64_t r = 0; r < rows; ++r)
      if (n_pow2 > k) OD_CUDA(cudaMemsetAsync(buf + r * n_pow2 + k, 0, (size_t)(n_pow2 - k) * 8, st));
    OD_CHECK(sort_u64_desc_launch(buf, rows, n_pow2, st));
    const dim3 g2((unsigned)((k + 255) / 256), (unsigned)rows);
    pad_emit_kernel<<<g2, 256, 0, st>>>(buf, k, ib, scores, row_stride, col_stride, n_pow2, idx_out, val_out);
    OD_LAUNCH_CHECK("pad_emit_kernel");
  }
  return OD_OK;
}

}  // namespace od

using namespace od;

extern "C" {

size_t od_topk_workspace_bytes(int64_t rows, int64_t cols, int64_t k) { return topk_workspace_bytes(rows, cols, k); }

int od_topk(const DLTensor* scores, int64_t k, DLTensor* values, DLTensor* indices, void* ws, size_t ws_bytes,
            void* stream) {
  DeviceScope scope;
  OD_CHECK(check_tensor(scores, "scores", F32, {kAny, kAny}, 4, scope, /*any_strides=*/true));
  const int64_t rows = scores->shape[0], cols = scores->shape[1];
  if (k < 0) OD_FAIL(OD_ERR_SHAPE, "indices: k = %lld is negative", (long long)k);
  OD_CHECK(check_tensor(indices, "indices", I32, {rows, k}, 4, scope));
  OD_CHECK(check_opt_tensor(values, "values", F32, {rows, k}, 4, scope));
  return topk_launch(dptr<float>(scores), rows, cols, stride_of(scores, 0), stride_of(scores, 1), k,
                     dptr<int32_t>(indices), dptr<float>(values), ws, ws_bytes, static_cast<cudaStream_t>(stream));
}

}  // extern "C"
