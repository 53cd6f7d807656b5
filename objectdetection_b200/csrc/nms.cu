// nms.cu — greedy hard NMS with tf.image.non_max_suppression semantics as a bitmask-IoU kernel
// plus a single-CTA keep scan. Call sites replaced: proposals_tf.py:234, detection.py:177.
//
//   mask layout : row-major words. With W = ceil(K/64) and Ws = W rounded up to even, word (i, w) at i*Ws + w says which
//                 boxes of chunk w box i suppresses (only w > i/64 is read). The diagonal tiles are kept TRANSPOSED in
//                 a second array diagT [W][64] (word j of chunk c = which earlier boxes of the chunk suppress box
//                 c*64+j), which is what the scan needs. The 64 rows of chunk c are one contiguous span of 64*Ws words.
//   mask kernel : a CTA owns 64 rows x 4 column tiles whose canonical boxes sit in shared memory; a thread owns row i
//                 and builds the words of two tiles. Pass 1 is branch-free: a pair is a candidate iff four fp32
//                 differences are all negative (sign-bit AND, one funnel shift per pair). Pass 2 evaluates the exact
//                 TF IoU (TF's operation order, IEEE division, `> thr`) for the candidates only.
//   scan kernel : one CTA per image walks the 64-box chunks in order. Inside a chunk the greedy recurrence
//                 kept_j = cand_j && !(sup_j & kept) is solved by warp-ballot fixed-point iteration (bit j is final
//                 after j+1 rounds; typically 2-4 rounds), then every later word of the `removed` bitmap is updated by
//                 two threads (one per half of the chunk's rows): each ORs that word of its kept rows (conflict-free
//                 shared-memory reads, no cross-lane reduction, one atomicOr). The rows and the diagonal tile of chunk c + nslots - 1 arrive
//                 through two cp.async.bulk (TMA) copies into a shared-memory ring, completion counted in bytes on
//                 an mbarrier per slot, while chunk c is resolved. Stops as soon as max_out boxes are kept.
#include "nms.cuh"
#include "tma.cuh"
#include "topk.cuh"

namespace od {

constexpr int kMaskColTiles = 4;                         // column tiles (of 64 boxes) per CTA
constexpr int kMaskThreads = 256;                        // 64 rows x kMaskGroups thread groups
constexpr int kMaskGroups = kMaskThreads / 64;           // group h owns column tiles h, h + kMaskGroups, ... of the span

template <bool FAST>  // FAST: thr >= 0, division skipped when the intersection is not positive
__global__ void __launch_bounds__(kMaskThreads)
nms_mask_kernel(const float4* __restrict__ boxes, const int32_t* __restrict__ num_valid,
                const int32_t* __restrict__ group, int K, int W, int rb_begin, float thr, int max_out,
                const int32_t* __restrict__ scan_state, int state_stride, int Ws, unsigned long long* __restrict__ mask,
                unsigned long long* __restrict__ diagT) {
  pdl_prologue();
  const int rb = rb_begin + blockIdx.y, b = blockIdx.z;
  const int cb0 = rb + blockIdx.x * kMaskColTiles;
  const int n = num_valid ? min(num_valid[b], K) : K;
  if (cb0 * 64 >= n) return;  // rb <= cb0: nothing valid in this span
  // second round of a two-round NMS: the first round's scan may already have kept max_out boxes
  if (scan_state && scan_state[(int64_t)b * state_stride] >= max_out) return;
  __shared__ float4 cbox[kMaskColTiles * 64];   // canonical corners; boxes >= n are zero-area (never hit)
  __shared__ float carea[kMaskColTiles * 64];
  __shared__ int32_t cgrp[kMaskColTiles * 64];
  const int t = threadIdx.x;
  const float4* bx = boxes + (int64_t)b * K;
  for (int q = t; q < kMaskColTiles * 64; q += kMaskThreads) {
    const int j = cb0 * 64 + q;
    const float4 v = (j < n) ? bx[j] : make_float4(0.f, 0.f, 0.f, 0.f);
    const CBox c = canon_box(v);
    cbox[q] = make_float4(c.ymin, c.xmin, c.ymax, c.xmax);
    carea[q] = c.area;
    cgrp[q] = (group && j < n) ? group[(int64_t)b * K + j] : -1;
  }
  __syncthreads();
  const int r = t & 63, half = t >> 6;   // (thread group)
  const int i = rb * 64 + r;
  const bool row_ok = i < n;
  const CBox my = canon_box(row_ok ? bx[i] : make_float4(0.f, 0.f, 0.f, 0.f));
  const int32_t g = (group && row_ok) ? group[(int64_t)b * K + i] : 0;
#pragma unroll
  for (int ct = 0; ct < kMaskColTiles / kMaskGroups; ++ct) {
    const int tile = half + kMaskGroups * ct;
    const int cb = cb0 + tile;
    if (cb * 64 >= n) break;   // uniform per thread group (two warps)
    unsigned long long bits = 0ull;
    const float4* cbp = cbox + tile * 64;
    const float* cap = carea + tile * 64;
    const int32_t* cgp = cgrp + tile * 64;
    if (FAST) {
      // pass 1, branch-free: candidates = a superset of the pairs whose intersection has positive height and width.
      // Everything else has inter == 0 (or NaN) in TF's arithmetic and can never exceed a threshold >= 0.
      // (min(a,b) > max(c,d) needs a > d and b > c; a > c / b > d are the boxes' own validity, which pass 2 settles.)
      // The four differences run on the FMA pipe; a pair is a candidate iff all four are negative, i.e. the AND of
      // their sign bits is set, which one funnel shift appends to the word (bit jj ends up at position jj).
      uint32_t cand_lo = 0u, cand_hi = 0u;
#pragma unroll
      for (int jj = 31; jj >= 0; --jj) {
        const float4 c = cbp[jj];
        const uint32_t sgn = __float_as_uint(c.x - my.ymax) & __float_as_uint(my.ymin - c.z) &
                             __float_as_uint(c.y - my.xmax) & __float_as_uint(my.xmin - c.w);
        cand_lo = __funnelshift_l(sgn, cand_lo, 1);
      }
#pragma unroll
      for (int jj = 31; jj >= 0; --jj) {
        const float4 c = cbp[32 + jj];
        const uint32_t sgn = __float_as_uint(c.x - my.ymax) & __float_as_uint(my.ymin - c.z) &
                             __float_as_uint(c.y - my.xmax) & __float_as_uint(my.xmin - c.w);
        cand_hi = __funnelshift_l(sgn, cand_hi, 1);
      }
      unsigned long long m = ((unsigned long long)cand_hi << 32) | cand_lo;
      if (cb == rb) m &= (r == 63) ? 0ull : ~((2ull << r) - 1ull);   // only j > i
      // pass 2, rare: the exact TF IoU (operation order, IEEE division) of the candidates
      while (m) {
        const int jj = __ffsll((long long)m) - 1;
        m &= m - 1ull;
        const float4 c = cbp[jj];
        const float ih = f_min(my.ymax, c.z) - f_max(my.ymin, c.x);
        const float iw = f_min(my.xmax, c.w) - f_max(my.xmin, c.y);
        const float inter = f_max(ih, 0.0f) * f_max(iw, 0.0f);
        // inter > 0 implies both areas > 0 (inter <= area under monotone rounding), TF's area guard is moot
        const bool hit = (inter > 0.0f) && (inter / (my.area + cap[jj] - inter) > thr) && (!group || g == cgp[jj]);
        bits |= (unsigned long long)hit << jj;
      }
    } else {
#pragma unroll 8
      for (int jj = 0; jj < 64; ++jj) {
        const float4 c = cbp[jj];
        CBox o;
        o.ymin = c.x; o.xmin = c.y; o.ymax = c.z; o.xmax = c.w; o.area = cap[jj];
        const bool hit = (cb * 64 + jj < n) && (tf_iou(my, o) > thr) && (!group || g == cgp[jj]);
        bits |= (unsigned long long)hit << jj;
      }
    }
    if (cb == rb) bits &= (r == 63) ? 0ull : ~((2ull << r) - 1ull);   // only j > i
    if (!row_ok) bits = 0ull;
    if (cb != rb) {
      OD_DBG_IDX(cb, Ws);
      if (row_ok) mask[((int64_t)b * K + i) * Ws + cb] = bits;
    } else {
      // diagonal tile, stored transposed: word jj, bit r = "box r of this chunk suppresses box jj"
      OD_DBG_IDX(cb, W);
      uint32_t* dt = reinterpret_cast<uint32_t*>(diagT + ((int64_t)b * W + cb) * 64);
      const int warp = (t >> 5) & 1, lane = t & 31;
#pragma unroll 8
      for (int jj = 0; jj < 64; ++jj) {
        const uint32_t bal = __ballot_sync(0xffffffffu, (bits >> jj) & 1ull);
        if (lane == 0) dt[jj * 2 + warp] = bal;
      }
    }
  }
}

constexpr int kScanThreads = 256;
constexpr int kScanMaxSlots = 8;
constexpr int kScanCopyParts = 4;   // bulk copies per chunk of 64 mask rows (issued by different lanes of the producer warp)
// named barriers (ids 1..4; 0 is __syncthreads): bar.arrive does not block, bar.sync does; both order shared memory
__device__ __forceinline__ void nb_sync(int id) { asm volatile("bar.sync %0, %1;" ::"r"(id), "n"(kScanThreads) : "memory"); }
__device__ __forceinline__ void nb_sync_n(int id, int n) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(n) : "memory"); }
__device__ __forceinline__ void nb_arrive_n(int id, int n) { asm volatile("bar.arrive %0, %1;" ::"r"(id), "r"(n) : "memory"); }
__device__ __forceinline__ void nb_arrive(int id) { asm volatile("bar.arrive %0, %1;" ::"r"(id), "n"(kScanThreads) : "memory"); }
// 64-bit OR into shared memory as two native 32-bit atomics (a 64-bit shared atomicOr is a compare-and-swap loop)
__device__ __forceinline__ void smem_or64(unsigned long long* p, unsigned long long v) {
  uint32_t* h = reinterpret_cast<uint32_t*>(p);
  if ((uint32_t)v) atomicOr(h, (uint32_t)v);
  if ((uint32_t)(v >> 32)) atomicOr(h + 1, (uint32_t)(v >> 32));
}

// STAGED: nslots >= 2 ring slots of (64 rows x Ws words + the diagonal tile) fit in shared memory (K <= ~12000);
// otherwise the rows are read from global memory (L2).
template <bool STAGED>
__global__ void __launch_bounds__(kScanThreads)
nms_scan_kernel(const unsigned long long* __restrict__ mask, const unsigned long long* __restrict__ diagT,
                const int32_t* __restrict__ num_valid, int K, int W, int Ws, int nslots, int max_out, int c_begin, int c_end,
                int final_round, int32_t* __restrict__ scan_state, int state_stride, int32_t* __restrict__ keep_pos,
                int32_t* __restrict__ num_kept, int32_t* __restrict__ keep_flag) {
  pdl_launch_dependents();
  extern __shared__ __align__(128) unsigned long long smem_u64[];
  const int Wr = (W + 15) & ~15;                 // keeps the ring 128-byte aligned
  unsigned long long* removed = smem_u64;        // [Wr]
  unsigned long long* stage = smem_u64 + Wr;     // [nslots][64*Ws + 64] when STAGED: rows of a chunk, then its diagonal tile
  const size_t slot_words = (size_t)64 * Ws + 64;
  __shared__ __align__(8) unsigned long long full_bar[kScanMaxSlots];
  __shared__ unsigned long long kept_word;
  __shared__ uint4 pipe_ring[2];   // pipelined loop, slot c & 1: keep word of chunk c (x, y), boxes kept before it (z), max_out reached (w)
  __shared__ int32_t pipe_out[2];               // kept_total, last chunk waited for
  const int b = blockIdx.x;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  // Shared-memory set-up touches nothing the previous kernel writes: done while that kernel is still running (the CTA
  // is resident early under programmatic dependent launch), global memory only after pdl_wait().
  for (int w = tid; w < Wr; w += kScanThreads) removed[w] = 0ull;
  if (STAGED && tid == 0) {
    for (int s = 0; s < nslots; ++s) mbar_init(&full_bar[s], 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  }
  pdl_wait();
  const int n = num_valid ? min(num_valid[b], K) : K;
  const int Wn = (n + 63) / 64;
  // scan_state (two-round NMS): [0] = boxes kept so far, then the `removed` bitmap as 2*Wr 32-bit halves
  int32_t* state = scan_state ? scan_state + (int64_t)b * state_stride : nullptr;
  const bool resume = state != nullptr && c_begin > 0;
  const int c_last = min(c_end, Wn);
  if (resume) {
    const unsigned long long* sr = reinterpret_cast<const unsigned long long*>(state + 2);
    for (int w = tid; w < Wr; w += kScanThreads) removed[w] = sr[w];
  } else if (keep_flag) {
    for (int i = tid; i < K; i += kScanThreads) keep_flag[(int64_t)b * K + i] = 0;
  }
  __syncthreads();
  const unsigned long long* mrow = mask + (int64_t)b * K * Ws;
  const unsigned long long* dimg = diagT + (int64_t)b * W * 64;

  int kept_total = resume ? state[0] : 0;
  const int c_first = (kept_total >= max_out) ? c_last : c_begin;   // nothing left to do: skip the loop
  // One thread of the last warp (off the fixed point's critical path) stages chunk c into ring slot (c - c_first) %
  // nslots with two bulk copies: its 64 mask rows (contiguous) and its transposed diagonal tile.
  auto stage_chunk = [&](int c) {
    if (STAGED && tid == kScanThreads - 32 && c < c_last) {
      const int slot = (c - c_first) % nslots;
      unsigned long long* bar = &full_bar[slot];
      unsigned long long* dst = stage + (size_t)slot * slot_words;
      const int rows = min(64, n - c * 64);
      const uint32_t row_bytes = (uint32_t)rows * (uint32_t)Ws * 8u;
      mbar_expect_tx(bar, row_bytes + 512u);
      bulk_g2s(dst, mrow + (size_t)c * 64 * Ws, row_bytes, bar);
      bulk_g2s(dst + (size_t)64 * Ws, dimg + (size_t)c * 64, 512u, bar);
    }
  };
  if (STAGED)
    for (int c = c_first; c < c_first + nslots - 1; ++c) stage_chunk(c);

  int c_waited = c_first - 1;
  if (STAGED) {
    // Only removed[c] is needed to resolve chunk c. Warp 0 resolves chunk c, ORs word c+1 of its kept rows itself and
    // goes on to chunk c+1; warps 1-7 OR the kept rows of chunk c into the words >= c+2 meanwhile, so the per-chunk
    // critical path is the 64x64 fixed point and one warp-wide OR instead of the whole row pass and two CTA barriers.
    // Warp 7 only issues the bulk copies. Barrier 1 + (c&1): keep word of chunk c published (all warps). Barrier
    // 3 + (c&1): the workers are done with chunk c (warp 0 waits for it before chunk c+2, whose word is the first one
    // they might still be updating).
    if (warp == 0) {
      // All 64-bit words are handled as 32-bit halves (lane l owns boxes l and l + 32 of the chunk): this warp's
      // instruction count is the critical path of the whole kernel.
      uint32_t own_lo = 0u, own_hi = 0u;   // word c of the rows kept in chunk c-1: computed here, never leaves the warp
      // Everything of chunk c that does not depend on removed[c] - the phase test of its slot, its diagonal tile, word
      // c+1 of my two rows - is fetched one chunk ahead, so that only one shared load sits between the workers' barrier
      // and the fixed point.
      uint2 sup0 = make_uint2(0u, 0u), sup1 = sup0, nx0 = sup0, nx1 = sup0;
      // (ring slot and phase parity of the chunk to fetch are advanced by hand: `% nslots` and `/ nslots` on a run-time
      //  value cost ~60 dependent instructions on the one warp everybody waits for)
      int f_slot = 0;
      uint32_t f_par = 0u;
      auto fetch = [&](int c) {
        mbar_wait(&full_bar[f_slot], f_par);   // chunk c has landed
        c_waited = c;
        const uint2* rows = reinterpret_cast<const uint2*>(stage + (size_t)f_slot * slot_words);
        if (++f_slot == nslots) {
          f_slot = 0;
          f_par ^= 1u;
        }
        const uint2* dt = rows + (size_t)64 * Ws;
        const int wn = min(c + 1, Wn - 1);
        sup0 = dt[lane];
        sup1 = dt[lane + 32];
        nx0 = rows[(size_t)lane * Ws + wn];
        nx1 = rows[(size_t)(lane + 32) * Ws + wn];
      };
      const uint32_t lbit = 1u << lane;
      const uint2* removed2 = reinterpret_cast<const uint2*>(removed);
      int c = c_first;
      if (c < c_last) fetch(c);
      for (; c < c_last; ++c) {
        if (c - c_first >= 2) nb_sync_n(3 + (c & 1), kScanThreads - 32);   // (workers + this warp; the producer warp is not part of it)
        const uint2 w = removed2[c];
        const int nrem = n - c * 64;
        const bool cand0 = (lane < nrem) && !((w.x | own_lo) & lbit);
        const bool cand1 = (lane + 32 < nrem) && !((w.y | own_hi) & lbit);
        uint32_t k_lo = __ballot_sync(0xffffffffu, cand0), k_hi = __ballot_sync(0xffffffffu, cand1);
        for (int it = 0; it < 64; ++it) {
          const bool k0 = cand0 && !((sup0.x & k_lo) | (sup0.y & k_hi));
          const bool k1 = cand1 && !((sup1.x & k_lo) | (sup1.y & k_hi));
          const uint32_t n_lo = __ballot_sync(0xffffffffu, k0), n_hi = __ballot_sync(0xffffffffu, k1);
          if (n_lo == k_lo && n_hi == k_hi) break;
          k_lo = n_lo;
          k_hi = n_hi;
        }
        int cnt = __popc(k_lo) + __popc(k_hi);
        const int allow = max_out - kept_total;
        if (cnt > allow) {   // respect max_out: drop the highest set bits beyond the allowance
          unsigned long long kept = ((unsigned long long)k_hi << 32) | k_lo;
          while (__popcll(kept) > allow) kept &= ~(1ull << (63 - __clzll((long long)kept)));
          k_lo = (uint32_t)kept;
          k_hi = (uint32_t)(kept >> 32);
          cnt = allow;
        }
        const int total = kept_total + cnt;
        const bool stop = total >= max_out;
        if (lane == 0) pipe_ring[c & 1] = make_uint4(k_lo, k_hi, (uint32_t)kept_total, stop ? 1u : 0u);
        nb_arrive(1 + (c & 1));
        kept_total = total;
        own_lo = own_hi = 0u;
        if (stop) break;
        const uint32_t m0 = 0u - ((k_lo >> lane) & 1u), m1 = 0u - ((k_hi >> lane) & 1u);
        const uint32_t v_lo = (nx0.x & m0) | (nx1.x & m1), v_hi = (nx0.y & m0) | (nx1.y & m1);
        if (c + 1 < c_last) fetch(c + 1);   // (its latency overlaps the reduction below and the workers' barrier)
        if (c + 1 < Wn) {   // (rows beyond n are never kept; whatever their slots hold is masked out)
          own_lo = __reduce_or_sync(0xffffffffu, v_lo);
          own_hi = __reduce_or_sync(0xffffffffu, v_hi);
        }
      }
      if (lane == 0) {
        OD_DBG_ASSERT(!(own_lo | own_hi) || (c >= 0 && c < Wr), "carried bits beyond the removed bitmap");
        if (own_lo | own_hi) smem_or64(&removed[c], ((unsigned long long)own_hi << 32) | own_lo);   // round boundary: the carried bitmap must be complete
        pipe_out[0] = kept_total;
        pipe_out[1] = c_waited;
      }
    } else if (warp == kScanThreads / 32 - 1) {
      // producer warp: refills the slot of chunk c-1 as soon as everybody has left it (issuing a bulk copy costs its
      // thread ~700 cycles, so the rows and the diagonal tile go out from two lanes and nobody else waits for them)
      int slot = nslots - 1;   // slot of chunk c + nslots - 1
      for (int c = c_first; c < c_last; ++c) {
        nb_sync(1 + (c & 1));
        const int cn = c + nslots - 1;
        if (cn < c_last && lane <= kScanCopyParts) {
          unsigned long long* bar = &full_bar[slot];
          unsigned long long* dst = stage + (size_t)slot * slot_words;
          const int rows = min(64, n - cn * 64);
          if (lane == 0) {
            mbar_expect_tx(bar, (uint32_t)rows * (uint32_t)Ws * 8u + 512u);
            bulk_g2s(dst + (size_t)64 * Ws, dimg + (size_t)cn * 64, 512u, bar);
          } else {   // the rows in kScanCopyParts pieces, one lane each
            constexpr int kPart = 64 / kScanCopyParts;
            const int r0 = (lane - 1) * kPart, nr = min(kPart, rows - r0);
            if (nr > 0) bulk_g2s(dst + (size_t)r0 * Ws, mrow + ((size_t)cn * 64 + r0) * Ws, (uint32_t)nr * (uint32_t)Ws * 8u, bar);
          }
        }
        __syncwarp();
        if (++slot == nslots) slot = 0;
        if (pipe_ring[c & 1].w) break;
      }
    } else {
      constexpr int kHalf = (kScanThreads - 64) / 2;   // warps 1-6: two threads per word (rows 0-31 / 32-63)
      const int wt = tid - 32, half = wt / kHalf, idx = wt - half * kHalf;
      int w_slot = 0;
      uint32_t w_par = 0u;
      for (int c = c_first; c < c_last; ++c) {
        mbar_wait(&full_bar[w_slot], w_par);   // (landed long ago; makes the rows visible to this thread)
        nb_sync(1 + (c & 1));        // keep word of chunk c is there; everybody is done with chunk c-1 and its slot
        const uint4 pr = pipe_ring[c & 1];
        const unsigned long long kept = ((unsigned long long)pr.y << 32) | pr.x;
        if (warp == 1) {   // the outputs of chunk c, off warp 0's path
          const int base = (int)pr.z;
#pragma unroll
          for (int h = 0; h < 2; ++h) {
            const int r = lane + 32 * h;
            if ((kept >> r) & 1ull) {
              const int pos = base + __popcll(kept & ((1ull << r) - 1ull));
              OD_DBG_IDX(pos, max_out);
              OD_DBG_IDX(c * 64 + r, K);
              if (keep_pos) keep_pos[(int64_t)b * max_out + pos] = c * 64 + r;
              if (keep_flag) keep_flag[(int64_t)b * K + c * 64 + r] = 1;
            }
          }
        }
        if (pr.w) break;
        if (kept != 0ull && c + 2 < Wn) {
          const unsigned long long* rows = stage + (size_t)w_slot * slot_words;
          const uint32_t kbits = half ? (uint32_t)(kept >> 32) : (uint32_t)kept;
          if (kbits)
            for (int w = c + 2 + idx; w < Wn; w += kHalf) {
              const unsigned long long* col = rows + (size_t)(32 * half) * Ws + w;
              unsigned long long acc = 0ull;
#pragma unroll
              for (int r0 = 0; r0 < 32; r0 += 16) {   // 16 unconditional loads in flight, masked afterwards
                unsigned long long v[16];
#pragma unroll
                for (int r = 0; r < 16; ++r) v[r] = col[(size_t)(r0 + r) * Ws];
#pragma unroll
                for (int r = 0; r < 16; ++r) acc |= v[r] & (0ull - (unsigned long long)((kbits >> (r0 + r)) & 1u));
              }
              OD_DBG_IDX(w, Wr);
              smem_or64(&removed[w], acc);
            }
        }
        nb_arrive_n(3 + (c & 1), kScanThreads - 32);
        if (++w_slot == nslots) {
          w_slot = 0;
          w_par ^= 1u;
        }
      }
    }
    __syncthreads();
    kept_total = pipe_out[0];
    c_waited = pipe_out[1];
  }
  // ---- global-memory path (!STAGED; K beyond the ring in a two-round call): lock-step loop, rows read through L2
  const int c_loop = STAGED ? c_last : c_first;
  unsigned long long nsup0 = 0ull, nsup1 = 0ull;
  if (!STAGED && warp == 0 && c_first < c_last) {
    nsup0 = __ldg(&dimg[(size_t)c_first * 64 + lane]);
    nsup1 = __ldg(&dimg[(size_t)c_first * 64 + lane + 32]);
  }
  for (int c = c_loop; c < c_last; ++c) {
    __syncthreads();   // removed[c] is final
    if (warp == 0) {
      // transposed diagonal tile: the one of the next chunk is loaded one chunk ahead
      const unsigned long long sup0 = nsup0, sup1 = nsup1;
      if (c + 1 < c_last) {
        nsup0 = __ldg(&dimg[(size_t)(c + 1) * 64 + lane]);
        nsup1 = __ldg(&dimg[(size_t)(c + 1) * 64 + lane + 32]);
      }
      const unsigned long long word = removed[c];
      const bool cand0 = (c * 64 + lane < n) && !((word >> lane) & 1ull);
      const bool cand1 = (c * 64 + lane + 32 < n) && !((word >> (lane + 32)) & 1ull);
      unsigned long long kept = (unsigned long long)__ballot_sync(0xffffffffu, cand0) |
                                ((unsigned long long)__ballot_sync(0xffffffffu, cand1) << 32);
      for (int it = 0; it < 64; ++it) {
        const bool k0 = cand0 && !(sup0 & kept);
        const bool k1 = cand1 && !(sup1 & kept);
        const unsigned long long nk = (unsigned long long)__ballot_sync(0xffffffffu, k0) |
                                      ((unsigned long long)__ballot_sync(0xffffffffu, k1) << 32);
        if (nk == kept) break;
        kept = nk;
      }
      // respect max_out: drop the highest set bits beyond the allowance
      const int allow = max_out - kept_total;
      while (__popcll(kept) > allow) kept &= ~(1ull << (63 - __clzll((long long)kept)));
      if (lane == 0) kept_word = kept;
    }
    __syncthreads();
    const unsigned long long kept = kept_word;
    if (kept != 0ull) {
      if (tid < 64 && ((kept >> tid) & 1ull)) {
        const int pos = kept_total + __popcll(kept & ((1ull << tid) - 1ull));
        OD_DBG_IDX(pos, max_out);
        OD_DBG_IDX(c * 64 + tid, K);
        if (keep_pos) keep_pos[(int64_t)b * max_out + pos] = c * 64 + tid;
        if (keep_flag) keep_flag[(int64_t)b * K + c * 64 + tid] = 1;
      }
      kept_total += __popcll(kept);
      if (kept_total >= max_out) break;
      // removed[w] |= OR of word w over the kept rows, for every later word w. Rows beyond n are never kept, so their
      // (unwritten) words are never selected.
      {
        // rows straight from global memory (L2): one owner thread per word (two words per thread and pass), 16 rows x 2
        // words = 32 unconditional loads in flight per thread, no atomics
        for (int w0 = c + 1 + tid; w0 < Wn; w0 += 2 * kScanThreads) {
          const int w1 = w0 + kScanThreads;
          const int w1c = min(w1, Wn - 1);
          unsigned long long acc0 = 0ull, acc1 = 0ull;
#pragma unroll 1
          for (int q = 0; q < 4; ++q) {
            const uint32_t kb = (uint32_t)(kept >> (16 * q)) & 0xFFFFu;
            if (kb == 0u) continue;   // uniform
            unsigned long long v0[16], v1[16];
#pragma unroll
            for (int r = 0; r < 16; ++r) {
              const size_t row = (size_t)min(c * 64 + 16 * q + r, K - 1) * Ws;
              v0[r] = __ldg(&mrow[row + w0]);
              v1[r] = __ldg(&mrow[row + w1c]);
            }
#pragma unroll
            for (int r = 0; r < 16; ++r) {
              acc0 |= ((kb >> r) & 1u) ? v0[r] : 0ull;
              acc1 |= ((kb >> r) & 1u) ? v1[r] : 0ull;
            }
          }
          OD_DBG_IDX(w0, Wr);
          removed[w0] |= acc0;
          if (w1 < Wn) removed[w1] |= acc1;
        }
      }
    }
  }
  if (STAGED) {
    // early exit: every bulk copy already issued (chunks < c_waited + nslots) must land before the CTA and its shared
    // memory go away
    for (int cc = c_waited + 1; cc < min(c_last, c_waited + nslots); ++cc)
      mbar_wait(&full_bar[(cc - c_first) % nslots], (uint32_t)(((cc - c_first) / nslots) & 1));
  }
  __syncthreads();
  if (state) {   // carry over to (or report to) the next round
    if (tid == 0) state[0] = kept_total;
    unsigned long long* sr = reinterpret_cast<unsigned long long*>(state + 2);
    for (int w = tid; w < Wr; w += kScanThreads) sr[w] = removed[w];
  }
  if (!final_round) return;
  if (keep_pos)
    for (int j = kept_total + tid; j < max_out; j += kScanThreads) keep_pos[(int64_t)b * max_out + j] = -1;
  if (num_kept && tid == 0) num_kept[b] = kept_total;
}

// ---- wide scan: K too large for the shared-memory ring (K > ~12000) -------------------------------------------------
// The serial part of greedy NMS is only the 64x64 diagonal fixed point per chunk; the OR of the kept rows into the
// `removed` bitmap is spread over G co-resident CTAs (cooperative launch). CTA g owns words [g*S, (g+1)*S) of the bitmap:
// it consumes the keep words the owners of earlier chunks publish (acquire/release flags, up to 32 chunks per step),
// ORs those rows' words of its slice, then resolves its own S chunks one after the other and publishes them. The
// hand-over between owners costs one flag round trip per S chunks; everything else overlaps.
constexpr int kWideThreads = 256;
constexpr int kWideBatch = 32;   // chunks consumed per step
constexpr int kWideMaxS = 128;   // most bitmap words per CTA
struct WideSync {
  unsigned long long keep;   // kept rows of the chunk
  int32_t cum;               // boxes kept up to and including the chunk
  int32_t flag;              // 0 pending, 1 published, 2 published and final (max_out reached or last chunk)
};
__device__ __forceinline__ int32_t ld_acquire(const int32_t* p) {
  int32_t v;
  asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_release(int32_t* p, int32_t v) {
  asm volatile("st.release.gpu.global.s32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}

constexpr int kWidePrefetchMaxS = 16;   // S*64 rows x S words of the diagonal block in shared memory: 128 KB at S = 16
template <bool PREFETCH>
__global__ void __launch_bounds__(kWideThreads)
nms_scan_wide_kernel(const unsigned long long* __restrict__ mask, const unsigned long long* __restrict__ diagT,
                     const int32_t* __restrict__ num_valid, int K, int W, int Ws, int S, int max_out, WideSync* __restrict__ sync,
                     int32_t* __restrict__ keep_pos, int32_t* __restrict__ num_kept, int32_t* __restrict__ keep_flag,
                     int two_blocks) {
  extern __shared__ __align__(16) unsigned long long wide_smem[];
  unsigned long long* removed = wide_smem;        // [S] my slice of the bitmap
  // PREFETCH: my own diagonal block (rows of my chunks x words of my slice), fetched while the earlier owners work, so
  // that the one-chunk-at-a-time phase below never waits for global memory
  unsigned long long* dtile = wide_smem + ((S + 1) & ~1);   // [S][64] transposed diagonal tiles of my chunks
  unsigned long long* blk = dtile + (size_t)S * 64;         // [S*64][S]
  // two_blocks: also the previous owner's rows x my words, so that the hand-over (his last chunks -> my first fixed
  // point) does not wait for global memory either
  unsigned long long* blk2 = blk + (size_t)64 * S * S;      // [S*64][S]
  __shared__ unsigned long long kb_s[kWideMaxS];   // keep words of my own chunks
  __shared__ int32_t rows_s[kWideBatch * 64];     // kept rows of the chunks of this step
  __shared__ int32_t ctl[4];                      // [0] chunks ready, [1] stop seen, [2] kept rows listed, [3] kept_total
  const int b = blockIdx.y, g = blockIdx.x;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int n = num_valid ? min(num_valid[b], K) : K;
  const int Wn = (n + 63) / 64;
  const int lo = g * S, hi = min(lo + S, Wn);
  const int prev_row0 = (lo - S) * 64;
  const unsigned long long* mrow = mask + (int64_t)b * K * Ws;
  const unsigned long long* dimg = diagT + (int64_t)b * W * 64;
  WideSync* sy = sync + (int64_t)b * W;
  if (Wn == 0) {   // empty image: CTA 0 reports
    if (g == 0) {
      if (keep_pos)
        for (int j = tid; j < max_out; j += kWideThreads) keep_pos[(int64_t)b * max_out + j] = -1;
      if (num_kept && tid == 0) num_kept[b] = 0;
    }
    return;
  }
  if (lo >= Wn) return;
  for (int j = tid; j < S; j += kWideThreads) removed[j] = 0ull;
  if (keep_flag)
    for (int i = lo * 64 + tid; i < min(hi * 64, K); i += kWideThreads) keep_flag[(int64_t)b * K + i] = 0;
  if (g == 0 && keep_flag)   // boxes past the valid ones belong to nobody's chunks
    for (int i = Wn * 64 + tid; i < K; i += kWideThreads) keep_flag[(int64_t)b * K + i] = 0;
  if (tid == 0) ctl[3] = 0;
  const int Sw = hi - lo;   // live words of my slice
  for (int i = tid; i < Sw * 64; i += kWideThreads) dtile[i] = __ldg(&dimg[(size_t)lo * 64 + i]);
  if (PREFETCH) {
    const int nrows = Sw * 64;
    for (int i = tid; i < nrows * Sw; i += kWideThreads) {
      const int r = i / Sw, j = i - r * Sw;
      blk[(size_t)r * S + j] = __ldg(&mrow[(size_t)min(lo * 64 + r, K - 1) * Ws + lo + j]);
    }
    if (two_blocks && lo > 0)
      for (int i = tid; i < S * 64 * Sw; i += kWideThreads) {
        const int r = i / Sw, j = i - r * Sw;
        blk2[(size_t)r * S + j] = __ldg(&mrow[(size_t)(prev_row0 + r) * Ws + lo + j]);
      }
  }
  __syncthreads();

  // ---- phase A: chunks owned by earlier CTAs
  int c = 0;
  while (c < lo) {
    if (warp == 0) {
      int f, nready;
      do {   // the other warps wait at the barrier below; only this warp polls
        f = 0;
        if (c + lane < lo) f = ld_acquire(&sy[c + lane].flag);
        const uint32_t ready = __ballot_sync(0xffffffffu, f != 0);
        nready = (ready == 0xffffffffu) ? 32 : (__ffs((int)~ready) - 1);
      } while (nready == 0);
      unsigned long long kb = 0ull;
      if (lane < nready) kb = sy[c + lane].keep;
      const uint32_t stop = __ballot_sync(0xffffffffu, lane < nready && f == 2);
      // list the kept rows of the ready chunks
      const int cnt = __popcll(kb);
      int incl = cnt;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int v = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += v;
      }
      int base = incl - cnt;
      unsigned long long bits = kb;
      while (bits) {
        const int r = __ffsll((long long)bits) - 1;
        bits &= bits - 1ull;
        OD_DBG_IDX(base, kWideBatch * 64);
        rows_s[base++] = (c + lane) * 64 + r;
      }
      if (lane == 31) ctl[2] = incl;
      if (lane == 0) {
        ctl[0] = nready;
        ctl[1] = stop != 0u;
      }
      if (nready > 0 && lane == nready - 1) ctl[3] = sy[c + lane].cum;
    }
    __syncthreads();
    const int nready = ctl[0], nrows = ctl[2];
    const bool stop = ctl[1] != 0;
    if (stop) return;   // max_out was reached before my chunks: nothing left for me
    if (nready > 0 && nrows > 0) {
      // thread -> (word j of my slice, row lane q): consecutive threads read consecutive words of one row
      const int j = tid % Sw, q0 = tid / Sw, qstep = kWideThreads / Sw;
      if (q0 < qstep) {
        unsigned long long acc = 0ull;
        for (int q = q0; q < nrows; q += 8 * qstep) {   // eight independent loads in flight (DRAM latency ~1 us)
          unsigned long long v[8];
#pragma unroll
          for (int u = 0; u < 8; ++u) {
            const int qq = q + u * qstep;
            unsigned long long x = 0ull;
            if (qq < nrows) {
              const int row = rows_s[qq];
              x = (PREFETCH && two_blocks && row >= prev_row0) ? blk2[(size_t)(row - prev_row0) * S + j]
                                                                : __ldg(&mrow[(size_t)row * Ws + lo + j]);
            }
            v[u] = x;
          }
#pragma unroll
          for (int u = 0; u < 8; ++u) acc |= v[u];
        }
        OD_DBG_IDX(j, S);
        smem_or64(&removed[j], acc);
      }
    }
    __syncthreads();
    c += nready;
  }

  // ---- phase B: my own chunks, one at a time
  int kept_total = ctl[3];
  const int kept_before = kept_total;
  bool final_mine = false;
  for (c = lo; c < hi; ++c) {
    if (warp == 0) {
      const unsigned long long sup0 = dtile[(c - lo) * 64 + lane], sup1 = dtile[(c - lo) * 64 + lane + 32];
      const unsigned long long word = removed[c - lo];
      const bool cand0 = (c * 64 + lane < n) && !((word >> lane) & 1ull);
      const bool cand1 = (c * 64 + lane + 32 < n) && !((word >> (lane + 32)) & 1ull);
      unsigned long long kept = (unsigned long long)__ballot_sync(0xffffffffu, cand0) |
                                ((unsigned long long)__ballot_sync(0xffffffffu, cand1) << 32);
      for (int it = 0; it < 64; ++it) {
        const bool k0 = cand0 && !(sup0 & kept);
        const bool k1 = cand1 && !(sup1 & kept);
        const unsigned long long nk = (unsigned long long)__ballot_sync(0xffffffffu, k0) |
                                      ((unsigned long long)__ballot_sync(0xffffffffu, k1) << 32);
        if (nk == kept) break;
        kept = nk;
      }
      const int allow = max_out - kept_total;
      while (__popcll(kept) > allow) kept &= ~(1ull << (63 - __clzll((long long)kept)));
      OD_DBG_IDX(c - lo, kWideMaxS);
      if (lane == 0) kb_s[c - lo] = kept;   // (kb_s has kWideBatch >= S entries when the results are buffered)
    }
    __syncthreads();
    const unsigned long long kept = kb_s[c - lo];
    kept_total += __popcll(kept);
    if (kept_total >= max_out || c == Wn - 1) {   // the final chunk is mine
      final_mine = true;
      ++c;
      break;
    }
    // OR my kept rows into the rest of my slice (words c+1-lo .. Sw-1)
    const int live = hi - c - 1;
    if (kept != 0ull && live > 0) {
      if (PREFETCH) {
        // a warp per word, a lane per row (two rows each): OR-reduce across the warp, no atomics
        const bool r0 = (kept >> lane) & 1ull, r1 = (kept >> (lane + 32)) & 1ull;
        for (int j = warp; j < live; j += kWideThreads / 32) {
          const unsigned long long* col = blk + (size_t)((c - lo) * 64) * S + c + 1 - lo + j;
          const unsigned long long v = (r0 ? col[(size_t)lane * S] : 0ull) | (r1 ? col[(size_t)(lane + 32) * S] : 0ull);
          const uint32_t vlo = __reduce_or_sync(0xffffffffu, (uint32_t)v), vhi = __reduce_or_sync(0xffffffffu, (uint32_t)(v >> 32));
          if (lane == 0) removed[c + 1 - lo + j] |= ((unsigned long long)vhi << 32) | vlo;
        }
      } else {
        const int j = tid % live, q0 = tid / live, qstep = kWideThreads / live;
        if (q0 < qstep) {
          unsigned long long acc = 0ull;
          for (int r = q0; r < 64; r += qstep)
            if ((kept >> r) & 1ull) acc |= __ldg(&mrow[(size_t)(c * 64 + r) * Ws + c + 1 + j]);
          OD_DBG_IDX(c + 1 - lo + j, S);
          smem_or64(&removed[c + 1 - lo + j], acc);
        }
      }
    }
    __syncthreads();
  }
  // My chunks lo .. c-1 are resolved (keep words in kb_s): publish them together - a release per chunk would sit on the
  // critical path - then write the outputs, which nobody waits for.
  const int done = c - lo;
  if (tid < done) {
    int cum = kept_before;
    for (int i = 0; i <= tid; ++i) cum += __popcll(kb_s[i]);
    sy[lo + tid].keep = kb_s[tid];
    sy[lo + tid].cum = cum;
    st_release(&sy[lo + tid].flag, (final_mine && tid == done - 1) ? 2 : 1);
  }
  for (int i = warp; i < done; i += kWideThreads / 32) {
    int base = kept_before;
    for (int q = 0; q < i; ++q) base += __popcll(kb_s[q]);
    const unsigned long long kept = kb_s[i];
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int r = lane + 32 * h;
      if ((kept >> r) & 1ull) {
        const int pos = base + __popcll(kept & ((1ull << r) - 1ull));
        OD_DBG_IDX(pos, max_out);
        OD_DBG_IDX((lo + i) * 64 + r, K);
        if (keep_pos) keep_pos[(int64_t)b * max_out + pos] = (lo + i) * 64 + r;
        if (keep_flag) keep_flag[(int64_t)b * K + (lo + i) * 64 + r] = 1;
      }
    }
  }
  if (final_mine) {
    if (keep_pos)
      for (int j = kept_total + tid; j < max_out; j += kWideThreads) keep_pos[(int64_t)b * max_out + j] = -1;
    if (num_kept && tid == 0) num_kept[b] = kept_total;
  }
}

// int32 words of per-image scan state for the two-round NMS: kept count (+ pad) and the removed bitmap
static int64_t scan_state_stride(int64_t W) { return 2 + 2 * ((W + 15) & ~(int64_t)15); }

size_t nms_sorted_workspace_bytes(int64_t B, int64_t K) {
  const int64_t W = (K + 63) / 64, Ws = nms_mask_stride(K);
  Workspace w(nullptr, 0);
  w.take<unsigned long long>((size_t)(B * K * Ws));
  w.take<unsigned long long>((size_t)(B * W * 64));
  w.take<unsigned long long>((size_t)(B * scan_state_stride(W) / 2 + 1));
  w.take<WideSync>((size_t)(B * W + 1));
  return w.off + 256;
}

// Words of the bitmap per CTA of the wide scan so that all B * ceil(W / S) CTAs are co-resident; 0 = not possible.
// *prefetch: the slice is small enough for the diagonal block to live in shared memory.
static size_t wide_scan_smem(int S, int blocks) {   // blocks of S*64 rows x S words staged in shared memory: 0, 1 or 2
  return ((size_t)((S + 1) & ~1) + (size_t)64 * S + (size_t)blocks * 64 * S * S) * sizeof(unsigned long long);
}
static int wide_scan_blocks(int S) { return wide_scan_smem(S, 2) <= 200 * 1024 ? 2 : 1; }
static int wide_scan_slice(int64_t B, int W, bool* prefetch) {
  int dev = 0, sms = 0, coop = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess ||
      cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, dev) != cudaSuccess || !coop)
    return 0;
  for (int pf = 1; pf >= 0; --pf) {
    // with the block in shared memory one CTA per SM is the plan; without it, whatever fits
    int occ = 1;
    if (!pf && cudaFuncSetAttribute(nms_scan_wide_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                    (int)wide_scan_smem(kWideMaxS, 0)) != cudaSuccess)
      return 0;
    if (!pf && cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, nms_scan_wide_kernel<false>, kWideThreads, wide_scan_smem(kWideMaxS, 0)) != cudaSuccess)
      return 0;
    const int64_t per_image = ((int64_t)sms * occ) / B;
    if (per_image < 1) continue;
    int64_t G = (W + 3) / 4;   // at least four words per CTA
    if (G > per_image) G = per_image;
    const int S = (int)((W + G - 1) / G);
    if (pf) {
      if (S > kWidePrefetchMaxS) continue;
      const size_t smem = wide_scan_smem(S, wide_scan_blocks(S));
      static const size_t wide_static = static_smem_bytes((const void*)nms_scan_wide_kernel<true>);
      if (smem + wide_static > 48 * 1024 &&
          cudaFuncSetAttribute(nms_scan_wide_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess)
        continue;
      if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, nms_scan_wide_kernel<true>, kWideThreads, smem) != cudaSuccess || occ < 1)
        continue;
    } else if (S > kWideMaxS) {
      continue;
    }
    *prefetch = pf != 0;
    return S;
  }
  return 0;
}

static int scan_round_launch(const unsigned long long* mask, const unsigned long long* diagT, const int32_t* num_valid,
                             int64_t B, int64_t K, int64_t mask_stride, int64_t max_out, int c_begin, int c_end,
                             int final_round, int32_t* scan_state, int32_t* keep_pos, int32_t* num_kept, int32_t* keep_flag,
                             WideSync* wide, cudaStream_t st) {
  const int W = (int)((K + 63) / 64), Ws = (int)mask_stride;
  if (Ws < W) OD_FAIL(OD_ERR_PARAM, "NMS mask stride %d < %d words", Ws, W);
  const size_t plain = (size_t)((W + 15) & ~15) * sizeof(unsigned long long);
  const size_t per_slot = ((size_t)64 * Ws + 64) * sizeof(unsigned long long);
  const size_t kSmemBudget = 200 * 1024;
  const int stride = (int)scan_state_stride(W);
  int nslots = 0;
  bool wide_prefetch = false;
  int wide_S = 0;
  if (W > 0 && Ws % 2 == 0 && reinterpret_cast<uintptr_t>(mask) % 16 == 0 && reinterpret_cast<uintptr_t>(diagT) % 16 == 0 &&
      plain + 2 * per_slot <= kSmemBudget) {
    nslots = (int)((kSmemBudget - plain) / per_slot);
    if (nslots > kScanMaxSlots) nslots = kScanMaxSlots;
    // short rows (DetectionLayer: K = 1000): four slots are plenty, and a 35 KB CTA disturbs the kernels it shares the
    // SMs with less than a 70 KB one (14x14 ROIAlign next to it: 118.1 -> 117.5 us)
    if (W <= 32 && nslots > 4) nslots = 4;
  }
  if (nslots >= 2) {
    const size_t smem = plain + (size_t)nslots * per_slot;
    static const size_t staged_static = static_smem_bytes((const void*)nms_scan_kernel<true>);
    if (smem + staged_static > 48 * 1024)
      OD_CUDA(cudaFuncSetAttribute(nms_scan_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    OD_CUDA(launch_pdl(nms_scan_kernel<true>, dim3((unsigned)B), dim3(kScanThreads), smem, st, mask, diagT, num_valid, (int)K, W, Ws, nslots, (int)max_out,
                                                                   c_begin, c_end, final_round, scan_state, stride, keep_pos,
                                                                   num_kept, keep_flag));
  } else if (wide && !scan_state && c_begin == 0 && c_end >= W && W >= 64 && (wide_S = wide_scan_slice(B, W, &wide_prefetch)) > 0) {
    // too many boxes for the ring: spread the OR phase over co-resident CTAs
    int S = wide_S, Ki = (int)K, mo = (int)max_out;
    const dim3 grid((unsigned)((W + S - 1) / S), (unsigned)B);
    OD_CUDA(cudaMemsetAsync(wide, 0, (size_t)B * W * sizeof(WideSync), st));
    int Wi = W, Wsi = Ws;
    const int blocks = wide_prefetch ? wide_scan_blocks(S) : 0;
    int two = blocks == 2;
    void* args[] = {(void*)&mask, (void*)&diagT, (void*)&num_valid, &Ki, &Wi, &Wsi, &S, &mo, &wide, &keep_pos, &num_kept, &keep_flag, &two};
    OD_CUDA(cudaLaunchCooperativeKernel(wide_prefetch ? (const void*)nms_scan_wide_kernel<true> : (const void*)nms_scan_wide_kernel<false>,
                                        grid, dim3(kWideThreads), args, wide_scan_smem(S, blocks), st));
    OD_LAUNCH_CHECK("nms_scan_wide_kernel");
    return OD_OK;
  } else {
    const size_t smem = plain > 0 ? plain : 128;
    static const size_t unstaged_static = static_smem_bytes((const void*)nms_scan_kernel<false>);
    if (smem + unstaged_static > 48 * 1024)
      OD_CUDA(cudaFuncSetAttribute(nms_scan_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    nms_scan_kernel<false><<<(unsigned)B, kScanThreads, smem, st>>>(mask, diagT, num_valid, (int)K, W, Ws, 0, (int)max_out, c_begin,
                                                                    c_end, final_round, scan_state, stride, keep_pos, num_kept,
                                                                    keep_flag);
  }
  OD_LAUNCH_CHECK("nms_scan_kernel");
  return OD_OK;
}

int nms_sorted_launch(const float4* boxes, const int32_t* num_valid, const int32_t* group, int64_t B, int64_t K,
                      float thr, int64_t max_out, int32_t* keep_pos, int32_t* num_kept, int32_t* keep_flag,
                      void* ws, size_t ws_bytes, cudaStream_t st) {
  if (B == 0) return OD_OK;
  if (B > 65535) OD_FAIL(OD_ERR_PARAM, "NMS batch %lld > 65535", (long long)B);
  if (K >= (1 << 22)) OD_FAIL(OD_ERR_PARAM, "NMS supports < 4M boxes per image");
  const int W = (int)((K + 63) / 64), Ws = (int)nms_mask_stride(K);
  Workspace w(ws, ws_bytes);
  unsigned long long* mask = w.take<unsigned long long>((size_t)(B * K * Ws));
  unsigned long long* diagT = w.take<unsigned long long>((size_t)(B * W * 64));
  int32_t* state = reinterpret_cast<int32_t*>(w.take<unsigned long long>((size_t)(B * scan_state_stride(W) / 2 + 1)));
  WideSync* wide = w.take<WideSync>((size_t)(B * W + 1));
  if (!ws || !w.ok()) OD_FAIL(OD_ERR_WORKSPACE, "NMS workspace %zu < %zu bytes", ws_bytes, w.off);
  if (K == 0)
    return scan_round_launch(mask, diagT, num_valid, B, K, Ws, max_out, 0, 0, 1, nullptr, keep_pos, num_kept, keep_flag, nullptr, st);
  if (W > 65535) OD_FAIL(OD_ERR_PARAM, "NMS tile grid too large");
  // Two rounds when far fewer boxes are wanted than offered (proposals: 1000 of 6000): the first round covers the row
  // chunks that normally suffice (1.5 x max_out boxes); the second one - the remaining rows - returns at once on the
  // device if max_out boxes are already kept. Costs two nearly empty launches, saves up to ~55 % of the pair tests.
  int c1 = (int)((max_out + max_out / 2 + 63) / 64);
  const bool two_rounds = c1 + 8 <= W;
  if (!two_rounds) c1 = W;
  const int stride = (int)scan_state_stride(W);
  for (int round = 0; round < (two_rounds ? 2 : 1); ++round) {
    const int rb0 = round == 0 ? 0 : c1, rb1 = round == 0 ? c1 : W;
    const dim3 grid((unsigned)((W - rb0 + kMaskColTiles - 1) / kMaskColTiles), (unsigned)(rb1 - rb0), (unsigned)B);
    const int32_t* st_in = round == 0 ? nullptr : state;
    if (thr >= 0.0f)
      OD_CUDA(launch_pdl(nms_mask_kernel<true>, grid, dim3(kMaskThreads), 0, st, boxes, num_valid, group, (int)K, W, rb0, thr, (int)max_out, st_in,
                                                           stride, Ws, mask, diagT));
    else
      OD_CUDA(launch_pdl(nms_mask_kernel<false>, grid, dim3(kMaskThreads), 0, st, boxes, num_valid, group, (int)K, W, rb0, thr, (int)max_out, st_in,
                                                            stride, Ws, mask, diagT));
    OD_LAUNCH_CHECK("nms_mask_kernel");
    OD_CHECK(scan_round_launch(mask, diagT, num_valid, B, K, Ws, max_out, rb0, rb1, round == (two_rounds ? 1 : 0),
                               two_rounds ? state : nullptr, keep_pos, num_kept, keep_flag, wide, st));
  }
  return OD_OK;
}

int nms_scan_launch(const unsigned long long* mask, const unsigned long long* diagT, const int32_t* num_valid, int64_t B,
                    int64_t K, int64_t mask_stride, int64_t max_out, int32_t* keep_pos, int32_t* num_kept,
                    int32_t* keep_flag, cudaStream_t st) {
  const int W = (int)((K + 63) / 64);
  return scan_round_launch(mask, diagT, num_valid, B, K, mask_stride, max_out, 0, W, 1, nullptr, keep_pos, num_kept,
                           keep_flag, nullptr, st);
}

// ---- unsorted front-end (tf.image.non_max_suppression on arbitrary score order)
__global__ void nms_build_keys_kernel(const float* __restrict__ scores, const int32_t* __restrict__ num_valid, int K,
                                      int64_t n_pow2, unsigned long long* __restrict__ keys) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int b = blockIdx.y;
  if (i >= n_pow2) return;
  const int n = num_valid ? min(num_valid[b], K) : K;
  keys[(int64_t)b * n_pow2 + i] = (i < n) ? composite_key(scores[(int64_t)b * K + i], (uint32_t)i) : 0ull;
}
__global__ void nms_gather_sorted_kernel(const float4* __restrict__ boxes, const unsigned long long* __restrict__ keys,
                                         const int32_t* __restrict__ num_valid, int K, int64_t n_pow2,
                                         float4* __restrict__ sorted) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int b = blockIdx.y;
  const int n = num_valid ? min(num_valid[b], K) : K;
  if (i >= K) return;
  sorted[(int64_t)b * K + i] =
      (i < n) ? boxes[(int64_t)b * K + composite_index(keys[(int64_t)b * n_pow2 + i])] : make_float4(0.f, 0.f, 0.f, 0.f);
}
__global__ void nms_map_back_kernel(const unsigned long long* __restrict__ keys, int64_t n_pow2, int max_out,
                                    int32_t* __restrict__ keep) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  const int b = blockIdx.y;
  if (j >= max_out) return;
  const int32_t pos = keep[(int64_t)b * max_out + j];
  if (pos >= 0) keep[(int64_t)b * max_out + j] = (int32_t)composite_index(keys[(int64_t)b * n_pow2 + pos]);
}

}  // namespace od

using namespace od;

extern "C" {

size_t od_nms_workspace_bytes(int64_t batch, int64_t num_boxes) {
  Workspace w(nullptr, 0);
  w.take<unsigned long long>((size_t)(batch * next_pow2(num_boxes > 0 ? num_boxes : 1)));
  w.take<float4>((size_t)(batch * num_boxes));
  return w.off + 256 + nms_sorted_workspace_bytes(batch, num_boxes);
}

int od_nms(const DLTensor* boxes, const DLTensor* scores, const DLTensor* num_valid, float iou_threshold,
           int64_t max_out, DLTensor* keep_idx, DLTensor* num_kept, void* ws, size_t ws_bytes, void* stream) {
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  DeviceScope scope;
  OD_CHECK(check_tensor(boxes, "boxes", F32, {kAny, kAny, 4}, 16, scope));
  const int64_t B = boxes->shape[0], K = boxes->shape[1];
  OD_CHECK(check_tensor(scores, "scores", F32, {B, K}, 4, scope));
  if (max_out < 0) OD_FAIL(OD_ERR_SHAPE, "keep_idx: max_out = %lld is negative", (long long)max_out);
  OD_CHECK(check_tensor(keep_idx, "keep_idx", I32, {B, max_out}, 4, scope));
  OD_CHECK(check_opt_tensor(num_valid, "num_valid", I32, {B}, 4, scope));
  OD_CHECK(check_opt_tensor(num_kept, "num_kept", I32, {B}, 4, scope));
  if (B == 0 || max_out == 0) return OD_OK;
  if (!ws) OD_FAIL(OD_ERR_WORKSPACE, "NMS workspace is NULL");
  const int64_t n_pow2 = next_pow2(K > 0 ? K : 1);
  Workspace w(ws, ws_bytes);
  unsigned long long* keys = w.take<unsigned long long>((size_t)(B * n_pow2));
  float4* sorted = w.take<float4>((size_t)(B * K));
  w.off = align_up(w.off, 256);
  if (!w.ok() || ws_bytes < w.off + nms_sorted_workspace_bytes(B, K) - 256)
    OD_FAIL(OD_ERR_WORKSPACE, "NMS workspace %zu bytes too small", ws_bytes);
  const int32_t* nv = dptr<int32_t>(num_valid);
  {
    const dim3 g((unsigned)((n_pow2 + 255) / 256), (unsigned)B);
    nms_build_keys_kernel<<<g, 256, 0, st>>>(dptr<float>(scores), nv, (int)K, n_pow2, keys);
    OD_LAUNCH_CHECK("nms_build_keys_kernel");
  }
  OD_CHECK(sort_u64_desc_launch(keys, B, n_pow2, st));
  if (K > 0) {
    const dim3 g((unsigned)((K + 255) / 256), (unsigned)B);
    nms_gather_sorted_kernel<<<g, 256, 0, st>>>(dptr<float4>(boxes), keys, nv, (int)K, n_pow2, sorted);
    OD_LAUNCH_CHECK("nms_gather_sorted_kernel");
  }
  OD_CHECK(nms_sorted_launch(sorted, nv, nullptr, B, K, iou_threshold, max_out, dptr<int32_t>(keep_idx),
                             dptr<int32_t>(num_kept), nullptr, w.base + w.off, ws_bytes - w.off, st));
  {
    const dim3 g((unsigned)((max_out + 255) / 256), (unsigned)B);
    nms_map_back_kernel<<<g, 256, 0, st>>>(keys, n_pow2, (int)max_out, dptr<int32_t>(keep_idx));
    OD_LAUNCH_CHECK("nms_map_back_kernel");
  }
  return OD_OK;
}

}  // extern "C"
