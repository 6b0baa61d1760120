// CIDEr-D of id captions against a reference corpus (recnet_cider_d; coco-caption's CiderScorer / CiderD with n = 4, sigma = 6).
// One warp per candidate row.  The row's caption (<= 64 ids) and its n-gram keys live in shared memory at fixed slots: order n
// (0-based) at [64 n, 64 n + 64), slot 64 n + i = the n-gram starting at word i.  Lane l owns slots l + 32 j, j = 0..7, so slots j
// and j + 1 of a lane are of order j / 2.  Each lane keeps, for the first occurrence of each of its n-grams, the key and the hypothesis
// weight count * (ref_len - log df) in registers; every reference of the row's video is staged into shared memory (when it fits) and
// binary-searched for those keys.  Each lane sums its share of every reference's cosine terms, already divided by the two norms and
// scaled by the length penalty; one butterfly reduction at the end gives the score, so the result does not depend on timing.
#pragma once
#include "common.cuh"

namespace cider {

constexpr int kMaxSteps = 64;             // the sampler's own limit on max_steps
constexpr int kStage = 256;               // reference entries staged in shared memory (4 * 65 - 6 fit: any reference of <= 65 words)
constexpr int kSlots = 4 * kMaxSteps;     // n-gram slots of a candidate
constexpr float kInvTwoSigmaSq = 1.0f / 72.0f;

// First index in a[0, n) whose key is >= k (n when there is none).
__device__ __forceinline__ int lower_bound(const uint64_t* a, int n, uint64_t k) {
  int lo = 0;
  while (n > 0) {
    const int half = n >> 1;
    if (a[lo + half] < k) { lo += half + 1; n -= half + 1; }
    else n = half;
  }
  return lo;
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

__global__ void __launch_bounds__(32) cider_d_kernel(recnet_cider_corpus c, const long long* __restrict__ ids, long long ld_step,
                                                      long long ld_row, int steps, const int* __restrict__ video_of_row,
                                                      long long eos_id, float* __restrict__ scores) {
  __shared__ int s_ids[kMaxSteps];
  __shared__ uint64_t s_keys[kSlots];
  __shared__ uint64_t s_ref_keys[kStage];
  __shared__ float s_ref_w[kStage];
  const int row = blockIdx.x, lane = threadIdx.x;

  // 1. the caption: ids before the first eos_id / <PAD> / negative id; an id above 65535 cannot be keyed and makes the score NaN
  bool stop[2], big[2];
#pragma unroll
  for (int h = 0; h < 2; ++h) {
    const int t = lane + 32 * h;
    const long long v = t < steps ? ids[t * ld_step + row * ld_row] : 0;
    stop[h] = v == eos_id || v <= 0;
    big[h] = v > 0xffff;
    s_ids[t] = (int)(v & 0xffff);
  }
  const unsigned m0 = __ballot_sync(0xffffffffu, stop[0]), m1 = __ballot_sync(0xffffffffu, stop[1]);
  const int len = m0 ? __ffs(m0) - 1 : (m1 ? 32 + __ffs(m1) - 1 : kMaxSteps);
  const bool too_big = __any_sync(0xffffffffu, (big[0] && lane < len) || (big[1] && lane + 32 < len));
  const int vid = video_of_row[row];
  if (too_big || vid < 0 || vid >= c.n_videos) {
    if (lane == 0) scores[row] = __int_as_float(0x7fc00000);
    return;
  }
  __syncwarp();

  // 2. n-gram keys of every slot
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const int s = lane + 32 * j, n = j >> 1, i = s & 63;
    uint64_t k = 0;
    if (i + n < len)
      for (int q = 0; q <= n; ++q) k |= (uint64_t)s_ids[i + q] << (48 - 16 * q);
    s_keys[s] = k;
  }
  __syncwarp();

  // 3. counts and df of the first occurrence of each n-gram -> hypothesis weights and the squared norms of this lane's share
  uint64_t key[8];
  float wh[8], nsq[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const int s = lane + 32 * j, n = j >> 1, i = s & 63;
    key[j] = 0;
    wh[j] = 0.f;
    if (i + n >= len) continue;
    const uint64_t k = s_keys[s];
    const uint64_t* blk = s_keys + 64 * n;
    bool first = true;
    int count = 0;
    for (int q = 0; q + n < len; ++q) {
      const bool eq = blk[q] == k;
      count += eq;
      first &= !(eq && q < i);
    }
    if (!first) continue;
    const int d = lower_bound(c.df_keys, c.n_df, k);
    const float lg = (d < c.n_df && c.df_keys[d] == k) ? c.df_log[d] : 0.f;
    key[j] = k;
    wh[j] = (float)count * (c.ref_len - lg);
    nsq[n] += wh[j] * wh[j];
  }
  float norm_h[4];
#pragma unroll
  for (int n = 0; n < 4; ++n) norm_h[n] = sqrtf(warp_sum(nsq[n]));
  const int length_h = len > 1 ? len - 1 : 0;

  // 4. every reference of the video: sum over this lane's n-grams of min(w_h, w_r) * w_r, per order, divided by the norms
  const int r0 = c.video_refs[vid], r1 = c.video_refs[vid + 1];
  float acc = 0.f;
  for (int r = r0; r < r1; ++r) {
    const int e0 = c.ref_entries[r], ne = c.ref_entries[r + 1] - e0;
    const uint64_t* rk = c.entry_keys + e0;
    const float* rw = c.entry_w + e0;
    if (ne <= kStage) {
      __syncwarp();
      for (int e = lane; e < ne; e += 32) { s_ref_keys[e] = rk[e]; s_ref_w[e] = rw[e]; }
      __syncwarp();
      rk = s_ref_keys;
      rw = s_ref_w;
    }
    float part[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      if (key[j] == 0) continue;
      const int e = lower_bound(rk, ne, key[j]);
      if (e < ne && rk[e] == key[j]) {
        const float wr = rw[e];
        part[j >> 1] += fminf(wh[j], wr) * wr;
      }
    }
    const float delta = (float)(length_h - c.ref_length[r]);
    const float pen = expf(-delta * delta * kInvTwoSigmaSq);
#pragma unroll
    for (int n = 0; n < 4; ++n) {
      const float nr = c.ref_norm[4 * r + n];
      const float v = (norm_h[n] != 0.f && nr != 0.f) ? part[n] / (norm_h[n] * nr) : part[n];
      acc += v * pen;
    }
  }
  acc = warp_sum(acc);
  if (lane == 0) scores[row] = r1 > r0 ? 10.f * acc / (4.f * (float)(r1 - r0)) : 0.f;
}

inline int launch(const recnet_cider_corpus& c, const long long* ids, long long ld_step, long long ld_row, int steps, int n_rows,
                  const int* video_of_row, long long eos_id, float* scores, cudaStream_t st) {
  cider_d_kernel<<<n_rows, 32, 0, st>>>(c, ids, ld_step, ld_row, steps, video_of_row, eos_id, scores);
  RN_LAUNCH_OK();
  return 0;
}

}  // namespace cider
