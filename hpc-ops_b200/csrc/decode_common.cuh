// Definitions shared by the paged decode attention kernels (fp8: decode_attn_fp8.cu, bf16:
// decode_attn_bf16.cu): task-map rows, kernel parameters, the split-k combine launcher.
#pragma once
#include "common.cuh"
#include "host_utils.h"

namespace b200 {
namespace decode {

constexpr int kTileN = 128;  // keys per tile == UMMA M
constexpr int kPage = 64;    // paged block size (tokens) of the fp8 caches
constexpr int kD = 128;      // head dim
constexpr int kTaskStride = 12;
constexpr int kSoftmaxBar = 1;

struct Params {
  const int* task_map;
  const int* block_ids;
  const float* qscale;
  const float* kscale;
  const float* vscale;
  float* split_out;
  float* lse;
  __nv_bfloat16* y;  // final output: tasks that are the only chunk of their (batch, kv head) write it directly
  int ld_y;
  int num_batch;
  int num_seq_q;
  int num_head_q;
  int num_head_kv;
  int group;
  int num_seq_max_blocks;
  int qscale_stride;
  int max_splitk;
  int lse_pad;
  int k_head_first;  // TMA dim order of the cache maps: (d, head, token, blk) or (d, token, head, blk)
  int v_head_first;
  float softmax_scale_log2;
  // k-per-token variant: in-cache scale rows (SURVEY.md Appendix A): float index
  //   blk * ks_blk + (t / 32) * ks_row + head * ks_head + t % 32     (t = token slot in the page)
  long long ks_blk, ks_row, ks_head;
  int rotate;  // walk each bin from the tile whose position on the per-head line is 0 (mod P)
  int kv_policy;  // L2 policy of the K/V loads: 0 evict_first, 1 evict_normal, 2 evict_last
  // fp8 kernel, dense token-major caches under the rotated walk: page-wide L2 prefetch pf_dist
  // tiles ahead (< 0: off). Page blk of K (all heads) is [pf_k + blk * pf_k_blk, + pf_bytes).
  int pf_dist;
  uint32_t pf_bytes;
  const uint8_t* pf_k;
  const uint8_t* pf_v;
  long long pf_k_blk, pf_v_blk;
};

struct Task {
  int ihead_kv, ibatch, ichunk, iseq_start;
  int num_seqkv, num_seqkvcache, num_tile_kv, num_tile_full;
  int is_causal;
};

__device__ __forceinline__ bool load_task(const int* row, Task& t) {
  int4 a = *reinterpret_cast<const int4*>(row);
  if (a.x < 0 || a.y < 0) return false;
  int4 b = *reinterpret_cast<const int4*>(row + 4);
  int c = row[8];
  t.ihead_kv = a.x;
  t.ibatch = a.y;
  t.ichunk = a.z;
  t.iseq_start = a.w;
  t.num_seqkv = b.x;
  t.num_seqkvcache = b.y;
  t.num_tile_kv = b.z;
  t.num_tile_full = b.w;
  t.is_causal = c;
  return true;
}

// ---- rotated bin walk -------------------------------------------------------------------------
// The task line lays the tiles of one kv head after those of the previous one, and bin i owns
// tiles [i P, (i+1) P) of it. Walked front to back, two CTAs that stream the same pages for
// neighbouring heads do so (TB mod P) tiles apart in time. With a token-major (NHD) cache the rows
// of neighbouring heads are neighbours in memory (128-byte runs), so the DRAM sees half-used
// 256-byte granules. Rotated so that every CTA processes, at step t, the tile whose position on
// its head's line is t (mod P), all heads of a page are streamed at the same time: the 256-byte L2
// promotion of one head's load is the other head's prefetch. The task a walk starts inside of is
// processed in two parts (its tail first, its head last) with the online-softmax state carried in
// registers in between; every task is still written exactly once, to the chunk slot the task map
// gives it. TB (tiles per head) is header int 6, written by both schedulers of this library; a
// map without it is walked front to back.
struct BinWalk {
  int m;   // task rows to visit (upper bound when the walk is not rotated: a terminator ends it)
  int ks;  // row the walk starts in
  int o;   // first tile of that row to process (0: the walk starts at a task boundary)
};

__device__ __forceinline__ int walk_start(const int* task_map, int icta) {
  const int P = task_map[0] - 1;
  const int TB = task_map[6];
  if (TB <= 0 || P <= 0) return 0;
  const long long x0 = static_cast<long long>(icta) * P;
  const int c = static_cast<int>((x0 % TB) % P);
  return (P - c) % P;
}

// Whole-warp scan of a bin's rows (tile counts in int 6 of each row): finds the row and tile the
// walk starts at and the number of rows. All results are warp-uniform.
__device__ __forceinline__ BinWalk scan_bin(const int* bin, int max_rows, int u0, int lane) {
  BinWalk w;
  w.m = max_rows;
  w.ks = 0;
  w.o = 0;
  if (u0 <= 0) return w;  // front to back: rows are read until the terminator
  w.m = 0;
  int before = 0;
  bool found = false;
  for (int base = 0; base < max_rows; base += 32) {
    const int i = base + lane;
    int c = 0;
    bool valid = false;
    if (i < max_rows) {
      const int* row = bin + static_cast<long long>(i) * kTaskStride;
      const int2 hb = *reinterpret_cast<const int2*>(row);
      valid = hb.x >= 0 && hb.y >= 0;
      if (valid) c = row[6];
    }
    const unsigned vm = __ballot_sync(0xffffffffu, valid);
    const int cnt = (vm == 0xffffffffu) ? 32 : __ffs(~vm) - 1;  // leading valid rows
    if (lane >= cnt) c = 0;
    int s = c;  // inclusive prefix sum of the tile counts
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const int v = __shfl_up_sync(0xffffffffu, s, d);
      if (lane >= d) s += v;
    }
    const int excl = before + s - c;
    const bool hit = (lane < cnt) && (u0 >= excl) && (u0 < excl + c);
    const unsigned hm = __ballot_sync(0xffffffffu, hit);
    if (hm != 0u && !found) {
      const int src = __ffs(hm) - 1;
      w.ks = base + src;
      w.o = u0 - __shfl_sync(0xffffffffu, excl, src);
      found = true;
    }
    before += __shfl_sync(0xffffffffu, s, 31);
    w.m += cnt;
    if (cnt < 32) break;
  }
  if (!found) {  // a short bin (the last one): front to back
    w.ks = 0;
    w.o = 0;
  }
  return w;
}

// Segment j of a walk: row index, tile range, and whether the softmax state is carried over.
struct Segment {
  int row;
  int tb, te;    // tiles [tb, te) of the row's task (te < 0: up to the task's last tile)
  bool save;     // first part of the split task: keep the state, write nothing
  bool restore;  // second part: continue from the kept state
};
__device__ __forceinline__ int num_segments(const BinWalk& w) { return w.m + (w.o > 0 ? 1 : 0); }
__device__ __forceinline__ Segment segment_of(const BinWalk& w, int j) {
  Segment s;
  int r = w.ks + j;
  if (r >= w.m) r -= w.m;
  s.row = r;
  s.tb = (j == 0) ? w.o : 0;
  s.te = (j == w.m) ? w.o : -1;
  s.save = (w.o > 0) && (j == 0);
  s.restore = (j == w.m);
  return s;
}

// split-k combine (decode_attn_fp8.cu): y = sum_c 2^(lse_c - m) O_c / sum_c 2^(lse_c - m) -> bf16;
// (batch, kv head) pairs with a single chunk were written by the attention kernel itself.
cudaError_t launch_combine(__nv_bfloat16* y, const float* split_out, const float* lse,
                           const int* task_map, int num_batch, int num_seq_q, int num_head_q,
                           int num_head_kv, int group, int max_splitk, int lse_pad, int ldY,
                           cudaStream_t stream);

}  // namespace decode
}  // namespace b200
