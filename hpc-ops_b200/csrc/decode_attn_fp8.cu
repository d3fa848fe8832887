// FP8 paged decode attention, q-per-token/per-head scale, k/v per-tensor scale, dynamic split-k
// task map. B200 (sm_100a) design, written from scratch:
//
//   * persistent grid = num_total_ctas (one CTA per SM); each CTA walks its bin of the task map
//   * warp 0  : TMA producer  - K/V 64-token pages -> 128B-swizzled smem ring (12 x 16 KB slots),
//                               Q rows of the task -> smem (double buffered)
//   * warp 1  : tcgen05 issuer - S^T[128 keys, NQ] = K_tile . Q^T     (kind::f8f6f4, K-major A/B)
//                                O^T[128 d, NQ]   = V_tile^T . P^T    (MN-major A and B: V is
//                                consumed exactly as it lies in the cache, no byte transpose)
//   * warps 2-5: softmax      - one thread per key: TMEM->regs, scale/mask, online softmax in the
//                               log2 domain, P*256 -> e4m3 -> smem, O tile TMEM->regs accumulate
//   accumulators live in TMEM (S^T and O^T double buffered, 4*NQ columns).
//
// Semantics follow reference
//   src/attention/decode/sm90/dynamic/smallm_fp8_qpertoken_perhead_kvpertensor_dim128_dynamic_splitk_kernels.cuh:29-437
//   src/attention/decode/sm90/util_kernels.cuh:280-305 (mask), :332-436 (online softmax),
//   :523-602 (final), :638-660 (lse)
// and the launcher contract of
//   src/attention/decode/decode.h:28-37 (attention_decode_fp8_async).
#include <cstdlib>

#include "decode_common.cuh"

namespace b200 {
namespace decode {

constexpr int kSlotBytes = kTileN * kD;  // 16 KB (fp8)
constexpr int kThreads = 192;

constexpr int kNumStages = 6;                 // (K tile + V tile) stages of 32 KB
constexpr int kStageBytes = 2 * kSlotBytes;

template <int NQ>
struct Smem {
  static constexpr int kPPlanes = NQ / 16;
  static constexpr int kPBytes = kPPlanes * kTileN * 16;  // one P buffer
  static constexpr int kOffStages = 0;
  static constexpr int kOffQ = kNumStages * kStageBytes;
  static constexpr int kOffP = kOffQ + 2 * 4096;  // Q buffers padded to 4 KB (1024-B aligned)
  static constexpr int kOffMax = kOffP + 2 * kPBytes;
  static constexpr int kOffBar = kOffMax + 2 * 4 * 32 * 4;
  static constexpr int kNumBars = 3 * kNumStages + 10;
  static constexpr int kOffTmem = kOffBar + kNumBars * 8;
  static constexpr int kTotal = kOffTmem + 16;
};

// Synchronisation protocol (all mbarriers, phase = use count parity):
//   k_full[st], v_full[st]  producer TMA bytes landed          -> MMA thread
//   stage_empty[st]         tcgen05.commit after PV of the tile -> producer (K and V slots free)
//   q_full/q_empty[qb]      Q rows of a task                    (producer <-> MMA thread)
//   s_full[buf]             commit after QK                     -> softmax warps
//   p_full[buf]             the 4 softmax warps wrote P^T       -> MMA thread
//   o_full[buf]             commit after PV                     -> softmax warps
// No "empty" barriers are needed for S, P and O: the MMA thread issues QK(n) only after it has
// waited p_full(n-2) (softmax threads arrive on it after their tcgen05.ld of S(n-2) and O(n-3)),
// and a softmax thread writes P(n) only after it has consumed O(n-2), i.e. PV(n-2) completed.
// kKPerToken: q per-token/head, k per-token/head (scales in the cache's extra rows), v per-head
// (reference .../smallm_fp8_qkpertoken_perhead_vperhead_dim128_dynamic_splitk_kernels.cuh:29);
// otherwise q per-token/head, k/v per-tensor.
template <int NQ, int RL, bool kKPerToken>
__global__ void __launch_bounds__(kThreads, 1)
    decode_attn_fp8_kernel(const __grid_constant__ CUtensorMap tmap_q,
                           const __grid_constant__ CUtensorMap tmap_k,
                           const __grid_constant__ CUtensorMap tmap_v, const Params p) {
  using L = Smem<NQ>;
  extern __shared__ __align__(1024) uint8_t smem[];

  uint8_t* stages = smem + L::kOffStages;
  uint8_t* q_smem = smem + L::kOffQ;
  uint8_t* p_smem = smem + L::kOffP;
  float* smax = reinterpret_cast<float*>(smem + L::kOffMax);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + L::kOffBar);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + L::kOffTmem);

  uint64_t* k_full = bars;
  uint64_t* v_full = bars + kNumStages;
  uint64_t* stage_empty = bars + 2 * kNumStages;
  uint64_t* q_full = bars + 3 * kNumStages;
  uint64_t* q_empty = q_full + 2;
  uint64_t* s_full = q_full + 4;
  uint64_t* p_full = q_full + 6;
  uint64_t* o_full = q_full + 8;

  const int tid = threadIdx.x;
  const int warp = tid >> 5;
  const int lane = tid & 31;

  // ---- one-time setup --------------------------------------------------------------------
  {
    // zero both Q buffers so padded query rows are exact zeros for the whole kernel
    uint4 z = make_uint4(0, 0, 0, 0);
    for (int i = tid; i < 2 * 4096 / 16; i += kThreads) {
      reinterpret_cast<uint4*>(q_smem)[i] = z;
    }
    fence_proxy_async_smem();
  }
  if (warp == 0 && lane == 0) {
    prefetch_tensormap(&tmap_q);
    prefetch_tensormap(&tmap_k);
    prefetch_tensormap(&tmap_v);
    for (int i = 0; i < kNumStages; i++) {
      mbar_init(&k_full[i], 1);
      mbar_init(&v_full[i], 1);
      mbar_init(&stage_empty[i], 1);
    }
    for (int i = 0; i < 2; i++) {
      mbar_init(&q_full[i], 1);
      mbar_init(&q_empty[i], 1);
      mbar_init(&s_full[i], 1);
      mbar_init(&p_full[i], 4);  // one arrive per softmax warp
      mbar_init(&o_full[i], 1);
    }
    fence_barrier_init();
  }
  if (warp == 1) {
    tmem_alloc(tmem_slot, 128);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  // PDL: all of the above overlapped the tail of the previous kernel (the task-map assign); from
  // here on its output is read. The combine kernel's CTAs may be scheduled now: they park at
  // their own pdl_wait() until this grid has completed.
  pdl_launch_dependents();
  pdl_wait();

  const int ntpc1 = p.task_map[0];
  const int* bin = p.task_map + (1 + static_cast<long long>(blockIdx.x) * ntpc1) * kTaskStride;
  // rotated walk (decode_common.cuh): every role derives the same segment sequence
  constexpr bool kRotate = RL <= 16;  // the carried softmax state costs 3 RL registers
  const int u0 = (kRotate && p.rotate) ? walk_start(p.task_map, blockIdx.x) : 0;
  const BinWalk walk = scan_bin(bin, ntpc1 - 1, u0, lane);
  const int nseg = num_segments(walk);

  if (warp == 0) {
    // =========================== TMA producer ===========================================
    const uint64_t pol_stream = p.kv_policy == 0 ? make_policy_evict_first()
                                : p.kv_policy == 1 ? make_policy_evict_normal()
                                                   : make_policy_evict_last();
    uint32_t n = 0;      // global tile counter of this CTA
    uint32_t qcnt = 0;   // task counter for the Q double buffer
    Task t;
    for (int j = 0; j < nseg; j++) {
      const Segment sg = segment_of(walk, j);
      if (!load_task(bin + static_cast<long long>(sg.row) * kTaskStride, t)) break;
      // The whole warp walks the task list with warp-uniform values and ONE elected lane issues:
      // operands of TMA / mbarrier instructions live in uniform registers, and values the compiler
      // cannot prove uniform (anything loaded from memory) would make it wrap each instruction in an
      // elect + R2UR.BROADCAST loop (~70 cycles apiece).
      t.ihead_kv = __shfl_sync(0xffffffffu, t.ihead_kv, 0);
      t.ibatch = __shfl_sync(0xffffffffu, t.ibatch, 0);
      t.num_tile_kv = __shfl_sync(0xffffffffu, t.num_tile_kv, 0);
      {
        const int qb = qcnt & 1;
        mbar_wait(&q_empty[qb], ((qcnt >> 1) & 1) ^ 1);
        if (elect_one()) {
          mbar_arrive_expect_tx(&q_full[qb], p.num_seq_q * p.group * kD);
          tma_load_3d(q_smem + qb * 4096, &tmap_q, &q_full[qb], 0, t.ihead_kv * p.group,
                      t.ibatch * p.num_seq_q);
        }
        __syncwarp();
      }
      qcnt++;
      const int nblk = (t.num_seqkv + kPage - 1) / kPage;
      const int* ids = p.block_ids + static_cast<long long>(t.ibatch) * p.num_seq_max_blocks +
                       t.iseq_start / kPage;
      const int ntiles = sg.te < 0 ? t.num_tile_kv : sg.te;  // tiles [sg.tb, ntiles) of the task
      const int kc1 = p.k_head_first ? t.ihead_kv : 0;
      const int kc2 = p.k_head_first ? 0 : t.ihead_kv;
      const int vc1 = p.v_head_first ? t.ihead_kv : 0;
      const int vc2 = p.v_head_first ? 0 : t.ihead_kv;
      // L2 prefetch duty: the Hkv CTAs that stream tile x of request b (one per kv head) do so in
      // about the same step of the rotated walk; the one with ihead_kv == (b + x) % Hkv fetches
      // that tile's two pages, K and V of all heads, into L2 pf_dist tiles before it loads tile x
      // itself, so DRAM sees each page as one contiguous read. Only tiles of the current segment
      // are prefetched: its first pf_dist tiles get none. pf_dist < 0: no prefetch.
      const int pf_dist = p.pf_dist;
      const int pf_phase = (__shfl_sync(0xffffffffu, t.ibatch + t.iseq_start / kTileN, 0) + pf_dist) %
                           p.num_head_kv;
      for (int g0 = sg.tb; g0 < ntiles; g0 += 16) {
        int bi = g0 * 2 + lane;
        bi = bi < nblk ? bi : nblk - 1;  // a missing 2nd page of the last tile re-reads the 1st
        const int my_id = __ldg(ids + bi);
        int pf_id = my_id;  // page ids pf_dist tiles ahead, same lane order
        if (pf_dist > 0) {  // (distance 0: the ids of the tiles loaded now)
          int pbi = (g0 + pf_dist) * 2 + lane;
          pbi = pbi < nblk ? pbi : nblk - 1;
          pf_id = __ldg(ids + pbi);
        }
        const int gt = (ntiles - g0) < 16 ? (ntiles - g0) : 16;
        for (int tt = 0; tt < gt; tt++) {
          const int id0 = __shfl_sync(0xffffffffu, my_id, 2 * tt);
          const int id1 = __shfl_sync(0xffffffffu, my_id, 2 * tt + 1);
          const int pf0 = __shfl_sync(0xffffffffu, pf_id, 2 * tt);
          const int pf1 = __shfl_sync(0xffffffffu, pf_id, 2 * tt + 1);
          const int pt = g0 + tt + pf_dist;  // tile of the task to prefetch
          const bool pf = pf_dist >= 0 && pt < ntiles &&
                          (pf_phase + g0 + tt) % p.num_head_kv == t.ihead_kv;
          const uint32_t st = n % kNumStages;
          mbar_wait(&stage_empty[st], ((n / kNumStages) & 1) ^ 1);
          if (elect_one()) {
            if (pf) {
              bulk_prefetch_l2(p.pf_k + pf0 * p.pf_k_blk, p.pf_bytes);
              bulk_prefetch_l2(p.pf_v + pf0 * p.pf_v_blk, p.pf_bytes);
              if (2 * pt + 1 < nblk) {
                bulk_prefetch_l2(p.pf_k + pf1 * p.pf_k_blk, p.pf_bytes);
                bulk_prefetch_l2(p.pf_v + pf1 * p.pf_v_blk, p.pf_bytes);
              }
            }
            uint8_t* dst = stages + st * kStageBytes;
            mbar_arrive_expect_tx(&k_full[st], kSlotBytes);
            tma_load_4d_hint(dst, &tmap_k, &k_full[st], 0, kc1, kc2, id0, pol_stream);
            tma_load_4d_hint(dst + kSlotBytes / 2, &tmap_k, &k_full[st], 0, kc1, kc2, id1,
                             pol_stream);
            mbar_arrive_expect_tx(&v_full[st], kSlotBytes);
            tma_load_4d_hint(dst + kSlotBytes, &tmap_v, &v_full[st], 0, vc1, vc2, id0,
                             pol_stream);
            tma_load_4d_hint(dst + kSlotBytes + kSlotBytes / 2, &tmap_v, &v_full[st], 0, vc1, vc2,
                             id1, pol_stream);
          }
          __syncwarp();
          n++;
        }
      }
    }
  } else if (warp == 1) {
    // =========================== tcgen05 issuer (whole warp, one elected lane issues) ========
    {
      const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_slot, 0);  // warp-uniform copy
      constexpr uint32_t idesc_qk = make_idesc(128, NQ, kFmtE4M3, kFmtE4M3, 0, 0);
      constexpr uint32_t idesc_pv = make_idesc(128, NQ, kFmtE4M3, kFmtE4M3, 1, 1);
      // Descriptor templates; per tile only the 14-bit start-address field (units of 16 B) moves.
      //  K tile / Q rows : K-major, 128B swizzle, 8-row groups 1024 B apart, K advances 32 B / MMA
      //  V tile          : MN-major (d contiguous, exactly as stored), 128B swizzle, 8-key groups
      //                    1024 B apart, one MMA consumes 32 keys = 4096 B
      //  P^T             : MN-major, no swizzle, [key][16 queries] planes: 8-key core matrices
      //                    128 B apart (LBO), second plane kTileN*16 B away (SBO); 512 B / MMA
      const uint64_t kdesc0 = make_smem_desc(smem_u32(stages), 16, 1024, kLayoutSW128);
      const uint64_t vdesc0 = make_smem_desc(smem_u32(stages) + kSlotBytes, 16, 1024, kLayoutSW128);
      const uint64_t qdesc0 = make_smem_desc(smem_u32(q_smem), 16, 1024, kLayoutSW128);
      const uint64_t pdesc0 = make_smem_desc(smem_u32(p_smem), 128, kTileN * 16, kLayoutNone);

      auto issue_pv = [&](uint32_t m) {
        const uint32_t st = m % kNumStages;
        const uint32_t buf = m & 1;
        mbar_wait(&p_full[buf], (m >> 1) & 1);
        mbar_wait(&v_full[st], (m / kNumStages) & 1);
        tc_fence_after();
        const uint64_t ad = vdesc0 + static_cast<uint64_t>(st * (kStageBytes >> 4));
        const uint64_t bd = pdesc0 + static_cast<uint64_t>(buf * (L::kPBytes >> 4));
        const uint32_t d = tmem_base + 2 * NQ + buf * NQ;
        if (elect_one()) {
#pragma unroll
          for (int k = 0; k < 4; k++) {
            umma_f8(d, ad + k * (4096 >> 4), bd + k * (512 >> 4), idesc_pv, k > 0);
          }
          umma_commit(&o_full[buf]);  // the softmax warps wait for this one: first
          umma_commit(&stage_empty[st]);
        }
        __syncwarp();
      };

      uint32_t n = 0;
      uint32_t qcnt = 0;
      Task t;
      for (int j = 0; j < nseg; j++) {
        const Segment sg = segment_of(walk, j);
        if (!load_task(bin + static_cast<long long>(sg.row) * kTaskStride, t)) break;
        const int qb = qcnt & 1;
        mbar_wait(&q_full[qb], (qcnt >> 1) & 1);
        const uint64_t bd = qdesc0 + static_cast<uint64_t>(qb * (4096 >> 4));
        const int ntiles = sg.te < 0 ? __shfl_sync(0xffffffffu, t.num_tile_kv, 0) : sg.te;
        for (int tt = sg.tb; tt < ntiles; tt++) {
          const uint32_t st = n % kNumStages;
          const uint32_t buf = n & 1;
          mbar_wait(&k_full[st], (n / kNumStages) & 1);
          tc_fence_after();
          const uint64_t ad = kdesc0 + static_cast<uint64_t>(st * (kStageBytes >> 4));
          const uint32_t d = tmem_base + buf * NQ;
          if (elect_one()) {
#pragma unroll
            for (int k = 0; k < 4; k++) {
              umma_f8(d, ad + k * (32 >> 4), bd + k * (32 >> 4), idesc_qk, k > 0);
            }
            umma_commit(&s_full[buf]);
            if (tt == ntiles - 1) umma_commit(&q_empty[qb]);
          }
          __syncwarp();
          if (n > 0) issue_pv(n - 1);
          n++;
        }
        qcnt++;
      }
      if (n > 0) issue_pv(n - 1);
    }
  } else {
    // =========================== softmax / epilogue warps =================================
    const int quad = warp & 3;           // TMEM lane quadrant this warp may access
    const int row_in_tile = quad * 32 + lane;  // key index (S^T) and d index (O^T)
    const int sw = warp - 2;             // 0..3 index for smem exchange
    const uint32_t lane_addr = tmem_base + (static_cast<uint32_t>(quad * 32) << 16);
    const float kscale = kKPerToken ? 1.f : p.kscale[0];
    const int* chunk_table = p.task_map + kTaskStride * (ntpc1 * p.task_map[1] + 1);  // num_chunks[h * B + b]
    float out_scale = kKPerToken ? 0.f : p.vscale[0] * (1.0f / 256.0f);

    uint32_t n = 0;
    Task t;
    // online-softmax state of the task the rotated walk started inside of, kept from its first
    // part (tail tiles) to its second part (head tiles) at the end of the walk
    float carry_m[kRotate ? RL : 1], carry_l[kRotate ? RL : 1], carry_acc[kRotate ? RL : 1];
    for (int j = 0; j < nseg; j++) {
      const Segment sg = segment_of(walk, j);
      if (!load_task(bin + static_cast<long long>(sg.row) * kTaskStride, t)) break;
      float c[RL], mrun[RL], lrun[RL], alpha_pend[RL];
      float acc[RL];
      {
        const float* qs = p.qscale +
                          static_cast<long long>(t.ibatch) * p.num_seq_q * p.qscale_stride +
                          t.ihead_kv * p.group;
#pragma unroll
        for (int r = 0; r < RL; r++) {
          const int sq = r / p.group;
          const int g = r - sq * p.group;
          const bool valid = sq < p.num_seq_q;
          const float qv = valid ? __ldg(qs + sq * p.qscale_stride + g) : 0.f;
          c[r] = qv * kscale * p.softmax_scale_log2;
          mrun[r] = -INFINITY;
          lrun[r] = 0.f;
          alpha_pend[r] = 1.f;
          acc[r] = 0.f;
        }
        if constexpr (kRotate) {
          if (sg.restore) {
#pragma unroll
            for (int r = 0; r < RL; r++) {
              mrun[r] = carry_m[r];
              lrun[r] = carry_l[r];
              acc[r] = carry_acc[r];
            }
          }
        }
      }
      const int lim_len = t.num_seqkv;
      const int lim_causal = t.num_seqkvcache;
      const int tile_begin = sg.tb;
      const int ntiles = sg.te < 0 ? t.num_tile_kv : sg.te;  // tiles [tile_begin, ntiles)
      // k-per-token: this thread's key of tile tt sits in page (2 tt + row / 64) of the task's
      // page list; its scale is fetched one tile ahead
      const int* page_ids = p.block_ids + static_cast<long long>(t.ibatch) * p.num_seq_max_blocks +
                            t.iseq_start / kPage;
      const int npages = (t.num_seqkv + kPage - 1) / kPage;
      auto key_scale = [&](int tile) -> float {
        int pg = 2 * tile + (row_in_tile >> 6);
        pg = pg < npages ? pg : npages - 1;
        if (pg < 0) return 0.f;
        const long long blk = __ldg(page_ids + pg);
        const int slot = row_in_tile & 63;
        return __ldg(p.kscale + blk * p.ks_blk + (slot >> 5) * p.ks_row + t.ihead_kv * p.ks_head +
                     (slot & 31));
      };
      float ks_next = 1.f;
      if constexpr (kKPerToken) {
        out_scale = __ldg(p.vscale + t.ihead_kv) * (1.0f / 256.0f);
        ks_next = ntiles > tile_begin ? key_scale(tile_begin) : 0.f;
      }

      auto consume_o = [&](uint32_t m) {
        const uint32_t buf = m & 1;
        mbar_wait(&o_full[buf], (m >> 1) & 1);
        tc_fence_after();
        uint32_t o[NQ];
        if constexpr (NQ == 16) {
          tmem_ld_x16(lane_addr + 2 * NQ + buf * NQ, o);
        } else {
          tmem_ld_x32(lane_addr + 2 * NQ + buf * NQ, o);
        }
        tmem_wait_ld();
#pragma unroll
        for (int r = 0; r < RL; r++) {
          acc[r] = acc[r] * alpha_pend[r] + __uint_as_float(o[r]);
        }
      };

      for (int tt = tile_begin; tt < ntiles; tt++) {
        const uint32_t buf = n & 1;
        const uint32_t ph = (n >> 1) & 1;
        const float ks_cur = ks_next;
        if constexpr (kKPerToken) {
          if (tt + 1 < ntiles) ks_next = key_scale(tt + 1);
        }
        mbar_wait(&s_full[buf], ph);
        tc_fence_after();
        uint32_t sraw[NQ];
        if constexpr (NQ == 16) {
          tmem_ld_x16(lane_addr + buf * NQ, sraw);
        } else {
          tmem_ld_x32(lane_addr + buf * NQ, sraw);
        }
        tmem_wait_ld();

        const int key = tt * kTileN + row_in_tile;
        const int lim_min = lim_len < lim_causal ? lim_len : lim_causal;
        const bool need_mask = (tt + 1) * kTileN > lim_min;
        float x[RL];
        float* mx = smax + (buf * 4 + sw) * 32;
#pragma unroll
        for (int r = 0; r < RL; r++) {
          float v = __uint_as_float(sraw[r]) * c[r];
          if constexpr (kKPerToken) v *= ks_cur;
          if (need_mask) {
            const int sq = r / p.group;
            const bool dead = (key >= lim_len) || (key > lim_causal + sq);
            v = dead ? -INFINITY : v;
          }
          x[r] = v;
          const float wm = warp_max_f32(v);
          if (lane == 0) mx[r] = wm;
        }
        named_bar_sync(kSoftmaxBar, 128);
        const float* mall = smax + buf * 4 * 32;
        float pv[RL];
#pragma unroll
        for (int r = 0; r < RL; r++) {
          const float tm = fmaxf(fmaxf(mall[r], mall[32 + r]), fmaxf(mall[64 + r], mall[96 + r]));
          const float mold = mrun[r];
          const float mnew = fmaxf(mold, tm);
          float a = 1.f, e = 0.f;
          if (mnew != -INFINITY) {
            a = exp2_approx(mold - mnew);
            e = exp2_approx(x[r] - mnew);
          }
          mrun[r] = mnew;
          lrun[r] = lrun[r] * a + e;
          pv[r] = e * 256.f;
          // alpha for the O tile of *this* key tile is applied when that tile is consumed
          x[r] = a;
        }
        // ---- P^T row of this key -> smem (e4m3), 16 queries per plane ----
        // (P buffer `buf` is free: this thread consumed O(n-2) last iteration => PV(n-2) done)
        {
          uint8_t* pb = p_smem + buf * L::kPBytes + row_in_tile * 16;
#pragma unroll
          for (int pl = 0; pl < L::kPPlanes; pl++) {
            float f[16];
#pragma unroll
            for (int i = 0; i < 16; i++) {
              const int r = pl * 16 + i;
              f[i] = (r < RL) ? pv[r < RL ? r : 0] : 0.f;
            }
            uint4 w;
            w.x = cvt_e4m3x4(f[0], f[1], f[2], f[3]);
            w.y = cvt_e4m3x4(f[4], f[5], f[6], f[7]);
            w.z = cvt_e4m3x4(f[8], f[9], f[10], f[11]);
            w.w = cvt_e4m3x4(f[12], f[13], f[14], f[15]);
            *reinterpret_cast<uint4*>(pb + pl * kTileN * 16) = w;
          }
        }
        fence_proxy_async_smem();
        tc_fence_before();  // orders this thread's tcgen05.ld of S(n) and O(n-2) before the arrive
        __syncwarp();
        if (lane == 0) mbar_arrive(&p_full[buf]);

        if (tt > tile_begin) consume_o(n - 1);
#pragma unroll
        for (int r = 0; r < RL; r++) alpha_pend[r] = x[r];
        n++;
      }
      if (ntiles > tile_begin) consume_o(n - 1);

      if constexpr (kRotate) {
        if (sg.save) {  // first part of the split task: its head tiles come last
#pragma unroll
          for (int r = 0; r < RL; r++) {
            carry_m[r] = mrun[r];
            carry_l[r] = lrun[r];
            carry_acc[r] = acc[r];
          }
          continue;
        }
      }

      // ---- task epilogue: 1/sum, v scale, partial O and LSE out ----
      float* red = smax;  // reuse: [4 warps][32]
      named_bar_sync(kSoftmaxBar, 128);
#pragma unroll
      for (int r = 0; r < RL; r++) {
        const float ws = warp_sum_f32(lrun[r]);
        if (lane == 0) red[sw * 32 + r] = ws;
      }
      named_bar_sync(kSoftmaxBar, 128);
      const long long chunk_row =
          static_cast<long long>(t.ibatch) * p.max_splitk + t.ichunk;
      // A (batch, kv head) pair that was not split needs no combine: its rows go out as bf16 right
      // here (the same fp32 value the combine kernel would round), and the combine kernel skips
      // pairs with one chunk. At C2 that is ~70 % of the pairs.
      const bool single = p.y != nullptr && __ldg(chunk_table + t.ihead_kv * p.num_batch + t.ibatch) == 1;
#pragma unroll
      for (int r = 0; r < RL; r++) {
        const int sq = r / p.group;
        const int g = r - sq * p.group;
        if (sq < p.num_seq_q) {
          const float tot = red[r] + red[32 + r] + red[64 + r] + red[96 + r];
          const float inv = tot != 0.f ? rcp_approx(tot) : 0.f;
          if (single) {
            p.y[(static_cast<long long>(t.ibatch) * p.num_seq_q + sq) * p.ld_y +
                (t.ihead_kv * p.group + g) * kD + row_in_tile] =
                __float2bfloat16_rn(acc[r] * inv * out_scale);
            continue;
          }
          const long long orow =
              (chunk_row * p.num_seq_q + sq) * p.num_head_q + t.ihead_kv * p.group + g;
          p.split_out[orow * kD + row_in_tile] = acc[r] * inv * out_scale;
          if (row_in_tile == r) {
            const float l = (mrun[r] == -INFINITY) ? -INFINITY : mrun[r] + log2_approx(tot);
            p.lse[((chunk_row * p.num_head_kv + t.ihead_kv) * p.num_seq_q + sq) * p.lse_pad + g] =
                l;
          }
        }
      }
      named_bar_sync(kSoftmaxBar, 128);  // red[] reused as smax by the next task
    }
  }

  // ---- teardown ----
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tmem_dealloc(tmem_base, 128);
  }
}

// ------------------------------------------------------------------------------------------------
// split-k combine: y = sum_c 2^(lse_c - m) O_c / sum_c 2^(lse_c - m)  -> bf16
// (reference src/attention/decode/splitk_combine_kernels.cuh:140-322)
// one 128-thread block per output row (b, s, hq); warp w handles chunks w, w+4, ...
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128)
    decode_combine_kernel(__nv_bfloat16* __restrict__ y, const float* __restrict__ split_out,
                          const float* __restrict__ lse, const int* __restrict__ task_map,
                          int num_batch, int num_seq_q, int num_head_q, int num_head_kv, int group,
                          int max_splitk, int lse_pad, int ldY, int direct_single) {
  __shared__ float4 s_acc[4][32];
  __shared__ float s_m[4];
  __shared__ float s_l[4];

  const int row = blockIdx.x;  // (b * Sq + s) * Hq + hq
  const int hq = row % num_head_q;
  const int bs = row / num_head_q;
  const int s = bs % num_seq_q;
  const int b = bs / num_seq_q;
  const int hkv = hq / group;
  const int g = hq - hkv * group;
  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  pdl_wait();               // the attention kernel's partials and LSEs are complete
  pdl_launch_dependents();  // whatever follows may set itself up

  const int ntpc1 = task_map[0];
  const int nctas = task_map[1];
  const int max_batch = task_map[3];
  (void)max_batch;
  const int* chunk_table = task_map + kTaskStride * (ntpc1 * nctas + 1);
  const int nchunks = chunk_table[hkv * num_batch + b];
  if (nchunks == 1 && direct_single) return;  // written by the attention kernel itself

  float m = -INFINITY;
  float l = 0.f;
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
  for (int c = warp; c < nchunks; c += 4) {
    const long long chunk_row = static_cast<long long>(b) * max_splitk + c;
    const float lc = __ldg(lse + ((chunk_row * num_head_kv + hkv) * num_seq_q + s) * lse_pad + g);
    const float4 o = ld_nc_f4(split_out +
                              ((chunk_row * num_seq_q + s) * num_head_q + hq) * (long long)kD +
                              lane * 4);
    if (lc == -INFINITY) continue;
    const float mn = fmaxf(m, lc);
    const float a = exp2_approx(m - mn);
    const float w = exp2_approx(lc - mn);
    acc.x = acc.x * a + o.x * w;
    acc.y = acc.y * a + o.y * w;
    acc.z = acc.z * a + o.z * w;
    acc.w = acc.w * a + o.w * w;
    l = l * a + w;
    m = mn;
  }
  s_acc[warp][lane] = acc;
  if (lane == 0) {
    s_m[warp] = m;
    s_l[warp] = l;
  }
  __syncthreads();
  if (warp == 0) {
    const float mg = fmaxf(fmaxf(s_m[0], s_m[1]), fmaxf(s_m[2], s_m[3]));
    float4 r = make_float4(0.f, 0.f, 0.f, 0.f);
    float lt = 0.f;
#pragma unroll
    for (int w = 0; w < 4; w++) {
      const float sc = (s_m[w] == -INFINITY) ? 0.f : exp2_approx(s_m[w] - mg);
      const float4 a = s_acc[w][lane];
      r.x += a.x * sc;
      r.y += a.y * sc;
      r.z += a.z * sc;
      r.w += a.w * sc;
      lt += s_l[w] * sc;
    }
    const float inv = lt > 0.f ? 1.f / lt : 0.f;
    __nv_bfloat162 lo = __floats2bfloat162_rn(r.x * inv, r.y * inv);
    __nv_bfloat162 hi = __floats2bfloat162_rn(r.z * inv, r.w * inv);
    uint2 pk;
    pk.x = *reinterpret_cast<uint32_t*>(&lo);
    pk.y = *reinterpret_cast<uint32_t*>(&hi);
    __nv_bfloat16* dst = y + static_cast<long long>(bs) * ldY + hq * kD + lane * 4;
    *reinterpret_cast<uint2*>(dst) = pk;
  }
}

cudaError_t launch_combine(__nv_bfloat16* y, const float* split_out, const float* lse,
                           const int* task_map, int num_batch, int num_seq_q, int num_head_q,
                           int num_head_kv, int group, int max_splitk, int lse_pad, int ldY,
                           cudaStream_t stream) {
  const int out_rows = num_batch * num_seq_q * num_head_q;
  return launch_pdl(decode_combine_kernel, dim3(out_rows), dim3(128), 0, stream, 1, y, split_out, lse,
                    task_map, num_batch, num_seq_q, num_head_q, num_head_kv, group, max_splitk,
                    lse_pad, ldY, 1);
}

template <int NQ, int RL, bool kKPerToken>
static int launch_attn(const CUtensorMap& tq, const CUtensorMap& tk, const CUtensorMap& tv,
                       const Params& p, int grid, cudaStream_t stream) {
  using L = Smem<NQ>;
  auto kern = decode_attn_fp8_kernel<NQ, RL, kKPerToken>;
  static bool configured[64] = {false};
  const int dev = device_slot();
  if (!configured[dev]) {
    HPC_CUDA_CHECK(
        cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, L::kTotal));
    configured[dev] = true;
  }
  HPC_CUDA_CHECK(launch_pdl(kern, dim3(grid), dim3(kThreads), L::kTotal, stream, 1, tq, tk, tv, p));
  return HPC_OK;
}

}  // namespace decode
}  // namespace b200

using namespace b200;  // NOLINT

static int decode_fp8_impl(
    bool run_attn, bool run_combine, void* y_ptr, void* lse_ptr, void* split_out_ptr, const int* task_map_ptr, const void* q_ptr,
    void* kcache_ptr, void* vcache_ptr, const int* block_ids_ptr, const int* num_seq_kvcache_ptr,
    const float* qscale_ptr, const float* kscale_ptr, const float* vscale_ptr, int* split_flag_ptr,
    int new_kv_included, int splitk, int splitk_min_len, int consumers, int quant_type,
    int num_batch, int num_seq_q, int num_head_q, int num_head_k, int num_head_v, int num_dim_qk,
    int num_dim_v, int num_kvcache_blocks, int block_size, int num_seq_max_blocks,
    int qscale_pad_stride, int ldY, int ldQ, int64_t kcache_block_stride,
    int64_t kcache_token_stride, int64_t kcache_head_stride, int64_t vcache_block_stride,
    int64_t vcache_token_stride, int64_t vcache_head_stride, cudaStream_t stream) {
  (void)num_seq_kvcache_ptr;  // lengths come from the task map (as in the reference dynamic path)
  (void)split_flag_ptr;
  (void)new_kv_included;
  (void)splitk_min_len;
  (void)consumers;
  // quant_type (reference hpc/attention.py QuantType): 0 = q,k per token/head + v per head,
  // 1 = q per token/head + k,v per tensor
  HPC_REQUIRE(quant_type == 0 || quant_type == 1,
              "attention_decode_fp8: quant_type %d is not implemented (0: q/k per token-head, v per "
              "head; 1: q per token-head, k/v per tensor)",
              quant_type);
  if (quant_type == 0) {
    // the per-token k scales live in the cache allocation's extra rows and share its strides
    // (reference src/attention/entry.cc:245-253): float strides = byte strides / 4
    HPC_REQUIRE((kcache_block_stride % 4) == 0 && (kcache_token_stride % 4) == 0 &&
                    (kcache_head_stride % 4) == 0 && kscale_ptr != nullptr &&
                    (reinterpret_cast<uintptr_t>(kscale_ptr) & 3) == 0,
                "attention_decode_fp8: k scale rows must be 4-byte aligned slices of the cache");
  }
  HPC_REQUIRE(task_map_ptr != nullptr, "attention_decode_fp8: a task_map is required on sm_100");
  HPC_REQUIRE(num_dim_qk == 128 && num_dim_v == 128, "head dim must be 128");
  HPC_REQUIRE(block_size == 64, "kvcache paged blocksize must be 64");
  HPC_REQUIRE(num_head_k == num_head_v && num_head_k > 0 && num_head_q % num_head_k == 0,
              "bad head counts q=%d k=%d v=%d", num_head_q, num_head_k, num_head_v);
  const int group = num_head_q / num_head_k;
  const int rows = group * num_seq_q;
  HPC_REQUIRE(rows >= 1 && rows <= 32 && group <= 16,
              "heads_per_group * num_seq_q = %d not in [1, 32]", rows);
  HPC_REQUIRE(splitk >= 1, "splitk (max chunks) must be >= 1");
  HPC_REQUIRE((reinterpret_cast<uintptr_t>(q_ptr) & 15) == 0 && (ldQ % 16) == 0,
              "q must be 16-byte aligned");
  HPC_REQUIRE((kcache_block_stride % 16) == 0 && (kcache_token_stride % 16) == 0 &&
                  (kcache_head_stride % 16) == 0 && (vcache_block_stride % 16) == 0 &&
                  (vcache_token_stride % 16) == 0 && (vcache_head_stride % 16) == 0,
              "kv cache strides must be multiples of 16 bytes");

  const int lse_pad_ = (group + 7) / 8 * 8;
  if (run_combine && !run_attn) {
    HPC_CUDA_CHECK(decode::launch_combine(static_cast<__nv_bfloat16*>(y_ptr),
                                          static_cast<const float*>(split_out_ptr),
                                          static_cast<const float*>(lse_ptr), task_map_ptr, num_batch,
                                          num_seq_q, num_head_q, num_head_k, group, splitk, lse_pad_,
                                          ldY, stream));
    return HPC_OK;
  }

  // Rotated bin walk: for token-major caches whose rows of neighbouring heads are neighbours in
  // memory (pairs of 128-byte runs inside 256-byte-aligned lines). HPC_B200_DECODE_ROTATE=0 disables.
  bool rotate = num_head_k >= 2 && (num_head_k % 2) == 0 && rows <= 16 &&
                kcache_head_stride == 128 && vcache_head_stride == 128 &&
                (kcache_token_stride % 256) == 0 && (vcache_token_stride % 256) == 0 &&
                (kcache_block_stride % 256) == 0 && (vcache_block_stride % 256) == 0 &&
                (reinterpret_cast<uintptr_t>(kcache_ptr) % 256) == 0 &&
                (reinterpret_cast<uintptr_t>(vcache_ptr) % 256) == 0;
  if (const char* e = getenv("HPC_B200_DECODE_ROTATE")) rotate = rotate && atoi(e) != 0;

  // Page-wide L2 prefetch (producer warp): when each cache is dense token-major, one page's rows of
  // all heads are one contiguous range, [blk * block_stride, + 64 * token_stride) (the k-per-token
  // scale rows follow it and are not prefetched). One bulk prefetch per page, so at most 8 kv heads
  // (64 KB, the size run on B200). HPC_B200_KV_PREFETCH=0 disables it, HPC_B200_KV_PREFETCH_DIST
  // sets the distance in tiles.
  const int64_t dense_row = static_cast<int64_t>(num_head_k) * 128;
  bool prefetch = rotate && num_head_k <= 8 && kcache_token_stride == dense_row &&
                  vcache_token_stride == dense_row;
  if (const char* e = getenv("HPC_B200_KV_PREFETCH")) prefetch = prefetch && atoi(e) != 0;
  int pf_dist = 1;
  if (const char* e = getenv("HPC_B200_KV_PREFETCH_DIST")) pf_dist = atoi(e);

  CUtensorMap tq, tk, tv;
  {
    uint64_t dims[3] = {128, static_cast<uint64_t>(num_head_q),
                        static_cast<uint64_t>(num_batch) * num_seq_q};
    uint64_t strides[2] = {128, static_cast<uint64_t>(ldQ)};
    uint32_t box[3] = {128, static_cast<uint32_t>(group), static_cast<uint32_t>(num_seq_q)};
    int rc = encode_tmap_u8(&tq, q_ptr, 3, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_128B);
    if (rc) return rc;
  }
  auto encode_cache = [&](CUtensorMap* tm, const void* base, int heads, int64_t blk_stride,
                          int64_t tok_stride, int64_t head_stride, int* head_first) -> int {
    // TMA wants strides ordered ascending: pick (d, head, token, blk) for NHD caches and
    // (d, token, head, blk) for HND caches; the smem image of the 64x128 box is identical.
    *head_first = head_stride <= tok_stride ? 1 : 0;
    uint64_t dims[4];
    uint64_t strides[3];
    uint32_t box[4];
    dims[0] = 128;
    box[0] = 128;
    if (*head_first) {
      dims[1] = static_cast<uint64_t>(heads);
      dims[2] = 64;
      strides[0] = static_cast<uint64_t>(head_stride);
      strides[1] = static_cast<uint64_t>(tok_stride);
      box[1] = 1;
      box[2] = 64;
    } else {
      dims[1] = 64;
      dims[2] = static_cast<uint64_t>(heads);
      strides[0] = static_cast<uint64_t>(tok_stride);
      strides[1] = static_cast<uint64_t>(head_stride);
      box[1] = 64;
      box[2] = 1;
    }
    dims[3] = static_cast<uint64_t>(num_kvcache_blocks);
    strides[2] = static_cast<uint64_t>(blk_stride);
    box[3] = 1;
    // L2 promotion must not exceed the contiguous run of one head's row: with token rows of
    // 128 B strided by Hkv*128 B (NHD) a 256 B promotion drags in the neighbouring head's row,
    // which is consumed by another CTA much later (measured: +49 % DRAM reads, profiles/).
    // ... unless the walk is rotated: then the neighbouring head's row is wanted by another CTA at
    // the same time and the wider fetch is its prefetch (decode_common.cuh).
    // With the page-wide prefetch the loads find their lines in L2 and the wider promotion only
    // adds reads (measured at C2: 172 vs 173 us, profiles/decode_prefetch_ab.json).
    CUtensorMapL2promotion promo = (tok_stride == 128 || (rotate && !prefetch))
                                       ? CU_TENSOR_MAP_L2_PROMOTION_L2_256B
                                       : CU_TENSOR_MAP_L2_PROMOTION_L2_128B;
    if (const char* e = getenv("HPC_B200_KV_PROMO")) {  // tuning knob: 0 none, 1 64B, 2 128B, 3 256B
      const int v = atoi(e);
      promo = v == 0 ? CU_TENSOR_MAP_L2_PROMOTION_NONE
                     : v == 1 ? CU_TENSOR_MAP_L2_PROMOTION_L2_64B
                              : v == 2 ? CU_TENSOR_MAP_L2_PROMOTION_L2_128B
                                       : CU_TENSOR_MAP_L2_PROMOTION_L2_256B;
    }
    return encode_tmap_u8(tm, base, 4, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_128B, promo);
  };
  int k_head_first = 1, v_head_first = 1;
  {
    int rc = encode_cache(&tk, kcache_ptr, num_head_k, kcache_block_stride, kcache_token_stride,
                          kcache_head_stride, &k_head_first);
    if (rc) return rc;
    rc = encode_cache(&tv, vcache_ptr, num_head_v, vcache_block_stride, vcache_token_stride,
                      vcache_head_stride, &v_head_first);
    if (rc) return rc;
  }

  decode::Params p;
  p.task_map = task_map_ptr;
  p.block_ids = block_ids_ptr;
  p.qscale = qscale_ptr;
  p.kscale = kscale_ptr;
  p.vscale = vscale_ptr;
  p.split_out = static_cast<float*>(split_out_ptr);
  p.lse = static_cast<float*>(lse_ptr);
  p.y = static_cast<__nv_bfloat16*>(y_ptr);
  p.ld_y = ldY;
  p.num_batch = num_batch;
  p.num_seq_q = num_seq_q;
  p.num_head_q = num_head_q;
  p.num_head_kv = num_head_k;
  p.group = group;
  p.num_seq_max_blocks = num_seq_max_blocks;
  p.qscale_stride = qscale_pad_stride;
  p.max_splitk = splitk;
  p.lse_pad = (group + 7) / 8 * 8;
  p.k_head_first = k_head_first;
  p.v_head_first = v_head_first;
  p.softmax_scale_log2 = 1.4426950408889634f / sqrtf(static_cast<float>(num_dim_qk));
  p.ks_blk = kcache_block_stride / 4;
  p.ks_row = kcache_token_stride / 4;
  p.ks_head = kcache_head_stride / 4;
  p.rotate = rotate ? 1 : 0;
  // streamed once: evict_first - except under the rotated walk, where the promoted half of a line
  // is another CTA's data a moment later and should not be the first thing to go (measured at C2:
  // 180 vs 199 us, profiles/r2_decode_rotate_ab2.json)
  p.kv_policy = rotate ? 1 : 0;
  if (const char* e = getenv("HPC_B200_KV_POLICY")) p.kv_policy = atoi(e);  // tuning knob
  p.pf_dist = prefetch && pf_dist >= 0 ? pf_dist : -1;
  p.pf_bytes = static_cast<uint32_t>(64 * dense_row);
  p.pf_k = static_cast<const uint8_t*>(kcache_ptr);
  p.pf_v = static_cast<const uint8_t*>(vcache_ptr);
  p.pf_k_blk = kcache_block_stride;
  p.pf_v_blk = vcache_block_stride;

  const int grid = splitk;  // == num_total_ctas of the task map
  int rc;
#define HPC_DECODE_LAUNCH(NQ_, RL_)                                                   \
  rc = (quant_type == 0) ? decode::launch_attn<NQ_, RL_, true>(tq, tk, tv, p, grid, stream) \
                         : decode::launch_attn<NQ_, RL_, false>(tq, tk, tv, p, grid, stream)
  if (rows <= 4) {
    HPC_DECODE_LAUNCH(16, 4);
  } else if (rows <= 8) {
    HPC_DECODE_LAUNCH(16, 8);
  } else if (rows <= 12) {
    HPC_DECODE_LAUNCH(16, 12);
  } else if (rows <= 16) {
    HPC_DECODE_LAUNCH(16, 16);
  } else if (rows <= 24) {
    HPC_DECODE_LAUNCH(32, 24);
  } else {
    HPC_DECODE_LAUNCH(32, 32);
  }
#undef HPC_DECODE_LAUNCH
  if (rc) return rc;
  if (!run_combine) return HPC_OK;

  HPC_CUDA_CHECK(decode::launch_combine(static_cast<__nv_bfloat16*>(y_ptr), p.split_out, p.lse,
                                        task_map_ptr, num_batch, num_seq_q, num_head_q, num_head_k,
                                        group, splitk, p.lse_pad, ldY, stream));
  return HPC_OK;
}

#define DECODE_FP8_ARGS                                                                           \
  lse_ptr, split_out_ptr, task_map_ptr, q_ptr, kcache_ptr, vcache_ptr, block_ids_ptr,             \
      num_seq_kvcache_ptr, qscale_ptr, kscale_ptr, vscale_ptr, split_flag_ptr, new_kv_included,   \
      splitk, splitk_min_len, consumers, quant_type, num_batch, num_seq_q, num_head_q,            \
      num_head_k, num_head_v, num_dim_qk, num_dim_v, num_kvcache_blocks, block_size,              \
      num_seq_max_blocks, qscale_pad_stride, ldY, ldQ, kcache_block_stride, kcache_token_stride,  \
      kcache_head_stride, vcache_block_stride, vcache_token_stride, vcache_head_stride, stream

#define DECODE_FP8_PARAMS                                                                         \
  void *lse_ptr, void *split_out_ptr, const int *task_map_ptr, const void *q_ptr,                 \
      void *kcache_ptr, void *vcache_ptr, const int *block_ids_ptr,                               \
      const int *num_seq_kvcache_ptr, const float *qscale_ptr, const float *kscale_ptr,           \
      const float *vscale_ptr, int *split_flag_ptr, int new_kv_included, int splitk,              \
      int splitk_min_len, int consumers, int quant_type, int num_batch, int num_seq_q,            \
      int num_head_q, int num_head_k, int num_head_v, int num_dim_qk, int num_dim_v,              \
      int num_kvcache_blocks, int block_size, int num_seq_max_blocks, int qscale_pad_stride,      \
      int ldY, int ldQ, int64_t kcache_block_stride, int64_t kcache_token_stride,                 \
      int64_t kcache_head_stride, int64_t vcache_block_stride, int64_t vcache_token_stride,       \
      int64_t vcache_head_stride, cudaStream_t stream

// attention (split partials + lse) followed by the combine: the reference launcher's contract
extern "C" int hpc_attention_decode_fp8_async(void* y_ptr, DECODE_FP8_PARAMS) {
  return decode_fp8_impl(true, true, y_ptr, DECODE_FP8_ARGS);
}
// the two stages separately (bench.py times the dominant kernel alone; same arguments)
extern "C" int hpc_attention_decode_fp8_partial_async(void* y_ptr, DECODE_FP8_PARAMS) {
  return decode_fp8_impl(true, false, y_ptr, DECODE_FP8_ARGS);
}
extern "C" int hpc_attention_decode_fp8_combine_async(void* y_ptr, DECODE_FP8_PARAMS) {
  return decode_fp8_impl(false, true, y_ptr, DECODE_FP8_ARGS);
}
