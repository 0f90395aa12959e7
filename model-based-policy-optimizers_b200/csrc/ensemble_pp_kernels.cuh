// Stage 4, fused, two row tiles per CTA ("ping-pong"): the dominant kernel of BASELINE config 4.
//
// Same computation as ensemble_kernels.cuh (vmap(vmap(rollout_actions)) through the learned ensemble,
// mbpo/utils/optimizer_utils.py:11-59 + icem_optimizer.py:155-160), same operand roundings, same layer
// formulation (all four layers on tcgen05, cta_group::2, weights resident in shared memory) -- but a
// CTA pair owns 512 candidate rows as two tiles X and Y of 256 rows (128 TMEM lanes per CTA each):
// while the tensor cores run layer l+1 of tile X, the 16 epilogue warps turn tile Y's accumulator
// into activations, and vice versa.  The epilogue warps never wait for an MMA in steady state, and
// because nothing forces them to a common barrier at a layer boundary they drift apart, which keeps
// the MUFU pipe (tanh, the bound of this kernel: 16/clk/SM) busy across boundaries.
//
//   TMEM      D_X = columns [0, 256), D_Y = columns [256, 512): ONE accumulator per tile, so layer l+1 of
//             a tile is issued only after its layer-l epilogue has published all four chunks.
//   A ring    the bf16 A operand exists only as a ring of five 16 KB chunks (64 K-columns x 128 rows):
//             the epilogue of one tile fills chunks while the MMAs of the other tile drain them; a full
//             A tile per row tile (2 x 64 KB) would not fit beside the 128 KB of resident weights.
//             stage[tile] (leader CTA, 32 warp arrivals)   all four chunks of the tile's next A operand are
//                                                          published by both CTAs (one arrive per warp per
//                                                          stage: the MMAs cannot start earlier anyway)
//             empty[slot][k] (both CTAs, tcgen05.commit)   the MMA that read K-step k (16 columns) of the chunk
//                                                          has completed; a warp rewrites only its own K-step
//   order     epilogue warps, per horizon step:  E0(X) E0(Y) E1(X) E1(Y) E2(X) E2(Y) E3(X) E3(Y)
//             MMA issuer,     per horizon step:  M0(X) M0(Y) M1(X) M1(Y) M2(X) M2(Y) M3(X) M3(Y)
//             (El = epilogue reading layer l's accumulator; E3 = output layer -> state update -> next
//             step's split-input row; Ml = the MMAs of layer l.)
#pragma once
#include "ensemble_kernels.cuh"

namespace mbpo {
namespace ens {

constexpr int PP_SLOTS = 5;
constexpr uint32_t PP_SLOT_BYTES = TILE_M * 64 * 2;     // 16384: 64 K-columns of 128 rows
constexpr int PP_ROUNDS = 4;                            // 64-column rounds per layer

struct PpSmem {
  static constexpr uint32_t RING = 0;                                    // 5 x 16 KB A chunks
  static constexpr uint32_t W1 = RING + PP_SLOTS * PP_SLOT_BYTES;        // W[e,0] rows [128*rank, +128)
  static constexpr uint32_t W2 = W1 + WH_BYTES;                          // W[e,1] rows [128*rank, +128)
  static constexpr uint32_t A0 = W2 + WH_BYTES;                          // 2 tiles x (128 x 16 bf16) split inputs
  static constexpr uint32_t W0 = A0 + 2 * TILE_M * 32;                   // 128 x 16 bf16 split layer-0 weights
  static constexpr uint32_t W3 = W0 + 128 * 32;                          // 8 x 256 bf16 output layer hi/lo rows
  static constexpr uint32_t HB = W3 + 8 * HID * 2;                       // float [2][256]: 0.5 * b_h
  static constexpr uint32_t B_OUT = HB + 2 * HID * 4;                    // float [4]
  static constexpr uint32_t BARS = B_OUT + 16;   // stage[2] empty[5][4] acc_done[2] out_done[2] a0_full[2] bar_w
  static constexpr uint32_t TMEM_PTR = BARS + (4 * PP_SLOTS + 9) * 8;
  static constexpr uint32_t TOTAL = TMEM_PTR + 16;
};
static_assert(PpSmem::TOTAL <= 227 * 1024, "ping-pong ensemble rollout shared memory plan exceeds 227 KB");

// The kernel body; TR as in ensemble_rollout_body.
template <bool TR>
__device__ __forceinline__ void ensemble_rollout_pp_body(const EnsArgs& a, const CUtensorMap& w_map, float* obs_out,
                                                         float* reward_out) {
  extern __shared__ __align__(1024) uint8_t smem[];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int quarter = warp >> 2;                       // which 16 of a round's 64 columns (epilogue warps)
  const int lrow = ((warp & 3) << 5) | lane;           // row within a tile = TMEM lane
  const uint32_t rank = cluster_ctarank();
  const bool leader = rank == 0;
  const bool row_owner = quarter == 3;   // warps 12-15 carry the rows' state: the warp scheduler favours the
                                          // highest warp ids, and the state update is the serial link between steps
  float* s_hb = reinterpret_cast<float*>(smem + PpSmem::HB);
  float* s_b_out = reinterpret_cast<float*>(smem + PpSmem::B_OUT);
  uint64_t* bar_stage = reinterpret_cast<uint64_t*>(smem + PpSmem::BARS);   // [2] leader: tile's A chunks published
  uint64_t* bar_empty = bar_stage + 2;
  uint64_t* bar_acc = bar_empty + 4 * PP_SLOTS;            // [2] accumulator of layer 0/1/2 of tile t complete
  uint64_t* bar_out = bar_acc + 2;                     // [2] output-layer accumulator of tile t complete
  uint64_t* bar_a0 = bar_out + 2;                      // [2] leader: split-input rows of tile t published
  uint64_t* bar_w = bar_a0 + 2;
  uint32_t* s_tmem = reinterpret_cast<uint32_t*>(smem + PpSmem::TMEM_PTR);

  // ---- one-time setup --------------------------------------------------------------------------
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(s_tmem)),
                 "r"(ENS_TMEM_COLS));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;");
  }
  if (tid == 0) {
    for (int s = 0; s < 4 * PP_SLOTS; ++s) mbar_init(bar_empty + s, 1);
    for (int t = 0; t < 2; ++t) {
      mbar_init(bar_stage + t, 2 * EPI_WARPS);
      mbar_init(bar_acc + t, 1);
      mbar_init(bar_out + t, 1);
      mbar_init(bar_a0 + t, 2 * 4);
    }
    mbar_init(bar_w, 1);
    fence_barrier_init();
  }
  for (int i = tid; i < 8 * HID * 2 / 16; i += ENS_THREADS)   // non-leader's output-layer rows stay zero
    reinterpret_cast<uint4*>(smem + PpSmem::W3)[i] = make_uint4(0u, 0u, 0u, 0u);
  fence_proxy_async();
  tc_fence_before();
  __syncthreads();
  cluster_sync();
  tc_fence_after();
  const uint32_t tmem_base = *s_tmem;
  const uint32_t tmem_lane = tmem_base + (static_cast<uint32_t>((warp & 3) * 32) << 16);
  const uint32_t bar_stage_leader = map_to_cta(smem_u32(bar_stage), 0);
  const uint32_t bar_a0_leader = map_to_cta(smem_u32(bar_a0), 0);
  constexpr uint32_t IDESC = umma_idesc_bf16(2 * TILE_M, HID);
  constexpr uint32_t IDESC_OUT = umma_idesc_bf16(2 * TILE_M, 16);
  uint32_t phase_w = 0;
  uint32_t ph_acc[2] = {0, 0}, ph_out[2] = {0, 0};   // epilogue warps
  uint32_t ph_a0[2] = {0, 0}, ph_stage[2] = {0, 0};  // MMA warp
  // position in the A-chunk ring: chunks produced (epilogue warps) / consumed (MMA warp) so far, kept as
  // (position % PP_SLOTS, position / PP_SLOTS)
  uint32_t ring_slot = 0, ring_use = 0;
  const PendulumConsts pc(a.reward);

  const int num_groups = (a.R + 4 * TILE_M - 1) / (4 * TILE_M);
  for (int group = blockIdx.x >> 1; group < num_groups; group += gridDim.x >> 1) {
    int row[2];
    bool valid[2];
    float x_init[2][3];
    const float* act[2];
#pragma unroll
    for (int tl = 0; tl < 2; ++tl) {
      row[tl] = group * 4 * TILE_M + tl * 2 * TILE_M + static_cast<int>(rank) * TILE_M + lrow;
      valid[tl] = row[tl] < a.R;
      const int rr = valid[tl] ? row[tl] : a.R - 1;
      const int b = rr / a.M;
      x_init[tl][0] = a.x0[3 * b]; x_init[tl][1] = a.x0[3 * b + 1]; x_init[tl][2] = a.x0[3 * b + 2];
      act[tl] = a.actions + static_cast<size_t>(rr) * a.H;
    }
    float summary[2] = {0.0f, 0.0f};

    for (int e = 0; e < a.num_members; ++e) {
      // ---- member e: hidden weight halves by TMA; the small layers are split into bf16 parts here ----
      __syncthreads();  // every MMA of the previous member has completed (row owners waited bar_out of both tiles)
      if (tid == 0) {
        mbar_expect_tx(bar_w, 2 * WH_BYTES);
        for (int l = 0; l < 2; ++l)
          for (int kc = 0; kc < KCHUNKS; ++kc)
            tma_load_2d(smem + (l ? PpSmem::W2 : PpSmem::W1) + kc * WH_LBO, &w_map, kc * 8,
                        (e * 2 + l) * HID + static_cast<int>(rank) * 128, bar_w);
      }
      if (tid < 128) {
        // layer 0, this CTA's 128 output units: per input [wh, wl, wh], then the bias [bh, bm, bl, 0]; all * 0.5
        const int n = static_cast<int>(rank) * 128 + tid;
        float wh[4], wl[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const float w = 0.5f * a.w_in[(static_cast<size_t>(e) * 4 + i) * HID + n];
          wh[i] = bf16_hi(w);
          wl[i] = w - wh[i];
        }
        const float bias = 0.5f * a.b_in[e * HID + n];
        const float bh = bf16_hi(bias), bm = bf16_hi(bias - bh), bl = (bias - bh) - bm;
        uint4 p0, p1;
        p0.x = pack_bf16(wh[0], wl[0]); p0.y = pack_bf16(wh[0], wh[1]);
        p0.z = pack_bf16(wl[1], wh[1]); p0.w = pack_bf16(wh[2], wl[2]);
        p1.x = pack_bf16(wh[2], wh[3]); p1.y = pack_bf16(wl[3], wh[3]);
        p1.z = pack_bf16(bh, bm);       p1.w = pack_bf16(bl, 0.0f);
        *reinterpret_cast<uint4*>(smem + PpSmem::W0 + tid * 16) = p0;
        *reinterpret_cast<uint4*>(smem + PpSmem::W0 + WH_LBO + tid * 16) = p1;
      } else if (tid < 128 + HID && leader) {
        // output layer: row j (j < 3) = hi part of w_out[:, j], row 3 + j = lo part; rows 6, 7 stay zero
        const int k = tid - 128;
#pragma unroll
        for (int j = 0; j < 3; ++j) {
          const float w = a.w_out[(static_cast<size_t>(e) * HID + k) * 3 + j];
          const __nv_bfloat16 h = __float2bfloat16_rn(w);
          const __nv_bfloat16 l = __float2bfloat16_rn(w - __bfloat162float(h));
          uint8_t* base = smem + PpSmem::W3 + (k >> 3) * W3_LBO + (k & 7) * 2;
          *reinterpret_cast<__nv_bfloat16*>(base + j * 16) = h;
          *reinterpret_cast<__nv_bfloat16*>(base + (3 + j) * 16) = l;
        }
      }
      for (int i = tid; i < 2 * HID; i += ENS_THREADS) s_hb[i] = 0.5f * a.b_h[e * 2 * HID + i];
      if (tid < 3) s_b_out[tid] = a.b_out[e * 3 + tid];
      fence_proxy_async();        // generic-proxy writes of W0 / W3 -> visible to the tensor core
      mbar_wait(bar_w, phase_w);  // every thread observes the TMA completion
      phase_w ^= 1;
      __syncthreads();

      if (warp == MMA_WARP) {
        // ================= MMA issuer: warp 16 of the leader CTA =====================================
        if (leader) {
          const uint32_t tmem_u = __shfl_sync(0xffffffffu, tmem_base, 0);
          const bool elected = elect_one();
          const uint64_t desc_ring = umma_desc(smem_u32(smem + PpSmem::RING), A_LBO, SBO);
          const uint64_t desc_a0 = umma_desc(smem_u32(smem + PpSmem::A0), A_LBO, SBO);
          const uint64_t desc_w0 = umma_desc(smem_u32(smem + PpSmem::W0), WH_LBO, SBO);
          const uint64_t desc_w1 = umma_desc(smem_u32(smem + PpSmem::W1), WH_LBO, SBO);
          const uint64_t desc_w2 = umma_desc(smem_u32(smem + PpSmem::W2), WH_LBO, SBO);
          const uint64_t desc_w3 = umma_desc(smem_u32(smem + PpSmem::W3), W3_LBO, SBO);
          constexpr uint32_t A_STEP = (2 * A_LBO) >> 4;          // one K = 16 step inside a chunk, descriptor units
          constexpr uint32_t SLOT_STEP = PP_SLOT_BYTES >> 4;
          constexpr uint32_t A0_TILE_STEP = (TILE_M * 32) >> 4;
#pragma unroll 1
          for (int t = 0; t < a.H; ++t) {
#pragma unroll
            for (int tl = 0; tl < 2; ++tl) {
              mbar_wait(bar_a0 + tl, ph_a0[tl]);
              ph_a0[tl] ^= 1;
              tc_fence_after();
              ENS_TRACE(lane == 0, tl);
              if (elected) {
                umma_bf16_ss_2sm(tmem_u + tl * HID, desc_a0 + static_cast<uint64_t>(tl * A0_TILE_STEP), desc_w0, IDESC, 0u);
                umma_commit_2sm(bar_acc + tl);
              }
            }
#pragma unroll
            for (int layer = 1; layer <= 3; ++layer) {
              const uint64_t desc_w = layer == 1 ? desc_w1 : (layer == 2 ? desc_w2 : desc_w3);
              const uint32_t w_step = (layer < 3 ? 2 * WH_LBO : 2 * W3_LBO) >> 4;
#pragma unroll
              for (int tl = 0; tl < 2; ++tl) {
                const uint32_t d = tmem_u + tl * HID;
                // the tile has ONE accumulator: its MMAs start when the previous epilogue has read all of it,
                // i.e. when every warp of both CTAs has published the stage
                mbar_wait(bar_stage + tl, ph_stage[tl]);
                ph_stage[tl] ^= 1;
                tc_fence_after();
                ENS_TRACE(lane == 0, 2 + ((layer - 1) * 2 + tl) * 2);
#pragma unroll
                for (int r = 0; r < PP_ROUNDS; ++r) {
                  if (elected) {
                    const uint64_t da = desc_ring + static_cast<uint64_t>(ring_slot * SLOT_STEP);
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                      umma_bf16_ss_2sm(d, da + static_cast<uint64_t>(j * A_STEP),
                                       desc_w + static_cast<uint64_t>((4 * r + j) * w_step),
                                       layer < 3 ? IDESC : IDESC_OUT, (r | j) ? 1u : 0u);
                      umma_commit_2sm(bar_empty + ring_slot * 4 + j);   // K-step j of the chunk may be rewritten
                    }
                    if (r == PP_ROUNDS - 1) umma_commit_2sm(layer < 3 ? bar_acc + tl : bar_out + tl);
                  }
                  if (++ring_slot == PP_SLOTS) { ring_slot = 0; ++ring_use; }
                }
                ENS_TRACE(lane == 0, 3 + ((layer - 1) * 2 + tl) * 2);
              }
            }
          }
        }
      } else {
        // ================= epilogue warps ============================================================
        float x[2][3], acc[2] = {0.0f, 0.0f}, u[2] = {0.0f, 0.0f};
#pragma unroll
        for (int tl = 0; tl < 2; ++tl) {
          x[tl][0] = x_init[tl][0]; x[tl][1] = x_init[tl][1]; x[tl][2] = x_init[tl][2];
          if (row_owner) {
            u[tl] = __ldg(act[tl]);
            build_a0_row(smem + PpSmem::A0 + tl * TILE_M * 32 + lrow * 16, x[tl][0], x[tl][1], x[tl][2], u[tl]);
            fence_proxy_async();
            __syncwarp();
            if (lane == 0) mbar_arrive_cluster(bar_a0_leader + tl * 8);
          }
        }
#pragma unroll 1
        for (int t = 0; t < a.H; ++t) {
          float u_next[2] = {0.0f, 0.0f};
          if (row_owner) {
#pragma unroll
            for (int tl = 0; tl < 2; ++tl) {
              // reward on the current state and the raw action (pendulum_reward.py:32-40)
              const float rw = reward_from(pc, atan2_bounded(x[tl][1], x[tl][0]), x[tl][2], u[tl]);
              if (TR && valid[tl]) {
                const size_t o = (static_cast<size_t>(row[tl]) * a.num_members + e) * a.H + t;
                obs_out[3 * o] = x[tl][0]; obs_out[3 * o + 1] = x[tl][1]; obs_out[3 * o + 2] = x[tl][2];
                reward_out[o] = rw;
              }
              acc[tl] = __fadd_rn(acc[tl], rw);
              if (t + 1 < a.H) u_next[tl] = __ldg(act[tl] + t + 1);
            }
          }
#pragma unroll
          for (int layer = 0; layer < 3; ++layer) {
#pragma unroll
            for (int tl = 0; tl < 2; ++tl) {
              mbar_wait(bar_acc + tl, ph_acc[tl]);   // accumulator of this layer of this tile complete
              ph_acc[tl] ^= 1;
              tc_fence_after();
              ENS_TRACE(tid == 0, 20 + (layer * 2 + tl) * 6);
              ENS_TRACE(tid == 480, 60 + (layer * 2 + tl) * 6);
              const uint32_t d_src = tmem_lane + tl * HID + quarter * 16;
              const float* hb = s_hb + (layer > 0 ? layer - 1 : 0) * HID + quarter * 16;
#pragma unroll
              for (int r = 0; r < PP_ROUNDS; ++r) {
                uint32_t v[16];
                tmem_ld16_nowait(d_src + r * 64, v);
                if (ring_use > 0) mbar_wait(bar_empty + ring_slot * 4 + quarter, (ring_use - 1) & 1);   // K-step drained
                tmem_wait_ld16(v);
                uint8_t* dst = smem + PpSmem::RING + ring_slot * PP_SLOT_BYTES + (2 * quarter) * A_LBO + lrow * 16;
                if (layer == 0) epilogue_round<16, false>(v, nullptr, dst);
                else epilogue_round<16, true>(v, hb + r * 64, dst);
                if (++ring_slot == PP_SLOTS) { ring_slot = 0; ++ring_use; }
                ENS_TRACE(tid == 0, 21 + (layer * 2 + tl) * 6 + r);
                ENS_TRACE(tid == 480, 61 + (layer * 2 + tl) * 6 + r);
              }
              publish_round(bar_stage_leader + tl * 8, lane);   // one fence + arrive per warp per stage
            }
          }
          if (row_owner) {
#pragma unroll
            for (int tl = 0; tl < 2; ++tl) {
              mbar_wait(bar_out + tl, ph_out[tl]);
              ph_out[tl] ^= 1;
              tc_fence_after();
              ENS_TRACE(tid == 384, 100 + tl);
              uint32_t o[8];
              tmem_ld8_nowait(tmem_lane + tl * HID, o);
              tmem_wait_ld8(o);
              tc_fence_before();
              x[tl][0] = __fadd_rn(x[tl][0], (__uint_as_float(o[0]) + __uint_as_float(o[3])) + s_b_out[0]);
              x[tl][1] = __fadd_rn(x[tl][1], (__uint_as_float(o[1]) + __uint_as_float(o[4])) + s_b_out[1]);
              x[tl][2] = __fadd_rn(x[tl][2], (__uint_as_float(o[2]) + __uint_as_float(o[5])) + s_b_out[2]);
              if (t + 1 < a.H) {
                u[tl] = u_next[tl];
                build_a0_row(smem + PpSmem::A0 + tl * TILE_M * 32 + lrow * 16, x[tl][0], x[tl][1], x[tl][2], u[tl]);
                fence_proxy_async();
                __syncwarp();
                if (lane == 0) mbar_arrive_cluster(bar_a0_leader + tl * 8);
                ENS_TRACE(tid == 384, 102 + tl);
              }
            }
          }
        }
        if (row_owner) {
#pragma unroll
          for (int tl = 0; tl < 2; ++tl) {
            const float ret = __fdiv_rn(acc[tl], static_cast<float>(a.H));
            if (a.summarize == MBPO_SUMMARIZE_MAX) summary[tl] = (e == 0) ? ret : fmaxf(summary[tl], ret);
            else summary[tl] = __fadd_rn(summary[tl], ret);
          }
        }
      }
    }
    if (row_owner && warp != MMA_WARP) {
#pragma unroll
      for (int tl = 0; tl < 2; ++tl) {
        float s = summary[tl];
        if (a.summarize != MBPO_SUMMARIZE_MAX) s = __fdiv_rn(s, static_cast<float>(a.num_members));
        if (!TR && valid[tl]) a.returns_out[row[tl]] = s;
      }
    }
  }

  // ---- teardown --------------------------------------------------------------------------------------
  tc_fence_before();
  __syncthreads();
  cluster_sync();
  if (warp == 0) {
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(ENS_TMEM_COLS));
  }
}

__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(ENS_THREADS, 1)
    ensemble_rollout_pp_kernel(const __grid_constant__ EnsArgs a, const __grid_constant__ CUtensorMap w_map) {
  ensemble_rollout_pp_body<false>(a, w_map, nullptr, nullptr);
}

__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(ENS_THREADS, 1)
    ensemble_transitions_pp_kernel(const __grid_constant__ EnsArgs a, const __grid_constant__ CUtensorMap w_map,
                                   float* __restrict__ obs_out, float* __restrict__ reward_out) {
  ensemble_rollout_pp_body<true>(a, w_map, obs_out, reward_out);
}

// Chooses the kernel: the two-tile kernel needs half as many CTA pairs per row, so it is used whenever the
// one-tile kernel would need more than one round of CTA pairs (throughput shapes); small row counts keep
// the one-tile kernel, which spreads them over more SMs (latency shapes).  The row count alone decides
// (no run-time switch); the tests reach each kernel through its own sizes.  obs_out / reward_out: as in
// launch_ensemble_rollout.
inline int launch_ensemble_rollout_auto(const MbpoMlpEnsembleParams& p, int horizon, const float* x0,
                                        const float* actions, int B, int M, int summarize, float* returns_out,
                                        float* obs_out, float* reward_out, cudaStream_t st, char* err, size_t errlen) {
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  const long long R = static_cast<long long>(B) * M;
  const bool use_pp = R > static_cast<long long>(2 * TILE_M) * (sms / 2);
  if (!use_pp)
    return launch_ensemble_rollout(p, horizon, x0, actions, B, M, summarize, returns_out, obs_out, reward_out, st, err,
                                   errlen);
  if (p.hidden != HID || p.x_dim != 3 || p.u_dim != 1 || p.num_members < 1) {
    snprintf(err, errlen,
             "ensemble rollout: the tcgen05 kernel needs hidden == 256, x_dim == 3, u_dim == 1 (got %d, %d, %d)",
             p.hidden, p.x_dim, p.u_dim);
    return MBPO_EUNSUPPORTED;
  }
  EncodeTiledFn enc = encode_tiled_fn();
  if (!enc) {
    snprintf(err, errlen, "ensemble rollout: cuTensorMapEncodeTiled is not available from the driver");
    return MBPO_ECUDA;
  }
  CUtensorMap map;
  const cuuint64_t dims[2] = {static_cast<cuuint64_t>(HID), static_cast<cuuint64_t>(p.num_members) * 2 * HID};
  const cuuint64_t strides[1] = {static_cast<cuuint64_t>(HID) * 2};
  const cuuint32_t box[2] = {8, 128};
  const cuuint32_t estr[2] = {1, 1};
  const CUresult cr = enc(&map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<uint16_t*>(p.w_h), dims, strides, box,
                          estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
                          CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (cr != CUDA_SUCCESS) {
    snprintf(err, errlen, "ensemble rollout: cuTensorMapEncodeTiled failed (CUresult %d)", static_cast<int>(cr));
    return MBPO_ECUDA;
  }
  EnsArgs a;
  a.num_members = p.num_members; a.R = B * M; a.H = horizon; a.M = M; a.summarize = summarize;
  a.w_in = p.w_in; a.b_in = p.b_in; a.b_h = p.b_h; a.w_out = p.w_out; a.b_out = p.b_out;
  a.x0 = x0; a.actions = actions; a.returns_out = returns_out; a.reward = p.reward;
  const bool tr = obs_out != nullptr;
  cudaError_t ce = cudaFuncSetAttribute(tr ? reinterpret_cast<const void*>(ensemble_transitions_pp_kernel)
                                           : reinterpret_cast<const void*>(ensemble_rollout_pp_kernel),
                                        cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(PpSmem::TOTAL));
  if (ce != cudaSuccess) {
    snprintf(err, errlen, "ensemble rollout: smem attribute: %s", cudaGetErrorString(ce));
    return MBPO_ECUDA;
  }
  const int groups = (a.R + 4 * TILE_M - 1) / (4 * TILE_M);
  const int pairs = groups < sms / 2 ? groups : sms / 2;
  if (tr) ensemble_transitions_pp_kernel<<<2 * pairs, ENS_THREADS, PpSmem::TOTAL, st>>>(a, map, obs_out, reward_out);
  else ensemble_rollout_pp_kernel<<<2 * pairs, ENS_THREADS, PpSmem::TOTAL, st>>>(a, map);
  return MBPO_OK;
}

}  // namespace ens
}  // namespace mbpo
