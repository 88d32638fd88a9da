// Fused transition block (FeedForward + residual) on tcgen05, CTA-pair (cta_group::2) MMA:
//
//   x <- x + W2 (a * gelu(g)) + b2,   [a | g] = W1' ((x - mean) * rstd) + b1'
//
// One pass per unit of 256 rows (128 per CTA of the pair); the hidden activations h never leave the SM.
//   * A tile: LN(x) of the CTA's 128 rows x d, bf16, produced by the SIMT LayerNorm producers of proj_tc.cuh
//     (proj_producer_loop) straight from fp32 x; the LN affine is folded into W1 / b1 on the host (pack_feed_forward).
//   * The hidden dimension is walked in chunks of 64 units.  Chunk c:
//       FF-1  acc1[c & 1] (128 TMEM columns: 64 value | 64 gate) = ones x bias block + A x W1(c)^T        M 256, N 128, K d
//       GEGLU the epilogue warps read acc1, compute a * gelu(g) (proj_finish32, the same arithmetic as proj_tc's GEGLU
//             epilogue) and write h as bf16 pairs with tcgen05.st OVER the value columns they have just read
//       FF-2  out (+)= h(c) x W2[:, c]^T with h as the TMEM A operand                                     M 256, N d, K 64
//     The MMA warp issues FF-1(c + 1) before FF-2(c), so the GEGLU of chunk c runs under the tensor work of FF-1(c + 1).
//     acc1[c & 1] is overwritten by FF-1(c + 2), which is issued after FF-2(c) by the same thread: the tensor core executes
//     one thread's MMAs in issue order (attention_tc.cuh relies on the same property), so no barrier guards that reuse.
//   * W1 chunks use the per-tile packing of the unfused path unchanged (w_cat: [128 value rows | 128 gate rows] per 256-row
//     tile): chunk c is rows tile * 256 + {0, 128} + (c & 1) * 64 of tile c / 2, so CTA rank r stages the 64 rows starting at
//     (c / 2) * 256 + r * 128 + (c & 1) * 64 and the pair MMA sees [64 value | 64 gate] columns.  The bias enters through one
//     K = 16 MMA step (ones x [bias hi | bias lo]) exactly as in proj_tc, from the same w_ext block.
//   * Residual epilogue once per unit: out accumulator -> registers, + b2, + x, stored in place.  Every epilogue warp stages
//     two 4 KB boxes (32 rows x 32 fp32) in the unit's A buffer, which no MMA reads once the output accumulator is complete;
//     the residual comes in and the result goes out by TMA, and the buffer returns to the producers after the last store has
//     read it.  Each row is read by the producer and later read and written by its own unit's epilogue only.
//
// TMEM (512 columns per CTA): [0, d) output accumulator (single buffered) | [256, 384) acc1[0] | [384, 512) acc1[1].
// The next unit's FF-1 chunks 0 and 1 are issued before the previous unit's last FF-2, so they overlap its drain.
//
// Shared memory per CTA (217 856 B of the 227 KB):
//   A        2 x 64 KB   LN(x) tiles, double buffered: producing one takes about a third of a unit's tensor time, and with a
//                        single buffer the tensor core would idle for all of it at every unit boundary
//   weights  5 x 16 KB   ring, in MMA order: W1(c+1) as nkb/2 slots of two 8 KB k-blocks (64 rows x 128 B), then W2(c)
//                        (d/2 rows x 64 hidden, 128 B rows); all 128B-swizzled
//   bias     2 x 2 KB    W1 bias block of a chunk (64 rows x 32 B, 32B swizzle)
//   ones     256 B       A operand of the bias step (one 8-row atom, stride 0)
//   barriers 512 B
// Per-warp residual boxes do not fit beside this, hence the reuse of the spent A buffer (a first version that loaded and stored
// x straight from registers, one row per thread, spent ~16k clk per unit on uncoalesced accesses: 141 us instead of 101 us).
//
// Warp roles (512 threads): 0 weight TMA producer | 1 MMA issuer (leader CTA) | 2 TMEM allocator | 3 idle |
// 4..11 epilogue (warp w: TMEM lanes 32 (w % 4) .., hidden half (w - 4) / 4 of every chunk; output columns 32-column
// chunks of parity (w - 4) / 4) | 12..15 LayerNorm producers.
#pragma once
#include "proj_tc.cuh"

namespace af2 {

constexpr int FF_THREADS = 512;
constexpr int FF_CHUNK = 64;            // hidden units per chunk

struct FfParams {
  float* x;                // [T, d] fp32 residual stream (read and written in place)
  const float* b2;         // [d]
  long long T;
  int d, hidden;
  float inv_d, eps;
  int m_units;             // ceil(T / 256)
};

struct FfSmem {
  static constexpr int STAGES = 5;
  static constexpr int STAGE = 16384;
  static constexpr int A_OFF = 0;
  static constexpr int W_OFF = 2 * PROJ_A_BUF;
  static constexpr int BIAS_OFF = W_OFF + STAGES * STAGE;
  static constexpr int BIAS_BYTES = 64 * 32;
  static constexpr int AEXT_OFF = BIAS_OFF + 2 * BIAS_BYTES;
  static constexpr int BAR_OFF = AEXT_OFF + 256;
  static constexpr int TOTAL = BAR_OFF + 512;
  static_assert(TOTAL <= 232448, "exceeds the 227 KB of shared memory a CTA can use");
};

// D[tmem of both CTAs] (+)= A[tmem of both CTAs, 128 rows each] * B[smem, N/2 rows each]; one thread of the leader CTA
__device__ __forceinline__ void umma_bf16_ts_pair(uint32_t d_tmem, uint32_t a_tmem, uint64_t bdesc, uint32_t idesc,
                                                  uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], [%1], %2, %3, p;\n\t}"
      ::"r"(d_tmem), "r"(a_tmem), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}

__global__ void __launch_bounds__(FF_THREADS, 1)
ff_tc_kernel(const __grid_constant__ CUtensorMap tmW1, const __grid_constant__ CUtensorMap tmB1,
             const __grid_constant__ CUtensorMap tmW2, const __grid_constant__ CUtensorMap tmX,
             const __grid_constant__ FfParams p) {
  using L = FfSmem;
  constexpr int STAGES = L::STAGES;
  extern __shared__ __align__(1024) uint8_t smem[];
  if ((smem_u32(smem) & 1023u) != 0) __trap();
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + L::BAR_OFF);   // [STAGES] weight slot landed (leader's)
  uint64_t* empty_bar = full_bar + STAGES;                                // [STAGES] weight slot consumed
  uint64_t* bfull_bar = empty_bar + STAGES;                               // [2] bias block landed (leader's)
  uint64_t* bempty_bar = bfull_bar + 2;                                   // [2] bias block consumed
  uint64_t* c1full_bar = bempty_bar + 2;                                  // [2] chunk accumulator ready
  uint64_t* hfull_bar = c1full_bar + 2;                                   // [2] h of the chunk written (leader's)
  uint64_t* afull_bar = hfull_bar + 2;                                    // [2] A tile produced (leader's)
  uint64_t* aempty_bar = afull_bar + 2;                                   // [2] A buffer free (unit drained)
  uint64_t* ofull_bar = aempty_bar + 2;                                   // output accumulator ready
  uint64_t* oempty_bar = ofull_bar + 1;                                   // output accumulator drained (leader's)
  uint64_t* res_bar = oempty_bar + 1;                                     // [8 epilogue warps][2] residual box landed
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(res_bar + 16);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const bool is_leader = rank == 0;
  const int cluster_id = blockIdx.x / 2;
  const int nclusters = gridDim.x / 2;
  constexpr uint32_t TMEM_COLS = 512;
  constexpr uint32_t ACC1_COL = 256;

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&tmW1);
    prefetch_tmap(&tmB1);
    prefetch_tmap(&tmW2);
    prefetch_tmap(&tmX);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(&bfull_bar[s], 1);
      mbar_init(&bempty_bar[s], 1);
      mbar_init(&c1full_bar[s], 1);
      mbar_init(&hfull_bar[s], 16);
      mbar_init(&afull_bar[s], 2 * PROJ_NPROD);
      mbar_init(&aempty_bar[s], 8);                   // the CTA's epilogue warps, after the unit's residual stores
    }
    mbar_init(ofull_bar, 1);
    mbar_init(oempty_bar, 16);
    for (int s = 0; s < 16; ++s) mbar_init(&res_bar[s], 1);
    fence_barrier_init();
  }
  if (warp == 2) tmem_alloc_pair(tmem_slot, TMEM_COLS);
  // ones block of the bias K-step (see proj_tc_kernel)
  for (int i = threadIdx.x; i < 256 / 16; i += FF_THREADS)
    *reinterpret_cast<uint4*>(smem + L::AEXT_OFF + i * 16) = make_uint4(0x3f803f80u, 0u, 0u, 0u);
  fence_proxy_async_smem();
  tc_fence_before();
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  pdl_launch_dependents();
  pdl_wait();

  // units (256 rows) dealt round-robin over the clusters; the chunk stream runs across this cluster's units
  const int my_units = p.m_units > cluster_id ? (p.m_units - 1 - cluster_id) / nclusters + 1 : 0;
  const int nch = p.hidden / FF_CHUNK;
  const int nchunks = my_units * nch;
  const int nkb = p.d / GEMM_BK;
  const int d_half = p.d >> 1;
  auto unit_of = [&](int it) { return cluster_id + it * nclusters; };

  if (warp == 0) {
    // ================================ weight TMA producer ================================
    if (lane == 0) {
      auto leader_bar = [&](uint64_t* bar) { return mapa_u32(smem_u32(bar), 0); };
      int stage = 0;
      uint32_t phase = 0;
      auto acquire = [&](int bytes) {
        mbar_wait(&empty_bar[stage], phase ^ 1);
        if (is_leader) mbar_arrive_expect_tx(&full_bar[stage], 2 * bytes);
        return smem + L::W_OFF + stage * L::STAGE;
      };
      auto advance = [&]() { if (++stage == STAGES) { stage = 0; phase ^= 1; } };
      auto load_w1 = [&](int g) {
        const int c = g % nch;
        const int row0 = (c >> 1) * 256 + static_cast<int>(rank) * 128 + (c & 1) * 64;
        const int b = g & 1;
        mbar_wait(&bempty_bar[b], ((g >> 1) & 1) ^ 1);
        if (is_leader) mbar_arrive_expect_tx(&bfull_bar[b], 2 * L::BIAS_BYTES);
        tma_load_2d_pair(smem + L::BIAS_OFF + b * L::BIAS_BYTES, &tmB1, leader_bar(&bfull_bar[b]), 0, row0);
        for (int kb = 0; kb < nkb; kb += 2) {
          uint8_t* sb = acquire(2 * 8192);
          tma_load_2d_pair(sb, &tmW1, leader_bar(&full_bar[stage]), kb * GEMM_BK, row0);
          tma_load_2d_pair(sb + 8192, &tmW1, leader_bar(&full_bar[stage]), (kb + 1) * GEMM_BK, row0);
          advance();
        }
      };
      auto load_w2 = [&](int g) {
        const int c = g % nch;
        uint8_t* sb = acquire(d_half * 128);
        tma_load_2d_pair(sb, &tmW2, leader_bar(&full_bar[stage]), c * FF_CHUNK, static_cast<int>(rank) * d_half);
        advance();
      };
      if (nchunks > 0) load_w1(0);
      for (int g = 0; g < nchunks; ++g) {
        if (g + 1 < nchunks) load_w1(g + 1);
        load_w2(g);
      }
    }
  } else if (warp == 1) {
    // ================================ MMA issuer (leader CTA) =================================
    if (is_leader) {
      const uint32_t idesc1 = umma_idesc_bf16(256, 128, 0, 0);
      const uint32_t idesc2 = umma_idesc_bf16(256, p.d, 0, 0);
      int stage = 0;
      uint32_t phase = 0;
      auto ff1 = [&](int g) {
        const int it = g / nch, c = g - it * nch;
        const int ab = it & 1;
        if (c == 0) mbar_wait(&afull_bar[ab], (it >> 1) & 1);
        const int b = g & 1;
        const uint32_t d_tmem = tmem_base + ACC1_COL + b * 128;
        mbar_wait(&bfull_bar[b], (g >> 1) & 1);
        tc_fence_after();
        if (elect_one()) {
          const uint64_t adesc = umma_smem_desc(smem_u32(smem + L::AEXT_OFF), 16, 0, SWZ_32);
          const uint64_t bdesc = umma_smem_desc(smem_u32(smem + L::BIAS_OFF + b * L::BIAS_BYTES), 16, 256, SWZ_32);
          umma_bf16_pair(d_tmem, adesc, bdesc, idesc1, 0u);
          umma_commit_pair(&bempty_bar[b], 3);
        }
        __syncwarp();
        const uint32_t sa0 = smem_u32(smem + L::A_OFF + ab * PROJ_A_BUF);
        for (int kb = 0; kb < nkb; kb += 2) {
          mbar_wait(&full_bar[stage], phase);
          tc_fence_after();
          if (elect_one()) {
            const uint32_t sb = smem_u32(smem + L::W_OFF + stage * L::STAGE);
#pragma unroll
            for (int h = 0; h < 2; ++h) {
#pragma unroll
              for (int k = 0; k < GEMM_BK / 16; ++k) {
                const uint64_t adesc = umma_smem_desc(sa0 + (kb + h) * 16384 + k * 32, 16, 1024, SWZ_128);
                const uint64_t bdesc = umma_smem_desc(sb + h * 8192 + k * 32, 16, 1024, SWZ_128);
                umma_bf16_pair(d_tmem, adesc, bdesc, idesc1, 1u);
              }
            }
            umma_commit_pair(&empty_bar[stage], 3);
            if (kb + 2 >= nkb) {
              umma_commit_pair(&c1full_bar[b], 3);
            }
          }
          __syncwarp();
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
      };
      auto ff2 = [&](int g) {
        const int it = g / nch, c = g - it * nch;
        const int b = g & 1;
        mbar_wait(&hfull_bar[b], (g >> 1) & 1);
        if (c == 0) mbar_wait(oempty_bar, (it & 1) ^ 1);
        mbar_wait(&full_bar[stage], phase);
        tc_fence_after();
        if (elect_one()) {
          const uint32_t sb = smem_u32(smem + L::W_OFF + stage * L::STAGE);
          const uint32_t a_tmem = tmem_base + ACC1_COL + b * 128;
#pragma unroll
          for (int k = 0; k < FF_CHUNK / 16; ++k) {
            // h of hidden units 16k .. 16k+15: packed bf16 pairs at columns (k / 2) * 32 + (k % 2) * 8 (see the epilogue)
            const uint64_t bdesc = umma_smem_desc(sb + k * 32, 16, 1024, SWZ_128);
            umma_bf16_ts_pair(tmem_base, a_tmem + (k >> 1) * 32 + (k & 1) * 8, bdesc, idesc2, (c != 0 || k != 0) ? 1u : 0u);
          }
          umma_commit_pair(&empty_bar[stage], 3);
          if (c == nch - 1) umma_commit_pair(ofull_bar, 3);
        }
        __syncwarp();
        if (++stage == STAGES) { stage = 0; phase ^= 1; }
      };
      if (nchunks > 0) ff1(0);
      for (int g = 0; g < nchunks; ++g) {
        if (g + 1 < nchunks) ff1(g + 1);
        ff2(g);
      }
    }
  } else if (warp >= 4 && warp < 12) {
    // ================================ epilogue ====================================
    const int q = warp & 3;
    const int grp = (warp - 4) >> 2;
    const uint32_t lane_sel = static_cast<uint32_t>(q * 32) << 16;
    const uint32_t oempty_remote = mapa_u32(smem_u32(oempty_bar), 0);
    const int ncc = p.d >> 6;                         // 32-column output chunks per warp
    int g = 0;
    uint32_t rc = 0;                                  // residual boxes this warp has loaded (barrier phases)
    for (int it = 0; it < my_units; ++it) {
      for (int c = 0; c < nch; ++c, ++g) {
        const int b = g & 1;
        mbar_wait(&c1full_bar[b], (g >> 1) & 1);
        tc_fence_after();
        // this warp: hidden units grp * 32 .. +31 of the chunk (value columns grp * 32.., gate columns 64 + grp * 32..)
        const uint32_t t_acc = tmem_base + lane_sel + ACC1_COL + b * 128 + grp * 32;
        uint32_t u[32], gt[32], pk[16];
        tmem_ld32(t_acc, u);
        tmem_ld32(t_acc + 64, gt);
        tmem_ld_wait();
        proj_finish32<EK_GATED_TOK_GELU>(u, gt, 1.0f, pk);
        // h goes over the first 16 of the 32 value columns this warp has just read (the other group's columns untouched)
        tmem_st16(t_acc, pk);
        tmem_st_wait();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive_cluster(mapa_u32(smem_u32(&hfull_bar[b]), 0));
      }
      // ---- residual epilogue of the unit: x = (out + b2) + x for this warp's 32 rows, output columns (grp + 2 j) * 32 ----
      // staged in the unit's A buffer, which the MMAs no longer read once the output accumulator is complete: two 4 KB boxes
      // per warp ([32 rows][128 B], 128B swizzle), residual in and result out by TMA (coalesced, rows beyond T clipped)
      const int m0w = (unit_of(it) * 2 + static_cast<int>(rank)) * 128 + q * 32;
      uint8_t* wbuf = smem + L::A_OFF + (it & 1) * PROJ_A_BUF + (warp - 4) * 8192;
      uint64_t* rbar = res_bar + (warp - 4) * 2;
      auto load_res = [&](int j) {                       // lane 0: residual box of output chunk j -> buffer j & 1
        mbar_arrive_expect_tx(&rbar[j & 1], 4096);
        tma_load_2d(wbuf + (j & 1) * 4096, &tmX, &rbar[j & 1], (grp + 2 * j) * 32, m0w);
      };
      mbar_wait(ofull_bar, it & 1);
      tc_fence_after();
      if (lane == 0) {
        load_res(0);
        if (ncc > 1) load_res(1);
      }
#pragma unroll 1
      for (int j = 0; j < ncc; ++j, ++rc) {
        const int col = (grp + 2 * j) * 32;
        uint32_t v[32];
        tmem_ld32(tmem_base + lane_sel + col, v);
        tmem_ld_wait();
        if (j == ncc - 1) {                            // this warp's loads of the accumulator have landed
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive_cluster(oempty_remote);
        }
        mbar_wait(&rbar[j & 1], (rc >> 1) & 1);
        uint8_t* eb = wbuf + (j & 1) * 4096;
        const float4* bias = reinterpret_cast<const float4*>(p.b2 + col);
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          float4* sp = reinterpret_cast<float4*>(eb + swz128_off(lane, e));
          const float4 r4 = *sp, b4 = __ldg(bias + e);
          // (acc + b2) + x: the order of gemm_tc's residual epilogue
          *sp = make_float4(__uint_as_float(v[4 * e]) + b4.x + r4.x, __uint_as_float(v[4 * e + 1]) + b4.y + r4.y,
                            __uint_as_float(v[4 * e + 2]) + b4.z + r4.z, __uint_as_float(v[4 * e + 3]) + b4.w + r4.w);
        }
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) {
          tma_store_2d(&tmX, eb, col, m0w);
          tma_store_commit();
          if (j + 2 < ncc) {
            tma_store_wait_read<0>();                  // the box is free again once this store has read it
            load_res(j + 2);
          }
        }
      }
      // the A buffer goes back to the LayerNorm producers once every store has read its box
      if (lane == 0) {
        tma_store_wait_read<0>();
        mbar_arrive(&aempty_bar[it & 1]);
      }
      __syncwarp();
    }
  } else if (warp >= 12) {
    // ================================ LayerNorm producers (warps 12..15) ====================================
    const int pi = warp - 12;
    auto item_row0 = [&](int it) { return static_cast<long long>(unit_of(it) * 2 + static_cast<int>(rank)) * 128; };
    auto wait_empty = [&](int it) { mbar_wait(&aempty_bar[it & 1], ((it >> 1) & 1) ^ 1); };
    auto signal_full = [&](int it) { mbar_arrive_cluster(mapa_u32(smem_u32(&afull_bar[it & 1]), 0)); };
    uint8_t* a_base = smem + L::A_OFF;
    if (p.d == 256) proj_producer_loop<8, PROJ_NPROD>(p.x, p.T, p.d, p.inv_d, p.eps, a_base, my_units, pi, lane, item_row0, wait_empty, signal_full, false, false);
    else proj_producer_loop<4, PROJ_NPROD>(p.x, p.T, p.d, p.inv_d, p.eps, a_base, my_units, pi, lane, item_row0, wait_empty, signal_full, false, false);
  }

  __syncwarp();
  tc_fence_before();
  cluster_sync_all();
  if (warp == 2) tmem_dealloc_pair(tmem_base, TMEM_COLS);
}

}  // namespace af2
