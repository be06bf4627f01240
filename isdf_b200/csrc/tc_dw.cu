// Weight-gradient kernel of the tensor-core path:  dW_l = sum over points of
//     delta_l^T  abar_{l-1}   (S3 term)   +   zbar_l^T  h_{l-1}   (S4 term)          (SURVEY.md 8a)
// as UMMA products with K = points.  The chain kernel left every operand in the "dW layout"
// (tc_common.cuh): each 16-point slice is an MN-major UMMA operand, 8 KB contiguous, fetched with one
// bulk copy.  A CTA owns one 128-row half of one 256x256 weight unit and a subset of the tiles; it
// accumulates in TMEM (256 fp32 columns) over all of them and flushes once with vector
// red.global.add.  Column sums (bias gradients, and d w_out from the v blob) ride on the same
// pipeline as N=16 products against a tile of ones.
//
// Warp roles (192 threads): warp 0 = producer, warp 1 = MMA issuer (+TMEM), warps 2-5 = flush.
#include "tc_path.cuh"

#define DW_THREADS 192

template <int kPasses> struct DwCfg {
  static constexpr int kXBytes = 4096 * (kPasses == 3 ? 2 : 1);
  static constexpr int kYBytes = 8192 * (kPasses == 3 ? 2 : 1);
  static constexpr int kStageBytes = kXBytes + kYBytes;
  static constexpr int kStages = (kPasses == 3) ? 8 : 12;
  static constexpr int kSmem = kStages * kStageBytes + 512 + 256;
};

struct DwSmemTail {
  uint64_t full[12], empty[12], done;
  uint32_t tmem_base;
};

template <int kPasses>
__global__ void __launch_bounds__(DW_THREADS, 1) tc_dw_kernel(const TcDwArgs args) {
  using Cfg = DwCfg<kPasses>;
  extern __shared__ __align__(1024) uint8_t smem[];
  uint8_t* ring = smem;
  uint8_t* ones = smem + Cfg::kStages * Cfg::kStageBytes;
  DwSmemTail* tail = reinterpret_cast<DwSmemTail*>(ones + 512);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  const int job_id = blockIdx.x % args.n_jobs;
  const int split = blockIdx.x / args.n_jobs;
  const int n_splits = ((int)gridDim.x - 1 - job_id) / args.n_jobs + 1;
  const int my_tiles = (args.n_tiles > split) ? (args.n_tiles - 1 - split) / n_splits + 1 : 0;
  const TcDwJob& job = args.jobs[job_id];

  if (threadIdx.x < 128) reinterpret_cast<uint32_t*>(ones)[threadIdx.x] = 0x3F803F80u;   // bf16 1.0 pairs
  if (threadIdx.x == 0) {
    for (int i = 0; i < Cfg::kStages; ++i) { mbar_init(smem_u32(&tail->full[i]), 1); mbar_init(smem_u32(&tail->empty[i]), 1); }
    mbar_init(smem_u32(&tail->done), 1);
    mbar_fence_init();
  }
  fence_proxy_async_smem();
  if (warp == 1) tmem_alloc(smem_u32(&tail->tmem_base), 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = tail->tmem_base;

  if (warp == 0) {
    if (elect_one()) {
      uint32_t j = 0;
      for (int it = 0; it < my_tiles; ++it) {
        const size_t tile_off = (size_t)(args.tile0 + split + it * n_splits) * TC_DWL_TILE_BYTES;
        for (int pi = 0; pi < job.n_pairs; ++pi) {
          const TcDwPair pr = job.pair[pi];
          const size_t xo = (size_t)pr.x_arr * args.dwl_stride + tile_off + (size_t)job.half * 4096;
          const size_t yo = (size_t)(pr.y_arr < 0 ? 0 : pr.y_arr) * args.dwl_stride + tile_off;
          const uint32_t bytes = Cfg::kXBytes + (pr.y_arr >= 0 ? Cfg::kYBytes : 0);
          for (int ks = 0; ks < 8; ++ks, ++j) {
            const uint32_t stage = j % Cfg::kStages, ph = (j / Cfg::kStages) & 1;
            mbar_wait(smem_u32(&tail->empty[stage]), ph ^ 1);
            const uint32_t bar = smem_u32(&tail->full[stage]);
            const uint32_t dst = smem_u32(ring + stage * Cfg::kStageBytes);
            mbar_arrive_expect_tx(bar, bytes);
            bulk_g2s(dst, args.dwl_hi + xo + (size_t)ks * 8192, 4096, bar);
            if (kPasses == 3) bulk_g2s(dst + 4096, args.dwl_lo + xo + (size_t)ks * 8192, 4096, bar);
            if (pr.y_arr >= 0) {
              bulk_g2s(dst + Cfg::kXBytes, args.dwl_hi + yo + (size_t)ks * 8192, 8192, bar);
              if (kPasses == 3) bulk_g2s(dst + Cfg::kXBytes + 8192, args.dwl_lo + yo + (size_t)ks * 8192, 8192, bar);
            }
          }
        }
      }
    }
  } else if (warp == 1) {
    constexpr uint32_t idesc_main = umma_idesc_bf16(128, 256, 1, 1);
    constexpr uint32_t idesc_ones = umma_idesc_bf16(128, 16, 1, 1);
    uint32_t j = 0;
    uint32_t acc_main = 0, acc_ones[2] = {0, 0};
    const uint64_t b_ones = umma_desc(smem_u32(ones), 128, 256);
    for (int it = 0; it < my_tiles; ++it) {
      for (int pi = 0; pi < job.n_pairs; ++pi) {
        const TcDwPair pr = job.pair[pi];
        for (int ks = 0; ks < 8; ++ks, ++j) {
          const uint32_t stage = j % Cfg::kStages, ph = (j / Cfg::kStages) & 1;
          mbar_wait(smem_u32(&tail->full[stage]), ph);
          tc_fence_after();
          if (elect_one()) {
            const uint32_t base = smem_u32(ring + stage * Cfg::kStageBytes);
            const uint64_t ah = umma_desc(base, 128, 256);
            const uint64_t al = umma_desc(base + 4096, 128, 256);
            if (pr.y_arr >= 0) {
              const uint64_t bh = umma_desc(base + Cfg::kXBytes, 128, 256);
              tc_mma_f16(tmem, ah, bh, idesc_main, acc_main);
              if (kPasses == 3) {
                const uint64_t bl = umma_desc(base + Cfg::kXBytes + 8192, 128, 256);
                tc_mma_f16(tmem, al, bh, idesc_main, 1);
                tc_mma_f16(tmem, ah, bl, idesc_main, 1);
              }
            }
            if (pr.ones) {
              const uint32_t d = tmem + 256 + (pr.ones - 1) * 16;
              tc_mma_f16(d, ah, b_ones, idesc_ones, acc_ones[pr.ones - 1]);
              if (kPasses == 3) tc_mma_f16(d, al, b_ones, idesc_ones, 1);
            }
            tc_commit(smem_u32(&tail->empty[stage]));
          }
          __syncwarp();
          if (pr.y_arr >= 0) acc_main = 1;
          if (pr.ones) acc_ones[pr.ones - 1] = 1;
        }
      }
    }
    if (my_tiles > 0 && elect_one()) tc_commit(smem_u32(&tail->done));
    __syncwarp();
  } else if (my_tiles > 0) {
    // flush: TMEM -> red.global.add into the packed gradient
    mbar_wait(smem_u32(&tail->done), 0);
    tc_fence_after();
    const int q = warp & 3;
    const uint32_t lane_addr = (uint32_t)(q * 32) << 16;
    const int row = job.half * 128 + q * 32 + lane;
    bool has_main = false, has_db = false, has_dw = false;
    for (int pi = 0; pi < job.n_pairs; ++pi) {
      has_main |= job.pair[pi].y_arr >= 0;
      has_db |= job.pair[pi].ones == 1;
      has_dw |= job.pair[pi].ones == 2;
    }
    float v[32];
    if (has_main) {
      float* grow = args.g_packed + job.g_off + (size_t)row * job.ld;
#pragma unroll 1
      for (int c = 0; c < 8; ++c) {
        tmem_ld32(tmem + lane_addr + c * 32, v);
        if (job.perm_half > 0) {     // embedding-fed unit: internal column order -> the reference's (pe_nat_col)
#pragma unroll
          for (int i = 0; i < 32; ++i) {
            const int nat = pe_nat_col(job.col0 + c * 32 + i, job.perm_half);
            if (nat < job.ld) grad_add(grow + nat, v[i], 0);      // internal padding columns have no home (and are zero)
          }
          continue;
        }
#pragma unroll
        for (int i = 0; i < 8; ++i) grad_add4(grow + c * 32 + i * 4, v[i * 4], v[i * 4 + 1], v[i * 4 + 2], v[i * 4 + 3], 0);
      }
    }
    if (has_db || has_dw) {
      tmem_ld32(tmem + lane_addr + 256, v);
      if (has_db) grad_add(args.g_packed + job.db_off + row, v[0], 0);
      if (has_dw) grad_add(args.g_packed + args.wout_off + row, args.scale_output * v[16], 0);
    }
    tc_fence_before();
  }
  if (args.g_mc && warp >= 2) {
    // C1 fused: the LAST CTA of a job (over all launches of the step) forwards the job's finished 128 x 256 tile
    // from the local staging buffer to every rank's gradient through the NVLink-multicast alias (multimem.red)
    // and clears the stage for the next step: 2 MB per rank per step cross the fabric, tile by tile as jobs finish.
    __shared__ int s_last;
    __threadfence();
    named_bar_sync(2, 128);
    if (threadIdx.x == 64) {
      const int prev = (my_tiles > 0) ? atomicAdd(args.counters + job_id, 1) : -1;
      s_last = (prev == args.expect[job_id] - 1) ? 1 : 0;
      if (s_last) args.counters[job_id] = 0;
    }
    named_bar_sync(2, 128);
    if (s_last) {
      __threadfence();
      const int q = warp & 3;
      const int row = job.half * 128 + q * 32 + lane;
      bool has_main = false, has_db = false, has_dw = false;
      for (int pi = 0; pi < job.n_pairs; ++pi) {
        has_main |= job.pair[pi].y_arr >= 0;
        has_db |= job.pair[pi].ones == 1;
        has_dw |= job.pair[pi].ones == 2;
      }
      if (has_main) {
        // the tile's 128 rows x 256 floats, 2 KB (two rows) per pass of the 128 flush threads, 8 loads in flight
        const int t = threadIdx.x - 64;                 // 0..127
        const size_t base = job.g_off + (size_t)(job.half * 128) * job.ld;
        float4* src = reinterpret_cast<float4*>(args.g_packed + base) + t;
        float* dst = args.g_mc_out + base + (size_t)t * 4;
#pragma unroll 1
        for (int it = 0; it < 64; it += 8) {
          float4 r[8];
#pragma unroll
          for (int u = 0; u < 8; ++u) r[u] = __ldcg(src + (size_t)(it + u) * 128);
#pragma unroll
          for (int u = 0; u < 8; ++u) {
            grad_add4(dst + (size_t)(it + u) * 512, r[u].x, r[u].y, r[u].z, r[u].w, 1);
            __stcg(src + (size_t)(it + u) * 128, make_float4(0.f, 0.f, 0.f, 0.f));
          }
        }
      }
      if (has_db) {
        float* p = args.g_packed + job.db_off + row;
        grad_add(args.g_mc_out + job.db_off + row, __ldcg(p), 1);
        __stcg(p, 0.f);
      }
      if (has_dw) {
        float* p = args.g_packed + args.wout_off + row;
        grad_add(args.g_mc_out + args.wout_off + row, __ldcg(p), 1);
        __stcg(p, 0.f);
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem, 512);
}

int tc_dw_launch(isdfb_ctx* ctx, const TcDwArgs& args, int passes, int grid, cudaStream_t st) {
  if (passes == 3) {
    tc_dw_kernel<3><<<grid, DW_THREADS, DwCfg<3>::kSmem, st>>>(args);
  } else {
    tc_dw_kernel<1><<<grid, DW_THREADS, DwCfg<1>::kSmem, st>>>(args);
  }
  ISDFB_LAUNCHED(ctx);
  ISDFB_CUDA_OK(ctx, cudaGetLastError());
  return ISDFB_OK;
}

int tc_dw_init(isdfb_ctx* ctx) {
  ISDFB_CUDA_OK(ctx, cudaFuncSetAttribute(tc_dw_kernel<3>, cudaFuncAttributeMaxDynamicSharedMemorySize, DwCfg<3>::kSmem));
  ISDFB_CUDA_OK(ctx, cudaFuncSetAttribute(tc_dw_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, DwCfg<1>::kSmem));
  return ISDFB_OK;
}
