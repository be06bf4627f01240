// K2/K3/K4 on tcgen05: one persistent kernel runs, for a 128-point tile, the whole chain
//   PE -> S1 (forward) -> S2 (input gradient) -> loss -> S3 -> S4   (SURVEY.md 8a, A4-A9)
// as a sequence of 128x256x256 UMMA products whose accumulators live in TMEM (two 256-column
// buffers, ping-pong) and whose A operand (the activations) stays in shared memory: the epilogue of
// step s reads D_s from TMEM, applies the element-wise stage (softplus / sigmoid products / loss),
// and writes the A operand of step s+1 in place.  Weights stream from L2 through a ring of bulk
// (TMA) copies of pre-packed operand images, one UMMA K-step (16) per stage.
//
// Warp roles (640 threads):
//   warps 0-15  epilogue: warp w owns TMEM lane quadrant w%4 (points 32(w%4)..+31) and 16 of the 64
//               columns of every K chunk of the next step's A operand; 4 warps per scheduler hide the
//               ALU/SFU/LSU latency of the element-wise math; chunk 0 of the next A operand is done
//               after a quarter of the epilogue, so the next MMA runs under the rest of it;
//   warp 16     MMA issuer (+ TMEM alloc);      warp 17   weight producer (+ L2 prefetch of side arrays);
//   warps 18-19 idle: they complete the helper WARPGROUP, which hands registers back (setmaxnreg.dec 32) so
//               that the four epilogue warpgroups can grow from the launch-time 96 to 112 registers per thread
//               (the launch bound is 65536 / 640 threads) -- room for operand prefetch two sub-pieces ahead.
//
// Precision: kPasses = 3 -> every product is A_hi*B_hi + A_lo*B_hi + A_hi*B_lo with bf16 hi/lo splits
// and fp32 accumulation (~fp32 accuracy); kPasses = 1 -> single bf16 pass (fast mode).
// kLean (precision "bf16x3g", the default): the per-point side state handed to the weight-gradient kernel, the S3
// read-back of delta_l and zbar2_l are single bf16 -- half the HBM traffic, sdf / d sdf/dx / losses unchanged.
// kNE = embedding halves of 256 internal columns (2: E = 381 / 465 of the realsense / franka configs): every
// embedding-fed product is then two products whose partial results are parked (EPI_RAW) and added (TcStep::addp).
// The step program itself is built on the host (tc_path.cu build_program; pinned by tests/test_abi.py).
#include "tc_chain.cuh"
#include "pe_loss.cuh"

#define EPI_WARPS 16
#define EPI_THREADS (EPI_WARPS * 32)
#define NUM_THREADS (EPI_THREADS + 128)   // + one helper warpgroup: MMA issuer, weight producer, two idle warps
#define EPI_REGS 112                     // setmaxnreg moves registers inside the CTA's launch-time pool (640 x 96):
#define HELPER_REGS 32                   // 512 x 112 + 128 x 32 = 61 440 = 640 x 96 exactly
#define K_STEP 16                        // K elements per weight-ring stage (one UMMA K step)
#define N_KSTEPS (TC_H / K_STEP)         // 16
#define A_IMG_BYTES (TC_TILE * TC_H * 2) // 64 KB
#define A_LBO (TC_TILE * 16)             // 2048
#define B_LBO (TC_H * 16)                // 4096
#define KSTEP_IMG_BYTES (TC_H * K_STEP * 2)   // 8 KB per precision part
#define SCRATCH_BYTES 8192

template <int kPasses> struct ChainCfg {
  static constexpr int kStageBytes = KSTEP_IMG_BYTES * (kPasses == 3 ? 2 : 1);
  static constexpr int kStages = (kPasses == 3) ? 5 : 8;
  static constexpr int kABytes = A_IMG_BYTES * (kPasses == 3 ? 2 : 1);
  static constexpr int kSmem = kABytes + kStages * kStageBytes + SCRATCH_BYTES + 256;
};

struct ChainSmemTail {       // lives after the operand buffers and the scratch
  uint64_t w_full[8], w_empty[8], a_ready[4], d_full[2];
  uint32_t tmem_base;
};

__device__ __forceinline__ float4 ld4(const float* p) { return *reinterpret_cast<const float4*>(p); }
// 16-byte load of per-tile side state: read once, never re-used by this SM -> do not allocate in the (tiny:
// 228 KB - 216 KB of shared memory) L1, whose lines would otherwise all be tied up by in-flight fills
__device__ __forceinline__ uint4 ld_stream(const void* p) {
  uint4 v;
  asm("ld.global.L1::no_allocate.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p));
  return v;
}
__device__ __forceinline__ void st4(float* p, float a, float b, float c, float d) {
  *reinterpret_cast<float4*>(p) = make_float4(a, b, c, d);
}

// ---------------------------------------------------------------------------------------------
// epilogue building blocks.  Thread (q, jg) handles point p = 32q + lane and, in every 64-column
// K chunk c, the 16 columns [64c + 16jg, +16) as two 8-column sub-pieces h = 0, 1.
// ---------------------------------------------------------------------------------------------
struct EpiT {                       // per-thread / per-tile constants (thread offsets folded in)
  uint8_t *a_hi, *a_lo;             // smem A images  + p*16 + (2 jg) A_LBO
  uint8_t *dwl_hi, *dwl_lo;         // dW-layout array 0 + tile + (p>>4) 8192 + (p&15) 16 + (2 jg) 256
  float* aux;                       // aux array 0 + tile + p*4 + (4 jg) 512        (floats)
  uint8_t* sig;                     // sigma16 layer 0 + tile + p*16 + (2 jg) 2048
  uint8_t* zb2h;                    // lean: zbar2 (bf16) layer 0, same addressing as sig
  size_t dwl_stride, aux_stride, sig_stride;
  int p, kcol;                      // kcol = 16 jg
  int c0;                           // first K chunk of this CTA's rotated order (rot_kstep)
};
struct EpiOps { uint4 s, b0, b1, e0, e1; };   // side-array operands of one sub-piece (e0/e1: own embedding values, S2_END)
struct EpiStepPtrs {                  // per-step pointers (thread offsets included)
  const uint8_t* sigp; uint8_t* sigw;
  const uint8_t *dhi, *dlo;           // delta_l (dW layout) for S3
  float* zb2;                         // zbar2_l  (fp32 side array; strict mode)
  uint8_t* zb2h;                      // zbar2_l  (bf16, sigma-image layout; lean mode)
  const float* part_in;               // partial sums consumed by this step
  float* part_out;                    // RAW: partial sums produced
  const float *bias, *wout;
  float* hlast;
  const float* e32;                   // this thread's slice of the fp32 embedding side array (same offsets as aux)
  int flags;                          // TcStep::flags (STF_*)
  int ecol0;                          // EPI_S2_END: first internal embedding column of this step's outputs (256 * eh)
};
__device__ __forceinline__ uint32_t sub_a(int c, int h) { return (uint32_t)(8 * c + h) * A_LBO; }
__device__ __forceinline__ uint32_t sub_d(int c, int h) { return (uint32_t)(8 * c + h) * 256u; }
__device__ __forceinline__ uint32_t sub_x(int c, int h) { return (uint32_t)(16 * c + 2 * h) * 512u; }

// kLean: the weight-gradient operands (dW layout) keep only their bf16 hi part -- the products of S1..S4 themselves
// stay hi/lo (A image), so sdf, d sdf/dx and the loss are unchanged; only dW sees the rounding.
template <int kPasses, bool kLean>
__device__ __forceinline__ void put8(const EpiT& T, const float* x, int c, int h, bool to_a, int dwl_arr) {
  uint4 hi, lo;
  if (kPasses == 3 && (to_a || !kLean)) split8(x, hi, lo); else hi = pack8_hi(x);
  if (to_a) {
    *reinterpret_cast<uint4*>(T.a_hi + sub_a(c, h)) = hi;
    if (kPasses == 3) *reinterpret_cast<uint4*>(T.a_lo + sub_a(c, h)) = lo;
  }
  if (dwl_arr >= 0) {
    const size_t off = (size_t)dwl_arr * T.dwl_stride + sub_d(c, h);
    *reinterpret_cast<uint4*>(T.dwl_hi + off) = hi;
    if (kPasses == 3 && !kLean) *reinterpret_cast<uint4*>(T.dwl_lo + off) = lo;
  }
}

template <int EPI, int kPasses, bool kLean>
__device__ __forceinline__ void epi_load(const EpiStepPtrs& P, bool l_is_cat, int c, int h, EpiOps& o) {
  auto ld = [&](const void* q) -> uint4 { return ld_stream(q); };   // read-once side state: never allocates in L1
  if (EPI == EPI_S2 || EPI == EPI_S3 || EPI == EPI_S3_LAST || EPI == EPI_S4)
    o.s = ld(P.sigp + sub_a(c, h));
  if (EPI == EPI_S3 || EPI == EPI_S3_LAST) {
    o.b0 = ld(P.dhi + sub_d(c, h));
    if (kPasses == 3 && !kLean) o.b1 = ld(P.dlo + sub_d(c, h));
  } else if (EPI == EPI_S4) {
    if (kLean) {
      o.b0 = ld(P.zb2h + sub_a(c, h));
    } else {
      o.b0 = ld(P.zb2 + sub_x(c, h));
      o.b1 = ld(P.zb2 + sub_x(c, h) + 512);
    }
  } else if (EPI == EPI_S2_END || ((EPI == EPI_S1 || EPI == EPI_S1_LAST) && l_is_cat)) {
    o.b0 = ld(P.part_in + sub_x(c, h));
    o.b1 = ld(P.part_in + sub_x(c, h) + 512);
    if (EPI == EPI_S2_END) {
      o.e0 = ld(P.e32 + sub_x(c, h));
      o.e1 = ld(P.e32 + sub_x(c, h) + 512);
    }
  }
}

struct EpiAcc { float raw_acc, gx, gy, gz; };

// Per-CTA rotation of the K order of every product: CTA b walks the four 64-column K chunks
// starting at chunk (b/4)%4 and the four K steps inside a chunk starting at b%4.  All CTAs stream the SAME
// weight images from L2 at the same pace; without the rotation the 148 SMs ask the same L2 lines for the same
// 8 KB block at the same moment and queue behind each other (measured: 12 k cycles per step for the weight
// ring alone).  The sum over K is order-independent up to fp32 rounding.
__device__ __forceinline__ int rot_kstep(int ks, int rot) {
  return ((((ks >> 2) + (rot >> 2)) & 3) << 2) | (((ks & 3) + rot) & 3);
}

template <int EPI, int kPasses, bool kLean, int kNE>
__device__ __forceinline__ void epi_sub(const TcChainArgs& args, const EpiT& T, const EpiStepPtrs& P, const EpiOps& o,
                                        float* v /* 8 accumulator columns of this sub-piece */, int c, int h, int l,
                                        bool l_is_cat, bool train, bool store_state, bool last_step, float sbar,
                                        EpiAcc& acc) {
  const int k0 = 64 * c + T.kcol + 8 * h;
  if (EPI == EPI_RAW) {
    if (kNE == 2 && (P.flags & STF_RAW_ADD)) {       // second embedding half: accumulate onto the parked partial product
      const float4 pa = ld4(P.part_out + sub_x(c, h)), pb = ld4(P.part_out + sub_x(c, h) + 512);
      v[0] += pa.x; v[1] += pa.y; v[2] += pa.z; v[3] += pa.w; v[4] += pb.x; v[5] += pb.y; v[6] += pb.z; v[7] += pb.w;
    }
    st4(P.part_out + sub_x(c, h), v[0], v[1], v[2], v[3]);
    st4(P.part_out + sub_x(c, h) + 512, v[4], v[5], v[6], v[7]);
  } else if (EPI == EPI_S1 || EPI == EPI_S1_LAST) {
    const float4 ba = ld4(P.bias + k0), bb = ld4(P.bias + k0 + 4);
    float z[8] = {v[0] + ba.x, v[1] + ba.y, v[2] + ba.z, v[3] + ba.w, v[4] + bb.x, v[5] + bb.y, v[6] + bb.z, v[7] + bb.w};
    if (l_is_cat) {
      z[0] += __uint_as_float(o.b0.x); z[1] += __uint_as_float(o.b0.y); z[2] += __uint_as_float(o.b0.z); z[3] += __uint_as_float(o.b0.w);
      z[4] += __uint_as_float(o.b1.x); z[5] += __uint_as_float(o.b1.y); z[6] += __uint_as_float(o.b1.z); z[7] += __uint_as_float(o.b1.w);
    }
    float hh[8], sg[8];
#pragma unroll
    for (int t = 0; t < 8; ++t) softplus100_fast(z[t], hh[t], sg[t]);
    if (store_state) *reinterpret_cast<uint4*>(P.sigw + sub_a(c, h)) = pack_unorm16x8(sg);
    if (EPI == EPI_S1) {
      put8<kPasses, kLean>(T, hh, c, h, true, (train && l + 1 < args.L) ? args.arr_yh + l + 1 : -1);
    } else {
      const float4 wa = ld4(P.wout + k0), wb = ld4(P.wout + k0 + 4);
      const float ww[8] = {wa.x, wa.y, wa.z, wa.w, wb.x, wb.y, wb.z, wb.w};
      if (train) {
        st4(P.hlast + sub_x(c, h), hh[0], hh[1], hh[2], hh[3]);
        st4(P.hlast + sub_x(c, h) + 512, hh[4], hh[5], hh[6], hh[7]);
      }
#pragma unroll
      for (int t = 0; t < 8; ++t) {
        acc.raw_acc = fmaf(hh[t], ww[t], acc.raw_acc);
        v[t] = args.scale_output * ww[t] * sg[t];          // delta_{L-1} = a_{L-1} * sigma
      }
      put8<kPasses, kLean>(T, v, c, h, args.mode != TC_MODE_FWD, train ? args.arr_xd + l : -1);
    }
  } else if (EPI == EPI_S2) {
    float sg[8];
    unpack_unorm16x8(o.s, sg);
#pragma unroll
    for (int t = 0; t < 8; ++t) v[t] *= sg[t];
    put8<kPasses, kLean>(T, v, c, h, true, train ? args.arr_xd + l : -1);
  } else if (EPI == EPI_S2_END) {
    // PE Jacobian in the internal column order (tc_common.cuh): columns (2i, 2i+1) = (sin, cos) of pair i, so
    // d e / d xb = (cos, -sin) is thread-local:  g_xs += D_d 2^f (cos a_sin - sin a_cos);  x y z follow the pairs
    const int two_half = 2 * ISDFB_NDIRS * args.pe.n_freqs;
    const float a[8] = {v[0] + __uint_as_float(o.b0.x), v[1] + __uint_as_float(o.b0.y), v[2] + __uint_as_float(o.b0.z), v[3] + __uint_as_float(o.b0.w),
                        v[4] + __uint_as_float(o.b1.x), v[5] + __uint_as_float(o.b1.y), v[6] + __uint_as_float(o.b1.z), v[7] + __uint_as_float(o.b1.w)};
    const float ev[8] = {__uint_as_float(o.e0.x), __uint_as_float(o.e0.y), __uint_as_float(o.e0.z), __uint_as_float(o.e0.w),
                         __uint_as_float(o.e1.x), __uint_as_float(o.e1.y), __uint_as_float(o.e1.z), __uint_as_float(o.e1.w)};
#pragma unroll
    for (int t = 0; t < 8; t += 2) {
      const int k = (kNE == 2 ? P.ecol0 : 0) + k0 + t;
      if (k < two_half) {
        const int pi = k >> 1, d = args.pair_d[pi];
        const float w = (ev[t + 1] * a[t] - ev[t] * a[t + 1]) * (float)(1 << args.pair_f[pi]);
        acc.gx = fmaf(w, c_ico[d][0], acc.gx);
        acc.gy = fmaf(w, c_ico[d][1], acc.gy);
        acc.gz = fmaf(w, c_ico[d][2], acc.gz);
      } else if (k == two_half) {
        acc.gx += a[t]; acc.gy += a[t + 1];
      } else if (k == two_half + 2) {
        acc.gz += a[t];
      }
    }
  } else if (EPI == EPI_S3 || EPI == EPI_S3_LAST) {
    float sg[8], dl[8], zb[8];
    unpack_unorm16x8(o.s, sg);
    unpack8(o.b0, dl);
    if (kPasses == 3 && !kLean) {
      float t8[8];
      unpack8(o.b1, t8);
#pragma unroll
      for (int t = 0; t < 8; ++t) dl[t] += t8[t];
    }
    if (l_is_cat) {
      const float4 pa = ld4(P.part_in + sub_x(c, h)), pb = ld4(P.part_in + sub_x(c, h) + 512);
      v[0] += pa.x; v[1] += pa.y; v[2] += pa.z; v[3] += pa.w; v[4] += pb.x; v[5] += pb.y; v[6] += pb.z; v[7] += pb.w;
    }
#pragma unroll
    for (int t = 0; t < 8; ++t) {
      const float om = 100.f * (1.f - sg[t]);   // sigma' / sigma; 0 in the saturated (linear) regime
      zb[t] = v[t] * dl[t] * om;           // zbar2 = dbar * delta * beta (1 - sigma)
      v[t] = v[t] * sg[t];                 // abar = dbar * sigma
    }
    if (EPI == EPI_S3) {
      if (kLean) {
        *reinterpret_cast<uint4*>(P.zb2h + sub_a(c, h)) = pack8_hi(zb);
      } else {
        st4(P.zb2 + sub_x(c, h), zb[0], zb[1], zb[2], zb[3]);
        st4(P.zb2 + sub_x(c, h) + 512, zb[4], zb[5], zb[6], zb[7]);
      }
      put8<kPasses, kLean>(T, v, c, h, true, (l + 1 < args.L) ? args.arr_ya + l + 1 : -1);
    } else {
      // v_blob = sbar * h_last + abar_last  (for d w_out);  A <- zbar_last = sbar c w_out sigma + zbar2
      const float4 ha = ld4(P.hlast + sub_x(c, h)), hb = ld4(P.hlast + sub_x(c, h) + 512);
      const float4 wa = ld4(P.wout + k0), wb = ld4(P.wout + k0 + 4);
      const float hh[8] = {ha.x, ha.y, ha.z, ha.w, hb.x, hb.y, hb.z, hb.w};
      const float ww[8] = {wa.x, wa.y, wa.z, wa.w, wb.x, wb.y, wb.z, wb.w};
      float vb[8];
#pragma unroll
      for (int t = 0; t < 8; ++t) {
        vb[t] = fmaf(sbar, hh[t], v[t]);
        zb[t] = fmaf(sbar * args.scale_output * ww[t], sg[t], zb[t]);
      }
      put8<kPasses, kLean>(T, vb, c, h, false, args.arr_v);
      put8<kPasses, kLean>(T, zb, c, h, true, args.arr_xz + l);
    }
  } else {   // EPI_S4
    float sg[8];
    unpack_unorm16x8(o.s, sg);
    float z2[8];
    if (kLean) {
      unpack8(o.b0, z2);
    } else {
      z2[0] = __uint_as_float(o.b0.x); z2[1] = __uint_as_float(o.b0.y); z2[2] = __uint_as_float(o.b0.z); z2[3] = __uint_as_float(o.b0.w);
      z2[4] = __uint_as_float(o.b1.x); z2[5] = __uint_as_float(o.b1.y); z2[6] = __uint_as_float(o.b1.z); z2[7] = __uint_as_float(o.b1.w);
    }
#pragma unroll
    for (int t = 0; t < 8; ++t) v[t] = fmaf(v[t], sg[t], z2[t]);
    put8<kPasses, kLean>(T, v, c, h, !last_step, args.arr_xz + l);
  }
}

// one whole step of the epilogue for this thread (8 sub-pieces), operands fetched two sub-pieces ahead
template <int EPI, int kPasses, bool kLean, int kNE>
__device__ __forceinline__ void epi_step(const TcChainArgs& args, const EpiT& T, const EpiStepPtrs& P, ChainSmemTail* tail,
                                         uint32_t d_tmem, uint32_t n, int l, bool train, bool store_state, bool last_step,
                                         float sbar, EpiAcc& acc, int lane) {
  const bool l_is_cat = P.part_in != nullptr;        // "a parked partial product is added" (concat layer, 2nd embedding half)
  // A operand left untouched by this epilogue -> the next step's MMA may start at once
  const bool early_release = (EPI == EPI_RAW && (kNE == 1 || !(P.flags & (STF_PE_E | STF_PE_ABAR)))) ||
                             (EPI == EPI_S2_END && kNE == 2 && !(P.flags & STF_END_LAST) && !last_step);
  const bool chunk_release = EPI != EPI_RAW && EPI != EPI_S2_END && !last_step;
  EpiOps oa, ob;
  oa.s = oa.b0 = oa.b1 = oa.e0 = oa.e1 = make_uint4(0, 0, 0, 0);
  ob = oa;
  epi_load<EPI, kPasses, kLean>(P, l_is_cat, T.c0, 0, oa);         // overlaps the tail of this step's MMA
  mbar_wait(smem_u32(&tail->d_full[n & 1]), (n >> 1) & 1);
  tc_fence_after();
  if (early_release) {
    // A is left untouched: release the next step now (its MMA overlaps this drain of D into a side
    // array).  Arriving only after d_full guarantees every warp finished the previous phase.
    __syncwarp();
    if (lane == 0) {
#pragma unroll
      for (int c = 0; c < 4; ++c) mbar_arrive(smem_u32(&tail->a_ready[c]));
    }
  }
  // operands of BOTH sub-pieces of the next chunk are requested before this chunk is processed: two sub-pieces
  // of lead on the side-state loads (L2 latency under load exceeds one) at the price of two more operand sets
  epi_load<EPI, kPasses, kLean>(P, l_is_cat, T.c0, 1, ob);
#pragma unroll 1
  for (int ci = 0; ci < 4; ++ci) {
    const int c = (ci + T.c0) & 3;
    EpiOps na = oa, nb = ob;
    if (ci < 3) {
      epi_load<EPI, kPasses, kLean>(P, l_is_cat, (c + 1) & 3, 0, na);
      epi_load<EPI, kPasses, kLean>(P, l_is_cat, (c + 1) & 3, 1, nb);
    }
    float v[8];
    tmem_ld8(d_tmem + 64 * c + T.kcol, v);
    epi_sub<EPI, kPasses, kLean, kNE>(args, T, P, oa, v, c, 0, l, l_is_cat, train, store_state, last_step, sbar, acc);
    tmem_ld8(d_tmem + 64 * c + T.kcol + 8, v);
    epi_sub<EPI, kPasses, kLean, kNE>(args, T, P, ob, v, c, 1, l, l_is_cat, train, store_state, last_step, sbar, acc);
    if (chunk_release) {
      fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) mbar_arrive(smem_u32(&tail->a_ready[c]));
    }
    oa = na; ob = nb;
  }
  tc_fence_before();
}

// kNE = embedding halves of 256 internal columns the program was built for (1: E <= 256 -- every shipped default
// config; 2: E <= 512).  A template parameter so that the single-half kernel carries none of the second half's
// run-time flag tests (they cost 2.6 % of the default workload's kernel time when they were run-time only).
template <int kPasses, bool kLean, int kNE>
__global__ void __launch_bounds__(NUM_THREADS, 1) tc_chain_kernel(const __grid_constant__ TcChainArgs args) {
  using Cfg = ChainCfg<kPasses>;
  extern __shared__ __align__(1024) uint8_t smem[];
  uint8_t* a_hi = smem;
  uint8_t* a_lo = smem + A_IMG_BYTES;                         // only valid when kPasses == 3
  uint8_t* w_ring = smem + Cfg::kABytes;
  float* red = reinterpret_cast<float*>(smem + Cfg::kABytes + Cfg::kStages * Cfg::kStageBytes);   // [3][4][128]
  float* bcast = red + 3 * 4 * 128;                                                               // [128][4]
  ChainSmemTail* tail = reinterpret_cast<ChainSmemTail*>(reinterpret_cast<uint8_t*>(red) + SCRATCH_BYTES);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n_steps = args.n_steps;

  if (threadIdx.x == 0) {
    for (int i = 0; i < Cfg::kStages; ++i) { mbar_init(smem_u32(&tail->w_full[i]), 1); mbar_init(smem_u32(&tail->w_empty[i]), 1); }
    for (int i = 0; i < 4; ++i) mbar_init(smem_u32(&tail->a_ready[i]), EPI_WARPS);
    for (int i = 0; i < 2; ++i) mbar_init(smem_u32(&tail->d_full[i]), 1);
    mbar_fence_init();
  }
  if (warp == EPI_WARPS) tmem_alloc(smem_u32(&tail->tmem_base), 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = tail->tmem_base;

  const int rot = (int)(blockIdx.x & 15u);
  const int my_tiles = (args.n_tiles > (int)blockIdx.x) ? (args.n_tiles - 1 - (int)blockIdx.x) / (int)gridDim.x + 1 : 0;

  // (setmaxnreg sits INSIDE each role branch: ptxas budgets registers per branch only when the re-allocation
  // dominates the branch; placed before the dispatch it constrains the whole kernel to the smallest value)
  if (warp >= EPI_WARPS + 2) {
    reg_dec<HELPER_REGS>();          // idle warps of the helper warpgroup
  } else if (warp == EPI_WARPS + 1) {
    reg_dec<HELPER_REGS>();
    // ===================== weight producer =====================
    if (elect_one()) {
      uint32_t j = 0;
      for (int it = 0; it < my_tiles; ++it) {
        const int tile = args.tile0 + blockIdx.x + it * gridDim.x;
        for (int s = 0; s < n_steps; ++s) {
          const TcStep st = args.steps[s];
          if (s + 1 < n_steps) {
            // pull the side arrays the NEXT step's epilogue will read from HBM into L2 while this step runs
            const TcStep nx = args.steps[s + 1];
            const float* aux_t = args.aux + (size_t)tile * TC_TILE_FLOATS;
            const size_t dwl_t = (size_t)tile * TC_DWL_TILE_BYTES;
            auto pf_aux = [&](int arr) { bulk_prefetch_l2(aux_t + (size_t)arr * args.aux_stride, TC_TILE_FLOATS * 4); };
            auto pf_sig = [&](int l_) { bulk_prefetch_l2(args.sig16 + (size_t)l_ * args.sig16_stride + dwl_t, TC_DWL_TILE_BYTES); };
            auto pf_dwl = [&](int arr) {
              bulk_prefetch_l2(args.dwl_hi + (size_t)arr * args.dwl_stride + dwl_t, TC_DWL_TILE_BYTES);
              if (kPasses == 3 && !kLean) bulk_prefetch_l2(args.dwl_lo + (size_t)arr * args.dwl_stride + dwl_t, TC_DWL_TILE_BYTES);
            };
            auto pf_zb2 = [&](int l_) {
              if (kLean) bulk_prefetch_l2(args.zb2h + (size_t)l_ * args.sig16_stride + dwl_t, TC_DWL_TILE_BYTES);
              else pf_aux(args.arr_zb2 + l_);
            };
            switch (nx.epi) {
              case EPI_S1: case EPI_S1_LAST: if (nx.addp >= 0) pf_aux(args.arr_part + nx.addp); break;
              case EPI_S2: pf_sig(nx.layer); break;
              case EPI_S2_END: pf_aux(args.arr_part + nx.addp); pf_aux(args.arr_e32 + nx.eh); break;
              case EPI_S3: case EPI_S3_LAST:
                pf_sig(nx.layer); pf_dwl(args.arr_xd + nx.layer);
                if (nx.addp >= 0) pf_aux(args.arr_part + nx.addp);
                if (nx.epi == EPI_S3_LAST) pf_aux(args.arr_hlast);
                break;
              case EPI_S4: pf_sig(nx.layer); pf_zb2(nx.layer); break;
              default: break;
            }
          }
          const uint8_t* img_hi = args.w_img + ((size_t)(st.unit * 2 + st.orient) * 2 + 0) * TC_IMG_BYTES;
          const uint8_t* img_lo = img_hi + TC_IMG_BYTES;
          for (int ks = 0; ks < N_KSTEPS; ++ks, ++j) {
            const uint32_t stage = j % Cfg::kStages, ph = (j / Cfg::kStages) & 1;
            mbar_wait(smem_u32(&tail->w_empty[stage]), ph ^ 1);
            const uint32_t bar = smem_u32(&tail->w_full[stage]);
            const uint32_t dst = smem_u32(w_ring + stage * Cfg::kStageBytes);
            const int kse = rot_kstep(ks, rot);
            mbar_arrive_expect_tx(bar, Cfg::kStageBytes);
            bulk_g2s(dst, img_hi + (size_t)kse * KSTEP_IMG_BYTES, KSTEP_IMG_BYTES, bar);
            if (kPasses == 3) bulk_g2s(dst + KSTEP_IMG_BYTES, img_lo + (size_t)kse * KSTEP_IMG_BYTES, KSTEP_IMG_BYTES, bar);
          }
        }
      }
    }
  } else if (warp == EPI_WARPS) {
    reg_dec<HELPER_REGS>();
    // ===================== MMA issuer =====================
    constexpr uint32_t idesc = umma_idesc_bf16(128, 256, 0, 0);
    uint32_t j = 0, n = 0;
    for (int it = 0; it < my_tiles; ++it) {
      for (int s = 0; s < n_steps; ++s, ++n) {
        const uint32_t d_tmem = tmem + (n & 1) * 256;
        for (int ks = 0; ks < N_KSTEPS; ++ks, ++j) {
          const int kse = rot_kstep(ks, rot);
          if ((ks & 3) == 0) mbar_wait(smem_u32(&tail->a_ready[kse >> 2]), n & 1);
          const uint32_t stage = j % Cfg::kStages, ph = (j / Cfg::kStages) & 1;
          mbar_wait(smem_u32(&tail->w_full[stage]), ph);
          tc_fence_after();
          if (elect_one()) {
            const uint32_t b_base = smem_u32(w_ring + stage * Cfg::kStageBytes);
            const uint64_t ah = umma_desc(smem_u32(a_hi) + kse * 2 * A_LBO, A_LBO, 128);
            const uint64_t bh = umma_desc(b_base, B_LBO, 128);
            tc_mma_f16(d_tmem, ah, bh, idesc, ks != 0);
            if (kPasses == 3) {
              const uint64_t al = umma_desc(smem_u32(a_lo) + kse * 2 * A_LBO, A_LBO, 128);
              const uint64_t bl = umma_desc(b_base + KSTEP_IMG_BYTES, B_LBO, 128);
              tc_mma_f16(d_tmem, al, bh, idesc, 1);
              tc_mma_f16(d_tmem, ah, bl, idesc, 1);
            }
            tc_commit(smem_u32(&tail->w_empty[stage]));
            if (ks == N_KSTEPS - 1) tc_commit(smem_u32(&tail->d_full[n & 1]));
          }
          __syncwarp();
        }
      }
    }
  } else {
    reg_inc<EPI_REGS>();
    // ===================== epilogue: thread = (point, 4 x 16 columns) =====================
    // Warp (q, jg) owns points 32q..32q+31 and, inside every 64-column K chunk c of the next A operand,
    // columns [64c+16jg, 64c+16jg+16): chunk 0 is complete after a quarter of the epilogue, so the MMA
    // of the next step runs under the rest of it.
    const int q = warp & 3, jg = warp >> 2;
    const int p = q * 32 + lane;                                  // row / TMEM lane
    const uint32_t lane_addr = (uint32_t)(q * 32) << 16;
    const float c_out = args.scale_output;
    const float* Wp = args.w_packed;
    const int two_half = 2 * ISDFB_NDIRS * args.pe.n_freqs;      // internal columns [0, two_half) are (sin, cos) pairs
    const bool train = args.mode == TC_MODE_TRAIN;
    const bool store_state = args.mode != TC_MODE_FWD;
    uint32_t n = 0;
    float lsum0 = 0.f, lsum1 = 0.f, lsum2 = 0.f, lsum3 = 0.f, sbsum = 0.f;

    for (int it = 0; it < my_tiles; ++it) {
      const int tile = args.tile0 + blockIdx.x + it * gridDim.x;
      const int64_t pl = (int64_t)tile * TC_TILE + p;             // point index inside the chunk
      const bool real = pl < args.n_points;
      EpiT T;
      T.p = p; T.kcol = 16 * jg; T.c0 = rot >> 2;
      T.a_hi = a_hi + p * 16 + (2 * jg) * A_LBO;
      T.a_lo = a_lo + p * 16 + (2 * jg) * A_LBO;
      const size_t dthr = (size_t)tile * TC_DWL_TILE_BYTES + (size_t)(p >> 4) * 8192u + (size_t)(p & 15) * 16u + (size_t)(2 * jg) * 256u;
      T.dwl_hi = args.dwl_hi + dthr;
      T.dwl_lo = args.dwl_lo + dthr;
      T.aux = args.aux + (size_t)tile * TC_TILE_FLOATS + p * 4 + (4 * jg) * 512;
      T.sig = args.sig16 + (size_t)tile * TC_DWL_TILE_BYTES + p * 16 + (2 * jg) * 2048;
      T.zb2h = args.zb2h + (size_t)tile * TC_DWL_TILE_BYTES + p * 16 + (2 * jg) * 2048;
      T.dwl_stride = args.dwl_stride; T.aux_stride = args.aux_stride; T.sig_stride = args.sig16_stride;
      float* e32_w = T.aux + (size_t)args.arr_e32 * args.aux_stride;
      auto chunk_ready = [&](int c) {
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) mbar_arrive(smem_u32(&tail->a_ready[c]));
      };

      // ---------------- PE stage: x -> e (A operand of the first step) ----------------
      float xs[3] = {0.f, 0.f, 0.f};
      if (real) {
        float xw0, xw1, xw2;
        if (args.grid.dim > 0) {             // lattice point (i, j, k) of torch.meshgrid(t, t, t), 'ij' order
          const int64_t pg = args.p0 + pl;
          const int d = args.grid.dim;
          const int64_t r = pg / d;
          const int k = (int)(pg - r * d), i = (int)(r / d), j = (int)(r - (int64_t)i * d);
          const float gx = __fmul_rn(args.grid.lin[i], args.grid.scale[0]);
          const float gy = __fmul_rn(args.grid.lin[j], args.grid.scale[1]);
          const float gz = __fmul_rn(args.grid.lin[k], args.grid.scale[2]);
          xw0 = gx; xw1 = gy; xw2 = gz;
          if (args.grid.has_transform) {     // (R_row * g).sum(-1) + t   (transform.py:291-302)
            const float* R = args.grid.R;
            xw0 = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(R[0], gx), __fmul_rn(R[1], gy)), __fmul_rn(R[2], gz)), args.grid.t[0]);
            xw1 = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(R[3], gx), __fmul_rn(R[4], gy)), __fmul_rn(R[5], gz)), args.grid.t[1]);
            xw2 = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(R[6], gx), __fmul_rn(R[7], gy)), __fmul_rn(R[8], gz)), args.grid.t[2]);
          }
        } else {
          const float* xp = args.x + pl * 3;
          xw0 = xp[0]; xw1 = xp[1]; xw2 = xp[2];
        }
        pe_scale_input(args.pe, xw0, xw1, xw2, xs);
      }
      // per-point state carried across steps
      float sdf_reg = 0.f, sbar = 0.f, u3[3] = {0.f, 0.f, 0.f};
      // embedding half eh (internal columns [256 eh, 256 eh + 256)) -> A image, its dW-layout copy and the fp32 side
      // array the PE Jacobian / its adjoint read back.  Called at the start of the tile (eh = 0) and, for padded
      // embeddings wider than 256, from the EPI_RAW step that parks the first half's partial product (STF_PE_E).
      auto write_e_half = [&](int eh) {
        float* e32_h = e32_w + (size_t)eh * args.aux_stride;
#pragma unroll 1
        for (int i = 0; i < 8; ++i) {
          const int c = i >> 1, h = i & 1;
          const int k0 = 256 * eh + 64 * c + T.kcol + 8 * h;
          float v[8];
#pragma unroll
          for (int jj = 0; jj < 8; jj += 2) {         // internal column order: (sin, cos) pairs, then x y z, then padding
            const int k = k0 + jj;
            float va = 0.f, vb = 0.f;
            if (real) {
              if (k < two_half) {
                const int pi = k >> 1;
                const float xb = pe_project(xs, args.pair_d[pi]) * (float)(1 << args.pair_f[pi]);
                va = sinf(xb);
                vb = sinf(__fadd_rn(xb, ISDFB_HALF_PI_F));
              } else if (k == two_half) {
                va = xs[0]; vb = xs[1];
              } else if (k == two_half + 2) {
                va = xs[2];
              }
            }
            v[jj] = va; v[jj + 1] = vb;
          }
          put8<kPasses, kLean>(T, v, c, h, true, train ? (eh ? args.arr_yh_e1 : args.arr_yh) : -1);
          if (store_state) {
            st4(e32_h + sub_x(c, h), v[0], v[1], v[2], v[3]);
            st4(e32_h + sub_x(c, h) + 512, v[4], v[5], v[6], v[7]);
          }
          if (h) chunk_ready(c);
        }
      };
      // adjoint of the embedding half eh, abar_e = (u . D_d) 2^f (cos, -sin) | u, -> A image (+ its dW-layout copy)
      auto write_abar_half = [&](int eh) {
        const float* e32_h = e32_w + (size_t)eh * args.aux_stride;
        float4 ea = ld4(e32_h + sub_x(0, 0)), eb = ld4(e32_h + sub_x(0, 0) + 512);
#pragma unroll 1
        for (int i = 0; i < 8; ++i) {
          const int c = i >> 1, h = i & 1;
          const int k0 = 256 * eh + 64 * c + T.kcol + 8 * h;
          const float ev[8] = {ea.x, ea.y, ea.z, ea.w, eb.x, eb.y, eb.z, eb.w};
          if (i < 7) {                       // own embedding values of the next sub-piece, one ahead
            const int cn = (i + 1) >> 1, hn = (i + 1) & 1;
            ea = ld4(e32_h + sub_x(cn, hn));
            eb = ld4(e32_h + sub_x(cn, hn) + 512);
          }
          float v[8];
#pragma unroll
          for (int jj = 0; jj < 8; jj += 2) {
            const int k = k0 + jj;
            float va = 0.f, vb = 0.f;
            if (k < two_half) {       // abar_e = (u . D_d) 2^f (cos, -sin)
              const int pi = k >> 1, d = args.pair_d[pi];
              const float ud = (u3[0] * c_ico[d][0] + u3[1] * c_ico[d][1] + u3[2] * c_ico[d][2]) * (float)(1 << args.pair_f[pi]);
              va = ud * ev[jj + 1];
              vb = -ud * ev[jj];
            } else if (k == two_half) {
              va = u3[0]; vb = u3[1];
            } else if (k == two_half + 2) {
              va = u3[2];
            }
            v[jj] = va; v[jj + 1] = vb;
          }
          put8<kPasses, kLean>(T, v, c, h, true, eh ? args.arr_ya_e1 : args.arr_ya);
          if (h) chunk_ready(c);
        }
      };
      write_e_half(0);

      EpiAcc gacc = {0.f, 0.f, 0.f, 0.f};                 // d sdf / d x_s partial sums over this thread's embedding columns

      for (int s = 0; s < n_steps; ++s, ++n) {
        const TcStep st = args.steps[s];
        const int l = st.layer;
        const int epi = st.epi;
        const bool last_step = (s == n_steps - 1);
        const uint32_t d_tmem = tmem + (n & 1) * 256 + lane_addr;
        EpiStepPtrs P;
        P.sigp = T.sig + (size_t)l * T.sig_stride;
        P.sigw = T.sig + (size_t)l * T.sig_stride;
        P.dhi = T.dwl_hi + (size_t)(args.arr_xd + l) * T.dwl_stride;
        P.dlo = T.dwl_lo + (size_t)(args.arr_xd + l) * T.dwl_stride;
        P.zb2 = T.aux + (size_t)(args.arr_zb2 + l) * T.aux_stride;
        P.zb2h = T.zb2h + (size_t)l * T.sig_stride;
        P.part_in = (st.addp >= 0) ? T.aux + (size_t)(args.arr_part + st.addp) * T.aux_stride : nullptr;
        P.part_out = T.aux + (size_t)(args.arr_part + st.aux) * T.aux_stride;
        P.bias = Wp + args.lay_b_off[l];
        P.wout = Wp + args.wout_off;
        P.hlast = T.aux + (size_t)args.arr_hlast * T.aux_stride;
        P.e32 = (kNE == 2) ? e32_w + (size_t)st.eh * args.aux_stride : e32_w;
        P.flags = st.flags;
        P.ecol0 = 256 * st.eh;
        EpiAcc acc_local = {0.f, 0.f, 0.f, 0.f};
        if (epi == EPI_S2_END && (kNE == 1 || (st.flags & STF_END_FIRST))) gacc = acc_local;
        EpiAcc& acc = (epi == EPI_S2_END) ? gacc : acc_local;
        switch (epi) {
          case EPI_RAW:     epi_step<EPI_RAW, kPasses, kLean, kNE>(args, T, P, tail, d_tmem, n, l, train, store_state, last_step, sbar, acc, lane); break;
          case EPI_S1:      epi_step<EPI_S1, kPasses, kLean, kNE>(args, T, P, tail, d_tmem, n, l, train, store_state, last_step, sbar, acc, lane); break;
          case EPI_S1_LAST: epi_step<EPI_S1_LAST, kPasses, kLean, kNE>(args, T, P, tail, d_tmem, n, l, train, store_state, last_step, sbar, acc, lane); break;
          case EPI_S2:      epi_step<EPI_S2, kPasses, kLean, kNE>(args, T, P, tail, d_tmem, n, l, train, store_state, last_step, sbar, acc, lane); break;
          case EPI_S2_END:  epi_step<EPI_S2_END, kPasses, kLean, kNE>(args, T, P, tail, d_tmem, n, l, train, store_state, last_step, sbar, acc, lane); break;
          case EPI_S3:      epi_step<EPI_S3, kPasses, kLean, kNE>(args, T, P, tail, d_tmem, n, l, train, store_state, last_step, sbar, acc, lane); break;
          case EPI_S3_LAST: epi_step<EPI_S3_LAST, kPasses, kLean, kNE>(args, T, P, tail, d_tmem, n, l, train, store_state, last_step, sbar, acc, lane); break;
          default:          epi_step<EPI_S4, kPasses, kLean, kNE>(args, T, P, tail, d_tmem, n, l, train, store_state, last_step, sbar, acc, lane); break;
        }

        if (kNE == 2 && epi == EPI_RAW) {
          // second embedding half of a wide embedding: its A operand replaces the first half's (whose products are done)
          if (st.flags & STF_PE_E) write_e_half(st.peh);
          if (st.flags & STF_PE_ABAR) write_abar_half(st.peh);
        } else if (epi == EPI_S1_LAST) {
          // out layer: combine the four column groups of every point
          red[jg * 128 + p] = acc.raw_acc;
          named_bar_sync(1, EPI_THREADS);
          if (jg == 0) {
            float raw = red[p] + red[128 + p] + red[256 + p] + red[384 + p] + Wp[args.bout_off];
            if (args.noise && real) raw += args.noise[pl] * args.noise_std;
            sdf_reg = raw * c_out;
            if (real) args.sdf_out[pl] = sdf_reg;
          }
          // the scratch is written again at S2_END (other warps, >= 3 steps later).  The a_ready / d_full chain already
          // orders that write after these reads, but compute-sanitizer's racecheck does not model mbarriers: one more
          // named barrier (~100 cycles per tile) keeps the kernel provably -- and tool-visibly -- hazard free
          named_bar_sync(1, EPI_THREADS);
        } else if (epi == EPI_S2_END && (kNE == 1 || (st.flags & STF_END_LAST))) {
          red[(0 * 4 + jg) * 128 + p] = acc.gx;
          red[(1 * 4 + jg) * 128 + p] = acc.gy;
          red[(2 * 4 + jg) * 128 + p] = acc.gz;
          named_bar_sync(1, EPI_THREADS);
          if (jg == 0) {
            const float gx = red[p] + red[128 + p] + red[256 + p] + red[384 + p];
            const float gy = red[512 + p] + red[640 + p] + red[768 + p] + red[896 + p];
            const float gz = red[1024 + p] + red[1152 + p] + red[1280 + p] + red[1408 + p];
            float ox = gx, oy = gy, oz = gz;     // g = s R^T g_xs
            if (args.pe.has_transform) {
              ox = args.pe.R[0] * gx + args.pe.R[3] * gy + args.pe.R[6] * gz;
              oy = args.pe.R[1] * gx + args.pe.R[4] * gy + args.pe.R[7] * gz;
              oz = args.pe.R[2] * gx + args.pe.R[5] * gy + args.pe.R[8] * gz;
            }
            const float g[3] = {args.pe.scale * ox, args.pe.scale * oy, args.pe.scale * oz};
            if (real && args.g_out) { args.g_out[pl * 3] = g[0]; args.g_out[pl * 3 + 1] = g[1]; args.g_out[pl * 3 + 2] = g[2]; }
            float sb = 0.f, gb[3] = {0.f, 0.f, 0.f};
            if (train) {
              float tot = 0.f;
              if (real) {
                const int64_t pg = args.p0 + pl;                 // global sample index = r*S + j
                const int64_t r = pg / args.S;
                const int jx = (int)(pg - r * args.S);
                const bool valid = args.ray_valid ? (args.ray_valid[r] != 0) : true;
                if (valid) {
                  float bnd, uu[3];
                  loss_bound_target(args.loss, pg, r, jx, args.dirs_C, args.depth, args.z_vals, args.T_WC, args.normals, bnd, uu);
                  const LossPoint o = loss_point(args.loss, sdf_reg, g, bnd, uu);
                  sb = o.sbar; gb[0] = o.gbar[0]; gb[1] = o.gbar[1]; gb[2] = o.gbar[2];
                  tot = o.total;
                  lsum0 += o.l_sdf; lsum1 += o.l_grad; lsum2 += o.l_eik; lsum3 += o.total;
                  sbsum += o.sbar;
                }
                args.loss_mat[pg] = tot;
              }
              // u = s R gbar
              float ux = gb[0], uy = gb[1], uz = gb[2];
              if (args.pe.has_transform) {
                ux = args.pe.R[0] * gb[0] + args.pe.R[1] * gb[1] + args.pe.R[2] * gb[2];
                uy = args.pe.R[3] * gb[0] + args.pe.R[4] * gb[1] + args.pe.R[5] * gb[2];
                uz = args.pe.R[6] * gb[0] + args.pe.R[7] * gb[1] + args.pe.R[8] * gb[2];
              }
              st4(bcast + p * 4, sb, ux * args.pe.scale, uy * args.pe.scale, uz * args.pe.scale);
            }
          }
          if (!train) named_bar_sync(1, EPI_THREADS);     // reads of the scratch done before anybody re-uses it (see S1_LAST)
          if (train) {
            named_bar_sync(1, EPI_THREADS);
            const float4 b4 = ld4(bcast + p * 4);
            sbar = b4.x; u3[0] = b4.y; u3[1] = b4.z; u3[2] = b4.w;
            write_abar_half(0);               // abar_e (first half) -> A operand of S3
          }
        }
      }
    }
    // loss sums: warp reduce, one atomic per warp (column group 0 holds the per-point values)
    if (args.mode == TC_MODE_TRAIN && jg == 0) {
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        lsum0 += __shfl_xor_sync(0xffffffffu, lsum0, o);
        lsum1 += __shfl_xor_sync(0xffffffffu, lsum1, o);
        lsum2 += __shfl_xor_sync(0xffffffffu, lsum2, o);
        lsum3 += __shfl_xor_sync(0xffffffffu, lsum3, o);
        sbsum += __shfl_xor_sync(0xffffffffu, sbsum, o);
      }
      if (lane == 0) {
        atomicAdd(args.loss_sums + 0, lsum0);
        atomicAdd(args.loss_sums + 1, lsum1);
        atomicAdd(args.loss_sums + 2, lsum2);
        atomicAdd(args.loss_sums + 3, lsum3);
        grad_add(args.g_packed + args.bout_off, c_out * sbsum, args.g_mc);     // d b_out = c * sum sbar
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == EPI_WARPS) tmem_dealloc(tmem, 512);
}

template <int kPasses, bool kLean, int kNE>
static void chain_launch_t(const TcChainArgs& args, int grid, cudaStream_t st) {
  tc_chain_kernel<kPasses, kLean, kNE><<<grid, NUM_THREADS, ChainCfg<kPasses>::kSmem, st>>>(args);
}

int tc_chain_launch(isdfb_ctx* ctx, const TcChainArgs& args, int passes, int grid, cudaStream_t st) {
  const bool two = args.n_eh == 2;
  if (passes == 3) {
    if (args.lean) { if (two) chain_launch_t<3, true, 2>(args, grid, st); else chain_launch_t<3, true, 1>(args, grid, st); }
    else if (two) chain_launch_t<3, false, 2>(args, grid, st);
    else chain_launch_t<3, false, 1>(args, grid, st);
  } else {
    if (two) chain_launch_t<1, false, 2>(args, grid, st);
    else chain_launch_t<1, false, 1>(args, grid, st);
  }
  ISDFB_LAUNCHED(ctx);
  ISDFB_CUDA_OK(ctx, cudaGetLastError());
  return ISDFB_OK;
}

template <int kPasses, bool kLean, int kNE>
static cudaError_t chain_attr_t() {
  return cudaFuncSetAttribute(tc_chain_kernel<kPasses, kLean, kNE>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                              ChainCfg<kPasses>::kSmem);
}

int tc_chain_init(isdfb_ctx* ctx) {
  ISDFB_CUDA_OK(ctx, (chain_attr_t<3, false, 1>()));
  ISDFB_CUDA_OK(ctx, (chain_attr_t<3, false, 2>()));
  ISDFB_CUDA_OK(ctx, (chain_attr_t<3, true, 1>()));
  ISDFB_CUDA_OK(ctx, (chain_attr_t<3, true, 2>()));
  ISDFB_CUDA_OK(ctx, (chain_attr_t<1, false, 1>()));
  ISDFB_CUDA_OK(ctx, (chain_attr_t<1, false, 2>()));
  return ISDFB_OK;
}
