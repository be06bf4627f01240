// Argument block and step program of the tcgen05 chain kernel (tc_chain.cu).
#pragma once
#include "tc_common.cuh"

enum { TC_MODE_FWD = 0, TC_MODE_FWD_GRAD = 1, TC_MODE_TRAIN = 2 };
enum { EPI_RAW = 0, EPI_S1, EPI_S1_LAST, EPI_S2, EPI_S2_END, EPI_S3, EPI_S3_LAST, EPI_S4 };

// Step flags.  With a padded embedding wider than 256 (n_embed_funcs 8 / 10: E = 381 / 465 -> two halves of 256 internal
// columns) every embedding-fed product is the sum of two 128x256x256 products whose A operands (e_h, abar_e_h) are
// generated one after the other into the same shared-memory image; the first partial result is parked in a side array
// (EPI_RAW) and added by the consumer (addp) or accumulated there (STF_RAW_ADD).
enum {
  STF_RAW_ADD = 1,     // EPI_RAW: part[aux] += D   (else part[aux] = D)
  STF_PE_E = 2,        // EPI_RAW: after the drain write the embedding half `peh` into A (S1)
  STF_PE_ABAR = 4,     // EPI_RAW: after the drain write the adjoint abar_e half `peh` into A (S3)
  STF_END_FIRST = 8,   // EPI_S2_END: first embedding half -> reset the d sdf/dx accumulators
  STF_END_LAST = 16    // EPI_S2_END: last embedding half -> reduce, loss, then abar_e half 0 into A
};
struct TcStep {
  int32_t unit;     // weight unit (tc_pack.cu)
  int32_t orient;   // 0: Y = X W^T (S1, S3)   1: Y = X W (S2, S4)
  int32_t epi;      // epilogue kind
  int16_t layer;    // hidden layer whose sigma / bias / side arrays the epilogue uses
  int16_t aux;      // EPI_RAW: partial-sum side array written (index relative to arr_part)
  int16_t addp;     // S1 / S3 / S2_END: partial-sum side array added to the accumulator (relative to arr_part), -1: none
  int16_t flags;    // STF_*
  int16_t peh;      // STF_PE_*: which embedding half to generate
  int16_t eh;       // EPI_S2_END: embedding half of this step's 256 output columns
};
#define TC_MAX_STEPS (4 * ISDFB_MAX_HIDDEN_LAYERS + 12)
#define TC_MAX_EH 2                               // embedding halves of 256 internal columns

// forward-only lattice evaluation (get_sdf_grid, trainer.py:1426-1444 + transform.py:273-304): the query points
// x = R (lin[i] s_x, lin[j] s_y, lin[k] s_z) + t are generated in the PE stage instead of being read from HBM
struct TcGrid {
  const float* lin;          // [dim] torch.linspace(lo, hi, dim) (passed in: bit-identical abscissae)
  int32_t dim;               // 0: off (points come from args.x)
  int32_t has_transform;
  float scale[3];
  float R[9], t[3];
};

struct TcChainArgs {
  TcStep steps[TC_MAX_STEPS];
  int32_t n_steps, mode, L, ic, E, S;
  int32_t n_tiles;           // tiles processed by this launch ...
  int32_t tile0;             // ... starting at this tile of the chunk
  int64_t n_points;          // real points in this chunk
  int64_t p0;                // global index of the chunk's first point (sample index r*S+j)
  PEParams pe;
  isdfb_loss_cfg loss;
  float scale_output, noise_std;
  // model
  const uint8_t* w_img;      // [unit][orient][hi|lo] bf16 K-major images
  const float* w_packed;     // packed fp32 params (biases, output layer)
  int64_t lay_b_off[ISDFB_MAX_HIDDEN_LAYERS];
  int64_t wout_off, bout_off;
  // inputs / outputs
  TcGrid grid;
  const float* x;            // [n_points,3] (chunk-local); unused when grid.dim > 0
  const float* noise;        // [n_points] or null
  float* sdf_out;            // [n_points]
  float* g_out;              // [n_points,3] or null
  const float *z_vals, *depth, *dirs_C, *T_WC, *normals;   // GLOBAL ray arrays (indexed via p0)
  const uint8_t* ray_valid;
  float* loss_mat;           // GLOBAL [R*S]
  float* loss_sums;          // [4]
  float* g_packed;           // packed gradient (d b_out is accumulated by the chain kernel)
  int32_t g_mc;              // 1: g_packed is a multicast address (multimem.red, see grad_add)
  // per-tile side state
  float* aux;                // fp32 arrays [arr][tile][256*128], aux layout
  size_t aux_stride;         // floats between arrays
  uint8_t *dwl_hi, *dwl_lo;  // bf16 arrays [arr][tile][64 KB], dW layout
  uint8_t* sig16;            // sigma_l as unorm16, [layer][tile][64 KB], K-major image layout [f/8][p][8]
  uint8_t* zb2h;             // lean mode: zbar2_l as bf16, same [layer][tile][64 KB] layout and stride as sig16
  int32_t lean;              // 1: weight-gradient operands, the S3 read of delta_l and zbar2_l are single bf16 (precision
                             //    "bf16x3g"): halves the per-point side state; sdf / d sdf/dx / loss are unaffected
  size_t sig16_stride;       // bytes between layers
  size_t dwl_stride;         // bytes between arrays
  int32_t arr_zb2, arr_part, arr_e32, arr_hlast;            // aux array indices (arr_e32 + h: embedding half h)
  int32_t arr_yh, arr_ya, arr_xd, arr_xz, arr_v;            // dW-layout array indices
  int32_t arr_yh_e1, arr_ya_e1;                             // dW-layout arrays of the second embedding half (e, abar_e)
  int32_t n_eh;                                             // embedding halves (1: E <= 256, 2: E <= 512)
  uint8_t pair_d[TC_MAX_EH * TC_H / 2], pair_f[TC_MAX_EH * TC_H / 2];   // internal PE column pair -> (direction, octave)
};

int tc_chain_launch(isdfb_ctx* ctx, const TcChainArgs& args, int passes, int grid, cudaStream_t st);
