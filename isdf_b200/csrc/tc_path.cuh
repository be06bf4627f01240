// Host-side state of the tensor-core path.
#pragma once
#include "tc_chain.cuh"

#define TC_PROF_MAX 512
struct TcUnitTable { TcUnit u[TC_MAX_UNITS]; };

// weight-gradient job: one 128-row half of one weight unit; up to three (X, Y) operand pairs
struct TcDwPair { int32_t x_arr, y_arr, ones; };      // y_arr < 0: no main product; ones: 0 none, 1 -> db, 2 -> d w_out
struct TcDwJob {
  int32_t half;            // which 128 output rows
  int32_t n_pairs;
  TcDwPair pair[3];
  int64_t g_off;           // packed-gradient offset of the unit's [256][ld] block
  int32_t ld;
  int64_t db_off;          // packed-gradient offset of the bias (or -1)
  int32_t perm_half;       // > 0: gradient columns are in the internal embedding order (pe_nat_col)
  int32_t col0;            //      ... starting at this internal column (second embedding half: 256)
};
#define TC_MAX_JOBS (2 * TC_MAX_UNITS)

struct TcDwArgs {
  TcDwJob jobs[TC_MAX_JOBS];
  int32_t n_jobs, n_tiles, tile0;
  const uint8_t *dwl_hi, *dwl_lo;
  size_t dwl_stride;
  float* g_packed;         // where the TMEM accumulators are flushed (red.global.add): the gradient itself, or with an
                           // exchange installed the LOCAL staging buffer
  int32_t g_mc;            // 1: exchange installed -- the last CTA of every job forwards the job's finished tile
  float* g_mc_out;         //    from the staging buffer to this MULTICAST address (multimem.red) and clears the stage
  int32_t* counters;       //    per-job arrival counters (self-resetting)
  int32_t expect[TC_MAX_JOBS];   // arrivals per job over ALL weight-gradient launches of the step
  int64_t wout_off;
  float scale_output;
};

struct TcState {
  int n_units, num_sms;
  TcUnitTable units;
  uint8_t* w_img;          // [unit][orient][hi|lo] x 128 KB
  float* aux;
  uint8_t *dwl_hi, *dwl_lo, *sig16;
  int64_t tiles_cap;
  size_t aux_stride, dwl_stride;
  int n_aux, n_dwl;
  TcChainArgs proto[3];    // per mode: steps and array indices filled in at create
  TcDwArgs dw;
  // optional kernel timing
  bool profiling;
  cudaEvent_t ev[TC_PROF_MAX][3];   // before chain, after chain, after dW
  int ev_kind[TC_PROF_MAX];         // 1: chain only, 2: chain + dW
  int n_ev;
  int32_t* dw_counters;    // device, [TC_MAX_JOBS], zero between steps
  cudaStream_t side;       // second stream: weight gradients of the first wave overlap the second wave
  cudaEvent_t ev_fork, ev_join;
};

int tc_dw_launch(isdfb_ctx* ctx, const TcDwArgs& args, int passes, int grid, cudaStream_t st);
