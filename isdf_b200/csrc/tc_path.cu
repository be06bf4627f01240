// Host orchestration of the tensor-core path: state, step programs, weight-gradient jobs, launches.
#include "tc_path.cuh"
#include <new>

static TcStep& add_step(TcChainArgs& a, int unit, int orient, int epi, int layer, int aux = 0) {
  TcStep& s = a.steps[a.n_steps++];
  s.unit = unit; s.orient = orient; s.epi = epi; s.layer = (int16_t)layer; s.aux = (int16_t)aux;
  s.addp = -1; s.flags = 0; s.peh = 0; s.eh = 0;
  return s;
}

// Partial-sum side arrays (indices relative to arr_part).  NE = 1: 0 concat(S1), 1 concat(S2), 2 concat(S3).
// NE = 2 adds 3: concat(S2) second half, 4: layer-0 first-half partial (S1), 5: the same for S3.
enum { PART_CAT_S1 = 0, PART_CAT_S2 = 1, PART_CAT_S3 = 2, PART_CAT_S2_H1 = 3, PART_L0_S1 = 4, PART_L0_S3 = 5 };

// Units: 0..L-1 = layer l's main block (layer 0: first embedding half), L = concat embedding part (first half),
// L+1 = layer 0 second embedding half, L+2 = concat embedding part second half.
static void build_program(const ModelLayout& lay, int mode, int NE, TcChainArgs& a) {
  const int L = lay.L, ic = lay.block + 1, UE = L, U0B = L + 1, UEB = L + 2;
  a.n_steps = 0;
  // ---- S1: e -> h_0 .. h_{L-1} -> sdf
  add_step(a, UE, 0, EPI_RAW, 0, PART_CAT_S1);                       // e_0 W_cat,e0^T  (A = e_0, kept)
  if (NE == 2) {
    TcStep& r = add_step(a, 0, 0, EPI_RAW, 0, PART_L0_S1);           // e_0 W_0,0^T parked; then e_1 -> A
    r.flags = STF_PE_E; r.peh = 1;
    add_step(a, UEB, 0, EPI_RAW, 0, PART_CAT_S1).flags = STF_RAW_ADD;   // += e_1 W_cat,e1^T  (A = e_1, kept)
  }
  for (int l = 0; l < L; ++l) {
    TcStep& t = add_step(a, (l == 0 && NE == 2) ? U0B : l, 0, l == L - 1 ? EPI_S1_LAST : EPI_S1, l);
    if (l == 0 && NE == 2) t.addp = PART_L0_S1;
    if (l == ic) t.addp = PART_CAT_S1;
  }
  if (mode == TC_MODE_FWD) return;
  // ---- S2: a_{L-1} .. a_e -> d sdf / d x
  for (int l = L - 1; l >= 1; --l) {
    if (l == ic) {
      add_step(a, UE, 1, EPI_RAW, l, PART_CAT_S2);                   // delta_ic W_cat,e0   (A = delta_ic, kept)
      if (NE == 2) add_step(a, UEB, 1, EPI_RAW, l, PART_CAT_S2_H1);
    }
    add_step(a, l, 1, EPI_S2, l - 1);
  }
  for (int h = 0; h < NE; ++h) {                                     // a_e half h = delta_0 W_0,h + concat part
    TcStep& t = add_step(a, h == 0 ? 0 : U0B, 1, EPI_S2_END, 0);
    t.addp = h == 0 ? PART_CAT_S2 : PART_CAT_S2_H1;
    t.eh = (int16_t)h;
    t.flags = (h == 0 ? STF_END_FIRST : 0) | (h == NE - 1 ? STF_END_LAST : 0);
  }
  if (mode == TC_MODE_FWD_GRAD) return;
  // ---- S3: abar_e -> dbar_0 .. (forward direction)
  add_step(a, UE, 0, EPI_RAW, 0, PART_CAT_S3);
  if (NE == 2) {
    TcStep& r = add_step(a, 0, 0, EPI_RAW, 0, PART_L0_S3);
    r.flags = STF_PE_ABAR; r.peh = 1;
    add_step(a, UEB, 0, EPI_RAW, 0, PART_CAT_S3).flags = STF_RAW_ADD;
  }
  for (int l = 0; l < L; ++l) {
    TcStep& t = add_step(a, (l == 0 && NE == 2) ? U0B : l, 0, l == L - 1 ? EPI_S3_LAST : EPI_S3, l);
    if (l == 0 && NE == 2) t.addp = PART_L0_S3;
    if (l == ic) t.addp = PART_CAT_S3;
  }
  // ---- S4 (reverse; the two d / d e products are not needed)
  for (int l = L - 1; l >= 1; --l) add_step(a, l, 1, EPI_S4, l - 1);
}

// Host-only view of the step program (no CUDA call, no context): what the chain kernel will run for a model shape.
// Each step is written as 8 int32: unit, orient, epi, layer, aux, addp, flags, (peh << 8 | eh).  Returns the number of
// steps, or a negative error.  Used by tests/test_abi.py to pin the programs (CPU suite) and by tools.
extern "C" int isdfb_debug_program(int32_t n_freqs, int32_t hidden, int32_t block, int32_t mode, int32_t* steps_out,
                                   int32_t max_steps) {
  if (!steps_out || n_freqs < 1 || block < 1 || 2 * block + 2 > ISDFB_MAX_HIDDEN_LAYERS || mode < 0 || mode > 2) return -1;
  ModelLayout lay;
  memset(&lay, 0, sizeof(lay));
  lay.n_freqs = n_freqs;
  lay.E = 2 * ISDFB_NDIRS * n_freqs + 3;
  lay.H = hidden;
  lay.block = block;
  lay.L = 2 * block + 2;
  if (lay.H != TC_H || lay.E > TC_MAX_EH * TC_H) return -2;          // shapes the tcgen05 path refuses
  TcChainArgs* a = new (std::nothrow) TcChainArgs();
  if (!a) return -3;
  memset(a, 0, sizeof(*a));
  build_program(lay, mode, lay.E > TC_H ? 2 : 1, *a);
  const int n = a->n_steps;
  if (n > max_steps || n > TC_MAX_STEPS) { delete a; return -4; }
  for (int i = 0; i < n; ++i) {
    const TcStep& t = a->steps[i];
    int32_t* o = steps_out + 8 * i;
    o[0] = t.unit; o[1] = t.orient; o[2] = t.epi; o[3] = t.layer; o[4] = t.aux; o[5] = t.addp; o[6] = t.flags;
    o[7] = (t.peh << 8) | t.eh;
  }
  delete a;
  return n;
}

void tc_destroy(isdfb_ctx* ctx) {
  TcState* tc = reinterpret_cast<TcState*>(ctx->tc);
  if (!tc) return;
  if (tc->w_img) cudaFree(tc->w_img);
  if (tc->aux) cudaFree(tc->aux);
  if (tc->dwl_hi) cudaFree(tc->dwl_hi);
  if (tc->dwl_lo) cudaFree(tc->dwl_lo);
  if (tc->sig16) cudaFree(tc->sig16);
  if (tc->dw_counters) cudaFree(tc->dw_counters);
  if (tc->side) cudaStreamDestroy(tc->side);
  if (tc->ev_fork) cudaEventDestroy(tc->ev_fork);
  if (tc->ev_join) cudaEventDestroy(tc->ev_join);
  for (int i = 0; i < TC_PROF_MAX; ++i)
    for (int k = 0; k < 3; ++k)
      if (tc->ev[i][k]) cudaEventDestroy(tc->ev[i][k]);
  delete tc;
  ctx->tc = nullptr;
}

int tc_chain_init(isdfb_ctx* ctx);
int tc_dw_init(isdfb_ctx* ctx);

int tc_create(isdfb_ctx* ctx) {
  const ModelLayout& lay = ctx->lay;
  if (lay.H != TC_H || lay.E > TC_MAX_EH * TC_H)
    ISDFB_FAIL(ctx, ISDFB_ERR_ARG,
               "tensor-core path supports hidden=256 and embedding <= 512 (n_embed_funcs <= 11); got hidden=%d E=%d. "
               "Use precision fp32 for other shapes.", lay.H, lay.E);
  const int NE = lay.E > TC_H ? 2 : 1;           // embedding halves of 256 internal columns
  { int rc = tc_chain_init(ctx); if (rc) return rc; rc = tc_dw_init(ctx); if (rc) return rc; }
  TcState* tc = new (std::nothrow) TcState();
  if (!tc) ISDFB_FAIL(ctx, ISDFB_ERR_ARG, "out of host memory");
  memset(tc, 0, sizeof(*tc));
  ctx->tc = tc;
  const int L = lay.L, ic = lay.block + 1;
  ISDFB_CUDA_OK(ctx, cudaDeviceGetAttribute(&tc->num_sms, cudaDevAttrMultiProcessorCount, ctx->device));
  ISDFB_CUDA_OK(ctx, cudaStreamCreateWithFlags(&tc->side, cudaStreamNonBlocking));
  ISDFB_CUDA_OK(ctx, cudaEventCreateWithFlags(&tc->ev_fork, cudaEventDisableTiming));
  ISDFB_CUDA_OK(ctx, cudaEventCreateWithFlags(&tc->ev_join, cudaEventDisableTiming));
  tc->n_units = L + 1 + (NE == 2 ? 2 : 0);
  const int pe_half = ISDFB_NDIRS * lay.n_freqs;
  for (int l = 0; l < L; ++l) {
    tc->units.u[l].w_off = lay.layer[l].w_off; tc->units.u[l].ld = lay.layer[l].k0;
    tc->units.u[l].perm_half = (l == 0) ? pe_half : 0;
    tc->units.u[l].col0 = 0;
  }
  tc->units.u[L].w_off = lay.layer[ic].we_off;
  tc->units.u[L].ld = lay.Ep;
  tc->units.u[L].perm_half = pe_half;
  tc->units.u[L].col0 = 0;
  if (NE == 2) {                                 // second embedding halves of layer 0 and of the concat layer
    tc->units.u[L + 1] = tc->units.u[0]; tc->units.u[L + 1].col0 = TC_H;
    tc->units.u[L + 2] = tc->units.u[L]; tc->units.u[L + 2].col0 = TC_H;
  }
  const bool lean = ctx->cfg.precision == ISDFB_PREC_BF16X3G;
  tc->tiles_cap = ctx->cap / TC_TILE;
  const int n_part = NE == 2 ? 6 : 3;
  tc->n_aux = n_part + NE + 1 + (lean ? 0 : L);     // partial sums, e32 per half, h_last (+ zbar2_l as fp32 unless lean)
  tc->n_dwl = 4 * L + 1 + (NE == 2 ? 2 : 0);
  tc->aux_stride = (size_t)tc->tiles_cap * TC_TILE_FLOATS;
  tc->dwl_stride = (size_t)tc->tiles_cap * TC_DWL_TILE_BYTES;
  ISDFB_CUDA_OK(ctx, cudaMalloc(&tc->w_img, (size_t)tc->n_units * 4 * TC_IMG_BYTES));
  ISDFB_CUDA_OK(ctx, cudaMalloc(&tc->aux, tc->aux_stride * tc->n_aux * sizeof(float)));
  ISDFB_CUDA_OK(ctx, cudaMalloc(&tc->dwl_hi, tc->dwl_stride * tc->n_dwl));
  ISDFB_CUDA_OK(ctx, cudaMalloc(&tc->sig16, tc->dwl_stride * L * (lean ? 2 : 1)));     // lean: + zbar2_l (bf16)
  if (ctx->cfg.precision == ISDFB_PREC_BF16X3) ISDFB_CUDA_OK(ctx, cudaMalloc(&tc->dwl_lo, tc->dwl_stride * tc->n_dwl));

  ISDFB_CUDA_OK(ctx, cudaMalloc(&tc->dw_counters, TC_MAX_JOBS * sizeof(int32_t)));
  ISDFB_CUDA_OK(ctx, cudaMemset(tc->dw_counters, 0, TC_MAX_JOBS * sizeof(int32_t)));
  for (int mode = 0; mode < 3; ++mode) {
    TcChainArgs& a = tc->proto[mode];
    memset(&a, 0, sizeof(a));
    build_program(lay, mode, NE, a);
    a.n_eh = NE;
    a.mode = mode; a.L = L; a.ic = ic; a.E = lay.E;
    a.pe = ctx->pe;
    a.scale_output = ctx->cfg.scale_output;
    a.w_img = tc->w_img;
    a.w_packed = ctx->w_packed;
    a.g_packed = ctx->g_packed;
    for (int l = 0; l < L; ++l) a.lay_b_off[l] = lay.layer[l].b_off;
    a.wout_off = lay.wout_off; a.bout_off = lay.bout_off;
    a.aux = tc->aux; a.aux_stride = tc->aux_stride;
    a.dwl_hi = tc->dwl_hi; a.dwl_lo = tc->dwl_lo; a.dwl_stride = tc->dwl_stride;
    a.sig16 = tc->sig16; a.sig16_stride = tc->dwl_stride;
    a.arr_part = 0; a.arr_e32 = n_part; a.arr_hlast = n_part + NE; a.arr_zb2 = n_part + NE + 1;   // zbar2 (fp32): absent in lean mode
    a.lean = lean ? 1 : 0;
    a.zb2h = lean ? tc->sig16 + tc->dwl_stride * L : nullptr;
    for (int i = 0; i < TC_MAX_EH * TC_H / 2; ++i) {      // pair i = (direction, octave) of internal columns 2i, 2i+1
      a.pair_d[i] = (uint8_t)(i < pe_half ? i / lay.n_freqs : 0);
      a.pair_f[i] = (uint8_t)(i < pe_half ? i % lay.n_freqs : 0);
    }
    a.arr_yh = 0; a.arr_ya = L; a.arr_xd = 2 * L; a.arr_xz = 3 * L; a.arr_v = 4 * L;
    a.arr_yh_e1 = 4 * L + 1; a.arr_ya_e1 = 4 * L + 2;
  }
  // weight-gradient jobs
  TcDwArgs& d = tc->dw;
  memset(&d, 0, sizeof(d));
  const TcChainArgs& a = tc->proto[TC_MODE_TRAIN];
  for (int u = 0; u < tc->n_units; ++u) {
    for (int half = 0; half < 2; ++half) {
      TcDwJob& j = d.jobs[d.n_jobs++];
      j.half = half;
      j.ld = tc->units.u[u].ld;
      j.perm_half = tc->units.u[u].perm_half;
      j.col0 = tc->units.u[u].col0;
      const bool second = (u > L);                       // second embedding half of layer 0 (L+1) / the concat layer (L+2)
      const int ya0 = second ? a.arr_ya_e1 : a.arr_ya, yh0 = second ? a.arr_yh_e1 : a.arr_yh;
      if (u < L) {
        j.g_off = lay.layer[u].w_off;
        j.db_off = lay.layer[u].b_off;
        j.pair[0] = {a.arr_xd + u, a.arr_ya + u, 0};
        j.pair[1] = {a.arr_xz + u, a.arr_yh + u, 1};
        j.n_pairs = 2;
        if (u == L - 1) { j.pair[2] = {a.arr_v, -1, 2}; j.n_pairs = 3; }
      } else if (u == L + 1) {                           // layer 0, second embedding half (bias rides with the first)
        j.g_off = lay.layer[0].w_off;
        j.db_off = -1;
        j.pair[0] = {a.arr_xd + 0, ya0, 0};
        j.pair[1] = {a.arr_xz + 0, yh0, 0};
        j.n_pairs = 2;
      } else {                                           // concat layer, embedding part (half 0 or 1)
        j.g_off = lay.layer[ic].we_off;
        j.db_off = -1;
        j.pair[0] = {a.arr_xd + ic, ya0, 0};
        j.pair[1] = {a.arr_xz + ic, yh0, 0};
        j.n_pairs = 2;
      }
    }
  }
  d.dwl_hi = tc->dwl_hi; d.dwl_lo = tc->dwl_lo; d.dwl_stride = tc->dwl_stride;
  d.g_packed = ctx->g_packed;
  d.wout_off = lay.wout_off;
  d.scale_output = ctx->cfg.scale_output;
  return ISDFB_OK;
}

static int prof_begin(TcState* tc, cudaStream_t st) {
  if (!tc->profiling || tc->n_ev >= TC_PROF_MAX) return -1;
  const int i = tc->n_ev++;
  for (int k = 0; k < 3; ++k)
    if (!tc->ev[i][k]) cudaEventCreate(&tc->ev[i][k]);
  tc->ev_kind[i] = 0;
  cudaEventRecord(tc->ev[i][0], st);
  return i;
}
static void prof_mark(TcState* tc, int i, int k, cudaStream_t st) {
  if (i < 0) return;
  cudaEventRecord(tc->ev[i][k], st);
  tc->ev_kind[i] = k;
}

static inline int passes_of(const isdfb_ctx* ctx) {
  return (ctx->cfg.precision == ISDFB_PREC_BF16X3 || ctx->cfg.precision == ISDFB_PREC_BF16X3G) ? 3 : 1;
}
// the weight-gradient kernel reads single-bf16 operands in lean mode
static inline int dw_passes_of(const isdfb_ctx* ctx) { return ctx->cfg.precision == ISDFB_PREC_BF16X3 ? 3 : 1; }

// A call over n points runs in chunks of at most cap points (the side state is sized for cap points): chunk
// [p0, p0 + nc) for p0 = 0, cap, 2 cap, ..., cut into tiles of TC_TILE points.  f(p0, nc, tiles) runs once per chunk,
// in order; a non-zero return stops the walk and is returned.
template <class F>
static int for_each_chunk(int64_t n, int64_t cap, F&& f) {
  for (int64_t p0 = 0; p0 < n; p0 += cap) {
    const int64_t nc = (n - p0 < cap) ? (n - p0) : cap;
    const int rc = f(p0, nc, (int)((nc + TC_TILE - 1) / TC_TILE));
    if (rc) return rc;
  }
  return ISDFB_OK;
}

// The launches of one training chunk.  A wave runs the chain kernel over tiles [tile0, tile0 + n_tiles) on chain_grid
// CTAs and then the weight-gradient kernel over the same tiles on dw_grid CTAs, on the side stream when dw_side.
struct TcWave { int tile0, n_tiles, chain_grid, dw_grid; bool dw_side; };
struct TcChunkPlan { int n_waves; TcWave wave[2]; };

// A chunk of more than one and less than two waves of tiles runs as two waves when overlap is allowed: the weight
// gradients of the full wave 1 run on the side stream underneath the partial wave 2, on the CTAs wave 2 leaves idle --
// but never fewer than one CTA per job: tc_dw_kernel maps CTA b to job b % n_jobs, so the jobs past a smaller grid
// would get no CTA and their gradient over wave 1 would be lost.  Otherwise one wave: the chain on at most num_sms
// persistent CTAs, then the dW on num_sms CTAs.
static TcChunkPlan chunk_plan(int tiles, int num_sms, int n_jobs, bool overlap) {
  TcChunkPlan pl;
  if (overlap && tiles > num_sms && tiles < 2 * num_sms) {
    const int rest = tiles - num_sms, idle = num_sms - rest;
    pl.n_waves = 2;
    pl.wave[0] = {0, num_sms, num_sms, idle > n_jobs ? idle : n_jobs, true};
    pl.wave[1] = {num_sms, rest, rest, num_sms, false};
  } else {
    pl.n_waves = 1;
    pl.wave[0] = {0, tiles, tiles < num_sms ? tiles : num_sms, num_sms, false};
  }
  return pl;
}

// Arrivals at job j's counter from one weight-gradient launch of `grid` CTAs (grid >= n_jobs) over `tiles` tiles:
// tc_dw_kernel maps CTA b to job b % n_jobs and tile split b / n_jobs, so job j has (grid - 1 - j) / n_jobs + 1 splits,
// and only a split that owns at least one tile arrives.
static inline int dw_arrivals(int j, int grid, int tiles, int n_jobs) {
  const int n_splits = (grid - 1 - j) / n_jobs + 1;
  return n_splits < tiles ? n_splits : tiles;
}

static int tc_forward_impl(isdfb_ctx* ctx, const float* x, const float* noise, float noise_std, int64_t n, float* sdf,
                           float* grad, cudaStream_t st, const TcGrid* grid) {
  TcState* tc = reinterpret_cast<TcState*>(ctx->tc);
  return for_each_chunk(n, ctx->cap, [&](int64_t p0, int64_t nc, int tiles) -> int {
    TcChainArgs a = tc->proto[grad ? TC_MODE_FWD_GRAD : TC_MODE_FWD];
    if (grid) a.grid = *grid;
    a.n_points = nc;
    a.n_tiles = tiles;
    a.p0 = p0;
    a.x = x ? x + p0 * 3 : nullptr;
    a.noise = noise ? noise + p0 : nullptr;
    a.noise_std = noise_std;
    a.sdf_out = sdf + p0;
    a.g_out = grad ? grad + p0 * 3 : nullptr;
    const TcWave w = chunk_plan(tiles, tc->num_sms, tc->dw.n_jobs, false).wave[0];
    const int pi = prof_begin(tc, st);
    const int rc = tc_chain_launch(ctx, a, passes_of(ctx), w.chain_grid, st);
    if (rc) return rc;
    prof_mark(tc, pi, 1, st);
    return ISDFB_OK;
  });
}

int tc_forward(isdfb_ctx* ctx, const float* x, const float* noise, float noise_std, int64_t n, float* sdf,
               float* grad, cudaStream_t st) {
  return tc_forward_impl(ctx, x, noise, noise_std, n, sdf, grad, st, nullptr);
}

// K2 over the dim^3 lattice of get_sdf_grid with the query points generated in the kernel (no [dim^3, 3] array in HBM)
int tc_forward_grid(isdfb_ctx* ctx, const float* lin, int dim, const float* scale, const float* transform, float* sdf,
                    cudaStream_t st) {
  TcGrid g;
  memset(&g, 0, sizeof(g));
  g.lin = lin; g.dim = dim;
  for (int i = 0; i < 3; ++i) g.scale[i] = scale ? scale[i] : 1.f;
  g.has_transform = transform ? 1 : 0;
  if (transform)
    for (int r = 0; r < 3; ++r) {
      for (int c = 0; c < 3; ++c) g.R[r * 3 + c] = transform[r * 4 + c];
      g.t[r] = transform[r * 4 + 3];
    }
  return tc_forward_impl(ctx, nullptr, nullptr, 0.f, (int64_t)dim * dim * dim, sdf, nullptr, st, &g);
}

int tc_train(isdfb_ctx* ctx, const float* pc, const float* z_vals, const float* depth_sample, const float* dirs_C,
             const float* T_WC_sample, const float* norm_sample, const float* noise, const uint8_t* ray_valid,
             int64_t n_rays, int32_t S, const isdfb_loss_cfg* loss, float* sdf, float* grad, float* loss_mat,
             float* loss_sums, cudaStream_t st) {
  TcState* tc = reinterpret_cast<TcState*>(ctx->tc);
  const int64_t n = n_rays * S;
  const int n_jobs = tc->dw.n_jobs;
  // kernel timing reads one (chain, dW) event pair per chunk, so profiling runs every chunk as one wave
  const bool overlap = !tc->profiling;
  // with a gradient exchange installed the last CTA of each job over ALL weight-gradient launches of the step
  // forwards the job's tile to the multicast buffer, so it must know how many arrive
  int32_t expect[TC_MAX_JOBS] = {0};
  if (ctx->g_xchg)
    for_each_chunk(n, ctx->cap, [&](int64_t, int64_t, int tiles) -> int {
      const TcChunkPlan pl = chunk_plan(tiles, tc->num_sms, n_jobs, overlap);
      for (int w = 0; w < pl.n_waves; ++w)
        for (int j = 0; j < n_jobs; ++j) expect[j] += dw_arrivals(j, pl.wave[w].dw_grid, pl.wave[w].n_tiles, n_jobs);
      return ISDFB_OK;
    });
  return for_each_chunk(n, ctx->cap, [&](int64_t p0, int64_t nc, int tiles) -> int {
    TcChainArgs a = tc->proto[TC_MODE_TRAIN];
    a.n_points = nc;
    a.p0 = p0;
    a.S = S;
    a.loss = *loss;
    a.x = pc + p0 * 3;
    a.noise = noise ? noise + p0 : nullptr;
    a.noise_std = loss->noise_std;
    a.sdf_out = sdf + p0;
    a.g_out = grad ? grad + p0 * 3 : nullptr;
    a.z_vals = z_vals; a.depth = depth_sample; a.dirs_C = dirs_C; a.T_WC = T_WC_sample; a.normals = norm_sample;
    a.ray_valid = ray_valid;
    a.loss_mat = loss_mat;
    a.loss_sums = loss_sums;
    a.g_packed = ctx->g_xchg ? ctx->g_mc[ctx->g_sel] : ctx->g_packed;
    a.g_mc = ctx->g_xchg ? 1 : 0;
    TcDwArgs d = tc->dw;
    d.g_mc = ctx->g_xchg ? 1 : 0;
    d.g_packed = ctx->g_xchg ? ctx->g_own : ctx->g_packed;      // exchange: accumulate in the local stage ...
    d.g_mc_out = ctx->g_xchg ? ctx->g_mc[ctx->g_sel] : nullptr; // ... the last CTA per job forwards it
    d.counters = tc->dw_counters;
    for (int j = 0; j < TC_MAX_JOBS; ++j) d.expect[j] = expect[j];
    const TcChunkPlan pl = chunk_plan(tiles, tc->num_sms, n_jobs, overlap);
    const int pi = prof_begin(tc, st);                // -1 (marks are no-ops) unless profiling, which plans one wave
    for (int w = 0; w < pl.n_waves; ++w) {
      const TcWave& wv = pl.wave[w];
      a.tile0 = d.tile0 = wv.tile0;
      a.n_tiles = d.n_tiles = wv.n_tiles;
      int rc = tc_chain_launch(ctx, a, passes_of(ctx), wv.chain_grid, st);
      if (rc) return rc;
      prof_mark(tc, pi, 1, st);
      if (wv.dw_side) {                                // fork: these weight gradients run underneath the next wave
        ISDFB_CUDA_OK(ctx, cudaEventRecord(tc->ev_fork, st));
        ISDFB_CUDA_OK(ctx, cudaStreamWaitEvent(tc->side, tc->ev_fork, 0));
        rc = tc_dw_launch(ctx, d, dw_passes_of(ctx), wv.dw_grid, tc->side);
        if (rc) return rc;
        ISDFB_CUDA_OK(ctx, cudaEventRecord(tc->ev_join, tc->side));
      } else {
        if (w > 0 && pl.wave[w - 1].dw_side) ISDFB_CUDA_OK(ctx, cudaStreamWaitEvent(st, tc->ev_join, 0));
        rc = tc_dw_launch(ctx, d, dw_passes_of(ctx), wv.dw_grid, st);
        if (rc) return rc;
        prof_mark(tc, pi, 2, st);
      }
    }
    return ISDFB_OK;
  });
}

extern "C" int isdfb_debug_buffers(isdfb_ctx* ctx, float** aux, int64_t* aux_stride_floats, void** dwl_hi,
                                   void** dwl_lo, int64_t* dwl_stride_bytes, int32_t* n_aux, int32_t* n_dwl,
                                   int64_t* tiles_cap, void** sig16) {
  if (!ctx) return ISDFB_ERR_ARG;
  TcState* tc = reinterpret_cast<TcState*>(ctx->tc);
  if (!tc) ISDFB_FAIL(ctx, ISDFB_ERR_STATE, "no tensor-core state (fp32 path)");
  *aux = tc->aux; *aux_stride_floats = (int64_t)tc->aux_stride;
  *dwl_hi = tc->dwl_hi; *dwl_lo = tc->dwl_lo; *dwl_stride_bytes = (int64_t)tc->dwl_stride;
  *n_aux = tc->n_aux; *n_dwl = tc->n_dwl; *tiles_cap = tc->tiles_cap; *sig16 = tc->sig16;
  return ISDFB_OK;
}

extern "C" int isdfb_profile_enable(isdfb_ctx* ctx, int32_t enable) {
  if (!ctx) return ISDFB_ERR_ARG;
  TcState* tc = reinterpret_cast<TcState*>(ctx->tc);
  if (!tc) ISDFB_FAIL(ctx, ISDFB_ERR_STATE, "kernel timing is available on the tensor-core path only");
  tc->profiling = enable != 0;
  tc->n_ev = 0;
  return ISDFB_OK;
}

extern "C" int isdfb_profile_read(isdfb_ctx* ctx, double* chain_ms, double* dw_ms, int64_t* n_chain, int64_t* n_dw) {
  if (!ctx || !chain_ms || !dw_ms || !n_chain || !n_dw) return ISDFB_ERR_ARG;
  TcState* tc = reinterpret_cast<TcState*>(ctx->tc);
  if (!tc) ISDFB_FAIL(ctx, ISDFB_ERR_STATE, "kernel timing is available on the tensor-core path only");
  ISDFB_CUDA_OK(ctx, cudaSetDevice(ctx->device));
  *chain_ms = *dw_ms = 0.0; *n_chain = *n_dw = 0;
  for (int i = 0; i < tc->n_ev; ++i) {
    const int k = tc->ev_kind[i];
    if (k < 1) continue;
    float ms = 0.f;
    ISDFB_CUDA_OK(ctx, cudaEventSynchronize(tc->ev[i][k]));
    ISDFB_CUDA_OK(ctx, cudaEventElapsedTime(&ms, tc->ev[i][0], tc->ev[i][1]));
    *chain_ms += ms; ++*n_chain;
    if (k == 2) {
      ISDFB_CUDA_OK(ctx, cudaEventElapsedTime(&ms, tc->ev[i][1], tc->ev[i][2]));
      *dw_ms += ms; ++*n_dw;
    }
  }
  tc->n_ev = 0;
  return ISDFB_OK;
}
