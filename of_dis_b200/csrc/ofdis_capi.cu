// C-ABI of libofdis_b200 (include/ofdis_b200.h): context, device workspaces,
// level loop (OFClass::OFClass, oflow.cpp:76-108,138-157,184-295) and transfers.
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <map>
#include <new>
#include <string>
#include <vector>

#include <nvtx3/nvToolsExt.h>

#include "../../include/ofdis_b200.h"
#include "ofdis_internal.cuh"

using namespace ofdis;

struct ofdis_ctx {
  int device = 0;
  cudaStream_t stream = nullptr;
  bool own_stream = false;
  ofdis_params prm{};
  int nop = 2, width = 0, height = 0, pad = 0, max_frames = 0;
  // usefbcon: every pair occupies two internal frames (2*f forward, 2*f+1 the grid on the swapped
  // images); dirs = 2, cap = max_frames * dirs internal frames are allocated
  int dirs = 1, cap = 0;
  int last_vr_fstep = 1;
  int sel_dir = -1;                // ofdis_set_direction: -1 = both directions / the forward grid
  // SOR band plan (sor_band_plan): levels of up to sor_single_max rows run in one CTA, taller ones in a
  // cluster of up to sor_max_cluster CTAs (8 = portable limit; 16 where the device grants it)
  int sor_single_max = 128, sor_max_cluster = 8, sor_dev_cluster = 8, sor_rt = 1;  // defaults set in ofdis_create
  // levels of few 32-row bands: pixel wavefront (sor_lane_kernel) instead of the block wavefront.  0 never, 1 always,
  // 2 (default) for launches of up to SOR_LANE_AUTO_FRAMES frames on levels of one or two bands (sor_lane_preferred):
  // there the kernel is 10-20 % faster per launch, but it needs
  // 200 KB of shared memory per CTA at 56-row levels (one CTA per SM), which costs 6 % of throughput when ten
  // streams of 64 frames overlap (bench.py `value`)
  int sor_lane = 2;
  int last_vr_lane = 0;  // layout of the last refinement (ofdis_debug_get)
  // programmatic dependent launch of the level loop's kernels (pdl_wait, ofdis_internal.cuh): 0 never, 1 always,
  // 2 (default) for launches of up to SOR_LANE_AUTO_FRAMES frames: one stream, graph replay, tools/pdl_ab.py:
  // 1 pair 0.349 -> 0.342 ms, 8 pairs 0.373 -> 0.356 ms, 64 pairs 0.558 -> 0.598 ms (waiting CTAs of the next kernel
  // take SM slots from the tail of the current one)
  int pdl = 2;
  int nlev = 0;                    // sc_f - sc_l + 1
  std::vector<LevelGeom> lev;      // index: level - sc_l
  std::vector<size_t> img_off;     // [lev][4] offsets (floats) inside one packed frame
  size_t frame_floats = 0;
  size_t images_floats = 0;        // leading part of a packed frame that holds I0,I1 of all levels
  float* d_img = nullptr;          // [max_frames][frame_floats]
  // lazily allocated staging of the pyramid / output stages (ofdis_upload_frames_u8,
  // ofdis_upload_finest_level, ofdis_get_flow_fullres)
  void* d_stage = nullptr;
  size_t stage_bytes = 0;
  float* d_full = nullptr;
  size_t full_floats = 0;
  std::vector<float*> d_flow;      // index level - sc_l, plus one extra entry for level sc_f+1 (initflow)
  std::vector<size_t> flow_floats;
  VarRefPlanes planes{};
  float* d_planes = nullptr;
  float* d_fast = nullptr;          // fast-mode records and (du,dv) ping-pong planes (ofdis_set_option "sor_fast")
  int last_vr_fcur = 0;
  PatchParams pp{};
  long launches = 0;
  int last_vr_level = -1, last_vr_f0 = 0;
  bool graph_mode = false;
  Profiler* prof = nullptr;         // non-null only inside ofdis_profile_run
  std::map<long, cudaGraphExec_t> graphs;
  std::map<long, long> graph_launches;
  std::string err;
};

namespace {
constexpr int SOR_LANE_AUTO_FRAMES = 16;

// NVTX range per stage and level ("patch L3", "densify L3", "varref L3", "pyramid", "upsample"): free
// when no profiler is attached, names the stages in Nsight Systems / ncu --nvtx timelines.
struct NvtxRange {
  NvtxRange(const char* stage, int level) {
    char name[48];
    if (level >= 0) snprintf(name, sizeof(name), "ofdis %s L%d", stage, level);
    else snprintf(name, sizeof(name), "ofdis %s", stage);
    nvtxRangePushA(name);
  }
  ~NvtxRange() { nvtxRangePop(); }
};

int fail(ofdis_ctx* c, int code, const char* what, cudaError_t e = cudaSuccess) {
  if (c) {
    c->err = what;
    if (e != cudaSuccess) {
      c->err += ": ";
      c->err += cudaGetErrorString(e);
    }
  }
  return code;
}

#define CK(call)                                                        \
  do {                                                                  \
    cudaError_t e__ = (call);                                           \
    if (e__ != cudaSuccess) return fail(ctx, OFDIS_ERR_CUDA, #call, e__); \
  } while (0)

// camparam / optparam derivation (oflow.cpp:81-92,142-157; patchgrid.cpp:42-48)
void make_level(LevelGeom& L, const ofdis_ctx* c, int sl) {
  const ofdis_params& p = c->prm;
  const float sc_fct = (float)pow(2, -sl);
  L.h = (int)(c->height * sc_fct);
  L.w = (int)(c->width * sc_fct);
  L.pad = c->pad;
  L.tmp_w = L.w + 2 * c->pad;
  L.tmp_h = L.h + 2 * c->pad;
  L.noc = p.noc;
  L.nop = c->nop;
  L.P = p.p_samp_s;
  L.novals = p.noc * p.p_samp_s * p.p_samp_s;
  L.steps = (int)floor(p.p_samp_s * (1 - p.patove));
  if (L.steps < 1) L.steps = 1;
  L.nopw = (int)ceil((float)L.w / (float)L.steps);
  L.noph = (int)ceil((float)L.h / (float)L.steps);
  L.np = L.nopw * L.noph;
  L.offw = (L.w - (L.nopw - 1) * L.steps) / 2;
  L.offh = (L.h - (L.noph - 1) * L.steps) / 2;
  L.level = sl;
  L.camlr = 0;
  L.pitch = ((L.w + 3) / 4) * 4;
  L.lb = -(float)p.p_samp_s / 2;
  L.ubw = (float)(L.w + p.p_samp_s / 2 - 2);
  L.ubh = (float)(L.h + p.p_samp_s / 2 - 2);
  L.outlierthresh = (float)p.p_samp_s / 2;
  L.pat_p = L.pat_w = nullptr;
  L.pat_conv = L.pat_cnt = nullptr;
  L.fb = 0;
  L.fstep = 1;
  L.fb_pos = nullptr;
  L.fb_wbil = nullptr;
  L.fb_reach = nullptr;
}

LevelGeom* level_of(ofdis_ctx* c, int level) {
  if (level < c->prm.sc_l || level > c->prm.sc_f) return nullptr;
  return &c->lev[level - c->prm.sc_l];
}

// copy of a level's geometry whose launches address every `fstep`-th internal frame
LevelGeom stepped(const LevelGeom& L, int fstep) {
  LevelGeom g = L;
  g.fstep = fstep;
  return g;
}

cudaMemcpyKind kind_in(int memkind) { return memkind == OFDIS_MEM_DEVICE ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice; }
cudaMemcpyKind kind_out(int memkind) { return memkind == OFDIS_MEM_DEVICE ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost; }

int run_levels(ofdis_ctx* ctx, int nframes, int use_initflow) {
  for (int sl = ctx->prm.sc_f; sl >= ctx->prm.sc_l; --sl) {
    const bool from_coarser = (sl < ctx->prm.sc_f) || use_initflow;
    if (ctx->prof) ctx->prof->level = sl;
    int rc = ofdis_patgrid_optimize(ctx, sl, 0, nframes, from_coarser ? 1 : 0);
    if (rc) return rc;
    rc = ofdis_patgrid_aggregate(ctx, sl, 0, nframes);
    if (rc) return rc;
    if (ctx->prm.usetvref) {
      rc = ofdis_varref_refine(ctx, sl, 0, nframes);
      if (rc) return rc;
    }
  }
  return OFDIS_OK;
}

}  // namespace

extern "C" {

const char* ofdis_version(void) { return "ofdis_b200 0.1 (sm_100a)"; }

const char* ofdis_last_error(const ofdis_ctx* ctx) { return ctx ? ctx->err.c_str() : "null context"; }

int ofdis_create(ofdis_ctx** out, int device, void* stream, const ofdis_params* prm, int nop, int width,
                 int height, int imgpadding, int max_frames) {
  if (!out || !prm) return OFDIS_ERR_ARG;
  *out = nullptr;
  if (nop != 1 && nop != 2) return OFDIS_ERR_ARG;
  if (prm->noc != 1 && prm->noc != 3) return OFDIS_ERR_ARG;
  if (prm->sc_l < 0 || prm->sc_f < prm->sc_l || prm->sc_f > 16) return OFDIS_ERR_ARG;
  if (prm->p_samp_s < 2 || (prm->p_samp_s & 1) || (prm->noc * prm->p_samp_s * prm->p_samp_s) % 4) return OFDIS_ERR_ARG;
  if (imgpadding < prm->p_samp_s) return OFDIS_ERR_ARG;  // window of a patch at the bounds must stay inside the padding
  if (width <= 0 || height <= 0 || (width % (1 << prm->sc_f)) || (height % (1 << prm->sc_f))) return OFDIS_ERR_ARG;
  if (max_frames < 1 || prm->max_iter < 0) return OFDIS_ERR_ARG;
  if (prm->usetvref && ((height >> prm->sc_f) < 4 || (width >> prm->sc_f) < 2)) return OFDIS_ERR_ARG;  // image.c:401-434 needs >= 4 rows
  if (prm->usetvref) {  // tallest refinement level: 256-row bands x a cluster of 16 CTAs at most (re-checked for the device below)
    VarRefPlanes probe{};
    if (!sor_band_plan(width >> prm->sc_l, height >> prm->sc_l, 4, 128, 16, nop, 1, &probe)) return OFDIS_ERR_UNSUPPORTED;
  }

  ofdis_ctx* ctx = new (std::nothrow) ofdis_ctx();
  if (!ctx) return OFDIS_ERR_NOMEM;
  ctx->device = device;
  ctx->prm = *prm;
  ctx->nop = nop;
  ctx->width = width;
  ctx->height = height;
  ctx->pad = imgpadding;
  ctx->max_frames = max_frames;
  ctx->dirs = prm->usefbcon ? 2 : 1;
  ctx->cap = max_frames * ctx->dirs;
  const int cap = ctx->cap;
  ctx->nlev = prm->sc_f - prm->sc_l + 1;
  cudaError_t e = cudaSetDevice(device);
  if (e != cudaSuccess) {
    delete ctx;
    return OFDIS_ERR_CUDA;
  }
  if (stream) ctx->stream = (cudaStream_t)stream;
  else {
    e = cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking);
    if (e != cudaSuccess) {
      delete ctx;
      return OFDIS_ERR_CUDA;
    }
    ctx->own_stream = true;
  }
  if (prm->usetvref) {  // tallest refinement level: 256-row bands x the largest cluster the device grants
    // Measured defaults (tools/big_configs.py, bench.py --opt): the largest cluster the device grants
    // (16 CTAs: -10..20 % on levels of 272..1024 rows against 8); two rows per SOR thread for stereo
    // (-23 % on configs[4]), one for flow (two rows: -3 % on configs[2], +4 % on the 56-row bench level).
    ctx->sor_dev_cluster = sor_max_cluster_size();
    ctx->sor_max_cluster = ctx->sor_dev_cluster;
    ctx->sor_rt = (nop == 1) ? 2 : 1;
    VarRefPlanes probe{};
    const int fw = width >> prm->sc_l, fh = height >> prm->sc_l;
    if (!sor_band_plan(fw, fh, ctx->sor_rt, 128, ctx->sor_max_cluster, nop, prm->tv_solverit, &probe)) {
      ofdis_destroy(ctx);
      return OFDIS_ERR_UNSUPPORTED;
    }
  }
  ctx->pp.max_iter = prm->max_iter;
  ctx->pp.min_iter = prm->min_iter;
  ctx->pp.costfct = prm->costfct;
  ctx->pp.patnorm = prm->patnorm;
  ctx->pp.dp_thresh_sq = prm->dp_thresh * prm->dp_thresh;  // oflow.cpp:88
  ctx->pp.dr_thresh = prm->dr_thresh;
  ctx->pp.res_thresh = prm->res_thresh;

  // geometry + packed image layout: per frame, level sc_f down to sc_l, I0 I0x I0y I1
  ctx->lev.resize(ctx->nlev);
  ctx->img_off.resize((size_t)ctx->nlev * 4);
  // packed frame: [for level sc_f..sc_l: I0, I1] then [for level sc_f..sc_l: I0x, I0y].  The image
  // block is contiguous so that ofdis_upload_packed_images can move it with one 2-D copy and derive
  // the gradients on the device.
  size_t off = 0;
  for (int pass = 0; pass < 2; ++pass)
    for (int sl = prm->sc_f; sl >= prm->sc_l; --sl) {
      LevelGeom& L = ctx->lev[sl - prm->sc_l];
      if (pass == 0) make_level(L, ctx, sl);
      const size_t n = (size_t)L.tmp_w * L.tmp_h * L.noc;
      const int which[2][2] = {{0, 3}, {1, 2}};  // pass 0: I0, I1; pass 1: I0x, I0y
      for (int k = 0; k < 2; ++k) {
        ctx->img_off[(size_t)(sl - prm->sc_l) * 4 + which[pass][k]] = off;
        off += (n + 3) / 4 * 4;  // keep every array 16-byte aligned
      }
    }
  ctx->frame_floats = off;
  ctx->images_floats = ctx->img_off[(size_t)(prm->sc_f - prm->sc_l) * 4 + 1];  // first gradient array starts where the images end

  auto dalloc = [&](void** p, size_t bytes) -> bool {
    return cudaMalloc(p, bytes ? bytes : 16) == cudaSuccess;
  };
  bool ok = dalloc((void**)&ctx->d_img, sizeof(float) * ctx->frame_floats * cap);
  ctx->d_flow.assign(ctx->nlev + 1, nullptr);
  ctx->flow_floats.assign(ctx->nlev + 1, 0);
  for (int li = 0; li <= ctx->nlev && ok; ++li) {
    const int sl = prm->sc_l + li;
    const size_t n = (size_t)(width >> sl) * (height >> sl) * nop;
    ctx->flow_floats[li] = n;
    ok = dalloc((void**)&ctx->d_flow[li], sizeof(float) * n * cap);
    if (ok) cudaMemsetAsync(ctx->d_flow[li], 0, sizeof(float) * n * cap, ctx->stream);
  }
  for (int li = 0; li < ctx->nlev && ok; ++li) {
    LevelGeom& L = ctx->lev[li];
    // device layout == the packed host frame: [frame][I0,I1 of all levels | I0x,I0y of all levels], so that
    // ofdis_upload_packed is ONE contiguous copy (two 64-row 2-D copies reached 44 of the link's 54 GB/s)
    for (int k = 0; k < 4; ++k) {
      L.img[k] = ctx->d_img + ctx->img_off[(size_t)li * 4 + k];
      L.img_fs[k] = ctx->frame_floats;
    }
    L.flow = ctx->d_flow[li];
    L.flow_frame_stride = ctx->flow_floats[li];
    L.flow_prev = ctx->d_flow[li + 1];
    L.flow_prev_frame_stride = ctx->flow_floats[li + 1];
    ok = ok && dalloc((void**)&L.pat_p, sizeof(float) * L.np * nop * cap);
    ok = ok && dalloc((void**)&L.pat_w, sizeof(float) * (size_t)L.np * L.novals * cap);
    ok = ok && dalloc((void**)&L.pat_conv, sizeof(int) * L.np * cap);
    ok = ok && dalloc((void**)&L.pat_cnt, sizeof(int) * L.np * cap);
    L.fb = ctx->dirs == 2 ? 1 : 0;
    L.fstep = 1;
    L.fb_pos = nullptr;
    L.fb_wbil = nullptr;
    L.fb_reach = nullptr;
    if (L.fb) {
      ok = ok && dalloc((void**)&L.fb_pos, sizeof(int) * 2 * L.np * cap);
      ok = ok && dalloc((void**)&L.fb_wbil, sizeof(float) * 4 * L.np * cap);
      ok = ok && dalloc((void**)&L.fb_reach, sizeof(int) * cap);
    }
  }
  if (ok && prm->usetvref) {
    // refinement planes sized for the finest level: mask, avg[C], 8 x deriv[C], and the SOR's lane rows
    const LevelGeom& Lf = ctx->lev[0];
    const size_t plane = (size_t)Lf.pitch * Lf.h;
    const int C = prm->noc;
    // band-skewed SOR array: nb bands x (W4 + hpad + 2) diagonals x hpad lanes x lpitch float4; sized for
    // the largest level under every plan ofdis_set_option can select
    size_t recf4 = 0;
    for (const LevelGeom& L : ctx->lev)
      for (int mc = 8; mc <= ctx->sor_dev_cluster; mc += 8)
        for (int sm = 32; sm <= 128; sm *= 2)
          for (int rt = 1; rt <= 4; rt *= 2) {
            VarRefPlanes t{};
            if (sor_band_plan(L.w, L.h, rt, sm, mc, nop, prm->tv_solverit, &t))
              recf4 = std::max(recf4, (size_t)t.nb * t.ndiag * t.hpad * t.lpitch);
          }
    for (const LevelGeom& L : ctx->lev)  // lane mode (sor_lane_kernel) of the levels it can take
      if (sor_lane_fits(L.h, 1)) recf4 = std::max(recf4, lane_frame_f4(L.w, L.h));
    const size_t per_frame = plane * (1 + C + 8 * C) + recf4 * 4;
    ok = dalloc((void**)&ctx->d_planes, sizeof(float) * per_frame * cap);
    if (ok) {
      // never-written lane rows (wavefront ramps, padded lanes) are read by idle SOR lanes: keep them finite
      cudaMemsetAsync(ctx->d_planes, 0, sizeof(float) * per_frame * cap, ctx->stream);
      float* q = ctx->d_planes;
      VarRefPlanes& P = ctx->planes;
      P.rec = reinterpret_cast<float4*>(q); q += recf4 * 4 * cap;   // first (alignment)
      P.mask = q; q += plane * cap;
      P.avg = q; q += plane * C * cap;
      for (int k = 0; k < 8; ++k) { P.deriv[k] = q; q += plane * C * cap; }
      P.plane = plane;
    }
  }
  if (!ok) {
    ofdis_destroy(ctx);
    return OFDIS_ERR_NOMEM;
  }
  *out = ctx;
  return OFDIS_OK;
}

int ofdis_destroy(ofdis_ctx* ctx) {
  if (!ctx) return OFDIS_OK;
  cudaSetDevice(ctx->device);
  if (ctx->stream) cudaStreamSynchronize(ctx->stream);
  for (auto& kv : ctx->graphs) cudaGraphExecDestroy(kv.second);
  cudaFree(ctx->d_img);
  cudaFree(ctx->d_stage);
  cudaFree(ctx->d_full);
  for (float* p : ctx->d_flow) cudaFree(p);
  for (LevelGeom& L : ctx->lev) {
    cudaFree(L.pat_p);
    cudaFree(L.pat_w);
    cudaFree(L.pat_conv);
    cudaFree(L.pat_cnt);
    cudaFree(L.fb_pos);
    cudaFree(L.fb_wbil);
    cudaFree(L.fb_reach);
  }
  cudaFree(ctx->d_planes);
  cudaFree(ctx->d_fast);
  if (ctx->own_stream) cudaStreamDestroy(ctx->stream);
  delete ctx;
  return OFDIS_OK;
}

int ofdis_set_camlr(ofdis_ctx* ctx, int camlr) {
  if (!ctx || (camlr != 0 && camlr != 1)) return OFDIS_ERR_ARG;
  for (LevelGeom& L : ctx->lev) L.camlr = camlr;
  for (auto& kv : ctx->graphs) cudaGraphExecDestroy(kv.second);  // kernel arguments changed
  ctx->graphs.clear();
  return OFDIS_OK;
}

int ofdis_set_dp_thresh_sq(ofdis_ctx* ctx, float dp_thresh_sq) {
  if (!ctx) return OFDIS_ERR_ARG;
  ctx->pp.dp_thresh_sq = dp_thresh_sq;
  for (auto& kv : ctx->graphs) cudaGraphExecDestroy(kv.second);
  ctx->graphs.clear();
  return OFDIS_OK;
}

int ofdis_level_info(const ofdis_ctx* ctx, int level, int* w, int* h, int* nopw, int* noph, int* steps) {
  if (!ctx) return OFDIS_ERR_ARG;
  const LevelGeom* L = level_of(const_cast<ofdis_ctx*>(ctx), level);
  if (!L) return OFDIS_ERR_ARG;
  if (w) *w = L->w;
  if (h) *h = L->h;
  if (nopw) *nopw = L->nopw;
  if (noph) *noph = L->noph;
  if (steps) *steps = L->steps;
  return OFDIS_OK;
}

int ofdis_upload_level(ofdis_ctx* ctx, int frame, int level, const float* i0, const float* i0x,
                       const float* i0y, const float* i1, int memkind) {
  if (!ctx) return OFDIS_ERR_ARG;
  LevelGeom* L = level_of(ctx, level);
  if (!L || frame < 0 || frame >= ctx->max_frames || !i0 || !i0x || !i0y || !i1) return fail(ctx, OFDIS_ERR_ARG, "upload_level: bad argument");
  CK(cudaSetDevice(ctx->device));
  if (ctx->dirs == 2) return fail(ctx, OFDIS_ERR_ARG, "upload_level: usefbcon needs the gradients of the second image, use ofdis_upload_level_fb");
  const size_t n = (size_t)L->tmp_w * L->tmp_h * L->noc;
  const float* src[4] = {i0, i0x, i0y, i1};
  for (int k = 0; k < 4; ++k)
    CK(cudaMemcpyAsync(const_cast<float*>(L->img[k]) + (size_t)frame * L->img_fs[k], src[k], sizeof(float) * n,
                       kind_in(memkind), ctx->stream));
  return OFDIS_OK;
}

int ofdis_upload_level_fb(ofdis_ctx* ctx, int frame, int level, const float* i0, const float* i0x, const float* i0y,
                          const float* i1, const float* i1x, const float* i1y, int memkind) {
  if (!ctx) return OFDIS_ERR_ARG;
  LevelGeom* L = level_of(ctx, level);
  if (!L || frame < 0 || frame >= ctx->max_frames || !i0 || !i0x || !i0y || !i1) return fail(ctx, OFDIS_ERR_ARG, "upload_level_fb: bad argument");
  if (ctx->dirs == 2 && (!i1x || !i1y)) return fail(ctx, OFDIS_ERR_ARG, "upload_level_fb: usefbcon needs i1x, i1y");
  CK(cudaSetDevice(ctx->device));
  const size_t n = (size_t)L->tmp_w * L->tmp_h * L->noc;
  // forward frame: template I0 (+ gradients), target I1; backward frame: the swapped pair (oflow.cpp:191-197)
  const float* src[2][4] = {{i0, i0x, i0y, i1}, {i1, i1x, i1y, i0}};
  for (int d = 0; d < ctx->dirs; ++d)
    for (int k = 0; k < 4; ++k)
      CK(cudaMemcpyAsync(const_cast<float*>(L->img[k]) + (size_t)(frame * ctx->dirs + d) * L->img_fs[k], src[d][k],
                         sizeof(float) * n, kind_in(memkind), ctx->stream));
  return OFDIS_OK;
}

int ofdis_get_level(ofdis_ctx* ctx, int frame, int level, int which, float* dst, int memkind) {
  if (!ctx) return OFDIS_ERR_ARG;
  LevelGeom* L = level_of(ctx, level);
  if (!L || frame < 0 || frame >= ctx->max_frames || which < 0 || which > 3 || !dst) return fail(ctx, OFDIS_ERR_ARG, "get_level: bad argument");
  CK(cudaSetDevice(ctx->device));
  const size_t n = (size_t)L->tmp_w * L->tmp_h * L->noc;
  CK(cudaMemcpyAsync(dst, L->img[which] + (size_t)frame * ctx->dirs * L->img_fs[which], sizeof(float) * n, kind_out(memkind), ctx->stream));
  if (memkind != OFDIS_MEM_DEVICE) CK(cudaStreamSynchronize(ctx->stream));
  return OFDIS_OK;
}

size_t ofdis_packed_frame_floats(const ofdis_ctx* ctx) { return ctx ? ctx->frame_floats : 0; }

size_t ofdis_packed_offset(const ofdis_ctx* ctx, int level, int which) {
  if (!ctx || level < ctx->prm.sc_l || level > ctx->prm.sc_f || which < 0 || which > 3) return (size_t)-1;
  return ctx->img_off[(size_t)(level - ctx->prm.sc_l) * 4 + which];
}

int ofdis_upload_packed(ofdis_ctx* ctx, int f0, int f1, const float* packed, int memkind) {
  if (!ctx) return OFDIS_ERR_ARG;
  if (f0 < 0 || f1 > ctx->max_frames || f0 >= f1 || !packed) return fail(ctx, OFDIS_ERR_ARG, "upload_packed: bad argument");
  if (ctx->dirs == 2) return fail(ctx, OFDIS_ERR_UNSUPPORTED, "upload_packed: a packed frame has no gradients of the second image; with usefbcon use ofdis_upload_level_fb or one of the image-only uploads");
  CK(cudaSetDevice(ctx->device));
  // host and device share the frame layout: one contiguous copy
  CK(cudaMemcpyAsync(ctx->d_img + (size_t)f0 * ctx->frame_floats, packed, sizeof(float) * ctx->frame_floats * (f1 - f0),
                     kind_in(memkind), ctx->stream));
  return OFDIS_OK;
}

// Images of the forward frames are in place: fill the backward frames with the swapped pair
// (usefbcon) and derive the template gradients of every internal frame on every level.
static int finish_gradients(ofdis_ctx* ctx, int f0, int f1) {
  const int D = ctx->dirs, q0 = f0 * D, q1 = f1 * D;
  for (int sl = ctx->prm.sc_f; sl >= ctx->prm.sc_l; --sl) {
    const LevelGeom& L = ctx->lev[sl - ctx->prm.sc_l];
    if (D == 2) {
      if (launch_swap_images(L, q0, q1, ctx->stream) < 0) return fail(ctx, OFDIS_ERR_CUDA, "swap_images_kernel launch", cudaGetLastError());
      ctx->launches += 1;
    }
    if (launch_sobel(L, q0, q1, ctx->stream) < 0) return fail(ctx, OFDIS_ERR_CUDA, "sobel_kernel launch", cudaGetLastError());
    ctx->launches += 1;
  }
  return OFDIS_OK;
}

size_t ofdis_packed_images_frame_floats(const ofdis_ctx* ctx) { return ctx ? ctx->images_floats : 0; }

int ofdis_upload_packed_images(ofdis_ctx* ctx, int f0, int f1, const float* packed, int memkind) {
  if (!ctx) return OFDIS_ERR_ARG;
  if (f0 < 0 || f1 > ctx->max_frames || f0 >= f1 || !packed) return fail(ctx, OFDIS_ERR_ARG, "upload_packed_images: bad argument");
  CK(cudaSetDevice(ctx->device));
  // the image part of every (forward) frame: one 2-D copy, a row per frame
  const int D = ctx->dirs;
  const size_t nif = ctx->images_floats;
  CK(cudaMemcpy2DAsync(ctx->d_img + (size_t)f0 * D * ctx->frame_floats, sizeof(float) * ctx->frame_floats * D, packed,
                       sizeof(float) * nif, sizeof(float) * nif, (size_t)(f1 - f0), kind_in(memkind), ctx->stream));
  return finish_gradients(ctx, f0, f1);
}

// Coarser levels by 2x2 box means (forward frames), then finish_gradients.
static int finish_pyramid(ofdis_ctx* ctx, int f0, int f1) {
  NvtxRange nvtx("pyramid", -1);
  const int D = ctx->dirs, q0 = f0 * D, nq = f1 - f0;
  for (int sl = ctx->prm.sc_l + 1; sl <= ctx->prm.sc_f; ++sl) {
    const LevelGeom gs = stepped(ctx->lev[sl - 1 - ctx->prm.sc_l], D), gd = stepped(ctx->lev[sl - ctx->prm.sc_l], D);
    if (launch_pyr_down(gs, gd, q0, q0 + nq, ctx->stream) < 0)
      return fail(ctx, OFDIS_ERR_CUDA, "pyr_down_kernel launch", cudaGetLastError());
    ctx->launches += 1;
  }
  return finish_gradients(ctx, f0, f1);
}

static int ensure_stage(ofdis_ctx* ctx, size_t bytes) {
  if (ctx->stage_bytes >= bytes) return OFDIS_OK;
  CK(cudaStreamSynchronize(ctx->stream));
  cudaFree(ctx->d_stage);
  ctx->d_stage = nullptr;
  ctx->stage_bytes = 0;
  if (cudaMalloc(&ctx->d_stage, bytes) != cudaSuccess) return fail(ctx, OFDIS_ERR_NOMEM, "staging buffer");
  ctx->stage_bytes = bytes;
  return OFDIS_OK;
}

static int org_padding(ofdis_ctx* ctx, int width_org, int height_org, int* padl, int* padt) {
  // run_dense.cpp:299-311: pad up to the next multiple of 2^lv_f, floor(pad/2) on the left/top
  const int scf = 1 << ctx->prm.sc_f;
  if (width_org <= 0 || height_org <= 0 || (width_org + scf - 1) / scf * scf != ctx->width ||
      (height_org + scf - 1) / scf * scf != ctx->height)
    return fail(ctx, OFDIS_ERR_ARG, "frame size does not pad to the context's width/height");
  *padl = (ctx->width - width_org) / 2;
  *padt = (ctx->height - height_org) / 2;
  return OFDIS_OK;
}

int ofdis_upload_frames_u8(ofdis_ctx* ctx, int f0, int f1, const unsigned char* frames, int width_org, int height_org,
                           int memkind) {
  if (!ctx) return OFDIS_ERR_ARG;
  if (f0 < 0 || f1 > ctx->max_frames || f0 >= f1 || !frames) return fail(ctx, OFDIS_ERR_ARG, "upload_frames_u8: bad argument");
  if (ctx->prm.sc_l > 8) return fail(ctx, OFDIS_ERR_UNSUPPORTED, "upload_frames_u8: box sums are exact in float32 up to level 8");
  PyrSourceU8 src;
  int rc = org_padding(ctx, width_org, height_org, &src.pad_left, &src.pad_top);
  if (rc) return rc;
  CK(cudaSetDevice(ctx->device));
  src.w_org = width_org;
  src.h_org = height_org;
  src.image_bytes = (size_t)width_org * height_org * ctx->prm.noc;
  src.frames = frames;
  if (memkind != OFDIS_MEM_DEVICE) {
    const size_t bytes = src.image_bytes * 2 * (size_t)(f1 - f0);
    rc = ensure_stage(ctx, src.image_bytes * 2 * (size_t)ctx->max_frames);
    if (rc) return rc;
    CK(cudaMemcpyAsync(ctx->d_stage, frames, bytes, cudaMemcpyHostToDevice, ctx->stream));
    src.frames = static_cast<const unsigned char*>(ctx->d_stage);
  }
  if (launch_pyr_from_u8(stepped(ctx->lev[0], ctx->dirs), f0 * ctx->dirs, f0 * ctx->dirs + (f1 - f0), src, ctx->stream) < 0)
    return fail(ctx, OFDIS_ERR_CUDA, "pyr_from_u8_kernel launch", cudaGetLastError());
  ctx->launches += 1;
  return finish_pyramid(ctx, f0, f1);
}

size_t ofdis_finest_level_frame_floats(const ofdis_ctx* ctx) {
  return ctx ? (size_t)2 * ctx->lev[0].w * ctx->lev[0].h * ctx->lev[0].noc : 0;
}

int ofdis_upload_finest_level(ofdis_ctx* ctx, int f0, int f1, const float* packed, int memkind) {
  if (!ctx) return OFDIS_ERR_ARG;
  if (f0 < 0 || f1 > ctx->max_frames || f0 >= f1 || !packed) return fail(ctx, OFDIS_ERR_ARG, "upload_finest_level: bad argument");
  CK(cudaSetDevice(ctx->device));
  const size_t per = ofdis_finest_level_frame_floats(ctx);
  const float* src = packed;
  if (memkind != OFDIS_MEM_DEVICE) {
    int rc = ensure_stage(ctx, sizeof(float) * per * (size_t)ctx->max_frames);
    if (rc) return rc;
    CK(cudaMemcpyAsync(ctx->d_stage, packed, sizeof(float) * per * (size_t)(f1 - f0), cudaMemcpyHostToDevice, ctx->stream));
    src = static_cast<const float*>(ctx->d_stage);
  }
  if (launch_pyr_from_level(stepped(ctx->lev[0], ctx->dirs), f0 * ctx->dirs, f0 * ctx->dirs + (f1 - f0), src, ctx->stream) < 0)
    return fail(ctx, OFDIS_ERR_CUDA, "pyr_from_level_kernel launch", cudaGetLastError());
  ctx->launches += 1;
  return finish_pyramid(ctx, f0, f1);
}

int ofdis_get_flow_fullres(ofdis_ctx* ctx, int f0, int f1, float* out, int width_org, int height_org, int memkind) {
  if (!ctx) return OFDIS_ERR_ARG;
  if (f0 < 0 || f1 > ctx->max_frames || f0 >= f1 || !out) return fail(ctx, OFDIS_ERR_ARG, "get_flow_fullres: bad argument");
  int cx, cy;
  int rc = org_padding(ctx, width_org, height_org, &cx, &cy);
  if (rc) return rc;
  NvtxRange nvtx("upsample", -1);
  CK(cudaSetDevice(ctx->device));
  const size_t per = (size_t)width_org * height_org * ctx->nop;
  float* dst = out;
  if (memkind != OFDIS_MEM_DEVICE) {
    const size_t need = per * (size_t)ctx->max_frames;
    if (ctx->full_floats < need) {
      CK(cudaStreamSynchronize(ctx->stream));
      cudaFree(ctx->d_full);
      ctx->d_full = nullptr;
      ctx->full_floats = 0;
      if (cudaMalloc((void**)&ctx->d_full, sizeof(float) * need) != cudaSuccess)
        return fail(ctx, OFDIS_ERR_NOMEM, "full-resolution flow buffer");
      ctx->full_floats = need;
    }
    dst = ctx->d_full;
  }
  if (launch_flow_upsample(stepped(ctx->lev[0], ctx->dirs), f0 * ctx->dirs, f0 * ctx->dirs + (f1 - f0), dst, width_org, height_org,
                           cx, cy, ctx->stream) < 0)
    return fail(ctx, OFDIS_ERR_CUDA, "flow_upsample_kernel launch", cudaGetLastError());
  ctx->launches += 1;
  if (memkind != OFDIS_MEM_DEVICE)
    CK(cudaMemcpyAsync(out, dst, sizeof(float) * per * (size_t)(f1 - f0), cudaMemcpyDeviceToHost, ctx->stream));
  return OFDIS_OK;
}

int ofdis_patgrid_optimize(ofdis_ctx* ctx, int level, int f0, int f1, int init_from_coarser) {
  if (!ctx) return OFDIS_ERR_ARG;
  LevelGeom* L = level_of(ctx, level);
  if (!L || f0 < 0 || f1 > ctx->max_frames || f0 >= f1) return fail(ctx, OFDIS_ERR_ARG, "patgrid_optimize: bad argument");
  CK(cudaSetDevice(ctx->device));
  if (ctx->sel_dir >= 0 && f1 != f0 + 1) return fail(ctx, OFDIS_ERR_ARG, "patgrid_optimize: one frame at a time while a direction is selected");
  NvtxRange nvtx("patch", level);
  const int q0 = ctx->sel_dir >= 0 ? f0 * ctx->dirs + ctx->sel_dir : f0 * ctx->dirs;
  const int q1 = ctx->sel_dir >= 0 ? q0 + 1 : f1 * ctx->dirs;
  L->pdl = (ctx->pdl == 1 || (ctx->pdl == 2 && q1 - q0 <= SOR_LANE_AUTO_FRAMES)) ? 1 : 0;
  const int n = launch_patch_optimize(*L, ctx->pp, q0, q1, init_from_coarser != 0, ctx->stream, ctx->prof);
  if (n < 0) return fail(ctx, OFDIS_ERR_CUDA, "patch_optimize_kernel launch", cudaGetLastError());
  ctx->launches += n;
  return OFDIS_OK;
}

int ofdis_patgrid_aggregate(ofdis_ctx* ctx, int level, int f0, int f1) {
  if (!ctx) return OFDIS_ERR_ARG;
  LevelGeom* L = level_of(ctx, level);
  if (!L || f0 < 0 || f1 > ctx->max_frames || f0 >= f1) return fail(ctx, OFDIS_ERR_ARG, "patgrid_aggregate: bad argument");
  CK(cudaSetDevice(ctx->device));
  NvtxRange nvtx("densify", level);
  L->pdl = (ctx->pdl == 1 || (ctx->pdl == 2 && (f1 - f0) * ctx->dirs <= SOR_LANE_AUTO_FRAMES)) ? 1 : 0;
  int n;
  if (ctx->dirs == 2) {
    // both grids' patch positions first; the backward flow is not densified on the last level (oflow.cpp:269-270)
    if (launch_fb_prepare(*L, f0 * 2, f1 * 2, ctx->stream) < 0) return fail(ctx, OFDIS_ERR_CUDA, "fb_prepare_kernel launch", cudaGetLastError());
    ctx->launches += 1;
    if (ctx->sel_dir >= 0)  // one grid of the couple (PatGridClass::AggregateFlowDense of either stand-alone grid)
      n = launch_densify(stepped(*L, 2), f0 * 2 + ctx->sel_dir, f0 * 2 + ctx->sel_dir + (f1 - f0), ctx->stream, ctx->prof);
    else
      n = (level == ctx->prm.sc_l) ? launch_densify(stepped(*L, 2), f0 * 2, f0 * 2 + (f1 - f0), ctx->stream, ctx->prof)
                                   : launch_densify(*L, f0 * 2, f1 * 2, ctx->stream, ctx->prof);
  } else {
    n = launch_densify(*L, f0, f1, ctx->stream, ctx->prof);
  }
  if (n < 0) return fail(ctx, OFDIS_ERR_CUDA, "densify_kernel launch", cudaGetLastError());
  ctx->launches += n;
  return OFDIS_OK;
}

static int varref_impl(ofdis_ctx* ctx, int level, int f0, int f1, int n_inner_override) {
  if (!ctx) return OFDIS_ERR_ARG;
  LevelGeom* L = level_of(ctx, level);
  if (!L || f0 < 0 || f1 > ctx->max_frames || f0 >= f1) return fail(ctx, OFDIS_ERR_ARG, "varref_refine: bad argument");
  if (!ctx->d_planes) return fail(ctx, OFDIS_ERR_ARG, "varref_refine: context created with usetvref=0");
  CK(cudaSetDevice(ctx->device));
  NvtxRange nvtx("varref", level);
  VarRefParams vp;
  // refine_variational.cpp:36-43
  vp.n_inner = n_inner_override >= 0 ? n_inner_override : ctx->prm.tv_innerit * (level + 1);
  vp.n_solver = ctx->prm.tv_solverit;
  vp.omega = ctx->prm.tv_sor;
  vp.quarter_alpha = 0.25f * ctx->prm.tv_alpha;
  vp.half_gamma_over3 = ctx->prm.tv_gamma * 0.5f / 3.0f;
  vp.half_delta_over3 = ctx->prm.tv_delta * 0.5f / 3.0f;
  VarRefPlanes pl = ctx->planes;
  pl.plane = (size_t)L->pitch * L->h;
  if (!sor_band_plan(L->w, L->h, ctx->sor_rt, ctx->sor_single_max, ctx->sor_max_cluster, ctx->nop, ctx->prm.tv_solverit, &pl))
    return fail(ctx, OFDIS_ERR_UNSUPPORTED, "varref_refine: level too tall for the largest SOR cluster");
  pl.rec_stride = (size_t)pl.nb * pl.ndiag * pl.hpad * pl.lpitch;
  pl.lane = 0;
  const int nlaunch = (f1 - f0) * ctx->dirs;  // frames per launch
  L->pdl = (ctx->pdl == 1 || (ctx->pdl == 2 && nlaunch <= SOR_LANE_AUTO_FRAMES)) ? 1 : 0;
  if ((ctx->sor_lane == 1 || (ctx->sor_lane == 2 && nlaunch <= SOR_LANE_AUTO_FRAMES && sor_lane_preferred(L->h, ctx->prm.tv_solverit))) &&
      !pl.fast && sor_lane_fits(L->h, 1)) {  // lane-skewed layout, bands of 32 rows
    pl.lane = 1;
    pl.nb = (L->h + 31) / 32;
    pl.ndiag = lane_ndiag(L->w);
    pl.rec_stride = lane_frame_f4(L->w, L->h);
  }
  pl.frec_stride = pl.plane * 8;   // fast mode: natural layout at this level's plane size
  pl.fdu_stride = pl.plane * 4;
  // usefbcon: both directions are refined except on the last level (oflow.cpp:285-294)
  const int D = ctx->dirs;
  const bool fwd_only = (D == 2 && level == ctx->prm.sc_l);
  const int n = fwd_only ? launch_varref(stepped(*L, 2), pl, vp, f0 * 2, f0 * 2 + (f1 - f0), ctx->stream, ctx->prof)
                         : launch_varref(*L, pl, vp, f0 * D, f1 * D, ctx->stream, ctx->prof);
  if (n < 0) return fail(ctx, OFDIS_ERR_CUDA, "varref kernels launch", cudaGetLastError());
  ctx->launches += n;
  ctx->last_vr_level = level;
  ctx->last_vr_lane = pl.lane;
  ctx->last_vr_fcur = vp.n_inner & 1;
  ctx->last_vr_f0 = f0;
  ctx->last_vr_fstep = fwd_only ? 1 : D;  // workspace slots per user frame
  return OFDIS_OK;
}

int ofdis_varref_refine(ofdis_ctx* ctx, int level, int f0, int f1) { return varref_impl(ctx, level, f0, f1, -1); }

int ofdis_debug_varref_iters(ofdis_ctx* ctx, int level, int f0, int f1, int n_inner) {
  return varref_impl(ctx, level, f0, f1, n_inner);
}

int ofdis_set_direction(ofdis_ctx* ctx, int dir) {
  if (!ctx || dir < -1 || dir > 1 || (dir >= 0 && ctx->dirs != 2)) return OFDIS_ERR_ARG;
  ctx->sel_dir = dir;
  return OFDIS_OK;
}

int ofdis_set_option(ofdis_ctx* ctx, const char* name, int value) {
  if (!ctx || !name) return OFDIS_ERR_ARG;
  if (!strcmp(name, "sor_single_max")) {
    if (value != 32 && value != 64 && value != 128) return fail(ctx, OFDIS_ERR_ARG, "sor_single_max: 32, 64 or 128");
    ctx->sor_single_max = value;
  } else if (!strcmp(name, "sor_max_cluster")) {
    if (value != 8 && value != 16) return fail(ctx, OFDIS_ERR_ARG, "sor_max_cluster: 8 or 16");
    if (value > ctx->sor_dev_cluster) return fail(ctx, OFDIS_ERR_UNSUPPORTED, "sor_max_cluster: the device does not grant clusters of 16 CTAs");
    VarRefPlanes probe{};
    if (ctx->prm.usetvref && !sor_band_plan(ctx->lev[0].w, ctx->lev[0].h, ctx->sor_rt, 128, value, ctx->nop, ctx->prm.tv_solverit, &probe))
      return fail(ctx, OFDIS_ERR_UNSUPPORTED, "sor_max_cluster: the finest level needs the larger cluster");
    ctx->sor_max_cluster = value;
  } else if (!strcmp(name, "sor_lane")) {
    if (value < 0 || value > 2) return fail(ctx, OFDIS_ERR_ARG, "sor_lane: 0, 1 or 2");
    ctx->sor_lane = value;
  } else if (!strcmp(name, "pdl")) {
    if (value < 0 || value > 2) return fail(ctx, OFDIS_ERR_ARG, "pdl: 0, 1 or 2");
    ctx->pdl = value;
  } else if (!strcmp(name, "sor_fast")) {
    if (value != 0 && value != 1) return fail(ctx, OFDIS_ERR_ARG, "sor_fast: 0 or 1");
    if (!ctx->d_planes) return fail(ctx, OFDIS_ERR_ARG, "sor_fast: context created with usetvref=0");
    if (value && rb_smem_limit_exceeded(ctx->nop, ctx->prm.tv_solverit))
      return fail(ctx, OFDIS_ERR_UNSUPPORTED, "sor_fast: too many sweeps for the tile's halo");
    if (value && !ctx->d_fast) {  // records 8 floats per pixel + 2 x 2 planes of (du,dv), finest level x frames
      const size_t plane = ctx->planes.plane;
      CK(cudaSetDevice(ctx->device));
      if (cudaMalloc((void**)&ctx->d_fast, sizeof(float) * plane * 12 * ctx->cap) != cudaSuccess)
        return fail(ctx, OFDIS_ERR_NOMEM, "sor_fast workspace");
      cudaMemsetAsync(ctx->d_fast, 0, sizeof(float) * plane * 12 * ctx->cap, ctx->stream);
      ctx->planes.frec = ctx->d_fast;
      ctx->planes.fdu = ctx->d_fast + plane * 8 * ctx->cap;
    }
    ctx->planes.fast = value;
  } else if (!strcmp(name, "sor_rows_per_thread")) {
    if (value != 1 && value != 2 && value != 4) return fail(ctx, OFDIS_ERR_ARG, "sor_rows_per_thread: 1, 2 or 4");
    VarRefPlanes probe{};
    if (ctx->prm.usetvref && !sor_band_plan(ctx->lev[0].w, ctx->lev[0].h, value, 128, ctx->sor_max_cluster, ctx->nop, ctx->prm.tv_solverit, &probe))
      return fail(ctx, OFDIS_ERR_UNSUPPORTED, "sor_rows_per_thread: the finest level needs more rows per thread or the larger cluster");
    ctx->sor_rt = value;
  } else {
    return fail(ctx, OFDIS_ERR_ARG, "set_option: unknown option");
  }
  for (auto& kv : ctx->graphs) cudaGraphExecDestroy(kv.second);  // launch geometry changed
  ctx->graphs.clear();
  return OFDIS_OK;
}

int ofdis_set_graph_mode(ofdis_ctx* ctx, int enabled) {
  if (!ctx) return OFDIS_ERR_ARG;
  ctx->graph_mode = enabled != 0;
  return OFDIS_OK;
}

int ofdis_run(ofdis_ctx* ctx, int nframes, int use_initflow) {
  if (!ctx) return OFDIS_ERR_ARG;
  if (nframes < 1 || nframes > ctx->max_frames) return fail(ctx, OFDIS_ERR_ARG, "run: bad frame count");
  CK(cudaSetDevice(ctx->device));
  NvtxRange nvtx(ctx->graph_mode ? "run (graph)" : "run", -1);
  if (!ctx->graph_mode) return run_levels(ctx, nframes, use_initflow);
  const long key = (long)nframes * 2 + (use_initflow ? 1 : 0);
  auto it = ctx->graphs.find(key);
  if (it == ctx->graphs.end()) {
    const long before = ctx->launches;
    cudaGraph_t graph = nullptr;
    CK(cudaStreamBeginCapture(ctx->stream, cudaStreamCaptureModeThreadLocal));
    const int rc = run_levels(ctx, nframes, use_initflow);
    cudaError_t e = cudaStreamEndCapture(ctx->stream, &graph);
    if (rc || e != cudaSuccess) {
      if (graph) cudaGraphDestroy(graph);
      return rc ? rc : fail(ctx, OFDIS_ERR_CUDA, "cudaStreamEndCapture", e);
    }
    cudaGraphExec_t exec = nullptr;
    e = cudaGraphInstantiate(&exec, graph, 0);
    cudaGraphDestroy(graph);
    if (e != cudaSuccess) return fail(ctx, OFDIS_ERR_CUDA, "cudaGraphInstantiate", e);
    ctx->graph_launches[key] = ctx->launches - before;
    ctx->launches = before;  // capture does not execute
    it = ctx->graphs.emplace(key, exec).first;
  }
  CK(cudaGraphLaunch(it->second, ctx->stream));
  ctx->launches += ctx->graph_launches[key];
  return OFDIS_OK;
}

int ofdis_sync(ofdis_ctx* ctx) {
  if (!ctx) return OFDIS_ERR_ARG;
  CK(cudaStreamSynchronize(ctx->stream));
  return OFDIS_OK;
}

static int flow_index(const ofdis_ctx* ctx, int level) {
  if (level < ctx->prm.sc_l || level > ctx->prm.sc_f + 1) return -1;
  return level - ctx->prm.sc_l;
}

int ofdis_get_flow(ofdis_ctx* ctx, int frame, int level, float* dst, int memkind) {
  if (!ctx) return OFDIS_ERR_ARG;
  const int li = flow_index(ctx, level);
  if (li < 0 || frame < 0 || frame >= ctx->max_frames || !dst) return fail(ctx, OFDIS_ERR_ARG, "get_flow: bad argument");
  CK(cudaMemcpyAsync(dst, ctx->d_flow[li] + (size_t)(frame * ctx->dirs + std::max(ctx->sel_dir, 0)) * ctx->flow_floats[li],
                     sizeof(float) * ctx->flow_floats[li], kind_out(memkind), ctx->stream));
  if (memkind == OFDIS_MEM_HOST) CK(cudaStreamSynchronize(ctx->stream));
  return OFDIS_OK;
}

int ofdis_set_flow(ofdis_ctx* ctx, int frame, int level, const float* src, int memkind) {
  if (!ctx) return OFDIS_ERR_ARG;
  const int li = flow_index(ctx, level);
  if (li < 0 || frame < 0 || frame >= ctx->max_frames || !src) return fail(ctx, OFDIS_ERR_ARG, "set_flow: bad argument");
  CK(cudaMemcpyAsync(ctx->d_flow[li] + (size_t)(frame * ctx->dirs + std::max(ctx->sel_dir, 0)) * ctx->flow_floats[li], src,
                     sizeof(float) * ctx->flow_floats[li], kind_in(memkind), ctx->stream));
  return OFDIS_OK;
}

int ofdis_get_flow_batch(ofdis_ctx* ctx, int f0, int f1, float* dst, int memkind) {
  if (!ctx) return OFDIS_ERR_ARG;
  if (f0 < 0 || f1 > ctx->max_frames || f0 >= f1 || !dst) return fail(ctx, OFDIS_ERR_ARG, "get_flow_batch: bad argument");
  const size_t nfl = ctx->flow_floats[0];
  if (ctx->dirs == 1)
    CK(cudaMemcpyAsync(dst, ctx->d_flow[0] + (size_t)f0 * nfl, sizeof(float) * nfl * (f1 - f0), kind_out(memkind), ctx->stream));
  else  // forward frames only
    CK(cudaMemcpy2DAsync(dst, sizeof(float) * nfl, ctx->d_flow[0] + (size_t)f0 * 2 * nfl, sizeof(float) * nfl * 2,
                         sizeof(float) * nfl, (size_t)(f1 - f0), kind_out(memkind), ctx->stream));
  return OFDIS_OK;
}

int ofdis_get_patches(ofdis_ctx* ctx, int frame, int level, float* p, float* pweight, int* conv, int* cnt) {
  if (!ctx) return OFDIS_ERR_ARG;
  LevelGeom* L = level_of(ctx, level);
  if (!L || frame < 0 || frame >= ctx->max_frames) return fail(ctx, OFDIS_ERR_ARG, "get_patches: bad argument");
  const size_t np = L->np;
  frame = frame * ctx->dirs + std::max(ctx->sel_dir, 0);  // the forward grid unless a direction is selected
  if (p) CK(cudaMemcpyAsync(p, L->pat_p + frame * np * L->nop, sizeof(float) * np * L->nop, cudaMemcpyDeviceToHost, ctx->stream));
  if (pweight) CK(cudaMemcpyAsync(pweight, L->pat_w + frame * np * L->novals, sizeof(float) * np * L->novals, cudaMemcpyDeviceToHost, ctx->stream));
  if (conv) CK(cudaMemcpyAsync(conv, L->pat_conv + frame * np, sizeof(int) * np, cudaMemcpyDeviceToHost, ctx->stream));
  if (cnt) CK(cudaMemcpyAsync(cnt, L->pat_cnt + frame * np, sizeof(int) * np, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  return OFDIS_OK;
}

long ofdis_debug_get(ofdis_ctx* ctx, const char* name, int frame, float* dst, size_t max_floats) {
  if (!ctx || !name || !dst || ctx->last_vr_level < 0) return OFDIS_ERR_ARG;
  LevelGeom* L = level_of(ctx, ctx->last_vr_level);
  const int fr = (frame - ctx->last_vr_f0) * ctx->last_vr_fstep;
  if (!L || fr < 0) return OFDIS_ERR_ARG;
  const size_t plane = (size_t)L->pitch * L->h;
  const int C = L->noc;
  static const char* dn[8] = {"Ix", "Iy", "Iz", "Ixx", "Ixy", "Iyy", "Ixz", "Iyz"};
  const float* src = nullptr;
  size_t n = 0;
  for (int k = 0; k < 8; ++k)
    if (!strcmp(name, dn[k])) {
      src = ctx->planes.deriv[k] + (size_t)fr * C * plane;
      n = plane * C;
    }
  if (!strcmp(name, "mask")) { src = ctx->planes.mask + (size_t)fr * plane; n = plane; }
  if (!strcmp(name, "dudv") || !strcmp(name, "rec")) {
    // stored skewed (see VarRefPlanes); returned in natural (h, pitch, per-pixel) order
    const bool is_rec = name[0] == 'r';
    if (ctx->planes.fast) {  // natural layout: records 8 floats per pixel, (du,dv) two planes of the current buffer
      const int per_f = is_rec ? (L->nop == 2 ? 8 : 5) : 2;
      if (plane * per_f > max_floats) return OFDIS_ERR_ARG;
      std::vector<float> raw(is_rec ? plane * 8 : plane * 2);
      const float* src_f = is_rec ? ctx->planes.frec + (size_t)fr * plane * 8
                                  : ctx->planes.fdu + (size_t)fr * plane * 4 + (size_t)ctx->last_vr_fcur * 2 * plane;
      if (cudaMemcpyAsync(raw.data(), src_f, sizeof(float) * raw.size(), cudaMemcpyDeviceToHost, ctx->stream) != cudaSuccess) return OFDIS_ERR_CUDA;
      if (cudaStreamSynchronize(ctx->stream) != cudaSuccess) return OFDIS_ERR_CUDA;
      for (size_t o = 0; o < plane; ++o)
        for (int e = 0; e < per_f; ++e) dst[o * per_f + e] = is_rec ? raw[o * 8 + e] : raw[(size_t)e * plane + o];
      return (long)(plane * per_f);
    }
    if (ctx->last_vr_lane) {  // lane-skewed layout (VarRefPlanes, lane mode)
      VarRefPlanes lp{};
      lp.nb = (L->h + 31) / 32;
      lp.ndiag = lane_ndiag(L->w);
      const int per_l = is_rec ? (L->nop == 2 ? 8 : 5) : 2;
      const size_t stride_l = lane_frame_f4(L->w, L->h);
      if (plane * per_l > max_floats) return OFDIS_ERR_ARG;
      std::vector<float> raw(stride_l * 4);
      if (cudaMemcpyAsync(raw.data(), ctx->planes.rec + (size_t)fr * stride_l, sizeof(float) * raw.size(), cudaMemcpyDeviceToHost, ctx->stream) != cudaSuccess) return OFDIS_ERR_CUDA;
      if (cudaStreamSynchronize(ctx->stream) != cudaSuccess) return OFDIS_ERR_CUDA;
      for (int j = 0; j < L->h; ++j)
        for (int i = 0; i < L->w; ++i)
          for (int e = 0; e < per_l; ++e)
            dst[((size_t)j * L->pitch + i) * per_l + e] =
                is_rec ? raw[lane_rec_f4(lp, i, j, e >> 2) * 4 + (e & 3)] : raw[lane_dudv_f(lp, i, j) + e];
      return (long)(plane * per_l);
    }
    VarRefPlanes bp{};
    if (!sor_band_plan(L->w, L->h, ctx->sor_rt, ctx->sor_single_max, ctx->sor_max_cluster, ctx->nop, ctx->prm.tv_solverit, &bp)) return OFDIS_ERR_UNSUPPORTED;
    const int per = is_rec ? bp.nq : 2;                              // floats per pixel
    const size_t stride = (size_t)bp.nb * bp.ndiag * bp.hpad * bp.lpitch;  // float4 per frame
    if (plane * per > max_floats) return OFDIS_ERR_ARG;
    std::vector<float> raw(stride * 4);
    const float4* base = ctx->planes.rec + (size_t)fr * stride;
    if (cudaMemcpyAsync(raw.data(), base, sizeof(float) * raw.size(), cudaMemcpyDeviceToHost, ctx->stream) != cudaSuccess) return OFDIS_ERR_CUDA;
    if (cudaStreamSynchronize(ctx->stream) != cudaSuccess) return OFDIS_ERR_CUDA;
    for (int j = 0; j < L->h; ++j)
      for (int i = 0; i < L->w; ++i)
        for (int e = 0; e < per; ++e) {
          // chunk e of the block's lane row holds field e of its 4 pixels; (du,dv) are chunks nq, nq+1
          const size_t f4 = band_f4(bp, i >> 2, j, is_rec ? e : bp.nq + e);
          dst[((size_t)j * L->pitch + i) * per + e] = raw[f4 * 4 + (i & 3)];
        }
    return (long)(plane * per);
  }
  if (!src || n > max_floats) return OFDIS_ERR_ARG;
  if (cudaMemcpyAsync(dst, src, sizeof(float) * n, cudaMemcpyDeviceToHost, ctx->stream) != cudaSuccess) return OFDIS_ERR_CUDA;
  if (cudaStreamSynchronize(ctx->stream) != cudaSuccess) return OFDIS_ERR_CUDA;
  return (long)n;
}

long ofdis_launch_count(const ofdis_ctx* ctx) { return ctx ? ctx->launches : 0; }

int ofdis_profile_run(ofdis_ctx* ctx, int nframes, int steps, double* ms_by_class, long* launches_by_class) {
  return ofdis_profile_levels(ctx, nframes, steps, ms_by_class, launches_by_class, nullptr);
}

int ofdis_profile_levels(ofdis_ctx* ctx, int nframes, int steps, double* ms_by_class, long* launches_by_class,
                         double* ms_by_level_class) {
  if (!ctx || steps < 1 || !ms_by_class || !launches_by_class) return OFDIS_ERR_ARG;
  if (nframes < 1 || nframes > ctx->max_frames) return fail(ctx, OFDIS_ERR_ARG, "profile_run: bad frame count");
  CK(cudaSetDevice(ctx->device));
  Profiler prof;
  prof.st = ctx->stream;
  ctx->prof = &prof;
  int rc = OFDIS_OK;
  for (int s = 0; s < steps && rc == OFDIS_OK; ++s) rc = run_levels(ctx, nframes, 0);
  ctx->prof = nullptr;
  cudaError_t e = cudaStreamSynchronize(ctx->stream);
  for (int k = 0; k < KC_COUNT; ++k) {
    ms_by_class[k] = 0.0;
    launches_by_class[k] = 0;
  }
  if (ms_by_level_class)
    for (int k = 0; k < ctx->nlev * KC_COUNT; ++k) ms_by_level_class[k] = 0.0;
  for (auto& r : prof.recs) {
    float ms = 0.f;
    if (e == cudaSuccess && cudaEventElapsedTime(&ms, r.a, r.b) == cudaSuccess) {
      ms_by_class[r.cls] += ms;
      launches_by_class[r.cls] += 1;
      if (ms_by_level_class && r.level >= ctx->prm.sc_l && r.level <= ctx->prm.sc_f)
        ms_by_level_class[(r.level - ctx->prm.sc_l) * KC_COUNT + r.cls] += ms;
    }
    cudaEventDestroy(r.a);
    cudaEventDestroy(r.b);
  }
  if (rc) return rc;
  if (e != cudaSuccess) return fail(ctx, OFDIS_ERR_CUDA, "profile_run sync", e);
  return OFDIS_OK;
}

}  // extern "C"
