// Internal declarations shared by the CUDA translation units of libofdis_b200.
// sm_100a only; compiled with -fmad=false (no FMA contraction) because results
// must be bitwise equal to the reference CPU build (DESIGN.md section 4).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <vector>

namespace ofdis {

// Per-level geometry, mirrors camparam/optparam (oflow.h:16-76) + grid (patchgrid.cpp:42-48).
struct LevelGeom {
  int w, h, pad, tmp_w, tmp_h;
  int noc, nop, P, novals, steps, nopw, noph, np, offw, offh;
  int level, camlr;
  int pdl;                 // launch the level loop's kernels with programmatic dependent launch (see pdl_wait)
  int pitch;               // row pitch (floats) of the planar refinement planes, multiple of 4
  float lb, ubw, ubh, outlierthresh;
  // device pointers (frame 0); frame f adds f * stride
  const float* img[4];     // I0, I0x, I0y, I1 (padded, interleaved)
  size_t img_fs[4];        // floats between consecutive frames of each array (images and gradients live in two blocks)
  float* flow;             // [frames][h][w][nop]
  size_t flow_frame_stride;
  const float* flow_prev;  // level+1 flow (or initflow), nullptr -> zero init
  size_t flow_prev_frame_stride;
  float* pat_p;            // [frames][np][nop]
  float* pat_w;            // [frames][np][novals]
  int* pat_conv;           // [frames][np]
  int* pat_cnt;            // [frames][np]
  // Forward-backward consistency (usefbcon, oflow.cpp:162-170): internal frame q = 2*pair + dir,
  // dir 1 = the grid on the swapped images; the complementary frame of q is q ^ 1.
  int fb;                  // 1: frames come in (forward, backward) couples; stereo camlr = q & 1
  int fstep;               // frame step of a launch: frame = f0 + index * fstep (2 = forward frames only)
  int* fb_pos;             // [frames][np][2]  integer patch position after optimisation (patchgrid.cpp:308-309)
  float* fb_wbil;          // [frames][np][4]  bilinear weights of that position (:313-318)
  int* fb_reach;           // [frames]         max |position - reference| over the frame's patches
};

__host__ __device__ __forceinline__ int frame_of(const LevelGeom& g, int f0, int idx) { return f0 + idx * g.fstep; }
__host__ __device__ __forceinline__ int camlr_of(const LevelGeom& g, int frame) { return g.fb ? (frame & 1) : g.camlr; }

struct PatchParams {
  int max_iter, min_iter, costfct, patnorm;
  float dp_thresh_sq, dr_thresh, res_thresh;
};

// Refinement workspace for one level (all frames), planar planes of pitch*h floats.
struct VarRefPlanes {
  float* mask;             // [frames]
  float* avg;              // [frames][C]   0.5*(I1w+I0)            (setup only)
  float* deriv[8];         // Ix Iy Iz Ixx Ixy Iyy Ixz Iyz, each [frames][C]
  // Band-skewed ("anti-diagonal major") storage shared by assemble_kernel and sor_wave_kernel.  The
  // rows of a level are cut into `nb` bands of hpad*rt rows (one band per CTA of the SOR launch); a
  // band has `hpad` lanes (threads of one sweep; a power of two) of `rt` consecutive rows each
  // (1, 2 or 4).  Everything one lane needs for the 4-pixel blocks (rows rl*rt .. rl*rt+rt-1 of the
  // band, columns 4I..4I+3) of one super-step is ONE contiguous "lane row":
  //     [band c][d = I + rl][lane rl][ rt x (NQ record fields | du x4 | dv x4) float4, pad to odd ]
  // so that (a) the lanes that hold a block on diagonal d -- max(0, d-W4+1) .. min(d, lanes-1) --
  // are one contiguous piece of memory: the SOR's producer fetches exactly the occupied part of a
  // diagonal with one bulk copy (no bytes for the empty corners of the skew), and (b) with an odd
  // number of 16-byte words per lane row the lanes of a warp read any one field without a
  // shared-memory bank conflict.  (du,dv) live in the same lane row as the records (the last sweep
  // writes them in place).
  float4* rec;             // [frames][nb][ndiag][hpad][lpitch] float4
  size_t plane;            // pitch*h (natural planes)
  size_t rec_stride;       // float4 per frame
  int hpad;                // lanes per band (threads of one sweep)
  int rt, rtshift;         // rows per lane, log2
  int hbshift;             // log2(rows per band = hpad*rt)
  int nb;                  // bands
  int ndiag;               // diagonals stored per band: W4 + hpad + 2
  int nq;                  // record fields per block: 8 (flow) / 5 (stereo); chunk nq = du, nq+1 = dv
  int lpitch;              // float4 per lane row: rt*(nq+2), made odd
  // "Fast" refinement (ofdis_set_option "sor_fast", SURVEY 8f rank 4; NOT bit-exact, see DESIGN.md): red-black
  // SOR on natural-layout arrays -- records [frames][h][pitch][8] (a11^-1 a12^-1 a22^-1 b1 b2 sh sv -; stereo
  // A11 b1 sh sv), (du,dv) as two ping-pong buffers of two planes each [frames][2][2][h*pitch].
  // Lane mode (sor_lane_kernel.cuh; exact, levels of few 32-row bands): nb = bands of 32 rows, ndiag = lane_ndiag(w),
  // records [frames][nb][t = x/2 + (y & 31)][q = 2 (x & 1) + half][lane = y & 31] float4 (flow: a11^-1 a12^-1 a22^-1
  // b1 | b2 sh sv sv_top; stereo: A11 b1 sh sv | sv_top - - -), then (du,dv) of the two pixels of a block as one
  // float4 [frames][nb][t][lane] behind them.
  int lane;                // 1 = lane-skewed layout + sor_lane_kernel for this level
  int fast;                // 0 = exact lexicographic SOR (default)
  int fcur;                // ping-pong buffer that holds the current (du,dv)
  float* frec;
  float* fdu;
  size_t frec_stride, fdu_stride;  // floats per frame
};

__host__ __device__ __forceinline__ int sor_lane_pitch(int nop, int rt) { return (rt * ((nop == 2 ? 8 : 5) + 2)) | 1; }

// float4 index of chunk q (0..nq-1 record fields, nq = du, nq+1 = dv) of block (I, j)
__host__ __device__ __forceinline__ size_t band_f4(const VarRefPlanes& pl, int I, int j, int q) {
  const int jl = j & ((pl.hpad << pl.rtshift) - 1), rl = jl >> pl.rtshift, s = jl & (pl.rt - 1);
  return ((size_t)((j >> pl.hbshift) * pl.ndiag + I + rl) * pl.hpad + rl) * pl.lpitch + s * (pl.nq + 2) + q;
}

// lane mode: rows in bands of 32 (lane = y & 31), columns in blocks of two; block I of lane l sits at t = I + l.
// float4 index of record half `half` (0, 1) and FLOAT index of du (dv = +1) of pixel (x, y), relative to the
// frame's pl.rec; entries per band; float4 per frame
__host__ __device__ __forceinline__ int lane_ndiag(int w) { return ((w + 1) >> 1) + 48; }
__host__ __device__ __forceinline__ size_t lane_rec_f4(const VarRefPlanes& pl, int x, int y, int half) {
  const int l = y & 31;
  return ((size_t)((y >> 5) * pl.ndiag + (x >> 1) + l) * 4 + 2 * (x & 1) + half) * 32 + l;
}
__host__ __device__ __forceinline__ size_t lane_dudv_f(const VarRefPlanes& pl, int x, int y) {
  const int l = y & 31;
  return ((size_t)pl.nb * pl.ndiag * 128 + (size_t)((y >> 5) * pl.ndiag + (x >> 1) + l) * 32 + l) * 4 + 2 * (x & 1);
}
__host__ __device__ __forceinline__ size_t lane_frame_f4(int w, int h) { return (size_t)((h + 31) / 32) * lane_ndiag(w) * 160; }

// Band plan of a level for the SOR (sor_wave_kernel.cuh).  `rt` rows per lane (tiles of 4 columns x
// rt rows per thread and super-step: the wavefront needs W/4 + h/rt super-steps).  Levels of up to
// `single_max` lanes run in one CTA (hpad = lanes padded to 32/64/128); taller ones are cut into the
// smallest bands that still fit a cluster of `max_cluster` CTAs.  Returns false when the level is
// too tall.
bool sor_fits(int nop, int hpad, int rt, int K);  // threads and shared memory of one CTA with K sweeps in flight
inline bool sor_band_plan(int w, int h, int rt, int single_max, int max_cluster, int nop, int K, VarRefPlanes* pl) {
  const int lanes = (h + rt - 1) / rt;  // lanes the whole level needs
  int hpad = 0;
  // all K sweeps in flight if some band size allows it, else one sweep per launch (K launches per solve)
  for (int kk = K < 1 ? 1 : K; !hpad; kk = 1) {
    for (int p = 32; p <= 128 && !hpad; p *= 2)
      if (lanes <= p && lanes <= single_max && sor_fits(nop, p, rt, kk)) hpad = p;
    for (int p = 32; p <= 256 && !hpad; p *= 2)
      if ((lanes + p - 1) / p <= max_cluster && sor_fits(nop, p, rt, kk)) hpad = p;
    if (kk == 1) break;
  }
  if (!hpad) return false;
  pl->hpad = hpad;
  pl->rt = rt;
  pl->rtshift = rt == 1 ? 0 : (rt == 2 ? 1 : 2);
  pl->hbshift = (hpad == 32 ? 5 : (hpad == 64 ? 6 : (hpad == 128 ? 7 : 8))) + pl->rtshift;
  pl->nb = (lanes + hpad - 1) / hpad;
  pl->ndiag = (w + 3) / 4 + hpad + 2;
  pl->nq = nop == 2 ? 8 : 5;
  pl->lpitch = sor_lane_pitch(nop, rt);
  return true;
}

struct VarRefParams {
  float quarter_alpha, half_gamma_over3, half_delta_over3, omega;
  int n_inner, n_solver;
};

// Optional per-kernel-class CUDA-event timing (bench.py roofline; eager mode only).
enum KernelClass { KC_PATCH = 0, KC_DENSIFY, KC_VR_SETUP, KC_VR_ASSEMBLE, KC_VR_SOR, KC_COUNT };
struct Profiler {
  cudaStream_t st = nullptr;
  struct Rec { int cls, level; cudaEvent_t a, b; };
  int level = 0;  // pyramid level of the launches being recorded
  std::vector<Rec> recs;
  cudaEvent_t cur = nullptr;
  int cur_cls = -1;
  void begin(int cls) {
    cudaEventCreate(&cur);
    cudaEventRecord(cur, st);
    cur_cls = cls;
  }
  void end() {
    cudaEvent_t b;
    cudaEventCreate(&b);
    cudaEventRecord(b, st);
    recs.push_back({cur_cls, level, cur, b});
  }
};
struct ProfScope {
  Profiler* p;
  ProfScope(Profiler* prof, int cls) : p(prof) { if (p) p->begin(cls); }
  ~ProfScope() { if (p) p->end(); }
};

// launchers (each returns the number of kernels launched, <0 on error)
int launch_patch_optimize(const LevelGeom& g, const PatchParams& pp, int f0, int f1, bool init_from_coarser,
                          cudaStream_t st, Profiler* prof = nullptr);
int launch_densify(const LevelGeom& g, int f0, int f1, cudaStream_t st, Profiler* prof = nullptr);
// usefbcon: positions/weights of every patch (all frames of [f0,f1)), then the merged gather
int launch_fb_prepare(const LevelGeom& g, int f0, int f1, cudaStream_t st);
int launch_swap_images(const LevelGeom& g, int f0, int f1, cudaStream_t st);
// pyramid_kernels.cu -- callers either side of the hot path (SURVEY 8f rank 1, 2)
struct PyrSourceU8 {
  const unsigned char* frames;  // [frame][2][h_org][w_org][noc], device
  size_t image_bytes;           // h_org * w_org * noc
  int w_org, h_org, pad_left, pad_top;
};
int launch_sobel(const LevelGeom& g, int f0, int f1, cudaStream_t st);
int launch_pyr_from_u8(const LevelGeom& g, int f0, int f1, const PyrSourceU8& s, cudaStream_t st);
int launch_pyr_from_level(const LevelGeom& g, int f0, int f1, const float* stage, cudaStream_t st);
int launch_pyr_down(const LevelGeom& gs, const LevelGeom& gd, int f0, int f1, cudaStream_t st);
int launch_flow_upsample(const LevelGeom& g, int f0, int f1, float* out, int w_org, int h_org, int crop_x, int crop_y,
                         cudaStream_t st);
int launch_varref(const LevelGeom& g, const VarRefPlanes& pl, const VarRefParams& vp, int f0, int f1,
                  cudaStream_t st, Profiler* prof = nullptr);

// fast mode: does the red-black kernel's staged tile (32 + 4K pixels square) exceed an SM's shared memory?
bool rb_smem_limit_exceeded(int nop, int K);
// can sor_lane_kernel (pixel wavefront, one CTA per frame) take a level of h rows with K sweeps?
bool sor_lane_fits(int h, int K);
bool sor_lane_preferred(int h, int K);  // ... and is it the faster of the two exact kernels there?
// largest thread-block cluster the SOR kernel can be launched with on the current device (8 or 16)
int sor_max_cluster_size();

// ---- programmatic dependent launch (PDL) ---------------------------------------
// Every kernel starts with pdl_wait(): a kernel launched with the programmatic-stream-serialization attribute may be
// scheduled while its predecessor in the stream still runs (its launch latency and CTA start-up overlap the
// predecessor's tail); griddepcontrol.wait then blocks until the predecessor has completed and its memory
// operations are visible, griddepcontrol.launch_dependents lets this kernel's own successor be scheduled as soon
// as all of this kernel's CTAs have started.  Without the attribute both instructions do nothing.
#ifdef __CUDACC__
__device__ __forceinline__ void pdl_wait() {
  asm volatile("griddepcontrol.wait;\n\tgriddepcontrol.launch_dependents;" ::: "memory");
}
// launch with or without the attribute (g.pdl, set per context: ofdis_set_option "pdl")
template <typename... KP, typename... A>
static inline cudaError_t launch_k(bool pdl, void (*kern)(KP...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, A... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = pdl ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kern, static_cast<KP>(args)...);
}
#endif

// ---- exact-arithmetic helpers -------------------------------------------------
// std::min/std::max semantics of the reference (operand order matters for +-0/NaN)
__device__ __forceinline__ float std_min(float a, float b) { return (b < a) ? b : a; }
__device__ __forceinline__ float std_max(float a, float b) { return (a < b) ? b : a; }
__device__ __forceinline__ int clampi(int v, int n) { return v < 0 ? 0 : (v > n - 1 ? n - 1 : v); }

}  // namespace ofdis
