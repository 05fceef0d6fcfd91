/* ofdis_b200.h -- C-ABI of the B200-native DIS optical-flow hot path.
 *
 * This is the drop-in boundary (DESIGN.md section 1): plain C, plain pointers
 * and sizes, no C++/torch types.  Everything the reference's three classes do
 * on the hot path is reachable from here:
 *
 *   reference interface (file:line)                       -> entry point
 *   ------------------------------------------------------------------------
 *   OFC::OFClass::OFClass            oflow.h:84-111,        ofdis_create + ofdis_upload_* +
 *                                    oflow.cpp:32-363        ofdis_run + ofdis_get_flow
 *   PatGridClass::InitializeGrid /   patchgrid.h:25-26,     ofdis_upload_level (binds I0,dI0,I1 of a level)
 *     SetTargetImage                 patchgrid.cpp:98-132
 *   PatGridClass::InitializeFromCoarserOF  patchgrid.cpp:195-211   ofdis_set_flow(level+1) / implicit in ofdis_run
 *   PatGridClass::Optimize           patchgrid.cpp:134-141  ofdis_patgrid_optimize
 *     (PatClass::InitializePatch, OptimizeIter  patch.cpp:57-88,119-212 -- fused into the same kernel)
 *   PatGridClass::AggregateFlowDense patchgrid.cpp:213-397  ofdis_patgrid_aggregate
 *   PatGridClass::SetComplGrid       patchgrid.h:36 + oflow.cpp:162-170   ofdis_params.usefbcon = 1 (both grids of a pair
 *                                                            live in the context; ofdis_upload_level_fb,
 *                                                            ofdis_set_direction)
 *   PatGridClass::GetQuePatchDis &c  patchgrid.h:42-44      ofdis_get_patches
 *   VarRefClass::VarRefClass         refine_variational.h:37-39,    ofdis_varref_refine
 *                                    refine_variational.cpp:25-116
 *     (image_warp, get_derivatives, compute_smoothness, compute_data[_DE],
 *      sub_laplacian, sor_coupled / sor_coupled_slow_but_readable_DE;
 *      FDF1.0.1/opticalflow_aux.c:17-548, solver.c:77-466 -- device kernels)
 *
 * Unlike the reference (no status, exit(1) on OOM, image.c:17-28) every call
 * returns an int status and never exits.  A context is bound to one CUDA
 * device and one stream; all work is asynchronous on that stream unless the
 * call copies to pageable host memory.  `frames` is the batch dimension that
 * sits BELOW the reference API: one context processes frame pairs
 * [0, max_frames) per launch.
 *
 * Arithmetic contract: IEEE binary32, no FMA contraction, expression order of
 * the reference, so results are bitwise equal to the reference CPU build on
 * the same inputs (tests/test_gpu_parity.py).
 */
#ifndef OFDIS_B200_H
#define OFDIS_B200_H

#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct ofdis_ctx ofdis_ctx;

/* The 21 run-time scalars of OFClass's constructor (oflow.h:93-111), CLI
 * semantics of run_dense.cpp:225-294.  dp_thresh is the un-squared CLI value. */
typedef struct ofdis_params {
  int sc_f, sc_l;          /* first (coarsest) / last (finest) pyramid level */
  int max_iter, min_iter;  /* Gauss-Newton iterations per patch */
  float dp_thresh, dr_thresh, res_thresh;
  int p_samp_s;            /* patch edge length P (even, P*P*noc % 4 == 0) */
  float patove;            /* patch overlap in [0,1) */
  int usefbcon;            /* forward-backward merge (oflow.cpp:162-170, patchgrid.cpp:278-375): doubles the patch work */
  int costfct;             /* 0 L2, 1 L1, 2 pseudo-Huber */
  int noc;                 /* image channels: 1 or 3 */
  int patnorm;             /* mean-normalise patches */
  int usetvref;            /* run the variational refinement */
  float tv_alpha, tv_gamma, tv_delta;
  int tv_innerit, tv_solverit;
  float tv_sor;
  int verbosity;
} ofdis_params;

enum {
  OFDIS_OK = 0,
  OFDIS_ERR_ARG = -1,         /* bad argument / unsupported geometry */
  OFDIS_ERR_CUDA = -2,        /* a CUDA call failed; see ofdis_last_error */
  OFDIS_ERR_UNSUPPORTED = -3, /* valid in the reference but not built here (refinement levels taller than ~256 rows x the largest thread-block cluster -- the SOR's shared-memory ring bounds the rows of one band --, i.e. 2048 rows, 4096 where the device grants 16-CTA clusters; ofdis_upload_packed with usefbcon) */
  OFDIS_ERR_NOMEM = -4
};
enum { OFDIS_MEM_HOST = 0, OFDIS_MEM_DEVICE = 1 };

/* nop: 2 = optical flow (run_OF_*), 1 = stereo disparity (run_DE_*).
 * width/height: level-0 size, divisible by 2^sc_f (oflow.h:87).  imgpadding:
 * border of every level image (run_dense.cpp:343 passes the patch size).
 * stream: a cudaStream_t to enqueue on, or NULL for a private stream. */
int ofdis_create(ofdis_ctx** out, int device, void* stream, const ofdis_params* prm, int nop,
                 int width, int height, int imgpadding, int max_frames);
int ofdis_destroy(ofdis_ctx* ctx);
const char* ofdis_last_error(const ofdis_ctx* ctx);
const char* ofdis_version(void);

/* camparam::camlr (oflow.h:28; 0 = left/forward grid clamps disparity <= 0, 1 = right/backward
 * clamps >= 0, patch.cpp:188-193, refine_variational.cpp:299-314).  Default 0, as OFClass's
 * forward grid uses.  Only meaningful for nop == 1; with usefbcon the forward grid is 0 and the
 * backward grid 1 whatever is set here. */
int ofdis_set_camlr(ofdis_ctx* ctx, int camlr);
/* optparam::dp_thresh is stored SQUARED by OFClass (oflow.cpp:88); callers that already hold
 * the squared value (PatGridClass built from an optparam) set it here bit-exactly. */
int ofdis_set_dp_thresh_sq(ofdis_ctx* ctx, float dp_thresh_sq);

/* level geometry (oflow.cpp:142-151, patchgrid.cpp:42-48) */
int ofdis_level_info(const ofdis_ctx* ctx, int level, int* w, int* h, int* nopw, int* noph, int* steps);

/* Images of one level of one frame pair: padded, row-major, channel-interleaved
 * float32, (h+2*pad) x (w+2*pad) x noc, exactly what OFClass receives
 * (oflow.h:84-86).  The gradients of I1 are only read by the forward-backward grid
 * (oflow.cpp:193-197); without usefbcon they are not needed (ofdis_upload_level_fb otherwise). */
int ofdis_upload_level(ofdis_ctx* ctx, int frame, int level, const float* i0, const float* i0x,
                       const float* i0y, const float* i1, int memkind);

/* Like ofdis_upload_level plus the gradients of the second image (im_bo_dx, im_bo_dy of oflow.h:84-86),
 * which the forward-backward grid needs as its template gradients (oflow.cpp:193-197).  Required when the
 * context was created with usefbcon = 1; i1x, i1y may be NULL otherwise. */
int ofdis_upload_level_fb(ofdis_ctx* ctx, int frame, int level, const float* i0, const float* i0x,
                          const float* i0y, const float* i1, const float* i1x, const float* i1y, int memkind);

/* Packed transfer: all levels sc_f..sc_l of frames [f0,f1) in the context's own
 * layout (per frame: I0,I1 of levels sc_f..sc_l, then I0x,I0y of the same levels; use
 * ofdis_packed_offset), one copy.  Not available with usefbcon (a packed frame has no gradients of
 * the second image: OFDIS_ERR_UNSUPPORTED); the image-only transfers below are. */
size_t ofdis_packed_frame_floats(const ofdis_ctx* ctx);
size_t ofdis_packed_offset(const ofdis_ctx* ctx, int level, int which /*0 I0,1 I0x,2 I0y,3 I1*/);
int ofdis_upload_packed(ofdis_ctx* ctx, int f0, int f1, const float* packed, int memkind);

/* Images-only transfer (extension, SURVEY 8f rank 1): the leading ofdis_packed_images_frame_floats()
 * floats of a packed frame are I0,I1 of all levels (offsets as ofdis_packed_offset reports them);
 * `packed` holds only those, frame after frame.  One 2-D copy, then the gradients of I0 are derived
 * on the device (Sobel 3x3 / 8, reflect101, zero border: run_dense.cpp:156-157,171-172). */
size_t ofdis_packed_images_frame_floats(const ofdis_ctx* ctx);
int ofdis_upload_packed_images(ofdis_ctx* ctx, int f0, int f1, const float* packed, int memkind);

/* Read-back of one padded array of the device pyramid (which: 0 I0, 1 I0x, 2 I0y, 3 I1); the
 * inverse of ofdis_upload_level, used to check the device-built pyramids. */
int ofdis_get_level(ofdis_ctx* ctx, int frame, int level, int which, float* dst, int memkind);

/* Pyramid on the device (extension, SURVEY 8f rank 1 == ConstructImgPyramide, run_dense.cpp:130-178
 * plus the divisibility padding of run_dense.cpp:298-311).
 * ofdis_upload_frames_u8: `frames` = [frame][2][height_org][width_org][noc] 8-bit pixels (I0 then I1
 *   of each pair); width_org/height_org must pad up to the context's width/height.  Builds levels
 *   sc_l..sc_f of I0, I1 (box means), I0x, I0y (Sobel/8) and both paddings on the device.
 * ofdis_upload_finest_level: `packed` = [frame][2][h][w][noc] float images of level sc_l WITHOUT
 *   the border padding (h = height >> sc_l, ...; ofdis_finest_level_frame_floats() per frame);
 *   coarser levels, gradients and paddings are derived on the device.  Smallest transfer that still
 *   defines the run's input exactly. */
int ofdis_upload_frames_u8(ofdis_ctx* ctx, int f0, int f1, const unsigned char* frames, int width_org, int height_org,
                           int memkind);
size_t ofdis_finest_level_frame_floats(const ofdis_ctx* ctx);
int ofdis_upload_finest_level(ofdis_ctx* ctx, int f0, int f1, const float* packed, int memkind);

/* Output stage on the device (extension, SURVEY 8f rank 2 == run_dense.cpp:407-414): flow of level
 * sc_l times 2^sc_l, bilinear upsampling by 2^sc_l (half-pixel centres, edge clamped), crop of the
 * divisibility padding.  `out` = [f1-f0][height_org][width_org][nop] floats. */
int ofdis_get_flow_fullres(ofdis_ctx* ctx, int f0, int f1, float* out, int width_org, int height_org, int memkind);

/* Stage operators on frames [f0,f1) of one level. */
int ofdis_patgrid_optimize(ofdis_ctx* ctx, int level, int f0, int f1, int init_from_coarser);
int ofdis_patgrid_aggregate(ofdis_ctx* ctx, int level, int f0, int f1);
int ofdis_varref_refine(ofdis_ctx* ctx, int level, int f0, int f1);

/* Whole coarse-to-fine run on frames [0,nframes): == OFClass ctor per frame.
 * use_initflow != 0 takes the flow stored at level sc_f+1 (ofdis_set_flow) as
 * the reference's `initflow` argument. */
int ofdis_run(ofdis_ctx* ctx, int nframes, int use_initflow);
int ofdis_sync(ofdis_ctx* ctx);

/* Dense flow of a level, (h x w x nop) interleaved float32.  Levels sc_l..sc_f+1
 * are addressable (sc_f+1 only as initflow). */
int ofdis_get_flow(ofdis_ctx* ctx, int frame, int level, float* dst, int memkind);
int ofdis_set_flow(ofdis_ctx* ctx, int frame, int level, const float* src, int memkind);
/* Final flow (level sc_l) of frames [f0,f1), contiguous, one copy. */
int ofdis_get_flow_batch(ofdis_ctx* ctx, int f0, int f1, float* dst, int memkind);

/* Per-patch results of the last ofdis_patgrid_optimize on `level` (any pointer may be
 * NULL): p[np*nop] displacement, pweight[np*novals] abs. residual, conv[np], cnt[np]. */
int ofdis_get_patches(ofdis_ctx* ctx, int frame, int level, float* p, float* pweight, int* conv,
                      int* cnt);

/* Test hook: raw internal planes of the last ofdis_varref_refine / debug run.
 * name in {"Ix","Iy","Iz","Ixx","Ixy","Iyy","Ixz","Iyz","mask","rec","dudv"};
 * returns the number of floats written (or a negative status). */
long ofdis_debug_get(ofdis_ctx* ctx, const char* name, int frame, float* dst, size_t max_floats);
/* Test hook: run only the first n_inner inner iterations of the refinement. */
int ofdis_debug_varref_iters(ofdis_ctx* ctx, int level, int f0, int f1, int n_inner);

/* Number of kernels this library has launched on the context since creation. */
long ofdis_launch_count(const ofdis_ctx* ctx);
/* Eager ofdis_run x steps with a CUDA-event pair around every launch group; sums per class
 * {0 patch, 1 densify, 2 refinement setup (warp+derivatives), 3 assemble, 4 SOR} into
 * ms_by_class[5] / launches_by_class[5] (launch groups, one per stage call). */
int ofdis_profile_run(ofdis_ctx* ctx, int nframes, int steps, double* ms_by_class, long* launches_by_class);
/* The same, additionally split by pyramid level: ms_by_level_class[(level - sc_l) * 5 + class] (may be NULL). */
int ofdis_profile_levels(ofdis_ctx* ctx, int nframes, int steps, double* ms_by_class, long* launches_by_class,
                         double* ms_by_level_class);
/* usefbcon contexts only: address ONE grid of every pair (0 = forward, 1 = the grid on the swapped images)
 * in the following ofdis_patgrid_optimize / ofdis_patgrid_aggregate (one frame per call) / ofdis_set_flow /
 * ofdis_get_flow / ofdis_get_patches calls; -1 (default) restores "both grids; flows and patches of the
 * forward one".  This is what two stand-alone PatGridClass objects joined by SetComplGrid
 * (patchgrid.h:36, oflow.cpp:162-170) are built on. */
int ofdis_set_direction(ofdis_ctx* ctx, int dir);
/* Options.  "sor_fast" 0 (default) | 1 switches the refinement's solver from the reference's lexicographic SOR to a
 *   red-black SOR (same system, omega and sweep count; SURVEY 8f rank 4): NOT bit-identical to the reference --
 *   the flow differs by a few hundredths of a pixel (bench.py reports the delta) -- and never covered by the parity
 *   claim.  All other options are launch geometry (tuning / test hook), results are bit-identical under every setting:
 *   "sor_lane"        2 (default) | 1 | 0: refinement levels of few 32-row bands (bands x sweeps <= 12 warps within the
 *                     shared memory of an SM; more sweeps than fit run in several launches) run the SOR as a wavefront of
 *                     two-pixel blocks whose warps synchronise through shared-memory flags instead of a CTA barrier
 *                     (sor_lane_kernel.cuh): 1 always, 0 never (the block wavefront of sor_wave_kernel everywhere),
 *                     2 for launches of up to 16 frames on levels of up to 64 rows -- there it is 10-20 % faster per
 *                     launch; it holds one CTA per SM at 56-row levels, which costs throughput when several streams of
 *                     large batches overlap, and every further band of rows adds start-up skew
 *   "pdl"             2 (default) | 1 | 0: programmatic dependent launch of the level loop's kernels (every kernel starts
 *                     with griddepcontrol.wait, so the next kernel's launch overlaps the tail of the current one):
 *                     1 always, 0 never, 2 for launches of up to 16 frames (2-5 % of the step there; larger batches lose)
 *   "sor_rows_per_thread" 1 (default for flow) | 2 (default for stereo) | 4: rows of the 4-column tile one SOR thread updates per super-step
 *                     (a level needs W/4 + h/rows super-steps; sor_wave_kernel.cuh)
 *   "sor_single_max"  32 | 64 | 128 (default): refinement levels of up to this many SOR lanes (= rows / rows per
 *                     thread) run their SOR in one CTA, taller ones in a thread-block cluster of row bands
 *   "sor_max_cluster" 8 (portable) | 16 (default where the device grants it) */
int ofdis_set_option(ofdis_ctx* ctx, const char* name, int value);
/* CUDA-graph replay of ofdis_run (captured on first use per nframes). */
int ofdis_set_graph_mode(ofdis_ctx* ctx, int enabled);

#ifdef __cplusplus
}
#endif
#endif
