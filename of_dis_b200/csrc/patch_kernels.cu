// Patch stage of the DIS hot path on sm_100a: K1 (template + Hessian), K2 (init
// from the coarser flow), K3 (inverse-compositional Gauss-Newton iterations)
// fused in one kernel, and K4 (densification) as a deterministic gather.
//
// Reference: PatClass / PatGridClass (patch.cpp:57-402, patchgrid.cpp:98-397).
//
// Mapping.  The reference reduces every P*P*C-vector with 8 strided partial
// sums (element e goes to partial e mod 8, added in increasing e) that are then
// folded 8 -> 4 -> 2 -> 1 (oracle/eigen_shim/Eigen/Core).  To be bit-identical
// the kernel gives one patch to a group of 8 lanes: lane l owns the elements
// e = l, l+8, l+16, ... and the fold is three xor-shuffles (4, 2, 1).  Four
// patches share a warp; a CTA of 256 threads holds 32 patches.  The template,
// its gradients and the residual of each lane live in shared memory as
// [slot][thread] columns (conflict free, private to the thread), staged once.
// The bilinear taps of I1 are plain LDGs: the (P+1)x(P+1) window of a patch
// moves by a fraction of a pixel per iteration and stays L1-resident.
#include "ofdis_internal.cuh"

namespace ofdis {

namespace {

constexpr unsigned FULL = 0xffffffffu;

// fold of the 8 partial sums of one patch (lanes l..l+7 of an aligned group)
__device__ __forceinline__ float fold8(float acc, float tailv, bool has_strided, bool has_tail) {
  float s;
  const float other = __shfl_xor_sync(FULL, acc, 4);
  if (has_strided) {
    s = acc + other;
    if (has_tail) s = s + tailv;
  } else {
    s = tailv;
  }
  const float t = s + __shfl_xor_sync(FULL, s, 2);
  return t + __shfl_xor_sync(FULL, t, 1);
}

template <int NOP>
__global__ void __launch_bounds__(256) patch_optimize_kernel(LevelGeom g, PatchParams pp, int f0,
                                                              int init_from_coarser) {
  pdl_wait();  // programmatic dependent launch: nothing of the previous kernel is touched before this
  extern __shared__ float smem[];
  const int tid = threadIdx.x, nthr = blockDim.x;
  const int l8 = tid & 7;
  const int frame = f0 + blockIdx.y;
  const int ip = blockIdx.x * (nthr >> 3) + (tid >> 3);
  const bool valid = ip < g.np;

  const int P = g.P, C = g.noc, n = g.novals;
  const int n8 = (n >> 3) << 3, nk = n8 >> 3;
  const bool has_tail = (n - n8) >= 4, has_strided = nk > 0;
  const int NK = nk + (has_tail ? 1 : 0);
  const float fn = (float)n;

  float* sT = smem + tid;
  float* sGx = sT + NK * nthr;
  float* sGy = sGx + NK * nthr;
  float* sD = sGy + NK * nthr;
  int* sOff = reinterpret_cast<int*>(sD + NK * nthr);
  const int rowC = g.tmp_w * C;

  const float* i0 = g.img[0] + (size_t)frame * g.img_fs[0];
  const float* i0x = g.img[1] + (size_t)frame * g.img_fs[1];
  const float* i0y = g.img[2] + (size_t)frame * g.img_fs[2];
  const float* i1 = g.img[3] + (size_t)frame * g.img_fs[3];

  // ---- patch geometry (patchgrid.cpp:62-69) ---------------------------------
  const int ipc = valid ? ip : 0;
  const int gx_i = ipc / g.noph, gy_i = ipc - gx_i * g.noph;
  const int cxi = gx_i * g.steps + g.offw, cyi = gy_i * g.steps + g.offh;
  const float refx = (float)cxi, refy = (float)cyi;

  // ---- K1: template, gradients, mean normalisation (patch.cpp:287-332) ------
  {
    const int base = ((cxi + g.pad - P / 2) + (cyi + g.pad - P / 2) * g.tmp_w) * C;
    float acc = 0.f, tailv = 0.f;
    for (int k = 0; k < NK; ++k) {
      const int e = (k < nk) ? (l8 + 8 * k) : (n8 + (l8 & 3));
      const int y = e / (P * C), rem = e - y * (P * C), x = rem / C, c = rem - x * C;
      const int off = y * rowC + x * C + c;
      sOff[k * nthr] = off;
      const float t = i0[base + off];
      sT[k * nthr] = t;
      sGx[k * nthr] = i0x[base + off];
      sGy[k * nthr] = i0y[base + off];
      if (k < nk) acc = (k == 0) ? t : acc + t;
      else tailv = t;
    }
    if (pp.patnorm > 0) {
      const float m = fold8(acc, tailv, has_strided, has_tail) / fn;
      for (int k = 0; k < NK; ++k) sT[k * nthr] = sT[k * nthr] - m;
    }
  }

  // ---- Hessian and its Cholesky factor (patch.cpp:71-88, Eigen LLT) ---------
  float L00, L10 = 0.f, L11 = 0.f;
  {
    float axx = 0.f, axy = 0.f, ayy = 0.f, txx = 0.f, txy = 0.f, tyy = 0.f;
    for (int k = 0; k < NK; ++k) {
      const float a = sGx[k * nthr], b = sGy[k * nthr];
      const float vxx = a * a, vxy = a * b, vyy = b * b;
      if (k < nk) {
        axx = (k == 0) ? vxx : axx + vxx;
        axy = (k == 0) ? vxy : axy + vxy;
        ayy = (k == 0) ? vyy : ayy + vyy;
      } else {
        txx = vxx; txy = vxy; tyy = vyy;
      }
    }
    float H00 = fold8(axx, txx, has_strided, has_tail);
    if (NOP == 2) {
      const float H01 = fold8(axy, txy, has_strided, has_tail);
      float H11 = fold8(ayy, tyy, has_strided, has_tail);
      if (H00 * H11 - H01 * H01 == 0.f) {
        H00 = (float)((double)H00 + 1e-10);
        H11 = (float)((double)H11 + 1e-10);
      }
      L00 = H00; L10 = H01; L11 = H11;
      if (H00 > 0.f) {
        L00 = sqrtf(H00);
        L10 = H01 / L00;
        const float x = H11 - L10 * L10;
        if (x > 0.f) L11 = sqrtf(x);
      }
    } else {
      if (H00 == 0.f) H00 = (float)((double)H00 + 1e-10);
      L00 = H00 > 0.f ? sqrtf(H00) : H00;
    }
  }

  // ---- K2: start value (patchgrid.cpp:195-211) ------------------------------
  float pin0 = 0.f, pin1 = 0.f;
  if (init_from_coarser && g.flow_prev != nullptr) {
    const float* fp = g.flow_prev + (size_t)frame * g.flow_prev_frame_stride;
    const int i = (cyi >> 1) * (g.w / 2) + (cxi >> 1);
    if (NOP == 2) {
      const float2 v = reinterpret_cast<const float2*>(fp)[i];
      pin0 = v.x * 2.f;
      pin1 = v.y * 2.f;
    } else {
      pin0 = fp[i] * 2.f;
    }
  }

  // ---- K3: OptimizeStart / OptimizeIter (patch.cpp:119-212, 264-284) --------
  float p0 = pin0, p1 = pin1, dp0 = 0.f, dp1 = 0.f;
  float ptx = refx + p0, pty = (NOP == 2) ? refy + p1 : refy;
  const float stx = ptx, sty = pty;
  float dpsq_init = 1e-10f, mares = 1e5f, mares_old = 1e20f;
  int cnt = 0, conv = 0;
  bool wrote_w = false;   // whether the residual column holds a valid error image
  bool finishing = false; // reset happened: one last error image, no test
  bool active = valid;
  if (active && (ptx < g.lb || pty < g.lb || ptx > g.ubw || pty > g.ubh)) {
    conv = 1;  // patch.cpp:135-141 (pweight stays zero-initialised)
    active = false;
  }

  while (__any_sync(FULL, active)) {
    // -- error image at (ptx, pty): getPatchStaticBil + LossComputeErrorImage --
    float b0 = 0.f, b1 = 0.f, sw = 0.f, tb0 = 0.f, tb1 = 0.f, tsw = 0.f;
    {
      float acc = 0.f, tailv = 0.f;
      int base = 0;
      float w0 = 0.f, w1 = 0.f, w2 = 0.f, w3 = 0.f;
      if (active) {
        const int pcx = (int)ceilf(ptx + .00001f), pcy = (int)ceilf(pty + .00001f);
        const int pfx = (int)floorf(ptx), pfy = (int)floorf(pty);
        const float rx = ptx - (float)pfx, ry = pty - (float)pfy;
        w0 = rx * ry;
        w1 = (1.f - rx) * ry;
        w2 = rx * (1.f - ry);
        w3 = (1.f - rx) * (1.f - ry);
        base = ((pcx + g.pad - P / 2) + (pcy + g.pad - P / 2) * g.tmp_w) * C;
        for (int k = 0; k < NK; ++k) {
          const float* a = i1 + base + sOff[k * nthr];
          const float v = w0 * __ldg(a) + w1 * __ldg(a - C) + w2 * __ldg(a - rowC) + w3 * __ldg(a - rowC - C);
          sD[k * nthr] = v;
          if (k < nk) acc = (k == 0) ? v : acc + v;
          else tailv = v;
        }
      }
      float m = 0.f;
      if (pp.patnorm > 0) m = fold8(acc, tailv, has_strided, has_tail) / fn;
      if (active) {
        for (int k = 0; k < NK; ++k) {
          float d = sD[k * nthr];
          if (pp.patnorm > 0) d = d - m;
          float r, w;
          if (pp.costfct == 0) {
            r = d - sT[k * nthr];
            w = fabsf(r);
          } else if (pp.costfct == 1) {
            const float t = d - sT[k * nthr];
            r = copysignf(sqrtf(fabsf(t)), t);
            w = fabsf(r);
          } else if (pp.costfct == 2) {
            const float t = d - sT[k * nthr];
            const float hh = sqrtf((sqrtf(1.0f + (t * t) / 25.0f) - 1.0f) * 50.0f);
            r = copysignf(hh, t);
            w = fabsf(r);
          } else {  // reference leaves pdiff/pweight untouched (patch.cpp:230-261)
            r = d;
            w = 0.f;
          }
          sD[k * nthr] = r;
          const float vx = sGx[k * nthr] * r, vy = sGy[k * nthr] * r;
          if (k < nk) {
            b0 = (k == 0) ? vx : b0 + vx;
            b1 = (k == 0) ? vy : b1 + vy;
            sw = (k == 0) ? w : sw + w;
          } else {
            tb0 = vx; tb1 = vy; tsw = w;
          }
        }
        wrote_w = (pp.costfct >= 0 && pp.costfct <= 2);
      }
    }
    b0 = fold8(b0, tb0, has_strided, has_tail);
    if (NOP == 2) b1 = fold8(b1, tb1, has_strided, has_tail);
    sw = fold8(sw, tsw, has_strided, has_tail);

    if (active) {
      if (finishing) {
        active = false;
      } else {
        // OptimizeComputeErrImg tail (patch.cpp:272-282)
        const float dpsq = (NOP == 2) ? dp0 * dp0 + dp1 * dp1 : dp0 * dp0;
        if (cnt == 1) dpsq_init = dpsq;
        mares_old = mares;
        mares = sw / fn;
        // the two ratio tests only count once min_iter is reached: skip their divisions before
        bool go = (cnt < pp.max_iter) & (mares > pp.res_thresh);
        if (go && cnt >= pp.min_iter)
          go = (dpsq / dpsq_init >= pp.dp_thresh_sq) & (mares / mares_old <= pp.dr_thresh);
        if (!go) {
          conv = 1;
          active = false;
        } else {
          // one Gauss-Newton step (patch.cpp:174-208)
          cnt++;
          if (NOP == 2) {
            const float y0 = b0 / L00;
            const float y1 = (b1 - L10 * y0) / L11;
            dp1 = y1 / L11;
            dp0 = (y0 - L10 * dp1) / L00;
            p0 = p0 - dp0;
            p1 = p1 - dp1;
            ptx = refx + p0;
            pty = refy + p1;
          } else {
            dp0 = (b0 / L00) / L00;
            p0 = p0 - dp0;
            p0 = (camlr_of(g, frame) == 0) ? std_min(p0, 0.0f) : std_max(p0, 0.0f);
            ptx = refx + p0;
          }
          const float ex = stx - ptx, ey = sty - pty;
          if (sqrtf(ex * ex + ey * ey) > g.outlierthresh || ptx < g.lb || pty < g.lb || ptx > g.ubw ||
              pty > g.ubh) {
            p0 = pin0;
            p1 = pin1;
            ptx = refx + p0;
            if (NOP == 2) pty = refy + p1;
            conv = 1;
            finishing = true;
          }
        }
      }
    }
  }

  if (valid) {
    float* pw = g.pat_w + ((size_t)frame * g.np + ip) * n;
    for (int k = 0; k < NK; ++k) {
      if (k < nk) pw[l8 + 8 * k] = wrote_w ? fabsf(sD[k * nthr]) : 0.f;
      else if (l8 < 4) pw[n8 + l8] = wrote_w ? fabsf(sD[k * nthr]) : 0.f;
    }
    if (l8 == 0) {
      float* po = g.pat_p + ((size_t)frame * g.np + ip) * NOP;
      po[0] = p0;
      if (NOP == 2) po[1] = p1;
      g.pat_conv[(size_t)frame * g.np + ip] = conv;
      g.pat_cnt[(size_t)frame * g.np + ip] = cnt;
    }
  }
}

// ---------------------------------------------------------------------------
// Specialisation for the common operating points 1/2 (P = 8, gray): the 8 lanes of a patch
// are its 8 columns, the 8 strided elements of a lane are the 8 rows of that column, so the
// template, its gradients and the residual live in 32 registers (no shared memory), and the
// bilinear taps of a lane are just two image columns of 9 rows (18 loads per iteration instead
// of 32, no per-element offsets).  Arithmetic and reduction order are those of the generic kernel.
template <int NOP>
__global__ void __launch_bounds__(256) patch_p8c1_kernel(LevelGeom g, PatchParams pp, int f0,
                                                          int init_from_coarser) {
  pdl_wait();  // programmatic dependent launch: nothing of the previous kernel is touched before this
  const int tid = threadIdx.x;
  const int l8 = tid & 7;
  const int frame = f0 + blockIdx.y;
  const int ip = blockIdx.x * (blockDim.x >> 3) + (tid >> 3);
  const bool valid = ip < g.np;
  constexpr int P = 8;
  const float fn = 64.0f;
  const int tw = g.tmp_w;
  const float* i0 = g.img[0] + (size_t)frame * g.img_fs[0];
  const float* i0x = g.img[1] + (size_t)frame * g.img_fs[1];
  const float* i0y = g.img[2] + (size_t)frame * g.img_fs[2];
  const float* i1 = g.img[3] + (size_t)frame * g.img_fs[3];

  const int ipc = valid ? ip : 0;
  const int gx_i = ipc / g.noph, gy_i = ipc - gx_i * g.noph;
  const int cxi = gx_i * g.steps + g.offw, cyi = gy_i * g.steps + g.offh;
  const float refx = (float)cxi, refy = (float)cyi;

  // K1: column l8 of the template and its gradients (patch.cpp:287-332)
  float T[8], GX[8], GY[8], R[8];
  {
    const int base = (cxi + g.pad - P / 2 + l8) + (cyi + g.pad - P / 2) * tw;
    float acc = 0.f;
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      T[k] = i0[base + k * tw];
      GX[k] = i0x[base + k * tw];
      GY[k] = i0y[base + k * tw];
      acc = (k == 0) ? T[k] : acc + T[k];
      R[k] = 0.f;
    }
    if (pp.patnorm > 0) {
      const float m = fold8(acc, 0.f, true, false) / fn;
#pragma unroll
      for (int k = 0; k < 8; ++k) T[k] = T[k] - m;
    }
  }
  // Hessian + Cholesky (patch.cpp:71-88)
  float L00, L10 = 0.f, L11 = 0.f;
  {
    float axx = 0.f, axy = 0.f, ayy = 0.f;
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      const float vxx = GX[k] * GX[k], vxy = GX[k] * GY[k], vyy = GY[k] * GY[k];
      axx = (k == 0) ? vxx : axx + vxx;
      axy = (k == 0) ? vxy : axy + vxy;
      ayy = (k == 0) ? vyy : ayy + vyy;
    }
    float H00 = fold8(axx, 0.f, true, false);
    if (NOP == 2) {
      const float H01 = fold8(axy, 0.f, true, false);
      float H11 = fold8(ayy, 0.f, true, false);
      if (H00 * H11 - H01 * H01 == 0.f) {
        H00 = (float)((double)H00 + 1e-10);
        H11 = (float)((double)H11 + 1e-10);
      }
      L00 = H00; L10 = H01; L11 = H11;
      if (H00 > 0.f) {
        L00 = sqrtf(H00);
        L10 = H01 / L00;
        const float x = H11 - L10 * L10;
        if (x > 0.f) L11 = sqrtf(x);
      }
    } else {
      if (H00 == 0.f) H00 = (float)((double)H00 + 1e-10);
      L00 = H00 > 0.f ? sqrtf(H00) : H00;
    }
  }
  // K2 (patchgrid.cpp:195-211)
  float pin0 = 0.f, pin1 = 0.f;
  if (init_from_coarser && g.flow_prev != nullptr) {
    const float* fp = g.flow_prev + (size_t)frame * g.flow_prev_frame_stride;
    const int i = (cyi >> 1) * (g.w / 2) + (cxi >> 1);
    if (NOP == 2) {
      const float2 v = reinterpret_cast<const float2*>(fp)[i];
      pin0 = v.x * 2.f;
      pin1 = v.y * 2.f;
    } else {
      pin0 = fp[i] * 2.f;
    }
  }
  // K3 (patch.cpp:119-212, 264-284)
  float p0 = pin0, p1 = pin1, dp0 = 0.f, dp1 = 0.f;
  float ptx = refx + p0, pty = (NOP == 2) ? refy + p1 : refy;
  const float stx = ptx, sty = pty;
  float dpsq_init = 1e-10f, mares = 1e5f, mares_old = 1e20f;
  int cnt = 0, conv = 0;
  bool wrote_w = false, finishing = false, active = valid;
  if (active && (ptx < g.lb || pty < g.lb || ptx > g.ubw || pty > g.ubh)) {
    conv = 1;
    active = false;
  }
  while (__any_sync(FULL, active)) {
    float b0 = 0.f, b1 = 0.f, sw = 0.f;
    {
      float V[8];
      float acc = 0.f;
      if (active) {
        const int pcx = (int)ceilf(ptx + .00001f), pcy = (int)ceilf(pty + .00001f);
        const int pfx = (int)floorf(ptx), pfy = (int)floorf(pty);
        const float rx = ptx - (float)pfx, ry = pty - (float)pfy;
        const float w0 = rx * ry, w1 = (1.f - rx) * ry, w2 = rx * (1.f - ry), w3 = (1.f - rx) * (1.f - ry);
        // window rows pcy-5 .. pcy+3, columns (pcx-5+l8) and (pcx-4+l8): d/c above, b/a below
        const float* q0 = i1 + (pcx + g.pad - P / 2 - 1 + l8) + (pcy + g.pad - P / 2 - 1) * tw;
        float cl = __ldg(q0), cr = __ldg(q0 + 1);  // row above: d, c
#pragma unroll
        for (int k = 0; k < 8; ++k) {
          const float* q = q0 + (k + 1) * tw;  // one IMAD.WIDE per row instead of a 64-bit add chain
          const float bl = __ldg(q), br = __ldg(q + 1);  // this row: b, a
          V[k] = w0 * br + w1 * bl + w2 * cr + w3 * cl;
          acc = (k == 0) ? V[k] : acc + V[k];
          cl = bl;
          cr = br;
        }
      } else {
#pragma unroll
        for (int k = 0; k < 8; ++k) V[k] = 0.f;
      }
      float m = 0.f;
      if (pp.patnorm > 0) m = fold8(acc, 0.f, true, false) / fn;
      if (active) {
#pragma unroll
        for (int k = 0; k < 8; ++k) {
          float d = V[k];
          if (pp.patnorm > 0) d = d - m;
          float r, w;
          if (pp.costfct == 0) {
            r = d - T[k];
            w = fabsf(r);
          } else if (pp.costfct == 1) {
            const float t = d - T[k];
            r = copysignf(sqrtf(fabsf(t)), t);
            w = fabsf(r);
          } else if (pp.costfct == 2) {
            const float t = d - T[k];
            const float hh = sqrtf((sqrtf(1.0f + (t * t) / 25.0f) - 1.0f) * 50.0f);
            r = copysignf(hh, t);
            w = fabsf(r);
          } else {
            r = d;
            w = 0.f;
          }
          R[k] = r;
          const float vx = GX[k] * r, vy = GY[k] * r;
          b0 = (k == 0) ? vx : b0 + vx;
          b1 = (k == 0) ? vy : b1 + vy;
          sw = (k == 0) ? w : sw + w;
        }
        wrote_w = (pp.costfct >= 0 && pp.costfct <= 2);
      }
    }
    b0 = fold8(b0, 0.f, true, false);
    if (NOP == 2) b1 = fold8(b1, 0.f, true, false);
    sw = fold8(sw, 0.f, true, false);
    if (active) {
      if (finishing) {
        active = false;
      } else {
        const float dpsq = (NOP == 2) ? dp0 * dp0 + dp1 * dp1 : dp0 * dp0;
        if (cnt == 1) dpsq_init = dpsq;
        mares_old = mares;
        mares = sw / fn;
        // the two ratio tests only count once min_iter is reached: skip their divisions before
        bool go = (cnt < pp.max_iter) & (mares > pp.res_thresh);
        if (go && cnt >= pp.min_iter)
          go = (dpsq / dpsq_init >= pp.dp_thresh_sq) & (mares / mares_old <= pp.dr_thresh);
        if (!go) {
          conv = 1;
          active = false;
        } else {
          cnt++;
          if (NOP == 2) {
            const float y0 = b0 / L00;
            const float y1 = (b1 - L10 * y0) / L11;
            dp1 = y1 / L11;
            dp0 = (y0 - L10 * dp1) / L00;
            p0 = p0 - dp0;
            p1 = p1 - dp1;
            ptx = refx + p0;
            pty = refy + p1;
          } else {
            dp0 = (b0 / L00) / L00;
            p0 = p0 - dp0;
            p0 = (camlr_of(g, frame) == 0) ? std_min(p0, 0.0f) : std_max(p0, 0.0f);
            ptx = refx + p0;
          }
          const float ex = stx - ptx, ey = sty - pty;
          if (sqrtf(ex * ex + ey * ey) > g.outlierthresh || ptx < g.lb || pty < g.lb || ptx > g.ubw ||
              pty > g.ubh) {
            p0 = pin0;
            p1 = pin1;
            ptx = refx + p0;
            if (NOP == 2) pty = refy + p1;
            conv = 1;
            finishing = true;
          }
        }
      }
    }
  }
  if (valid) {
    float* pw = g.pat_w + ((size_t)frame * g.np + ip) * 64;
#pragma unroll
    for (int k = 0; k < 8; ++k) pw[l8 + 8 * k] = wrote_w ? fabsf(R[k]) : 0.f;
    if (l8 == 0) {
      float* po = g.pat_p + ((size_t)frame * g.np + ip) * NOP;
      po[0] = p0;
      if (NOP == 2) po[1] = p1;
      g.pat_conv[(size_t)frame * g.np + ip] = conv;
      g.pat_cnt[(size_t)frame * g.np + ip] = cnt;
    }
  }
}

// ---------------------------------------------------------------------------
// Specialisation for P = 12 (operating points 3 and 4; gray and RGB): same 8-lanes-per-patch
// mapping and reduction order as the generic kernel, but
//   * the template and the residual of a lane (P*P*C/8 = 18 or 54 elements) live in registers, the
//     template gradients too for gray (RGB keeps them in shared-memory columns);
//   * the bilinear taps of I1 come from a per-patch WINDOW in shared memory -- the (P+1+2M)^2 pixels
//     around the patch's current integer position (M = 2 pixels of slack; stereo: P+1 rows, the row
//     never moves) -- staged by the patch's own 8 lanes and re-staged only when the position leaves
//     the slack.  The generic kernel issues 4 LDGs per element and iteration whose 32 lanes touch 4
//     patches x 1..2 sectors each: the L1 tag stage, not the math, bounded it (profiles/).  From
//     shared memory the same taps are 4 LDS with at most a 2-way bank conflict between patches;
//   * element offsets are walked incrementally (no offset table).
// Arithmetic (operand order, reduction tree, stop tests) is that of patch_optimize_kernel.
//
// The window is filled with LDG: a TMA tensor-tile fill was measured and loses (DESIGN.md section 5.2).
template <int V> struct CostTag { static constexpr int value = V; };
template <int NOP, int C> struct PwCfg {
  static constexpr int P = 12, M = 2, W = P + 1 + 2 * M, PC = P * C, N = P * P * C, NK = N / 8;
  static constexpr int WH = (NOP == 2) ? W : P + 1;  // window rows
  static constexpr int WC = W * C;                    // floats per window row
  static constexpr int WIN = WH * WC;                 // floats per window
};

template <int NOP, int C>
__global__ void __launch_bounds__(256, C == 1 ? 2 : 1) patch_p12_kernel(LevelGeom g, PatchParams pp, int f0,
                                                                        int init_from_coarser) {
  pdl_wait();  // programmatic dependent launch: nothing of the previous kernel is touched before this
  using Cfg = PwCfg<NOP, C>;
  constexpr int P = Cfg::P, M = Cfg::M, W = Cfg::W, PC = Cfg::PC, N = Cfg::N, NK = Cfg::NK;
  constexpr int WH = Cfg::WH, WC = Cfg::WC, WIN = Cfg::WIN;
  constexpr int SY = WH - P - 1;  // rows of slack (stereo: none, the row never moves)
  constexpr bool G_REG = (C == 1);            // template gradients in registers
  extern __shared__ float smem[];
  const int tid = threadIdx.x, nthr = blockDim.x;
  const int l8 = tid & 7;
  const int frame = f0 + blockIdx.y;
  const int ip = blockIdx.x * (nthr >> 3) + (tid >> 3);
  const bool valid = ip < g.np;
  const float fn = (float)N;
  float* const win = smem + (tid >> 3) * WIN;                  // this patch's window
  float* const sGx = smem + (nthr >> 3) * WIN + tid;           // RGB: gradient columns [k][thread]
  float* const sGy = sGx + NK * nthr;
  const int rowC = g.tmp_w * C;

  const float* i0 = g.img[0] + (size_t)frame * g.img_fs[0];
  const float* i0x = g.img[1] + (size_t)frame * g.img_fs[1];
  const float* i0y = g.img[2] + (size_t)frame * g.img_fs[2];
  const float* i1 = g.img[3] + (size_t)frame * g.img_fs[3];

  const int ipc = valid ? ip : 0;
  const int gx_i = ipc / g.noph, gy_i = ipc - gx_i * g.noph;
  const int cxi = gx_i * g.steps + g.offw, cyi = gy_i * g.steps + g.offh;
  const float refx = (float)cxi, refy = (float)cyi;

  // ---- K1: template, gradients, mean normalisation (patch.cpp:287-332) ------
  float T[NK], R[NK], GX[G_REG ? NK : 1], GY[G_REG ? NK : 1];
  {
    const int base = ((cxi + g.pad - P / 2) + (cyi + g.pad - P / 2) * g.tmp_w) * C;
    float acc = 0.f;
    int rem = l8, off = l8;  // element e = l8 + 8k: rem = e mod P*C, off = image offset
#pragma unroll
    for (int k = 0; k < NK; ++k) {
      T[k] = i0[base + off];
      const float gx = i0x[base + off], gy = i0y[base + off];
      if (G_REG) {
        GX[k] = gx;
        GY[k] = gy;
      } else {
        sGx[k * nthr] = gx;
        sGy[k * nthr] = gy;
      }
      acc = (k == 0) ? T[k] : acc + T[k];
      R[k] = 0.f;
      rem += 8;
      off += 8;
      if (rem >= PC) {
        rem -= PC;
        off += rowC - PC;
      }
    }
    if (pp.patnorm > 0) {
      const float m = fold8(acc, 0.f, true, false) / fn;
#pragma unroll
      for (int k = 0; k < NK; ++k) T[k] = T[k] - m;
    }
  }
  // ---- Hessian and its Cholesky factor (patch.cpp:71-88) ---------------------
  float L00, L10 = 0.f, L11 = 0.f;
  {
    float axx = 0.f, axy = 0.f, ayy = 0.f;
#pragma unroll
    for (int k = 0; k < NK; ++k) {
      const float a = G_REG ? GX[k] : sGx[k * nthr], b = G_REG ? GY[k] : sGy[k * nthr];
      const float vxx = a * a, vxy = a * b, vyy = b * b;
      axx = (k == 0) ? vxx : axx + vxx;
      axy = (k == 0) ? vxy : axy + vxy;
      ayy = (k == 0) ? vyy : ayy + vyy;
    }
    float H00 = fold8(axx, 0.f, true, false);
    if (NOP == 2) {
      const float H01 = fold8(axy, 0.f, true, false);
      float H11 = fold8(ayy, 0.f, true, false);
      if (H00 * H11 - H01 * H01 == 0.f) {
        H00 = (float)((double)H00 + 1e-10);
        H11 = (float)((double)H11 + 1e-10);
      }
      L00 = H00; L10 = H01; L11 = H11;
      if (H00 > 0.f) {
        L00 = sqrtf(H00);
        L10 = H01 / L00;
        const float x = H11 - L10 * L10;
        if (x > 0.f) L11 = sqrtf(x);
      }
    } else {
      if (H00 == 0.f) H00 = (float)((double)H00 + 1e-10);
      L00 = H00 > 0.f ? sqrtf(H00) : H00;
    }
  }
  // ---- K2 (patchgrid.cpp:195-211) ---------------------------------------------
  float pin0 = 0.f, pin1 = 0.f;
  if (init_from_coarser && g.flow_prev != nullptr) {
    const float* fp = g.flow_prev + (size_t)frame * g.flow_prev_frame_stride;
    const int i = (cyi >> 1) * (g.w / 2) + (cxi >> 1);
    if (NOP == 2) {
      const float2 v = reinterpret_cast<const float2*>(fp)[i];
      pin0 = v.x * 2.f;
      pin1 = v.y * 2.f;
    } else {
      pin0 = fp[i] * 2.f;
    }
  }
  // ---- K3 (patch.cpp:119-212, 264-284) ------------------------------------------
  float p0 = pin0, p1 = pin1, dp0 = 0.f, dp1 = 0.f;
  float ptx = refx + p0, pty = (NOP == 2) ? refy + p1 : refy;
  const float stx = ptx, sty = pty;
  float dpsq_init = 1e-10f, mares = 1e5f, mares_old = 1e20f;
  int cnt = 0, conv = 0;
  bool wrote_w = false, finishing = false, active = valid;
  if (active && (ptx < g.lb || pty < g.lb || ptx > g.ubw || pty > g.ubh)) {
    conv = 1;
    active = false;
  }
  // window origin in padded-image pixels; far away = nothing staged yet
  int wx0 = -(1 << 20), wy0 = -(1 << 20);

  while (__any_sync(FULL, active)) {
    float b0 = 0.f, b1 = 0.f, sw = 0.f;
    {
      float acc = 0.f;
      float w0 = 0.f, w1 = 0.f, w2 = 0.f, w3 = 0.f;
      int ux = 0, uy = 0;
      bool restage = false;
      if (active) {
        const int pcx = (int)ceilf(ptx + .00001f), pcy = (int)ceilf(pty + .00001f);
        const int pfx = (int)floorf(ptx), pfy = (int)floorf(pty);
        const float rx = ptx - (float)pfx, ry = pty - (float)pfy;
        w0 = rx * ry;
        w1 = (1.f - rx) * ry;
        w2 = rx * (1.f - ry);
        w3 = (1.f - rx) * (1.f - ry);
        // top-left tap of element (0,0): padded-image pixel (tx, ty)
        const int tx = pcx + g.pad - P / 2 - 1, ty = pcy + g.pad - P / 2 - 1;
        ux = tx - wx0;
        uy = ty - wy0;
        restage = (ux < 0) | (ux > W - P - 1) | (uy < 0) | (uy > SY);
        if (restage) {
          wx0 = tx - M;
          wy0 = (NOP == 2) ? ty - M : ty;
          ux = tx - wx0;
          uy = (NOP == 2) ? M : 0;
        }
      }
      if (__any_sync(FULL, restage)) {
        __syncwarp();  // every lane has finished reading the previous window
        if (restage) {
          const int xlo = wx0 * C, xmax = g.tmp_w * C - 1;
          for (int idx = l8; idx < WIN; idx += 8) {
            const int row = idx / WC, cc = idx - row * WC;
            int sy = wy0 + row, sx = xlo + cc;  // coordinates outside the padded image are never used as taps
            sy = sy < 0 ? 0 : (sy > g.tmp_h - 1 ? g.tmp_h - 1 : sy);
            sx = sx < 0 ? 0 : (sx > xmax ? xmax : sx);
            win[idx] = __ldg(i1 + (size_t)sy * rowC + sx);
          }
        }
        __syncwarp();
      }
      if (active) {
        const float* q = win + uy * WC + ux * C;  // tap d of element 0
        int rem = l8, off = l8;
#pragma unroll
        for (int k = 0; k < NK; ++k) {
          const float* a = q + off;
          const float v = w0 * a[WC + C] + w1 * a[WC] + w2 * a[C] + w3 * a[0];
          R[k] = v;
          acc = (k == 0) ? v : acc + v;
          rem += 8;
          off += 8;
          if (rem >= PC) {
            rem -= PC;
            off += WC - PC;
          }
        }
      }
      float m = 0.f;
      if (pp.patnorm > 0) m = fold8(acc, 0.f, true, false) / fn;
      if (active) {
        // the cost function is uniform over the launch: one copy of the loop per cost instead of a
        // three-way branch per element (LossComputeErrorImage, patch.cpp:223-262)
        auto residuals = [&](auto cost_tag) {
          constexpr int COST = decltype(cost_tag)::value;
#pragma unroll
          for (int k = 0; k < NK; ++k) {
            float d = R[k];
            if (pp.patnorm > 0) d = d - m;
            float r, w;
            if (COST == 0) {
              r = d - T[k];
              w = fabsf(r);
            } else if (COST == 1) {
              const float t = d - T[k];
              r = copysignf(sqrtf(fabsf(t)), t);
              w = fabsf(r);
            } else if (COST == 2) {
              const float t = d - T[k];
              const float hh = sqrtf((sqrtf(1.0f + (t * t) / 25.0f) - 1.0f) * 50.0f);
              r = copysignf(hh, t);
              w = fabsf(r);
            } else {  // reference leaves pdiff/pweight untouched (patch.cpp:230-261)
              r = d;
              w = 0.f;
            }
            R[k] = r;
            const float gx = G_REG ? GX[k] : sGx[k * nthr], gy = G_REG ? GY[k] : sGy[k * nthr];
            const float vx = gx * r, vy = gy * r;
            b0 = (k == 0) ? vx : b0 + vx;
            b1 = (k == 0) ? vy : b1 + vy;
            sw = (k == 0) ? w : sw + w;
          }
        };
        if (pp.costfct == 0) residuals(CostTag<0>{});
        else if (pp.costfct == 1) residuals(CostTag<1>{});
        else if (pp.costfct == 2) residuals(CostTag<2>{});
        else residuals(CostTag<3>{});
        wrote_w = (pp.costfct >= 0 && pp.costfct <= 2);
      }
    }
    b0 = fold8(b0, 0.f, true, false);
    if (NOP == 2) b1 = fold8(b1, 0.f, true, false);
    sw = fold8(sw, 0.f, true, false);
    if (active) {
      if (finishing) {
        active = false;
      } else {
        const float dpsq = (NOP == 2) ? dp0 * dp0 + dp1 * dp1 : dp0 * dp0;
        if (cnt == 1) dpsq_init = dpsq;
        mares_old = mares;
        mares = sw / fn;
        bool go = (cnt < pp.max_iter) & (mares > pp.res_thresh);
        if (go && cnt >= pp.min_iter)
          go = (dpsq / dpsq_init >= pp.dp_thresh_sq) & (mares / mares_old <= pp.dr_thresh);
        if (!go) {
          conv = 1;
          active = false;
        } else {
          cnt++;
          if (NOP == 2) {
            const float y0 = b0 / L00;
            const float y1 = (b1 - L10 * y0) / L11;
            dp1 = y1 / L11;
            dp0 = (y0 - L10 * dp1) / L00;
            p0 = p0 - dp0;
            p1 = p1 - dp1;
            ptx = refx + p0;
            pty = refy + p1;
          } else {
            dp0 = (b0 / L00) / L00;
            p0 = p0 - dp0;
            p0 = (camlr_of(g, frame) == 0) ? std_min(p0, 0.0f) : std_max(p0, 0.0f);
            ptx = refx + p0;
          }
          const float ex = stx - ptx, ey = sty - pty;
          if (sqrtf(ex * ex + ey * ey) > g.outlierthresh || ptx < g.lb || pty < g.lb || ptx > g.ubw ||
              pty > g.ubh) {
            p0 = pin0;
            p1 = pin1;
            ptx = refx + p0;
            if (NOP == 2) pty = refy + p1;
            conv = 1;
            finishing = true;
          }
        }
      }
    }
  }
  if (valid) {
    float* pw = g.pat_w + ((size_t)frame * g.np + ip) * N;
#pragma unroll
    for (int k = 0; k < NK; ++k) pw[l8 + 8 * k] = wrote_w ? fabsf(R[k]) : 0.f;
    if (l8 == 0) {
      float* po = g.pat_p + ((size_t)frame * g.np + ip) * NOP;
      po[0] = p0;
      if (NOP == 2) po[1] = p1;
      g.pat_conv[(size_t)frame * g.np + ip] = conv;
      g.pat_cnt[(size_t)frame * g.np + ip] = cnt;
    }
  }
}

// 8 lanes per patch; dynamic shared memory: the patches' windows, then (RGB) the gradient columns
template <int NOP, int C>
void launch_patch_p12(const LevelGeom& g, const PatchParams& pp, int f0, int f1, int init, cudaStream_t st) {
  using Cfg = PwCfg<NOP, C>;
  const int threads = 256;
  const dim3 grid((g.np + threads / 8 - 1) / (threads / 8), f1 - f0);
  const size_t sm = sizeof(float) * ((size_t)(threads / 8) * Cfg::WIN + (C == 1 ? 0 : (size_t)2 * Cfg::NK * threads));
  if (sm > 48 * 1024) cudaFuncSetAttribute(patch_p12_kernel<NOP, C>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm);
  patch_p12_kernel<NOP, C><<<grid, threads, sm, st>>>(g, pp, f0, init);
}

// usefbcon, second loop of AggregateFlowDense (patchgrid.cpp:278-375) as a gather: the patches of
// the complementary frame `cq`, at their displaced positions, add their NEGATED flow with bilinear
// weights.  The reference's scatter visits patches in ascending ip and the pixels of a patch in
// raster order, so this cell receives at most four terms per patch -- from the patch pixels at
// (xi,yi) [wbil0], (xi+1,yi) [wbil1], (xi,yi+1) [wbil2], (xi+1,yi+1) [wbil3], in that order.  Only
// patches whose reference lies within `reach` (+ patch extent) of the cell can contribute.
template <int NOP>
__device__ __forceinline__ void densify_merge_complement(const LevelGeom& g, int cq, int xi, int yi, float& we,
                                                         float& a0, float& a1) {
  const int P = g.P, C = g.noc, n = g.novals, lb = -P / 2, ub = P / 2 - 1;
  const float* pp = g.pat_p + (size_t)cq * g.np * NOP;
  const float* pw = g.pat_w + (size_t)cq * g.np * n;
  const int* pos = g.fb_pos + (size_t)cq * g.np * 2;
  const float* wb = g.fb_wbil + (size_t)cq * g.np * 4;
  const int reach = g.fb_reach[cq];
  // a patch at position pos covers cells pos+lb-1 .. pos+ub; |pos - ref| <= reach
  int gx0 = xi - ub - reach - g.offw, gx1 = xi - lb + 1 + reach - g.offw;
  gx0 = gx0 <= 0 ? 0 : (gx0 + g.steps - 1) / g.steps;
  gx1 = gx1 < 0 ? -1 : gx1 / g.steps;
  if (gx1 > g.nopw - 1) gx1 = g.nopw - 1;
  int gy0 = yi - ub - reach - g.offh, gy1 = yi - lb + 1 + reach - g.offh;
  gy0 = gy0 <= 0 ? 0 : (gy0 + g.steps - 1) / g.steps;
  gy1 = gy1 < 0 ? -1 : gy1 / g.steps;
  if (gy1 > g.noph - 1) gy1 = g.noph - 1;
  for (int gx = gx0; gx <= gx1; ++gx)
    for (int gy = gy0; gy <= gy1; ++gy) {
      const int ip = gx * g.noph + gy;
      const int p0 = pos[2 * ip], p1 = pos[2 * ip + 1];
      if (xi < p0 + lb - 1 || xi > p0 + ub || yi < p1 + lb - 1 || yi > p1 + ub) continue;
      // in-image rectangle of this patch (the reference tests xt>=1, yt>=1, xt<w-1, yt<h-1), patch coordinates
      int x0 = 1 - p0 - lb, x1 = g.w - 2 - p0 - lb, y0 = 1 - p1 - lb;
      x0 = x0 < 0 ? 0 : x0;
      x1 = x1 > P - 1 ? P - 1 : x1;
      y0 = y0 < 0 ? 0 : y0;
      const float f0v = pp[ip * NOP], f1v = (NOP == 2) ? pp[ip * NOP + 1] : 0.f;
#pragma unroll
      for (int t = 0; t < 4; ++t) {
        const int xt = xi + (t & 1), yt = yi + (t >> 1);
        const int rx = xt - p0 - lb, ry = yt - p1 - lb;
        if (rx < 0 || rx > P - 1 || ry < 0 || ry > P - 1) continue;
        if (!(xt >= 1 && yt >= 1 && xt < g.w - 1 && yt < g.h - 1)) continue;
        // weight cursor: +1 per pixel and +(C-1) per in-image pixel before this one (patchgrid.cpp:331-339)
        const float* q = pw + (size_t)ip * n + (ry * P + rx) + (C - 1) * ((ry - y0) * (x1 - x0 + 1) + (rx - x0));
        float absw;
        if (C == 1) {
          absw = 1.0f / std_max(2.0f, q[0]);
        } else {
          absw = std_max(2.0f, q[0]);
          for (int c = 1; c < C; ++c) absw += std_max(2.0f, q[c]);
          absw = 1.0f / absw;
        }
        const float wt = wb[4 * ip + t];
        we += wt * absw;
        a0 -= wt * (f0v * absw);
        if (NOP == 2) a1 -= wt * (f1v * absw);
      }
    }
}

// K4: PatGridClass::AggregateFlowDense (patchgrid.cpp:213-275,377-394) as a
// per-pixel gather.  The reference scatters patch by patch in ip = x*noph + y
// order; visiting the covering patches of a pixel in ascending (x, y) grid order
// performs the same float additions in the same order, without atomics.
template <int NOP>
__global__ void __launch_bounds__(256) densify_kernel(LevelGeom g, int f0) {
  pdl_wait();  // programmatic dependent launch: nothing of the previous kernel is touched before this
  const int xi = blockIdx.x * blockDim.x + threadIdx.x;
  const int yi = blockIdx.y * blockDim.y + threadIdx.y;
  const int frame = frame_of(g, f0, blockIdx.z);
  if (xi >= g.w || yi >= g.h) return;
  const int P = g.P, C = g.noc, n = g.novals, hp = P / 2;
  const float* pp = g.pat_p + (size_t)frame * g.np * NOP;
  const float* pw = g.pat_w + (size_t)frame * g.np * n;
  // grid columns whose patch covers xi: xi - hp + 1 <= cx <= xi + hp
  int gx0 = (xi - hp + 1 - g.offw + g.steps - 1);
  gx0 = gx0 < 0 ? 0 : gx0 / g.steps;
  int gx1 = xi + hp - g.offw;
  gx1 = gx1 < 0 ? -1 : gx1 / g.steps;
  if (gx1 > g.nopw - 1) gx1 = g.nopw - 1;
  int gy0 = (yi - hp + 1 - g.offh + g.steps - 1);
  gy0 = gy0 < 0 ? 0 : gy0 / g.steps;
  int gy1 = yi + hp - g.offh;
  gy1 = gy1 < 0 ? -1 : gy1 / g.steps;
  if (gy1 > g.noph - 1) gy1 = g.noph - 1;

  float we = 0.f, a0 = 0.f, a1 = 0.f;
  for (int gx = gx0; gx <= gx1; ++gx) {
    const int cx = gx * g.steps + g.offw, rx = xi - cx + hp;
    for (int gy = gy0; gy <= gy1; ++gy) {
      const int cy = gy * g.steps + g.offh, ry = yi - cy + hp;
      const int ip = gx * g.noph + gy;
      float absw;
      if (C == 1) {
        absw = 1.0f / std_max(2.0f, pw[(size_t)ip * n + ry * P + rx]);
      } else {
        // patchgrid.cpp:243-259: the weight cursor advances by 1 for a patch pixel
        // outside the image and by C for one inside.
        const int x0 = cx - hp < 0 ? hp - cx : 0, y0 = cy - hp < 0 ? hp - cy : 0;
        const int x1 = cx + hp - 1 > g.w - 1 ? g.w - 1 - cx + hp : P - 1;
        const int inb = (ry - y0) * (x1 - x0 + 1) + (rx - x0);
        const float* q = pw + (size_t)ip * n + (ry * P + rx) + (C - 1) * inb;
        absw = std_max(2.0f, q[0]);
        for (int c = 1; c < C; ++c) absw += std_max(2.0f, q[c]);
        absw = 1.0f / absw;
      }
      we += absw;
      a0 += pp[ip * NOP] * absw;
      if (NOP == 2) a1 += pp[ip * NOP + 1] * absw;
    }
  }
  if (g.fb) densify_merge_complement<NOP>(g, frame ^ 1, xi, yi, we, a0, a1);
  float* out = g.flow + (size_t)frame * g.flow_frame_stride + ((size_t)yi * g.w + xi) * NOP;
  if (we > 0.f) {
    a0 = a0 / we;
    a1 = a1 / we;
  }
  out[0] = a0;
  if (NOP == 2) out[1] = a1;
}

// Swapped copy of the image pair into the backward frame of every couple: its template is I1,
// its target I0 (oflow.cpp:193-197).  Gradients are derived afterwards by sobel_kernel.
__global__ void __launch_bounds__(256) swap_images_kernel(LevelGeom g, int f0) {
  pdl_wait();  // programmatic dependent launch: nothing of the previous kernel is touched before this
  const size_t n = (size_t)g.tmp_w * g.tmp_h * g.noc;
  const int fwd = f0 + 2 * blockIdx.y, bwd = fwd + 1;
  const float* a = g.img[0] + (size_t)fwd * g.img_fs[0];
  const float* b = g.img[3] + (size_t)fwd * g.img_fs[3];
  float* a2 = const_cast<float*>(g.img[0]) + (size_t)bwd * g.img_fs[0];
  float* b2 = const_cast<float*>(g.img[3]) + (size_t)bwd * g.img_fs[3];
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    a2[i] = b[i];
    b2[i] = a[i];
  }
}

// usefbcon, first half of the second loop of AggregateFlowDense (patchgrid.cpp:296-318): per patch the
// integer position after optimisation and its bilinear weights; per frame how far any patch moved
// (bounds the gather window of densify_merge_complement exactly).  One CTA per frame.
template <int NOP>
__global__ void __launch_bounds__(256) fb_prepare_kernel(LevelGeom g, int f0) {
  pdl_wait();  // programmatic dependent launch: nothing of the previous kernel is touched before this
  __shared__ int s_max[256];
  const int frame = f0 + blockIdx.x;
  const float* pp = g.pat_p + (size_t)frame * g.np * NOP;
  int* pos = g.fb_pos + (size_t)frame * g.np * 2;
  float* wb = g.fb_wbil + (size_t)frame * g.np * 4;
  int reach = 0;
  for (int ip = threadIdx.x; ip < g.np; ip += blockDim.x) {
    const int gx = ip / g.noph, gy = ip - gx * g.noph;
    const int cx = gx * g.steps + g.offw, cy = gy * g.steps + g.offh;
    // GetPointPos() == pt_ref + p_iter (patch.cpp:214-221; stereo keeps the row)
    const float rpx = (float)cx + pp[ip * NOP], rpy = (NOP == 2) ? (float)cy + pp[ip * NOP + 1] : (float)cy;
    const int p0 = (int)ceil((double)rpx + .00001), p1 = (int)ceil((double)rpy + .00001);  // double literal in the reference
    const float r0 = rpx - (float)(int)floorf(rpx), r1 = rpy - (float)(int)floorf(rpy);
    pos[2 * ip] = p0;
    pos[2 * ip + 1] = p1;
    wb[4 * ip] = r0 * r1;
    wb[4 * ip + 1] = (1.f - r0) * r1;
    wb[4 * ip + 2] = r0 * (1.f - r1);
    wb[4 * ip + 3] = (1.f - r0) * (1.f - r1);
    const int dx = p0 > cx ? p0 - cx : cx - p0, dy = p1 > cy ? p1 - cy : cy - p1;
    reach = max(reach, max(dx, dy));
  }
  s_max[threadIdx.x] = reach;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if (threadIdx.x < o) s_max[threadIdx.x] = max(s_max[threadIdx.x], s_max[threadIdx.x + o]);
    __syncthreads();
  }
  if (threadIdx.x == 0) g.fb_reach[frame] = s_max[0];
}


}  // namespace

int launch_patch_optimize(const LevelGeom& g, const PatchParams& pp, int f0, int f1, bool init_from_coarser,
                          cudaStream_t st, Profiler* prof) {
  ProfScope scope(prof, KC_PATCH);
  if (g.P == 8 && g.noc == 1) {  // register-resident specialisation (operating points 1 and 2)
    const dim3 grid8((g.np + 31) / 32, f1 - f0);
    if (g.nop == 2) launch_k(g.pdl && !prof, patch_p8c1_kernel<2>, dim3(grid8), dim3(256), 0, st, g, pp, f0, init_from_coarser ? 1 : 0);
    else launch_k(g.pdl && !prof, patch_p8c1_kernel<1>, dim3(grid8), dim3(256), 0, st, g, pp, f0, init_from_coarser ? 1 : 0);
    return cudaGetLastError() == cudaSuccess ? 1 : -1;
  }
  if (g.P == 12 && g.pad >= 12 && (g.noc == 1 || g.noc == 3)) {  // window-staged specialisation (operating points 3 and 4)
    const int init = init_from_coarser ? 1 : 0;
    if (g.nop == 2 && g.noc == 1) launch_patch_p12<2, 1>(g, pp, f0, f1, init, st);
    else if (g.nop == 2) launch_patch_p12<2, 3>(g, pp, f0, f1, init, st);
    else if (g.noc == 1) launch_patch_p12<1, 1>(g, pp, f0, f1, init, st);
    else launch_patch_p12<1, 3>(g, pp, f0, f1, init, st);
    return cudaGetLastError() == cudaSuccess ? 1 : -1;
  }
  const int n = g.novals;
  const int NK = (n / 8) + (((n % 8) >= 4) ? 1 : 0);
  int threads = 256;
  while (threads > 32 && (size_t)5 * NK * threads * sizeof(float) > 200 * 1024) threads >>= 1;
  const size_t smem = (size_t)5 * NK * threads * sizeof(float);
  const dim3 grid((g.np + threads / 8 - 1) / (threads / 8), f1 - f0);
  if (g.nop == 2) {
    if (smem > 48 * 1024)
      cudaFuncSetAttribute(patch_optimize_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    patch_optimize_kernel<2><<<grid, threads, smem, st>>>(g, pp, f0, init_from_coarser ? 1 : 0);
  } else {
    if (smem > 48 * 1024)
      cudaFuncSetAttribute(patch_optimize_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    patch_optimize_kernel<1><<<grid, threads, smem, st>>>(g, pp, f0, init_from_coarser ? 1 : 0);
  }
  return cudaGetLastError() == cudaSuccess ? 1 : -1;
}

int launch_fb_prepare(const LevelGeom& g, int f0, int f1, cudaStream_t st) {
  if (g.nop == 2) fb_prepare_kernel<2><<<f1 - f0, 256, 0, st>>>(g, f0);
  else fb_prepare_kernel<1><<<f1 - f0, 256, 0, st>>>(g, f0);
  return cudaGetLastError() == cudaSuccess ? 1 : -1;
}

int launch_swap_images(const LevelGeom& g, int f0, int f1, cudaStream_t st) {  // [f0,f1): internal frames, couples
  const size_t n = (size_t)g.tmp_w * g.tmp_h * g.noc;
  const dim3 grid((unsigned)((n + 1023) / 1024 > 64 ? 64 : (n + 1023) / 1024), (f1 - f0) / 2);
  swap_images_kernel<<<grid, 256, 0, st>>>(g, f0);
  return cudaGetLastError() == cudaSuccess ? 1 : -1;
}

// [f0,f1) are launch indices: frame = f0 + index * g.fstep
int launch_densify(const LevelGeom& g, int f0, int f1, cudaStream_t st, Profiler* prof) {
  ProfScope scope(prof, KC_DENSIFY);
  const dim3 block(32, 8), grid((g.w + 31) / 32, (g.h + 7) / 8, f1 - f0);
  if (g.nop == 2) launch_k(g.pdl && !prof, densify_kernel<2>, grid, block, 0, st, g, f0);
  else launch_k(g.pdl && !prof, densify_kernel<1>, grid, block, 0, st, g, f0);
  return cudaGetLastError() == cudaSuccess ? 1 : -1;
}

}  // namespace ofdis
