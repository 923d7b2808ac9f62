// project_bwd.cu -- K6: per-Gaussian backward of the projection (App. A.5), fused: conic -> 2D covariance -> 3D
// covariance -> scale / quaternion, EWA Jacobian -> mean, perspective projection -> mean, depth -> mean, SH -> coeffs
// and view direction -> mean.  Replaces the reference rasteriser's two backward preprocess kernels (SURVEY.md
// section 2.3 rows 9-10).  Every output element is written (zeros for culled Gaussians), so the host allocates
// the gradient tensors uninitialised and no memset kernels run.
//
// Conventions kept from the published backward (App. A.6): 1/(det^2 + 1e-7), frustum-clamped t.x / t.y pass no direct
// gradient, gradient is w.r.t. the un-normalised quaternion, dL/dmeans2D is NDC-scaled (x 0.5 W, 0.5 H) with z = 0
// -- the quantity ExAvatar thresholds for densification (module.py:155-157,176; config.py:21).
#include "gaussian_math.cuh"

namespace b2r {

// Body of K6 for one Gaussian.  `shrow` (shared memory, may be null) holds the Gaussian's SH coefficients on entry and
// its SH gradient on exit (row layout k*3 + c, as in global memory); see the staging in the kernel below.
__device__ __forceinline__ void project_bwd_one(const B2RScene& sc, const Ctx& cx, const B2RBackwardArgs& out,
                                                const float* __restrict__ gacc, const int i, const size_t oi,
                                                const bool visible, const int4 aux, float* shrow,
                                                const float* wrow) {
  const int M = sc.sh_coeffs;
  const bool accumulate = (out.flags & B2R_BWD_ACCUMULATE) != 0;

  float dm[3] = {0.f, 0.f, 0.f}, dm2[2] = {0.f, 0.f}, dcol[3] = {0.f, 0.f, 0.f}, dop = 0.f;
  float dS[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  float dscale[3] = {0.f, 0.f, 0.f}, dq[4] = {0.f, 0.f, 0.f, 0.f};
  uint32_t clamp_bits = 0;
  float3 p = make_float3(0.f, 0.f, 0.f);
  Cam cam;
  Skin skin;
  // gradient arriving at the posed position itself (other ExAvatar modules read it, model.py:172-173): also for
  // Gaussians this render culled
  const bool posed_in = wrow != nullptr && out.dL_dposed != nullptr;
  if (posed_in && !visible) skin = skin_position(sc, i, wrow);

  if (visible) {
    cam = load_cam(sc);
    const float4 q0 = reinterpret_cast<const float4*>(gacc)[3 * (size_t)i];
    const float4 q1 = reinterpret_cast<const float4*>(gacc)[3 * (size_t)i + 1];
    const float4 q2 = reinterpret_cast<const float4*>(gacc)[3 * (size_t)i + 2];
    dm2[0] = (0.5f * (float)sc.width * INV_LOG2E) * q0.x;
    dm2[1] = (0.5f * (float)sc.height * INV_LOG2E) * q0.y;
    const float dcon[3] = {-0.5f * q0.z, -0.5f * q0.w, -0.5f * q1.x};
    dop = q1.y;
    const float ddep = q1.z;
    dcol[0] = q2.x; dcol[1] = q2.y; dcol[2] = q2.z;
    clamp_bits = __float_as_uint(reinterpret_cast<const float4*>(cx.geom + i)[2].w) >> 29;

    if (wrow) {
      skin = skin_position(sc, i, wrow);
      p = skin.world;
    } else {
      p = make_float3(__ldg(sc.means3D + 3 * (size_t)i), __ldg(sc.means3D + 3 * (size_t)i + 1),
                      __ldg(sc.means3D + 3 * (size_t)i + 2));
    }
    float c6[6];
    float3 scl = make_float3(0.f, 0.f, 0.f);
    float4 q = make_float4(1.f, 0.f, 0.f, 0.f);
    if (sc.cov3D_precomp) {
#pragma unroll
      for (int k = 0; k < 6; k++) c6[k] = __ldg(sc.cov3D_precomp + 6 * (size_t)i + k);
    } else {
      scl = make_float3(__ldg(sc.scales + 3 * (size_t)i), __ldg(sc.scales + 3 * (size_t)i + 1),
                        __ldg(sc.scales + 3 * (size_t)i + 2));
      const float* qp = sc.rotations + 4 * (size_t)i;
      q = make_float4(__ldg(qp), __ldg(qp + 1), __ldg(qp + 2), __ldg(qp + 3));
      cov3d_from_scale_rot(scl, sc.scale_modifier, q, c6);
    }
    const float3 pv = xform4x3(p, cam.v);
    Ewa e;
    ewa_project(pv, c6, cam, e);

    // conic -> (a, b, c)
    const float a = e.a, b = e.b, c = e.c;
    const float denom = a * c - b * b;
    const float d2inv = 1.f / (denom * denom + K_EPS_W);
    float dLa = 0.f, dLb = 0.f, dLc = 0.f;
    if (d2inv != 0.f) {
      dLa = d2inv * (-c * c * dcon[0] + 2.f * b * c * dcon[1] + (denom - a * c) * dcon[2]);
      dLc = d2inv * (-a * a * dcon[2] + 2.f * a * b * dcon[1] + (denom - a * c) * dcon[0]);
      dLb = d2inv * 2.f * (b * c * dcon[0] - (denom + 2.f * b * b) * dcon[1] + a * b * dcon[2]);
      const float* A0 = e.A0;
      const float* A1 = e.A1;
      dS[0] = A0[0] * A0[0] * dLa + A0[0] * A1[0] * dLb + A1[0] * A1[0] * dLc;
      dS[3] = A0[1] * A0[1] * dLa + A0[1] * A1[1] * dLb + A1[1] * A1[1] * dLc;
      dS[5] = A0[2] * A0[2] * dLa + A0[2] * A1[2] * dLb + A1[2] * A1[2] * dLc;
      dS[1] = 2.f * A0[0] * A0[1] * dLa + (A0[0] * A1[1] + A0[1] * A1[0]) * dLb + 2.f * A1[0] * A1[1] * dLc;
      dS[2] = 2.f * A0[0] * A0[2] * dLa + (A0[0] * A1[2] + A0[2] * A1[0]) * dLb + 2.f * A1[0] * A1[2] * dLc;
      dS[4] = 2.f * A0[2] * A0[1] * dLa + (A0[1] * A1[2] + A0[2] * A1[1]) * dLb + 2.f * A1[1] * A1[2] * dLc;
    }
    // (a,b,c) -> rows of A = J Rv -> J -> t -> mean
    const float S[9] = {c6[0], c6[1], c6[2], c6[1], c6[3], c6[4], c6[2], c6[4], c6[5]};
    float dA0[3], dA1[3];
#pragma unroll
    for (int k = 0; k < 3; k++) {
      const float SA0 = e.A0[0] * S[3 * k] + e.A0[1] * S[3 * k + 1] + e.A0[2] * S[3 * k + 2];
      const float SA1 = e.A1[0] * S[3 * k] + e.A1[1] * S[3 * k + 1] + e.A1[2] * S[3 * k + 2];
      dA0[k] = 2.f * SA0 * dLa + SA1 * dLb;
      dA1[k] = 2.f * SA1 * dLc + SA0 * dLb;
    }
    const float* v = cam.v;
    const float dJ00 = dA0[0] * v[0] + dA0[1] * v[4] + dA0[2] * v[8];
    const float dJ02 = dA0[0] * v[2] + dA0[1] * v[6] + dA0[2] * v[10];
    const float dJ11 = dA1[0] * v[1] + dA1[1] * v[5] + dA1[2] * v[9];
    const float dJ12 = dA1[0] * v[2] + dA1[1] * v[6] + dA1[2] * v[10];
    const float tz = 1.f / e.t[2], tz2 = tz * tz, tz3 = tz2 * tz;
    const float dtx = e.xmul * -cam.fx * tz2 * dJ02;
    const float dty = e.ymul * -cam.fy * tz2 * dJ12;
    const float dtz = -cam.fx * tz2 * dJ00 - cam.fy * tz2 * dJ11 + (2.f * cam.fx * e.t[0]) * tz3 * dJ02 +
                      (2.f * cam.fy * e.t[1]) * tz3 * dJ12;
    dm[0] = v[0] * dtx + v[1] * dty + v[2] * dtz;
    dm[1] = v[4] * dtx + v[5] * dty + v[6] * dtz;
    dm[2] = v[8] * dtx + v[9] * dty + v[10] * dtz;

    // perspective projection of the centre
    const float* pm = cam.p;
    const float4 mh = xform4x4(p, pm);
    const float mw = 1.f / (mh.w + K_EPS_W);
    const float mul1 = mh.x * mw * mw, mul2 = mh.y * mw * mw;
    dm[0] += (pm[0] * mw - pm[3] * mul1) * dm2[0] + (pm[1] * mw - pm[3] * mul2) * dm2[1];
    dm[1] += (pm[4] * mw - pm[7] * mul1) * dm2[0] + (pm[5] * mw - pm[7] * mul2) * dm2[1];
    dm[2] += (pm[8] * mw - pm[11] * mul1) * dm2[0] + (pm[9] * mw - pm[11] * mul2) * dm2[1];
    // depth = row 2 of V . [p,1]
    dm[0] += v[2] * ddep;
    dm[1] += v[6] * ddep;
    dm[2] += v[10] * ddep;

    // Sigma = R S^2 R^T
    if (!sc.cov3D_precomp) {
      float R[9];
      quat_to_R(q, R);
      const float mod = sc.scale_modifier;
      const float s[3] = {mod * scl.x, mod * scl.y, mod * scl.z};
      const float G3[9] = {dS[0], 0.5f * dS[1], 0.5f * dS[2], 0.5f * dS[1], dS[3], 0.5f * dS[4], 0.5f * dS[2], 0.5f * dS[4], dS[5]};
      float dR[9];
#pragma unroll
      for (int k = 0; k < 3; k++) {
        float dN[3];
#pragma unroll
        for (int r = 0; r < 3; r++)
          dN[r] = 2.f * (G3[3 * r] * R[k] * s[k] + G3[3 * r + 1] * R[3 + k] * s[k] + G3[3 * r + 2] * R[6 + k] * s[k]);
        dscale[k] = mod * (R[k] * dN[0] + R[3 + k] * dN[1] + R[6 + k] * dN[2]);
#pragma unroll
        for (int r = 0; r < 3; r++) dR[3 * r + k] = dN[r] * s[k];
      }
      const float r = q.x, x = q.y, y = q.z, z = q.w;
      dq[0] = 2.f * (-z * dR[1] + y * dR[2] + z * dR[3] - x * dR[5] - y * dR[6] + x * dR[7]);
      dq[1] = 2.f * (y * dR[1] + z * dR[2] + y * dR[3] - 2.f * x * dR[4] - r * dR[5] + z * dR[6] + r * dR[7] - 2.f * x * dR[8]);
      dq[2] = 2.f * (-2.f * y * dR[0] + x * dR[1] + r * dR[2] + x * dR[3] + z * dR[5] - r * dR[6] + z * dR[7] - 2.f * y * dR[8]);
      dq[3] = 2.f * (-2.f * z * dR[0] - r * dR[1] + x * dR[2] + r * dR[3] - 2.f * z * dR[4] + y * dR[5] + x * dR[6] + y * dR[7]);
    }
  }

  // ---- SH (App. A.7): dL/dshs replaces the coefficients in `shrow`; the view-direction term is added to dL/dmean ----
  if (shrow) {
    if (!visible) {
      for (int k = 0; k < M * 3; k++) shrow[k] = 0.f;
    } else {
      const int deg = sc.sh_degree;
      const int used = (deg + 1) * (deg + 1);
      const float ddx = p.x - cam.campos[0], ddy = p.y - cam.campos[1], ddz = p.z - cam.campos[2];
      const float n = sqrtf(ddx * ddx + ddy * ddy + ddz * ddz);
      const float x = ddx / n, y = ddy / n, z = ddz / n;
      const float xx = x * x, yy = y * y, zz = z * z, xy = x * y, yz = y * z, xz = x * z;
      float ddir[3] = {0.f, 0.f, 0.f};
#pragma unroll
      for (int c = 0; c < 3; c++) {
        const float gc = ((clamp_bits >> c) & 1u) ? 0.f : dcol[c];
        float shv[16];  // this channel's coefficients, read before the gradient overwrites them in place
#pragma unroll
        for (int k = 0; k < 16; k++) shv[k] = k < used ? shrow[k * 3 + c] : 0.f;
        auto SH = [&](int k) { return shv[k]; };
        auto DSH = [&](int k, float basis) { shrow[k * 3 + c] = basis * gc; };
        float drx = 0.f, dry = 0.f, drz = 0.f;
        DSH(0, B2R_SH_C0);
        if (deg > 0) {
          DSH(1, -B2R_SH_C1 * y); DSH(2, B2R_SH_C1 * z); DSH(3, -B2R_SH_C1 * x);
          drx += -B2R_SH_C1 * SH(3); dry += -B2R_SH_C1 * SH(1); drz += B2R_SH_C1 * SH(2);
          if (deg > 1) {
            DSH(4, c_SH_C2[0] * xy); DSH(5, c_SH_C2[1] * yz); DSH(6, c_SH_C2[2] * (2.f * zz - xx - yy));
            DSH(7, c_SH_C2[3] * xz); DSH(8, c_SH_C2[4] * (xx - yy));
            drx += c_SH_C2[0] * y * SH(4) - 2.f * c_SH_C2[2] * x * SH(6) + c_SH_C2[3] * z * SH(7) + 2.f * c_SH_C2[4] * x * SH(8);
            dry += c_SH_C2[0] * x * SH(4) + c_SH_C2[1] * z * SH(5) - 2.f * c_SH_C2[2] * y * SH(6) - 2.f * c_SH_C2[4] * y * SH(8);
            drz += c_SH_C2[1] * y * SH(5) + 4.f * c_SH_C2[2] * z * SH(6) + c_SH_C2[3] * x * SH(7);
            if (deg > 2) {
              DSH(9, c_SH_C3[0] * y * (3.f * xx - yy));
              DSH(10, c_SH_C3[1] * xy * z);
              DSH(11, c_SH_C3[2] * y * (4.f * zz - xx - yy));
              DSH(12, c_SH_C3[3] * z * (2.f * zz - 3.f * xx - 3.f * yy));
              DSH(13, c_SH_C3[4] * x * (4.f * zz - xx - yy));
              DSH(14, c_SH_C3[5] * z * (xx - yy));
              DSH(15, c_SH_C3[6] * x * (xx - 3.f * yy));
              drx += c_SH_C3[0] * SH(9) * 6.f * xy + c_SH_C3[1] * SH(10) * yz - c_SH_C3[2] * SH(11) * 2.f * xy -
                     c_SH_C3[3] * SH(12) * 6.f * xz + c_SH_C3[4] * SH(13) * (4.f * zz - 3.f * xx - yy) +
                     c_SH_C3[5] * SH(14) * 2.f * xz + c_SH_C3[6] * SH(15) * 3.f * (xx - yy);
              dry += c_SH_C3[0] * SH(9) * 3.f * (xx - yy) + c_SH_C3[1] * SH(10) * xz +
                     c_SH_C3[2] * SH(11) * (4.f * zz - xx - 3.f * yy) - c_SH_C3[3] * SH(12) * 6.f * yz -
                     c_SH_C3[4] * SH(13) * 2.f * xy - c_SH_C3[5] * SH(14) * 2.f * yz - c_SH_C3[6] * SH(15) * 6.f * xy;
              drz += c_SH_C3[1] * SH(10) * xy + c_SH_C3[2] * SH(11) * 8.f * yz +
                     c_SH_C3[3] * SH(12) * 3.f * (2.f * zz - xx - yy) + c_SH_C3[4] * SH(13) * 8.f * xz +
                     c_SH_C3[5] * SH(14) * (xx - yy);
            }
          }
        }
        for (int k = used; k < M; k++) shrow[k * 3 + c] = 0.f;
        ddir[0] += drx * gc;
        ddir[1] += dry * gc;
        ddir[2] += drz * gc;
      }
      const float dot = x * ddir[0] + y * ddir[1] + z * ddir[2];
      dm[0] += (ddir[0] - x * dot) / n;
      dm[1] += (ddir[1] - y * dot) / n;
      dm[2] += (ddir[2] - z * dot) / n;
    }
  }

  if (posed_in) {
    dm[0] += __ldg(out.dL_dposed + 3 * (size_t)i);
    dm[1] += __ldg(out.dL_dposed + 3 * (size_t)i + 1);
    dm[2] += __ldg(out.dL_dposed + 3 * (size_t)i + 2);
  }
  const bool track = visible && (out.densify_rows == 0u || (uint32_t)i < out.densify_rows);
  if (track && out.densify_grad_accum) out.densify_grad_accum[oi] += sqrtf(dm2[0] * dm2[0] + dm2[1] * dm2[1]);
  if (track && out.densify_count) out.densify_count[oi] += 1.f;
  if (track && out.densify_radius_max) out.densify_radius_max[oi] = fmaxf(out.densify_radius_max[oi], (float)aux.z);
  auto put3 = [&](float* base, const float* v) {
    if (!base) return;
    float* d = base + 3 * oi;
    if (accumulate) { d[0] += v[0]; d[1] += v[1]; d[2] += v[2]; }
    else { d[0] = v[0]; d[1] = v[1]; d[2] = v[2]; }
  };
  // fused skinning: world-space gradient -> canonical position and the outer product the joint-transform GEMM needs
  if (wrow && (out.dL_dskin_xyz || out.dL_dskin_G)) {
    float gc[3] = {dm[0], dm[1], dm[2]}, dx[3] = {0.f, 0.f, 0.f}, G[12];
    float xs[4] = {0.f, 0.f, 0.f, 0.f};
    if (visible || posed_in) {
      if (sc.skin_cam_Rinv) {  // g_cam = Rinv^T g_world
        const float* R = sc.skin_cam_Rinv;
        gc[0] = __ldg(R) * dm[0] + __ldg(R + 3) * dm[1] + __ldg(R + 6) * dm[2];
        gc[1] = __ldg(R + 1) * dm[0] + __ldg(R + 4) * dm[1] + __ldg(R + 7) * dm[2];
        gc[2] = __ldg(R + 2) * dm[0] + __ldg(R + 5) * dm[1] + __ldg(R + 8) * dm[2];
      }
#pragma unroll
      for (int c = 0; c < 3; c++) dx[c] = skin.M[c] * gc[0] + skin.M[4 + c] * gc[1] + skin.M[8 + c] * gc[2];
      xs[0] = skin.x.x; xs[1] = skin.x.y; xs[2] = skin.x.z; xs[3] = 1.f;
    }
#pragma unroll
    for (int r = 0; r < 3; r++)
#pragma unroll
      for (int c = 0; c < 4; c++) G[4 * r + c] = gc[r] * xs[c];
    put3(out.dL_dskin_xyz, dx);
    if (out.dL_dskin_G) {
      float* d = out.dL_dskin_G + 12 * oi;
#pragma unroll
      for (int k = 0; k < 12; k++) { if (accumulate) d[k] += G[k]; else d[k] = G[k]; }
    }
  }
  const float dm2z[3] = {dm2[0], dm2[1], 0.f};
  put3(out.dL_dmeans3D, dm);
  put3(out.dL_dmeans2D, dm2z);
  // a scene with both colour sources (sh_rows > 0): the colour gradient of an SH row went to its coefficients above;
  // its dL_dcolors row is written zero, or left as it is when accumulating
  float* dcolors = out.dL_dcolors;
  if (i < sc.sh_rows) {
    dcol[0] = dcol[1] = dcol[2] = 0.f;
    if (accumulate) dcolors = nullptr;
  }
  put3(dcolors, dcol);
  put3(out.dL_dscales, dscale);
  if (out.dL_dopacities) {
    if (accumulate) out.dL_dopacities[oi] += dop; else out.dL_dopacities[oi] = dop;
  }
  if (out.dL_drotations) {
#pragma unroll
    for (int k = 0; k < 4; k++) {
      float* d = out.dL_drotations + 4 * oi + k;
      if (accumulate) *d += dq[k]; else *d = dq[k];
    }
  }
  if (out.dL_dcov3D) {
#pragma unroll
    for (int k = 0; k < 6; k++) {
      float* d = out.dL_dcov3D + 6 * oi + k;
      const float v = sc.cov3D_precomp ? dS[k] : 0.f;
      if (accumulate) *d += v; else *d = v;
    }
  }
}

// K6.  The per-Gaussian body above reads / writes everything with one thread per Gaussian, which is fine for the
// 3..4-float rows but not for SH: (P,16,3) rows are 192 bytes apart, so a per-thread walk touches 32 different
// 128-byte lines per load instruction.  SH rows therefore move through shared memory: every warp copies the
// contiguous block of its 32 rows in with coalesced 128-byte accesses (odd row stride: conflict-free), the body
// turns each row into its gradient in place, and the warp writes (or accumulates) the block back the same way.
#ifndef PBWD_MIN_BLOCKS
#define PBWD_MIN_BLOCKS 3  // 80 registers (64 bytes spilled): three CTAs per SM measured faster than two at 116; tuning hook
#endif
__global__ void __launch_bounds__(256, PBWD_MIN_BLOCKS) project_bwd_kernel(const B2RScene sc, const Ctx cx, const B2RBackwardArgs out,
                                                          const float* __restrict__ gacc) {
  extern __shared__ float sh_stage[];
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const bool in_range = i < sc.P;
  const bool accumulate = (out.flags & B2R_BWD_ACCUMULATE) != 0;
  int4 aux = make_int4(0, 0, 0, 0);
  if (in_range) aux = cx.aux[i];
  const bool visible = aux.z > 0;
  // out.first_row: Gaussians below it are a detached prefix (ExAvatar renders cat(scene.detach(), human),
  // model.py:117-125): nothing is written for them and Gaussian i lands in output row i - first_row
  const int first_row = (int)out.first_row;
  // an invisible Gaussian has nothing to add -- unless a gradient arrives at its posed position
  const bool active = in_range && i >= first_row && !(accumulate && !visible && out.dL_dposed == nullptr);
  const bool use_sh = sc.shs != nullptr && out.dL_dshs != nullptr;
  const int L = sc.sh_coeffs * 3, S = L | 1;
  float* wstage = sh_stage + (size_t)warp * 32 * S;
  const int row0 = blockIdx.x * blockDim.x + warp * 32;
  const int nrows = min(32, sc.P - row0);
  // rows [0, sh_rows) are coloured from SH (all rows when B2RScene.sh_rows == 0); the others from colors_precomp
  const int sh_rows = sc.sh_rows > 0 ? sc.sh_rows : sc.P;
  const int nsh = min(32, sh_rows - row0);
  if (use_sh && nsh > 0) {
    stage_rows<0>(wstage, const_cast<float*>(sc.shs) + (size_t)row0 * L, L, nsh, 0xffffffffu);
    __syncwarp();
  }
  float* shrow = use_sh && i < sh_rows ? wstage + lane * S : nullptr;
  const float* wrow = nullptr;
  if (sc.skin_xyz) {  // skinning weight rows, staged like the SH rows (after them in shared memory)
    const int J = sc.skin_J, SJ = J | 1;
    float* kstage = sh_stage + (use_sh ? (size_t)8 * 32 * S : 0) + (size_t)warp * 32 * SJ;
    if (nrows > 0) stage_rows<0>(kstage, const_cast<float*>(sc.skin_weights) + (size_t)row0 * J, J, nrows, 0xffffffffu);
    __syncwarp();
    wrow = kstage + lane * SJ;
  }
  if (active) project_bwd_one(sc, cx, out, gacc, i, (size_t)(i - first_row), visible, aux, shrow, wrow);
  if ((out.flags & B2R_BWD_SCRATCH_ZEROED) && in_range && visible) {  // leave the accumulator clean for the next render
    float4* row = reinterpret_cast<float4*>(const_cast<float*>(gacc)) + 3 * (size_t)i;
    row[0] = row[1] = row[2] = make_float4(0.f, 0.f, 0.f, 0.f);
  }
  if (use_sh && nsh > 0) {
    const unsigned rows_active = __ballot_sync(0xffffffffu, active && i < sh_rows);
    __syncwarp();  // every lane's row is complete before the block is written out cooperatively
    // rows below first_row and from sh_rows on are masked off, never touched
    float* dst = out.dL_dshs + ((ptrdiff_t)row0 - first_row) * L;
    if (accumulate) stage_rows<2>(wstage, dst, L, nsh, rows_active);
    else stage_rows<1>(wstage, dst, L, nsh, rows_active);
  }
}

int launch_project_bwd(const B2RScene& sc, const Ctx& cx, const B2RBackwardArgs& a, const float* gacc, cudaStream_t st) {
  ProfScope p(K_PROJECT_BWD, st, sc.P > 0 ? 1 : 0);
  if (sc.P > 0) {
    const bool use_sh = sc.shs != nullptr && a.dL_dshs != nullptr;
    const size_t smem = (use_sh ? (size_t)8 * 32 * ((sc.sh_coeffs * 3) | 1) * sizeof(float) : 0) +
                        (sc.skin_xyz ? (size_t)8 * 32 * (sc.skin_J | 1) * sizeof(float) : 0);
    cudaFuncSetAttribute(project_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 128 * 1024);  // per device
    launch_k(project_bwd_kernel, (sc.P + 255) / 256, 256, smem, st, true, sc, cx, a, gacc);
  }
  return check_launch();
}

}  // namespace b2r
