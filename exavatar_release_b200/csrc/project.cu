// project.cu -- K1: per-Gaussian projection + exact tile counting, and the tile-offset scan.
//
// Replaces, for ExAvatar's render path (avatar/common/nets/module.py:632-640), the reference rasteriser's
// preprocess kernel, its CUB inclusive scan over Gaussians and the device->host copy of the duplicate count
// (SURVEY.md section 2.3 rows 1-3; algorithm App. A.1).  Design differences from that pipeline:
//   * one 48-byte packed record per Gaussian (three 16-byte vectors) instead of five SoA arrays, so the
//     composites gather a splat with three vector loads from one 64-byte-aligned neighbourhood;
//   * the conic is stored pre-scaled for exp2 (one MUFU.EX2, no multiply in the inner loop);
//   * tiles are counted per TILE (histogram with L2 reductions), not per Gaussian, so the later scatter writes each
//     tile's list contiguously and the sort is a per-tile shared-memory sort instead of a global 64-bit radix sort;
//   * a (splat, tile) pair is dropped when the splat provably cannot reach alpha >= 1/255 at any pixel centre of
//     the tile -- output-preserving (every dropped pair would have been skipped per pixel by App. A.3) and cuts
//     list length for anisotropic / low-opacity splats.
#include "gaussian_math.cuh"

namespace b2r {

int g_last_cuda_error = 0;

__device__ __forceinline__ void sh_to_rgb(int deg, const float* __restrict__ sh, const float3 mean, const Cam& cam,
                                          float* rgb, uint32_t& clamp_bits) {
  float dx = mean.x - cam.campos[0], dy = mean.y - cam.campos[1], dz = mean.z - cam.campos[2];
  const float n = sqrtf(dx * dx + dy * dy + dz * dz);
  const float x = dx / n, y = dy / n, z = dz / n;
  clamp_bits = 0;
#pragma unroll
  for (int c = 0; c < 3; c++) {
    auto SH = [&](int k) { return sh[k * 3 + c]; };  // `sh` is the Gaussian's row in the warp's shared-memory stage
    float r = B2R_SH_C0 * SH(0);
    if (deg > 0) {
      r = r - B2R_SH_C1 * y * SH(1) + B2R_SH_C1 * z * SH(2) - B2R_SH_C1 * x * SH(3);
      if (deg > 1) {
        const float xx = x * x, yy = y * y, zz = z * z, xy = x * y, yz = y * z, xz = x * z;
        r = r + c_SH_C2[0] * xy * SH(4) + c_SH_C2[1] * yz * SH(5) + c_SH_C2[2] * (2.f * zz - xx - yy) * SH(6) +
            c_SH_C2[3] * xz * SH(7) + c_SH_C2[4] * (xx - yy) * SH(8);
        if (deg > 2) {
          r = r + c_SH_C3[0] * y * (3.f * xx - yy) * SH(9) + c_SH_C3[1] * xy * z * SH(10) +
              c_SH_C3[2] * y * (4.f * zz - xx - yy) * SH(11) + c_SH_C3[3] * z * (2.f * zz - 3.f * xx - 3.f * yy) * SH(12) +
              c_SH_C3[4] * x * (4.f * zz - xx - yy) * SH(13) + c_SH_C3[5] * z * (xx - yy) * SH(14) +
              c_SH_C3[6] * x * (xx - 3.f * yy) * SH(15);
        }
      }
    }
    r += 0.5f;
    if (r < 0.f) clamp_bits |= 1u << c;
    rgb[c] = fmaxf(r, 0.f);
  }
}

#ifndef PROJ_MIN_BLOCKS
#define PROJ_MIN_BLOCKS 4  // 64 registers: four CTAs per SM; tuning hook (build_ext.py B2R_NVCC_EXTRA)
#endif
__global__ void __launch_bounds__(256, PROJ_MIN_BLOCKS) project_kernel(const B2RScene sc, const Ctx cx, int32_t* __restrict__ radii,
                                                      const int aggregate) {
  // CTA-level histogram in shared memory: atomics of different warps to the SAME global address serialise in L2
  // (~15 ns each measured on the hot avatar tiles), so each CTA adds to a tile's counter at most once.
  extern __shared__ uint32_t s_cnt[];
  if (aggregate) {
    for (int t = threadIdx.x; t < cx.tiles; t += blockDim.x) s_cnt[t] = 0u;
    __syncthreads();
  }
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  // SH rows (192 bytes apart for degree 3) are staged through shared memory: each warp copies the contiguous block of
  // its 32 rows with coalesced 128-byte loads; a thread then reads its own row (odd row stride: conflict-free).
  // Only rows below sh_rows have coefficients (B2RScene.sh_rows); a warp wholly above them stages nothing and its
  // lanes take their colour from colors_precomp.
  const float* shrow = nullptr;
  if (sc.shs) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int L = sc.sh_coeffs * 3, S = L | 1;
    const int sh_rows = sc.sh_rows > 0 ? sc.sh_rows : sc.P;
    float* wstage = reinterpret_cast<float*>(s_cnt + (aggregate ? cx.tiles : 0)) + (size_t)warp * 32 * S;
    const int row0 = blockIdx.x * blockDim.x + warp * 32;
    const int nrows = min(32, sh_rows - row0);
    if (nrows > 0) stage_rows<0>(wstage, const_cast<float*>(sc.shs) + (size_t)row0 * L, L, nrows, 0xffffffffu);
    __syncwarp();
    if (i < sh_rows) shrow = wstage + lane * S;
  }
  // fused skinning: the warp's 32 weight rows (J floats each) take the same staged route as the SH rows
  const float* wrow = nullptr;
  if (sc.skin_xyz) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int J = sc.skin_J, S = J | 1;
    float* base = reinterpret_cast<float*>(s_cnt + (aggregate ? cx.tiles : 0));
    if (sc.shs) base += (size_t)8 * 32 * ((sc.sh_coeffs * 3) | 1);
    float* wstage = base + (size_t)warp * 32 * S;
    const int row0 = blockIdx.x * blockDim.x + warp * 32;
    const int nrows = min(32, sc.P - row0);
    if (nrows > 0) stage_rows<0>(wstage, const_cast<float*>(sc.skin_weights) + (size_t)row0 * J, J, nrows, 0xffffffffu);
    __syncwarp();
    wrow = wstage + lane * S;
  }
  const Cam cam = load_cam(sc);
  bool visible = false;
  Geom g;
  g.g0 = make_float4(0.f, 0.f, 0.f, 0.f);
  g.g1 = make_float4(0.f, 0.f, 0.f, INFINITY);
  g.g2 = make_float4(0.f, 0.f, 0.f, 0.f);
  int4 aux = make_int4(0, 0, 0, 0);
  if (i < sc.P) {
    float3 p;
    if (wrow) {
      p = skin_position(sc, i, wrow).world;
      if (sc.skin_means_out) {
        sc.skin_means_out[3 * (size_t)i] = p.x;
        sc.skin_means_out[3 * (size_t)i + 1] = p.y;
        sc.skin_means_out[3 * (size_t)i + 2] = p.z;
      }
    } else {
      p = make_float3(__ldg(sc.means3D + 3 * (size_t)i), __ldg(sc.means3D + 3 * (size_t)i + 1),
                      __ldg(sc.means3D + 3 * (size_t)i + 2));
    }
    const float3 pv = xform4x3(p, cam.v);
    if (pv.z > K_NEAR) {  // App. A.1 step 1
      // Homogeneous position and pixel centre WITHOUT fma contraction, operation for operation as the oracle's C
      // expression (App. A.1 steps 2, 7).  One ulp of a pixel coordinate near 1000 is 6e-5 px; through a sharp splat's
      // exponent that is a 1e-4 relative change of alpha, enough to flip alpha >= 1/255 decisions the oracle's threshold
      // margins do not expect (seen at 1024^2 / 1080p, profiles/r02_notes.md).  Bit-identical centres remove that source.
      const float ph_x = dot4_rn(cam.p[0], p.x, cam.p[4], p.y, cam.p[8], p.z, cam.p[12]);
      const float ph_y = dot4_rn(cam.p[1], p.x, cam.p[5], p.y, cam.p[9], p.z, cam.p[13]);
      const float ph_w = dot4_rn(cam.p[3], p.x, cam.p[7], p.y, cam.p[11], p.z, cam.p[15]);
      const float pw = __fdiv_rn(1.f, __fadd_rn(ph_w, K_EPS_W));
      float c6[6];
      if (sc.cov3D_precomp) {
#pragma unroll
        for (int k = 0; k < 6; k++) c6[k] = __ldg(sc.cov3D_precomp + 6 * (size_t)i + k);
      } else {
        const float3 s = make_float3(__ldg(sc.scales + 3 * (size_t)i), __ldg(sc.scales + 3 * (size_t)i + 1),
                                     __ldg(sc.scales + 3 * (size_t)i + 2));
        const float* qp = sc.rotations + 4 * (size_t)i;  // scalar loads: the tensor may be a 4-byte-aligned view
        const float4 q = make_float4(__ldg(qp), __ldg(qp + 1), __ldg(qp + 2), __ldg(qp + 3));
        cov3d_from_scale_rot(s, sc.scale_modifier, q, c6);
      }
      Ewa e;
      ewa_project(pv, c6, cam, e);
      const float det = e.a * e.c - e.b * e.b;
      if (det != 0.f) {  // step 5
        const float det_inv = 1.f / det;
        const float conx = e.c * det_inv, cony = -e.b * det_inv, conz = e.a * det_inv;
        const float mid = 0.5f * (e.a + e.c);
        const float root = sqrtf(fmaxf(K_EIG_FLOOR, mid * mid - det));
        const float lam = fmaxf(mid + root, mid - root);
        const int radius = (int)ceilf(3.f * sqrtf(lam));
        const float px = __fmul_rn(__fadd_rn(__fmul_rn(__fadd_rn(__fmul_rn(ph_x, pw), 1.f), (float)cam.W), -1.f), 0.5f);
        const float py = __fmul_rn(__fadd_rn(__fmul_rn(__fadd_rn(__fmul_rn(ph_y, pw), 1.f), (float)cam.H), -1.f), 0.5f);
        int x0 = (int)((px - (float)radius) / (float)TILE), y0 = (int)((py - (float)radius) / (float)TILE);
        int x1 = (int)((px + (float)radius + (float)(TILE - 1)) / (float)TILE);
        int y1 = (int)((py + (float)radius + (float)(TILE - 1)) / (float)TILE);
        x0 = min(cx.gx, max(0, x0)); y0 = min(cx.gy, max(0, y0));
        x1 = min(cx.gx, max(0, x1)); y1 = min(cx.gy, max(0, y1));
        if ((x1 - x0) * (y1 - y0) != 0) {  // step 8
          visible = true;
          const float o = __ldg(sc.opacities + i);
          float rgb[3];
          uint32_t bits = 0;
          if (shrow) {  // the SH clamp bits are set for SH rows only
            sh_to_rgb(sc.sh_degree, shrow, p, cam, rgb, bits);
          } else {
            rgb[0] = __ldg(sc.colors_precomp + 3 * (size_t)i);
            rgb[1] = __ldg(sc.colors_precomp + 3 * (size_t)i + 1);
            rgb[2] = __ldg(sc.colors_precomp + 3 * (size_t)i + 2);
          }
          const float A2 = -0.5f * LOG2E * conx, B2 = -LOG2E * cony, C2 = -0.5f * LOG2E * conz;
          // thr2: smallest log2-exponent at which opacity * 2^p2 can still reach 1/255
          float thr2;
          const bool concave = (A2 < 0.f) && (C2 < 0.f) && (4.f * A2 * C2 > B2 * B2) && (det > 0.f);
          if (!(o > 0.f)) thr2 = INFINITY;            // alpha <= 0 < 1/255 everywhere
          else if (!concave) thr2 = -INFINITY;        // degenerate conic: never cull, evaluate per pixel
          else thr2 = -log2f(255.f * o) - CULL_MARGIN2;
          g.g0 = make_float4(px, py, A2, B2);
          g.g1 = make_float4(C2, o, pv.z, thr2);
          g.g2 = make_float4(rgb[0], rgb[1], rgb[2], __uint_as_float((bits << 29) | (uint32_t)i));  // id rides with the record
          aux = make_int4(x0 | (y0 << 16), x1 | (y1 << 16), radius, 0);
        }
      }
    }
    radii[i] = aux.z;
    float4* gp = reinterpret_cast<float4*>(cx.geom + i);
    gp[0] = g.g0;
    gp[1] = g.g1;
    gp[2] = g.g2;
  }
  // per-tile histogram of kept (splat, tile) pairs -- warp-cooperative, exact culling unless disabled; the kept mask of a
  // rect of <= 32 tiles rides in aux.w for the scatter
  {
    const int gx = cx.gx;
    uint32_t* tile_count = aggregate ? s_cnt : cx.tile_count;
    aux.w = (int)warp_count_kept_tiles(visible, aux.x & 0xffff, aux.x >> 16, aux.y & 0xffff, aux.y >> 16, g.g0.x, g.g0.y,
                                       g.g0.z, g.g0.w, g.g1.x, g.g1.w, (sc.flags & B2R_FLAG_NO_TILE_CULL) != 0, sc.width,
                                       sc.height, gx, tile_count);
    if (i < sc.P) cx.aux[i] = aux;
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) cx.classes[CLS_SCAN_FINAL] = 0u;  // new counts: no final scan yet
  const unsigned vis = __ballot_sync(0xffffffffu, visible);
  if ((threadIdx.x & 31) == 0 && vis) atomicAdd(&cx.classes[CLS_VIS_ACC], (uint32_t)__popc(vis));
  if (aggregate) {
    __syncthreads();
    for (int t = threadIdx.x; t < cx.tiles; t += blockDim.x) {
      const uint32_t c = s_cnt[t];
      if (c) atomicAdd(cx.tile_count + t, c);
    }
  }
}

// Exclusive scan of the per-tile counts (one block; tiles <= a few 10^4).  Writes ranges[t] = [start, end) clamped to
// the duplicate capacity, primes the scatter cursors with `start`, and publishes the total.
// `final`: this scan's ranges are the ones the binning will use (a duplicate capacity was given), so the per-tile
// counters are consumed: the kernel leaves them -- and the other accumulators of the ctx -- zero for the next render,
// which can then skip status_reset_kernel (B2R_FLAG_CTX_CLEAN).
// `final` = 2: the re-scan of b2r_forward_render.  If the projection phase already ran a final scan (it was given a
// capacity), the counters are gone and its ranges stand: nothing to do (B2RStatus.overflow still tells the caller when
// that capacity was too small).
__global__ void __launch_bounds__(1024) tile_scan_kernel(const Ctx cx, const int final) {
  if (final == 2 && cx.classes[CLS_SCAN_FINAL] != 0u) return;
  __shared__ uint64_t warp_sums[32];
  __shared__ uint64_t carry_s;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (threadIdx.x == 0) carry_s = 0;
  __syncthreads();
  for (int base = 0; base < cx.tiles; base += 1024) {
    const int t = base + threadIdx.x;
    const uint64_t v = t < cx.tiles ? cx.tile_count[t] : 0;
    uint64_t inc = v;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const uint64_t n = __shfl_up_sync(0xffffffffu, inc, d);
      if (lane >= d) inc += n;
    }
    if (lane == 31) warp_sums[warp] = inc;
    __syncthreads();
    if (warp == 0) {
      uint64_t w = warp_sums[lane];
#pragma unroll
      for (int d = 1; d < 32; d <<= 1) {
        const uint64_t n = __shfl_up_sync(0xffffffffu, w, d);
        if (lane >= d) w += n;
      }
      warp_sums[lane] = w;
    }
    __syncthreads();
    const uint64_t carry = carry_s;
    const uint64_t excl = carry + (warp > 0 ? warp_sums[warp - 1] : 0) + inc - v;
    if (t < cx.tiles) {
      const uint64_t cap = cx.dup_capacity;
      const uint32_t s = (uint32_t)(excl < cap ? excl : cap);
      const uint32_t e = (uint32_t)(excl + v < cap ? excl + v : cap);
      cx.ranges[t] = make_uint2(s, e);
      cx.tile_cursor[t] = s;
    }
    __syncthreads();
    if (threadIdx.x == 1023) carry_s = carry + warp_sums[31];
    __syncthreads();
  }
  // Longest-list-first processing order for the per-tile kernels (sort, composites): counting sort of the tiles
  // by floor(log2(n)) descending.  Tile cost is ~linear in n and spans three orders of magnitude, so launching in
  // index order leaves most SMs idle behind a few heavy tiles that happened to start late.
  __shared__ uint32_t bin_cursor[34];
  __shared__ uint32_t n_large_s, n_multi_s;
  if (threadIdx.x < 34) bin_cursor[threadIdx.x] = 0;
  __syncthreads();
  auto bin_of = [](uint32_t n) { return n == 0 ? 33 : __clz(n); };  // clz = 31 - floor(log2 n): small bin = long list
  for (int t = threadIdx.x; t < cx.tiles; t += blockDim.x) atomicAdd(&bin_cursor[bin_of(cx.tile_count[t])], 1u);
  __syncthreads();
  if (threadIdx.x == 0) {
    uint32_t run = 0;
    for (int b = 0; b < 34; b++) {
      const uint32_t c = bin_cursor[b];
      bin_cursor[b] = run;
      run += c;
    }
    // class boundaries of the per-tile sort (binning.cu): bins 0..20 hold n >= 2048 (sorted in chunks), bins 0..31-s hold
    // n >= 2^s = SORT_CTA_MIN (one CTA per list; shorter lists are sorted eight to a CTA, one per warp)
    cx.status->reserved[0] = (unsigned long long)bin_cursor[21] | ((unsigned long long)bin_cursor[32 - SORT_CTA_SHIFT] << 32);
    n_large_s = bin_cursor[21];
    // segmented composites: tiles of >= SEG (256) entries are the bins 0..23; cut only when there is room for checkpoints
    n_multi_s = cx.ckpt ? bin_cursor[32 - SEG_SHIFT] : 0u;  // bins 0..31-s hold n >= 2^s
    cx.classes[CLS_N_LARGE] = bin_cursor[21];
    cx.classes[CLS_N_GE512] = bin_cursor[23];
    cx.classes[CLS_N_GE1024] = bin_cursor[22];
    cx.classes[CLS_N_MULTI] = n_multi_s;
  }
  __syncthreads();
  for (int t = threadIdx.x; t < cx.tiles; t += blockDim.x) {
    const uint32_t pos = atomicAdd(&bin_cursor[bin_of(cx.tile_count[t])], 1u);
    cx.tile_order[pos] = (uint32_t)t;
  }
  __syncthreads();
  // Block-wide exclusive scan of ceil(n / 2^shift) over the first n_tiles entries of tile_order (all threads call it;
  // the total is returned to every thread).  One pass of 1024 tiles covers every workload measured so far.
  __shared__ uint32_t wsum[32];
  auto scan_units = [&](const uint32_t n_tiles, const int shift, uint32_t* out) -> uint32_t {
    uint32_t run = 0;
    for (uint32_t base = 0; base < n_tiles; base += 1024) {
      const uint32_t t = base + threadIdx.x;
      uint32_t c = 0;
      if (t < n_tiles) {
        const uint2 r = cx.ranges[cx.tile_order[t]];
        c = (r.y - r.x + (1u << shift) - 1u) >> shift;
      }
      uint32_t incl = c;
#pragma unroll
      for (int d = 1; d < 32; d <<= 1) {
        const uint32_t v = __shfl_up_sync(0xffffffffu, incl, d);
        if (lane >= d) incl += v;
      }
      if (lane == 31) wsum[warp] = incl;
      __syncthreads();
      if (warp == 0) {
        uint32_t w = wsum[lane];
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
          const uint32_t v = __shfl_up_sync(0xffffffffu, w, d);
          if (lane >= d) w += v;
        }
        wsum[lane] = w;
      }
      __syncthreads();
      if (t < n_tiles) out[t] = run + (warp > 0 ? wsum[warp - 1] : 0u) + incl - c;
      run += wsum[31];
      __syncthreads();  // wsum is rewritten by the next round
    }
    return run;
  };
  static_assert(SORT_CHUNK == 2048 && SEG == (1 << SEG_SHIFT), "scan_units takes the unit as a shift");
  // Tiles of >= 2048 entries are sorted in chunks of SORT_CHUNK by separate CTAs and merged afterwards (binning.cu):
  // chunk_start[t] = first chunk of the t-th tile of tile_order, reserved[1] = number of chunks.
  const uint32_t n_chunks = scan_units(n_large_s, 11, cx.chunk_start);
  // Segment table of the multi-segment tiles (composite_fwd4.cu / composite_bwd4.cu): seg_start[t] = segments of all
  // earlier such tiles = index of the tile's first checkpoint record.
  uint32_t segs = scan_units(n_multi_s, SEG_SHIFT, cx.seg_start);
  __syncthreads();
  if (threadIdx.x == 0) {
    cx.status->reserved[1] = n_chunks;
    cx.classes[CLS_N_CHUNKS] = n_chunks;
    // cannot exceed the store by construction (sum of ceil(n / 256) <= capacity / 256 + tiles); guard all the same
    if (segs > cx.max_segs) { segs = 0; cx.classes[CLS_N_MULTI] = 0; n_multi_s = 0; }
    cx.classes[CLS_TOTAL_SEGS] = segs;
  }
  __syncthreads();
  for (uint32_t t = threadIdx.x; t < n_multi_s; t += blockDim.x) {  // one (tile, segment) entry per backward work item
    const uint2 r = cx.ranges[cx.tile_order[t]];
    const uint32_t c = (r.y - r.x + SEG - 1) / SEG, s0 = cx.seg_start[t];
    for (uint32_t k = 0; k < c; k++) cx.seg_table[s0 + k] = make_uint2(t, k);
  }
  if (final) {  // every read of the counters happened before the barrier above
    for (int t = threadIdx.x; t < cx.tiles; t += blockDim.x) {
      cx.tile_count[t] = 0u;
      cx.tile_maxid[t] = 0u;
    }
  }
  if (threadIdx.x == 0) {
    const uint64_t total = carry_s;
    cx.status->num_visible = cx.classes[CLS_VIS_ACC];
    if (final) {
      cx.classes[CLS_VIS_ACC] = 0u;
      cx.classes[CLS_SCAN_FINAL] = 1u;
    }
    cx.status->consumed_fwd = 0;
    cx.status->consumed_bwd = 0;
    cx.status->num_dups = total;
    cx.status->dup_capacity = cx.dup_capacity;
    cx.status->overflow = total > cx.dup_capacity ? 1u : 0u;
    cx.status->token = cx.status_token;
    if (cx.status_mirror) {
      volatile uint64_t* m = cx.status_mirror;
      m[0] = total;
      __threadfence_system();
      m[1] = cx.status_token;
    }
  }
}

// resets the status block and the per-tile counters the projection kernel accumulates into
__global__ void status_reset_kernel(const Ctx cx) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t < cx.tiles) {
    cx.tile_count[t] = 0u;
    cx.tile_maxid[t] = 0u;
  }
  if (t == 0) {
    B2RStatus* s = cx.status;
    s->num_dups = 0;
    s->overflow = 0;
    s->num_visible = 0;
    s->consumed_fwd = 0;
    s->consumed_bwd = 0;
    cx.classes[CLS_VIS_ACC] = 0u;
    cx.classes[CLS_SCAN_FINAL] = 0u;
  }
}

__global__ void mark_visible_kernel(int P, const float* __restrict__ means3D, const float* __restrict__ view,
                                    uint8_t* __restrict__ present) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= P) return;
  const float x = means3D[3 * (size_t)i], y = means3D[3 * (size_t)i + 1], z = means3D[3 * (size_t)i + 2];
  const float vz = dot4_rn(view[2], x, view[6], y, view[10], z, view[14]);
  present[i] = vz > K_NEAR ? 1 : 0;
}

int launch_project(const B2RScene& sc, const Ctx& cx, int32_t* radii, cudaStream_t st) {
  const bool clean = (sc.flags & B2R_FLAG_CTX_CLEAN) != 0;  // the previous render's final scan left the counters zero
  if (!clean) { ProfScope p(K_MISC, st); launch_k(status_reset_kernel, (cx.tiles + 1023) / 1024, 1024, 0, st, true, cx); }
  if (sc.P > 0) {
    ProfScope p(K_PROJECT, st);
    const int aggregate = cx.tiles <= 2048;  // beyond that the per-CTA sweeps over the tile table cost more than they save
    const size_t smem = (aggregate ? (size_t)cx.tiles * 4 : 0) +
                        (sc.shs ? (size_t)8 * 32 * ((sc.sh_coeffs * 3) | 1) * sizeof(float) : 0) +
                        (sc.skin_xyz ? (size_t)8 * 32 * (sc.skin_J | 1) * sizeof(float) : 0);
    cudaFuncSetAttribute(project_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024);  // per device
    launch_k(project_kernel, (sc.P + 255) / 256, 256, smem, st, true, sc, cx, radii, aggregate);
  }
  { ProfScope p(K_TILE_SCAN, st); launch_k(tile_scan_kernel, 1, 1024, 0, st, true, cx, cx.dup_capacity > 0 ? 1 : 0); }
  return check_launch();
}

void launch_tile_scan(const Ctx& cx, cudaStream_t st) {
  ProfScope p(K_TILE_SCAN, st);
  launch_k(tile_scan_kernel, 1, 1024, 0, st, true, cx, 2);
}

int launch_mark_visible(int P, const float* means3D, const float* view, uint8_t* present, cudaStream_t st) {
  ProfScope p(K_MISC, st, P > 0 ? 1 : 0);
  if (P > 0) launch_k(mark_visible_kernel, (P + 255) / 256, 256, 0, st, true, P, means3D, view, present);
  return check_launch();
}

}  // namespace b2r
