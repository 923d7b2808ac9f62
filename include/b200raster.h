/*
 * b200raster.h -- C ABI of the B200-native differentiable 3D-Gaussian rasteriser.
 *
 * Drop-in boundary for the one hot path of mks0601/ExAvatar_RELEASE: the rasteriser that
 * `GaussianRenderer.forward` reaches through `GaussianRasterizer(raster_settings)(...)`
 * (avatar/common/nets/module.py:609-640).  The reference binds that path through a third-party
 * pybind module (`diff_gaussian_rasterization_depth._C`, module.py:11, not vendored); the entry
 * points below are what that binding would call instead:
 *
 *   reference interface (file:line / upstream symbol)                    replaced by
 *   ------------------------------------------------------------------   -------------------------
 *   _C.rasterize_gaussians(...)        <- module.py:632-640 forward      b2r_forward_project +
 *                                                                        b2r_forward_render (or b2r_forward)
 *   _C.rasterize_gaussians_backward(.) <- loss.backward(), train.py:46   b2r_backward
 *   _C.mark_visible(...)               <- GaussianRasterizer.markVisible b2r_mark_visible
 *   geom/binning/img byte arenas owned by the autograd ctx               B2RWorkspace (caller-owned)
 *
 * Rules of the boundary: plain pointers and sizes only (no torch / STL types); every pointer is a
 * DEVICE pointer unless its comment says host; the library never allocates device memory, never
 * synchronises the stream and never throws -- it returns 0 or a negative B2R_E_* code.  All work is
 * enqueued on the caller's `stream` (a cudaStream_t passed as void*).
 *
 * Matrix layout (what ExAvatar hands over, module.py:605-607): `viewmatrix` / `projmatrix` are 16
 * floats with element (r,c) of the mathematical matrix at [4*c + r].
 */
#ifndef B200RASTER_H_
#define B200RASTER_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B2R_ABI_VERSION 3

#define B2R_OK 0
#define B2R_E_INVALID (-1)      /* bad argument (null pointer, negative size, both / neither colour source ...) */
#define B2R_E_WORKSPACE (-2)    /* ctx / scratch buffer smaller than b2r_*_bytes() reports */
#define B2R_E_CUDA (-3)         /* a CUDA launch failed; b2r_last_cuda_error() has the cudaError_t */
#define B2R_E_DUP_OVERFLOW (-4) /* only ever reported through B2RStatus.overflow (device side) */

/* flags */
#define B2R_FLAG_NO_TILE_CULL 1u /* keep every tile of the 3-sigma rect (reference list membership, for list parity tests) */
#define B2R_FLAG_DEBUG 2u        /* reference `debug=True` (module.py:621): the host wrapper syncs and checks after the call */
#define B2R_FLAG_CTX_CLEAN 4u    /* the ctx buffer's counters are zero: its last use was a b2r_forward / b2r_forward_project
                                    with dup_capacity > 0 (or b2r_forward_render) of this library, which leave them zero
                                    again -- the projection then skips its reset launch.  Never set it for a fresh buffer. */

/* Scene description shared by forward and backward: the fields of GaussianRasterizationSettings
 * (module.py:609-622) plus the per-Gaussian inputs of the call (module.py:632-640). */
typedef struct B2RScene {
  int32_t P;              /* number of Gaussians */
  int32_t width, height;  /* image_width, image_height */
  int32_t sh_degree;      /* active SH degree (0..3); ignored when shs == NULL */
  int32_t sh_coeffs;      /* M: coefficients per Gaussian in `shs` (0 when shs == NULL) */
  uint32_t flags;         /* B2R_FLAG_* */
  float scale_modifier;
  float tanfovx, tanfovy;
  const float* bg;            /* (3) */
  const float* viewmatrix;    /* (16) world->view, [4c+r] */
  const float* projmatrix;    /* (16) full projection (proj*view), [4c+r] */
  const float* campos;        /* (3) */
  const float* means3D;       /* (P,3) */
  const float* shs;           /* (P,M,3) or NULL; (sh_rows,M,3) when sh_rows > 0 */
  const float* colors_precomp;/* (P,3) or NULL  (exactly one of shs / colors_precomp, unless sh_rows > 0: see there) */
  const float* opacities;     /* (P) */
  const float* scales;        /* (P,3) or NULL */
  const float* rotations;     /* (P,4) (r,x,y,z), used un-normalised, or NULL */
  const float* cov3D_precomp; /* (P,6) or NULL  (exactly one of scales+rotations / cov3D_precomp) */
  /* Optional fused linear-blend skinning in front of the projection (SURVEY section 8f-2).  ExAvatar poses its human
   * Gaussians with  M_i = sum_j w_ij A_j,  posed_i = M_i [xyz_i, 1] + trans,  world_i = Rinv (posed_i - t)
   * (avatar/common/nets/module.py:413-422 `get_transform_mat_vertex` / `lbs`, module.py:555-557) as five PyTorch
   * kernels that write a (P,4,4) matrix per Gaussian.  With skin_xyz != NULL the projection kernels evaluate this per
   * Gaussian in registers instead of reading `means3D` (which may then be NULL); the backward emits the gradient with
   * respect to the canonical positions and the per-Gaussian outer products the joint-transform gradient is a GEMM of
   * (B2RBackwardArgs.dL_dskin_xyz / dL_dskin_G). */
  const float* skin_xyz;        /* (P,3) canonical ("big pose") positions, or NULL = no skinning */
  const float* skin_weights;    /* (P,J) skinning weights of each Gaussian (rows already gathered, module.py:414) */
  const float* skin_joint_mats; /* (J,16) row-major 4x4 transform per joint (module.py:385-411) */
  const float* skin_trans;      /* (3) root translation added after blending (module.py:421) */
  const float* skin_cam_Rinv;   /* (9) row-major inverse camera rotation, or NULL to stay in the posed frame */
  const float* skin_cam_t;      /* (3) camera translation (used with skin_cam_Rinv) */
  float* skin_means_out;        /* (P,3) optional OUTPUT: the posed world positions (other ExAvatar modules read them) */
  int32_t skin_J;               /* joints (55 for SMPL-X); <= 64 */
  /* Two colour sources in one scene (SURVEY section 8f-4 inside the merged frame of 8f-3): ExAvatar colours its scene
   * Gaussians from SH and its human Gaussians from rgb, and a merged pass renders cat(scene, human).
   *   sh_rows == 0:        one colour source for every row -- exactly one of shs (P,M,3) / colors_precomp (P,3).
   *   0 < sh_rows <= P:    rows [0, sh_rows) are coloured from `shs`, which is then (sh_rows,M,3) at `sh_degree`; rows
   *                        [sh_rows, P) from `colors_precomp`, which stays (P,3) indexed by Gaussian id (its rows below
   *                        sh_rows are never read).  colors_precomp is required iff sh_rows < P.  Not with skin_xyz.
   *   Backward (b2r_backward / b2r_backward_project): rows first_row <= i < sh_rows receive their SH gradient in
   *   dL_dshs row i - first_row and the view-direction term in dL_dmeans3D; their dL_dcolors row is written zero (left
   *   untouched with B2R_BWD_ACCUMULATE).  Rows >= sh_rows receive dL_dcolors.  first_row must be 0 or >= sh_rows;
   *   with first_row >= sh_rows no SH row takes part and dL_dshs may be NULL. */
  int32_t sh_rows;
} B2RScene;

/* Device-side status block; lives at offset 0 of the ctx buffer (read it back with a 64-byte D2H copy). */
typedef struct B2RStatus {
  uint64_t num_dups;      /* (tile, Gaussian) pairs the binning wants to emit */
  uint64_t dup_capacity;  /* capacity the render phase ran with */
  uint32_t overflow;      /* 1 if num_dups > dup_capacity: outputs are truncated, re-run with more room */
  uint32_t num_visible;   /* Gaussians with radii > 0 */
  uint64_t consumed_fwd;  /* list entries staged by the forward composite per tile (C_f of the roofline model), x 8 */
  uint64_t consumed_bwd;  /* list entries staged by the backward composite per tile (C_b), x 4 (one count per quarter tile) */
  uint64_t token;         /* B2RWorkspace.status_token of the project phase that filled this block */
  uint64_t reserved[2];
} B2RStatus; /* 64 bytes */

/* Caller-owned memory for one forward->backward context. */
typedef struct B2RWorkspace {
  void* ctx;             /* >= b2r_ctx_bytes(P,W,H); saved until backward */
  size_t ctx_bytes;
  uint32_t* dup_ids;     /* dup_capacity sorted per-tile Gaussian ids; saved until backward */
  uint64_t dup_capacity;
  void* scratch;         /* >= b2r_scratch_bytes(P,W,H,dup_capacity); free after the call returns + stream order */
  size_t scratch_bytes;
  uint64_t* status_mirror; /* optional device-accessible pointer to 2 x uint64 in pinned HOST memory: the project
                              phase stores {num_dups, status_token} there (in that order) so the host can learn the
                              duplicate count by polling, without a stream synchronisation */
  uint64_t status_token;   /* caller-chosen, e.g. a call counter */
  /* Optional (ABI v3): room for the segment table + per-pixel blend-state checkpoints the forward composite stores at
   * every 512-entry cut of a tile's list, >= b2r_checkpoint_bytes(width, height, dup_capacity); saved until backward.
   * With it the backward composite replays every (quarter tile, 512-entry segment) as an independent work item instead
   * of walking a 2000-entry list on one warp.  NULL: lists are not cut (same results, longer serial chains). */
  void* checkpoints;
  size_t checkpoint_bytes;
} B2RWorkspace;

/* A VIEW of a binned scene (ABI v3; SURVEY section 8f-3).  ExAvatar renders one camera five times per training frame
 * (avatar/main/model.py:130-162): the scene Gaussians, the human Gaussians, and cat(scene, human) -- the same
 * projections, tile lists and depth order every time.  Project + bin cat(scene, human) ONCE (b2r_forward_project,
 * b2r_forward_bin) and composite it several times, each view keeping only the Gaussians of an index range, with its own
 * background and its own per-pixel state; b2r_backward_composite accumulates every view's screen-space gradients into
 * one scratch, b2r_backward_project turns them into parameter gradients once. */
typedef struct B2RView {
  uint32_t id_begin, id_end; /* Gaussians [id_begin, id_end) take part; the others are skipped as if absent */
  const float* bg;           /* (3) background of this view; NULL = scene->bg */
  float* final_T;            /* (H*W) per-pixel final transmittance of this view, saved until its backward; NULL = in ctx */
  uint32_t* n_contrib;       /* (H*W) per-pixel position of the last applied list entry; NULL = in ctx */
  void* checkpoints;         /* this view's checkpoint store (see B2RWorkspace.checkpoints); NULL = the workspace's */
  size_t checkpoint_bytes;
  uint32_t skip_below;       /* != 0: tiles whose list holds no Gaussian of index >= skip_below are SKIPPED -- the forward
                                leaves their pixels of `out` (and of final_T / n_contrib) untouched, the backward adds
                                nothing for them.  For cat(scene.detach(), human) with skip_below = #scene: where no human
                                Gaussian reaches a tile the combined render equals the scene-only view (copy its image
                                into `out` first) and nothing of it carries gradient (model.py:117-125). */
  uint32_t reserved;
} B2RView;

typedef struct B2RForwardOutputs {
  float* color;   /* (3,H,W) */
  float* depth;   /* (H,W)  sum z*alpha*T, no background term */
  float* alpha;   /* (H,W)  sum alpha*T */
  int32_t* radii; /* (P)    3-sigma pixel radius, 0 when culled */
} B2RForwardOutputs;

typedef struct B2RBackwardArgs {
  const float* dL_dcolor; /* (3,H,W) */
  const float* dL_ddepth; /* (H,W) or NULL */
  const float* dL_dalpha; /* (H,W) or NULL */
  /* outputs; every element is written (zeros for culled Gaussians).  Any may be NULL. */
  float* dL_dmeans3D;   /* (P,3) */
  float* dL_dmeans2D;   /* (P,3) NDC-scaled screen gradient, z = 0 (module.py:626-629 reads its .grad) */
  float* dL_dshs;       /* (P,M,3) */
  float* dL_dcolors;    /* (P,3) */
  float* dL_dopacities; /* (P) */
  float* dL_dscales;    /* (P,3) */
  float* dL_drotations; /* (P,4) */
  float* dL_dcov3D;     /* (P,6) */
  uint32_t flags;       /* B2R_BWD_ACCUMULATE: outputs += gradient instead of outputs = gradient, so the frames a rank
                           renders in one step sum into a single bucket that is all-reduced once (SURVEY section 8e) */
  uint32_t first_row;   /* Gaussians [0, first_row) are a DETACHED PREFIX: no gradient is written for them and Gaussian i
                           goes to row i - first_row of every output (outputs then have P - first_row rows).  This is
                           ExAvatar's "scene + human" render, cat(scene.detach(), human) (avatar/main/model.py:117-125):
                           the human part of the gradient lands directly in the human bucket.  0 = off. */
  /* Optional fused densification bookkeeping (SURVEY section 8f-1), each (P) or NULL, updated IN PLACE for Gaussians
   * with radii > 0 exactly as ExAvatar does after backward (avatar/common/nets/module.py:155-157,
   * avatar/main/model.py:283-285):  grad_accum += ||dL/dmeans2D.xy||,  count += 1,  radius_max = max(radius_max, radii). */
  float* densify_grad_accum;
  float* densify_count;
  float* densify_radius_max;
  /* Fused skinning (B2RScene.skin_*), each may be NULL:
   *   dL_dskin_xyz (P,3):  gradient w.r.t. the canonical positions,  (M_i[:3,:3])^T Rinv^T dL/dworld_i
   *   dL_dskin_G   (P,12): row-major 3x4 outer product  (Rinv^T dL/dworld_i) [xyz_i, 1]^T ; the joint-transform gradient
   *                        is the plain GEMM  dL/dA[:, :3, :] = W^T G  and  dL/dtrans = sum_i G_i[:, 3].
   * Both follow `flags` (write / accumulate) and `first_row` like every other output. */
  float* dL_dskin_xyz;
  float* dL_dskin_G;
  /* INPUT (ABI v3), (P,3) or NULL: gradient arriving at the posed world positions the forward wrote to
   * B2RScene.skin_means_out (other ExAvatar modules read them: face_mesh_renderer, avatar/main/model.py:172-173); it is
   * added to dL/dworld_i before the skinning transpose, so it reaches dL_dskin_xyz / dL_dskin_G (and dL_dmeans3D). */
  const float* dL_dposed;
  /* (ABI v3) the densification statistics above are updated for Gaussians [0, densify_rows) only; 0 = all.  A merged
   * cat(scene, human) pass keeps ExAvatar's bookkeeping to the scene Gaussians this way (model.py:193). */
  uint32_t densify_rows;
  uint32_t reserved;
} B2RBackwardArgs;
#define B2R_BWD_ACCUMULATE 1u
/* The caller guarantees `bwd_scratch` is all zero on entry; b2r_backward then skips its memset and leaves the scratch
 * all zero again on return (the backward projection kernel clears each row after consuming it).  For callers that
 * keep one scratch buffer alive across steps (plan.py): one graph node and one 48 B/Gaussian memset less per render. */
#define B2R_BWD_SCRATCH_ZEROED 2u

int b2r_abi_version(void);
const char* b2r_strerror(int code);
int b2r_last_cuda_error(void);
/* sizeof() of the ABI structs, for bindings to verify their mirror: 0 B2RScene, 1 B2RStatus, 2 B2RWorkspace,
 * 3 B2RForwardOutputs, 4 B2RBackwardArgs, 5 B2RView; 0 for anything else. */
size_t b2r_sizeof(int which);

size_t b2r_ctx_bytes(int32_t P, int32_t width, int32_t height);
size_t b2r_scratch_bytes(int32_t P, int32_t width, int32_t height, uint64_t dup_capacity);
size_t b2r_backward_scratch_bytes(int32_t P);
size_t b2r_checkpoint_bytes(int32_t width, int32_t height, uint64_t dup_capacity);

/* Phase A: projection, tile counting, tile scan.  Writes radii and B2RStatus.num_dups.  With ws->dup_capacity == 0 it
 * only counts (two-phase use: size the lists from num_dups, then b2r_forward_render).  With a capacity it also prepares
 * the binning (b2r_forward_bin may follow directly); if that capacity then turns out too small (B2RStatus.overflow), run
 * the whole forward again with more room -- the tile counters are consumed. */
int b2r_forward_project(const B2RScene* scene, const B2RWorkspace* ws, int32_t* radii, void* stream);
/* Phase B: duplicate-with-keys, per-tile sort, forward composite (needs phase A on the same ws).  After a count-only
 * phase A it re-derives the per-tile ranges for ws->dup_capacity; after a phase A that was given a capacity it uses the
 * ranges that phase prepared (same capacity expected). */
int b2r_forward_render(const B2RScene* scene, const B2RWorkspace* ws, const B2RForwardOutputs* out, void* stream);
/* Both phases with a capacity chosen up front. */
int b2r_forward(const B2RScene* scene, const B2RWorkspace* ws, const B2RForwardOutputs* out, void* stream);

/* Backward composite + backward projection.  `ws` is the forward's; `bwd_scratch` >= b2r_backward_scratch_bytes(P). */
int b2r_backward(const B2RScene* scene, const B2RWorkspace* ws, const B2RBackwardArgs* args, void* bwd_scratch,
                 size_t bwd_scratch_bytes, void* stream);

/* The same pipeline in separately callable stages (ABI v3), for several views of one binned scene:
 *   b2r_forward_project -> b2r_forward_bin -> b2r_forward_composite (once per view)
 *   b2r_backward_composite (once per view, same scratch) -> b2r_backward_project (once).
 * b2r_forward_render == bin + composite(view = NULL); b2r_backward == composite(view = NULL) + project.
 * b2r_backward_composite reads only dL_dcolor / dL_ddepth / dL_dalpha, `flags` (B2R_BWD_SCRATCH_ZEROED: the caller zeroed
 * the scratch before the FIRST view; later views must pass it too, so nothing is cleared in between) and `first_row`
 * (Gaussians below it receive nothing from this view: the detached prefix of cat(scene.detach(), human)). */
int b2r_forward_bin(const B2RScene* scene, const B2RWorkspace* ws, void* stream);
int b2r_forward_composite(const B2RScene* scene, const B2RWorkspace* ws, const B2RView* view,
                          const B2RForwardOutputs* out, void* stream);
int b2r_backward_composite(const B2RScene* scene, const B2RWorkspace* ws, const B2RView* view, const B2RBackwardArgs* args,
                           void* bwd_scratch, size_t bwd_scratch_bytes, void* stream);
int b2r_backward_project(const B2RScene* scene, const B2RWorkspace* ws, const B2RBackwardArgs* args, void* bwd_scratch,
                         size_t bwd_scratch_bytes, void* stream);

/* present[i] = 1 iff Gaussian i passes the near-plane test (z_view > 0.2). */
int b2r_mark_visible(int32_t P, const float* means3D, const float* viewmatrix, uint8_t* present, void* stream);

/* Measurement hooks (host side).  Kernel ids: 0 project, 1 tile_scan, 2 scatter, 3 sort (all lists, long ones in chunks), 4 sort_merge (chunks of the long lists),
 * 5 composite_fwd, 6 composite_bwd, 7 project_bwd, 8 misc (status reset).  With profiling on, every kernel launch
 * is bracketed by CUDA events on the caller's stream; b2r_profile_read() waits for them and returns the summed
 * milliseconds and launch counts per kernel id (arrays of B2R_NUM_KERNELS).  b2r_launch_count() counts kernel
 * launches made by this library since it was loaded, profiling or not. */
#define B2R_NUM_KERNELS 9
void b2r_profile_enable(int on);
int b2r_profile_read(double* ms_sum, uint64_t* counts, int reset);
uint64_t b2r_launch_count(void);
const char* b2r_kernel_name(int id);

/* Stage-level introspection for parity tests (device pointers into ctx; valid until ctx is reused).
 * geom: P x 12 floats {px, py, A2, B2 | C2, opacity, depth, thr2 | r, g, b, bits};  A2,B2,C2 are the conic
 * pre-scaled for exp2: A2 = -0.5*log2(e)*conic.x, B2 = -log2(e)*conic.y, C2 = -0.5*log2(e)*conic.z.
 * aux: P x 4 int32 {rect_min (x | y<<16), rect_max (x | y<<16), radius, tiles_kept}.
 * ranges: Tn x 2 uint32 [start,end) into dup_ids.  pixel_state: per pixel {final_T (float), n_contrib (uint32)}. */
const float* b2r_ctx_geom(const B2RWorkspace* ws, int32_t P, int32_t width, int32_t height);
const int32_t* b2r_ctx_aux(const B2RWorkspace* ws, int32_t P, int32_t width, int32_t height);
const uint32_t* b2r_ctx_ranges(const B2RWorkspace* ws, int32_t P, int32_t width, int32_t height);
const float* b2r_ctx_final_T(const B2RWorkspace* ws, int32_t P, int32_t width, int32_t height);
const uint32_t* b2r_ctx_n_contrib(const B2RWorkspace* ws, int32_t P, int32_t width, int32_t height);

#ifdef __cplusplus
}
#endif
#endif /* B200RASTER_H_ */
