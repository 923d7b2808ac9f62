// api.cu -- the extern "C" boundary declared in include/b200raster.h.
#include "common.cuh"

using namespace b2r;

namespace {

int validate_scene(const B2RScene* sc) {
  if (!sc) return B2R_E_INVALID;
  if (sc->P < 0 || sc->width <= 0 || sc->height <= 0) return B2R_E_INVALID;
  if (sc->P >= (1 << 29)) return B2R_E_INVALID;  // the splat record carries id in 29 bits (common.cuh Geom)
  if (sc->width > 65535 * TILE || sc->height > 32767 * TILE) return B2R_E_INVALID;
  if (!(sc->tanfovx > 0.f) || !(sc->tanfovy > 0.f)) return B2R_E_INVALID;
  if (!sc->bg || !sc->viewmatrix || !sc->projmatrix || !sc->campos) return B2R_E_INVALID;
  if (sc->sh_rows < 0 || sc->sh_rows > sc->P) return B2R_E_INVALID;  // SH rows of a two-source scene
  if (sc->P > 0) {
    if (!sc->opacities) return B2R_E_INVALID;
    if (sc->skin_xyz) {  // fused skinning replaces means3D
      if (!sc->skin_weights || !sc->skin_joint_mats || !sc->skin_trans) return B2R_E_INVALID;
      if (sc->skin_J <= 0 || sc->skin_J > 64) return B2R_E_INVALID;
      if (sc->skin_cam_Rinv && !sc->skin_cam_t) return B2R_E_INVALID;
    } else if (!sc->means3D) {
      return B2R_E_INVALID;
    }
    if (sc->sh_rows == 0) {
      if ((sc->shs != nullptr) == (sc->colors_precomp != nullptr)) return B2R_E_INVALID;  // exactly one colour source
    } else {  // SH rows [0, sh_rows), colours for the rest
      if (!sc->shs) return B2R_E_INVALID;
      if (sc->sh_rows < sc->P && !sc->colors_precomp) return B2R_E_INVALID;
      if (sc->skin_xyz) return B2R_E_INVALID;
    }
    const bool sr = sc->scales != nullptr && sc->rotations != nullptr;
    if (sr == (sc->cov3D_precomp != nullptr)) return B2R_E_INVALID;                      // exactly one covariance source
    if ((sc->scales != nullptr) != (sc->rotations != nullptr)) return B2R_E_INVALID;
    if (sc->shs) {
      if (sc->sh_degree < 0 || sc->sh_degree > 3) return B2R_E_INVALID;
      if (sc->sh_coeffs < (sc->sh_degree + 1) * (sc->sh_degree + 1)) return B2R_E_INVALID;
      if (sc->sh_coeffs > 16) return B2R_E_INVALID;  // rows are staged through shared memory (project.cu)
    }
  }
  return B2R_OK;
}

int validate_ws(const B2RScene* sc, const B2RWorkspace* ws, bool need_scratch) {
  if (!ws || !ws->ctx) return B2R_E_INVALID;
  if (ws->ctx_bytes < b2r_ctx_bytes(sc->P, sc->width, sc->height)) return B2R_E_WORKSPACE;
  if (ws->dup_capacity > 0xfffffff0ull) return B2R_E_INVALID;  // list positions are 32-bit
  if (need_scratch) {
    if (!ws->scratch) return B2R_E_INVALID;
    if (ws->scratch_bytes < b2r_scratch_bytes(sc->P, sc->width, sc->height, ws->dup_capacity)) return B2R_E_WORKSPACE;
  }
  if (ws->dup_capacity > 0 && !ws->dup_ids) return B2R_E_INVALID;
  if (ws->checkpoints && ws->checkpoint_bytes < b2r_checkpoint_bytes(sc->width, sc->height, ws->dup_capacity)) return B2R_E_WORKSPACE;
  return B2R_OK;
}

// where the backward projection writes the SH gradient.  One colour source: every row needs dL_dshs.  SH rows
// [0, sh_rows) before colour rows: the detached prefix may not cut the SH rows (first_row is 0 or >= sh_rows), and
// dL_dshs may only be NULL when no SH row is past first_row.
bool sh_grad_ok(const B2RScene* sc, const B2RBackwardArgs* a) {
  if (sc->sh_rows == 0) return !(sc->shs && a->dL_dshs == nullptr && sc->P > 0);
  const int64_t fr = (int64_t)a->first_row;
  if (fr > 0 && fr < sc->sh_rows) return false;
  return a->dL_dshs != nullptr || fr >= sc->sh_rows;
}

}  // namespace

extern "C" {

int b2r_abi_version(void) { return B2R_ABI_VERSION; }

const char* b2r_strerror(int code) {
  switch (code) {
    case B2R_OK: return "ok";
    case B2R_E_INVALID: return "invalid argument";
    case B2R_E_WORKSPACE: return "workspace buffer too small";
    case B2R_E_CUDA: return "CUDA launch failed";
    case B2R_E_DUP_OVERFLOW: return "duplicate capacity exceeded";
    default: return "unknown error";
  }
}

int b2r_last_cuda_error(void) { return g_last_cuda_error; }

size_t b2r_sizeof(int which) {
  switch (which) {
    case 0: return sizeof(B2RScene);
    case 1: return sizeof(B2RStatus);
    case 2: return sizeof(B2RWorkspace);
    case 3: return sizeof(B2RForwardOutputs);
    case 4: return sizeof(B2RBackwardArgs);
    case 5: return sizeof(B2RView);
    default: return 0;
  }
}

size_t b2r_ctx_bytes(int32_t P, int32_t width, int32_t height) { return ctx_layout(P, width, height).total; }

size_t b2r_scratch_bytes(int32_t P, int32_t width, int32_t height, uint64_t dup_capacity) {
  return scratch_layout(P, width, height, dup_capacity).total;
}

size_t b2r_backward_scratch_bytes(int32_t P) { return align_up((size_t)(P > 0 ? P : 1) * 12 * sizeof(float)); }

size_t b2r_checkpoint_bytes(int32_t width, int32_t height, uint64_t dup_capacity) {
  const CtxLayout L = ctx_layout(0, width, height);
  const uint32_t ms = max_segments(L.tiles, dup_capacity);
  return seg_table_bytes(ms) + (size_t)ms * CK_REC_BYTES;
}

int b2r_forward_project(const B2RScene* scene, const B2RWorkspace* ws, int32_t* radii, void* stream) {
  int rc = validate_scene(scene);
  if (rc) return rc;
  rc = validate_ws(scene, ws, false);
  if (rc) return rc;
  if (scene->P > 0 && !radii) return B2R_E_INVALID;
  const Ctx cx = resolve(ws, scene->P, scene->width, scene->height);
  return launch_project(*scene, cx, radii, (cudaStream_t)stream);
}

static int forward_render(const B2RScene* scene, const B2RWorkspace* ws, const B2RForwardOutputs* out, bool rescan,
                          void* stream) {
  int rc = validate_scene(scene);
  if (rc) return rc;
  rc = validate_ws(scene, ws, true);
  if (rc) return rc;
  if (!out || !out->color || !out->depth || !out->alpha) return B2R_E_INVALID;
  const Ctx cx = resolve(ws, scene->P, scene->width, scene->height);
  rc = launch_binning(*scene, cx, rescan, (cudaStream_t)stream);
  if (rc) return rc;
  return launch_composite_fwd(*scene, cx, *out, (cudaStream_t)stream);
}

// a view narrows the Gaussian range, swaps the background and redirects the per-pixel state / checkpoint records
static int apply_view(Ctx& cx, const B2RScene* scene, const B2RWorkspace* ws, const B2RView* v) {
  if (!v) return B2R_OK;
  if (v->id_end < v->id_begin || (int64_t)v->id_end > (int64_t)scene->P) return B2R_E_INVALID;
  if ((v->final_T != nullptr) != (v->n_contrib != nullptr)) return B2R_E_INVALID;
  cx.id_begin = v->id_begin;
  cx.id_span = v->id_end - v->id_begin;
  cx.bg = v->bg;
  cx.skip_below = v->skip_below;
  if (v->final_T) { cx.final_T = v->final_T; cx.n_contrib = v->n_contrib; }
  if (v->checkpoints && cx.ckpt) {  // records only; the segment table is the workspace's (one per binned scene)
    const size_t need = seg_table_bytes(cx.max_segs) + (size_t)cx.max_segs * CK_REC_BYTES;
    if (v->checkpoint_bytes < need) return B2R_E_WORKSPACE;
    cx.ckpt = (float*)((char*)v->checkpoints + seg_table_bytes(cx.max_segs));
  }
  (void)ws;
  return B2R_OK;
}

int b2r_forward_bin(const B2RScene* scene, const B2RWorkspace* ws, void* stream) {
  int rc = validate_scene(scene);
  if (rc) return rc;
  rc = validate_ws(scene, ws, true);
  if (rc) return rc;
  const Ctx cx = resolve(ws, scene->P, scene->width, scene->height);
  return launch_binning(*scene, cx, false, (cudaStream_t)stream);
}

int b2r_forward_composite(const B2RScene* scene, const B2RWorkspace* ws, const B2RView* view,
                          const B2RForwardOutputs* out, void* stream) {
  int rc = validate_scene(scene);
  if (rc) return rc;
  rc = validate_ws(scene, ws, false);
  if (rc) return rc;
  if (!out || !out->color || !out->depth || !out->alpha) return B2R_E_INVALID;
  Ctx cx = resolve(ws, scene->P, scene->width, scene->height);
  rc = apply_view(cx, scene, ws, view);
  if (rc) return rc;
  return launch_composite_fwd(*scene, cx, *out, (cudaStream_t)stream);
}

int b2r_forward_render(const B2RScene* scene, const B2RWorkspace* ws, const B2RForwardOutputs* out, void* stream) {
  return forward_render(scene, ws, out, true, stream);
}

int b2r_forward(const B2RScene* scene, const B2RWorkspace* ws, const B2RForwardOutputs* out, void* stream) {
  if (!out) return B2R_E_INVALID;
  int rc = b2r_forward_project(scene, ws, out->radii, stream);
  if (rc) return rc;
  return forward_render(scene, ws, out, false, stream);
}

int b2r_backward(const B2RScene* scene, const B2RWorkspace* ws, const B2RBackwardArgs* args, void* bwd_scratch,
                 size_t bwd_scratch_bytes, void* stream) {
  int rc = validate_scene(scene);
  if (rc) return rc;
  rc = validate_ws(scene, ws, false);
  if (rc) return rc;
  if (!args || !args->dL_dcolor || !bwd_scratch) return B2R_E_INVALID;
  if (!sh_grad_ok(scene, args)) return B2R_E_INVALID;
  if (bwd_scratch_bytes < b2r_backward_scratch_bytes(scene->P)) return B2R_E_WORKSPACE;
  if ((int64_t)args->first_row > (int64_t)scene->P) return B2R_E_INVALID;
  if (args->dL_dposed && !scene->skin_xyz) return B2R_E_INVALID;
  const Ctx cx = resolve(ws, scene->P, scene->width, scene->height);
  float* gacc = (float*)bwd_scratch;
  rc = launch_composite_bwd(*scene, cx, *args, gacc, (cudaStream_t)stream);
  if (rc) return rc;
  return launch_project_bwd(*scene, cx, *args, gacc, (cudaStream_t)stream);
}

int b2r_backward_composite(const B2RScene* scene, const B2RWorkspace* ws, const B2RView* view, const B2RBackwardArgs* args,
                           void* bwd_scratch, size_t bwd_scratch_bytes, void* stream) {
  int rc = validate_scene(scene);
  if (rc) return rc;
  rc = validate_ws(scene, ws, false);
  if (rc) return rc;
  if (!args || !args->dL_dcolor || !bwd_scratch) return B2R_E_INVALID;
  if (bwd_scratch_bytes < b2r_backward_scratch_bytes(scene->P)) return B2R_E_WORKSPACE;
  if ((int64_t)args->first_row > (int64_t)scene->P) return B2R_E_INVALID;
  Ctx cx = resolve(ws, scene->P, scene->width, scene->height);
  rc = apply_view(cx, scene, ws, view);
  if (rc) return rc;
  return launch_composite_bwd(*scene, cx, *args, (float*)bwd_scratch, (cudaStream_t)stream);
}

int b2r_backward_project(const B2RScene* scene, const B2RWorkspace* ws, const B2RBackwardArgs* args, void* bwd_scratch,
                         size_t bwd_scratch_bytes, void* stream) {
  int rc = validate_scene(scene);
  if (rc) return rc;
  rc = validate_ws(scene, ws, false);
  if (rc) return rc;
  if (!args || !bwd_scratch) return B2R_E_INVALID;
  if (!sh_grad_ok(scene, args)) return B2R_E_INVALID;
  if (bwd_scratch_bytes < b2r_backward_scratch_bytes(scene->P)) return B2R_E_WORKSPACE;
  if ((int64_t)args->first_row > (int64_t)scene->P) return B2R_E_INVALID;
  if (args->dL_dposed && !scene->skin_xyz) return B2R_E_INVALID;
  const Ctx cx = resolve(ws, scene->P, scene->width, scene->height);
  return launch_project_bwd(*scene, cx, *args, (const float*)bwd_scratch, (cudaStream_t)stream);
}

int b2r_mark_visible(int32_t P, const float* means3D, const float* viewmatrix, uint8_t* present, void* stream) {
  if (P < 0 || (P > 0 && (!means3D || !present)) || !viewmatrix) return B2R_E_INVALID;
  return launch_mark_visible(P, means3D, viewmatrix, present, (cudaStream_t)stream);
}

const float* b2r_ctx_geom(const B2RWorkspace* ws, int32_t P, int32_t width, int32_t height) {
  return (const float*)((const char*)ws->ctx + ctx_layout(P, width, height).geom);
}
const int32_t* b2r_ctx_aux(const B2RWorkspace* ws, int32_t P, int32_t width, int32_t height) {
  return (const int32_t*)((const char*)ws->ctx + ctx_layout(P, width, height).aux);
}
const uint32_t* b2r_ctx_ranges(const B2RWorkspace* ws, int32_t P, int32_t width, int32_t height) {
  return (const uint32_t*)((const char*)ws->ctx + ctx_layout(P, width, height).ranges);
}
const float* b2r_ctx_final_T(const B2RWorkspace* ws, int32_t P, int32_t width, int32_t height) {
  return (const float*)((const char*)ws->ctx + ctx_layout(P, width, height).final_T);
}
const uint32_t* b2r_ctx_n_contrib(const B2RWorkspace* ws, int32_t P, int32_t width, int32_t height) {
  return (const uint32_t*)((const char*)ws->ctx + ctx_layout(P, width, height).n_contrib);
}

}  // extern "C"
