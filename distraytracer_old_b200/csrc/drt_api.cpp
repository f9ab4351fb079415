// C ABI (include/drt.h) over the host interpreter/flattener and the device renderer.
#include "../../include/drt.h"
#include "renderer.h"
#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <initializer_list>
#include <memory>
#include <stdexcept>
#include <zlib.h>

using namespace drt;

namespace drt { double hostPhiloxU01(uint64_t seed, uint32_t stream, uint32_t a, uint32_t b, uint32_t c, uint32_t d); }

typedef std::chrono::duration<double, std::milli> MsD;
static double wallMs() { return MsD(std::chrono::steady_clock::now().time_since_epoch()).count(); }

struct drt_ctx {
  drt_config cfg;
  std::unique_ptr<HostScene> scene;
  std::unique_ptr<Renderer> renderer;
  std::string err, texDir, dataDir;
  drt_image_loader_fn loader = nullptr; void* loaderUser = nullptr;
  int spp = 0; long long photons = -1;
  bool finalized = false; double msUpload = 0;
  void freshScene() {
    scene.reset(new HostScene(cfg.cols, cfg.rows)); scene->setSeed(cfg.seed); finalized = false;
    if (!texDir.empty()) scene->setTexDir(texDir);
    if (renderer) {     // median-split BVHs over large object lists are ordered on the device (csrc/refbvh.cuh); DRT_REFBVH_MIN=<objects> moves the threshold
      Renderer* r = renderer.get(); HostScene* sc = scene.get(); const char* e = getenv("DRT_REFBVH_MIN");
      scene->setBvhOrderer([r, sc](int n, const double* keys, int32_t* ord) { double ms = 0; const bool ok = r->orderBvh(n, keys, ord, &ms); sc->msBvhOrderDevice += ms; return ok; }, e ? atoi(e) : 4096);
    }
    if (loader) { drt_image_loader_fn fn = loader; void* u = loaderUser;
      scene->setImageLoader([fn, u](const std::string& name, HostImage& out) { int32_t w = 0, h = 0; const int32_t* px = nullptr; if (fn(u, name.c_str(), &w, &h, &px) != 0 || !px) return false; out.w = w; out.h = h; out.px.assign(px, px + (size_t)w * h); return true; }); }
  }
};

static void toStats(const RenderStats& r, drt_stats* s) {
  if (!s) return;
  s->rays_primary = r.primary; s->rays_shadow = r.shadow; s->rays_reflect = r.reflect; s->rays_refract = r.refract; s->rays_photon = r.photonSeg;
  s->box_tests = r.boxTests; s->prim_tests = r.primTests; s->photons_stored = r.photonsStored; s->kernel_launches = r.kernelLaunches; s->box_tests_closest = r.boxTestsClosest; s->prim_tests_closest = r.primTestsClosest;
  s->ms_trace = r.msTrace; s->ms_shade = r.msShade; s->ms_light = r.msLight; s->ms_other = r.msOther; s->ms_total = r.msTotal;
  s->rays_deferred = r.deferred; s->frame_retries = r.retries; s->host_syncs = r.hostSyncs;
}
#define NEED_DEV(ctx) if ((ctx) && !(ctx)->renderer) { (ctx)->err = "host-only context: no CUDA device, and this library has no CPU fallback"; return DRT_ERR_NO_DEVICE; }
#define GUARD(ctx, body, code) if (!(ctx)) return DRT_ERR_BAD_ARG; try { body; return DRT_OK; } catch (std::exception& e) { (ctx)->err = e.what(); return code; }

extern "C" {

int drt_create(const drt_config* cfg, drt_ctx** out) {
  if (!cfg || !out) return DRT_ERR_BAD_ARG;
  *out = nullptr; drt_ctx* c = new drt_ctx; c->cfg = *cfg;
  if (c->cfg.cols <= 0) c->cfg.cols = 300; if (c->cfg.rows <= 0) c->cfg.rows = 300;
  if (cfg->device >= 0) {     // device < 0: host-only context (interpreter + flattener); every render entry point then fails with DRT_ERR_NO_DEVICE
    try { c->renderer.reset(new Renderer(cfg->device)); } catch (std::exception& e) { fprintf(stderr, "drt_create: %s\n", e.what()); delete c; return DRT_ERR_NO_DEVICE; }
    if (cfg->batch_rays > 0) c->renderer->setBatchRays(cfg->batch_rays);
    c->renderer->setCounters(cfg->counters != 0);
  }
  c->freshScene(); *out = c; return DRT_OK;
}
void drt_destroy(drt_ctx* ctx) { delete ctx; }
const char* drt_last_error(drt_ctx* ctx) { return ctx ? ctx->err.c_str() : "null context"; }

int drt_set_image_loader(drt_ctx* ctx, drt_image_loader_fn fn, void* user) { GUARD(ctx, { ctx->loader = fn; ctx->loaderUser = user; ctx->freshScene(); }, DRT_ERR_SCENE) }
int drt_set_texture_dir(drt_ctx* ctx, const char* dir) { GUARD(ctx, { ctx->texDir = dir ? dir : ""; if (ctx->scene) ctx->scene->setTexDir(ctx->texDir); }, DRT_ERR_SCENE) }
int drt_scene_reset(drt_ctx* ctx) { GUARD(ctx, ctx->freshScene(), DRT_ERR_SCENE) }
int drt_scene_command(drt_ctx* ctx, const char* line) { GUARD(ctx, { if (!line) throw std::runtime_error("null line"); ctx->scene->command(line); }, DRT_ERR_SCENE) }
int drt_scene_load_cli(drt_ctx* ctx, const char* file, const char* data_dir) {
  GUARD(ctx, { if (!file || !data_dir) throw std::runtime_error("null path"); ctx->freshScene(); ctx->scene->loadFile(file, data_dir); }, DRT_ERR_SCENE)
}
int drt_scene_override(drt_ctx* ctx, int32_t spp, int64_t photons) { GUARD(ctx, { ctx->spp = spp; ctx->photons = photons; }, DRT_ERR_SCENE) }
int drt_scene_finalize(drt_ctx* ctx, int32_t accel_mode) {
  GUARD(ctx, {
    if (accel_mode < 0 || accel_mode > 2) throw std::runtime_error("unknown acceleration mode (use DRT_ACCEL_REFERENCE, DRT_ACCEL_REFERENCE_FAST or DRT_ACCEL_LBVH)");
    ctx->scene->overrideSpp(ctx->spp); ctx->scene->overridePhotons(ctx->photons);
    ctx->scene->finalize();
    if (ctx->renderer) { ctx->renderer->setAccelMode(accel_mode); const double t0 = wallMs(); ctx->renderer->upload(*ctx->scene); ctx->msUpload = wallMs() - t0; ctx->finalized = true; } }, DRT_ERR_SCENE)
}
int drt_scene_reupload(drt_ctx* ctx) { NEED_DEV(ctx) GUARD(ctx, { if (!ctx->finalized) throw std::runtime_error("scene not finalized"); ctx->renderer->upload(*ctx->scene, true); }, DRT_ERR_STATE) }
int drt_accel_info(drt_ctx* ctx, double* out4) { NEED_DEV(ctx) GUARD(ctx, { if (!ctx->finalized || !out4) throw std::runtime_error("scene not finalized"); ctx->renderer->accelInfo(out4); }, DRT_ERR_STATE) }
int drt_build_info(drt_ctx* ctx, double* o) {
  GUARD(ctx, { if (!o) throw std::runtime_error("null output"); const HostScene& s = *ctx->scene;
    o[0] = s.msParse; o[1] = s.msBvhOrder; o[2] = s.msBvhOrderDevice; o[3] = s.msBvhShape; o[4] = s.msFinalize; o[5] = (double)s.bvhDeviceBuilds; o[6] = (double)s.bvhObjects; o[7] = ctx->msUpload; }, DRT_ERR_SCENE)
}
int drt_bvh_order(drt_ctx* ctx, int32_t n, const double* keys, int32_t* ord, int32_t on_device) {
  if (on_device) { NEED_DEV(ctx) }
  GUARD(ctx, { if (n < 0 || (n > 0 && (!keys || !ord))) throw std::runtime_error("bad order buffers");
    if (!on_device) HostScene::refOrderHost(n, keys, ord);
    else { double ms = 0; if (!ctx->renderer->orderBvh(n, keys, ord, &ms)) throw std::runtime_error("the device declined this key set (fewer than 2 objects, NaN keys or undefined spans)"); } }, DRT_ERR_SCENE)
}
int64_t drt_lbvh_probe(drt_ctx* ctx, int32_t fast_index, int32_t which, double* box6, double* verts9, int32_t* prim_serial, int32_t* links2, double* boxes12, int64_t cap_tris) {
  if (!ctx) return DRT_ERR_BAD_ARG; if (which) { NEED_DEV(ctx) }
  try {
    if (!ctx->finalized && which) throw std::runtime_error("scene not finalized");
    ctx->scene->finalize(); const HostScene& hs = *ctx->scene; std::vector<FTri> tris; std::vector<FNode> nodes; int32_t info[4] = {0, 0, 0, 0}; long long n = -1; int k = 0;
    for (const FBvh& B : hs.bvhs) if (B.fast && k++ == fast_index) {
      if (box6) { for (int i = 0; i < 3; ++i) { box6[i] = B.bmin[i]; box6[3 + i] = B.bmax[i]; } }
      if (!which) { tris.assign(hs.tris.begin() + B.triStart, hs.tris.begin() + B.triStart + B.triCount); n = B.triCount; info[0] = B.triStart; }
      else n = ctx->renderer->probeFastBvh(fast_index, tris, nodes, info);
      break;
    }
    if (n < 0) return DRT_ERR_BAD_ARG;            // no such fast BVH
    for (long long i = 0; i < n && i < cap_tris; ++i) { if (verts9) std::memcpy(verts9 + 9 * i, tris[i].v, 72); if (prim_serial) prim_serial[i] = hs.prims[tris[i].prim].serial; }
    // links: >= 0 inner node (relative to the BVH's first LBVH node), < 0: -(1 + leaf number), leaf j = triangles 4j .. 4j+3 of the resident order
    if (n <= cap_tris) for (size_t i = 0; i < nodes.size(); ++i) { const FNode& N = nodes[i];
      if (links2) { links2[2 * i] = N.left >= 0 ? N.left - info[1] : -(1 + ((N.triL >> 3) - info[0]) / 4); links2[2 * i + 1] = N.right >= 0 ? N.right - info[1] : -(1 + ((N.triR >> 3) - info[0]) / 4); }
      if (boxes12) std::memcpy(boxes12 + 12 * i, N.lmin, 96); }
    return n;
  } catch (std::exception& e) { ctx->err = e.what(); return DRT_ERR_SCENE; }
}
int drt_scene_counts(drt_ctx* ctx, int64_t* o) {
  GUARD(ctx, { if (!o) throw std::runtime_error("null output"); ctx->scene->finalize(); const HostScene& s = *ctx->scene; std::memset(o, 0, 8 * sizeof(int64_t));
    o[0] = (int64_t)s.tris.size(); for (const FBvh& B : s.bvhs) if (B.fast) { ++o[1]; o[3] += B.triCount; } for (const FPrim& P : s.prims) if (P.pad0 >= 0) ++o[2];
    o[4] = (int64_t)s.children.size(); o[5] = (int64_t)s.pdata.size(); }, DRT_ERR_SCENE)
}
int drt_scene_info(drt_ctx* ctx, int32_t* o) {
  GUARD(ctx, { ctx->scene->finalize(); const HostScene& s = *ctx->scene; std::memset(o, 0, 16 * sizeof(int32_t));
    o[0] = s.g.cols; o[1] = s.g.rows; o[2] = s.g.spp; o[3] = (int)s.top.size(); o[4] = (int)s.lights.size(); o[5] = (int)s.prims.size(); o[6] = (int)s.instances.size(); o[7] = s.g.photonKind;
    o[8] = (int)s.shaders.size(); o[9] = (int)s.nodes.size(); o[10] = (int)s.xforms.size(); o[11] = (int)s.lists.size(); o[12] = (int)s.bvhs.size(); o[13] = (int)s.images.size(); o[14] = (int)s.warnings.size(); o[15] = s.g.numPhotonsCast; }, DRT_ERR_SCENE)
}

int drt_emit_photons(drt_ctx* ctx, drt_stats* stats) { NEED_DEV(ctx) GUARD(ctx, { if (!ctx->finalized) throw std::runtime_error("scene not finalized"); RenderStats rs; std::memset(&rs, 0, sizeof(rs)); ctx->renderer->emitPhotons(&rs); toStats(rs, stats); }, DRT_ERR_CUDA) }
int drt_emit_photons_range(drt_ctx* ctx, int64_t i0, int64_t i1, drt_stats* stats) { NEED_DEV(ctx) GUARD(ctx, { if (!ctx->finalized) throw std::runtime_error("scene not finalized"); RenderStats rs; std::memset(&rs, 0, sizeof(rs)); ctx->renderer->emitPhotonsRange(i0, i1, &rs); toStats(rs, stats); }, DRT_ERR_CUDA) }
int64_t drt_photons_export_device(drt_ctx* ctx, double* dst, int64_t cap) { if (!ctx) return DRT_ERR_BAD_ARG; NEED_DEV(ctx) try { return ctx->renderer->exportPhotonsDevice(dst, cap); } catch (std::exception& e) { ctx->err = e.what(); return DRT_ERR_CUDA; } }
int drt_photons_build_device(drt_ctx* ctx, const double* src, int64_t n, drt_stats* stats) { NEED_DEV(ctx) GUARD(ctx, { if (!ctx->finalized) throw std::runtime_error("scene not finalized"); RenderStats rs; std::memset(&rs, 0, sizeof(rs)); ctx->renderer->buildPhotonsFromDevice(src, n, &rs); toStats(rs, stats); }, DRT_ERR_CUDA) }
int drt_photon_probe(drt_ctx* ctx, int64_t n, const double* pts, double* out5) { NEED_DEV(ctx) GUARD(ctx, { if (!ctx->finalized) throw std::runtime_error("scene not finalized"); if (n < 0 || !pts || !out5) throw std::runtime_error("bad probe buffers"); ctx->renderer->probePhotons(n, pts, out5); }, DRT_ERR_CUDA) }
int drt_render_aov(drt_ctx* ctx, int32_t* argb, int32_t* hp, int32_t* hi, double* rgb, double* t, drt_stats* stats) {
  NEED_DEV(ctx) GUARD(ctx, { if (!ctx->finalized) throw std::runtime_error("scene not finalized"); RenderStats rs; std::memset(&rs, 0, sizeof(rs)); ctx->renderer->renderToHost(argb, hp, hi, rgb, t, &rs); toStats(rs, stats); }, DRT_ERR_CUDA)
}
int drt_render(drt_ctx* ctx, int32_t* argb, drt_stats* stats) { return drt_render_aov(ctx, argb, nullptr, nullptr, nullptr, nullptr, stats); }
int drt_render_device(drt_ctx* ctx, int64_t pix0, int64_t pix1, int32_t* argb_dev, drt_stats* stats) {
  NEED_DEV(ctx) GUARD(ctx, { if (!ctx->finalized) throw std::runtime_error("scene not finalized"); RenderStats rs; std::memset(&rs, 0, sizeof(rs)); RenderOutputs o; std::memset(&o, 0, sizeof(o)); o.argb = argb_dev;
    ctx->renderer->renderRange(pix0, pix1, o, &rs); toStats(rs, stats); }, DRT_ERR_CUDA)
}

int drt_render_device_chunks(drt_ctx* ctx, int32_t world, int32_t rank, int32_t chunk_rows, int32_t* argb_dev, drt_stats* stats) {
  NEED_DEV(ctx) GUARD(ctx, { if (!ctx->finalized) throw std::runtime_error("scene not finalized"); if (world < 1 || rank < 0 || rank >= world || chunk_rows < 1) throw std::runtime_error("bad partition");
    RenderStats rs; std::memset(&rs, 0, sizeof(rs)); RenderOutputs o; std::memset(&o, 0, sizeof(o)); o.argb = argb_dev;
    ctx->renderer->renderChunks(0, 0, world, rank, chunk_rows, o, &rs); toStats(rs, stats); }, DRT_ERR_CUDA)
}

int drt_comm_unique_id(uint8_t* id128) { if (!id128) return DRT_ERR_BAD_ARG; try { Renderer::commUniqueId(id128); return DRT_OK; } catch (std::exception& e) { fprintf(stderr, "drt_comm_unique_id: %s\n", e.what()); return DRT_ERR_CUDA; } }
int drt_comm_init(drt_ctx* ctx, const uint8_t* id128, int32_t world, int32_t rank) { NEED_DEV(ctx) GUARD(ctx, { if (!id128 && world > 1) throw std::runtime_error("null id"); unsigned char z[128] = {0}; ctx->renderer->commInit(id128 ? id128 : z, world, rank); }, DRT_ERR_CUDA) }
int drt_comm_destroy(drt_ctx* ctx) { NEED_DEV(ctx) GUARD(ctx, ctx->renderer->commDestroy(), DRT_ERR_CUDA) }
int drt_render_distributed(drt_ctx* ctx, int32_t* argb_host, int32_t* argb_dev, int32_t chunk_rows, int32_t reemit, drt_stats* stats) {
  NEED_DEV(ctx) GUARD(ctx, { if (!ctx->finalized) throw std::runtime_error("scene not finalized"); RenderStats rs; std::memset(&rs, 0, sizeof(rs));
    ctx->renderer->renderDistributed(argb_host, argb_dev, chunk_rows, reemit != 0, &rs); toStats(rs, stats); }, DRT_ERR_CUDA)
}

int64_t drt_dist_rank_pixels(int32_t cols, int32_t rows, int32_t world, int32_t rank, int32_t chunk_rows) { if (cols < 1 || rows < 1 || world < 1 || rank < 0 || rank >= world || chunk_rows < 1) return DRT_ERR_BAD_ARG; return Renderer::distRankPixels(cols, rows, world, rank, chunk_rows); }
int64_t drt_dist_abs_pixel(int32_t cols, int32_t rows, int32_t world, int32_t rank, int32_t chunk_rows, int64_t compact) { if (cols < 1 || rows < 1 || world < 1 || rank < 0 || rank >= world || chunk_rows < 1 || compact < 0) return DRT_ERR_BAD_ARG; return Renderer::distAbsPixel(cols, rows, world, rank, chunk_rows, compact); }
int drt_dist_photon_range(int64_t n, int32_t world, int32_t rank, int64_t* out2) { if (!out2 || world < 1 || rank < 0 || rank >= world || n < 0) return DRT_ERR_BAD_ARG; long long o[2]; Renderer::distPhotonRange(n, world, rank, o); out2[0] = o[0]; out2[1] = o[1]; return DRT_OK; }

int drt_scene_refine(drt_ctx* ctx) { if (!ctx) return DRT_ERR_BAD_ARG; return ctx->scene->refine ? 1 : 0; }
int32_t drt_refine_steps(int32_t cols, int32_t rows, int32_t* steps16) {          // myScene.setRefine (:796-803)
  if (cols < 1 || rows < 1) return 0;
  const int refIDX = (int)(std::log10(.5 * (cols + rows) / 16.0) / std::log10(2.0));
  if (refIDX < 0 || refIDX > 15) return 0;                                         // `new int[refIDX + 1]` / pow2[] of the reference
  for (int i = refIDX; i >= 0; --i) if (steps16) steps16[refIDX - i] = 1 << i;
  return refIDX + 1;
}
int drt_refine_pass(const int32_t* full, int32_t cols, int32_t rows, int32_t step, int32_t* out) {     // the pass loop of draw() + writePxlSpan
  if (!full || !out || cols < 1 || rows < 1 || step < 1) return DRT_ERR_BAD_ARG;
  for (int row = 0; row < rows; row += step) for (int col = 0; col < cols; col += step) {
    const int32_t c = full[(size_t)row * cols + col]; const int rEnd = std::min(row + step, rows), cEnd = std::min(col + step, cols);
    for (int r = row; r < rEnd; ++r) for (int q = col; q < cEnd; ++q) out[(size_t)r * cols + q] = c;
  }
  return DRT_OK;
}

// PNG (8-bit RGB, zlib deflate) -- PImage.save of an RGB image
int drt_save_png(const char* path, const int32_t* argb, int32_t cols, int32_t rows) {
  if (!path || !argb || cols <= 0 || rows <= 0) return DRT_ERR_BAD_ARG;
  std::vector<unsigned char> raw((size_t)rows * (1 + 3 * (size_t)cols));
  for (int y = 0; y < rows; ++y) { unsigned char* r = &raw[(size_t)y * (1 + 3 * cols)]; r[0] = 0;
    for (int x = 0; x < cols; ++x) { uint32_t c = (uint32_t)argb[(size_t)y * cols + x]; r[1 + 3 * x] = (c >> 16) & 255; r[2 + 3 * x] = (c >> 8) & 255; r[3 + 3 * x] = c & 255; } }
  uLongf zlen = compressBound(raw.size()); std::vector<unsigned char> z(zlen);
  if (compress2(z.data(), &zlen, raw.data(), raw.size(), 6) != Z_OK) return DRT_ERR_BAD_ARG;
  FILE* f = fopen(path, "wb"); if (!f) return DRT_ERR_BAD_ARG;
  auto be32 = [](unsigned char* p, uint32_t v) { p[0] = v >> 24; p[1] = v >> 16; p[2] = v >> 8; p[3] = v; };
  auto chunk = [&](const char* type, const unsigned char* data, uint32_t len) { unsigned char hd[8]; be32(hd, len); memcpy(hd + 4, type, 4); fwrite(hd, 1, 8, f); if (len) fwrite(data, 1, len, f);
    uLong crc = crc32(0, (const Bytef*)type, 4); if (len) crc = crc32(crc, data, len); unsigned char c4[4]; be32(c4, (uint32_t)crc); fwrite(c4, 1, 4, f); };
  static const unsigned char sig[8] = {137, 80, 78, 71, 13, 10, 26, 10}; fwrite(sig, 1, 8, f);
  unsigned char ihdr[13]; be32(ihdr, cols); be32(ihdr + 4, rows); ihdr[8] = 8; ihdr[9] = 2; ihdr[10] = 0; ihdr[11] = 0; ihdr[12] = 0;
  chunk("IHDR", ihdr, 13); chunk("IDAT", z.data(), (uint32_t)zlen); chunk("IEND", nullptr, 0); fclose(f); return DRT_OK;
}

int drt_trace_rays(drt_ctx* ctx, int64_t n, const double* org, const double* dir, int32_t* ids2, double* t) { NEED_DEV(ctx) GUARD(ctx, { if (!ctx->finalized) throw std::runtime_error("scene not finalized"); ctx->renderer->traceRays(n, org, dir, ids2, t); }, DRT_ERR_CUDA) }
// shared argument checks of the ray queries: device, finalized scene, n >= 0, required pointers present when there are rays
static int queryArgs(drt_ctx* ctx, int64_t n, std::initializer_list<const void*> required) {
  if (!ctx) return DRT_ERR_BAD_ARG;
  NEED_DEV(ctx)
  if (!ctx->finalized) { ctx->err = "scene not finalized"; return DRT_ERR_STATE; }
  if (n < 0) { ctx->err = "negative ray count"; return DRT_ERR_BAD_ARG; }
  if (n > 0) for (const void* p : required) if (!p) { ctx->err = "a required ray or output buffer is NULL"; return DRT_ERR_BAD_ARG; }
  return DRT_OK;
}
int drt_query_closest(drt_ctx* ctx, int64_t n, const double* org3, const double* dir3, const double* tmax, int32_t* ids2, double* t, double* pos3, double* nrm3, drt_stats* stats) {
  if (const int rc = queryArgs(ctx, n, {org3, dir3, ids2, t})) return rc;
  GUARD(ctx, { RenderStats rs; ctx->renderer->queryClosest(n, org3, dir3, tmax, ids2, t, pos3, nrm3, &rs); toStats(rs, stats); }, DRT_ERR_CUDA)
}
int drt_query_occluded(drt_ctx* ctx, int64_t n, const double* org3, const double* dir3, const double* dist, uint8_t* occluded, drt_stats* stats) {
  if (const int rc = queryArgs(ctx, n, {org3, dir3, dist, occluded})) return rc;
  GUARD(ctx, { RenderStats rs; ctx->renderer->queryOccluded(n, org3, dir3, dist, occluded, &rs); toStats(rs, stats); }, DRT_ERR_CUDA)
}
int drt_eval_texture(drt_ctx* ctx, int32_t serial, int64_t n, const double* hl, const double* fl, double* rgb) {
  NEED_DEV(ctx) GUARD(ctx, { if (!ctx->finalized) throw std::runtime_error("scene not finalized"); if (serial < 0 || serial >= (int)ctx->scene->shaderOfSerial.size()) throw std::runtime_error("no such shader"); ctx->renderer->evalTexture(ctx->scene->shaderOfSerial[serial], n, hl, fl ? fl : hl, rgb); }, DRT_ERR_CUDA)
}
int64_t drt_dump_bvh(drt_ctx* ctx, int32_t topIdx, int32_t* out, int64_t cap, double* box6) {
  if (!ctx) return DRT_ERR_BAD_ARG;
  try { std::vector<int32_t> v; double b[6] = {0, 0, 0, 0, 0, 0}; ctx->scene->finalize(); ctx->scene->dumpBvh(topIdx, v, b); if (v.empty()) return -1;
    for (size_t i = 0; i < v.size() && (int64_t)i < cap; ++i) out[i] = v[i]; if (box6) memcpy(box6, b, sizeof(b)); return (int64_t)v.size(); } catch (std::exception& e) { ctx->err = e.what(); return DRT_ERR_SCENE; }
}
int drt_obj_ctm(drt_ctx* ctx, int32_t topIdx, double* out16) {
  GUARD(ctx, { ctx->scene->finalize(); if (topIdx < 0 || topIdx >= (int)ctx->scene->top.size()) throw std::runtime_error("index"); memcpy(out16, ctx->scene->xforms[ctx->scene->top[topIdx].xform].m, 128); }, DRT_ERR_SCENE)
}
double drt_sample_u01(uint64_t seed, uint32_t stream, uint32_t a, uint32_t b, uint32_t c, uint32_t d) { return hostPhiloxU01(seed, stream, a, b, c, d); }
int64_t drt_get_photons(drt_ctx* ctx, double* out6, int64_t cap) { if (!ctx) return DRT_ERR_BAD_ARG; NEED_DEV(ctx) try { return ctx->renderer->getPhotons(out6, cap); } catch (std::exception& e) { ctx->err = e.what(); return DRT_ERR_CUDA; } }

}  // extern "C"
