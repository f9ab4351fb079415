/* drt.h -- C ABI of the B200 wavefront renderer that replaces the render path of
 * jturner65/distRayTracer_old (package rayTracerDistAccelShdPhtnMap).
 *
 * The reference has no plugin/FFI seam; its render path sits behind
 *   myRTFileReader.readRTFile()  (myRTFileReader.java:15-349, one switch per .cli line, `write` renders, :86-93)
 *   myScene.initRender()/draw()  (myScene.java:1096-1099, :1481-1531, :1408-1443, :1589-1643, :1704-1753)
 * whose only product is PImage.pixels (int ARGB, row-major, alpha 0xFF; myObjShader.java:671).
 * A Java host binds these entry points through JNI or Panama FFM (see INTEGRATION.md): the interpreter loop
 * forwards every .cli line to drt_scene_command(), `write` calls drt_scene_finalize() + drt_render().
 *
 * Conventions: every function returns 0 on success or a negative drt_status; the message is available
 * from drt_last_error(). There is NO CPU fallback: without a CUDA device drt_create fails with DRT_ERR_NO_DEVICE.
 * One context is used by one host thread at a time (the reference is single threaded).
 * The caller owns all input strings/arrays (copied during the call) and all output buffers.
 */
#ifndef DRT_H
#define DRT_H
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

typedef struct drt_ctx drt_ctx;

typedef enum { DRT_OK = 0, DRT_ERR_NO_DEVICE = -1, DRT_ERR_BAD_ARG = -2, DRT_ERR_SCENE = -3, DRT_ERR_CUDA = -4, DRT_ERR_STATE = -5 } drt_status;

/* acceleration-structure / traversal modes (drt_scene_finalize) */
enum { DRT_ACCEL_REFERENCE = 0,   /* reference-topology BVH, reference traversal order and box rules (parity mode) */
       DRT_ACCEL_REFERENCE_FAST = 1, /* same topology and hit rules, near-first ordered traversal with global pruning */
       DRT_ACCEL_LBVH = 2 };      /* GPU-built 30-bit-Morton LBVH over triangle meshes (performance mode) */

typedef struct drt_config {
  int32_t device;          /* CUDA ordinal; < 0 = host-only context (interpret + flatten only, every render call fails) */
  int32_t cols, rows;      /* output resolution (the reference hard-codes 300x300, DistRayTracer.java:15-16) */
  int32_t counters;        /* !=0: count box / primitive tests (slower) */
  uint64_t seed;           /* sampler seed (replaces the reference's unseeded ThreadLocalRandom) */
  int64_t batch_rays;      /* primary rays per wavefront batch, 0 = default */
} drt_config;

typedef struct drt_stats {
  uint64_t rays_primary, rays_shadow, rays_reflect, rays_refract, rays_photon;  /* logical rays, not the reference's copy count (myRay.java:30) */
  uint64_t box_tests, prim_tests, photons_stored, kernel_launches;
  uint64_t box_tests_closest, prim_tests_closest;                                 /* the closest-hit (k_trace) share of the two counters above */
  double ms_trace, ms_shade, ms_light, ms_other, ms_total;                      /* CUDA-event times of the call */
  uint64_t rays_deferred, frame_retries, host_syncs;                             /* work the lean kernels handed to the generic pass; frames re-rendered after a failed speculation; host<->device syncs of the call */
} drt_stats;

/* host image decoder: PApplet.loadImage(name).pixels (myRTFileReader.java:133,265). Return 0 and fill w,h and a
 * pointer to w*h ARGB ints that stays valid until the callback returns to the library (it copies). */
typedef int (*drt_image_loader_fn)(void* user, const char* name, int32_t* w, int32_t* h, const int32_t** argb);

int drt_create(const drt_config* cfg, drt_ctx** out);
void drt_destroy(drt_ctx* ctx);
const char* drt_last_error(drt_ctx* ctx);

/* ---- scene description: replaces myRTFileReader.readRTFile + the myScene builders ---- */
int drt_set_image_loader(drt_ctx* ctx, drt_image_loader_fn fn, void* user);
int drt_set_texture_dir(drt_ctx* ctx, const char* dir);          /* fallback decoder cache: <dir>/<name>.argb */
int drt_scene_reset(drt_ctx* ctx);                               /* new myFOVScene, fov 60 (myRTFileReader.java:27-28) */
int drt_scene_command(drt_ctx* ctx, const char* line);           /* one .cli line (myRTFileReader.java:47-346) */
int drt_scene_load_cli(drt_ctx* ctx, const char* file, const char* data_dir); /* whole file incl. nested `read` */
int drt_scene_override(drt_ctx* ctx, int32_t spp, int64_t photons); /* <=0 / <0 keep the file's values */
int drt_scene_finalize(drt_ctx* ctx, int32_t accel_mode);        /* flatten, build acceleration structures, upload to HBM */
int drt_scene_reupload(drt_ctx* ctx);                            /* host->device copy of the flattened scene again (used by end-to-end timing) */
int drt_accel_info(drt_ctx* ctx, double* out4);                  /* after finalize: GPU LBVH build ms, triangles and nodes it covers, scene bytes resident in HBM */
/* host wall clock (ms) of the build phases of the current scene: [0] .cli interpretation (includes [1],[3]), [1] median-split object ordering
   (myBVH.addObjList / buildSortedObjAras, myGeomBase.java:338-386) host or device, [2] the device part of [1] (CUDA events), [3] node / leaf-list
   construction from the order, [4] finalize (packed triangles, FP32 node mirror), [5] BVHs ordered on the device, [6] objects ordered, [7] upload */
int drt_build_info(drt_ctx* ctx, double* out8);
/* parity probe: object order of the reference's median-split BVH (myBVH.addObjList, myGeomBase.java:338-386) over n objects with centroid keys
   keys3n = [3][n]; ord[n] = leaves left to right, each in the order the reference's leaf list holds them, the object dropped at the root
   (SURVEY Q2) last.  on_device != 0: the device builder (segmented radix sorts), else the host recursion -- the two must agree bit for bit. */
int drt_bvh_order(drt_ctx* ctx, int32_t n, const double* keys3n, int32_t* ord, int32_t on_device);
/* parity probe for the fast BVHs (north star subsystem 2: "Morton/BVH ordering must be bit-exact"): packed triangles of fast BVH number
   fast_index (scene order) -- 9 vertex coordinates + primitive serial each -- in the order of the host flattener (which = 0: the reference
   tree's DFS order = the input order of the Morton sort) or as resident in HBM (which = 1: after the device LBVH build in DRT_ACCEL_LBVH mode),
   the BVH's root box, and (which = 1, LBVH mode) the built nodes: child links (>= 0 node, < 0: -(1 + leaf), leaf j = resident triangles
   4j..4j+3) and both child boxes.  Returns the triangle count (DRT_ERR_BAD_ARG: no such BVH; DRT_ERR_NO_DEVICE: which = 1 on a host-only context); arrays are filled only
   when cap_tris >= count.
   Buffers: verts9[9n], prim_serial[n], links2[2(ceil(n/4)-1)], boxes12[12(ceil(n/4)-1)]; any may be NULL. */
int64_t drt_lbvh_probe(drt_ctx* ctx, int32_t fast_index, int32_t which, double* box6, double* verts9, int32_t* prim_serial, int32_t* links2, double* boxes12, int64_t cap_tris);
int drt_scene_counts(drt_ctx* ctx, int64_t* out8);               /* flattener products of the fast paths: packed triangles, fast BVHs, packed top-level triangles, triangles in fast BVHs, children, pdata doubles, 0, 0 */
int drt_scene_info(drt_ctx* ctx, int32_t* out16);                /* cols, rows, spp, top objects, lights, prims, instances, photon kind, shaders, nodes, xforms, lists, ... */

/* ---- rendering: replaces myScene.initRender + draw; argb layout == PImage.pixels ---- */
int drt_emit_photons(drt_ctx* ctx, drt_stats* stats);            /* myScene.sendCausticPhotons / sendDiffusePhotons (:952-1091) */
/* multi-GPU photon pass (the reference emits serially, myScene.java:961,1009): rank r emits photon indices [i0,i1) of every light into
 * canonical-order records {x,y,z,r,g,b} (6 doubles) on its device, the host all-gathers the records (NCCL) and every rank builds the grid
 * from the full set.  Record order -- hence every later floating-point sum -- is independent of how the index range was split. */
int drt_emit_photons_range(drt_ctx* ctx, int64_t i0, int64_t i1, drt_stats* stats);
int64_t drt_photons_export_device(drt_ctx* ctx, double* dst6_dev, int64_t cap);    /* copies min(count,cap) records to a DEVICE buffer; returns count */
int drt_photons_build_device(drt_ctx* ctx, const double* src6_dev, int64_t n, drt_stats* stats);  /* n records in a DEVICE buffer -> photon grid */
int drt_render(drt_ctx* ctx, int32_t* argb_out, drt_stats* stats);                 /* host buffer, cols*rows */
int drt_render_aov(drt_ctx* ctx, int32_t* argb_out, int32_t* hit_prim, int32_t* hit_inst, double* rgb, double* t, drt_stats* stats); /* any may be NULL */
/* device-resident variant for multi-GPU hosts: render pixels [pix0,pix1) into caller-owned DEVICE buffers of cols*rows ints */
int drt_render_device(drt_ctx* ctx, int64_t pix0, int64_t pix1, int32_t* argb_dev, drt_stats* stats);
/* multi-GPU tiles: render this rank's interleaved row chunks (chunk c of the rank = rows [(c*world+rank)*chunk_rows, +chunk_rows)) at their
 * absolute positions of a full cols*rows DEVICE buffer; pixels of other ranks are left untouched */
int drt_render_device_chunks(drt_ctx* ctx, int32_t world, int32_t rank, int32_t chunk_rows, int32_t* argb_dev, drt_stats* stats);
/* ---- multi-GPU inside the library (no reference counterpart: the reference renders serially, myScene.java:1481-1531).  One context per GPU
 * (one process per GPU, or several contexts in one host process on different threads).  Rank 0 creates an id, the host ships its 128 bytes
 * to the other ranks by any transport, every rank calls drt_comm_init (collective).  drt_render_distributed (collective) renders this rank's
 * interleaved row chunks, gathers them to rank 0 over NCCL (send / recv into the frame) and, for photon scenes, splits the emission by
 * photon index, all-gathers the records and builds the grid on every rank.  The frame is bit-identical for every world size. */
int drt_comm_unique_id(uint8_t* id128);
int drt_comm_init(drt_ctx* ctx, const uint8_t* id128, int32_t world, int32_t rank);
int drt_comm_destroy(drt_ctx* ctx);
/* argb_host_rank0 / argb_dev_rank0: cols*rows ints on rank 0 (either may be NULL), ignored on other ranks.  reemit_photons != 0: redo the photon pass even if a map exists (the reference emits inside every draw) */
int drt_render_distributed(drt_ctx* ctx, int32_t* argb_host_rank0, int32_t* argb_dev_rank0, int32_t chunk_rows, int32_t reemit_photons, drt_stats* stats);
/* the partition behind drt_render_distributed as pure host functions (no device needed): compact pixels rank `rank` renders (whole chunks),
 * absolute pixel of one of its compact slots (-1 = padding beyond the frame), photon index range [out2[0], out2[1]) it emits */
int64_t drt_dist_rank_pixels(int32_t cols, int32_t rows, int32_t world, int32_t rank, int32_t chunk_rows);
int64_t drt_dist_abs_pixel(int32_t cols, int32_t rows, int32_t world, int32_t rank, int32_t chunk_rows, int64_t compact_index);
int drt_dist_photon_range(int64_t n_cast, int32_t world, int32_t rank, int64_t* out2);
int drt_save_png(const char* path, const int32_t* argb, int32_t cols, int32_t rows);  /* PImage.save (myScene.java:1194) */
/* ---- progressive refinement display (`refine on`: myScene.setRefine :796-803, the pass loop of draw() :1493-1526, writePxlSpan :1171-1177).
 * The reference shows a sequence of previews: pass k traces every step_k-th pixel of every step_k-th row (step = 2^refIDX ... 2, 1 with
 * refIDX = (int)(log10(.5 (cols + rows) / 16) / log10(2))) and paints each result over a step x step block.  It re-traces the pixels on every
 * pass; with this library's seeded sampler a pixel's colour does not depend on the pass, so every preview is a function of the finished frame:
 * block (r, c) shows the frame's pixel at the block's top-left corner.  drt_scene_refine: 1 when the scene said `refine on`;
 * drt_refine_steps: the step sequence (returns its length, 0 when the reference's formula yields none: frames smaller than 16 pixels mean size);
 * drt_refine_pass: the preview of one step from the finished frame (pure host functions: the frame itself comes from drt_render). */
int drt_scene_refine(drt_ctx* ctx);
int32_t drt_refine_steps(int32_t cols, int32_t rows, int32_t* steps16);
int drt_refine_pass(const int32_t* argb_full, int32_t cols, int32_t rows, int32_t step, int32_t* argb_out);

/* ---- ray queries: the caller's own rays against the finalized scene (visibility, ambient occlusion, picking, depth / normal buffers).
 * Every pointer is DEVICE memory of the context's GPU; n rays, origin org3[3i..] and direction dir3[3i..] in FP64 world space (the direction
 * is normalised on the device; it need not be unit length).  Ray time is 0: moving spheres are queried at their start position.  A ray whose
 * origin or direction is not finite, or whose direction has a zero (or non-finite) FP64 length, is not traced: a miss / not occluded.
 * The rays run through the same traversal, kernel variants and fix-up pass as the renderer's closest-hit and shadow rays, on the context's
 * stream; the call returns when the outputs are complete (one host sync).  The caller makes its own producers of the inputs finish first.
 * Returns DRT_ERR_NO_DEVICE on a host-only context, DRT_ERR_STATE before drt_scene_finalize, DRT_ERR_BAD_ARG for n < 0 or a required pointer
 * that is NULL while n > 0; n == 0 does nothing.  stats (may be NULL): kernel_launches, rays_deferred (rays the lean kernel left to the generic
 * one), host_syncs, ms_trace (closest) or ms_light (occlusion) and ms_total (CUDA events); every other field is 0.
 *
 * drt_query_closest: the closest hit, reported as a miss unless t < tmax[i] (tmax NULL = +inf; a NaN tmax is a miss).  ids2[2i] = primitive
 * serial, ids2[2i+1] = instance serial (-1, -1 on a miss), t[i] (0 on a miss) -- the conventions of drt_trace_rays, whose ids and t these are
 * bit for bit.  Optional pos3 / nrm3 (NULL: skipped): the world hit point and unit normal the renderer shades with (0 on a miss).  SURVEY Q6/Q7
 * apply: for a mesh in a transformed BVH pos is the reference's CTM-applied-twice point, and through a scaled instance t is measured in the
 * instance's direction units, so pos is not org + t * dir in general.
 * drt_query_occluded: occluded[i] = 1 when something is hit with (dist[i] - t) > 1e-7 -- the renderer's shadow test (box rules and instance
 * trees included) -- else 0.  dist may be +inf; a NaN dist is not occluded.
 * No Java binding covers these entry points (device pointers). */
int drt_query_closest(drt_ctx* ctx, int64_t n, const double* org3, const double* dir3, const double* tmax, int32_t* ids2, double* t, double* pos3, double* nrm3, drt_stats* stats);
int drt_query_occluded(drt_ctx* ctx, int64_t n, const double* org3, const double* dir3, const double* dist, uint8_t* occluded, drt_stats* stats);

/* ---- parity probes (used by tests; not needed by a host) ---- */
/* drt_trace_rays: drt_query_closest's generic kernel on HOST arrays, without tmax, pos3 / nrm3 or the lean kernel variants: the same ids2 and
 * t.  So a ray whose origin or direction is not finite, or whose direction has a zero (or non-finite) FP64 length, is a miss (-1, -1, 0). */
int drt_trace_rays(drt_ctx* ctx, int64_t n, const double* org, const double* dir, int32_t* ids2, double* t);
int drt_eval_texture(drt_ctx* ctx, int32_t shader_serial, int64_t n, const double* hit_loc, const double* fwd_loc, double* rgb);
int64_t drt_dump_bvh(drt_ctx* ctx, int32_t top_index, int32_t* out, int64_t cap, double* root_box6);
int drt_obj_ctm(drt_ctx* ctx, int32_t top_index, double* out16);
double drt_sample_u01(uint64_t seed, uint32_t stream, uint32_t a, uint32_t b, uint32_t c, uint32_t d);
int64_t drt_get_photons(drt_ctx* ctx, double* out6, int64_t cap);   /* x,y,z,r,g,b per stored photon */
/* kNN radiance gather at explicit world points (myKD_Tree.find_near + getIrradianceFromPhtnTree): out5 = {sum r, sum g, sum b, d^2 of the farthest, gather tier taken: 0 no photon in range, 1 lane sum, 2 lane selection, 3 warp over coarse rows, 4 warp over a fine cube} */
int drt_photon_probe(drt_ctx* ctx, int64_t n, const double* pts3, double* out5);

#ifdef __cplusplus
}
#endif
#endif
