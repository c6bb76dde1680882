/* rtfs_b200.h — C ABI of the B200-native path-tracing core for Smaug123/ray-tracing-fsharp.
 *
 * This is the drop-in boundary for the reference's per-pixel render loop.  The reference has no
 * FFI of its own; the seam it offers is the F# function
 *
 *   Scene.render : (float<progress> -> unit) -> (string -> unit) -> maxWidthCoord:int ->
 *                  maxHeightCoord:int -> Camera -> Scene -> float<progress> * Image
 *                                                            (RayTracing/Scene.fs:196-204)
 *   Scene.make   : Hittable array -> Scene                   (RayTracing/Scene.fs:15-28)
 *
 * so every entry point below cites the reference function it replaces.  The F#-side P/Invoke
 * binding a maintainer would add is in INTEGRATION.md and shim/RayTracing.Gpu.fs.
 *
 * Conventions
 *   - plain C types only; doubles on the ABI because the host types are double
 *     (RayTracing/Point.fs:8-11); the device computes in FP32 (see DESIGN.md for the three
 *     places where FP64 is used on the device for exactness).
 *   - every function returns RT_OK (0) or a negative RT_ERR_* code; nothing throws or aborts across
 *     the boundary; rt_last_error() gives a thread-local message for the last failure.
 *   - the caller owns every buffer it passes; the library copies what it needs.  Opaque handles
 *     (RtScene*) own device memory and are released with rt_scene_destroy.  A handle is not
 *     thread-safe; distinct handles are independent.
 *   - there is NO CPU fallback: entry points that compute fail with RT_ERR_NO_DEVICE when no
 *     CUDA device is present.  Host-side helpers (camera basis, BVH build, P3 writer) run anywhere.
 */
#ifndef RTFS_B200_H
#define RTFS_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RT_ABI_VERSION 6

/* ---- error codes --------------------------------------------------------------------------- */
#define RT_OK 0
#define RT_ERR_INVALID_ARGUMENT (-1)
#define RT_ERR_CUDA (-2)
#define RT_ERR_NO_DEVICE (-3)
#define RT_ERR_UNSUPPORTED (-4) /* e.g. a texture the device cannot evaluate (F# closures)       */
#define RT_ERR_DEGENERATE (-5)  /* where the reference would throw from ValueOption.get          */
#define RT_ERR_IO (-6)

/* ---- scene description --------------------------------------------------------------------- */

/* Hittable cases, RayTracing/Hittable.fs:3-6. */
enum RtShape { RT_SHAPE_SPHERE = 0, RT_SHAPE_UNBOUNDED_SPHERE = 1, RT_SHAPE_INFINITE_PLANE = 2 };

/* SphereStyle cases, RayTracing/Sphere.fs:10-37.  InfinitePlaneStyle (InfinitePlane.fs:3-13) uses
 * the subset LIGHT_SOURCE, PURE_REFLECTION, LAMBERT_REFLECTION, FUZZED_REFLECTION. */
enum RtStyle {
    RT_STYLE_LIGHT_SOURCE = 0,
    RT_STYLE_LIGHT_SOURCE_CAP = 1,
    RT_STYLE_PURE_REFLECTION = 2,
    RT_STYLE_FUZZED_REFLECTION = 3,
    RT_STYLE_LAMBERT_REFLECTION = 4,
    RT_STYLE_DIELECTRIC = 5,
    RT_STYLE_GLASS = 6
};

/* Texture / ParameterisedTexture cases, RayTracing/Texture.fs:5-22.  F# closures
 * (Texture.Arbitrary, ParameterisedTexture.Arbitrary) cannot cross the ABI; the shim must pass the
 * structure (image, checker) before ParameterisedTexture.toTexture erases it (Texture.fs:69-72). */
enum RtTextureKind { RT_TEX_COLOUR = 0, RT_TEX_IMAGE = 1, RT_TEX_CHECKERED = 2 };

typedef struct RtTexture {
    int32_t kind;        /* RtTextureKind                                                        */
    uint8_t colour[3];   /* RT_TEX_COLOUR                                                        */
    uint8_t _pad0;
    int32_t width;       /* RT_TEX_IMAGE: img.[0].Length                                         */
    int32_t height;      /* RT_TEX_IMAGE: img.Length                                             */
    const uint8_t *rgb8; /* RT_TEX_IMAGE: the Pixel[][] of ParameterisedTexture.Image, row-major
                            img.[y].[x], 3 bytes per texel, i.e. AFTER ofImage's row flip
                            (Texture.fs:30-48)                                                   */
    int32_t even;        /* RT_TEX_CHECKERED: texture index used when sin(g u) sin(g v) < 0      */
    int32_t odd;         /* RT_TEX_CHECKERED: texture index used otherwise (Texture.fs:56-62)    */
    double grid_size;    /* RT_TEX_CHECKERED                                                     */
    /* the `interpret` closure is always Sphere.planeMapInverse radius centre (Sphere.fs:55-61) */
    double map_centre[3];
    double map_radius;
} RtTexture;

/* One element of the Hittable array handed to Scene.make (Scene.fs:15).  Array order is
 * significant: it is the reference's tie-break order (Scene.fs:47, :77-86). */
typedef struct RtHittable {
    int32_t shape;     /* RtShape                                                                */
    int32_t style;     /* RtStyle                                                                */
    double p[3];       /* Sphere.Centre (Sphere.fs:305) or InfinitePlane.Point (InfinitePlane.fs:105) */
    double n[3];       /* InfinitePlane.Normal (unit); ignored for spheres                       */
    double radius;     /* Sphere.Radius; negative radius is legal (Sphere.fs:160-182)            */
    double albedo;     /* float<albedo>                                                          */
    double fuzz;       /* float<fuzz>,  FUZZED_REFLECTION                                        */
    double ior;        /* float<ior>,   DIELECTRIC / GLASS                                       */
    double prob;       /* float<prob>,  DIELECTRIC: probability of refraction                    */
    int32_t texture;   /* index into textures[], or -1: constant `colour`                        */
    uint8_t colour[3]; /* Texture.Colour / LightSourceCap colour / plane colour                  */
    uint8_t _pad0;
} RtHittable;

/* Camera record, RayTracing/Camera.fs:3-28.  ViewportYAxis' origin is never read by the render
 * loop (Scene.fs:139-140 uses only its Vector) so only the direction crosses the ABI. */
typedef struct RtCamera {
    double view_origin[3];  /* View.Origin                                                      */
    double view_dir[3];     /* View.Vector                                                      */
    double xaxis_origin[3]; /* ViewportXAxis.Origin                                             */
    double xaxis_dir[3];    /* ViewportXAxis.Vector                                             */
    double yaxis_dir[3];    /* ViewportYAxis.Vector                                             */
    double viewport_width;
    double viewport_height;
    double focal_length;
    int32_t samples_per_pixel;
    int32_t bounce_depth;
} RtCamera;

enum RtMode { RT_MODE_MEGAKERNEL = 0, RT_MODE_WAVEFRONT = 1 };
enum RtBvhKind { RT_BVH_SAH = 0, RT_BVH_REFERENCE = 1 };

typedef struct RtRenderOpts {
    uint64_t seed;    /* key of the counter-based RNG; replaces `FloatProducer (Random ())` (Scene.fs:205) */
    int32_t adaptive; /* 1: the reference's early-out rule (Scene.fs:172-194); 0: always spp samples */
    int32_t mode;     /* RtMode                                                                  */
    int32_t gamma;    /* rt_render only: 1 = apply PixelOutput.correct (ImageOutput.fs:11-18) on the device */
    int32_t flags;    /* RT_FLAG_* bits                                                           */
} RtRenderOpts;

/* RtRenderOpts.flags */
#define RT_FLAG_COUNTERS 1 /* also count the device traversal's box / primitive tests (slower kernel variant) */
#define RT_FLAG_NO_SMEM 2  /* read the BVH from global memory even when it would fit in shared memory      */
#define RT_FLAG_WIDE_BVH 4 /* walk the 8-wide compressed tree (read from global memory) instead of the binary one:
                              measured slower on B200 for every scene tried (DESIGN.md), kept selectable          */
#define RT_FLAG_BVH2 8     /* walk the binary tree (the default; overrides RT_FLAG_WIDE_BVH)                      */
#define RT_FLAG_LOCKSTEP 16 /* the default schedule, spelt out: the 32 lanes of a warp trace one ray each per pass      */
#define RT_FLAG_FLOW 32     /* the flow schedule: every warp keeps a ring of 64 rays in shared memory, lanes pull walks
                              from it in quanta, scatters run in full-width passes.  Bit-identical frames; measured
                              slower than lockstep on B200 (DESIGN.md), kept selectable                          */
#define RT_FLAG_NO_LEAN 64  /* do not pick the kernel specialised for scenes without FP64 unbounded objects and without
                              texture lookups even where the scene allows it (A/B tests; frames are bit-identical)      */
#define RT_FLAG_NOISE 128   /* rt_frame_begin only: also keep per pixel the sum of r^2 + g^2 + b^2 over its samples, for the
                              noise estimate of rt_frame_noise.  Not with RT_FLAG_FLOW or RT_FLAG_COUNTERS
                              (RT_ERR_UNSUPPORTED).  Every other entry point ignores the bit                           */

typedef struct RtStats {
    uint64_t paths;     /* traceOnce calls (Scene.fs:118)                                        */
    uint64_t rays;      /* hitObject calls (Scene.fs:99)                                         */
    uint64_t box_tests; /* slab tests executed by the device traversal (its own, not the reference's) */
    uint64_t prim_tests;
    double kernel_ms;   /* device time of the trace kernels (CUDA events)                        */
    double total_ms;    /* device time of the whole call incl. copies                            */
    uint64_t pixels_early_out;
    int32_t launches;   /* kernels launched by this call                                         */
    int32_t _pad0;
    double main_ms;     /* device time of the main-phase kernel alone (compact + render_kernel<PROBE=0>) */
    uint64_t main_rays; /* hitObject calls of that launch (this rank's)                          */
    uint64_t degenerate_paths; /* paths ended where the reference would throw (Ray.make' / ValueOption.get failing):
                                  rendered Black, counted here; 0 on non-degenerate scenes        */
} RtStats;

typedef struct RtScene RtScene;

/* ---- library ------------------------------------------------------------------------------- */
int rt_abi_version(void);
const char *rt_last_error(void);
/* number of CUDA devices visible (0 on a CPU-only host; never fails) */
int rt_device_count(void);

/* ---- host-side helpers (no GPU needed) ------------------------------------------------------ */

/* Camera.makeBasic (RayTracing/Camera.fs:34-59) incl. Plane.makeNormalTo' and Plane.basis
 * (RayTracing/Plane.fs:22-38, :82-97).  bounce_depth is set to 150 as in the reference
 * (Camera.fs:58); callers override the field afterwards like `{ camera with BounceDepth = 50 }`. */
int rt_camera_make_basic(int32_t samples_per_pixel, double focal_length, double aspect_ratio,
                         const double origin[3], const double view_direction[3],
                         const double view_up[3], RtCamera *out);

/* ImageOutput.writePpm (RayTracing/ImageOutput.fs:163-197): P3 text, byte-identical format.
 * `rgb` is rows*cols*3, row 0 first.  gamma_correct applies PixelOutput.correct.  Writes at most
 * `cap` bytes into `out` and returns the full length in *len (call with cap = 0 to size it). */
int rt_ppm_format(const uint8_t *rgb, int32_t rows, int32_t cols, int32_t gamma_correct, char *out,
                  size_t cap, size_t *len);
int rt_ppm_write_file(const uint8_t *rgb, int32_t rows, int32_t cols, int32_t gamma_correct,
                      const char *path);
/* PixelOutput.correct (ImageOutput.fs:11-18) for one byte (host). */
uint8_t rt_gamma_correct(uint8_t b);

/* ---- scene --------------------------------------------------------------------------------- */

/* Scene.make (Scene.fs:15-28) + BoundingBoxTree.make (BoundingBoxTree.fs:9-43), rebuilt as a
 * flattened BVH in device memory.  `device` is a CUDA ordinal.  Pass device = -1 to build the
 * host side only (no GPU required; for rt_scene_bvh_* inspection). */
int rt_scene_create(const RtHittable *objects, int32_t n_objects, const RtTexture *textures,
                    int32_t n_textures, int32_t device, RtScene **out);
void rt_scene_destroy(RtScene *scene);

/* Inspection of the two host-built trees (CPU tests use these).
 * Node layout (flattened, DFS pre-order, left child = i+1):
 *   bounds[6*i..] = min xyz, max xyz ; right[i] = index of right child, or -1 for a leaf ;
 *   prim[i] = index into the caller's Hittable array for a leaf, else -1. */
int rt_scene_bvh_node_count(const RtScene *scene, int32_t which /* RtBvhKind */);
int rt_scene_bvh_nodes(const RtScene *scene, int32_t which, double *bounds, int32_t *right,
                       int32_t *prim);
/* The third tree: the 8-wide compressed BVH the render kernels walk for scenes read from global memory (quantised
 * child boxes, 80-byte nodes; replaces BoundingBoxTree.fs:9-43 / Scene.fs:30-60 for those scenes).  Builds it on the
 * host if need be and verifies it: every bounded sphere in exactly one leaf slot, every decoded box containing what
 * lies below it (RT_ERR_DEGENERATE otherwise).  Outputs are optional. */
int rt_scene_wide_bvh_check(RtScene *scene, int32_t *n_nodes, int32_t *depth, int32_t *n_spheres,
                            double *mean_children);
/* The tree as the render kernels read it (binary SAH tree, child boxes as centre / half-extent with the left and right child's
 * values side by side for the packed FP32 slab test; replaces BoundingBoxTree.fs:9-43 / Scene.fs:30-60): verifies on the host
 * that no converted box is smaller than the box it was made from, that every bounded sphere of non-negative radius is the leaf
 * of exactly one node and lies inside that leaf's box, and that the tree is no deeper than the walk stacks assume
 * (RT_ERR_DEGENERATE otherwise).  Outputs are optional. */
int rt_scene_device_bvh_check(RtScene *scene, int32_t *n_nodes, int32_t *depth, int32_t *n_spheres);
/* bytes of scene data resident on the device (nodes + primitives + materials + textures) */
size_t rt_scene_device_bytes(const RtScene *scene);
/* bytes of BVH + spheres + materials that every persistent block stages in shared memory; 0 when the scene
 * is too large for that and is read from global memory (L1 / L2) instead */
size_t rt_scene_shared_memory_bytes(const RtScene *scene);

/* ---- editing a scene in place ----------------------------------------------------------------- */
/* Changes objects and textures of a scene on its device and refits its tree there: for selection and recolouring, nudging
 * an object, or the next step of an animation, without rt_scene_create's host build and full upload.
 *
 * Object object_index[i] of the caller's array becomes objects[i]; texture texture_index[j] becomes textures[j].  After the
 * call the scene is the scene rt_scene_create would make from the edited arrays, except that the SAH tree keeps its
 * topology, its leaf order and the device primitive ids: the boxes of every node above a moved sphere are recomputed on the
 * device, bottom-up, as the host build computes them (directed roundings of each FP32 sphere, exact unions).  So every entry
 * point (rt_render, views, windows, progressive frames opened after the call, features and denoise; sums, RGB8, Q, stats
 * and rays) gives bit for bit the frame of a freshly created scene of the edited arrays, wherever no closest hit is an exact
 * tie in t between two bounded spheres (the condition under which the binary and the 8-wide trees already agree).  A tree
 * refit over moved spheres may become slower to walk than a fresh build; DESIGN.md section 20 says when to recreate.
 *
 * Structure must stay: the object count, each object's shape, whether each bounded sphere's radius is >= 0, the texture
 * count, each texture's kind, an image texture's width and height.  Anything else may change (centre, radius, normal,
 * style, albedo, fuzz, ior, prob, colour, texture index, checker parameters, map centre and radius, image texels).  A
 * structural change needs a new scene.
 * Refusals (RT_ERR_INVALID_ARGUMENT, before any device work, leaving the scene as it was): a structural change, an index
 * out of range, a duplicate index, a negative count, a NULL array with a non-zero count, and anything rt_scene_create
 * would refuse in the edited arrays.  A scene created with device = -1: RT_ERR_UNSUPPORTED.
 * Frames.  A progressive frame opened before the call is stale: rt_frame_advance, _extend, _set_convergence, _features
 *   and _denoise refuse it (RT_ERR_INVALID_ARGUMENT); _read, _noise, _view_noise, _convergence and _destroy still work on
 *   what it holds.
 * Returns with its device work complete.  info optional.  A caller detects the feature by the symbol rt_scene_update. */
typedef struct RtSceneUpdate {
    int32_t objects;       /* object records that changed                                                         */
    int32_t textures;      /* texture records that changed                                                        */
    int32_t spheres_moved; /* bounded spheres whose device sphere (FP32 centre, radius) changed                    */
    int32_t nodes_refit;   /* tree nodes whose child boxes were recomputed                                          */
    uint64_t generation;   /* the scene's edit count after this call (0 = as created)                              */
    double device_ms;      /* device time of the copy and the kernels (CUDA events)                                */
    int32_t launches;
    int32_t _pad0;
} RtSceneUpdate;
int rt_scene_update(RtScene *scene, const int32_t *object_index, const RtHittable *objects, int32_t n_objects,
                    const int32_t *texture_index, const RtTexture *textures, int32_t n_textures,
                    RtSceneUpdate *info /* optional */);

/* Removes and appends objects of a scene and builds its tree anew on the device: for adding or deleting an object of a live
 * scene, and for renewing a tree that rt_scene_update's refits have left slow to walk, without rt_scene_create's host build
 * and full upload, and without closing the scene's handle.
 *
 * The objects remove[0..n_remove) (indices into the caller's array) are taken out; the others keep their order and are
 * renumbered densely; then append[0..n_append) are added at the end.  After the call the scene is rt_scene_create(new array,
 * the same textures), except that its tree comes from the device builder (PLOC over the FP32 sphere boxes, DESIGN.md section
 * 22): every entry point (rt_render, views, windows, progressive frames opened after the call, features with the new object
 * indices, denoise; sums, RGB8, Q, stats, rays, every flag) gives bit for bit the frame of a freshly created scene of the new
 * array, wherever no closest hit is an exact tie in t between two bounded spheres (rt_scene_update's condition).  With
 * n_remove = n_append = 0 the call rebuilds the tree of the current objects.
 * Determinism.  The tree is a pure function of the object array after the call: two scenes that reach the same array by any
 *   edit sequences hold identical trees, byte for byte.
 * Fallback.  A device tree deeper than the walk stacks allow (60) is replaced by the host SAH tree rt_scene_create builds
 *   (on_device = 0); the call does not fail for that reason.
 * Refusals (RT_ERR_INVALID_ARGUMENT, before any change or device work, leaving the scene as it was): a remove index out of
 * range or repeated, a negative count, a NULL array with a non-zero count, and anything rt_scene_create would refuse in an
 * appended object (such as a texture index out of range).  Textures cannot be added or removed here (rt_scene_update
 * replaces a texture's content).  A scene created with device = -1: RT_ERR_UNSUPPORTED.
 * Frames opened before the call are stale, as after rt_scene_update; rt_scene_update refits the new tree.
 * Returns with its device work complete.  info optional.  A caller detects the feature by the symbol rt_scene_rebuild. */
typedef struct RtSceneRebuild {
    int32_t objects_removed, objects_appended;
    int32_t n_objects; /* the caller's array after the call                                                       */
    int32_t n_bounded; /* spheres in the tree                                                                     */
    int32_t nodes;     /* of the new tree                                                                         */
    int32_t depth;     /* of the new tree: internal nodes on its longest root-to-leaf path                        */
    int32_t on_device; /* 1: the device build; 0: the host SAH build (the device tree was deeper than 60)         */
    int32_t launches;
    uint64_t generation; /* the scene's edit count after the call                                                 */
    double device_ms;    /* CUDA events around the device work                                                   */
} RtSceneRebuild;
int rt_scene_rebuild(RtScene *scene, const int32_t *remove, int32_t n_remove, const RtHittable *append, int32_t n_append,
                     RtSceneRebuild *info /* optional */);

/* ---- host buffers ----------------------------------------------------------------------------- */
/* Page-locks a host buffer the caller owns (an output frame it renders into again and again) so that the device->host
 * copy of rt_render / rt_multi_render / rt_comm_render runs at PCIe speed and asynchronously instead of through the
 * driver's staging buffer (2.9 MB C2 frame: ~0.25 ms -> ~0.1 ms).  Optional: every entry point accepts pageable memory.
 * The F# host: GCHandle.Alloc(array, GCHandleType.Pinned) + rt_host_pin(AddrOfPinnedObject, length).  Unpin before freeing. */
int rt_host_pin(void *ptr, size_t bytes);
int rt_host_unpin(void *ptr);

/* ---- render (host buffers) ------------------------------------------------------------------ */

/* Scene.render + Image.render (Scene.fs:196-236, Domain.fs:23-24) on one GPU.
 * rgb_out: rows*cols*3 bytes, rows = 2*max_height_coord+1, cols = 2*max_width_coord+1
 * (Scene.fs:208-209), row 0 = top row — exactly the Pixel[][] that Image.render yields
 * (pre-gamma truncated means, Pixel.fs:103-108) unless opts->gamma is set.
 * sums_out (optional): rows*cols*4 int32 {sumR,sumG,sumB,count} as PixelStats holds them
 * (Pixel.fs:78-85).  stats optional. */
int rt_render(RtScene *scene, const RtCamera *camera, int32_t max_width_coord,
              int32_t max_height_coord, const RtRenderOpts *opts, uint8_t *rgb_out,
              int32_t *sums_out, RtStats *stats);

/* ---- many views of one scene (host buffers; one GPU) -------------------------------------------- */
/* n_views frames of one scene, same extents, in one submission: a turntable, a camera path, stereo pairs, a contact sheet
 * of previews.  The views are stacked as one tall frame of n_views * rows rows, so the batch pays rt_render's fixed costs
 * once (the launches of one probe, one main phase and one output tail, the tail of the persistent kernel, one device->host
 * copy and one synchronisation) instead of once per view.
 *
 * View v is cameras[v] with seed seeds[v] (seeds NULL: opts->seed for every view).  rgb_out: n_views*rows*cols*3, view v at
 * offset v*rows*cols*3; sums_out (optional) n_views*rows*cols*4 int32, view v at offset v*rows*cols*4.  Every sample is
 * keyed by (seed, pixel, sample index) with the pixel counted within its view, and the sums are integers, so view v's bytes
 * are bit for bit rt_render(scene, &cameras[v], max_w, max_h, opts with seed = seeds[v]).
 * What may differ between views: origin, view direction, axes, viewport width and height, focal length, seed.
 * What must be the same: samples_per_pixel and bounce_depth on every camera (the probe's firstTrial and the chunk table are
 *   shared): RT_ERR_INVALID_ARGUMENT otherwise.
 * Other argument errors (RT_ERR_INVALID_ARGUMENT): n_views < 1; cameras or rgb_out NULL; n_views * rows * cols >= 2^31;
 *   and those of rt_render.
 * Options.  RT_MODE_WAVEFRONT, RT_FLAG_FLOW and RT_FLAG_COUNTERS: RT_ERR_UNSUPPORTED (no batched wavefront, flow-schedule
 *   or counting kernels).  RT_FLAG_NOISE is ignored, as rt_render ignores it (a batch that keeps its noise estimate is a
 *   progressive frame: rt_frame_begin_views, below).  RT_FLAG_NO_SMEM, RT_FLAG_WIDE_BVH,
 *   RT_FLAG_BVH2, RT_FLAG_NO_LEAN, RT_FLAG_LOCKSTEP, adaptive and gamma act as in rt_render.
 * Stats (optional): paths, rays, degenerate_paths and pixels_early_out are sums over the views; the _ms fields and
 *   launches describe the batch; box_tests and prim_tests are 0.
 * Like rt_render, the call returns with its device work complete, and rt_render or progressive frames may use the scene
 * between two batches. */
int rt_render_views(RtScene *scene, const RtCamera *cameras, const uint64_t *seeds, int32_t n_views,
                    int32_t max_width_coord, int32_t max_height_coord, const RtRenderOpts *opts,
                    uint8_t *rgb_out, int32_t *sums_out, RtStats *stats);

/* ---- progressive frames (host buffers; one GPU) -------------------------------------------------- */
/* rt_render's frame in sample passes, with progress between them (the reference calls progressIncrement as rows finish,
 * Scene.fs:232), an image to look at after every pass, early stopping and continuation to more samples.
 *
 * Open a frame once (rt_frame_begin: the probe phase, Scene.fs:172-188, and the compaction of the flagged pixels), then
 * advance it in passes (rt_frame_advance: the third loop, Scene.fs:191-192, over a window of sample indices).  Every
 * sample is keyed by (seed, pixel, sample index) and the sums are integers, so after any pass the frame's sums are bit for
 * bit those of rt_render with samples_per_pixel = samples_done (same scene, camera, extents, seed, adaptive and flags).
 * The rule's firstTrial = min(5, spp / 2) is the same at samples_done and at the target once the probe is done.
 *
 * Pass sizing.  A pass covers the sample window [samples_done, samples_done + k).  k is the smallest of max_samples
 * (if > 0); the number of sample indices predicted to take target_ms of device time (if > 0), from the measured device
 * time per sample index of the last pass, or of the probe for the first pass (a frame with adaptive = 0 has no probe:
 * its first paced pass takes one sample index); and what is left.  k is never below 1.  max_samples = 0 and
 * target_ms = 0 take everything that is left.  Only the number of passes depends on their sizes, never the result.
 * Stopping.  A caller stops early by not calling rt_frame_advance again: one pass is the longest it waits.
 * Extending.  rt_frame_extend raises (or lowers) the target to samples_per_pixel.  It accepts a value only if the target
 *   it gives is >= samples_done, samples_per_pixel <= 2^22, and firstTrial stays what it is (6 -> 64 would change the
 *   probe: RT_ERR_INVALID_ARGUMENT).  A frame opened at spp <= 2 firstTrial + 1 runs no main phase but keeps which pixels
 *   would go on, so it can be extended.
 * Modes.  RT_MODE_MEGAKERNEL only (RT_MODE_WAVEFRONT: RT_ERR_UNSUPPORTED); the RT_FLAG_* bits act as in rt_render, and
 *   RT_FLAG_NOISE also keeps the per-pixel sum of squares for rt_frame_noise (below).
 * Ownership.  A frame owns its sum, flag, list and image buffers and its work counters: rt_render and other frames may
 *   run on the same scene between two passes.  Every call returns with the device work it issued complete.  A frame is
 *   not thread-safe (like its scene) and must be destroyed before its scene. */
typedef struct RtFrame RtFrame;
typedef struct RtFrameProgress {
    int32_t samples_done;    /* every flagged pixel holds sample indices [0, samples_done): the frame equals
                                rt_render's at samples_per_pixel = samples_done                                   */
    int32_t samples_target;  /* max(2 firstTrial + 1, spp) with the early-out, spp without; or what rt_frame_extend set */
    uint64_t paths_done;     /* traceOnce calls so far (probe + passes), from the device counters               */
    uint64_t paths_target;   /* n_pixels * n_probe + pixels_flagged * (samples_target - n_probe); exact          */
    uint64_t pixels_flagged; /* pixels that go on after the probe (every pixel without the early-out)             */
    double last_pass_ms;     /* device time of the last pass (CUDA events)                                        */
    double device_ms;        /* device time of the probe and compaction plus every pass so far                     */
    int32_t passes;          /* rt_frame_advance calls that traced something                                      */
    int32_t done;            /* samples_done == samples_target                                                    */
} RtFrameProgress;
/* probe + compaction, synchronous.  progress optional. */
int rt_frame_begin(RtScene *scene, const RtCamera *camera, int32_t max_width_coord,
                   int32_t max_height_coord, const RtRenderOpts *opts, RtFrame **out,
                   RtFrameProgress *progress);
/* one pass (nothing when done).  progress optional. */
int rt_frame_advance(RtFrame *frame, int32_t max_samples, double target_ms, RtFrameProgress *progress);
/* the current image as rt_render gives it: rgb_out rows*cols*3 (gamma as opts->gamma of rt_render), sums_out
 * rows*cols*4 int32 {sumR,sumG,sumB,count}; either may be NULL */
int rt_frame_read(RtFrame *frame, int32_t gamma, uint8_t *rgb_out, int32_t *sums_out);
int rt_frame_extend(RtFrame *frame, int32_t samples_per_pixel);
void rt_frame_destroy(RtFrame *frame);

/* Noise estimate of a progressive frame opened with RT_FLAG_NOISE.  Per pixel the frame holds, besides the channel sums
 * T_c and the count n, Q = the sum over the pixel's samples of r^2 + g^2 + b^2 (8-bit levels).  Then
 *     D = n Q - (T_r^2 + T_g^2 + T_b^2)          exact in int64 (every term < 3.5e18 at n <= 2^22)
 *     E = sqrt(D / (3 n^2 (n - 1)))              in double, the denominator evaluated left to right as written
 * is the RMS over the three channels of the standard error of the channel mean, in 8-bit levels; E = +inf where n < 2.
 * Like the sums, Q is an integer keyed by (seed, pixel, sample index): it does not depend on how the frame was paced.
 * rt_frame_noise returns, each optional: se_out rows*cols float E of every pixel, sq_out rows*cols uint64 Q, and the
 * summary over the flagged pixels (those later passes still sample, in pixel order): how many, how many have
 * E > tolerance, the largest and the mean E.  The summary is bit-identical from call to call (fixed-order reduction).
 * RT_ERR_INVALID_ARGUMENT if the frame was opened without RT_FLAG_NOISE or tolerance is negative or NaN. */
typedef struct RtFrameNoise {
    uint64_t pixels;       /* flagged pixels (every pixel without the early-out)                        */
    uint64_t pixels_above; /* of them, those with E > tolerance                                         */
    double max_se;         /* the largest E over them (0 when there are none)                           */
    double mean_se;        /* the mean E over them (0 when there are none)                              */
    double tolerance;      /* as given                                                                  */
} RtFrameNoise;
int rt_frame_noise(RtFrame *frame, double tolerance, float *se_out, uint64_t *sq_out, RtFrameNoise *summary);
/* The same E from saved moments, on the host (no device needed): sums n*4 int32 {T_r, T_g, T_b, n} as rt_render and
 * rt_frame_read give them, sq n uint64 Q, se_out n float. */
int rt_pixel_noise(const int32_t *sums, const uint64_t *sq, size_t n, float *se_out);

/* Convergence rule of a progressive frame opened with RT_FLAG_NOISE: stop sampling each pixel once its E has converged.
 * rt_frame_set_convergence(tolerance tau, min_samples m, interval k) before the first pass; a second call before it
 * replaces the rule.  RT_ERR_INVALID_ARGUMENT without RT_FLAG_NOISE, after a pass, for tau negative or NaN, k < 1,
 * m < 2 or m <= samples_done (the probe's samples).
 *   Checkpoints are the sample counts c = m + j k (j >= 0), a fixed lattice: they do not depend on the target, the
 *   pacing or rt_frame_extend.  A pass never crosses one: rt_frame_advance also cuts its window at the next checkpoint.
 *   When a pass ends on a checkpoint c, the same rt_frame_advance call runs the check: every pixel still being sampled
 *   whose E over samples [0, c) is <= tau (E in double, exactly as rt_frame_noise computes it: the complement of its
 *   summary's E > tolerance) stops there, with its sums, count and Q.
 *   So every pixel p holds samples [0, n_p): n_p = n_probe for a pixel the probe stopped, the first checkpoint at which it
 *   converged, or samples_done for a pixel still being sampled; bit for bit rt_render's pixel p at samples_per_pixel =
 *   n_p.  n_p is a function of the frame's inputs and the rule only: the frame is the same whatever the pacing, and a
 *   frame extended from 256 to 512 samples is the frame opened at 512.
 *   Progress: samples_done is the count of the pixels still being sampled; pixels_flagged keeps its meaning;
 *   paths_target = paths_done + pixels_active (samples_target - samples_done), exact if nothing more converges, so it
 *   never grows between two rt_frame_extend calls; when a check leaves no pixel active, samples_done becomes
 *   samples_target (done) without a launch.  rt_frame_noise's summary covers the pixels still being sampled: right after
 *   a check, pixels_above == pixels at tolerance tau.  The check (one thread per pixel, then the compaction of the
 *   remaining flags) is part of its pass's last_pass_ms.
 * rt_frame_convergence fails (RT_ERR_INVALID_ARGUMENT) on a frame without a rule. */
typedef struct RtFrameConvergence {
    double tolerance;          /* tau, as set                                                                        */
    int32_t min_samples;       /* m                                                                                  */
    int32_t interval;          /* k                                                                                  */
    int32_t next_check;        /* the first checkpoint above samples_done                                            */
    int32_t checks;            /* checks run so far                                                                  */
    uint64_t pixels_active;    /* pixels still being sampled (pixels_flagged before the first check)                 */
    uint64_t pixels_converged; /* pixels stopped by a check; pixels_active + pixels_converged == pixels_flagged       */
} RtFrameConvergence;
int rt_frame_set_convergence(RtFrame *frame, double tolerance, int32_t min_samples, int32_t interval);
int rt_frame_convergence(RtFrame *frame, RtFrameConvergence *out);

/* ---- progressive frames of many views (host buffers; one GPU) ------------------------------------ */
/* A progressive frame whose pixels are a batch of views: rt_render_views' tall frame (n_views * rows rows, view v at
 * offset v*rows*cols) driven in passes, with the noise estimate and the convergence rule above.  A turntable rendered to
 * a noise target pays each pass's fixed costs (the tail of the persistent kernel, a synchronisation, a counter copy) once
 * for the batch instead of once per view.
 *
 * These two functions were added without a change of RT_ABI_VERSION (still 6): no struct and no existing prototype
 * changed.  A caller detects the feature by the presence of the symbol rt_frame_begin_views.
 *
 * rt_frame_begin_views returns an ordinary RtFrame: rt_frame_advance, _read, _extend, _noise, _set_convergence,
 * _convergence and _destroy accept it unchanged.  rt_frame_read writes n_views*rows*cols*3 bytes (sums
 * n_views*rows*cols*4); rt_frame_noise's maps and its summary cover the whole batch; the counts of RtFrameProgress and
 * RtFrameConvergence are sums over the views.
 *   Arguments as rt_render_views: n_views >= 1, cameras non-NULL, the same samples_per_pixel and bounce_depth on every
 *   camera, n_views * rows * cols < 2^31 (RT_ERR_INVALID_ARGUMENT otherwise); seeds NULL: opts->seed for every view.
 *   Modes as rt_frame_begin: RT_MODE_MEGAKERNEL only; RT_FLAG_FLOW and RT_FLAG_COUNTERS: RT_ERR_UNSUPPORTED, with or
 *   without RT_FLAG_NOISE.
 *   The frame owns its table of view cameras and keys: rt_render_views, rt_render and other frames may run on the scene
 *   between two passes.
 * Exactness.  Every sample is keyed by (view seed, pixel within the view, sample index) and the sums, Q and counts are
 *   integers, so after any pass view v is bit for bit the progressive frame of cameras[v] and seeds[v] at the same
 *   samples_done (and rt_render's frame at that samples_per_pixel).  Under a convergence rule each pixel's stopping count
 *   depends only on its own samples and the checkpoint lattice: view v of a converging batch is a converging frame of
 *   camera v with the same rule, whatever the pacing of either.
 * rt_frame_view_noise fills per_view[0 .. n_views) (n_views = 1 for a frame of rt_frame_begin): view v's summary over its
 *   pixels still being sampled, bit for bit rt_frame_noise's summary of the frame of camera v and seed v in the same state
 *   (the same fixed-order reduction over the view's pixels).  pixels == 0: the view is finished.  RT_ERR_INVALID_ARGUMENT
 *   for a frame opened without RT_FLAG_NOISE, a NULL per_view, or a negative or NaN tolerance. */
int rt_frame_begin_views(RtScene *scene, const RtCamera *cameras, const uint64_t *seeds, int32_t n_views,
                         int32_t max_width_coord, int32_t max_height_coord, const RtRenderOpts *opts,
                         RtFrame **out, RtFrameProgress *progress);
int rt_frame_view_noise(RtFrame *frame, double tolerance, RtFrameNoise *per_view /* n_views entries */);

/* ---- a window of a frame (host buffers; one GPU) ------------------------------------------------- */
/* Any rectangle of rt_render's frame, bit for bit, without tracing the rest: a closer look at one part of the image (a
 * caustic, a reflection) at the frame's own camera, or a tile of a frame rendered by several processes, which assemble
 * into the frame with nothing to blend at the seams.
 *
 * These two functions were added without a change of RT_ABI_VERSION (still 6): no struct and no existing prototype
 * changed.  A caller detects the feature by the presence of the symbol rt_render_window.
 *
 * The window is [row0, row0 + rows) x [col0, col0 + cols), rows and cols counted as rt_render's output (row 0 = top row;
 * the frame is (2 max_h + 1) x (2 max_w + 1)).  rgb_out rows*cols*3, sums_out (optional) rows*cols*4 int32, row-major over
 * the window.
 * Exactness.  Every sample is keyed by (seed, frame pixel, sample index), a path depends only on that key and the camera's
 *   full extents, and the sums are integers; the probe's flag of a pixel depends only on its own samples.  So window pixel
 *   (r, c) is bit for bit pixel (row0 + r, col0 + c) of rt_render(scene, camera, max_w, max_h, opts): sums, RGB8 and gamma
 *   RGB8, whatever the window, and tiles of any grid reassemble into rt_render's frame.
 * Argument errors (RT_ERR_INVALID_ARGUMENT): rows < 1 or cols < 1; row0 < 0 or col0 < 0; row0 + rows > 2 max_h + 1 or
 *   col0 + cols > 2 max_w + 1; rgb_out (or out) NULL; and those of rt_render.
 * Options.  RT_MODE_WAVEFRONT, RT_FLAG_FLOW and RT_FLAG_COUNTERS: RT_ERR_UNSUPPORTED (no window wavefront, flow-schedule or
 *   counting kernels).  RT_FLAG_NO_SMEM, RT_FLAG_WIDE_BVH, RT_FLAG_BVH2, RT_FLAG_NO_LEAN, RT_FLAG_LOCKSTEP, adaptive and
 *   gamma act as in rt_render; RT_FLAG_NOISE acts as in rt_frame_begin, and rt_render_window ignores it.
 * Stats (optional): the window's own paths, rays, degenerate_paths and pixels_early_out (of its pixels); the _ms fields and
 *   launches describe the call; box_tests and prim_tests are 0.  A window that is the whole frame is rt_render in every
 *   output, stats included.
 * Like rt_render, the call returns with its device work complete. */
int rt_render_window(RtScene *scene, const RtCamera *camera, int32_t max_width_coord, int32_t max_height_coord,
                     int32_t row0, int32_t col0, int32_t rows, int32_t cols, const RtRenderOpts *opts,
                     uint8_t *rgb_out, int32_t *sums_out, RtStats *stats);
/* A progressive frame over that window: an ordinary RtFrame (rt_frame_advance, _read, _extend, _noise, _view_noise,
 * _set_convergence, _convergence and _destroy take it unchanged; read and the noise maps are rows*cols, and
 * rt_frame_view_noise gives one entry).  The counts of RtFrameProgress and RtFrameConvergence cover the window's pixels.
 * Arguments and modes as rt_render_window.  After any pass, and under a convergence rule, window pixel (r, c) is bit for
 * bit pixel (row0 + r, col0 + c) of rt_frame_begin's frame of the same camera, extents, opts and rule: sums, counts, Q and
 * the E map (each pixel's stopping count depends only on its own samples and the checkpoint lattice). */
int rt_frame_begin_window(RtScene *scene, const RtCamera *camera, int32_t max_width_coord, int32_t max_height_coord,
                          int32_t row0, int32_t col0, int32_t rows, int32_t cols, const RtRenderOpts *opts,
                          RtFrame **out, RtFrameProgress *progress);

/* ---- denoised previews of progressive frames (host buffers; one GPU) ----------------------------- */
/* A clean preview of a progressive frame after its first passes, and the first-hit feature buffers it is guided by: an
 * object-id map for selection masks, depth, normals and albedo for compositing or an external denoiser.  Both work on any
 * RtFrame (rt_frame_begin, rt_frame_begin_views, rt_frame_begin_window); outputs have rt_frame_read's layout (the tall
 * frame of a batch, the window's pixels of a window).
 *
 * These two functions were added without a change of RT_ABI_VERSION (still 6): no existing struct or prototype changed.
 * A caller detects the feature by the presence of the symbol rt_frame_denoise.
 *
 * rt_frame_features: for each pixel, sample s < samples is the camera ray that the frame's path for (seed, pixel, s)
 *   starts with (for a batch, the view's camera and seed; for a window, the frame's pixel), one closest hit (the binary
 *   tree walk, as rt_test_hit_object with traversal 0) and one first scatter (Hittable.Reflection) of a white colour:
 *     prim_out    the caller's Hittable index hit by sample 0; -1 for a miss;
 *     albedo_out  per channel the integer sum over the samples of the colour the scatter leaves in the path
 *                 (darken(albedo, combine(white, surface)) for a scattering surface, the emitted colour for an absorbing
 *                 one, black for a miss or a scatter that fails), divided by samples with truncation (PixelStats.mean);
 *     normal_out  the shading normal scatter computes (oriented against the ray, F10, F11), summed in float32 in sample
 *                 order over the samples that hit and divided by their number; (0, 0, 0) if none hit;
 *     depth_out   the hit distance t, summed and divided the same way; +inf if none hit.
 *   The features are exact functions of (seed, pixel, samples): the same before and after any pass, under any pacing,
 *   convergence rule or rt_frame_extend.  The frame keeps them (computed once per samples value).  Each output is optional.
 *   RT_ERR_INVALID_ARGUMENT for a NULL frame or samples outside [1, 64].
 *
 * rt_frame_denoise: an edge-avoiding a-trous wavelet filter (Dammertz et al. 2010) over the frame's current means, its colour
 *   weight scaled by each pixel's standard error E (as SVGF scales it by its variance, Schied et al. 2017) and stopped at
 *   edges by the features of feature_samples samples.  It reads the frame and writes buffers of its own: the sums, Q,
 *   flags, list and counters are untouched, so a frame that is denoised between passes ends as one that never was.  It
 *   needs Q: RT_ERR_INVALID_ARGUMENT for a frame opened without RT_FLAG_NOISE, a NULL frame or opts, iterations outside
 *   [1, 10], feature_samples outside [1, 64], or a sigma that is not > 0 and finite as a float32; the options are checked
 *   first, before any device work.  Suggested options and where they come from: DESIGN.md section 19.
 *   Every operation below is an IEEE float32 operation rounded to nearest, evaluated as written, left to right:
 *     input     c_p = float(T_c) / float(n), v_p = float(E_p) * float(E_p) (E as rt_frame_noise); a pixel with n = 0 is
 *               output black and is no pixel's neighbour;
 *     level k   (k = 0 .. iterations - 1) out_p = sum_q w_pq c_q / sum_q w_pq over the taps q = (r + 2^k j, c + 2^k i),
 *               j outer, i inner, both -2..2, skipping taps outside the frame, outside p's view (a batch) and pixels with
 *               n = 0; c is the previous level's output (the input at k = 0), v always the input's;
 *     weight    w_pq = h_j h_i * W(x_c) * W(x_n) * W(x_a) * W(x_z), h = (1, 4, 6, 4, 1) (the product h_j h_i is exact),
 *               W(x) = 1 / (1 + x * (1 + 0.5 * x));
 *     colour    d = |c_p - c_q|^2 = (dr*dr + dg*dg) + db*db; x_c = 0 if d == 0, else d / (s_k * s_k * (v_p + v_q)) with
 *               s_k = float(sigma_colour) * 2^-k, the product s_k * s_k first;
 *     normal    x_n = |n_p - n_q|^2 / (s_n * s_n), s_n = float(sigma_normal);
 *     albedo    x_a = |a_p - a_q|^2 / (s_a * s_a), 8-bit levels, s_a = float(sigma_albedo);
 *     depth     x_z = 0 if z_p == z_q; +inf if either is +inf; else t * t with t = (z_p - z_q) / (s_z * z_p),
 *               s_z = float(sigma_depth).
 *   linear_out (optional, n_pixels*3 float) is the last level; rgb_out (optional, n_pixels*3) is that value clamped to
 *   [0, 255], truncated, and passed through PixelOutput.correct when gamma is non-zero, as rt_frame_read's gamma.
 * Both calls return with their device work complete, like every rt_frame_* call. */
int rt_frame_features(RtFrame *frame, int32_t samples,
                      int32_t *prim_out,   /* n_pixels                  */
                      uint8_t *albedo_out, /* n_pixels*3                */
                      float *normal_out,   /* n_pixels*3                */
                      float *depth_out);   /* n_pixels                  */
typedef struct RtDenoiseOpts {
    int32_t iterations;      /* a-trous levels; level k uses tap spacing 2^k; 1..10                         */
    int32_t feature_samples; /* F of the guide features, 1..64                                              */
    double sigma_colour;     /* > 0: scales the per-pixel standard errors in the colour weight; halved per level */
    double sigma_normal;     /* > 0                                                                         */
    double sigma_albedo;     /* > 0, 8-bit levels                                                           */
    double sigma_depth;      /* > 0, relative to the centre pixel's depth                                   */
    int32_t gamma;           /* rgb_out through PixelOutput.correct, as rt_frame_read                       */
    int32_t _pad0;
} RtDenoiseOpts;
int rt_frame_denoise(RtFrame *frame, const RtDenoiseOpts *opts,
                     uint8_t *rgb_out,   /* n_pixels*3, optional                               */
                     float *linear_out); /* n_pixels*3 filtered means in 8-bit levels, optional */

/* The same frame split over the GPUs of this process (the F# host is one process): replicated scene,
 * sample-index split (Scene.fs:191-192 shared out by sample index), probe tiles shared out by tile.
 * The devices exchange flags and sums through NVLink peer memory inside the kernels that consume them
 * (no separate collective): the last kernel sums every device's PixelStats buffer for its slice of the
 * pixels with peer loads, divides (Pixel.fs:103-108), applies gamma and stores RGB8 to pinned host
 * memory.  Results are bit-identical for every device count (integer sums keyed by sample index).
 * All devices must have peer access to one another (RT_ERR_UNSUPPORTED otherwise). */
typedef struct RtMulti RtMulti;
int rt_multi_create(const RtHittable *objects, int32_t n_objects, const RtTexture *textures,
                    int32_t n_textures, const int32_t *devices, int32_t n_devices, RtMulti **out);
int rt_multi_render(RtMulti *multi, const RtCamera *camera, int32_t max_width_coord,
                    int32_t max_height_coord, const RtRenderOpts *opts, uint8_t *rgb_out,
                    int32_t *sums_out, RtStats *stats);
void rt_multi_destroy(RtMulti *multi);
/* A progressive frame split over the devices of an RtMulti: rt_frame_begin's frame, with its passes, noise estimate,
 * convergence rule, features and denoised previews, at the speed of several GPUs.
 *
 * This function was added without a change of RT_ABI_VERSION (still 6): no struct and no existing prototype changed.  A
 * caller detects the feature by the presence of the symbol rt_multi_frame_begin.
 *
 * It returns an ordinary RtFrame: rt_frame_advance, _read, _extend, _noise, _view_noise (one entry), _set_convergence,
 * _convergence, _features, _denoise and _destroy take it unchanged.
 *   Arguments, modes and refusals are rt_frame_begin's, checked before any device work: RT_MODE_WAVEFRONT and RT_FLAG_NOISE
 *   with RT_FLAG_FLOW or RT_FLAG_COUNTERS are RT_ERR_UNSUPPORTED; a NULL multi or out is RT_ERR_INVALID_ARGUMENT, and *out
 *   is NULL after any failure.  RT_FLAG_FLOW and RT_FLAG_COUNTERS without RT_FLAG_NOISE are accepted and act as in
 *   rt_frame_begin (the split kernels of rt_multi_render).
 * Exactness.  Device r probes the tiles t with t mod world == r and, in a pass over [s, s + k), traces the sample
 *   indices s + r + j world (j >= 0) into buffers of its own; the sums, counts and Q are integers keyed by (seed, pixel, sample index), and the first device sums
 *   them over the devices before anything reads them.  So after every pass, and under a convergence rule, the frame is bit
 *   for bit rt_frame_begin's frame of the same camera, extents, opts and rule on one device of the same scene: sums,
 *   counts, RGB8 and gamma RGB8; Q, the E map and the RtFrameNoise summary (the same fixed-order reduction, on the first
 *   device); every field of RtFrameProgress and RtFrameConvergence except the _ms fields and passes; rt_frame_features and
 *   rt_frame_denoise.  This holds for every device count: only the number of passes may depend on it.
 * Pacing.  As rt_frame_begin's, with the device time per sample index of the slowest device; a paced window that neither
 *   max_samples, a checkpoint nor the target cuts is rounded down to a multiple of the device count when it holds at least
 *   that many indices, so that no device idles.
 * Timing.  last_pass_ms is the largest of the devices' own spans of the pass (as rt_multi_render's kernel_ms), device_ms
 *   the sum of those pass times and the slowest device's probe.
 * Ownership.  The frame owns its buffers on every device (about 29 bytes per pixel on each, 25 more on the first), so
 *   rt_multi_render and other frames may run on the same RtMulti between two passes.  Every call returns with its device
 *   work complete on every device.  The frame must be destroyed before its RtMulti. */
int rt_multi_frame_begin(RtMulti *multi, const RtCamera *camera, int32_t max_width_coord, int32_t max_height_coord,
                         const RtRenderOpts *opts, RtFrame **out, RtFrameProgress *progress);
/* A batch of views split over the devices of an RtMulti, in one call or as a progressive frame: rt_render_views' and
 * rt_frame_begin_views' tall frame (n_views * rows rows, view v at rows [v rows, (v + 1) rows)), split by sample index as
 * rt_multi_render splits one frame.  A batch of small views makes each device's share of the work large again, where one
 * rt_multi_render per view would give each device 1 / world of a frame already too small to hide its fixed costs.
 *
 * These two functions were added without a change of RT_ABI_VERSION (still 6): no struct and no existing prototype
 * changed.  A caller detects the feature by the presence of the symbol rt_multi_render_views.
 *
 *   Arguments are the union of rt_render_views' and rt_multi_render's (rt_frame_begin_views' and rt_multi_frame_begin's),
 *   checked before any device work: a NULL multi, out or rgb_out, n_views < 1, NULL cameras, cameras with differing
 *   samples_per_pixel or bounce_depth, and n_views * rows * cols >= 2^31 are RT_ERR_INVALID_ARGUMENT; RT_MODE_WAVEFRONT,
 *   RT_FLAG_FLOW and RT_FLAG_COUNTERS are RT_ERR_UNSUPPORTED (the kernels of a batch have no such variant).  *out is NULL
 *   after any failure.  seeds may be NULL (every view then has opts->seed).
 * Exactness.  Device r probes the tiles t with t mod world == r of the tall frame (a tile may straddle two views) and traces
 *   the sample indices s + r + j world; every device holds its own copy of the table of view cameras and keys.  So
 *   rt_multi_render_views equals rt_render_views on one device of the same arrays bit for bit, for every device count: RGB8
 *   with and without gamma, the sums, and the RtStats paths, rays, degenerate_paths and pixels_early_out (box_tests and
 *   prim_tests are 0; the _ms fields describe the slowest device, as in rt_multi_render).  rt_multi_frame_begin_views
 *   returns an ordinary RtFrame, and after every pass, under a convergence rule too, it is rt_frame_begin_views' frame on
 *   one device in everything rt_multi_frame_begin's frame equals rt_frame_begin's, and in every entry of
 *   rt_frame_view_noise; only the number of passes may depend on the device count, and rt_multi_frame_begin's pacing
 *   applies.
 * Ownership.  As rt_multi_frame_begin's frame, plus its table of views on every device; the frame must be destroyed before
 *   its RtMulti. */
int rt_multi_render_views(RtMulti *multi, const RtCamera *cameras, const uint64_t *seeds, int32_t n_views,
                          int32_t max_width_coord, int32_t max_height_coord, const RtRenderOpts *opts,
                          uint8_t *rgb_out, int32_t *sums_out, RtStats *stats);
int rt_multi_frame_begin_views(RtMulti *multi, const RtCamera *cameras, const uint64_t *seeds, int32_t n_views,
                               int32_t max_width_coord, int32_t max_height_coord, const RtRenderOpts *opts,
                               RtFrame **out, RtFrameProgress *progress);
/* ---- saving a progressive frame and resuming it ---------------------------------------------------- */
/* A progressive frame written to bytes and opened again later, in this process or another, on one device or on an RtMulti
 * of any device count: a frame that took minutes survives its process, and a one-GPU preview can be finished on eight.
 *
 * These three functions were added without a change of RT_ABI_VERSION (still 6): no existing struct or prototype changed.  A
 * caller detects the feature by the presence of the symbol rt_frame_save.
 *
 * rt_frame_save writes the frame into out[0, *len).  *len is always set: out == NULL with cap == 0 only sizes the snapshot
 *   (no device work); a cap below *len writes nothing (RT_ERR_INVALID_ARGUMENT).  It takes every frame (one camera, a batch
 *   of views or a window, of one device or of an RtMulti) at any point: right after its opener, between passes, on a
 *   checkpoint, after rt_frame_extend, or done.  A frame whose scene was edited since it opened is refused
 *   (RT_ERR_INVALID_ARGUMENT), as rt_frame_advance refuses it.  The frame itself is not changed.  The copy into out is fast
 *   if the caller pinned it (rt_host_pin).
 * rt_frame_resume and rt_multi_frame_resume open an ordinary RtFrame from a snapshot; every rt_frame_* call takes it.
 *   Exactness: after resuming, and after every further pass, the frame equals the saved frame continued without
 *   interruption in everything rt_multi_frame_begin's frame equals rt_frame_begin's (sums, counts, RGB8, Q, the E map,
 *   rt_frame_noise and rt_frame_view_noise, every RtFrameProgress and RtFrameConvergence field except the _ms fields and
 *   passes, rt_frame_extend, rt_frame_features and rt_frame_denoise), whatever the device counts at save and at resume.
 *   passes continues from the snapshot; last_pass_ms and device_ms cover this process only (device_ms starts with the
 *   restore).  The first paced pass is sized from the saved device time per sample index, scaled by the ratio of the
 *   device counts.  rt_frame_set_convergence is accepted exactly when the saved frame would have accepted it.
 *   Refusals, before any device allocation, with *out NULL: RT_ERR_INVALID_ARGUMENT for a NULL argument, a bad magic,
 *   version, length or checksum, and a scene whose content differs from the saved one (its fingerprint, object count or
 *   texture count); RT_ERR_UNSUPPORTED for a scene created with device = -1, and for a window given to
 *   rt_multi_frame_resume (windows run on one GPU); then every refusal of the frame's opener for the saved arguments.  A
 *   snapshot that passes these checks but whose pixels break the frame's rules (below) is refused with
 *   RT_ERR_INVALID_ARGUMENT naming the first bad pixel; the half-built frame is freed.
 *   The scene fingerprint hashes the object array and texture table as the scene holds them now (every field but padding
 *   and pointers, and the texels), not its tree: a snapshot taken after rt_scene_update or rt_scene_rebuild resumes on
 *   rt_scene_create of the same arrays, bit for bit except where a closest hit is an exact tie in t (rt_scene_update).
 *
 * Format (little-endian; version 1).  RtSnapshotHeader, then for a batch of views n_views entries of {RtCamera, uint64
 * seed} (the caller's cameras and seeds), then the pixel sections of n_pixels pixels (the tall frame of a batch, the
 * window's pixels of a window):
 *   sums    n_pixels x int32[4] {sumR, sumG, sumB, count}, as rt_frame_read gives them;
 *   Q       n_pixels x uint64, only when opts.flags has RT_FLAG_NOISE;
 *   flags   the pixels still being sampled, bit p % 32 of uint32 word p / 32, the words padded to an even count (zeros).
 * checksum = sum over i of mix(i, w_i) mod 2^64, w_i the i-th little-endian uint64 word of the file with the checksum
 *   field read as 0, and mix(i, w) = f(w + (i + 1) 0x9E3779B97F4A7C15) with splitmix64's finalizer
 *   f(z): z = (z ^ z >> 30) 0xBF58476D1CE4E5B9; z = (z ^ z >> 27) 0x94D049BB133111EB; z ^ z >> 31.
 * Each pixel satisfies: a pixel still being sampled has count == samples_done; any other has count == n_probe or a
 *   checkpoint of the rule m + j k <= samples_done; each channel sum lies in [0, 255 count] and Q in [0, 3 255^2 count].
 *   Over the frame: the counts sum to paths_done, pixels_active pixels are still sampled, and pixels_flagged pixels are
 *   still sampled or hold more than n_probe samples.
 * A frame with RT_FLAG_NOISE takes about 24 bytes a pixel (8.3 M pixels: about 200 MB), 16 without. */
#define RT_SNAPSHOT_VERSION 1
enum RtFrameKind { RT_FRAME_CAMERA = 0, RT_FRAME_VIEWS = 1, RT_FRAME_WINDOW = 2 };
typedef struct RtSnapshotHeader {
    char magic[8];              /* "RTFSSNAP"                                                                  */
    uint32_t version;           /* RT_SNAPSHOT_VERSION                                                         */
    uint32_t header_bytes;      /* sizeof(RtSnapshotHeader) = 344                                              */
    uint64_t total_bytes;       /* the whole snapshot                                                          */
    uint64_t checksum;          /* above                                                                       */
    uint64_t scene_fingerprint; /* of the scene the frame traced                                               */
    int32_t n_objects, n_textures;
    int32_t kind;               /* RtFrameKind                                                                 */
    int32_t n_views;            /* 1 unless kind == RT_FRAME_VIEWS                                             */
    RtCamera camera;            /* the opener's camera (the first view's for a batch)                          */
    int32_t max_width_coord, max_height_coord;
    int32_t window[4];          /* RT_FRAME_WINDOW: row0, col0, rows, cols                                     */
    RtRenderOpts opts;          /* the opener's                                                                */
    int32_t samples_per_pixel;  /* the frame's, after any rt_frame_extend                                      */
    int32_t samples_done, samples_target, n_probe, passes, _pad0;
    uint64_t n_pixels, pixels_flagged, pixels_active, paths_done;
    double conv_tolerance;      /* the convergence rule (conv_interval == 0: none)                             */
    int32_t conv_min, conv_interval, conv_checks;
    int32_t pace_devices;       /* the device count ms_per_sample was measured at                              */
    double ms_per_sample;       /* the pacing estimate (< 0: none yet)                                         */
} RtSnapshotHeader;
int rt_frame_save(RtFrame *frame, void *out, size_t cap, size_t *len);
int rt_frame_resume(RtScene *scene, const void *snapshot, size_t len, RtFrame **out, RtFrameProgress *progress);
int rt_multi_frame_resume(RtMulti *multi, const void *snapshot, size_t len, RtFrame **out, RtFrameProgress *progress);

/* create + render + destroy in one call */
int rt_render_multi(const RtHittable *objects, int32_t n_objects, const RtTexture *textures,
                    int32_t n_textures, const int32_t *devices, int32_t n_devices,
                    const RtCamera *camera, int32_t max_width_coord, int32_t max_height_coord,
                    const RtRenderOpts *opts, uint8_t *rgb_out, int32_t *sums_out, RtStats *stats);

/* ---- render (device buffers; one rank of a sample-split job) -------------------------------- */
/* All d_* pointers are device pointers on the scene's device; `stream` is a cudaStream_t.
 * d_stats: rows*cols*4 int32 {sumR,sumG,sumB,count}; d_flags: rows*cols uint8.
 *
 * Phase 1 — renderPixel's first two loops (Scene.fs:172-188) for the pixel tiles owned by
 * rank/world: adds the 2*firstTrial+1 probe samples into d_stats and sets d_flags[p] = 1 where the
 * two truncated means differ (the pixel continues).  With adaptive = 0 this only sets flags.
 * Buffers must be zeroed by the caller before phase 1. */
int rt_device_probe(RtScene *scene, const RtCamera *camera, int32_t max_width_coord,
                    int32_t max_height_coord, const RtRenderOpts *opts, int32_t rank, int32_t world,
                    int32_t *d_stats, uint8_t *d_flags, void *stream, RtStats *stats);
/* Phase 2 — the third loop (Scene.fs:191-192): for every flagged pixel, this rank's share of the
 * remaining sample indices (index mod world == rank) is added into d_stats.  d_flags must hold
 * the combined flags of all ranks (all-reduce max/sum between the phases when world > 1). */
int rt_device_main(RtScene *scene, const RtCamera *camera, int32_t max_width_coord,
                   int32_t max_height_coord, const RtRenderOpts *opts, int32_t rank, int32_t world,
                   int32_t *d_stats, const uint8_t *d_flags, void *stream, RtStats *stats);
/* Work counters of this scene accumulated since its last rt_device_probe call: paths, rays, (with
 * RT_FLAG_COUNTERS) box_tests / prim_tests; pixels_early_out holds the number of pixels that went ON to
 * phase 2.  One small device->host copy and a synchronisation of `stream`; call it outside timed regions. */
int rt_device_counters(RtScene *scene, void *stream, RtStats *stats);
/* PixelStats.mean (Pixel.fs:103-108) + optional PixelOutput.correct: d_stats (after the sum
 * all-reduce) -> d_rgb rows*cols*3. */
int rt_device_finalize(int32_t device, const int32_t *d_stats, int32_t n_pixels, int32_t gamma,
                       uint8_t *d_rgb, void *stream);

/* ---- render (one process per GPU; the collectives are issued by the library) -------------------- */
/* The sample-split frame of SURVEY.md 8e for a job of `world` processes, one per GPU, each holding a replica of
 * the scene: rank r probes its share of the tiles (Scene.fs:172-188), the flags are all-reduced (MAX), rank r
 * adds its share of the remaining sample indices (Scene.fs:191-192), the PixelStats sums are reduce-scattered
 * (int32 SUM) so that every rank divides (Pixel.fs:103-108) and gamma-corrects (ImageOutput.fs:11-18) one slice
 * of the pixels, and the RGB8 slices are all-gathered (as ONE kernel over NVLink peer memory where the ranks' buffers can
 * be mapped into one another, see rt_comm_uses_peer_memory; else with ncclReduceScatter / ncclAllGather).  All of it — kernels and NCCL calls — is enqueued by
 * rt_comm_render on one stream; the image is bit-identical to rt_render's for every world size.
 * NCCL (libnccl.so.2) is bound at run time on first use: RT_ERR_UNSUPPORTED if it cannot be loaded.
 *
 * Bootstrap as with NCCL itself: one rank calls rt_comm_unique_id, the host program hands the 128 bytes to every
 * rank (the F# host: a file, a pipe or MPI; bench.py: torch.distributed's store), every rank calls rt_comm_create
 * (collective).  `stream`: the cudaStream_t to enqueue on, or NULL for a stream owned by the communicator. */
#define RT_COMM_ID_BYTES 128
typedef struct RtComm RtComm;
int rt_comm_unique_id(uint8_t *id_out /* RT_COMM_ID_BYTES */);
int rt_comm_create(const uint8_t *id, int32_t rank, int32_t world, int32_t device, void *stream,
                   RtComm **out);
void rt_comm_destroy(RtComm *comm); /* collective, like rt_comm_create */
/* 1 when the ranks' sum and frame buffers are mapped into one another (CUDA IPC over NVLink peer access) and the tail of a
 * frame — sum over ranks, divide, gamma, gather — is ONE kernel of peer loads and peer stores between two 4-byte barriers;
 * 0 when that mapping was refused on some rank (or RTFS_COMM_NO_PEER=1) and the tail is ncclReduceScatter + finalize +
 * ncclAllGather.  Decided collectively whenever the communicator (re)allocates its buffers. */
int rt_comm_uses_peer_memory(const RtComm *comm);
/* version (e.g. 22809) and file name of the NCCL build the library bound */
int rt_comm_nccl_version(int32_t *version_out, char *path_out, size_t path_cap);
/* One frame (collective: every rank calls it with the same camera, extents and opts, on its own replica of the
 * scene).  rgb_out / sums_out: host buffers as for rt_render, or NULL on ranks that do not want them (the
 * frame is complete in device memory on every rank either way; passing sums_out makes the ranks all-reduce the
 * sums instead of reduce-scattering them).  stats: THIS rank's paths and rays.  With rgb_out, sums_out and
 * stats all NULL the call only enqueues work and returns without synchronising (device-resident use). */
int rt_comm_render(RtComm *comm, RtScene *scene, const RtCamera *camera, int32_t max_width_coord,
                   int32_t max_height_coord, const RtRenderOpts *opts, uint8_t *rgb_out,
                   int32_t *sums_out, RtStats *stats);
/* Timing and work counters of the last rt_comm_render that was enqueued with rgb_out, sums_out and stats all
 * NULL, once the caller has synchronised the stream: kernel_ms, main_ms, total_ms from the events the call
 * recorded; paths, rays, main_rays from counter snapshots it copied to pinned memory. */
int rt_comm_last_stats(RtComm *comm, RtScene *scene, RtStats *stats);
/* device pointers of the last frame: RGB8 rows*cols*3, and the sum buffer (complete only after a call with
 * sums_out or world == 1; otherwise only this rank's slice holds totals).  Valid until the next call. */
int rt_comm_frame(RtComm *comm, const uint8_t **d_rgb_out, const int32_t **d_stats_out);

/* ---- per-primitive conformance entry points (device) ---------------------------------------- */
/* Each runs one thread per vector through exactly the __device__ function the render kernels call.
 * Inputs/outputs are host pointers; doubles are rounded to FP32 on upload where the device
 * function takes FP32. */

/* Sphere.firstIntersection (Sphere.fs:349-386).  t_out[i] = NaN when there is no hit. */
int rt_test_sphere_hit(int32_t device, int32_t n, const double *origin, const double *dir,
                       const double *centre, const double *radius, double *t_out);
/* InfinitePlane.intersection (InfinitePlane.fs:125-136). */
int rt_test_plane_hit(int32_t device, int32_t n, const double *origin, const double *dir,
                      const double *point, const double *normal, double *t_out);
/* BoundingBox.hits with inverseDirections (BoundingBox.fs:25-94): the decision-exact slab test that the
 * reference-order traversal (rt_test_hit_object traversal = 1) runs.  The render traversal uses a
 * conservative variant of it (padded, culled by the best hit); that one is covered by
 * rt_test_hit_object traversal = 0. */
int rt_test_aabb_hit(int32_t device, int32_t n, const double *origin, const double *dir,
                     const double *box_min, const double *box_max, uint8_t *hit_out);
/* Scene.hitObject (Scene.fs:62-91).  prim_out = index into the caller's Hittable array or -1;
 * traversal: 0 = the render kernels' ordered/culled traversal of the binary SAH tree,
 *            1 = exhaustive left-then-right DFS of the reference-topology tree (F12),
 *            2 = the render kernels' traversal of the 8-wide compressed tree (big scenes, RT_FLAG_WIDE_BVH). */
int rt_test_hit_object(RtScene *scene, int32_t traversal, int32_t n, const double *origin,
                       const double *dir, int32_t *prim_out, double *t_out, double *strike_out);
/* Hittable.Reflection (Hittable.fs:8-12 -> Sphere.fs:150-300 / InfinitePlane.fs:43-99) with
 * explicit uniforms: uniforms[4*i..] are the FloatProducer draws for vector i (GetThree uses
 * [0..2], Get uses [0]); retries re-use the same draws rotated by one (they never happen on
 * non-degenerate inputs).  absorbed_out[i] = 1 when the reference returns ValueSome colour. */
int rt_test_reflection(RtScene *scene, int32_t n, const int32_t *prim, const double *origin,
                       const double *dir, const double *strike, const uint8_t *colour_in,
                       const double *uniforms, uint8_t *absorbed_out, uint8_t *colour_out,
                       double *origin_out, double *dir_out, uint8_t *inside_out);
/* traceOnce's ray generation (Scene.fs:129-144): one ray per (row, col, rand1, rand2), where
 * row/col are the signed coordinates renderPixel receives. */
int rt_test_camera_rays(int32_t device, const RtCamera *camera, int32_t max_width_coord,
                        int32_t max_height_coord, int32_t n, const int32_t *row, const int32_t *col,
                        const double *rand1, const double *rand2, double *origin_out, double *dir_out);
/* Texture.colourAt on the primitive's texture (Texture.fs:12-15, :50-67). */
int rt_test_texture(RtScene *scene, int32_t n, const int32_t *prim, const double *point,
                    uint8_t *colour_out);
/* Pixel.combine + Pixel.darken (Pixel.fs:136-151) on the device, explicit albedo. */
int rt_test_combine_darken(int32_t device, int32_t n, const uint8_t *a, const uint8_t *b,
                           const double *albedo, uint8_t *out);
/* The counter-based RNG: uniforms of (seed, pixel, sample, bounce, retry) as the device draws them. */
int rt_test_rng(int32_t device, uint64_t seed, int32_t n, const uint32_t *pixel,
                const uint32_t *sample, const uint32_t *bounce, const uint32_t *retry,
                uint32_t *words_out /* 4n */, double *uniforms_out /* 4n */);
/* traceOnce for explicit (pixel row/col, sample index): the final Pixel of that one path. */
int rt_test_trace_samples(RtScene *scene, const RtCamera *camera, int32_t max_width_coord,
                          int32_t max_height_coord, uint64_t seed, int32_t n, const int32_t *row_idx,
                          const int32_t *col_idx, const int32_t *sample, uint8_t *colour_out,
                          int32_t *rays_out);

/* FP32 FMA microbenchmark used as the roofline denominator (DESIGN.md §roofline): returns
 * measured TFLOP/s of a dependent-chain FFMA kernel filling the device. */
int rt_measure_fp32_peak(int32_t device, double *tflops_out);

#ifdef __cplusplus
}
#endif
#endif /* RTFS_B200_H */
