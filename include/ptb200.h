/* ptb200.h -- C-ABI of libptb200.so: the B200-native drop-in for the ray-cast +
 * radiance-integration path of OclPathTracer.
 *
 * The reference drives this path through ADL's header-template C++ API
 * (adl::DeviceUtils / Buffer<T> / Launcher, no ABI of its own).  Every entry
 * point below names the ADL call it replaces (paths relative to the reference
 * root).  Plain pointers and sizes only; every function returns 0 on success or
 * a negative PTB_E_* code, and ptb_last_error() holds a thread-local message
 * (the reference reports nothing in release builds: ADLASSERT expands to
 * `if(x){}`, Adl/AdlError.h:51).
 *
 * Threading: like ADL (one in-order queue per device, Adl/CL/AdlCL.cpp:215) a
 * ptb_device owns ONE CUDA stream and is single-host-thread.
 *
 * There is no CPU fallback: without a CUDA device ptb_device_create fails.
 */
#ifndef PTB200_H
#define PTB200_H

#include <stddef.h>
#include <stdint.h>

#include "SharedHeader.h"

#ifdef __cplusplus
extern "C" {
#endif

#define PTB_OK 0
#define PTB_E_INVALID -1   /* bad argument */
#define PTB_E_CUDA -2      /* a CUDA runtime call or kernel launch failed */
#define PTB_E_NODEVICE -3  /* no usable CUDA device */
#define PTB_E_IO -4        /* file could not be read / parsed */
#define PTB_E_NOTFOUND -5  /* unknown kernel name */
#define PTB_E_NOMEM -6

typedef struct ptb_device ptb_device;
typedef struct ptb_buffer ptb_buffer;
typedef struct ptb_kernel ptb_kernel;
typedef struct ptb_scene ptb_scene;

const char* ptb_last_error(void);
int ptb_version(void);

/* ---- device: adl::init + DeviceUtils::allocate / deallocate ---------------------
 * Adl/Adl.h:96,125-126; Adl/Adl.cpp:39-58,160-208.  Like DeviceCL::initialize
 * (Adl/CL/AdlCL.cpp:154) the index is clamped to the last device.              */
int ptb_device_count(int* count);
int ptb_device_create(int device_index, ptb_device** out);
/* same, but enqueue on a caller-owned cudaStream_t (e.g. torch's current stream) */
int ptb_device_create_on_stream(int device_index, void* cuda_stream, ptb_device** out);
int ptb_device_destroy(ptb_device* dev);
/* DeviceUtils::waitForCompletion(const Device*)  Adl/Adl.h:127, Adl/CL/AdlCL.cpp:282-285 */
int ptb_device_sync(ptb_device* dev);
/* Device::getDeviceVersion(char[128])  Adl/Adl.h:164 (names the PPM) */
int ptb_device_name(ptb_device* dev, char out[128]);
int ptb_device_sm_count(ptb_device* dev, int* sm_count);
/* Device::getMaxAllocationSize / memory accounting  Adl/Adl.h:168-170,173 */
int ptb_device_memory(ptb_device* dev, size_t* free_bytes, size_t* total_bytes);
void* ptb_device_stream(ptb_device* dev);

/* ---- buffers: adl::Buffer<T>  Adl/Adl.h:203-265, Adl/Adl.inl:145-253 ------------
 * Buffer(device, nElems) -> create(bytes); ~Buffer -> destroy;
 * write/read (Adl.h:218-220, async on the device queue) -> write/read;
 * getHostPtr/returnHostPtr (Adl.h:230-232, Adl/CL/AdlCL.inl:434-455: map whole
 * buffer RW, caller then waits; unmap publishes writes) -> map/unmap.          */
int ptb_buffer_create(ptb_device* dev, size_t bytes, ptb_buffer** out);
/* non-owning view of caller-allocated device memory (a torch tensor's storage) */
int ptb_buffer_wrap(ptb_device* dev, void* device_ptr, size_t bytes, ptb_buffer** out);
int ptb_buffer_destroy(ptb_buffer* buf);
int ptb_buffer_write(ptb_buffer* buf, const void* host_src, size_t bytes, size_t dst_offset);
int ptb_buffer_read(ptb_buffer* buf, void* host_dst, size_t bytes, size_t src_offset);
int ptb_buffer_map(ptb_buffer* buf, void** host_ptr);
int ptb_buffer_unmap(ptb_buffer* buf, void* host_ptr);
int ptb_buffer_clear(ptb_buffer* buf); /* Buffer<T>::clear  Adl/Adl.h:226 */
void* ptb_buffer_device_ptr(ptb_buffer* buf);
/* ptb_launch1d keys its resident scene and its frame-ahead batch on the buffers' contents as written through THIS API
 * (write / unmap / clear).  A tBuffer or matBuffer rewritten behind its back -- by a kernel or copy using
 * ptb_buffer_device_ptr, or by an IPC peer -- must be marked, or the old scene keeps rendering.                   */
int ptb_buffer_mark_dirty(ptb_buffer* buf);
size_t ptb_buffer_size(ptb_buffer* buf);

/* ---- kernel + launcher -----------------------------------------------------------
 * Device::getKernel(fileName, funcName)  Adl/Adl.h:166, Adl/CL/AdlCL.cpp:490-493,
 * KernelManager::query Adl/AdlKernel.cpp:94-224: name -> kernel, cached for the
 * device's lifetime, NULL when unknown.  Here the table holds AOT-compiled CUDA
 * entry points; file_name may carry the reference's path
 * ("../test/ClKernels/GenerateColors") -- only its basename is matched.        */
int ptb_kernel_get(ptb_device* dev, const char* file_name, const char* func_name, ptb_kernel** out);
/* the reference's compile-time #defines (GenerateColors.cl:5-6) as run-time
 * options: "NUM_TRIANGLES" (36), "BOUNCES" (16), "ACCEL" (PTB_ACCEL_*),
 * "INTEGRATOR" (PTB_INTEGRATOR_*), and "FRAME_AHEAD" (1): when the caller steps
 * through consecutive frame indices (the loop at RaytraceTest.cpp:248-262) the
 * samples of the following frames are traced together in one launch that fills
 * the GPU and each ptb_launch1d folds its own frame into the framebuffer --
 * bit-identical to FRAME_AHEAD 0 (one integrator launch per call).            */
int ptb_kernel_set_int(ptb_kernel* k, const char* name, int value);
/* Launcher::setBuffers + setConst + launch1D  Adl/AdlKernel.h:166-184,
 * Adl/AdlKernel.inl:179-184, Adl/CL/AdlKernelUtilsCL.cpp:399-500.  Positional:
 * buffers first, then the by-value constant block.  For "GenerateColors":
 * bufs = {tBuffer, matBuffer, gDst}, consts = ptb_int4{W, H, frame, -}; one
 * call = one sample per pixel + the gamma-space running mean
 * (GenerateColors.cl:302-322).  n_threads must equal W*H (the reference rounds
 * the grid up to 64 and has no guard; this one guards).                        */
int ptb_launch1d(ptb_device* dev, ptb_kernel* k, ptb_buffer* const* bufs, int n_bufs, const void* consts,
                 size_t const_bytes, int n_threads, int local_size);

/* Launch capture / replay: Launcher::serializeToFile / deserializeFromFile
 * (Adl/AdlKernel.h:185-188, Adl/CL/AdlKernelUtilsCL.cpp:509-620).  Same byte layout as the reference writes:
 * int32 nArgs; per argument { int32 isBuffer; int32 sizeInBytes; bytes }; then ExecInfo
 * { int32 nWIs[3]; int32 wgSize[3]; int32 nDim } -- so a dump taken from the reference's OpenCL run of
 * GenerateColors replays here.  _serialize reads the buffers back (it synchronises); _deserialize creates one
 * ptb_buffer per buffer argument (caller destroys them) and returns the by-value block and the launch shape. */
int ptb_launch_serialize(ptb_device* dev, const char* path, ptb_buffer* const* bufs, int n_bufs, const void* consts,
                         size_t const_bytes, int n_threads, int local_size);
int ptb_launch_deserialize(ptb_device* dev, const char* path, ptb_buffer** bufs_out, int buf_cap, int* n_bufs,
                           void* consts_out /* >= 64 bytes */, size_t* const_bytes, int* n_threads, int* local_size);

/* ---- host-side scene helpers: RaytraceTest.cpp:87-198 loadModel -------------------- */
int ptb_load_model(const char* path, ptb_triangle** tris, int* n_tris, ptb_material** mats, int* n_mats);
/* BUILD-DEFINED C5 scene: each quad (triangle pair) -> k x k sub-quads */
int ptb_tessellate(const ptb_triangle* tris, int n_tris, int k, ptb_triangle** out, int* n_out);
int ptb_light_from_quad(const ptb_triangle* tris, int n_tris, int quad, float p1[3], float ea[3], float eb[3]);
void ptb_free(void* p);
/* RaytraceTest.cpp:78-83,:277-287: sqrt, x255, truncate, clamp -> ASCII "P3" */
int ptb_to_rgb8(const float* rgba, int n_pixels, uint8_t* rgb);
/* the same transform on the device (identical bytes): float4 frame buffer -> 3 bytes per pixel in rgb (>= 3 * n_pixels
 * bytes, 16-byte aligned), asynchronous on the frame buffer's device stream */
int ptb_buffer_to_rgb8(ptb_buffer* frame, int n_pixels, ptb_buffer* rgb);
int ptb_write_ppm(const char* path, const float* rgba, int width, int height);

/* ---- resident scene: triangles re-laid out + BVH (BUILD-DEFINED) --------------------- */
typedef struct ptb_bvh_params {
    int32_t max_leaf;   /* 1..8, default 4 */
    float pad_rel;      /* child boxes are grown by pad_rel * scene diagonal, default 1e-4.  Must be finite and > 0: 0, negative
                           and NaN are refused, because without a pad the fp32 boxes of FLAT and 4-wide scenes lose hits
                           (measured on a planar scene).  The smallest value at which every form still equals the brute-force
                           loop for ray origins within 100 scene diagonals is 1e-5 on the generated scenes of
                           tests/test_traversal_scenes.py; at 3e-6 the planar scenes already lose hits (DESIGN.md section 4) */
    int32_t n_bins;     /* SAH bins, default 16 */
    int32_t smem_nodes; /* top-of-tree nodes laid out first (BFS) for shared-memory staging, default 1024 */
    float traverse_cost; /* SAH cost of one node visit relative to one triangle test (<= 0: default 1.2) */
    int32_t force_width; /* 0 = pick the scene class (below); 1 | 4 | 2 = force the FLAT / 4-wide / binary form (A/B runs and tests;
                            ptb_scene_create fails when the scene does not qualify for the forced form) */
    int32_t builder;    /* the tree the device entry points (ptb_scene_create_gpu, ptb_scene_create_from_device) build:
                           PTB_BUILDER_LBVH (default; max_leaf and pad_rel apply) or PTB_BUILDER_SAH: on the device, the tree
                           ptb_scene_create(force_width = 2) builds on the host from the same records, byte for byte (nodes,
                           tri_order, ptb_scene_info, quantised nodes, so every render, intersect and shade result); max_leaf,
                           pad_rel, n_bins, smem_nodes and traverse_cost apply as on the host.  Other values are refused.  The host
                           entry points (ptb_scene_create, ptb_bvh_build_host) have one builder and ignore the field. */
    int32_t reserved[1];
} ptb_bvh_params;
#define PTB_BUILDER_LBVH 0 /* Morton-order LBVH (csrc/lbvh.cuh): the fastest build, more node visits per ray */
#define PTB_BUILDER_SAH 1  /* the host's binned-SAH tree, built on the device (csrc/sah_build.cuh) */
void ptb_bvh_params_default(ptb_bvh_params* p);

/* host-only build (no device needed): returns malloc'd arrays, release with ptb_free.  width = 2: ptb_bvh_node
 * records; width = 4: ptb_bvh_node4 records (the same tree collapsed; built for scenes of <= 2048 triangles);
 * width = 1: ptb_bvh_leafbox records (the FLAT form: <= 32 leaves and <= 64 triangles) */
int ptb_bvh_build_host(const ptb_triangle* tris, int n_tris, const ptb_bvh_params* bvh_params, int width, void** nodes,
                       int* n_nodes, int32_t** tri_order, ptb_bvh_tri** ordered_tris, int* depth, int* smem_nodes);

int ptb_scene_create(ptb_device* dev, const ptb_triangle* tris, int n_tris, const ptb_material* mats, int n_mats,
                     const ptb_bvh_params* bvh_params /* NULL = default */, ptb_scene** out);
/* same, but the BVH is built ON the device: milliseconds for millions of triangles instead of seconds.  By default the
 * Morton-order LBVH (csrc/lbvh.cuh), of lower tree quality than the host SAH build; bvh_params->builder = PTB_BUILDER_SAH builds
 * the host's SAH tree instead.  Needs >= 2 triangles.                                                                        */
int ptb_scene_create_gpu(ptb_device* dev, const ptb_triangle* tris, int n_tris, const ptb_material* mats, int n_mats,
                         const ptb_bvh_params* bvh_params /* NULL = default */, ptb_scene** out);
/* The same scene from records that already live on the device (triangles a torch pipeline made or deformed): tris holds n_tris
 * ptb_triangle and mats n_mats ptb_material records (64 bytes each, 16-byte aligned; a ptb_buffer_create buffer or a tensor's
 * storage through ptb_buffer_wrap, both of `dev`).  The tree, node bytes, tri_order, quantised nodes, grid, ptb_scene_info and
 * every render, intersect and shade result equal ptb_scene_create_gpu's for the same records.  bvh_params: builder selects the
 * tree (see ptb_bvh_params); force_width must be 0 or 2 (the FLAT and 4-wide forms need the host builder).  Needs 2 <= n_tris < 2^28 and
 * n_mats >= 1.  The records are checked on the device as ptb_scene_create_gpu checks them on the host (every id in
 * [0, n_mats); every vertex float, w included, |v| <= 3e38), and the message names the lowest offending triangle.  Read on
 * the device's stream, so a device made with ptb_device_create_on_stream on torch's current stream sees the work that wrote
 * them; synchronises and returns when the scene is ready.  The scene keeps its own copies: the caller may overwrite or free
 * tris and mats at once.                                                                                                    */
int ptb_scene_create_from_device(ptb_device* dev, ptb_buffer* tris, int n_tris, ptb_buffer* mats, int n_mats,
                                 const ptb_bvh_params* bvh_params /* NULL = default */, ptb_scene** out);
int ptb_scene_destroy(ptb_scene* scene);
int ptb_scene_info(ptb_scene* scene, int* n_nodes, int* n_tris, int* depth, int* smem_nodes);
/* form of the resident scene: 1 (FLAT: ptb_bvh_leafbox records, scenes of <= 32 leaves and <= 64 triangles), 4
 * (ptb_bvh_node4, scenes that fit a 32 KB shared-memory budget) or 2 (binary ptb_bvh_node, traversed from L2/HBM through
 * its quantised encoding ptb_bvh_nodeq) */
int ptb_scene_bvh_width(ptb_scene* scene);
/* form a render of `mode` (PTB_MODE_*) walks: a FLAT scene keeps its 4-wide tree resident too and uses it where the rays of a
 * warp are coherent (PTB_MODE_DIRECT); results are identical, the visit statistics follow the form */
int ptb_scene_mode_width(ptb_scene* scene, int mode);
/* host copies of the built tree (n_nodes records of the scene's width), for structural validation and tests */
int ptb_scene_copy_bvh(ptb_scene* scene, void* nodes, int32_t* tri_order);
/* width-2 scenes: the 32-byte quantised encoding of the binary tree that the kernels traverse (ptb_bvh_nodeq, n_nodes records)
 * and its grid (SharedHeader.h); qnodes may be NULL to fetch the grid only */
int ptb_scene_copy_bvh_quantized(ptb_scene* scene, uint32_t* qnodes, float grid_lo[3], float grid_step[3]);

/* ---- the hot path -------------------------------------------------------------------
 * per-pixel statistics of the LAST frame of a call (collect_stats = 1)          */
typedef struct ptb_pixel_stats {
    int32_t tri;               /* primary hit: index into the caller's triangle array, -1 miss */
    int32_t quad;              /* primary hit: Triangle.id */
    uint32_t t_bits;           /* primary hit: bits of t */
    uint32_t visits_primary;   /* BVH nodes fetched by the primary query */
    uint32_t visits_secondary; /* ... by every other query of the sample */
    uint32_t count;            /* AO: unoccluded rays; DIRECT: lit; PATH: segments traced */
    uint32_t id_hash;          /* h = h*31 + (tri+2) over secondary queries in order */
    uint32_t tri_tests;        /* Moller-Trumbore tests started by the sample */
} ptb_pixel_stats;

void ptb_render_params_default(ptb_render_params* p);
int ptb_render_local_pixels(const ptb_render_params* p);

/* Renders frames [first_frame, first_frame + n_frames) of this shard's pixels.
 * frame: float4 per local pixel (in/out for PTB_ACCUM_REFERENCE when
 * first_frame > 0).  stats: ptb_pixel_stats per local pixel or NULL.
 * counters: host pointer or NULL; when given the call synchronises.
 * Asynchronous on the device's stream otherwise.                               */
int ptb_render(ptb_device* dev, ptb_scene* scene, const ptb_render_params* params, ptb_buffer* frame,
               ptb_buffer* stats, ptb_counters* counters);

/* Scene queries on rays that already live on the device (a caller's camera, shadow or visibility rays, a torch pipeline).
 * rays: n_rays ptb_ray records (>= 32 * n_rays bytes, 32-byte aligned); hits: n_rays ptb_hit records (>= 16 * n_rays bytes);
 * stats: NULL or 2 x uint32 per ray (BVH nodes fetched, triangle tests started; >= 8 * n_rays bytes).  query = PTB_QUERY_*.
 * Results, visit and test counts are those of the render paths' queries on the scene's form (FLAT, 4-wide or quantised binary;
 * DESIGN.md section 4).  Like ptb_render: asynchronous on the device's stream, no allocation per call; counters (host pointer
 * or NULL) synchronise and return rays_closest / rays_any, and nodes / tri_tests when stats is given; the cumulative mode of
 * ptb_device_counters applies.  n_rays = 0 does nothing.                                                                 */
int ptb_scene_intersect(ptb_device* dev, ptb_scene* scene, int query, ptb_buffer* rays, int n_rays, ptb_buffer* hits,
                        ptb_buffer* stats, ptb_counters* counters);

/* Render-mode samples along rays that already live on the device (another viewpoint or lens, adaptively chosen pixels, rays a
 * torch pipeline produced).  Sample i is exactly what ptb_render computes for one pixel-frame after its camera step, with
 * rays[i].o, rays[i].d and rays[i].seed in place of the camera ray and the post-camera RNG state (ptb_sample_ray).
 *   rays      n_rays ptb_sample_ray records (>= 32 * n_rays bytes, 32-byte aligned)
 *   radiance  float4 per ray (>= 16 * n_rays bytes, 16-byte aligned): xyz after max(., 0), w = 1, the value ptb_render writes
 *             into a sample slot
 *   stats     NULL or ptb_pixel_stats per ray (>= 32 * n_rays bytes, 16-byte aligned), fields as for ptb_render
 * Read from params: mode, max_depth, ao_samples, ao_max_dist, light_quad and light_p1 / ea / eb (the light comes from light_quad
 * when ea is all zero, as for ptb_render).  Ignored: the image size, frames, accum, shard, output and frames_per_batch.
 * Refused: accel = PTB_ACCEL_BRUTE and integrator = PTB_INTEGRATOR_WAVEFRONT.  Every closest-hit query runs to tmax 1e20, as
 * the reference's do.  Asynchronous on the device's stream, no allocation per call; counters (host pointer or NULL)
 * synchronise and return the rays, nodes and tri_tests (with stats) and samples = n_rays; the cumulative mode of
 * ptb_device_counters applies.  n_rays = 0 does nothing.                                                              */
int ptb_scene_shade(ptb_device* dev, ptb_scene* scene, const ptb_render_params* params, ptb_buffer* rays, int n_rays,
                    ptb_buffer* radiance, ptb_buffer* stats, ptb_counters* counters);

/* End-to-end convenience with HOST buffers: uploads the scene records (H2D),
 * (re)builds the resident scene if the records changed, renders, reads the frame
 * (and stats) back (D2H) and synchronises.  out_rgba: float4 per local pixel. */
/* Image sharding with the exchange fused into the render (BUILD-DEFINED; the reference is single-device).  Every
 * rank owns a FULL image; ptb_buffer_ipc_export / _import map the images of the other ranks' processes (CUDA IPC:
 * peer memory over NVLink / NVSwitch).  ptb_render_gather renders this rank's shard (params->shard_*) and stores
 * each finished pixel at its global position in full_frame and in every peer image, so no collective and no
 * un-interleave pass follows -- only a barrier before the images are read.  With accum = REFERENCE the running state
 * is read from full_frame.  Results are bit-identical to a single-device ptb_render of the whole image.          */
int ptb_buffer_ipc_export(ptb_buffer* buf, void* handle64 /* 64 bytes out */);
int ptb_buffer_ipc_import(ptb_device* dev, const void* handle64, size_t bytes, ptb_buffer** out);
int ptb_render_gather(ptb_device* dev, ptb_scene* scene, const ptb_render_params* params, ptb_buffer* full_frame,
                      ptb_buffer* const* peer_frames, int n_peers /* 0..PTB_MAX_PEERS */, ptb_counters* counters);

int ptb_render_host(ptb_device* dev, const ptb_triangle* tris, int n_tris, const ptb_material* mats, int n_mats,
                    const ptb_render_params* params, float* out_rgba, ptb_pixel_stats* out_stats,
                    ptb_counters* counters);

/* With params->output = PTB_OUTPUT_RGB8 both host entry points run the reference's output transform on the device
 * (RaytraceTest.cpp:78-83,:283; identical bytes to ptb_to_rgb8 of the float4 frame) and out_rgba receives 3 bytes per
 * local pixel instead of 16 -- the image a PPM writer needs, at a fifth of the PCIe traffic.
 *
 * Pipelined form: _async enqueues H2D + render + D2H and returns; ptb_job_wait blocks until that job's
 * frame (and stats) are in the caller's buffers and releases the job (waiting twice for one job is an error).  At
 * most two jobs may be in flight (double buffering: job j's D2H overlaps job j+1's render).  Buffers from
 * ptb_host_alloc are pinned, so the copies go straight to / from them; pageable buffers are staged.  Counters are
 * not available here.
 * Accumulation across calls: accum = LINEAR carries nothing (every call returns the mean of ITS frames).  accum =
 * REFERENCE with first_frame > 0 continues the gamma-space running mean from the caller's out_rgba, which is read at
 * SUBMIT time -- so such a call is refused while another job is in flight (wait for it first): the reference's
 * progressive loop is sequential by definition (GenerateColors.cl:318-321).                                     */
typedef struct ptb_job ptb_job;
int ptb_render_host_async(ptb_device* dev, const ptb_triangle* tris, int n_tris, const ptb_material* mats, int n_mats,
                          const ptb_render_params* params, float* out_rgba, ptb_pixel_stats* out_stats,
                          ptb_job** job);
int ptb_job_wait(ptb_job* job);
int ptb_host_alloc(size_t bytes, void** out); /* page-locked host memory */
int ptb_host_free(void* p);

/* ---- several GPUs in one process (BUILD-DEFINED; the reference picks ONE device, Adl/CL/AdlCL.cpp:154) --------------
 * ptb_device_add_helper gives `dev` another device of the box that renders part of its work; peer access helper -> dev is
 * enabled (NVLink / NVSwitch).  Results never change: pixels are independent and a sample depends on (scene, W, H, pixel,
 * frame) only (GenerateColors.cl:305-308).  From then on
 *   - ptb_launch1d(dev, ...) deals the frames of its frame-ahead batch over dev and its helpers (each traces into its
 *     slice of the batch on dev through peer memory), so the unmodified RayCast loop uses every GPU;
 *   - ptb_render_multi shards ONE image over dev and its helpers (64-pixel blocks round-robin); every device's resolve
 *     kernel stores its pixels at their global position in the image on dev, which is then read back once.
 * One host thread drives all devices (asynchronous launches ordered with events).  A helper serves one device; destroy
 * helpers before or after their device in any order.                                                            */
int ptb_device_add_helper(ptb_device* dev, ptb_device* helper);
int ptb_device_helper_count(ptb_device* dev);
/* HOST buffers in, ONE host image out: out_rgba receives float4 per pixel of the whole image (or 3 bytes per pixel with
 * params->output = PTB_OUTPUT_RGB8); in/out for accum = REFERENCE with first_frame > 0.  params->shard_* must be unset.
 * Bit-identical to ptb_render_host on one device.  Synchronises.                                                */
int ptb_render_multi(ptb_device* dev, const ptb_triangle* tris, int n_tris, const ptb_material* mats, int n_mats,
                     const ptb_render_params* params, float* out_rgba, ptb_counters* counters);

/* ---- measurement hooks ----------------------------------------------------------------
 * (the reference's analogue: Device::toggleProfiling + the ms launch1D returns,
 * Adl/Adl.h:143-171, Adl/CL/AdlKernelUtilsCL.cpp:470-499).  With profiling on, every
 * render batch is bracketed by CUDA events on the device's stream; _read synchronises
 * and returns the totals since the previous read.  kernel_launches counts this
 * library's own kernel launches (always on).                                      */
int ptb_device_profile(ptb_device* dev, int enable);
/* Ray / node / test counters of the device.  By default every render call starts them at zero (and returns them when
 * asked).  cumulative = 1: the counters keep adding up over render calls until this function reads them (out != NULL:
 * synchronises, returns the totals since the previous read and clears them) -- exact ray counts over a whole timed
 * region without a synchronisation inside it.  cumulative = 0 restores the default; -1 leaves the mode as it is.      */
int ptb_device_counters(ptb_device* dev, int cumulative, ptb_counters* out);
/* experiment knobs for A/B measurements (results never change; DESIGN.md section 5); 0 = the default everywhere.  index:
 *  0  waiting lanes that trigger path regeneration (default 6; 4 in the large-scene state-machine kernel)
 *  1  log2 multiplier of the frame-ahead batch of ptb_launch1d
 *  2  = 2: keep the traversal stack of large scenes in shared memory instead of local memory
 *  3  CTA size 64 | 32 (default 128) of the megakernels
 *  4  BVH nodes staged per CTA for large scenes (default 0: none)
 *  5  PATH kernel: 1 = one sample per thread, 2 = while-while query inside a persistent path segment (k_mega_path_regen),
 *     3 = per-lane state machine (k_path_sm) for every scene form; default: state machine for large scenes, 2 otherwise
 *  6  = 1: wavefront stages without persistent ray fetch;  7  idle-lane count that triggers a wavefront refill (default 8)
 *  9  > 0: extra KB of shared memory per CTA, < 0: -n resident CTAs per SM (occupancy / latency sensitivity runs)
 *  10 lanes waiting for the shade phase, 11 lanes at a leaf, that make the state-machine kernels switch phase (defaults 20 | 16, 10)
 *  12 large-scene PATH kernel: 1 = registers-only k_path_sm (8 CTAs per SM), 9 = the same at 9 CTAs; default k_path_sm2 (path state
 *     parked in shared memory, 11 CTAs), 28 | 29 | 30 = at 8 | 9 | 10 CTAs, 32 | 33 = 4 | 8 node visits per vote at 10 CTAs (default 6)
 *  13 = 1: wavefront extend stage as a state machine for large scenes (default: while-while with dynamic fetch); = 2: FLAT scenes
 *     without the pooled triangle phase
 *  14 registers-only k_path_sm: 1 | 2 | 4 node visits per vote
 *  15 log2 of the sample slots kept in flight per launch (default 2^27 for PATH, 2^22 otherwise)                              */
int ptb_device_set_tuning(ptb_device* dev, int index, int value);
int ptb_device_profile_read(ptb_device* dev, float* integrator_ms, float* resolve_ms, int* integrator_launches,
                            uint64_t* kernel_launches);

/* ---- unit access for parity tests -----------------------------------------------------
 * scene query on caller-supplied rays (host arrays: o, d = 3 floats per ray).   */
int ptb_trace(ptb_device* dev, ptb_scene* scene, int accel, int any_hit, int n_rays, const float* o,
              const float* d, const float* tmax, int32_t* out_tri, float* out_t, float* out_u, float* out_v,
              uint32_t* out_visits, uint32_t* out_tests);
int ptb_test_sincos(ptb_device* dev, const float* x, int n, float* s, float* c);
int ptb_test_pow(ptb_device* dev, const float* x, int n, float y, float* out);
/* the branch-reduced IEEE helpers of the kernels: out6n = [1/x | sqrt(x) | safe reciprocal | normalize(x, x/2, 2x).xyz] */
int ptb_test_ieee(ptb_device* dev, const float* x, int n, float* out6n);
int ptb_test_rng(ptb_device* dev, uint32_t gid, uint32_t frame, int n, uint32_t* states, float* values);
int ptb_test_camera(ptb_device* dev, int width, int height, int frame, int n, const int32_t* gids, float* o,
                    float* d, uint32_t* seeds);

#ifdef __cplusplus
}
#endif
#endif /* PTB200_H */
