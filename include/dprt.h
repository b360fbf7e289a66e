/*
 * dprt.h -- C ABI of libdprt.so: the B200-native per-sample / per-bounce inner loop of the PG2024
 * data-parallel ray tracer, one opaque context per rank (= per GPU = per scene-chunk owner).
 *
 * The reference has no plugin/FFI layer; its boundary is the set of call sites inside
 * src/render/renderer.cpp:runSample (SURVEY.md section 8b). Each entry point below names the reference call
 * site it replaces (paths relative to the reference tree). Plain pointers and sizes only; every function
 * returns 0 on success or a negative dprt_error, never aborts, never throws across the boundary.
 * All "host" pointers are caller-owned host memory; the context owns every device buffer.
 * A context is driven by one host thread; all work is enqueued on one CUDA stream per context.
 */
#ifndef DPRT_H
#define DPRT_H

#include "dprt_types.h"

#ifdef __cplusplus
extern "C" {
#endif

typedef struct dprt_ctx dprt_ctx;
typedef struct dprt_bvh8 dprt_bvh8;

/* ---- lifecycle ------------------------------------------------------------------------------- */
/* MPI_Init + cudaSetDevice + buffer allocation (renderer.cpp:547-741 mallocBuffers/deferredMallocBuffers).
 * nccl_unique_id: 128 bytes from dprt_get_unique_id() on rank 0 (broadcast by the caller), or NULL for a
 * context that is only driven single-rank or through dprt_*_group(). */
int  dprt_get_unique_id(void* out128);
int  dprt_create(const dprt_config* cfg, int rank, int world, int device, const void* nccl_unique_id, dprt_ctx** out);
/* A second context of the same rank (other frame size / scene) that SHARES the parent's NCCL communicator instead of
 * creating one (several frames in one MPI job share MPI_COMM_WORLD the same way). Collective like dprt_create; the
 * communicator lives until the last context on it is destroyed (any order); the contexts' collectives must not interleave
 * across ranks. */
int  dprt_create_shared(const dprt_config* cfg, dprt_ctx* parent, dprt_ctx** out);
void dprt_destroy(dprt_ctx* ctx);
const char* dprt_last_error(const dprt_ctx* ctx);   /* ctx may be NULL: last create-time error */
int  dprt_synchronize(dprt_ctx* ctx);
int  dprt_get_stats(const dprt_ctx* ctx, dprt_stats* out);
int  dprt_reset_stats(dprt_ctx* ctx);

/* ---- scene (renderer.cpp:1725-1849: lights, AccelerationStructure table; GAS build is OptiX's) -- */
/* Host-side BVH8 build, exposed so that harnesses can inspect the structure the kernels walk. */
int  dprt_bvh8_build(const float* verts9, const int32_t* mat_ids, int64_t ntris, float pad, dprt_bvh8** out);
int  dprt_bvh8_info(const dprt_bvh8* b, int64_t* nnodes, int64_t* ntris, int32_t* max_depth);
int  dprt_bvh8_copy(const dprt_bvh8* b, dprt_bvh8_node* nodes_out, dprt_bvh8_tri* tris_out);
void dprt_bvh8_free(dprt_bvh8* b);

/* Scene object `scene_index` is real geometry on this rank: verts9 = ntris*9 floats, normals9 = ntris*9
 * floats (per-corner shading normals, HitGroupData.normals/normalIndices of pipeline_helper.cpp:182-193),
 * mat_ids = ntris ints into the material table. */
int  dprt_upload_chunk(dprt_ctx* ctx, int scene_index, const dprt_object_desc* desc, const float* verts9,
                       const float* normals9, const int32_t* mat_ids, int64_t ntris);
/* ---- BVH8 refit: moved vertices, same triangles (the counterpart of an OptiX acceleration-structure update) ------------
 * dprt_refit_chunk rewrites the device geometry of local chunk `scene_index` in place for new corner positions verts9
 * (ntris*9 floats, indexed by the original triangle index = primID, like the upload's) and, when the chunk was uploaded with
 * them, new normals9: the BVH8 keeps its topology and every node box is recomputed by the builder's own rule (DESIGN.md 3.9),
 * so the structure stays exact and conservative and hits are the ones of a fresh upload of the new vertices. Materials and
 * texture coordinates stay as uploaded. Returns after the context's stream is synchronised.
 * DPRT_ERR_INVALID with a message, and nothing on the device changed: a null array or context, an index that holds no local
 * chunk, ntris different from the upload's, a non-finite coordinate, a vertex outside the object's aabbMin / aabbMax (the box
 * other ranks route by and hold proxies of), normals9 given for a chunk uploaded without normals or missing for one with them.
 * The device memory is shared with every context that adopted the scene (dprt_adopt_scene): they all see the new geometry,
 * and none of them may have work in flight (the precondition of a re-upload). Proxies of this chunk trained on other ranks
 * are NOT retrained: they keep answering for the old geometry. A different triangle count needs dprt_upload_chunk, and so does
 * a deformation that scatters neighbouring triangles: the old grouping then makes every ray visit far more nodes (DESIGN.md 3.9).
 * dprt_refit_chunk_device: the same on device arrays; the checks run on the device (one reduction, one read-back).
 * dprt_spec_bvh8_refit: the refit on caller-owned host arrays (a dprt_bvh8_copy or dprt_chunk_bvh8_copy blob), in place, no
 * device; rejects, leaving the arrays unchanged, a blob whose childBase / triBase / primID point outside the arrays or whose
 * children do not follow their parent, and non-finite vertices. dprt_chunk_bvh8_copy reads back a chunk's device blob
 * (triangle records without the texture-coordinate tail); NULL outputs only query the sizes. */
int  dprt_refit_chunk(dprt_ctx* ctx, int scene_index, const float* verts9, const float* normals9, int64_t ntris);
int  dprt_refit_chunk_device(dprt_ctx* ctx, int scene_index, const void* verts9_dev, const void* normals9_dev, int64_t ntris);
int  dprt_spec_bvh8_refit(dprt_bvh8_node* nodes, int64_t nnodes, dprt_bvh8_tri* tris, int64_t ntris, const float* verts9);
int  dprt_chunk_bvh8_copy(dprt_ctx* ctx, int scene_index, int64_t* nnodes, int64_t* ntris, dprt_bvh8_node* nodes_out,
                          dprt_bvh8_tri* tris_out);
/* ---- BVH8 build on the GPU: new triangles (the counterpart of an OptiX acceleration-structure build) ----------------------
 * dprt_build_chunk makes local chunk `scene_index` out of verts9 (ntris*9 floats), normals9 (ntris*9 floats or NULL), uv6
 * (ntris*6 floats or NULL) and mat_ids (ntris ints or NULL), like dprt_upload_chunk_uv, but builds the BVH8 on the device
 * (Morton order, PLOC, the host builder's SAH-optimal collapse; DESIGN.md 3.10). The host arrays are staged through the
 * context's I/O buffer. The tree differs from the host builder's, the hits do not: a built chunk renders bit for bit like an
 * uploaded one. Everything after the build is dprt_upload_chunk_uv's: normals, the texture-coordinate tail, the depth levels
 * a later dprt_refit_chunk walks; the old geometry at the index is released once the context's streams are idle.
 * Returns after the context's stream is synchronised. DPRT_ERR_INVALID with a message, and the object at the index unchanged:
 * a null context, description or vertex array, an index out of range, ntris <= 0, a nodeID outside the world, a material id
 * outside [0, DPRT_MAX_MATERIALS), a non-finite coordinate. DPRT_ERR_CAPACITY: ntris >= 2^27 (checked before any array is
 * read) or a BVH8 deeper than 36 levels.
 * dprt_build_chunk_device: the same on device arrays; no triangle data goes through the host (the checks run on the device:
 * one reduction, one read-back; the build reads back one count per clustering iteration and per tree level).
 * dprt_spec_bvh8_build_gpu: the host twin of the device build (no device): the blob dprt_build_chunk_device makes, bit for
 * bit, as a handle for dprt_bvh8_info / dprt_bvh8_copy / dprt_bvh8_free (triangle records without texture coordinates).
 * DPRT_ERR_INVALID: null vertices or handle, ntris <= 0 or >= 2^27, a non-finite coordinate. */
int  dprt_build_chunk(dprt_ctx* ctx, int scene_index, const dprt_object_desc* desc, const float* verts9, const float* normals9,
                      const float* uv6, const int32_t* mat_ids, int64_t ntris);
int  dprt_build_chunk_device(dprt_ctx* ctx, int scene_index, const dprt_object_desc* desc, const void* verts9_dev,
                             const void* normals9_dev, const void* uv6_dev, const void* mat_ids_dev, int64_t ntris);
int  dprt_spec_bvh8_build_gpu(const float* verts9, const int32_t* mat_ids, int64_t ntris, dprt_bvh8** out);
/* Scene object `scene_index` is a proxy on this rank: AABB + world->object transform + the two proxy MLPs
 * (torch::jit::load of vis/depth modules, renderer.cpp:1884-1905). Weight blobs use the packed fp32 layout
 * documented in DESIGN.md ("proxy weight blob"); either may be NULL ("padding" entries of the reference). */
int  dprt_upload_proxy(dprt_ctx* ctx, int scene_index, const dprt_object_desc* desc, const void* vis_blob,
                       size_t vis_bytes, const void* depth_blob, size_t depth_bytes);
/* ---- real-scene front end (SURVEY.md 8f row 3: pipeline_helper.cpp:145-220, kernel.cu:190-292,311-359,
 * distributed_traversal_kernel.cu:82-158, renderer.cpp:1621-1721) -------------------------------------------------------
 * Geometry arrives the way the reference's SBT records hold it -- meshes with INDEXED normals and texture coordinates, placed
 * by (nested, host-composed) instance transforms -- and is flattened at upload: world-space corners, per-corner normals
 * (inverse-transpose of the instance matrix) and per-corner texture coordinates, primitive id = running index over
 * (instance, triangle). The closest-hit program then reads 36 + 24 contiguous bytes per hit instead of chasing two index
 * arrays (180 GB of HBM buy that; a two-level BVH for Moana-scale instancing is what comes next, DESIGN.md 6). The flatten is
 * host code and callable without a device: count first, then fill caller-owned arrays. uv6 may be NULL; has_uv (may be
 * NULL) tells whether any mesh carries texture coordinates. */
int64_t dprt_flatten_count(const dprt_mesh_desc* meshes, int n_meshes, const dprt_instance_desc* instances, int64_t n_instances);
int  dprt_flatten_instances(const dprt_mesh_desc* meshes, int n_meshes, const dprt_instance_desc* instances, int64_t n_instances,
                            float* verts9, float* normals9, float* uv6, int32_t* mat_ids, int* has_uv);
/* dprt_upload_chunk with per-corner texture coordinates (uv6 = ntris*6 floats: u0 v0 u1 v1 u2 v2; NULL = none). */
int  dprt_upload_chunk_uv(dprt_ctx* ctx, int scene_index, const dprt_object_desc* desc, const float* verts9, const float* normals9,
                          const float* uv6, const int32_t* mat_ids, int64_t ntris);
/* flatten + dprt_upload_chunk_uv: one scene object from its meshes and instances (GAS build + SBT records of the reference) */
int  dprt_upload_instanced_chunk(dprt_ctx* ctx, int scene_index, const dprt_object_desc* desc, const dprt_mesh_desc* meshes,
                                 int n_meshes, const dprt_instance_desc* instances, int64_t n_instances);
/* ---- instanced objects built and moved on the GPU (the counterparts of an OptiX IAS build and IAS update; DESIGN.md 3.11) ----
 * dprt_build_instanced_chunk: dprt_upload_instanced_chunk's object, made on the device. The indexed arrays and the instance
 * table (not the flattened triangles) are copied through the context; the device flattens them, bit for bit as
 * dprt_flatten_instances does, straight into dprt_build_chunk's GPU build. The chunk keeps its own copy of the indexed meshes
 * (shared with the contexts that adopt the scene, freed with the geometry) for dprt_update_instances. Returns after the
 * context's stream is synchronised. The checks are dprt_upload_instanced_chunk's (mesh and instance descriptions, the flattened
 * triangle count against 2^27 before any array is copied: DPRT_ERR_CAPACITY) and dprt_build_chunk's; DPRT_ERR_INVALID, with
 * the object at the index unchanged, also for a position, normal or texture-coordinate index outside its mesh's array and for a
 * singular or non-finite instance transform (checked on the device, read back with the other checks).
 * dprt_update_instances: new transforms for the instance list of the build (same count, same mesh per instance): flattened on
 * the device and refitted exactly as dprt_refit_chunk does it with the flattened moved instances. DPRT_ERR_INVALID, with
 * nothing changed: an index that holds no chunk made by dprt_build_instanced_chunk (a proxy, an uploaded chunk), another
 * instance count, an instance naming another mesh, a singular or non-finite transform, a vertex outside the object's
 * aabbMin / aabbMax. Preconditions as for dprt_refit_chunk: no context that shares the scene (dprt_adopt_scene) may have work
 * in flight, and proxies of this chunk on other ranks are not retrained. */
int  dprt_build_instanced_chunk(dprt_ctx* ctx, int scene_index, const dprt_object_desc* desc, const dprt_mesh_desc* meshes,
                                int n_meshes, const dprt_instance_desc* instances, int64_t n_instances);
int  dprt_update_instances(dprt_ctx* ctx, int scene_index, const dprt_instance_desc* instances, int64_t n_instances);
/* params.albedoTextures[texture_index] (renderer.cpp:1621-1721): width*height RGBA float texels, row 0 first (v = 0), filtered
 * bilinearly with wrap addressing on normalised coordinates like the reference's texture descriptor -- in software, in exact
 * binary32 (DESIGN.md 4), not by the texture unit's 9-bit fixed-point weights. rgba = NULL removes the texture. */
int  dprt_set_texture(dprt_ctx* ctx, int texture_index, const float* rgba, int width, int height);
/* HitGroupData.textureIndex per material (pipeline_helper.cpp:185): -1 = untextured. A textured material takes its base
 * colour from the texture (kernel.cu:251-281) and drops intersections whose opacity (alpha) is below 0.05 in EVERY trace --
 * the __anyhit__ah program of all five pipelines (kernel.cu:311-359, distributed_traversal_kernel.cu:110-158, ...). */
int  dprt_set_material_textures(dprt_ctx* ctx, const int32_t* texture_index, int n);
/* params.envLightTexture (renderer.cpp:1851; calculateEnvironmentLighting kernel.cu:28-48): lat-long RGBA float map looked up
 * at (phi / 2pi, theta / pi) after phi += rotation_offset; wraps in u, clamps in v. rgba = NULL restores the analytic sky
 * of cfg.envColor. */
int  dprt_set_env_map(dprt_ctx* ctx, const float* rgba, int width, int height, float rotation_offset);
/* Rough conductor (bsdfType 2, DESIGN.md 3.12): a GGX microfacet metal with Schlick Fresnel, F0 = the material's albedo
 * (baseColor, or the albedo-map texel of a textured material), Smith height-correlated masking, visible-normal sampling for
 * the next path and f(wi, wo) in place of albedo / pi for the light samples. roughness[m] in [0, 1] is material m's GGX
 * roughness (alpha = max(r^2, 1e-3)); 0 is a perfect mirror, a delta lobe that takes no light samples, like Water. The table
 * holds DPRT_MAX_MATERIALS entries, all 0 at create, shared by dprt_adopt_scene, and read only for bsdfType 2 and 3 materials.
 * For the glossy plastic (bsdfType 3, DESIGN.md 3.13) it is the roughness of the coat's specular lobe; 0 is a smooth coat whose
 * specular lobe is a mirror, while its diffuse base still takes the light samples.
 * DPRT_ERR_INVALID with the table unchanged: n outside [1, DPRT_MAX_MATERIALS], an entry not finite or outside [0, 1].
 * Waits for the context's streams, then replaces entries [0, n). */
int  dprt_set_material_roughness(dprt_ctx* ctx, const float* roughness, int n);
/* The two texture look-ups above on host arrays, compiled from the very source the kernels use (dprt_math.cuh): lets a
 * machine without a GPU compare the arithmetic with the oracle. out4 = n RGBA results. */
int  dprt_spec_texture_sample(const float* rgba, int width, int height, const float* u, const float* v, int64_t n, int clamp_v,
                              float* out4);
int  dprt_spec_env_lookup(const float* rgba, int width, int height, float rotation_offset, const float* dirs3, int64_t n, float* out3);
/* The conductor on host arrays, from the source the shading kernel compiles (conductor.cuh), per entry i: f0[3i..3i+2],
 * roughness[i], the local outgoing direction wo[3i..3i+2] (+z = the face-forwarded shading normal). _sample takes the two
 * uniforms xi[2i], xi[2i+1] and writes the next direction wi and the throughput factor weight (both 0 when the path ends);
 * _eval writes f(wi, wo) per channel. */
int  dprt_spec_conductor_sample(const float* f0, const float* roughness, const float* wo, const float* xi, int64_t n, float* wi,
                                float* weight);
int  dprt_spec_conductor_eval(const float* f0, const float* roughness, const float* wo, const float* wi, int64_t n, float* f);
/* The glossy plastic on host arrays, from the source the shading kernel compiles (plastic.cuh), per entry i: the diffuse colour
 * albedo[3i..3i+2], roughness[i], wo[3i..3i+2] as above. _sample takes three uniforms xi[3i..3i+2] (the third chooses the lobe)
 * and writes wi and weight (both 0 when the path ends); _eval writes f(wi, wo) per channel. */
int  dprt_spec_plastic_sample(const float* albedo, const float* roughness, const float* wo, const float* xi, int64_t n, float* wi,
                              float* weight);
int  dprt_spec_plastic_eval(const float* albedo, const float* roughness, const float* wo, const float* wi, int64_t n, float* f);

int  dprt_set_materials(dprt_ctx* ctx, const dprt_material* mats, int n);
int  dprt_set_lights(dprt_ctx* ctx, const dprt_light_tri* lights, int n);   /* renderer.cpp:1798-1808 */
int  dprt_set_camera(dprt_ctx* ctx, const dprt_camera* cam);                /* params.camera, :1990 */

/* ---- stage entry points: one per reference call site ----------------------------------------- */
int  dprt_reset_frame(dprt_ctx* ctx);                 /* resetFrameBuffers            renderer.cpp:416-451 */
int  dprt_begin_sample(dprt_ctx* ctx, int sample);    /* resetSampleBuffers + params  renderer.cpp:1497-1512 */
int  dprt_path_gen(dprt_ctx* ctx);                    /* optixLaunch(PathGen)         renderer.cpp:1514-1527 */
int  dprt_traverse(dprt_ctx* ctx);                    /* optixLaunch(TraRay)          renderer.cpp:1232-1243 */
int  dprt_partition(dprt_ctx* ctx);                   /* Work_Efficient_Scan          cuda_compaction.cu:352 */
int  dprt_exchange(dprt_ctx* ctx, int* done);         /* Alltoall+Alltoallv+Allreduce renderer.cpp:1254-1314 */
/* The host half of dprt_exchange, callable without a device: from the gathered W x (W+1) matrix of every rank's
 * transferOffset row (row s, column d = where rank s's segment for destination d starts) derive what rank `rank`
 * sends (send_count[W]), where each source's records land in its path buffer (recv_offset[W+1], recv_count[W]) --
 * the sendCount/recvCount/recvOffset vectors of renderer.cpp:1256-1277 -- and the termination flag of
 * renderer.cpp:1292-1298 (all_local = no record crossed ranks anywhere). Output pointers may be NULL. */
int  dprt_plan_exchange(const int32_t* gathered_offsets, int world, int rank, int32_t* send_count, int32_t* recv_offset,
                        int32_t* recv_count, int64_t* recv_total, int* all_local);
/* Host half of the settled-deque exchange (cfg.referenceMigrate == 0; DESIGN.md 3.4), callable without a device. The
 * partition of the travelling paths has W + 1 buckets: 0..W-1 by destination, W = the second piece of the self segment
 * (records that stay on the rank and came from HIGHER ranks; bucket `rank` holds the ones that came from lower ranks).
 * rows: W rows of W + 2 offsets. Outputs for rank `rank`: send_count[W] / recv_count[W] (the self entries are 0),
 * dst_offset[W] = where this rank's bucket d starts among the arrivals of rank d (arrivals are ordered by source rank),
 * piece[4] = {offset, count of the first self piece, offset, count of the second}, new_nl = records arriving from lower
 * ranks (they precede the ones from higher ranks in the new active set), new_active = all arrivals, all_local =
 * termination flag of renderer.cpp:1292-1298. Output pointers may be NULL. */
int  dprt_plan_exchange_deque(const int32_t* rows, int world, int rank, int32_t* send_count, int32_t* recv_count,
                              int32_t* dst_offset, int32_t* piece, int32_t* new_nl, int32_t* new_active, int* all_local);
int  dprt_shade(dprt_ctx* ctx);                       /* optixLaunch(MainRay)         renderer.cpp:1320-1347 */
int  dprt_reset_nn(dprt_ctx* ctx);                    /* resetNNBuffers               renderer.cpp:367-414 */
int  dprt_shadow_trace(dprt_ctx* ctx);                /* optixLaunch(ShadowRay)       renderer.cpp:1366-1379 */
int  dprt_secondary_trace(dprt_ctx* ctx);             /* optixLaunch(SecondaryRay)    renderer.cpp:1426-1437 */
/* which: 0 = shadow queries (mc*shadowPathSize slots), 1 = secondary queries (mc*pathSize slots).
 * inside_only != 0 is Work_Efficient_Scan_For_NN_HIT_INSIDE (cuda_compaction.cu:532), else ..._For_NN (:441). */
int  dprt_bucket_queries(dprt_ctx* ctx, int which, int inside_only, int* total);
/* kind: 0 = vis model -> pred[0..total), 1 = depth model -> pred[pred_offset..): the batched
 * torch::jit forward loops of renderer.cpp:768-839 (depth, offset 0), :841-1011, :1014-1159. */
int  dprt_proxy_infer(dprt_ctx* ctx, int kind, int pred_offset);
int  dprt_frame_buffer_update(dprt_ctx* ctx);         /* Frame_Buffer_Update   frame_buffer_update.cu:129 */
int  dprt_depth_buffer_update(dprt_ctx* ctx);         /* Depth_Buffer_Update   frame_buffer_update.cu:194 */
int  dprt_target_node_update(dprt_ctx* ctx);          /* Target_Node_Update    frame_buffer_update.cu:326 */
/* composite modules, same order as the reference helpers. The composites may schedule differently from a plain
 * sequence of the stage calls above -- the migrate loop keeps settled paths out of the per-iteration work
 * (cfg.referenceMigrate), dprt_render_sample runs the ShadowRay module beside the next TraRay loop on a second stream
 * (cfg.serialStages), MainRay reuses TraRay's hit (cfg.mainRayRetrace) -- but every buffer the reference defines holds the
 * same bytes when they return (DESIGN.md 3.1, 3.4). */
int  dprt_primary_ray_module(dprt_ctx* ctx);          /* primaryRayModule          renderer.cpp:1212-1318 */
int  dprt_shadow_ray_module(dprt_ctx* ctx);           /* shadowRayModuleBasedNN    renderer.cpp:1349-1405 */
int  dprt_secondary_ray_module(dprt_ctx* ctx);        /* secondaryRayModuleBasedNN renderer.cpp:1407-1452 */
int  dprt_render_sample(dprt_ctx* ctx, int sample);   /* runSample                 renderer.cpp:1457-1574 */
/* (direct+env)/spp on device, ncclReduce(sum) to root, copy to out_host (3*N floats, root only; may be NULL
 * elsewhere): renderer.cpp:2031-2052. */
int  dprt_reduce_image(dprt_ctx* ctx, int root, float* out_host);

/* ---- first-hit guide buffers (AOVs) for a denoiser ------------------------------------------------------------------
 * The reference's launch() takes normalImage and albedoImage beside the colour image (renderer.cpp:1576-1589); the
 * semantics here are this project's own (DESIGN.md 4). Off by default. dprt_enable_aov(ctx, 1) allocates, on the first
 * enable, one zeroed buffer of 6N floats (DPRT_BUF_AOV: albedo sums 3N, then normal sums 3N), which dprt_reset_frame clears.
 * Rule: dprt_begin_sample arms the context, and the first dprt_shade after it -- the camera paths' first surface hits on
 * this rank -- adds, per hit record, the albedo the shading program uses (material baseColor or albedo-map texel) and the
 * interpolated, normalised, face-forwarded shading normal to the record's pixel. Later dprt_shade calls of the sample add
 * nothing; a camera ray that hits nothing adds nothing. The per-stage entry points and dprt_render_sample[_group] follow
 * the same rule. dprt_accumulate_from adds the AOV sums too when both contexts have them on (DPRT_ERR_STATE when only one
 * does). dprt_reduce_aov: albedo/spp and normal/spp on device (not renormalised), ncclReduce(sum) to root when W > 1,
 * 3N floats each to albedo_host / normal_host on root (may be NULL elsewhere); collective like dprt_reduce_image.
 * dprt_reduce_aov_group sums the ranks in rank order on the host. Both return DPRT_ERR_STATE when AOVs were never enabled. */
int  dprt_enable_aov(dprt_ctx* ctx, int enable);
int  dprt_reduce_aov(dprt_ctx* ctx, int root, float* albedo_host, float* normal_host);
int  dprt_reduce_aov_group(dprt_ctx** ctxs, int world, int root, float* albedo_host, float* normal_host);

/* ---- denoiser: edge-avoiding a-trous wavelet filter guided by the first-hit albedo and normal --------------------------
 * The reference hands its colour, albedo and normal images to OptiX's denoiser (renderer.cpp:1576-1589); this build has no
 * OptiX, so it filters them itself (Dammertz et al. 2010, on albedo-demodulated colour; DESIGN.md 3.8 is the arithmetic
 * specification, bit for bit on GPU and host). Inputs are width x height pixels of 3 floats each, pixel (x, y) at
 * y * width + x: the layouts dprt_reduce_image and dprt_reduce_aov return. p == NULL selects the defaults: iterations 3,
 * sigma_color 2.0, sigma_normal 1.0, sigma_albedo 0.3 (DPRT_DENOISE_DEFAULT_*). The output may alias any input.
 * DPRT_ERR_INVALID, with nothing enqueued: a null context or array, width or height < 1, more than DPRT_DENOISE_MAX_PIXELS
 * pixels, iterations outside 1..10, a sigma that is not finite and > 0, or one whose weight constant 4^(L-1) / sigma_color^2,
 * 1 / sigma_normal^2 or 1 / sigma_albedo^2 is not finite and > 0 in binary32.
 * dprt_denoise / dprt_denoise_device run on the context's device and stream (the frame size need not be the context's;
 * not collective: call it on whichever rank holds the reduced frame) and return after the stream is synchronised. The
 * context keeps the scratch (56 bytes per pixel), grown to the largest call and freed by dprt_destroy; never allocated
 * when the denoiser is not used. dprt_spec_denoise runs the same arithmetic on the host, without a device. */
int  dprt_denoise(dprt_ctx* ctx, const dprt_denoise_params* p, int width, int height, const float* color_host,
                  const float* albedo_host, const float* normal_host, float* out_host);
int  dprt_denoise_device(dprt_ctx* ctx, const dprt_denoise_params* p, int width, int height, const void* color_dev,
                         const void* albedo_dev, const void* normal_dev, void* out_dev);
int  dprt_spec_denoise(const dprt_denoise_params* p, int width, int height, const float* color, const float* albedo,
                       const float* normal, float* out);

/* ---- samples in flight ----------------------------------------------------------------------------
 * Samples of a frame are independent (renderer.cpp:1993-2022 runs them one after the other). The late bounces and the later
 * migrate iterations of a sample carry 10^4..10^5 rays -- launches that last as long as their longest ray and leave most of
 * the GPU idle -- so a host may keep K samples in flight: K contexts of the same rank (dprt_create_shared), one host thread
 * each, context j rendering samples j, j + K, ... with dprt_render_sample. dprt_adopt_scene makes a context use another
 * one's uploaded scene (chunk geometry, proxies and their networks: shared device memory, freed with the last context that
 * uses it; materials, lights, camera: copied) -- a later re-upload on either side no longer reaches the other. dprt_accumulate_from adds another context's directLighting (plane 0) and
 * envLighting sums into this one's, after which dprt_reduce_image averages and reduces the whole frame. Each sample's
 * arithmetic is unchanged; only the order of the per-pixel sum over samples differs. The image is exact against the
 * per-context composition: each context's sums are those of its own samples in order (bit for bit the one-context result
 * of the same sample list), added into the first context in the order of the dprt_accumulate_from calls, then averaged
 * (tests/test_gpu_inflight.py). */
int  dprt_adopt_scene(dprt_ctx* ctx, dprt_ctx* from);
int  dprt_accumulate_from(dprt_ctx* ctx, dprt_ctx* other);

/* ---- peer-memory exchange (the data plane of dprt_primary_ray_module when every rank's buffers are reachable over
 * NVLink: MPI_Alltoall + MPI_Alltoallv + MPI_Allreduce of renderer.cpp:1254-1298 without a host round trip; DESIGN.md 3.4).
 * A context created with an NCCL id wires itself up inside dprt_create (and falls back to ncclSend/ncclRecv on all ranks
 * when any rank cannot; DPRT_P2P=0 forces the fallback). A host with its own bootstrap and no NCCL does it by hand:
 * every rank exports DPRT_P2P_HANDLE_BYTES, the host all-gathers them, every rank connects, the host agrees on
 * min(*connected) and tells every rank the verdict. All three calls are collective over the job. */
int  dprt_p2p_export(dprt_ctx* ctx, void* handle_out);
int  dprt_p2p_connect(dprt_ctx* ctx, const void* all_handles, int* connected);
int  dprt_p2p_enable(dprt_ctx* ctx, int enable);
int  dprt_p2p_enabled(const dprt_ctx* ctx);

/* ---- in-process rank group: W contexts driven by one thread (tests on fewer GPUs than ranks) --- */
int  dprt_exchange_group(dprt_ctx** ctxs, int world, int* done);
int  dprt_render_sample_group(dprt_ctx** ctxs, int world, int sample);
int  dprt_reduce_image_group(dprt_ctx** ctxs, int world, int root, float* out_host);

/* ---- state access for harnesses -------------------------------------------------------------- */
int  dprt_get_path_size(const dprt_ctx* ctx, int* path_size, int* shadow_path_size);
int  dprt_set_path_size(dprt_ctx* ctx, int path_size);
int  dprt_buffer_bytes(const dprt_ctx* ctx, int buffer_id, size_t* bytes);
int  dprt_download(dprt_ctx* ctx, int buffer_id, size_t offset_bytes, void* host, size_t bytes);
int  dprt_upload(dprt_ctx* ctx, int buffer_id, size_t offset_bytes, const void* host, size_t bytes);
int  dprt_enable_hit_prim(dprt_ctx* ctx, int enable);

/* ---- standalone operators --------------------------------------------------------------------- */
/* Closest hit of n host rays against this rank's local geometry: H2D, trace, D2H (the optixTrace closest-hit
 * launch of BASELINE config 2 through host buffers). */
int  dprt_trace_closest(dprt_ctx* ctx, const dprt_ray* rays_host, int64_t n, dprt_hit* hits_host);
/* Same on device-resident buffers obtained from dprt_device_alloc. */
int  dprt_trace_closest_device(dprt_ctx* ctx, const void* rays_dev, int64_t n, void* hits_dev);
/* Proxy MLP forward of scene object `scene_index`: x_host [n,5] fp16 -> y_host [n] fp16 (module.forward,
 * renderer.cpp:809-816). kind 0 = vis, 1 = depth. */
int  dprt_mlp_infer(dprt_ctx* ctx, int scene_index, int kind, const dprt_half* x_host, int64_t n, dprt_half* y_host);
int  dprt_mlp_infer_device(dprt_ctx* ctx, int scene_index, int kind, const void* x_dev, int64_t n, void* y_dev);

/* Training samples of the proxy of scene object `scene_index` (a LOCAL object of this rank): the Vis pipeline,
 * optix/vis_ray_kernel.cu:98-161 + copyOutputBuffersForTrainData renderer.cpp:264-285. Closest hit of each ray
 * against that object only (the reference uses tMin 1e-5, tMax inf: put them in the ray records);
 * features_host[5n] = ((o - aabbMin) / (aabbMax - aabbMin), phi / 2pi, theta / pi) of the ray in object space,
 * labels_host[n] = t / maxLength for a hit, exactly 1.0 for a miss -- the encoding trainingcode/datasets.py:149-227 reads. */
int  dprt_gen_train_data(dprt_ctx* ctx, int scene_index, const dprt_ray* rays_host, int64_t n, float* features_host,
                         float* labels_host);

/* The Precom pipeline, optix/precom_ray_kernel.cu:193-299 (+ copyOutputBuffersForTrainData renderer.cpp:264-285): the other
 * training-set generator. Each ray (a camera path: tMin 1e-2, tMax = path.tMax in the record) is intersected with the proxied
 * object's AABB -- front face, or back face with the direction reversed when the origin is inside -- and the MLP input is taken
 * AT THE AABB HIT: features_host[5n] = ((p_aabb - aabbMin) / (aabbMax - aabbMin), phi / 2pi, theta / pi) in object space; then
 * the object's original geometry is traced with tMax = inf and labels_host[n] = (t_geo - t_aabb) / maxLength. A ray that hits
 * the AABB but not the geometry gets the loaders' miss value 1.0 (the reference leaves the buffer's reset value there);
 * valid_host[n] = 0 for rays that miss the AABB (features 0: the reference writes nothing for them). */
int  dprt_gen_precom_data(dprt_ctx* ctx, int scene_index, const dprt_ray* rays_host, int64_t n, float* features_host,
                          float* labels_host, uint8_t* valid_host);

int  dprt_device_alloc(dprt_ctx* ctx, size_t bytes, void** dev_ptr);
int  dprt_device_free(dprt_ctx* ctx, void* dev_ptr);
int  dprt_memcpy_h2d(dprt_ctx* ctx, void* dev, const void* host, size_t bytes);
int  dprt_memcpy_d2h(dprt_ctx* ctx, void* host, const void* dev, size_t bytes);
/* CUDA-event timing on the context's stream (the harness times stages the way the kernels are launched). */
int  dprt_timer_start(dprt_ctx* ctx);
int  dprt_timer_stop(dprt_ctx* ctx, float* ms);
int  dprt_flush_l2(dprt_ctx* ctx);
/* Per-stage device time: when enabled every stage launch is bracketed by a CUDA-event pair on the context's
 * stream (the Timing::start/end sections of renderer.cpp:1245-1251,1262-1283 as device-side measurements).
 * ms_out / launches_out hold DPRT_STAGE_COUNT entries, accumulated since the last dprt_reset_stats. */
int  dprt_stage_profile(dprt_ctx* ctx, int enable);
int  dprt_get_stage_times(dprt_ctx* ctx, double* ms_out, int64_t* launches_out);
/* Instrumented traversal: when enabled the traversal kernels run in a counting variant that accumulates BVH8
 * nodes visited and triangles tested per stage (the algorithmic-byte basis of the roofline, DESIGN.md).
 * counts_out holds 2*DPRT_STAGE_COUNT entries {nodes, tris}. Results are unchanged; timing is not representative. */
int  dprt_enable_counters(dprt_ctx* ctx, int enable);
int  dprt_get_counters(dprt_ctx* ctx, uint64_t* counts_out);

#ifdef __cplusplus
}
#endif
#endif /* DPRT_H */
