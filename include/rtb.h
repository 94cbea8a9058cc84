/* rtb.h -- C ABI of the B200 ray-tracing hot path (librtb200.so).
 *
 * This is the drop-in boundary for ONE path of windy32/win32-ray-tracing-demo: per-pixel camera
 * ray generation -> ray/scene intersection through the regular-grid / flat-grid / k-d (median,
 * SAH) accelerators and the plane / sphere / triangle primitives -> Whitted `trace` and
 * Monte-Carlo `radiance` shading.  Every entry point cites the reference interface it replaces
 * (paths relative to the reference's src/RayTracingOpt/).
 *
 * Plain pointers and sizes only; no C++ / torch types.  The caller owns every host buffer it
 * passes; the library owns device memory behind the opaque handles.  All functions return
 * RTB_OK (0) or a negative rtb_status and are re-entrant per context (one context = one CUDA
 * device + one stream).  There is NO CPU fallback: without a CUDA device rtb_init fails.
 *
 * Host-side builders (grid, k-d tree: reference Tunnel.cpp:346-784) stay on the host and hand
 * their output over as the flattened SoA buffers of rtb_flat_scene.
 */
#ifndef RTB_H
#define RTB_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RTB_ABI_VERSION 5

typedef enum rtb_status {
    RTB_OK = 0,
    RTB_ERR_INVALID = -1,     /* bad argument / inconsistent flat scene          */
    RTB_ERR_NO_DEVICE = -2,   /* no usable CUDA device (there is no CPU path)    */
    RTB_ERR_CUDA = -3,        /* CUDA runtime error; see rtb_last_error          */
    RTB_ERR_UNSUPPORTED = -4, /* valid request outside the implemented path      */
    RTB_ERR_OOM = -5
} rtb_status;

/* ---- materials: reference Material.h:7-38 and subclasses, flattened to a tagged POD ------- */
enum { RTB_MAT_SOLID = 0,            /* SolidColorMaterial.cpp:11-19 (GlassMaterial.cpp:3-7 is SOLID white, (0,0,1), n=1.46) */
       RTB_MAT_CHECKER = 1,          /* CheckerMaterial.cpp:11-23                 */
       RTB_MAT_RADIANCE_CHECKER = 2, /* RadianceCheckerMaterial.cpp:12-29         */
       RTB_MAT_PHONG = 3 };          /* PhongMaterial.cpp:13-29                   */
enum { RTB_DIR_XOZ = 0, RTB_DIR_XOY = 1, RTB_DIR_YOZ = 2 }; /* CheckerMaterial.h:9 */

typedef struct rtb_material {
    int32_t kind;
    float diffusiveness, reflectiveness, refractiveness, refractive_index; /* Material.h:18-24 */
    float a[3];   /* SOLID: local colour;  PHONG: diffuse  */
    float b[3];   /* SOLID: emission;      PHONG: specular */
    float scale;  /* checker scale                         */
    float p;      /* RADIANCE_CHECKER: radiance; PHONG: shininess */
    int32_t dir;  /* RTB_DIR_*                             */
    int32_t pad_[2];
} rtb_material;   /* 64 bytes */

/* ---- top-level geometries: reference GeometrySet.cpp:95-110 iterates them in insertion order */
enum { RTB_PRIM_PLANE = 0,     /* Plane.cpp:3-34: v = normal xyz, position xyz, dist              */
       RTB_PRIM_SPHERE = 1,    /* Sphere.cpp:4-37: v = center xyz, radius                         */
       RTB_PRIM_TRIANGLES = 2, /* run of loose Triangle geometries (GeometrySet.cpp:33-86): first/count index loose_tri */
       RTB_PRIM_TUNNEL = 3,    /* the Tunnel geometry (Tunnel.cpp:1299-1309), traversed with `accel` */
       /* A triangle MESH (a loaded model; no reference counterpart): the fields of a TRIANGLES run -- first/count index
        * loose_tri (count >= 1), one material, triangle k has hit id base_id + k -- traversed through a bounding-volume
        * hierarchy that rtb_scene_upload builds on the device (one per record, also when ranges overlap).  Contract: the
        * nearest hit is the one the run of the same triangles returns -- the smallest t the reference's triangle test accepts, ties to the lowest k, compared with
        * the earlier records by the same strict `<` -- except when the run's winning pair lies in the grazing band
        * described in csrc/rtb_bvh.h (ray almost in the triangle's plane), where the reference's t is rounding noise.   */
       RTB_PRIM_MESH = 4 };

typedef struct rtb_prim {
    int32_t type;
    int32_t material; /* index into materials (ignored for TUNNEL: per-triangle) */
    int32_t base_id;  /* top-level geometry index of this record (of its first triangle for a run) */
    int32_t first, count; /* TRIANGLES, MESH: range in loose_tri */
    float v[7];
} rtb_prim;           /* 48 bytes */

/* ---- accelerators: reference Tunnel.h:16-22 ---------------------------------------------- */
enum { RTB_ACCEL_LINEAR = 0,       /* Tunnel.cpp:786-804  */
       RTB_ACCEL_REGULAR_GRID = 1, /* Tunnel.cpp:346-465 (uniform cell = maxExtent/399), 819-970 */
       RTB_ACCEL_FLAT_GRID = 2,    /* 400^3 anisotropic cells                                  */
       RTB_ACCEL_KD_MEDIAN = 3,    /* Tunnel.cpp:546-669, 1163-1297                            */
       RTB_ACCEL_KD_SAH = 4,       /* Tunnel.cpp:671-784                                       */
       RTB_ACCEL_CONVEX = 5,        /* PerformanceTest/ConvexAcc.cpp (Tunnel.cpp:972-1161): polygon-to-polygon walk,  */
       RTB_ACCEL_CONVEX_SIMPLE = 6 }; /* first accepted triangle of the wall segment, table-ordered / list-ordered     */

/* 8-byte k-d node, nodes stored in pre-order (left child = index + 1).
 *   inner: a = float bits of the split position, b = (right_child_index << 2) | axis (0,1,2)
 *   leaf : a = first index into kd_leaf_tris,    b = (count << 2) | 3                          */
typedef struct rtb_kdnode { uint32_t a, b; } rtb_kdnode;

/* Sparse grid cell directory: one word pair per 32 consecutive linear cell indices
 * ((x*ny + y)*nz + z, reference Tunnel.h:63-66): `bits` marks non-empty cells, `rank` is the
 * number of non-empty cells before this word.  Non-empty cell r owns
 * grid_cell_tris[grid_cell_start[r] .. grid_cell_start[r+1]).                                   */
typedef struct rtb_cellword { uint32_t bits, rank; } rtb_cellword;

typedef struct rtb_flat_scene {
    int32_t n_prims;      const rtb_prim *prims;
    int32_t n_materials;  const rtb_material *materials;
    int32_t n_top;        /* number of top-level geometries; tunnel triangle k has hit id n_top + k */
    int32_t n_loose;      const float *loose_tri;  /* [n_loose][12]: a, b, c, normal (Triangle.h:10-11) */
    int32_t n_tris;       const float *tri;        /* [n_tris][12] tunnel triangles in surface[seg][j] order */
                          const int32_t *tri_material; /* [n_tris] */
    int32_t accel;        /* RTB_ACCEL_* used by the TUNNEL prim */
    /* grid (RTB_ACCEL_REGULAR_GRID / FLAT_GRID): reference Tunnel.h:51-67 */
    float grid_origin[3], grid_cell[3];
    int32_t grid_dims[3];
    int32_t grid_build_resolution; /* > 1 with grid_words == NULL: the library builds the grid ON THE DEVICE from `tri`
                                      with the reference's rules (Tunnel.cpp:346-465; 400 in the reference): REGULAR
                                      cuts the longest extent into resolution - 1 cubic cells, FLAT every extent;
                                      grid_origin / grid_cell / grid_dims and the three arrays below are ignored        */
    int64_t n_cellwords;  const rtb_cellword *grid_words;      /* ceil(nx*ny*nz / 32)        */
    int64_t n_cells_used; const uint32_t *grid_cell_start;     /* [n_cells_used + 1]         */
    int64_t n_cell_refs;  const uint32_t *grid_cell_tris;      /* [n_cell_refs]              */
    /* k-d tree (RTB_ACCEL_KD_*): reference Tunnel.h:75-93 */
    float kd_min[3], kd_max[3];                                 /* root box                   */
    int32_t n_kd_nodes;   const rtb_kdnode *kd_nodes;
    int64_t n_kd_refs;    const uint32_t *kd_leaf_tris;
    /* convex accelerator (RTB_ACCEL_CONVEX*): reference PerformanceTest/ConvexAcc.h:8-28.  The tunnel is n_cx_path - 1
     * segments of 2 * n_cx_edges triangles each (tri order = surface[seg][j]).                                        */
    int32_t n_cx_path;    const float *cx_frames;  /* [n_cx_path][8]: path vertex xyz, ring normal xyz, cos / sin of the
                                                       rotation that maps the ring's plane to z = 0 (ConvexAcc.cpp:12-18;
                                                       host cosf / sinf / atan2f, as the reference evaluates them)        */
    int32_t n_cx_edges;   const float *cx_edges;   /* [n_cx_edges][3]: A, B, C of A*x + B*y + C > 0 (ConvexAcc.cpp:183-214) */
    float cx_width, cx_height;                      /* bounding rectangle of the cross section (Tunnel.h:19-20)              */
    int32_t cx_table_size;                          /* T: cells per side of the lookup over the cross section's bounding
                                                       rectangle -- 100 in PerformanceTest (ConvexAcc.h:12), 400 in
                                                       RayTracingOpt (Tunnel.cpp:255-284)                                     */
    int32_t cx_round_bins;                          /* direction bin of the order table: 1 = (int)(deg + 0.5) % 360
                                                       (ConvexAcc.cpp:372), 0 = (int)deg (Tunnel.cpp:1042)                    */
    const uint8_t *cx_cell_status;                  /* [T*T] 0 Hit, 1 Partial, 2 Miss (ConvexAcc.cpp:216-247)                */
    const int16_t *cx_cell_range;                   /* [T*T][2] first / last edge to test in a Partial cell (RayTracingOpt
                                                       tests them all: 0 .. n_cx_edges - 1)                                   */
    const uint16_t *cx_order;                       /* RTB_ACCEL_CONVEX: [100][360][2*n_cx_edges] triangle order per
                                                       (height, angle) bin (ConvexAcc.cpp:249-270)                           */
    int32_t grid_build_exact;                       /* device grid build (grid_build_resolution): 1 = a triangle enters a cell only
                                                       if it passes the reference's exact overlap test Triangle::intersectWithGrid
                                                       (Triangle.cpp:152-199), the alternative the reference compiles out at
                                                       Tunnel.cpp:435-445 ("8 times faster" to build without, "20% slower" to
                                                       traverse); 0 = bounding-box binning as the reference ships               */
    /* RTB_ACCEL_KD_SAH with kd_nodes == NULL and kd_build_max_depth > 0: the library builds the tree ON THE DEVICE from `tri`
     * with the reference's builder (Tunnel.cpp:546-638, 671-784): leaf when the list holds <= kd_build_leaf_size triangles or
     * depth > kd_build_max_depth (reference: 8 and 18), kd_build_candidates - 1 uniform planes per axis (reference: 100 - 1).
     * kd_min / kd_max / n_kd_* and the two arrays are ignored.                                                                */
    int32_t kd_build_leaf_size, kd_build_max_depth, kd_build_candidates;
    /* 1 = the arrays above are page-locked host memory (rtb_host_alloc / rtb_host_register) AND stay unchanged until a render
     * of the uploaded scene has returned or the scene has been freed: the upload then copies host -> device straight out of
     * them (truly asynchronous copies, no staging pass over the 4.5 MB of a 45,900-triangle scene, 0.6 -> 0.3 ms per upload).
     * 0 = the arrays may be pageable and may be reused as soon as the upload call returns (they are staged).  An array that
     * is not page-locked is staged whatever the flag says.                                                                  */
    int32_t arrays_page_locked;
} rtb_flat_scene;

/* ---- camera: reference Camera.h:7-23; the derived fields are computed on the host exactly as
 * Camera.cpp:4-18 does (fovScale needs the host tanf)                                        */
typedef struct rtb_camera {
    float eye[3], front[3], up[3], right[3];
    float xcenter, fov_scale, forward;
} rtb_camera;

/* ---- render policy: reference RenderSetting.h:6-79 ---------------------------------------- */
typedef struct rtb_render_setting {
    int32_t enable_monte_carlo;
    int32_t max_depth, termination_depth, single_tracing_depth;
} rtb_render_setting;

/* ---- frame description: the file-statics width/height/samples of reference
 * MainWindow.cpp:33-36 plus the tile-row shard this device renders.
 * Rows are dealt to ranks in blocks of `row_block` rows, block b going to rank b % world
 * (the reference's `omp parallel for schedule(dynamic,1)` over y, MainWindow.cpp:267-269, made
 * static across devices).  The output holds this rank's rows only, in increasing y, row-major
 * [local_row][x][3] float RGB -- unless RTB_LAYOUT_REFERENCE is set (world must be 1), which
 * gives the reference framebuffer order index = x*height + y (MainWindow.cpp:276).          */
enum { RTB_LAYOUT_ROWMAJOR = 0, RTB_LAYOUT_REFERENCE = 1,
       /* OR-able: the output buffer is the WHOLE frame, row-major [height][width][3], and this rank stores only the
        * pixels of its shard into it, at their place in the frame (slot = y * width + x).  Every rank of a frame is
        * given the same buffer -- rank 0's device frame opened on the peers through CUDA IPC (rtb_ipc_*: the stores
        * cross NVLink while the shard renders; no gather, no unshard pass), or one page-locked host frame that all
        * devices of a process store into (rtb_multi_render).  The reference has exactly one framebuffer
        * (MainWindow.cpp:257); this is that buffer, filled by several devices.                                     */
       RTB_LAYOUT_GLOBAL = 2,
       /* OR-able: the output buffer holds 3 BYTES per pixel (R, G, B) produced by the reference's output
        * stage -- saturate (upper clamp only) then (int)(c * 255), MainWindow.cpp:305-311 -- instead of 3
        * floats.  A quarter of the bytes to read back; the float framebuffer is what parity is judged on. */
       RTB_OUTPUT_RGB8 = 4,
       /* OR-able, Monte Carlo only: the output buffer holds SIX floats per pixel -- the sum over this call's samples of
        * the per-sample radiance (R, G, B; the reference accumulates radiance * (1 / samples), MainWindow.cpp:288: here
        * the plain sum) and the sum of its squares -- the accumulation buffer (sum, sum of squares, spp) of a progressive
        * or sample-sharded render: buffers of disjoint sample ranges add up, mean = sum / spp,
        * variance = (sumsq - sum^2 / spp) / (spp - 1).  Not with RTB_OUTPUT_RGB8 / RTB_LAYOUT_REFERENCE.            */
       RTB_OUTPUT_MOMENTS = 8 };
typedef struct rtb_frame {
    int32_t width, height;
    int32_t samples;      /* spp when enable_monte_carlo                                      */
    uint64_t seed;        /* counter-based RNG frame seed (key = pixel, sample)               */
    int32_t rank, world;  /* shard selector; 0,1 = whole frame                                */
    int32_t row_block;    /* rows per dealt block (multiple of 8; 0 = default 8)              */
    int32_t layout;       /* RTB_LAYOUT_*                                                     */
    int32_t counters;     /* 1: also count triangle tests / traversal steps (slower); 2: as 1 and write a
                             per-pixel cost map (thread cycles, rays, steps + tests) instead of the colour
                             (profiling aid, Whitted chain kernel only)                          */
    int32_t col_block;    /* 0: the shard is whole rows (blocks of row_block rows dealt round-robin).  > 0 (with world
                             > 1): COLUMN-BLOCK shard -- every rank renders every row and, of block row
                             by = y / row_block, the column blocks bx = x / col_block with (bx + by) % world == rank;
                             its output is a local image [height][width / world] in which local column block c holds
                             global block c * world + (rank - by) mod world.  Multiple of 8, width a multiple of
                             world * col_block, row-major layout.  The tunnel frames concentrate their cost around
                             the vanishing point: narrow column blocks give every rank the same mix of tiles.
                             (Occupies what was tail padding of this struct: zero-initialised callers get rows.)  */
    int32_t sample_first; /* Monte Carlo SAMPLE shard: this call renders samples [sample_first, sample_first +   */
    int32_t sample_count; /* sample_count) of the frame's `samples` (0 = all of them).  The RNG is keyed by (pixel,
                             sample index) and every sample is weighted 1 / samples, so the images of disjoint ranges
                             ADD UP to the full frame (float rounding of the per-pixel sum aside: the order of the
                             additions differs from the single pass): low-resolution / high-spp frames shard over
                             samples instead of rows, one NCCL reduce (sum) assembles them (SURVEY 8e).              */
} rtb_frame;

typedef struct rtb_stats {
    int64_t n_rays;        /* scene intersections issued (primary + secondary)                */
    int64_t n_tri_tests;   /* frame.counters only                                             */
    int64_t n_steps;       /* cells / k-d nodes visited; frame.counters only                  */
    int64_t n_local_rows;  /* rows rendered by this rank                                      */
    float kernel_ms;       /* CUDA-event time of the render kernel(s) on the context stream   */
    float total_ms;        /* CUDA-event time of the whole call incl. copies                  */
    int32_t n_launches;    /* kernels launched by the call                                    */
    int32_t pad_;
} rtb_stats;

typedef struct rtb_ctx rtb_ctx;
typedef struct rtb_scene rtb_scene;

/* Context = one CUDA device.  `stream` may be 0 (library-owned stream) or a caller's
 * cudaStream_t cast to void* (e.g. torch's current stream) for rtb_render_device.            */
int rtb_init(int device, rtb_ctx **ctx);
int rtb_shutdown(rtb_ctx *ctx);
const char *rtb_last_error(const rtb_ctx *ctx); /* ctx may be NULL: last global error       */
int rtb_abi_version(void);

/* Page-locked host memory for the host-buffer calls (optional: any host pointer is accepted, but
 * device->host copies into pageable memory are staged by the driver and several times slower).   */
int rtb_host_alloc(size_t bytes, void **out);
int rtb_host_free(void *p);
/* Page-lock memory the caller already owns (the arrays of a flat scene, see rtb_flat_scene.arrays_page_locked; a frame
 * buffer): every device of the process may copy from / store into it.  Unregister before the memory is freed.          */
int rtb_host_register(void *p, size_t bytes);
int rtb_host_unregister(void *p);

/* Number of rows / first-row list of a shard (pure host arithmetic; no device needed).       */
int64_t rtb_shard_rows(const rtb_frame *frame);
/* width of the shard's local image: frame->width, or frame->width / world for a column-block shard */
int64_t rtb_shard_width(const rtb_frame *frame);

/* Host-only check (no device needed) that nodes[0 .. n) is a well-formed pre-order k-d array as rtb_scene_upload
 * requires it: every inner node's right child lies behind its left subtree and before the end of the enclosing
 * subtree, every node belongs to exactly one subtree, no node is deeper than 64.  RTB_OK and *max_depth (root = 0)
 * or RTB_ERR_INVALID.  rtb_scene_upload runs the same check (and refuses trees whose traversal stack,
 * 2 * max_depth + 2 entries, would exceed the reference's 50, Tunnel.cpp:1176).                                   */
int rtb_kd_validate(const rtb_kdnode *nodes, int32_t n, int32_t *max_depth);

/* Upload a flattened scene.  Replaces nothing in the reference (it has no device); it is the
 * device-side image of GeometrySet + Tunnel::grid / Tunnel::root.                           */
int rtb_scene_upload(rtb_ctx *ctx, const rtb_flat_scene *flat, rtb_scene **scene);
int rtb_scene_free(rtb_ctx *ctx, rtb_scene *scene);
int64_t rtb_scene_device_bytes(const rtb_scene *scene);
/* bytes rtb_scene_upload copied from host memory for this scene (raw triangle records, materials, accelerator arrays);
 * the packed triangle streams and the pair stream of the list scans are produced on the device                      */
int64_t rtb_scene_upload_bytes(const rtb_scene *scene);
/* Inspection: canonical structure hash of the grid resident on the device (the arrays are read back), the hash
 * tests/golden and the host API use for grids; stats = {dims x, y, z, occupied cells, triangle references, longest
 * cell list}.  RTB_ERR_UNSUPPORTED for other accelerators.                                                          */
int rtb_scene_grid_hash(rtb_ctx *ctx, const rtb_scene *scene, uint64_t *hash, int64_t stats[6]);
/* Inspection: the k-d tree resident on the device (uploaded, or built there) read back in the layout of rtb_flat_scene:
 * nodes[counts[0]] in pre-order, leaf_tris[counts[1]]; counts[2] = levels of a device build (0 otherwise); box = root box
 * (min xyz, size xyz).  Either array may be NULL to query the counts first.                                            */
int rtb_scene_kd_download(rtb_ctx *ctx, const rtb_scene *scene, rtb_kdnode *nodes, int64_t node_cap, uint32_t *leaf_tris,
                          int64_t ref_cap, int64_t counts[3], float box[6]);

/* Bounding-volume hierarchy of an RTB_PRIM_MESH record (built on the device by rtb_scene_upload, csrc/rtb_build_bvh.cuh).
 * A mesh of n triangles has max(n - 1, 1) inner nodes, node 0 is the root.  Each node holds the boxes of its two children
 * (a child's box is the union of the boxes below it; a leaf's box is its triangle's box widened by the barycentric slack,
 * csrc/rtb_bvh.h) and the two child links: c >= 0 is inner node c, c < 0 is the leaf at position ~c of the mesh's leaf
 * order (one triangle per leaf; a one-triangle mesh has both links -1).  tri_order[p] = local index k (0 .. n - 1) of the
 * triangle at leaf position p.                                                                                          */
typedef struct rtb_bvhnode {
    float lo[2][3], hi[2][3]; /* [child][axis] */
    int32_t child[2];
    int32_t pad_[2];
} rtb_bvhnode;              /* 64 bytes */
/* Inspection: the tree of the mesh record `mesh_index` (0 = the first MESH record in prims order).  counts = {inner nodes,
 * triangles, depth (the root's children are at depth 1; leaves count)}.  nodes / tri_order may be NULL to query the counts. */
int rtb_scene_mesh_download(rtb_ctx *ctx, const rtb_scene *scene, int32_t mesh_index, rtb_bvhnode *nodes, int64_t node_cap,
                            uint32_t *tri_order, int64_t tri_cap, int64_t counts[3]);

/* Replace the triangles of the MESH record `mesh_index` (0 = first MESH record in prims order): `tri` = [n][12] records in
 * the loose_tri format (a, b, c, normal), n == the record's count.  `tri` is host memory (pageable or page-locked; staged,
 * reusable when the call returns) or device memory of the context's device (16-byte aligned; read in place, no PCIe);
 * managed memory is read in place on the device like device memory.
 * Enqueued behind the work already on `stream` (0 = the context's stream, which is not ordered with the legacy default
 * stream: pass cudaStreamLegacy for that) and behind every launch that reads the scene;
 * later work on `stream` and later renders on any stream see the new triangles.  No host synchronisation for a device source.
 * The scene becomes the one rtb_scene_upload gives for the same flat scene with loose_tri[first, first + count) replaced:
 * TRIANGLES runs over that range see the new records, and every other MESH record that intersects the range must lie inside
 * it (its records are a slice of `tri`; it gets the same operation) -- one that overlaps it only in part is
 * RTB_ERR_UNSUPPORTED.  Every rejection leaves the scene unchanged: n != count and device memory of another device or
 * misaligned are RTB_ERR_INVALID, no such mesh is RTB_ERR_UNSUPPORTED.
 *   RTB_MESH_REBUILD: the hierarchy is built again as rtb_scene_upload builds it (byte-identical tree, identical results).
 *   RTB_MESH_REFIT:   child links and leaf order are kept, every box is recomputed from the new records (the bound of the
 *                     node test holds for any tree shape: the mesh contract holds; the tree's quality decays with large motion). */
enum { RTB_MESH_REBUILD = 0, RTB_MESH_REFIT = 1 };
int rtb_scene_mesh_update(rtb_ctx *ctx, rtb_scene *scene, int32_t mesh_index, const float *tri, int64_t n,
                          int32_t flags, void *stream);

/* Replaces `int Render(GeometrySet&, PerspectiveCamera&, RenderSetting&, ProgressCallback)`
 * (reference MainWindow.cpp:251-303, the RenderProc of Scripts.h:11-12): ray generation,
 * trace()/radiance() and the framebuffer store for this rank's rows.  `rgb_out` is a HOST
 * buffer of rtb_shard_rows(frame)*width*3 floats (bytes with RTB_OUTPUT_RGB8, which also runs the
 * output stage of MainWindow.cpp:305-311); the device->host copy is part of the call.         */
int rtb_render(rtb_ctx *ctx, const rtb_scene *scene, const rtb_camera *camera,
               const rtb_render_setting *setting, const rtb_frame *frame, void *rgb_out,
               rtb_stats *stats);

/* Same, writing to a DEVICE buffer on `stream` without synchronising (stats are filled only if
 * non-NULL, which forces a sync).  Used to keep the framebuffer resident for the NCCL gather.   */
int rtb_render_device(rtb_ctx *ctx, const rtb_scene *scene, const rtb_camera *camera,
                      const rtb_render_setting *setting, const rtb_frame *frame,
                      void *rgb_device, void *stream, rtb_stats *stats);

/* Multi-GPU assembly: `gathered` is the NCCL all-gather of every rank's rtb_render_device output,
 * [world][rows_per_rank][width][3] floats (each rank's rows padded to rows_per_rank); writes the
 * frame in image row order [height][width][3] to `image`.  Both are DEVICE buffers; asynchronous
 * on `stream`.  (The reference has a single framebuffer, MainWindow.cpp:257; this is its
 * reassembly after tile-row sharding.)                                                        */
int rtb_unshard_device(rtb_ctx *ctx, const void *gathered, void *image, int32_t width, int32_t height,
                       int32_t world, int32_t row_block, int64_t rows_per_rank, void *stream);

/* Parity hook: primary rays only (pixel centres, MainWindow.cpp:294-297) through
 * GeometrySet::intersect.  Arrays are row-major [y*width + x] HOST buffers, any may be NULL.
 * seq_* record the accelerator steps of the TUNNEL prim (cell indices / pre-order node ids):
 * seq_hash folds h = (h ^ id) * 0x100000001b3 from 0xcbf29ce484222325; seq_buf keeps the first
 * seq_cap ids per ray (-1 padded).                                                            */
int rtb_trace_primary(rtb_ctx *ctx, const rtb_scene *scene, const rtb_camera *camera,
                      int32_t width, int32_t height, int32_t *hit_id, float *hit_t,
                      int32_t *seq_len, uint64_t *seq_hash, int32_t *seq_buf, int32_t seq_cap);

/* Replaces `IntersectResult Geometry::intersect(Ray&)` (reference Geometry.h:17) and PT's
 * `Accelerator::intersect` (PerformanceTest/Accelerator.h:6-15) for a BATCH of rays:
 * rays = [n][6] origin, direction (HOST); outputs (HOST, any may be NULL): hit id (-1 miss),
 * distance, position xyz, normal xyz (the stored, unflipped normal).                         */
int rtb_intersect_rays(rtb_ctx *ctx, const rtb_scene *scene, int64_t n, const float *rays,
                       int32_t *hit_id, float *hit_t, float *position, float *normal);

/* Ray queries on DEVICE buffers, stream-ordered (no host synchronisation, no allocation): for a physics or robotics step,
 * a sensor model or a renderer outside this library that keep their rays on the device.
 * rays = [n][6] origin, direction: memory of the context's device or managed memory, 8-byte aligned.  tmax = [n] per-ray
 * bounds in the same kind of memory, or NULL: tmax_all for every ray.  Every other buffer is such memory too.
 *   RTB_QUERY_CLOSEST: hit_id, hit_t, position, normal (any may be NULL; occluded must be NULL) as rtb_intersect_rays
 *     writes them.  The bound is STRICT: a ray's result is rtb_intersect_rays's result for it when that hit has t < tmax,
 *     otherwise a miss (id -1, t -1, zeros).  A bound at or above FLT_MAX (+inf included) is no bound: NULL with tmax_all =
 *     INFINITY is rtb_intersect_rays bit for bit.  A NaN bound, or one <= 0.0005 (the reference's least distance), is a miss.
 *     The search starts at the bound, so the records' own strict `<` apply it: exact for PLANE, SPHERE, TRIANGLES and the
 *     TUNNEL under every accelerator; a MESH record's hierarchy prunes against it, and its result is the masked unbounded one
 *     except for rays whose winning pair lies in the grazing band (the mesh's contract, RTB_PRIM_MESH above).
 *   RTB_QUERY_ANY: occluded[n] (required; the other outputs must be NULL) = 1 exactly when RTB_QUERY_CLOSEST with the same
 *     bound would hit, else 0 (the grazing-band exception applies to meshes).  The walk stops at the first hit under the bound.
 * Enqueued on `stream` (0 = the context's stream, not ordered with the legacy default stream: pass cudaStreamLegacy for that)
 * behind the scene's upload and mesh updates; queries on different streams are ordered among themselves, and later mesh
 * updates and rtb_scene_free wait for them.  Renders are not ordered against queries (both only read the scene).
 * Checks come before anything is enqueued, and a refused call writes nothing: host memory, memory of another device, a
 * misaligned buffer, n < 0, unknown flags or outputs that do not match them are RTB_ERR_INVALID.  n == 0 does nothing.   */
enum { RTB_QUERY_CLOSEST = 0, RTB_QUERY_ANY = 1 };
int rtb_query_rays(rtb_ctx *ctx, const rtb_scene *scene, int64_t n, const float *rays, const float *tmax, float tmax_all,
                   int32_t flags, int32_t *hit_id, float *hit_t, float *position, float *normal, uint8_t *occluded,
                   void *stream);

/* Closest-point queries on DEVICE buffers, stream-ordered like rtb_query_rays (no host synchronisation, no allocation): the
 * nearest point on the scene's triangles within a per-point radius, for contact generation, clearance checks or distance
 * sampling in a physics or robotics step.  points = [n][3], rmax = [n] per-point radii or NULL: rmax_all for every point;
 * every buffer is memory of the context's device or managed memory, 4-byte aligned (near: 1-byte).
 * Records considered: TRIANGLES and MESH records only, in prims order (a MESH record is walked through its hierarchy and
 * returns what the run of the same triangles returns, bit for bit, with no exception).  PLANE, SPHERE and TUNNEL records are
 * ignored (upload the tunnel's triangles as a mesh to include them); a scene without triangle records returns misses.
 * Distance: csrc/rtb_closest.h, one function compiled identically for host and device; d2 = the squared distance from the
 * point to its closest point q on the triangle.  The winner is the smallest d2: ties within a record go to the lowest k, across
 * records to the earlier record.  The bound is STRICT and squared: a pair counts when d2 < fl(r * r); r = +inf is no bound,
 * r <= 0 or NaN is a miss, and so is a NaN point.
 *   RTB_QUERY_CLOSEST: hit_id (base_id + k), distance = sqrtf(d2), position = q, normal = the stored, unflipped normal (any
 *     may be NULL; near must be NULL).  A miss writes -1, -1, zeros, zeros.
 *   RTB_QUERY_ANY: near[n] (required; the other outputs must be NULL) = 1 exactly when RTB_QUERY_CLOSEST with the same radius
 *     hits, else 0.  The search stops at the first triangle within the radius.
 * Ordering and refusals as rtb_query_rays: enqueued on `stream` (0 = the context's stream) behind the scene's upload and mesh
 * updates, ordered with the other queries, awaited by later mesh updates and rtb_scene_free; host memory, memory of another
 * device, a misaligned buffer, n < 0, unknown flags or outputs that do not match them are RTB_ERR_INVALID, and a refused call
 * writes nothing.  n == 0 does nothing.                                                                                    */
int rtb_query_points(rtb_ctx *ctx, const rtb_scene *scene, int64_t n, const float *points, const float *rmax, float rmax_all,
                     int32_t flags, int32_t *hit_id, float *distance, float *position, float *normal, uint8_t *near,
                     void *stream);

/* First-order moments of every MESH record's hierarchy, for rtb_query_winding: per node and child the area vector, the
 * area-weighted centre and a radius about it (64 bytes per node slot; rtb_scene_device_bytes grows by 64 x the scene's mesh
 * triangles).  Opt-in: rtb_scene_upload does not build them.  Once built, rtb_scene_mesh_update (rebuild and refit) keeps
 * them current with no new allocation.  Ordered like rtb_scene_mesh_update: enqueued on the context's stream behind `stream`
 * (0 = the context's stream) and every launch that has read the scene, and `stream` waits for it.  A second call, and a call
 * on a scene without MESH records, does nothing.                                                                          */
int rtb_scene_mesh_moments(rtb_ctx *ctx, rtb_scene *scene, void *stream);

/* Winding-number queries on DEVICE buffers, stream-ordered like rtb_query_points: inside / outside tests for occupancy,
 * penetration depth or SDF sampling.  points = [n][3]; winding = [n] float, inside = [n] uint8, either may be NULL but not
 * both; every buffer is memory of the context's device or managed memory, 4-byte aligned (inside: 1-byte).
 * winding[i] = the generalised winding number sum_t Omega_t(p) / 4 pi over the TRIANGLES and MESH records, in prims order
 * (overlapping records count once each; PLANE, SPHERE and TUNNEL records are ignored): 1 inside and 0 outside a closed
 * surface whose facets follow the right-hand rule outwards (the vertex order decides, never the stored normal), fractional
 * for open soups.  inside[i] = winding[i] > 0.5.  Solid angles: csrc/rtb_winding.h, one function compiled identically for
 * host and device.  A TRIANGLES run sums every triangle exactly, in k order.  A MESH record walks its hierarchy: a leaf adds
 * its exact solid angle, an inner child whose centre lies farther than beta x its radius adds its dipole (Barill et al.
 * 2018), any other child is descended into.  beta = +inf sums every triangle exactly; beta must be >= 1 (2 is the usual
 * choice).  A NaN point gives NaN / 0.
 * Refused with RTB_ERR_INVALID, writing nothing: n < 0, beta NaN or below 1, no output, a scene with MESH records but no
 * moments (rtb_scene_mesh_moments), and the buffer refusals of rtb_query_points.  n == 0 does nothing.                     */
int rtb_query_winding(rtb_ctx *ctx, const rtb_scene *scene, int64_t n, const float *points, float beta, float *winding,
                      uint8_t *inside, void *stream);

/* Triangle intersection queries on DEVICE buffers, stream-ordered like rtb_query_points: which of the scene's triangles a
 * batch of triangles touches, for contact between a deforming body and a scene, cloth against a body, or checking that an
 * edit or an optimisation step does not make two parts interpenetrate.  tris = [n][12] in the loose_tri format (a, b, c,
 * normal; the normal is ignored), 16-byte aligned; n <= INT32_MAX.  Records considered: TRIANGLES and MESH records, in prims
 * order (PLANE, SPHERE and TUNNEL records are ignored); a scene triangle k is (a, fl(a - e1), fl(a - e2)) of its packed record,
 * with hit id base_id + k, so a triangle inside two overlapping records is reported once per record.
 * A pair is reported EXACTLY when the two closed triangles share at least one point in exact real arithmetic: touching counts
 * (a shared vertex, a vertex on the other's face, coplanar triangles that overlap or touch); there is no tolerance.  The one
 * exception: DEGENERATE triangles, on either side -- three exactly collinear vertices (repeated vertices included) or a
 * non-finite coordinate -- are never reported.  The decision is csrc/rtb_tritri.h, exact orientation predicates compiled for
 * host and device; a MESH record prunes its hierarchy by closed boxes and gives what a loop over its triangles gives.
 *   RTB_QUERY_ANY: hit[n] (uint8, 1-byte aligned, required) = 1 exactly when RTB_QUERY_PAIRS reports a pair for triangle i,
 *     else 0; pairs and count must be NULL and capacity 0.  A triangle's search stops at its first pair.
 *   RTB_QUERY_PAIRS: *count (int64, 8-byte aligned, required) is zeroed on the stream, then holds the number of pairs, even
 *     when it exceeds capacity.  pairs = [capacity][2] int32 (i, hit_id), 8-byte aligned: slots 0 .. min(count, capacity) - 1
 *     are written and nothing beyond them.  The order is unspecified; the set is deterministic.  capacity = 0 with pairs NULL
 *     counts only; size the buffer from *count and call again.  hit must be NULL.
 * Ordering as rtb_query_points; no host synchronisation, no allocation.  Refused with RTB_ERR_INVALID, writing nothing: n < 0 or
 * above INT32_MAX, capacity < 0, capacity > 0 with pairs NULL, unknown flags, outputs that do not match them, host memory,
 * memory of another device, a misaligned buffer.  n == 0 launches nothing (PAIRS still zeroes *count).                   */
enum { RTB_QUERY_PAIRS = 2 };
int rtb_query_triangles(rtb_ctx *ctx, const rtb_scene *scene, int64_t n, const float *tris, int32_t flags, uint8_t *hit,
                        int32_t *pairs, int64_t capacity, int64_t *count, void *stream);

/* Replaces the ray loop of the reference's PerformanceTest console benchmark
 * (src/PerformanceTest/main.cpp:29-59 `trace`, 151-162): every ray of the batch [n][6] (HOST) is
 * mirror-reflected off whatever it hits until it reaches a PLANE geometry (the plane closing the tunnel
 * exit), misses, or has been traced max_depth times (reference: 200).  Outputs (HOST, any may be NULL):
 * reached (1 = stopped on a plane), depth (hits counted), hit id and position of the last hit,
 * the total number of rays traced and the kernel's CUDA-event time.                                   */
int rtb_bounce_rays(rtb_ctx *ctx, const rtb_scene *scene, int64_t n, const float *rays, int32_t max_depth,
                    int32_t *reached, int32_t *depth, int32_t *last_id, float *last_pos, int64_t *total_rays,
                    float *kernel_ms);

/* As rtb_unshard_device for column-block shards (rtb_frame.col_block): `gathered` = [world][height][width / world][3]. */
int rtb_unshard_cols_device(rtb_ctx *ctx, const void *gathered, void *image, int32_t width, int32_t height,
                            int32_t world, int32_t row_block, int32_t col_block, void *stream);

/* Self-test of the list scans' rejection test (csrc/rtb_pretest.h): n random (ray, triangle) pairs -- triangles of
 * widely varying size, slivers, rays aimed at the triangle's boundary -- are decided by the scalar function (the one
 * tests/ checks against the oracle on the CPU) and by the packed-FP32 two-triangle variant the kernels run;
 * *mismatches = pairs on which the two disagree (must be 0), *rejected = pairs the test rejects (so a caller can see
 * that both outcomes occur).  No reference counterpart: diagnostic entry point.                                     */
int rtb_selftest_pretest(rtb_ctx *ctx, int64_t n, uint64_t seed, int64_t *mismatches, int64_t *rejected);

/* Progress reporting -- replaces `progress(y + 1, height)` of the reference's row loop (MainWindow.cpp:271; the
 * ProgressCallback of Scripts.h:9).  While rtb_render / rtb_multi_render wait for the frame they poll the number of
 * finished tiles (a device counter, read over a side stream; the kernels are not interrupted) and call `fn` from the
 * calling host thread, every ~0.25 ms and once more when the frame is complete (done == total).  NULL turns it off.  */
typedef void (*rtb_progress_fn)(int64_t tiles_done, int64_t tiles_total, void *user);
int rtb_set_progress(rtb_ctx *ctx, rtb_progress_fn fn, void *user);

/* Forget the tile schedule the context has learnt (heaviest-first order and latency tiers of the last view): the next
 * frame runs like the first frame of a new view -- raster order, one throughput kernel, every tile measured.  The
 * reference renderer keeps no state between frames (MainWindow.cpp:251-303); this makes that case measurable.       */
int rtb_forget_schedule(rtb_ctx *ctx);

/* ---- one frame buffer, several devices (RTB_LAYOUT_GLOBAL) -------------------------------------------------------
 * Replaces the single framebuffer `colors` every OpenMP thread of the reference's Render writes its rows into
 * (MainWindow.cpp:257, 267-276).
 *
 * A: one process per device (torch.distributed / MPI plumbing).  The owner rank allocates the frame with
 *    rtb_device_alloc (plain cudaMalloc memory: exportable), exports it with rtb_ipc_export, sends the 64 handle bytes
 *    to its peers by any means, each peer maps it with rtb_ipc_open (peer access over NVLink is enabled as needed) and
 *    passes the mapped pointer to rtb_render_device with RTB_LAYOUT_GLOBAL.  A barrier of the caller closes the step. */
#define RTB_IPC_HANDLE_BYTES 64
int rtb_device_alloc(rtb_ctx *ctx, size_t bytes, void **out);
int rtb_device_free(rtb_ctx *ctx, void *p);
int rtb_device_download(rtb_ctx *ctx, const void *device_ptr, void *host, size_t bytes); /* synchronous read-back of such a frame */
int rtb_ipc_export(rtb_ctx *ctx, void *device_ptr, unsigned char handle[RTB_IPC_HANDLE_BYTES]);
int rtb_ipc_open(rtb_ctx *ctx, const unsigned char handle[RTB_IPC_HANDLE_BYTES], void **mapped);
int rtb_ipc_close(rtb_ctx *ctx, void *mapped);
/* Alternative to rendering straight into the mapped frame: render the shard into a LOCAL device buffer (row-major layout of
 * rtb_render_device), then move it to its place in the whole frame with one streaming pass of 128-bit copies on `stream`
 * (the frame may be peer-mapped: one bulk NVLink transfer instead of tile-sized stores issued while the kernels render).
 * `frame` describes the shard (rank / world / row_block / col_block); float frames only.                              */
int rtb_scatter_shard_device(rtb_ctx *ctx, const void *local, void *frame_buffer, const rtb_frame *frame, void *stream);

/* B: ONE host thread drives n devices (SURVEY 8b threading row; the drop-in behind Scripts.h:11-12 RenderProc).
 *    rtb_multi_render shards the frame over the devices (tile rows up to 4 devices, column blocks above), every device
 *    stores its tiles straight into `rgb_out` -- ONE assembled host frame, row-major [height][width][3] floats (bytes
 *    with RTB_OUTPUT_RGB8), or the reference order with RTB_LAYOUT_REFERENCE -- and the call returns when all devices
 *    are done.  `rgb_out` from rtb_host_alloc is written directly over PCIe by all devices at once; any other host
 *    buffer goes through a page-locked frame owned by the library and one host copy.  frame->rank / world are ignored.
 *    stats: counts are summed over the devices, kernel_ms / total_ms are the maximum.                                */
typedef struct rtb_multi rtb_multi;
typedef struct rtb_multi_scene rtb_multi_scene;
int rtb_multi_init(int n_devices, const int *devices /* NULL: 0 .. n_devices - 1 */, rtb_multi **out);
int rtb_multi_shutdown(rtb_multi *m);
int rtb_multi_count(const rtb_multi *m);
rtb_ctx *rtb_multi_ctx(rtb_multi *m, int i);
const char *rtb_multi_last_error(const rtb_multi *m);
int rtb_multi_set_progress(rtb_multi *m, rtb_progress_fn fn, void *user);
int rtb_multi_scene_upload(rtb_multi *m, const rtb_flat_scene *flat, rtb_multi_scene **scene); /* replicated on every device */
int rtb_multi_scene_free(rtb_multi *m, rtb_multi_scene *scene);
int64_t rtb_multi_scene_upload_bytes(const rtb_multi_scene *scene); /* summed over the devices */
int rtb_multi_render(rtb_multi *m, const rtb_multi_scene *scene, const rtb_camera *camera,
                     const rtb_render_setting *setting, const rtb_frame *frame, void *rgb_out, rtb_stats *stats);
/* rtb_scene_mesh_update on every device of the scene; `tri` is host memory (device and managed memory are RTB_ERR_INVALID). */
int rtb_multi_scene_mesh_update(rtb_multi *m, rtb_multi_scene *scene, int32_t mesh_index, const float *tri, int64_t n,
                                int32_t flags);

#ifdef __cplusplus
}
#endif
#endif /* RTB_H */
