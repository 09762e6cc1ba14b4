/*
 * pcv.h — C ABI of the B200-native octree builder / LOD + frustum point-query engine.
 *
 * This is the drop-in boundary for point_cloud_viewer's hot path: each entry point replaces a Rust
 * function or trait method of crate `point_viewer` (citations = reference file:line).  The reference
 * has no FFI of its own; INTEGRATION.md shows the Rust `extern "C"` block + shim a maintainer adds.
 *
 * Conventions
 *  - plain pointers and sizes only; every function returns 0 (PCV_OK) or a negative pcv_status and
 *    never unwinds across the boundary; pcv_last_error() returns the text for the calling thread.
 *  - "host" entry points take host memory (pinned or pageable) and copy inside the call; "_device"
 *    entry points take device pointers already resident in HBM on the context's GPU.
 *  - positions are f64; element i of a coordinate array is at ptr[i * stride] so both the SoA layout
 *    (stride 1, three arrays) and the crate's AoS `Vec<Point3<f64>>` (stride 3, y = x+1, z = x+2) are
 *    accepted without a host-side transpose.
 *  - matrices are column-major like nalgebra::Matrix4<f64>; isometries are tx,ty,tz,qi,qj,qk,qw.
 *  - NodeId is the crate's u128 (level << 120 | octal path index, src/octree/node.rs:52-111) passed
 *    as (high, low) u64 halves exactly like proto::NodeId (node.rs:101-106).
 *  - there is no CPU fallback: without a CUDA device every compute entry point fails with
 *    PCV_ERR_CUDA.
 */
#ifndef PCV_H
#define PCV_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct pcv_ctx pcv_ctx;       /* one per device; internally stream ordered              */
typedef struct pcv_octree pcv_octree; /* a built / loaded octree, node data resident in HBM     */

typedef enum pcv_status {
    PCV_OK = 0,
    PCV_ERR_INVALID = -1,     /* bad argument                                                    */
    PCV_ERR_CUDA = -2,        /* CUDA runtime error or no device                                 */
    PCV_ERR_IO = -3,          /* file system error (the reference unwrap()s these)               */
    PCV_ERR_NOT_FOUND = -4,   /* ErrorKind::NodeNotFound (src/errors.rs)                         */
    PCV_ERR_CANCELLED = -5,   /* callback returned non-zero == ErrorKind::Channel                */
    PCV_ERR_UNSUPPORTED = -6, /* e.g. more than 2^32-1 points per context, depth > 40            */
    PCV_ERR_SINGULAR = -7     /* get_visible_nodes: "Invalid projection matrix." (mod.rs:230)    */
} pcv_status;

/* PositionEncoding (src/read_write/codec.rs:22-28, proto.proto:78-84) */
enum { PCV_ENC_UINT8 = 1, PCV_ENC_UINT16 = 2, PCV_ENC_FLOAT32 = 3, PCV_ENC_FLOAT64 = 4 };

typedef struct pcv_config {
    uint64_t max_points_per_node; /* MAX_POINTS_PER_NODE, generation.rs:37; 0 -> 100000          */
    uint32_t levels_per_pass;     /* kept for ABI stability: the split phase resolves 2 levels/pass */
    uint32_t reserved;
} pcv_config;

typedef struct pcv_points {
    const double* x; /* element i at x[i*stride]                                                 */
    const double* y;
    const double* z;
    uint64_t stride;        /* 1 = SoA, 3 = AoS xyz                                              */
    const uint8_t* rgb;     /* n * 3, "color" U8Vec3 (mandatory: on_disk.rs:23-33)               */
    const float* intensity; /* n or NULL ("intensity" F32, octree/mod.rs:62-74)                  */
    uint64_t n;
} pcv_points;

typedef struct pcv_node_meta {
    uint64_t id_high, id_low; /* NodeId u128 halves                                              */
    int64_t num_points;       /* may be 0: such nodes stay in meta.pb (generation.rs:241-243)    */
    int32_t position_encoding;
    int32_t level;
    double cube_min[3]; /* NodeId::find_bounding_cube (node.rs:157-172)                          */
    double cube_edge;
    uint64_t point_offset;    /* first point of the node in the node-contiguous arrays           */
    uint64_t xyz_byte_offset; /* first byte of the node's .xyz content                           */
} pcv_node_meta;

/* PointLocation (src/iterator.rs:13-20).  Same field layout as the oracle's orc_location. */
enum { PCV_LOC_ALL = 0, PCV_LOC_AABB = 1, PCV_LOC_FRUSTUM = 2, PCV_LOC_OBB = 3 };
typedef struct pcv_location {
    int32_t kind;
    int32_t pad;
    double aabb_min[3], aabb_max[3];                 /* Aabb{mins,maxs}        aabb.rs:12-16     */
    double clip_from_query[16], query_from_clip[16]; /* Frustum fields         frustum.rs:95-98  */
    double query_from_obb[7], obb_from_query[7];     /* Obb fields             obb.rs:13-17      */
    double half_extent[3];
} pcv_location;

typedef struct pcv_interval { /* ClosedInterval<f64> on "intensity" (math/mod.rs:65-89)          */
    double lo, hi;
} pcv_interval;

/* A PointsBatch (src/lib.rs:102-107) delivered to the consumer: AoS positions + SoA attributes.  */
typedef struct pcv_batch {
    uint64_t n;
    const double* xyz;         /* n * 3                                                          */
    const uint8_t* rgb;        /* n * 3                                                          */
    const float* intensity;    /* n or NULL                                                      */
    const uint64_t* src_index; /* provenance: index of the point in the build input              */
} pcv_batch;
typedef int (*pcv_batch_cb)(void* user, const pcv_batch* batch); /* non-zero return cancels      */

/* ---- context ------------------------------------------------------------------------------- */
int pcv_create(int device, const pcv_config* cfg, pcv_ctx** out);
void pcv_destroy(pcv_ctx* ctx);
const char* pcv_last_error(void);
int pcv_device_count(void);

/* ---- a1: find_bounding_box (generation.rs:256-270, aabb.rs:41-44) -------------------------- */
int pcv_bbox(pcv_ctx* ctx, const pcv_points* host_points, double out_min[3], double out_max[3]);
int pcv_bbox_device(pcv_ctx* ctx, const pcv_points* dev_points, double out_min[3], double out_max[3]);

/* ---- a2-a8: build_octree (generation.rs:289-403) -------------------------------------------- */
int pcv_build_octree(pcv_ctx* ctx, const pcv_points* host_points, double resolution, const double bbox_min[3],
                     const double bbox_max[3], pcv_octree** out);
int pcv_build_octree_device(pcv_ctx* ctx, const pcv_points* dev_points, double resolution, const double bbox_min[3],
                            const double bbox_max[3], pcv_octree** out);
void pcv_octree_free(pcv_octree* o);

/* ---- a8-a10: node table, node bytes, on-disk layout ----------------------------------------- */
int pcv_octree_info(const pcv_octree* o, uint64_t* num_nodes, uint64_t* num_points, uint64_t* xyz_bytes, double* resolution,
                    double bbox_min[3], double bbox_max[3], int* has_intensity);
int pcv_octree_nodes(const pcv_octree* o, pcv_node_meta* out, uint64_t cap); /* sorted by NodeId   */
/* Octree::get_node_data (octree/mod.rs:285-307): raw .xyz / .rgb bytes (+ intensity, provenance). */
int pcv_octree_node_data(const pcv_octree* o, uint64_t id_high, uint64_t id_low, void* xyz_out, uint8_t* rgb_out,
                         float* intensity_out, uint64_t* src_index_out);
/* The web viewer's `/nodes_data` reply (octree_web_viewer/src/backend.rs:66-75, 92-165): for every requested node, in
 * request order: cube min (3 f64 LE), edge (f64), num_points (u32), bytes per coordinate (u8), zero padding to 8 bytes,
 * position bytes, padding, colour bytes, padding.  ids_hi_lo = num_nodes x (high, low).  out == NULL: size query.
 * An unknown id or a node without points is PCV_ERR_NOT_FOUND (get_node_data -> NodeNotFound: no files). */
int pcv_nodes_data_blob(const pcv_octree* o, const uint64_t* ids_hi_lo, uint32_t num_nodes, void* out, uint64_t cap, uint64_t* size_out);
/* LOD draw order (sdl_viewer/src/node_drawer.rs:34-43,185-205: the viewer shuffles every node it loads so that "the first N"
 * points are a uniform subsample; octree/mod.rs:286-287 asks for that order to be applied when the node is written).
 * pcv_octree_shuffle_nodes permutes positions, colours, intensity and provenance of every node in place (on the GPU) with the
 * keyed permutation pcv_lod_order(seed, node id, n) returns on the host: shuffled[i] = original[new_order[i]] (`reshuffle`). */
int pcv_octree_shuffle_nodes(pcv_octree* o, uint64_t seed);
int pcv_lod_order(uint64_t seed, uint64_t id_high, uint64_t id_low, uint64_t n, uint64_t* new_order_out);
/* All nodes at once into caller (ideally pinned) buffers: node n occupies points [point_offset, +num_points) and
 * bytes [xyz_byte_offset, +num_points*3*bpc) of these arrays (offsets from pcv_octree_nodes; no particular order). */
int pcv_octree_download(const pcv_octree* o, void* xyz_out, uint8_t* rgb_out, float* intensity_out, uint64_t* src_index_out);
/* Device views of the same arrays (valid until pcv_octree_free). */
int pcv_octree_device_arrays(const pcv_octree* o, const void** xyz, const uint8_t** rgb, const float** intensity,
                             const uint32_t** src_index);
/* <dir>/<NodeId>.xyz|.rgb|.intensity + meta.pb (on_disk.rs:17-33, lib.rs:49,74-80, proto.proto:68-149). */
int pcv_octree_write_dir(const pcv_octree* o, const char* dir);
int pcv_octree_load_dir(pcv_ctx* ctx, const char* dir, pcv_octree** out); /* Octree::from_data_provider, mod.rs:156-215 */

/* ---- a11-a14: nodes_in_location (octree/mod.rs:309-323, octree_iterator.rs:30-43) ---------- */
int pcv_nodes_in_location(const pcv_octree* o, const pcv_location* loc, uint64_t* ids_hi_lo, uint64_t cap, uint64_t* n_out);

/* ---- a17: Octree::get_visible_nodes (octree/mod.rs:228-283) --------------------------------- */
int pcv_visible_nodes(const pcv_octree* o, const double clip_from_world[16], uint64_t* ids_hi_lo, uint64_t cap, uint64_t* n_out);

/* ---- a15-a16: PointQuery streaming (iterator.rs:66-119,255-333) ----------------------------- */
/* Streams every point of every node in `loc` that passes the culling + interval filters, re-chunked
 * into batches of exactly batch_size points (last one short), on the caller's thread. */
int pcv_query_points(const pcv_octree* o, const pcv_location* loc, const pcv_interval* filters, uint32_t nfilt,
                     uint64_t batch_size, pcv_batch_cb cb, void* user);
/* Survivors of pcv_query_batch_device, written to caller-owned device buffers of `cap` points.  Inside one location
 * every point appears at most once; the order across and inside locations is unspecified.  Survivors beyond `cap`
 * are counted in counts_out but not stored. */
typedef struct pcv_query_out {
    double* xyz;         /* cap * 3, decoded positions                                           */
    uint8_t* rgb;        /* cap * 3                                                              */
    float* intensity;    /* cap, or NULL (ignored when the octree has no intensity)              */
    uint32_t* src_index; /* cap: the u32 source index the octree holds                           */
    uint32_t* loc;       /* cap, or NULL: index into locs[] of each survivor                     */
    uint64_t cap;
    uint64_t stored;     /* out: survivors written, = min(cap, sum of counts_out)                */
} pcv_query_out;
/* Throughput form: nloc locations in one call; survivors stay compacted in HBM.  counts_out[i] =
 * survivors of location i, tested_out[i] = points decoded + tested for location i.  out == NULL: the
 * survivors go to scratch buffers (capacity min(points tested, 192 Mi)) that are freed before the call returns. */
int pcv_query_batch_device(const pcv_octree* o, const pcv_location* locs, uint32_t nloc, const pcv_interval* filters,
                           uint32_t nfilt, uint64_t* counts_out, uint64_t* tested_out, pcv_query_out* out);

/* Timing / traffic of the last pcv_query_batch_device call on the context (CUDA events on the context's stream). */
typedef struct pcv_query_stats {
    float ms_device;            /* first kernel to last kernel of the call                                   */
    float ms_select;            /* node selection: per-level frontier kernels + work-list build              */
    float ms_cull;              /* the culling kernel                                                        */
    uint32_t kernel_launches;
    uint64_t algorithmic_bytes; /* SURVEY 8(d) B_query: sum over visited (location, node) of n (3 bpc + 3) + 27 per survivor */
    uint64_t tested_points, returned_points, stored_points; /* stored <= returned: survivors beyond the output capacity are only counted */
    uint64_t visited_pairs;     /* (location, node) pairs with points that were culled                       */
} pcv_query_stats;
int pcv_last_query_stats(pcv_ctx* ctx, pcv_query_stats* out);

/* ---- a19: X-ray leaf tile (xray/src/generation.rs:108-127,159-198,464-513) ------------------ */
/* query_from_global: 7 doubles or NULL.  rgba_out: w*h*4.  Returns any_points_out=0 for an empty tile
 * (the reference returns None). zbits_out (optional): w*h*32 u32 z-bucket bitsets. */
int pcv_xray_tile(const pcv_octree* o, const double tile_min[3], const double tile_max[3], uint32_t w, uint32_t h,
                  const double* query_from_global, uint8_t* rgba_out, uint32_t* zbits_out, int* any_points_out);
/* Timing / traffic of the last pcv_xray_tile[_attr] call on the context. */
typedef struct pcv_xray_stats {
    float ms_device;            /* CUDA events around the call's kernels                                    */
    uint32_t kernel_launches;
    uint64_t points;            /* points of the nodes the tile intersects (decoded + tested)               */
    uint64_t algorithmic_bytes; /* SURVEY 8(d) B_xray: sum over nodes of n (3 bpc + 3) + 4 W H               */
} pcv_xray_stats;
int pcv_last_xray_stats(pcv_ctx* ctx, pcv_xray_stats* out);
/* The other ColoringStrategyKinds (xray/src/generation.rs:76-97): point colour mean (:294-363), intensity mean brightened
 * by ln(mean - min) / ln(max - min) (:210-290; p0 = min, p1 = max), height standard deviation through the Jet (0) or
 * Purplish (1) colormap (:365-405, xray/src/colormap.rs; p0 = max_stddev).  Binning = None.  The reference accumulates in
 * arrival order from several threads, so results are defined up to rounding: expect +-1 per channel. */
enum { PCV_XRAY_COLORED = 1, PCV_XRAY_INTENSITY = 2, PCV_XRAY_HEIGHT_STDDEV = 3 };
int pcv_xray_tile_attr(const pcv_octree* o, const double tile_min[3], const double tile_max[3], uint32_t w, uint32_t h,
                       const double* query_from_global /* 7 or NULL */, int strategy, float p0, float p1, int colormap, uint8_t* rgba_out,
                       int* any_out);

/* Pixels no point falls into are TRANSPARENT.to_u8() = (255, 255, 255, 0) in every tile (src/color.rs:154-159,
 * xray/src/generation.rs:506-511). */

/* ---- f3: the rest of the X-ray pipeline (xray/src/generation.rs:129-157, 410-451, 515-759) ---- */
/* Colored / ColoredWithIntensity with Binning = Some(("intensity", bin_size)) (:66-67, :129-157): per pixel and bin
 * (bin = (intensity as f64 / bin_size) as i64) the mean colour / intensity, per pixel the mean of its bins' means
 * (:276-290, :339-346).  Needs an octree with intensities ("Binning attribute needs to be available").  The reference sums
 * in arrival / hash-map order: results are defined up to f32 rounding (+-1 per channel). */
int pcv_xray_tile_attr_binned(const pcv_octree* o, const double tile_min[3], const double tile_max[3], uint32_t w, uint32_t h,
                              const double* query_from_global /* 7 or NULL */, int strategy /* PCV_XRAY_COLORED | PCV_XRAY_INTENSITY */,
                              float p0, float p1, double bin_size, uint8_t* rgba_out, int* any_out);
/* assign_background (:695-720): every pixel with alpha < 128 becomes `background` (RGBA), in place (host buffer). */
int pcv_xray_assign_background(pcv_ctx* ctx, uint8_t* rgba, uint64_t num_pixels, const uint8_t background[4]);
/* build_node (:722-759) for one parent: build_parent's 2 x 2 mosaic of the four child images (:410-451; children[i] =
 * child_px x child_px RGBA of quadtree child i or NULL -> background; child 1 top left, 0 bottom left, 3 top right, 2 bottom
 * right) reduced to tile_px x tile_px with image 0.23's `imageops::resize(.., FilterType::Lanczos3)` (vertical pass into
 * u8, then horizontal pass; f32 weights; round-to-nearest conversion - restated, the crate is not vendored).  Host buffers. */
int pcv_xray_build_parent(pcv_ctx* ctx, const uint8_t* const children[4], uint32_t child_px, const uint8_t background[4],
                          uint32_t tile_px, uint8_t* rgba_out /* tile_px * tile_px * 4 */);
/* build_xray_quadtree (:560-622) as one call: bounding rect and levels (:515-533), every leaf tile at the deepest level
 * (:535-551, :624-667) with the chosen strategy, assign_background on the created leaves, then level by level the parents
 * (:669-693).  Every image stays in HBM until its parent is built; each finished tile is handed to `on_tile` (host
 * pointer, valid during the call; return non-zero to cancel -> PCV_ERR_CANCELLED; must not call into the same context).
 * What the reference writes as <id>.png and meta.pb is what on_tile receives plus `info`; PNG encoding stays on the host. */
typedef struct pcv_xray_quadtree_params {
    int32_t strategy;             /* 0 = XRay, or PCV_XRAY_COLORED / _INTENSITY / _HEIGHT_STDDEV                 */
    float p0, p1;                 /* as in pcv_xray_tile_attr                                                     */
    int32_t colormap;
    double bin_size;              /* 0: Binning = None                                                            */
    int32_t has_query_from_global;
    double query_from_global[7];  /* tx,ty,tz, qi,qj,qk,qw                                                        */
    uint8_t background[4];        /* tile_background_color: WHITE (255,255,255,255) or TRANSPARENT (255,255,255,0) */
    uint32_t tile_size_px;
    double pixel_size_m;
    uint8_t root_level;           /* root_node_id (quadtree/src/lib.rs:143-150); NodeId::root() = (0, 0)          */
    uint64_t root_index;
} pcv_xray_quadtree_params;
typedef struct pcv_xray_quadtree_info {
    double rect_min_x, rect_min_y, rect_edge; /* Meta::bounding_rect = the (sub-)root node's rect                 */
    uint8_t deepest_level;                    /* Meta::deepest_level                                              */
    uint32_t tile_size_px;                    /* Meta::tile_size                                                  */
    uint32_t num_nodes, num_leaves;           /* Meta::nodes = the ids on_tile received                           */
    float ms_leaves, ms_parents;              /* CUDA events: leaf tiles + background; parent kernels             */
    uint32_t kernel_launches;
    uint64_t leaf_points;                     /* XRay strategy: points decoded for the leaf tiles                 */
} pcv_xray_quadtree_info;
typedef int (*pcv_xray_tile_fn)(void* user, uint8_t level, uint64_t index, const uint8_t* rgba, uint32_t tile_size_px);
int pcv_xray_quadtree(const pcv_octree* o, const pcv_xray_quadtree_params* params, pcv_xray_tile_fn on_tile, void* user,
                      pcv_xray_quadtree_info* info_out);

/* ... with the reference's outputs: <directory>/<node id>.png for every tile ("r", "r0", "r123323": quadtree/src/lib.rs:216-233;
 * 8-bit RGBA, deflated on the host with zlib) and the quadtree's meta file (xray Meta, version 3: bounding_rect, deepest_level,
 * tile_size, nodes; "meta.pb" for the root, "meta<digits>.pb" for a sub-root: xray/src/utils.rs:7-11, lib.rs:88-139). */
int pcv_xray_quadtree_write_dir(const pcv_octree* o, const pcv_xray_quadtree_params* params, const char* directory,
                                pcv_xray_quadtree_info* info_out);

/* ---- f4: the S2-cell point cloud (src/read_write/s2.rs, src/s2_cells/mod.rs, src/geometry/s2_cell_union.rs) ---- */
/* Cell ids are the S2 library's 64-bit CellID values (face, Hilbert position, level marker bit); the arithmetic is the `s2`
 * crate's, restated (csrc/s2.h): integer and IEEE +, *, /, sqrt only, identical on host and device. */
/* CellID::from_point(p).parent(level) for every point (src/math/mod.rs:119-131). */
int pcv_s2_cell_ids(pcv_ctx* ctx, const pcv_points* host_points, uint32_t level, uint64_t* ids_out);
/* S2Splitter::write over the cloud + get_meta (read_write/s2.rs:52-125,165-173; DEFAULT_S2_SPLIT_LEVEL = 20): every point must
 * be a valid ECEF point (|p| in [6 352 800, 6 384 400] m, else PCV_ERR_INVALID with the reference's message); points are grouped
 * by cell - cells in id order, inside a cell in input order - as Plain-encoded f64 positions plus colour / intensity. */
typedef struct pcv_s2cloud pcv_s2cloud;
int pcv_s2_build(pcv_ctx* ctx, const pcv_points* host_points, uint32_t split_level, pcv_s2cloud** out);
int pcv_s2_build_device(pcv_ctx* ctx, const pcv_points* dev_points, uint32_t split_level, pcv_s2cloud** out);
void pcv_s2_free(pcv_s2cloud* cloud);
/* S2Meta: cells + num_points (mod.rs:23-41), bounding box, attributes. */
int pcv_s2_info(const pcv_s2cloud* cloud, uint64_t* num_cells, uint64_t* num_points, uint32_t* split_level, double bbox_min[3],
                double bbox_max[3], int* has_color, int* has_intensity);
int pcv_s2_cells(const pcv_s2cloud* cloud, uint64_t* ids_out, uint64_t* num_points_out);
/* Device time of the build (CUDA events: keys, sort, run starts, gather; the bounding-box pass and the host reads between them
 * included), kernel launches, and the compulsory bytes: every point read once and written once into its cell. */
int pcv_s2_build_stats(const pcv_s2cloud* cloud, float* ms_device, uint32_t* kernel_launches, uint64_t* algorithmic_bytes);
/* points_in_node (mod.rs:174-190): one cell's arrays; PCV_ERR_NOT_FOUND for an id the cloud does not hold. */
int pcv_s2_cell_data(const pcv_s2cloud* cloud, uint64_t cell_id, double* xyz_out /* n*3 */, uint8_t* rgb_out, float* intensity_out,
                     uint64_t* src_index_out);
/* nodes_in_location for PointLocation::AllPoints (union_ids == NULL) and PointLocation::S2Cells (mod.rs:157-168, 233-241:
 * the cells whose id range intersects the union's; the union is normalised first).  ids_out may be NULL to count. */
int pcv_s2_cells_in_union(const pcv_s2cloud* cloud, const uint64_t* union_ids, uint32_t n_union, uint64_t* ids_out, uint64_t cap,
                          uint64_t* n_out);
/* The FilteredIterator over those cells with the CellUnion as PointCulling (s2_cell_union.rs:27-31): survivors in cell order,
 * input order inside a cell.  n_out = number of survivors (may exceed cap: only cap are written). */
int pcv_s2_query_union(const pcv_s2cloud* cloud, const uint64_t* union_ids, uint32_t n_union, double* xyz_out, uint8_t* rgb_out,
                       float* intensity_out, uint64_t* src_index_out, uint64_t cap, uint64_t* n_out, uint64_t* tested_out);
/* The directory an S2Splitter<RawNodeWriter> leaves behind (read_write/s2.rs:127-145, raw.rs): per cell `<to_token()>.xyz`
 * (f64 LE x, y, z), `.rgb`, `.intensity`, and meta.pb = Meta { version 13, bounding_box, s2 { cells, attributes } }
 * (s2_cells/mod.rs:77-104); load = S2Cells::from_data_provider over such a directory (:106-147, :203-216; versions < 12 and
 * octree metas are rejected with the reference's messages). */
int pcv_s2_write_dir(const pcv_s2cloud* cloud, const char* directory);
int pcv_s2_load_dir(pcv_ctx* ctx, const char* directory, pcv_s2cloud** out);
/* CellUnion::contains for arbitrary points: mask_out[i] = union.contains_cellid(CellID::from_point(p_i)). */
int pcv_s2_union_contains(pcv_ctx* ctx, const pcv_points* host_points, const uint64_t* union_ids, uint32_t n_union, uint8_t* mask_out);

/* ---- multi-GPU helpers (points shard by level-k path prefix; SURVEY.md 8e) ------------------ */
/* Per-point level-k cell (first k steps of the re-quantising descent on the raw positions) ->
 * 8^k histogram; then a stable pack of the points of each destination rank into contiguous send
 * buffers.  The exchange itself is one NCCL all-to-all issued by the host layer. */
int pcv_prefix_histogram_device(pcv_ctx* ctx, const pcv_points* dev_points, double resolution, const double bbox_min[3],
                                const double bbox_max[3], uint32_t k, uint64_t* counts_out /* 8^k, host */);
/* The same histogram with find_bounding_box (generation.rs:256-270) of the local points folded into the one read of the
 * positions.  Both histogram calls keep the per-point cells on the context for exactly ONE following pack call over the same
 * device arrays, box and resolution, which reuses them instead of repeating the descent and then drops them (the caller must not
 * modify the points between the histogram and that pack; a pack without a fresh histogram recomputes the cells). */
int pcv_prefix_histogram_bbox_device(pcv_ctx* ctx, const pcv_points* dev_points, double resolution, const double bbox_min[3],
                                     const double bbox_max[3], uint32_t k, uint64_t* counts_out, double data_min[3], double data_max[3]);
int pcv_prefix_pack_device(pcv_ctx* ctx, const pcv_points* dev_points, const uint64_t* dev_global_index /* or NULL */,
                           uint64_t global_index_base /* used when dev_global_index == NULL: index = base + i */, double resolution,
                           const double bbox_min[3], const double bbox_max[3], uint32_t k,
                           const int32_t* cell_to_rank /* 8^k, host */, uint32_t nranks, double* dev_xyz_out /* n*3 AoS */,
                           uint8_t* dev_rgb_out, float* dev_intensity_out, uint64_t* dev_index_out,
                           uint64_t* rank_counts_out /* nranks, host */);
/* Fused pack + exchange: the same stable pack, but every record is stored straight into the destination rank's receive
 * arrays (SoA: x, y, z f64; global index u64; intensity f32; colour packed r | g << 8 | b << 16 as u32) - local memory
 * for the own rank, peer memory mapped through CUDA IPC (below) for the others, so the transfer over NVLink / NVSwitch
 * overlaps the ranking; there is no send buffer and no collective call.  dst_*[r]: base pointers of rank r's arrays as
 * mapped in THIS process; dst_first[r]: first slot of this rank's block inside them (sum of the counts of lower ranks).
 * The call returns after the kernel has completed; the caller then runs one inter-process barrier. */
int pcv_prefix_pack_exchange_device(pcv_ctx* ctx, const pcv_points* dev_points, const uint64_t* dev_global_index /* or NULL */,
                                    uint64_t global_index_base, double resolution, const double bbox_min[3], const double bbox_max[3],
                                    uint32_t k, const int32_t* cell_to_rank /* 8^k, host */, uint32_t nranks,
                                    const uint64_t* dst_first /* nranks, host */, void* const* dst_x, void* const* dst_y, void* const* dst_z,
                                    void* const* dst_index, void* const* dst_intensity /* or NULL */, void* const* dst_colour,
                                    uint64_t* rank_counts_out /* nranks, host */);
int pcv_unpack_colours_device(pcv_ctx* ctx, const uint32_t* dev_colour, uint64_t n, uint8_t* dev_rgb /* n * 3 */);
/* Exportable device memory (plain cudaMalloc + cudaIpcGetMemHandle) and its mapping in a peer process. */
int pcv_ipc_alloc(pcv_ctx* ctx, uint64_t bytes, void** dev_ptr, uint8_t handle_out[64]);
int pcv_ipc_free(pcv_ctx* ctx, void* dev_ptr);
int pcv_ipc_open(pcv_ctx* ctx, const uint8_t handle[64], void** dev_ptr);
int pcv_ipc_close(pcv_ctx* ctx, void* dev_ptr);
/* ---- exchange of ingested records (SURVEY.md 8e, round 2): every rank runs the first step of the chain on its own points, the
 * records (three level-1 codes 12 B + packed colour 4 B as one 16-byte record, digits 1 B [+ intensity 4 B]; Float64 trees: 32-byte
 * records + a separate colour array) move once into the owners' receive slabs, and every owner's build starts at its first
 * partition pass - nothing is computed twice and 17 instead of 40 bytes per point cross NVLink.
 *   pcv_shard_ingest_device   ingest kernel + per-tile digit histogram of the local points; counts_out = their 8^k level-k cells
 *   pcv_shard_exchange_device one kernel: rank every record by destination and store it straight into the destination slab
 *                             (dst_*[r] = rank r's slab arrays as mapped in THIS process, capacity + 64 bytes of slack each;
 *                             dst_first[r] = first slot of this rank's block in them).  idx of a stored record = its slot.
 *                             Returns after the kernel has completed; the caller then runs one inter-process barrier.
 *   pcv_shard_send_dest       per local point the rank it went to (device, n bytes; valid until pcv_shard_send_free)
 *   pcv_build_octree_from_records_device  the owner's build over its slab (dev_col == NULL: narrow records carrying their colour,
 *                             as pcv_shard_exchange_device stores them; the slab is reused as scratch by the build). */
typedef struct pcv_shard_send pcv_shard_send;
int pcv_shard_ingest_device(pcv_ctx* ctx, const pcv_points* dev_points, double resolution, const double bbox_min[3], const double bbox_max[3],
                            uint32_t k, uint64_t* counts_out /* 8^k, host */, pcv_shard_send** out);
int pcv_shard_exchange_device(pcv_shard_send* s, uint32_t k, const int32_t* cell_to_rank /* 8^k, host */, uint32_t nranks,
                              const uint64_t* dst_first /* nranks, host */, void* const* dst_rec, void* const* dst_col, void* const* dst_dig,
                              void* const* dst_intensity /* or NULL */, uint64_t* rank_counts_out /* nranks, host */);
int pcv_shard_send_info(const pcv_shard_send* s, int* wide_records /* 1: 32-byte records (a Float64 level exists) */, int* digit_levels);
int pcv_shard_send_dest(const pcv_shard_send* s, const uint8_t** dev_dest, uint64_t* n);
void pcv_shard_send_free(pcv_shard_send* s);
int pcv_build_octree_from_records_device(pcv_ctx* ctx, void* dev_rec, uint32_t* dev_col, uint8_t* dev_dig, const float* dev_intensity, uint64_t n,
                                         double resolution, const double bbox_min[3], const double bbox_max[3], uint32_t k,
                                         const uint64_t* prefix_counts, pcv_octree** out);
/* ---- fused exchange pass: the sender's first partition pass (root -> level-2 cells, two levels of the chain finished, the next
 * pass's first step done) stores every bucket straight into the buffers of the cell's owner - peer memory over NVLink - so the
 * transfer overlaps the partition tile by tile and the owner's build starts at its SECOND pass.  Narrow records that continue travel
 * as {codes, colour} + 1 digit byte (17 B per point), their index implied by their position (= slot); records of level-2 leaves go
 * to the owner's arena with an explicit slot.  Needs prefix depth 2; everything follows from the gathered histograms:
 *   hist_all[s * 64 + c]  points of sender s in level-2 cell c (all-gather of pcv_shard_ingest_device's counts at k = 2)
 *   dst[r]                rank r's buffers as mapped in THIS process (capacity >= slots_out[r] entries + 64 bytes of slack each)
 *   slots_out[r]          slots rank r owns; first_bins_out: this rank's own per-cell counts (input of the owner's build)
 * Returns PCV_ERR_UNSUPPORTED when the layout does not allow it (the caller then uses pcv_shard_exchange_device). */
typedef struct pcv_shard_bufs {
    void* rec_next;   /* slots x 16 B (32 B for wide records) */
    void* col_next;   /* wide records only: slots x 4 B, else NULL */
    void* dig_next;   /* slots x 1 B */
    void* arena;      /* slots x 16 / 32 B: leaf records (the whole build's leaf arena) */
    void* col_arena;  /* slots x 4 B */
    void* intensity;  /* slots x 4 B or NULL */
} pcv_shard_bufs;
int pcv_shard_pass_device(pcv_shard_send* s, uint32_t nranks, uint32_t rank, const int32_t* cell_to_rank /* 64 */, const uint64_t* hist_all,
                          const pcv_shard_bufs* dst /* nranks */, uint64_t* slots_out /* nranks or NULL */, uint64_t* first_bins_out /* 64 or NULL */);
/* after pcv_shard_pass_device: per local point its level-2 cell (device, n bytes; valid until pcv_shard_send_free) */
int pcv_shard_send_cells(const pcv_shard_send* s, const uint8_t** dev_cells, uint64_t* n);
/* the owner's build after every sender's pcv_shard_pass_device has completed (one inter-process barrier in between) */
int pcv_build_octree_after_pass_device(pcv_ctx* ctx, const pcv_shard_bufs* own, uint64_t nslots, const uint64_t* first_bins /* 64 */, double resolution,
                                       const double bbox_min[3], const double bbox_max[3], const uint64_t* prefix_counts /* levels 1..2 */, pcv_octree** out);
/* Local part of a sharded build: like pcv_build_octree_device, but nodes of levels <= k take their split decision from
 * the GLOBAL counts (`prefix_counts`: levels 1..k concatenated, 8 + 64 + .. entries, host), and the nodes of level k-1
 * collect the every-8th points of their local children for pcv_assemble_top. */
int pcv_build_octree_sharded_device(pcv_ctx* ctx, const pcv_points* dev_points, double resolution, const double bbox_min[3],
                                    const double bbox_max[3], uint32_t k, const uint64_t* prefix_counts, pcv_octree** out);
/* n(X): size of node X at the moment it is subsampled into its parent (needed from every level-k node by the assembly). */
int pcv_octree_node_nsub(const pcv_octree* o, uint64_t id_high, uint64_t id_low, uint64_t* nsub_out);
int pcv_octree_nsub_all(const pcv_octree* o, uint64_t* out, uint64_t cap); /* same order as pcv_octree_nodes */
/* Nodes of levels 0..k-1 from the gathered collector content (host buffers; level k-1 nodes in index order, inside a
 * node child order, positions as node-file bytes in the collector's encoding).  src_index of the result = position in
 * the gathered arrays. */
int pcv_assemble_top(pcv_ctx* ctx, double resolution, const double bbox_min[3], const double bbox_max[3], uint32_t k,
                     const uint64_t* prefix_counts, const uint64_t* unit_nsub /* 8^k */, const void* xyz_codes, const uint8_t* rgb,
                     const float* intensity, uint64_t npoints, pcv_octree** out);

/* ---- the whole sharded build as ONE call per rank (SURVEY.md 8e).  The three collectives come from the caller (NCCL, MPI,
 * torch.distributed ...: anything that offers them over host buffers), everything else - ingest, global histogram, cells -> ranks,
 * the slab set-up over CUDA IPC (cached per context), the fused record exchange over NVLink, the owner's build, the assembly of the
 * nodes above level k on rank 0 - happens behind this boundary.  Every callback returns 0 on success.  All ranks must call with the
 * same resolution / bbox / prefix_levels (1 or 2); one process per GPU on one node.
 *   local_out: this rank's nodes of levels >= k (and the collectors it contributed to); top_out: rank 0 only, levels < k
 *   k_out: the prefix depth actually used (<= prefix_levels, distributed.py usable_prefix_levels)
 *   cell_to_rank_out / unit_nsub_out: optional, 8^prefix_levels entries each (the first 8^k are written)
 *   recv_points_out: optional, the points this rank owns
 *   send_out: optional; when given, the caller owns the handle and frees it with pcv_shard_send_free.  It keeps one byte per
 *   local point - its level-2 cell (pcv_shard_send_cells) after the fused exchange pass, else the rank it went to
 *   (pcv_shard_send_dest) - which together with the gathered histograms reconstructs the provenance of every slot.
 * PCV_NO_FUSED_PASS=1 (environment) forces the exchange of ingested records + the owner's full build. */
typedef struct pcv_comm {
    void* user;
    int rank, world;
    int (*allreduce_sum_u64)(void* user, uint64_t* inout, uint64_t count);
    int (*allgather)(void* user, const void* send, uint64_t bytes, void* recv /* world * bytes, rank order */);
    int (*barrier)(void* user);
} pcv_comm;
int pcv_build_octree_sharded(pcv_ctx* ctx, const pcv_comm* comm, const pcv_points* dev_points, double resolution, const double bbox_min[3],
                             const double bbox_max[3], uint32_t prefix_levels, pcv_octree** local_out, pcv_octree** top_out, uint32_t* k_out,
                             int32_t* cell_to_rank_out, uint64_t* unit_nsub_out, uint64_t* recv_points_out, pcv_shard_send** send_out);
/* Wall-clock milliseconds of the last pcv_build_octree_sharded on this context, per phase (each ends in a stream synchronisation or
 * a barrier): ingest + histogram, all-reduce + plan (+ slab set-up on the first call), exchange, local build, top assembly;
 * out[5] = 1 when the exchange was the fused exchange pass. */
int pcv_sharded_phases(pcv_ctx* ctx, double out[6]);
/* Releases the receive slab pcv_build_octree_sharded caches on the context (collective: every rank calls it). */
int pcv_sharded_release(pcv_ctx* ctx, const pcv_comm* comm);

/* ---- PLY input (SURVEY.md 8f rank 1): src/read_write/ply.rs:126-229 (parse_header), :327-450
 * (PlyIterator::from_file), :453-556 (batches), src/octree/generation.rs:256-287 (find_bounding_box,
 * build_octree_from_file).  The file body goes to the GPU as raw vertex records through a pinned,
 * double-buffered staging ring; one kernel turns the records into the SoA arrays pcv_build_octree_device
 * takes (position = (x, y, z) as f64 + header offset, colour r,g,b, intensity) and reduces the bounding box
 * in the same pass (the reference reads the whole file twice). ------------------------------------- */
enum {  /* property types, ply.rs:43-73 */
    PCV_PLY_I8 = 0, PCV_PLY_U8, PCV_PLY_I16, PCV_PLY_U16, PCV_PLY_I32, PCV_PLY_U32, PCV_PLY_I64, PCV_PLY_U64, PCV_PLY_F32, PCV_PLY_F64
};
typedef struct pcv_ply_info {
    uint64_t num_points;   /* `element vertex N`                                                   */
    uint64_t header_bytes; /* the body starts here (the vertex element must come first)            */
    uint32_t record_bytes; /* bytes per vertex, skipped properties included                        */
    int32_t has_color;     /* uchar red/green/blue (or r/g/b) present                              */
    int32_t has_intensity; /* float `intensity` present                                            */
    int32_t type_xyz[3];   /* PCV_PLY_* of x, y, z (cast to f64 like `as f64`; int8 reads unsigned) */
    uint32_t off_xyz[3];   /* byte offsets inside the record                                       */
    uint32_t off_rgb[3];
    uint32_t off_intensity;
    double offset[3];      /* `comment offset: x y z`, added to every position                     */
} pcv_ply_info;
/* Parses the header with the reference's rules and error conditions (where the reference panics — no vertex element,
 * not binary_little_endian, missing x/y/z — this returns PCV_ERR_INVALID; unreadable file: PCV_ERR_IO). */
int pcv_ply_read_header(const char* path, pcv_ply_info* out);
/* Kernel-level entry: `n` raw records already in device memory (16-byte aligned) -> SoA arrays (device).  rgb /
 * intensity may be NULL.  bbox_min/max (host, may be NULL) receive the component-wise min/max of the positions
 * (Aabb::grow, aabb.rs:41-44); for n == 0 they are Aabb::zero (generation.rs:269). */
int pcv_ply_unpack_device(pcv_ctx* ctx, const pcv_ply_info* info, const void* dev_records, uint64_t n, double* dev_x,
                          double* dev_y, double* dev_z, uint8_t* dev_rgb, float* dev_intensity, double bbox_min[3],
                          double bbox_max[3]);
/* File -> device SoA arrays (capacity info->num_points each) + bounding box; a truncated body is PCV_ERR_IO. */
int pcv_ply_load_device(pcv_ctx* ctx, const char* path, const pcv_ply_info* info, double* dev_x, double* dev_y,
                        double* dev_z, uint8_t* dev_rgb, float* dev_intensity, double bbox_min[3], double bbox_max[3]);
/* build_octree_from_file (generation.rs:272-287): bounding box of the file's points, then build_octree.  Colour is
 * mandatory; `with_intensity` mirrors "intensity" in the reference's `attributes` argument. */
int pcv_build_octree_from_file(pcv_ctx* ctx, const char* path, double resolution, int with_intensity, pcv_octree** out);

/* ---- synthetic inputs for benchmarks / parity tests (integer-only, counter based) ----------- */
enum { PCV_SYNTH_SLAB_ECEF = 1, PCV_SYNTH_GAUSS_CLUSTERS = 2 };
int pcv_synth_points_device(pcv_ctx* ctx, int kind, uint64_t seed, uint64_t first_index, uint64_t n, double* dev_x,
                            double* dev_y, double* dev_z, uint8_t* dev_rgb);
int pcv_synth_points_host(int kind, uint64_t seed, uint64_t first_index, uint64_t n, double* x, double* y, double* z, uint8_t* rgb);
int pcv_synth_bbox(int kind, double bbox_min[3], double bbox_max[3], double* resolution);

/* ---- device memory from the context's stream-ordered pool (so that callers' staging buffers, e.g. the all-to-all
 * send/receive buffers of the sharded build, share one allocator with the build's working set) --------------------- */
int pcv_device_alloc(pcv_ctx* ctx, uint64_t bytes, void** out); /* usable on any stream after the call returns */
int pcv_device_free(pcv_ctx* ctx, void* ptr);                   /* caller guarantees its own streams are done with it */

/* ---- instrumentation ------------------------------------------------------------------------ */
typedef struct pcv_build_stats {
    uint64_t kernel_launches; /* CUDA kernels launched by the last build on this context           */
    uint32_t passes;
    uint32_t deepest_level;
    uint64_t num_nodes;
    uint64_t algorithmic_bytes; /* 27*N + sum_nodes n*(3*bpc+3) (+8*N with intensity)             */
    float ms_host_plan, ms_partition, ms_place, ms_total; /* ms_partition/place/total: CUDA events on the context's stream;
                                                             ms_host_plan: host time spent planning passes (inside ms_total) */
    float ms_host_wait;                                   /* host time blocked on the per-pass histogram read-back       */
} pcv_build_stats;
/* Work buffers are recycled inside the context (by exact size, at most half of the device memory) and in the device's stream-ordered
 * pool, so that repeated builds make no allocator calls.  This returns all of it to the driver (e.g. before another library needs
 * the memory). */
int pcv_release_cached_memory(pcv_ctx* ctx);
int pcv_last_build_stats(pcv_ctx* ctx, pcv_build_stats* out);
/* Optional per-kernel timing: CUDA events on the context's stream around every launch of the build kernels.
 * Off by default (the events serialise nothing but cost host time); turn on for a measurement build. */
typedef struct pcv_kernel_stat {
    char name[24];
    uint64_t launches;
    uint64_t algorithmic_bytes; /* bytes the launches had to move (reads of inputs/records + writes of records/outputs) */
    double ms;
} pcv_kernel_stat;
int pcv_set_profiling(pcv_ctx* ctx, int on); /* also resets the accumulated statistics */
int pcv_kernel_stats(pcv_ctx* ctx, pcv_kernel_stat* out, uint32_t cap, uint32_t* n_out);
uint64_t pcv_kernel_launch_count(pcv_ctx* ctx); /* cumulative, all entry points                    */

#ifdef __cplusplus
}
#endif
#endif /* PCV_H */
