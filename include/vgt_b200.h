/*
 * vgt_b200.h -- C-ABI of the B200 (sm_100a) backend for the occupancy -> SDF hot path of
 * calderpg/voxelized_geometry_tools. Plain C: raw pointers, sizes, no C++/Eigen/torch types.
 *
 * Every entry point names the reference interface it replaces (paths relative to the
 * reference checkout). Grids use the reference's storage convention
 * (common_robotics_utilities VoxelGrid; mirrored at
 * src/voxelized_geometry_tools/cuda_voxelization_helpers.cu:281-282):
 *     linear index = x * (ny * nz) + y * nz + z        (x slowest, z contiguous)
 * OccupancyMap raw data is a packed float[nx*ny*nz] (include/.../occupancy_map.hpp:28-58).
 *
 * Conventions
 *   - every function returns VGT_B200_OK (0) or an error code; vgt_b200_last_error() returns a
 *     thread-local message for the last failing call on the calling thread.
 *   - "host" entry points take HOST pointers and do their own H2D/D2H; "_dev" entry points take
 *     DEVICE pointers on `device` plus a cudaStream_t (passed as void*; NULL = legacy default
 *     stream) and never synchronise the host unless stated.
 *   - all functions may be called concurrently from several host threads (each call sets the
 *     device it needs and works on its own streams and buffers). Process-wide state is limited
 *     to mutex-protected caches that cannot change a result: the pinned staging slots and host
 *     copy threads of the host-pointer entries, the A/B switches read once from the environment
 *     (vgt_b200_reload_tuning) and a launch counter; the error string is thread-local.
 *   - there is NO CPU fallback: without a usable CUDA device every compute call fails with
 *     VGT_B200_ERR_DEVICE.
 */
#ifndef VGT_B200_H_
#define VGT_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define VGT_B200_API __attribute__((visibility("default")))

enum
{
  VGT_B200_OK = 0,
  /* maps to std::invalid_argument in the C++ adapter (sdfgen.hpp:123-126, pcv_if.hpp:30-41,267-288) */
  VGT_B200_ERR_INVALID_ARGUMENT = 1,
  /* maps to std::runtime_error (cuda.cu:26-33 "[msg] Cuda error [str]", dev_pcv.hpp:34-46) */
  VGT_B200_ERR_DEVICE = 2,
  VGT_B200_ERR_UNSUPPORTED = 3,
  /* maps to std::runtime_error("Triangle is not contained by occupancy map")
   * (mesh_rasterizer.cpp:191-196) */
  VGT_B200_ERR_NOT_CONTAINED = 4,
  /* maps to std::out_of_range (vertices.at() / triangles.at(), mesh_rasterizer.cpp:122-125) */
  VGT_B200_ERR_OUT_OF_RANGE = 5
};

/* "no opposite-class voxel anywhere": the reference's +inf squared distance. */
#define VGT_B200_SQ_INF INT32_MAX

/* Largest supported voxel count per axis (squared distances must stay below 2^31). */
#define VGT_B200_MAX_AXIS 8192

VGT_B200_API const char* vgt_b200_last_error(void);
VGT_B200_API const char* vgt_b200_version(void);

/* Experiment / test aid (no reference counterpart). The library reads its VGT_B200_* A/B
 * switches (which kernel variant serves the strided passes; none of them changes a result) from
 * the environment once, at the first SDF call of the process. This re-reads them, for tests
 * that force each variant inside one process. */
VGT_B200_API void vgt_b200_reload_tuning(void);

/* Measurement aid (no reference counterpart): the number of CUDA kernels this library has
 * launched in this process so far, over all threads and devices. bench.py reports the difference
 * across its timed region as "gpu_launches". */
VGT_B200_API uint64_t vgt_b200_kernel_launch_count(void);

/* Replaces cuda_helpers::GetAvailableDevices() / IsAvailable()
 * (src/.../cuda_voxelization_helpers.cu:562-637, 769-822). Returns the number of usable
 * sm_100 devices (0 when there is none or the driver is missing; never an error). */
VGT_B200_API int vgt_b200_device_count(void);

/* ---------------------------------------------------------------------------------------------
 * Signed distance field generation
 * ------------------------------------------------------------------------------------------- */

/* Replaces OccupancyMap::ExtractSignedDistanceField<float> -> internal::ExtractSignedDistanceField
 * (include/.../occupancy_map.hpp:174-210, include/.../signed_distance_field_generation.hpp:39-113
 * and :115-285 for add_virtual_border) followed by SignedDistanceField::Lock()
 * (include/.../signed_distance_field.hpp:765-787).
 *   occupancy          host float[nx*ny*nz]; filled iff occ > 0.5 or (unknown_is_filled and occ == 0.5)
 *   resolution         voxel edge length (> 0, finite); the grid must be uniform (sdfgen.hpp:123-126)
 *   sdf_out            host float[nx*ny*nz]: +d outside, -d inside, +/-inf when a class is absent
 *   out_min, out_max   may be NULL; the values Lock() would cache
 */
VGT_B200_API int vgt_b200_sdf_f32(
    const float* occupancy, int64_t nx, int64_t ny, int64_t nz, double resolution,
    int unknown_is_filled, int add_virtual_border, int device, float* sdf_out, float* out_min,
    float* out_max);

/* The same call on SEVERAL devices of one box, from one process: the grid is cut into x-slabs
 * (one per listed device), the z and y passes run slab-local with the exchange fused into the
 * y pass (NVLink peer stores into the other devices' receive buffers; peer access is enabled
 * between the listed devices), the x pass + finalize on y-slabs, and every device copies its
 * y-slab into its rows of sdf_out. Same result, bit for bit, as vgt_b200_sdf_f32.
 * Replaces the same reference code (include/.../occupancy_map.hpp:174-210); the reference's only
 * parallelism is the OpenMP split over lines (src/.../signed_distance_field_generation.cpp:286-389).
 *   devices, num_devices   1..8 distinct device ordinals; 1 device = vgt_b200_sdf_f32.
 * Fails with VGT_B200_ERR_DEVICE when two of the devices cannot reach each other as peers (no
 * fallback). Uses one host thread per device for the duration of the call. */
VGT_B200_API int vgt_b200_sdf_f32_multi(
    const float* occupancy, int64_t nx, int64_t ny, int64_t nz, double resolution,
    int unknown_is_filled, int add_virtual_border, const int* devices, int num_devices,
    float* sdf_out, float* out_min, float* out_max);

/* Same for SignedDistanceField<double> (ExtractSignedDistanceFieldDouble, occupancy_map.cpp:250-254). */
VGT_B200_API int vgt_b200_sdf_f64(
    const float* occupancy, int64_t nx, int64_t ny, int64_t nz, double resolution,
    int unknown_is_filled, int add_virtual_border, int device, double* sdf_out, double* out_min,
    double* out_max);

/* vgt_b200_sdf_f64 on SEVERAL devices of one box (ExtractSignedDistanceFieldDouble,
 * occupancy_map.cpp:250-254): the x-slab / y-slab cut, the exchange and the rules of
 * vgt_b200_sdf_f32_multi; the same bytes as vgt_b200_sdf_f64 (field, min and max).
 *   devices, num_devices   1..8 distinct ordinals in [0, 64), no more than nx or ny;
 *                          1 device = vgt_b200_sdf_f64.
 *   Device memory, per slab on its device: 4 B per voxel of its x-slab for the occupancy and 4 B
 *   per voxel for the local-pass scratch; a receive buffer of 4 * nx * ceil(ny / num_devices) * nz
 *   bytes, kept for the life of the process; 8 B per voxel of its y-slab for the SDF; a magnitude
 *   table of at most 8 MB.
 * Every argument, the device list included, is checked before the first device call. Fails with
 * VGT_B200_ERR_DEVICE when two of the devices cannot reach each other as peers (no fallback). */
VGT_B200_API int vgt_b200_sdf_f64_multi(
    const float* occupancy, int64_t nx, int64_t ny, int64_t nz, double resolution,
    int unknown_is_filled, int add_virtual_border, const int* devices, int num_devices,
    double* sdf_out, double* out_min, double* out_max);

/* For grids whose filled predicate is an opaque std::function (the other map types,
 * include/.../signed_distance_field_generation.hpp:115-121): the adapter evaluates the predicate
 * on the host into filled_mask (uint8, non-zero = filled) and calls this. */
VGT_B200_API int vgt_b200_sdf_from_mask_f32(
    const uint8_t* filled_mask, int64_t nx, int64_t ny, int64_t nz, double resolution,
    int add_virtual_border, int device, float* sdf_out, float* out_min, float* out_max);

VGT_B200_API int vgt_b200_sdf_from_mask_f64(
    const uint8_t* filled_mask, int64_t nx, int64_t ny, int64_t nz, double resolution,
    int add_virtual_border, int device, double* sdf_out, double* out_min, double* out_max);

/* ---- the other map types (SURVEY.md section 8f, rank 1) ----
 * OccupancyComponentMap, TaggedObjectOccupancyMap and TaggedObjectOccupancyComponentMap store
 * packed cells of 8 or 16 bytes whose first word is the float occupancy and whose second word is
 * the object id (tagged maps) or the component (component map, never read here):
 *   include/.../occupancy_component_map.hpp:28-64, tagged_object_occupancy_map.hpp:28-68,
 *   tagged_object_occupancy_component_map.hpp:17-60 (static_asserts pin the sizes).
 * `cells` is GetImmutableRawData().data() of such a map; the filled predicate runs on the device.
 *
 * vgt_b200_sdf_from_cells_*: replaces ExtractSignedDistanceField<T>(objects_to_use, parameters)
 *   (tagged_object_occupancy_map.hpp:199-247, tagged_object_occupancy_component_map.hpp:360-410)
 *   and, with num_object_ids == 0, OccupancyComponentMap::ExtractSignedDistanceField<T>
 *   (occupancy_component_map.hpp:270-306): a cell is filled iff the occupancy rule holds and
 *   (num_object_ids == 0 or its object id is listed). */
VGT_B200_API int vgt_b200_sdf_from_cells_f32(
    const void* cells, int cell_bytes, int64_t nx, int64_t ny, int64_t nz, double resolution,
    int unknown_is_filled, int add_virtual_border, const uint32_t* object_ids,
    int64_t num_object_ids, int device, float* sdf_out, float* out_min, float* out_max);

VGT_B200_API int vgt_b200_sdf_from_cells_f64(
    const void* cells, int cell_bytes, int64_t nx, int64_t ny, int64_t nz, double resolution,
    int unknown_is_filled, int add_virtual_border, const uint32_t* object_ids,
    int64_t num_object_ids, int device, double* sdf_out, double* out_min, double* out_max);

/* Replaces MakeSeparateObjectSDFs<T>(object_ids, parameters)
 * (tagged_object_occupancy_map.hpp:249-262): one SDF per listed object, the cells uploaded once.
 * sdf_out holds num_object_ids grids back to back, out_min / out_max one value per object. */
VGT_B200_API int vgt_b200_sdf_per_object_f32(
    const void* cells, int cell_bytes, int64_t nx, int64_t ny, int64_t nz, double resolution,
    int unknown_is_filled, int add_virtual_border, const uint32_t* object_ids,
    int64_t num_object_ids, int device, float* sdf_out, float* out_min, float* out_max);

VGT_B200_API int vgt_b200_sdf_per_object_f64(
    const void* cells, int cell_bytes, int64_t nx, int64_t ny, int64_t nz, double resolution,
    int unknown_is_filled, int add_virtual_border, const uint32_t* object_ids,
    int64_t num_object_ids, int device, double* sdf_out, double* out_min, double* out_max);

/* Replaces ExtractFreeAndNamedObjectsSignedDistanceField<T>(parameters)
 * (tagged_object_occupancy_map.hpp:293-378): the SDF of all filled cells and the SDF of the
 * filled cells of named objects (id > 0), merged (free >= 0 -> free; else named <= -0 -> named;
 * else 0), min/max of the merged field. */
VGT_B200_API int vgt_b200_sdf_free_and_named_f32(
    const void* cells, int cell_bytes, int64_t nx, int64_t ny, int64_t nz, double resolution,
    int unknown_is_filled, int add_virtual_border, int device, float* sdf_out, float* out_min,
    float* out_max);

VGT_B200_API int vgt_b200_sdf_free_and_named_f64(
    const void* cells, int cell_bytes, int64_t nx, int64_t ny, int64_t nz, double resolution,
    int unknown_is_filled, int add_virtual_border, int device, double* sdf_out, double* out_min,
    double* out_max);

/* The three cell entries above on SEVERAL devices of one box, for maps one device cannot hold;
 * they replace the same reference code (tagged_object_occupancy_map.hpp:199-262, :293-378,
 * occupancy_component_map.hpp:270-306). Each takes the argument list of its host entry with
 * `int device` replaced by `devices, num_devices`, and follows vgt_b200_sdf_f32_multi: slab g
 * of the cells (x-slab) is uploaded to devices[g] once and classified there, the z and y passes
 * run slab-local with the exchange fused into the y pass (peer stores), and the x pass + finalize
 * runs on y-slab g. The result is the same bytes as the host entry: every field and min/max pair.
 *   devices, num_devices   1..8 distinct ordinals in [0, 64), no more than nx or ny;
 *                          1 device = the host entry.
 *   vgt_b200_sdf_from_cells_*_multi     one round: the filled mask, the passes.
 *   vgt_b200_sdf_free_and_named_*_multi two rounds on the resident cell slab (all filled cells,
 *                                       then named objects), merged on each y-slab.
 *   vgt_b200_sdf_per_object_*_multi     one round per listed id; the slab is classified once per
 *                                       group of 255 distinct ids (the slot map of the _dev
 *                                       batch). sdf_out is T[num_object_ids][nx*ny*nz], out_min /
 *                                       out_max one value per listed id. Repeated ids and ids
 *                                       absent from the map are allowed; num_object_ids == 0
 *                                       launches nothing. num_object_ids * nx*ny*nz * sizeof(T)
 *                                       beyond int64 is refused.
 *   Device memory, per slab on its device: its x-slab of cells (cell_bytes per voxel), 1 B per
 *   voxel of the x-slab for the mask (the slot map of the batch) and 4 B for the local-pass
 *   scratch; a receive buffer of 4 * nx * ceil(ny / num_devices) * nz bytes, kept for the life
 *   of the process; sizeof(T) per voxel of its y-slab for the SDF (two y-slabs for
 *   free-and-named); a magnitude table of at most 4 / 8 MB.
 * Every argument, the device list included, is checked before the first device call. Fails with
 * VGT_B200_ERR_DEVICE when two of the devices cannot reach each other as peers (no fallback). */
VGT_B200_API int vgt_b200_sdf_from_cells_f32_multi(
    const void* cells, int cell_bytes, int64_t nx, int64_t ny, int64_t nz, double resolution,
    int unknown_is_filled, int add_virtual_border, const uint32_t* object_ids,
    int64_t num_object_ids, const int* devices, int num_devices,
    float* sdf_out, float* out_min, float* out_max);

VGT_B200_API int vgt_b200_sdf_from_cells_f64_multi(
    const void* cells, int cell_bytes, int64_t nx, int64_t ny, int64_t nz, double resolution,
    int unknown_is_filled, int add_virtual_border, const uint32_t* object_ids,
    int64_t num_object_ids, const int* devices, int num_devices,
    double* sdf_out, double* out_min, double* out_max);

VGT_B200_API int vgt_b200_sdf_per_object_f32_multi(
    const void* cells, int cell_bytes, int64_t nx, int64_t ny, int64_t nz, double resolution,
    int unknown_is_filled, int add_virtual_border, const uint32_t* object_ids,
    int64_t num_object_ids, const int* devices, int num_devices,
    float* sdf_out, float* out_min, float* out_max);

VGT_B200_API int vgt_b200_sdf_per_object_f64_multi(
    const void* cells, int cell_bytes, int64_t nx, int64_t ny, int64_t nz, double resolution,
    int unknown_is_filled, int add_virtual_border, const uint32_t* object_ids,
    int64_t num_object_ids, const int* devices, int num_devices,
    double* sdf_out, double* out_min, double* out_max);

VGT_B200_API int vgt_b200_sdf_free_and_named_f32_multi(
    const void* cells, int cell_bytes, int64_t nx, int64_t ny, int64_t nz, double resolution,
    int unknown_is_filled, int add_virtual_border, const int* devices, int num_devices,
    float* sdf_out, float* out_min, float* out_max);

VGT_B200_API int vgt_b200_sdf_free_and_named_f64_multi(
    const void* cells, int cell_bytes, int64_t nx, int64_t ny, int64_t nz, double resolution,
    int unknown_is_filled, int add_virtual_border, const int* devices, int num_devices,
    double* sdf_out, double* out_min, double* out_max);

/* The three cell entries above on a map that lives on the device; they replace the same reference
 * code (tagged_object_occupancy_map.hpp:199-262, :293-378, occupancy_component_map.hpp:270-306).
 * Each takes the argument list of its host entry, except that
 *   d_cells      device cells (4-byte aligned), the layout of `cells` above
 *   d_sdf_out    device T[nx*ny*nz] (T[num_object_ids][nx*ny*nz] for the batch)
 *   d_min_max    device T[2] (T[num_object_ids][2] for the batch) or NULL
 *   stream       a cudaStream_t; the call is asynchronous and stream-ordered on it, its scratch
 *                comes from the device's stream-ordered pool
 * object_ids stays a host array; it has been read when the call returns. Every argument is checked
 * before the first device call, as in the host entries; the batch also refuses num_object_ids *
 * nx*ny*nz * sizeof(T) bytes beyond int64.
 * vgt_b200_sdf_from_cells_*_dev classifies the cells into a 1-byte mask, as the host entry does.
 * vgt_b200_sdf_per_object_*_dev classifies them once per group of 255 distinct ids into a 1-byte
 * slot map (1 + the id's position in the group; 0 = not filled or another group), and each SDF of
 * the group runs on "slot == its id's slot": the cells are read ceil(distinct ids / 255) times,
 * not once per object. Repeated ids and ids absent from the map are allowed; num_object_ids == 0
 * launches nothing. */
VGT_B200_API int vgt_b200_sdf_from_cells_f32_dev(
    const void* d_cells, int cell_bytes, int64_t nx, int64_t ny, int64_t nz, double resolution,
    int unknown_is_filled, int add_virtual_border, const uint32_t* object_ids,
    int64_t num_object_ids, int device, float* d_sdf_out, float* d_min_max, void* stream);

VGT_B200_API int vgt_b200_sdf_from_cells_f64_dev(
    const void* d_cells, int cell_bytes, int64_t nx, int64_t ny, int64_t nz, double resolution,
    int unknown_is_filled, int add_virtual_border, const uint32_t* object_ids,
    int64_t num_object_ids, int device, double* d_sdf_out, double* d_min_max, void* stream);

VGT_B200_API int vgt_b200_sdf_per_object_f32_dev(
    const void* d_cells, int cell_bytes, int64_t nx, int64_t ny, int64_t nz, double resolution,
    int unknown_is_filled, int add_virtual_border, const uint32_t* object_ids,
    int64_t num_object_ids, int device, float* d_sdf_out, float* d_min_max, void* stream);

VGT_B200_API int vgt_b200_sdf_per_object_f64_dev(
    const void* d_cells, int cell_bytes, int64_t nx, int64_t ny, int64_t nz, double resolution,
    int unknown_is_filled, int add_virtual_border, const uint32_t* object_ids,
    int64_t num_object_ids, int device, double* d_sdf_out, double* d_min_max, void* stream);

VGT_B200_API int vgt_b200_sdf_free_and_named_f32_dev(
    const void* d_cells, int cell_bytes, int64_t nx, int64_t ny, int64_t nz, double resolution,
    int unknown_is_filled, int add_virtual_border, int device, float* d_sdf_out, float* d_min_max,
    void* stream);

VGT_B200_API int vgt_b200_sdf_free_and_named_f64_dev(
    const void* d_cells, int cell_bytes, int64_t nx, int64_t ny, int64_t nz, double resolution,
    int unknown_is_filled, int add_virtual_border, int device, double* d_sdf_out,
    double* d_min_max, void* stream);

/* Replaces internal::ComputeDistanceFieldTransformInPlace(DegreeOfParallelism, VoxelGrid<double>&)
 * (include/.../signed_distance_field_generation.hpp:34-37, src/.../signed_distance_field_generation.cpp:258-391):
 * the in-place 3-D squared distance transform D(p) = min over q of f(q) + |p - q|^2 (voxel
 * units) of an arbitrary sampled function, passes along X, Y, Z, axes of one voxel skipped.
 *   field   host double[nx*ny*nz], GetMutableRawData().data() of the EDTDistanceField; on return
 *           it holds the transform. Samples must be +inf ("no site") or non-negative integers --
 *           what every caller in the reference stores (0 / +inf marks, sdfgen.hpp:47-74) and what
 *           keeps the transform exact; anything else, or values whose transform could pass 2^29,
 *           fails with VGT_B200_ERR_UNSUPPORTED and leaves the field untouched.
 * The reference's DegreeOfParallelism argument has no device meaning and is not passed. */
VGT_B200_API int vgt_b200_edt_transform_inplace_f64(
    double* field, int64_t nx, int64_t ny, int64_t nz, int device);

/* Parity hook for internal::ComputeDistanceFieldTransformInPlace on the two 0/inf fields
 * (include/.../signed_distance_field_generation.hpp:34-37, 47-80): both squared fields in voxel
 * units as int32, VGT_B200_SQ_INF where the reference holds +inf. Host pointers. */
VGT_B200_API int vgt_b200_edt_sq_i32(
    const float* occupancy, int64_t nx, int64_t ny, int64_t nz, int unknown_is_filled, int device,
    int32_t* dist_to_filled_sq, int32_t* dist_to_free_sq);

/* Device-resident variants of the entry points above (no host copies, asynchronous on `stream`);
 * they replace the same reference code (include/.../occupancy_map.hpp:174-210,
 * include/.../signed_distance_field_generation.hpp:39-113, :115-285).
 *   d_occupancy   device float[nx*ny*nz]
 *   d_sdf_out     device float[nx*ny*nz]; also used as the first intermediate of the integer
 *                 passes (a second, 4 bytes per voxel, comes from the device's stream-ordered pool)
 *   d_min_max     device float[2] (min, max) or NULL; written by the last kernel on `stream`
 */
VGT_B200_API int vgt_b200_sdf_f32_dev(
    const float* d_occupancy, int64_t nx, int64_t ny, int64_t nz, double resolution,
    int unknown_is_filled, int add_virtual_border, int device, float* d_sdf_out, float* d_min_max,
    void* stream);

/* Measurement aid for bench.py / profiles: the same three kernels as vgt_b200_sdf_f32_dev with
 * CUDA events between them on `stream`. Synchronises the stream. out_pass_ms[5] receives the
 * duration of the z scan, the y envelope pass and the x envelope pass + finalize (each pass =
 * pilot probe + decision + window kernel + stack kernel over the hand-over list), then the
 * duration of the y pass's and of the x pass's main window-kernel launch alone (0 when that
 * kernel did not run). */
VGT_B200_API int vgt_b200_sdf_f32_dev_profile(
    const float* d_occupancy, int64_t nx, int64_t ny, int64_t nz, double resolution,
    int unknown_is_filled, int add_virtual_border, int device, float* d_sdf_out, float* d_min_max,
    void* stream, float* out_pass_ms);

VGT_B200_API int vgt_b200_sdf_f64_dev(
    const float* d_occupancy, int64_t nx, int64_t ny, int64_t nz, double resolution,
    int unknown_is_filled, int add_virtual_border, int device, double* d_sdf_out,
    double* d_min_max, void* stream);

VGT_B200_API int vgt_b200_sdf_from_mask_f32_dev(
    const uint8_t* d_filled_mask, int64_t nx, int64_t ny, int64_t nz, double resolution,
    int add_virtual_border, int device, float* d_sdf_out, float* d_min_max, void* stream);

/* ---- staged passes, for the slab-sharded multi-GPU path (SURVEY.md section 8e) ----
 * The sign-fused intermediate is one int32 per voxel: bit 31 = class (1 = filled), bits 0..30 =
 * partial squared distance to the opposite class (0x7fffffff = none yet).
 *
 * vgt_b200_edt_local_passes_dev: passes along z (contiguous) and y on an x-slab
 *   [nx_local, ny, nz]; both are independent per x, so a slab needs no neighbours.
 *   Replaces the Y and Z loops of ComputeDistanceFieldTransformInPlace (sdfgen.cpp:315-390) for
 *   both fields at once plus the marking loop (sdfgen.hpp:57-74).
 *   send_parts <= 1: d_out has the slab's own layout [nx_local][ny][nz].
 *   send_parts = G > 1: d_out is written in SEND LAYOUT -- y is cut into G near-equal parts (the
 *   first ny % G parts one row longer) and part h is stored as the block [nx_local][rows_h][nz],
 *   blocks back to back: block h is exactly what the all-to-all sends to rank h, so no packing
 *   pass is needed. Returns VGT_B200_ERR_UNSUPPORTED when ny > 1024 (caller packs instead).
 * vgt_b200_edt_final_pass_f32_dev: the pass along x on a y-slab laid out [nx, ny_local, nz]
 *   (after the all-to-all), fused with the sqrt*resolution combine (sdfgen.hpp:85-108) and the
 *   min/max of Lock(). y_offset / ny_total / (x,z are whole) locate the slab inside the full grid
 *   for the virtual border. d_in is DESTROYED (the envelope stacks are built in place in it) and
 *   must not alias d_sdf_out.
 */
VGT_B200_API int vgt_b200_edt_local_passes_dev(
    const float* d_occupancy, int64_t nx_local, int64_t ny, int64_t nz, int unknown_is_filled,
    int send_parts, int device, int32_t* d_out, void* stream);

/* Fused compute + exchange: the same two passes, but the y pass stores part h of every line
 * straight into rank h's receive buffer through peer-mapped device pointers (NVLink stores), so
 * the kernel IS the all-to-all (the reference has no counterpart: SURVEY.md section 2.2). The
 * passes are the Z and Y loops of ComputeDistanceFieldTransformInPlace
 * (src/.../signed_distance_field_generation.cpp:315-390) on this rank's x-slab.
 *   rank, num_ranks       this rank and the number of x-slabs (2..8). Rank g sweeps the parts of
 *                         its lines starting with the part of rank g + 1, so that at any moment
 *                         the ranks store into different peers.
 *   x_offset, nx_total    first x row of this rank's slab inside the full grid, and its x size.
 *   peer_receive_buffers  host array of num_ranks device addresses, entry h = base of rank h's
 *                         receive buffer laid out [nx_total][rows_h][nz] (rows_h = rank h's share
 *                         of ny), mapped into this process (CUDA IPC / symmetric memory);
 *                         entry [own rank] is the local buffer.
 *   receive_capacity_words  size of EVERY receive buffer in 32-bit words; the call fails with
 *                         VGT_B200_ERR_INVALID_ARGUMENT when nx_total * ceil(ny / num_ranks) * nz
 *                         words do not fit (a peer store must never land outside a buffer).
 * The caller synchronises the ranks (a barrier on `stream`) before any rank reads its buffer. */
VGT_B200_API int vgt_b200_edt_local_passes_scatter_dev(
    const float* d_occupancy, int64_t nx_local, int64_t ny, int64_t nz, int unknown_is_filled,
    int num_ranks, int rank, int64_t x_offset, int64_t nx_total,
    const uint64_t* peer_receive_buffers, int64_t receive_capacity_words, int device,
    void* stream);

/* The remaining X pass (signed_distance_field_generation.cpp:276-312) fused with the combine loop
 * and Lock() (signed_distance_field_generation.hpp:85-111) on this rank's y-slab after the
 * exchange. d_in is destroyed. */
VGT_B200_API int vgt_b200_edt_final_pass_f32_dev(
    int32_t* d_in, int64_t nx, int64_t ny_local, int64_t nz, int64_t y_offset,
    int64_t ny_total, double resolution, int add_virtual_border, int device, float* d_sdf_out,
    float* d_min_max, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Signed distance field queries (the consumers right after the path: planners keep the SDF on
 * the device and ask it about many points at once)
 * ------------------------------------------------------------------------------------------- */

/* A device-resident SignedDistanceField<float>: the grid vgt_b200_sdf_f32_dev wrote plus the
 * pose VoxelGridBase keeps (OriginTransform, column-major 4x4 as Eigen's .data() gives it). */
typedef struct vgt_b200_sdf_view
{
  const float* d_sdf; /* device float[nx*ny*nz] */
  int64_t nx;
  int64_t ny;
  int64_t nz;
  double resolution;
  double origin_transform[16];
} vgt_b200_sdf_view;

/* d_valid[i] after a query: */
#define VGT_B200_QUERY_NO_VALUE 0 /* the reference returns an empty query / ProjectedPosition */
#define VGT_B200_QUERY_VALUE 1
#define VGT_B200_QUERY_THROWS 2   /* the reference throws std::runtime_error for this point */

/* All four: d_points_xyz = device double[num_points*3], WORLD frame; one thread per point;
 * asynchronous on `stream`; outputs are 0 where d_valid is not VGT_B200_QUERY_VALUE.
 *
 * vgt_b200_sdf_estimate_distance_dev replaces SignedDistanceField::EstimateLocationDistance4d
 *   (include/.../signed_distance_field.hpp:823-838 with the helpers at :259-357): trilinear
 *   interpolation of the half-cell-corrected distances of the 8 surrounding cell centres.
 * vgt_b200_sdf_coarse_gradient_dev replaces GetLocationCoarseGradient4d (:887-900, :903-1025):
 *   central differences of the neighbouring cells, one-sided at the grid faces when
 *   enable_edge_gradients, rotated into the world frame; d_gradients_xyz = double[num_points*3].
 * vgt_b200_sdf_fine_gradient_dev replaces GetLocationFineGradient (:1051-1092, :213-255):
 *   differences of seven distance estimates at +/- |nominal_window_size|.
 * vgt_b200_sdf_project_out_of_collision_dev replaces
 *   ProjectLocationOutOfCollisionToMinimumDistance4d (:1159-1203): gradient steps of at most
 *   resolution * stepsize_multiplier until the estimate exceeds minimum_distance. The
 *   reference's loop is unbounded; a point still in collision after max_steps steps reports
 *   VGT_B200_QUERY_THROWS. */
VGT_B200_API int vgt_b200_sdf_estimate_distance_dev(
    const vgt_b200_sdf_view* sdf, const double* d_points_xyz, int64_t num_points, int device,
    double* d_distances, uint8_t* d_valid, void* stream);

VGT_B200_API int vgt_b200_sdf_coarse_gradient_dev(
    const vgt_b200_sdf_view* sdf, const double* d_points_xyz, int64_t num_points,
    int enable_edge_gradients, int device, double* d_gradients_xyz, uint8_t* d_valid,
    void* stream);

VGT_B200_API int vgt_b200_sdf_fine_gradient_dev(
    const vgt_b200_sdf_view* sdf, const double* d_points_xyz, int64_t num_points,
    double nominal_window_size, int device, double* d_gradients_xyz, uint8_t* d_valid,
    void* stream);

VGT_B200_API int vgt_b200_sdf_project_out_of_collision_dev(
    const vgt_b200_sdf_view* sdf, const double* d_points_xyz, int64_t num_points,
    double minimum_distance, double stepsize_multiplier, int64_t max_steps, int device,
    double* d_projected_xyz, uint8_t* d_valid, void* stream);

/* Replaces SignedDistanceField::ComputeLocalExtremaMap
 * (include/voxelized_geometry_tools/signed_distance_field.hpp:1207-1231 with :360-476, :478-545):
 * for every cell the centre (grid frame) of the cell its gradient walk ends at, +inf when the walk leaves the grid. Walks that run into a loop take the
 * cell where the first walk of that basin (in storage order, as the reference's sequential loop
 * starts them) enters the loop, so the result equals the reference's memoised sequential result.
 *   d_extrema_xyz   device double[nx*ny*nz*3] (VoxelGrid<Eigen::Vector3d> raw data)
 * Grids of fewer than 2^31 cells; uses 32 bytes of stream-ordered scratch per cell. */
VGT_B200_API int vgt_b200_sdf_local_extrema_map_dev(
    const vgt_b200_sdf_view* sdf, int device, double* d_extrema_xyz, void* stream);

/* A device-resident SignedDistanceField<double>: the grid vgt_b200_sdf_f64_dev (or a double
 * ExtractSignedDistanceField entry) wrote, with the same fields as vgt_b200_sdf_view. */
typedef struct vgt_b200_sdf_view_f64
{
  const double* d_sdf; /* device double[nx*ny*nz] */
  int64_t nx;
  int64_t ny;
  int64_t nz;
  double resolution;
  double origin_transform[16];
} vgt_b200_sdf_view_f64;

/* The same five calls on a SignedDistanceField<double>, with the argument lists, outputs,
 * statuses and limits of the float entries above. They replace the ScalarType = double
 * instantiations of the same members (include/.../signed_distance_field.hpp:823-838,
 * :887-1025, :1051-1092, :1159-1203, :1207-1231). A cell is read as a double and never rounded
 * through float; where the reference computes in ScalarType, the interior gradient's difference
 * of two neighbours (:932-943) and the sign test of the extrema walk (:494-534), that arithmetic
 * is double. */
VGT_B200_API int vgt_b200_sdf_estimate_distance_f64_dev(
    const vgt_b200_sdf_view_f64* sdf, const double* d_points_xyz, int64_t num_points, int device,
    double* d_distances, uint8_t* d_valid, void* stream);

VGT_B200_API int vgt_b200_sdf_coarse_gradient_f64_dev(
    const vgt_b200_sdf_view_f64* sdf, const double* d_points_xyz, int64_t num_points,
    int enable_edge_gradients, int device, double* d_gradients_xyz, uint8_t* d_valid,
    void* stream);

VGT_B200_API int vgt_b200_sdf_fine_gradient_f64_dev(
    const vgt_b200_sdf_view_f64* sdf, const double* d_points_xyz, int64_t num_points,
    double nominal_window_size, int device, double* d_gradients_xyz, uint8_t* d_valid,
    void* stream);

VGT_B200_API int vgt_b200_sdf_project_out_of_collision_f64_dev(
    const vgt_b200_sdf_view_f64* sdf, const double* d_points_xyz, int64_t num_points,
    double minimum_distance, double stepsize_multiplier, int64_t max_steps, int device,
    double* d_projected_xyz, uint8_t* d_valid, void* stream);

VGT_B200_API int vgt_b200_sdf_local_extrema_map_f64_dev(
    const vgt_b200_sdf_view_f64* sdf, int device, double* d_extrema_xyz, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Mesh rasterizer (an occupancy producer in front of the SDF path)
 * ------------------------------------------------------------------------------------------- */

/* Replaces mesh_rasterizer::RasterizeMesh (src/voxelized_geometry_tools/mesh_rasterizer.cpp:205-230,
 * per triangle :105-203) for OccupancyMap (cell_bytes 4) and OccupancyComponentMap (cell_bytes 8,
 * the float occupancy first): every cell whose centre is within sqrt(3)/2 voxels of a triangle
 * (the reference's conservative closest-point test, evaluated in its operation order) gets
 * occupancy 1.0; all other cell contents are left as they are.
 *   vertices_xyz    double[num_vertices*3], the frame the map's origin transform maps into
 *   triangles       int32[num_triangles*3] vertex indices
 *   cells           host, nx*ny*nz cells of cell_bytes, x slowest, modified in place
 *   x_wg, x_gw      the map's origin transform and its inverse, 4x4 column-major (Eigen .data())
 *   enforce_contains  a touched cell outside the map is an error (VGT_B200_ERR_NOT_CONTAINED;
 *                   the reference throws at the first one, so the map contents after an error
 *                   are unspecified there and here)
 * A triangle naming a missing vertex gives VGT_B200_ERR_OUT_OF_RANGE. */
VGT_B200_API int vgt_b200_rasterize_mesh_f64(
    const double* vertices_xyz, int64_t num_vertices, const int32_t* triangles,
    int64_t num_triangles, void* cells, int cell_bytes, int64_t nx, int64_t ny, int64_t nz,
    double resolution, const double* x_wg, const double* x_gw, int enforce_contains, int device);

/* The same on device-resident arrays, asynchronous on `stream` (RasterizeMeshImpl,
 * mesh_rasterizer.cpp:205-230). d_flags is one device int the kernel ORs its findings into;
 * read it back after the stream has finished and pass it to vgt_b200_rasterize_status. */
VGT_B200_API int vgt_b200_rasterize_mesh_dev(
    const double* d_vertices_xyz, int64_t num_vertices, const int32_t* d_triangles,
    int64_t num_triangles, void* d_cells, int cell_bytes, int64_t nx, int64_t ny, int64_t nz,
    double resolution, const double* x_wg /* host, 16 */, const double* x_gw /* host, 16 */,
    int enforce_contains, int device, int* d_flags, void* stream);

/* The status (and error text) for a flag word of vgt_b200_rasterize_mesh_dev: the two throw
 * sites of RasterizeTriangleImpl (mesh_rasterizer.cpp:122-125 and :191-196). */
VGT_B200_API int vgt_b200_rasterize_status(int flags);

/* ---------------------------------------------------------------------------------------------
 * Point cloud voxelization
 * ------------------------------------------------------------------------------------------- */

/* One cloud, as the adapter extracts it from a PointCloudWrapper
 * (include/.../pointcloud_voxelization_interface.hpp:94-202). */
typedef struct vgt_b200_cloud
{
  const double* points_xyz; /* num_points * 3 doubles, cloud frame (CopyPointLocationIntoDoublePtr) */
  int64_t num_points;       /* PointCloudWrapper::Size() */
  double x_gc[16];          /* X_GC = X_GW * X_WC, column-major 4x4 (Eigen .data(); cpu_pcv.cpp:176) */
  double max_range;         /* PointCloudWrapper::MaxRange(), may be +inf */
} vgt_b200_cloud;

/* The same for a cloud whose points are float32 (what a sensor_msgs/PointCloud2 carries; the
 * reference's PointCloud2Wrapper widens them per point,
 * include/.../pointcloud_voxelization_ros_interface.hpp:35-97): 12 bytes per point cross the bus
 * and are widened on the device. Counts are identical to the double entry on the same values. */
typedef struct vgt_b200_cloud_f32
{
  const float* points_xyz; /* num_points * 3 floats, cloud frame */
  int64_t num_points;
  double x_gc[16];
  double max_range;
} vgt_b200_cloud_f32;

/* PointCloudVoxelizationFilterOptions (pointcloud_voxelization_interface.hpp:20-92). */
typedef struct vgt_b200_filter_options
{
  double percent_seen_free;         /* (0, 1] */
  int32_t outlier_points_threshold; /* > 0 */
  int32_t num_cameras_seen_free;    /* > 0 */
} vgt_b200_filter_options;

/* Replaces <Backend>PointCloudVoxelizer::DoVoxelizePointClouds
 * (src/.../cpu_pointcloud_voxelization.cpp:133-165 for semantics -- double-precision DDA,
 * src/.../device_pointcloud_voxelization.cpp:65-181 for the call position). Host pointers.
 *   static_occupancy   host float[V], copied to out_occupancy first (pcv_if.hpp:252)
 *   out_occupancy      host float[V]
 *   out_counts         optional host int32[num_clouds][V][2] = {seen_free, seen_filled} per cloud
 *                      (the CpuVoxelizationTrackingCell layout, cpu_pcv.hpp:24-32); NULL to skip
 *   out_seconds        optional double[2] = {raycasting, filtering} (VoxelizerRuntime, pcv_if.hpp:206-229)
 */
VGT_B200_API int vgt_b200_voxelize_f64(
    const float* static_occupancy, int64_t nx, int64_t ny, int64_t nz, double voxel_size,
    const vgt_b200_cloud* clouds, int32_t num_clouds, const vgt_b200_filter_options* filter,
    int device, float* out_occupancy, int32_t* out_counts, double* out_seconds);

/* vgt_b200_voxelize_f64 for float32 clouds (see vgt_b200_cloud_f32): the same replacement of
 * DoVoxelizePointClouds (src/.../cpu_pointcloud_voxelization.cpp:133-165) for clouds that arrive
 * through the reference's PointCloud2 wrapper
 * (include/.../pointcloud_voxelization_ros_interface.hpp:35-97). */
VGT_B200_API int vgt_b200_voxelize_f32(
    const float* static_occupancy, int64_t nx, int64_t ny, int64_t nz, double voxel_size,
    const vgt_b200_cloud_f32* clouds, int32_t num_clouds, const vgt_b200_filter_options* filter,
    int device, float* out_occupancy, int32_t* out_counts, double* out_seconds);

/* Device-resident pieces (asynchronous on `stream`).
 * vgt_b200_raycast_f64_dev accumulates one cloud into d_counts (int32[V][2], caller zeroes it).
 *   Replaces CpuPointCloudVoxelizer::DoRaycastPointCloud (cpu_pcv.cpp:167-206) and, positionally,
 *   DeviceVoxelizationHelperInterface::RaycastPoints (device_voxelization_interface.hpp:149-156).
 * vgt_b200_filter_dev applies the per-camera rule and the combine to d_occupancy in place.
 *   Replaces DoCombineAndFilterGrids (cpu_pcv.cpp:438-497) / FilterTrackingGrids
 *   (device_voxelization_interface.hpp:162-167). d_counts is int32[num_grids][V][2].
 */
VGT_B200_API int vgt_b200_raycast_f64_dev(
    const double* d_points_xyz, int64_t num_points, const double* x_gc /* host, 16 */,
    double max_range, int64_t nx, int64_t ny, int64_t nz, double voxel_size, int device,
    int32_t* d_counts, void* stream);

/* vgt_b200_raycast_f64_dev for device float[num_points*3] points (DoRaycastPointCloud,
 * src/.../cpu_pointcloud_voxelization.cpp:167-206, on widened float32 points). */
VGT_B200_API int vgt_b200_raycast_f32_dev(
    const float* d_points_xyz, int64_t num_points, const double* x_gc /* host, 16 */,
    double max_range, int64_t nx, int64_t ny, int64_t nz, double voxel_size, int device,
    int32_t* d_counts, void* stream);

VGT_B200_API int vgt_b200_filter_dev(
    const int32_t* d_counts, int32_t num_grids, int64_t num_voxels,
    const vgt_b200_filter_options* filter, int device, float* d_occupancy, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Connected components of the component maps (topology)
 * ------------------------------------------------------------------------------------------- */

/* Replaces ComputeConnectedComponents (include/voxelized_geometry_tools/topology_computation.hpp:138-196)
 * as OccupancyComponentMap and TaggedObjectOccupancyComponentMap call it: every cell's component
 * word gets the number of its connected component, counted from 1 over the 6 face neighbours,
 * component k being the one whose smallest linear index is the k-th smallest of all components'
 * smallest indices (the order of the reference's scan). Two face neighbours are connected iff
 *   cell_bytes 8  (OccupancyComponentCell, component = word 1):
 *       (occupancy_a > 0.5) == (occupancy_b > 0.5)
 *   cell_bytes 16 (TaggedObjectOccupancyComponentCell, component = word 2):
 *       the same and object_id_a == object_id_b
 * (so unknown cells, 0.5, and NaN join the free cells). Every other byte of every cell is left as
 * it was. The result does not depend on thread timing.
 *   cells               host, nx*ny*nz cells (GetMutableRawData().data()), modified in place
 *   out_num_components  host; the number of components (the reference's return value)
 * Grids of 2^32 cells or more fail with VGT_B200_ERR_UNSUPPORTED. */
VGT_B200_API int vgt_b200_connected_components(
    void* cells, int cell_bytes, int64_t nx, int64_t ny, int64_t nz, int device,
    uint32_t* out_num_components);

/* The same on device-resident cells (ComputeConnectedComponents,
 * topology_computation.hpp:138-196), asynchronous on `stream`; the count is written to device
 * memory. Scratch comes from the device's stream-ordered pool: 4 bytes per cell plus about
 * 0.25 bytes per cell for the ranks. d_cells must be 4-byte aligned. */
VGT_B200_API int vgt_b200_connected_components_dev(
    void* d_cells, int cell_bytes, int64_t nx, int64_t ny, int64_t nz, int device,
    uint32_t* d_num_components, void* stream);

/* vgt_b200_connected_components (ComputeConnectedComponents, topology_computation.hpp:138-196)
 * on the map cut into num_slabs x-slabs (the cut of vgt_b200_sdf_f32_multi), slab g on
 * devices[g]; a device may be listed more than once, so one device labels a map of 2^32 cells or
 * more when its memory allows. The same bytes and count as vgt_b200_connected_components on every
 * map that entry accepts. Each slab is labelled on its own, the edges across the x-faces between
 * slabs are resolved on every slab's device, and every slab then writes the reference's numbers.
 *   1 <= num_slabs <= 8, num_slabs <= nx; num_slabs == 1 is vgt_b200_connected_components.
 *   Device memory, per slab on its device: the slab's cells + 4 B per cell + about 0.25 B per
 *   cell + about 4.25 B per component local to the slab, and up to 64 B per face edge, at most
 *   (num_slabs - 1) * ny * nz edges.
 * Slabs of 2^32 cells or more fail with VGT_B200_ERR_UNSUPPORTED before any device call, and so
 * does a map of more than 0xFFFFFFFF components, before any cell is written (cells unchanged). */
VGT_B200_API int vgt_b200_connected_components_multi(
    void* cells, int cell_bytes, int64_t nx, int64_t ny, int64_t nz, const int* devices,
    int num_slabs, uint32_t* out_num_components);

/* The phases of vgt_b200_connected_components_multi for one x-slab whose cells are already on
 * its device, one slab per process (DESIGN.md section 8): the caller moves what crosses slabs
 * (collectives) and owns every array that lives from one phase to the next. Every entry is
 * asynchronous on `stream`; values the caller needs on the host are written to device memory.
 * Slab r holds the x-planes [x0_r, x1_r) of the map; its base is x0_r * ny * nz, the global index
 * of its first cell. In order, on every slab:
 *   scan_bytes, local, face_edges (every slab but the first), resolve, count, publish, write.
 * Arguments are checked before any device call: VGT_B200_ERR_INVALID_ARGUMENT for a null
 * pointer, a cell size other than 8 or 16, bad dimensions or ranges (a slab has at least one
 * x-plane), VGT_B200_ERR_UNSUPPORTED for a slab of 2^32 cells or more. */

/* The bytes of scan storage the local and count phases of a slab of nx*ny*nz cells need
 * (ComputeConnectedComponents, topology_computation.hpp:138-196, per slab). */
VGT_B200_API int vgt_b200_components_slab_scan_bytes(
    int64_t nx, int64_t ny, int64_t nz, int device, size_t* out_bytes);

/* Labels the slab as a grid of its own (32-bit local indices; topology_computation.hpp:138-196).
 *   d_parent       uint32[nx*ny*nz]            the local union-find, kept until the write phase
 *   d_mask         uint32[words]               words = (nx*ny*nz + 31) / 32: the local roots
 *   d_word_prefix  uint32[words + 1]           their ranks; K_g, the number of local
 *                                              components, ends in d_word_prefix[words]
 *   d_scan_storage scan_bytes bytes            (vgt_b200_components_slab_scan_bytes)
 *   d_face_roots   uint32[ny*nz] or NULL       the local roots of the slab's last x-plane, for
 *                                              the slab above (NULL on the last slab) */
VGT_B200_API int vgt_b200_components_slab_local(
    void* d_cells, int cell_bytes, int64_t nx, int64_t ny, int64_t nz, int device,
    uint32_t* d_parent, uint32_t* d_mask, uint32_t* d_word_prefix, void* d_scan_storage,
    size_t scan_bytes, uint32_t* d_face_roots, void* stream);

/* The edges of the x-face below the slab (the face neighbours of topology_computation.hpp:138-196
 * that lie in two slabs): d_below_cells (ny*nz cells as stored) and
 * d_below_roots (their local roots, d_face_roots of the local phase there) are the last x-plane
 * of the slab below, whose base is below_base. Writes up to ny*nz edges
 * d_edges[e] = {global root below, global root above} (int64[ny*nz][2]) and their number to
 * *d_edge_count. */
VGT_B200_API int vgt_b200_components_slab_face_edges(
    const void* d_below_cells, const uint32_t* d_below_roots, int64_t below_base, void* d_cells,
    int cell_bytes, int64_t nx, int64_t ny, int64_t nz, int64_t base, int device,
    uint32_t* d_parent, int64_t* d_edges, uint32_t* d_edge_count, void* stream);

/* The edges of all faces of a map of num_cells cells (topology_computation.hpp:138-196), in any order (d_edges may be NULL without
 * edges), sorted and made unique into nodes and joined; every slab that passes the same edges
 * gets the same nodes and compact roots. d_nodes (int64) and d_node_roots (uint32) hold
 * max(1, 2*num_edges) entries; d_node_range[3] = {number of nodes, first node of the slab
 * [base, end), one past its last}. */
VGT_B200_API int vgt_b200_components_resolve(
    const int64_t* d_edges, int64_t num_edges, int64_t num_cells, int64_t base, int64_t end,
    int device, int64_t* d_nodes, uint32_t* d_node_roots, uint32_t* d_node_range, void* stream);

/* The slab's global roots (topology_computation.hpp:138-196): its local components that are not merged into a component whose
 * smallest index lies in a lower slab. num_components = K_g; num_nodes, first_node and
 * num_slab_nodes from d_node_range. d_bits uint32[bit_words], d_bit_prefix uint32[bit_words + 1]
 * with bit_words = (K_g + 31) / 32; count_g ends in d_bit_prefix[bit_words]. */
VGT_B200_API int vgt_b200_components_slab_count(
    int64_t nx, int64_t ny, int64_t nz, int64_t base, int64_t num_components, int device,
    const uint32_t* d_mask, const uint32_t* d_word_prefix, const int64_t* d_nodes,
    const uint32_t* d_node_roots, int64_t num_nodes, int64_t first_node, int64_t num_slab_nodes,
    uint32_t* d_bits, uint32_t* d_bit_prefix, void* d_scan_storage, size_t scan_bytes,
    void* stream);

/* The reference's numbers (topology_computation.hpp:138-196) of the slab's global roots:
 * offset = the sum of count_g over the slabs below (the caller refuses a map whose total is
 * above 0xFFFFFFFF before this phase). Writes d_final_ids (uint32[K_g]) and the ids of the slab's
 * nodes into d_node_ids (uint32[num_nodes], zero-filled by the caller; the slab writes only its
 * own nodes, 0 for those whose compact root is another node). */
VGT_B200_API int vgt_b200_components_slab_publish(
    int64_t nx, int64_t ny, int64_t nz, int64_t base, int64_t num_components, int64_t offset,
    int device, const uint32_t* d_mask, const uint32_t* d_word_prefix, const int64_t* d_nodes,
    int64_t num_nodes, int64_t first_node, int64_t num_slab_nodes, const uint32_t* d_bits,
    const uint32_t* d_bit_prefix, uint32_t* d_final_ids, uint32_t* d_node_ids, void* stream);

/* The component words (topology_computation.hpp:138-196). d_node_ids = the sum over all slabs
 * of their published arrays (each entry is written by one
 * slab only). Every node takes its compact root's id, then the component word of every cell of
 * the slab is written; every other word of every cell stays as it was. */
VGT_B200_API int vgt_b200_components_slab_write(
    void* d_cells, int cell_bytes, int64_t nx, int64_t ny, int64_t nz, int64_t base,
    int64_t num_components, int device, uint32_t* d_parent, const uint32_t* d_mask,
    const uint32_t* d_word_prefix, const int64_t* d_nodes, const uint32_t* d_node_roots,
    int64_t num_nodes, int64_t first_node, int64_t num_slab_nodes, uint32_t* d_node_ids,
    uint32_t* d_final_ids, void* stream);

/* ------------------------------------------------------------------------------------------------
 * On-disk formats (SURVEY.md section 8 f3): the reference's own grid files, so that results
 * computed here round-trip through
 *   SignedDistanceField<T>::SaveToFile / LoadFromFile ("SDFZ" / "SDFR";
 *     include/voxelized_geometry_tools/signed_distance_field.hpp:622-722, members :551-596) and
 *   OccupancyMap::SaveToFile / LoadFromFile ("CMGZ" / "CMGR";
 *     src/voxelized_geometry_tools/occupancy_map.cpp:100-193, members :56-84, cells :23-46).
 * Host functions (no device needed, except _save_dev). The bytes between the magic and the
 * derived members are common_robotics_utilities' VoxelGridBase form, restated in
 * csrc/grid_files.cu (that library is not in the reference tree: parity unpinned at that layer).
 * Errors are VGT_B200_ERR_INVALID_ARGUMENT with the reference's messages ("File does not exist",
 * "File is too small", "File has invalid header [....]").
 * ---------------------------------------------------------------------------------------------- */
enum
{
  VGT_B200_GRID_FILE_SDF_F32 = 0,   /* SignedDistanceField<float>:  float cells  */
  VGT_B200_GRID_FILE_SDF_F64 = 1,   /* SignedDistanceField<double>: double cells */
  VGT_B200_GRID_FILE_OCCUPANCY = 2  /* OccupancyMap: one float per cell          */
};

typedef struct vgt_b200_grid_file_info
{
  int64_t nx, ny, nz;
  double voxel_size[3];               /* must be uniform (sdf.hpp:612-620) */
  double origin_transform[16];         /* 4x4 column-major, rigid */
  double inverse_origin_transform[16]; /* filled by probe / load; save computes it */
  double default_value;
  double oob_value;
  int32_t initialized;
  int32_t locked;                      /* SDF only (sdf.hpp:558-559, 579-592) */
  int64_t frame_length;                /* filled by probe / load */
  int64_t payload_bytes;               /* filled by probe / load: size of the serialized grid */
} vgt_b200_grid_file_info;

/* SaveToFile (sdf.hpp:643-668, occupancy_map.cpp:116-141): cells = host T[nx*ny*nz], x slowest. */
VGT_B200_API int vgt_b200_grid_file_save(
    const char* path, int kind, int compress, const void* cells,
    const vgt_b200_grid_file_info* info, const char* frame);

/* SaveToFile (signed_distance_field.hpp:643-668) for a grid that lives on `device` (copied out
 * on `stream`, which is synchronised). */
VGT_B200_API int vgt_b200_grid_file_save_dev(
    const char* path, int kind, int compress, const void* d_cells,
    const vgt_b200_grid_file_info* info, const char* frame, int device, void* stream);

/* LoadFromFile in two steps (sdf.hpp:670-722, occupancy_map.cpp:143-193): probe fills `info`
 * and the frame name (truncated to frame_capacity - 1 characters), load also copies the cells
 * into the caller's buffer of cell_capacity cells. */
VGT_B200_API int vgt_b200_grid_file_probe(
    const char* path, int kind, vgt_b200_grid_file_info* info, char* frame,
    int64_t frame_capacity);
/* LoadFromFile (signed_distance_field.hpp:670-722, occupancy_map.cpp:143-193), second step. */
VGT_B200_API int vgt_b200_grid_file_load(
    const char* path, int kind, void* cells, int64_t cell_capacity,
    vgt_b200_grid_file_info* info, char* frame, int64_t frame_capacity);

#ifdef __cplusplus
}
#endif

#endif /* VGT_B200_H_ */
