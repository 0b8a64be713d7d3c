// C++ host adapter: the reference's SDF generation signatures, bodies marshalled to the B200
// C-ABI (include/vgt_b200.h). Header-only; compiles against the reference's own headers
// (Eigen, common_robotics_utilities, voxelized_geometry_tools/signed_distance_field.hpp).
//
// Same names, argument meaning and error behaviour as
//   include/voxelized_geometry_tools/signed_distance_field_generation.hpp:115-121 (the internal
//   seam every map type's ExtractSignedDistanceField goes through) and
//   include/voxelized_geometry_tools/occupancy_map.hpp:174-216 (the OccupancyMap fast path),
// in namespace voxelized_geometry_tools::signed_distance_field_generation::b200 so it can sit
// next to the CPU implementation while a maintainer switches call sites (INTEGRATION.md).
#pragma once

#include <cstdint>
#include <functional>
#include <stdexcept>
#include <string>
#include <vector>

#include <common_robotics_utilities/voxel_grid.hpp>
#include <voxelized_geometry_tools/signed_distance_field.hpp>
#include <voxelized_geometry_tools/vgt_namespace.hpp>

#include "vgt_b200.h"

namespace voxelized_geometry_tools
{
VGT_NAMESPACE_BEGIN
namespace signed_distance_field_generation
{
namespace b200
{
using common_robotics_utilities::voxel_grid::GridIndex;

// C-ABI status -> the exception type the reference throws for the same condition.
inline void ThrowOnError(const int status)
{
  if (status == VGT_B200_OK)
  {
    return;
  }
  const std::string message = vgt_b200_last_error();
  if (status == VGT_B200_ERR_INVALID_ARGUMENT)
  {
    throw std::invalid_argument(message);
  }
  throw std::runtime_error(message);
}

// Locks a finished SDF. The reference's Lock() re-derives the extrema with a serial
// std::minmax_element over every value (signed_distance_field.hpp:765-787) - at 512^3 that is
// longer than the whole device computation. The device already returns the same pair, so with
// the one-line accessor INTEGRATION.md proposes for SignedDistanceField (install known extrema
// and lock; define VGT_B200_SDF_HAS_LOCK_WITH_KNOWN_EXTREMA when it is there) the scan is
// skipped; without it the adapter calls Lock() like the reference.
template <typename ScalarType>
inline void FinishAndLock(SignedDistanceField<ScalarType>& sdf, const ScalarType minimum,
                          const ScalarType maximum)
{
#ifdef VGT_B200_SDF_HAS_LOCK_WITH_KNOWN_EXTREMA
  sdf.LockWithKnownExtrema(minimum, maximum);
#else
  (void)minimum;
  (void)maximum;
  sdf.Lock();
#endif
}

// Drop-in for internal::ComputeDistanceFieldTransformInPlace(parallelism, distance_field)
// (signed_distance_field_generation.hpp:34-37): the squared distance transform of the sampled
// function in `distance_field`, in place, on the device. `parallelism` is accepted and ignored.
// The device transform is exact integer arithmetic: samples must be +inf or non-negative
// integers (all the reference's callers store 0 / +inf); anything else throws
// std::runtime_error and leaves the field untouched.
template <typename DistanceFieldType, typename ParallelismType>
inline void ComputeDistanceFieldTransformInPlace(
    const ParallelismType& /* parallelism */, DistanceFieldType& distance_field,
    const int device = 0)
{
  static_assert(sizeof(distance_field.GetMutableRawData()[0]) == sizeof(double),
                "EDTDistanceField is a VoxelGrid<double> (sdfgen.hpp:30-32)");
  ThrowOnError(vgt_b200_edt_transform_inplace_f64(
      distance_field.GetMutableRawData().data(), distance_field.NumXVoxels(),
      distance_field.NumYVoxels(), distance_field.NumZVoxels(), device));
}

namespace detail
{
inline int CallMask(const uint8_t* mask, int64_t nx, int64_t ny, int64_t nz, double resolution,
                    bool border, int device, float* out, float* lo, float* hi)
{
  return vgt_b200_sdf_from_mask_f32(mask, nx, ny, nz, resolution, border ? 1 : 0, device, out, lo,
                                    hi);
}
inline int CallMask(const uint8_t* mask, int64_t nx, int64_t ny, int64_t nz, double resolution,
                    bool border, int device, double* out, double* lo, double* hi)
{
  return vgt_b200_sdf_from_mask_f64(mask, nx, ny, nz, resolution, border ? 1 : 0, device, out, lo,
                                    hi);
}
inline int CallOccupancy(const float* occ, int64_t nx, int64_t ny, int64_t nz, double resolution,
                         bool unknown_is_filled, bool border, int device, float* out, float* lo,
                         float* hi)
{
  return vgt_b200_sdf_f32(occ, nx, ny, nz, resolution, unknown_is_filled ? 1 : 0, border ? 1 : 0,
                          device, out, lo, hi);
}
inline int CallOccupancy(const float* occ, int64_t nx, int64_t ny, int64_t nz, double resolution,
                         bool unknown_is_filled, bool border, int device, double* out, double* lo,
                         double* hi)
{
  return vgt_b200_sdf_f64(occ, nx, ny, nz, resolution, unknown_is_filled ? 1 : 0, border ? 1 : 0,
                          device, out, lo, hi);
}
inline int CallOccupancy(const float* occ, int64_t nx, int64_t ny, int64_t nz, double resolution,
                         bool unknown_is_filled, bool border, const std::vector<int>& devices,
                         float* out, float* lo, float* hi)
{
  return vgt_b200_sdf_f32_multi(occ, nx, ny, nz, resolution, unknown_is_filled ? 1 : 0,
                                border ? 1 : 0, devices.data(), static_cast<int>(devices.size()),
                                out, lo, hi);
}
inline int CallOccupancy(const float* occ, int64_t nx, int64_t ny, int64_t nz, double resolution,
                         bool unknown_is_filled, bool border, const std::vector<int>& devices,
                         double* out, double* lo, double* hi)
{
  return vgt_b200_sdf_f64_multi(occ, nx, ny, nz, resolution, unknown_is_filled ? 1 : 0,
                                border ? 1 : 0, devices.data(), static_cast<int>(devices.size()),
                                out, lo, hi);
}
}  // namespace detail

// Drop-in for internal::ExtractSignedDistanceField(grid, is_filled_fn, frame, parameters)
// (signed_distance_field_generation.hpp:115-285). The opaque host predicate is evaluated once per
// voxel into a byte mask (the reference calls it once per voxel too, sdfgen.hpp:57-74); everything
// after that runs on the GPU. parameters.Parallelism() is accepted and ignored.
template <typename T, typename BackingStore, typename SDFScalarType>
inline SignedDistanceField<SDFScalarType> ExtractSignedDistanceField(
    const common_robotics_utilities::voxel_grid::VoxelGridBase<T, BackingStore>& grid,
    const std::function<bool(const GridIndex&)>& is_filled_fn, const std::string& frame,
    const SignedDistanceFieldGenerationParameters<SDFScalarType>& parameters,
    const int device = 0)
{
  if (!grid.HasUniformVoxelSize())
  {
    throw std::invalid_argument("Grid must have uniform resolution");
  }
  const int64_t nx = grid.NumXVoxels();
  const int64_t ny = grid.NumYVoxels();
  const int64_t nz = grid.NumZVoxels();
  std::vector<uint8_t> mask(static_cast<size_t>(nx * ny * nz));
  size_t at = 0;
  for (int64_t x = 0; x < nx; x++)
  {
    for (int64_t y = 0; y < ny; y++)
    {
      for (int64_t z = 0; z < nz; z++)
      {
        mask[at++] = is_filled_fn(GridIndex(x, y, z)) ? 1 : 0;
      }
    }
  }
  SignedDistanceField<SDFScalarType> new_sdf(
      grid.OriginTransform(), frame, grid.ControlSizes(), parameters.OOBValue());
  SDFScalarType minimum = 0;
  SDFScalarType maximum = 0;
  ThrowOnError(detail::CallMask(
      mask.data(), nx, ny, nz, grid.VoxelXSize(), parameters.AddVirtualBorder(), device,
      new_sdf.GetMutableRawData().data(), &minimum, &maximum));
  FinishAndLock(new_sdf, minimum, maximum);
  return new_sdf;
}

// Drop-in for OccupancyMap::ExtractSignedDistanceField<ScalarType> (occupancy_map.hpp:174-210):
// the occupancy floats go to the device as they are and the predicate
// `occ > 0.5 || (unknown_is_filled && occ == 0.5)` is evaluated there.
template <typename OccupancyMapType, typename SDFScalarType>
inline SignedDistanceField<SDFScalarType> ExtractSignedDistanceFieldFromOccupancyMap(
    const OccupancyMapType& map,
    const SignedDistanceFieldGenerationParameters<SDFScalarType>& parameters,
    const int device = 0)
{
  if (!map.HasUniformVoxelSize())
  {
    throw std::invalid_argument("Grid must have uniform resolution");
  }
  static_assert(sizeof(typename std::remove_reference<
                           decltype(map.GetImmutableRawData())>::type::value_type)
                    == sizeof(float),
                "occupancy cells must be one float (occupancy_map.hpp:56-58)");
  const float* occupancy = reinterpret_cast<const float*>(map.GetImmutableRawData().data());
  SignedDistanceField<SDFScalarType> new_sdf(
      map.OriginTransform(), map.Frame(), map.ControlSizes(), parameters.OOBValue());
  SDFScalarType minimum = 0;
  SDFScalarType maximum = 0;
  ThrowOnError(detail::CallOccupancy(
      occupancy, map.NumXVoxels(), map.NumYVoxels(), map.NumZVoxels(), map.VoxelXSize(),
      parameters.UnknownIsFilled(), parameters.AddVirtualBorder(), device,
      new_sdf.GetMutableRawData().data(), &minimum, &maximum));
  FinishAndLock(new_sdf, minimum, maximum);
  return new_sdf;
}
// The same on several devices of the box (vgt_b200_sdf_f32_multi / vgt_b200_sdf_f64_multi:
// x-slabs, one per device, the exchange fused into the y pass as NVLink peer stores).
template <typename OccupancyMapType, typename SDFScalarType>
inline SignedDistanceField<SDFScalarType> ExtractSignedDistanceFieldFromOccupancyMap(
    const OccupancyMapType& map,
    const SignedDistanceFieldGenerationParameters<SDFScalarType>& parameters,
    const std::vector<int>& devices)
{
  if (!map.HasUniformVoxelSize())
  {
    throw std::invalid_argument("Grid must have uniform resolution");
  }
  const float* occupancy = reinterpret_cast<const float*>(map.GetImmutableRawData().data());
  SignedDistanceField<SDFScalarType> new_sdf(
      map.OriginTransform(), map.Frame(), map.ControlSizes(), parameters.OOBValue());
  SDFScalarType minimum = 0;
  SDFScalarType maximum = 0;
  ThrowOnError(detail::CallOccupancy(
      occupancy, map.NumXVoxels(), map.NumYVoxels(), map.NumZVoxels(), map.VoxelXSize(),
      parameters.UnknownIsFilled(), parameters.AddVirtualBorder(), devices,
      new_sdf.GetMutableRawData().data(), &minimum, &maximum));
  FinishAndLock(new_sdf, minimum, maximum);
  return new_sdf;
}
}  // namespace b200
}  // namespace signed_distance_field_generation
VGT_NAMESPACE_END
}  // namespace voxelized_geometry_tools
