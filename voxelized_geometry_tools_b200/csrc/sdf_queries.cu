// Batched SignedDistanceField queries on a device-resident SDF (sm_100a) and their C-ABI entry
// points: trilinear distance estimate, coarse and fine gradient, projection out of collision.
// One thread per query point; the SDF stays where the generation pass left it.
//
// Replaces, per point, the reference's SignedDistanceField<float> and SignedDistanceField<double>
// members (include/voxelized_geometry_tools/signed_distance_field.hpp):
//   EstimateLocationDistance4d            :823-838, :259-357 (interpolation helpers)
//   GetLocationCoarseGradient4d           :887-900, :903-1025
//   GetLocationFineGradient               :1051-1092, :213-255
//   ProjectLocationOutOfCollisionToMinimumDistance4d :1159-1203
// Every kernel that reads cells is a template on the stored ScalarType; the two instantiations
// differ in two statements only, the interior gradient's subtraction and the sign test of the
// extrema walk, both of which the reference evaluates in ScalarType.
//
// THIS TRANSLATION UNIT IS COMPILED WITH -fmad=false so that every expression below evaluates
// as written (the numpy restatement the tests check against then matches bit for bit).
// What is pinned by the reference's own source and what is not:
//   * the coarse gradient, the axis index selection, the half-cell correction, the fine-gradient
//     window logic and the projection loop are in-tree arithmetic and are mirrored operation by
//     operation (including the ScalarType subtraction of the interior gradient, :932-943, against
//     the double subtraction of the edge gradient, :977-1006);
//   * the trilinear blend itself lives in common_robotics_utilities::math::TrilinearInterpolate,
//     which is not in the reference tree (unvendored, unpinned dependency). It is restated here
//     as: ratio = (q - low) / (high - low) clamped to [0, 1]; Interpolate(a, b, r) =
//     a * (1 - r) + b * r; x first, then y, then z. Another evaluation order changes the last
//     bits only: the tests state 1e-12 relative as the tolerance of that one function against
//     the library ("parity unpinned" for it), bit-exact against the restatement.
#include <cmath>

#include "common.cuh"

namespace vgt_b200
{
namespace queries
{
namespace
{
// T = the SDF's ScalarType (float or double). A cell is read as T and widened to double where
// the reference widens it; it never passes through float when T is double.
template <typename T>
struct SdfView
{
  const T* sdf;
  int64_t nx;
  int64_t ny;
  int64_t nz;
  double resolution;
  double inverse_resolution;
  double x_wg[16];  // OriginTransform, column-major (pose of the grid in the world)
  double x_gw[16];  // its inverse
};

struct Vec3
{
  double x;
  double y;
  double z;
};

// Isometry3d * (p, 1): row r = ((m(r,0)*x + m(r,1)*y) + m(r,2)*z) + m(r,3) -- the fixed order of
// the front ends (grids.compose_rigid).
__device__ __forceinline__ Vec3 TransformPoint(const double* m, const Vec3& p)
{
  return Vec3{((m[0] * p.x + m[4] * p.y) + m[8] * p.z) + m[12],
              ((m[1] * p.x + m[5] * p.y) + m[9] * p.z) + m[13],
              ((m[2] * p.x + m[6] * p.y) + m[10] * p.z) + m[14]};
}

// Isometry3d * (v, 0): the rotation only (the translation column is multiplied by w = 0).
__device__ __forceinline__ Vec3 RotateVector(const double* m, const Vec3& v)
{
  return Vec3{((m[0] * v.x + m[4] * v.y) + m[8] * v.z) + m[12] * 0.0,
              ((m[1] * v.x + m[5] * v.y) + m[9] * v.z) + m[13] * 0.0,
              ((m[2] * v.x + m[6] * v.y) + m[10] * v.z) + m[14] * 0.0};
}

template <typename T>
__device__ __forceinline__ double Stored(const SdfView<T>& v, int64_t x, int64_t y, int64_t z)
{
  return static_cast<double>(v.sdf[(x * v.ny + y) * v.nz + z]);
}

template <typename T>
__device__ __forceinline__ T StoredScalar(const SdfView<T>& v, int64_t x, int64_t y, int64_t z)
{
  return v.sdf[(x * v.ny + y) * v.nz + z];
}

template <typename T>
__device__ __forceinline__ bool InBounds(const SdfView<T>& v, int64_t x, int64_t y, int64_t z)
{
  return x >= 0 && x < v.nx && y >= 0 && y < v.ny && z >= 0 && z < v.nz;
}

// LocationToGridIndex4d: grid-frame location and its cell.
template <typename T>
__device__ __forceinline__ void Locate(const SdfView<T>& v, const Vec3& world, Vec3* grid,
                                       int64_t* x, int64_t* y, int64_t* z)
{
  *grid = TransformPoint(v.x_gw, world);
  *x = static_cast<int64_t>(floor(grid->x * v.inverse_resolution));
  *y = static_cast<int64_t>(floor(grid->y * v.inverse_resolution));
  *z = static_cast<int64_t>(floor(grid->z * v.inverse_resolution));
}

// GetCorrectedCenterDistance (:259-273).
template <typename T>
__device__ __forceinline__ double CorrectedCenterDistance(const SdfView<T>& v, int64_t x, int64_t y,
                                                          int64_t z)
{
  const double nominal = Stored(v, x, y, z);
  const double offset = v.resolution * 0.5;
  return (nominal >= 0.0) ? nominal - offset : nominal + offset;
}

// GetAxisInterpolationIndices (:276-308).
__device__ __forceinline__ void AxisInterpolationIndices(int64_t initial, int64_t size,
                                                         double offset, int64_t* lower,
                                                         int64_t* upper)
{
  *lower = initial;
  *upper = initial;
  if (offset >= 0.0)
  {
    *upper = initial + 1;
    if (*upper >= size)
    {
      *upper = initial;
      *lower = initial - 1;
      if (*lower < 0)
      {
        *lower = initial;
      }
    }
  }
  else
  {
    *lower = initial - 1;
    if (*lower < 0)
    {
      *upper = initial + 1;
      *lower = initial;
      if (*upper >= size)
      {
        *upper = initial;
      }
    }
  }
}

__device__ __forceinline__ double Interpolate(double a, double b, double ratio)
{
  return (a * (1.0 - ratio)) + (b * ratio);
}

__device__ __forceinline__ double AxisRatio(double query, double low, double high)
{
  const double ratio = (query - low) / (high - low);
  return fmin(fmax(ratio, 0.0), 1.0);
}

// EstimateLocationDistance4d (:823-838): false = the location is outside the grid.
template <typename T>
__device__ bool EstimateDistance(const SdfView<T>& v, const Vec3& world, double* distance)
{
  Vec3 q;
  int64_t ix, iy, iz;
  Locate(v, world, &q, &ix, &iy, &iz);
  if (!InBounds(v, ix, iy, iz))
  {
    return false;
  }
  // EstimateDistanceInterpolateFromNeighbors (:311-357)
  const double cx = v.resolution * (static_cast<double>(ix) + 0.5);
  const double cy = v.resolution * (static_cast<double>(iy) + 0.5);
  const double cz = v.resolution * (static_cast<double>(iz) + 0.5);
  int64_t x0, x1, y0, y1, z0, z1;
  AxisInterpolationIndices(ix, v.nx, q.x - cx, &x0, &x1);
  AxisInterpolationIndices(iy, v.ny, q.y - cy, &y0, &y1);
  AxisInterpolationIndices(iz, v.nz, q.z - cz, &z0, &z1);
  const double lx = v.resolution * (static_cast<double>(x0) + 0.5);
  const double ly = v.resolution * (static_cast<double>(y0) + 0.5);
  const double lz = v.resolution * (static_cast<double>(z0) + 0.5);
  const double mmm = CorrectedCenterDistance(v, x0, y0, z0);
  const double mmp = CorrectedCenterDistance(v, x0, y0, z1);
  const double mpm = CorrectedCenterDistance(v, x0, y1, z0);
  const double mpp = CorrectedCenterDistance(v, x0, y1, z1);
  const double pmm = CorrectedCenterDistance(v, x1, y0, z0);
  const double pmp = CorrectedCenterDistance(v, x1, y0, z1);
  const double ppm = CorrectedCenterDistance(v, x1, y1, z0);
  const double ppp = CorrectedCenterDistance(v, x1, y1, z1);
  // TrilinearInterpolate(low corner, low corner + voxel sizes, ..., query) -- see the header
  const double rx = AxisRatio(q.x, lx, lx + v.resolution);
  const double ry = AxisRatio(q.y, ly, ly + v.resolution);
  const double rz = AxisRatio(q.z, lz, lz + v.resolution);
  const double mm = Interpolate(mmm, pmm, rx);
  const double mp = Interpolate(mmp, pmp, rx);
  const double pm = Interpolate(mpm, ppm, rx);
  const double pp = Interpolate(mpp, ppp, rx);
  const double m = Interpolate(mm, pm, ry);
  const double p = Interpolate(mp, pp, ry);
  *distance = Interpolate(m, p, rz);
  return true;
}

// GetGridAlignedIndexCoarseGradient + the rotation into the world frame (:903-1025).
template <typename T>
__device__ bool CoarseGradientAtIndex(const SdfView<T>& v, int64_t x, int64_t y, int64_t z,
                                      bool enable_edge_gradients, Vec3* gradient)
{
  if (!InBounds(v, x, y, z))
  {
    return false;
  }
  Vec3 aligned;
  if (x > 0 && y > 0 && z > 0 && x < v.nx - 1 && y < v.ny - 1 && z < v.nz - 1)
  {
    // (the difference of two ScalarType values is a ScalarType -- a float subtraction for float,
    // a double one for double; then times a double)
    const double inv_twice_resolution = 1.0 / (2.0 * v.resolution);
    aligned.x = static_cast<double>(StoredScalar(v, x + 1, y, z) - StoredScalar(v, x - 1, y, z))
        * inv_twice_resolution;
    aligned.y = static_cast<double>(StoredScalar(v, x, y + 1, z) - StoredScalar(v, x, y - 1, z))
        * inv_twice_resolution;
    aligned.z = static_cast<double>(StoredScalar(v, x, y, z + 1) - StoredScalar(v, x, y, z - 1))
        * inv_twice_resolution;
  }
  else if (enable_edge_gradients)
  {
    const int64_t low_x = max(static_cast<int64_t>(0), x - 1);
    const int64_t high_x = min(v.nx - 1, x + 1);
    const int64_t low_y = max(static_cast<int64_t>(0), y - 1);
    const int64_t high_y = min(v.ny - 1, y + 1);
    const int64_t low_z = max(static_cast<int64_t>(0), z - 1);
    const int64_t high_z = min(v.nz - 1, z + 1);
    const double x_increment = static_cast<double>(high_x - low_x) * v.resolution;
    const double y_increment = static_cast<double>(high_y - low_y) * v.resolution;
    const double z_increment = static_cast<double>(high_z - low_z) * v.resolution;
    aligned = Vec3{0.0, 0.0, 0.0};
    if (x_increment > 0.0)
    {
      aligned.x = (Stored(v, high_x, y, z) - Stored(v, low_x, y, z)) * (1.0 / x_increment);
    }
    if (y_increment > 0.0)
    {
      aligned.y = (Stored(v, x, high_y, z) - Stored(v, x, low_y, z)) * (1.0 / y_increment);
    }
    if (z_increment > 0.0)
    {
      aligned.z = (Stored(v, x, y, high_z) - Stored(v, x, y, low_z)) * (1.0 / z_increment);
    }
  }
  else
  {
    return false;
  }
  *gradient = RotateVector(v.x_wg, aligned);
  return true;
}

template <typename T>
__device__ bool CoarseGradientAtLocation(const SdfView<T>& v, const Vec3& world,
                                         bool enable_edge_gradients, Vec3* gradient)
{
  Vec3 q;
  int64_t ix, iy, iz;
  Locate(v, world, &q, &ix, &iy, &iz);
  return CoarseGradientAtIndex(v, ix, iy, iz, enable_edge_gradients, gradient);
}

// ComputeAxisFineGradient (:213-255): false = the reference throws ("window too large").
__device__ bool AxisFineGradient(bool has_point, double point, bool has_minus, double minus,
                                 bool has_plus, double plus, double query_axis, double minus_axis,
                                 double plus_axis, double* gradient)
{
  if (has_point && has_minus && has_plus)
  {
    *gradient = (plus - minus) / (plus_axis - minus_axis);
    return true;
  }
  if (has_point && has_minus)
  {
    *gradient = (point - minus) / (query_axis - minus_axis);
    return true;
  }
  if (has_point && has_plus)
  {
    *gradient = (plus - point) / (plus_axis - query_axis);
    return true;
  }
  return false;
}

constexpr uint8_t kInvalid = 0;
constexpr uint8_t kValid = 1;
constexpr uint8_t kThrows = 2;   // where the reference throws std::runtime_error

template <typename T>
__global__ void EstimateDistanceKernel(SdfView<T> view, const double* __restrict__ points,
                                       int64_t count, double* __restrict__ distances,
                                       uint8_t* __restrict__ valid)
{
  const int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= count)
  {
    return;
  }
  double distance = 0.0;
  const bool ok =
      EstimateDistance(view, Vec3{points[3 * i], points[3 * i + 1], points[3 * i + 2]}, &distance);
  distances[i] = ok ? distance : 0.0;
  valid[i] = ok ? kValid : kInvalid;
}

template <typename T>
__global__ void CoarseGradientKernel(SdfView<T> view, const double* __restrict__ points,
                                     int64_t count, int enable_edge_gradients,
                                     double* __restrict__ gradients, uint8_t* __restrict__ valid)
{
  const int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= count)
  {
    return;
  }
  Vec3 gradient{0.0, 0.0, 0.0};
  const bool ok = CoarseGradientAtLocation(
      view, Vec3{points[3 * i], points[3 * i + 1], points[3 * i + 2]}, enable_edge_gradients != 0,
      &gradient);
  gradients[3 * i] = ok ? gradient.x : 0.0;
  gradients[3 * i + 1] = ok ? gradient.y : 0.0;
  gradients[3 * i + 2] = ok ? gradient.z : 0.0;
  valid[i] = ok ? kValid : kInvalid;
}

// GetLocationFineGradient (:1051-1092).
template <typename T>
__global__ void FineGradientKernel(SdfView<T> view, const double* __restrict__ points,
                                   int64_t count, double nominal_window_size,
                                   double* __restrict__ gradients, uint8_t* __restrict__ valid)
{
  const int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= count)
  {
    return;
  }
  const double window = fabs(nominal_window_size);
  const Vec3 p{points[3 * i], points[3 * i + 1], points[3 * i + 2]};
  uint8_t status = kInvalid;
  Vec3 gradient{0.0, 0.0, 0.0};
  Vec3 q;
  int64_t ix, iy, iz;
  Locate(view, p, &q, &ix, &iy, &iz);
  if (InBounds(view, ix, iy, iz))   // CheckLocationInBounds
  {
    double d_point = 0.0, d_mx = 0.0, d_px = 0.0, d_my = 0.0, d_py = 0.0, d_mz = 0.0, d_pz = 0.0;
    const bool has_point = EstimateDistance(view, p, &d_point);
    const bool has_mx = EstimateDistance(view, Vec3{p.x - window, p.y, p.z}, &d_mx);
    const bool has_px = EstimateDistance(view, Vec3{p.x + window, p.y, p.z}, &d_px);
    const bool has_my = EstimateDistance(view, Vec3{p.x, p.y - window, p.z}, &d_my);
    const bool has_py = EstimateDistance(view, Vec3{p.x, p.y + window, p.z}, &d_py);
    const bool has_mz = EstimateDistance(view, Vec3{p.x, p.y, p.z - window}, &d_mz);
    const bool has_pz = EstimateDistance(view, Vec3{p.x, p.y, p.z + window}, &d_pz);
    const bool ok_x = AxisFineGradient(has_point, d_point, has_mx, d_mx, has_px, d_px, p.x,
                                       p.x - window, p.x + window, &gradient.x);
    const bool ok_y = AxisFineGradient(has_point, d_point, has_my, d_my, has_py, d_py, p.y,
                                       p.y - window, p.y + window, &gradient.y);
    const bool ok_z = AxisFineGradient(has_point, d_point, has_mz, d_mz, has_pz, d_pz, p.z,
                                       p.z - window, p.z + window, &gradient.z);
    status = (ok_x && ok_y && ok_z) ? kValid : kThrows;
  }
  const bool ok = status == kValid;
  gradients[3 * i] = ok ? gradient.x : 0.0;
  gradients[3 * i + 1] = ok ? gradient.y : 0.0;
  gradients[3 * i + 2] = ok ? gradient.z : 0.0;
  valid[i] = status;
}

// ProjectLocationOutOfCollisionToMinimumDistance4d (:1159-1203). The reference's loop has no
// iteration bound; here a point that is still in collision after max_steps steps reports
// kThrows (never seen with the default multiplier: a step is resolution / 10).
template <typename T>
__global__ void ProjectOutOfCollisionKernel(SdfView<T> view, const double* __restrict__ points,
                                            int64_t count, double minimum_distance,
                                            double stepsize_multiplier, int64_t max_steps,
                                            double* __restrict__ projected,
                                            uint8_t* __restrict__ valid)
{
  const int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= count)
  {
    return;
  }
  Vec3 location{points[3 * i], points[3 * i + 1], points[3 * i + 2]};
  uint8_t status = kValid;
  Vec3 q;
  int64_t ix, iy, iz;
  Locate(view, location, &q, &ix, &iy, &iz);
  if (InBounds(view, ix, iy, iz))
  {
    const double margin_distance =
        minimum_distance + view.resolution * stepsize_multiplier * 1e-3;
    const double max_stepsize = view.resolution * stepsize_multiplier;
    double sdf_distance = 0.0;
    EstimateDistance(view, location, &sdf_distance);
    int64_t steps = 0;
    while (sdf_distance <= minimum_distance)
    {
      Vec3 gradient;
      if (!CoarseGradientAtLocation(view, location, true, &gradient))
      {
        status = kInvalid;   // ran off the grid
        break;
      }
      // Vector4d::norm() with w = 0
      const double norm = sqrt(((gradient.x * gradient.x + gradient.y * gradient.y)
                                + gradient.z * gradient.z) + 0.0 * 0.0);
      if (!(norm > view.resolution * 0.25))
      {
        status = kInvalid;   // gradient too small to be productive
        break;
      }
      const double step_distance = fmin(max_stepsize, margin_distance - sdf_distance);
      // normalized(): v / norm (Eigen leaves the vector as it is only when the norm is 0)
      location.x = location.x + (gradient.x / norm) * step_distance;
      location.y = location.y + (gradient.y / norm) * step_distance;
      location.z = location.z + (gradient.z / norm) * step_distance;
      if (!EstimateDistance(view, location, &sdf_distance))
      {
        // (the reference calls .Value() on an empty query here and throws)
        status = kThrows;
        break;
      }
      if (++steps >= max_steps)
      {
        status = kThrows;
        break;
      }
    }
  }
  const bool ok = status == kValid;
  projected[3 * i] = ok ? location.x : 0.0;
  projected[3 * i + 1] = ok ? location.y : 0.0;
  projected[3 * i + 2] = ok ? location.z : 0.0;
  valid[i] = status;
}

// ------------------------------------------------------------------------------------------------
// ComputeLocalExtremaMap (signed_distance_field.hpp:1207-1231 with :360-476, :478-545): every cell
// follows the coarse gradient (edge gradients on; uphill outside obstacles, downhill inside) one
// of its 26 neighbours at a time until it reaches a cell with an effectively flat gradient (its
// own centre is the extremum), leaves the grid (+inf), or runs into a loop.
//
// The reference walks the cells one after the other in storage order and memoises: a walk stops
// at the first cell that already has a value, and a walk that closes a loop takes the centre of
// the first cell it visits twice. For cells that drain into a flat cell or off the grid the
// result does not depend on that order (every walk ends at the same terminal). For cells that
// drain into a loop it does: the whole basin gets the centre of the cell where the FIRST walk of
// that basin (the one from its smallest cell index, the walks being started in index order)
// enters the loop. The parallel version reproduces exactly that:
//   1. successor of every cell (itself = terminal; a marker = off the grid);
//   2. pointer jumping, ceil(log2 V) + 1 rounds: the cell each cell ends at, and the smallest
//      cell index met on the way (for a cell on a loop: the smallest index of the loop = its id);
//   3. per loop: the smallest cell index of its basin (atomicMin);
//   4. per loop: one thread replays the walk from that cell and finds the entry cell;
//   5. every cell writes the centre of its terminal / its loop's entry cell.
// ------------------------------------------------------------------------------------------------
constexpr uint32_t kOffGrid = 0xffffffffu;

template <typename T>
__global__ void ExtremaSuccessorKernel(SdfView<T> view, uint32_t* __restrict__ successor)
{
  const int64_t cell = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  const int64_t count = view.nx * view.ny * view.nz;
  if (cell >= count)
  {
    return;
  }
  const int64_t z = cell % view.nz;
  const int64_t y = (cell / view.nz) % view.ny;
  const int64_t x = cell / (view.nz * view.ny);
  Vec3 gradient;
  CoarseGradientAtIndex(view, x, y, z, true, &gradient);
  // GradientIsEffectiveFlat (:478-492) and GetNextFromGradient (:494-534)
  const double step = view.resolution * 0.06125;
  uint32_t next = static_cast<uint32_t>(cell);
  const bool flat = fabs(gradient.x) <= step && fabs(gradient.y) <= step && fabs(gradient.z) <= step;
  if (!flat)
  {
    if (StoredScalar(view, x, y, z) < static_cast<T>(0))
    {
      gradient = Vec3{gradient.x * -1.0, gradient.y * -1.0, gradient.z * -1.0};
    }
    int64_t nx = x, ny = y, nz = z;
    if (gradient.x > step) { nx += 1; } else if (gradient.x < -step) { nx -= 1; }
    if (gradient.y > step) { ny += 1; } else if (gradient.y < -step) { ny -= 1; }
    if (gradient.z > step) { nz += 1; } else if (gradient.z < -step) { nz -= 1; }
    next = InBounds(view, nx, ny, nz)
        ? static_cast<uint32_t>((nx * view.ny + ny) * view.nz + nz)
        : kOffGrid;
  }
  successor[cell] = next;
}

// One round of pointer jumping: target' = target[target], lowest' = min(lowest, lowest[target]).
__global__ void ExtremaJumpKernel(const uint32_t* __restrict__ target_in,
                                  const uint32_t* __restrict__ lowest_in, int64_t count,
                                  uint32_t* __restrict__ target_out,
                                  uint32_t* __restrict__ lowest_out)
{
  const int64_t cell = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (cell >= count)
  {
    return;
  }
  const uint32_t target = target_in[cell];
  uint32_t lowest = lowest_in[cell];
  uint32_t next = target;
  if (target != kOffGrid)
  {
    next = target_in[target];
    lowest = min(lowest, lowest_in[target]);
  }
  target_out[cell] = next;
  lowest_out[cell] = lowest;
}

// After the jumps target[c] is a terminal (successor == itself), off the grid, or a cell on a
// loop; for the latter lowest[target[c]] is the loop's id. Smallest basin cell per loop.
__global__ void ExtremaBasinKernel(const uint32_t* __restrict__ successor,
                                   const uint32_t* __restrict__ target,
                                   const uint32_t* __restrict__ lowest, int64_t count,
                                   uint32_t* __restrict__ basin_first)
{
  const int64_t cell = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (cell >= count)
  {
    return;
  }
  const uint32_t end = target[cell];
  if (end != kOffGrid && successor[end] != end)
  {
    atomicMin(basin_first + lowest[end], static_cast<uint32_t>(cell));
  }
}

// One thread per loop (the thread of the basin's smallest cell): replays the reference's walk
// from that cell, stamping the cells it visits, until it steps on a stamped cell: the entry.
__global__ void ExtremaEntryKernel(const uint32_t* __restrict__ successor,
                                   const uint32_t* __restrict__ target,
                                   const uint32_t* __restrict__ lowest,
                                   const uint32_t* __restrict__ basin_first, int64_t count,
                                   uint32_t* __restrict__ stamp, uint32_t* __restrict__ entry)
{
  const int64_t cell = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (cell >= count)
  {
    return;
  }
  const uint32_t end = target[cell];
  if (end == kOffGrid || successor[end] == end)
  {
    return;
  }
  const uint32_t loop = lowest[end];
  if (basin_first[loop] != static_cast<uint32_t>(cell))
  {
    return;
  }
  // (the walks of different loops never share a cell, so the stamps need no loop id)
  uint32_t current = static_cast<uint32_t>(cell);
  stamp[current] = 1u;
  while (true)
  {
    current = successor[current];
    if (stamp[current] != 0u)
    {
      entry[loop] = current;
      return;
    }
    stamp[current] = 1u;
  }
}

template <typename T>
__global__ void ExtremaWriteKernel(SdfView<T> view, const uint32_t* __restrict__ successor,
                                   const uint32_t* __restrict__ target,
                                   const uint32_t* __restrict__ lowest,
                                   const uint32_t* __restrict__ entry,
                                   double* __restrict__ extrema)
{
  const int64_t cell = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  const int64_t count = view.nx * view.ny * view.nz;
  if (cell >= count)
  {
    return;
  }
  uint32_t end = target[cell];
  const double infinity = __longlong_as_double(0x7ff0000000000000LL);
  double ex = infinity, ey = infinity, ez = infinity;
  if (end != kOffGrid)
  {
    if (successor[end] != end)
    {
      end = entry[lowest[end]];
    }
    const int64_t z = end % view.nz;
    const int64_t y = (end / view.nz) % view.ny;
    const int64_t x = end / (view.nz * view.ny);
    // GridIndexToLocationInGridFrame
    ex = view.resolution * (static_cast<double>(x) + 0.5);
    ey = view.resolution * (static_cast<double>(y) + 0.5);
    ez = view.resolution * (static_cast<double>(z) + 0.5);
  }
  extrema[3 * cell] = ex;
  extrema[3 * cell + 1] = ey;
  extrema[3 * cell + 2] = ez;
}

__global__ void FillWordsKernel(uint32_t* words, int64_t count, uint32_t value, bool iota)
{
  const int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i < count)
  {
    words[i] = iota ? static_cast<uint32_t>(i) : value;
  }
}

// Inverse of a rigid transform in the front ends' fixed order (grids.inverse_rigid).
void InverseRigid(const double* m, double* out)
{
  for (int i = 0; i < 16; i++)
  {
    out[i] = 0.0;
  }
  out[15] = 1.0;
  for (int r = 0; r < 3; r++)
  {
    for (int c = 0; c < 3; c++)
    {
      out[c * 4 + r] = m[r * 4 + c];
    }
  }
  for (int r = 0; r < 3; r++)
  {
    out[12 + r] = -((out[0 * 4 + r] * m[12] + out[1 * 4 + r] * m[13]) + out[2 * 4 + r] * m[14]);
  }
}

// CView = vgt_b200_sdf_view (float) or vgt_b200_sdf_view_f64 (double); its d_sdf must be a
// const T*.
template <typename CView, typename T>
int MakeView(const CView* sdf, SdfView<T>* view)
{
  if (sdf == nullptr || sdf->d_sdf == nullptr)
  {
    return FailInvalid("null SDF view");
  }
  if (!ValidDims(sdf->nx, sdf->ny, sdf->nz))
  {
    return FailInvalid("SDF dimensions out of range");
  }
  if (!(sdf->resolution > 0.0) || !std::isfinite(sdf->resolution))
  {
    return FailInvalid("resolution must be positive and finite");
  }
  view->sdf = sdf->d_sdf;
  view->nx = sdf->nx;
  view->ny = sdf->ny;
  view->nz = sdf->nz;
  view->resolution = sdf->resolution;
  view->inverse_resolution = 1.0 / sdf->resolution;
  for (int i = 0; i < 16; i++)
  {
    view->x_wg[i] = sdf->origin_transform[i];
  }
  InverseRigid(sdf->origin_transform, view->x_gw);
  return VGT_B200_OK;
}

int CheckBatch(const void* points, int64_t count, const void* out, const void* valid)
{
  if (count < 0 || (count > 0 && (points == nullptr || out == nullptr || valid == nullptr)))
  {
    return FailInvalid("null query buffer or negative count");
  }
  if (count > 0x7fffffffLL * 128)
  {
    return FailInvalid("too many query points for one launch");
  }
  return VGT_B200_OK;
}

constexpr int kThreads = 128;
inline unsigned Blocks(int64_t count) { return static_cast<unsigned>((count + kThreads - 1) / kThreads); }

// The bodies of the C-ABI entries, one per query; T is the SDF's ScalarType.
template <typename T, typename CView>
int EstimateDistanceEntry(const CView* sdf, const double* d_points_xyz, int64_t num_points,
                          int device, double* d_distances, uint8_t* d_valid, void* stream)
{
  SdfView<T> view;
  int status = MakeView(sdf, &view);
  if (status == VGT_B200_OK)
  {
    status = CheckBatch(d_points_xyz, num_points, d_distances, d_valid);
  }
  if (status != VGT_B200_OK || num_points == 0)
  {
    return status;
  }
  ScopedDevice scoped(device);
  VGT_CUDA_TRY(scoped.Status(), "cudaSetDevice");
  EstimateDistanceKernel<<<Blocks(num_points), kThreads, 0, static_cast<cudaStream_t>(stream)>>>(
      view, d_points_xyz, num_points, d_distances, d_valid); NoteKernelLaunch();
  VGT_CUDA_TRY(cudaGetLastError(), "EstimateDistanceKernel launch");
  return VGT_B200_OK;
}

template <typename T, typename CView>
int CoarseGradientEntry(const CView* sdf, const double* d_points_xyz, int64_t num_points,
                        int enable_edge_gradients, int device, double* d_gradients_xyz,
                        uint8_t* d_valid, void* stream)
{
  SdfView<T> view;
  int status = MakeView(sdf, &view);
  if (status == VGT_B200_OK)
  {
    status = CheckBatch(d_points_xyz, num_points, d_gradients_xyz, d_valid);
  }
  if (status != VGT_B200_OK || num_points == 0)
  {
    return status;
  }
  ScopedDevice scoped(device);
  VGT_CUDA_TRY(scoped.Status(), "cudaSetDevice");
  CoarseGradientKernel<<<Blocks(num_points), kThreads, 0, static_cast<cudaStream_t>(stream)>>>(
      view, d_points_xyz, num_points, enable_edge_gradients, d_gradients_xyz, d_valid); NoteKernelLaunch();
  VGT_CUDA_TRY(cudaGetLastError(), "CoarseGradientKernel launch");
  return VGT_B200_OK;
}

template <typename T, typename CView>
int FineGradientEntry(const CView* sdf, const double* d_points_xyz, int64_t num_points,
                      double nominal_window_size, int device, double* d_gradients_xyz,
                      uint8_t* d_valid, void* stream)
{
  SdfView<T> view;
  int status = MakeView(sdf, &view);
  if (status == VGT_B200_OK)
  {
    status = CheckBatch(d_points_xyz, num_points, d_gradients_xyz, d_valid);
  }
  if (status != VGT_B200_OK || num_points == 0)
  {
    return status;
  }
  ScopedDevice scoped(device);
  VGT_CUDA_TRY(scoped.Status(), "cudaSetDevice");
  FineGradientKernel<<<Blocks(num_points), kThreads, 0, static_cast<cudaStream_t>(stream)>>>(
      view, d_points_xyz, num_points, nominal_window_size, d_gradients_xyz, d_valid); NoteKernelLaunch();
  VGT_CUDA_TRY(cudaGetLastError(), "FineGradientKernel launch");
  return VGT_B200_OK;
}

template <typename T, typename CView>
int LocalExtremaMapEntry(const CView* sdf, int device, double* d_extrema_xyz, void* stream)
{
  SdfView<T> view;
  const int status = MakeView(sdf, &view);
  if (status != VGT_B200_OK)
  {
    return status;
  }
  if (d_extrema_xyz == nullptr)
  {
    return FailInvalid("null extrema buffer");
  }
  const int64_t count = view.nx * view.ny * view.nz;
  if (count >= 0x7fffffffLL)
  {
    return FailInvalid("grids of 2^31 cells or more are not supported by the extrema map");
  }
  ScopedDevice scoped(device);
  VGT_CUDA_TRY(scoped.Status(), "cudaSetDevice");
  KeepPoolMemory(device);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  StreamScratch<uint32_t> successor, target_a, target_b, lowest_a, lowest_b, basin_first, entry,
      stamp;
  for (StreamScratch<uint32_t>* buffer :
       {&successor, &target_a, &target_b, &lowest_a, &lowest_b, &basin_first, &entry, &stamp})
  {
    VGT_CUDA_TRY(buffer->Allocate(count, s), "extrema map scratch allocation");
  }
  const unsigned blocks = Blocks(count);
  ExtremaSuccessorKernel<<<blocks, kThreads, 0, s>>>(view, successor.get()); NoteKernelLaunch();
  VGT_CUDA_TRY(cudaMemcpyAsync(target_a.get(), successor.get(), sizeof(uint32_t) * count,
                               cudaMemcpyDeviceToDevice, s),
               "copy successors");
  FillWordsKernel<<<blocks, kThreads, 0, s>>>(lowest_a.get(), count, 0u, true); NoteKernelLaunch();
  FillWordsKernel<<<blocks, kThreads, 0, s>>>(basin_first.get(), count, 0xffffffffu, false); NoteKernelLaunch();
  VGT_CUDA_TRY(cudaMemsetAsync(stamp.get(), 0, sizeof(uint32_t) * count, s), "stamp reset");
  uint32_t* target_in = target_a.get();
  uint32_t* target_out = target_b.get();
  uint32_t* lowest_in = lowest_a.get();
  uint32_t* lowest_out = lowest_b.get();
  int rounds = 1;
  while ((int64_t{1} << rounds) < count)
  {
    rounds++;
  }
  for (int round = 0; round <= rounds; round++)
  {
    ExtremaJumpKernel<<<blocks, kThreads, 0, s>>>(target_in, lowest_in, count, target_out,
                                                  lowest_out); NoteKernelLaunch();
    uint32_t* swap = target_in;
    target_in = target_out;
    target_out = swap;
    swap = lowest_in;
    lowest_in = lowest_out;
    lowest_out = swap;
  }
  ExtremaBasinKernel<<<blocks, kThreads, 0, s>>>(successor.get(), target_in, lowest_in, count,
                                                 basin_first.get()); NoteKernelLaunch();
  ExtremaEntryKernel<<<blocks, kThreads, 0, s>>>(successor.get(), target_in, lowest_in,
                                                 basin_first.get(), count, stamp.get(),
                                                 entry.get()); NoteKernelLaunch();
  ExtremaWriteKernel<<<blocks, kThreads, 0, s>>>(view, successor.get(), target_in, lowest_in,
                                                 entry.get(), d_extrema_xyz); NoteKernelLaunch();
  VGT_CUDA_TRY(cudaGetLastError(), "local extrema map kernels");
  return VGT_B200_OK;
}

template <typename T, typename CView>
int ProjectOutOfCollisionEntry(const CView* sdf, const double* d_points_xyz,
                               int64_t num_points, double minimum_distance,
                               double stepsize_multiplier, int64_t max_steps, int device,
                               double* d_projected_xyz, uint8_t* d_valid, void* stream)
{
  SdfView<T> view;
  int status = MakeView(sdf, &view);
  if (status == VGT_B200_OK)
  {
    status = CheckBatch(d_points_xyz, num_points, d_projected_xyz, d_valid);
  }
  if (status == VGT_B200_OK && (!(stepsize_multiplier > 0.0) || max_steps < 1))
  {
    status = FailInvalid("stepsize_multiplier must be positive and max_steps >= 1");
  }
  if (status != VGT_B200_OK || num_points == 0)
  {
    return status;
  }
  ScopedDevice scoped(device);
  VGT_CUDA_TRY(scoped.Status(), "cudaSetDevice");
  ProjectOutOfCollisionKernel<<<Blocks(num_points), kThreads, 0,
                                static_cast<cudaStream_t>(stream)>>>(
      view, d_points_xyz, num_points, minimum_distance, stepsize_multiplier, max_steps,
      d_projected_xyz, d_valid); NoteKernelLaunch();
  VGT_CUDA_TRY(cudaGetLastError(), "ProjectOutOfCollisionKernel launch");
  return VGT_B200_OK;
}
}  // namespace
}  // namespace queries
}  // namespace vgt_b200

using namespace vgt_b200;

extern "C"
{
int vgt_b200_sdf_estimate_distance_dev(
    const vgt_b200_sdf_view* sdf, const double* d_points_xyz, int64_t num_points, int device,
    double* d_distances, uint8_t* d_valid, void* stream)
{
  return queries::EstimateDistanceEntry<float>(sdf, d_points_xyz, num_points, device,
                                               d_distances, d_valid, stream);
}

int vgt_b200_sdf_estimate_distance_f64_dev(
    const vgt_b200_sdf_view_f64* sdf, const double* d_points_xyz, int64_t num_points, int device,
    double* d_distances, uint8_t* d_valid, void* stream)
{
  return queries::EstimateDistanceEntry<double>(sdf, d_points_xyz, num_points, device,
                                                d_distances, d_valid, stream);
}

int vgt_b200_sdf_coarse_gradient_dev(
    const vgt_b200_sdf_view* sdf, const double* d_points_xyz, int64_t num_points,
    int enable_edge_gradients, int device, double* d_gradients_xyz, uint8_t* d_valid, void* stream)
{
  return queries::CoarseGradientEntry<float>(sdf, d_points_xyz, num_points,
                                             enable_edge_gradients, device, d_gradients_xyz,
                                             d_valid, stream);
}

int vgt_b200_sdf_coarse_gradient_f64_dev(
    const vgt_b200_sdf_view_f64* sdf, const double* d_points_xyz, int64_t num_points,
    int enable_edge_gradients, int device, double* d_gradients_xyz, uint8_t* d_valid, void* stream)
{
  return queries::CoarseGradientEntry<double>(sdf, d_points_xyz, num_points,
                                              enable_edge_gradients, device, d_gradients_xyz,
                                              d_valid, stream);
}

int vgt_b200_sdf_fine_gradient_dev(
    const vgt_b200_sdf_view* sdf, const double* d_points_xyz, int64_t num_points,
    double nominal_window_size, int device, double* d_gradients_xyz, uint8_t* d_valid,
    void* stream)
{
  return queries::FineGradientEntry<float>(sdf, d_points_xyz, num_points, nominal_window_size,
                                           device, d_gradients_xyz, d_valid, stream);
}

int vgt_b200_sdf_fine_gradient_f64_dev(
    const vgt_b200_sdf_view_f64* sdf, const double* d_points_xyz, int64_t num_points,
    double nominal_window_size, int device, double* d_gradients_xyz, uint8_t* d_valid,
    void* stream)
{
  return queries::FineGradientEntry<double>(sdf, d_points_xyz, num_points, nominal_window_size,
                                            device, d_gradients_xyz, d_valid, stream);
}

int vgt_b200_sdf_local_extrema_map_dev(
    const vgt_b200_sdf_view* sdf, int device, double* d_extrema_xyz, void* stream)
{
  return queries::LocalExtremaMapEntry<float>(sdf, device, d_extrema_xyz, stream);
}

int vgt_b200_sdf_local_extrema_map_f64_dev(
    const vgt_b200_sdf_view_f64* sdf, int device, double* d_extrema_xyz, void* stream)
{
  return queries::LocalExtremaMapEntry<double>(sdf, device, d_extrema_xyz, stream);
}

int vgt_b200_sdf_project_out_of_collision_dev(
    const vgt_b200_sdf_view* sdf, const double* d_points_xyz, int64_t num_points,
    double minimum_distance, double stepsize_multiplier, int64_t max_steps, int device,
    double* d_projected_xyz, uint8_t* d_valid, void* stream)
{
  return queries::ProjectOutOfCollisionEntry<float>(sdf, d_points_xyz, num_points,
                                                    minimum_distance, stepsize_multiplier,
                                                    max_steps, device, d_projected_xyz, d_valid,
                                                    stream);
}

int vgt_b200_sdf_project_out_of_collision_f64_dev(
    const vgt_b200_sdf_view_f64* sdf, const double* d_points_xyz, int64_t num_points,
    double minimum_distance, double stepsize_multiplier, int64_t max_steps, int device,
    double* d_projected_xyz, uint8_t* d_valid, void* stream)
{
  return queries::ProjectOutOfCollisionEntry<double>(sdf, d_points_xyz, num_points,
                                                     minimum_distance, stepsize_multiplier,
                                                     max_steps, device, d_projected_xyz, d_valid,
                                                     stream);
}
}  // extern "C"
