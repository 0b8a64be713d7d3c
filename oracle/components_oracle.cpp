// =============================================================================
// TEST INFRASTRUCTURE ONLY -- CPU oracle for the connected components of the
// component maps.
//
// From-scratch restatement of the reference's labelling. Only tests/ may use it;
// the product path never does.
//
// Parity status: RESTATED, NOT PINNED. The reference's own member bodies are not
// compiled into oracle/_ref; the two connection rules below are a reading of
// them and each sits in one function, so that it can be checked and changed in
// one place.
//
// What it follows (path relative to the reference checkout):
//   include/voxelized_geometry_tools/topology_computation.hpp:138-196
//       ComputeConnectedComponents: every component set to 0, then a scan in
//       storage order (x slowest, z fastest); at each cell whose component is
//       still 0 the count is incremented and a breadth-first flood fill marks
//       every cell reached, neighbours in the order -x, +x, -y, +y, -z, +z, a
//       neighbour being added when are_connected_fn(current, neighbour) holds.
//       Returns the count.
// =============================================================================
#include <cstdint>
#include <cstring>
#include <list>
#include <unordered_set>

namespace
{
float Occupancy(const uint32_t* cell)
{
  float occupancy;
  std::memcpy(&occupancy, cell, sizeof(occupancy));
  return occupancy;
}

// OccupancyComponentMap: connected iff both cells are on the same side of 0.5
// (the float promoted to double against the literal, as the reference compares).
bool OccupancyComponentsConnected(const uint32_t* a, const uint32_t* b)
{
  return (static_cast<double>(Occupancy(a)) > 0.5) == (static_cast<double>(Occupancy(b)) > 0.5);
}

// TaggedObjectOccupancyComponentMap: the same, and the same object id.
bool TaggedObjectComponentsConnected(const uint32_t* a, const uint32_t* b)
{
  return (static_cast<double>(Occupancy(a)) > 0.5) == (static_cast<double>(Occupancy(b)) > 0.5)
      && a[1] == b[1];
}

template <typename Connected>
uint32_t ComputeConnectedComponents(uint32_t* cells, int cell_words, int component_word,
                                    int64_t nx, int64_t ny, int64_t nz, Connected are_connected)
{
  const int64_t count = nx * ny * nz;
  const auto cell = [&](int64_t i) { return cells + i * cell_words; };
  for (int64_t i = 0; i < count; i++)
  {
    cell(i)[component_word] = 0u;
  }
  uint32_t components = 0;
  for (int64_t x = 0; x < nx; x++)
  {
    for (int64_t y = 0; y < ny; y++)
    {
      for (int64_t z = 0; z < nz; z++)
      {
        const int64_t start = (x * ny + y) * nz + z;
        if (cell(start)[component_word] != 0u)
        {
          continue;
        }
        components++;
        std::list<int64_t> queue{start};
        std::unordered_set<int64_t> visited{start};
        while (!queue.empty())
        {
          const int64_t current = queue.front();
          queue.pop_front();
          cell(current)[component_word] = components;
          const int64_t cz = current % nz;
          const int64_t cy = (current / nz) % ny;
          const int64_t cx = current / (ny * nz);
          const int64_t neighbours[6][3] = {{cx - 1, cy, cz}, {cx + 1, cy, cz}, {cx, cy - 1, cz},
                                            {cx, cy + 1, cz}, {cx, cy, cz - 1}, {cx, cy, cz + 1}};
          for (const auto& n : neighbours)
          {
            if (n[0] < 0 || n[0] >= nx || n[1] < 0 || n[1] >= ny || n[2] < 0 || n[2] >= nz)
            {
              continue;
            }
            const int64_t neighbour = (n[0] * ny + n[1]) * nz + n[2];
            if (visited.count(neighbour) == 0 && are_connected(cell(current), cell(neighbour)))
            {
              visited.insert(neighbour);
              queue.push_back(neighbour);
            }
          }
        }
      }
    }
  }
  return components;
}
}  // namespace

extern "C"
{
// cells: nx*ny*nz packed cells of cell_bytes (8: {occupancy, component}; 16: {occupancy,
// object_id, component, spatial_segment}), component word rewritten in place.
// Returns 0, or 1 for an unsupported cell size.
int vgt_oracle_connected_components(void* cells, int cell_bytes, int64_t nx, int64_t ny,
                                    int64_t nz, uint32_t* out_num_components)
{
  uint32_t* words = static_cast<uint32_t*>(cells);
  if (cell_bytes == 8)
  {
    *out_num_components = ComputeConnectedComponents(words, 2, 1, nx, ny, nz,
                                                     OccupancyComponentsConnected);
    return 0;
  }
  if (cell_bytes == 16)
  {
    *out_num_components = ComputeConnectedComponents(words, 4, 2, nx, ny, nz,
                                                     TaggedObjectComponentsConnected);
    return 0;
  }
  return 1;
}
}  // extern "C"
