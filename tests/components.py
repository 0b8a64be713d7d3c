"""Shared pieces of the connected-component tests: cell arrays, scenes, a numpy model of the
device algorithm (csrc/connected_components.cu) and the scipy labelling renumbered the way the
reference numbers components (by the first cell of each component in storage order)."""
import numpy as np

from voxelized_geometry_tools_b200.grids import (OCCUPANCY_COMPONENT_CELL,
                                                 TAGGED_OBJECT_OCCUPANCY_COMPONENT_CELL)


def make_cells(occupancy, object_id=None, rng=None):
    """Packed cells around an occupancy grid: 8-byte cells without object ids, 16-byte cells with
    them; the component word (and the spatial segment) hold garbage when rng is given."""
    occupancy = np.asarray(occupancy, dtype=np.float32)
    if object_id is None:
        cells = np.zeros(occupancy.shape, dtype=OCCUPANCY_COMPONENT_CELL)
    else:
        cells = np.zeros(occupancy.shape, dtype=TAGGED_OBJECT_OCCUPANCY_COMPONENT_CELL)
        cells["object_id"] = object_id
        if rng is not None:
            cells["spatial_segment"] = rng.integers(0, 2 ** 32, occupancy.shape, dtype=np.uint32)
    cells["occupancy"] = occupancy
    if rng is not None:
        cells["component"] = rng.integers(0, 2 ** 32, occupancy.shape, dtype=np.uint32)
    return cells


def keys(cells):
    """The connection key of every cell: neighbours are connected iff their keys are equal."""
    filled = (cells["occupancy"] > np.float32(0.5)).astype(np.int64)
    if "object_id" in cells.dtype.names:
        return filled + 2 * cells["object_id"].astype(np.int64)
    return filled


def renumber_by_first_occurrence(labels, count=None):
    """Labels (any integers, one per component) -> 1, 2, ... in the order of each component's
    first cell in storage order, and the number of components. With `count` given the labels
    must already be 0 .. count - 1 (no sort needed)."""
    flat = np.ascontiguousarray(labels).reshape(-1)
    if count is None:
        _, dense = np.unique(flat, return_inverse=True)
        dense = dense.reshape(-1)
        count = int(dense.max()) + 1 if dense.size else 0
    else:
        dense = flat
    first = np.empty(count, dtype=np.int64)
    # repeated indices: the last assignment wins, so reversed order leaves the smallest index
    first[dense[::-1]] = np.arange(flat.size - 1, -1, -1, dtype=np.int64)
    order = np.empty(count, dtype=np.int64)
    order[np.argsort(first, kind="stable")] = np.arange(1, count + 1)
    return order[dense].reshape(np.shape(labels)).astype(np.uint32), count


def scipy_components(cells):
    """scipy.ndimage.label (6-connectivity) per key class, renumbered by first occurrence."""
    from scipy import ndimage
    key = keys(cells)
    labels = np.zeros(key.shape, dtype=np.int64)
    offset = 0
    for value in np.unique(key):
        mask = key == value
        labelled, count = ndimage.label(mask)
        labels[mask] = labelled[mask].astype(np.int64) + (offset - 1)
        offset += count
    return renumber_by_first_occurrence(labels, offset)


def model_components(cells, rng, tile=8):
    """The device algorithm, step by step, on the host: parent = start of the z run inside tiles
    of `tile` consecutive cells; unions (the larger root hung under the smaller) with -y, -x and,
    at tile heads, -z, the implied ones skipped, in a shuffled order; flatten; rank of the roots.
    Returns (ids, count)."""
    nx, ny, nz = cells.shape
    key = keys(cells).reshape(-1)
    count = key.size
    index = np.arange(count, dtype=np.int64)
    z = index % nz
    y = (index // nz) % ny
    x = index // (ny * nz)
    parent = np.empty(count, dtype=np.int64)
    for first in range(0, count, tile):
        start = first
        for i in range(first, min(count, first + tile)):
            if i == first or z[i] == 0 or key[i] != key[i - 1]:
                start = i
            parent[i] = start

    def find(i):
        while parent[i] != i:
            parent[i] = parent[parent[i]]
            i = parent[i]
        return i

    edges = []
    for i in range(count):
        same_below = z[i] > 0 and key[i - 1] == key[i]
        if same_below and i % tile == 0:
            edges.append((i, i - 1))
        for stride, coordinate in ((nz, y), (ny * nz, x)):
            if coordinate[i] > 0:
                j = i - stride
                if key[j] == key[i] and not (same_below and key[j - 1] == key[i]):
                    edges.append((i, j))
    for e in rng.permutation(len(edges)):
        a, b = find(edges[e][0]), find(edges[e][1])
        if a != b:
            parent[max(a, b)] = min(a, b)
    roots = np.array([find(i) for i in range(count)], dtype=np.int64)
    assert np.all(roots <= index)
    is_root = roots == index
    rank = np.cumsum(is_root) - 1
    return (rank[roots] + 1).astype(np.uint32).reshape(cells.shape), int(is_root.sum())


# ---- scenes ------------------------------------------------------------------------------------
def checkerboard(shape):
    x, y, z = np.indices(shape)
    return ((x + y + z) % 2).astype(np.float32)


def serpentine(shape):
    """One filled path through every second row of every second x plane, the rows of a plane
    joined at alternating ends and the planes joined at y = z = 0: one filled component whose
    union-find chains are as deep as the grid allows."""
    nx, ny, nz = shape
    occupancy = np.zeros(shape, dtype=np.float32)
    for x in range(0, nx, 2):
        for y in range(0, ny, 2):
            occupancy[x, y, :] = 1.0
            if y + 2 < ny:
                occupancy[x, y + 1, nz - 1 if (y // 2) % 2 == 0 else 0] = 1.0
        if x + 2 < nx:
            occupancy[x + 1, 0, 0] = 1.0
    return occupancy


def nested_shells(shape, thickness=2):
    """Concentric box shells, alternately filled and free, from the outer faces inwards."""
    index = np.indices(shape)
    depth = np.min([np.minimum(i, n - 1 - i) for i, n in zip(index, shape)], axis=0)
    return ((depth // thickness) % 2 == 0).astype(np.float32)


SPECIAL_VALUES = np.array([0.5, np.nan, 0.0, -0.0, np.nextafter(np.float32(0.5), np.float32(1)),
                           np.inf, -np.inf, 1.0, 0.25, 0.75], dtype=np.float32)


def special_values(rng, shape):
    """Occupancies of exactly 0.5, NaN (with assorted payloads), +-0, the float after 0.5,
    +-inf and ordinary values."""
    occupancy = rng.choice(SPECIAL_VALUES, size=shape).astype(np.float32)
    bits = occupancy.view(np.uint32)
    nan = np.isnan(occupancy)
    payload = rng.integers(1, 1 << 22, size=shape, dtype=np.uint32)
    sign = rng.integers(0, 2, size=shape, dtype=np.uint32) << np.uint32(31)
    bits[nan] = (np.uint32(0x7f800000) | payload | sign)[nan]
    return occupancy
