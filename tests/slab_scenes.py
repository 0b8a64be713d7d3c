"""Scenes for the x-slab connected-component tests (the CPU model and the GPU entry): shapes whose
labelling depends on what happens across the x-faces between slabs."""
import numpy as np


def x_serpentine(shape):
    """One filled path along x through every second y row at z = 0, the rows joined at alternating
    x ends: it crosses every x-face once per row, and every slab holds many pieces of it that only
    the other slabs join."""
    nx, ny, nz = shape
    occupancy = np.zeros(shape, dtype=np.float32)
    for y in range(0, ny, 2):
        occupancy[:, y, 0] = 1.0
        if y + 2 < ny:
            occupancy[nx - 1 if (y // 2) % 2 == 0 else 0, y + 1, 0] = 1.0
    return occupancy


def ring_closed_in_slab(shape, closing_x):
    """Two filled arms along x from x = 0, at y = 0 and y = ny - 1 (z = 1), joined only at
    x = closing_x: in every slab below closing_x they are two separate pieces."""
    nx, ny, nz = shape
    z = min(1, nz - 1)
    occupancy = np.zeros(shape, dtype=np.float32)
    occupancy[:closing_x + 1, 0, z] = 1.0
    occupancy[:closing_x + 1, ny - 1, z] = 1.0
    occupancy[closing_x, :, z] = 1.0
    return occupancy


def last_slab_components(shape, first_x):
    """Free space with filled boxes that begin at x = first_x and a filled U opening towards -x
    there: components whose smallest index lies at or above first_x, one of them joined only
    through its own slab."""
    nx, ny, nz = shape
    occupancy = np.zeros(shape, dtype=np.float32)
    occupancy[first_x:, 0:2, 0:2] = 1.0
    occupancy[first_x:, ny - 1, nz - 1] = 1.0
    occupancy[nx - 1, ny // 2, :] = 1.0
    occupancy[first_x:, ny // 2, 0] = 1.0
    occupancy[first_x:, ny // 2, nz - 1] = 1.0
    return occupancy
