"""TEST INFRASTRUCTURE (oracle): pure-Python restatement of the reference's Multiresolution IsoSurface Extraction
(code/src/libmise/mise.pyx, the Cython octree of Occupancy Networks that utils/meshing.py:9-72 drives), kept with the
reference's own data structures: a list of voxels with child links, grid points in insertion order, a hash from lattice index
to grid point.  It is pinned to a run of the reference's compiled module recorded in profiles/r02_bench_aux.jsonl (replayed by
tests/test_cpu_mise.py), and it is independent of the dense-array restatement the CUDA kernels run
(hold_b200/csrc/mise_phases.h), which is held to it bit for bit (tests/test_cpu_mise.py on the host, tests/test_gpu_mise.py on
the GPU).  `MISE` has the interface of the compiled module's class (oracle/build_ref_mise.py builds it from a reference tree),
so either can drive the same loop."""
import numpy as np


class MISE:
    def __init__(self, resolution_0, depth, threshold):
        self.resolution_0, self.depth, self.threshold = int(resolution_0), int(depth), float(threshold)
        self.voxel_size_0 = 1 << self.depth
        self.resolution = self.resolution_0 * self.voxel_size_0
        # voxels (mise.pyx Voxel): location of the lower corner, level, leaf flag, children [2][2][2] flattened
        self._vloc, self._vlevel, self._vleaf, self._vchild = [], [], [], []
        r0, s0 = self.resolution_0, self.voxel_size_0
        for i in range(r0):
            for j in range(r0):
                for k in range(r0):    # index == vec_to_idx((i, j, k), resolution_0)
                    self._add_voxel((i * s0, j * s0, k * s0), 0)
        # grid points (mise.pyx GridPoint) and the hash lattice index -> grid point
        self._ploc, self._pval, self._pknown, self._phash = [], [], [], {}
        for i in range(r0 + 1):
            for j in range(r0 + 1):
                for k in range(r0 + 1):
                    self._add_grid_point((i * s0, j * s0, k * s0))

    def _add_voxel(self, loc, level):
        self._vloc.append(loc)
        self._vlevel.append(level)
        self._vleaf.append(True)
        self._vchild.append(None)

    def _key(self, loc):
        n = self.resolution + 1
        return (loc[0] * n + loc[1]) * n + loc[2]

    def _add_grid_point(self, loc):
        self._phash[self._key(loc)] = len(self._ploc)
        self._ploc.append(loc)
        self._pval.append(0.0)
        self._pknown.append(False)

    def query(self):
        """Every grid point without a value, in insertion order, as int64 [N, 3]."""
        pts = [p for p, known in zip(self._ploc, self._pknown) if not known]
        return np.asarray(pts, np.int64).reshape(-1, 3)

    def update(self, points, values):
        """Store the values of `points`, then subdivide every active voxel."""
        points, values = np.asarray(points), np.asarray(values, np.float64)
        assert points.ndim == 2 and points.shape[1] == 3 and points.shape[0] == values.shape[0]
        for p, v in zip(points.tolist(), values.tolist()):
            idx = self._phash.get(self._key(p))
            if idx is None:
                raise ValueError("Point not in grid!")
            self._pval[idx], self._pknown[idx] = v, True
        self._subdivide_voxels()

    def to_dense(self):
        """Values on the (resolution + 1)^3 lattice, forward-filled along x, then y, then z."""
        G = self.resolution + 1
        out = np.full((G, G, G), np.nan)
        for (x, y, z), v in zip(self._ploc, self._pval):
            out[x, y, z] = v
        for axis in range(3):
            o = np.moveaxis(out, axis, 0)      # a view: the fill runs in place
            for i in range(1, G):
                m = np.isnan(o[i])
                o[i][m] = o[i - 1][m]
        assert not np.isnan(out).any()
        return out

    def _voxel_idx(self, x, y, z):
        """Leaf voxel containing the finest cell whose lower corner is (x, y, z); -1 outside the grid (get_voxel_idx)."""
        R, d = self.resolution, self.depth
        if not (0 <= x < R and 0 <= y < R and 0 <= z < R):
            return -1
        x0, y0, z0 = x >> d, y >> d, z >> d
        idx = (x0 * self.resolution_0 + y0) * self.resolution_0 + z0
        rx, ry, rz = x - (x0 << d), y - (y0 << d), z - (z0 << d)
        size = self.voxel_size_0
        leaf, child = self._vleaf, self._vchild
        while not leaf[idx]:
            size >>= 1
            ox, oy, oz = int(rx >= size), int(ry >= size), int(rz >= size)
            idx = child[idx][(ox * 2 + oy) * 2 + oz]
            rx, ry, rz = rx - ox * size, ry - oy * size, rz - oz * size
        return idx

    def _subdivide_voxels(self):
        n = len(self._vloc)
        pos, neg = [False] * n, [False] * n
        thr = self.threshold
        voxel_idx = self._voxel_idx
        offsets = [(i, j, k) for i in (-1, 0) for j in (-1, 0) for k in (-1, 0)]
        for (x, y, z), v, known in zip(self._ploc, self._pval, self._pknown):
            if not known:
                continue
            is_pos, is_neg = v >= thr, v <= thr
            for i, j, k in offsets:
                idx = voxel_idx(x + i, y + j, z + k)
                if idx == -1:
                    continue
                if is_pos:
                    pos[idx] = True
                if is_neg:
                    neg[idx] = True
        # only the voxels that existed before this update: the ones created here carry no marks yet
        for idx in range(n):
            if self._vleaf[idx] and self._vlevel[idx] != self.depth and pos[idx] and neg[idx]:
                self._subdivide_voxel(idx)

    def _subdivide_voxel(self, idx):
        x0, y0, z0 = self._vloc[idx]
        level = self._vlevel[idx] + 1
        size = 1 << (self.depth - level)
        self._vleaf[idx] = False
        children = []
        for i in range(2):
            for j in range(2):
                for k in range(2):
                    children.append(len(self._vloc))
                    self._add_voxel((x0 + i * size, y0 + j * size, z0 + k * size), level)
        self._vchild[idx] = children
        for i in range(3):
            for j in range(3):
                for k in range(3):
                    loc = (x0 + i * size, y0 + j * size, z0 + k * size)
                    if self._key(loc) not in self._phash:
                        self._add_grid_point(loc)
