// SURVEY §8f rank 4 (first half): Multiresolution IsoSurface Extraction — the reference's only native code
// (code/src/libmise/mise.pyx, a CPU octree in Cython/C++ driven by utils/meshing.py:9-72) — restated for the GPU with
// dense per-level arrays instead of a pointer octree + hash map.  Semantics are those of mise.pyx, round by round:
//   query()  : every grid point that exists and has no value yet                               (mise.pyx:113-136)
//   update() : store the values; mark each LEAF voxel touched by a known point as next-to-positive (value >= threshold)
//              / next-to-negative (value <= threshold); subdivide every leaf with both marks and level < depth into 8,
//              adding the 27 lattice points of the finer level                                  (mise.pyx:96-111,183-273)
//   to_dense(): known values on the (R+1)^3 lattice, NaN elsewhere, forward-filled along x, then y, then z (:138-166)
// The per-item functions below compile for the host too (tests/host/mise_host.cpp), where they are checked against the
// oracle's restatement of mise.pyx (oracle/mise_oracle.py, pinned to a recorded run of the reference's compiled MISE).
#pragma once
#include <math.h>
#include <stdint.h>

#if defined(__CUDACC__)
#define HOLD_HD __host__ __device__ __forceinline__
#else
#ifndef HOLD_HD
#define HOLD_HD inline
#endif
#endif
#if defined(__CUDA_ARCH__)
#define HOLD_ATOMIC_OR(p, v) atomicOr((p), (v))
#else
#define HOLD_ATOMIC_OR(p, v) (*(p) |= (v))
#endif

namespace hold {
namespace mise {

constexpr int kMaxDepth = 6;
enum : uint8_t { kNoPoint = 0, kUnknown = 1, kKnown = 2 };

struct Grid {
  int res0, depth, R, G;             // coarse voxels per axis, levels, finest voxels per axis (res0 << depth), lattice R + 1
  float threshold;
  float* val;                        // [G^3] lattice values
  uint8_t* state;                    // [G^3] kNoPoint / kUnknown / kKnown
  uint8_t* sub[kMaxDepth];           // level L < depth: [(res0 << L)^3] 1 = voxel subdivided (it exists and is not a leaf)
  unsigned int* mark[kMaxDepth];     // level L < depth: bit 0 next-to-positive, bit 1 next-to-negative (leaves only)
};

HOLD_HD size_t pidx(const Grid& g, int x, int y, int z) { return ((size_t)x * g.G + y) * g.G + z; }  // vec_to_idx(loc, R + 1)
HOLD_HD size_t vidx(const Grid& g, int L, int x, int y, int z) {
  const size_t n = (size_t)g.res0 << L;
  return ((size_t)x * n + y) * n + z;
}

// Leaf voxel containing the finest cell (cx, cy, cz): get_voxel_idx (mise.pyx:275-336).  Returns its level.
HOLD_HD int leaf_of_cell(const Grid& g, int cx, int cy, int cz, size_t& v) {
  for (int L = 0;; ++L) {
    const int sh = g.depth - L;
    v = vidx(g, L, cx >> sh, cy >> sh, cz >> sh);
    if (L == g.depth || !g.sub[L][v]) return L;
  }
}

// subdivide_voxels, first loop (mise.pyx:199-223): one KNOWN lattice point marks the <= 8 leaves around it
HOLD_HD void mark_point(const Grid& g, int x, int y, int z) {
  const float value = g.val[pidx(g, x, y, z)];
  unsigned int bits = 0;
  if (value >= g.threshold) bits |= 1u;
  if (value <= g.threshold) bits |= 2u;
  for (int i = -1; i < 1; ++i)
    for (int j = -1; j < 1; ++j)
      for (int k = -1; k < 1; ++k) {
        const int cx = x + i, cy = y + j, cz = z + k;
        if (cx < 0 || cy < 0 || cz < 0 || cx >= g.R || cy >= g.R || cz >= g.R) continue;
        size_t v;
        const int L = leaf_of_cell(g, cx, cy, cz, v);
        if (L < g.depth) HOLD_ATOMIC_OR(&g.mark[L][v], bits);   // leaves at the finest level never subdivide
      }
}

// subdivide_voxels, second half + subdivide_voxel (mise.pyx:225-273) for the level-L voxel (vx, vy, vz):
// a leaf with both marks becomes 8 children; the 27 lattice points of the children are added (unknown if new).
// Returns true if the voxel was subdivided.
HOLD_HD bool subdivide_voxel(const Grid& g, int L, int vx, int vy, int vz) {
  const size_t v = vidx(g, L, vx, vy, vz);
  if (g.sub[L][v]) return false;                                                   // not a leaf
  if (L > 0 && !g.sub[L - 1][vidx(g, L - 1, vx >> 1, vy >> 1, vz >> 1)]) return false;  // does not exist
  if (g.mark[L][v] != 3u) return false;
  g.sub[L][v] = 1;
  const int size = 1 << (g.depth - L), half = size >> 1;
  const int x0 = vx * size, y0 = vy * size, z0 = vz * size;
  for (int i = 0; i < 3; ++i)
    for (int j = 0; j < 3; ++j)
      for (int k = 0; k < 3; ++k) {
        uint8_t* s = g.state + pidx(g, x0 + i * half, y0 + j * half, z0 + k * half);
        if (*s == kNoPoint) *s = kUnknown;   // concurrent writers all store kUnknown
      }
  return true;
}

// to_dense forward fills (mise.pyx:144-166); out holds NaN where no value is known
HOLD_HD void fill_x(const Grid& g, float* out, int j, int k) {
  for (int i = 1; i < g.G; ++i) {
    float* o = out + pidx(g, i, j, k);
    if (isnan(*o)) *o = out[pidx(g, i - 1, j, k)];
  }
}
HOLD_HD void fill_y(const Grid& g, float* out, int i, int k) {
  for (int j = 1; j < g.G; ++j) {
    float* o = out + pidx(g, i, j, k);
    if (isnan(*o)) *o = out[pidx(g, i, j - 1, k)];
  }
}
HOLD_HD void fill_z(const Grid& g, float* out, int i, int j) {
  for (int k = 1; k < g.G; ++k) {
    float* o = out + pidx(g, i, j, k);
    if (isnan(*o)) *o = out[pidx(g, i, j, k - 1)];
  }
}

}  // namespace mise
}  // namespace hold
