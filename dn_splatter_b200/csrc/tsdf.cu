// TSDF fusion and mesh extraction on the device: the `gs-mesh o3dtsdf` exporter (reference
// dn_splatter/export_mesh.py:931-1047), i.e. Open3D's legacy ScalableTSDFVolume (Integrate, ExtractTriangleMesh) and
// the cluster filter that follows it.  The numpy statement of the same contract is oracle/mesh_ref.py; built with
// -fmad=false and written in the oracle's operation order, so the two agree bit for bit.
//
// Volume: units of 16^3 voxels; an open-addressing hash (packed 63-bit unit key -> pool slot) with a per-entry stamp of
// the last view that touched it.  Allocation: one thread per stride-4 depth pixel inserts the units of its
// [p - trunc, p + trunc] box and appends each unit to the view's touched list the first time the view sees it.
// Integration: a grid-stride loop of CTAs over the touched list, 256 threads = the 16x16 voxel columns of a unit, each
// walking z as Open3D does.  Extraction: unit keys sorted with cub; a count pass flags the crossed edges each voxel
// owns (+x, +y, +z) and counts triangles per cell; cub scans give vertex ids and triangle offsets; an emit pass writes
// both.  Cluster filter: radix-sorted edge keys, union-find by atomic hooking, cluster sizes, the threshold, and a
// compaction of triangles and vertices.
#include <cub/cub.cuh>

#include "common.cuh"
#include "mc_tables.cuh"

namespace {

constexpr int RES = 16;
constexpr int UNIT_VOXELS = RES * RES * RES;
constexpr int STRIDE = 4;
constexpr int KEY_BIAS = 1 << 20;
constexpr unsigned long long EMPTY = ~0ull;
constexpr int INTEGRATE_CTAS = 2048;

__host__ size_t align256(size_t x) { return (x + 255) & ~size_t(255); }

__device__ __forceinline__ unsigned long long pack_key(int x, int y, int z) {
  return ((unsigned long long)(x + KEY_BIAS) << 42) | ((unsigned long long)(y + KEY_BIAS) << 21) |
         (unsigned long long)(z + KEY_BIAS);
}
__device__ __forceinline__ int key_axis(unsigned long long k, int shift) { return (int)((k >> shift) & 0x1FFFFF) - KEY_BIAS; }

__device__ __forceinline__ uint32_t hash_key(unsigned long long k) {  // splitmix64 finaliser
  k ^= k >> 30;
  k *= 0xbf58476d1ce4e5b9ull;
  k ^= k >> 27;
  k *= 0x94d049bb133111ebull;
  k ^= k >> 31;
  return (uint32_t)k;
}

__device__ __forceinline__ int hash_find(const unsigned long long* __restrict__ keys, const int32_t* __restrict__ vals,
                                         uint32_t mask, unsigned long long key) {
  uint32_t h = hash_key(key) & mask;
  for (uint32_t probe = 0; probe <= mask; ++probe) {
    const unsigned long long k = keys[h];
    if (k == key) return vals[h];
    if (k == EMPTY) return -1;
    h = (h + 1) & mask;
  }
  return -1;
}

// depth as the integration sees it: truncated and masked to 0
__device__ __forceinline__ float view_depth(const DnrTsdfView& v, float depth_trunc, int u, int y) {
  const int i = y * v.width + u;
  float d = v.depth[i];
  if (d > depth_trunc) d = 0.f;
  if (v.mask && !v.mask[i]) d = 0.f;
  return d;
}

__global__ void tsdf_allocate_kernel(DnrTsdfVolume vol, DnrTsdfView view) {
  const int w4 = (view.width + STRIDE - 1) / STRIDE, h4 = (view.height + STRIDE - 1) / STRIDE;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= w4 * h4) return;
  const int u = (i % w4) * STRIDE, v = (i / w4) * STRIDE;
  const float df = view_depth(view, vol.depth_trunc, u, v);
  if (!(df > 0.f)) return;
  const double z = (double)df;
  const double x = ((double)u - (double)view.cx) * z / (double)view.fx;
  const double y = ((double)v - (double)view.cy) * z / (double)view.fy;
  const double* P = view.pose;
  const double unit_len = vol.voxel_size * RES;
  int lo[3], hi[3];
  for (int a = 0; a < 3; ++a) {
    const double p = ((P[4 * a] * x + P[4 * a + 1] * y) + P[4 * a + 2] * z) + P[4 * a + 3];
    const double l = floor((p - vol.sdf_trunc) / unit_len), h = floor((p + vol.sdf_trunc) / unit_len);
    if (!(l >= -(double)KEY_BIAS && h < (double)KEY_BIAS)) {
      atomicAdd((int32_t*)vol.counters + 3, 1);
      return;
    }
    lo[a] = (int)l;
    hi[a] = (int)h;
  }
  unsigned long long* keys = (unsigned long long*)vol.hash_keys;
  int32_t* vals = (int32_t*)vol.hash_vals;
  int32_t* stamp = (int32_t*)vol.hash_stamp;
  int32_t* counters = (int32_t*)vol.counters;
  const uint32_t mask = (uint32_t)vol.hash_size - 1;
  for (int ux = lo[0]; ux <= hi[0]; ++ux)
    for (int uy = lo[1]; uy <= hi[1]; ++uy)
      for (int uz = lo[2]; uz <= hi[2]; ++uz) {
        const unsigned long long key = pack_key(ux, uy, uz);
        uint32_t h = hash_key(key) & mask;
        bool found = false;
        for (uint32_t probe = 0; probe <= mask; ++probe) {
          const unsigned long long prev = atomicCAS((unsigned long long*)keys + h, EMPTY, key);
          if (prev == EMPTY) {
            const int s = atomicAdd(counters, 1);
            vals[h] = s < vol.capacity ? s : -1;
            found = true;
            break;
          }
          if (prev == key) {
            found = true;
            break;
          }
          h = (h + 1) & mask;
        }
        if (!found) {
          atomicExch(counters + 2, 1);
          continue;
        }
        if (atomicExch(stamp + h, view.stamp) != view.stamp) ((int32_t*)vol.touched)[atomicAdd(counters + 1, 1)] = (int32_t)h;
      }
}

__global__ void __launch_bounds__(256) tsdf_integrate_kernel(DnrTsdfVolume vol, DnrTsdfView view) {
  const int n_touched = ((const int32_t*)vol.counters)[1];
  const int lx = threadIdx.x & 15, ly = threadIdx.x >> 4;
  const float fx = view.fx, fy = view.fy, cx = view.cx, cy = view.cy;
  const float vox = (float)vol.voxel_size;
  const float half = vox * 0.5f;
  const float trunc = (float)vol.sdf_trunc;
  const float trunc_inv = 1.0f / trunc;
  const float safe_w = (float)view.width - 0.0001f, safe_h = (float)view.height - 0.0001f;
  const float inv_fx = 1.0f / fx, inv_fy = 1.0f / fy;
  const double unit_len = vol.voxel_size * RES;
  const float* E = view.extrinsic;
  const float step0 = E[2] * vox, step1 = E[6] * vox, step2 = E[10] * vox;
  for (int t = blockIdx.x; t < n_touched; t += gridDim.x) {
    const int h = ((const int32_t*)vol.touched)[t];
    const int slot = ((const int32_t*)vol.hash_vals)[h];
    if (slot < 0) continue;  // the pool overflowed: the host fuses again with a larger one
    const unsigned long long key = ((const unsigned long long*)vol.hash_keys)[h];
    const double ox = (double)key_axis(key, 42) * unit_len, oy = (double)key_axis(key, 21) * unit_len,
                 oz = (double)key_axis(key, 0) * unit_len;
    const float px = (float)((double)(half + vox * (float)lx) + ox);
    const float py = (float)((double)(half + vox * (float)ly) + oy);
    const float pz = (float)((double)half + oz);
    float c0 = ((E[0] * px + E[1] * py) + E[2] * pz) + E[3];
    float c1 = ((E[4] * px + E[5] * py) + E[6] * pz) + E[7];
    float c2 = ((E[8] * px + E[9] * py) + E[10] * pz) + E[11];
    float* base = (float*)vol.voxels + (size_t)slot * 5 * UNIT_VOXELS + lx + RES * ly;
    for (int z = 0; z < RES; ++z, c0 += step0, c1 += step1, c2 += step2) {
      if (!(c2 > 0.f)) continue;
      const float uf = (c0 * fx) / c2 + cx + 0.5f;
      const float vf = (c1 * fy) / c2 + cy + 0.5f;
      if (!(uf >= 0.0001f && uf < safe_w && vf >= 0.0001f && vf < safe_h)) continue;
      const int u = (int)uf, v = (int)vf;
      const float d = view_depth(view, vol.depth_trunc, u, v);
      if (!(d > 0.f)) continue;
      const float xx = ((float)u - cx) * inv_fx, yy = ((float)v - cy) * inv_fy;
      const float sdf = (d - c2) * sqrtf(xx * xx + yy * yy + 1.0f);
      if (!(sdf > -trunc)) continue;
      const float tsdf = fminf(1.0f, sdf * trunc_inv);
      float* p = base + RES * RES * z;
      const float w = p[UNIT_VOXELS];
      const float wn = w + 1.0f;
      p[0] = (p[0] * w + tsdf) / wn;
      const float* rgb = view.rgb + 3 * ((size_t)v * view.width + u);
      for (int ch = 0; ch < 3; ++ch) {
        const float c8 = (float)(int)fminf(fmaxf(rgb[ch] * 255.0f, 0.f), 255.f);
        p[(2 + ch) * UNIT_VOXELS] = (p[(2 + ch) * UNIT_VOXELS] * w + c8) / wn;
      }
      p[UNIT_VOXELS] = wn;
    }
  }
}

// ------------------------------------------------------------------------------------------------ extraction
struct ExtractLayout {
  size_t totals, gather_keys, gather_slots, keys, slots, rank_of_slot, n_gather, flags, vcnt, voff, tcnt, toff, cub_temp, total;
  size_t cub_bytes;
};

ExtractLayout extract_layout(int32_t n) {
  const size_t N = (size_t)n * UNIT_VOXELS;
  ExtractLayout L;
  size_t off = 0;
  L.totals = off; off = align256(off + 4 * sizeof(int64_t));
  L.gather_keys = off; off = align256(off + sizeof(uint64_t) * (size_t)n);
  L.gather_slots = off; off = align256(off + sizeof(int32_t) * (size_t)n);
  L.keys = off; off = align256(off + sizeof(uint64_t) * (size_t)n);
  L.slots = off; off = align256(off + sizeof(int32_t) * (size_t)n);
  L.rank_of_slot = off; off = align256(off + sizeof(int32_t) * (size_t)n);
  L.n_gather = off; off = align256(off + sizeof(int32_t));
  L.flags = off; off = align256(off + sizeof(uint32_t) * N);
  L.vcnt = off; off = align256(off + sizeof(int32_t) * (N + 1));
  L.voff = off; off = align256(off + sizeof(int32_t) * (N + 1));
  L.tcnt = off; off = align256(off + sizeof(int32_t) * (N + 1));
  L.toff = off; off = align256(off + sizeof(int32_t) * (N + 1));
  size_t sort_b = 0, scan_b = 0;
  cub::DeviceRadixSort::SortPairs(nullptr, sort_b, (const uint64_t*)nullptr, (uint64_t*)nullptr, (const int32_t*)nullptr,
                                  (int32_t*)nullptr, n, 0, 63);
  cub::DeviceScan::ExclusiveSum(nullptr, scan_b, (const int32_t*)nullptr, (int32_t*)nullptr, (int)(N + 1));
  L.cub_bytes = sort_b > scan_b ? sort_b : scan_b;
  L.cub_temp = off; off = align256(off + L.cub_bytes);
  L.total = off;
  return L;
}

struct Grid {  // sorted units + hash, as the extraction kernels see them
  const unsigned long long* hkeys;
  const int32_t* hvals;
  uint32_t hmask;
  const unsigned long long* keys;  // [n] sorted
  const int32_t* slots;            // [n] pool slot of each sorted unit
  const int32_t* rank_of_slot;
  const float* voxels;
  int32_t n;
};

// rank of the unit at offset (dx, dy, dz) in {0,1}^3 from unit `rank` (cached per thread), -1 if not allocated
__device__ __forceinline__ int neighbour_rank(const Grid& g, int rank, int nb, int* cache) {
  if (nb == 0) return rank;
  if (cache[nb] != -2) return cache[nb];
  const unsigned long long k = g.keys[rank];
  const unsigned long long key = pack_key(key_axis(k, 42) + (nb & 1), key_axis(k, 21) + ((nb >> 1) & 1), key_axis(k, 0) + (nb >> 2));
  const int s = hash_find(g.hkeys, g.hvals, g.hmask, key);
  return cache[nb] = s < 0 ? -1 : g.rank_of_slot[s];
}

// global voxel id (rank * 4096 + local) of local voxel (x, y, z) in [0, 16]^3 of unit `rank`, -1 if not allocated
__device__ __forceinline__ int voxel_id(const Grid& g, int rank, int x, int y, int z, int* cache) {
  const int nb = (x >> 4) | ((y >> 4) << 1) | ((z >> 4) << 2);
  const int r = neighbour_rank(g, rank, nb, cache);
  return r < 0 ? -1 : r * UNIT_VOXELS + (x & 15) + RES * (y & 15) + RES * RES * (z & 15);
}

__device__ __forceinline__ const float* voxel_ptr(const Grid& g, int id) {
  return g.voxels + (size_t)g.slots[id >> 12] * 5 * UNIT_VOXELS + (id & (UNIT_VOXELS - 1));
}

__global__ void gather_units_kernel(DnrTsdfVolume vol, uint64_t* keys, int32_t* slots, int32_t* count, int32_t n) {
  const int h = blockIdx.x * blockDim.x + threadIdx.x;
  if (h >= vol.hash_size) return;
  const unsigned long long k = ((const unsigned long long*)vol.hash_keys)[h];
  const int s = ((const int32_t*)vol.hash_vals)[h];
  if (k == EMPTY || s < 0) return;
  const int i = atomicAdd(count, 1);
  if (i < n) {
    keys[i] = k;
    slots[i] = s;
  }
}

__global__ void rank_kernel(const int32_t* slots, int32_t n, int32_t* rank_of_slot) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r < n) rank_of_slot[slots[r]] = r;
}

// one thread per cell (its origin voxel): case, triangle count, and the crossed edges flagged on their owner voxels.
// flags bits 0-2: the voxel's +x / +y / +z edge carries a vertex; bits 8-15: the cell's case (valid cells only).
__global__ void __launch_bounds__(256) extract_count_kernel(Grid g, uint32_t* flags, int32_t* tcnt) {
  const int id = blockIdx.x * blockDim.x + threadIdx.x;
  if (id >= g.n * UNIT_VOXELS) return;
  const int rank = id >> 12, loc = id & (UNIT_VOXELS - 1);
  const int x = loc & 15, y = (loc >> 4) & 15, z = loc >> 8;
  int cache[8];
  for (int i = 0; i < 8; ++i) cache[i] = -2;
  int cube = 0;
  bool valid = true;
  for (int i = 0; i < 8 && valid; ++i) {
    const int c = voxel_id(g, rank, x + kMcCorner[i][0], y + kMcCorner[i][1], z + kMcCorner[i][2], cache);
    if (c < 0) {
      valid = false;
      break;
    }
    const float* p = voxel_ptr(g, c);
    if (p[UNIT_VOXELS] == 0.0f) valid = false;
    else if (p[0] < 0.0f) cube |= 1 << i;
  }
  if (!valid || cube == 0 || cube == 255) {
    tcnt[id] = 0;
    return;
  }
  tcnt[id] = kMcTriCount[cube];
  atomicOr(flags + id, (uint32_t)cube << 8);
  const int em = kMcEdgeTable[cube];
  for (int e = 0; e < 12; ++e) {
    if (!((em >> e) & 1)) continue;
    const int o = voxel_id(g, rank, x + kMcEdgeOwner[e][0], y + kMcEdgeOwner[e][1], z + kMcEdgeOwner[e][2], cache);
    atomicOr(flags + o, 1u << kMcEdgeOwner[e][3]);
  }
}

__global__ void popcount_kernel(const uint32_t* flags, int64_t n, int32_t* vcnt) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) vcnt[i] = __popc(flags[i] & 7u);
}

__global__ void totals_kernel(const int32_t* a, int64_t na, const int32_t* b, int64_t nb, int64_t* totals) {
  totals[0] = a[na];
  totals[1] = b[nb];
}

__global__ void __launch_bounds__(256) extract_emit_kernel(Grid g, const uint32_t* flags, const int32_t* voff,
                                                           const int32_t* toff, double voxel, float* vertices,
                                                           float* colors, int32_t* tris) {
  const int id = blockIdx.x * blockDim.x + threadIdx.x;
  if (id >= g.n * UNIT_VOXELS) return;
  const uint32_t f = flags[id];
  if (!f) return;
  const int rank = id >> 12, loc = id & (UNIT_VOXELS - 1);
  const int x = loc & 15, y = (loc >> 4) & 15, z = loc >> 8;
  int cache[8];
  for (int i = 0; i < 8; ++i) cache[i] = -2;
  const unsigned long long k = g.keys[rank];
  const int gx = key_axis(k, 42) * RES + x, gy = key_axis(k, 21) * RES + y, gz = key_axis(k, 0) * RES + z;
  // vertices owned by this voxel
  int vid = voff[id];
  const float* p0 = voxel_ptr(g, id);
  for (int a = 0; a < 3; ++a) {
    if (!((f >> a) & 1)) continue;
    const int n1 = voxel_id(g, rank, x + (a == 0), y + (a == 1), z + (a == 2), cache);
    const float* p1 = voxel_ptr(g, n1);
    const double f0 = fabs((double)p0[0]), f1 = fabs((double)p1[0]);
    double pos[3] = {0.5 * voxel + voxel * (double)gx, 0.5 * voxel + voxel * (double)gy, 0.5 * voxel + voxel * (double)gz};
    pos[a] += f0 * voxel / (f0 + f1);
    for (int c = 0; c < 3; ++c) {
      const double c0 = (double)p0[(2 + c) * UNIT_VOXELS], c1 = (double)p1[(2 + c) * UNIT_VOXELS];
      vertices[3 * (size_t)vid + c] = (float)pos[c];
      colors[3 * (size_t)vid + c] = (float)((c0 * f1 + c1 * f0) / (f0 + f1) / 255.0);
    }
    ++vid;
  }
  // triangles of the cell at this voxel
  const int cube = (f >> 8) & 0xFF;
  if (!cube) return;
  int edge_vid[12];
  const int em = kMcEdgeTable[cube];
  for (int e = 0; e < 12; ++e) {
    if (!((em >> e) & 1)) continue;
    const int o = voxel_id(g, rank, x + kMcEdgeOwner[e][0], y + kMcEdgeOwner[e][1], z + kMcEdgeOwner[e][2], cache);
    edge_vid[e] = voff[o] + __popc(flags[o] & ((1u << kMcEdgeOwner[e][3]) - 1u));
  }
  int32_t* out = tris + 3 * (size_t)toff[id];
  for (int i = 0; kMcTriTable[cube][i] >= 0; i += 3, out += 3) {
    out[0] = edge_vid[kMcTriTable[cube][i]];
    out[1] = edge_vid[kMcTriTable[cube][i + 2]];
    out[2] = edge_vid[kMcTriTable[cube][i + 1]];
  }
}

int check_volume(const DnrTsdfVolume* v) {
  if (!v || !v->hash_keys || !v->hash_vals || !v->hash_stamp || !v->voxels || !v->touched || !v->counters) return DNR_E_NULL;
  if (!(v->voxel_size > 0.0) || !(v->sdf_trunc > 0.0) || !(v->depth_trunc > 0.f) || v->capacity <= 0 || v->hash_size <= 0 ||
      (v->hash_size & (v->hash_size - 1)) || v->hash_size < v->capacity)
    return DNR_E_SIZE;
  return 0;
}

int check_view(const DnrTsdfView* w) {
  if (!w || !w->depth || !w->rgb) return DNR_E_NULL;
  if (w->width <= 0 || w->height <= 0 || w->stamp < 0 || !(w->fx != 0.f) || !(w->fy != 0.f)) return DNR_E_SIZE;
  return 0;
}

Grid make_grid(const DnrTsdfVolume* vol, char* base, const ExtractLayout& L, int32_t n) {
  Grid g;
  g.hkeys = (const unsigned long long*)vol->hash_keys;
  g.hvals = (const int32_t*)vol->hash_vals;
  g.hmask = (uint32_t)vol->hash_size - 1;
  g.keys = (const unsigned long long*)(base + L.keys);
  g.slots = (const int32_t*)(base + L.slots);
  g.rank_of_slot = (const int32_t*)(base + L.rank_of_slot);
  g.voxels = (const float*)vol->voxels;
  g.n = n;
  return g;
}

// ------------------------------------------------------------------------------------------------ cluster filter
struct ClusterLayout {
  size_t totals, ekeys, evals, ekeys_s, evals_s, parent, size, size_sorted, thr, keep, koff, used, uoff, cub_temp, total;
  size_t cub_bytes;
};

ClusterLayout cluster_layout(int32_t T, int32_t V) {
  ClusterLayout L;
  const size_t E = 3 * (size_t)T;
  size_t off = 0;
  L.totals = off; off = align256(off + 4 * sizeof(int64_t));
  L.ekeys = off; off = align256(off + sizeof(uint64_t) * E);
  L.evals = off; off = align256(off + sizeof(int32_t) * E);
  L.ekeys_s = off; off = align256(off + sizeof(uint64_t) * E);
  L.evals_s = off; off = align256(off + sizeof(int32_t) * E);
  L.parent = off; off = align256(off + sizeof(int32_t) * (size_t)T);
  L.size = off; off = align256(off + sizeof(int32_t) * (size_t)T);
  L.size_sorted = off; off = align256(off + sizeof(int32_t) * (size_t)T);
  L.thr = off; off = align256(off + sizeof(int32_t));
  L.keep = off; off = align256(off + sizeof(int32_t) * ((size_t)T + 1));
  L.koff = off; off = align256(off + sizeof(int32_t) * ((size_t)T + 1));
  L.used = off; off = align256(off + sizeof(int32_t) * ((size_t)V + 1));
  L.uoff = off; off = align256(off + sizeof(int32_t) * ((size_t)V + 1));
  size_t a = 0, b = 0, c = 0, d = 0;
  cub::DeviceRadixSort::SortPairs(nullptr, a, (const uint64_t*)nullptr, (uint64_t*)nullptr, (const int32_t*)nullptr,
                                  (int32_t*)nullptr, (int)E, 0, 64);
  cub::DeviceRadixSort::SortKeysDescending(nullptr, b, (const int32_t*)nullptr, (int32_t*)nullptr, T, 0, 32);
  cub::DeviceScan::ExclusiveSum(nullptr, c, (const int32_t*)nullptr, (int32_t*)nullptr, T + 1);
  cub::DeviceScan::ExclusiveSum(nullptr, d, (const int32_t*)nullptr, (int32_t*)nullptr, V + 1);
  L.cub_bytes = std::max(std::max(a, b), std::max(c, d));
  L.cub_temp = off; off = align256(off + L.cub_bytes);
  L.total = off;
  return L;
}

__global__ void edge_keys_kernel(const int32_t* tris, int32_t T, uint64_t* keys, int32_t* vals) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= T) return;
  const uint32_t v[3] = {(uint32_t)tris[3 * t], (uint32_t)tris[3 * t + 1], (uint32_t)tris[3 * t + 2]};
  for (int e = 0; e < 3; ++e) {
    const uint32_t a = v[e], b = v[(e + 1) % 3];
    keys[3 * (size_t)t + e] = ((uint64_t)min(a, b) << 32) | max(a, b);
    vals[3 * (size_t)t + e] = t;
  }
}

__global__ void iota_kernel(int32_t* p, int32_t n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) p[i] = i;
}

__device__ __forceinline__ int find_root(volatile int32_t* parent, int x) {
  while (true) {
    const int px = parent[x];
    if (px == x) return x;
    const int ppx = parent[px];
    if (ppx != px) parent[x] = ppx;  // path halving: ppx is still an ancestor of x
    x = px;
  }
}

// hook the larger root under the smaller one; a lost CAS means the root was hooked meanwhile: retry from there
__global__ void union_kernel(const uint64_t* keys, const int32_t* vals, int64_t E, int32_t* parent) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i == 0 || i >= E || keys[i] != keys[i - 1]) return;
  int a = vals[i - 1], b = vals[i];
  while (true) {
    a = find_root(parent, a);
    b = find_root(parent, b);
    if (a == b) return;
    if (a > b) {
      const int t = a;
      a = b;
      b = t;
    }
    if (atomicCAS(parent + b, b, a) == b) return;
  }
}

__global__ void cluster_size_kernel(int32_t* parent, int32_t T, int32_t* size) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= T) return;
  const int r = find_root(parent, t);
  atomicAdd(size + r, 1);
}

__global__ void threshold_kernel(const int32_t* sorted, int32_t T, int32_t keep_largest, int32_t min_triangles, int32_t* thr) {
  const int kth = keep_largest <= T ? sorted[keep_largest - 1] : 0;
  *thr = max(kth, min_triangles);
}

__global__ void keep_kernel(const int32_t* tris, const int32_t* parent, const int32_t* size, const int32_t* thr, int32_t T,
                            int32_t* keep, int32_t* used) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= T) return;
  const bool k = size[find_root((int32_t*)parent, t)] >= *thr;
  keep[t] = k;
  if (k)
    for (int e = 0; e < 3; ++e) used[tris[3 * t + e]] = 1;
}

__global__ void cluster_emit_kernel(const int32_t* tris, const float* vertices, const float* colors, int32_t T, int32_t V,
                                    const int32_t* koff, const int32_t* uoff, int32_t* out_tris, float* out_vertices,
                                    float* out_colors) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < T && koff[i + 1] != koff[i])
    for (int e = 0; e < 3; ++e) out_tris[3 * (size_t)koff[i] + e] = uoff[tris[3 * i + e]];
  if (i < V && uoff[i + 1] != uoff[i])
    for (int c = 0; c < 3; ++c) {
      out_vertices[3 * (size_t)uoff[i] + c] = vertices[3 * (size_t)i + c];
      out_colors[3 * (size_t)uoff[i] + c] = colors[3 * (size_t)i + c];
    }
}

int blocks(int64_t n, int b = 256) { return (int)((n + b - 1) / b); }

}  // namespace

extern "C" int dnr_tsdf_reset(const DnrTsdfVolume* vol, void* stream) {
  const int rc = check_volume(vol);
  if (rc) return rc;
  cudaStream_t s = (cudaStream_t)stream;
  DNR_CUDA(cudaMemsetAsync(vol->hash_keys, 0xFF, sizeof(uint64_t) * (size_t)vol->hash_size, s));
  DNR_CUDA(cudaMemsetAsync(vol->hash_vals, 0xFF, sizeof(int32_t) * (size_t)vol->hash_size, s));
  DNR_CUDA(cudaMemsetAsync(vol->hash_stamp, 0xFF, sizeof(int32_t) * (size_t)vol->hash_size, s));
  DNR_CUDA(cudaMemsetAsync(vol->voxels, 0, sizeof(float) * 5 * UNIT_VOXELS * (size_t)vol->capacity, s));
  DNR_CUDA(cudaMemsetAsync(vol->counters, 0, 4 * sizeof(int32_t), s));
  return 0;
}

extern "C" int dnr_tsdf_allocate(const DnrTsdfVolume* vol, const DnrTsdfView* view, void* stream) {
  int rc = check_volume(vol);
  if (!rc) rc = check_view(view);
  if (rc) return rc;
  cudaStream_t s = (cudaStream_t)stream;
  DNR_CUDA(cudaMemsetAsync((int32_t*)vol->counters + 1, 0, sizeof(int32_t), s));
  const int64_t n = (int64_t)((view->width + STRIDE - 1) / STRIDE) * ((view->height + STRIDE - 1) / STRIDE);
  tsdf_allocate_kernel<<<blocks(n), 256, 0, s>>>(*vol, *view);
  DNR_CHECK_LAUNCH();
  return 0;
}

extern "C" int dnr_tsdf_integrate(const DnrTsdfVolume* vol, const DnrTsdfView* view, void* stream) {
  int rc = check_volume(vol);
  if (!rc) rc = check_view(view);
  if (rc) return rc;
  const int grid = vol->hash_size < INTEGRATE_CTAS ? vol->hash_size : INTEGRATE_CTAS;
  tsdf_integrate_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(*vol, *view);
  DNR_CHECK_LAUNCH();
  return 0;
}

extern "C" int64_t dnr_tsdf_extract_workspace_bytes(int32_t n_units) {
  if (n_units < 0 || (int64_t)n_units * UNIT_VOXELS >= ((int64_t)1 << 31) - 1) return DNR_E_SIZE;
  return (int64_t)extract_layout(n_units).total;
}

extern "C" int dnr_tsdf_extract_count(const DnrTsdfVolume* vol, int32_t n_units, void* ws, int64_t ws_bytes, void* stream) {
  if (!vol || !ws) return DNR_E_NULL;
  int rc = check_volume(vol);
  if (rc) return rc;
  if (n_units < 0 || n_units > vol->capacity || dnr_tsdf_extract_workspace_bytes(n_units) < 0) return DNR_E_SIZE;
  const ExtractLayout L = extract_layout(n_units);
  if ((int64_t)L.total > ws_bytes) return DNR_E_WORKSPACE;
  cudaStream_t s = (cudaStream_t)stream;
  char* base = (char*)ws;
  const int64_t N = (int64_t)n_units * UNIT_VOXELS;
  DNR_CUDA(cudaMemsetAsync(base + L.totals, 0, 4 * sizeof(int64_t), s));
  if (n_units == 0) return 0;
  DNR_CUDA(cudaMemsetAsync(base + L.n_gather, 0, sizeof(int32_t), s));
  gather_units_kernel<<<blocks(vol->hash_size), 256, 0, s>>>(*vol, (uint64_t*)(base + L.gather_keys),
                                                             (int32_t*)(base + L.gather_slots), (int32_t*)(base + L.n_gather),
                                                             n_units);
  DNR_CHECK_LAUNCH();
  size_t temp = L.cub_bytes;
  DNR_CUDA(cub::DeviceRadixSort::SortPairs(base + L.cub_temp, temp, (const uint64_t*)(base + L.gather_keys),
                                           (uint64_t*)(base + L.keys), (const int32_t*)(base + L.gather_slots),
                                           (int32_t*)(base + L.slots), n_units, 0, 63, s));
  rank_kernel<<<blocks(n_units), 256, 0, s>>>((const int32_t*)(base + L.slots), n_units, (int32_t*)(base + L.rank_of_slot));
  DNR_CHECK_LAUNCH();
  DNR_CUDA(cudaMemsetAsync(base + L.flags, 0, sizeof(uint32_t) * N, s));
  DNR_CUDA(cudaMemsetAsync(base + L.vcnt + sizeof(int32_t) * N, 0, sizeof(int32_t), s));
  DNR_CUDA(cudaMemsetAsync(base + L.tcnt + sizeof(int32_t) * N, 0, sizeof(int32_t), s));
  const Grid g = make_grid(vol, base, L, n_units);
  extract_count_kernel<<<blocks(N), 256, 0, s>>>(g, (uint32_t*)(base + L.flags), (int32_t*)(base + L.tcnt));
  DNR_CHECK_LAUNCH();
  popcount_kernel<<<blocks(N), 256, 0, s>>>((const uint32_t*)(base + L.flags), N, (int32_t*)(base + L.vcnt));
  DNR_CHECK_LAUNCH();
  temp = L.cub_bytes;
  DNR_CUDA(cub::DeviceScan::ExclusiveSum(base + L.cub_temp, temp, (const int32_t*)(base + L.vcnt), (int32_t*)(base + L.voff),
                                         (int)(N + 1), s));
  temp = L.cub_bytes;
  DNR_CUDA(cub::DeviceScan::ExclusiveSum(base + L.cub_temp, temp, (const int32_t*)(base + L.tcnt), (int32_t*)(base + L.toff),
                                         (int)(N + 1), s));
  totals_kernel<<<1, 1, 0, s>>>((const int32_t*)(base + L.voff), N, (const int32_t*)(base + L.toff), N, (int64_t*)(base + L.totals));
  DNR_CHECK_LAUNCH();
  return 0;
}

extern "C" int dnr_tsdf_extract_emit(const DnrTsdfVolume* vol, int32_t n_units, void* ws, int64_t ws_bytes, float* vertices,
                                     float* colors, int32_t* triangles, void* stream) {
  if (!vol || !ws) return DNR_E_NULL;
  int rc = check_volume(vol);
  if (rc) return rc;
  if (n_units < 0 || n_units > vol->capacity || dnr_tsdf_extract_workspace_bytes(n_units) < 0) return DNR_E_SIZE;
  const ExtractLayout L = extract_layout(n_units);
  if ((int64_t)L.total > ws_bytes) return DNR_E_WORKSPACE;
  if (n_units == 0) return 0;
  if (!vertices || !colors || !triangles) return DNR_E_NULL;
  char* base = (char*)ws;
  const int64_t N = (int64_t)n_units * UNIT_VOXELS;
  extract_emit_kernel<<<blocks(N), 256, 0, (cudaStream_t)stream>>>(
      make_grid(vol, base, L, n_units), (const uint32_t*)(base + L.flags), (const int32_t*)(base + L.voff),
      (const int32_t*)(base + L.toff), vol->voxel_size, vertices, colors, triangles);
  DNR_CHECK_LAUNCH();
  return 0;
}

extern "C" int64_t dnr_mesh_cluster_workspace_bytes(int32_t n_triangles, int32_t n_vertices) {
  if (n_triangles < 0 || n_vertices < 0 || (int64_t)n_triangles * 3 >= ((int64_t)1 << 31) - 1) return DNR_E_SIZE;
  return (int64_t)cluster_layout(n_triangles, n_vertices).total;
}

extern "C" int dnr_mesh_cluster_count(const int32_t* triangles, int32_t n_triangles, int32_t n_vertices, int32_t keep_largest,
                                      int32_t min_triangles, void* ws, int64_t ws_bytes, void* stream) {
  if (!ws || (n_triangles > 0 && !triangles)) return DNR_E_NULL;
  if (keep_largest <= 0 || dnr_mesh_cluster_workspace_bytes(n_triangles, n_vertices) < 0) return DNR_E_SIZE;
  const ClusterLayout L = cluster_layout(n_triangles, n_vertices);
  if ((int64_t)L.total > ws_bytes) return DNR_E_WORKSPACE;
  cudaStream_t s = (cudaStream_t)stream;
  char* base = (char*)ws;
  const int32_t T = n_triangles, V = n_vertices;
  const int64_t E = 3 * (int64_t)T;
  DNR_CUDA(cudaMemsetAsync(base + L.totals, 0, 4 * sizeof(int64_t), s));
  if (T == 0) return 0;
  int32_t* parent = (int32_t*)(base + L.parent);
  int32_t* size = (int32_t*)(base + L.size);
  edge_keys_kernel<<<blocks(T), 256, 0, s>>>(triangles, T, (uint64_t*)(base + L.ekeys), (int32_t*)(base + L.evals));
  DNR_CHECK_LAUNCH();
  size_t temp = L.cub_bytes;
  DNR_CUDA(cub::DeviceRadixSort::SortPairs(base + L.cub_temp, temp, (const uint64_t*)(base + L.ekeys),
                                           (uint64_t*)(base + L.ekeys_s), (const int32_t*)(base + L.evals),
                                           (int32_t*)(base + L.evals_s), (int)E, 0, 64, s));
  iota_kernel<<<blocks(T), 256, 0, s>>>(parent, T);
  DNR_CHECK_LAUNCH();
  union_kernel<<<blocks(E), 256, 0, s>>>((const uint64_t*)(base + L.ekeys_s), (const int32_t*)(base + L.evals_s), E, parent);
  DNR_CHECK_LAUNCH();
  DNR_CUDA(cudaMemsetAsync(size, 0, sizeof(int32_t) * (size_t)T, s));
  cluster_size_kernel<<<blocks(T), 256, 0, s>>>(parent, T, size);
  DNR_CHECK_LAUNCH();
  temp = L.cub_bytes;
  DNR_CUDA(cub::DeviceRadixSort::SortKeysDescending(base + L.cub_temp, temp, (const int32_t*)size,
                                                    (int32_t*)(base + L.size_sorted), T, 0, 32, s));
  threshold_kernel<<<1, 1, 0, s>>>((const int32_t*)(base + L.size_sorted), T, keep_largest, min_triangles,
                                   (int32_t*)(base + L.thr));
  DNR_CHECK_LAUNCH();
  DNR_CUDA(cudaMemsetAsync(base + L.keep + sizeof(int32_t) * (size_t)T, 0, sizeof(int32_t), s));
  DNR_CUDA(cudaMemsetAsync(base + L.used, 0, sizeof(int32_t) * ((size_t)V + 1), s));
  keep_kernel<<<blocks(T), 256, 0, s>>>(triangles, parent, size, (const int32_t*)(base + L.thr), T, (int32_t*)(base + L.keep),
                                        (int32_t*)(base + L.used));
  DNR_CHECK_LAUNCH();
  temp = L.cub_bytes;
  DNR_CUDA(cub::DeviceScan::ExclusiveSum(base + L.cub_temp, temp, (const int32_t*)(base + L.keep), (int32_t*)(base + L.koff),
                                         T + 1, s));
  temp = L.cub_bytes;
  DNR_CUDA(cub::DeviceScan::ExclusiveSum(base + L.cub_temp, temp, (const int32_t*)(base + L.used), (int32_t*)(base + L.uoff),
                                         V + 1, s));
  totals_kernel<<<1, 1, 0, s>>>((const int32_t*)(base + L.uoff), V, (const int32_t*)(base + L.koff), T, (int64_t*)(base + L.totals));
  DNR_CHECK_LAUNCH();
  return 0;
}

extern "C" int dnr_mesh_cluster_emit(const int32_t* triangles, const float* vertices, const float* colors, int32_t n_triangles,
                                     int32_t n_vertices, void* ws, int64_t ws_bytes, int32_t* out_triangles,
                                     float* out_vertices, float* out_colors, void* stream) {
  if (!ws || (n_triangles > 0 && (!triangles || !out_triangles)) || (n_vertices > 0 && (!vertices || !colors || !out_vertices || !out_colors)))
    return DNR_E_NULL;
  if (dnr_mesh_cluster_workspace_bytes(n_triangles, n_vertices) < 0) return DNR_E_SIZE;
  const ClusterLayout L = cluster_layout(n_triangles, n_vertices);
  if ((int64_t)L.total > ws_bytes) return DNR_E_WORKSPACE;
  if (n_triangles == 0) return 0;
  char* base = (char*)ws;
  const int32_t n = n_triangles > n_vertices ? n_triangles : n_vertices;
  cluster_emit_kernel<<<blocks(n), 256, 0, (cudaStream_t)stream>>>(
      triangles, vertices, colors, n_triangles, n_vertices, (const int32_t*)(base + L.koff), (const int32_t*)(base + L.uoff),
      out_triangles, out_vertices, out_colors);
  DNR_CHECK_LAUNCH();
  return 0;
}
