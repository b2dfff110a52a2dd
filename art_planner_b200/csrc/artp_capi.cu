// art_planner_b200/csrc/artp_capi.cu -- C ABI (include/artp.h) over the sm_100a kernels.
// Host side mirrors the reference's checker objects: artp_create ~ StateValidityChecker ctor,
// artp_set_map ~ setMap + updateHeightField (HeightMapBoxChecker::setHeightField,
// art_planner/src/validity_checker/height_map_box_checker.cpp:38-54), artp_check_* ~ isValid / checkMotion.
// No CPU fallback: every entry point fails with ARTP_E_CUDA if the device or the kernel image is unusable.
#include <cuda.h>
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <chrono>
#include <cstring>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/artp.h"
#include "artp_cnn.h"
#include "artp_kernels.cuh"
#include "artp_tiles.cuh"
#include "artp_sampler.cuh"
#include "artp_basic.cuh"
#include "artp_roadmap.cuh"

namespace {

thread_local std::string g_create_error;
constexpr int kCopyEvents = 16;
constexpr int kMaxSlices = 64;   // H2D pipeline slices per round of the host-buffer calls

struct Handle {
  artp_params p;
  int device = 0;
  int sm_count = 0;
  artp::Checker chk;
  float* d_H[2] = {nullptr, nullptr};
  float2* d_T[2][artp::kMaxLevel + 1] = {};
  uint32_t* d_NF[2][artp::kMaxLevel + 1] = {};   // bit-packed window flags (2 bits per entry)
  int pitch = 0;
  int rows = 0, cols = 0;           // full map
  int win_row0 = 0, win_rows = 0;   // rows held by this handle (artp_set_map_window); whole map: 0, rows
  bool has_map = false;
  // [0] warp-stage claim counter, [1] defer count, [2] reach-vertex claim counter, [3] warp-queue count,
  // [4] reach-queue count, [5], [6] unused, [7] scratch (sampler CDF validation), [8] group-queue count, [9] its claim counter
  uint32_t* d_ctr = nullptr;
  uint32_t* d_defer = nullptr;      // deferred record list (bit 31: reach-box queue)
  size_t defer_cap = 0;
  artp::BoxRec* d_recs = nullptr;   // classify -> warp-stage box queue (torso boxes, reach boxes of unusual size)
  artp::BoxRec* d_recs_f = nullptr; // classify -> reach-box queue (one warp per box: zones with -inf or mergeable planes)
  artp::BoxRec* d_recs_g = nullptr; // classify -> reach-box queue of the 8-lane-group kernel (all-finite, merge-free zones)
  int group_grid = 0, group_smem = 0;
  size_t recs_cap = 0;
  uint32_t* d_block_counts = nullptr;
  size_t block_counts_cap = 0;
  void* d_stage = nullptr;          // device staging for the host-buffer API
  size_t stage_cap = 0;
  cudaStream_t stream = nullptr;    // internal compute stream for the host-buffer API
  cudaStream_t copy_stream = nullptr;   // H2D slices of the host-buffer API
  cudaStream_t group_stream = nullptr;  // the 8-lane-group kernel of slice i (host-fed rounds), beside the other box kernels
  cudaEvent_t group_ev = nullptr;
  cudaStream_t box_stream = nullptr;    // box stages of slice i, concurrent with the copy + classify of slice i + 1
  cudaEvent_t copy_ev[16] = {};
  cudaEvent_t slice_ev[kMaxSlices] = {};   // classify of slice i done (box_stream waits on it)
  cudaEvent_t box_ev = nullptr;            // box stages of a round done (stream waits on it)
  int trace = 0;                           // env ARTP_TRACE: print the timeline of host-fed rounds (debug)
  cudaEvent_t tr_ev[6] = {};
  cudaEvent_t tr_slice[8][4] = {};   // ARTP_TRACE: per slice: copy landed, classify start, classify done, box stages done
  uint32_t* d_slices = nullptr;            // per slice, 8 words: {group-queue end, claim, reach-queue end, claim, big-tile-queue end, claim}
  int k1_grid = 0, k2_grid = 0, k2_smem = 0, k2_tcap = 0;
  // stage B (artp_tiles.cuh): [0] big tiles (torso queue, 4 warps per CTA), [1] small tiles (reach-box queue, 8 warps)
  artp::TileCfg tile_cfg[2] = {};
  int tile_grid[2] = {0, 0}, tile_smem[2] = {0, 0}, tile_warps[2] = {8, 8};
  CUtensorMap tile_map[2][2];       // [cfg][layer]: 2-D tile maps over elevation / elevation_masked
  size_t fork_items = (size_t)1 << 30;   // rounds up to this size run their box kernels side by side (env ARTP_FORK_ITEMS; 0 = serial)
  int pipe_tune = 0;                // env ARTP_PIPE_TUNE (experiments on the host-fed pipeline)
  int pipe_cap_g = 4, pipe_cap_f = 4;   // host-fed slices: grid caps of the group / one-warp-per-box reach kernels, in half SM counts (0: none)
  int k0_flags = 0;                 // tuning switch of the classify stage (env ARTP_K0_FLAGS: 2 = no vertex probes)
  bool slice_override = false;
  float sched_override[9] = {0};    // env ARTP_SLICE_SCHEDULE="0.1,0.3,0.6": slice fractions of the host-fed rounds
  size_t slice_items_f64 = 128 * 1024, slice_items_f32 = 256 * 1024;   // H2D pipeline slices of the host-buffer calls (env ARTP_SLICE_ITEMS)
  int mode = 0;
  artp_cnn::State* cnn = nullptr;
  int cnn_mode = 0;
  // sampler (artp_set_sampler): device copies of the per-cell layers, scratch of the fused sample->check->compact path
  artp::SamplerDev samp{};
  float* d_samp_layers = nullptr;   // normal_x | normal_y | normal_z | std_dev | cum_prob | cum_row
  size_t samp_layers_cap = 0;
  bool has_sampler = false;
  bool has_device_normals = false;  // artp_estimate_normals filled normal_x/y/z/std_dev of d_samp_layers for this map
  bool has_device_cdf = false;      // artp_compute_sample_cdf filled cum_prob / cum_row of d_samp_layers for this map
  void* d_samp_scratch = nullptr;
  size_t samp_scratch_cap = 0;
  uint8_t* h_small_out = nullptr;   // mapped pinned host bytes the latency-path kernel writes its verdicts to
  int timing = 0;
  cudaEvent_t ev[6] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};   // classify | warp | reach vertex | reach plane | group
  bool ev_valid = false;
  bool deferred_unread = false;
  // Cross-stream ordering of the per-handle scratch (ADVICE r1): calls may come on different streams; every call that
  // uses a scratch group first makes its stream wait for the previous user of that group, and records an event after.
  // group 0: d_ctr / d_recs / d_defer / d_stage / d_samp_scratch (check, sampler);  group 1: d_block_counts (compaction)
  cudaEvent_t chain_ev[2] = {nullptr, nullptr};
  cudaStream_t chain_stream[2] = {nullptr, nullptr};
  bool chain_busy[2] = {false, false};
  // Sticky error word in mapped pinned host memory: the plane-grouping stage sets it when a zone does not fit its
  // shared-memory store (the item is then marked INVALID -- fail closed). Host-buffer calls return ARTP_E_LIMIT from the
  // call that caused it; device-buffer (asynchronous) calls surface it through artp_poll_error().
  uint32_t* h_err = nullptr;        // host view
  uint32_t* d_err = nullptr;        // device view of the same word
  int tcap_override = 0;            // test hook (artp_debug_set_group_capacity)
  // map change layer (artp_compute_change): the new map's `updated` layer, one bit per cell, and that map's geometry;
  // the roadmap calls read both until the next artp_compute_change
  uint32_t* d_chg_bits = nullptr;
  size_t chg_words_cap = 0;
  bool has_change = false;
  int chg_rows = 0, chg_cols = 0;
  double chg_res = 0, chg_cx = 0, chg_cy = 0;
  artp_stats stats{};
  std::string err;
  std::recursive_mutex mtx;   // recursive: host-buffer entry points hold it across their nested *_device call
};

#define CU_TRY(h, expr)                                                                          \
  do {                                                                                           \
    cudaError_t _e = (expr);                                                                     \
    if (_e != cudaSuccess) {                                                                     \
      (h)->err = std::string(#expr) + ": " + cudaGetErrorString(_e);                             \
      return ARTP_E_CUDA;                                                                        \
    }                                                                                            \
  } while (0)

// H[x + z*nx] = layer[x + (nz-1-z)*nx] (+0.0f canonicalises -0 like GetHeight's (h*scale)+offset,
// ode/ode/src/heightfield.cpp:383).
__global__ void reverse_columns_kernel(const float* __restrict__ layer, float* __restrict__ H, int nx, int nz, int pitch) {
  const size_t total = (size_t)pitch * nz;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const int z = (int)(i / pitch), x = (int)(i - (size_t)z * pitch);
    H[i] = (x < nx) ? layer[x + (size_t)(nz - 1 - z) * nx] * 1.0f + 0.0f : 0.0f;   // pad columns are never read
  }
}

// Range-table level k from level k-1 (level 0 = the heights themselves): reduction over the 2^k x 2^k window
// starting at (x,z) = op of the four 2^(k-1) windows at offsets {0,half} (clamped at the border; clamped windows
// are never queried). (max over all h, min over finite h or +inf, any non-finite).
__global__ void build_level_kernel(const float* __restrict__ H, const float2* __restrict__ prevT,
                                   const unsigned char* __restrict__ prevNF, const unsigned char* __restrict__ mergeable,
                                   float2* __restrict__ T, unsigned char* __restrict__ NF, int nx, int nz, int pitch, int half) {
  const size_t total = (size_t)pitch * nz;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const int z = (int)(i / pitch), x = (int)(i - (size_t)z * pitch);
    if (x >= nx) { T[i] = make_float2(0.f, 0.f); NF[i] = 0; continue; }
    const int x2 = min(x + half, nx - 1), z2 = min(z + half, nz - 1);
    const size_t id[4] = {(size_t)z * pitch + x, (size_t)z * pitch + x2, (size_t)z2 * pitch + x, (size_t)z2 * pitch + x2};
    float mx = -CUDART_INF_F, mn = CUDART_INF_F;
    unsigned char nf = 0;
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      if (prevT) {
        const float2 v = prevT[id[q]];
        mx = fmaxf(mx, v.x); mn = fminf(mn, v.y); nf |= prevNF[id[q]];
      } else {
        const float h = H[id[q]];
        mx = fmaxf(mx, h);
        if (fabsf(h) < CUDART_INF_F) mn = fminf(mn, h); else nf |= 1;
        nf |= mergeable[id[q]];      // 0 or 2: the cell starting at this vertex holds a mergeable triangle
      }
    }
    T[i] = make_float2(mx, mn);
    NF[i] = nf;
  }
}

// ---------------------------------------------------------------------------------------------------------------
// Plane tables: which cells hold a triangle whose plane equals (within eps, the greedy grouping's test,
// heightfield.cpp:1541-1546) the plane of ANOTHER triangle of the layer? A zone without such a cell cannot merge
// anything: every kept triangle is its own plane group whatever the box, and the warp stage skips its merge screen.
// All triangle planes (exact, the collider's arithmetic) go into a hash table keyed by their (n0, n2, d) buckets; a
// second pass looks every triangle's +-2 eps neighbour buckets up. Natural terrain flags nothing; flat or terraced
// maps flag almost everything and keep the screen / the exact grouping stage.
struct PlaneSlot { unsigned long long key; uint32_t lo, hi; };
constexpr unsigned long long kEmptyKey = ~0ull;
__device__ __forceinline__ unsigned long long plane_key(int kx, int kz, int kd) {
  return ((unsigned long long)(uint32_t)(kx & 0xffff) << 48) | ((unsigned long long)(uint32_t)(kz & 0xffff) << 32) | (uint32_t)kd;
}
__device__ __forceinline__ uint32_t plane_slot_hash(unsigned long long k) {
  k ^= k >> 33; k *= 0xff51afd7ed558ccdull; k ^= k >> 33; k *= 0xc4ceb9fe1a85ec53ull; k ^= k >> 33;
  return (uint32_t)k;
}
__global__ void plane_table_clear_kernel(PlaneSlot* tab, size_t cap) {
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < cap; i += (size_t)gridDim.x * blockDim.x) {
    tab[i].key = kEmptyKey; tab[i].lo = 0xffffffffu; tab[i].hi = 0u;
  }
}
// Exact plane of triangle u of cell (x, z), or false if one of its vertices is not finite (never kept).
__device__ __forceinline__ bool cell_tri_plane(const artp::Field& f, int x, int x_off, int z, int u, float pl[4]) {
  float hA, hB, hC, hD;
  artp::load_cell(f, x, z, hA, hB, hC, hD);
  const bool ok = u == 0 ? (artp::finitef(hA) && artp::finitef(hB) && artp::finitef(hC))
                         : (artp::finitef(hD) && artp::finitef(hB) && artp::finitef(hC));
  if (!ok) return false;
  artp::cell_plane(f, u == 0, x + x_off, z, hA, hB, hC, hD, pl);   // vertex coordinates are those of the full map
  return true;
}
__global__ void plane_table_insert_kernel(const artp::Field f, int x_off, PlaneSlot* tab, uint32_t mask) {
  const size_t ncell = (size_t)(f.nx - 1) * (f.nz - 1);
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < 2 * ncell; i += (size_t)gridDim.x * blockDim.x) {
    const size_t c = i >> 1;
    const int u = (int)(i & 1), z = (int)(c / (f.nx - 1)), x = (int)(c - (size_t)z * (f.nx - 1));
    float pl[4];
    if (!cell_tri_plane(f, x, x_off, z, u, pl)) continue;
    const uint32_t id = (uint32_t)(((size_t)z * f.pitch + x) * 2 + u);
    const unsigned long long key = plane_key((int)floorf((pl[0] + 1.0f) * artp::kKeyScale), (int)floorf((pl[2] + 1.0f) * artp::kKeyScale),
                                             artp::dkey(pl[3]));
    uint32_t s = plane_slot_hash(key) & mask;
    for (;;) {
      const unsigned long long old = atomicCAS(&tab[s].key, kEmptyKey, key);
      if (old == kEmptyKey || old == key) {
        // (lo, hi) only has to tell "one triangle" from "several": skip the atomics once id lies strictly inside
        if (!(tab[s].lo < id && tab[s].hi > id)) { atomicMin(&tab[s].lo, id); atomicMax(&tab[s].hi, id); }
        break;
      }
      s = (s + 1) & mask;
    }
  }
}
__global__ void plane_table_query_kernel(const artp::Field f, int x_off, const PlaneSlot* __restrict__ tab, uint32_t mask,
                                         unsigned char* __restrict__ mergeable) {
  const size_t ncell = (size_t)(f.nx - 1) * (f.nz - 1);
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < 2 * ncell; i += (size_t)gridDim.x * blockDim.x) {
    const size_t c = i >> 1;
    const int u = (int)(i & 1), z = (int)(c / (f.nx - 1)), x = (int)(c - (size_t)z * (f.nx - 1));
    float pl[4];
    if (!cell_tri_plane(f, x, x_off, z, u, pl)) continue;
    const uint32_t id = (uint32_t)(((size_t)z * f.pitch + x) * 2 + u);
    const float e2 = 2.0f * ARTP_EPS;
    const int kx0 = (int)floorf((pl[0] - e2 + 1.0f) * artp::kKeyScale), kx1 = (int)floorf((pl[0] + e2 + 1.0f) * artp::kKeyScale);
    const int kz0 = (int)floorf((pl[2] - e2 + 1.0f) * artp::kKeyScale), kz1 = (int)floorf((pl[2] + e2 + 1.0f) * artp::kKeyScale);
    const int kd0 = artp::dkey(pl[3] - e2), kd1 = artp::dkey(pl[3] + e2);
    bool dup = false;
    for (int kx = kx0; kx <= kx1 && !dup; ++kx)
      for (int kz = kz0; kz <= kz1 && !dup; ++kz)
        for (int kd = kd0; kd <= kd1 && !dup; ++kd) {
          const unsigned long long key = plane_key(kx, kz, kd);
          uint32_t s = plane_slot_hash(key) & mask;
          for (;;) {
            const unsigned long long k = tab[s].key;
            if (k == kEmptyKey) break;
            if (k == key) { dup = tab[s].lo != id || tab[s].hi != id; break; }
            s = (s + 1) & mask;
          }
        }
    if (dup) mergeable[(size_t)z * f.pitch + x] = 2;   // races write the same value
  }
}

// 16 flag bytes (values 0..3) -> one word of 2-bit fields; the tail of the last word is zero
__global__ void pack_flags_kernel(const unsigned char* __restrict__ nf, size_t n, uint32_t* __restrict__ out) {
  const size_t words = (n + 15) / 16;
  for (size_t w = blockIdx.x * (size_t)blockDim.x + threadIdx.x; w < words; w += (size_t)gridDim.x * blockDim.x) {
    uint32_t v = 0;
    for (int i = 0; i < 16; ++i) {
      const size_t e = w * 16 + i;
      if (e < n) v |= (uint32_t)(nf[e] & 3) << (2 * i);
    }
    out[w] = v;
  }
}

__global__ void fill_u8_kernel(uint8_t* p, size_t n, uint8_t v) {
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) p[i] = v;
}

// PathLengthObjective::motionCost (art_planner/src/objectives/path_length_objective.cpp:26-70), double.
__global__ void path_length_kernel(const double* __restrict__ s1, const double* __restrict__ s2, size_t n,
                                   double* __restrict__ cost, int directional, double v_lon, double v_lat,
                                   double v_ang) {
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    const double* a = s1 + 7 * i;
    const double* b = s2 + 7 * i;
    const double x_dif = b[0] - a[0], y_dif = b[1] - a[1], z_dif = b[2] - a[2];
    if (!directional) {
      cost[i] = sqrt(x_dif * x_dif + y_dif * y_dif + z_dif * z_dif) / v_lon;
      continue;
    }
    // getYawFromSO3 returns `Scalar` = float (utils.h:80-88)
    const double yaw1 = (double)(float)atan2(2 * (a[6] * a[5] + a[3] * a[4]), 1 - 2 * (a[4] * a[4] + a[5] * a[5]));
    const double yaw2 = (double)(float)atan2(2 * (b[6] * b[5] + b[3] * b[4]), 1 - 2 * (b[4] * b[4] + b[5] * b[5]));
    const double d = fabs(yaw1 - yaw2);
    const double yaw_dif = (d > 3.14159265358979323846) ? 2.0 * 3.14159265358979323846 - d : d;
    const double lon_dif = cos(yaw1) * x_dif + sin(yaw1) * y_dif;
    const double lat_dif = -sin(yaw1) * x_dif + cos(yaw1) * y_dif;
    const double t_yaw = fabs(yaw_dif) / v_ang, t_lon = fabs(lon_dif) / v_lon, t_lat = fabs(lat_dif) / v_lat;
    const double m = t_lon > t_lat ? t_lon : t_lat;
    cost[i] = m > t_yaw ? m : t_yaw;
  }
}

// Ordered compaction: (A) per-block counts, (B) single-block exclusive scan, (C) scatter.
constexpr int kCompactBlock = 1024;
// BITS: the mask is bit-packed (item i = bit i&31 of word i>>5, artp_pack_valid_bits_device), else one byte per item.
template <bool BITS>
__device__ __forceinline__ int mask_at(const uint8_t* __restrict__ valid, size_t i) {
  if (BITS) return (int)((reinterpret_cast<const uint32_t*>(valid)[i >> 5] >> (i & 31)) & 1u);
  return valid[i] != 0;
}
template <bool BITS>
__global__ void compact_count_kernel(const uint8_t* __restrict__ valid, size_t n, uint32_t* __restrict__ counts) {
  const size_t i = (size_t)blockIdx.x * kCompactBlock + threadIdx.x;
  const int v = (i < n) && mask_at<BITS>(valid, i);
  const int c = __syncthreads_count(v);
  if (threadIdx.x == 0) counts[blockIdx.x] = (uint32_t)c;
}
__global__ void compact_scan_kernel(uint32_t* counts, size_t nb, uint32_t* total) {
  __shared__ uint32_t carry;
  __shared__ uint32_t wsum[32];
  if (threadIdx.x == 0) carry = 0;
  __syncthreads();
  for (size_t b0 = 0; b0 < nb; b0 += blockDim.x) {
    const size_t i = b0 + threadIdx.x;
    const uint32_t v = i < nb ? counts[i] : 0u;
    uint32_t x = v;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    for (int o = 1; o < 32; o <<= 1) { const uint32_t y = __shfl_up_sync(0xffffffffu, x, o); if (lane >= o) x += y; }
    if (lane == 31) wsum[wid] = x;
    __syncthreads();
    if (wid == 0) {
      uint32_t s = lane < (int)(blockDim.x >> 5) ? wsum[lane] : 0u;
      for (int o = 1; o < 32; o <<= 1) { const uint32_t y = __shfl_up_sync(0xffffffffu, s, o); if (lane >= o) s += y; }
      wsum[lane] = s;
    }
    __syncthreads();
    const uint32_t before = carry + (wid ? wsum[wid - 1] : 0u) + x - v;
    if (i < nb) counts[i] = before;
    __syncthreads();
    if (threadIdx.x == blockDim.x - 1) carry = before + v;
    __syncthreads();
  }
  if (threadIdx.x == 0) *total = carry;
}
template <bool BITS, typename IndexT>
__global__ void compact_scatter_kernel(const uint8_t* __restrict__ valid, size_t n, int64_t base,
                                       const uint32_t* __restrict__ offsets, IndexT* __restrict__ out) {
  __shared__ uint32_t wsum[32];
  const size_t i = (size_t)blockIdx.x * kCompactBlock + threadIdx.x;
  const int v = (i < n) && mask_at<BITS>(valid, i);
  const unsigned bal = __ballot_sync(0xffffffffu, v);
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  if (lane == 0) wsum[wid] = __popc(bal);
  __syncthreads();
  if (wid == 0) {
    uint32_t s = wsum[lane];
    for (int o = 1; o < 32; o <<= 1) { const uint32_t y = __shfl_up_sync(0xffffffffu, s, o); if (lane >= o) s += y; }
    wsum[lane] = s;
  }
  __syncthreads();
  if (v) {
    const uint32_t pos = offsets[blockIdx.x] + (wid ? wsum[wid - 1] : 0u) + __popc(bal & ((1u << lane) - 1u));
    out[pos] = (IndexT)(base + (int64_t)i);
  }
}

// bits[w] bit b = valid[32*w + b] != 0; one warp ballot per word, tail bits zero.
__global__ void pack_bits_kernel(const uint8_t* __restrict__ valid, size_t n, uint32_t* __restrict__ bits) {
  const size_t words = (n + 31) / 32;
  const size_t warps = ((size_t)gridDim.x * blockDim.x) >> 5, wid = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  for (size_t w = wid; w < words; w += warps) {
    const size_t i = w * 32 + lane;
    const unsigned bal = __ballot_sync(0xffffffffu, i < n && valid[i] != 0);
    if (lane == 0) bits[w] = bal;
  }
}

constexpr size_t kChunkItems = 1u << 20;   // work items per internal launch round (bounds the box queue)

int ensure_queues(Handle* h, size_t n_items, cudaStream_t s) {
  (void)s;
  const size_t need = 5 * std::min(n_items, kChunkItems);
  if (h->recs_cap >= need) return ARTP_OK;
  CU_TRY(h, cudaDeviceSynchronize());   // rare (growth only): users on any stream must be done before the free
  cudaFree(h->d_defer); cudaFree(h->d_recs); cudaFree(h->d_recs_f); cudaFree(h->d_recs_g);
  h->d_defer = nullptr; h->d_recs = nullptr; h->d_recs_f = nullptr; h->d_recs_g = nullptr; h->recs_cap = 0;
  const size_t cap = std::max<size_t>(need, 1u << 16);
  CU_TRY(h, cudaMalloc(&h->d_recs, cap * sizeof(artp::BoxRec)));
  CU_TRY(h, cudaMalloc(&h->d_recs_f, cap * sizeof(artp::BoxRec)));
  CU_TRY(h, cudaMalloc(&h->d_recs_g, cap * sizeof(artp::BoxRec)));
  CU_TRY(h, cudaMalloc(&h->d_defer, cap * sizeof(uint32_t)));
  h->recs_cap = cap; h->defer_cap = cap;
  return ARTP_OK;
}

int ensure_stage(Handle* h, size_t bytes) {
  if (h->stage_cap >= bytes) return ARTP_OK;
  CU_TRY(h, cudaDeviceSynchronize());
  if (h->d_stage) CU_TRY(h, cudaFree(h->d_stage));
  h->d_stage = nullptr;
  CU_TRY(h, cudaMalloc(&h->d_stage, bytes));
  h->stage_cap = bytes;
  return ARTP_OK;
}

// Scratch-group ordering across streams (see Handle::chain_ev).
int chain_begin(Handle* h, int g, cudaStream_t s) {
  if (h->chain_busy[g] && h->chain_stream[g] != s) CU_TRY(h, cudaStreamWaitEvent(s, h->chain_ev[g], 0));
  return ARTP_OK;
}
int chain_end(Handle* h, int g, cudaStream_t s) {
  CU_TRY(h, cudaEventRecord(h->chain_ev[g], s));
  h->chain_stream[g] = s;
  h->chain_busy[g] = true;
  return ARTP_OK;
}
struct ChainScope {   // begin on construction, end on destruction (every return path)
  Handle* h; int g; cudaStream_t s; int rc;
  ChainScope(Handle* h_, int g_, cudaStream_t s_) : h(h_), g(g_), s(s_), rc(chain_begin(h_, g_, s_)) {}
  ~ChainScope() { if (rc == ARTP_OK) chain_end(h, g, s); }
};

// Sticky plane-grouping overflow (set by the device, see Handle::h_err): read and clear.
int take_sticky_error(Handle* h) {
  if (h->h_err && *(volatile uint32_t*)h->h_err) {
    const uint32_t e = *(volatile uint32_t*)h->h_err;
    *(volatile uint32_t*)h->h_err = 0;
    if (e & artp::kRoadmapBadEdge) {
      h->err = "an edge referenced a vertex index >= nv (artp_roadmap_updates_device); its flag was set to 1";
      return ARTP_E_INVALID;
    }
    if (e & 2u) {
      h->err = "a box reached outside this handle's map window (artp_set_map_window: route samples to the shard that holds them, "
               "halo >= box half-diagonal + offsets); affected poses were marked invalid";
      return ARTP_E_WINDOW;
    }
    h->err = "plane-grouping stage overflow: a zone exceeded its shared-memory store; affected poses were marked invalid";
    return ARTP_E_LIMIT;
  }
  return ARTP_OK;
}

// Optional host feed of a call: the states are copied H2D in slices on the copy stream while the kernels of the
// previous slice run on the compute stream.
struct HostFeed {
  const char* host;        // host states
  char* dev;               // device destination (same layout)
  size_t bytes_per_item;
  size_t slice_items;      // classic equal slices (small calls, env override)
  // Slice schedule of a full round as fractions (0-terminated; empty: equal slices): a small first slice so that the
  // kernels start early, then equal ones. Every slice costs its kernels' latency floors (~0.1 ms of chain per slice,
  // profiles/stage_vs_n.py), which is why five or six slices beat both fewer (long tail after the last byte) and more, and
  // why shrinking the last slices below ~15 % buys nothing (measured with ARTP_SLICE_SCHEDULE / ARTP_TRACE).
  float schedule[8];
};

// The claim counters of the consumer stages restart where the next slice's producers will append (the persistent
// consumers of the previous slice overshoot their counters).
__global__ void restart_claims_kernel(uint32_t* ctr) {
  ctr[0] = ctr[3]; ctr[2] = ctr[4]; ctr[9] = ctr[8];
}

// Slice i of a piped round is closed: its box stages consume the queue entries [end of slice i-1, current count).
__global__ void close_slice_kernel(const uint32_t* ctr, uint32_t* slices, int i) {
  const uint32_t g0 = i ? slices[8 * (i - 1)] : 0u, f0 = i ? slices[8 * (i - 1) + 2] : 0u, w0 = i ? slices[8 * (i - 1) + 4] : 0u;
  slices[8 * i] = ctr[8]; slices[8 * i + 1] = g0;        // group queue: end, claim counter (starts at the slice's begin)
  slices[8 * i + 2] = ctr[4]; slices[8 * i + 3] = f0;    // reach-box queue
  slices[8 * i + 4] = ctr[3]; slices[8 * i + 5] = w0;    // big-tile queue
}

// Host-fed round (the host-buffer entry points): the states arrive in slices over PCIe. Four streams:
//   copy_stream    H2D of slice i+1
//   s              classify of slice i as soon as its copy has landed (appends to the three box queues)
//   box_stream     one-warp-per-box kernels of slice i (reach-box queue, then big-tile queue) over exactly the queue entries
//                  its classify appended (per-slice claim counters, close_slice_kernel), then the grouping stage once per round
//   group_stream   the 8-lane-group kernel of slice i, beside them
// so the copy, the classify stage and the box stages of consecutive slices overlap; s waits for box_stream at the end.
int run_round_piped(Handle* h, artp::Work w, cudaStream_t s, const HostFeed* feed, size_t base, size_t end, size_t slice,
                    uint32_t& launches, size_t& ev_i) {
  CU_TRY(h, cudaMemsetAsync(h->d_ctr, 0, 16 * sizeof(uint32_t), s));
  // slice boundaries
  size_t cut[kMaxSlices + 1];
  int ncut = 0;
  cut[0] = base;
  const float* sched = feed->schedule;
  if (h->sched_override[0] > 0.0f) sched = h->sched_override;          // ARTP_SLICE_SCHEDULE (experiments)
  if (sched[0] > 0.0f && end - base >= (1u << 18) && !h->slice_override) {
    double acc = 0.0;
    for (int i = 0; i < 8 && sched[i] > 0.0f; ++i) {
      acc += sched[i];
      size_t c = base + (size_t)((double)(end - base) * acc);
      c = std::min(end, (c + 127) & ~(size_t)127);
      if (c > cut[ncut]) cut[++ncut] = c;
    }
    if (cut[ncut] != end) cut[++ncut] = end;
  } else {
    for (size_t lo = base; lo < end; lo += slice) cut[++ncut] = std::min(end, lo + slice);
  }
  const auto cpu_t0 = std::chrono::steady_clock::now();
  double cpu_ms[kMaxSlices + 2] = {0};
  if (h->trace) { cudaEventRecord(h->tr_ev[0], s); cudaStreamWaitEvent(h->copy_stream, h->tr_ev[0], 0); cudaEventRecord(h->tr_ev[1], h->copy_stream); }
  for (int si = 0; si < ncut; ++si) {
    const size_t lo = cut[si], hi = cut[si + 1];
    CU_TRY(h, cudaMemcpyAsync(feed->dev + lo * feed->bytes_per_item, feed->host + lo * feed->bytes_per_item,
                              (hi - lo) * feed->bytes_per_item, cudaMemcpyHostToDevice, h->copy_stream));
    cudaEvent_t ev = h->copy_ev[ev_i++ % kCopyEvents];
    CU_TRY(h, cudaEventRecord(ev, h->copy_stream));
    CU_TRY(h, cudaStreamWaitEvent(s, ev, 0));
    if (h->trace && si < 8) { cudaEventRecord(h->tr_slice[si][0], h->copy_stream); cudaEventRecord(h->tr_slice[si][1], s); }
    w.item_base = (uint32_t)lo;
    w.n_items = (uint32_t)hi;
    artp::classify_items_kernel<<<(unsigned)((hi - lo + 127) / 128), 128, 0, s>>>(
        h->chk, w, h->d_recs, h->d_recs_f, h->group_grid ? h->d_recs_g : nullptr, h->d_ctr + 3, h->d_ctr + 4, h->d_ctr + 8,
        (h->mode == 1 ? 1 : 0) | h->k0_flags);
    close_slice_kernel<<<1, 1, 0, s>>>(h->d_ctr, h->d_slices, si);
    CU_TRY(h, cudaGetLastError());
    if (h->trace && si < 8) cudaEventRecord(h->tr_slice[si][2], s);
    CU_TRY(h, cudaEventRecord(h->slice_ev[si], s));
    CU_TRY(h, cudaStreamWaitEvent(h->box_stream, h->slice_ev[si], 0));
    const size_t nb = hi - lo;
    if (h->group_grid) {
      CU_TRY(h, cudaStreamWaitEvent(h->group_stream, h->slice_ev[si], 0));
      unsigned grid_g = (unsigned)std::min<size_t>((size_t)h->group_grid, (nb + 7) / 8);
      if (h->pipe_cap_g) grid_g = std::min<unsigned>(grid_g, (unsigned)(h->pipe_cap_g * h->sm_count / 2));
      artp::reach_groups_kernel<<<grid_g, artp::kMaxTileWarps * 32, h->group_smem, h->group_stream>>>(
          h->chk, h->tile_map[1][1], h->tile_cfg[1], w, h->d_recs_g, h->d_slices + 8 * si, h->d_slices + 8 * si + 1);
      launches += 1;
    }
    if (h->chk.reach_tw) {
      const int wpc = h->tile_warps[1];
      unsigned grid_f = (unsigned)std::min<size_t>((size_t)h->tile_grid[1], (4 * nb + wpc - 1) / wpc);
      if (h->pipe_cap_f) grid_f = std::min<unsigned>(grid_f, (unsigned)(h->pipe_cap_f * h->sm_count / 2));
      artp::box_tiles_warp_kernel<<<grid_f, wpc * 32, h->tile_smem[1], h->box_stream>>>(
          h->chk, h->tile_map[1][1], h->tile_map[1][1], h->tile_cfg[1], w, h->d_recs_f, h->d_slices + 8 * si + 2, h->d_slices + 8 * si + 3,
          h->d_ctr + 1, h->d_defer, artp::kDeferReachBit, h->mode == 1);
      launches += 1;
    }
    {
      // the big-tile queue (torso boxes: few) of this slice, behind its reach-box queue
      const int wpc = h->tile_warps[0];
      const unsigned grid_w = (unsigned)std::min<size_t>((size_t)h->tile_grid[0], (nb + wpc - 1) / wpc);
      artp::box_tiles_warp_kernel<<<grid_w, wpc * 32, h->tile_smem[0], h->box_stream>>>(
          h->chk, h->tile_map[0][0], h->tile_map[0][1], h->tile_cfg[0], w, h->d_recs, h->d_slices + 8 * si + 4, h->d_slices + 8 * si + 5,
          h->d_ctr + 1, h->d_defer, 0u, h->mode == 1);
      launches += 1;
    }
    CU_TRY(h, cudaGetLastError());
    launches += 2;
    if (h->trace && si < 8) cudaEventRecord(h->tr_slice[si][3], h->box_stream);
    if (h->trace) cpu_ms[si] = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - cpu_t0).count();
  }
  if (h->group_grid) {
    // the grouping stage (box_stream) runs last: the group kernels must not clear a verdict after it has been copied out
    CU_TRY(h, cudaEventRecord(h->group_ev, h->group_stream));
    CU_TRY(h, cudaStreamWaitEvent(h->box_stream, h->group_ev, 0));
  }
  if (h->trace) { cudaEventRecord(h->tr_ev[2], h->copy_stream); cudaEventRecord(h->tr_ev[3], s); cudaEventRecord(h->tr_ev[4], h->box_stream); }
  w.item_base = (uint32_t)base;
  w.n_items = (uint32_t)end;
  const unsigned grid_c = (unsigned)std::min<size_t>((size_t)h->k2_grid, 5 * (end - base));
  artp::box_items_block_kernel<<<grid_c, artp::kBlockStageThreads, h->k2_smem, h->box_stream>>>(h->chk, w, h->d_recs, h->d_recs_f, h->d_ctr + 1,
                                                                                             h->d_defer, h->k2_tcap, h->d_err);
  CU_TRY(h, cudaGetLastError());
  launches += 1;
  CU_TRY(h, cudaEventRecord(h->box_ev, h->box_stream));
  CU_TRY(h, cudaStreamWaitEvent(s, h->box_ev, 0));
  if (h->trace) {
    cudaEventRecord(h->tr_ev[5], s);
    cudaEventSynchronize(h->tr_ev[5]);
    float t[5];
    for (int i = 0; i < 5; ++i) cudaEventElapsedTime(&t[i], h->tr_ev[0], h->tr_ev[i + 1]);
    std::fprintf(stderr, "[artp trace] copies start %.3f end %.3f | classify end %.3f | box stages end %.3f | grouping end %.3f ms | cpu submit",
                 t[0], t[1], t[2], t[3], t[4]);
    for (int i = 0; i < ncut; ++i) std::fprintf(stderr, " %.3f", cpu_ms[i]);
    std::fprintf(stderr, "\n[artp trace]   per slice (copy landed, classify start, classify done, box done):");
    for (int i = 0; i < ncut && i < 8; ++i) {
      float u[4];
      for (int j = 0; j < 4; ++j) cudaEventElapsedTime(&u[j], h->tr_ev[0], h->tr_slice[i][j]);
      std::fprintf(stderr, "  [%.3f %.3f %.3f %.3f]", u[0], u[1], u[2], u[3]);
    }
    std::fprintf(stderr, "\n");
  }
  return ARTP_OK;
}

// Launch the pipeline for a prepared Work (items 0 .. w.n_items = the whole call) on stream s, in rounds of
// kChunkItems work items (bounds the box queues). Within a round the stages run slice by slice -- classify (A), warp
// stage (W: torso boxes), reach vertex scan (F1), reach plane stage (F2); the queues and claim counters simply keep
// growing -- and the plane-grouping stage (C) runs ONCE over all boxes deferred in the round (its sequential greedy has
// a fixed latency of tens of microseconds per launch).
int run_items(Handle* h, artp::Work w, cudaStream_t s, const HostFeed* feed = nullptr) {
  const size_t n_total = w.n_items;
  int rc = ensure_queues(h, n_total, s);
  if (rc) return rc;
  uint32_t launches = 0;
  size_t ev_i = 0;
  for (size_t base = 0; base < n_total; base += kChunkItems) {
    const size_t end = std::min(n_total, base + kChunkItems);
    const bool last_round = end == n_total;
    if (feed && feed->slice_items < end - base && (end - base + feed->slice_items - 1) / feed->slice_items < (size_t)kMaxSlices &&
        !h->timing) {
      rc = run_round_piped(h, w, s, feed, base, end, feed->slice_items, launches, ev_i);
      if (rc) return rc;
      continue;
    }
    CU_TRY(h, cudaMemsetAsync(h->d_ctr, 0, 16 * sizeof(uint32_t), s));
    const size_t slice = (feed && feed->slice_items < end - base) ? feed->slice_items : (end - base);
    for (size_t lo = base; lo < end; lo += slice) {
      const size_t hi = std::min(end, lo + slice);
      const bool last = last_round && hi == end;
      if (feed) {
        const bool piped = slice < end - base;
        cudaStream_t cs = piped ? h->copy_stream : s;
        CU_TRY(h, cudaMemcpyAsync(feed->dev + lo * feed->bytes_per_item, feed->host + lo * feed->bytes_per_item,
                                  (hi - lo) * feed->bytes_per_item, cudaMemcpyHostToDevice, cs));
        if (piped) {
          cudaEvent_t ev = h->copy_ev[ev_i++ % kCopyEvents];
          CU_TRY(h, cudaEventRecord(ev, h->copy_stream));
          CU_TRY(h, cudaStreamWaitEvent(s, ev, 0));
        }
      }
      w.item_base = (uint32_t)lo;
      w.n_items = (uint32_t)hi;
      if (lo != base) { restart_claims_kernel<<<1, 1, 0, s>>>(h->d_ctr); launches += 1; }
      if (h->timing && last) CU_TRY(h, cudaEventRecord(h->ev[0], s));
      artp::classify_items_kernel<<<(unsigned)((hi - lo + 127) / 128), 128, 0, s>>>(
          h->chk, w, h->d_recs, h->d_recs_f, h->group_grid ? h->d_recs_g : nullptr, h->d_ctr + 3, h->d_ctr + 4, h->d_ctr + 8,
        (h->mode == 1 ? 1 : 0) | h->k0_flags);
      CU_TRY(h, cudaGetLastError());
      if (h->timing && last) CU_TRY(h, cudaEventRecord(h->ev[1], s));
      // small batches (the planner's one-state isValid calls): no more CTAs than there can be boxes
      const size_t nb = hi - lo;
      // The three box kernels are independent of each other (each only clears verdicts). Batches too small to fill the GPU
      // with any one of them (each has a latency floor of 20-30 us) run them side by side: the two reach-box kernels fork
      // onto box_stream / group_stream after the classify stage and join before the grouping stage.
      const bool fork = !h->timing && nb <= h->fork_items && h->chk.reach_tw;
      cudaStream_t s_f = fork ? h->box_stream : s, s_g = fork ? h->group_stream : s;
      if (fork) {
        CU_TRY(h, cudaEventRecord(h->slice_ev[0], s));
        CU_TRY(h, cudaStreamWaitEvent(h->box_stream, h->slice_ev[0], 0));
        if (h->group_grid) CU_TRY(h, cudaStreamWaitEvent(h->group_stream, h->slice_ev[0], 0));
      }
      {
        const int wpc = h->tile_warps[0];
        const unsigned grid_w = (unsigned)std::min<size_t>((size_t)h->tile_grid[0], (5 * nb + wpc - 1) / wpc);
        artp::box_tiles_warp_kernel<<<grid_w, wpc * 32, h->tile_smem[0], s>>>(h->chk, h->tile_map[0][0], h->tile_map[0][1], h->tile_cfg[0],
                                                                               w, h->d_recs, h->d_ctr + 3, h->d_ctr, h->d_ctr + 1, h->d_defer,
                                                                               0u, h->mode == 1);
        CU_TRY(h, cudaGetLastError());
      }
      if (h->timing && last) CU_TRY(h, cudaEventRecord(h->ev[2], s));
      if (h->chk.reach_tw) {
        const int wpc = h->tile_warps[1];
        const unsigned grid_f = (unsigned)std::min<size_t>((size_t)h->tile_grid[1], (4 * nb + wpc - 1) / wpc);
        artp::box_tiles_warp_kernel<<<grid_f, wpc * 32, h->tile_smem[1], s_f>>>(h->chk, h->tile_map[1][1], h->tile_map[1][1], h->tile_cfg[1],
                                                                                 w, h->d_recs_f, h->d_ctr + 4, h->d_ctr + 2, h->d_ctr + 1,
                                                                                 h->d_defer, artp::kDeferReachBit, h->mode == 1);
        CU_TRY(h, cudaGetLastError());
        launches += 1;
      }
      if (h->timing && last) CU_TRY(h, cudaEventRecord(h->ev[3], s));
      if (h->group_grid) {
        const unsigned grid_g = (unsigned)std::min<size_t>((size_t)h->group_grid, (nb + 7) / 8);
        artp::reach_groups_kernel<<<grid_g, artp::kMaxTileWarps * 32, h->group_smem, s_g>>>(h->chk, h->tile_map[1][1], h->tile_cfg[1], w,
                                                                                             h->d_recs_g, h->d_ctr + 8, h->d_ctr + 9);
        CU_TRY(h, cudaGetLastError());
        launches += 1;
      }
      if (fork) {
        CU_TRY(h, cudaEventRecord(h->box_ev, h->box_stream));
        CU_TRY(h, cudaStreamWaitEvent(s, h->box_ev, 0));
        if (h->group_grid) {
          CU_TRY(h, cudaEventRecord(h->group_ev, h->group_stream));
          CU_TRY(h, cudaStreamWaitEvent(s, h->group_ev, 0));
        }
      }
      if (h->timing && last) CU_TRY(h, cudaEventRecord(h->ev[4], s));
      launches += 2;
    }
    w.item_base = (uint32_t)base;
    w.n_items = (uint32_t)end;
    const unsigned grid_c = (unsigned)std::min<size_t>((size_t)h->k2_grid, 5 * (end - base));
    artp::box_items_block_kernel<<<grid_c, artp::kBlockStageThreads, h->k2_smem, s>>>(h->chk, w, h->d_recs, h->d_recs_f, h->d_ctr + 1,
                                                                      h->d_defer, h->k2_tcap, h->d_err);
    CU_TRY(h, cudaGetLastError());
    if (h->timing && last_round) { CU_TRY(h, cudaEventRecord(h->ev[5], s)); h->ev_valid = true; }
    launches += 1;
  }
  h->stats.kernel_launches += launches;
  h->stats.last_launches = launches;
  h->deferred_unread = true;
  return ARTP_OK;
}

int check_common(Handle* h, size_t n) {
  if (!h->has_map) { h->err = "no map set"; return ARTP_E_NOMAP; }
  if (n >= (size_t)0xFFFFFFF0u) { h->err = "too many items for one call"; return ARTP_E_LIMIT; }
  return ARTP_OK;
}

}  // namespace

extern "C" {

const char* artp_version(void) { return "artp 0.1 sm_100a"; }

const char* artp_last_error(const artp_handle* hh) {
  if (!hh) return g_create_error.c_str();
  return reinterpret_cast<const Handle*>(hh)->err.c_str();
}

int artp_create(const artp_params* params, artp_handle** out) {
  if (!params || !out) { g_create_error = "null argument"; return ARTP_E_INVALID; }
  *out = nullptr;
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0) {
    g_create_error = std::string("no CUDA device: ") + cudaGetErrorString(e);
    return ARTP_E_CUDA;
  }
  if (params->device < 0 || params->device >= ndev) { g_create_error = "bad device ordinal"; return ARTP_E_INVALID; }
  if (!(params->torso_length > 0 && params->torso_width > 0 && params->torso_height > 0 && params->reach_x > 0 &&
        params->reach_y > 0 && params->reach_z > 0)) {
    g_create_error = "box dimensions must be positive";
    return ARTP_E_INVALID;
  }
  Handle* h = new Handle();
  h->p = *params;
  h->device = params->device;
  auto fail = [&](const char* what, cudaError_t ce) {
    g_create_error = std::string(what) + ": " + cudaGetErrorString(ce);
    delete h;
    return ARTP_E_CUDA;
  };
  if ((e = cudaSetDevice(h->device)) != cudaSuccess) return fail("cudaSetDevice", e);
  cudaDeviceProp prop;
  if ((e = cudaGetDeviceProperties(&prop, h->device)) != cudaSuccess) return fail("cudaGetDeviceProperties", e);
  h->sm_count = prop.multiProcessorCount;
  cudaFuncAttributes fa;
  if ((e = cudaFuncGetAttributes(&fa, artp::box_tiles_warp_kernel)) != cudaSuccess)
    return fail("no usable kernel image (built for sm_100a)", e);
  {
    // experiment switch ARTP_PIPE_TUNE: bit 0 = the call's own stream (classify) gets the highest priority, the box-stage
    // streams the lowest (measured: no effect); ARTP_PIPE_CAPS: see pipe_cap_g / pipe_cap_f
    if (const char* pt = std::getenv("ARTP_PIPE_TUNE")) h->pipe_tune = std::atoi(pt);
    if (const char* fi = std::getenv("ARTP_FORK_ITEMS")) h->fork_items = (size_t)std::atoll(fi);
    if (const char* pc = std::getenv("ARTP_PIPE_CAPS")) std::sscanf(pc, "%d,%d", &h->pipe_cap_g, &h->pipe_cap_f);   // "g,f" in half SM counts
    int lo_p = 0, hi_p = 0;
    cudaDeviceGetStreamPriorityRange(&lo_p, &hi_p);
    const bool prio = (h->pipe_tune & 1) != 0;
    if ((e = cudaStreamCreateWithPriority(&h->stream, cudaStreamNonBlocking, prio ? hi_p : 0)) != cudaSuccess) return fail("cudaStreamCreate", e);
    if ((e = cudaStreamCreateWithPriority(&h->copy_stream, cudaStreamNonBlocking, prio ? hi_p : 0)) != cudaSuccess) return fail("cudaStreamCreate", e);
    if ((e = cudaStreamCreateWithPriority(&h->box_stream, cudaStreamNonBlocking, prio ? lo_p : 0)) != cudaSuccess) return fail("cudaStreamCreate", e);
    if ((e = cudaStreamCreateWithPriority(&h->group_stream, cudaStreamNonBlocking, prio ? lo_p : 0)) != cudaSuccess) return fail("cudaStreamCreate", e);
  }
  if ((e = cudaEventCreateWithFlags(&h->group_ev, cudaEventDisableTiming)) != cudaSuccess) return fail("cudaEventCreate", e);
  for (int i = 0; i < kMaxSlices; ++i)
    if ((e = cudaEventCreateWithFlags(&h->slice_ev[i], cudaEventDisableTiming)) != cudaSuccess) return fail("cudaEventCreate", e);
  if ((e = cudaEventCreateWithFlags(&h->box_ev, cudaEventDisableTiming)) != cudaSuccess) return fail("cudaEventCreate", e);
  if ((e = cudaMalloc(&h->d_slices, kMaxSlices * 8 * sizeof(uint32_t))) != cudaSuccess) return fail("cudaMalloc", e);
  for (int i = 0; i < kCopyEvents; ++i)
    if ((e = cudaEventCreateWithFlags(&h->copy_ev[i], cudaEventDisableTiming)) != cudaSuccess) return fail("cudaEventCreate", e);
  if ((e = cudaMalloc(&h->d_ctr, 16 * sizeof(uint32_t))) != cudaSuccess) return fail("cudaMalloc", e);
  for (int g = 0; g < 2; ++g)
    if ((e = cudaEventCreateWithFlags(&h->chain_ev[g], cudaEventDisableTiming)) != cudaSuccess) return fail("cudaEventCreate", e);
  if ((e = cudaHostAlloc((void**)&h->h_err, 64, cudaHostAllocMapped)) != cudaSuccess) return fail("cudaHostAlloc", e);
  *h->h_err = 0;
  if ((e = cudaHostGetDevicePointer((void**)&h->d_err, h->h_err, 0)) != cudaSuccess) return fail("cudaHostGetDevicePointer", e);
  if (const char* kf = std::getenv("ARTP_K0_FLAGS")) h->k0_flags = std::atoi(kf) & 2;
  if (std::getenv("ARTP_TRACE")) {
    h->trace = 1;
    for (auto& te : h->tr_ev) cudaEventCreate(&te);
    for (auto& ts : h->tr_slice) for (auto& te : ts) cudaEventCreate(&te);
  }
  if (const char* sl = std::getenv("ARTP_SLICE_ITEMS")) {
    const long v = std::atol(sl);
    if (v >= 1024) { h->slice_items_f64 = (size_t)v; h->slice_items_f32 = (size_t)v; h->slice_override = true; }
  }
  if (const char* sc = std::getenv("ARTP_SLICE_SCHEDULE")) {
    int i = 0;
    for (const char* p = sc; *p && i < 8;) {
      char* q = nullptr;
      const float v = std::strtof(p, &q);
      if (q == p) break;
      if (v > 0.0f) h->sched_override[i++] = v;
      p = (*q == ',') ? q + 1 : q;
    }
  }
  h->cnn = artp_cnn::create(h->device, h->sm_count);
  // checker constants (float casts as the reference's ctor/Pose3FromXYZ arguments make them)
  artp::Checker& c = h->chk;
  std::memset(&c, 0, sizeof(c));
  c.side[0][0] = (float)params->torso_length; c.side[0][1] = (float)params->torso_width; c.side[0][2] = (float)params->torso_height;
  c.side[1][0] = (float)params->reach_x; c.side[1][1] = (float)params->reach_y; c.side[1][2] = (float)params->reach_z;
  c.torso_off[0] = (float)params->torso_off_x; c.torso_off[1] = (float)params->torso_off_y;
  c.torso_off[2] = (float)(params->torso_off_z - params->feet_off_z);
  c.feet_ox = (float)params->feet_off_x; c.feet_oy = (float)params->feet_off_y;
  c.unknown_untraversable = params->unknown_space_untraversable ? 1 : 0;
  *out = reinterpret_cast<artp_handle*>(h);
  return ARTP_OK;
}

void artp_destroy(artp_handle* hh) {
  if (!hh) return;
  Handle* h = reinterpret_cast<Handle*>(hh);
  cudaSetDevice(h->device);
  if (h->stream) { cudaStreamSynchronize(h->stream); cudaStreamDestroy(h->stream); }
  if (h->copy_stream) { cudaStreamSynchronize(h->copy_stream); cudaStreamDestroy(h->copy_stream); }
  for (int i = 0; i < kCopyEvents; ++i) if (h->copy_ev[i]) cudaEventDestroy(h->copy_ev[i]);
  if (h->box_stream) { cudaStreamSynchronize(h->box_stream); cudaStreamDestroy(h->box_stream); }
  if (h->group_stream) { cudaStreamSynchronize(h->group_stream); cudaStreamDestroy(h->group_stream); }
  if (h->group_ev) cudaEventDestroy(h->group_ev);
  for (int i = 0; i < kMaxSlices; ++i) if (h->slice_ev[i]) cudaEventDestroy(h->slice_ev[i]);
  if (h->box_ev) cudaEventDestroy(h->box_ev);
  cudaFree(h->d_slices);
  for (int k = 0; k < 2; ++k) for (int l = 0; l <= artp::kMaxLevel; ++l) { cudaFree(h->d_T[k][l]); cudaFree(h->d_NF[k][l]); }
  cudaFree(h->d_H[0]); cudaFree(h->d_H[1]); cudaFree(h->d_ctr); cudaFree(h->d_defer); cudaFree(h->d_stage);
  cudaFree(h->d_block_counts); cudaFree(h->d_recs); cudaFree(h->d_recs_f); cudaFree(h->d_recs_g); cudaFree(h->d_samp_layers); cudaFree(h->d_samp_scratch);
  cudaFree(h->d_chg_bits);
  if (h->h_small_out) cudaFreeHost(h->h_small_out);
  if (h->h_err) cudaFreeHost(h->h_err);
  for (int g = 0; g < 2; ++g) if (h->chain_ev[g]) cudaEventDestroy(h->chain_ev[g]);
  artp_cnn::destroy(h->cnn);
  for (int i = 0; i < 6; ++i) if (h->ev[i]) cudaEventDestroy(h->ev[i]);
  delete h;
}

int artp_has_map(const artp_handle* hh) { return hh && reinterpret_cast<const Handle*>(hh)->has_map ? 1 : 0; }

int artp_set_mode(artp_handle* hh, int mode) {
  if (!hh || mode < 0 || mode > 1) return ARTP_E_INVALID;
  reinterpret_cast<Handle*>(hh)->mode = mode;
  return ARTP_OK;
}

int artp_set_timing(artp_handle* hh, int enable) {
  if (!hh) return ARTP_E_INVALID;
  Handle* h = reinterpret_cast<Handle*>(hh);
  std::lock_guard<std::recursive_mutex> lk(h->mtx);
  CU_TRY(h, cudaSetDevice(h->device));
  if (enable && !h->ev[0]) for (int i = 0; i < 6; ++i) CU_TRY(h, cudaEventCreate(&h->ev[i]));
  h->timing = enable ? 1 : 0;
  h->ev_valid = false;
  return ARTP_OK;
}

int artp_get_last_timing(artp_handle* hh, float* ms3) {
  if (!hh || !ms3) return ARTP_E_INVALID;
  Handle* h = reinterpret_cast<Handle*>(hh);
  std::lock_guard<std::recursive_mutex> lk(h->mtx);
  if (!h->timing || !h->ev_valid) { h->err = "timing not enabled or no call recorded"; return ARTP_E_INVALID; }
  CU_TRY(h, cudaSetDevice(h->device));
  CU_TRY(h, cudaEventSynchronize(h->ev[5]));
  CU_TRY(h, cudaEventElapsedTime(ms3 + 0, h->ev[0], h->ev[1]));   // classify
  CU_TRY(h, cudaEventElapsedTime(ms3 + 1, h->ev[1], h->ev[4]));   // box stages: warp + reach vertex + reach plane
  CU_TRY(h, cudaEventElapsedTime(ms3 + 2, h->ev[4], h->ev[5]));   // plane grouping
  return ARTP_OK;
}

int artp_get_last_stage_timing(artp_handle* hh, float* ms5) {
  if (!hh || !ms5) return ARTP_E_INVALID;
  Handle* h = reinterpret_cast<Handle*>(hh);
  std::lock_guard<std::recursive_mutex> lk(h->mtx);
  if (!h->timing || !h->ev_valid) { h->err = "timing not enabled or no call recorded"; return ARTP_E_INVALID; }
  CU_TRY(h, cudaSetDevice(h->device));
  CU_TRY(h, cudaEventSynchronize(h->ev[5]));
  for (int i = 0; i < 5; ++i) CU_TRY(h, cudaEventElapsedTime(ms5 + i, h->ev[i], h->ev[i + 1]));
  return ARTP_OK;
}

// Pinned host memory for the adapter's staging buffers (the contiguous n x 7 state batch it gathers the OMPL states into,
// the verdict bytes): cudaHostAlloc'd pages reach the device at PCIe line rate (measured 55 GB/s on the B200 boxes, where
// memory pinned after the fact -- cudaHostRegister, torch's pin_memory -- reached 17-25 GB/s; profiles/pcie_probe.cu).
void* artp_host_alloc(size_t bytes) {
  void* p = nullptr;
  if (bytes == 0 || cudaHostAlloc(&p, bytes, cudaHostAllocPortable) != cudaSuccess) return nullptr;
  return p;
}
void artp_host_free(void* p) { if (p) cudaFreeHost(p); }

int artp_poll_error(artp_handle* hh) {
  if (!hh) return ARTP_E_INVALID;
  Handle* h = reinterpret_cast<Handle*>(hh);
  std::lock_guard<std::recursive_mutex> lk(h->mtx);
  return take_sticky_error(h);
}

int artp_debug_set_group_capacity(artp_handle* hh, int max_triangles) {
  if (!hh || max_triangles < 0) return ARTP_E_INVALID;
  Handle* h = reinterpret_cast<Handle*>(hh);
  std::lock_guard<std::recursive_mutex> lk(h->mtx);
  h->tcap_override = max_triangles;   // takes effect at the next artp_set_map
  return ARTP_OK;
}

int artp_get_stats(artp_handle* hh, artp_stats* out) {
  if (!hh || !out) return ARTP_E_INVALID;
  Handle* h = reinterpret_cast<Handle*>(hh);
  std::lock_guard<std::recursive_mutex> lk(h->mtx);
  CU_TRY(h, cudaSetDevice(h->device));
  uint32_t ctr[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  CU_TRY(h, cudaMemcpy(ctr, h->d_ctr, sizeof(ctr), cudaMemcpyDeviceToHost));   // synchronises the device
  h->stats.last_deferred = ctr[1];
  uint32_t cg = 0;
  CU_TRY(h, cudaMemcpy(&cg, h->d_ctr + 8, sizeof(cg), cudaMemcpyDeviceToHost));
  h->stats.last_queued_boxes = ctr[3] + ctr[4] + cg;
  h->stats.last_queued_warp_stage = ctr[3];
  h->stats.last_queued_reach_stage = ctr[4];
  h->stats.last_reach_plane_stage = cg;
  if (h->deferred_unread) { h->stats.poses_deferred += ctr[1]; h->deferred_unread = false; }
  *out = h->stats;
  return take_sticky_error(h);
}

int artp_set_map(artp_handle* hh, const float* elevation, const float* elevation_masked, int rows, int cols, double res,
                 double cx, double cy) {
  return artp_set_map_window(hh, elevation, elevation_masked, rows, cols, res, cx, cy, 0, rows);
}

// Spatial shard of a map (SURVEY 8e): this handle holds only rows [row0, row0 + nrows) of the rows x cols layers --
// its slab plus the halo the caller chose -- but keeps the geometry of the FULL map (sample spacing L / (N - 1), vertex
// coordinates, isInside), so every verdict is bit-identical to a handle holding the whole map. The device pointers
// of the layer / range tables are shifted by -row0, so the kernels keep indexing with global vertex indices.
int artp_set_map_window(artp_handle* hh, const float* elevation, const float* elevation_masked, int rows, int cols, double res,
                        double cx, double cy, int row0, int nrows) {
  if (!hh) return ARTP_E_INVALID;
  Handle* h = reinterpret_cast<Handle*>(hh);
  std::lock_guard<std::recursive_mutex> lk(h->mtx);
  if (!elevation || !elevation_masked || rows < 2 || cols < 2 || !(res > 0)) { h->err = "bad map arguments"; return ARTP_E_INVALID; }
  if (row0 < 0 || nrows < 2 || row0 + nrows > rows || (row0 & 3)) {
    h->err = "bad map window (row0 must be a multiple of 4, 0 <= row0, row0 + nrows <= rows, nrows >= 2)"; return ARTP_E_INVALID;
  }
  CU_TRY(h, cudaSetDevice(h->device));
  const size_t ncell = (size_t)nrows * cols;
  // geometry exactly as dxHeightfieldData::SetData computes it in fp32 (heightfield.cpp:130-169)
  const double Lx = rows * res, Ly = cols * res;   // grid_map: length = size * resolution
  artp::Field f;
  f.nx = rows; f.nz = cols;
  f.W = (float)Lx; f.D = (float)Ly;
  f.hW = f.W / 2.0f; f.hD = f.D / 2.0f;
  f.sW = f.W / (f.nx - 1.0f);
  f.sD = f.D / (f.nz - 1.0f);
  f.asp = f.sD / f.sW;
  f.iW = 1.0f / f.sW;
  f.iD = 1.0f / f.sD;
  f.px = (float)cx; f.py = (float)cy;
  // K2 shared-memory plane store: bound the zone of either box by its half-diagonal; same bound -> table levels
  int tcap = 0, kmax[2] = {0, 0};
  for (int k = 0; k < 2; ++k) {
    const float* sd = h->chk.side[k];
    const double r = 0.5 * std::sqrt((double)sd[0] * sd[0] + (double)sd[1] * sd[1] + (double)sd[2] * sd[2]);
    const int nxm = std::min(rows, (int)std::ceil(2.0 * r * f.iW) + 4), nzm = std::min(cols, (int)std::ceil(2.0 * r * f.iD) + 4);
    tcap = std::max(tcap, 2 * (nxm - 1) * (nzm - 1));
    int kk = 0;
    while ((2 << kk) <= std::min(nxm, nzm) && kk < artp::kMaxLevel) ++kk;   // floor(log2(min dim bound))
    kmax[k] = kk;
  }
  if (h->tcap_override > 0) tcap = std::min(tcap, h->tcap_override);   // test hook: force the overflow path
  tcap = (tcap + 3) & ~3;
  const int smem = tcap * 21 + 64;
  if (smem > 200 * 1024) {
    h->err = "box/map resolution combination exceeds the plane-grouping kernel's shared-memory store";
    return ARTP_E_LIMIT;
  }
  CU_TRY(h, cudaFuncSetAttribute(artp::box_items_block_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
  int per_sm = 0;
  CU_TRY(h, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, artp::box_items_block_kernel, artp::kBlockStageThreads, smem));
  h->k2_smem = smem; h->k2_tcap = tcap; h->k2_grid = h->sm_count * std::max(per_sm, 1);
  // upload (the previous map may still be in use by asynchronous calls on the caller's streams)
  CU_TRY(h, cudaDeviceSynchronize());
  h->chain_busy[0] = h->chain_busy[1] = false;
  const int pitch = (nrows + 3) & ~3;
  const size_t npad = (size_t)pitch * cols;
  if (h->win_rows != nrows || h->cols != cols) {
    for (int k = 0; k < 2; ++k) {
      cudaFree(h->d_H[k]); h->d_H[k] = nullptr;
      for (int l = 0; l <= artp::kMaxLevel; ++l) { cudaFree(h->d_T[k][l]); cudaFree(h->d_NF[k][l]); h->d_T[k][l] = nullptr; h->d_NF[k][l] = nullptr; }
      CU_TRY(h, cudaMalloc(&h->d_H[k], npad * sizeof(float)));
    }
  }
  for (int k = 0; k < 2; ++k)
    for (int l = 1; l <= kmax[k]; ++l)
      if (!h->d_T[k][l]) {
        CU_TRY(h, cudaMalloc(&h->d_T[k][l], npad * sizeof(float2)));
        CU_TRY(h, cudaMalloc(&h->d_NF[k][l], ((npad + 15) / 16) * sizeof(uint32_t)));
      }
  int rc = ensure_stage(h, ncell * sizeof(float));
  if (rc) return rc;
  const float* src[2] = {elevation, elevation_masked};
  // plane tables (temporary): 4 slots per cell = load factor 0.5 for the 2 triangles of a cell
  size_t cap = 1;
  while (cap < 4 * ncell) cap <<= 1;
  PlaneSlot* d_tab = nullptr;
  unsigned char* d_merge = nullptr;   // [0, npad): mergeable cells; [npad, 3 npad): two byte-flag levels (ping-pong while building)
  CU_TRY(h, cudaMalloc(&d_tab, cap * sizeof(PlaneSlot)));
  if (cudaMalloc(&d_merge, 3 * npad) != cudaSuccess) { cudaFree(d_tab); h->err = "cudaMalloc (plane tables)"; return ARTP_E_CUDA; }
  for (int k = 0; k < 2; ++k) {
    CU_TRY(h, cudaMemcpyAsync(h->d_stage, src[k], ncell * sizeof(float), cudaMemcpyHostToDevice, h->stream));
    reverse_columns_kernel<<<h->sm_count * 4, 256, 0, h->stream>>>((const float*)h->d_stage, h->d_H[k], nrows, cols, pitch);
    CU_TRY(h, cudaGetLastError());
    artp::Field fk = f;                     // local storage, global geometry: cell x of the window is global cell x + row0
    fk.H = h->d_H[k]; fk.pitch = pitch; fk.nx = nrows;
    plane_table_clear_kernel<<<h->sm_count * 8, 256, 0, h->stream>>>(d_tab, cap);
    CU_TRY(h, cudaMemsetAsync(d_merge, 0, npad, h->stream));
    plane_table_insert_kernel<<<h->sm_count * 8, 256, 0, h->stream>>>(fk, row0, d_tab, (uint32_t)(cap - 1));
    plane_table_query_kernel<<<h->sm_count * 8, 256, 0, h->stream>>>(fk, row0, d_tab, (uint32_t)(cap - 1), d_merge);
    CU_TRY(h, cudaGetLastError());
    h->stats.kernel_launches += 4;
    for (int l = 1; l <= kmax[k]; ++l) {
      unsigned char* nf_prev = d_merge + npad * (size_t)(1 + ((l - 1) & 1));
      unsigned char* nf_cur = d_merge + npad * (size_t)(1 + (l & 1));
      build_level_kernel<<<h->sm_count * 4, 256, 0, h->stream>>>(h->d_H[k], l > 1 ? h->d_T[k][l - 1] : nullptr,
                                                                  l > 1 ? nf_prev : nullptr, d_merge, h->d_T[k][l], nf_cur, nrows,
                                                                  cols, pitch, 1 << (l - 1));
      pack_flags_kernel<<<h->sm_count * 4, 256, 0, h->stream>>>(nf_cur, npad, h->d_NF[k][l]);
      CU_TRY(h, cudaGetLastError());
      h->stats.kernel_launches += 2;
    }
  }
  CU_TRY(h, cudaStreamSynchronize(h->stream));
  cudaFree(d_tab); cudaFree(d_merge);
  h->rows = rows; h->cols = cols; h->pitch = pitch; h->win_row0 = row0; h->win_rows = nrows;
  f.pitch = pitch;
  f.x_lo = row0; f.x_hi = row0 + nrows - 1;
  for (int k = 0; k < 2; ++k) {
    f.H = h->d_H[k] - row0;                 // indexed with GLOBAL vertex indices x in [x_lo, x_hi]
    f.kmax = kmax[k];
    for (int l = 0; l <= artp::kMaxLevel; ++l) {
      f.T[l] = (l >= 1 && l <= kmax[k]) ? h->d_T[k][l] - row0 : nullptr;
      f.NF[l] = (l >= 1 && l <= kmax[k]) ? h->d_NF[k][l] : nullptr;   // bit-packed: indexed with LOCAL entry numbers, see below
    }
    h->chk.f[k] = f;
  }
  h->chk.err_word = h->d_err;
  h->chk.Lx = Lx; h->chk.Ly = Ly; h->chk.cx = cx; h->chk.cy = cy;
  h->chk.cell_margin = 0.02f + 2e-6f * (float)std::max(rows, cols);
  // Stage B tiles (artp_tiles.cuh): a zone spans at most ceil(2 r / s) + 3 vertices per axis (r = box half-diagonal);
  // + 3 columns because the tile starts at x0 & ~3; width rounded up to a multiple of 4 floats (16-byte rows).
  {
    typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                      const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                      CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres) != cudaSuccess || !fn) {
      h->err = "cuTensorMapEncodeTiled not available from the driver"; return ARTP_E_CUDA;
    }
    h->chk.reach_tw = 0; h->chk.reach_th = 0;
    for (int q = 0; q < 2; ++q) {          // 0: big tiles (torso box bound), 1: small tiles (reach box bound)
      const float* sd = h->chk.side[q];
      const double r = 0.5 * std::sqrt((double)sd[0] * sd[0] + (double)sd[1] * sd[1] + (double)sd[2] * sd[2]);
      int tw = ((int)std::ceil(2.0 * r * f.iW) + 3 + 3 + 3) & ~3, th = (int)std::ceil(2.0 * r * f.iD) + 3;
      tw = std::min(tw, 256); th = std::min(th, 256);
      artp::TileCfg tc;
      tc.tw = tw; tc.th = th; tc.bytes = (uint32_t)tw * th * 4; tc.stride = (tc.bytes + 127u) & ~127u;
      // big tiles: one slot per warp (three 8-warp CTAs per SM hide the copy latency better than a second 7 KB slot);
      // small tiles: two slots, the next box's tile is in flight while this one is decided
      tc.slots = (tc.stride > 2048) ? 1 : 2;
      int wpc = 8;
      while (wpc > 1 && (size_t)wpc * tc.slots * tc.stride + 128 > 72 * 1024) wpc >>= 1;
      if ((size_t)wpc * tc.slots * tc.stride + 128 > 200 * 1024) {
        if (q == 1) continue;              // no reach-box queue: everything takes the big-tile queue
        // boxes this large relative to the cells: tiles capped, oversized zones go to the grouping stage
        tc.tw = 64; tc.th = 64; tc.bytes = 64 * 64 * 4; tc.stride = tc.bytes; tc.slots = 1; wpc = 4;
      }
      const cuuint64_t gdim[2] = {(cuuint64_t)pitch, (cuuint64_t)cols};
      const cuuint64_t gstr[1] = {(cuuint64_t)pitch * sizeof(float)};
      const cuuint32_t box[2] = {(cuuint32_t)tc.tw, (cuuint32_t)tc.th};
      const cuuint32_t one[2] = {1, 1};
      for (int layer = 0; layer < 2; ++layer) {
        const CUresult cr = reinterpret_cast<EncodeTiledFn>(fn)(&h->tile_map[q][layer], CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, h->d_H[layer], gdim,
                                                                gstr, box, one, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
                                                                CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (cr != CUDA_SUCCESS) { h->err = "cuTensorMapEncodeTiled failed (" + std::to_string((int)cr) + ")"; return ARTP_E_CUDA; }
      }
      tc.x_off = row0;
      h->tile_cfg[q] = tc; h->tile_warps[q] = wpc;
      h->tile_smem[q] = (int)((size_t)wpc * tc.slots * tc.stride + 128);
      if (q == 1) { h->chk.reach_tw = tc.tw; h->chk.reach_th = tc.th; }
    }
    h->group_grid = 0;
    if (h->chk.reach_tw && h->tile_cfg[1].tw <= 127 && h->tile_cfg[1].th <= 255) {   // task packing: 7 + 8 bits of cell coordinates
      const int gsm = artp::kMaxTileWarps * 8 * (int)h->tile_cfg[1].stride + 128;
      if (gsm <= 160 * 1024 && !std::getenv("ARTP_NO_GROUPS")) {   // ARTP_NO_GROUPS: every reach box takes the one-warp-per-box queue
        CU_TRY(h, cudaFuncSetAttribute(artp::reach_groups_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, gsm));
        int ps = 0;
        CU_TRY(h, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ps, artp::reach_groups_kernel, artp::kMaxTileWarps * 32, gsm));
        h->group_grid = h->sm_count * std::max(ps, 1);
        h->group_smem = gsm;
      }
    }
    const int smax = std::max(h->tile_smem[0], h->tile_smem[1]);
    CU_TRY(h, cudaFuncSetAttribute(artp::box_tiles_warp_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smax));
    for (int q = 0; q < 2; ++q) {
      int ps = 0;
      CU_TRY(h, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ps, artp::box_tiles_warp_kernel, h->tile_warps[q] * 32, h->tile_smem[q]));
      h->tile_grid[q] = h->sm_count * std::max(ps, 1);
    }
  }
  h->has_map = true;
  h->has_sampler = false;      // its layers belong to the previous map
  h->has_device_normals = false;
  h->has_device_cdf = false;
  return ARTP_OK;
}

int artp_check_poses_device(artp_handle* hh, const double* d_states, size_t n, uint8_t* d_valid, void* stream) {
  if (!hh) return ARTP_E_INVALID;
  Handle* h = reinterpret_cast<Handle*>(hh);
  std::lock_guard<std::recursive_mutex> lk(h->mtx);
  int rc = check_common(h, n);
  if (rc) return rc;
  if (n == 0) return ARTP_OK;
  if (!d_states || !d_valid) { h->err = "null buffer"; return ARTP_E_INVALID; }
  CU_TRY(h, cudaSetDevice(h->device));
  artp::Work w;
  w.s1 = nullptr; w.s2 = d_states; w.s2f = nullptr; w.valid = d_valid; w.item_base = 0; w.n_items = (uint32_t)n; w.steps = 0; w.edge_mode = 0;
  ChainScope cs(h, 0, (cudaStream_t)stream);
  if (cs.rc) return cs.rc;
  rc = run_items(h, w, (cudaStream_t)stream);
  if (rc) return rc;
  h->stats.poses_checked += n;
  return ARTP_OK;
}

// Latency path for n <= kSmallBatch host states (doubles): one launch, verdicts through mapped host memory.
static int check_poses_small(Handle* h, const artp::SmallBatch& sb, size_t n, uint8_t* valid, int steps = -1) {
  if (!h->h_small_out) {
    CU_TRY(h, cudaHostAlloc((void**)&h->h_small_out, 64, cudaHostAllocMapped));
    CU_TRY(h, cudaFuncSetAttribute(artp::pose_small_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
  }
  uint8_t* d_out = nullptr;
  CU_TRY(h, cudaHostGetDevicePointer((void**)&d_out, h->h_small_out, 0));
  { int rc0 = chain_begin(h, 0, h->stream); if (rc0) return rc0; }
  artp::pose_small_kernel<<<(unsigned)n, 256, h->k2_smem, h->stream>>>(h->chk, sb, d_out, h->k2_tcap, h->d_err,
                                                                        h->mode == 1, steps);
  CU_TRY(h, cudaGetLastError());
  CU_TRY(h, cudaStreamSynchronize(h->stream));
  if (steps < 0) {
    std::memcpy(valid, h->h_small_out, n);
  } else {   // n = edges * (steps + 1) state verdicts -> one flag per edge
    const size_t per = (size_t)steps + 1;
    for (size_t e = 0; e < n / per; ++e) {
      uint8_t ok = 1;
      for (size_t j = 0; j < per; ++j) ok &= h->h_small_out[e * per + j];
      valid[e] = ok;
    }
  }
  h->stats.kernel_launches += 1;
  h->stats.last_launches = 1;
  h->stats.poses_checked += n;
  h->ev_valid = false;
  if (h->chain_stream[0] == h->stream || !h->chain_busy[0]) h->chain_busy[0] = false;   // everything of this group has completed
  return take_sticky_error(h);
}

int artp_check_poses(artp_handle* hh, const double* states, size_t n, uint8_t* valid) {
  if (!hh) return ARTP_E_INVALID;
  Handle* h = reinterpret_cast<Handle*>(hh);
  std::lock_guard<std::recursive_mutex> lk(h->mtx);
  int rc = check_common(h, n);
  if (rc) return rc;
  if (n == 0) return ARTP_OK;
  if (!states || !valid) { h->err = "null buffer"; return ARTP_E_INVALID; }
  CU_TRY(h, cudaSetDevice(h->device));
  if (n <= (size_t)artp::kSmallBatch && !h->timing) {
    artp::SmallBatch sb;
    std::memcpy(sb.s, states, n * 7 * sizeof(double));
    return check_poses_small(h, sb, n, valid);
  }
  const size_t in_bytes = n * 7 * sizeof(double), out_off = (in_bytes + 255) & ~(size_t)255;
  rc = ensure_stage(h, out_off + n);
  if (rc) return rc;
  double* d_states = (double*)h->d_stage;
  uint8_t* d_valid = (uint8_t*)h->d_stage + out_off;
  // the H2D copy of slice i+1 (copy stream) overlaps the kernels of slice i (compute stream); results return once
  artp::Work w;
  w.s1 = nullptr; w.s2 = d_states; w.s2f = nullptr; w.valid = d_valid; w.item_base = 0; w.n_items = (uint32_t)n;
  w.steps = 0; w.edge_mode = 0;
  HostFeed feed{(const char*)states, (char*)d_states, 7 * sizeof(double), h->slice_items_f64, {0.06f, 0.14f, 0.20f, 0.20f, 0.20f, 0.20f, 0.f, 0.f}};
  rc = chain_begin(h, 0, h->stream);
  if (rc) return rc;
  rc = run_items(h, w, h->stream, &feed);
  if (rc) return rc;
  CU_TRY(h, cudaMemcpyAsync(valid, d_valid, n, cudaMemcpyDeviceToHost, h->stream));
  CU_TRY(h, cudaStreamSynchronize(h->stream));
  h->chain_busy[0] = false;
  h->stats.poses_checked += n;
  return take_sticky_error(h);
}

// float32 states: the caller has already applied the double -> float cast that Pose3FromSE3 (utils.h:25-38) performs
// first, so the result is identical to the double entry point while the H2D stream is 28 B/pose instead of 56.
int artp_check_poses_f32_device(artp_handle* hh, const float* d_states, size_t n, uint8_t* d_valid, void* stream) {
  if (!hh) return ARTP_E_INVALID;
  Handle* h = reinterpret_cast<Handle*>(hh);
  std::lock_guard<std::recursive_mutex> lk(h->mtx);
  int rc = check_common(h, n);
  if (rc) return rc;
  if (n == 0) return ARTP_OK;
  if (!d_states || !d_valid) { h->err = "null buffer"; return ARTP_E_INVALID; }
  CU_TRY(h, cudaSetDevice(h->device));
  artp::Work w;
  w.s1 = nullptr; w.s2 = nullptr; w.s2f = d_states; w.valid = d_valid; w.item_base = 0; w.n_items = (uint32_t)n; w.steps = 0;
  w.edge_mode = 0;
  ChainScope cs(h, 0, (cudaStream_t)stream);
  if (cs.rc) return cs.rc;
  rc = run_items(h, w, (cudaStream_t)stream);
  if (rc) return rc;
  h->stats.poses_checked += n;
  return ARTP_OK;
}

int artp_check_poses_f32(artp_handle* hh, const float* states, size_t n, uint8_t* valid) {
  if (!hh) return ARTP_E_INVALID;
  Handle* h = reinterpret_cast<Handle*>(hh);
  std::lock_guard<std::recursive_mutex> lk(h->mtx);
  int rc = check_common(h, n);
  if (rc) return rc;
  if (n == 0) return ARTP_OK;
  if (!states || !valid) { h->err = "null buffer"; return ARTP_E_INVALID; }
  CU_TRY(h, cudaSetDevice(h->device));
  if (n <= (size_t)artp::kSmallBatch && !h->timing) {
    artp::SmallBatch sb;
    for (size_t i = 0; i < n * 7; ++i) (&sb.s[0][0])[i] = (double)states[i];   // exact; cast back to float in the kernel
    return check_poses_small(h, sb, n, valid);
  }
  const size_t in_bytes = n * 7 * sizeof(float), out_off = (in_bytes + 255) & ~(size_t)255;
  rc = ensure_stage(h, out_off + n);
  if (rc) return rc;
  float* d_states = (float*)h->d_stage;
  uint8_t* d_valid = (uint8_t*)h->d_stage + out_off;
  artp::Work w;
  w.s1 = nullptr; w.s2 = nullptr; w.s2f = d_states; w.valid = d_valid; w.item_base = 0; w.n_items = (uint32_t)n;
  w.steps = 0; w.edge_mode = 0;
  HostFeed feed{(const char*)states, (char*)d_states, 7 * sizeof(float), h->slice_items_f32, {0.08f, 0.17f, 0.25f, 0.25f, 0.25f, 0.f, 0.f, 0.f}};
  rc = chain_begin(h, 0, h->stream);
  if (rc) return rc;
  rc = run_items(h, w, h->stream, &feed);
  if (rc) return rc;
  CU_TRY(h, cudaMemcpyAsync(valid, d_valid, n, cudaMemcpyDeviceToHost, h->stream));
  CU_TRY(h, cudaStreamSynchronize(h->stream));
  h->chain_busy[0] = false;
  h->stats.poses_checked += n;
  return take_sticky_error(h);
}

int artp_check_motions_device(artp_handle* hh, const double* d_s1, const double* d_s2, size_t n, int n_steps,
                              uint8_t* d_valid, void* stream) {
  if (!hh) return ARTP_E_INVALID;
  Handle* h = reinterpret_cast<Handle*>(hh);
  std::lock_guard<std::recursive_mutex> lk(h->mtx);
  if (n_steps < 0) { h->err = "n_steps < 0"; return ARTP_E_INVALID; }
  const size_t items = n * ((size_t)n_steps + 1);
  int rc = check_common(h, items);
  if (rc) return rc;
  if (n == 0) return ARTP_OK;
  if (!d_s1 || !d_s2 || !d_valid) { h->err = "null buffer"; return ARTP_E_INVALID; }
  CU_TRY(h, cudaSetDevice(h->device));
  cudaStream_t s = (cudaStream_t)stream;
  ChainScope cs(h, 0, s);
  if (cs.rc) return cs.rc;
  fill_u8_kernel<<<std::min<size_t>((n + 255) / 256, (size_t)h->sm_count * 8), 256, 0, s>>>(d_valid, n, 1);
  CU_TRY(h, cudaGetLastError());
  artp::Work w;
  w.s1 = d_s1; w.s2 = d_s2; w.s2f = nullptr; w.valid = d_valid; w.item_base = 0; w.n_items = (uint32_t)items; w.steps = n_steps; w.edge_mode = 1;
  rc = run_items(h, w, s);
  if (rc) return rc;
  h->stats.kernel_launches += 1;
  h->stats.last_launches += 1;
  h->stats.poses_checked += items;
  return ARTP_OK;
}

int artp_check_motions(artp_handle* hh, const double* s1, const double* s2, size_t n, int n_steps, uint8_t* valid) {
  if (!hh) return ARTP_E_INVALID;
  Handle* h = reinterpret_cast<Handle*>(hh);
  if (n > 0 && n_steps >= 0 && n * ((size_t)n_steps + 1) <= (size_t)artp::kSmallBatch && 2 * n <= (size_t)artp::kSmallBatch &&
      s1 && s2 && valid) {
    // latency path (a single checkMotion call): one fused launch, interpolation on the device as in the pipeline
    std::lock_guard<std::recursive_mutex> lk(h->mtx);
    if (h->has_map && !h->timing) {
      CU_TRY(h, cudaSetDevice(h->device));
      artp::SmallBatch sb;
      for (size_t e = 0; e < n; ++e) {
        std::memcpy(sb.s[2 * e], s1 + 7 * e, 7 * sizeof(double));
        std::memcpy(sb.s[2 * e + 1], s2 + 7 * e, 7 * sizeof(double));
      }
      return check_poses_small(h, sb, n * ((size_t)n_steps + 1), valid, n_steps);
    }
  }
  const size_t sb = n * 7 * sizeof(double), sb_al = (sb + 255) & ~(size_t)255;
  std::lock_guard<std::recursive_mutex> lk(h->mtx);   // held across stage -> launch -> D2H: d_stage is per handle
  if (!h->has_map) { h->err = "no map set"; return ARTP_E_NOMAP; }
  if (n == 0) return ARTP_OK;
  if (!s1 || !s2 || !valid) { h->err = "null buffer"; return ARTP_E_INVALID; }
  CU_TRY(h, cudaSetDevice(h->device));
  int rc = chain_begin(h, 0, h->stream);
  if (rc) return rc;
  rc = ensure_stage(h, 2 * sb_al + n);
  if (rc) return rc;
  CU_TRY(h, cudaMemcpyAsync(h->d_stage, s1, sb, cudaMemcpyHostToDevice, h->stream));
  CU_TRY(h, cudaMemcpyAsync((char*)h->d_stage + sb_al, s2, sb, cudaMemcpyHostToDevice, h->stream));
  uint8_t* d_valid = (uint8_t*)h->d_stage + 2 * sb_al;
  rc = artp_check_motions_device(hh, (const double*)h->d_stage, (const double*)((char*)h->d_stage + sb_al), n, n_steps,
                                 d_valid, h->stream);
  if (rc) return rc;
  CU_TRY(h, cudaMemcpyAsync(valid, d_valid, n, cudaMemcpyDeviceToHost, h->stream));
  CU_TRY(h, cudaStreamSynchronize(h->stream));
  h->chain_busy[0] = false;
  return take_sticky_error(h);
}

// valid_prefix[e] = number of leading 1s in item_valid[item_off[e] .. item_off[e+1])
__global__ void edge_prefix_kernel(const uint8_t* __restrict__ item_valid, const uint32_t* __restrict__ item_off, size_t n,
                                   int32_t* __restrict__ valid_prefix) {
  for (size_t e = blockIdx.x * (size_t)blockDim.x + threadIdx.x; e < n; e += (size_t)gridDim.x * blockDim.x) {
    const uint32_t o0 = item_off[e], o1 = item_off[e + 1];
    uint32_t k = o0;
    while (k < o1 && item_valid[k]) ++k;
    valid_prefix[e] = (int32_t)(k - o0);
  }
}

static int check_items_prefix(artp_handle* hh, const double* d_s1, const double* d_s2, size_t n, const uint32_t* d_item_off,
                              size_t total_items, uint8_t* d_item_valid, int32_t* d_valid_prefix, void* stream, int quotient);

int artp_check_edge_interiors_device(artp_handle* hh, const double* d_s1, const double* d_s2, size_t n,
                                     const uint32_t* d_item_off, size_t total_items, uint8_t* d_item_valid,
                                     int32_t* d_valid_prefix, void* stream) {
  return check_items_prefix(hh, d_s1, d_s2, n, d_item_off, total_items, d_item_valid, d_valid_prefix, stream, 0);
}

static int check_items_prefix(artp_handle* hh, const double* d_s1, const double* d_s2, size_t n, const uint32_t* d_item_off,
                              size_t total_items, uint8_t* d_item_valid, int32_t* d_valid_prefix, void* stream, int quotient) {
  if (!hh) return ARTP_E_INVALID;
  Handle* h = reinterpret_cast<Handle*>(hh);
  std::lock_guard<std::recursive_mutex> lk(h->mtx);
  int rc = check_common(h, total_items);
  if (rc) return rc;
  if (n == 0) return ARTP_OK;
  if (!d_s1 || !d_s2 || !d_item_off || !d_valid_prefix || (total_items && !d_item_valid)) {
    h->err = "null buffer"; return ARTP_E_INVALID;
  }
  if (n >= 0xFFFFFFFFull) { h->err = "too many edges"; return ARTP_E_INVALID; }
  CU_TRY(h, cudaSetDevice(h->device));
  cudaStream_t s = (cudaStream_t)stream;
  ChainScope cs(h, 0, s);
  if (cs.rc) return cs.rc;
  h->stats.last_launches = 0;
  if (total_items) {
    artp::Work w;
    w.s1 = d_s1; w.s2 = d_s2; w.s2f = nullptr; w.valid = d_item_valid; w.item_base = 0; w.n_items = (uint32_t)total_items;
    w.steps = 0; w.edge_mode = 0; w.item_off = d_item_off; w.n_edges = (uint32_t)n; w.quotient = quotient;
    rc = run_items(h, w, s);
    if (rc) return rc;
  }
  edge_prefix_kernel<<<std::min<size_t>((n + 255) / 256, (size_t)h->sm_count * 8), 256, 0, s>>>(d_item_valid, d_item_off, n,
                                                                                                  d_valid_prefix);
  CU_TRY(h, cudaGetLastError());
  h->stats.kernel_launches += 1;
  h->stats.last_launches += 1;
  h->stats.poses_checked += total_items;
  return ARTP_OK;
}

int artp_check_edge_interiors(artp_handle* hh, const double* s1, const double* s2, size_t n, const int32_t* n_interp,
                              double max_lateral, int32_t* valid_prefix) {
  if (!hh) return ARTP_E_INVALID;
  Handle* h = reinterpret_cast<Handle*>(hh);
  std::vector<uint32_t> off;
  size_t total = 0, sb_al = 0, ob_al = 0, pb_al = 0;
  std::lock_guard<std::recursive_mutex> lk(h->mtx);   // held across stage -> launch -> D2H
  {
    if (!h->has_map) { h->err = "no map set"; return ARTP_E_NOMAP; }
    if (n == 0) return ARTP_OK;
    if (!s1 || !s2 || !valid_prefix) { h->err = "null buffer"; return ARTP_E_INVALID; }
    if (!n_interp && !(max_lateral > 0.0)) { h->err = "n_interp == NULL needs max_lateral > 0"; return ARTP_E_INVALID; }
    off.resize(n + 1);
    for (size_t e = 0; e < n; ++e) {
      off[e] = (uint32_t)total;
      long long ne;
      if (n_interp) {
        ne = n_interp[e];
      } else {   // lateralDistance (utils.h:52-61) / max_lateral truncated like prm_motion_cost.cpp:341-343
        const double dx = s2[7 * e] - s1[7 * e], dy = s2[7 * e + 1] - s1[7 * e + 1];
        ne = (long long)(unsigned int)(std::sqrt(dx * dx + dy * dy) / max_lateral);
      }
      if (ne < 0) { h->err = "n_interp < 0"; return ARTP_E_INVALID; }
      total += (size_t)ne;
      if (total >= 0xFFFFFFFFull) { h->err = "too many interior states (>= 2^32)"; return ARTP_E_INVALID; }
    }
    off[n] = (uint32_t)total;
    const size_t sb = n * 7 * sizeof(double);
    sb_al = (sb + 255) & ~(size_t)255;
    ob_al = ((n + 1) * sizeof(uint32_t) + 255) & ~(size_t)255;
    pb_al = (n * sizeof(int32_t) + 255) & ~(size_t)255;
    CU_TRY(h, cudaSetDevice(h->device));
    int rc = chain_begin(h, 0, h->stream);
    if (rc) return rc;
    rc = ensure_stage(h, 2 * sb_al + ob_al + pb_al + total + 256);
    if (rc) return rc;
    char* base = (char*)h->d_stage;
    CU_TRY(h, cudaMemcpyAsync(base, s1, sb, cudaMemcpyHostToDevice, h->stream));
    CU_TRY(h, cudaMemcpyAsync(base + sb_al, s2, sb, cudaMemcpyHostToDevice, h->stream));
    CU_TRY(h, cudaMemcpyAsync(base + 2 * sb_al, off.data(), (n + 1) * sizeof(uint32_t), cudaMemcpyHostToDevice, h->stream));
  }
  char* base = (char*)h->d_stage;
  int32_t* d_prefix = (int32_t*)(base + 2 * sb_al + ob_al);
  int rc = artp_check_edge_interiors_device(hh, (const double*)base, (const double*)(base + sb_al), n,
                                            (const uint32_t*)(base + 2 * sb_al), total,
                                            (uint8_t*)(base + 2 * sb_al + ob_al + pb_al), d_prefix, h->stream);
  if (rc) return rc;
  CU_TRY(h, cudaMemcpyAsync(valid_prefix, d_prefix, n * sizeof(int32_t), cudaMemcpyDeviceToHost, h->stream));
  CU_TRY(h, cudaStreamSynchronize(h->stream));   // `off` must outlive its H2D copy: it does, we synchronise here
  h->chain_busy[0] = false;
  return take_sticky_error(h);
}

// ompl::base::CompoundStateSpace::validSegmentCount for SE3 = max over the R^3 and SO(3) sub-spaces of
// (unsigned)ceil(distance / (maximum extent * longest valid segment fraction)) (OMPL 1.4.2 StateSpace.cpp;
// RealVectorStateSpace: Euclidean distance, extent = |high - low|; SO3StateSpace: arc length acos(|q1.q2|) with
// the 1e-9 clamp, extent pi/2). Host arithmetic, doubles, like OMPL.
int artp_valid_segment_count(const artp_se3_space* sp, const double* s1, const double* s2, size_t n, int32_t* nd) {
  if (!sp || (n && (!s1 || !s2 || !nd))) return ARTP_E_INVALID;
  const double frac = sp->longest_valid_segment_fraction > 0 ? sp->longest_valid_segment_fraction : 0.01;
  double e2 = 0;
  for (int i = 0; i < 3; ++i) e2 += (sp->high[i] - sp->low[i]) * (sp->high[i] - sp->low[i]);
  const double seg_r3 = std::sqrt(e2) * frac, seg_so3 = 0.5 * 3.14159265358979323846 * frac;
  if (!(seg_r3 > 0)) return ARTP_E_INVALID;
  for (size_t i = 0; i < n; ++i) {
    const double* a = s1 + 7 * i;
    const double* b = s2 + 7 * i;
    const double dx = a[0] - b[0], dy = a[1] - b[1], dz = a[2] - b[2];
    const double d3 = std::sqrt(dx * dx + dy * dy + dz * dz);
    const double dq = std::fabs(a[3] * b[3] + a[4] * b[4] + a[5] * b[5] + a[6] * b[6]);
    const double ds = (dq > 1.0 - 1e-9) ? 0.0 : std::acos(dq);
    const unsigned n3 = (unsigned)std::ceil(d3 / seg_r3), ns = (unsigned)std::ceil(ds / seg_so3);
    nd[i] = (int32_t)std::max(n3, ns);
  }
  return ARTP_OK;
}

int artp_check_motions_segments(artp_handle* hh, const double* s1, const double* s2, size_t n, const int32_t* nd,
                                const artp_se3_space* sp, uint8_t* valid, double* last_valid_t) {
  if (!hh) return ARTP_E_INVALID;
  Handle* h = reinterpret_cast<Handle*>(hh);
  std::lock_guard<std::recursive_mutex> lk(h->mtx);   // held across stage -> launch -> D2H
  if (!h->has_map) { h->err = "no map set"; return ARTP_E_NOMAP; }
  if (n == 0) return ARTP_OK;
  if (!s1 || !s2 || !valid || (!nd && !sp)) { h->err = "null buffer (nd == NULL needs the space parameters)"; return ARTP_E_INVALID; }
  std::vector<int32_t> seg(n);
  if (nd) std::copy(nd, nd + n, seg.begin());
  else { const int rc = artp_valid_segment_count(sp, s1, s2, n, seg.data()); if (rc) { h->err = "bad SE3 space parameters"; return rc; } }
  std::vector<uint32_t> off(n + 1);
  size_t total = 0;
  for (size_t e = 0; e < n; ++e) {
    if (seg[e] < 0) { h->err = "segment count < 0"; return ARTP_E_INVALID; }
    if (seg[e] < 1) seg[e] = 1;                 // nd = 0 (identical states): only s2 is checked
    off[e] = (uint32_t)total;
    total += (size_t)seg[e];
    if (total >= 0xFFFFFFFFull) { h->err = "too many states (>= 2^32)"; return ARTP_E_INVALID; }
  }
  off[n] = (uint32_t)total;
  const size_t sb = n * 7 * sizeof(double), sb_al = (sb + 255) & ~(size_t)255;
  const size_t ob_al = ((n + 1) * sizeof(uint32_t) + 255) & ~(size_t)255, pb_al = (n * sizeof(int32_t) + 255) & ~(size_t)255;
  CU_TRY(h, cudaSetDevice(h->device));
  int rc = chain_begin(h, 0, h->stream);
  if (rc) return rc;
  rc = ensure_stage(h, 2 * sb_al + ob_al + pb_al + total + 256);
  if (rc) return rc;
  char* base = (char*)h->d_stage;
  CU_TRY(h, cudaMemcpyAsync(base, s1, sb, cudaMemcpyHostToDevice, h->stream));
  CU_TRY(h, cudaMemcpyAsync(base + sb_al, s2, sb, cudaMemcpyHostToDevice, h->stream));
  CU_TRY(h, cudaMemcpyAsync(base + 2 * sb_al, off.data(), (n + 1) * sizeof(uint32_t), cudaMemcpyHostToDevice, h->stream));
  int32_t* d_prefix = (int32_t*)(base + 2 * sb_al + ob_al);
  rc = check_items_prefix(hh, (const double*)base, (const double*)(base + sb_al), n, (const uint32_t*)(base + 2 * sb_al), total,
                          (uint8_t*)(base + 2 * sb_al + ob_al + pb_al), d_prefix, h->stream, 1);
  if (rc) return rc;
  std::vector<int32_t> prefix(n);
  CU_TRY(h, cudaMemcpyAsync(prefix.data(), d_prefix, n * sizeof(int32_t), cudaMemcpyDeviceToHost, h->stream));
  CU_TRY(h, cudaStreamSynchronize(h->stream));
  h->chain_busy[0] = false;
  for (size_t e = 0; e < n; ++e) {
    // DiscreteMotionValidator::checkMotion(s1, s2, lastValid): the first invalid state in the order j = 1 .. nd-1, s2
    // is state index p (0-based) => lastValid.second = p / nd  ((j-1)/nd for an interior state, (nd-1)/nd for s2)
    valid[e] = prefix[e] == seg[e] ? 1 : 0;
    if (last_valid_t) last_valid_t[e] = valid[e] ? 1.0 : (double)prefix[e] / (double)seg[e];
  }
  return take_sticky_error(h);
}

// Rows [tx, ty, tyaw, sx, sy, syaw] of the MotionCostFunc edge matrix from SE(3) states exactly as
// PRMMotionCostMaintainer::updateEdges / computeCostForVertexEdges fill them (prm_motion_cost.cpp:27-128): x, y cast
// double -> float by the assignment into the float matrix, yaw = getYawFromSO3 (utils.h:80-88: double atan2, float result).
__global__ void edge_matrix_kernel(const double* __restrict__ s_start, const double* __restrict__ s_target, size_t n,
                                   float* __restrict__ edges) {
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    const double* a = s_start + 7 * i;
    const double* b = s_target + 7 * i;
    float* o = edges + 6 * i;
    o[0] = (float)b[0]; o[1] = (float)b[1];
    o[2] = (float)atan2(2 * (b[6] * b[5] + b[3] * b[4]), 1 - 2 * (b[4] * b[4] + b[5] * b[5]));
    o[3] = (float)a[0]; o[4] = (float)a[1];
    o[5] = (float)atan2(2 * (a[6] * a[5] + a[3] * a[4]), 1 - 2 * (a[4] * a[4] + a[5] * a[5]));
  }
}
// getCost / isFeasible per row (motion_cost_objective.h:54-66); infeasible edges get +inf like updateEdges (:56-59)
__global__ void combine_cost_kernel(const float* __restrict__ cost3, size_t n, float we, float wt, float wr, float thr,
                                    double* __restrict__ cost, uint8_t* __restrict__ feasible) {
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    const float ce = cost3[3 * i], ct = cost3[3 * i + 1], cr = cost3[3 * i + 2];
    const bool ok = (double)cr <= (double)thr;
    feasible[i] = ok ? 1 : 0;
    cost[i] = ok ? (double)ce * (double)we + (double)ct * (double)wt + (double)cr * (double)wr : CUDART_INF;
  }
}

int artp_edge_matrix_from_states(const double* s_start, const double* s_target, size_t n, float* edges) {
  if (n && (!s_start || !s_target || !edges)) return ARTP_E_INVALID;
  for (size_t i = 0; i < n; ++i) {
    const double* a = s_start + 7 * i;
    const double* b = s_target + 7 * i;
    float* o = edges + 6 * i;
    o[0] = (float)b[0]; o[1] = (float)b[1];
    o[2] = (float)std::atan2(2 * (b[6] * b[5] + b[3] * b[4]), 1 - 2 * (b[4] * b[4] + b[5] * b[5]));
    o[3] = (float)a[0]; o[4] = (float)a[1];
    o[5] = (float)std::atan2(2 * (a[6] * a[5] + a[3] * a[4]), 1 - 2 * (a[4] * a[4] + a[5] * a[5]));
  }
  return ARTP_OK;
}

int artp_motion_cost_states(artp_handle* hh, const double* s_start, const double* s_target, size_t n, double* cost,
                            uint8_t* feasible, float* cost3) {
  if (!hh) return ARTP_E_INVALID;
  Handle* h = reinterpret_cast<Handle*>(hh);
  std::lock_guard<std::recursive_mutex> lk(h->mtx);   // held across stage -> launch -> D2H
  if (n == 0) return ARTP_OK;
  if (!s_start || !s_target || !cost || !feasible) { h->err = "null buffer"; return ARTP_E_INVALID; }
  CU_TRY(h, cudaSetDevice(h->device));
  const size_t sb = n * 7 * sizeof(double), sb_al = (sb + 255) & ~(size_t)255, eb_al = (n * 6 * sizeof(float) + 255) & ~(size_t)255,
               cb_al = (n * 3 * sizeof(float) + 255) & ~(size_t)255, db_al = (n * sizeof(double) + 255) & ~(size_t)255;
  int rc = chain_begin(h, 0, h->stream);
  if (rc) return rc;
  rc = ensure_stage(h, 2 * sb_al + eb_al + cb_al + db_al + n);
  if (rc) return rc;
  char* base = (char*)h->d_stage;
  float* d_edges = (float*)(base + 2 * sb_al);
  float* d_c3 = (float*)(base + 2 * sb_al + eb_al);
  double* d_cost = (double*)(base + 2 * sb_al + eb_al + cb_al);
  uint8_t* d_feas = (uint8_t*)(base + 2 * sb_al + eb_al + cb_al + db_al);
  CU_TRY(h, cudaMemcpyAsync(base, s_start, sb, cudaMemcpyHostToDevice, h->stream));
  CU_TRY(h, cudaMemcpyAsync(base + sb_al, s_target, sb, cudaMemcpyHostToDevice, h->stream));
  const unsigned grid = (unsigned)std::min<size_t>((n + 255) / 256, (size_t)h->sm_count * 8);
  edge_matrix_kernel<<<grid, 256, 0, h->stream>>>((const double*)base, (const double*)(base + sb_al), n, d_edges);
  CU_TRY(h, cudaGetLastError());
  rc = artp_cnn::motion_cost(h->cnn, d_edges, n, d_c3, h->stream, h->err);
  if (rc) return rc;
  combine_cost_kernel<<<grid, 256, 0, h->stream>>>(d_c3, n, h->p.cost_w_energy, h->p.cost_w_time, h->p.cost_w_risk, h->p.risk_threshold, d_cost,
                                                   d_feas);
  CU_TRY(h, cudaGetLastError());
  CU_TRY(h, cudaMemcpyAsync(cost, d_cost, n * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  CU_TRY(h, cudaMemcpyAsync(feasible, d_feas, n, cudaMemcpyDeviceToHost, h->stream));
  if (cost3) CU_TRY(h, cudaMemcpyAsync(cost3, d_c3, n * 3 * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
  CU_TRY(h, cudaStreamSynchronize(h->stream));
  h->chain_busy[0] = false;
  h->stats.kernel_launches += 3;
  h->stats.last_launches = 3;
  return ARTP_OK;
}

int artp_path_length_cost_device(artp_handle* hh, const double* d_s1, const double* d_s2, size_t n, double* d_cost,
                                 void* stream) {
  if (!hh) return ARTP_E_INVALID;
  Handle* h = reinterpret_cast<Handle*>(hh);
  std::lock_guard<std::recursive_mutex> lk(h->mtx);
  if (n == 0) return ARTP_OK;
  if (!d_s1 || !d_s2 || !d_cost) { h->err = "null buffer"; return ARTP_E_INVALID; }
  CU_TRY(h, cudaSetDevice(h->device));
  path_length_kernel<<<std::min<size_t>((n + 255) / 256, (size_t)h->sm_count * 8), 256, 0, (cudaStream_t)stream>>>(
      d_s1, d_s2, n, d_cost, h->p.use_directional_cost, h->p.max_lon_vel, h->p.max_lat_vel, h->p.max_ang_vel);
  CU_TRY(h, cudaGetLastError());
  h->stats.kernel_launches += 1;
  h->stats.last_launches = 1;
  return ARTP_OK;
}

int artp_path_length_cost(artp_handle* hh, const double* s1, const double* s2, size_t n, double* cost) {
  if (!hh) return ARTP_E_INVALID;
  Handle* h = reinterpret_cast<Handle*>(hh);
  const size_t sb = n * 7 * sizeof(double), sb_al = (sb + 255) & ~(size_t)255;
  std::lock_guard<std::recursive_mutex> lk(h->mtx);   // held across stage -> launch -> D2H
  if (n == 0) return ARTP_OK;
  if (!s1 || !s2 || !cost) { h->err = "null buffer"; return ARTP_E_INVALID; }
  CU_TRY(h, cudaSetDevice(h->device));
  int rc = chain_begin(h, 0, h->stream);
  if (rc) return rc;
  rc = ensure_stage(h, 2 * sb_al + n * sizeof(double));
  if (rc) return rc;
  CU_TRY(h, cudaMemcpyAsync(h->d_stage, s1, sb, cudaMemcpyHostToDevice, h->stream));
  CU_TRY(h, cudaMemcpyAsync((char*)h->d_stage + sb_al, s2, sb, cudaMemcpyHostToDevice, h->stream));
  double* d_cost = (double*)((char*)h->d_stage + 2 * sb_al);
  rc = artp_path_length_cost_device(hh, (const double*)h->d_stage, (const double*)((char*)h->d_stage + sb_al), n, d_cost,
                                    h->stream);
  if (rc) return rc;
  CU_TRY(h, cudaMemcpyAsync(cost, d_cost, n * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  CU_TRY(h, cudaStreamSynchronize(h->stream));
  h->chain_busy[0] = false;
  return ARTP_OK;
}

static int compact_valid_impl(Handle* h, const uint8_t* d_valid, size_t n, int64_t base, void* d_indices,
                              uint32_t* d_count, cudaStream_t s, bool bits = false, bool u32 = false) {
  if (n == 0) { CU_TRY(h, cudaMemsetAsync(d_count, 0, sizeof(uint32_t), s)); return ARTP_OK; }
  ChainScope cs(h, 1, s);
  if (cs.rc) return cs.rc;
  const size_t nb = (n + kCompactBlock - 1) / kCompactBlock;
  if (h->block_counts_cap < nb) {
    CU_TRY(h, cudaDeviceSynchronize());   // every stream that may still read the old buffer
    cudaFree(h->d_block_counts);
    h->d_block_counts = nullptr;
    CU_TRY(h, cudaMalloc(&h->d_block_counts, nb * sizeof(uint32_t)));
    h->block_counts_cap = nb;
  }
  if (bits) compact_count_kernel<true><<<(unsigned)nb, kCompactBlock, 0, s>>>(d_valid, n, h->d_block_counts);
  else compact_count_kernel<false><<<(unsigned)nb, kCompactBlock, 0, s>>>(d_valid, n, h->d_block_counts);
  compact_scan_kernel<<<1, 1024, 0, s>>>(h->d_block_counts, nb, d_count);
  if (bits) compact_scatter_kernel<true, int64_t><<<(unsigned)nb, kCompactBlock, 0, s>>>(d_valid, n, base, h->d_block_counts, (int64_t*)d_indices);
  else if (u32) compact_scatter_kernel<false, uint32_t><<<(unsigned)nb, kCompactBlock, 0, s>>>(d_valid, n, base, h->d_block_counts, (uint32_t*)d_indices);
  else compact_scatter_kernel<false, int64_t><<<(unsigned)nb, kCompactBlock, 0, s>>>(d_valid, n, base, h->d_block_counts, (int64_t*)d_indices);
  CU_TRY(h, cudaGetLastError());
  h->stats.kernel_launches += 3;
  h->stats.last_launches = 3;
  return ARTP_OK;
}

int artp_compact_valid_device(artp_handle* hh, const uint8_t* d_valid, size_t n, int64_t base, int64_t* d_indices,
                              uint32_t* d_count, void* stream) {
  if (!hh) return ARTP_E_INVALID;
  Handle* h = reinterpret_cast<Handle*>(hh);
  std::lock_guard<std::recursive_mutex> lk(h->mtx);
  if (!d_valid || !d_indices || !d_count) { h->err = "null buffer"; return ARTP_E_INVALID; }
  CU_TRY(h, cudaSetDevice(h->device));
  return compact_valid_impl(h, d_valid, n, base, d_indices, d_count, (cudaStream_t)stream);
}

int artp_compact_valid_u32_device(artp_handle* hh, const uint8_t* d_valid, size_t n, uint32_t base, uint32_t* d_indices,
                                  uint32_t* d_count, void* stream) {
  if (!hh) return ARTP_E_INVALID;
  Handle* h = reinterpret_cast<Handle*>(hh);
  std::lock_guard<std::recursive_mutex> lk(h->mtx);
  if (!d_valid || !d_indices || !d_count) { h->err = "null buffer"; return ARTP_E_INVALID; }
  if (n + (size_t)base > 0xFFFFFFFFull) { h->err = "indices do not fit 32 bits"; return ARTP_E_INVALID; }
  CU_TRY(h, cudaSetDevice(h->device));
  return compact_valid_impl(h, d_valid, n, (int64_t)base, d_indices, d_count, (cudaStream_t)stream, false, true);
}

// isValid for a shard + the bit-packed verdicts the multi-GPU exchange sends, in one call on one stream.
int artp_check_poses_bits_device(artp_handle* hh, const double* d_states, size_t n, uint8_t* d_valid, uint32_t* d_bits, void* stream) {
  if (!hh) return ARTP_E_INVALID;
  Handle* h = reinterpret_cast<Handle*>(hh);
  std::lock_guard<std::recursive_mutex> lk(h->mtx);
  int rc = artp_check_poses_device(hh, d_states, n, d_valid, stream);
  if (rc) return rc;
  return artp_pack_valid_bits_device(hh, d_valid, n, d_bits, stream);
}

int artp_pack_valid_bits_device(artp_handle* hh, const uint8_t* d_valid, size_t n, uint32_t* d_bits, void* stream) {
  if (!hh) return ARTP_E_INVALID;
  Handle* h = reinterpret_cast<Handle*>(hh);
  std::lock_guard<std::recursive_mutex> lk(h->mtx);
  if (n == 0) return ARTP_OK;
  if (!d_valid || !d_bits) { h->err = "null buffer"; return ARTP_E_INVALID; }
  CU_TRY(h, cudaSetDevice(h->device));
  const size_t words = (n + 31) / 32;
  pack_bits_kernel<<<(unsigned)std::min<size_t>((words * 32 + 255) / 256, (size_t)h->sm_count * 8), 256, 0,
                     (cudaStream_t)stream>>>(d_valid, n, d_bits);
  CU_TRY(h, cudaGetLastError());
  h->stats.kernel_launches += 1;
  h->stats.last_launches = 1;
  return ARTP_OK;
}

int artp_compact_bits_device(artp_handle* hh, const uint32_t* d_bits, size_t n, int64_t base, int64_t* d_indices,
                             uint32_t* d_count, void* stream) {
  if (!hh) return ARTP_E_INVALID;
  Handle* h = reinterpret_cast<Handle*>(hh);
  std::lock_guard<std::recursive_mutex> lk(h->mtx);
  if (!d_bits || !d_indices || !d_count) { h->err = "null buffer"; return ARTP_E_INVALID; }
  CU_TRY(h, cudaSetDevice(h->device));
  return compact_valid_impl(h, reinterpret_cast<const uint8_t*>(d_bits), n, base, d_indices, d_count, (cudaStream_t)stream, true);
}

// ---------------------------------------------------------------------------------------------------------------
// Sampler: SE3FromSE2Sampler::sampleUniform on the device (artp_sampler.cuh)
// ---------------------------------------------------------------------------------------------------------------
static int ensure_sampler_layers(Handle* h) {
  const size_t ncell = (size_t)h->rows * h->cols;
  const size_t need = (5 * ncell + (size_t)h->rows + 64) * sizeof(float);
  if (h->samp_layers_cap >= need) return ARTP_OK;
  CU_TRY(h, cudaStreamSynchronize(h->stream));
  cudaFree(h->d_samp_layers);
  h->d_samp_layers = nullptr; h->samp_layers_cap = 0;
  h->has_device_normals = false;
  h->has_device_cdf = false;
  CU_TRY(h, cudaMalloc(&h->d_samp_layers, need));
  h->samp_layers_cap = need;
  return ARTP_OK;
}

int artp_estimate_normals(artp_handle* hh, double estimation_radius, float* normal_x, float* normal_y, float* normal_z,
                          float* plane_fit_std_dev) {
  if (!hh) return ARTP_E_INVALID;
  Handle* h = reinterpret_cast<Handle*>(hh);
  std::lock_guard<std::recursive_mutex> lk(h->mtx);
  if (!h->has_map) { h->err = "no map set"; return ARTP_E_NOMAP; }
  if (h->win_rows != h->rows) { h->err = "not available on a map window (artp_set_map_window)"; return ARTP_E_INVALID; }
  if (!(estimation_radius >= 0.0)) { h->err = "estimation_radius < 0"; return ARTP_E_INVALID; }
  CU_TRY(h, cudaSetDevice(h->device));
  int rc = chain_begin(h, 0, h->stream);
  if (rc) return rc;
  rc = ensure_sampler_layers(h);
  if (rc) return rc;
  const size_t ncell = (size_t)h->rows * h->cols;
  const double res = h->chk.Lx / h->rows;
  float* base = h->d_samp_layers;
  const int r_cells = (int)(estimation_radius / res), r_diag = (int)(estimation_radius * 0.70710678118 / res);   // utils.cpp:226-227
  artp::estimate_normals_kernel<<<(unsigned)std::min<size_t>((ncell + 127) / 128, (size_t)h->sm_count * 32), 128, 0, h->stream>>>(
      h->d_H[0], h->pitch, h->rows, h->cols, res, h->chk.cx, h->chk.cy, r_cells, r_diag, base, base + ncell, base + 2 * ncell,
      base + 3 * ncell);
  CU_TRY(h, cudaGetLastError());
  float* dst[4] = {normal_x, normal_y, normal_z, plane_fit_std_dev};
  for (int k = 0; k < 4; ++k)
    if (dst[k]) CU_TRY(h, cudaMemcpyAsync(dst[k], base + k * ncell, ncell * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
  CU_TRY(h, cudaStreamSynchronize(h->stream));
  h->has_device_normals = true;
  h->has_sampler = false;          // the sampler must be (re)armed with artp_set_sampler
  h->stats.kernel_launches += 1;
  h->stats.last_launches = 1;
  return ARTP_OK;
}

int artp_compute_sample_cdf(artp_handle* hh, const float* sample_probability, float* cum_prob, float* cum_prob_rowwise) {
  if (!hh) return ARTP_E_INVALID;
  Handle* h = reinterpret_cast<Handle*>(hh);
  std::lock_guard<std::recursive_mutex> lk(h->mtx);
  if (!h->has_map) { h->err = "no map set"; return ARTP_E_NOMAP; }
  if (h->win_rows != h->rows) { h->err = "not available on a map window (artp_set_map_window)"; return ARTP_E_INVALID; }
  if (!sample_probability) { h->err = "null buffer"; return ARTP_E_INVALID; }
  CU_TRY(h, cudaSetDevice(h->device));
  int rc = chain_begin(h, 0, h->stream);
  if (rc) return rc;
  rc = ensure_sampler_layers(h);
  if (rc) return rc;
  const size_t ncell = (size_t)h->rows * h->cols;
  rc = ensure_stage(h, ncell * sizeof(float));
  if (rc) return rc;
  float* d_cum = h->d_samp_layers + 4 * ncell;
  float* d_row = h->d_samp_layers + 5 * ncell;
  CU_TRY(h, cudaMemcpyAsync(h->d_stage, sample_probability, ncell * sizeof(float), cudaMemcpyHostToDevice, h->stream));
  artp::cdf_rows_kernel<<<(h->rows + 63) / 64, 64, 0, h->stream>>>((const float*)h->d_stage, h->rows, h->cols, d_cum, d_row);
  artp::cdf_rowwise_kernel<<<1, 32, 0, h->stream>>>(d_row, h->rows);
  CU_TRY(h, cudaGetLastError());
  if (cum_prob) CU_TRY(h, cudaMemcpyAsync(cum_prob, d_cum, ncell * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
  if (cum_prob_rowwise)
    CU_TRY(h, cudaMemcpyAsync(cum_prob_rowwise, d_row, (size_t)h->rows * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
  CU_TRY(h, cudaStreamSynchronize(h->stream));
  h->has_device_cdf = true;
  h->has_sampler = false;          // the sampler must be (re)armed with artp_set_sampler
  h->stats.kernel_launches += 2;
  h->stats.last_launches = 2;
  return ARTP_OK;
}

int artp_set_sampler(artp_handle* hh, const artp_sampler_params* sp, const float* normal_x, const float* normal_y,
                     const float* normal_z, const float* plane_fit_std_dev, const float* cum_prob,
                     const float* cum_prob_rowwise) {
  if (!hh) return ARTP_E_INVALID;
  Handle* h = reinterpret_cast<Handle*>(hh);
  std::lock_guard<std::recursive_mutex> lk(h->mtx);
  if (!h->has_map) { h->err = "no map set"; return ARTP_E_NOMAP; }
  if (h->win_rows != h->rows) { h->err = "not available on a map window (artp_set_map_window)"; return ARTP_E_INVALID; }
  const bool host_normals = normal_x && normal_y && normal_z && plane_fit_std_dev;
  if (!sp) { h->err = "null sampler params"; return ARTP_E_INVALID; }
  if (!host_normals && (normal_x || normal_y || normal_z || plane_fit_std_dev)) {
    h->err = "pass all four normal / plane-fit layers or none"; return ARTP_E_INVALID;
  }
  if (!host_normals && !h->has_device_normals) {
    h->err = "no normal layers: pass them or call artp_estimate_normals after artp_set_map"; return ARTP_E_INVALID;
  }
  const bool host_cdf = cum_prob && cum_prob_rowwise;
  if (sp->sample_from_distribution && !host_cdf && !(h->has_device_cdf && !cum_prob && !cum_prob_rowwise)) {
    h->err = "sample_from_distribution needs the cum_prob layers (pass both, or call artp_compute_sample_cdf first)";
    return ARTP_E_INVALID;
  }
  if (!sp->sample_from_distribution && !(sp->high[0] > sp->low[0] && sp->high[1] > sp->low[1])) {
    h->err = "empty sampling bounds"; return ARTP_E_INVALID;
  }
  CU_TRY(h, cudaSetDevice(h->device));
  const size_t ncell = (size_t)h->rows * h->cols;
  {
    int rc = chain_begin(h, 0, h->stream);
    if (rc) return rc;
    rc = ensure_sampler_layers(h);
    if (rc) return rc;
  }
  float* base = h->d_samp_layers;
  if (host_normals) {
    const float* src[4] = {normal_x, normal_y, normal_z, plane_fit_std_dev};
    for (int k = 0; k < 4; ++k)
      CU_TRY(h, cudaMemcpyAsync(base + k * ncell, src[k], ncell * sizeof(float), cudaMemcpyHostToDevice, h->stream));
    h->has_device_normals = false;   // overwritten by the caller's layers
  }
  artp::SamplerDev& m = h->samp;
  m.elevation_rev = h->d_H[0]; m.pitch = h->pitch;
  m.normal_x = base; m.normal_y = base + ncell; m.normal_z = base + 2 * ncell; m.std_dev = base + 3 * ncell;
  m.cum_prob = nullptr; m.cum_row = nullptr;
  m.rows = h->rows; m.cols = h->cols;
  m.res = h->chk.Lx / h->rows; m.cx = h->chk.cx; m.cy = h->chk.cy;
  m.max_roll_pert = sp->max_roll_pert; m.max_pitch_pert = sp->max_pitch_pert;
  m.from_distribution = sp->sample_from_distribution ? 1 : 0;
  m.low[0] = sp->low[0]; m.low[1] = sp->low[1]; m.high[0] = sp->high[0]; m.high[1] = sp->high[1];
  m.reach_z = h->p.reach_z;
  if (m.from_distribution) {
    if (host_cdf) {
      CU_TRY(h, cudaMemcpyAsync(base + 4 * ncell, cum_prob, ncell * sizeof(float), cudaMemcpyHostToDevice, h->stream));
      CU_TRY(h, cudaMemcpyAsync(base + 5 * ncell, cum_prob_rowwise, (size_t)h->rows * sizeof(float), cudaMemcpyHostToDevice,
                                h->stream));
      h->has_device_cdf = false;   // overwritten by the caller's layers
    }
    m.cum_prob = base + 4 * ncell; m.cum_row = base + 5 * ncell;
    // the binary searches need monotone (or all-NaN) CDF rows: refuse anything else
    CU_TRY(h, cudaMemsetAsync(h->d_ctr + 7, 0, sizeof(uint32_t), h->stream));
    artp::validate_cdf_kernel<<<(h->rows + 127) / 128, 128, 0, h->stream>>>(m.cum_prob, h->rows, h->cols, (size_t)h->rows, 1,
                                                                             h->d_ctr + 7);
    artp::validate_cdf_kernel<<<1, 32, 0, h->stream>>>(m.cum_row, 1, h->rows, 1, 0, h->d_ctr + 7);
    CU_TRY(h, cudaGetLastError());
    uint32_t bad = 0;
    CU_TRY(h, cudaMemcpyAsync(&bad, h->d_ctr + 7, sizeof(uint32_t), cudaMemcpyDeviceToHost, h->stream));
    CU_TRY(h, cudaStreamSynchronize(h->stream));
    h->stats.kernel_launches += 2;
    if (bad) { h->err = "cum_prob layers are not cumulative distributions (rows must be non-decreasing or all NaN)"; return ARTP_E_INVALID; }
  } else {
    CU_TRY(h, cudaStreamSynchronize(h->stream));
  }
  h->has_sampler = true;
  return ARTP_OK;
}

static int sampler_ready(Handle* h) {
  if (!h->has_map) { h->err = "no map set"; return ARTP_E_NOMAP; }
  if (!h->has_sampler) { h->err = "no sampler layers set (artp_set_sampler after artp_set_map)"; return ARTP_E_NOMAP; }
  return ARTP_OK;
}

static inline unsigned grid_for(Handle* h, size_t n, int block) {
  return (unsigned)std::min<size_t>((n + block - 1) / block, (size_t)h->sm_count * 16);
}

int artp_sampler_uniforms(artp_handle* hh, uint64_t seed, uint64_t first_sample, size_t n, double* u) {
  if (!hh) return ARTP_E_INVALID;
  Handle* h = reinterpret_cast<Handle*>(hh);
  std::lock_guard<std::recursive_mutex> lk(h->mtx);
  if (n == 0) return ARTP_OK;
  if (!u) { h->err = "null buffer"; return ARTP_E_INVALID; }
  CU_TRY(h, cudaSetDevice(h->device));
  int rc = chain_begin(h, 0, h->stream);
  if (rc) return rc;
  rc = ensure_stage(h, n * 6 * sizeof(double));
  if (rc) return rc;
  artp::sampler_uniforms_kernel<<<grid_for(h, n, 256), 256, 0, h->stream>>>(seed, first_sample, n, (double*)h->d_stage);
  CU_TRY(h, cudaGetLastError());
  CU_TRY(h, cudaMemcpyAsync(u, h->d_stage, n * 6 * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  CU_TRY(h, cudaStreamSynchronize(h->stream));
  h->stats.kernel_launches += 1;
  return ARTP_OK;
}

int artp_sample_states_device(artp_handle* hh, const double* d_u, uint64_t seed, uint64_t first_sample, size_t n,
                              double* d_states, int32_t* d_rowcol, void* stream) {
  if (!hh) return ARTP_E_INVALID;
  Handle* h = reinterpret_cast<Handle*>(hh);
  std::lock_guard<std::recursive_mutex> lk(h->mtx);
  int rc = sampler_ready(h);
  if (rc) return rc;
  if (n == 0) return ARTP_OK;
  if (!d_states) { h->err = "null buffer"; return ARTP_E_INVALID; }
  CU_TRY(h, cudaSetDevice(h->device));
  artp::sample_states_kernel<<<grid_for(h, n, 128), 128, 0, (cudaStream_t)stream>>>(h->samp, d_u, seed, first_sample, n, d_states,
                                                                                   nullptr, d_rowcol);
  CU_TRY(h, cudaGetLastError());
  h->stats.kernel_launches += 1;
  h->stats.last_launches = 1;
  return ARTP_OK;
}

int artp_sample_states(artp_handle* hh, const double* u, uint64_t seed, uint64_t first_sample, size_t n, double* states,
                       int32_t* rowcol) {
  if (!hh) return ARTP_E_INVALID;
  Handle* h = reinterpret_cast<Handle*>(hh);
  const size_t ub = (n * 6 * sizeof(double) + 255) & ~(size_t)255, sb = (n * 7 * sizeof(double) + 255) & ~(size_t)255;
  std::lock_guard<std::recursive_mutex> lk(h->mtx);   // held across stage -> launch -> D2H
  int rc = sampler_ready(h);
  if (rc) return rc;
  if (n == 0) return ARTP_OK;
  if (!states) { h->err = "null buffer"; return ARTP_E_INVALID; }
  CU_TRY(h, cudaSetDevice(h->device));
  rc = chain_begin(h, 0, h->stream);
  if (rc) return rc;
  rc = ensure_stage(h, ub + sb + n * 2 * sizeof(int32_t));
  if (rc) return rc;
  if (u) CU_TRY(h, cudaMemcpyAsync(h->d_stage, u, n * 6 * sizeof(double), cudaMemcpyHostToDevice, h->stream));
  char* base = (char*)h->d_stage;
  rc = artp_sample_states_device(hh, u ? (const double*)base : nullptr, seed, first_sample, n, (double*)(base + ub),
                                 rowcol ? (int32_t*)(base + ub + sb) : nullptr, h->stream);
  if (rc) return rc;
  CU_TRY(h, cudaMemcpyAsync(states, base + ub, n * 7 * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  if (rowcol) CU_TRY(h, cudaMemcpyAsync(rowcol, base + ub + sb, n * 2 * sizeof(int32_t), cudaMemcpyDeviceToHost, h->stream));
  CU_TRY(h, cudaStreamSynchronize(h->stream));
  return ARTP_OK;
}

// running total += chunk count (device-side, stream ordered)
__global__ void add_count_kernel(uint32_t* total, const uint32_t* chunk) { *total += *chunk; }

// out + 7 * (*total) .. : ordered gather of this chunk's valid candidates behind the previous chunks'
__global__ void gather_chunk_kernel(const double* __restrict__ states, const int64_t* __restrict__ idx,
                                    const uint32_t* __restrict__ chunk_count, const uint32_t* __restrict__ total_before,
                                    size_t capacity, double* __restrict__ out) {
  const size_t before = *total_before;
  const size_t room = capacity > before ? capacity - before : 0;
  const size_t cc = *chunk_count;
  const size_t keep = cc < room ? cc : room;
  const size_t n = keep * 7;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    const size_t k = i / 7, c = i - k * 7;
    out[before * 7 + i] = states[(size_t)idx[k] * 7 + c];
  }
}

static constexpr size_t kSampleChunk = (size_t)1 << 21;

int artp_sample_valid_device(artp_handle* hh, uint64_t seed, uint64_t first_sample, size_t n_draw, double* d_states_out,
                             size_t capacity, uint32_t* d_count, void* stream) {
  if (!hh) return ARTP_E_INVALID;
  Handle* h = reinterpret_cast<Handle*>(hh);
  std::lock_guard<std::recursive_mutex> lk(h->mtx);
  int rc = sampler_ready(h);
  if (rc) return rc;
  if (!d_count || (capacity && !d_states_out)) { h->err = "null buffer"; return ARTP_E_INVALID; }
  CU_TRY(h, cudaSetDevice(h->device));
  cudaStream_t s = (cudaStream_t)stream;
  CU_TRY(h, cudaMemsetAsync(d_count, 0, sizeof(uint32_t), s));
  if (n_draw == 0) return ARTP_OK;
  ChainScope cs(h, 0, s);
  if (cs.rc) return cs.rc;
  const size_t chunk = std::min(n_draw, kSampleChunk);
  // scratch: states f64 | states f32 | indices | valid | chunk count
  const size_t o_f32 = chunk * 7 * sizeof(double), o_idx = o_f32 + ((chunk * 7 * sizeof(float) + 255) & ~(size_t)255),
               o_val = o_idx + chunk * sizeof(int64_t), o_cnt = o_val + ((chunk + 255) & ~(size_t)255), total = o_cnt + 256;
  if (h->samp_scratch_cap < total) {
    CU_TRY(h, cudaDeviceSynchronize());
    cudaFree(h->d_samp_scratch);
    h->d_samp_scratch = nullptr; h->samp_scratch_cap = 0;
    CU_TRY(h, cudaMalloc(&h->d_samp_scratch, total));
    h->samp_scratch_cap = total;
  }
  char* sc = (char*)h->d_samp_scratch;
  double* d_st = (double*)sc;
  float* d_sf = (float*)(sc + o_f32);
  int64_t* d_idx = (int64_t*)(sc + o_idx);
  uint8_t* d_val = (uint8_t*)(sc + o_val);
  uint32_t* d_cnt = (uint32_t*)(sc + o_cnt);
  uint32_t launches = 0;
  for (size_t done = 0; done < n_draw; done += chunk) {
    const size_t m = std::min(chunk, n_draw - done);
    artp::sample_states_kernel<<<grid_for(h, m, 128), 128, 0, s>>>(h->samp, nullptr, seed, first_sample + done, m, d_st, d_sf,
                                                                   nullptr);
    CU_TRY(h, cudaGetLastError());
    artp::Work w;
    w.s1 = nullptr; w.s2 = nullptr; w.s2f = d_sf; w.valid = d_val; w.item_base = 0; w.n_items = (uint32_t)m; w.steps = 0;
    w.edge_mode = 0;
    rc = run_items(h, w, s);
    if (rc) return rc;
    launches += h->stats.last_launches + 1;
    if (!h->samp.from_distribution) {   // rejected (outside-map) candidates carry NaN states
      artp::reject_nan_kernel<<<grid_for(h, m, 256), 256, 0, s>>>(d_st, m, d_val);
      launches += 1;
    }
    rc = compact_valid_impl(h, d_val, m, 0, d_idx, d_cnt, s);
    if (rc) return rc;
    gather_chunk_kernel<<<grid_for(h, m * 7, 256), 256, 0, s>>>(d_st, d_idx, d_cnt, d_count, capacity, d_states_out);
    add_count_kernel<<<1, 1, 0, s>>>(d_count, d_cnt);
    CU_TRY(h, cudaGetLastError());
    launches += 5;
    h->stats.kernel_launches += 3 + (h->samp.from_distribution ? 0 : 1);
    h->stats.poses_checked += m;
  }
  h->stats.last_launches = launches;
  return ARTP_OK;
}

int artp_sample_valid(artp_handle* hh, uint64_t seed, uint64_t first_sample, size_t n_draw, double* states, size_t capacity,
                      size_t* n_valid) {
  if (!hh) return ARTP_E_INVALID;
  Handle* h = reinterpret_cast<Handle*>(hh);
  const size_t cap = std::min(capacity, n_draw);
  std::lock_guard<std::recursive_mutex> lk(h->mtx);   // held across stage -> launch -> D2H
  int rc = sampler_ready(h);
  if (rc) return rc;
  if (!n_valid || (cap && !states)) { h->err = "null buffer"; return ARTP_E_INVALID; }
  CU_TRY(h, cudaSetDevice(h->device));
  rc = chain_begin(h, 0, h->stream);
  if (rc) return rc;
  rc = ensure_stage(h, cap * 7 * sizeof(double) + 256);
  if (rc) return rc;
  uint32_t* d_count = (uint32_t*)((char*)h->d_stage + cap * 7 * sizeof(double));
  rc = artp_sample_valid_device(hh, seed, first_sample, n_draw, (double*)h->d_stage, cap, d_count, h->stream);
  if (rc) return rc;
  uint32_t cnt = 0;
  CU_TRY(h, cudaMemcpyAsync(&cnt, d_count, sizeof(uint32_t), cudaMemcpyDeviceToHost, h->stream));
  CU_TRY(h, cudaStreamSynchronize(h->stream));
  const size_t keep = std::min<size_t>(cnt, cap);
  if (keep) {
    CU_TRY(h, cudaMemcpyAsync(states, h->d_stage, keep * 7 * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    CU_TRY(h, cudaStreamSynchronize(h->stream));
  }
  *n_valid = cnt;      // > capacity means the output was truncated to `capacity` states
  return ARTP_OK;
}

// cv::circle(kernel, (r, r), r, 255, FILLED) on a size x size zero image, r = size / 2 (utils.cpp:106-111): OpenCV's
// integer midpoint circle (imgproc/src/drawing.cpp, Circle()): for every step (dx, dy) of the octant walk the rows
// cy -+ dy get the span cx -+ dx and the rows cy -+ dx the span cx -+ dy, everything clipped to the image.
static artp::MorphKernel make_circular_kernel(int size) {
  artp::MorphKernel k;
  std::memset(&k, 0, sizeof(k));
  if (size <= 0) {   // empty element: cv::erode / cv::dilate fall back to the 3 x 3 box, anchor (1, 1)
    k.size = 3; k.anchor = 1;
    for (int r = 0; r < 3; ++r) { k.lo[r] = 0; k.hi[r] = 2; }
    return k;
  }
  k.size = size; k.anchor = size / 2;
  for (int r = 0; r < size; ++r) { k.lo[r] = 127; k.hi[r] = -1; }
  const int radius = size / 2, cx = radius, cy = radius;
  auto span = [&](int y, int x0, int x1) {
    if (y < 0 || y >= size) return;
    x0 = std::max(x0, 0); x1 = std::min(x1, size - 1);
    if (x0 > x1) return;
    k.lo[y] = (int8_t)std::min<int>(k.lo[y], x0); k.hi[y] = (int8_t)std::max<int>(k.hi[y], x1);
  };
  int err = 0, dx = radius, dy = 0, plus = 1, minus = (radius << 1) - 1;
  while (dx >= dy) {
    span(cy - dy, cx - dx, cx + dx); span(cy + dy, cx - dx, cx + dx);
    span(cy - dx, cx - dy, cx + dy); span(cy + dx, cx - dy, cx + dy);
    dy++; err += plus; plus += 2;
    const int mask = (err <= 0) - 1;
    err -= minus & mask; dx += mask; minus -= mask & 2;
  }
  return k;
}

int artp_debug_circular_kernel(int size, uint8_t* out) {   // test hook: the size x size element as 0 / 1 bytes (row-major)
  if (size > artp::kMaxMorph || !out) return ARTP_E_INVALID;
  const artp::MorphKernel k = make_circular_kernel(size);
  for (int r = 0; r < k.size; ++r) for (int c = 0; c < k.size; ++c) out[r * k.size + c] = (c >= k.lo[r] && c <= k.hi[r]) ? 1 : 0;
  return k.size;
}

int artp_process_basic(artp_handle* hh, const float* elevation, const float* traversability, const float* observed, int rows,
                       int cols, double res, const artp_basic_params* bp, float* elevation_masked, float* traversability_thresholded) {
  if (!hh) return ARTP_E_INVALID;
  Handle* h = reinterpret_cast<Handle*>(hh);
  std::lock_guard<std::recursive_mutex> lk(h->mtx);
  if (!elevation || !traversability || !bp || !elevation_masked || rows < 1 || cols < 1 || !(res > 0)) {
    h->err = "bad arguments"; return ARTP_E_INVALID;
  }
  if (bp->unknown_space_untraversable && !observed) { h->err = "unknown_space_untraversable needs the observed layer"; return ARTP_E_INVALID; }
  // basic.cpp:65-74: cell counts of the structuring elements
  const int foothold = (int)std::ceil(bp->foothold_size / res), margin = (int)std::ceil(2 * bp->foothold_margin / res),
            hole = (int)std::floor(bp->foothold_margin_max_hole_size / res),
            search = (int)std::ceil(2 * bp->foothold_margin_max_drop_search_radius / res);
  if (std::max(std::max(foothold, margin), std::max(hole, search)) > artp::kMaxMorph) {
    h->err = "structuring element larger than 64 cells"; return ARTP_E_LIMIT;
  }
  CU_TRY(h, cudaSetDevice(h->device));
  const size_t n = (size_t)rows * cols, lb = n * sizeof(float);
  int rc = chain_begin(h, 0, h->stream);
  if (rc) return rc;
  rc = ensure_stage(h, 9 * lb);
  if (rc) return rc;
  float* L = (float*)h->d_stage;   // 0 elev, 1 trav, 2 observed, 3 T0, 4 A, 5 B, 6 elev eroded, 7 elev dilated, 8 out
  cudaStream_t s = h->stream;
  CU_TRY(h, cudaMemcpyAsync(L, elevation, lb, cudaMemcpyHostToDevice, s));
  CU_TRY(h, cudaMemcpyAsync(L + n, traversability, lb, cudaMemcpyHostToDevice, s));
  if (observed) CU_TRY(h, cudaMemcpyAsync(L + 2 * n, observed, lb, cudaMemcpyHostToDevice, s));
  const unsigned grid = (unsigned)std::min<size_t>((n + 255) / 256, (size_t)h->sm_count * 16);
  auto morph = [&](bool dil, const float* src, float* dst, int size) {
    const artp::MorphKernel k = make_circular_kernel(size);
    if (dil) artp::morph_kernel<true><<<grid, 256, 0, s>>>(src, dst, rows, cols, k);
    else artp::morph_kernel<false><<<grid, 256, 0, s>>>(src, dst, rows, cols, k);
  };
  float *E = L, *T0 = L + 3 * n, *A = L + 4 * n, *B = L + 5 * n, *Elo = L + 6 * n, *Ehi = L + 7 * n, *O = L + 8 * n;
  artp::basic_threshold_kernel<<<grid, 256, 0, s>>>(L + n, L + 2 * n, bp->unknown_space_untraversable ? 1 : 0, bp->traversability_thres, n, T0);
  morph(true, T0, A, hole); morph(false, A, B, hole);                    // dilateAndErode: close holes (:72)
  morph(false, E, Elo, search);                                          // elevation - erode(elevation) (:75-77)
  morph(true, E, Ehi, margin);                                           // dilate(elevation) - elevation (:84)
  artp::basic_select_kernel<<<grid, 256, 0, s>>>(0, E, Elo, Ehi, T0, B, (float)bp->foothold_margin_max_drop, (float)bp->foothold_margin_min_step, n, A);
  morph(false, A, B, margin);                                            // erode by the safety margin (:90)
  artp::basic_select_kernel<<<grid, 256, 0, s>>>(1, E, Elo, Ehi, T0, B, (float)bp->foothold_margin_max_drop, (float)bp->foothold_margin_min_step, n, A);
  morph(false, A, B, foothold); morph(true, B, A, foothold);             // erodeAndDilate: remove small patches (:95)
  artp::basic_final_kernel<<<grid, 256, 0, s>>>(E, T0, A, n, B, O);
  CU_TRY(h, cudaGetLastError());
  CU_TRY(h, cudaMemcpyAsync(elevation_masked, O, lb, cudaMemcpyDeviceToHost, s));
  if (traversability_thresholded) CU_TRY(h, cudaMemcpyAsync(traversability_thresholded, B, lb, cudaMemcpyDeviceToHost, s));
  CU_TRY(h, cudaStreamSynchronize(s));
  h->chain_busy[0] = false;
  h->stats.kernel_launches += 11;
  h->stats.last_launches = 11;
  return ARTP_OK;
}

// ---------------------------------------------------------------------------------------------------------------
// Map change + roadmap reuse (artp_roadmap.cuh): processors::computeChange (change.cpp:9-51) and the per-vertex /
// per-edge questions of LazyPRMStarMinUpdateMaintainer::update (lazy_prm_star_min_update.cpp:18-91, 123-135)
// ---------------------------------------------------------------------------------------------------------------
// grid_map::boundPositionToRange for one coordinate: epsilon = 10 * DBL_EPSILON, times |p| when |p| > 1.
static void gm_bound(double* p, double L, double c) {
  const double vto = 0.5 * L;
  double s = (*p - c) + vto;
  double eps = 10.0 * 2.220446049250313080847e-16;
  if (std::fabs(*p) > 1.0) eps *= std::fabs(*p);
  if (s <= 0.0) s = eps;
  else if (s >= L) s = L - eps;
  *p = (s + c) - vto;
}

// grid_map::SubmapGeometry(map, position, length) (getSubmapInformation): corners clamped into the map, converted to
// indices; size = br - tl + 1; fails when the requested centre is outside the resulting submap (or a corner index is
// outside the map, which only rounding can cause).
static bool gm_submap(const artp_grid* m, double rx, double ry, double rlx, double rly, int start[2], int size[2]) {
  const double Lx = m->rows * m->res, Ly = m->cols * m->res;
  double tl[2] = {rx + 0.5 * rlx, ry + 0.5 * rly}, br[2] = {rx - 0.5 * rlx, ry - 0.5 * rly};
  gm_bound(&tl[0], Lx, m->cx); gm_bound(&tl[1], Ly, m->cy);
  gm_bound(&br[0], Lx, m->cx); gm_bound(&br[1], Ly, m->cy);
  int ti, tj, bi, bj;
  if (!artp::grid_index(m->rows, m->cols, m->res, m->cx, m->cy, tl[0], tl[1], ti, tj)) return false;
  if (!artp::grid_index(m->rows, m->cols, m->res, m->cx, m->cy, br[0], br[1], bi, bj)) return false;
  // getPositionFromIndex(top-left) + 0.5 res: the submap's corner
  const double cx = ((m->cx + (0.5 * Lx - 0.5 * m->res)) + m->res * (-(double)ti)) + 0.5 * m->res;
  const double cy = ((m->cy + (0.5 * Ly - 0.5 * m->res)) + m->res * (-(double)tj)) + 0.5 * m->res;
  start[0] = ti; start[1] = tj;
  size[0] = bi - ti + 1; size[1] = bj - tj + 1;
  const double slx = size[0] * m->res, sly = size[1] * m->res;
  const double spx = cx - 0.5 * slx, spy = cy - 0.5 * sly;
  const double tx = -((rx - spx) - 0.5 * slx), ty = -((ry - spy) - 0.5 * sly);
  return tx >= 0.0 && ty >= 0.0 && tx < slx && ty < sly;
}

static bool grid_ok(const artp_grid* m) {
  return m && m->elevation && m->traversability_thresholded && m->rows > 0 && m->cols > 0 && m->res > 0.0 &&
         (size_t)m->rows * (size_t)m->cols < ((size_t)1 << 31);
}

int artp_compute_change_device(artp_handle* hh, const artp_grid* map_new, const artp_grid* map_old,
                               float height_change_for_update, float* d_updated, void* stream) {
  if (!hh) return ARTP_E_INVALID;
  Handle* h = reinterpret_cast<Handle*>(hh);
  std::lock_guard<std::recursive_mutex> lk(h->mtx);
  if (!grid_ok(map_new) || !grid_ok(map_old)) { h->err = "bad map (null layer, empty, res <= 0 or >= 2^31 cells)"; return ARTP_E_INVALID; }
  CU_TRY(h, cudaSetDevice(h->device));
  const cudaStream_t s = (cudaStream_t)stream;
  ChainScope cs(h, 0, s);
  if (cs.rc) return cs.rc;
  const size_t ncell = (size_t)map_new->rows * map_new->cols, words = (ncell + 31) / 32;
  if (h->chg_words_cap < words) {
    CU_TRY(h, cudaDeviceSynchronize());   // growth only: earlier readers on any stream must be done
    cudaFree(h->d_chg_bits);
    h->d_chg_bits = nullptr; h->chg_words_cap = 0; h->has_change = false;
    CU_TRY(h, cudaMalloc(&h->d_chg_bits, words * sizeof(uint32_t)));
    h->chg_words_cap = words;
  }
  // change.cpp:15-25: both submap geometries, once, in double on the host
  int sn[2], zn[2], so[2], zo[2];
  const bool ok = gm_submap(map_new, map_old->cx, map_old->cy, map_old->rows * map_old->res, map_old->cols * map_old->res, sn, zn) &&
                  gm_submap(map_old, map_new->cx, map_new->cy, map_new->rows * map_new->res, map_new->cols * map_new->res, so, zo);
  artp::ChangeArgs a{};
  a.e_new = map_new->elevation; a.t_new = map_new->traversability_thresholded;
  a.e_old = map_old->elevation; a.t_old = map_old->traversability_thresholded;
  a.rows_new = (uint32_t)map_new->rows; a.rows_old = (uint32_t)map_old->rows; a.ncell = (uint32_t)ncell;
  if (ok) {
    a.sn0 = sn[0]; a.sn1 = sn[1]; a.so0 = so[0]; a.so1 = so[1];
    a.sx = std::min(zn[0], zo[0]); a.sy = std::min(zn[1], zo[1]);
  }
  a.thr = height_change_for_update;
  a.bits = h->d_chg_bits;
  a.upd = d_updated;
  const unsigned grid = (unsigned)std::min<size_t>((ncell + 255) / 256, (size_t)h->sm_count * 16);
  artp::change_kernel<<<grid, 256, 0, s>>>(a);
  CU_TRY(h, cudaGetLastError());
  h->has_change = true;
  h->chg_rows = map_new->rows; h->chg_cols = map_new->cols;
  h->chg_res = map_new->res; h->chg_cx = map_new->cx; h->chg_cy = map_new->cy;
  h->stats.kernel_launches += 1;
  h->stats.last_launches = 1;
  return ARTP_OK;
}

int artp_compute_change(artp_handle* hh, const artp_grid* map_new, const artp_grid* map_old, float height_change_for_update,
                        float* updated) {
  if (!hh) return ARTP_E_INVALID;
  Handle* h = reinterpret_cast<Handle*>(hh);
  std::lock_guard<std::recursive_mutex> lk(h->mtx);   // held across stage -> launch -> D2H
  if (!grid_ok(map_new) || !grid_ok(map_old)) { h->err = "bad map (null layer, empty, res <= 0 or >= 2^31 cells)"; return ARTP_E_INVALID; }
  CU_TRY(h, cudaSetDevice(h->device));
  int rc = chain_begin(h, 0, h->stream);
  if (rc) return rc;
  const size_t nn = (size_t)map_new->rows * map_new->cols, no = (size_t)map_old->rows * map_old->cols;
  const size_t bn = (nn * sizeof(float) + 255) & ~(size_t)255, bo = (no * sizeof(float) + 255) & ~(size_t)255;
  rc = ensure_stage(h, 3 * bn + 2 * bo);
  if (rc) return rc;
  char* st = (char*)h->d_stage;
  artp_grid dn = *map_new, dold = *map_old;
  dn.elevation = (const float*)st; dn.traversability_thresholded = (const float*)(st + bn);
  dold.elevation = (const float*)(st + 2 * bn); dold.traversability_thresholded = (const float*)(st + 2 * bn + bo);
  float* d_out = updated ? (float*)(st + 2 * bn + 2 * bo) : nullptr;
  CU_TRY(h, cudaMemcpyAsync((void*)dn.elevation, map_new->elevation, nn * sizeof(float), cudaMemcpyHostToDevice, h->stream));
  CU_TRY(h, cudaMemcpyAsync((void*)dn.traversability_thresholded, map_new->traversability_thresholded, nn * sizeof(float),
                            cudaMemcpyHostToDevice, h->stream));
  CU_TRY(h, cudaMemcpyAsync((void*)dold.elevation, map_old->elevation, no * sizeof(float), cudaMemcpyHostToDevice, h->stream));
  CU_TRY(h, cudaMemcpyAsync((void*)dold.traversability_thresholded, map_old->traversability_thresholded, no * sizeof(float),
                            cudaMemcpyHostToDevice, h->stream));
  rc = artp_compute_change_device(hh, &dn, &dold, height_change_for_update, d_out, h->stream);
  if (rc) return rc;
  if (updated) CU_TRY(h, cudaMemcpyAsync(updated, d_out, nn * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
  CU_TRY(h, cudaStreamSynchronize(h->stream));
  h->chain_busy[0] = false;
  return ARTP_OK;
}

int artp_roadmap_updates_device(artp_handle* hh, const double* d_vertex_states, size_t nv, const uint32_t* d_edges, size_t ne,
                                uint8_t* d_vertex_flags, uint8_t* d_edge_flags, void* stream) {
  if (!hh) return ARTP_E_INVALID;
  Handle* h = reinterpret_cast<Handle*>(hh);
  std::lock_guard<std::recursive_mutex> lk(h->mtx);
  if (!h->has_change) { h->err = "no change layer (artp_compute_change first)"; return ARTP_E_NOMAP; }
  if ((nv && (!d_vertex_states || !d_vertex_flags)) || (ne && (!d_edges || !d_edge_flags))) { h->err = "null buffer"; return ARTP_E_INVALID; }
  if (nv == 0 && ne == 0) return ARTP_OK;
  CU_TRY(h, cudaSetDevice(h->device));
  const cudaStream_t s = (cudaStream_t)stream;
  ChainScope cs(h, 0, s);
  if (cs.rc) return cs.rc;
  const artp::RoadmapGeom g{h->d_chg_bits, h->chg_rows, h->chg_cols, h->chg_res, h->chg_cx, h->chg_cy};
  const size_t threads = std::max(nv, ne * 32);
  const unsigned grid = (unsigned)std::min<size_t>((threads + 255) / 256, (size_t)h->sm_count * 16);
  artp::roadmap_kernel<<<grid, 256, 0, s>>>(g, d_vertex_states, nv, d_edges, ne, d_vertex_flags, d_edge_flags, h->d_err);
  CU_TRY(h, cudaGetLastError());
  h->stats.kernel_launches += 1;
  h->stats.last_launches = 1;
  return ARTP_OK;
}

int artp_roadmap_updates(artp_handle* hh, const double* vertex_states, size_t nv, const uint32_t* edges, size_t ne,
                         uint8_t* vertex_flags, uint8_t* edge_flags) {
  if (!hh) return ARTP_E_INVALID;
  Handle* h = reinterpret_cast<Handle*>(hh);
  std::lock_guard<std::recursive_mutex> lk(h->mtx);   // held across stage -> launch -> D2H
  if (!h->has_change) { h->err = "no change layer (artp_compute_change first)"; return ARTP_E_NOMAP; }
  if ((nv && (!vertex_states || !vertex_flags)) || (ne && (!edges || !edge_flags))) { h->err = "null buffer"; return ARTP_E_INVALID; }
  for (size_t k = 0; k < 2 * ne; ++k)
    if (edges[k] >= nv) { h->err = "edge " + std::to_string(k / 2) + " references a vertex index >= nv"; return ARTP_E_INVALID; }
  if (nv == 0 && ne == 0) return ARTP_OK;
  CU_TRY(h, cudaSetDevice(h->device));
  int rc = chain_begin(h, 0, h->stream);
  if (rc) return rc;
  const size_t bs = (nv * 7 * sizeof(double) + 255) & ~(size_t)255, be = (ne * 2 * sizeof(uint32_t) + 255) & ~(size_t)255;
  const size_t bv = (nv + 255) & ~(size_t)255;
  rc = ensure_stage(h, bs + be + bv + ne);
  if (rc) return rc;
  char* st = (char*)h->d_stage;
  double* d_s = (double*)st;
  uint32_t* d_e = (uint32_t*)(st + bs);
  uint8_t* d_vf = (uint8_t*)(st + bs + be);
  uint8_t* d_ef = d_vf + bv;
  if (nv) CU_TRY(h, cudaMemcpyAsync(d_s, vertex_states, nv * 7 * sizeof(double), cudaMemcpyHostToDevice, h->stream));
  if (ne) CU_TRY(h, cudaMemcpyAsync(d_e, edges, ne * 2 * sizeof(uint32_t), cudaMemcpyHostToDevice, h->stream));
  rc = artp_roadmap_updates_device(hh, d_s, nv, d_e, ne, d_vf, d_ef, h->stream);
  if (rc) return rc;
  if (nv) CU_TRY(h, cudaMemcpyAsync(vertex_flags, d_vf, nv, cudaMemcpyDeviceToHost, h->stream));
  if (ne) CU_TRY(h, cudaMemcpyAsync(edge_flags, d_ef, ne, cudaMemcpyDeviceToHost, h->stream));
  CU_TRY(h, cudaStreamSynchronize(h->stream));
  h->chain_busy[0] = false;
  return take_sticky_error(h);
}

size_t artp_cost_weights_size(void) { return artp_cnn::blob_floats(); }

int artp_set_cost_weights(artp_handle* hh, const float* blob, size_t n_floats) {
  if (!hh || !blob) return ARTP_E_INVALID;
  Handle* h = reinterpret_cast<Handle*>(hh);
  std::lock_guard<std::recursive_mutex> lk(h->mtx);
  return artp_cnn::set_weights(h->cnn, blob, n_floats, h->stream, h->err);
}

int artp_update_features(artp_handle* hh) {
  if (!hh) return ARTP_E_INVALID;
  Handle* h = reinterpret_cast<Handle*>(hh);
  std::lock_guard<std::recursive_mutex> lk(h->mtx);
  if (!h->has_map) { h->err = "no map set"; return ARTP_E_NOMAP; }
  if (h->win_rows != h->rows) { h->err = "not available on a map window (artp_set_map_window)"; return ARTP_E_INVALID; }
  artp_cnn::set_base_offset_mode(h->cnn, (h->cnn_mode & 2) ? 1 : 0);
  artp_cnn::set_conv15_mode(h->cnn, (h->cnn_mode >> 2) & 3);
  return artp_cnn::update_features(h->cnn, h->d_H[0], h->rows, h->cols, h->pitch, h->chk.Lx / h->rows, h->chk.cx, h->chk.cy,
                                   h->stream, h->cnn_mode & 1, h->err);
}

int artp_motion_cost_device(artp_handle* hh, const float* d_edges, size_t n, float* d_cost3, void* stream) {
  if (!hh) return ARTP_E_INVALID;
  Handle* h = reinterpret_cast<Handle*>(hh);
  std::lock_guard<std::recursive_mutex> lk(h->mtx);
  if (n && (!d_edges || !d_cost3)) { h->err = "null buffer"; return ARTP_E_INVALID; }
  int rc = artp_cnn::motion_cost(h->cnn, d_edges, n, d_cost3, (cudaStream_t)stream, h->err);
  if (rc == 0 && n) { h->stats.kernel_launches += 1; h->stats.last_launches = 1; }
  return rc;
}

int artp_motion_cost(artp_handle* hh, const float* edges, size_t n, float* cost3) {
  if (!hh) return ARTP_E_INVALID;
  Handle* h = reinterpret_cast<Handle*>(hh);
  if (n == 0) return ARTP_OK;
  const size_t in_b = n * 6 * sizeof(float), in_al = (in_b + 255) & ~(size_t)255;
  std::lock_guard<std::recursive_mutex> lk(h->mtx);   // held across stage -> launch -> D2H
  if (!edges || !cost3) { h->err = "null buffer"; return ARTP_E_INVALID; }
  CU_TRY(h, cudaSetDevice(h->device));
  int rc = chain_begin(h, 0, h->stream);
  if (rc) return rc;
  rc = ensure_stage(h, in_al + n * 3 * sizeof(float));
  if (rc) return rc;
  CU_TRY(h, cudaMemcpyAsync(h->d_stage, edges, in_b, cudaMemcpyHostToDevice, h->stream));
  float* d_cost = (float*)((char*)h->d_stage + in_al);
  rc = artp_motion_cost_device(hh, (const float*)h->d_stage, n, d_cost, h->stream);
  if (rc) return rc;
  CU_TRY(h, cudaMemcpyAsync(cost3, d_cost, n * 3 * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
  CU_TRY(h, cudaStreamSynchronize(h->stream));
  return ARTP_OK;
}

int artp_combine_cost(artp_handle* hh, const float* cost3, size_t n, double* cost, uint8_t* feasible) {
  if (!hh || (n && (!cost3 || !cost || !feasible))) return ARTP_E_INVALID;
  Handle* h = reinterpret_cast<Handle*>(hh);
  const float we = h->p.cost_w_energy, wt = h->p.cost_w_time, wr = h->p.cost_w_risk;
  for (size_t i = 0; i < n; ++i) {
    const float ce = cost3[3 * i], ct = cost3[3 * i + 1], cr = cost3[3 * i + 2];
    // getCost: getEnergy/getTime/getRisk return double (motion_cost_objective.h:30-46), so the weighted sum is evaluated
    // in double on exact float products
    cost[i] = (double)ce * (double)we + (double)ct * (double)wt + (double)cr * (double)wr;
    feasible[i] = (double)cr <= (double)h->p.risk_threshold ? 1 : 0;   // isFeasible (getRisk returns double)
  }
  return ARTP_OK;
}

int artp_get_features(artp_handle* hh, float* out, size_t n_floats, int* hf, int* wf) {
  if (!hh || !hf || !wf) return ARTP_E_INVALID;
  Handle* h = reinterpret_cast<Handle*>(hh);
  std::lock_guard<std::recursive_mutex> lk(h->mtx);
  artp_cnn::feature_shape(h->cnn, hf, wf);
  if (!out) return ARTP_OK;
  return artp_cnn::copy_features(h->cnn, out, n_floats, h->err);
}

int artp_set_cnn_mode(artp_handle* hh, int mode) {
  if (!hh) return ARTP_E_INVALID;
  reinterpret_cast<Handle*>(hh)->cnn_mode = mode;
  return ARTP_OK;
}

int artp_get_cnn_timing(artp_handle* hh, float* ms3) {
  if (!hh || !ms3) return ARTP_E_INVALID;
  artp_cnn::last_times(reinterpret_cast<Handle*>(hh)->cnn, ms3);
  return ARTP_OK;
}

}  // extern "C"
