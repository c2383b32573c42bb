// cloud.cu -- PointCloud2 post-processing (north-star extensions; no reference counterpart).
//
// oracle/cloud_oracle.cpp is the definition (PARITY UNPINNED: the reference has no
// polar->Cartesian, outlier or voxel code).  Steps 1-3 (window, stable key order, polar->xyz)
// run inside the scan kernels (scan_tma.cu / scan_general.cu, `xyzi` payload) and leave, per
// scan, the kept points in angle order as (x, y, 0, intensity).  This file holds
//   * the trig table those kernels read: (float)cos((double)angle_rad(key)), built on the host
//     with the same libm the oracle uses, so x = r * c is bit-identical on both sides,
//   * step 4, statistical outlier removal over the +-16 angular neighbours, statistics taken
//     with exact integer sums (order independent => bit reproducible),
//   * step 5, the voxel grid: shared hash table per scan, centroids from exact integer sums,
//     cells emitted in order of their first member,
//   * the fuse step that packs the per-scan clouds of a batch into one dense cloud (the per-GPU
//     payload of the multi-GPU all-gather).
#include <cmath>
#include <vector>

#include "cloud_args.h"
#include "rpl_device.cuh"

namespace rpl {

namespace {

constexpr int CT = 256;  // threads per CTA of the post-processing kernels
constexpr int kHalfWindow = 16;

// One hash-table entry.  The table is kept CLEAN between scans (every cell a scan touched is reset by
// the thread that emits it), so no per-scan clear of the whole table is needed.
struct __align__(32) VoxelCell {
  unsigned long long key;  // packed (ix, iy), kVoxelEmpty when free
  long long sx, sy;        // sums of llrintf(v * 65536)
  unsigned long long nsi;  // count << 32 | intensity sum
};
// no cell has ix == INT_MIN: |x| <= range_max < 1000 m and voxel >= 1e-6 m (checked by the C-ABI)
constexpr unsigned long long kVoxelEmpty = 0x8000000000000000ull;

struct CloudScratch {  // per CTA, sized for max_nodes
  unsigned long long* q;  // [max_nodes] SOR: fixed-point mean neighbour distance (llrintf)
  uint32_t* slot;      // [max_nodes] voxel: hash slot of every point
  VoxelCell* cell;     // [hsize] one 32-byte sector per cell: key + the three integer sums
  uint2* first_order;  // [hsize] (first member, output position)
};

__device__ __forceinline__ CloudScratch carve(void* base, size_t per_cta, uint32_t max_nodes, uint32_t hsize) {
  unsigned char* p = static_cast<unsigned char*>(base) + (size_t)blockIdx.x * per_cta;
  CloudScratch s;
  s.cell = reinterpret_cast<VoxelCell*>(p); p += (size_t)hsize * sizeof(VoxelCell);
  s.first_order = reinterpret_cast<uint2*>(p); p += (size_t)hsize * 8;
  s.q = reinterpret_cast<unsigned long long*>(p); p += (size_t)max_nodes * 8;
  s.slot = reinterpret_cast<uint32_t*>(p);
  return s;
}

__host__ __device__ inline uint32_t hash_size_for(uint32_t max_nodes) {
  uint32_t h = 64;
  while (h < 2u * max_nodes) h <<= 1;
  return h;
}

__device__ __forceinline__ uint32_t block_exclusive_scan_u32(uint32_t v, uint32_t* smem_warp, uint32_t* total) {
  const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const uint32_t inc = warp_inclusive_scan(v);
  if (lane == 31) smem_warp[warp] = inc;
  __syncthreads();
  uint32_t base = 0, tot = 0;
#pragma unroll
  for (int w = 0; w < CT / 32; ++w) {
    const uint32_t t = smem_warp[w];
    if ((uint32_t)w < warp) base += t;
    tot += t;
  }
  __syncthreads();
  *total = tot;
  return base + inc - v;
}

// ---- step 4: statistical outlier removal (oracle/cloud_oracle.cpp step 4) -----------------
// K = compile-time bound of sor_k: the K smallest distances live in a sorted register array (branch-free
// insertion), the neighbours' coordinates are staged through shared memory once per chunk of CT points.
template <int K>
__global__ void __launch_bounds__(CT) cloud_sor_kernel(float4* xyzi, uint32_t* point_counts, uint32_t n_scans,
                                                       uint32_t stride, uint32_t sor_k, float sor_alpha,
                                                       void* scratch, size_t per_cta, uint32_t max_nodes,
                                                       const uint32_t* list, const uint32_t* list_count) {
  __shared__ float2 s_xy[CT + 2 * kHalfWindow];
  __shared__ uint32_t s_warp[CT / 32];
  __shared__ long long s_s1[CT / 32];
  __shared__ unsigned long long s_s2[CT / 32];
  __shared__ double s_thr;
  const CloudScratch sc = carve(scratch, per_cta, max_nodes, hash_size_for(max_nodes));
  const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  // `list` (nullable): only these scans (the duplicate-key scans the shared-memory kernel handed on)
  const uint32_t n_work = list ? min(*list_count, n_scans) : n_scans;
  for (uint32_t sj = blockIdx.x; sj < n_work; sj += gridDim.x) {
    const uint32_t s = list ? list[sj] : sj;
    float4* pts = xyzi + (size_t)s * stride;
    const uint32_t m = point_counts[s];
    if (m < 2 || m > max_nodes) continue;  // fewer than 2 points keep everything
    const bool all_others = (m - 1) <= 2u * kHalfWindow;
    long long s1 = 0;
    unsigned long long s2 = 0;
    for (uint32_t c0 = 0; c0 < m; c0 += CT) {
      // stage (x, y) of this chunk's points and their +-16 neighbours (all points when the scan is tiny)
      __syncthreads();
      if (all_others) {
        for (uint32_t t = tid; t < m; t += CT) {
          const float4 o = pts[t];
          s_xy[t] = make_float2(o.x, o.y);
        }
      } else {
        for (uint32_t t = tid; t < (uint32_t)(CT + 2 * kHalfWindow); t += CT) {
          uint32_t j = c0 + t + m - (uint32_t)kHalfWindow;  // index c0 + t - 16, modulo m
          j %= m;
          const float4 o = pts[j];
          s_xy[t] = make_float2(o.x, o.y);
        }
      }
      __syncthreads();
      const uint32_t i = c0 + tid;
      if (i >= m) continue;
      const float2 me = all_others ? s_xy[i] : s_xy[tid + kHalfWindow];
      float top[K];  // ascending; +inf = empty
#pragma unroll
      for (int t = 0; t < K; ++t) top[t] = __int_as_float(0x7f800000);
      uint32_t nd = 0;
      auto add = [&](float2 o) {
        const float dx = __fsub_rn(o.x, me.x), dy = __fsub_rn(o.y, me.y);
        float v = __fsqrt_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)));
#pragma unroll
        for (int t = 0; t < K; ++t) {
          const float lo = fminf(top[t], v), hi = fmaxf(top[t], v);
          top[t] = lo;
          v = hi;
        }
        ++nd;
      };
      if (all_others) {
        for (uint32_t j = 0; j < m; ++j)
          if (j != i) add(s_xy[j]);
      } else {
#pragma unroll 4
        for (uint32_t o = 1; o <= (uint32_t)kHalfWindow; ++o) {
          add(s_xy[tid + kHalfWindow - o]);
          add(s_xy[tid + kHalfWindow + o]);
        }
      }
      const uint32_t k = min(sor_k, nd);
      float sum = 0.0f;
#pragma unroll
      for (int t = 0; t < K; ++t)
        if ((uint32_t)t < k) sum = __fadd_rn(sum, top[t]);
      const float mean = __fdiv_rn(sum, __uint2float_rn(k));
      const long long q = __float2ll_rn(__fmul_rn(mean, 65536.0f));  // llrintf
      sc.q[i] = (unsigned long long)q;
      s1 += q;
      s2 += (unsigned long long)q * (unsigned long long)q;
    }
    // exact block sums
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      s1 += __shfl_xor_sync(0xffffffffu, s1, o);
      s2 += __shfl_xor_sync(0xffffffffu, s2, o);
    }
    if (lane == 0) {
      s_s1[warp] = s1;
      s_s2[warp] = s2;
    }
    __syncthreads();
    if (tid == 0) {
      long long t1 = 0;
      unsigned long long t2 = 0;
      for (int w = 0; w < CT / 32; ++w) {
        t1 += s_s1[w];
        t2 += s_s2[w];
      }
      const double dn = (double)m;
      const double mean = __ddiv_rn((double)t1, dn);
      const double sq = __ddiv_rn(__dmul_rn((double)t1, (double)t1), dn);
      double var = __ddiv_rn(__dsub_rn((double)t2, sq), __dsub_rn(dn, 1.0));
      if (!(var > 0.0)) var = 0.0;
      s_thr = __dadd_rn(mean, __dmul_rn((double)sor_alpha, __dsqrt_rn(var)));
    }
    __syncthreads();
    const double thr = s_thr;
    // in-place stable compaction, chunk by chunk (destinations never pass sources)
    uint32_t done = 0;
    for (uint32_t c0 = 0; c0 < m; c0 += CT) {
      const uint32_t i = c0 + tid;
      float4 me = make_float4(0, 0, 0, 0);
      uint32_t keep = 0;
      if (i < m) {
        me = pts[i];
        keep = ((double)(long long)sc.q[i] <= thr) ? 1u : 0u;
      }
      uint32_t tot = 0;
      const uint32_t pos = block_exclusive_scan_u32(keep, s_warp, &tot);  // syncs: chunk fully read
      if (keep) pts[done + pos] = me;
      done += tot;
      __syncthreads();
    }
    if (tid == 0) point_counts[s] = done;
    __syncthreads();
  }
}

// ---- step 5: voxel grid (oracle/cloud_oracle.cpp step 5) -----------------------------------
__global__ void cloud_table_init_kernel(void* scratch, size_t per_cta, uint32_t max_nodes) {
  const uint32_t hsize = hash_size_for(max_nodes);
  const CloudScratch sc = carve(scratch, per_cta, max_nodes, hsize);
  for (uint32_t j = threadIdx.x; j < hsize; j += blockDim.x) {
    sc.cell[j] = VoxelCell{kVoxelEmpty, 0, 0, 0};
    sc.first_order[j] = make_uint2(0xFFFFFFFFu, 0u);
  }
}

__global__ void __launch_bounds__(CT) cloud_voxel_kernel(float4* xyzi, uint32_t* point_counts, uint32_t n_scans,
                                                         uint32_t stride, float voxel, void* scratch, size_t per_cta,
                                                         uint32_t max_nodes, const uint32_t* list,
                                                         const uint32_t* list_count) {
  __shared__ uint32_t s_warp[CT / 32];
  // the whole table (>= 2 * max_nodes slots) is clean on entry; a scan uses a prefix sized to its own
  // point count so that the slots all resident CTAs touch stay inside the L2
  const CloudScratch sc = carve(scratch, per_cta, max_nodes, hash_size_for(max_nodes));
  const uint32_t tid = threadIdx.x, lane = tid & 31;
  const uint32_t n_work = list ? min(*list_count, n_scans) : n_scans;
  for (uint32_t sj = blockIdx.x; sj < n_work; sj += gridDim.x) {
    const uint32_t s = list ? list[sj] : sj;
    float4* pts = xyzi + (size_t)s * stride;
    const uint32_t m = point_counts[s];
    if (m == 0 || m > max_nodes) continue;
    uint32_t hs = 64;
    while (hs < m + (m >> 2)) hs <<= 1;  // load factor <= 0.8 even if every point had its own cell
    // insert: exact integer sums, first member by atomicMin.  Points arrive in angular order, so the
    // members of a cell are mostly neighbours: every warp first folds runs of equal cells among its 32
    // consecutive points (segmented suffix sums with shuffles) and only the head of a run touches the
    // table -- all sums are integers, so the grouping cannot change the result.
    for (uint32_t c0 = 0; c0 < m; c0 += CT) {
      const uint32_t i = c0 + tid;
      const bool valid = i < m;
      float4 p = make_float4(0.f, 0.f, 0.f, 0.f);
      if (valid) {  // read once: keep the table, not the points, in the L2
        const uint4 r = ld_hint_v4(pts + i, l2_policy_evict_first());
        p = make_float4(__uint_as_float(r.x), __uint_as_float(r.y), __uint_as_float(r.z), __uint_as_float(r.w));
      }
      const int ix = __float2int_rd(__fdiv_rn(p.x, voxel));  // floorf(x / voxel)
      const int iy = __float2int_rd(__fdiv_rn(p.y, voxel));
      // lanes past the end get the key no cell can have
      const unsigned long long key = valid ? (((unsigned long long)(uint32_t)ix << 32) | (uint32_t)iy) : kVoxelEmpty;
      const unsigned long long key_prev = __shfl_up_sync(0xffffffffu, key, 1);
      const bool head = lane == 0 || key != key_prev;
      int hl = head ? (int)lane : 0;  // lane of this point's run head
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int t = __shfl_up_sync(0xffffffffu, hl, o);
        if ((int)lane >= o) hl = max(hl, t);
      }
      long long sx = __float2ll_rn(__fmul_rn(p.x, 65536.0f));
      long long sy = __float2ll_rn(__fmul_rn(p.y, 65536.0f));
      unsigned long long nsi = (1ull << 32) + (unsigned long long)__float2ll_rn(p.w);  // count | intensity sum
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int hl_o = __shfl_down_sync(0xffffffffu, hl, o);
        const long long sx_o = __shfl_down_sync(0xffffffffu, sx, o);
        const long long sy_o = __shfl_down_sync(0xffffffffu, sy, o);
        const unsigned long long nsi_o = __shfl_down_sync(0xffffffffu, nsi, o);
        if ((int)lane + o < 32 && hl_o == hl) {
          sx += sx_o;
          sy += sy_o;
          nsi += nsi_o;
        }
      }
      uint32_t h = 0;
      if (head && valid) {
        h = (uint32_t)(mix64(key) & (hs - 1));
        for (;;) {
          const unsigned long long prev = atomicCAS(&sc.cell[h].key, kVoxelEmpty, key);
          if (prev == kVoxelEmpty || prev == key) break;
          h = (h + 1) & (hs - 1);
        }
        atomicAdd(reinterpret_cast<unsigned long long*>(&sc.cell[h].sx), (unsigned long long)sx);
        atomicAdd(reinterpret_cast<unsigned long long*>(&sc.cell[h].sy), (unsigned long long)sy);
        atomicAdd(&sc.cell[h].nsi, nsi);
        atomicMin(&sc.first_order[h].x, i);
      }
      h = __shfl_sync(0xffffffffu, h, hl);
      if (valid) sc.slot[i] = h;
    }
    __syncthreads();
    // cells in order of their first member: exclusive scan over "i is a first member"
    uint32_t done = 0;
    for (uint32_t c0 = 0; c0 < m; c0 += CT) {
      const uint32_t i = c0 + tid;
      uint32_t rep = 0, h = 0;
      if (i < m) {
        h = sc.slot[i];
        rep = (sc.first_order[h].x == i) ? 1u : 0u;
      }
      uint32_t tot = 0;
      const uint32_t pos = block_exclusive_scan_u32(rep, s_warp, &tot);
      if (rep) sc.first_order[h].y = done + pos;
      done += tot;
    }
    __syncthreads();
    // emit centroids (all reads of the point array happened before the first barrier above) and hand
    // the cell back clean
    for (uint32_t i = tid; i < m; i += CT) {
      const uint32_t h = sc.slot[i];
      const uint2 fo = sc.first_order[h];
      if (fo.x != i) continue;
      const VoxelCell c = sc.cell[h];
      const double cnt = (double)(uint32_t)(c.nsi >> 32);
      const double den = __dmul_rn(65536.0, cnt);
      float4 o;
      o.x = __double2float_rn(__ddiv_rn((double)c.sx, den));
      o.y = __double2float_rn(__ddiv_rn((double)c.sy, den));
      o.z = 0.0f;
      o.w = __double2float_rn(__ddiv_rn((double)(long long)(c.nsi & 0xFFFFFFFFull), cnt));
      pts[fo.y] = o;
      sc.cell[h] = VoxelCell{kVoxelEmpty, 0, 0, 0};
      sc.first_order[h] = make_uint2(0xFFFFFFFFu, 0u);
    }
    if (tid == 0) point_counts[s] = done;
    __syncthreads();
  }
}

// ---- fuse: per-scan clouds -> one dense cloud ------------------------------------------------
__global__ void cloud_offsets_kernel(const uint32_t* counts, uint32_t n, uint32_t* offsets, uint32_t* total) {
  // single CTA exclusive scan (n_scans is small next to the point data)
  __shared__ uint32_t s_warp[32];
  __shared__ uint32_t s_carry;
  if (threadIdx.x == 0) s_carry = 0;
  __syncthreads();
  for (uint32_t c0 = 0; c0 < n; c0 += blockDim.x) {
    const uint32_t i = c0 + threadIdx.x;
    const uint32_t v = i < n ? counts[i] : 0u;
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint32_t inc = warp_inclusive_scan(v);
    if (lane == 31) s_warp[warp] = inc;
    __syncthreads();
    uint32_t base = 0, tot = 0;
    for (uint32_t w = 0; w < blockDim.x / 32; ++w) {
      if (w < warp) base += s_warp[w];
      tot += s_warp[w];
    }
    const uint32_t carry = s_carry;
    if (i < n) offsets[i] = carry + base + inc - v;
    __syncthreads();
    if (threadIdx.x == 0) s_carry = carry + tot;
    __syncthreads();
  }
  if (threadIdx.x == 0) *total = s_carry;
}

__global__ void cloud_pack_kernel(const float4* xyzi, const uint32_t* counts, const uint32_t* offsets,
                                  uint32_t n_scans, uint32_t stride, float4* fused, uint32_t capacity) {
  const uint64_t pol = l2_policy_evict_first();
  for (uint32_t s = blockIdx.y; s < n_scans; s += gridDim.y) {
    const uint32_t m = counts[s], off = offsets[s];
    const float4* src = xyzi + (size_t)s * stride;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < m; i += gridDim.x * blockDim.x) {
      if (off + i >= capacity) break;  // the reader sees total > capacity and knows the slot overflowed
      st_f32x4_if(fused + off + i, src[i], pol, 1u);
    }
  }
}

// fuse + all-gather in one kernel: every point of this rank's fused cloud is stored straight into slot
// `rank` of EVERY rank's gather buffer (the peers' buffers are mapped through CUDA IPC, the stores travel
// over NVLink), so the dense per-GPU cloud is never written locally and read again by a collective.
// Gather buffer layout: [256-byte header: point count of every rank][world][slot_points][16 B].
__global__ void cloud_push_kernel(const float4* xyzi, const uint32_t* counts, const uint32_t* offsets,
                                  const uint32_t* total, uint32_t n_scans, uint32_t stride, PeerBases peers,
                                  uint32_t world, uint32_t rank, uint32_t slot_points) {
  if (blockIdx.x == 0 && blockIdx.y == 0 && threadIdx.x < world)
    reinterpret_cast<uint32_t*>(peers.base[threadIdx.x])[rank] = *total;  // > slot_points tells the reader it overflowed
  const size_t slot0 = (size_t)rank * slot_points;
  for (uint32_t s = blockIdx.y; s < n_scans; s += gridDim.y) {
    const uint32_t m = counts[s], off = offsets[s];
    const float4* src = xyzi + (size_t)s * stride;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < m; i += gridDim.x * blockDim.x) {
      if (off + i >= slot_points) break;
      const float4 v = src[i];
      for (uint32_t p = 0; p < world; ++p)
        reinterpret_cast<float4*>(peers.base[p] + kPeerHeaderBytes)[slot0 + off + i] = v;
    }
  }
}

}  // namespace

cudaError_t launch_cloud_fuse_push(const float4* xyzi, const uint32_t* point_counts, uint32_t n_scans,
                                   uint32_t stride, const PeerBases& peers, uint32_t world, uint32_t rank,
                                   uint32_t slot_points, uint32_t* offsets, uint32_t* total, cudaStream_t stream,
                                   int* launched) {
  // an empty batch still runs both kernels: *total = 0 and the header entries must not keep an earlier step's count
  cloud_offsets_kernel<<<1, 1024, 0, stream>>>(point_counts, n_scans, offsets, total);
  const uint32_t gy = max(1u, min(n_scans, 65535u));
  const uint32_t gx = max(1u, min(32u, (stride + 255u) / 256u));
  cloud_push_kernel<<<dim3(gx, gy), 256, 0, stream>>>(xyzi, point_counts, offsets, total, n_scans, stride, peers,
                                                      world, rank, slot_points);
  if (launched) *launched += 2;
  return cudaGetLastError();
}

cudaError_t cloud_configure() { return cudaSuccess; }

cudaError_t cloud_workspace_alloc(CloudWorkspace& ws, int num_sms, uint32_t max_nodes) {
  // trig table: (float)cos((double)angle_rad), (float)sin(...) with angle_rad exactly as
  // publish_scan computes it (reference rplidar_node.cpp:586-587)
  std::vector<float2> h(65536), ang(65536);
  const double two_pi = 2.0 * 3.14159265358979323846;
  for (uint32_t k = 0; k < 65536; ++k) {
    const float deg = static_cast<float>(k) * 90.0f / 16384.0f;
    const float rad = static_cast<float>(static_cast<double>(deg) * (3.14159265358979323846 / 180.0));
    h[k].x = static_cast<float>(std::cos(static_cast<double>(rad)));
    h[k].y = static_cast<float>(std::sin(static_cast<double>(rad)));
    // Mode A angles (reference rplidar_node.cpp:641-649): plain and inverted
    float inv = static_cast<float>(two_pi - static_cast<double>(rad));
    if (static_cast<double>(inv) >= two_pi) inv = static_cast<float>(static_cast<double>(inv) - two_pi);
    ang[k].x = rad;
    ang[k].y = inv;
  }
  cudaError_t e = cudaMalloc(reinterpret_cast<void**>(&ws.trig), h.size() * sizeof(float2));
  if (e != cudaSuccess) return e;
  e = cudaMemcpy(ws.trig, h.data(), h.size() * sizeof(float2), cudaMemcpyHostToDevice);
  if (e != cudaSuccess) return e;
  e = cudaMalloc(reinterpret_cast<void**>(&ws.angle), ang.size() * sizeof(float2));
  if (e != cudaSuccess) return e;
  e = cudaMemcpy(ws.angle, ang.data(), ang.size() * sizeof(float2), cudaMemcpyHostToDevice);
  if (e != cudaSuccess) return e;
  ws.max_nodes = max_nodes;
  const uint32_t hsize = hash_size_for(max_nodes);
  ws.scratch_per_cta = (size_t)hsize * (sizeof(VoxelCell) + 8) + (size_t)max_nodes * 12 + 64;
  ws.scratch_per_cta = (ws.scratch_per_cta + 255) & ~(size_t)255;
  // the post kernels wait on L2 atomics and block scans: 4 CTAs of 256 threads per SM hide that latency;
  // fewer when the per-CTA tables are large (at most 1 GiB of scratch per lane, at least 2 CTAs per SM)
  const size_t budget_ctas = ((size_t)1 << 30) / ws.scratch_per_cta;
  ws.ctas = (int)std::min<size_t>((size_t)num_sms * 4, std::max<size_t>((size_t)num_sms * 2, budget_ctas));
  e = cudaMalloc(&ws.scratch, ws.scratch_per_cta * ws.ctas);
  if (e != cudaSuccess) return e;
  cloud_table_init_kernel<<<ws.ctas, 256>>>(ws.scratch, ws.scratch_per_cta, max_nodes);  // tables start clean
  e = cudaGetLastError();
  if (e != cudaSuccess) return e;
  return cudaDeviceSynchronize();
}

void cloud_workspace_free(CloudWorkspace& ws) {
  cudaFree(ws.trig);
  cudaFree(ws.angle);
  cudaFree(ws.scratch);
  ws = CloudWorkspace{};
}

cudaError_t launch_cloud_post(float4* xyzi, uint32_t* point_counts, uint32_t n_scans, uint32_t stride,
                              uint32_t sor_k, float sor_alpha, float voxel, const CloudWorkspace& ws,
                              const uint32_t* list, const uint32_t* list_count, cudaStream_t stream, int* launched) {
  // with a list the work is a handful of scans: a small grid finds out on the device
  const int grid = list ? (int)min((uint32_t)ws.ctas, min(n_scans, 64u)) : (int)min((uint32_t)ws.ctas, n_scans);
  if (sor_k > 0) {
    auto k = cloud_sor_kernel<32>;
    if (sor_k <= 4) k = cloud_sor_kernel<4>;
    else if (sor_k <= 8) k = cloud_sor_kernel<8>;
    else if (sor_k <= 16) k = cloud_sor_kernel<16>;
    k<<<grid, CT, 0, stream>>>(xyzi, point_counts, n_scans, stride, sor_k, sor_alpha, ws.scratch, ws.scratch_per_cta,
                               ws.max_nodes, list, list_count);
    if (launched) ++*launched;
  }
  if (voxel > 0.0f) {
    cloud_voxel_kernel<<<grid, CT, 0, stream>>>(xyzi, point_counts, n_scans, stride, voxel, ws.scratch,
                                                ws.scratch_per_cta, ws.max_nodes, list, list_count);
    if (launched) ++*launched;
  }
  return cudaGetLastError();
}

cudaError_t launch_cloud_fuse(const float4* xyzi, const uint32_t* point_counts, uint32_t n_scans,
                              uint32_t stride, float4* fused, uint32_t capacity, uint32_t* offsets, uint32_t* total,
                              cudaStream_t stream, int* launched) {
  // an empty batch still runs the offsets kernel: it writes *total = 0 (the caller's count, or a gather slot's header)
  cloud_offsets_kernel<<<1, 1024, 0, stream>>>(point_counts, n_scans, offsets, total);
  const uint32_t gy = max(1u, min(n_scans, 65535u));
  const uint32_t gx = max(1u, min(32u, (stride + 255u) / 256u));
  cloud_pack_kernel<<<dim3(gx, gy), 256, 0, stream>>>(xyzi, point_counts, offsets, n_scans, stride, fused, capacity);
  if (launched) *launched += 2;
  return cudaGetLastError();
}

}  // namespace rpl
