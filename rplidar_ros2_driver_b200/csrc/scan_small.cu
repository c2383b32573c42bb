// scan_small.cu -- the scan kernels for revolutions that fit shared memory (stride <= 8192 nodes, the SDK's own
// holder capacity: what a spinning lidar delivers; the S2/S3 produce 3200 at 10 Hz).  The PointCloud2 chain with
// SOR / voxel grid fused needs more shared memory per node and serves strides up to 4096.
//
// Same contract as scan_tma.cu / scan_fast.cu (ascendScanData_ + publish_scan, reference
// src/sdk/src/sl_lidar_driver.cpp:128-184 and src/rplidar_node.cpp:581-677; the PointCloud2 steps of
// oracle/cloud_oracle.cpp), different cost structure.  The big-scan kernels pay a fixed 128 KB of
// shared-memory traffic per scan (clearing and folding a 64 KB byte map) and stream the tile twice;
// at 3200 nodes that fixed work costs as much as the nodes themselves (round 1: 42 % of the HBM
// roofline against 74 % at 32768 nodes).  Here
//   * the whole revolution is staged ONCE into shared memory by one bulk-TMA copy (cp.async.bulk +
//     mbarrier; plain loads when the scan base is not 16-byte aligned), and both passes read it there;
//   * keys are marked straight into the 8 KB presence BITMAP with shared-memory atomicOr -- at
//     <= 4096 nodes per revolution neighbouring keys are >= 16 apart, so lanes rarely share a word
//     (the reason the 32768-node kernel uses a byte map instead) -- which removes the byte map, its
//     clear and its fold; the rank table is the bitmap + a 4 KB u16 prefix;
//   * Mode A is a scatter-min over its bins (per bin the smallest dist_m, then the smallest key among the
//     points that hold it: two shared atomics per point, no ranks, no bitmap of the measured keys), the
//     ascended buffer is a second bitmap over the final keys, and the PointCloud2 chain runs to the end
//     in shared memory: the kept
//     points are placed in angle order as (x, y) + intensity, statistical outlier removal and the
//     voxel grid (open-addressing table of cell leaders in the dead tile buffer, 32-bit integer
//     accumulators relative to the leader) work on them there, and only the final cloud -- rho x 16 B
//     per input node -- is written to HBM.  The three HBM round trips and the global hash tables of
//     the round-1 post kernels are gone.
// Duplicate keys among the measured nodes (popcount != count) go to the general kernel through the device-side
// list; Mode A only does so when a duplicate would change its result, and up to 16 shared FINAL keys per
// revolution (a fill key landing on a measured key) are placed here, in buffer order (stable rule).
#include <algorithm>
#include <type_traits>

#include "rpl_device.cuh"
#include "scan_args.h"
#include "scan_common.cuh"

namespace rpl {

namespace {

struct SmallCtl {
  unsigned long long full;  // mbarrier of the tile copy
  long long s1;
  unsigned long long s2;
  double thr;
  uint32_t red[3 * 32];
  uint32_t totV, totA, first_valid, front_key, fallback, count_out;
  union {
    uint32_t chunk_base[128];  // PointCloud2 chain, voxel ordering: per (chunk, warp) counts -> exclusive bases
    struct {                   // ascended buffer: the few nodes whose final key is already taken (see the place pass)
      uint16_t dupkey[16];     // final key of every node beyond the first with that key
      uint16_t dupnode[32];    // nodes whose key appears in dupkey: placed by the fix-up after the place pass
      uint32_t ndup, ndupnode;
    } d;
  };
};
constexpr uint32_t kMaxDup = 16;
static_assert(sizeof(SmallCtl) <= 1024, "control block");
constexpr uint32_t kCtl = 1024;

__device__ __forceinline__ uint32_t s_u32(const void* p) { return static_cast<uint32_t>(__cvta_generic_to_shared(p)); }
__device__ __forceinline__ void s_mbar_init(void* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(s_u32(bar)), "r"(count));
}
__device__ __forceinline__ void s_mbar_wait(void* bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "LAB_WAIT:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra DONE;\n"
      "bra LAB_WAIT;\n"
      "DONE:\n"
      "}\n" ::"r"(s_u32(bar)),
      "r"(parity)
      : "memory");
}
__device__ __forceinline__ void s_mbar_expect_tx(void* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(s_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void s_tma_load_1d(void* dst, const void* src, uint32_t bytes, void* bar, uint64_t policy) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;" ::
          "r"(s_u32(dst)),
      "l"(src), "r"(bytes), "r"(s_u32(bar)), "l"(policy)
      : "memory");
}

__device__ __forceinline__ uint32_t rank2(const uint32_t* bits, const uint16_t* pref, uint32_t key) {
  return (uint32_t)pref[key >> 5] + __popc(bits[key >> 5] & ((1u << (key & 31)) - 1u));
}

// ---- statistical outlier removal: mean of the k smallest neighbour distances (cloud_oracle.cpp step 4) ----
// The k smallest d are the square roots of the k smallest d^2 (sqrt is monotonic and correctly rounded), and
// they are added in ascending order either way -- so the selection runs on d^2 and only k square roots are taken.
template <int K>
struct TopK {
  float v[K];
  __device__ __forceinline__ void init() {
#pragma unroll
    for (int t = 0; t < K; ++t) v[t] = __int_as_float(0x7f800000);
  }
  __device__ __forceinline__ void insert(float x) {  // branch-free insertion into the ascending array
#pragma unroll
    for (int t = 0; t < K; ++t) {
      const float lo = fminf(v[t], x), hi = fmaxf(v[t], x);
      v[t] = lo;
      x = hi;
    }
  }
};
__device__ __forceinline__ float dist2(float2 o, float2 me) {
  const float dx = __fsub_rn(o.x, me.x), dy = __fsub_rn(o.y, me.y);
  return __fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy));
}
__device__ __forceinline__ void cswap(float& a, float& b) {
  const float lo = fminf(a, b), hi = fmaxf(a, b);
  a = lo;
  b = hi;
}
// optimal 19-exchange sorting network for 8 values (ascending)
__device__ __forceinline__ void sort8(float* v) {
  cswap(v[0], v[2]); cswap(v[1], v[3]); cswap(v[4], v[6]); cswap(v[5], v[7]);
  cswap(v[0], v[4]); cswap(v[1], v[5]); cswap(v[2], v[6]); cswap(v[3], v[7]);
  cswap(v[0], v[1]); cswap(v[2], v[3]); cswap(v[4], v[5]); cswap(v[6], v[7]);
  cswap(v[2], v[4]); cswap(v[3], v[5]);
  cswap(v[1], v[4]); cswap(v[3], v[6]);
  cswap(v[1], v[2]); cswap(v[3], v[4]); cswap(v[5], v[6]);
}
// a[0..8) and b[0..8) ascending -> a = the 8 smallest of the 16, ascending
__device__ __forceinline__ void merge_low8(float* a, const float* b) {
#pragma unroll
  for (int i = 0; i < 8; ++i) a[i] = fminf(a[i], b[7 - i]);  // bitonic
  cswap(a[0], a[4]); cswap(a[1], a[5]); cswap(a[2], a[6]); cswap(a[3], a[7]);
  cswap(a[0], a[2]); cswap(a[1], a[3]); cswap(a[4], a[6]); cswap(a[5], a[7]);
  cswap(a[0], a[1]); cswap(a[2], a[3]); cswap(a[4], a[5]); cswap(a[6], a[7]);
}
__device__ __forceinline__ float mean_of_smallest(const float* d2_sorted, int kmax, uint32_t k) {
  float sum = 0.0f;
#pragma unroll
  for (int t = 0; t < 32; ++t)
    if (t < kmax && (uint32_t)t < k) sum = __fadd_rn(sum, __fsqrt_rn(d2_sorted[t]));
  return __fdiv_rn(sum, __uint2float_rn(k));
}
// window form (more than 33 points), sor_k <= 8: sorting networks over the 32 candidates, 8 at a time
template <bool WRAP>
__device__ __forceinline__ float sor_mean_win8(const float2* px, uint32_t m, uint32_t i, uint32_t k) {
  const float2 me = px[i];
  float best[8], cur[8];
#pragma unroll
  for (int g = 0; g < 4; ++g) {
    float* dst = g == 0 ? best : cur;
#pragma unroll
    for (int t = 0; t < 4; ++t) {
      const uint32_t o = (uint32_t)(g * 4 + t + 1);
      uint32_t jm = i - o, jp = i + o;
      if (WRAP) {  // (i - o) mod m, (i + o) mod m with o <= 16 < m; interior points (WRAP = false) need neither
        jm = i + m - o;
        if (jm >= m) jm -= m;
        if (jp >= m) jp -= m;
      }
      dst[2 * t] = dist2(px[jm], me);
      dst[2 * t + 1] = dist2(px[jp], me);
    }
    if (g == 0) {
      sort8(best);
    } else {
      // the neighbours further away in angle rarely beat the eight nearest found so far: when no lane of the warp
      // holds a candidate below its current eighth-smallest, sorting and merging the group would change nothing
      const float lo = fminf(fminf(fminf(cur[0], cur[1]), fminf(cur[2], cur[3])), fminf(fminf(cur[4], cur[5]), fminf(cur[6], cur[7])));
      if (__any_sync(__activemask(), lo < best[7])) {
        sort8(cur);
        merge_low8(best, cur);
      }
    }
  }
  return mean_of_smallest(best, 8, k);
}
// any k <= 32, window or all-others form
__device__ __noinline__ float sor_mean_generic(const float2* px, uint32_t m, uint32_t i, uint32_t sor_k, bool all_others) {
  const float2 me = px[i];
  TopK<32> top;
  top.init();
  uint32_t nd = 0;
  if (all_others) {
    for (uint32_t j = 0; j < m; ++j)
      if (j != i) {
        top.insert(dist2(px[j], me));
        ++nd;
      }
  } else {
    for (uint32_t o = 1; o <= 16u; ++o) {
      uint32_t jm = i + m - o, jp = i + o;
      if (jm >= m) jm -= m;
      if (jp >= m) jp -= m;
      top.insert(dist2(px[jm], me));
      top.insert(dist2(px[jp], me));
    }
    nd = 32;
  }
  return mean_of_smallest(top.v, 32, min(sor_k, nd));
}

// floorf(x / v) without the division for all but a handful of points: q0 = x * RN(1/v) is within 2.4e-7 |q0| of the
// correctly rounded quotient, so both floor to the same integer unless q0 sits that close to one -- then (about 1 %
// of the points, the exact multiples of the voxel size among them) the division is done after all.
__device__ __forceinline__ int floor_div(float x, float v, float rv) {
  const float q0 = __fmul_rn(x, rv);
  const float n = rintf(q0);
  if (fabsf(__fsub_rn(q0, n)) <= __fmul_rn(fabsf(q0), 4e-7f)) return __float2int_rd(__fdiv_rn(x, v));
  return __float2int_rd(q0);
}
// voxel cell of a point (cloud_oracle.cpp step 5): (floorf(x / voxel), floorf(y / voxel)) packed into 32 bits;
// the host admits this kernel only when |cell index| < 32768 (range_max / voxel < 32000)
__device__ __forceinline__ uint32_t cell_key(float2 p, float voxel, float rvoxel) {
  const int ix = floor_div(p.x, voxel, rvoxel);
  const int iy = floor_div(p.y, voxel, rvoxel);
  return ((uint32_t)ix << 16) | ((uint32_t)iy & 0xFFFFu);
}
// llrintf(v * 65536) as a 32-bit integer: the host admits the fused voxel grid only for range_max < 1000 m
__device__ __forceinline__ int fix16(float v) { return __float2int_rn(__fmul_rn(v, 65536.0f)); }

// MODE: 0 LaserScan Mode B, 1 LaserScan Mode A, 2 PointCloud2.  EMIT: also write the ascended node buffer
// (MODE 0/1).  POST: (MODE 2) SOR and/or voxel grid in shared memory before anything is written.
// ---- rare paths of Mode B with duplicate measured keys, kept out of line so that they do not set the kernel's
// register count ---------------------------------------------------------------------------------------------------
// Which keys are held by more than one measured node?  Every measured node clears its key's bit and looks at what was
// there: the first node of a key finds it set, every further one finds it cleared and lists the key; then the bitmap is
// marked again.  Called by the whole block.
__device__ __noinline__ void vdup_list_keys(const uint2* tile, uint32_t n, uint32_t* bitsV, uint32_t* ndup,
                                            uint16_t* dupkey, uint32_t tid, uint32_t nthreads) {
  for (uint32_t i = tid; i < n; i += nthreads) {
    const uint2 nd = tile[i];
    if (__funnelshift_r(nd.x, nd.y, 16) != 0) {
      const uint32_t k = nd.x & 0xFFFFu, bit = 1u << (k & 31);
      if (!(atomicAnd(&bitsV[k >> 5], ~bit) & bit)) dupkey[atomicAdd(ndup, 1u)] = (uint16_t)k;
    }
  }
  __syncthreads();
  for (uint32_t i = tid; i < n; i += nthreads) {
    const uint2 nd = tile[i];
    if (__funnelshift_r(nd.x, nd.y, 16) != 0) atomicOr(&bitsV[(nd.x & 0xFFFFu) >> 5], 1u << (nd.x & 31u));
  }
  __syncthreads();
}
// Place pass of such a revolution (Mode B): every measured node beyond the first of a key shifts the larger keys by
// one; the measured nodes that share a key are set aside for vdup_place_shared.
__device__ __noinline__ void vdup_place_all(const uint2* tile, uint32_t n, const uint32_t* bitsV, const uint16_t* prefV,
                                            const uint16_t* dupkey, uint32_t n_listed, uint16_t* dupnode, uint32_t* n_shared,
                                            float* ranges, float* intens, uint32_t ob, uint32_t os, uint32_t q_shift,
                                            uint32_t q_mask, uint32_t tid, uint32_t nthreads) {
  for (uint32_t i = tid; i < n; i += nthreads) {
    const uint2 nd = tile[i];
    const uint32_t dist = __funnelshift_r(nd.x, nd.y, 16);
    if (dist == 0) continue;
    const uint32_t k = nd.x & 0xFFFFu;
    uint32_t rk = rank2(bitsV, prefV, k);
    bool shared = false;
    for (uint32_t j = 0; j < n_listed; ++j) {
      const uint32_t dk = dupkey[j];
      rk += (dk < k) ? 1u : 0u;
      shared = shared || (dk == k);
    }
    if (shared) {
      dupnode[atomicAdd(n_shared, 1u)] = (uint16_t)i;  // <= 2 * n_listed entries
    } else {
      const uint32_t o = ob + os * rk;
      ranges[o] = dist_to_m(dist);
      intens[o] = __fsub_rn(__uint_as_float(((nd.y >> q_shift) & q_mask) | 0x4B000000u), 8388608.0f);
    }
  }
}
// The measured nodes whose key is listed: one warp per node counts the measured nodes with the same key earlier in the
// buffer and stores the node's range and intensity at its slot.
__device__ __noinline__ void vdup_place_shared(const uint2* tile, const uint32_t* bitsV, const uint16_t* prefV,
                                               const uint16_t* dupkey, uint32_t n_listed, const uint16_t* dupnode,
                                               uint32_t n_shared, float* ranges, float* intens, uint32_t ob, uint32_t os,
                                               uint32_t q_shift, uint32_t q_mask, uint32_t warp, uint32_t lane,
                                               uint32_t nwarps) {
  for (uint32_t e = warp; e < n_shared; e += nwarps) {
    const uint32_t i = dupnode[e];
    const uint2 me = tile[i];
    const uint32_t k = me.x & 0xFFFFu;
    uint32_t before = 0;
    for (uint32_t j = lane; j < i; j += 32) {
      const uint2 o2 = tile[j];
      before += ((o2.x & 0xFFFFu) == k && __funnelshift_r(o2.x, o2.y, 16) != 0) ? 1u : 0u;
    }
    before = warp_sum(before);
    if (lane == 0) {
      uint32_t r = rank2(bitsV, prefV, k) + before;
      for (uint32_t j = 0; j < n_listed; ++j) r += (dupkey[j] < k) ? 1u : 0u;
      const uint32_t o = ob + os * r;
      ranges[o] = dist_to_m(__funnelshift_r(me.x, me.y, 16));
      intens[o] = __fsub_rn(__uint_as_float(((me.y >> q_shift) & q_mask) | 0x4B000000u), 8388608.0f);
    }
  }
}

template <int MODE, bool EMIT, bool POST, int TS>
__global__ void __launch_bounds__(TS, POST ? 2 : (EMIT ? 4 : (MODE == 0 ? 5 : 1))) scan_small_kernel(ScanBatchArgs a, SmallArgs p) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  constexpr bool MODE_A = (MODE == 1);
  constexpr bool CLOUD = (MODE == 2);
  constexpr int NW = TS / 32;
  constexpr uint32_t WPT = kWords / TS;  // bitmap words per thread in the prefix step
  static_assert(!(EMIT && CLOUD) && !(POST && !CLOUD), "variant");
  static_assert(kWords % TS == 0 && WPT % 4 == 0, "prefix layout");
  SmallCtl& ctl = *reinterpret_cast<SmallCtl*>(smem_raw);
  const uint32_t cap = p.cap;
  uint2* const tile0 = reinterpret_cast<uint2*>(smem_raw + kCtl);  // cap + 2 nodes
  unsigned char* q = smem_raw + kCtl + (size_t)cap * 8 + 16;
  float2* px = nullptr;
  uint8_t* pi = nullptr;
  uint32_t* bitsV = nullptr;
  uint16_t* prefV = nullptr;
  uint32_t* bitsA = nullptr;
  uint16_t* prefA = nullptr;
  unsigned char* acc = nullptr;
  if (POST) {
    px = reinterpret_cast<float2*>(q); q += (size_t)cap * 8;
    pi = q; q += cap;
    acc = q;  // 16 * cap bytes; the rank table lives at its start until the place pass is over
  }
  // Mode A needs no ranks among the measured points (see below): no bitmap of their keys
  constexpr bool USE_V = !MODE_A;
  // Mode B without the ascended buffer places a few duplicate MEASURED keys itself (see the place pass)
  constexpr bool VDUP = (MODE == 0) && !EMIT;
  if (USE_V) {
    bitsV = reinterpret_cast<uint32_t*>(q); q += kWords * 4;
    prefV = reinterpret_cast<uint16_t*>(q); q += kWords * 2;
  }
  if (EMIT) {
    bitsA = reinterpret_cast<uint32_t*>(q); q += kWords * 4;
    prefA = reinterpret_cast<uint16_t*>(q); q += kWords * 2;
  }
  // Mode A: per bin the smallest dist_m (as bits) and, among the points that have it, the smallest key | quality
  uint32_t* minv = nullptr;
  uint32_t* wkey = nullptr;
  if (MODE_A) {
    minv = reinterpret_cast<uint32_t*>(q);
    wkey = minv + cap;
  }


  const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const bool new_proto = a.is_new_protocol != 0;
  const bool inverted = a.inverted != 0;
  const uint64_t pol_stream = l2_policy_evict_first();
  const uint32_t q_shift = new_proto ? 16u : 18u, q_mask = new_proto ? 0xFFu : 0x3Fu;
  const float w_rmin = a.range_min, w_rmax = a.range_max, w_imin = a.intensity_min;
  auto intensity_of = [&](uint32_t y) {
    return __fsub_rn(__uint_as_float(((y >> q_shift) & q_mask) | 0x4B000000u), 8388608.0f);
  };
  const bool want_scan = CLOUD ? false : (EMIT ? (a.ranges != nullptr) : true);

  if (tid == 0) {
    s_mbar_init(&ctl.full, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  uint32_t parity = 0;

  for (uint32_t s = blockIdx.x; s < a.n_scans; s += gridDim.x) {
    const uint2 view = a.views ? a.views[s] : make_uint2(0u, a.counts[s]);  // {first, count}
    const uint32_t n = view.y;
    // caller error (a count above the stride or the context's limit, a view that runs past the node buffer):
    // report, touch nothing
    if (n > a.stride || n > p.max_nodes || (a.views && (unsigned long long)view.x + n > a.nodes_total)) {
      if (tid == 0) {
        if (a.status) a.status[s] = 0x80008000u;  // SL_RESULT_INVALID_DATA
        if (a.path) a.path[s] = 0u;
        if (a.beam_counts) a.beam_counts[s] = 0u;
        if (a.angle_inc) a.angle_inc[s] = 0.0f;
      }
      continue;
    }
    if (n == 0) {  // ascendScanData: OPERATION_FAIL; publish_scan: nodes.empty() -> return
      if (tid == 0) {
        if (a.status) a.status[s] = a.apply_ascend ? kResultOperationFail : kResultOk;
        if (a.path) a.path[s] = 0u;
        if (a.beam_counts) a.beam_counts[s] = 0u;
        if (a.angle_inc) a.angle_inc[s] = 0.0f;
      }
      continue;
    }
    const uint2* base = a.views ? a.nodes + view.x : a.nodes + (size_t)s * a.stride;

    // ---- stage the revolution (every thread is past the previous scan: its last barrier) -----------
    // Bulk copies move whole 16-byte units from 16-byte aligned addresses.  A batch scan starts aligned (even
    // stride) and an odd count is rounded up into the scan's own stride; a VIEW may start on an odd node: the
    // copy then starts one node early and the tile is read from `shift` on.  A view whose rounded copy would run
    // past the end of the node buffer is staged with ordinary loads instead.
    uint32_t shift = 0;
    bool bulk = p.use_tma != 0;
    if (a.views) {
      shift = (uint32_t)((reinterpret_cast<uintptr_t>(base) >> 3) & 1u);
      const unsigned long long first = view.x;
      bulk = bulk && (first - shift + ((n + shift + 1u) & ~1u) <= a.nodes_total);
    }
    const uint2* const tile = tile0 + shift;
    if (bulk) {
      if (tid == 0) {
        // the tile region may have been written with ordinary stores (voxel table): order them before the
        // asynchronous-proxy write of the copy
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        const uint32_t bytes = ((n + shift + 1u) & ~1u) * 8u;
        s_mbar_expect_tx(&ctl.full, bytes);
        s_tma_load_1d(tile0, base - shift, bytes, &ctl.full, pol_stream);
      }
    } else {
      for (uint32_t i = tid; i < n; i += TS) tile0[shift + i] = ld_stream_v2(base + i);
    }
    {
      if (USE_V) {
        uint4* b4 = reinterpret_cast<uint4*>(bitsV);
        for (uint32_t w = tid; w < kWords / 4; w += TS) b4[w] = make_uint4(0, 0, 0, 0);
      }
      if (EMIT) {
        uint4* a4 = reinterpret_cast<uint4*>(bitsA);
        for (uint32_t w = tid; w < kWords / 4; w += TS) a4[w] = make_uint4(0, 0, 0, 0);
      }
      if (MODE_A) {  // "nothing in this bin yet" for every bin (minv and wkey are adjacent; cap is a multiple of 64)
        uint4* f4 = reinterpret_cast<uint4*>(minv);
        for (uint32_t w = tid; w < cap / 2; w += TS) f4[w] = make_uint4(0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu);
      }
      if (tid == 0) {
        ctl.first_valid = 0xFFFFFFFFu;
        ctl.fallback = 0;
        if (EMIT || VDUP) {
          ctl.d.ndup = 0;
          ctl.d.ndupnode = 0;
        }
      }
    }
    __syncthreads();
    if (bulk) {
      s_mbar_wait(&ctl.full, parity);
      parity ^= 1u;
    }

    // ---- mark: one shared-memory atomicOr per kept key -----------------------------------------------
    uint32_t cnt = 0, fmin = 0xFFFFFFFFu;
    // Mode A (no bitmap of the measured keys) and the ascended-buffer variants (which mark the measured keys together
    // with the final keys, below) only need the number of measured nodes and the first of them here: two nodes per
    // 128-bit load
    const bool light = (!USE_V || EMIT) && !CLOUD && shift == 0;
    if (light) {
      const uint4* t4 = reinterpret_cast<const uint4*>(tile0);
#pragma unroll 4
      for (uint32_t w = tid; w < n / 2; w += TS) {
        const uint4 v = t4[w];
        const uint32_t m0 = (((v.x & 0xFFFF0000u) | (v.y & 0xFFFFu)) != 0u) ? 1u : 0u;
        const uint32_t m1 = (((v.z & 0xFFFF0000u) | (v.w & 0xFFFFu)) != 0u) ? 1u : 0u;
        cnt += m0 + m1;
        if (EMIT && (m0 | m1)) fmin = min(fmin, 2u * w + (m0 ^ 1u));
      }
      if ((n & 1u) && tid == 0) {
        const uint2 v = tile0[n - 1];
        if (((v.x & 0xFFFF0000u) | (v.y & 0xFFFFu)) != 0u) {
          ++cnt;
          if (EMIT) fmin = min(fmin, n - 1u);
        }
      }
    } else {
#pragma unroll 4
      for (uint32_t i = tid; i < n; i += TS) {
        const uint2 nd = tile[i];
        const uint32_t dist = __funnelshift_r(nd.x, nd.y, 16);
        bool valid = dist != 0;
        if (CLOUD) valid = valid && cloud_keep(dist_to_m(dist), intensity_of(nd.y), w_rmin, w_rmax, w_imin);
        if (valid) {
          if (USE_V) {
            const uint32_t k = nd.x & 0xFFFFu;
            atomicOr(&bitsV[k >> 5], 1u << (k & 31));
          }
          ++cnt;
          if (EMIT) fmin = min(fmin, i);
        }
      }
    }
    cnt = warp_sum(cnt);
    if (lane == 0) ctl.red[warp] = cnt;
    if (EMIT) {
      fmin = warp_min(fmin);
      if (lane == 0 && fmin != 0xFFFFFFFFu) atomicMin(&ctl.first_valid, fmin);
    }
    __syncthreads();
    uint32_t M = 0;
#pragma unroll
    for (int w = 0; w < NW; ++w) M += ctl.red[w];

    if (M == 0) {
      // ascendScanData: OPERATION_FAIL, buffer untouched; publish_scan: nothing to publish
      if (tid == 0) {
        if (a.status) a.status[s] = a.apply_ascend ? kResultOperationFail : kResultOk;
        if (a.path) a.path[s] = 0u;
        if (a.beam_counts) a.beam_counts[s] = 0u;
        if (a.angle_inc) a.angle_inc[s] = 0.0f;
      }
      if (EMIT) {
        uint2* out = a.nodes_out + (size_t)s * a.stride;
        for (uint32_t i = tid; i < n; i += TS) out[i] = tile[i];
      }
      __syncthreads();
      continue;
    }

    // ---- ascended buffer: final keys of ALL nodes into the second bitmap --------------------------------
    const float step = ascend_step(n);
    uint32_t front_key = 0;
    float front_deg = 0.0f;
    if (EMIT) {
      if (tid == 0) {
        // head tune: serial, only node 0's result survives (reference sl_lidar_driver.cpp:133-147)
        const uint32_t f = ctl.first_valid;
        ctl.front_key = ascend_head_key(node_key(tile[f]), f, step);
      }
      __syncthreads();
      front_key = ctl.front_key;
      front_deg = key_to_deg(front_key);
#pragma unroll 2
      for (uint32_t i = tid; i < n; i += TS) {
        const uint2 nd = tile[i];
        const uint32_t dist = __funnelshift_r(nd.x, nd.y, 16);
        uint32_t fk = nd.x & 0xFFFFu;
        if (dist == 0) {
          // the final key of an unmeasured node is written back into the shared-memory copy: the place pass then
          // reads every node's final key where it reads the node
          fk = (i == 0) ? front_key : ascend_fill_key(front_deg, i, step);
          tile0[shift + i].x = (nd.x & 0xFFFF0000u) | fk;
        } else if (USE_V && light) {
          atomicOr(&bitsV[fk >> 5], 1u << (fk & 31));  // (the light first pass marks nothing)
        }
        atomicOr(&bitsA[fk >> 5], 1u << (fk & 31));
      }
      __syncthreads();
    }

    // ---- exclusive popcount prefix over the bitmap words ------------------------------------------------
    if constexpr (USE_V || EMIT) {
      uint32_t wv[WPT], wa[WPT];
      uint32_t sv = 0, sa = 0;
#pragma unroll
      for (uint32_t j = 0; j < WPT / 4; ++j) {
        if (USE_V) {
          const uint4 t = reinterpret_cast<const uint4*>(bitsV)[tid * (WPT / 4) + j];
          wv[4 * j] = t.x; wv[4 * j + 1] = t.y; wv[4 * j + 2] = t.z; wv[4 * j + 3] = t.w;
        } else {
          wv[4 * j] = wv[4 * j + 1] = wv[4 * j + 2] = wv[4 * j + 3] = 0u;
        }
        if (EMIT) {
          const uint4 u = reinterpret_cast<const uint4*>(bitsA)[tid * (WPT / 4) + j];
          wa[4 * j] = u.x; wa[4 * j + 1] = u.y; wa[4 * j + 2] = u.z; wa[4 * j + 3] = u.w;
        }
      }
#pragma unroll
      for (uint32_t j = 0; j < WPT; ++j) {
        if (USE_V) sv += __popc(wv[j]);
        if (EMIT) sa += __popc(wa[j]);
      }
      const uint32_t iv = USE_V ? warp_inclusive_scan(sv) : 0u;
      const uint32_t ia = EMIT ? warp_inclusive_scan(sa) : 0u;
      if (lane == 31) {
        ctl.red[32 + warp] = iv;
        ctl.red[64 + warp] = ia;
      }
      __syncthreads();
      if (warp == 0) {
        const uint32_t tv = lane < NW ? ctl.red[32 + lane] : 0u;
        const uint32_t ta = lane < NW ? ctl.red[64 + lane] : 0u;
        const uint32_t cv = warp_inclusive_scan(tv), ca = warp_inclusive_scan(ta);
        if (lane < NW) {
          ctl.red[32 + lane] = cv - tv;
          ctl.red[64 + lane] = ca - ta;
        }
        if (lane == 31) {
          ctl.totV = cv;
          ctl.totA = ca;
        }
      }
      __syncthreads();
      uint32_t pv = ctl.red[32 + warp] + iv - sv;
      uint32_t pa = ctl.red[64 + warp] + ia - sa;
#pragma unroll
      for (uint32_t j = 0; j < WPT; ++j) {
        if (USE_V) {
          prefV[tid * WPT + j] = (uint16_t)pv;
          pv += __popc(wv[j]);
        }
        if (EMIT) {
          prefA[tid * WPT + j] = (uint16_t)pa;
          pa += __popc(wa[j]);
        }
      }
      __syncthreads();
    }

    // duplicate keys among the measured nodes (fewer distinct keys than kept nodes) -> general kernel (stable tie
    // rule); Mode A looks only for the duplicates that matter to it, in its winner pass below.  Duplicates among the
    // FINAL keys (typically the fill key of an unmeasured node landing on a measured node's key) only move entries of
    // the ascended buffer: up to kMaxDup of them are resolved here (place pass + fix-up), more go to the general kernel.
    // The same goes for duplicate MEASURED keys in Mode B without the ascended buffer (e.g. the first and the last
    // node of a revolution meeting on one key: ~1 % of the revolutions of the capsule -> LaserScan chain).
    const uint32_t D = EMIT ? n - ctl.totA : 0u;  // nodes beyond the first of their final key
    const uint32_t DV = VDUP ? M - ctl.totV : 0u;  // measured nodes beyond the first of their key
    if ((USE_V && !VDUP && ctl.totV != M) || (VDUP && DV > kMaxDup) || (EMIT && D > kMaxDup)) {
      if (tid == 0) a.fallback_list[atomicAdd(a.fallback_count, 1u)] = s;
      __syncthreads();
      continue;
    }
    if (EMIT && D) {
      // (rare) which keys are they?  Every node clears its key's bit and looks at what was there: the first node of
      // a key finds it set, every further one finds it cleared and lists the key; then the bitmap is marked again.
      for (uint32_t i = tid; i < n; i += TS) {
        const uint32_t fk = tile[i].x & 0xFFFFu, bit = 1u << (fk & 31);
        if (!(atomicAnd(&bitsA[fk >> 5], ~bit) & bit)) ctl.d.dupkey[atomicAdd(&ctl.d.ndup, 1u)] = (uint16_t)fk;  // D entries
      }
      __syncthreads();
      for (uint32_t i = tid; i < n; i += TS) {
        const uint32_t fk = tile[i].x & 0xFFFFu;
        atomicOr(&bitsA[fk >> 5], 1u << (fk & 31));
      }
      __syncthreads();
    }

    // ---- place ------------------------------------------------------------------------------------------
    float* ranges = want_scan ? a.ranges + (size_t)s * a.stride : nullptr;
    float* intens = want_scan ? a.intensities + (size_t)s * a.stride : nullptr;
    float4* cloud = CLOUD ? a.xyzi + (size_t)s * a.stride : nullptr;
    uint2* nodes_out = EMIT ? a.nodes_out + (size_t)s * a.stride : nullptr;
    const float inc = angle_increment(M, MODE_A);
    // Mode B output slot = ob + os * rank in wrapping u32 arithmetic (reference rplidar_node.cpp:673)
    const uint32_t ob = inverted ? M - 1u : 0u, os = inverted ? 0xFFFFFFFFu : 1u;
    const ptrdiff_t i_minus_r = reinterpret_cast<char*>(intens) - reinterpret_cast<char*>(ranges);
    // (two instances: revolutions with shared final keys are rare and must not slow the loop of the others down)
    auto place = [&](auto has_dup) {
      constexpr bool HAS_DUP = decltype(has_dup)::value;
      constexpr int kUnroll = HAS_DUP ? 1 : 4;  // (the rare instance must not set the kernel's register count)
#pragma unroll kUnroll
      for (uint32_t i = tid; i < n; i += TS) {
        const uint2 nd = tile[i];
        const uint32_t k = nd.x & 0xFFFFu;
        const uint32_t dist = __funnelshift_r(nd.x, nd.y, 16);
        uint32_t measured = dist != 0 ? 1u : 0u;
        if (EMIT) {  // k is the FINAL key here
          uint32_t rA = rank2(bitsA, prefA, k);  // rank among the distinct final keys
          bool defer = false;
          if constexpr (HAS_DUP) {
            // every node beyond the first of a key shifts the larger keys by one; the nodes that share a key are
            // ordered by buffer position (stable rule) in the fix-up below
            for (uint32_t j = 0; j < D; ++j) {
              const uint32_t dk = ctl.d.dupkey[j];
              rA += (dk < k) ? 1u : 0u;
              defer = defer || (dk == k);
            }
            if (defer) ctl.d.dupnode[atomicAdd(&ctl.d.ndupnode, 1u)] = (uint16_t)i;  // <= 2 * D entries
          }
          if (!defer) st_hint_v2(nodes_out + rA, nd, pol_stream);
        }
        if (!CLOUD && !want_scan) continue;
        const float dm = dist_to_m(dist);
        if (MODE_A) {
          // Mode A needs no order at all (reference rplidar_node.cpp:630-660): a bin keeps the smallest dist_m of the
          // points that fall into it -- dist_m >= 0, so its bit pattern orders like the value
          if (measured) {
            const uint32_t b = (uint32_t)mode_a_bin_fast(k, M, inc, inverted);  // < M <= 8192
            atomicMin(&minv[b], __float_as_uint(dm));
          }
          continue;
        }
        const uint32_t rk = rank2(bitsV, prefV, k);
        if (CLOUD) {  // polar -> xyz at the rank among kept points (oracle/cloud_oracle.cpp steps 1-3)
          const float it = intensity_of(nd.y);
          if (!cloud_keep(dm, it, w_rmin, w_rmax, w_imin)) measured = 0;
          const float2 cs = __ldg(a.trig + k);
          const float x = __fmul_rn(dm, cs.x), y = __fmul_rn(dm, cs.y);
          if (POST) {
            if (measured) {
              px[rk] = make_float2(x, y);
              pi[rk] = (uint8_t)((nd.y >> q_shift) & q_mask);
            }
          } else {
            st_f32x4_if(cloud + rk, make_float4(x, y, 0.0f, it), pol_stream, measured);
          }
        } else {  // Mode B: reference rplidar_node.cpp:661-677
          const uint32_t o = ob + os * rk;
          const float it = intensity_of(nd.y);
          float* pr = ranges + o;
          st_f32_if(pr, dm, pol_stream, measured);
          st_f32_if(reinterpret_cast<float*>(reinterpret_cast<char*>(pr) + i_minus_r), it, pol_stream, measured);
        }
      }
    };
    if (VDUP && DV) {  // (rare) the whole place pass of such a revolution runs out of line
      vdup_list_keys(tile, n, bitsV, &ctl.d.ndup, ctl.d.dupkey, tid, TS);
      vdup_place_all(tile, n, bitsV, prefV, ctl.d.dupkey, DV, ctl.d.dupnode, &ctl.d.ndupnode, ranges, intens, ob, os, q_shift, q_mask,
                     tid, TS);
    } else if (EMIT && D) {
      place(std::true_type{});
    } else {
      place(std::false_type{});
    }
    __syncthreads();

    // ---- ascended buffer, nodes with a shared final key: position = nodes with a smaller key + nodes with the same
    // key earlier in the buffer (stable rule); one warp per such node counts the latter over the tile
    if (EMIT && D) {
      const uint32_t nshared = ctl.d.ndupnode;
      for (uint32_t e = warp; e < nshared; e += NW) {
        const uint32_t i = ctl.d.dupnode[e];
        const uint2 me = tile[i];
        const uint32_t k = me.x & 0xFFFFu;
        uint32_t before = 0;
        for (uint32_t j = lane; j < i; j += 32) before += ((tile[j].x & 0xFFFFu) == k) ? 1u : 0u;
        before = warp_sum(before);
        if (lane == 0) {
          uint32_t r = rank2(bitsA, prefA, k) + before;
          for (uint32_t j = 0; j < D; ++j) r += (ctl.d.dupkey[j] < k) ? 1u : 0u;
          nodes_out[r] = me;
        }
      }
    }

    // ---- Mode B, measured nodes with a shared key: slot = measured nodes with a smaller key + measured nodes with the
    // same key earlier in the buffer (stable rule)
    if (VDUP && DV)
      vdup_place_shared(tile, bitsV, prefV, ctl.d.dupkey, DV, ctl.d.dupnode, ctl.d.ndupnode, ranges, intens, ob, os, q_shift,
                        q_mask, warp, lane, NW);

    // ---- Mode A, continued: among the points that hold their bin's minimum the first in ascending key order wins
    // (strict '<' in the reference) -- the smallest key | quality; then one thread per bin writes (dist_m, intensity)
    // or (+inf, 0) for a bin nothing fell into.  Lanes hold consecutive bins: coalesced stores.
    // Duplicate keys: equal keys fall into the same bin, and the order among them only matters when two of them hold
    // the bin's minimum with different qualities (the stable rule then takes the first in buffer order).  The second
    // of two such points to arrive finds the first one's key in the value its atomicMin returns -- unless a smaller
    // key is already there, and then neither wins.  Such a scan goes to the general kernel, like every scan with
    // duplicate keys does in the other modes.
    if constexpr (MODE_A) if (want_scan) {
      bool conflict = false;
#pragma unroll 4
      for (uint32_t i = tid; i < n; i += TS) {
        const uint2 nd = tile[i];
        const uint32_t dist = __funnelshift_r(nd.x, nd.y, 16);
        if (dist != 0) {
          const uint32_t k = nd.x & 0xFFFFu;
          const uint32_t b = (uint32_t)mode_a_bin_fast(k, M, inc, inverted);
          if (__float_as_uint(dist_to_m(dist)) == minv[b]) {
            const uint32_t v = (k << 8) | ((nd.y >> 16) & 0xFFu);
            const uint32_t old = atomicMin(&wkey[b], v);
            conflict = conflict || ((old ^ v) - 1u < 255u);  // same key, another quality
          }
        }
      }
      if (conflict) ctl.fallback = 1u;
      __syncthreads();
      if (ctl.fallback != 0u) {  // block-uniform: set before the barrier, cleared at the start of the next scan
        if (tid == 0) a.fallback_list[atomicAdd(a.fallback_count, 1u)] = s;
        __syncthreads();
        continue;
      }
      const float kInf = __int_as_float(0x7f800000);
      for (uint32_t b = tid; b < M; b += TS) {
        const uint32_t mb = minv[b];
        const bool hit = mb != 0xFFFFFFFFu;
        st_f32_if(ranges + b, hit ? __uint_as_float(mb) : kInf, pol_stream, 1u);
        st_f32_if(intens + b, hit ? quality_to_intensity(wkey[b] & 0xFFu, new_proto) : 0.0f, pol_stream, 1u);
      }
    }

    uint32_t m_out = M;
    if constexpr (POST) {
      uint32_t m = M;
      // ---- step 4: statistical outlier removal over the +-16 angular neighbours --------------------------
      if (p.sor_k > 0 && m >= 2) {
        unsigned long long* qv = reinterpret_cast<unsigned long long*>(acc);  // [cap] (rank table is dead)
        const bool all_others = (m - 1) <= 32u;
        long long s1 = 0;
        unsigned long long s2 = 0;
        for (uint32_t i = tid; i < m; i += TS) {
          float mean;
          if (all_others || p.sor_k > 8u) {
            mean = sor_mean_generic(px, m, i, p.sor_k, all_others);
          } else if (__all_sync(__activemask(), i >= 16u && i + 16u < m)) {  // the whole warp is clear of both ends
            mean = sor_mean_win8<false>(px, m, i, p.sor_k);
          } else {
            mean = sor_mean_win8<true>(px, m, i, p.sor_k);
          }
          const long long qq = __float2ll_rn(__fmul_rn(mean, 65536.0f));  // llrintf
          qv[i] = (unsigned long long)qq;
          s1 += qq;
          s2 += (unsigned long long)qq * (unsigned long long)qq;
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
          s1 += __shfl_xor_sync(0xffffffffu, s1, o);
          s2 += __shfl_xor_sync(0xffffffffu, s2, o);
        }
        if (tid == 0) {
          ctl.s1 = 0;
          ctl.s2 = 0;
        }
        __syncthreads();
        if (lane == 0) {  // exact integer sums: the order of the atomics cannot change them
          atomicAdd(reinterpret_cast<unsigned long long*>(&ctl.s1), (unsigned long long)s1);
          atomicAdd(&ctl.s2, s2);
        }
        __syncthreads();
        if (tid == 0) {
          const double dn = (double)m;
          const double t1 = (double)ctl.s1, t2 = (double)ctl.s2;
          const double mean = __ddiv_rn(t1, dn);
          const double sq = __ddiv_rn(__dmul_rn(t1, t1), dn);
          double var = __ddiv_rn(__dsub_rn(t2, sq), __dsub_rn(dn, 1.0));
          if (!(var > 0.0)) var = 0.0;
          ctl.thr = __dadd_rn(mean, __dmul_rn((double)p.sor_alpha, __dsqrt_rn(var)));
        }
        __syncthreads();
        const double thr = ctl.thr;
        // stable in-place compaction: every thread owns a contiguous run of at most 8 points
        constexpr uint32_t PMAX = kSmallPostMaxNodes / TS;
        const uint32_t P = (m + TS - 1) / TS;
        const uint32_t lo = tid * P;
        float2 kx[PMAX];
        uint8_t ki[PMAX];
        uint32_t mask = 0, nk = 0;
#pragma unroll
        for (uint32_t j = 0; j < PMAX; ++j) {
          const uint32_t i = lo + j;
          kx[j] = make_float2(0.f, 0.f);
          ki[j] = 0;
          if (j < P && i < m) {
            kx[j] = px[i];
            ki[j] = pi[i];
            if ((double)(long long)qv[i] <= thr) {
              mask |= 1u << j;
              ++nk;
            }
          }
        }
        const uint32_t inc_w = warp_inclusive_scan(nk);
        if (lane == 31) ctl.red[warp] = inc_w;
        __syncthreads();  // all reads of px/pi/qv are done
        uint32_t wbase = 0, tot = 0;
#pragma unroll
        for (int w = 0; w < NW; ++w) {
          const uint32_t t = ctl.red[w];
          if ((uint32_t)w < warp) wbase += t;
          tot += t;
        }
        uint32_t pos = wbase + inc_w - nk;
#pragma unroll
        for (uint32_t j = 0; j < PMAX; ++j)
          if (mask & (1u << j)) {
            px[pos] = kx[j];
            pi[pos] = ki[j];
            ++pos;
          }
        m = tot;
        __syncthreads();
      }
      m_out = m;

      if (p.voxel > 0.0f && m > 0) {
        // ---- step 5: voxel grid -------------------------------------------------------------------------
        // acc: key32[cap] | dx[cap] | dy[cap] | cs[cap]; table of cell leaders in the (dead) tile buffer
        uint32_t* key32 = reinterpret_cast<uint32_t*>(acc);
        int* dxs = reinterpret_cast<int*>(acc + (size_t)cap * 4);
        int* dys = reinterpret_cast<int*>(acc + (size_t)cap * 8);
        uint32_t* cs = reinterpret_cast<uint32_t*>(acc + (size_t)cap * 12);
        uint32_t* table = reinterpret_cast<uint32_t*>(tile0);
        const uint32_t nslots = 2u * cap;
        constexpr uint32_t kEmpty = 0xFFFFFFFFu;
        constexpr uint32_t PMAX = kSmallPostMaxNodes / TS;
        {
          uint4* t4 = reinterpret_cast<uint4*>(table);
          const uint4 e = make_uint4(kEmpty, kEmpty, kEmpty, kEmpty);
          for (uint32_t w = tid; w < nslots / 4; w += TS) t4[w] = e;
        }
        const float rvoxel = __frcp_rn(p.voxel);
        for (uint32_t i = tid; i < m; i += TS) {
          key32[i] = cell_key(px[i], p.voxel, rvoxel);
          dxs[i] = 0;
          dys[i] = 0;
          cs[i] = 0;
        }
        __syncthreads();
        // insert: a slot holds the smallest point index seen so far of ONE cell (the key of a slot never
        // changes once it is taken: atomicMin only swaps members of the same cell).  Points arrive in angle
        // order, so the members of a cell are mostly neighbours: within a warp only the first point of a run of
        // equal cells goes to the table, the others take its slot by shuffle (they cannot be the cell's leader).
        uint32_t myslot[PMAX];
#pragma unroll
        for (uint32_t j = 0; j < PMAX; ++j) {
          myslot[j] = 0;
          if (j * TS >= m) continue;  // (uniform) chunks past the end of the cloud: nothing to do
          const uint32_t i = tid + j * TS;
          const bool live = i < m;
          const uint32_t key = live ? key32[i] : 0u;
          const uint32_t kprev = __shfl_up_sync(0xffffffffu, key, 1);
          const bool head = live && (lane == 0 || key != kprev);
          uint32_t h = 0;
          if (head) {
            h = __umulhi(key * 0x9E3779B1u, nslots);
            for (;;) {
              uint32_t v = *reinterpret_cast<volatile uint32_t*>(&table[h]);
              if (v == kEmpty) {
                v = atomicCAS(&table[h], kEmpty, i);
                if (v == kEmpty) break;
              }
              if (key32[v] == key) {
                atomicMin(&table[h], i);
                break;
              }
              if (++h == nslots) h = 0;
            }
          }
          __syncwarp();
          const uint32_t heads = __ballot_sync(0xffffffffu, head);
          const uint32_t below = heads & (0xFFFFFFFFu >> (31u - lane));  // heads at or below this lane (lane 0 is one)
          const int src = 31 - __clz((int)(below | 1u));
          myslot[j] = __shfl_sync(0xffffffffu, h, src);
        }
        __syncthreads();
        // accumulate relative to the cell leader (32-bit integers: |delta| <= voxel * 65536 + 2 and the host
        // admits voxel <= 4 m, so 4096 members cannot overflow), leaders flagged for the ordering
        uint32_t leadflag = 0;
#pragma unroll
        for (uint32_t j = 0; j < PMAX; ++j) {
          if (j * TS >= m) {  // (uniform)
            if (lane == 0) ctl.chunk_base[j * NW + warp] = 0u;
            continue;
          }
          const uint32_t i = tid + j * TS;
          bool is_lead = false;
          if (i < m) {
            const uint32_t lead = table[myslot[j]];
            const uint32_t inten = pi[i];
            if (lead == i) {
              is_lead = true;
              atomicAdd(&cs[i], inten);
            } else {
              const float2 me = px[i], ld = px[lead];
              atomicAdd(&dxs[lead], fix16(me.x) - fix16(ld.x));
              atomicAdd(&dys[lead], fix16(me.y) - fix16(ld.y));
              atomicAdd(&cs[lead], (1u << 20) + inten);
            }
          }
          const uint32_t bal = __ballot_sync(0xffffffffu, is_lead);
          if (is_lead) leadflag |= 1u << j;
          if (lane == 0) ctl.chunk_base[j * NW + warp] = __popc(bal);
          // position of this leader among the leaders of its (chunk, warp) group
          myslot[j] = __popc(bal & ((1u << lane) - 1u));
        }
        __syncthreads();
        // cells are emitted in the order of their first member = index order of the leaders: exclusive scan
        // over the (chunk, warp) counts, chunk-major
        if (warp == 0) {
          constexpr uint32_t G = PMAX * NW;          // groups
          constexpr uint32_t GPL = (G + 31) / 32;     // per lane
          uint32_t v[GPL], sum = 0;
#pragma unroll
          for (uint32_t t = 0; t < GPL; ++t) {
            const uint32_t g = lane * GPL + t;
            v[t] = g < G ? ctl.chunk_base[g] : 0u;
            sum += v[t];
          }
          const uint32_t incl = warp_inclusive_scan(sum);
          uint32_t run = incl - sum;
#pragma unroll
          for (uint32_t t = 0; t < GPL; ++t) {
            const uint32_t g = lane * GPL + t;
            if (g < G) ctl.chunk_base[g] = run;
            run += v[t];
          }
          if (lane == 31) ctl.count_out = incl;
        }
        __syncthreads();
        // The leaders are a third of the points, scattered over the lanes: writing their cells from where they sit
        // would run the (double-precision) body for every warp with a third of its lanes.  So the leaders are first
        // listed densely in output order (the cell keys are dead: their array holds the list), then one thread per
        // CELL does the arithmetic -- full warps, and the stores of a warp are 512 contiguous bytes.
        uint16_t* lead16 = reinterpret_cast<uint16_t*>(key32);
#pragma unroll
        for (uint32_t j = 0; j < PMAX; ++j)
          if (leadflag & (1u << j)) lead16[ctl.chunk_base[j * NW + warp] + myslot[j]] = (uint16_t)(tid + j * TS);
        __syncthreads();
        const uint32_t n_cells = ctl.count_out;
        for (uint32_t pos = tid; pos < n_cells; pos += TS) {
          const uint32_t i = lead16[pos];
          const float2 ld = px[i];
          const uint32_t c = cs[i];
          const int qx = fix16(ld.x), qy = fix16(ld.y);
          float4 o;
          o.z = 0.0f;
          if ((c >> 20) == 0u) {
            // a cell of one point: sum / 65536 is exact in float (an integer below 2^24, or a float-valued integer)
            o.x = __fmul_rn(__int2float_rn(qx), 1.52587890625e-05f);
            o.y = __fmul_rn(__int2float_rn(qy), 1.52587890625e-05f);
            o.w = __uint2float_rn(c);
          } else {
            // (float)((double)sum / (65536.0 * count)): the double quotient from the correctly rounded reciprocal
            // and one residual step (Markstein) -- bit-identical to the division, a third of its instructions
            const uint32_t members = (c >> 20) + 1u;
            const double sx = (double)((long long)members * qx + (long long)dxs[i]);
            const double sy = (double)((long long)members * qy + (long long)dys[i]);
            const double cntd = (double)members;
            const double den = __dmul_rn(65536.0, cntd);
            const double rden = __drcp_rn(den);
            const double rcnt = __dmul_rn(rden, 65536.0);  // = RN(1 / count): scaling by 2^16 is exact
            auto quot = [](double a, double d, double r) {
              const double q0 = __dmul_rn(a, r);
              const double e = __fma_rn(-q0, d, a);
              return __fma_rn(e, r, q0);
            };
            o.x = __double2float_rn(quot(sx, den, rden));
            o.y = __double2float_rn(quot(sy, den, rden));
            o.w = __double2float_rn(quot((double)(c & 0xFFFFFu), cntd, rcnt));
          }
          st_f32x4_if(cloud + pos, o, pol_stream, 1u);
        }
        m_out = ctl.count_out;
        // the table was written with ordinary stores and the next scan's bulk copy lands on it
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      } else {
        // SOR only: the surviving points, in angle order
        for (uint32_t i = tid; i < m; i += TS) {
          const float2 v = px[i];
          st_f32x4_if(cloud + i, make_float4(v.x, v.y, 0.0f, small_uint_to_float(pi[i])), pol_stream, 1u);
        }
      }
    }

    __syncthreads();
    if (tid == 0) {
      if (a.status) a.status[s] = kResultOk;
      if (a.path) a.path[s] = 0u;
      if (a.beam_counts) a.beam_counts[s] = m_out;
      if (a.angle_inc) a.angle_inc[s] = inc;
    }
    // (the barrier at the top of the next scan's mark phase orders ctl reuse; the tile is not touched
    // before every thread has passed the barrier above)
  }
}

template <int MODE, bool EMIT, bool POST, int TS>
cudaError_t configure_one() {
  return cudaFuncSetAttribute(scan_small_kernel<MODE, EMIT, POST, TS>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                              227 * 1024);
}

template <int MODE, bool EMIT, bool POST, int TS>
cudaError_t launch_one(const ScanBatchArgs& a, const SmallArgs& p, size_t smem, int num_sms, cudaStream_t stream) {
  int occ = 0;
  cudaError_t e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, scan_small_kernel<MODE, EMIT, POST, TS>, TS, smem);
  if (e != cudaSuccess) return e;
  if (occ < 1) return cudaErrorLaunchOutOfResources;
  const int grid = (int)std::min<uint32_t>((uint32_t)(occ * num_sms), a.n_scans);
  scan_small_kernel<MODE, EMIT, POST, TS><<<grid, TS, smem, stream>>>(a, p);
  return cudaGetLastError();
}

}  // namespace

constexpr int kSmallThreads = 256;      // LaserScan variants
constexpr int kSmallPostThreads = 512;  // PointCloud2 chain

size_t scan_small_smem_bytes(uint32_t cap, int mode, bool emit, bool post) {
  size_t b = kCtl + (size_t)cap * 8 + 16;  // control block + tile (+ one node either side for unaligned views)
  if (post)  // (x, y) + intensity + accumulators (the rank table sits at their start during the place pass)
    return b + (size_t)cap * 8 + cap + std::max<size_t>((size_t)cap * 16, kWords * 6);
  b += kWords * 6;
  if (emit) b += kWords * 6;
  if (mode == 1) b += (size_t)cap * 8 - kWords * 6;  // per bin: min dist_m bits, winner key | quality; no bitmap
  return b;
}

bool scan_small_applies(uint32_t stride) { return stride != 0 && stride <= kSmallMaxNodes; }
bool scan_small_post_applies(uint32_t stride) { return stride != 0 && stride <= kSmallPostMaxNodes; }

cudaError_t scan_small_configure() {
  cudaError_t e;
  if ((e = configure_one<0, false, false, kSmallThreads>()) != cudaSuccess) return e;
  if ((e = configure_one<0, true, false, kSmallThreads>()) != cudaSuccess) return e;
  if ((e = configure_one<1, false, false, kSmallThreads>()) != cudaSuccess) return e;
  if ((e = configure_one<1, true, false, kSmallThreads>()) != cudaSuccess) return e;
  if ((e = configure_one<2, false, false, kSmallThreads>()) != cudaSuccess) return e;
  return configure_one<2, false, true, kSmallPostThreads>();
}

cudaError_t launch_scan_small(const ScanBatchArgs& a, uint32_t max_nodes, uint32_t sor_k, float sor_alpha, float voxel,
                              int num_sms, cudaStream_t stream) {
  SmallArgs p{};
  p.cap = (a.stride + 63u) & ~63u;
  p.max_nodes = max_nodes;
  p.use_tma = ((reinterpret_cast<uintptr_t>(a.nodes) & 15u) == 0 && (a.stride & 1u) == 0) ? 1u : 0u;
  p.sor_k = sor_k;
  p.sor_alpha = sor_alpha;
  p.voxel = voxel;
  const bool cloud = a.xyzi != nullptr;
  const bool emit = !cloud && a.nodes_out != nullptr && a.apply_ascend != 0;
  const bool post = cloud && (sor_k > 0 || voxel > 0.0f);
  const int mode = cloud ? 2 : (a.mode_a ? 1 : 0);
  const size_t sh = scan_small_smem_bytes(p.cap, mode, emit, post);
  if (cloud) {
    if (post) return launch_one<2, false, true, kSmallPostThreads>(a, p, sh, num_sms, stream);
    return launch_one<2, false, false, kSmallThreads>(a, p, sh, num_sms, stream);
  }
  if (mode == 1) {
    if (emit) return launch_one<1, true, false, kSmallThreads>(a, p, sh, num_sms, stream);
    return launch_one<1, false, false, kSmallThreads>(a, p, sh, num_sms, stream);
  }
  if (emit) return launch_one<0, true, false, kSmallThreads>(a, p, sh, num_sms, stream);
  return launch_one<0, false, false, kSmallThreads>(a, p, sh, num_sms, stream);
}

}  // namespace rpl
