// scan_general.cu -- the general scan kernel: any node count, duplicate keys allowed.
//
// Same contract as scan_fast.cu (ascendScanData_ + publish_scan, reference
// src/sdk/src/sl_lidar_driver.cpp:128-184 and src/rplidar_node.cpp:581-677) but built on an
// explicit STABLE sort, so equal angle_z_q14 keep buffer order -- the documented tie rule
// (the reference's std::sort leaves tie order to libstdc++'s introsort).  It serves the
// scans the fast kernel hands over (duplicate keys, > 65536 nodes) and, with
// RPL_FLAG_FORCE_GENERAL, every scan: an independent second implementation that the tests
// play against the fast kernel.
//
// One CTA of 128 threads per scan.  The sort is a 2-pass (8 bits each) LSD radix sort in
// which every thread owns a contiguous slice of the sequence and a private histogram column
// in shared memory: no atomics, deterministic, stable by construction.
#include "rpl_device.cuh"
#include "scan_args.h"

namespace rpl {

namespace {

constexpr int GT = kGeneralThreads;  // 128
constexpr int kRow = GT + 1;         // padded histogram row: conflict-free row walks
constexpr int kBins = 256;

struct GeneralSmem {
  uint32_t hist[kBins * kRow];
  uint32_t row_base[kBins];
  uint32_t red[2 * (GT / 32)];
  uint32_t seg[GT];
  uint32_t valid_count;
  uint32_t first_valid;
  uint32_t front_key;
};

__device__ __forceinline__ uint32_t block_exclusive_scan(GeneralSmem& sm, uint32_t v, uint32_t* total) {
  const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const uint32_t inc = warp_inclusive_scan(v);
  if (lane == 31) sm.red[warp] = inc;
  __syncthreads();
  uint32_t base = 0, tot = 0;
#pragma unroll
  for (int w = 0; w < GT / 32; ++w) {
    const uint32_t t = sm.red[w];
    if ((uint32_t)w < warp) base += t;
    tot += t;
  }
  __syncthreads();
  if (total) *total = tot;
  return base + inc - v;
}

// one stable counting pass over `n` entries; entry j is index in[j] (identity when in == 0)
__device__ void radix_pass(GeneralSmem& sm, const uint16_t* keyf, const uint32_t* in, uint32_t* out,
                           uint32_t n, uint32_t shift) {
  const uint32_t tid = threadIdx.x;
  const uint32_t len = (n + GT - 1) / GT;
  const uint32_t lo = min(n, tid * len), hi = min(n, lo + len);
  for (uint32_t j = tid; j < (uint32_t)(kBins * kRow); j += GT) sm.hist[j] = 0;
  __syncthreads();
  for (uint32_t j = lo; j < hi; ++j) {
    const uint32_t i = in ? in[j] : j;
    const uint32_t d = (keyf[i] >> shift) & 0xFFu;
    sm.hist[d * kRow + tid] += 1;
  }
  __syncthreads();
  for (uint32_t r = tid; r < (uint32_t)kBins; r += GT) {
    uint32_t run = 0;
    for (uint32_t t = 0; t < (uint32_t)GT; ++t) {
      const uint32_t v = sm.hist[r * kRow + t];
      sm.hist[r * kRow + t] = run;
      run += v;
    }
    sm.row_base[r] = run;
  }
  __syncthreads();
  if (tid == 0) {
    uint32_t run = 0;
    for (uint32_t r = 0; r < (uint32_t)kBins; ++r) {
      const uint32_t v = sm.row_base[r];
      sm.row_base[r] = run;
      run += v;
    }
  }
  __syncthreads();
  for (uint32_t j = lo; j < hi; ++j) {
    const uint32_t i = in ? in[j] : j;
    const uint32_t d = (keyf[i] >> shift) & 0xFFu;
    const uint32_t pos = sm.row_base[d] + sm.hist[d * kRow + tid];
    sm.hist[d * kRow + tid] += 1;
    out[pos] = i;
  }
  __syncthreads();
}

__global__ void __launch_bounds__(GT, 1)
    scan_general_kernel(ScanBatchArgs a, GeneralWorkspace ws, int all_scans) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  GeneralSmem& sm = *reinterpret_cast<GeneralSmem*>(smem_raw);
  const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const bool new_proto = a.is_new_protocol != 0;
  const bool mode_a = a.mode_a != 0;
  const bool inverted = a.inverted != 0;
  const bool ascend = a.apply_ascend != 0;
  const bool cloud = a.xyzi != nullptr;  // PointCloud2 payload: window filter + polar->xyz
  const bool want_scan = a.ranges != nullptr || cloud;
  auto kept = [&](uint2 nd) {
    const uint32_t d = node_dist(nd);
    if (d == 0) return false;
    if (!cloud) return true;
    return cloud_keep(dist_to_m(d), quality_to_intensity(node_quality(nd), new_proto), a.range_min, a.range_max,
                      a.intensity_min);
  };

  const size_t wo = (size_t)blockIdx.x * ws.max_nodes;
  uint16_t* keyf = ws.keyf + wo;
  uint32_t* idx0 = ws.idx0 + wo;
  uint32_t* idx1 = ws.idx1 + wo;
  uint32_t* vidx = ws.vidx + wo;
  unsigned long long* cell = ws.cell + wo;

  const uint32_t n_work = all_scans ? a.n_scans : *a.fallback_count;
  for (uint32_t work = blockIdx.x; work < n_work; work += gridDim.x) {
    const uint32_t s = all_scans ? work : a.fallback_list[work];
    const uint32_t n = a.views ? a.views[s].y : a.counts[s];
    const uint2* base = a.views ? a.nodes + a.views[s].x : a.nodes + (size_t)s * a.stride;
    uint2* nodes_out = a.nodes_out ? a.nodes_out + (size_t)s * a.stride : nullptr;

    // caller error (a count above the stride or the context's limit, a view that runs past the node buffer):
    // report, touch nothing
    if (n > a.stride || n > ws.max_nodes || (a.views && (unsigned long long)a.views[s].x + n > a.nodes_total)) {
      if (tid == 0) {
        if (a.status) a.status[s] = 0x80008000u;  // SL_RESULT_INVALID_DATA
        if (a.path) a.path[s] = 1u;
        if (a.beam_counts) a.beam_counts[s] = 0u;
        if (a.angle_inc) a.angle_inc[s] = 0.0f;
      }
      continue;
    }

    // ---- measured count, first measured node ---------------------------------------------
    uint32_t cnt = 0, first = 0xFFFFFFFFu;
    for (uint32_t i = tid; i < n; i += GT) {
      const uint2 nd = base[i];
      if (kept(nd)) ++cnt;
      if (node_dist(nd) != 0) first = min(first, i);
    }
    cnt = warp_sum(cnt);
    first = warp_min(first);
    if (lane == 0) {
      sm.red[warp] = cnt;
      sm.red[GT / 32 + warp] = first;
    }
    __syncthreads();
    if (tid == 0) {
      uint32_t c = 0, f = 0xFFFFFFFFu;
      for (int w = 0; w < GT / 32; ++w) {
        c += sm.red[w];
        f = min(f, sm.red[GT / 32 + w]);
      }
      sm.valid_count = c;
      sm.first_valid = f;
      // head tune (reference sl_lidar_driver.cpp:133-147)
      sm.front_key = (f != 0xFFFFFFFFu && ascend) ? ascend_head_key(node_key(base[f]), f, ascend_step(n)) : 0u;
    }
    __syncthreads();
    const uint32_t M = sm.valid_count;
    const float inc = (M != 0) ? angle_increment(M, mode_a) : 0.0f;
    if (tid == 0) {
      if (a.status) a.status[s] = (ascend && M == 0) ? kResultOperationFail : kResultOk;
      if (a.path) a.path[s] = 1u;
      if (a.beam_counts) a.beam_counts[s] = M;
      if (a.angle_inc) a.angle_inc[s] = inc;
    }
    if (M == 0) {  // OPERATION_FAIL: buffer untouched; publish_scan returns early
      if (nodes_out)
        for (uint32_t i = tid; i < n; i += GT) nodes_out[i] = base[i];
      __syncthreads();
      continue;
    }

    // ---- final key of every node (fill: reference sl_lidar_driver.cpp:170-178) ------------
    const float step = ascend_step(n);
    const uint32_t front_key = sm.front_key;
    const float front_deg = key_to_deg(front_key);
    for (uint32_t i = tid; i < n; i += GT) {
      const uint2 nd = base[i];
      uint32_t k = node_key(nd);
      if (ascend && node_dist(nd) == 0) k = (i == 0) ? front_key : ascend_fill_key(front_deg, i, step);
      keyf[i] = (uint16_t)k;
    }
    __syncthreads();

    // ---- stable sort of all nodes by final key --------------------------------------------
    radix_pass(sm, keyf, nullptr, idx0, n, 0);
    radix_pass(sm, keyf, idx0, idx1, n, 8);

    // ---- ascended node buffer ---------------------------------------------------------------
    if (nodes_out) {
      if (ascend) {
        for (uint32_t r = tid; r < n; r += GT) {
          const uint32_t i = idx1[r];
          nodes_out[r] = node_with_key(base[i], keyf[i]);
        }
      } else {
        for (uint32_t i = tid; i < n; i += GT) nodes_out[i] = base[i];
      }
    }
    if (!want_scan) {
      __syncthreads();
      continue;
    }

    // ---- measured nodes in sorted order (stable filter) ------------------------------------
    {
      const uint32_t len = (n + GT - 1) / GT;
      const uint32_t lo = min(n, tid * len), hi = min(n, lo + len);
      uint32_t c = 0;
      for (uint32_t r = lo; r < hi; ++r) c += kept(base[idx1[r]]) ? 1u : 0u;
      uint32_t v = block_exclusive_scan(sm, c, nullptr);
      for (uint32_t r = lo; r < hi; ++r) {
        const uint32_t i = idx1[r];
        if (kept(base[i])) vidx[v++] = i;
      }
    }
    __syncthreads();

    if (cloud) {  // oracle/cloud_oracle.cpp steps 1-3
      float4* out = a.xyzi + (size_t)s * a.stride;
      for (uint32_t v = tid; v < M; v += GT) {
        const uint2 nd = base[vidx[v]];
        const float dm = dist_to_m(node_dist(nd));
        const float2 cs = a.trig[node_key(nd)];
        out[v] = make_float4(__fmul_rn(dm, cs.x), __fmul_rn(dm, cs.y), 0.0f,
                             quality_to_intensity(node_quality(nd), new_proto));
      }
      __syncthreads();
      continue;
    }
    float* ranges = a.ranges + (size_t)s * a.stride;
    float* intens = a.intensities + (size_t)s * a.stride;
    if (!mode_a) {  // Mode B (reference rplidar_node.cpp:661-677)
      for (uint32_t v = tid; v < M; v += GT) {
        const uint2 nd = base[vidx[v]];
        const uint32_t o = inverted ? (M - 1 - v) : v;
        ranges[o] = dist_to_m(node_dist(nd));
        intens[o] = quality_to_intensity(node_quality(nd), new_proto);
      }
    } else {  // Mode A (reference rplidar_node.cpp:630-660): first strict minimum per bin
      for (uint32_t b = tid; b < M; b += GT) cell[b] = ~0ull;
      __syncthreads();
      for (uint32_t v = tid; v < M; v += GT) {
        const uint2 nd = base[vidx[v]];
        const int b = mode_a_bin(node_key(nd), inc, inverted);
        if (b >= 0 && b < (int)M) {
          const unsigned long long c =
              ((unsigned long long)__float_as_uint(dist_to_m(node_dist(nd))) << 32) | v;
          atomicMin(&cell[b], c);
        }
      }
      __syncthreads();
      for (uint32_t b = tid; b < M; b += GT) {
        const unsigned long long c = cell[b];
        if (c == ~0ull) {
          ranges[b] = __int_as_float(0x7f800000);
          intens[b] = 0.0f;
        } else {
          ranges[b] = __uint_as_float((uint32_t)(c >> 32));
          intens[b] = quality_to_intensity(node_quality(base[vidx[(uint32_t)c]]), new_proto);
        }
      }
    }
    __syncthreads();
  }
}

}  // namespace

size_t scan_general_smem_bytes() { return sizeof(GeneralSmem); }

cudaError_t launch_scan_general(const ScanBatchArgs& a, const GeneralWorkspace& ws, int grid,
                                bool all_scans, cudaStream_t stream) {
  scan_general_kernel<<<grid, GT, sizeof(GeneralSmem), stream>>>(a, ws, all_scans ? 1 : 0);
  return cudaGetLastError();
}

cudaError_t scan_general_configure() {
  return cudaFuncSetAttribute(scan_general_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                              (int)sizeof(GeneralSmem));
}

}  // namespace rpl
