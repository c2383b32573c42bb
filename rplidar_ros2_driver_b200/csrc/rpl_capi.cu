// rpl_capi.cu -- the C-ABI of librplidar_b200.so (include/rpl_b200.h).
//
// Host-side glue only: context, workspaces, streams, the chunked host<->device pipeline of
// the host-buffer entry points, and kernel launches.  There is no CPU implementation of the
// path in this library: every entry point either runs the CUDA kernels or fails.
#include <cuda_runtime.h>

#include <algorithm>
#include <cstdio>
#include <cstring>
#include <new>
#include <string>
#include <utility>
#include <vector>

#include "../../include/rpl_b200.h"
#include "cloud_args.h"
#include "cdr_args.h"
#include "decode_args.h"
#include "scan_args.h"

namespace rpl {
cudaError_t launch_synth(uint64_t first_scan_id, uint32_t n_scans, uint32_t n, uint32_t stride,
                         int variant, uint2* nodes, uint32_t* counts, cudaStream_t stream);
}

static_assert(sizeof(rpl_node_hq) == 8, "packed node must be 8 bytes");

#include "rpl_ctx.h"

namespace {

template <class P>
cudaError_t dev_alloc(P** p, size_t count) {
  return cudaMalloc(reinterpret_cast<void**>(p), std::max<size_t>(count, 1) * sizeof(P));
}

void free_lane(Lane& l) {
  cudaFree(l.fallback_list);
  cudaFree(l.fallback_count);
  cudaFree(l.fws.group);
  cudaFree(l.gws.keyf);
  cudaFree(l.gws.idx0);
  cudaFree(l.gws.idx1);
  cudaFree(l.gws.vidx);
  cudaFree(l.gws.cell);
  if (l.owns_cws) rpl::cloud_workspace_free(l.cws);
  cudaFree(l.d_nodes);
  cudaFree(l.d_nodes_out);
  cudaFree(l.d_counts);
  cudaFree(l.d_ranges);
  cudaFree(l.d_intens);
  cudaFree(l.d_beams);
  cudaFree(l.d_inc);
  cudaFree(l.d_status);
  cudaFree(l.d_path);
  cudaFree(l.d_xyzi);
  cudaFree(l.d_pcount);
  cudaFree(l.d_chain);
  if (l.stream) cudaStreamDestroy(l.stream);
  l = Lane{};
}

rpl_result ensure_staging(rpl_ctx* c, Lane& l, uint32_t scans, size_t nodes, bool cloud) {
  if (l.staged_nodes < nodes || l.staged_scans < scans) {
    cudaFree(l.d_nodes);
    cudaFree(l.d_nodes_out);
    cudaFree(l.d_ranges);
    cudaFree(l.d_intens);
    cudaFree(l.d_counts);
    cudaFree(l.d_beams);
    cudaFree(l.d_inc);
    cudaFree(l.d_status);
    cudaFree(l.d_path);
    cudaFree(l.d_xyzi);
    cudaFree(l.d_pcount);
    l.d_nodes = l.d_nodes_out = nullptr;
    l.d_ranges = l.d_intens = l.d_inc = l.d_xyzi = nullptr;
    l.d_counts = l.d_beams = l.d_status = l.d_path = l.d_pcount = nullptr;
    l.staged_nodes = 0;
    l.staged_scans = 0;
    const rpl_result oom = RPL_RESULT_INSUFFICIENT_MEMORY;
    RPL_CUDA(c, dev_alloc(&l.d_nodes, nodes), oom);
    RPL_CUDA(c, dev_alloc(&l.d_nodes_out, nodes), oom);
    RPL_CUDA(c, dev_alloc(&l.d_ranges, nodes), oom);
    RPL_CUDA(c, dev_alloc(&l.d_intens, nodes), oom);
    RPL_CUDA(c, dev_alloc(&l.d_counts, scans), oom);
    RPL_CUDA(c, dev_alloc(&l.d_beams, scans), oom);
    RPL_CUDA(c, dev_alloc(&l.d_inc, scans), oom);
    RPL_CUDA(c, dev_alloc(&l.d_status, scans), oom);
    RPL_CUDA(c, dev_alloc(&l.d_path, scans), oom);
    RPL_CUDA(c, dev_alloc(&l.d_pcount, scans), oom);
    l.staged_nodes = nodes;
    l.staged_scans = scans;
  }
  if (cloud && !l.d_xyzi) RPL_CUDA(c, dev_alloc(&l.d_xyzi, l.staged_nodes * 4), RPL_RESULT_INSUFFICIENT_MEMORY);
  return RPL_RESULT_OK;
}

// PointCloud2 steps 4-5 a launch may fuse into the shared-memory kernel (scan_small.cu)
struct PostParams {
  uint32_t sor_k = 0;
  float sor_alpha = 0.0f;
  float voxel = 0.0f;
};
rpl_result enqueue_args(rpl_ctx* c, Lane& l, rpl::ScanBatchArgs a, uint32_t flags, cudaStream_t stream,
                        const PostParams* post = nullptr, bool* post_fused = nullptr);

// queue the scan kernels for one device-resident batch on `stream`
rpl_result enqueue_scan(rpl_ctx* c, Lane& l, const rpl_node_hq* nodes, const uint32_t* counts,
                        uint32_t n_scans, uint32_t stride, const rpl_scan_params* p,
                        rpl_node_hq* nodes_out, float* ranges, float* intens, uint32_t* beams,
                        float* inc, uint32_t* status, uint32_t* path, cudaStream_t stream,
                        const uint2* views = nullptr, unsigned long long nodes_total = 0) {
  if (n_scans == 0) return RPL_RESULT_OK;
  if (!nodes || !counts || !p) {
    c->err = "null nodes/counts/params";
    return RPL_RESULT_INVALID_DATA;
  }
  if (n_scans > c->max_scans) {
    c->err = "n_scans exceeds the context's max_scans";
    return RPL_RESULT_INVALID_DATA;
  }
  if ((ranges == nullptr) != (intens == nullptr)) {
    c->err = "ranges and intensities must be given together";
    return RPL_RESULT_INVALID_DATA;
  }
  if (nodes_out && static_cast<const void*>(nodes_out) == static_cast<const void*>(nodes)) {
    c->err = "nodes_out must not alias nodes on the device path";
    return RPL_RESULT_INVALID_DATA;
  }
  if (misaligned8(nodes) || misaligned8(nodes_out)) {
    c->err = "node buffers must be 8-byte aligned";
    return RPL_RESULT_INVALID_DATA;
  }
  rpl::ScanBatchArgs a{};
  a.xyzi = nullptr;
  a.trig = nullptr;
  a.angle = l.cws.angle;
  a.nodes = reinterpret_cast<const uint2*>(nodes);
  a.nodes_out = reinterpret_cast<uint2*>(nodes_out);
  a.counts = counts;
  a.n_scans = n_scans;
  a.stride = stride;
  a.ranges = ranges;
  a.intensities = intens;
  a.beam_counts = beams;
  a.angle_inc = inc;
  a.status = status;
  a.path = path;
  a.fallback_list = l.fallback_list;
  a.fallback_count = l.fallback_count;
  a.is_new_protocol = p->is_new_protocol;
  a.mode_a = p->scan_processing;
  a.inverted = p->inverted;
  a.apply_ascend = p->apply_ascend;
  a.views = views;
  a.nodes_total = nodes_total;
  return enqueue_args(c, l, a, p->flags, stream);
}

rpl_result enqueue_args(rpl_ctx* c, Lane& l, rpl::ScanBatchArgs a, uint32_t flags, cudaStream_t stream,
                        const PostParams* post, bool* post_fused) {
  const uint32_t n_scans = a.n_scans, stride = a.stride;
  bool force_general = (flags & RPL_FLAG_FORCE_GENERAL) != 0;
  if (post_fused) *post_fused = false;
  if (a.nodes_out && !a.apply_ascend) {
    // no geometric correction requested: the buffer passes through unchanged
    // (reference lidar_driver_wrapper.cpp:330-337); a plain device copy, not kernel work
    RPL_CUDA(c, cudaMemcpy2DAsync(a.nodes_out, (size_t)stride * 8, a.nodes, (size_t)stride * 8,
                                  (size_t)stride * 8, n_scans, cudaMemcpyDeviceToDevice, stream),
             RPL_RESULT_OPERATION_FAIL);
    a.nodes_out = nullptr;
  }
  // status-only calls (no LaserScan, no ascended buffer) take the general kernel
  if (!a.ranges && !a.nodes_out && !a.xyzi) force_general = true;
  // revolutions that fit shared memory (what a lidar delivers) have their own kernels
  const bool small = !force_general && rpl::scan_small_applies(stride) && (flags & RPL_FLAG_NO_SMALL) == 0;
  // above that the PointCloud2 payload exists in the TMA kernel and the general kernel only
  if (a.xyzi && !small && ((reinterpret_cast<uintptr_t>(a.nodes) & 15u) != 0 || (stride & 1u) != 0)) force_general = true;
  if (!force_general) {
    RPL_CUDA(c, cudaMemsetAsync(l.fallback_count, 0, sizeof(uint32_t), stream), RPL_RESULT_OPERATION_FAIL);
    // the TMA-ring kernel needs every scan base 16-byte aligned
    const bool emit = a.nodes_out != nullptr;
    const bool aligned = (reinterpret_cast<uintptr_t>(a.nodes) & 15u) == 0 && (stride & 1u) == 0;
    const bool use_tma = !emit && aligned && ((flags & RPL_FLAG_NO_TMA) == 0 || a.xyzi != nullptr);
    const int grid = (int)std::min<uint32_t>(n_scans, (uint32_t)(use_tma ? c->tma_grid : c->fast_grid));
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    if (c->profile) {
      cudaEventCreate(&e0);
      cudaEventCreate(&e1);
      cudaEventRecord(e0, stream);
    }
    if (small) {
      // SOR / voxel grid run inside the kernel when the 32-bit cell keys and accumulators are exact:
      // |cell index| < 32768 and voxel <= 4 m (scan_small.cu); otherwise as separate passes
      bool fuse = false;
      if (a.xyzi && post && (post->sor_k > 0 || post->voxel > 0.0f) && rpl::scan_small_post_applies(stride))
        fuse = post->voxel == 0.0f || (post->voxel <= 4.0f && a.range_max / post->voxel < 32000.0f);
      RPL_CUDA(c, rpl::launch_scan_small(a, l.fws.max_nodes, fuse ? post->sor_k : 0u, fuse ? post->sor_alpha : 0.0f,
                                         fuse ? post->voxel : 0.0f, c->num_sms, stream),
               RPL_RESULT_OPERATION_FAIL);
      if (post_fused) *post_fused = fuse;
    } else if (use_tma) {
      RPL_CUDA(c, rpl::launch_scan_tma(a, l.fws, grid, stream), RPL_RESULT_OPERATION_FAIL);
    } else {
      RPL_CUDA(c, rpl::launch_scan_fast(a, l.fws, grid, stream), RPL_RESULT_OPERATION_FAIL);
    }
    if (c->profile) {
      cudaEventRecord(e1, stream);
      c->prof_fast.emplace_back(e0, e1);
    }
    c->launches++;
  }
  const int ggrid = (int)std::min<uint32_t>(n_scans, (uint32_t)c->general_grid);
  cudaEvent_t g0 = nullptr, g1 = nullptr;
  if (c->profile) {
    cudaEventCreate(&g0);
    cudaEventCreate(&g1);
    cudaEventRecord(g0, stream);
  }
  RPL_CUDA(c, rpl::launch_scan_general(a, l.gws, ggrid, force_general, stream), RPL_RESULT_OPERATION_FAIL);
  if (c->profile) {
    cudaEventRecord(g1, stream);
    c->prof_general.emplace_back(g0, g1);
  }
  c->launches++;
  return RPL_RESULT_OK;
}

}  // namespace

extern "C" {

uint32_t rpl_abi_version(void) { return RPL_ABI_VERSION; }

rpl_result rpl_ctx_create(int device, uint32_t max_nodes, uint32_t max_scans, rpl_ctx** out) {
  if (!out || max_nodes == 0 || max_scans == 0) return RPL_RESULT_INVALID_DATA;
  *out = nullptr;
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || device < 0 || device >= ndev) {
    // no CPU fallback by design
    return RPL_RESULT_OPERATION_NOT_SUPPORT;
  }
  rpl_ctx* c = new (std::nothrow) rpl_ctx();
  if (!c) return RPL_RESULT_INSUFFICIENT_MEMORY;
  c->device = device;
  c->max_nodes = max_nodes;
  c->max_scans = max_scans;
  auto fail = [&](rpl_result r) {
    std::fprintf(stderr, "[rpl_b200] rpl_ctx_create failed: %s\n", c->err.c_str());
    rpl_ctx_destroy(c);
    return r;
  };
  if (!cuda_ok(c, cudaSetDevice(device), "cudaSetDevice")) return fail(RPL_RESULT_OPERATION_FAIL);
  cudaDeviceProp prop{};
  if (!cuda_ok(c, cudaGetDeviceProperties(&prop, device), "cudaGetDeviceProperties"))
    return fail(RPL_RESULT_OPERATION_FAIL);
  if (prop.major < 10) {
    c->err = "librplidar_b200 is built for sm_100a (B200) only";
    return fail(RPL_RESULT_OPERATION_NOT_SUPPORT);
  }
  c->num_sms = prop.multiProcessorCount;
  if (!cuda_ok(c, rpl::scan_fast_configure(), "scan_fast_configure") ||
      !cuda_ok(c, rpl::scan_tma_configure(), "scan_tma_configure") ||
      !cuda_ok(c, rpl::scan_small_configure(), "scan_small_configure") ||
      !cuda_ok(c, rpl::scan_general_configure(), "scan_general_configure") ||
      !cuda_ok(c, rpl::cloud_configure(), "cloud_configure") ||
      !cuda_ok(c, rpl::decode_configure(), "decode_configure") ||
      !cuda_ok(c, rpl::decode_formats_configure(), "decode_formats_configure"))
    return fail(RPL_RESULT_OPERATION_FAIL);
  const int occ = std::max(1, rpl::scan_fast_max_ctas_per_sm());
  c->fast_grid = c->num_sms * occ;
  c->tma_grid = c->num_sms * std::max(1, rpl::scan_tma_max_ctas_per_sm());
  c->general_grid = c->num_sms;

  for (int i = 0; i < kLanes; ++i) {
    Lane& l = c->lane[i];
    const rpl_result oom = RPL_RESULT_INSUFFICIENT_MEMORY;
    if (!cuda_ok(c, cudaStreamCreateWithFlags(&l.stream, cudaStreamNonBlocking), "cudaStreamCreate"))
      return fail(RPL_RESULT_OPERATION_FAIL);
    const size_t fast_nodes = (size_t)std::max(c->fast_grid, c->tma_grid) * max_nodes;
    const size_t gen_nodes = (size_t)c->general_grid * max_nodes;
    l.fws.max_nodes = max_nodes;
    l.gws.max_nodes = max_nodes;
    if (!cuda_ok(c, dev_alloc(&l.fallback_list, max_scans), "cudaMalloc") ||
        !cuda_ok(c, dev_alloc(&l.fallback_count, 1), "cudaMalloc") ||
        !cuda_ok(c, dev_alloc(&l.fws.group, fast_nodes), "cudaMalloc") ||
        !cuda_ok(c, dev_alloc(&l.gws.keyf, gen_nodes), "cudaMalloc") ||
        !cuda_ok(c, dev_alloc(&l.gws.idx0, gen_nodes), "cudaMalloc") ||
        !cuda_ok(c, dev_alloc(&l.gws.idx1, gen_nodes), "cudaMalloc") ||
        !cuda_ok(c, dev_alloc(&l.gws.vidx, gen_nodes), "cudaMalloc") ||
        !cuda_ok(c, dev_alloc(&l.gws.cell, gen_nodes), "cudaMalloc") ||
        false)
      return fail(oom);
    if (i == 0) {
      if (!cuda_ok(c, rpl::cloud_workspace_alloc(l.cws, c->num_sms, max_nodes), "cloud workspace")) return fail(oom);
      l.owns_cws = true;
    } else {  // read-only tables shared with lane 0; the PointCloud2 post passes run on lane 0 only
      l.cws = rpl::CloudWorkspace{};
      l.cws.trig = c->lane[0].cws.trig;
      l.cws.angle = c->lane[0].cws.angle;
    }
    if (!cuda_ok(c, cudaMemset(l.fallback_count, 0, sizeof(uint32_t)), "cudaMemset"))
      return fail(RPL_RESULT_OPERATION_FAIL);
  }
  if (!cuda_ok(c, cudaHostAlloc(reinterpret_cast<void**>(&c->h_counts), (size_t)max_scans * 4, cudaHostAllocDefault),
               "cudaHostAlloc") ||
      !cuda_ok(c, cudaHostAlloc(reinterpret_cast<void**>(&c->h_small), (size_t)max_scans * 16, cudaHostAllocDefault),
               "cudaHostAlloc"))
    return fail(RPL_RESULT_INSUFFICIENT_MEMORY);
  {
    c->one_stride = ((size_t)max_nodes + 1) & ~(size_t)1;
    const size_t bytes = c->one_stride * (8 + 8 + 4 + 4) + 64;
    if (!cuda_ok(c, cudaHostAlloc(reinterpret_cast<void**>(&c->h_one), bytes, cudaHostAllocDefault), "cudaHostAlloc") ||
        !cuda_ok(c, cudaMalloc(reinterpret_cast<void**>(&c->d_one), bytes), "cudaMalloc"))
      return fail(RPL_RESULT_INSUFFICIENT_MEMORY);
  }
  *out = c;
  return RPL_RESULT_OK;
}

void rpl_ctx_destroy(rpl_ctx* c) {
  if (!c) return;
  cudaSetDevice(c->device);
  for (int i = 0; i < kLanes; ++i) {
    if (c->lane[i].stream) cudaStreamSynchronize(c->lane[i].stream);
    free_lane(c->lane[i]);
  }
  if (c->asm_done) cudaEventDestroy(c->asm_done);
  cudaFree(c->d_state_tmp);
  cudaFree(c->d_reset_prefix);
  cudaFree(c->d_desc);
  if (c->h_one) cudaFreeHost(c->h_one);
  cudaFree(c->d_one);
  if (c->h_counts) cudaFreeHost(c->h_counts);
  if (c->h_small) cudaFreeHost(c->h_small);
  delete c;
}

const char* rpl_last_error(const rpl_ctx* c) { return c ? c->err.c_str() : "null context"; }

rpl_result rpl_ctx_synchronize(rpl_ctx* c) {
  if (!c) return RPL_RESULT_INVALID_DATA;
  for (int i = 0; i < kLanes; ++i)
    RPL_CUDA(c, cudaStreamSynchronize(c->lane[i].stream), RPL_RESULT_OPERATION_FAIL);
  return RPL_RESULT_OK;
}

rpl_result rpl_host_alloc(size_t bytes, void** out) {
  if (!out) return RPL_RESULT_INVALID_DATA;
  *out = nullptr;
  return cudaHostAlloc(out, std::max<size_t>(bytes, 1), cudaHostAllocDefault) == cudaSuccess
             ? RPL_RESULT_OK
             : RPL_RESULT_INSUFFICIENT_MEMORY;
}
void rpl_host_free(void* p) {
  if (p) cudaFreeHost(p);
}

uint64_t rpl_ctx_launch_count(const rpl_ctx* c) { return c ? c->launches : 0; }

rpl_result rpl_ctx_profile(rpl_ctx* c, int enable) {
  if (!c) return RPL_RESULT_INVALID_DATA;
  c->profile = enable != 0;
  return RPL_RESULT_OK;
}

rpl_result rpl_ctx_profile_read(rpl_ctx* c, double* fast_ms, uint32_t* fast_launches,
                                double* general_ms, uint32_t* general_launches) {
  if (!c) return RPL_RESULT_INVALID_DATA;
  RPL_CUDA(c, cudaSetDevice(c->device), RPL_RESULT_OPERATION_FAIL);
  auto drain = [&](std::vector<std::pair<cudaEvent_t, cudaEvent_t>>& v, double* ms, uint32_t* n) {
    double sum = 0.0;
    for (auto& pr : v) {
      cudaEventSynchronize(pr.second);
      float t = 0.f;
      if (cudaEventElapsedTime(&t, pr.first, pr.second) == cudaSuccess) sum += t;
      cudaEventDestroy(pr.first);
      cudaEventDestroy(pr.second);
    }
    if (ms) *ms = sum;
    if (n) *n = (uint32_t)v.size();
    v.clear();
  };
  drain(c->prof_fast, fast_ms, fast_launches);
  drain(c->prof_general, general_ms, general_launches);
  return RPL_RESULT_OK;
}

// ---- device-resident batch ----------------------------------------------------------------
rpl_result rpl_scan_batch_dev(rpl_ctx* c, const rpl_node_hq* nodes, const uint32_t* counts,
                              uint32_t n_scans, uint32_t stride, const rpl_scan_params* params,
                              rpl_node_hq* nodes_out, float* ranges, float* intensities,
                              uint32_t* beam_counts, float* angle_increment, uint32_t* status,
                              uint32_t* path, void* stream) {
  if (!c) return RPL_RESULT_INVALID_DATA;
  RPL_CUDA(c, cudaSetDevice(c->device), RPL_RESULT_OPERATION_FAIL);
  if (n_scans != 0 && stride == 0) {
    c->err = "stride == 0";
    return RPL_RESULT_INVALID_DATA;
  }
  // counts[] live on the device: a scan with counts[s] > stride or > the context's max_nodes is reported
  // through status[s] = RPL_RESULT_INVALID_DATA by the kernels (nothing else is written for it)
  cudaStream_t st = stream ? static_cast<cudaStream_t>(stream) : c->lane[0].stream;
  return enqueue_scan(c, c->lane[0], nodes, counts, n_scans, stride, params, nodes_out, ranges,
                      intensities, beam_counts, angle_increment, status, path, st);
}

// ---- host-buffer batch: chunked over the two lanes so that the H2D copy of chunk i+1, the
// kernels of chunk i and the D2H copy of chunk i-1 overlap ---------------------------------
rpl_result rpl_scan_batch(rpl_ctx* c, const rpl_node_hq* nodes, const uint32_t* counts,
                          uint32_t n_scans, uint32_t stride, const rpl_scan_params* params,
                          rpl_node_hq* nodes_out, float* ranges, float* intensities,
                          uint32_t* beam_counts, float* angle_increment, uint32_t* status,
                          uint32_t* path) {
  if (!c) return RPL_RESULT_INVALID_DATA;
  if (n_scans == 0) return RPL_RESULT_OK;
  if (!nodes || !counts || !params) {
    c->err = "null nodes/counts/params";
    return RPL_RESULT_INVALID_DATA;
  }
  if (n_scans > c->max_scans || stride == 0) {
    c->err = "n_scans exceeds max_scans (or stride == 0)";
    return RPL_RESULT_INVALID_DATA;
  }
  for (uint32_t s = 0; s < n_scans; ++s)
    if (counts[s] > stride || counts[s] > c->max_nodes) {
      c->err = "counts[s] exceeds stride or the context's max_nodes";
      return RPL_RESULT_INVALID_DATA;
    }
  RPL_CUDA(c, cudaSetDevice(c->device), RPL_RESULT_OPERATION_FAIL);

  // chunk: about 32 MiB of nodes, at least one scan
  const size_t target_nodes = (32u << 20) / sizeof(rpl_node_hq);
  uint32_t chunk = (uint32_t)std::max<size_t>(1, target_nodes / stride);
  chunk = std::min(chunk, n_scans);
  const bool want_scan = ranges != nullptr;
  for (int i = 0; i < kLanes; ++i) {
    rpl_result r = ensure_staging(c, c->lane[i], chunk, (size_t)chunk * stride, false);
    if (r != RPL_RESULT_OK) return r;
  }
  const cudaMemcpyKind h2d = cudaMemcpyHostToDevice, d2h = cudaMemcpyDeviceToHost;
  std::memcpy(c->h_counts, counts, (size_t)n_scans * sizeof(uint32_t));
  uint32_t* hs_beams = c->h_small;
  uint32_t* hs_inc = c->h_small + c->max_scans;
  uint32_t* hs_status = c->h_small + 2 * (size_t)c->max_scans;
  uint32_t* hs_path = c->h_small + 3 * (size_t)c->max_scans;
  // one chunk through one lane; any failure leaves the loop with copies possibly still in flight
  auto run_chunk = [&](Lane& l, uint32_t s0, uint32_t ns) -> rpl_result {
    const size_t off = (size_t)s0 * stride, cnt = (size_t)ns * stride;
    // the lane's previous chunk (2 chunks ago) must have left its staging buffers
    RPL_CUDA(c, cudaStreamSynchronize(l.stream), RPL_RESULT_OPERATION_FAIL);
    RPL_CUDA(c, cudaMemcpyAsync(l.d_nodes, nodes + off, cnt * sizeof(rpl_node_hq), h2d, l.stream),
             RPL_RESULT_OPERATION_FAIL);
    RPL_CUDA(c, cudaMemcpyAsync(l.d_counts, c->h_counts + s0, ns * sizeof(uint32_t), h2d, l.stream),
             RPL_RESULT_OPERATION_FAIL);
    // The kernels write only the first counts[s] nodes of a scan they ascend (nothing for an empty or
    // unmeasured scan: the reference leaves those buffers untouched).  The whole [ns][stride] region goes
    // back to the caller, so it starts out as the caller's own bytes, not as leftovers of an earlier chunk.
    if (nodes_out && params->apply_ascend)
      RPL_CUDA(c, cudaMemcpyAsync(l.d_nodes_out, l.d_nodes, cnt * sizeof(rpl_node_hq), cudaMemcpyDeviceToDevice, l.stream),
               RPL_RESULT_OPERATION_FAIL);
    rpl_result r = enqueue_scan(c, l, reinterpret_cast<rpl_node_hq*>(l.d_nodes), l.d_counts, ns, stride,
                                params, nodes_out ? reinterpret_cast<rpl_node_hq*>(l.d_nodes_out) : nullptr,
                                want_scan ? l.d_ranges : nullptr, want_scan ? l.d_intens : nullptr,
                                l.d_beams, l.d_inc, l.d_status, l.d_path, l.stream);
    if (r != RPL_RESULT_OK) return r;
    if (nodes_out)
      RPL_CUDA(c, cudaMemcpyAsync(nodes_out + off, l.d_nodes_out, cnt * sizeof(rpl_node_hq), d2h, l.stream),
               RPL_RESULT_OPERATION_FAIL);
    if (want_scan) {
      RPL_CUDA(c, cudaMemcpyAsync(ranges + off, l.d_ranges, cnt * sizeof(float), d2h, l.stream),
               RPL_RESULT_OPERATION_FAIL);
      RPL_CUDA(c, cudaMemcpyAsync(intensities + off, l.d_intens, cnt * sizeof(float), d2h, l.stream),
               RPL_RESULT_OPERATION_FAIL);
    }
    if (beam_counts)
      RPL_CUDA(c, cudaMemcpyAsync(hs_beams + s0, l.d_beams, ns * sizeof(uint32_t), d2h, l.stream),
               RPL_RESULT_OPERATION_FAIL);
    if (angle_increment)
      RPL_CUDA(c, cudaMemcpyAsync(hs_inc + s0, l.d_inc, ns * sizeof(float), d2h, l.stream),
               RPL_RESULT_OPERATION_FAIL);
    if (status)
      RPL_CUDA(c, cudaMemcpyAsync(hs_status + s0, l.d_status, ns * sizeof(uint32_t), d2h, l.stream),
               RPL_RESULT_OPERATION_FAIL);
    if (path)
      RPL_CUDA(c, cudaMemcpyAsync(hs_path + s0, l.d_path, ns * sizeof(uint32_t), d2h, l.stream),
               RPL_RESULT_OPERATION_FAIL);
    return RPL_RESULT_OK;
  };
  uint32_t ci = 0;
  for (uint32_t s0 = 0; s0 < n_scans; s0 += chunk, ++ci) {
    const rpl_result r = run_chunk(c->lane[ci % kLanes], s0, std::min(chunk, n_scans - s0));
    if (r != RPL_RESULT_OK) {
      // nothing may still be writing into the caller's buffers when the error is reported
      const std::string why = c->err;
      for (int i = 0; i < kLanes; ++i) cudaStreamSynchronize(c->lane[i].stream);
      c->err = why;
      return r;
    }
  }
  const rpl_result rs = rpl_ctx_synchronize(c);
  if (rs != RPL_RESULT_OK) return rs;
  if (beam_counts) std::memcpy(beam_counts, hs_beams, (size_t)n_scans * 4);
  if (angle_increment) std::memcpy(angle_increment, hs_inc, (size_t)n_scans * 4);
  if (status) std::memcpy(status, hs_status, (size_t)n_scans * 4);
  if (path) std::memcpy(path, hs_path, (size_t)n_scans * 4);
  return RPL_RESULT_OK;
}

rpl_result rpl_ascend_scan_batch(rpl_ctx* c, rpl_node_hq* nodes, const uint32_t* counts,
                                 uint32_t n_scans, uint32_t stride, uint32_t* status) {
  rpl_scan_params p{};
  p.apply_ascend = 1;
  return rpl_scan_batch(c, nodes, counts, n_scans, stride, &p, nodes, nullptr, nullptr, nullptr,
                        nullptr, status, nullptr);
}

rpl_result rpl_laserscan_batch(rpl_ctx* c, const rpl_node_hq* nodes, const uint32_t* counts,
                               uint32_t n_scans, uint32_t stride, const rpl_scan_params* params,
                               float* ranges, float* intensities, uint32_t* beam_counts,
                               float* angle_increment) {
  if (!params) return RPL_RESULT_INVALID_DATA;
  rpl_scan_params p = *params;
  p.apply_ascend = 0;  // the LaserScan never depends on the ascended buffer (see DESIGN.md)
  return rpl_scan_batch(c, nodes, counts, n_scans, stride, &p, nullptr, ranges, intensities,
                        beam_counts, angle_increment, nullptr, nullptr);
}

// ---- single scan (the reference-shaped calls) ----------------------------------------------
namespace {

struct OneSmall {  // the 64-byte control block between the input and the outputs
  uint32_t count;
  uint32_t fallback_count;
  uint32_t fallback_list;
  uint32_t beams;
  float inc;
  uint32_t status;
  uint32_t path;
  uint32_t pad[9];
};
static_assert(sizeof(OneSmall) == 64, "control block");

// One lidar revolution: the operating point of the reference (one scan thread, ~10 Hz).  What
// matters here is latency, so the scan travels in one pinned block each way and the general
// kernel is launched only when the fast kernel reports a duplicate-key scan.
rpl_result scan_single(rpl_ctx* c, const rpl_node_hq* nodes_in, size_t count, const rpl_scan_params* p,
                       rpl_node_hq* nodes_out, float* ranges, float* intensities, uint32_t* beam_count,
                       float* angle_increment, rpl_result* ascend_status) {
  RPL_CUDA(c, cudaSetDevice(c->device), RPL_RESULT_OPERATION_FAIL);
  Lane& l = c->lane[0];
  const size_t S = c->one_stride, n = count;
  const size_t off_small = S * 8, off_nout = off_small + 64, off_r = off_nout + S * 8, off_i = off_r + S * 4;
  const size_t total = off_i + S * 4;
  std::memcpy(c->h_one, nodes_in, n * 8);
  OneSmall* hs = reinterpret_cast<OneSmall*>(c->h_one + off_small);
  std::memset(hs, 0, sizeof(OneSmall));
  hs->count = (uint32_t)n;
  // H2D: live nodes + control block (two copies only when the scan is much shorter than max_nodes)
  if (n * 8 + 4096 >= off_small) {
    RPL_CUDA(c, cudaMemcpyAsync(c->d_one, c->h_one, off_small + 64, cudaMemcpyHostToDevice, l.stream),
             RPL_RESULT_OPERATION_FAIL);
  } else {
    RPL_CUDA(c, cudaMemcpyAsync(c->d_one, c->h_one, n * 8, cudaMemcpyHostToDevice, l.stream), RPL_RESULT_OPERATION_FAIL);
    RPL_CUDA(c, cudaMemcpyAsync(c->d_one + off_small, hs, 64, cudaMemcpyHostToDevice, l.stream),
             RPL_RESULT_OPERATION_FAIL);
  }
  OneSmall* ds = reinterpret_cast<OneSmall*>(c->d_one + off_small);
  const bool want_nodes = nodes_out != nullptr && p->apply_ascend;
  const bool want_scan = ranges != nullptr;
  rpl::ScanBatchArgs a{};
  a.nodes = reinterpret_cast<const uint2*>(c->d_one);
  a.nodes_out = want_nodes ? reinterpret_cast<uint2*>(c->d_one + off_nout) : nullptr;
  a.counts = &ds->count;
  a.n_scans = 1;
  a.stride = (uint32_t)S;
  a.ranges = want_scan ? reinterpret_cast<float*>(c->d_one + off_r) : nullptr;
  a.intensities = want_scan ? reinterpret_cast<float*>(c->d_one + off_i) : nullptr;
  a.beam_counts = &ds->beams;
  a.angle_inc = &ds->inc;
  a.status = &ds->status;
  a.path = &ds->path;
  a.fallback_list = &ds->fallback_list;
  a.fallback_count = &ds->fallback_count;
  a.is_new_protocol = p->is_new_protocol;
  a.mode_a = p->scan_processing;
  a.inverted = p->inverted;
  a.apply_ascend = p->apply_ascend;
  a.angle = l.cws.angle;
  const bool force_general = (p->flags & RPL_FLAG_FORCE_GENERAL) != 0 || (!want_nodes && !want_scan);
  // D2H extent: control block + whatever was produced, trimmed to the live part
  auto copy_back = [&]() -> rpl_result {
    size_t end = off_nout;
    if (want_nodes) end = off_nout + n * 8;
    if (want_scan) end = off_i + n * 4;
    (void)total;
    if (want_scan && (end - off_small) > 3 * (64 + n * 16) + 8192) {
      // short scan in a large context: three small copies beat one copy across the gaps
      RPL_CUDA(c, cudaMemcpyAsync(hs, ds, 64 + (want_nodes ? n * 8 : 0), cudaMemcpyDeviceToHost, l.stream),
               RPL_RESULT_OPERATION_FAIL);
      RPL_CUDA(c, cudaMemcpyAsync(c->h_one + off_r, c->d_one + off_r, n * 4, cudaMemcpyDeviceToHost, l.stream),
               RPL_RESULT_OPERATION_FAIL);
      RPL_CUDA(c, cudaMemcpyAsync(c->h_one + off_i, c->d_one + off_i, n * 4, cudaMemcpyDeviceToHost, l.stream),
               RPL_RESULT_OPERATION_FAIL);
    } else {
      RPL_CUDA(c, cudaMemcpyAsync(hs, ds, end - off_small, cudaMemcpyDeviceToHost, l.stream),
               RPL_RESULT_OPERATION_FAIL);
    }
    RPL_CUDA(c, cudaStreamSynchronize(l.stream), RPL_RESULT_OPERATION_FAIL);
    return RPL_RESULT_OK;
  };
  if (!force_general) {
    const bool use_tma = !want_nodes && (p->flags & RPL_FLAG_NO_TMA) == 0;  // d_one and S keep bases 16-byte aligned
    if (use_tma)
      RPL_CUDA(c, rpl::launch_scan_tma(a, l.fws, 1, l.stream), RPL_RESULT_OPERATION_FAIL);
    else
      RPL_CUDA(c, rpl::launch_scan_fast(a, l.fws, 1, l.stream), RPL_RESULT_OPERATION_FAIL);
    c->launches++;
    rpl_result r = copy_back();
    if (r != RPL_RESULT_OK) return r;
  }
  if (force_general || hs->fallback_count != 0) {
    RPL_CUDA(c, rpl::launch_scan_general(a, l.gws, 1, true, l.stream), RPL_RESULT_OPERATION_FAIL);
    c->launches++;
    rpl_result r = copy_back();
    if (r != RPL_RESULT_OK) return r;
  }
  const uint32_t m = hs->beams;
  if (beam_count) *beam_count = m;
  if (angle_increment) *angle_increment = hs->inc;
  if (ascend_status) *ascend_status = hs->status;
  if (hs->status == RPL_RESULT_INVALID_DATA) return RPL_RESULT_INVALID_DATA;
  if (want_nodes) std::memcpy(nodes_out, c->h_one + off_nout, n * 8);
  if (want_scan && m) {
    std::memcpy(ranges, c->h_one + off_r, (size_t)m * 4);
    std::memcpy(intensities, c->h_one + off_i, (size_t)m * 4);
  }
  return RPL_RESULT_OK;
}

}  // namespace

rpl_result rpl_ascend_scan(rpl_ctx* c, rpl_node_hq* nodes, size_t count) {
  if (!c) return RPL_RESULT_INVALID_DATA;
  if (count == 0) return RPL_RESULT_OPERATION_FAIL;  // reference: i == count -> FAIL
  if (!nodes || count > c->max_nodes) return RPL_RESULT_INVALID_DATA;
  rpl_scan_params p{};
  p.apply_ascend = 1;
  rpl_result status = RPL_RESULT_OPERATION_FAIL;
  rpl_result r = scan_single(c, nodes, count, &p, nodes, nullptr, nullptr, nullptr, nullptr, &status);
  return r != RPL_RESULT_OK ? r : status;
}

rpl_result rpl_laserscan(rpl_ctx* c, const rpl_node_hq* nodes, size_t count,
                         const rpl_scan_params* params, float* ranges, float* intensities,
                         uint32_t* beam_count, float* angle_increment) {
  if (!c || !beam_count || !params) return RPL_RESULT_INVALID_DATA;
  *beam_count = 0;
  if (angle_increment) *angle_increment = 0.0f;
  if (count == 0) return RPL_RESULT_OK;  // publish_scan: nodes.empty() -> return
  if (!nodes || !ranges || !intensities || count > c->max_nodes) return RPL_RESULT_INVALID_DATA;
  rpl_scan_params p = *params;
  p.apply_ascend = 0;  // the LaserScan never depends on the ascended buffer (see DESIGN.md)
  return scan_single(c, nodes, count, &p, nullptr, ranges, intensities, beam_count, angle_increment, nullptr);
}

rpl_result rpl_scan(rpl_ctx* c, rpl_node_hq* nodes, size_t count, const rpl_scan_params* params,
                    float* ranges, float* intensities, uint32_t* beam_count,
                    float* angle_increment, rpl_result* ascend_status) {
  if (!c || !beam_count || !params) return RPL_RESULT_INVALID_DATA;
  *beam_count = 0;
  if (angle_increment) *angle_increment = 0.0f;
  if (ascend_status) *ascend_status = params->apply_ascend ? RPL_RESULT_OPERATION_FAIL : RPL_RESULT_OK;
  if (count == 0) return RPL_RESULT_OK;
  if (!nodes || !ranges || !intensities || count > c->max_nodes) return RPL_RESULT_INVALID_DATA;
  return scan_single(c, nodes, count, params, params->apply_ascend ? nodes : nullptr, ranges, intensities,
                     beam_count, angle_increment, ascend_status);
}

// ---- dense-capsule decode (SURVEY.md 8(f) rank 1) ---------------------------------------------
rpl_result rpl_decode_dense_batch_dev(rpl_ctx* c, const uint8_t* capsules, const uint32_t* capsule_counts,
                                      uint32_t n_streams, uint32_t stride_capsules, uint32_t sample_duration_us,
                                      const uint32_t* sync_state_in, rpl_node_hq* nodes_out,
                                      uint32_t* node_counts, uint32_t* capsule_status,
                                      uint32_t* capsule_node_offset, uint32_t* sync_state_out, void* stream) {
  return rpl_decode_dense_batch_starts_dev(c, capsules, capsule_counts, n_streams, stride_capsules, sample_duration_us,
                                           sync_state_in, nodes_out, node_counts, capsule_status, capsule_node_offset,
                                           sync_state_out, nullptr, 0, nullptr, stream);
}

rpl_result rpl_decode_dense_batch_starts_dev(rpl_ctx* c, const uint8_t* capsules, const uint32_t* capsule_counts,
                                             uint32_t n_streams, uint32_t stride_capsules, uint32_t sample_duration_us,
                                             const uint32_t* sync_state_in, rpl_node_hq* nodes_out,
                                             uint32_t* node_counts, uint32_t* capsule_status,
                                             uint32_t* capsule_node_offset, uint32_t* sync_state_out,
                                             uint32_t* scan_starts, uint32_t starts_stride, uint32_t* scan_start_counts,
                                             void* stream) {
  if (!c || !capsules || !capsule_counts || !nodes_out) return RPL_RESULT_INVALID_DATA;
  if ((scan_starts == nullptr) != (scan_start_counts == nullptr) || (scan_starts && starts_stride == 0)) {
    c->err = "scan_starts and scan_start_counts go together (starts_stride > 0)";
    return RPL_RESULT_INVALID_DATA;
  }
  if (sample_duration_us == 0 || sample_duration_us > 1000000u) {
    c->err = "sample_duration_us must be in [1, 1000000]";
    return RPL_RESULT_INVALID_DATA;
  }
  if ((reinterpret_cast<uintptr_t>(capsules) & 3u) != 0 || misaligned8(nodes_out)) {
    c->err = "capsule buffer must be 4-byte aligned, nodes_out 8-byte aligned";
    return RPL_RESULT_INVALID_DATA;
  }
  if (n_streams == 0) return RPL_RESULT_OK;
  RPL_CUDA(c, cudaSetDevice(c->device), RPL_RESULT_OPERATION_FAIL);
  cudaStream_t st = stream ? static_cast<cudaStream_t>(stream) : c->lane[0].stream;
  rpl::DecodeArgs a{};
  a.capsules = capsules;
  a.counts = capsule_counts;
  a.n_streams = n_streams;
  a.stride_capsules = stride_capsules;
  a.sample_duration_us = sample_duration_us;
  a.sync_state_in = sync_state_in;
  a.nodes_out = reinterpret_cast<uint2*>(nodes_out);
  a.node_counts = node_counts;
  a.capsule_status = capsule_status;
  a.capsule_node_offset = capsule_node_offset;
  a.sync_state_out = sync_state_out;
  a.scan_starts = scan_starts;
  a.scan_start_counts = scan_start_counts;
  a.starts_stride = starts_stride;
  const int grid = (int)std::min<uint32_t>(n_streams, (uint32_t)c->num_sms * 4u);
  RPL_CUDA(c, rpl::launch_decode_dense(a, grid, st), RPL_RESULT_OPERATION_FAIL);
  c->launches++;
  return RPL_RESULT_OK;
}

rpl_result rpl_decode_dense(rpl_ctx* c, const uint8_t* capsules, uint32_t n_capsules, uint32_t sample_duration_us,
                            uint32_t* sync_state, rpl_node_hq* nodes_out, uint32_t* node_count,
                            uint32_t* capsule_status, uint32_t* capsule_node_offset) {
  if (!c || !node_count || (n_capsules && (!capsules || !nodes_out))) return RPL_RESULT_INVALID_DATA;
  *node_count = 0;
  if (n_capsules == 0) return RPL_RESULT_OK;
  RPL_CUDA(c, cudaSetDevice(c->device), RPL_RESULT_OPERATION_FAIL);
  cudaStream_t st = c->lane[0].stream;
  const size_t cb = (size_t)n_capsules * 84, nb = (size_t)n_capsules * 40 * 8, sb = (size_t)n_capsules * 4;
  unsigned char* d = nullptr;  // [capsules | pad][nodes][status][offsets][count, n_nodes, sync in, sync out]
  const size_t o_nodes = (cb + 15) & ~(size_t)15, o_st = o_nodes + nb, o_off = o_st + sb, o_small = o_off + sb;
  RPL_CUDA(c, cudaMalloc(reinterpret_cast<void**>(&d), o_small + 16), RPL_RESULT_INSUFFICIENT_MEMORY);
  uint32_t small[4] = {n_capsules, 0u, sync_state ? (*sync_state & 1u) : 0u, 0u};
  rpl_result r = RPL_RESULT_OK;
  auto bail = [&](rpl_result code) {
    cudaFree(d);
    return code;
  };
  if (!cuda_ok(c, cudaMemcpyAsync(d, capsules, cb, cudaMemcpyHostToDevice, st), "H2D") ||
      !cuda_ok(c, cudaMemcpyAsync(d + o_small, small, 16, cudaMemcpyHostToDevice, st), "H2D"))
    return bail(RPL_RESULT_OPERATION_FAIL);
  uint32_t* ds = reinterpret_cast<uint32_t*>(d + o_small);
  r = rpl_decode_dense_batch_dev(c, d, ds, 1, n_capsules, sample_duration_us, ds + 2,
                                 reinterpret_cast<rpl_node_hq*>(d + o_nodes), ds + 1,
                                 reinterpret_cast<uint32_t*>(d + o_st), reinterpret_cast<uint32_t*>(d + o_off), ds + 3, st);
  if (r != RPL_RESULT_OK) return bail(r);
  if (!cuda_ok(c, cudaMemcpyAsync(small, ds, 16, cudaMemcpyDeviceToHost, st), "D2H") ||
      !cuda_ok(c, cudaStreamSynchronize(st), "sync"))
    return bail(RPL_RESULT_OPERATION_FAIL);
  *node_count = small[1];
  if (sync_state) *sync_state = small[3];
  if (!cuda_ok(c, cudaMemcpy(nodes_out, d + o_nodes, (size_t)small[1] * 8, cudaMemcpyDeviceToHost), "D2H"))
    return bail(RPL_RESULT_OPERATION_FAIL);
  if (capsule_status && !cuda_ok(c, cudaMemcpy(capsule_status, d + o_st, sb, cudaMemcpyDeviceToHost), "D2H"))
    return bail(RPL_RESULT_OPERATION_FAIL);
  if (capsule_node_offset && !cuda_ok(c, cudaMemcpy(capsule_node_offset, d + o_off, sb, cudaMemcpyDeviceToHost), "D2H"))
    return bail(RPL_RESULT_OPERATION_FAIL);
  return bail(RPL_RESULT_OK);
}

// ---- the other answer formats (SURVEY.md 8(f) rank 1) ----------------------------------------------
uint32_t rpl_capsule_bytes(uint32_t ans_type) {
  switch (ans_type) {
    case 0x82: return 84;
    case 0x83: return 781;
    case 0x84: return 132;
    case 0x85: return 84;
    case 0x86: return 170;
    default: return 0;
  }
}
uint32_t rpl_capsule_nodes(uint32_t ans_type) {
  switch (ans_type) {
    case 0x82: return 32;
    case 0x83: return 96;
    case 0x84: return 96;
    case 0x85: return 40;
    case 0x86: return 64;
    default: return 0;
  }
}

namespace {
// word 0 of every [2]-state pair, strided: the dense kernel keeps a single word per stream
__global__ void gather_state_kernel(const uint32_t* in2, uint32_t* out1, uint32_t n) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out1[i] = in2[2 * i] & 1u;
}
__global__ void scatter_state_kernel(const uint32_t* in1, uint32_t* out2, uint32_t n) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) {
    out2[2 * i] = in1[i];
    out2[2 * i + 1] = 0u;
  }
}
}  // namespace

rpl_result rpl_decode_capsules_batch_dev(rpl_ctx* c, uint32_t ans_type, const uint8_t* capsules,
                                         const uint32_t* capsule_counts, uint32_t n_streams,
                                         uint32_t stride_capsules, uint32_t sample_duration_us,
                                         const uint32_t* state_in, rpl_node_hq* nodes_out, uint32_t* node_counts,
                                         uint32_t* capsule_status, uint32_t* capsule_node_offset,
                                         uint32_t* state_out, void* stream) {
  if (!c || !capsules || !capsule_counts || !nodes_out) return RPL_RESULT_INVALID_DATA;
  if (rpl_capsule_bytes(ans_type) == 0) {
    c->err = "unknown answer type (capsule formats are 0x82..0x86)";
    return RPL_RESULT_INVALID_DATA;
  }
  if (misaligned8(nodes_out)) {
    c->err = "nodes_out must be 8-byte aligned";
    return RPL_RESULT_INVALID_DATA;
  }
  if (sample_duration_us == 0 || sample_duration_us > 1000000u) {
    c->err = "sample_duration_us must be in [1, 1000000]";
    return RPL_RESULT_INVALID_DATA;
  }
  if (n_streams == 0) return RPL_RESULT_OK;
  RPL_CUDA(c, cudaSetDevice(c->device), RPL_RESULT_OPERATION_FAIL);
  cudaStream_t st = stream ? static_cast<cudaStream_t>(stream) : c->lane[0].stream;
  if (ans_type == 0x85) {  // the dense kernel keeps one state word per stream
    uint32_t* tmp = nullptr;
    if (state_in || state_out) {
      if (n_streams > c->state_tmp_cap) {
        cudaFree(c->d_state_tmp);
        c->d_state_tmp = nullptr;
        RPL_CUDA(c, dev_alloc(&c->d_state_tmp, (size_t)2 * n_streams), RPL_RESULT_INSUFFICIENT_MEMORY);
        c->state_tmp_cap = n_streams;
      }
      tmp = c->d_state_tmp;
    }
    const uint32_t blocks = (n_streams + 255) / 256;
    if (state_in) gather_state_kernel<<<blocks, 256, 0, st>>>(state_in, tmp, n_streams);
    rpl_result r = rpl_decode_dense_batch_dev(c, capsules, capsule_counts, n_streams, stride_capsules,
                                              sample_duration_us, state_in ? tmp : nullptr, nodes_out, node_counts,
                                              capsule_status, capsule_node_offset,
                                              state_out ? tmp + n_streams : nullptr, st);
    if (r != RPL_RESULT_OK) return r;
    if (state_out) scatter_state_kernel<<<blocks, 256, 0, st>>>(tmp + n_streams, state_out, n_streams);
    RPL_CUDA(c, cudaGetLastError(), RPL_RESULT_OPERATION_FAIL);
    return RPL_RESULT_OK;
  }
  rpl::CapsuleDecodeArgs a{};
  a.capsules = capsules;
  a.counts = capsule_counts;
  a.n_streams = n_streams;
  a.stride_capsules = stride_capsules;
  a.sample_duration_us = sample_duration_us;
  a.state_in = state_in;
  a.nodes_out = reinterpret_cast<uint2*>(nodes_out);
  a.node_counts = node_counts;
  a.capsule_status = capsule_status;
  a.capsule_node_offset = capsule_node_offset;
  a.state_out = state_out;
  // one CTA per stream while they fit (express / ultra: five CTAs per SM by shared memory, ultra-dense two)
  const int grid = (int)std::min<uint32_t>(n_streams, (uint32_t)c->num_sms * 8u);
  RPL_CUDA(c, rpl::launch_decode_capsules(ans_type, a, grid, st), RPL_RESULT_OPERATION_FAIL);
  c->launches++;
  return RPL_RESULT_OK;
}

namespace {
// one stream from host buffers through a device-side entry: shared by the capsule and byte decoders
struct HostDecode {
  unsigned char* d = nullptr;
  size_t o_nodes = 0, o_st = 0, o_off = 0, o_small = 0;
  ~HostDecode() { cudaFree(d); }
};
}  // namespace

rpl_result rpl_decode_capsules(rpl_ctx* c, uint32_t ans_type, const uint8_t* capsules, uint32_t n_capsules,
                               uint32_t sample_duration_us, uint32_t* state, rpl_node_hq* nodes_out,
                               uint32_t* node_count, uint32_t* capsule_status, uint32_t* capsule_node_offset,
                               const rpl_timing* timing, const uint64_t* capsule_rx_us, uint64_t* node_ts_us) {
  if (!c || !node_count || (n_capsules && (!capsules || !nodes_out))) return RPL_RESULT_INVALID_DATA;
  const bool want_ts = timing || capsule_rx_us || node_ts_us;
  if (want_ts && !(timing && capsule_rx_us && node_ts_us)) {
    c->err = "timing, capsule_rx_us and node_ts_us go together";
    return RPL_RESULT_INVALID_DATA;
  }
  if (want_ts) sample_duration_us = timing->sample_duration_us;
  *node_count = 0;
  const uint32_t cbytes = rpl_capsule_bytes(ans_type), per = rpl_capsule_nodes(ans_type);
  if (cbytes == 0) {
    c->err = "unknown answer type (capsule formats are 0x82..0x86)";
    return RPL_RESULT_INVALID_DATA;
  }
  if (n_capsules == 0) return RPL_RESULT_OK;
  RPL_CUDA(c, cudaSetDevice(c->device), RPL_RESULT_OPERATION_FAIL);
  cudaStream_t st = c->lane[0].stream;
  const size_t cb = (size_t)n_capsules * cbytes, nb = (size_t)n_capsules * per * 8, sb = (size_t)n_capsules * 4;
  HostDecode h;  // [capsules | pad][nodes][status][offsets][count, n_nodes, state in x2, state out x2][rx][ts]
  h.o_nodes = (cb + 15) & ~(size_t)15;
  h.o_st = h.o_nodes + nb;
  h.o_off = h.o_st + sb;
  h.o_small = h.o_off + sb;
  const size_t o_rx = (h.o_small + 32 + 7) & ~(size_t)7, o_ts = o_rx + (size_t)n_capsules * 8;
  const size_t total_bytes = want_ts ? o_ts + (size_t)n_capsules * per * 8 : h.o_small + 32;
  RPL_CUDA(c, cudaMalloc(reinterpret_cast<void**>(&h.d), total_bytes), RPL_RESULT_INSUFFICIENT_MEMORY);
  uint32_t small[8] = {n_capsules, 0u, state ? state[0] : 0u, state ? state[1] : 0u, 0u, 0u, 0u, 0u};
  RPL_CUDA(c, cudaMemcpyAsync(h.d, capsules, cb, cudaMemcpyHostToDevice, st), RPL_RESULT_OPERATION_FAIL);
  RPL_CUDA(c, cudaMemcpyAsync(h.d + h.o_small, small, 32, cudaMemcpyHostToDevice, st), RPL_RESULT_OPERATION_FAIL);
  uint32_t* ds = reinterpret_cast<uint32_t*>(h.d + h.o_small);
  rpl_result r = rpl_decode_capsules_batch_dev(c, ans_type, h.d, ds, 1, n_capsules, sample_duration_us, ds + 2,
                                               reinterpret_cast<rpl_node_hq*>(h.d + h.o_nodes), ds + 1,
                                               reinterpret_cast<uint32_t*>(h.d + h.o_st),
                                               reinterpret_cast<uint32_t*>(h.d + h.o_off), ds + 4, st);
  if (r != RPL_RESULT_OK) return r;
  if (want_ts) {
    RPL_CUDA(c, cudaMemcpyAsync(h.d + o_rx, capsule_rx_us, (size_t)n_capsules * 8, cudaMemcpyHostToDevice, st),
             RPL_RESULT_OPERATION_FAIL);
    r = rpl_node_timestamps_dev(c, ans_type, timing, reinterpret_cast<const uint64_t*>(h.d + o_rx),
                                reinterpret_cast<uint32_t*>(h.d + h.o_st), reinterpret_cast<uint32_t*>(h.d + h.o_off), ds,
                                1, n_capsules, reinterpret_cast<uint64_t*>(h.d + o_ts), st);
    if (r != RPL_RESULT_OK) return r;
  }
  RPL_CUDA(c, cudaMemcpyAsync(small, ds, 32, cudaMemcpyDeviceToHost, st), RPL_RESULT_OPERATION_FAIL);
  RPL_CUDA(c, cudaStreamSynchronize(st), RPL_RESULT_OPERATION_FAIL);
  *node_count = small[1];
  if (state) {
    state[0] = small[4];
    state[1] = small[5];
  }
  if (want_ts)
    RPL_CUDA(c, cudaMemcpy(node_ts_us, h.d + o_ts, (size_t)small[1] * 8, cudaMemcpyDeviceToHost),
             RPL_RESULT_OPERATION_FAIL);
  RPL_CUDA(c, cudaMemcpy(nodes_out, h.d + h.o_nodes, (size_t)small[1] * 8, cudaMemcpyDeviceToHost),
           RPL_RESULT_OPERATION_FAIL);
  if (capsule_status)
    RPL_CUDA(c, cudaMemcpy(capsule_status, h.d + h.o_st, sb, cudaMemcpyDeviceToHost), RPL_RESULT_OPERATION_FAIL);
  if (capsule_node_offset)
    RPL_CUDA(c, cudaMemcpy(capsule_node_offset, h.d + h.o_off, sb, cudaMemcpyDeviceToHost), RPL_RESULT_OPERATION_FAIL);
  return RPL_RESULT_OK;
}

rpl_result rpl_frame_capsules_dev(rpl_ctx* c, uint32_t ans_type, const uint8_t* bytes, const uint32_t* byte_counts,
                                  uint32_t n_streams, uint32_t stride_bytes, uint8_t* capsules_out,
                                  uint32_t stride_capsules, uint32_t* capsule_counts_out, uint32_t* bytes_left_out,
                                  void* stream) {
  if (!c || !bytes || !byte_counts || !capsules_out || !capsule_counts_out) return RPL_RESULT_INVALID_DATA;
  const uint32_t cb = rpl_capsule_bytes(ans_type);
  if (cb == 0 || ans_type == 0x83) {
    c->err = "byte-level framing serves the capsule formats with sync nibbles: 0x82, 0x84, 0x85, 0x86";
    return RPL_RESULT_INVALID_DATA;
  }
  if (n_streams == 0) return RPL_RESULT_OK;
  RPL_CUDA(c, cudaSetDevice(c->device), RPL_RESULT_OPERATION_FAIL);
  cudaStream_t st = stream ? static_cast<cudaStream_t>(stream) : c->lane[0].stream;
  rpl::FrameArgs a{};
  a.bytes = bytes;
  a.byte_counts = byte_counts;
  a.n_streams = n_streams;
  a.stride_bytes = stride_bytes;
  a.capsule_bytes = cb;
  a.capsules_out = capsules_out;
  a.stride_capsules = stride_capsules;
  a.capsule_counts_out = capsule_counts_out;
  a.bytes_left_out = bytes_left_out;
  const int grid = (int)std::min<uint32_t>(n_streams, (uint32_t)c->num_sms * 8u);
  RPL_CUDA(c, rpl::launch_frame_capsules(a, grid, st), RPL_RESULT_OPERATION_FAIL);
  c->launches++;
  return RPL_RESULT_OK;
}

rpl_result rpl_decode_normal_batch_dev(rpl_ctx* c, const uint8_t* bytes, const uint32_t* byte_counts,
                                       uint32_t n_streams, uint32_t stride_bytes, rpl_node_hq* nodes_out,
                                       uint32_t* node_counts, uint32_t* fsm_state_out, uint32_t* node_end,
                                       void* stream) {
  if (!c || !bytes || !byte_counts || !nodes_out) return RPL_RESULT_INVALID_DATA;
  if (misaligned8(nodes_out)) {
    c->err = "nodes_out must be 8-byte aligned";
    return RPL_RESULT_INVALID_DATA;
  }
  if (n_streams == 0) return RPL_RESULT_OK;
  RPL_CUDA(c, cudaSetDevice(c->device), RPL_RESULT_OPERATION_FAIL);
  cudaStream_t st = stream ? static_cast<cudaStream_t>(stream) : c->lane[0].stream;
  rpl::NormalDecodeArgs a{};
  a.bytes = bytes;
  a.byte_counts = byte_counts;
  a.n_streams = n_streams;
  a.stride_bytes = stride_bytes;
  a.nodes_out = reinterpret_cast<uint2*>(nodes_out);
  a.node_counts = node_counts;
  a.fsm_state_out = fsm_state_out;
  a.node_end = node_end;
  const int grid = (int)std::min<uint32_t>(n_streams, (uint32_t)c->num_sms * 8u);
  RPL_CUDA(c, rpl::launch_decode_normal(a, grid, st), RPL_RESULT_OPERATION_FAIL);
  c->launches++;
  return RPL_RESULT_OK;
}

rpl_result rpl_decode_normal(rpl_ctx* c, const uint8_t* bytes, uint32_t n_bytes, rpl_node_hq* nodes_out,
                             uint32_t* node_count) {
  if (!c || !node_count || (n_bytes && (!bytes || !nodes_out))) return RPL_RESULT_INVALID_DATA;
  *node_count = 0;
  if (n_bytes < 5) return RPL_RESULT_OK;
  RPL_CUDA(c, cudaSetDevice(c->device), RPL_RESULT_OPERATION_FAIL);
  cudaStream_t st = c->lane[0].stream;
  HostDecode h;  // [bytes | pad][nodes][byte count, node count]
  h.o_nodes = ((size_t)n_bytes + 15) & ~(size_t)15;
  h.o_small = h.o_nodes + (size_t)(n_bytes / 5) * 8;
  RPL_CUDA(c, cudaMalloc(reinterpret_cast<void**>(&h.d), h.o_small + 16), RPL_RESULT_INSUFFICIENT_MEMORY);
  uint32_t small[2] = {n_bytes, 0u};
  RPL_CUDA(c, cudaMemcpyAsync(h.d, bytes, n_bytes, cudaMemcpyHostToDevice, st), RPL_RESULT_OPERATION_FAIL);
  RPL_CUDA(c, cudaMemcpyAsync(h.d + h.o_small, small, 8, cudaMemcpyHostToDevice, st), RPL_RESULT_OPERATION_FAIL);
  uint32_t* ds = reinterpret_cast<uint32_t*>(h.d + h.o_small);
  rpl_result r = rpl_decode_normal_batch_dev(c, h.d, ds, 1, n_bytes, reinterpret_cast<rpl_node_hq*>(h.d + h.o_nodes),
                                             ds + 1, nullptr, nullptr, st);
  if (r != RPL_RESULT_OK) return r;
  RPL_CUDA(c, cudaMemcpyAsync(small, ds, 8, cudaMemcpyDeviceToHost, st), RPL_RESULT_OPERATION_FAIL);
  RPL_CUDA(c, cudaStreamSynchronize(st), RPL_RESULT_OPERATION_FAIL);
  *node_count = small[1];
  RPL_CUDA(c, cudaMemcpy(nodes_out, h.d + h.o_nodes, (size_t)small[1] * 8, cudaMemcpyDeviceToHost),
           RPL_RESULT_OPERATION_FAIL);
  return RPL_RESULT_OK;
}

// ---- scan assembly (SURVEY.md 8(f) rank 2) ------------------------------------------------------
}  // extern "C"

namespace {
// copy mode (scans_out) or view mode (views_out + writable nodes)
rpl_result assemble_common(rpl_ctx* c, const rpl_node_hq* nodes, const uint32_t* node_counts,
                                  uint32_t n_streams, uint32_t stride_nodes, const uint32_t* capsule_status,
                                  const uint32_t* capsule_node_offset, const uint32_t* capsule_counts,
                                  uint32_t stride_capsules, uint32_t max_nodes, uint32_t max_scans,
                                  uint32_t scan_stride, rpl_node_hq* scans_out, rpl_scan_view* views_out, uint32_t* scan_len,
                                  uint32_t* scans_per_stream, const uint64_t* node_ts_us,
                                  uint64_t* scan_begin_ts_us, void* stream, const uint32_t* scan_starts = nullptr,
                                  uint32_t starts_stride = 0, const uint32_t* scan_start_counts = nullptr) {
  if (!c || !nodes || !node_counts || (!scans_out && !views_out) || !scan_len || !scans_per_stream) return RPL_RESULT_INVALID_DATA;
  const bool any = capsule_status || capsule_node_offset || capsule_counts;
  if (any && !(capsule_status && capsule_node_offset && capsule_counts)) {
    c->err = "capsule_status, capsule_node_offset and capsule_counts go together";
    return RPL_RESULT_INVALID_DATA;
  }
  if (max_nodes == 0 || max_scans == 0 || scan_stride < max_nodes) {
    c->err = "need max_nodes > 0, max_scans > 0, scan_stride >= max_nodes";
    return RPL_RESULT_INVALID_DATA;
  }
  if (misaligned8(nodes) || misaligned8(scans_out) || misaligned8(node_ts_us) || misaligned8(scan_begin_ts_us)) {
    c->err = "node and timestamp buffers must be 8-byte aligned";
    return RPL_RESULT_INVALID_DATA;
  }
  if (n_streams == 0) return RPL_RESULT_OK;
  RPL_CUDA(c, cudaSetDevice(c->device), RPL_RESULT_OPERATION_FAIL);
  const size_t need_rp = (size_t)n_streams * std::max<uint32_t>(stride_capsules, 1u);
  const size_t need_desc = (size_t)n_streams * max_scans;
  if (need_rp > c->reset_prefix_cap) {
    cudaFree(c->d_reset_prefix);
    c->d_reset_prefix = nullptr;
    RPL_CUDA(c, dev_alloc(&c->d_reset_prefix, need_rp), RPL_RESULT_INSUFFICIENT_MEMORY);
    c->reset_prefix_cap = need_rp;
  }
  if (need_desc > c->desc_cap) {
    cudaFree(c->d_desc);
    c->d_desc = nullptr;
    RPL_CUDA(c, dev_alloc(&c->d_desc, need_desc), RPL_RESULT_INSUFFICIENT_MEMORY);
    c->desc_cap = need_desc;
  }
  cudaStream_t st = stream ? static_cast<cudaStream_t>(stream) : c->lane[0].stream;
  rpl::AssembleArgs a{};
  a.nodes = reinterpret_cast<const uint2*>(nodes);
  a.node_counts = node_counts;
  a.n_streams = n_streams;
  a.stride_nodes = stride_nodes;
  a.capsule_status = capsule_status;
  a.capsule_node_offset = capsule_node_offset;
  a.capsule_counts = capsule_counts;
  a.stride_capsules = std::max<uint32_t>(stride_capsules, 1u);
  a.max_nodes = max_nodes;
  a.max_scans = max_scans;
  a.scan_stride = scan_stride;
  a.scans_out = reinterpret_cast<uint2*>(scans_out);
  a.views_out = reinterpret_cast<uint2*>(views_out);
  a.nodes_mut = views_out ? reinterpret_cast<uint2*>(const_cast<rpl_node_hq*>(nodes)) : nullptr;
  a.scan_len = scan_len;
  a.scans_per_stream = scans_per_stream;
  a.node_ts_us = reinterpret_cast<const unsigned long long*>(node_ts_us);
  a.scan_begin_ts_us = reinterpret_cast<unsigned long long*>(scan_begin_ts_us);
  a.scan_starts = scan_starts;
  a.scan_start_counts = scan_start_counts;
  a.starts_stride = starts_stride;
  a.reset_prefix = c->d_reset_prefix;
  a.desc = c->d_desc;
  const int grid = (int)std::min<uint32_t>(n_streams, (uint32_t)c->num_sms * 4u);
  RPL_CUDA(c, rpl::launch_assemble(a, grid, st), RPL_RESULT_OPERATION_FAIL);
  c->launches++;
  return RPL_RESULT_OK;
}
}  // namespace

extern "C" {

rpl_result rpl_assemble_scans_dev(rpl_ctx* c, const rpl_node_hq* nodes, const uint32_t* node_counts,
                                  uint32_t n_streams, uint32_t stride_nodes, const uint32_t* capsule_status,
                                  const uint32_t* capsule_node_offset, const uint32_t* capsule_counts,
                                  uint32_t stride_capsules, uint32_t max_nodes, uint32_t max_scans,
                                  uint32_t scan_stride, rpl_node_hq* scans_out, uint32_t* scan_len,
                                  uint32_t* scans_per_stream, const uint64_t* node_ts_us,
                                  uint64_t* scan_begin_ts_us, void* stream) {
  if (!scans_out) return RPL_RESULT_INVALID_DATA;
  return assemble_common(c, nodes, node_counts, n_streams, stride_nodes, capsule_status, capsule_node_offset,
                         capsule_counts, stride_capsules, max_nodes, max_scans, scan_stride, scans_out, nullptr, scan_len,
                         scans_per_stream, node_ts_us, scan_begin_ts_us, stream);
}

rpl_result rpl_assemble_scan_views_dev(rpl_ctx* c, rpl_node_hq* nodes, const uint32_t* node_counts,
                                       uint32_t n_streams, uint32_t stride_nodes, const uint32_t* capsule_status,
                                       const uint32_t* capsule_node_offset, const uint32_t* capsule_counts,
                                       uint32_t stride_capsules, uint32_t max_nodes, uint32_t max_scans,
                                       rpl_scan_view* views_out, uint32_t* scan_len, uint32_t* scans_per_stream,
                                       const uint64_t* node_ts_us, uint64_t* scan_begin_ts_us, void* stream) {
  if (!views_out) return RPL_RESULT_INVALID_DATA;
  if ((unsigned long long)n_streams * stride_nodes > 0xFFFFFFFFull) {
    if (c) c->err = "view mode addresses nodes with 32 bits: n_streams * stride_nodes must stay below 2^32";
    return RPL_RESULT_INVALID_DATA;
  }
  return assemble_common(c, nodes, node_counts, n_streams, stride_nodes, capsule_status, capsule_node_offset,
                         capsule_counts, stride_capsules, max_nodes, max_scans, max_nodes, nullptr, views_out, scan_len,
                         scans_per_stream, node_ts_us, scan_begin_ts_us, stream);
}

rpl_result rpl_assemble_scan_views_starts_dev(rpl_ctx* c, rpl_node_hq* nodes, const uint32_t* node_counts,
                                              uint32_t n_streams, uint32_t stride_nodes, const uint32_t* capsule_status,
                                              const uint32_t* capsule_node_offset, const uint32_t* capsule_counts,
                                              uint32_t stride_capsules, const uint32_t* scan_starts,
                                              uint32_t starts_stride, const uint32_t* scan_start_counts,
                                              uint32_t max_nodes, uint32_t max_scans, rpl_scan_view* views_out,
                                              uint32_t* scan_len, uint32_t* scans_per_stream, const uint64_t* node_ts_us,
                                              uint64_t* scan_begin_ts_us, void* stream) {
  if (!views_out || !scan_starts || !scan_start_counts || starts_stride == 0) return RPL_RESULT_INVALID_DATA;
  if ((unsigned long long)n_streams * stride_nodes > 0xFFFFFFFFull) {
    if (c) c->err = "view mode addresses nodes with 32 bits: n_streams * stride_nodes must stay below 2^32";
    return RPL_RESULT_INVALID_DATA;
  }
  return assemble_common(c, nodes, node_counts, n_streams, stride_nodes, capsule_status, capsule_node_offset,
                         capsule_counts, stride_capsules, max_nodes, max_scans, max_nodes, nullptr, views_out, scan_len,
                         scans_per_stream, node_ts_us, scan_begin_ts_us, stream, scan_starts, starts_stride,
                         scan_start_counts);
}

rpl_result rpl_scan_views_dev(rpl_ctx* c, const rpl_node_hq* nodes, uint64_t nodes_total, const rpl_scan_view* views,
                              uint32_t n_scans, uint32_t stride, const rpl_scan_params* params, rpl_node_hq* nodes_out,
                              float* ranges, float* intensities, uint32_t* beam_counts, float* angle_increment,
                              uint32_t* status, uint32_t* path, void* stream) {
  if (!c || !views || !nodes || !params) return RPL_RESULT_INVALID_DATA;
  if (!rpl::scan_small_applies(stride) || (params->flags & RPL_FLAG_NO_SMALL)) {
    c->err = "scan views are served by the shared-memory kernels: stride (the longest scan) must be <= 8192 nodes";
    return RPL_RESULT_INVALID_DATA;
  }
  if ((reinterpret_cast<uintptr_t>(nodes) & 15u) != 0) {
    c->err = "the node buffer of a view batch must be 16-byte aligned";
    return RPL_RESULT_INVALID_DATA;
  }
  if (nodes_out && !params->apply_ascend) {
    // the batch path's pass-through is one strided copy of [n_scans][stride] nodes, which views do not have
    c->err = "nodes_out of a view batch needs apply_ascend (the unascended nodes are the views themselves)";
    return RPL_RESULT_INVALID_DATA;
  }
  RPL_CUDA(c, cudaSetDevice(c->device), RPL_RESULT_OPERATION_FAIL);
  cudaStream_t st = stream ? static_cast<cudaStream_t>(stream) : c->lane[0].stream;
  return enqueue_scan(c, c->lane[0], nodes, reinterpret_cast<const uint32_t*>(views), n_scans, stride, params, nodes_out,
                      ranges, intensities, beam_counts, angle_increment, status, path, st,
                      reinterpret_cast<const uint2*>(views), nodes_total);
}

// ---- wire bytes -> LaserScan in one host call --------------------------------------------------------------------
rpl_result rpl_chain_dense_laserscan(rpl_ctx* c, const uint8_t* capsules, const uint32_t* capsule_counts,
                                     uint32_t n_streams, uint32_t stride_capsules, uint32_t sample_duration_us,
                                     const rpl_scan_params* params, uint32_t max_nodes, uint32_t max_scans,
                                     float* ranges, float* intensities, uint32_t* beam_counts, float* angle_increment,
                                     uint32_t* scans_per_stream) {
  if (!c || !capsules || !capsule_counts || !params || !ranges || !intensities || !beam_counts || !scans_per_stream)
    return RPL_RESULT_INVALID_DATA;
  if (n_streams == 0) return RPL_RESULT_OK;
  if (max_nodes == 0 || max_nodes > rpl::kSmallMaxNodes || (max_nodes & 1u) || max_scans == 0 || stride_capsules == 0) {
    c->err = "need an even max_nodes in [2, 8192] (the longest revolution), max_scans > 0, stride_capsules > 0";
    return RPL_RESULT_INVALID_DATA;
  }
  if (max_nodes > c->max_nodes) {
    // the scan kernels would report every longer revolution as INVALID_DATA into a status nobody reads
    c->err = "max_nodes exceeds the context's max_nodes";
    return RPL_RESULT_INVALID_DATA;
  }
  for (uint32_t s = 0; s < n_streams; ++s)
    if (capsule_counts[s] > stride_capsules) {
      c->err = "capsule_counts[s] exceeds stride_capsules";
      return RPL_RESULT_INVALID_DATA;
    }
  RPL_CUDA(c, cudaSetDevice(c->device), RPL_RESULT_OPERATION_FAIL);
  // chunk: about 16 MiB of capsules (~64 MiB of decoded nodes), whole streams
  const size_t cap_bytes_stream = (size_t)stride_capsules * 84;
  uint32_t chunk = (uint32_t)std::max<size_t>(1, ((size_t)16 << 20) / cap_bytes_stream);
  chunk = std::min(chunk, n_streams);
  if ((size_t)chunk * max_scans > c->max_scans) chunk = c->max_scans / max_scans;
  if (chunk == 0) {
    c->err = "the context's max_scans is smaller than max_scans of one stream";
    return RPL_RESULT_INVALID_DATA;
  }
  const size_t nodes_stream = (size_t)stride_capsules * 40;
  if ((size_t)chunk * nodes_stream > 0xFFFFFFFFull) {
    c->err = "chunk too large for 32-bit views";
    return RPL_RESULT_INVALID_DATA;
  }
  auto up = [](size_t v) { return (v + 255) & ~(size_t)255; };
  const size_t NS = (size_t)chunk * max_scans;
  const uint32_t starts_stride = 2 * max_scans + 64;  // scan starts per stream the decoder may list
  const size_t o_caps = 0, o_ccnt = o_caps + up(chunk * cap_bytes_stream), o_nodes = o_ccnt + up((size_t)chunk * 4),
               o_ncnt = o_nodes + up(chunk * nodes_stream * 8), o_st = o_ncnt + up((size_t)chunk * 4),
               o_off = o_st + up((size_t)chunk * stride_capsules * 4), o_views = o_off + up((size_t)chunk * stride_capsules * 4),
               o_slen = o_views + up(NS * 8), o_sps = o_slen + up(NS * 4), o_r = o_sps + up((size_t)chunk * 4),
               o_i = o_r + up(NS * max_nodes * 4), o_b = o_i + up(NS * max_nodes * 4), o_inc = o_b + up(NS * 4),
               o_starts = o_inc + up(NS * 4), o_scnt = o_starts + up((size_t)chunk * starts_stride * 4),
               total = o_scnt + up((size_t)chunk * 4);
  for (int i = 0; i < kLanes; ++i) {
    Lane& l = c->lane[i];
    if (l.chain_bytes < total) {
      RPL_CUDA(c, cudaStreamSynchronize(l.stream), RPL_RESULT_OPERATION_FAIL);
      cudaFree(l.d_chain);
      l.d_chain = nullptr;
      l.chain_bytes = 0;
      RPL_CUDA(c, cudaMalloc(reinterpret_cast<void**>(&l.d_chain), total), RPL_RESULT_INSUFFICIENT_MEMORY);
      l.chain_bytes = total;
    }
  }
  const cudaMemcpyKind h2d = cudaMemcpyHostToDevice, d2h = cudaMemcpyDeviceToHost;
  auto run_chunk = [&](Lane& l, uint32_t s0, uint32_t ns) -> rpl_result {
    unsigned char* d = l.d_chain;
    const size_t nsc = (size_t)ns * max_scans;
    RPL_CUDA(c, cudaStreamSynchronize(l.stream), RPL_RESULT_OPERATION_FAIL);  // the lane's previous chunk has left
    RPL_CUDA(c, cudaMemcpyAsync(d + o_caps, capsules + (size_t)s0 * cap_bytes_stream, ns * cap_bytes_stream, h2d, l.stream),
             RPL_RESULT_OPERATION_FAIL);
    RPL_CUDA(c, cudaMemcpyAsync(d + o_ccnt, capsule_counts + s0, (size_t)ns * 4, h2d, l.stream), RPL_RESULT_OPERATION_FAIL);
    rpl_result r = rpl_decode_dense_batch_starts_dev(
        c, d + o_caps, reinterpret_cast<uint32_t*>(d + o_ccnt), ns, stride_capsules, sample_duration_us, nullptr,
        reinterpret_cast<rpl_node_hq*>(d + o_nodes), reinterpret_cast<uint32_t*>(d + o_ncnt),
        reinterpret_cast<uint32_t*>(d + o_st), reinterpret_cast<uint32_t*>(d + o_off), nullptr,
        reinterpret_cast<uint32_t*>(d + o_starts), starts_stride, reinterpret_cast<uint32_t*>(d + o_scnt), l.stream);
    if (r != RPL_RESULT_OK) return r;
    // the assembler's scratch belongs to the context, not to the lane: one assemble kernel at a time
    if (!c->asm_done) RPL_CUDA(c, cudaEventCreateWithFlags(&c->asm_done, cudaEventDisableTiming), RPL_RESULT_OPERATION_FAIL);
    RPL_CUDA(c, cudaStreamWaitEvent(l.stream, c->asm_done, 0), RPL_RESULT_OPERATION_FAIL);
    r = rpl_assemble_scan_views_starts_dev(c, reinterpret_cast<rpl_node_hq*>(d + o_nodes), reinterpret_cast<uint32_t*>(d + o_ncnt), ns,
                                    (uint32_t)nodes_stream, reinterpret_cast<uint32_t*>(d + o_st),
                                    reinterpret_cast<uint32_t*>(d + o_off), reinterpret_cast<uint32_t*>(d + o_ccnt),
                                    stride_capsules, reinterpret_cast<uint32_t*>(d + o_starts), starts_stride,
                                    reinterpret_cast<uint32_t*>(d + o_scnt), max_nodes, max_scans,
                                    reinterpret_cast<rpl_scan_view*>(d + o_views),
                                    reinterpret_cast<uint32_t*>(d + o_slen), reinterpret_cast<uint32_t*>(d + o_sps), nullptr,
                                    nullptr, l.stream);
    if (r != RPL_RESULT_OK) return r;
    RPL_CUDA(c, cudaEventRecord(c->asm_done, l.stream), RPL_RESULT_OPERATION_FAIL);
    r = enqueue_scan(c, l, reinterpret_cast<rpl_node_hq*>(d + o_nodes), reinterpret_cast<uint32_t*>(d + o_slen),
                     (uint32_t)nsc, max_nodes, params, nullptr, reinterpret_cast<float*>(d + o_r),
                     reinterpret_cast<float*>(d + o_i), reinterpret_cast<uint32_t*>(d + o_b),
                     reinterpret_cast<float*>(d + o_inc), nullptr, nullptr, l.stream,
                     reinterpret_cast<const uint2*>(d + o_views), (unsigned long long)ns * nodes_stream);
    if (r != RPL_RESULT_OK) return r;
    const size_t so = (size_t)s0 * max_scans;
    RPL_CUDA(c, cudaMemcpyAsync(ranges + so * max_nodes, d + o_r, nsc * max_nodes * 4, d2h, l.stream), RPL_RESULT_OPERATION_FAIL);
    RPL_CUDA(c, cudaMemcpyAsync(intensities + so * max_nodes, d + o_i, nsc * max_nodes * 4, d2h, l.stream),
             RPL_RESULT_OPERATION_FAIL);
    RPL_CUDA(c, cudaMemcpyAsync(beam_counts + so, d + o_b, nsc * 4, d2h, l.stream), RPL_RESULT_OPERATION_FAIL);
    if (angle_increment)
      RPL_CUDA(c, cudaMemcpyAsync(angle_increment + so, d + o_inc, nsc * 4, d2h, l.stream), RPL_RESULT_OPERATION_FAIL);
    RPL_CUDA(c, cudaMemcpyAsync(scans_per_stream + s0, d + o_sps, (size_t)ns * 4, d2h, l.stream), RPL_RESULT_OPERATION_FAIL);
    return RPL_RESULT_OK;
  };
  uint32_t ci = 0;
  for (uint32_t s0 = 0; s0 < n_streams; s0 += chunk, ++ci) {
    const rpl_result r = run_chunk(c->lane[ci % kLanes], s0, std::min(chunk, n_streams - s0));
    if (r != RPL_RESULT_OK) {
      const std::string why = c->err;
      for (int i = 0; i < kLanes; ++i) cudaStreamSynchronize(c->lane[i].stream);
      c->err = why;
      return r;
    }
  }
  return rpl_ctx_synchronize(c);
}

// ---- LaserScan / PointCloud2 -> CDR (SURVEY.md 8(f) rank 3) -------------------------------------
namespace {
struct CdrWriter {  // XCDR1 little endian; alignment counts from the byte after the encapsulation header
  uint8_t* b;
  uint32_t n = 0;
  explicit CdrWriter(uint8_t* buf) : b(buf) {
    const uint8_t enc[4] = {0x00, 0x01, 0x00, 0x00};
    std::memcpy(b, enc, 4);
    n = 4;
  }
  void align(uint32_t a) {
    while ((n - 4) % a) b[n++] = 0;
  }
  void u32(uint32_t v) {
    align(4);
    std::memcpy(b + n, &v, 4);
    n += 4;
  }
  void u8(uint8_t v) { b[n++] = v; }
  void str(const char* s, uint32_t len) {
    u32(len + 1);
    std::memcpy(b + n, s, len);
    n += len;
    b[n++] = 0;
  }
};
uint32_t header_bytes(uint32_t frame_id_len) { return 4 + ((12 + frame_id_len + 1 + 3) & ~3u); }
}  // namespace

uint32_t rpl_laserscan_cdr_size(uint32_t frame_id_len, uint32_t beam_count) {
  return header_bytes(frame_id_len) + 28 + 4 + 4 * beam_count + 4 + 4 * beam_count;
}

uint32_t rpl_pointcloud2_cdr_size(uint32_t frame_id_len, uint32_t n_points) {
  // height, width, fields count; x/y/z (20 bytes each), intensity (28); is_bigendian + pad; point_step,
  // row_step, data length; data; is_dense
  return header_bytes(frame_id_len) + 12 + 3 * 20 + 28 + 4 + 12 + 16 * n_points + 1;
}

rpl_result rpl_laserscan_cdr_batch_dev(rpl_ctx* c, const rpl_laserscan_meta* meta, const float* angle_increment,
                                       const char* frame_id, const float* ranges, const float* intensities,
                                       const uint32_t* beam_counts, uint32_t n_scans, uint32_t stride,
                                       uint8_t* cdr_out, uint32_t cdr_stride, uint32_t* cdr_sizes, void* stream) {
  if (!c || !meta || !frame_id || !ranges || !intensities || !beam_counts || !cdr_out) return RPL_RESULT_INVALID_DATA;
  const size_t L = std::strlen(frame_id);
  if (L > 255) {
    c->err = "frame_id longer than 255 characters";
    return RPL_RESULT_INVALID_DATA;
  }
  if ((cdr_stride & 3u) || cdr_stride < rpl_laserscan_cdr_size((uint32_t)L, stride) ||
      (reinterpret_cast<uintptr_t>(cdr_out) & 3u)) {
    c->err = "cdr_out must be 4-byte aligned, cdr_stride a multiple of 4 and >= rpl_laserscan_cdr_size(len, stride)";
    return RPL_RESULT_INVALID_DATA;
  }
  if (n_scans == 0) return RPL_RESULT_OK;
  RPL_CUDA(c, cudaSetDevice(c->device), RPL_RESULT_OPERATION_FAIL);
  cudaStream_t st = stream ? static_cast<cudaStream_t>(stream) : c->lane[0].stream;
  rpl::CdrTemplate t{};
  CdrWriter w(t.prefix);
  w.u32(0);  // stamp.sec     (patched)
  w.u32(0);  // stamp.nanosec (patched)
  w.str(frame_id, (uint32_t)L);
  for (int i = 0; i < 7; ++i) w.u32(0);  // angle_min .. range_max (patched)
  w.u32(0);                              // ranges count (patched)
  t.prefix_bytes = w.n;
  rpl::LaserScanCdrArgs a{};
  a.meta = reinterpret_cast<const rpl::LaserScanMeta*>(meta);
  a.angle_increment = angle_increment;
  a.ranges = ranges;
  a.intensities = intensities;
  a.beam_counts = beam_counts;
  a.n_scans = n_scans;
  a.stride = stride;
  a.cdr_out = cdr_out;
  a.cdr_stride = cdr_stride;
  a.cdr_sizes = cdr_sizes;
  RPL_CUDA(c, rpl::launch_laserscan_cdr(a, t, st), RPL_RESULT_OPERATION_FAIL);
  c->launches++;
  return RPL_RESULT_OK;
}

rpl_result rpl_pointcloud2_cdr_batch_dev(rpl_ctx* c, const uint32_t* stamps, const char* frame_id,
                                         const float* xyzi, const uint32_t* point_counts, uint32_t n_clouds,
                                         uint32_t stride, uint8_t* cdr_out, uint32_t cdr_stride,
                                         uint32_t* cdr_sizes, void* stream) {
  if (!c || !stamps || !frame_id || !xyzi || !point_counts || !cdr_out) return RPL_RESULT_INVALID_DATA;
  const size_t L = std::strlen(frame_id);
  if (L > 255) {
    c->err = "frame_id longer than 255 characters";
    return RPL_RESULT_INVALID_DATA;
  }
  if ((cdr_stride & 15u) || cdr_stride < rpl_pointcloud2_cdr_size((uint32_t)L, stride) ||
      (reinterpret_cast<uintptr_t>(cdr_out) & 15u)) {
    c->err = "cdr_out must be 16-byte aligned, cdr_stride a multiple of 16 and >= rpl_pointcloud2_cdr_size(len, stride)";
    return RPL_RESULT_INVALID_DATA;
  }
  if (n_clouds == 0) return RPL_RESULT_OK;
  RPL_CUDA(c, cudaSetDevice(c->device), RPL_RESULT_OPERATION_FAIL);
  cudaStream_t st = stream ? static_cast<cudaStream_t>(stream) : c->lane[0].stream;
  rpl::CdrTemplate t{};
  CdrWriter w(t.prefix);
  w.u32(0);
  w.u32(0);
  w.str(frame_id, (uint32_t)L);
  w.u32(1);  // height
  w.align(4);
  t.patch_width = w.n;
  w.u32(0);  // width (patched)
  w.u32(4);  // fields
  const char* names[4] = {"x", "y", "z", "intensity"};
  for (uint32_t f = 0; f < 4; ++f) {
    w.str(names[f], (uint32_t)std::strlen(names[f]));
    w.u32(4 * f);  // offset
    w.u8(7);       // datatype FLOAT32
    w.u32(1);      // count
  }
  w.u8(0);         // is_bigendian
  w.u32(16);       // point_step
  w.align(4);
  t.patch_row_step = w.n;
  w.u32(0);        // row_step (patched)
  w.u32(0);        // data length (patched)
  t.prefix_bytes = w.n;
  rpl::PointCloudCdrArgs a{};
  a.stamps = stamps;
  a.xyzi = xyzi;
  a.point_counts = point_counts;
  a.n_clouds = n_clouds;
  a.stride = stride;
  a.cdr_out = cdr_out;
  a.cdr_stride = cdr_stride;
  a.cdr_sizes = cdr_sizes;
  RPL_CUDA(c, rpl::launch_pointcloud2_cdr(a, t, st), RPL_RESULT_OPERATION_FAIL);
  c->launches++;
  return RPL_RESULT_OK;
}

// ---- per-sample timestamps (SURVEY.md 8(f) rank 4) ----------------------------------------------
rpl_result rpl_node_timestamps_dev(rpl_ctx* c, uint32_t ans_type, const rpl_timing* timing,
                                   const uint64_t* capsule_rx_us, const uint32_t* capsule_status,
                                   const uint32_t* capsule_node_offset, const uint32_t* capsule_counts,
                                   uint32_t n_streams, uint32_t stride_capsules, uint64_t* node_ts_us, void* stream) {
  if (!c || !timing || !capsule_rx_us || !capsule_status || !capsule_node_offset || !capsule_counts || !node_ts_us)
    return RPL_RESULT_INVALID_DATA;
  if (misaligned8(capsule_rx_us) || misaligned8(node_ts_us)) {
    c->err = "timestamp buffers must be 8-byte aligned";
    return RPL_RESULT_INVALID_DATA;
  }
  if (rpl_capsule_bytes(ans_type) == 0) {
    c->err = "unknown answer type (capsule formats are 0x82..0x86)";
    return RPL_RESULT_INVALID_DATA;
  }
  if (n_streams == 0) return RPL_RESULT_OK;
  RPL_CUDA(c, cudaSetDevice(c->device), RPL_RESULT_OPERATION_FAIL);
  cudaStream_t st = stream ? static_cast<cudaStream_t>(stream) : c->lane[0].stream;
  rpl::TimingDesc t{timing->sample_duration_us, timing->native_baudrate, timing->linkage_delay_us,
                    timing->native_interface_type};
  rpl::TimestampArgs a{};
  a.capsule_rx_us = reinterpret_cast<const unsigned long long*>(capsule_rx_us);
  a.capsule_status = capsule_status;
  a.capsule_node_offset = capsule_node_offset;
  a.capsule_counts = capsule_counts;
  a.n_streams = n_streams;
  a.stride_capsules = stride_capsules;
  a.node_ts_us = reinterpret_cast<unsigned long long*>(node_ts_us);
  RPL_CUDA(c, rpl::launch_node_timestamps(ans_type, t, a, st), RPL_RESULT_OPERATION_FAIL);
  c->launches++;
  return RPL_RESULT_OK;
}

rpl_result rpl_normal_timestamps_dev(rpl_ctx* c, const rpl_timing* timing, const uint32_t* node_end,
                                     const uint32_t* node_counts, uint32_t n_streams, uint32_t stride_nodes,
                                     uint32_t chunk_bytes, const uint64_t* chunk_rx_us, uint32_t stride_chunks,
                                     uint64_t* node_ts_us, void* stream) {
  if (!c || !timing || !node_end || !node_counts || !chunk_rx_us || !node_ts_us || chunk_bytes == 0)
    return RPL_RESULT_INVALID_DATA;
  if (misaligned8(chunk_rx_us) || misaligned8(node_ts_us)) {
    c->err = "timestamp buffers must be 8-byte aligned";
    return RPL_RESULT_INVALID_DATA;
  }
  if (n_streams == 0) return RPL_RESULT_OK;
  RPL_CUDA(c, cudaSetDevice(c->device), RPL_RESULT_OPERATION_FAIL);
  cudaStream_t st = stream ? static_cast<cudaStream_t>(stream) : c->lane[0].stream;
  rpl::TimingDesc t{timing->sample_duration_us, timing->native_baudrate, timing->linkage_delay_us,
                    timing->native_interface_type};
  rpl::NormalTimestampArgs a{};
  a.node_end = node_end;
  a.node_counts = node_counts;
  a.n_streams = n_streams;
  a.stride_nodes = stride_nodes;
  a.chunk_bytes = chunk_bytes;
  a.stride_chunks = stride_chunks;
  a.chunk_rx_us = reinterpret_cast<const unsigned long long*>(chunk_rx_us);
  a.node_ts_us = reinterpret_cast<unsigned long long*>(node_ts_us);
  RPL_CUDA(c, rpl::launch_normal_timestamps(t, a, st), RPL_RESULT_OPERATION_FAIL);
  c->launches++;
  return RPL_RESULT_OK;
}

// ---- synthetic streams ------------------------------------------------------------------------
rpl_result rpl_synth_batch_dev(rpl_ctx* c, uint64_t first_scan_id, uint32_t n_scans, uint32_t n,
                               uint32_t stride, int variant, rpl_node_hq* nodes, uint32_t* counts,
                               void* stream) {
  if (!c || !nodes || n > stride || variant < 0 || variant > 4) return RPL_RESULT_INVALID_DATA;
  RPL_CUDA(c, cudaSetDevice(c->device), RPL_RESULT_OPERATION_FAIL);
  cudaStream_t st = stream ? static_cast<cudaStream_t>(stream) : c->lane[0].stream;
  RPL_CUDA(c, rpl::launch_synth(first_scan_id, n_scans, n, stride, variant,
                                reinterpret_cast<uint2*>(nodes), counts, st),
           RPL_RESULT_OPERATION_FAIL);
  c->launches++;
  return RPL_RESULT_OK;
}

// ---- PointCloud2 path ----------------------------------------------------------------------------
rpl_result rpl_cloud_batch_dev(rpl_ctx* c, const rpl_node_hq* nodes, const uint32_t* counts,
                               uint32_t n_scans, uint32_t stride, const rpl_cloud_params* params,
                               float* xyzi, uint32_t* point_counts, void* stream) {
  if (!c || !nodes || !counts || !params || !xyzi || !point_counts) return RPL_RESULT_INVALID_DATA;
  if (n_scans == 0) return RPL_RESULT_OK;
  if (n_scans > c->max_scans || params->sor_k > 32) {
    c->err = "n_scans exceeds max_scans or sor_k > 32";
    return RPL_RESULT_INVALID_DATA;
  }
  if (params->voxel_size != 0.0f && !(params->voxel_size >= 1e-6f && params->range_max < 1000.0f)) {
    c->err = "voxel grid: voxel_size must be >= 1e-6 m and range_max < 1000 m (cell indices must fit 31 bits)";
    return RPL_RESULT_INVALID_DATA;
  }
  RPL_CUDA(c, cudaSetDevice(c->device), RPL_RESULT_OPERATION_FAIL);
  cudaStream_t st = stream ? static_cast<cudaStream_t>(stream) : c->lane[0].stream;
  rpl::ScanBatchArgs a{};
  a.nodes = reinterpret_cast<const uint2*>(nodes);
  a.counts = counts;
  a.n_scans = n_scans;
  a.stride = stride;
  a.beam_counts = point_counts;  // points kept per scan
  a.fallback_list = c->lane[0].fallback_list;
  a.fallback_count = c->lane[0].fallback_count;
  a.is_new_protocol = params->is_new_protocol;
  a.xyzi = reinterpret_cast<float4*>(xyzi);
  a.trig = c->lane[0].cws.trig;
  a.angle = c->lane[0].cws.angle;
  a.range_min = params->range_min;
  a.range_max = params->range_max;
  a.intensity_min = params->intensity_min;
  // Revolutions of at most 4096 nodes: the whole chain (window, xyz, SOR, voxel grid) in one kernel, in shared
  // memory (scan_small.cu); the separate in-place post passes then only see the duplicate-key scans that kernel
  // handed to the general kernel.  Larger revolutions: steps 1-3 inside the scan kernels, steps 4-5 as post passes.
  PostParams pp;
  pp.sor_k = params->sor_k;
  pp.sor_alpha = params->sor_alpha;
  pp.voxel = params->voxel_size;
  bool fused = false;
  const uint32_t flags = (params->flags & RPL_CLOUD_NO_FUSED) ? RPL_FLAG_NO_SMALL : 0u;
  rpl_result r = enqueue_args(c, c->lane[0], a, flags, st, &pp, &fused);
  if (r != RPL_RESULT_OK) return r;
  if (params->sor_k > 0 || params->voxel_size > 0.0f) {
    int launched = 0;
    RPL_CUDA(c, rpl::launch_cloud_post(a.xyzi, point_counts, n_scans, stride, params->sor_k, params->sor_alpha,
                                       params->voxel_size, c->lane[0].cws, fused ? a.fallback_list : nullptr,
                                       fused ? a.fallback_count : nullptr, st, &launched),
             RPL_RESULT_OPERATION_FAIL);
    c->launches += launched;
  }
  return RPL_RESULT_OK;
}

rpl_result rpl_cloud_batch(rpl_ctx* c, const rpl_node_hq* nodes, const uint32_t* counts,
                           uint32_t n_scans, uint32_t stride, const rpl_cloud_params* params,
                           float* xyzi, uint32_t* point_counts) {
  if (!c || !nodes || !counts || !params || !xyzi || !point_counts) return RPL_RESULT_INVALID_DATA;
  if (n_scans == 0) return RPL_RESULT_OK;
  if (n_scans > c->max_scans) return RPL_RESULT_INVALID_DATA;
  RPL_CUDA(c, cudaSetDevice(c->device), RPL_RESULT_OPERATION_FAIL);
  Lane& l = c->lane[0];
  rpl_result r = ensure_staging(c, l, n_scans, (size_t)n_scans * stride, true);
  if (r != RPL_RESULT_OK) return r;
  const size_t cnt = (size_t)n_scans * stride;
  RPL_CUDA(c, cudaMemcpyAsync(l.d_nodes, nodes, cnt * sizeof(rpl_node_hq), cudaMemcpyHostToDevice, l.stream),
           RPL_RESULT_OPERATION_FAIL);
  RPL_CUDA(c, cudaMemcpyAsync(l.d_counts, counts, n_scans * sizeof(uint32_t), cudaMemcpyHostToDevice, l.stream),
           RPL_RESULT_OPERATION_FAIL);
  r = rpl_cloud_batch_dev(c, reinterpret_cast<rpl_node_hq*>(l.d_nodes), l.d_counts, n_scans, stride, params,
                          l.d_xyzi, l.d_pcount, l.stream);
  if (r != RPL_RESULT_OK) return r;
  RPL_CUDA(c, cudaMemcpyAsync(xyzi, l.d_xyzi, cnt * 4 * sizeof(float), cudaMemcpyDeviceToHost, l.stream),
           RPL_RESULT_OPERATION_FAIL);
  RPL_CUDA(c, cudaMemcpyAsync(point_counts, l.d_pcount, n_scans * sizeof(uint32_t), cudaMemcpyDeviceToHost, l.stream),
           RPL_RESULT_OPERATION_FAIL);
  RPL_CUDA(c, cudaStreamSynchronize(l.stream), RPL_RESULT_OPERATION_FAIL);
  return RPL_RESULT_OK;
}

rpl_result rpl_cloud_fuse_dev(rpl_ctx* c, const float* xyzi, const uint32_t* point_counts,
                              uint32_t n_scans, uint32_t stride, float* fused, uint32_t* offsets,
                              uint32_t* total, void* stream) {
  if (!c || !xyzi || !point_counts || !fused || !offsets || !total) return RPL_RESULT_INVALID_DATA;
  RPL_CUDA(c, cudaSetDevice(c->device), RPL_RESULT_OPERATION_FAIL);
  cudaStream_t st = stream ? static_cast<cudaStream_t>(stream) : c->lane[0].stream;
  int launched = 0;
  RPL_CUDA(c, rpl::launch_cloud_fuse(reinterpret_cast<const float4*>(xyzi), point_counts, n_scans, stride,
                                     reinterpret_cast<float4*>(fused), 0xFFFFFFFFu, offsets, total, st, &launched),
           RPL_RESULT_OPERATION_FAIL);
  c->launches += launched;
  return RPL_RESULT_OK;
}

// ---- peer memory: fuse + all-gather in one kernel (SURVEY.md 8(e)) ---------------------------------
size_t rpl_peer_gather_bytes(uint32_t world, uint32_t slot_points) {
  return (size_t)rpl::kPeerHeaderBytes + (size_t)world * slot_points * 16;
}

rpl_result rpl_peer_alloc(rpl_ctx* c, size_t bytes, void** dev_ptr, uint8_t* handle_out) {
  if (!c || !dev_ptr || !handle_out || bytes == 0) return RPL_RESULT_INVALID_DATA;
  static_assert(sizeof(cudaIpcMemHandle_t) == RPL_IPC_HANDLE_BYTES, "IPC handle size");
  RPL_CUDA(c, cudaSetDevice(c->device), RPL_RESULT_OPERATION_FAIL);
  void* p = nullptr;
  RPL_CUDA(c, cudaMalloc(&p, bytes), RPL_RESULT_INSUFFICIENT_MEMORY);
  cudaIpcMemHandle_t h;
  if (!cuda_ok(c, cudaMemset(p, 0, bytes), "cudaMemset") || !cuda_ok(c, cudaIpcGetMemHandle(&h, p), "cudaIpcGetMemHandle")) {
    cudaFree(p);
    return RPL_RESULT_OPERATION_FAIL;
  }
  std::memcpy(handle_out, &h, sizeof(h));
  *dev_ptr = p;
  return RPL_RESULT_OK;
}

rpl_result rpl_peer_open(rpl_ctx* c, const uint8_t* handle, void** peer_ptr) {
  if (!c || !handle || !peer_ptr) return RPL_RESULT_INVALID_DATA;
  RPL_CUDA(c, cudaSetDevice(c->device), RPL_RESULT_OPERATION_FAIL);
  cudaIpcMemHandle_t h;
  std::memcpy(&h, handle, sizeof(h));
  RPL_CUDA(c, cudaIpcOpenMemHandle(peer_ptr, h, cudaIpcMemLazyEnablePeerAccess), RPL_RESULT_OPERATION_FAIL);
  return RPL_RESULT_OK;
}

rpl_result rpl_peer_close(rpl_ctx* c, void* peer_ptr) {
  if (!c || !peer_ptr) return RPL_RESULT_INVALID_DATA;
  RPL_CUDA(c, cudaSetDevice(c->device), RPL_RESULT_OPERATION_FAIL);
  RPL_CUDA(c, cudaIpcCloseMemHandle(peer_ptr), RPL_RESULT_OPERATION_FAIL);
  return RPL_RESULT_OK;
}

rpl_result rpl_peer_free(rpl_ctx* c, void* dev_ptr) {
  if (!c || !dev_ptr) return RPL_RESULT_INVALID_DATA;
  RPL_CUDA(c, cudaSetDevice(c->device), RPL_RESULT_OPERATION_FAIL);
  RPL_CUDA(c, cudaFree(dev_ptr), RPL_RESULT_OPERATION_FAIL);
  return RPL_RESULT_OK;
}

rpl_result rpl_cloud_fuse_push_dev(rpl_ctx* c, const float* xyzi, const uint32_t* point_counts, uint32_t n_scans,
                                   uint32_t stride, void* const* peer_bases, uint32_t world, uint32_t rank,
                                   uint32_t slot_points, uint32_t* offsets, uint32_t* total, void* stream) {
  if (!c || !xyzi || !point_counts || !peer_bases || !offsets || !total) return RPL_RESULT_INVALID_DATA;
  if (world == 0 || world > rpl::kMaxPeers || rank >= world) {
    c->err = "world must be in [1, 16] and rank < world";
    return RPL_RESULT_INVALID_DATA;
  }
  rpl::PeerBases peers{};
  for (uint32_t p = 0; p < world; ++p) {
    if (!peer_bases[p] || (reinterpret_cast<uintptr_t>(peer_bases[p]) & 15u)) {
      c->err = "peer buffers must be non-null and 16-byte aligned";
      return RPL_RESULT_INVALID_DATA;
    }
    peers.base[p] = static_cast<unsigned char*>(peer_bases[p]);
  }
  RPL_CUDA(c, cudaSetDevice(c->device), RPL_RESULT_OPERATION_FAIL);
  cudaStream_t st = stream ? static_cast<cudaStream_t>(stream) : c->lane[0].stream;
  int launched = 0;
  RPL_CUDA(c, rpl::launch_cloud_fuse_push(reinterpret_cast<const float4*>(xyzi), point_counts, n_scans, stride, peers,
                                          world, rank, slot_points, offsets, total, st, &launched),
           RPL_RESULT_OPERATION_FAIL);
  c->launches += launched;
  return RPL_RESULT_OK;
}

}  // extern "C"
