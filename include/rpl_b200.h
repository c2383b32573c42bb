/* include/rpl_b200.h -- C-ABI of librplidar_b200.so (the drop-in boundary).
 *
 * B200-native (sm_100a) replacement for the per-scan point-processing hot path of
 * frozenreboot/rplidar_ros2_driver.  Every entry point is extern "C", POD-only, caller owns
 * all memory, nothing throws across the boundary, and results are sl_result-style uint32_t
 * (reference src/sdk/include/sl_types.h:70-81).  There is NO CPU fallback: without a CUDA
 * device rpl_ctx_create fails and nothing else can be called.
 *
 * What each entry point replaces in the reference:
 *
 *   rpl_ascend_scan          sl::ILidarDriver::ascendScanData(node*, count)
 *                              src/sdk/include/sl_lidar_driver.h:477
 *                              (body src/sdk/src/sl_lidar_driver.cpp:128-184, entry :957-960)
 *   rpl_laserscan            the compute body of RPlidarNode::publish_scan
 *                              src/rplidar_node.cpp:581-677 (filter+unpack :581-600, sort
 *                              :605-607, Mode A :630-660, Mode B :661-677)
 *   rpl_scan                 both, fused: RealLidarDriver::grab_scan_data's "ascend if the
 *                              profile asks" (src/lidar_driver_wrapper.cpp:328-329) followed by
 *                              publish_scan -- one host<->device round trip per scan
 *   rpl_*_batch              the same per scan over [n_scans][stride] buffers (the reference
 *                              has no batched form: one scan thread per node,
 *                              src/rplidar_node.cpp:220)
 *   rpl_*_batch_dev          the batched forms on buffers already resident in HBM
 *   rpl_cloud_batch[_dev]    north-star extensions with no reference counterpart (polar->xyz
 *                              PointCloud2 packing, range/intensity window, statistical
 *                              outlier removal, voxel grid); defined by oracle/cloud_oracle.cpp
 *   rpl_synth_batch_dev      synthetic scan streams of SURVEY.md 8(d) generated in HBM
 *
 * and, either side of that path (SURVEY.md 8(f)):
 *
 *   rpl_decode_*             the SDK's sample-data unpackers, all six measurement answer types
 *                              src/sdk/src/dataunpacker/unpacker/handler_{capsules,normalnode,hqnode}.cpp
 *   rpl_node_timestamps_dev  the timestamp the unpackers attach to every node (_getSampleDelayOffsetIn*Mode)
 *   rpl_assemble_scans_dev   ScanDataHolder::pushScanNodeData / rewindCurrentScanData
 *                              src/sdk/src/sl_lidar_driver.cpp:272-315
 *   rpl_*_cdr_batch_dev      the serialised form of the message scan_pub_->publish hands to the RMW layer
 *                              src/rplidar_node.cpp:679
 *   rpl_cloud_fuse_push_dev  (with rpl_peer_*) the fused cloud's all-gather across GPUs, in the pack kernel
 *
 * Buffer contract of the *_dev entry points: every count array entry must be <= its stride (counts are
 * read on the device and not clamped), device pointers must belong to the context's device, and work is
 * ordered on the stream passed in (NULL = the context's own stream).  The context's own stream is a non-blocking
 * stream: it does not wait for work the caller has in flight on other streams (the legacy default stream included).
 * A caller that fills its device buffers on a stream of its own either passes that stream, or synchronises before the
 * call and calls rpl_ctx_synchronize before it reads the results.
 *
 * Tie rule.  The reference sorts with std::sort (unstable); on equal angle_z_q14 its order
 * is whatever libstdc++'s introsort produces.  This library defines the order: equal keys
 * keep buffer order (stable).  On tie-free scans results are bit-identical to the reference.
 *
 * Threading (reference: one scan thread holding driver_mutex_, src/rplidar_node.cpp:420-439):
 * a context is single-threaded; use one context per thread.  No global state.
 */
#ifndef RPL_B200_H_
#define RPL_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RPL_ABI_VERSION 1u

typedef uint32_t rpl_result;
/* reference src/sdk/include/sl_types.h:72-81 */
#define RPL_RESULT_OK 0u
#define RPL_RESULT_FAIL_BIT 0x80000000u
#define RPL_RESULT_INVALID_DATA 0x80008000u
#define RPL_RESULT_OPERATION_FAIL 0x80008001u
#define RPL_RESULT_OPERATION_TIMEOUT 0x80008002u
#define RPL_RESULT_OPERATION_NOT_SUPPORT 0x80008004u
#define RPL_RESULT_INSUFFICIENT_MEMORY 0x80008006u
#define RPL_IS_OK(x) (((x) & RPL_RESULT_FAIL_BIT) == 0u)

/* reference src/sdk/include/sl_lidar_cmd.h:272-278 (sizeof 8, offsets 0/2/6/7) */
typedef struct __attribute__((packed)) rpl_node_hq {
  uint16_t angle_z_q14; /* 90 deg / 16384 per unit; 65536 = 360 deg */
  uint32_t dist_mm_q2;  /* quarter millimetres; 0 = no measurement   */
  uint8_t quality;
  uint8_t flag;         /* bit0 = scan start sync (sl_lidar_cmd.h:178) */
} rpl_node_hq;

typedef struct rpl_scan_params {
  uint8_t is_new_protocol; /* intensity = quality (1) or quality>>2 (0); rplidar_node.cpp:575-590 */
  uint8_t scan_processing; /* 1 = Mode A resample, 0 = Mode B raw map; rplidar_node.cpp:630 */
  uint8_t inverted;        /* rplidar_node.cpp:644,673 */
  uint8_t apply_ascend;    /* angle_compensate; lidar_driver_wrapper.cpp:107,328 */
  uint32_t flags;          /* RPL_FLAG_* */
} rpl_scan_params;

#define RPL_FLAG_FORCE_GENERAL 1u /* route every scan through the general (radix-sort) kernel */
#define RPL_FLAG_NO_TMA 2u        /* use the register-streamed fast kernel (scan_fast.cu) even when the
                                     TMA-ring kernel (scan_tma.cu) applies; for A/B measurements */
#define RPL_FLAG_NO_SMALL 4u      /* do not use the shared-memory-resident kernels (scan_small.cu) for
                                     revolutions of at most 8192 nodes; for A/B measurements */

/* per-scan path report (optional output) */
#define RPL_PATH_FAST 0u    /* tie-free scan: bitmap-rank kernel */
#define RPL_PATH_GENERAL 1u /* duplicate keys (or forced): stable radix-sort kernel */

typedef struct rpl_cloud_params {
  float range_min;     /* keep range_min <= r <= range_max */
  float range_max;
  float intensity_min; /* keep intensity >= intensity_min */
  float voxel_size;    /* metres; 0 disables the voxel grid */
  uint32_t sor_k;      /* 0 disables statistical outlier removal; <= 32 */
  float sor_alpha;
  uint8_t is_new_protocol;
  uint8_t flags;       /* RPL_CLOUD_* */
  uint8_t pad[2];
} rpl_cloud_params;
#define RPL_CLOUD_NO_FUSED 1u /* run SOR / voxel grid as separate passes even where the shared-memory kernel
                                 could fuse them (A/B measurements, second implementation for the tests) */

typedef struct rpl_ctx rpl_ctx;

/* ---- context -------------------------------------------------------------------------- */
uint32_t rpl_abi_version(void);
/* device: CUDA ordinal.  max_nodes: largest scan (nodes) the context will see; max_scans:
 * largest batch for the HOST-buffer entry points (device staging is sized from these). */
rpl_result rpl_ctx_create(int device, uint32_t max_nodes, uint32_t max_scans, rpl_ctx** out);
void rpl_ctx_destroy(rpl_ctx* ctx);
const char* rpl_last_error(const rpl_ctx* ctx);
/* Block until everything queued by this context has finished. */
rpl_result rpl_ctx_synchronize(rpl_ctx* ctx);
/* Pinned host memory for the host-buffer entry points (optional; pageable works, slower). */
rpl_result rpl_host_alloc(size_t bytes, void** out);
void rpl_host_free(void* p);
/* Number of kernels this context has launched so far (bench.py's gpu_launches). */
uint64_t rpl_ctx_launch_count(const rpl_ctx* ctx);
/* Kernel timing for roofline reports: when enabled, every scan-kernel launch is bracketed by
 * CUDA events on the stream it is launched on.  rpl_ctx_profile_read synchronises, returns
 * the summed durations (ms) and launch counts since the last read, and clears them. */
rpl_result rpl_ctx_profile(rpl_ctx* ctx, int enable);
rpl_result rpl_ctx_profile_read(rpl_ctx* ctx, double* fast_ms, uint32_t* fast_launches,
                                double* general_ms, uint32_t* general_launches);

/* ---- single scan, host buffers (the reference-shaped calls) --------------------------- */
/* In place, like ascendScanData.  RPL_RESULT_OPERATION_FAIL when no node is measured
 * (buffer untouched) or count == 0. */
rpl_result rpl_ascend_scan(rpl_ctx* ctx, rpl_node_hq* nodes, size_t count);
/* ranges / intensities: `count` floats each; the first *beam_count are written.
 * *beam_count == 0 means the reference would not publish (no measured node). */
rpl_result rpl_laserscan(rpl_ctx* ctx, const rpl_node_hq* nodes, size_t count,
                         const rpl_scan_params* params, float* ranges, float* intensities,
                         uint32_t* beam_count, float* angle_increment);
/* Fused grab_scan_data glue + publish_scan: nodes are ascended in place when
 * params->apply_ascend (its sl_result goes to *ascend_status, may be NULL), then converted. */
rpl_result rpl_scan(rpl_ctx* ctx, rpl_node_hq* nodes, size_t count, const rpl_scan_params* params,
                    float* ranges, float* intensities, uint32_t* beam_count,
                    float* angle_increment, rpl_result* ascend_status);

/* ---- batches, host buffers ------------------------------------------------------------ */
/* nodes: [n_scans][stride]; counts[s] <= stride nodes are live in scan s.
 * nodes_out (may be NULL, may equal nodes): ascended node buffers, same layout.
 * ranges/intensities: [n_scans][stride] floats; beam_counts/angle_increment/status/path:
 * [n_scans] (each may be NULL).  status[s] = ascendScanData's sl_result when apply_ascend,
 * else RPL_RESULT_OK. */
rpl_result rpl_scan_batch(rpl_ctx* ctx, const rpl_node_hq* nodes, const uint32_t* counts,
                          uint32_t n_scans, uint32_t stride, const rpl_scan_params* params,
                          rpl_node_hq* nodes_out, float* ranges, float* intensities,
                          uint32_t* beam_counts, float* angle_increment, uint32_t* status,
                          uint32_t* path);
rpl_result rpl_ascend_scan_batch(rpl_ctx* ctx, rpl_node_hq* nodes, const uint32_t* counts,
                                 uint32_t n_scans, uint32_t stride, uint32_t* status);
rpl_result rpl_laserscan_batch(rpl_ctx* ctx, const rpl_node_hq* nodes, const uint32_t* counts,
                               uint32_t n_scans, uint32_t stride, const rpl_scan_params* params,
                               float* ranges, float* intensities, uint32_t* beam_counts,
                               float* angle_increment);

/* ---- batches, device buffers (asynchronous on `stream`, a cudaStream_t; NULL = the
 * context's own stream).  Same layout as above; nodes_out must not alias nodes. ---------- */
rpl_result rpl_scan_batch_dev(rpl_ctx* ctx, const rpl_node_hq* nodes, const uint32_t* counts,
                              uint32_t n_scans, uint32_t stride, const rpl_scan_params* params,
                              rpl_node_hq* nodes_out, float* ranges, float* intensities,
                              uint32_t* beam_counts, float* angle_increment, uint32_t* status,
                              uint32_t* path, void* stream);

/* ---- PointCloud2 path (extensions; oracle/cloud_oracle.cpp is the definition) --------- */
/* xyzi: [n_scans][stride][4] floats (x, y, z, intensity = PointCloud2 point_step 16);
 * point_counts[s] = points written for scan s. */
rpl_result rpl_cloud_batch_dev(rpl_ctx* ctx, const rpl_node_hq* nodes, const uint32_t* counts,
                               uint32_t n_scans, uint32_t stride, const rpl_cloud_params* params,
                               float* xyzi, uint32_t* point_counts, void* stream);
rpl_result rpl_cloud_batch(rpl_ctx* ctx, const rpl_node_hq* nodes, const uint32_t* counts,
                           uint32_t n_scans, uint32_t stride, const rpl_cloud_params* params,
                           float* xyzi, uint32_t* point_counts);
/* Packs the per-scan clouds of a batch into one dense cloud (the per-GPU "fused cloud" that
 * is all-gathered across ranks): fused[0..*total) points, 16 B each; offsets[s] = first point
 * of scan s.  fused must hold n_scans*stride points.  An empty batch (n_scans == 0) sets *total = 0, as do the push
 * and the exchange below for the count they publish. */
rpl_result rpl_cloud_fuse_dev(rpl_ctx* ctx, const float* xyzi, const uint32_t* point_counts,
                              uint32_t n_scans, uint32_t stride, float* fused, uint32_t* offsets,
                              uint32_t* total, void* stream);

/* ---- fuse + all-gather through peer memory (SURVEY.md 8(e): one process per GPU, NVLink P2P) ---- */
/* rpl_cloud_fuse_dev + one NCCL all-gather writes the dense cloud locally and lets the collective read
 * it again.  rpl_cloud_fuse_push_dev does both in ONE kernel: every point is stored straight into slot
 * `rank` of every rank's gather buffer.  The buffers are allocated with rpl_peer_alloc (cudaMalloc +
 * cudaIpcGetMemHandle), the 64-byte handles are exchanged by the host (torch.distributed in this repo) and
 * opened with rpl_peer_open (cudaIpcOpenMemHandle: NVLink peer mapping).  Gather buffer layout:
 * [256-byte header: uint32 point count of every rank][world][slot_points][16 B]; size
 * rpl_peer_gather_bytes(world, slot_points).  peer_bases: HOST array [world] of device pointers, entry
 * `rank` = this rank's own buffer.  Completion: the stores are visible on the peers once this rank's
 * kernel has finished; a consumer needs one barrier over all ranks after the call (any tiny collective on
 * the same stream) and must not let the next push overwrite a buffer that is still being read
 * (rplidar_ros2_driver_b200/multi_gpu.py::PeerCloudGather alternates two buffers). */
#define RPL_IPC_HANDLE_BYTES 64u
#define RPL_MAX_PEERS 16u
size_t rpl_peer_gather_bytes(uint32_t world, uint32_t slot_points);
rpl_result rpl_peer_alloc(rpl_ctx* ctx, size_t bytes, void** dev_ptr, uint8_t* handle_out /* [64] */);
rpl_result rpl_peer_open(rpl_ctx* ctx, const uint8_t* handle /* [64] */, void** peer_ptr);
rpl_result rpl_peer_close(rpl_ctx* ctx, void* peer_ptr);
rpl_result rpl_peer_free(rpl_ctx* ctx, void* dev_ptr);
rpl_result rpl_cloud_fuse_push_dev(rpl_ctx* ctx, const float* xyzi, const uint32_t* point_counts, uint32_t n_scans,
                                   uint32_t stride, void* const* peer_bases, uint32_t world, uint32_t rank,
                                   uint32_t slot_points, uint32_t* offsets, uint32_t* total, void* stream);

/* ---- the exchange as a host-side C++ object (SURVEY.md 8(e): one process per GPU, ONE all-gather of the fused
 * cloud per step over NVLink, overlapped with the next batch's kernels) ------------------------------------
 * The reference has no analogue (it publishes one scan: src/rplidar_node.cpp:679); parity = every rank ends up
 * with the concatenation, in rank order, of what the ranks produce on their own.  NCCL is loaded at run time
 * (dlopen libnccl.so.2); the embedding process only carries the 128-byte unique id from rank 0 to the others.
 * rpl_exchange_create is collective (every rank, same id / world / slot_points); it creates the communicator
 * (ncclCommInitRank), a high-priority exchange stream, two gather buffers of `world` slots
 * [16-byte header: uint32 point count][slot_points x 16 B] and -- unless RPL_EXCHANGE_NO_PEER_MAP -- maps every
 * peer's buffers (CUDA IPC handles all-gathered through the communicator).
 * rpl_exchange_allgather packs the per-scan clouds of rpl_cloud_batch_dev (xyzi [n_scans][stride][4],
 * point_counts) into this rank's slot on `stream` and starts the transfer on the exchange stream:
 *   RPL_EXCHANGE_NCCL  one in-place ncclAllGather of the slot;
 *   RPL_EXCHANGE_COPY  world-1 peer-to-peer copies of the slot by the copy engines (no SM), then a 4-byte
 *                      all-reduce as the barrier.
 * `stream` is NOT made to wait for the transfer: the caller's next batch overlaps it.  *buffer_index (0/1) names
 * the buffer this step fills; a consumer calls rpl_exchange_wait(index, its stream) before reading the slots
 * (rpl_exchange_slot) and rpl_exchange_release(index, its stream) after its last read -- the exchange that reuses
 * the buffer two steps later waits for that.  A slot whose count exceeds slot_points overflowed (points dropped). */
#define RPL_EXCHANGE_ID_BYTES 128u
#define RPL_EXCHANGE_NCCL 0u
#define RPL_EXCHANGE_COPY 1u
#define RPL_EXCHANGE_NO_PEER_MAP 1u /* create flag: NCCL mode only, no CUDA IPC mappings */
typedef struct rpl_exchange rpl_exchange;
rpl_result rpl_exchange_unique_id(uint8_t* id_out /* [128], call on rank 0 */);
rpl_result rpl_exchange_create(rpl_ctx* ctx, const uint8_t* id /* [128]; may be NULL when world == 1 */, uint32_t world,
                               uint32_t rank, uint32_t slot_points, uint32_t flags, rpl_exchange** out);
void rpl_exchange_destroy(rpl_exchange* ex); /* collective when world > 1 */
rpl_result rpl_exchange_allgather(rpl_exchange* ex, const float* xyzi, const uint32_t* point_counts, uint32_t n_scans,
                                  uint32_t stride, uint32_t mode, void* stream, uint32_t* buffer_index);
rpl_result rpl_exchange_wait(rpl_exchange* ex, uint32_t buffer_index, void* stream);
rpl_result rpl_exchange_release(rpl_exchange* ex, uint32_t buffer_index, void* stream);
rpl_result rpl_exchange_slot(rpl_exchange* ex, uint32_t buffer_index, uint32_t rank, const float** points,
                             const uint32_t** count);
rpl_result rpl_exchange_synchronize(rpl_exchange* ex);

/* ---- dense-capsule decode (SURVEY.md 8(f) rank 1: the step before the hot path) ------- */
/* Replaces UnpackerHandler_DenseCapsuleNode (reference
 * src/sdk/src/dataunpacker/unpacker/handler_capsules.cpp:639-791) for FRAMED capsules: answer
 * type 0x85, 84 bytes each (src/sdk/include/sl_lidar_cmd.h:223-234), one capsule per protocol
 * message.  capsules: [n_streams][stride_capsules][84]; nodes_out: [n_streams][stride_capsules*40]
 * HQ nodes in the order the reference's listener receives them; node_counts[s] = nodes decoded.
 * capsule_status (nullable): RPL_CAPSULE_* bits per capsule; capsule_node_offset (nullable):
 * nodes decoded before each capsule (so scan-reset / error events keep their place in the node
 * stream).  sync_state_in/out (nullable): the reference's function-static lastNodeSyncBit
 * entering / leaving every stream (0 = fresh process).  sample_duration_us:
 * SlamtecLidarTimingDesc::sample_duration_uS (sets the angular-jump discard threshold). */
#define RPL_DENSE_CAPSULE_BYTES 84u
#define RPL_CAPSULE_OK 1u                /* sync nibbles and checksum fine */
#define RPL_CAPSULE_SYNC 2u              /* first capsule of a revolution: scan reset requested */
#define RPL_CAPSULE_EMIT 4u              /* released the previous capsule's 40 nodes */
#define RPL_CAPSULE_DISCARD 8u           /* angular jump above the 100 Hz bound: nothing released */
#define RPL_CAPSULE_CHECKSUM_ERR 16u     /* ERR_EVENT_ON_EXP_CHECKSUM_ERR */
#define RPL_CAPSULE_ENCODER_RESET_ERR 32u /* ERR_EVENT_ON_EXP_ENCODER_RESET */
#define RPL_CAPSULE_BAD_FRAME 64u        /* wrong sync nibbles: outside the framed contract */
rpl_result rpl_decode_dense_batch_dev(rpl_ctx* ctx, const uint8_t* capsules, const uint32_t* capsule_counts,
                                      uint32_t n_streams, uint32_t stride_capsules, uint32_t sample_duration_us,
                                      const uint32_t* sync_state_in, rpl_node_hq* nodes_out,
                                      uint32_t* node_counts, uint32_t* capsule_status,
                                      uint32_t* capsule_node_offset, uint32_t* sync_state_out, void* stream);
/* The same, and the decoder also lists where the revolutions start: scan_starts [n_streams][starts_stride] = node
 * offsets of the scan-start nodes of every stream (in no particular order), scan_start_counts[s] = how many there are
 * (more than starts_stride: the list is incomplete and must not be used).  rpl_assemble_scan_views_starts_dev takes
 * the list instead of reading every decoded node again. */
rpl_result rpl_decode_dense_batch_starts_dev(rpl_ctx* ctx, const uint8_t* capsules, const uint32_t* capsule_counts,
                                             uint32_t n_streams, uint32_t stride_capsules, uint32_t sample_duration_us,
                                             const uint32_t* sync_state_in, rpl_node_hq* nodes_out,
                                             uint32_t* node_counts, uint32_t* capsule_status,
                                             uint32_t* capsule_node_offset, uint32_t* sync_state_out,
                                             uint32_t* scan_starts, uint32_t starts_stride, uint32_t* scan_start_counts,
                                             void* stream);
/* One stream, host buffers.  nodes_out must hold 40 * n_capsules nodes. */
rpl_result rpl_decode_dense(rpl_ctx* ctx, const uint8_t* capsules, uint32_t n_capsules,
                            uint32_t sample_duration_us, uint32_t* sync_state, rpl_node_hq* nodes_out,
                            uint32_t* node_count, uint32_t* capsule_status, uint32_t* capsule_node_offset);

/* ---- the other measurement answer formats (SURVEY.md 8(f) rank 1) ----------------------- */
/* ans_type is the SDK's answer type (reference src/sdk/include/sl_lidar_cmd.h:144-151):
 *   0x82 express capsules      84 B -> 32 nodes   UnpackerHandler_CapsuleNode           handler_capsules.cpp:109-266
 *   0x83 HQ capsules          781 B -> 96 nodes   UnpackerHandler_HQNode                handler_hqnode.cpp:93-172
 *   0x84 ultra capsules       132 B -> 96 nodes   UnpackerHandler_UltraCapsuleNode      handler_capsules.cpp:324-580
 *   0x85 dense capsules        84 B -> 40 nodes   (same kernel as rpl_decode_dense_batch_dev)
 *   0x86 ultra-dense capsules 170 B -> 64 nodes   UnpackerHandler_UltraDenseCapsuleNode handler_capsules.cpp:852-1047
 * (reference src/sdk/src/dataunpacker/unpacker/).  Framed input as for the dense decoder:
 * capsules [n_streams][stride_capsules][rpl_capsule_bytes(ans_type)], nodes_out
 * [n_streams][stride_capsules * rpl_capsule_nodes(ans_type)].  state_in / state_out (nullable):
 * [n_streams][2] = {scan-start flag of the last node, last distance} -- the decoder state the SDK
 * keeps across capsules for the dense (word 0) and ultra-dense (both) formats; 0 on a fresh decoder.
 * The per-capsule status words are the RPL_CAPSULE_* bits above. */
/* sl::SlamtecLidarTimingDesc (reference src/sdk/include/sl_lidar_driver.h:156-166). */
typedef struct rpl_timing {
  uint32_t sample_duration_us;
  uint32_t native_baudrate;        /* 0 = the per-format default the SDK assumes */
  uint32_t linkage_delay_us;
  uint32_t native_interface_type;  /* sl::LIDARInterfaceType: 0 UART, 1 ETHERNET, 2 USB, 5 CANBUS */
} rpl_timing;
#define RPL_ANS_MEASUREMENT 0x81u
#define RPL_ANS_MEASUREMENT_CAPSULED 0x82u
#define RPL_ANS_MEASUREMENT_HQ 0x83u
#define RPL_ANS_MEASUREMENT_CAPSULED_ULTRA 0x84u
#define RPL_ANS_MEASUREMENT_DENSE_CAPSULED 0x85u
#define RPL_ANS_MEASUREMENT_ULTRA_DENSE_CAPSULED 0x86u
uint32_t rpl_capsule_bytes(uint32_t ans_type); /* 0 for an unknown type */
uint32_t rpl_capsule_nodes(uint32_t ans_type);
rpl_result rpl_decode_capsules_batch_dev(rpl_ctx* ctx, uint32_t ans_type, const uint8_t* capsules,
                                         const uint32_t* capsule_counts, uint32_t n_streams,
                                         uint32_t stride_capsules, uint32_t sample_duration_us,
                                         const uint32_t* state_in, rpl_node_hq* nodes_out, uint32_t* node_counts,
                                         uint32_t* capsule_status, uint32_t* capsule_node_offset,
                                         uint32_t* state_out, void* stream);
/* One stream, host buffers.  state: in/out [2] (nullable).  timing / capsule_rx_us / node_ts_us (nullable
 * together): also return the per-node stamps of rpl_node_timestamps_dev (below) for the receive times
 * capsule_rx_us[n_capsules]; sample_duration_us is then taken from timing. */
rpl_result rpl_decode_capsules(rpl_ctx* ctx, uint32_t ans_type, const uint8_t* capsules, uint32_t n_capsules,
                               uint32_t sample_duration_us, uint32_t* state, rpl_node_hq* nodes_out,
                               uint32_t* node_count, uint32_t* capsule_status, uint32_t* capsule_node_offset,
                               const rpl_timing* timing, const uint64_t* capsule_rx_us, uint64_t* node_ts_us);
/* Byte-level framing of RAW capsule streams (0x82, 0x84, 0x85, 0x86) with the SDK's resynchronisation: the hunt for
 * the two sync nibbles of UnpackerHandler_{Capsule,UltraCapsule,DenseCapsule,UltraDenseCapsule}Node::onData
 * (reference src/sdk/src/dataunpacker/unpacker/handler_capsules.cpp:107-135, 324-353, 639-668, 852-880).
 * bytes [n_streams][stride_bytes] -> capsules_out [n_streams][stride_capsules][rpl_capsule_bytes(ans_type)], the
 * input of the decoders above; every stretch of bytes the SDK would skip becomes ONE all-zero capsule (decoded as
 * RPL_CAPSULE_BAD_FRAME: the decoders then forget the previous capsule, as the SDK does).  capsule_counts_out[s] >
 * stride_capsules means the output overflowed (a stream of B bytes needs at most 2 * (B / frame size) + 2 slots);
 * bytes_left_out (nullable): bytes of an unfinished frame at the end of the stream -- prepend them to the next
 * piece of the stream. */
rpl_result rpl_frame_capsules_dev(rpl_ctx* ctx, uint32_t ans_type, const uint8_t* bytes, const uint32_t* byte_counts,
                                  uint32_t n_streams, uint32_t stride_bytes, uint8_t* capsules_out,
                                  uint32_t stride_capsules, uint32_t* capsule_counts_out, uint32_t* bytes_left_out,
                                  void* stream);
/* 0x81 standard measurement nodes (5 bytes each) from RAW byte streams, with the byte-level
 * resynchronisation of UnpackerHandler_NormalNode::onData (handler_normalnode.cpp:88-141): exact on
 * misframed / corrupted streams.  bytes [n_streams][stride_bytes]; nodes_out
 * [n_streams][stride_bytes / 5]; fsm_state_out (nullable): bytes still buffered at the end; node_end
 * (nullable, [n_streams][stride_bytes / 5]): index of the last byte of each decoded record (what
 * rpl_normal_timestamps_dev needs to find the piece of the stream a record arrived in). */
rpl_result rpl_decode_normal_batch_dev(rpl_ctx* ctx, const uint8_t* bytes, const uint32_t* byte_counts,
                                       uint32_t n_streams, uint32_t stride_bytes, rpl_node_hq* nodes_out,
                                       uint32_t* node_counts, uint32_t* fsm_state_out, uint32_t* node_end,
                                       void* stream);
rpl_result rpl_decode_normal(rpl_ctx* ctx, const uint8_t* bytes, uint32_t n_bytes, rpl_node_hq* nodes_out,
                             uint32_t* node_count);

/* ---- scan assembly (SURVEY.md 8(f) rank 2: node stream -> scans, on the device) -------- */
/* Replaces ScanDataHolder::pushScanNodeData / rewindCurrentScanData (reference
 * src/sdk/src/sl_lidar_driver.cpp:272-315).  nodes: [n_streams][stride_nodes] decoded streams
 * (rpl_decode_dense_batch_dev output).  capsule_status / capsule_node_offset / capsule_counts
 * (nullable together): the decoder's per-capsule report, from which the scan-reset requests are
 * taken (one before every RPL_CAPSULE_SYNC capsule).  max_nodes: holder capacity (8192 in the SDK);
 * scan_stride >= max_nodes.  scans_out: [n_streams][max_scans][scan_stride]; scan_len:
 * [n_streams][max_scans]; scans_per_stream[s] = scans published (only the first max_scans stored).
 * The output is laid out as the input of rpl_scan_batch_dev (n_scans = n_streams * max_scans with
 * scan_len as counts; unused slots must be zeroed by the caller or have length 0).
 * node_ts_us (nullable, [n_streams][stride_nodes]) / scan_begin_ts_us (nullable,
 * [n_streams][max_scans]): every published scan reports the stamp of the scan-start node that opened
 * it (ScanDataHolder::_scan_begin_timestamp_uS, :293,:326-328; what grabScanDataHqWithTimeStamp returns). */
rpl_result rpl_assemble_scans_dev(rpl_ctx* ctx, const rpl_node_hq* nodes, const uint32_t* node_counts,
                                  uint32_t n_streams, uint32_t stride_nodes, const uint32_t* capsule_status,
                                  const uint32_t* capsule_node_offset, const uint32_t* capsule_counts,
                                  uint32_t stride_capsules, uint32_t max_nodes, uint32_t max_scans,
                                  uint32_t scan_stride, rpl_node_hq* scans_out, uint32_t* scan_len,
                                  uint32_t* scans_per_stream, const uint64_t* node_ts_us,
                                  uint64_t* scan_begin_ts_us, void* stream);

/* The same cut WITHOUT the copy: a published scan is returned as a view {first node, count} into the node buffer
 * itself (first counts from the start of `nodes`, across streams), and rpl_scan_views_dev reads the revolutions
 * where the decoder left them -- the capsule -> LaserScan chain then moves every node through HBM once less in
 * each direction.  views_out / scan_len: [n_streams][max_scans], unused entries are {0, 0}.  The holder's capacity
 * rule (a scan longer than max_nodes keeps overwriting its last entry) is applied IN PLACE: node first+max_nodes-1
 * of such a scan is overwritten with the scan's last node (the nodes behind it are dropped either way), which is
 * why `nodes` is not const here. */
typedef struct rpl_scan_view {
  uint32_t first; /* index of the scan's first node in the whole node buffer */
  uint32_t count;
} rpl_scan_view;
rpl_result rpl_assemble_scan_views_dev(rpl_ctx* ctx, rpl_node_hq* nodes, const uint32_t* node_counts,
                                       uint32_t n_streams, uint32_t stride_nodes, const uint32_t* capsule_status,
                                       const uint32_t* capsule_node_offset, const uint32_t* capsule_counts,
                                       uint32_t stride_capsules, uint32_t max_nodes, uint32_t max_scans,
                                       rpl_scan_view* views_out, uint32_t* scan_len, uint32_t* scans_per_stream,
                                       const uint64_t* node_ts_us, uint64_t* scan_begin_ts_us, void* stream);
/* rpl_assemble_scan_views_dev with the decoder's scan-start list (rpl_decode_dense_batch_starts_dev): a stream whose
 * list is complete is cut without touching its nodes; one whose list overflowed falls back to reading them. */
rpl_result rpl_assemble_scan_views_starts_dev(rpl_ctx* ctx, rpl_node_hq* nodes, const uint32_t* node_counts,
                                              uint32_t n_streams, uint32_t stride_nodes, const uint32_t* capsule_status,
                                              const uint32_t* capsule_node_offset, const uint32_t* capsule_counts,
                                              uint32_t stride_capsules, const uint32_t* scan_starts,
                                              uint32_t starts_stride, const uint32_t* scan_start_counts,
                                              uint32_t max_nodes, uint32_t max_scans, rpl_scan_view* views_out,
                                              uint32_t* scan_len, uint32_t* scans_per_stream, const uint64_t* node_ts_us,
                                              uint64_t* scan_begin_ts_us, void* stream);
/* rpl_scan_batch_dev over views: scan s = views[s].count nodes from nodes[views[s].first]; nodes_total = nodes in
 * the buffer; outputs laid out [n_scans][stride] as before (stride >= every count, stride <= 8192: the views are
 * served by the shared-memory kernels).  `nodes` must be 16-byte aligned.  A view with first + count > nodes_total
 * is reported like a count above the stride: status[s] = RPL_RESULT_INVALID_DATA, beam count 0, nothing else written.
 * nodes_out requires params->apply_ascend (RPL_RESULT_INVALID_DATA otherwise, nothing enqueued): without the ascend
 * the unchanged nodes are the views themselves. */
rpl_result rpl_scan_views_dev(rpl_ctx* ctx, const rpl_node_hq* nodes, uint64_t nodes_total, const rpl_scan_view* views,
                              uint32_t n_scans, uint32_t stride, const rpl_scan_params* params, rpl_node_hq* nodes_out,
                              float* ranges, float* intensities, uint32_t* beam_counts, float* angle_increment,
                              uint32_t* status, uint32_t* path, void* stream);

/* Wire bytes -> LaserScan in ONE host call: framed dense (0x85) capsules in host memory -> H2D -> decode ->
 * scan views -> scan kernel -> D2H, chunked over the two lanes so that copies and kernels overlap.  Per stream this is
 * the reference's whole data path after the protocol codec: UnpackerHandler_DenseCapsuleNode::onData
 * (src/sdk/src/dataunpacker/unpacker/handler_capsules.cpp:639-791) -> ScanDataHolder::pushScanNodeData
 * (src/sdk/src/sl_lidar_driver.cpp:272-315) -> grab_scan_data with ascendScanData (src/lidar_driver_wrapper.cpp:307-342,
 * src/sdk/src/sl_lidar_driver.cpp:128-184) -> publish_scan (src/rplidar_node.cpp:556-680).  2.1 bytes per
 * point cross the host link on the way in instead of the 8 of a decoded node.  capsules: host
 * [n_streams][stride_capsules][84]; outputs: host ranges / intensities [n_streams * max_scans][max_nodes],
 * beam_counts / angle_increment (nullable) [n_streams * max_scans] (slot k of stream s at s * max_scans + k; unused
 * slots have beam count 0), scans_per_stream [n_streams].  max_nodes: even, <= 8192, at most the context's max_nodes
 * (RPL_RESULT_INVALID_DATA otherwise), at least the longest revolution (longer ones are cut by the holder's capacity
 * rule); the context's max_scans must cover
 * max_scans of at least one stream.  Pinned host memory (rpl_host_alloc) keeps the copies asynchronous. */
rpl_result rpl_chain_dense_laserscan(rpl_ctx* ctx, const uint8_t* capsules, const uint32_t* capsule_counts,
                                     uint32_t n_streams, uint32_t stride_capsules, uint32_t sample_duration_us,
                                     const rpl_scan_params* params, uint32_t max_nodes, uint32_t max_scans,
                                     float* ranges, float* intensities, uint32_t* beam_counts, float* angle_increment,
                                     uint32_t* scans_per_stream);

/* ---- LaserScan / PointCloud2 -> wire (SURVEY.md 8(f) rank 3) ---------------------------- */
/* The serialised message the RMW layer would produce from the message the reference publishes
 * (scan_pub_->publish, reference src/rplidar_node.cpp:679): XCDR1 little endian, 4-byte
 * encapsulation header, members in declaration order.  The host publishes the bytes as they are
 * (rclcpp::SerializedMessage, INTEGRATION.md 4c).  The reference tree holds no serialiser (it is in
 * the RMW dependency): the format follows the OMG CDR rules; parity unpinned. */
typedef struct rpl_laserscan_meta { /* sensor_msgs/LaserScan minus frame_id and the arrays */
  int32_t stamp_sec;
  uint32_t stamp_nanosec;
  float angle_min, angle_max, angle_increment, time_increment, scan_time, range_min, range_max;
} rpl_laserscan_meta;
uint32_t rpl_laserscan_cdr_size(uint32_t frame_id_len, uint32_t beam_count);
/* meta: [n_scans] on the device; angle_increment (nullable, device [n_scans]): the scan kernel's
 * output, overrides meta[s].angle_increment; ranges / intensities [n_scans][stride] and beam_counts
 * as rpl_scan_batch_dev wrote them.  cdr_out: [n_scans][cdr_stride] with cdr_stride % 4 == 0 and
 * cdr_stride >= rpl_laserscan_cdr_size(strlen(frame_id), stride); cdr_sizes (nullable): bytes used. */
rpl_result rpl_laserscan_cdr_batch_dev(rpl_ctx* ctx, const rpl_laserscan_meta* meta, const float* angle_increment,
                                       const char* frame_id, const float* ranges, const float* intensities,
                                       const uint32_t* beam_counts, uint32_t n_scans, uint32_t stride,
                                       uint8_t* cdr_out, uint32_t cdr_stride, uint32_t* cdr_sizes, void* stream);
uint32_t rpl_pointcloud2_cdr_size(uint32_t frame_id_len, uint32_t n_points);
/* sensor_msgs/PointCloud2 with fields x, y, z, intensity (float32, point_step 16, height 1, is_dense),
 * the layout laser_geometry produces and rpl_cloud_batch_dev writes.  stamps: device [n_clouds][2]
 * {sec, nanosec}; xyzi [n_clouds][stride][4]; cdr_stride % 16 == 0. */
rpl_result rpl_pointcloud2_cdr_batch_dev(rpl_ctx* ctx, const uint32_t* stamps, const char* frame_id,
                                         const float* xyzi, const uint32_t* point_counts, uint32_t n_clouds,
                                         uint32_t stride, uint8_t* cdr_out, uint32_t cdr_stride,
                                         uint32_t* cdr_sizes, void* stream);

/* ---- per-sample timestamps (SURVEY.md 8(f) rank 4) -------------------------------------- */
/* (rpl_timing is declared with the decoders above.) */
/* The stamp the SDK's unpackers attach to every node: receive time of a capsule minus
 * _getSampleDelayOffsetIn{Legacy,Express,HQ,UltraBoost,Dense,UltraDense}Mode (handler_normalnode.cpp:49-68,
 * handler_capsules.cpp:55-76,272-293,586-607,795-816, handler_hqnode.cpp:53-72).  capsule_rx_us:
 * [n_streams][stride_capsules] receive times; capsule_status / capsule_node_offset: the decoder's report;
 * node_ts_us: [n_streams][stride_capsules * rpl_capsule_nodes(ans_type)], written for released nodes. */
rpl_result rpl_node_timestamps_dev(rpl_ctx* ctx, uint32_t ans_type, const rpl_timing* timing,
                                   const uint64_t* capsule_rx_us, const uint32_t* capsule_status,
                                   const uint32_t* capsule_node_offset, const uint32_t* capsule_counts,
                                   uint32_t n_streams, uint32_t stride_capsules, uint64_t* node_ts_us, void* stream);
/* Standard nodes: the record ending at byte node_end[i] is stamped with the receive time of the
 * chunk_bytes-sized piece of the stream that byte arrived in (chunk_rx_us [n_streams][stride_chunks]). */
rpl_result rpl_normal_timestamps_dev(rpl_ctx* ctx, const rpl_timing* timing, const uint32_t* node_end,
                                     const uint32_t* node_counts, uint32_t n_streams, uint32_t stride_nodes,
                                     uint32_t chunk_bytes, const uint64_t* chunk_rx_us, uint32_t stride_chunks,
                                     uint64_t* node_ts_us, void* stream);

/* ---- synthetic scan streams (SURVEY.md 8(d)) ------------------------------------------ */
/* variant 0: tie-free rotated revolution, 5% unmeasured, quality 188; 1: same, quality
 * U[0,255]; 2: iid U[0,65535] keys (ties); 3: tie-free keys in pseudo-random order; 4: a
 * "room" (16 constant-range arcs of 2..10 m + 2 cm noise; non-trivial 5 cm voxels).
 * Also writes counts[s] = n when counts != NULL. */
rpl_result rpl_synth_batch_dev(rpl_ctx* ctx, uint64_t first_scan_id, uint32_t n_scans, uint32_t n,
                               uint32_t stride, int variant, rpl_node_hq* nodes, uint32_t* counts,
                               void* stream);

#ifdef __cplusplus
}
#endif
#endif /* RPL_B200_H_ */
