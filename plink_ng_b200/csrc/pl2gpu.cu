// pl2gpu.cu - C-ABI entry points (include/plink2_b200.h): context, staging, KING job driver.
#include <dlfcn.h>
#include <nccl.h>

#include <algorithm>
#include <cstdarg>
#include <cstring>
#include <mutex>
#include <vector>

#include "../../include/plink2_b200.h"
#include "common.cuh"
#include "king_kernels.cuh"
#include "king_ts_kernel.cuh"
#include "king_pairs_kernel.cuh"
#include "umma_probe.cuh"

namespace pl2 {

static thread_local char g_err[1024] = "";

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}
const char* get_error() { return g_err; }

// ---- tile list over the strict lower triangle restricted to rows [row_start,row_end) ----
static uint32_t ColTilesForRowTile(uint32_t rt, uint32_t row_end, bool include_diag, uint32_t tile_cols) {
  uint32_t tile_row_end = (rt + 1) * kTileRows;
  if (tile_row_end > row_end) tile_row_end = row_end;
  // columns 0 .. tile_row_end-2 are needed (.. tile_row_end-1 with the diagonal)
  const uint32_t cols = include_diag ? tile_row_end : (tile_row_end ? tile_row_end - 1 : 0);
  if (!cols) return 0;
  return DivUpU32(cols, tile_cols);
}

uint64_t CountTiles(uint32_t row_start, uint32_t row_end, bool include_diag, uint32_t tile_cols) {
  if (row_end <= row_start) return 0;
  uint64_t n = 0;
  for (uint32_t rt = row_start / kTileRows; rt * kTileRows < row_end; ++rt) n += ColTilesForRowTile(rt, row_end, include_diag, tile_cols);
  return n;
}

int BuildTileList(uint32_t row_start, uint32_t row_end, bool include_diag, TileList* tl, uint32_t tile_cols) {
  std::vector<uint32_t> rt_v, tc_v, off_v;
  tl->row_tile_first = row_start / kTileRows;
  uint32_t rt = tl->row_tile_first;
  // an empty row range (a rank of a multi-GPU team that owns no rows) has no tiles at all
  for (; row_end > row_start && rt * kTileRows < row_end; ++rt) {
    off_v.push_back(static_cast<uint32_t>(rt_v.size()));
    const uint32_t nct = ColTilesForRowTile(rt, row_end, include_diag, tile_cols);
    for (uint32_t tc = 0; tc < nct; ++tc) {
      rt_v.push_back(rt);
      tc_v.push_back(tc);
    }
  }
  off_v.push_back(static_cast<uint32_t>(rt_v.size()));
  tl->row_tile_ct = rt - tl->row_tile_first;
  tl->tile_ct = static_cast<uint32_t>(rt_v.size());
  const size_t nb = (rt_v.size() + 1) * sizeof(uint32_t);
  PL2_CUDA_OK(cudaMalloc(&tl->d_tile_rt, nb));
  PL2_CUDA_OK(cudaMalloc(&tl->d_tile_tc, nb));
  PL2_CUDA_OK(cudaMalloc(&tl->d_rowtile_offset, off_v.size() * sizeof(uint32_t)));
  if (!rt_v.empty()) {
    PL2_CUDA_OK(cudaMemcpy(tl->d_tile_rt, rt_v.data(), rt_v.size() * sizeof(uint32_t), cudaMemcpyHostToDevice));
    PL2_CUDA_OK(cudaMemcpy(tl->d_tile_tc, tc_v.data(), tc_v.size() * sizeof(uint32_t), cudaMemcpyHostToDevice));
  }
  PL2_CUDA_OK(cudaMemcpy(tl->d_rowtile_offset, off_v.data(), off_v.size() * sizeof(uint32_t), cudaMemcpyHostToDevice));
  tl->h_rowtile_offset = off_v;
  // launch order: blocks of kBand x kBand tiles (~ one wave of 148 CTAs) so that the CTAs resident at
  // the same time stream the same few row/column sample ranges and hit in L2
  constexpr uint32_t kBand = 12;
  std::vector<uint32_t> order;
  order.reserve(rt_v.size());
  const uint32_t n_rt = tl->row_tile_ct;
  for (uint32_t rb = 0; rb < n_rt; rb += kBand) {
    const uint32_t rb_end = std::min(n_rt, rb + kBand);
    uint32_t max_cols = 0;
    for (uint32_t r = rb; r < rb_end; ++r) max_cols = std::max(max_cols, off_v[r + 1] - off_v[r]);
    for (uint32_t cb = 0; cb < max_cols; cb += kBand) {
      for (uint32_t r = rb; r < rb_end; ++r) {
        const uint32_t ncols = off_v[r + 1] - off_v[r];
        for (uint32_t c = cb; c < std::min(ncols, cb + kBand); ++c) order.push_back(off_v[r] + c);
      }
    }
  }
  PL2_CUDA_OK(cudaMalloc(&tl->d_tile_order, nb));
  if (!order.empty()) PL2_CUDA_OK(cudaMemcpy(tl->d_tile_order, order.data(), order.size() * sizeof(uint32_t), cudaMemcpyHostToDevice));
  return 0;
}

void FreeTileList(TileList* tl) {
  cudaFree(tl->d_tile_rt);
  cudaFree(tl->d_tile_tc);
  cudaFree(tl->d_rowtile_offset);
  cudaFree(tl->d_tile_order);
  tl->d_tile_order = nullptr;
  tl->d_tile_rt = tl->d_tile_tc = tl->d_rowtile_offset = nullptr;
}

// ---- TMA tensor maps ----
typedef CUresult (*TensorMapEncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static TensorMapEncodeFn GetTensorMapEncode() {
  static TensorMapEncodeFn encode = nullptr;
  if (!encode) {
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres) != cudaSuccess || qres != cudaDriverEntryPointSuccess || !fn) {
      cudaGetLastError();
      set_error("cuTensorMapEncodeTiled is not available from this driver");
      return nullptr;
    }
    encode = reinterpret_cast<TensorMapEncodeFn>(fn);
  }
  return encode;
}

// 3-D uint8 tensor map over a sample-major copy raw_x[kstep_ct][sample_ct][16] (geno_tile_samples_kernel) with box
// {16, box_samples, box_ksteps}: one TMA copy lands box_ksteps consecutive [box_samples][16] blocks in shared memory.
static int MakeSampleMajorTensorMap(CUtensorMap* out, void* base, uint32_t sample_ct, uint32_t kstep_ct, uint32_t box_samples, uint32_t box_ksteps) {
  const TensorMapEncodeFn encode = GetTensorMapEncode();
  if (!encode) return 1;
  const cuuint64_t dims[3] = {16, sample_ct, kstep_ct};
  const cuuint64_t strides[2] = {16, 16ull * sample_ct};  // bytes, dimensions 1 and 2
  const cuuint32_t box[3] = {16, box_samples, box_ksteps};
  const cuuint32_t elem_strides[3] = {1, 1, 1};
  const CUresult r = encode(out, CU_TENSOR_MAP_DATA_TYPE_UINT8, 3, base, dims, strides, box, elem_strides, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed (%d) for a %u-sample x %u-k-step copy", static_cast<int>(r), sample_ct, kstep_ct);
    return 1;
  }
  return 0;
}

int MakeRawTensorMap(CUtensorMap* out, void* base, uint32_t pitch, uint32_t rows, uint32_t box_bytes, uint32_t box_rows) {
  const TensorMapEncodeFn encode = GetTensorMapEncode();
  if (!encode) return 1;
  const cuuint64_t dims[2] = {pitch, rows};
  const cuuint64_t strides[1] = {pitch};  // bytes, dimension 1
  const cuuint32_t box[2] = {box_bytes, box_rows};
  const cuuint32_t elem_strides[2] = {1, 1};
  const CUresult r = encode(out, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, base, dims, strides, box, elem_strides, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed (%d) for a %u x %u-byte block", static_cast<int>(r), rows, pitch);
    return 1;
  }
  return 0;
}

// ---- NCCL, loaded on first use: the library has no link-time dependency on it, and inside a process that
// already carries an NCCL (torch.distributed) the same copy is shared ----
namespace {
struct NcclApi {
  ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
  ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
  ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
  ncclResult_t (*AllGather)(const void*, void*, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*AllReduce)(const void*, void*, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
  const char* (*GetErrorString)(ncclResult_t) = nullptr;
  bool ok = false;
};
NcclApi g_nccl;
std::once_flag g_nccl_once;

void LoadNccl() {
  void* h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
  if (!h) h = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
  if (!h) return;
  g_nccl.GetUniqueId = reinterpret_cast<decltype(g_nccl.GetUniqueId)>(dlsym(h, "ncclGetUniqueId"));
  g_nccl.CommInitRank = reinterpret_cast<decltype(g_nccl.CommInitRank)>(dlsym(h, "ncclCommInitRank"));
  g_nccl.CommDestroy = reinterpret_cast<decltype(g_nccl.CommDestroy)>(dlsym(h, "ncclCommDestroy"));
  g_nccl.AllGather = reinterpret_cast<decltype(g_nccl.AllGather)>(dlsym(h, "ncclAllGather"));
  g_nccl.AllReduce = reinterpret_cast<decltype(g_nccl.AllReduce)>(dlsym(h, "ncclAllReduce"));
  g_nccl.GetErrorString = reinterpret_cast<decltype(g_nccl.GetErrorString)>(dlsym(h, "ncclGetErrorString"));
  g_nccl.ok = g_nccl.GetUniqueId && g_nccl.CommInitRank && g_nccl.CommDestroy && g_nccl.AllGather && g_nccl.AllReduce && g_nccl.GetErrorString;
}
bool HaveNccl() {
  std::call_once(g_nccl_once, LoadNccl);
  if (!g_nccl.ok) set_error("NCCL (libnccl.so.2) could not be loaded: %s", dlerror() ? dlerror() : "symbols missing");
  return g_nccl.ok;
}
}  // namespace

#define PL2_NCCL_OK(expr)                                                                              \
  do {                                                                                                 \
    ncclResult_t r__ = (expr);                                                                         \
    if (r__ != ncclSuccess) {                                                                          \
      pl2::set_error("%s failed at %s:%d: %s", #expr, __FILE__, __LINE__, g_nccl.GetErrorString(r__)); \
      return 1;                                                                                        \
    }                                                                                                  \
  } while (0)

int CommAllGatherInPlace(Ctx* ctx, void* buf, uint64_t bytes_per_rank, cudaStream_t stream) {
  if (!ctx->comm) {
    set_error("no communicator attached to the context");
    return 1;
  }
  const uint8_t* mine = static_cast<const uint8_t*>(buf) + static_cast<uint64_t>(ctx->comm_rank) * bytes_per_rank;
  PL2_NCCL_OK(g_nccl.AllGather(mine, buf, bytes_per_rank, ncclUint8, static_cast<ncclComm_t>(ctx->comm), stream));
  return 0;
}

int CommAllReduceSumF64(Ctx* ctx, double* buf, uint64_t count, cudaStream_t stream) {
  if (!ctx->comm) {
    set_error("no communicator attached to the context");
    return 1;
  }
  PL2_NCCL_OK(g_nccl.AllReduce(buf, buf, count, ncclDouble, ncclSum, static_cast<ncclComm_t>(ctx->comm), stream));
  return 0;
}

// ---- staged genotype block on the device ----
int StageAlloc(uint32_t sample_ct, uint32_t variant_cap, GenoStage* gs, uint32_t sample_pad) {
  gs->sample_ct = sample_ct;
  gs->sample_ct_padded = RoundUpU32(sample_ct, sample_pad);
  gs->pitch = gs->sample_ct_padded / 4;
  gs->variant_cap = RoundUpU32(variant_cap, kVariantPad);
  if (cudaMalloc(&gs->d_raw, static_cast<uint64_t>(gs->variant_cap) * gs->pitch) != cudaSuccess) {
    cudaGetLastError();
    gs->d_raw = nullptr;
    set_error("insufficient device memory for a %u-variant x %u-sample genotype stage", gs->variant_cap, sample_ct);
    return 1;
  }
  return 0;
}

int LaunchPadGenotypes(Ctx* ctx, uint8_t* dst, uint32_t pitch, uint32_t sample_ct, uint32_t variant_ct, uint32_t variant_ct_padded, cudaStream_t stream) {
  if (!variant_ct_padded) return 0;
  pad_genotypes_kernel<<<variant_ct_padded, 128, 0, stream ? stream : ctx->stream>>>(dst, pitch, sample_ct, variant_ct, variant_ct_padded);
  ctx->launches++;
  PL2_CUDA_OK(cudaGetLastError());
  return 0;
}

void StageFree(GenoStage* gs) {
  cudaFree(gs->d_raw);
  gs->d_raw = nullptr;
}

int StageUpload(Ctx* ctx, GenoStage* gs, const void* src, uint64_t src_stride, uint32_t variant_ct, int src_is_device, uint32_t* padded_ct_ptr, uint32_t dst_row, uint32_t pad_to) {
  const uint32_t padded = RoundUpU32(variant_ct, pad_to);
  if (dst_row + padded > gs->variant_cap) {
    set_error("StageUpload: %u + %u rows exceed the stage capacity %u", dst_row, padded, gs->variant_cap);
    return 1;
  }
  const uint32_t width = DivUpU32(gs->sample_ct, 4);
  uint8_t* dst = gs->d_raw + static_cast<uint64_t>(dst_row) * gs->pitch;
  if (variant_ct) {
    PL2_CUDA_OK(cudaMemcpy2DAsync(dst, gs->pitch, src, src_stride, width, variant_ct, src_is_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, ctx->stream));
  }
  if (padded) {
    pad_genotypes_kernel<<<padded, 128, 0, ctx->stream>>>(dst, gs->pitch, gs->sample_ct, variant_ct, padded);
    ctx->launches++;
    PL2_CUDA_OK(cudaGetLastError());
  }
  *padded_ct_ptr = padded;
  return 0;
}

}  // namespace pl2

using namespace pl2;

struct Pl2KingJob {
  Pl2GpuCtx* ctx = nullptr;
  uint32_t sample_ct = 0, row_start = 0, row_end = 0;
  int algo = kPl2KingAlgoTensor;
  TileList tiles;
  // TS path: two staged blocks + two sample-major copies, so that the copy / all-gather, padding and
  // re-tiling of batch k+1 (prep stream) overlap the tensor kernel of batch k (compute stream).
  // The other algorithms use buffer 0 on the compute stream only.
  GenoStage stage[2];
  uint8_t* d_raw_t[2] = {nullptr, nullptr};  // TS path: sample-major copy of samples [0, ts_samples) (geno_tile_samples_kernel)
  uint32_t ts_samples = 0;                   // TS path: samples in that copy, a multiple of kTsSamplePad covering the row tiles
  CUtensorMap tmap_i[2], tmap_j[2];          // TS path: 3-D tensor maps over d_raw_t[b], row-tile and column-tile boxes
  cudaEvent_t ev_prep_done[2] = {nullptr, nullptr};
  cudaEvent_t ev_kernel_start[2] = {nullptr, nullptr};  // timing-enabled pair around the tensor kernel (pl2gpu_king_last_kernel_ms)
  cudaEvent_t ev_kernel_done[2] = {nullptr, nullptr};
  int last_buf = -1;
  bool kernel_pending[2] = {false, false};
  uint32_t buf_idx = 0;
  uint32_t* d_planes = nullptr;  // popcount path only
  uint32_t tile_cols = kTileCols;
  int32_t* d_raw_acc = nullptr;
  void* d_out_stage = nullptr;   // bounded staging for host downloads
  uint64_t out_stage_bytes = 0;
  uint64_t variants_added = 0;
  cudaEvent_t ev_copied = nullptr;     // the caller's buffer has been consumed (prep stream)
  cudaEvent_t ev_src_ready = nullptr;  // device sources ordered on the compute stream
};

extern "C" {

int pl2gpu_abi_version(void) { return 2; }

const char* pl2gpu_last_error(void) { return get_error(); }

int pl2gpu_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) {
    cudaGetLastError();
    return 0;
  }
  return n;
}

int pl2gpu_ctx_create(int device_idx, Pl2GpuCtx** ctx_ptr) {
  *ctx_ptr = nullptr;
  int n = 0;
  PL2_CUDA_OK(cudaGetDeviceCount(&n));
  if (device_idx < 0 || device_idx >= n) {
    set_error("pl2gpu_ctx_create: device %d out of range (%d CUDA devices visible); there is no CPU fallback", device_idx, n);
    return 1;
  }
  cudaDeviceProp prop;
  PL2_CUDA_OK(cudaGetDeviceProperties(&prop, device_idx));
  if (prop.major != 10) {
    set_error("pl2gpu_ctx_create: device %d is sm_%d%d; this library contains sm_100a code only", device_idx, prop.major, prop.minor);
    return 1;
  }
  PL2_CUDA_OK(cudaSetDevice(device_idx));
  Pl2GpuCtx* ctx = new Pl2GpuCtx();
  ctx->c.device = device_idx;
  ctx->c.sm_count = prop.multiProcessorCount;
  PL2_CUDA_OK(cudaStreamCreateWithFlags(&ctx->c.stream, cudaStreamNonBlocking));
  {
    // the prep stream outranks the compute stream: its short copy / pad / re-tile / all-gather kernels must get
    // SM slots while a long tensor kernel keeps every SM busy
    int prio_lo = 0, prio_hi = 0;
    PL2_CUDA_OK(cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi));
    PL2_CUDA_OK(cudaStreamCreateWithPriority(&ctx->c.copy_stream, cudaStreamNonBlocking, prio_hi));
  }
  PL2_CUDA_OK(cudaFuncSetAttribute(king_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kTcSmemBytes));
  PL2_CUDA_OK(cudaFuncSetAttribute(umma_probe_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kProbeSmemBytes));
  PL2_CUDA_OK(cudaFuncSetAttribute(umma_probe_ts_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kProbeSmemBytes));
  PL2_CUDA_OK(cudaFuncSetAttribute(king_ts_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kTsSmemBytes));
  *ctx_ptr = ctx;
  return 0;
}

int pl2gpu_ctx_destroy(Pl2GpuCtx* ctx) {
  if (!ctx) return 0;
  cudaSetDevice(ctx->c.device);
  pl2gpu_comm_destroy(ctx);
  if (ctx->c.stream) cudaStreamDestroy(ctx->c.stream);
  if (ctx->c.copy_stream) cudaStreamDestroy(ctx->c.copy_stream);
  for (auto& e : ctx->c.events)
    if (e) cudaEventDestroy(e);
  delete ctx;
  return 0;
}

int pl2gpu_ctx_synchronize(Pl2GpuCtx* ctx) {
  PL2_CUDA_OK(cudaSetDevice(ctx->c.device));
  PL2_CUDA_OK(cudaStreamSynchronize(ctx->c.stream));
  return 0;
}

void* pl2gpu_ctx_stream(Pl2GpuCtx* ctx) { return ctx ? static_cast<void*>(ctx->c.stream) : nullptr; }

uint64_t pl2gpu_ctx_launch_count(Pl2GpuCtx* ctx) { return ctx ? ctx->c.launches : 0; }

int pl2gpu_ctx_mem_info(Pl2GpuCtx* ctx, uint64_t* free_bytes, uint64_t* total_bytes) {
  if (!ctx) {
    set_error("pl2gpu_ctx_mem_info: null context");
    return 1;
  }
  PL2_CUDA_OK(cudaSetDevice(ctx->c.device));
  size_t f = 0, t = 0;
  PL2_CUDA_OK(cudaMemGetInfo(&f, &t));
  if (free_bytes) *free_bytes = f;
  if (total_bytes) *total_bytes = t;
  return 0;
}

int pl2gpu_host_alloc(uint64_t bytes, void** ptr) {
  *ptr = nullptr;
  PL2_CUDA_OK(cudaHostAlloc(ptr, bytes ? bytes : 1, cudaHostAllocDefault));
  return 0;
}

int pl2gpu_host_free(void* ptr) {
  if (ptr) PL2_CUDA_OK(cudaFreeHost(ptr));
  return 0;
}

int pl2gpu_ctx_event_record(Pl2GpuCtx* ctx, int slot) {
  if (!ctx || slot < 0 || slot >= 16) {
    set_error("pl2gpu_ctx_event_record: bad arguments");
    return 1;
  }
  PL2_CUDA_OK(cudaSetDevice(ctx->c.device));
  if (!ctx->c.events[slot]) PL2_CUDA_OK(cudaEventCreate(&ctx->c.events[slot]));
  PL2_CUDA_OK(cudaEventRecord(ctx->c.events[slot], ctx->c.stream));
  return 0;
}

int pl2gpu_ctx_event_elapsed_ms(Pl2GpuCtx* ctx, int slot_from, int slot_to, float* ms) {
  if (!ctx || slot_from < 0 || slot_from >= 16 || slot_to < 0 || slot_to >= 16 || !ctx->c.events[slot_from] || !ctx->c.events[slot_to]) {
    set_error("pl2gpu_ctx_event_elapsed_ms: bad arguments");
    return 1;
  }
  PL2_CUDA_OK(cudaSetDevice(ctx->c.device));
  PL2_CUDA_OK(cudaEventSynchronize(ctx->c.events[slot_to]));
  PL2_CUDA_OK(cudaEventElapsedTime(ms, ctx->c.events[slot_from], ctx->c.events[slot_to]));
  return 0;
}

// ------------------------------------------------------------------------------------------ communicator

int pl2gpu_comm_unique_id(uint8_t* id_out) {
  if (!id_out || !HaveNccl()) {
    if (!id_out) set_error("pl2gpu_comm_unique_id: null output");
    return 1;
  }
  static_assert(sizeof(ncclUniqueId) == PL2GPU_COMM_ID_BYTES, "ncclUniqueId size");
  ncclUniqueId id;
  PL2_NCCL_OK(g_nccl.GetUniqueId(&id));
  memcpy(id_out, &id, sizeof(id));
  return 0;
}

int pl2gpu_comm_init(Pl2GpuCtx* ctx, int rank, int world, const uint8_t* id) {
  if (!ctx || !id || world < 1 || rank < 0 || rank >= world) {
    set_error("pl2gpu_comm_init: bad arguments");
    return 1;
  }
  if (ctx->c.comm) {
    set_error("pl2gpu_comm_init: the context already has a communicator");
    return 1;
  }
  if (!HaveNccl()) return 1;
  PL2_CUDA_OK(cudaSetDevice(ctx->c.device));
  ncclUniqueId uid;
  memcpy(&uid, id, sizeof(uid));
  ncclComm_t comm = nullptr;
  PL2_NCCL_OK(g_nccl.CommInitRank(&comm, world, uid, rank));
  ctx->c.comm = comm;
  ctx->c.comm_rank = rank;
  ctx->c.comm_world = world;
  return 0;
}

int pl2gpu_comm_destroy(Pl2GpuCtx* ctx) {
  if (!ctx || !ctx->c.comm) return 0;
  cudaSetDevice(ctx->c.device);
  cudaStreamSynchronize(ctx->c.stream);
  cudaStreamSynchronize(ctx->c.copy_stream);
  g_nccl.CommDestroy(static_cast<ncclComm_t>(ctx->c.comm));
  ctx->c.comm = nullptr;
  ctx->c.comm_rank = 0;
  ctx->c.comm_world = 1;
  return 0;
}

int pl2gpu_comm_allreduce_sum_f64(Pl2GpuCtx* ctx, double* device_buf, uint64_t count) {
  if (!ctx || !device_buf) {
    set_error("pl2gpu_comm_allreduce_sum_f64: bad arguments");
    return 1;
  }
  PL2_CUDA_OK(cudaSetDevice(ctx->c.device));
  return CommAllReduceSumF64(&ctx->c, device_buf, count, ctx->c.stream);
}

// ------------------------------------------------------------------------------------------ KING

static uint32_t ClampStageCap(uint32_t max_variants_per_add) {
  uint32_t cap = max_variants_per_add ? max_variants_per_add : kMaxStageVariants;
  if (cap > kMaxStageVariantsEx) cap = kMaxStageVariantsEx;
  return RoundUpU32(cap, kVariantPad);
}
constexpr uint64_t kKingOutStageBytes = 256ull << 20;

uint64_t pl2gpu_king_mem_required(uint32_t sample_ct, uint32_t row_start, uint32_t row_end, uint32_t max_variants_per_add) {
  // Upper bound over the algorithms (the caller does not pass one) of exactly what pl2gpu_king_begin_ex
  // allocates for the same max_variants_per_add: accumulators + staged block(s) and their per-algorithm
  // re-layouts + tile lists + the output staging buffer, plus slack for allocator granularity.
  const uint64_t cap = ClampStageCap(max_variants_per_add);
  const uint64_t slack = 128ull << 20;
  // SS tensor / popcount: 128 x 96 tiles, raw block + 3 bit planes (popcount only)
  const uint64_t tiles = CountTiles(row_start, row_end, false);
  const uint64_t npad = RoundUpU32(sample_ct, kSamplePad);
  const uint64_t need_ss = tiles * kKingTileAccWords * 4 + cap * (npad / 4) + 3ull * (cap / 32) * npad * 4 + tiles * 16;
  // TS tensor (the default): 128 x 80 tiles, two raw blocks + two sample-major copies of samples [0, row_end)
  // (a row block's column tiles reach back to sample 0)
  const uint64_t tiles_ts = CountTiles(row_start, row_end, false, kTsCols);
  const uint64_t npad_ts = RoundUpU32(sample_ct, kTsSamplePad);
  const uint64_t copy_samples = row_end > row_start ? RoundUpU32(row_end, kTsSamplePad) : 0;
  const uint64_t need_ts = tiles_ts * kTsTileAccWords * 4 + 2 * cap * (npad_ts / 4) + 2 * copy_samples * (cap / 4) + tiles_ts * 16;
  return (need_ss > need_ts ? need_ss : need_ts) + kKingOutStageBytes + slack;
}

int pl2gpu_king_begin(Pl2GpuCtx* ctx, uint32_t sample_ct, uint32_t row_start, uint32_t row_end, int algo, Pl2KingJob** job_ptr) {
  return pl2gpu_king_begin_ex(ctx, sample_ct, row_start, row_end, algo, 0, job_ptr);
}

int pl2gpu_king_begin_ex(Pl2GpuCtx* ctx, uint32_t sample_ct, uint32_t row_start, uint32_t row_end, int algo, uint32_t max_variants_per_add, Pl2KingJob** job_ptr) {
  *job_ptr = nullptr;
  if (!ctx) {
    set_error("pl2gpu_king_begin: null context");
    return 1;
  }
  if (sample_ct < 2 || row_end > sample_ct || row_start > row_end) {  // row_start == row_end: a rank that only takes part in the all-gathers
    set_error("pl2gpu_king_begin: bad row range [%u,%u) for %u samples", row_start, row_end, sample_ct);
    return 1;
  }
  if (algo == kPl2KingAlgoAuto) algo = kPl2KingAlgoTensorTS;
  if (algo != kPl2KingAlgoPopcount && algo != kPl2KingAlgoTensor && algo != kPl2KingAlgoTensorTS) {
    set_error("pl2gpu_king_begin: unknown algo %d", algo);
    return 1;
  }
  PL2_CUDA_OK(cudaSetDevice(ctx->c.device));
  Pl2KingJob* job = new Pl2KingJob();
  job->ctx = ctx;
  job->sample_ct = sample_ct;
  job->row_start = row_start;
  job->row_end = row_end;
  job->algo = algo;
  auto fail = [&]() {
    pl2gpu_king_end(job);
    return 1;
  };
  const bool ts = algo == kPl2KingAlgoTensorTS;
  const uint32_t cap = ClampStageCap(max_variants_per_add);
  bool ev_ok = cudaEventCreateWithFlags(&job->ev_copied, cudaEventDisableTiming) == cudaSuccess && cudaEventCreateWithFlags(&job->ev_src_ready, cudaEventDisableTiming) == cudaSuccess;
  for (int b = 0; b < 2 && ev_ok; ++b) {
    ev_ok = cudaEventCreateWithFlags(&job->ev_prep_done[b], cudaEventDisableTiming) == cudaSuccess && cudaEventCreate(&job->ev_kernel_start[b]) == cudaSuccess && cudaEventCreate(&job->ev_kernel_done[b]) == cudaSuccess;
  }
  if (!ev_ok) {
    set_error("pl2gpu_king_begin: cudaEventCreate failed");
    return fail();
  }
  job->tile_cols = ts ? kTsCols : kTileCols;
  if (BuildTileList(row_start, row_end, false, &job->tiles, job->tile_cols)) return fail();
  for (int b = 0; b < (ts ? 2 : 1); ++b) {
    if (StageAlloc(sample_ct, cap, &job->stage[b], ts ? kTsSamplePad : kSamplePad)) return fail();
    if (ts && job->tiles.tile_ct) {
      // the row tiles end at or before sample_ct_padded (a multiple of kTsSamplePad), so the copy fits the stage
      job->ts_samples = RoundUpU32((job->tiles.row_tile_first + job->tiles.row_tile_ct) * kTileRows, kTsSamplePad);
      const uint32_t ksteps = job->stage[b].variant_cap / kTsKstep;
      if (cudaMalloc(&job->d_raw_t[b], static_cast<uint64_t>(job->ts_samples) * (job->stage[b].variant_cap / 4)) != cudaSuccess) {
        cudaGetLastError();
        set_error("pl2gpu_king_begin: insufficient device memory for the sample-major genotype copy");
        return fail();
      }
      if (MakeSampleMajorTensorMap(&job->tmap_i[b], job->d_raw_t[b], job->ts_samples, ksteps, kTileRows, kTsRingKsteps) ||
          MakeSampleMajorTensorMap(&job->tmap_j[b], job->d_raw_t[b], job->ts_samples, ksteps, kTsCols, kTsRingKsteps))
        return fail();
    }
  }
  const uint64_t acc_bytes = static_cast<uint64_t>(job->tiles.tile_ct) * (5ull * job->tile_cols * kTileRows) * sizeof(int32_t);
  if (cudaMalloc(&job->d_raw_acc, acc_bytes ? acc_bytes : 4) != cudaSuccess) {
    cudaGetLastError();
    set_error("pl2gpu_king_begin: insufficient device memory for %u pair tiles (%.1f GB of accumulators); narrow the row range", job->tiles.tile_ct, acc_bytes / 1e9);
    return fail();
  }
  if (cudaMemsetAsync(job->d_raw_acc, 0, acc_bytes, ctx->c.stream) != cudaSuccess) {
    set_error("pl2gpu_king_begin: cudaMemsetAsync failed: %s", cudaGetErrorString(cudaGetLastError()));
    return fail();
  }
  if (algo == kPl2KingAlgoPopcount) {
    const uint64_t plane_bytes = 3ull * (job->stage[0].variant_cap / 32) * job->stage[0].sample_ct_padded * sizeof(uint32_t);
    if (cudaMalloc(&job->d_planes, plane_bytes) != cudaSuccess) {
      cudaGetLastError();
      set_error("pl2gpu_king_begin: insufficient device memory for bit planes");
      return fail();
    }
  }
  job->out_stage_bytes = kKingOutStageBytes;
  if (cudaMalloc(&job->d_out_stage, job->out_stage_bytes) != cudaSuccess) {
    cudaGetLastError();
    set_error("pl2gpu_king_begin: insufficient device memory for output staging");
    return fail();
  }
  *job_ptr = job;
  return 0;
}

// TS path: the staged block stage[b] holds `cur` variants (rows [0, cur)); pad it, re-tile samples
// [0, ts_samples) sample-major and queue the tensor kernel.  Everything up to the kernel runs on the prep stream.
static int KingTsPrepAndLaunch(Pl2KingJob* job, uint32_t b, uint32_t cur, bool pad_valid_rows) {
  Ctx* c = &job->ctx->c;
  cudaStream_t prep = c->copy_stream;
  GenoStage& st = job->stage[b];
  const uint32_t padded = RoundUpU32(cur, kVariantPad);
  // pad_valid_rows == false: the valid rows were already padded slice by slice (sharded add); only the tail rows remain
  if (pad_valid_rows) {
    PL2_TRY(LaunchPadGenotypes(c, st.d_raw, st.pitch, st.sample_ct, cur, padded, prep));
  } else if (padded > cur) {
    PL2_TRY(LaunchPadGenotypes(c, st.d_raw + static_cast<uint64_t>(cur) * st.pitch, st.pitch, st.sample_ct, 0, padded - cur, prep));
  }
  if (!job->tiles.tile_ct) {  // nothing to count on this rank: only order later reuse of the buffer behind the gather
    PL2_CUDA_OK(cudaEventRecord(job->ev_kernel_done[b], prep));
    job->kernel_pending[b] = true;
    return 0;
  }
  geno_tile_samples_kernel<<<dim3(padded / kTsKstep, job->ts_samples / 64), 256, 0, prep>>>(st.d_raw, st.pitch, job->ts_samples, job->d_raw_t[b]);
  c->launches++;
  PL2_CUDA_OK(cudaGetLastError());
  PL2_CUDA_OK(cudaEventRecord(job->ev_prep_done[b], prep));
  PL2_CUDA_OK(cudaStreamWaitEvent(c->stream, job->ev_prep_done[b], 0));
  PL2_CUDA_OK(cudaEventRecord(job->ev_kernel_start[b], c->stream));
  king_ts_kernel<<<job->tiles.tile_ct, kTsThreads, kTsSmemBytes, c->stream>>>(job->tmap_i[b], job->tmap_j[b], padded, job->tiles.d_tile_order, job->tiles.d_tile_rt, job->tiles.d_tile_tc, job->d_raw_acc);
  c->launches++;
  PL2_CUDA_OK(cudaGetLastError());
  PL2_CUDA_OK(cudaEventRecord(job->ev_kernel_done[b], c->stream));
  job->kernel_pending[b] = true;
  job->last_buf = static_cast<int>(b);
  return 0;
}

int pl2gpu_king_add_variants(Pl2KingJob* job, const void* genovecs, uint64_t variant_stride_bytes, uint32_t variant_ct, int src_is_device) {
  if (!job) {
    set_error("pl2gpu_king_add_variants: null job");
    return 1;
  }
  Ctx* c = &job->ctx->c;
  PL2_CUDA_OK(cudaSetDevice(c->device));
  const uint64_t min_stride = 8ull * DivUpU32(job->sample_ct, 32);
  if (variant_stride_bytes < DivUpU32(job->sample_ct, 4)) {
    set_error("pl2gpu_king_add_variants: variant stride %llu < %u bytes of genotype data (PgrGet rows are %llu bytes)", static_cast<unsigned long long>(variant_stride_bytes), DivUpU32(job->sample_ct, 4), static_cast<unsigned long long>(min_stride));
    return 1;
  }
  const uint8_t* src = static_cast<const uint8_t*>(genovecs);
  const bool ts = job->algo == kPl2KingAlgoTensorTS;
  uint32_t done = 0;
  while (done < variant_ct) {
    uint32_t cur = variant_ct - done;
    if (cur > job->stage[0].variant_cap) cur = job->stage[0].variant_cap;
    const uint8_t* src_cur = src + static_cast<uint64_t>(done) * variant_stride_bytes;
    if (ts && job->tiles.tile_ct) {
      // Double-buffered: copy + pad + row re-tiling on the prep stream while the previous batch's tensor
      // kernel (which reads the OTHER staged block through its tensor map) is still running.
      const uint32_t b = job->buf_idx;
      job->buf_idx ^= 1;
      GenoStage& st = job->stage[b];
      cudaStream_t prep = c->copy_stream;
      if (job->kernel_pending[b]) PL2_CUDA_OK(cudaStreamWaitEvent(prep, job->ev_kernel_done[b], 0));
      if (src_is_device == 1) {
        // device source produced by work the caller ordered on the context's stream
        PL2_CUDA_OK(cudaEventRecord(job->ev_src_ready, c->stream));
        PL2_CUDA_OK(cudaStreamWaitEvent(prep, job->ev_src_ready, 0));
      }
      PL2_CUDA_OK(cudaMemcpy2DAsync(st.d_raw, st.pitch, src_cur, variant_stride_bytes, DivUpU32(st.sample_ct, 4), cur, src_is_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, prep));
      PL2_CUDA_OK(cudaEventRecord(job->ev_copied, prep));
      PL2_TRY(KingTsPrepAndLaunch(job, b, cur, true));
      if (!src_is_device) PL2_CUDA_OK(cudaEventSynchronize(job->ev_copied));  // the caller may reuse its buffer; the kernels keep running
    } else {
      uint32_t padded = 0;
      PL2_TRY(StageUpload(c, &job->stage[0], src_cur, variant_stride_bytes, cur, src_is_device, &padded));
      if (job->tiles.tile_ct) {
        if (job->algo == kPl2KingAlgoPopcount) {
          const uint32_t word_ct = padded / 32;
          const uint64_t warps = static_cast<uint64_t>(job->stage[0].sample_ct_padded / 32) * word_ct;
          split_transpose_kernel<<<static_cast<uint32_t>(DivUpU64(warps, 8)), 256, 0, c->stream>>>(job->stage[0].d_raw, job->stage[0].pitch, job->stage[0].sample_ct_padded, word_ct, job->d_planes);
          c->launches++;
          king_popc_kernel<<<job->tiles.tile_ct * 2, 256, 0, c->stream>>>(job->d_planes, job->stage[0].sample_ct_padded, word_ct, job->tiles.d_tile_rt, job->tiles.d_tile_tc, job->d_raw_acc);
          c->launches++;
        } else {
          king_tc_kernel<<<job->tiles.tile_ct, kTcThreads, kTcSmemBytes, c->stream>>>(job->stage[0].d_raw, job->stage[0].pitch, padded, job->tiles.d_tile_order, job->tiles.d_tile_rt, job->tiles.d_tile_tc, job->d_raw_acc);
          c->launches++;
        }
        PL2_CUDA_OK(cudaGetLastError());
      }
      // host source on the compute stream: it has been consumed once the stream reaches here
      if (!src_is_device) PL2_CUDA_OK(cudaStreamSynchronize(c->stream));
    }
    done += cur;
  }
  job->variants_added += variant_ct;
  return 0;
}

int pl2gpu_king_add_variants_sharded(Pl2KingJob* job, const void* slice, uint64_t variant_stride_bytes, uint32_t slice_variant_ct, int src_is_device) {
  if (!job || !job->ctx->c.comm) {
    set_error("pl2gpu_king_add_variants_sharded: %s", job ? "no communicator attached to the context (pl2gpu_comm_init)" : "null job");
    return 1;
  }
  Ctx* c = &job->ctx->c;
  PL2_CUDA_OK(cudaSetDevice(c->device));
  if (job->algo != kPl2KingAlgoTensorTS) {
    set_error("pl2gpu_king_add_variants_sharded: only the default (TS tensor) algorithm is sharded");
    return 1;
  }
  const uint64_t total64 = static_cast<uint64_t>(slice_variant_ct) * c->comm_world;
  if (!slice_variant_ct || total64 > job->stage[0].variant_cap) {
    set_error("pl2gpu_king_add_variants_sharded: %u variants x %d ranks exceed the stage capacity %u", slice_variant_ct, c->comm_world, job->stage[0].variant_cap);
    return 1;
  }
  if (variant_stride_bytes < DivUpU32(job->sample_ct, 4)) {
    set_error("pl2gpu_king_add_variants_sharded: variant stride too small");
    return 1;
  }
  const uint32_t total = static_cast<uint32_t>(total64);
  const uint32_t b = job->buf_idx;
  job->buf_idx ^= 1;
  GenoStage& st = job->stage[b];
  cudaStream_t prep = c->copy_stream;
  if (job->kernel_pending[b]) PL2_CUDA_OK(cudaStreamWaitEvent(prep, job->ev_kernel_done[b], 0));
  if (src_is_device == 1) {
    PL2_CUDA_OK(cudaEventRecord(job->ev_src_ready, c->stream));
    PL2_CUDA_OK(cudaStreamWaitEvent(prep, job->ev_src_ready, 0));
  }
  // this rank's variants land at rows [rank * slice, (rank + 1) * slice) of the staged block, are padded
  // there, and ONE in-place all-gather of the genotype column tile makes the block complete on every GPU
  uint8_t* mine = st.d_raw + static_cast<uint64_t>(c->comm_rank) * slice_variant_ct * st.pitch;
  PL2_CUDA_OK(cudaMemcpy2DAsync(mine, st.pitch, slice, variant_stride_bytes, DivUpU32(st.sample_ct, 4), slice_variant_ct, src_is_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, prep));
  PL2_CUDA_OK(cudaEventRecord(job->ev_copied, prep));
  PL2_TRY(LaunchPadGenotypes(c, mine, st.pitch, st.sample_ct, slice_variant_ct, slice_variant_ct, prep));
  PL2_TRY(CommAllGatherInPlace(c, st.d_raw, static_cast<uint64_t>(slice_variant_ct) * st.pitch, prep));
  PL2_TRY(KingTsPrepAndLaunch(job, b, total, false));
  if (!src_is_device) PL2_CUDA_OK(cudaEventSynchronize(job->ev_copied));
  job->variants_added += total;
  return 0;
}

static int KingGet(Pl2KingJob* job, uint32_t r0, uint32_t r1, void* dst, int dst_is_device, bool kinship) {
  if (!job) {
    set_error("pl2gpu_king_get: null job");
    return 1;
  }
  if (r0 < job->row_start || r1 > job->row_end || r0 > r1) {
    set_error("pl2gpu_king_get: rows [%u,%u) outside the job's [%u,%u)", r0, r1, job->row_start, job->row_end);
    return 1;
  }
  Ctx* c = &job->ctx->c;
  PL2_CUDA_OK(cudaSetDevice(c->device));
  const uint64_t bytes_per_pair = kinship ? 8 : 20;
  auto tri = [](uint64_t r) { return r ? r * (r - 1) / 2 : 0ull; };
  uint8_t* out = static_cast<uint8_t*>(dst);
  uint32_t cur0 = r0;
  while (cur0 < r1) {
    uint32_t cur1;
    void* d_dst;
    if (dst_is_device) {
      cur1 = r1;
      d_dst = out;
    } else {
      // largest row block whose pairs fit the staging buffer (at least one row)
      cur1 = cur0 + 1;
      while (cur1 < r1 && (tri(cur1 + 1) - tri(cur0)) * bytes_per_pair <= job->out_stage_bytes) ++cur1;
      if ((tri(cur1) - tri(cur0)) * bytes_per_pair > job->out_stage_bytes) {
        set_error("pl2gpu_king_get: a single row exceeds the staging buffer");
        return 1;
      }
      d_dst = job->d_out_stage;
    }
    const uint64_t pairs = tri(cur1) - tri(cur0);
    if (pairs) {
      const uint32_t rt_a = cur0 / kTileRows - job->tiles.row_tile_first;
      const uint32_t rt_b = (cur1 - 1) / kTileRows - job->tiles.row_tile_first;
      const uint32_t tile_a = job->tiles.h_rowtile_offset[rt_a];
      const uint32_t tile_b = job->tiles.h_rowtile_offset[rt_b + 1];
      if (tile_b > tile_a) {
        const uint32_t grid = (tile_b - tile_a) * 8;
        const int32_t* acc0 = job->d_raw_acc + static_cast<uint64_t>(tile_a) * (5ull * job->tile_cols * kTileRows);
        const uint32_t* trt = job->tiles.d_tile_rt + tile_a;
        const uint32_t* ttc = job->tiles.d_tile_tc + tile_a;
        if (job->tile_cols == kTsCols) {
          if (kinship) king_finalize_kernel<true, kTsCols><<<grid, 256, 0, c->stream>>>(acc0, trt, ttc, job->sample_ct, cur0, cur1, nullptr, static_cast<double*>(d_dst));
          else king_finalize_kernel<false, kTsCols><<<grid, 256, 0, c->stream>>>(acc0, trt, ttc, job->sample_ct, cur0, cur1, static_cast<uint32_t*>(d_dst), nullptr);
        } else {
          if (kinship) king_finalize_kernel<true, kTileCols><<<grid, 256, 0, c->stream>>>(acc0, trt, ttc, job->sample_ct, cur0, cur1, nullptr, static_cast<double*>(d_dst));
          else king_finalize_kernel<false, kTileCols><<<grid, 256, 0, c->stream>>>(acc0, trt, ttc, job->sample_ct, cur0, cur1, static_cast<uint32_t*>(d_dst), nullptr);
        }
        c->launches++;
        PL2_CUDA_OK(cudaGetLastError());
      }
      if (!dst_is_device) {
        PL2_CUDA_OK(cudaMemcpyAsync(out, d_dst, pairs * bytes_per_pair, cudaMemcpyDeviceToHost, c->stream));
        PL2_CUDA_OK(cudaStreamSynchronize(c->stream));
        out += pairs * bytes_per_pair;
      }
    }
    cur0 = cur1;
  }
  if (dst_is_device) {
    // caller synchronises through pl2gpu_ctx_synchronize / its own stream ordering
  }
  return 0;
}

int pl2gpu_king_get_counts(Pl2KingJob* job, uint32_t out_row_start, uint32_t out_row_end, uint32_t* dst, int dst_is_device) {
  return KingGet(job, out_row_start, out_row_end, dst, dst_is_device, false);
}

int pl2gpu_king_get_kinship(Pl2KingJob* job, uint32_t out_row_start, uint32_t out_row_end, double* dst, int dst_is_device) {
  return KingGet(job, out_row_start, out_row_end, dst, dst_is_device, true);
}

int pl2gpu_king_get_filtered(Pl2KingJob* job, uint32_t r0, uint32_t r1, double min_kinship, uint64_t max_out, uint32_t* pairs_out, uint32_t* counts_out, double* kinship_out, uint64_t* n_found) {
  if (!job || !n_found || (max_out && (!pairs_out || !counts_out || !kinship_out))) {
    set_error("pl2gpu_king_get_filtered: bad arguments");
    return 1;
  }
  if (r0 < job->row_start || r1 > job->row_end || r0 > r1) {
    set_error("pl2gpu_king_get_filtered: rows [%u,%u) outside the job's [%u,%u)", r0, r1, job->row_start, job->row_end);
    return 1;
  }
  *n_found = 0;
  Ctx* c = &job->ctx->c;
  PL2_CUDA_OK(cudaSetDevice(c->device));
  if (!job->tiles.tile_ct || r0 == r1) return 0;
  unsigned long long* d_found = nullptr;
  uint32_t *d_pairs = nullptr, *d_counts = nullptr;
  double* d_kin = nullptr;
  const uint64_t cap = max_out ? max_out : 1;
  int rc = 1;
  do {
    if (cudaMalloc(&d_found, 8) != cudaSuccess || cudaMalloc(&d_pairs, cap * 8) != cudaSuccess || cudaMalloc(&d_counts, cap * 20) != cudaSuccess || cudaMalloc(&d_kin, cap * 8) != cudaSuccess) {
      cudaGetLastError();
      set_error("pl2gpu_king_get_filtered: insufficient device memory for %llu result slots", static_cast<unsigned long long>(max_out));
      break;
    }
    if (cudaMemsetAsync(d_found, 0, 8, c->stream) != cudaSuccess) break;
    if (job->tile_cols == kTsCols) {
      king_filter_kernel<kTsCols><<<job->tiles.tile_ct, kTileRows, 0, c->stream>>>(job->d_raw_acc, job->tiles.d_tile_rt, job->tiles.d_tile_tc, job->sample_ct, r0, r1, min_kinship, max_out, d_found, d_pairs, d_counts, d_kin);
    } else {
      king_filter_kernel<kTileCols><<<job->tiles.tile_ct, kTileRows, 0, c->stream>>>(job->d_raw_acc, job->tiles.d_tile_rt, job->tiles.d_tile_tc, job->sample_ct, r0, r1, min_kinship, max_out, d_found, d_pairs, d_counts, d_kin);
    }
    c->launches++;
    unsigned long long found = 0;
    if (cudaGetLastError() != cudaSuccess || cudaMemcpyAsync(&found, d_found, 8, cudaMemcpyDeviceToHost, c->stream) != cudaSuccess || cudaStreamSynchronize(c->stream) != cudaSuccess) {
      set_error("pl2gpu_king_get_filtered: %s", cudaGetErrorString(cudaGetLastError()));
      break;
    }
    *n_found = found;
    const uint64_t k = found < max_out ? found : max_out;
    if (k) {
      std::vector<uint32_t> hp(2 * k), hc(5 * k);
      std::vector<double> hk(k);
      if (cudaMemcpy(hp.data(), d_pairs, k * 8, cudaMemcpyDeviceToHost) != cudaSuccess || cudaMemcpy(hc.data(), d_counts, k * 20, cudaMemcpyDeviceToHost) != cudaSuccess || cudaMemcpy(hk.data(), d_kin, k * 8, cudaMemcpyDeviceToHost) != cudaSuccess) {
        set_error("pl2gpu_king_get_filtered: %s", cudaGetErrorString(cudaGetLastError()));
        break;
      }
      std::vector<uint64_t> order(k);
      for (uint64_t q = 0; q < k; ++q) order[q] = q;
      std::sort(order.begin(), order.end(), [&](uint64_t a, uint64_t b) { return hp[2 * a] != hp[2 * b] ? hp[2 * a] < hp[2 * b] : hp[2 * a + 1] < hp[2 * b + 1]; });
      for (uint64_t q = 0; q < k; ++q) {
        const uint64_t src = order[q];
        pairs_out[2 * q] = hp[2 * src];
        pairs_out[2 * q + 1] = hp[2 * src + 1];
        memcpy(counts_out + 5 * q, &hc[5 * src], 20);
        kinship_out[q] = hk[src];
      }
    }
    rc = 0;
  } while (0);
  cudaFree(d_found);
  cudaFree(d_pairs);
  cudaFree(d_counts);
  cudaFree(d_kin);
  return rc;
}

uint64_t pl2gpu_king_variants_added(Pl2KingJob* job) { return job ? job->variants_added : 0; }

int pl2gpu_king_last_kernel_ms(Pl2KingJob* job, float* ms) {
  if (!job || !ms || job->last_buf < 0) {
    set_error("pl2gpu_king_last_kernel_ms: no tensor-kernel launch has been recorded (TS algorithm only)");
    return 1;
  }
  PL2_CUDA_OK(cudaSetDevice(job->ctx->c.device));
  PL2_CUDA_OK(cudaEventSynchronize(job->ev_kernel_done[job->last_buf]));
  PL2_CUDA_OK(cudaEventElapsedTime(ms, job->ev_kernel_start[job->last_buf], job->ev_kernel_done[job->last_buf]));
  return 0;
}

int pl2gpu_king_end(Pl2KingJob* job) {
  if (!job) return 0;
  if (job->ctx) {
    cudaSetDevice(job->ctx->c.device);
    cudaStreamSynchronize(job->ctx->c.stream);
    if (job->ctx->c.copy_stream) cudaStreamSynchronize(job->ctx->c.copy_stream);
  }
  if (job->ev_copied) cudaEventDestroy(job->ev_copied);
  if (job->ev_src_ready) cudaEventDestroy(job->ev_src_ready);
  FreeTileList(&job->tiles);
  for (int b = 0; b < 2; ++b) {
    if (job->ev_prep_done[b]) cudaEventDestroy(job->ev_prep_done[b]);
    if (job->ev_kernel_start[b]) cudaEventDestroy(job->ev_kernel_start[b]);
    if (job->ev_kernel_done[b]) cudaEventDestroy(job->ev_kernel_done[b]);
    StageFree(&job->stage[b]);
    cudaFree(job->d_raw_t[b]);
  }
  cudaFree(job->d_planes);
  cudaFree(job->d_raw_acc);
  cudaFree(job->d_out_stage);
  cudaGetLastError();
  delete job;
  return 0;
}

// ------------------------------------------------------------------------------------------ pair list

struct Pl2KingPairJob {
  Pl2GpuCtx* ctx = nullptr;
  uint32_t sample_ct = 0;
  uint64_t pair_ct = 0;
  GenoStage stage;
  uint8_t* d_raw_t = nullptr;   // sample-major 2-bit copy of the staged block
  uint32_t* d_pairs = nullptr;  // [pair][2]
  uint32_t* d_counts = nullptr; // [pair][5]
};

int pl2gpu_king_pairs_begin(Pl2GpuCtx* ctx, uint32_t sample_ct, const uint32_t* pairs_host, uint64_t pair_ct, Pl2KingPairJob** job_ptr) {
  if (job_ptr) *job_ptr = nullptr;
  if (!ctx || !job_ptr || !sample_ct || (pair_ct && !pairs_host)) {
    set_error("pl2gpu_king_pairs_begin: bad arguments");
    return 1;
  }
  for (uint64_t p = 0; p < 2 * pair_ct; ++p) {
    if (pairs_host[p] >= sample_ct) {
      set_error("pl2gpu_king_pairs_begin: pair %llu names sample %u of %u", static_cast<unsigned long long>(p / 2), pairs_host[p], sample_ct);
      return 1;
    }
  }
  PL2_CUDA_OK(cudaSetDevice(ctx->c.device));
  Pl2KingPairJob* job = new Pl2KingPairJob();
  job->ctx = ctx;
  job->sample_ct = sample_ct;
  job->pair_ct = pair_ct;
  auto fail = [&]() {
    pl2gpu_king_pairs_end(job);
    return 1;
  };
  if (StageAlloc(sample_ct, kMaxStageVariants, &job->stage, 64)) return fail();
  const uint64_t n_alloc = pair_ct ? pair_ct : 1;
  if (cudaMalloc(&job->d_raw_t, static_cast<uint64_t>(job->stage.sample_ct_padded) * (job->stage.variant_cap / 4)) != cudaSuccess || cudaMalloc(&job->d_pairs, n_alloc * 8) != cudaSuccess ||
      cudaMalloc(&job->d_counts, n_alloc * 20) != cudaSuccess) {
    cudaGetLastError();
    set_error("pl2gpu_king_pairs_begin: insufficient device memory for %llu pairs", static_cast<unsigned long long>(pair_ct));
    return fail();
  }
  if (cudaMemcpyAsync(job->d_pairs, pairs_host, pair_ct * 8, cudaMemcpyHostToDevice, ctx->c.stream) != cudaSuccess || cudaMemsetAsync(job->d_counts, 0, n_alloc * 20, ctx->c.stream) != cudaSuccess ||
      cudaStreamSynchronize(ctx->c.stream) != cudaSuccess) {
    set_error("pl2gpu_king_pairs_begin: %s", cudaGetErrorString(cudaGetLastError()));
    return fail();
  }
  *job_ptr = job;
  return 0;
}

int pl2gpu_king_pairs_add_variants(Pl2KingPairJob* job, const void* genovecs, uint64_t variant_stride_bytes, uint32_t variant_ct, int src_is_device) {
  if (!job || (!genovecs && variant_ct)) {
    set_error("pl2gpu_king_pairs_add_variants: bad arguments");
    return 1;
  }
  Ctx* c = &job->ctx->c;
  PL2_CUDA_OK(cudaSetDevice(c->device));
  const uint64_t min_stride = static_cast<uint64_t>(DivUpU32(job->sample_ct, 4));
  if (variant_stride_bytes < min_stride) {
    set_error("pl2gpu_king_pairs_add_variants: variant stride %llu < %llu bytes of genotype data", static_cast<unsigned long long>(variant_stride_bytes), static_cast<unsigned long long>(min_stride));
    return 1;
  }
  const uint8_t* src = static_cast<const uint8_t*>(genovecs);
  uint32_t done = 0;
  while (done < variant_ct) {
    uint32_t cur = variant_ct - done;
    if (cur > job->stage.variant_cap) cur = job->stage.variant_cap;
    uint32_t padded = 0;
    PL2_TRY(StageUpload(c, &job->stage, src + static_cast<uint64_t>(done) * variant_stride_bytes, variant_stride_bytes, cur, src_is_device, &padded));
    if (job->pair_ct) {
      const uint32_t pitch_t = padded / 4;
      geno_transpose_kernel<<<dim3(padded / 64, job->stage.sample_ct_padded / 64), 256, 0, c->stream>>>(job->stage.d_raw, job->stage.pitch, job->d_raw_t, pitch_t);
      king_pairs_kernel<<<static_cast<uint32_t>(DivUpU64(job->pair_ct, 8)), 256, 0, c->stream>>>(job->d_raw_t, pitch_t, padded / 32, job->d_pairs, job->pair_ct, job->d_counts);
      c->launches += 2;
      PL2_CUDA_OK(cudaGetLastError());
    }
    if (!src_is_device) PL2_CUDA_OK(cudaStreamSynchronize(c->stream));
    done += cur;
  }
  return 0;
}

int pl2gpu_king_pairs_get_counts(Pl2KingPairJob* job, uint64_t pair_start, uint64_t pair_end, uint32_t* dst, int dst_is_device) {
  if (!job || pair_start > pair_end || pair_end > job->pair_ct || (!dst && pair_end > pair_start)) {
    set_error("pl2gpu_king_pairs_get_counts: bad arguments");
    return 1;
  }
  Ctx* c = &job->ctx->c;
  PL2_CUDA_OK(cudaSetDevice(c->device));
  if (pair_end > pair_start) {
    PL2_CUDA_OK(cudaMemcpyAsync(dst, job->d_counts + 5 * pair_start, (pair_end - pair_start) * 20, dst_is_device ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost, c->stream));
  }
  PL2_CUDA_OK(cudaStreamSynchronize(c->stream));
  return 0;
}

int pl2gpu_king_pairs_end(Pl2KingPairJob* job) {
  if (!job) return 0;
  if (job->ctx) {
    cudaSetDevice(job->ctx->c.device);
    cudaStreamSynchronize(job->ctx->c.stream);
  }
  StageFree(&job->stage);
  cudaFree(job->d_raw_t);
  cudaFree(job->d_pairs);
  cudaFree(job->d_counts);
  cudaGetLastError();
  delete job;
  return 0;
}

// ------------------------------------------------------------------------------------------ probe

int pl2gpu_int8_peak(Pl2GpuCtx* ctx, uint32_t n_cols, int form, double min_seconds, double* tops_out, double* seconds_out) {
  if (!ctx || !tops_out || n_cols < 16 || n_cols > 240 || (n_cols & 15) || (form != 0 && form != 1)) {
    set_error("pl2gpu_int8_peak: bad arguments (n_cols must be a multiple of 16 in [16,240])");
    return 1;
  }
  Ctx* c = &ctx->c;
  PL2_CUDA_OK(cudaSetDevice(c->device));
  PL2_CUDA_OK(cudaFuncSetAttribute(umma_peak_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kProbeSmemBytes));
  cudaEvent_t e0 = nullptr, e1 = nullptr;
  PL2_CUDA_OK(cudaEventCreate(&e0));
  PL2_CUDA_OK(cudaEventCreate(&e1));
  const uint32_t blocks = 4096;  // x 32 UMMAs x 2 issuer warps: ~15-35 ms per launch
  const double ops_per_launch = 2.0 * 128 * n_cols * 32 * 32.0 * 2 * blocks * c->sm_count;
  umma_peak_kernel<<<c->sm_count, 128, kProbeSmemBytes, c->stream>>>(n_cols, blocks, static_cast<uint32_t>(form));  // warm-up
  c->launches++;
  PL2_CUDA_OK(cudaStreamSynchronize(c->stream));
  double total_s = 0, total_ops = 0;
  uint32_t per_batch = 8;
  while (total_s < min_seconds) {
    PL2_CUDA_OK(cudaEventRecord(e0, c->stream));
    for (uint32_t k = 0; k < per_batch; ++k) umma_peak_kernel<<<c->sm_count, 128, kProbeSmemBytes, c->stream>>>(n_cols, blocks, static_cast<uint32_t>(form));
    c->launches += per_batch;
    PL2_CUDA_OK(cudaEventRecord(e1, c->stream));
    PL2_CUDA_OK(cudaEventSynchronize(e1));
    PL2_CUDA_OK(cudaGetLastError());
    float ms = 0;
    PL2_CUDA_OK(cudaEventElapsedTime(&ms, e0, e1));
    total_s += ms * 1e-3;
    total_ops += ops_per_launch * per_batch;
    if (min_seconds <= 0) break;
  }
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  *tops_out = total_ops / total_s / 1e12;
  if (seconds_out) *seconds_out = total_s;
  return 0;
}



int pl2gpu_debug_umma(Pl2GpuCtx* ctx, const uint8_t* a_img, uint32_t a_bytes, const uint8_t* b_img, uint32_t b_bytes, uint32_t a_lbo, uint32_t a_sbo, uint32_t b_lbo, uint32_t b_sbo, uint32_t a_step_bytes, uint32_t b_step_bytes, uint32_t k_steps, uint32_t idesc, uint32_t n, int32_t* d_out_host) {
  if (!ctx) {
    set_error("pl2gpu_debug_umma: null context");
    return 1;
  }
  Ctx* c = &ctx->c;
  PL2_CUDA_OK(cudaSetDevice(c->device));
  UmmaProbeParams prm;
  prm.a_bytes = a_bytes;
  prm.b_bytes = b_bytes;
  prm.b_smem_off = RoundUpU32(a_bytes, 1024);
  if (prm.b_smem_off + b_bytes + 1024 > kProbeSmemBytes || n > 256 || (n & 15)) {
    set_error("pl2gpu_debug_umma: images too large or bad n");
    return 1;
  }
  prm.a_lbo = a_lbo;
  prm.a_sbo = a_sbo;
  prm.b_lbo = b_lbo;
  prm.b_sbo = b_sbo;
  prm.a_step_bytes = a_step_bytes;
  prm.b_step_bytes = b_step_bytes;
  prm.k_steps = k_steps;
  prm.idesc = idesc;
  prm.n = n;
  uint8_t *d_a = nullptr, *d_b = nullptr;
  int32_t* d_d = nullptr;
  PL2_CUDA_OK(cudaMalloc(&d_a, a_bytes));
  PL2_CUDA_OK(cudaMalloc(&d_b, b_bytes));
  PL2_CUDA_OK(cudaMalloc(&d_d, 128ull * n * 4));
  PL2_CUDA_OK(cudaMemcpyAsync(d_a, a_img, a_bytes, cudaMemcpyHostToDevice, c->stream));
  PL2_CUDA_OK(cudaMemcpyAsync(d_b, b_img, b_bytes, cudaMemcpyHostToDevice, c->stream));
  umma_probe_kernel<<<1, 128, kProbeSmemBytes, c->stream>>>(d_a, d_b, prm, d_d);
  c->launches++;
  PL2_CUDA_OK(cudaGetLastError());
  PL2_CUDA_OK(cudaMemcpyAsync(d_out_host, d_d, 128ull * n * 4, cudaMemcpyDeviceToHost, c->stream));
  PL2_CUDA_OK(cudaStreamSynchronize(c->stream));
  cudaFree(d_a);
  cudaFree(d_b);
  cudaFree(d_d);
  return 0;
}

// kind::mxf4 checks behind king_ts_kernel (umma_probe.cuh):
//  * layout: random 0/+-1 operands, M = 128, N = 160, two k-steps of K = 64; A rows in tensor memory with element k
//    in nibble k % 2 (low first) of byte k / 2, B K-major in king_ts_kernel's core-matrix arrangement (K chunk of
//    32 at kTsLboJ-style stride, 8-sample groups at kCoreBytes), unit scales at tensor-memory columns [496, 512);
//  * precision: the F32 accumulator must add single +-1 products exactly once it has passed 2^20, the largest count
//    one launch can reach.
static int SelftestMxf4(Pl2GpuCtx* ctx, int verbose) {
  Ctx* c = &ctx->c;
  PL2_CUDA_OK(cudaFuncSetAttribute(umma_probe_mxf4_ts_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kProbeSmemBytes));
  PL2_CUDA_OK(cudaFuncSetAttribute(umma_mxf4_exact_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kProbeSmemBytes));
  constexpr uint32_t M = 128, N = 160, KS = 2, K = 64 * KS;
  constexpr uint32_t lbo = (N / 8) * kCoreBytes + 64, step = 2 * lbo;
  std::vector<int> av(M * K), bv(N * K);
  uint32_t seed = 4242;
  auto rnd = [&]() {
    seed = seed * 1664525u + 1013904223u;
    return static_cast<int>((seed >> 24) % 3) - 1;
  };
  auto nib = [](int v) -> uint32_t { return v == 0 ? 0u : (v > 0 ? 0x2u : 0xAu); };
  for (auto& x : av) x = rnd();
  for (auto& x : bv) x = rnd();
  std::vector<uint8_t> a_rows(M * K / 2, 0), b(KS * step, 0);
  for (uint32_t m = 0; m < M; ++m)
    for (uint32_t k = 0; k < K; ++k) a_rows[m * (K / 2) + k / 2] |= nib(av[m * K + k]) << (4 * (k & 1));
  for (uint32_t n = 0; n < N; ++n)
    for (uint32_t k = 0; k < K; ++k) {
      const uint32_t off = (k / 64) * step + ((k % 64) / 32) * lbo + (n / 8) * kCoreBytes + (n % 8) * 16 + (k % 32) / 2;
      b[off] |= nib(bv[n * K + k]) << (4 * (k & 1));
    }
  UmmaProbeParams prm{};
  prm.b_bytes = static_cast<uint32_t>(b.size());
  prm.b_lbo = lbo;
  prm.b_sbo = kCoreBytes;
  prm.b_step_bytes = step;
  prm.k_steps = KS;
  prm.idesc = make_idesc_mxf4(M, N);
  prm.n = N;
  uint8_t *d_a = nullptr, *d_b = nullptr;
  uint32_t* d_d = nullptr;
  std::vector<uint32_t> d(M * N);
  PL2_CUDA_OK(cudaMalloc(&d_a, a_rows.size()));
  PL2_CUDA_OK(cudaMalloc(&d_b, b.size()));
  PL2_CUDA_OK(cudaMalloc(&d_d, d.size() * 4));
  PL2_CUDA_OK(cudaMemcpyAsync(d_a, a_rows.data(), a_rows.size(), cudaMemcpyHostToDevice, c->stream));
  PL2_CUDA_OK(cudaMemcpyAsync(d_b, b.data(), b.size(), cudaMemcpyHostToDevice, c->stream));
  umma_probe_mxf4_ts_kernel<<<1, 128, kProbeSmemBytes, c->stream>>>(d_a, d_b, prm, d_d);
  c->launches++;
  PL2_CUDA_OK(cudaGetLastError());
  PL2_CUDA_OK(cudaMemcpyAsync(d.data(), d_d, d.size() * 4, cudaMemcpyDeviceToHost, c->stream));
  PL2_CUDA_OK(cudaStreamSynchronize(c->stream));
  uint32_t bad = 0;
  for (uint32_t m = 0; m < M; ++m)
    for (uint32_t n = 0; n < N; ++n) {
      int ref = 0;
      for (uint32_t k = 0; k < K; ++k) ref += av[m * K + k] * bv[n * K + k];
      float got;
      memcpy(&got, &d[m * N + n], 4);
      if (got != static_cast<float>(ref)) {
        if (verbose && bad < 8) fprintf(stderr, "selftest_umma(mxf4) mismatch m=%u n=%u got=%g want=%d\n", m, n, got, ref);
        ++bad;
      }
    }
  // precision: 2^20 / 64 + 1 all-ones UMMAs, then five single +-1 products (umma_mxf4_exact_kernel)
  uint32_t bad_exact = 0;
  const uint32_t base = (1u << 20) / 64 + 1;
  umma_mxf4_exact_kernel<<<1, 128, kProbeSmemBytes, c->stream>>>(base, lbo, kCoreBytes, d_d);
  c->launches++;
  PL2_CUDA_OK(cudaGetLastError());
  PL2_CUDA_OK(cudaMemcpyAsync(d.data(), d_d, 128 * 16 * 4, cudaMemcpyDeviceToHost, c->stream));
  PL2_CUDA_OK(cudaStreamSynchronize(c->stream));
  for (uint32_t m = 0; m < 128; ++m)
    for (uint32_t n = 0; n < 16; ++n) {
      int64_t want = 64ll * base + 1;
      for (uint32_t j = 1; j <= 4; ++j) want += ((n >> (j - 1)) & 1) ? -1 : 1;
      float got;
      memcpy(&got, &d[m * 16 + n], 4);
      if (static_cast<double>(got) != static_cast<double>(want)) {
        if (verbose && bad_exact < 8) fprintf(stderr, "selftest_umma(mxf4 precision) m=%u n=%u got=%.1f want=%lld\n", m, n, got, static_cast<long long>(want));
        ++bad_exact;
      }
    }
  cudaFree(d_a);
  cudaFree(d_b);
  cudaFree(d_d);
  if (bad) {
    set_error("pl2gpu_selftest_umma: kind::mxf4 TS form: %u of %u accumulator entries differ from the scalar reference", bad, M * N);
    return 1;
  }
  if (bad_exact) {
    set_error("pl2gpu_selftest_umma: kind::mxf4 accumulator is not exact past 2^20 (%u of 2048 entries differ)", bad_exact);
    return 1;
  }
  return 0;
}

int pl2gpu_mxf4_peak(Pl2GpuCtx* ctx, uint32_t n_cols, double min_seconds, double* tops_out, double* seconds_out) {
  if (!ctx || !tops_out || n_cols < 16 || n_cols > 240 || (n_cols & 15)) {
    set_error("pl2gpu_mxf4_peak: bad arguments (n_cols must be a multiple of 16 in [16,240])");
    return 1;
  }
  Ctx* c = &ctx->c;
  PL2_CUDA_OK(cudaSetDevice(c->device));
  PL2_CUDA_OK(cudaFuncSetAttribute(umma_mxf4_peak_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kProbeSmemBytes));
  cudaEvent_t e0 = nullptr, e1 = nullptr;
  PL2_CUDA_OK(cudaEventCreate(&e0));
  PL2_CUDA_OK(cudaEventCreate(&e1));
  const uint32_t blocks = 4096;  // x 32 UMMAs x 2 issuer warps
  const double ops_per_launch = 2.0 * 128 * n_cols * 64 * 32.0 * 2 * blocks * c->sm_count;
  umma_mxf4_peak_kernel<<<c->sm_count, 128, kProbeSmemBytes, c->stream>>>(n_cols, blocks);  // warm-up
  c->launches++;
  PL2_CUDA_OK(cudaStreamSynchronize(c->stream));
  double total_s = 0, total_ops = 0;
  const uint32_t per_batch = 8;
  while (total_s < min_seconds) {
    PL2_CUDA_OK(cudaEventRecord(e0, c->stream));
    for (uint32_t k = 0; k < per_batch; ++k) umma_mxf4_peak_kernel<<<c->sm_count, 128, kProbeSmemBytes, c->stream>>>(n_cols, blocks);
    c->launches += per_batch;
    PL2_CUDA_OK(cudaEventRecord(e1, c->stream));
    PL2_CUDA_OK(cudaEventSynchronize(e1));
    PL2_CUDA_OK(cudaGetLastError());
    float ms = 0;
    PL2_CUDA_OK(cudaEventElapsedTime(&ms, e0, e1));
    total_s += ms * 1e-3;
    total_ops += ops_per_launch * per_batch;
    if (min_seconds <= 0) break;
  }
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  *tops_out = total_ops / total_s / 1e12;
  if (seconds_out) *seconds_out = total_s;
  return 0;
}

int pl2gpu_selftest_umma(Pl2GpuCtx* ctx, int verbose) {
  if (getenv("PL2_UMMA_BENCH")) {  // diagnostic: tcgen05.mma issue / execution rate (umma_probe.cuh)
    Ctx* c = &ctx->c;
    long long* d_out = nullptr;
    PL2_CUDA_OK(cudaMalloc(&d_out, 64));
    PL2_CUDA_OK(cudaFuncSetAttribute(umma_issue_bench_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kProbeSmemBytes));
    const uint32_t reps = 512;
    for (uint32_t mode = 0; mode < 4; ++mode)
      for (uint32_t issuers = 1; issuers <= 2; ++issuers)
        for (uint32_t n : {80u, 160u, 224u})
          for (uint32_t ce : {0u, 1u}) {
            if (n * issuers > 448) continue;
            umma_issue_bench_kernel<<<1, 128, kProbeSmemBytes, c->stream>>>(n, reps, mode, issuers, ce, d_out);
            long long h[8] = {0};
            PL2_CUDA_OK(cudaMemcpyAsync(h, d_out, 64, cudaMemcpyDeviceToHost, c->stream));
            PL2_CUDA_OK(cudaStreamSynchronize(c->stream));
            printf("umma_bench style=%s mode=%s issuers=%u n=%3u commit_every=%u: issue %.1f clk/mma, complete %.1f clk/mma (floor %.0f)\n", (mode >> 1) ? "elect" : "lane0", (mode & 1) ? "TS" : "SS", issuers, n, ce, double(h[0]) / reps, double(h[1]) / reps, n / 2.0 * issuers);
          }
    cudaFree(d_out);
  }
  // Production operand layout (geno_expand.cuh operand_offset), M=128, N=96, K=64 (two k-steps).
  const uint32_t M = 128, N = 96, K = 64;
  const uint32_t lbo_a = operand_lbo(M), lbo_b = operand_lbo(N);
  std::vector<uint8_t> a(M * K), b(N * K);
  std::vector<int8_t> av(M * K), bv(N * K);
  uint32_t seed = 12345;
  auto rnd = [&]() {
    seed = seed * 1664525u + 1013904223u;
    return static_cast<int8_t>((seed >> 24) % 7) - 3;
  };
  for (uint32_t m = 0; m < M; ++m)
    for (uint32_t k = 0; k < K; ++k) {
      const int8_t v = rnd();
      av[m * K + k] = v;
      a[operand_offset(k, m / 16, lbo_a) + (m % 16)] = static_cast<uint8_t>(v);
    }
  for (uint32_t n = 0; n < N; ++n)
    for (uint32_t k = 0; k < K; ++k) {
      const int8_t v = rnd();
      bv[n * K + k] = v;
      b[operand_offset(k, n / 16, lbo_b) + (n % 16)] = static_cast<uint8_t>(v);
    }
  std::vector<int32_t> d(128 * N);
  const uint32_t idesc = make_idesc_i8(M, N, true, true);
  PL2_TRY(pl2gpu_debug_umma(ctx, a.data(), M * K, b.data(), N * K, lbo_a, kCoreBytes, lbo_b, kCoreBytes, 4 * lbo_a, 4 * lbo_b, K / 32, idesc, N, d.data()));
  uint32_t bad = 0;
  for (uint32_t m = 0; m < M; ++m)
    for (uint32_t n = 0; n < N; ++n) {
      int32_t ref = 0;
      for (uint32_t k = 0; k < K; ++k) ref += static_cast<int32_t>(av[m * K + k]) * bv[n * K + k];
      if (ref != d[m * N + n]) {
        if (verbose && bad < 8) fprintf(stderr, "selftest_umma mismatch m=%u n=%u got=%d want=%d\n", m, n, d[m * N + n], ref);
        ++bad;
      }
    }
  if (bad) {
    set_error("pl2gpu_selftest_umma: %u of %u accumulator entries differ from the scalar reference", bad, M * N);
    return 1;
  }
  // TS form: same B image, A rows written to tensor memory with tcgen05.st (K-major, 4 K-bytes per column)
  {
    Ctx* c = &ctx->c;
    std::vector<uint8_t> a_rows(M * K);
    for (uint32_t m = 0; m < M; ++m)
      for (uint32_t k = 0; k < K; ++k) a_rows[m * K + k] = static_cast<uint8_t>(av[m * K + k]);
    UmmaProbeParams prm{};
    prm.b_bytes = N * K;
    prm.b_lbo = lbo_b;
    prm.b_sbo = kCoreBytes;
    prm.b_step_bytes = 4 * lbo_b;
    prm.k_steps = K / 32;
    prm.idesc = make_idesc_i8(M, N, false, true);
    prm.n = N;
    uint8_t *d_a = nullptr, *d_b = nullptr;
    int32_t* d_d = nullptr;
    PL2_CUDA_OK(cudaMalloc(&d_a, M * K));
    PL2_CUDA_OK(cudaMalloc(&d_b, N * K));
    PL2_CUDA_OK(cudaMalloc(&d_d, 128ull * N * 4));
    PL2_CUDA_OK(cudaMemcpyAsync(d_a, a_rows.data(), M * K, cudaMemcpyHostToDevice, c->stream));
    PL2_CUDA_OK(cudaMemcpyAsync(d_b, b.data(), N * K, cudaMemcpyHostToDevice, c->stream));
    umma_probe_ts_kernel<<<1, 128, kProbeSmemBytes, c->stream>>>(d_a, d_b, prm, d_d);
    c->launches++;
    PL2_CUDA_OK(cudaGetLastError());
    PL2_CUDA_OK(cudaMemcpyAsync(d.data(), d_d, 128ull * N * 4, cudaMemcpyDeviceToHost, c->stream));
    PL2_CUDA_OK(cudaStreamSynchronize(c->stream));
    cudaFree(d_a);
    cudaFree(d_b);
    cudaFree(d_d);
    bad = 0;
    for (uint32_t m = 0; m < M; ++m)
      for (uint32_t n = 0; n < N; ++n) {
        int32_t ref = 0;
        for (uint32_t k = 0; k < K; ++k) ref += static_cast<int32_t>(av[m * K + k]) * bv[n * K + k];
        if (ref != d[m * N + n]) {
          if (verbose && bad < 8) fprintf(stderr, "selftest_umma(TS) mismatch m=%u n=%u got=%d want=%d\n", m, n, d[m * N + n], ref);
          ++bad;
        }
      }
    if (bad) {
      set_error("pl2gpu_selftest_umma: TS form: %u of %u accumulator entries differ from the scalar reference", bad, M * N);
      return 3;
    }
  }
  PL2_TRY(SelftestMxf4(ctx, verbose));
  return 0;
}

}  // extern "C"
