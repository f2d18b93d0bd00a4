// opb_api.cu -- C ABI of libopb.so (see include/opb.h).  Host-side orchestration of the
// sm_100a kernels: weight repacking, activation buffers, TMA tensor maps, the 92-conv chain of
// models/CocoPoseNet.py:132-262 as ~60 launches, and the post-process of
// pose_detector.py:501-517.  No CPU compute fallback exists in this file.
#include <cuda.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <dlfcn.h>

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <string>
#include <queue>
#include <vector>

#include "../../include/opb.h"
#include "conv_first.cuh"
#include "conv_mlp2.cuh"
#include "ingest.cuh"
#include "overlay.cuh"
#include "keypoints.cuh"
#include "conv_tcgen05.cuh"
#include "conv_tcgen05_pair.cuh"
#include "conv_tcgen05_swap.cuh"
#include "conv_tcgen05_swap7.cuh"
#include "paf.cuh"
#include "peaks.cuh"
#include "peaks_sep.cuh"
#include "pool.cuh"
#include "upsample.cuh"

using namespace opb;

static_assert(sizeof(opb_person) == sizeof(PersonOut), "opb_person layout");
static_assert(sizeof(opb_person) == 240, "opb_person size");
static_assert(sizeof(opb_image_header) == sizeof(ImageHeader), "opb_image_header layout");

namespace {

struct OpbNcclId { char internal[128]; };   // == ncclUniqueId (passed BY VALUE to ncclCommInitRank)

thread_local std::string g_create_error;

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

struct HostLayer {
  int cin = 0, cout = 0, ks = 0;
  std::vector<float> W, b;
};

struct PackedW {          // one "B" operand: [cout_pad][ks*ks][k_per_tap] fp16
  __half* w = nullptr;
  float* bias = nullptr;  // [cout_pad]
  int cout_pad = 0, k_per_tap = 0, cin_pad = 0, ks = 0;
  float acc_scale = 1.f;  // compensated precision: 2^-S (the fp16 weights are stored pre-scaled by 2^S)
};

struct Act {              // NHWC fp16 activation tensor, channels [hi C | lo C]
  __half* p = nullptr;
  int N = 0, H = 0, W = 0, C = 0, Ctot = 0;
  size_t bytes() const { return static_cast<size_t>(N) * H * W * Ctot * sizeof(__half); }
};

enum OpKind { OP_FIRST, OP_CONV, OP_POOL, OP_MLP2 };

struct Op {
  OpKind kind;
  std::string tag;
  // OP_CONV
  int ks = 0, bn = 0, mt = 1;
  bool drain = false;
  bool pair = false;   // cta_group::2 kernel (cluster of 2 CTAs)
  bool swap = false;   // weights-as-A kernel (16x16 pixel tiles as the N=256 operand)
  int cluster = 1;     // swap kernel: CTAs per cluster sharing every weight tile through multicast TMA (1 or 2)
  bool swap7 = false;  // 7x7 swap launches use the lean-issue kernel (conv_tcgen05_swap7.cuh)
  CUtensorMap tmP16[2];
  CUtensorMap tmA[2], tmB[2];
  ConvParams P;
  Mlp2Params M;        // OP_MLP2 (fused 1x1 -> ReLU -> 1x1): tmA = input, tmB = first weights, tmP16 = second weights
  int grid = 0;
  // OP_FIRST / OP_POOL
  const __half* in = nullptr;
  __half* out = nullptr;
  int N = 0, H = 0, W = 0, C = 0, cstride = 0, lo_off = 0;
};

struct Chain {            // everything cached for one (N, H, W)
  int N = 0, H = 0, W = 0;
  std::vector<Op> ops;
  std::vector<void*> allocs;
  float* paf_lo = nullptr;   // [N][38][h][w]
  float* heat_lo = nullptr;  // [N][19][h][w]  (keypoint nets: [N][kp_out][h][w])
  uint8_t* img_u8 = nullptr;
  float* img_f32 = nullptr;
  const uint8_t* img_u8_src = nullptr;   // where conv1_1 reads uint8 frames (img_u8, or the caller's device buffer)
};

struct PostWs {           // post-process workspace for (N, map_h, map_w)
  int N = 0, H = 0, W = 0;
  float* pafs = nullptr;      // [N][38][H][W]
  float* heat = nullptr;      // [N][19][H][W]
  PeakKey* keys = nullptr;    // [N][max_peaks]
  float* tile_max = nullptr;  // cell maxima [N*18][ceil(H/8)][ceil(W/8)]
  int* peak_counts = nullptr; // [N]
  PeakD* peaks = nullptr;     // [N][max_peaks]
  int* idx_list = nullptr;
  int* type_start = nullptr;  // [N][19]
  int* status = nullptr;      // [N]
  Candidate* cands = nullptr; // [N][19][max_cand]
  Candidate* cands_alt = nullptr;  // ping-pong partner of cands for limb_assign's per-round compaction
  int* cand_counts = nullptr; // [N][19]
  Connection* conns = nullptr;  // [N][19][conn_cap]
  int* conn_counts = nullptr;
  double* subsets_out = nullptr;
  ImageHeader* headers = nullptr;
  PersonOut* persons = nullptr;
  const float* last_paf_lo = nullptr;   // low-res maps the last opb_detect_batch upsampled (network or injected)
  const float* last_heat_lo = nullptr;
  int last_h8 = 0, last_w8 = 0;         // their size
  float* sep_wy = nullptr;              // smooth_nms_sep_kernel: per-row / per-column operator records ([H][8], [W][8] floats)
  float* sep_wx = nullptr;
  int sep_h = 0, sep_w = 0;             // low-resolution size the records were built for (0: none); -1: not representable
  float* lo_stage = nullptr;            // opb_postprocess_batch: device copy of host low-res maps [N][57][h8][w8]
  size_t lo_cap = 0;                    // floats
  double last_img_len = 0;
  std::vector<void*> allocs;
};

struct KpWs {             // face / hand post-process workspace (grown on demand)
  size_t cap = 0;             // floats per buffer
  int records = 0;
  size_t stage_cap = 0;       // bytes of h_stage
  float* up = nullptr;        // upsampled maps of every crop of a chunk, [planes][h_i][w_i] back to back
  float* tmp = nullptr;       // after the axis-0 pass
  ChannelMax* res = nullptr;  // [crops][planes]
  ChannelMax* h_res = nullptr;  // pinned
  uint8_t* h_stage = nullptr;   // pinned: [crop tables | crops] of one upload
};

}  // namespace

struct opb_ctx {
  int device = 0;
  int num_sms = 148;
  cudaStream_t stream = nullptr;
  cudaStream_t own_stream = nullptr;
  opb_params prm;
  PafConsts pc;
  GaussTaps taps;
  std::string err;
  int64_t launches = 0;
  EncodeTiledFn encode = nullptr;
  int precision = -1;
  int kp_out = 0;            // 0: CocoPoseNet; 71 / 22: FaceNet / HandNet (channels of the final 1x1, incl. background)
  float u8_denom = 255.f;    // uint8 normalisation: /255 (pose_detector.py:429) or /256 (face_detector.py:32)
  KpWs* kp_ws = nullptr;
  std::map<std::string, HostLayer> host_layers;
  std::map<std::string, PackedW> packed;
  float* w_first = nullptr;  // conv1_1 [27][64] fp32
  __half* w_first_h = nullptr;  // conv1_1 [64][32] fp16 (tensor-core variant)
  __half* w_first_x = nullptr;  // conv1_1 [2][64][64] fp16: exact tensor-core variant (hi / lo of W/255 and of the -0.5*sum_c W indicator taps, x 2^S)
  float first_x_scale = 1.f;    // 2^-S
  float* b_first = nullptr;
  std::vector<void*> weight_allocs;
  std::map<long long, Chain*> chains;
  Chain* last_chain = nullptr;
  std::map<long long, PostWs*> posts;
  PostWs* last_post = nullptr;
  uint8_t* ingest_buf = nullptr;   // staging for the original frame(s) of opb_detect_image
  float* precise_mid = nullptr;    // x8 cubic intermediate of the precise path
  uint8_t* ov_buf = nullptr;       // overlay scratch: [frame in | frame out | priority plane | int poses | flag]
  size_t ov_bytes = 0;
  size_t precise_mid_cap = 0;
  size_t ingest_bytes = 0;
  // streaming mode (opb_stream_submit / opb_stream_collect): two slots, pinned staging, a copy stream
  struct StreamSlot {
    uint8_t* d_frames = nullptr; size_t d_bytes = 0;     // device copy of the submitted frames (original size)
    uint8_t* h_frames = nullptr; size_t h_bytes = 0;     // pinned staging for pageable caller buffers
    uint8_t* h_result = nullptr; size_t r_bytes = 0;     // pinned [headers | persons] of the slot
    cudaEvent_t h2d_done = nullptr, done = nullptr;
    int n = 0; bool busy = false;
    const void* post = nullptr;                          // PostWs of the submitted batch (record block of opb_allgather_results)
    // CUDA-graph replay of the slot's pipeline: the launch sequence of one (shape, buffers) combination is captured
    // the second time it is submitted and replayed afterwards
    struct Key {
      int n, oh, ow, ih, iw, mh, mw; double img_len; const void *ip, *ih_, *frames, *result, *chain, *post;
      uint64_t epoch;
      bool operator==(const Key& o) const {
        return n == o.n && oh == o.oh && ow == o.ow && ih == o.ih && iw == o.iw && mh == o.mh && mw == o.mw &&
               img_len == o.img_len && ip == o.ip && ih_ == o.ih_ && frames == o.frames && result == o.result &&
               chain == o.chain && post == o.post && epoch == o.epoch;
      }
    } key{};
    int key_seen = 0;               // consecutive submits with `key`
    cudaGraphExec_t gexec = nullptr;
    int64_t graph_launches = 0;
  } slots[2];
  cudaStream_t copy_stream = nullptr;
  int cur_slot = 0;                // streaming slot whose chain / workspace get_chain / get_post hand out
  cudaStream_t stream_b = nullptr; // compute stream of streaming slot 1 (slot 0 uses `stream`)
  uint64_t cache_epoch = 0;        // bumped whenever cached chains / workspaces / weights are freed (invalidates graphs)
  int two_streams = 1;             // OPB_TWO_STREAMS=0: both streaming slots share `stream` and one set of buffers
  int use_graphs = 1;              // OPB_GRAPH=0: streaming mode launches kernel by kernel
  // Post-process variants (A/B on a B200: profiles/r02_lowres_ab.txt; bit-exact against the oracle in every combination):
  int fused_peaks = 3;             // OPB_FUSED_PEAKS=1: the peak kernel interpolates its tiles from the low-res heat maps;
                                   // =3: candidates from the separable (bilinear o Gaussian) operator on the low-res maps (peaks_sep.cuh);
                                   // =2: materialised maps, but the tile-skip bound comes from the low-res maps (no cell_max pass)
  int paf_lowres = 1;              // OPB_PAF_LOWRES=1: PAF line integrals sample the low-res PAFs on demand
  int peaks_v2 = 0;                // OPB_PEAKS_V2=1 (with OPB_FUSED_PEAKS=2): smoothing passes spread over all 256 threads
  int conn_cap = kAssignMaxType;
  bool profile = false;                       // OPB_PROFILE=1: cudaEvent after every launch of a batch
  std::vector<std::pair<std::string, cudaEvent_t>> marks;
};

namespace {

#define OPB_CUDA(ctx, expr)                                                                       \
  do {                                                                                            \
    cudaError_t e__ = (expr);                                                                     \
    if (e__ != cudaSuccess) {                                                                     \
      (ctx)->err = std::string(#expr) + ": " + cudaGetErrorString(e__) + " (" __FILE__ ":" +      \
                   std::to_string(__LINE__) + ")";                                                \
      return OPB_ERR_CUDA;                                                                        \
    }                                                                                             \
  } while (0)

#define OPB_FAIL(ctx, code, msg) \
  do {                           \
    (ctx)->err = (msg);          \
    return (code);               \
  } while (0)

int round_up(int v, int m) { return (v + m - 1) / m * m; }

void prof_mark(opb_ctx* ctx, const std::string& name) {
  if (!ctx->profile) return;
  cudaEvent_t e;
  cudaEventCreate(&e);
  cudaEventRecord(e, ctx->stream);
  ctx->marks.emplace_back(name, e);
}

void prof_report(opb_ctx* ctx) {
  if (!ctx->profile || ctx->marks.size() < 2) return;
  cudaStreamSynchronize(ctx->stream);
  std::map<std::string, std::pair<int, float>> agg;
  std::vector<std::string> order;
  float total = 0.f;
  for (size_t i = 1; i < ctx->marks.size(); ++i) {
    float ms = 0.f;
    cudaEventElapsedTime(&ms, ctx->marks[i - 1].second, ctx->marks[i].second);
    auto& a = agg[ctx->marks[i].first];
    if (a.first == 0) order.push_back(ctx->marks[i].first);
    a.first++;
    a.second += ms;
    total += ms;
  }
  fprintf(stderr, "[opb profile] total %.3f ms\n", total);
  for (auto& k : order) fprintf(stderr, "[opb profile] %-16s n=%3d %9.3f ms %5.1f%%\n", k.c_str(), agg[k].first, agg[k].second, 100.f * agg[k].second / total);
  for (auto& m : ctx->marks) cudaEventDestroy(m.second);
  ctx->marks.clear();
}

template <typename T>
int dev_alloc(opb_ctx* ctx, T** p, size_t count, std::vector<void*>& owner, bool zero = true) {
  void* q = nullptr;
  OPB_CUDA(ctx, cudaMalloc(&q, std::max<size_t>(count * sizeof(T), 256)));
  if (zero) OPB_CUDA(ctx, cudaMemsetAsync(q, 0, std::max<size_t>(count * sizeof(T), 256), ctx->stream));
  owner.push_back(q);
  *p = static_cast<T*>(q);
  return OPB_OK;
}

void free_all(std::vector<void*>& v) {
  for (void* p : v) cudaFree(p);
  v.clear();
}

// ------------------------------------------------------------------ tensor maps
int make_act_map(opb_ctx* ctx, CUtensorMap* tm, const Act& a, int coff, int ks, int box_w = 8) {
  cuuint64_t dims[4] = {static_cast<cuuint64_t>(a.Ctot - coff), static_cast<cuuint64_t>(a.W),
                        static_cast<cuuint64_t>(a.H), static_cast<cuuint64_t>(a.N)};
  cuuint64_t strides[3] = {static_cast<cuuint64_t>(a.Ctot) * 2, static_cast<cuuint64_t>(a.W) * a.Ctot * 2,
                           static_cast<cuuint64_t>(a.H) * a.W * a.Ctot * 2};
  cuuint32_t box[4] = {64, static_cast<cuuint32_t>(box_w), static_cast<cuuint32_t>(16 + ks - 1), 1};
  cuuint32_t estr[4] = {1, 1, 1, 1};
  CUresult r = ctx->encode(tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 4, a.p + coff, dims, strides, box, estr,
                           CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                           CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) OPB_FAIL(ctx, OPB_ERR_CUDA, "cuTensorMapEncodeTiled(activation) failed: " + std::to_string(r));
  return OPB_OK;
}

int make_w_map(opb_ctx* ctx, CUtensorMap* tm, const PackedW& w, int bn) {
  const cuuint64_t ktot = static_cast<cuuint64_t>(w.ks) * w.ks * w.k_per_tap;
  cuuint64_t dims[2] = {ktot, static_cast<cuuint64_t>(w.cout_pad)};
  cuuint64_t strides[1] = {ktot * 2};
  cuuint32_t box[2] = {64, static_cast<cuuint32_t>(bn)};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = ctx->encode(tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, w.w, dims, strides, box, estr,
                           CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                           CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) OPB_FAIL(ctx, OPB_ERR_CUDA, "cuTensorMapEncodeTiled(weights) failed: " + std::to_string(r));
  return OPB_OK;
}

// ------------------------------------------------------------------ conv launch
template <int KS, int BN, int MT, int NSA, int NSB, int ACC, bool DRAIN = false, bool BRES = false>
int launch_conv_t(opb_ctx* ctx, const Op& op) {
  using Cfg = ConvCfg<KS, BN, MT, NSA, NSB, ACC>;
  auto kern = conv_tcgen05_kernel<KS, BN, MT, NSA, NSB, ACC, DRAIN, BRES>;
  static bool attr_set[64] = {};
  if (!attr_set[ctx->device & 63]) {
    OPB_CUDA(ctx, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM_BYTES));
    attr_set[ctx->device & 63] = true;
  }
  kern<<<op.grid, DRAIN ? kConvThreads : kConvThreads2, Cfg::SMEM_BYTES, ctx->stream>>>(op.tmA[0], op.tmB[0], op.tmA[1], op.tmB[1], op.P);
  ctx->launches++;
  OPB_CUDA(ctx, cudaGetLastError());
  return OPB_OK;
}

template <int KS, int BN, int MT, int NSA, int NSB, int ACC, bool DRAIN = false>
int launch_conv_pair_t(opb_ctx* ctx, const Op& op) {
  using Cfg = ConvPairCfg<KS, BN, MT, NSA, NSB, ACC>;
  auto kern = conv_tcgen05_pair_kernel<KS, BN, MT, NSA, NSB, ACC, DRAIN>;
  static bool attr_set[64] = {};
  if (!attr_set[ctx->device & 63]) {
    OPB_CUDA(ctx, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM_BYTES));
    attr_set[ctx->device & 63] = true;
  }
  kern<<<op.grid, DRAIN ? kPairDrainThreads : kConvThreads2, Cfg::SMEM_BYTES, ctx->stream>>>(op.tmA[0], op.tmB[0], op.tmA[1], op.tmB[1], op.P);
  ctx->launches++;
  OPB_CUDA(ctx, cudaGetLastError());
  return OPB_OK;
}

template <int KS, int NSP, int NSW, bool DRAIN = false, int CL = 1>
int launch_conv_swap_t(opb_ctx* ctx, const Op& op) {
  using Cfg = ConvSwapCfg<KS, NSP, NSW>;
  auto kern = conv_tcgen05_swap_kernel<KS, NSP, NSW, DRAIN, CL>;
  static bool attr_set[64] = {};
  if (!attr_set[ctx->device & 63]) {
    OPB_CUDA(ctx, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM_BYTES));
    attr_set[ctx->device & 63] = true;
  }
  kern<<<op.grid, DRAIN ? kSwapDrainThreads : kConvThreads, Cfg::SMEM_BYTES, ctx->stream>>>(
      op.tmP16[0], op.tmA[0], op.tmB[0], op.tmP16[1], op.tmA[1], op.tmB[1], op.P);
  ctx->launches++;
  OPB_CUDA(ctx, cudaGetLastError());
  return OPB_OK;
}

template <bool COMP, bool DRAIN>
int launch_conv_swap7_t(opb_ctx* ctx, const Op& op) {
  using Cfg = ConvSwap7Cfg;
  auto kern = conv_tcgen05_swap7_kernel<COMP, DRAIN>;
  static bool attr_set[64] = {};
  if (!attr_set[ctx->device & 63]) {
    OPB_CUDA(ctx, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM_BYTES));
    attr_set[ctx->device & 63] = true;
  }
  kern<<<op.grid, DRAIN ? kSwapDrainThreads : kConvThreads, Cfg::SMEM_BYTES, ctx->stream>>>(
      op.tmP16[0], op.tmA[0], op.tmB[0], op.tmP16[1], op.tmA[1], op.tmB[1], op.P);
  ctx->launches++;
  OPB_CUDA(ctx, cudaGetLastError());
  return OPB_OK;
}

int launch_conv(opb_ctx* ctx, const Op& op) {
  const int key = op.ks * 10000 + op.bn * 10 + op.mt;
  if (op.swap) {
    if (op.ks == 7 && op.cluster != 2 && op.swap7) {   // lean-issue variant (conv_tcgen05_swap7.cuh); OPB_SWAP7=0 disables
      if (op.P.comp) return op.drain ? launch_conv_swap7_t<true, true>(ctx, op) : launch_conv_swap7_t<true, false>(ctx, op);
      return op.drain ? launch_conv_swap7_t<false, true>(ctx, op) : launch_conv_swap7_t<false, false>(ctx, op);
    }
    if (op.ks == 7 && op.cluster == 2)
      return op.drain ? launch_conv_swap_t<7, 3, 5, true, 2>(ctx, op) : launch_conv_swap_t<7, 3, 5, false, 2>(ctx, op);
    if (op.ks == 7) return op.drain ? launch_conv_swap_t<7, 3, 5, true>(ctx, op) : launch_conv_swap_t<7, 3, 5>(ctx, op);
    if (op.ks == 3) return op.drain ? launch_conv_swap_t<3, 3, 6, true>(ctx, op) : launch_conv_swap_t<3, 3, 6>(ctx, op);
    OPB_FAIL(ctx, OPB_ERR_UNSUPPORTED, "no swap-mode conv variant");
  }
  if (op.pair) {    // CTA-pair kernels (fast precision)
    switch (key) {
      case 7 * 10000 + 128 * 10 + 2: return launch_conv_pair_t<7, 128, 2, 3, 6, 2>(ctx, op);
      case 7 * 10000 + 128 * 10 + 1: return launch_conv_pair_t<7, 128, 1, 4, 8, 2>(ctx, op);
      case 7 * 10000 + 256 * 10 + 1:
        return op.drain ? launch_conv_pair_t<7, 256, 1, 4, 6, 2, true>(ctx, op) : launch_conv_pair_t<7, 256, 1, 4, 6, 2>(ctx, op);
      case 3 * 10000 + 128 * 10 + 2: return launch_conv_pair_t<3, 128, 2, 3, 6, 2>(ctx, op);
      case 3 * 10000 + 256 * 10 + 1: return launch_conv_pair_t<3, 256, 1, 4, 6, 2>(ctx, op);
      case 3 * 10000 + 64 * 10 + 2: return launch_conv_pair_t<3, 64, 2, 3, 6, 2>(ctx, op);
      case 1 * 10000 + 128 * 10 + 1: return launch_conv_pair_t<1, 128, 1, 4, 6, 2>(ctx, op);
      case 1 * 10000 + 256 * 10 + 1: return launch_conv_pair_t<1, 256, 1, 4, 6, 2>(ctx, op);
      default: OPB_FAIL(ctx, OPB_ERR_UNSUPPORTED, "no pair-mode conv variant for key " + std::to_string(key));
    }
  }
  if (op.drain) {   // parity precision: two-level accumulation variants (BN <= 128, MT = 1)
    switch (key) {
      case 7 * 10000 + 128 * 10 + 1: return launch_conv_t<7, 128, 1, 3, 6, 2, true>(ctx, op);
      case 7 * 10000 + 64 * 10 + 1: return launch_conv_t<7, 64, 1, 3, 6, 2, true>(ctx, op);
      case 7 * 10000 + 48 * 10 + 1: return launch_conv_t<7, 48, 1, 3, 6, 2, true>(ctx, op);
      case 3 * 10000 + 128 * 10 + 1: return launch_conv_t<3, 128, 1, 3, 6, 2, true>(ctx, op);
      case 3 * 10000 + 64 * 10 + 1: return launch_conv_t<3, 64, 1, 3, 6, 2, true>(ctx, op);
      case 3 * 10000 + 48 * 10 + 1: return launch_conv_t<3, 48, 1, 3, 6, 2, true>(ctx, op);
      case 1 * 10000 + 128 * 10 + 1: return launch_conv_t<1, 128, 1, 4, 6, 2, true>(ctx, op);
      case 1 * 10000 + 64 * 10 + 1: return launch_conv_t<1, 64, 1, 4, 6, 2, true>(ctx, op);
      case 1 * 10000 + 48 * 10 + 1: return launch_conv_t<1, 48, 1, 4, 6, 2, true>(ctx, op);
      default: OPB_FAIL(ctx, OPB_ERR_UNSUPPORTED, "no drain-mode conv variant for key " + std::to_string(key));
    }
  }
  switch (key) {
    case 7 * 10000 + 128 * 10 + 1: return launch_conv_t<7, 128, 1, 3, 6, 2>(ctx, op);
    case 7 * 10000 + 128 * 10 + 2: return launch_conv_t<7, 128, 2, 3, 5, 2>(ctx, op);
    case 7 * 10000 + 256 * 10 + 1: return launch_conv_t<7, 256, 1, 3, 4, 2>(ctx, op);
    case 3 * 10000 + 64 * 10 + 1: return launch_conv_t<3, 64, 1, 3, 6, 2>(ctx, op);
    case 3 * 10000 + 64 * 10 + 2:
      // conv1_2 (64->64): the 72 KB weight matrix stays resident in shared memory (9 stages, one per tap)
      if (op.P.n_pairs == 1 && op.P.n_problems == 1 && op.P.n_blocks == 1 && !(getenv("OPB_NO_BRES") && atoi(getenv("OPB_NO_BRES"))))
        return launch_conv_t<3, 64, 2, 3, 9, 2, false, true>(ctx, op);
      return launch_conv_t<3, 64, 2, 3, 6, 2>(ctx, op);
    case 7 * 10000 + 64 * 10 + 2: return launch_conv_t<7, 64, 2, 3, 6, 2>(ctx, op);
    case 3 * 10000 + 128 * 10 + 1: return launch_conv_t<3, 128, 1, 3, 6, 2>(ctx, op);
    case 3 * 10000 + 128 * 10 + 2: return launch_conv_t<3, 128, 2, 3, 6, 2>(ctx, op);
    case 3 * 10000 + 256 * 10 + 1: return launch_conv_t<3, 256, 1, 3, 4, 2>(ctx, op);
    case 1 * 10000 + 128 * 10 + 1: return launch_conv_t<1, 128, 1, 4, 6, 2>(ctx, op);
    case 1 * 10000 + 256 * 10 + 1: return launch_conv_t<1, 256, 1, 4, 4, 2>(ctx, op);
    case 1 * 10000 + 48 * 10 + 1: return launch_conv_t<1, 48, 1, 4, 6, 2>(ctx, op);
    case 3 * 10000 + 48 * 10 + 1: return launch_conv_t<3, 48, 1, 3, 6, 2>(ctx, op);
    case 7 * 10000 + 48 * 10 + 1: return launch_conv_t<7, 48, 1, 3, 6, 2>(ctx, op);
    case 7 * 10000 + 64 * 10 + 1: return launch_conv_t<7, 64, 1, 3, 6, 2>(ctx, op);
    case 1 * 10000 + 64 * 10 + 1: return launch_conv_t<1, 64, 1, 4, 6, 2>(ctx, op);
    default: OPB_FAIL(ctx, OPB_ERR_UNSUPPORTED, "no conv kernel variant for ks/bn/mt key " + std::to_string(key));
  }
}

int launch_op(opb_ctx* ctx, const Chain* ch, const Op& op) {
  if (op.kind == OP_CONV) return launch_conv(ctx, op);
  if (op.kind == OP_MLP2) {
    static bool attr_set[64] = {};
    if (!attr_set[ctx->device & 63]) {
      OPB_CUDA(ctx, cudaFuncSetAttribute(conv_mlp2_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kMlp2Smem));
      OPB_CUDA(ctx, cudaFuncSetAttribute(conv_mlp2_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kMlp2SmemComp));
      attr_set[ctx->device & 63] = true;
    }
    if (op.M.corr_off)   // compensated precision
      conv_mlp2_kernel<true><<<op.grid, 128, kMlp2SmemComp, ctx->stream>>>(op.tmA[0], op.tmB[0], op.tmP16[0], op.tmA[1], op.tmB[1],
                                                                          op.tmP16[1], op.M);
    else
      conv_mlp2_kernel<false><<<op.grid, 128, kMlp2Smem, ctx->stream>>>(op.tmA[0], op.tmB[0], op.tmP16[0], op.tmA[1], op.tmB[1],
                                                                       op.tmP16[1], op.M);
    ctx->launches++;
    OPB_CUDA(ctx, cudaGetLastError());
    return OPB_OK;
  }
  if (op.kind == OP_POOL) {
    const size_t total = static_cast<size_t>(op.N) * (op.H / 2) * (op.W / 2) * (op.C / 8);
    const int grid = static_cast<int>(std::min<size_t>((total + 255) / 256, static_cast<size_t>(ctx->num_sms) * 16));
    maxpool2x2_kernel<<<grid, 256, 0, ctx->stream>>>(op.in, op.out, op.N, op.H, op.W, op.C, op.cstride, op.lo_off);
    ctx->launches++;
    OPB_CUDA(ctx, cudaGetLastError());
    return OPB_OK;
  }
  // OP_FIRST
  if (op.C == 1 && ctx->precision == OPB_PRECISION_FAST && !(getenv("OPB_NO_TC_FIRST") && atoi(getenv("OPB_NO_TC_FIRST")))) {
    const int tiles = op.N * ((op.H + 15) / 16) * ((op.W + 7) / 8);
    const int grid = std::min(tiles, ctx->num_sms * 8);
    conv_first_tc_kernel<<<grid, 128, 0, ctx->stream>>>(ch->img_u8_src ? ch->img_u8_src : ch->img_u8, ctx->w_first_h,
                                                        ctx->b_first, op.tmA[0], op.N, op.H, op.W, ctx->u8_denom);
    ctx->launches++;
    OPB_CUDA(ctx, cudaGetLastError());
    return OPB_OK;
  }
  if (op.C == 1 && ctx->precision != OPB_PRECISION_FAST && !(getenv("OPB_NO_TC_FIRST") && atoi(getenv("OPB_NO_TC_FIRST")))) {
    // uint8 frames in a precision inside the map tolerance: exact tensor-core conv1_1 (raw pixel values + in-image indicators)
    const int tiles = op.N * ((op.H + 15) / 16) * ((op.W + 7) / 8);
    const int grid = std::min(tiles, ctx->num_sms * 3);   // 3 CTAs of 66 KB per SM
    static bool attr_set[64] = {};
    if (!attr_set[ctx->device & 63]) {
      OPB_CUDA(ctx, cudaFuncSetAttribute(conv_first_tcx_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kFirstTcxSmem));
      attr_set[ctx->device & 63] = true;
    }
    conv_first_tcx_kernel<<<grid, 128, kFirstTcxSmem, ctx->stream>>>(ch->img_u8_src ? ch->img_u8_src : ch->img_u8, ctx->w_first_x, ctx->b_first,
                                                         op.tmA[0], op.N, op.H, op.W,
                                                         ctx->precision == OPB_PRECISION_COMP ? 2 : 1, ctx->first_x_scale);
    ctx->launches++;
    OPB_CUDA(ctx, cudaGetLastError());
    return OPB_OK;
  }
  const int tiles = op.N * ((op.H + CF_TH - 1) / CF_TH) * ((op.W + CF_TW - 1) / CF_TW);
  const int grid = std::min(tiles, ctx->num_sms * 8);
  conv_first_kernel<<<grid, 256, 0, ctx->stream>>>(op.C == 1 ? (ch->img_u8_src ? ch->img_u8_src : ch->img_u8) : nullptr,
                                                   op.C == 1 ? nullptr : ch->img_f32, ctx->w_first, ctx->b_first,
                                                   op.out, op.N, op.H, op.W, op.cstride, op.lo_off, ctx->u8_denom,
                                                   ctx->precision == OPB_PRECISION_COMP ? 1 : 0);
  ctx->launches++;
  OPB_CUDA(ctx, cudaGetLastError());
  return OPB_OK;
}

// ------------------------------------------------------------------ weight packing
// rows: list of (layer, n_rows_pad); cin_map[d] = reference input channel of device channel d
// (or -1 = zero).  Output [sum rows_pad][ks*ks][cin_pad * (split ? 2 : 1)].
// Compensated precision (prec == OPB_PRECISION_COMP): per tap [W_hi * 2^S : cin_pad halves][per 64-channel chunk:
// e4m3(W * 2^kW) 64 B | e4m3(W_lo * 2^S) 64 B], S = kW + 11, 2^kW * max|W| in (8, 16] (one power of two per packed matrix).
int pack_weights(opb_ctx* ctx, const std::string& key, const std::vector<std::pair<std::string, int>>& rows,
                 const std::vector<int>& cin_map, int ks, int prec) {
  const bool split = prec == OPB_PRECISION_PARITY, comp = prec == OPB_PRECISION_COMP;
  const int cin_pad = static_cast<int>(cin_map.size());
  const int kpt = cin_pad * ((split || comp) ? 2 : 1);
  int cout_pad = 0;
  for (auto& r : rows) cout_pad += r.second;
  const size_t ktot = static_cast<size_t>(ks) * ks * kpt;
  std::vector<__half> hw(static_cast<size_t>(cout_pad) * ktot, __float2half(0.f));
  std::vector<float> hb(cout_pad, 0.f);
  int kW = 0, S = 0;
  if (comp) {
    float mx = 0.f;
    for (auto& r : rows) {
      auto it = ctx->host_layers.find(r.first);
      if (it == ctx->host_layers.end()) OPB_FAIL(ctx, OPB_ERR_STATE, "weights for layer " + r.first + " were not loaded");
      for (float v : it->second.W) mx = std::max(mx, std::fabs(v));
    }
    if (mx > 0.f && std::isfinite(mx)) {
      kW = static_cast<int>(std::floor(std::log2(16.0 / static_cast<double>(mx))));
      kW = std::max(-100, std::min(100, kW));
      S = kW + 11;
    }
  }
  int row0 = 0;
  for (auto& r : rows) {
    auto it = ctx->host_layers.find(r.first);
    if (it == ctx->host_layers.end()) OPB_FAIL(ctx, OPB_ERR_STATE, "weights for layer " + r.first + " were not loaded");
    const HostLayer& L = it->second;
    if (L.ks != ks) OPB_FAIL(ctx, OPB_ERR_ARG, "ksize mismatch for " + r.first);
    for (int o = 0; o < L.cout; ++o) {
      hb[row0 + o] = L.b[o];
      for (int t = 0; t < ks * ks; ++t) {
        __half* dst = hw.data() + (static_cast<size_t>(row0 + o) * ks * ks + t) * kpt;
        for (int d = 0; d < cin_pad; ++d) {
          const int c = cin_map[d];
          if (c < 0 || c >= L.cin) continue;
          const float v = L.W[(static_cast<size_t>(o) * L.cin + c) * ks * ks + t];
          if (comp) {
            const __half hs = __float2half_rn(std::ldexp(v, S));                     // W_hi * 2^S (exact scaling)
            dst[d] = hs;
            const double lo_s = std::ldexp(static_cast<double>(v), S) - static_cast<double>(__half2float(hs));   // W_lo * 2^S
            uint8_t* cb = reinterpret_cast<uint8_t*>(dst + cin_pad) + comp_byte_off(d);
            cb[0] = f32_to_e4m3(std::ldexp(v, kW));
            cb[64] = f32_to_e4m3(static_cast<float>(lo_s));
            continue;
          }
          const __half hi = __float2half_rn(v);
          dst[d] = hi;
          if (split) dst[cin_pad + d] = __float2half_rn(v - __half2float(hi));
        }
      }
    }
    row0 += r.second;
  }
  PackedW pw;
  pw.cout_pad = cout_pad;
  pw.k_per_tap = kpt;
  pw.cin_pad = cin_pad;
  pw.ks = ks;
  pw.acc_scale = comp ? std::ldexp(1.f, -S) : 1.f;
  int rc = dev_alloc(ctx, &pw.w, hw.size(), ctx->weight_allocs, false);
  if (rc) return rc;
  rc = dev_alloc(ctx, &pw.bias, hb.size() + 64, ctx->weight_allocs, true);
  if (rc) return rc;
  OPB_CUDA(ctx, cudaMemcpyAsync(pw.w, hw.data(), hw.size() * sizeof(__half), cudaMemcpyHostToDevice, ctx->stream));
  OPB_CUDA(ctx, cudaMemcpyAsync(pw.bias, hb.data(), hb.size() * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
  OPB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));  // host vectors die here
  ctx->packed[key] = pw;
  return OPB_OK;
}

std::vector<int> identity_map(int cin, int cin_pad) {
  std::vector<int> m(cin_pad, -1);
  for (int i = 0; i < cin; ++i) m[i] = i;
  return m;
}

// ------------------------------------------------------------------ chain construction
struct ConvSpec {
  const Act* in[2];
  int in_coff[2];
  std::string wkey[2];
  const Act* out[2];
  int out_coff[2];
  int cout_valid[2];
  float* out32[2];
  int n_problems;
  int relu;
  int pool;
};

int add_conv(opb_ctx* ctx, Chain* ch, const std::string& tag, const ConvSpec& s) {
  Op op;
  op.kind = OP_CONV;
  op.tag = tag;
  const PackedW& w0 = ctx->packed.at(s.wkey[0]);
  const bool split = ctx->precision == OPB_PRECISION_PARITY;
  const bool comp = ctx->precision == OPB_PRECISION_COMP;
  op.ks = w0.ks;
  const int per_problem_cout_pad = w0.cout_pad;
  op.drain = split;
  op.bn = std::min(per_problem_cout_pad, split ? 128 : 256);
  op.mt = 1;
  {  // MT=2: two 8-column sub-tiles share every weight stage (7x7/3x3, BN=128); OPB_MT=1 disables
    const char* e = getenv("OPB_MT");
    const int want = e ? atoi(e) : 2;   // measured: 7x7 128->128 grouped launch 10.1 -> 7.9 ms with MT=2
    if (want == 2 && !split && (op.bn == 128 || op.bn == 64) && (op.ks == 7 || op.ks == 3)) op.mt = 2;
    // (conv1_2 in compensated precision with its 144 KB of main + correction weights resident in shared memory and one
    //  sub-tile per CTA was measured SLOWER than this shape, 2.45 vs 2.07 ms per batch of 32, and removed.)
  }
  const Act& a0 = *s.in[0];
  if (a0.H < 16 + op.ks - 1 || a0.W < 8)
    OPB_FAIL(ctx, OPB_ERR_UNSUPPORTED, "feature map smaller than one TMA box (min 22 x 8); image too small");
  {  // OPB_PAIR: bit mask of kernel families that run on CTA pairs (cta_group::2): 1 = 7x7, 2 = 3x3, 4 = 1x1
    const char* e = getenv("OPB_PAIR");
    const int mask = e ? atoi(e) : -1;
    const int fam = op.ks == 7 ? 1 : op.ks == 3 ? 2 : 4;
    // default (-1): only the fused Mconv1 launch (7x7, N=256): measured 2.07 -> 1.92 ms per 5 launches.
    // The N=128 families lose more to the 16-column pair granularity (82 -> 96 columns) than they gain.
    // OPB_PAIR64=1 (experiment): additionally the N=64 3x3 layers (conv1_2): a pair halves the MMA instructions per SM.
    const char* e64 = getenv("OPB_PAIR64");
    const bool pair64 = e64 && atoi(e64) && op.ks == 3 && op.bn == 64;
    const bool use_pair = pair64 || ((mask < 0) ? (op.ks == 7 && op.bn == 256) : ((mask & fam) != 0));
    if (!split && use_pair && op.bn >= 64 && op.bn != 48) {
      op.pair = true;
      if (op.bn == 256 || op.ks == 1) op.mt = 1;
      const char* d = getenv("OPB_COMP_DRAIN");   // two-level accumulation of the fused Mconv1 launch (1176 chained MMAs)
      if (comp && op.ks == 7 && op.bn == 256 && !(d && atoi(d) == 0)) op.drain = true;
    }
  }
  {  // weights-as-A kernel (N = 256-pixel tiles) for the Cout=128 7x7 layers: measured 6.63 -> 5.23 ms on the
     // 20 grouped launches (1452 TFLOP/s).  OPB_SWAP=0 disables, bit 1 also enables it for 3x3 (slower there:
     // with K = 1152 the channel-per-thread epilogue dominates).
    const char* e = getenv("OPB_SWAP");
    const int want = e ? atoi(e) : 1;
    if (want && !split && !op.pair && per_problem_cout_pad % 128 == 0 && op.bn == 128 &&
        (op.ks == 7 || (op.ks == 3 && (want & 2))) && !s.pool && !s.out32[0] && a0.W >= 16) {
      op.swap = true;
      op.mt = 1;
      // compensated precision: two-level accumulation on the long-K 7x7 layers (784 chained MMAs each; the tensor core's
      // round-toward-zero accumulate is most of the remaining map error -- profiles/r02_precision_ladder.txt).
      // OPB_COMP_DRAIN=0 disables.
      const char* d = getenv("OPB_COMP_DRAIN");
      if (comp && !(d && atoi(d) == 0)) op.drain = true;
    }
  }
  {  // Small batches (one camera frame): the throughput-optimal shapes above leave most SMs idle (a 46x62 map is 12
     // 16x16 tiles).  When the launch would fill less than half a wave, trade per-instruction efficiency for
     // parallelism: plain kernel, one 16x8 sub-tile per CTA, and halve the channel block (down to 64) while the
     // launch still fits one wave.  OPB_SMALL_BATCH=0 disables.
    const char* e = getenv("OPB_SMALL_BATCH");
    auto tiles_of = [&](bool swap, bool pair, int mt, int bn) {
      const int tw = (pair ? 16 : 8) * mt;
      int tx = (a0.W + tw - 1) / tw;
      if (swap) tx = a0.W / 16 + ((a0.W % 16) ? 1 : 0);
      return s.n_problems * (per_problem_cout_pad / bn) * a0.N * ((a0.H + 15) / 16) * tx / (pair ? 1 : 1);
    };
    const bool enabled = !(e && atoi(e) == 0);
    if (enabled && op.bn >= 64 && op.bn != 48 && tiles_of(op.swap, op.pair, op.mt, op.bn) * 2 <= ctx->num_sms) {
      op.swap = false;
      op.pair = false;
      op.mt = 1;
      if (op.bn > 128 && per_problem_cout_pad % 128 == 0 && tiles_of(false, false, 1, op.bn) * 2 <= ctx->num_sms) op.bn = 128;
      if (op.bn == 128 && !s.pool && tiles_of(false, false, 1, 128) * 2 <= ctx->num_sms) op.bn = 64;
      if (comp) {   // the plain kernel's two-level accumulation variants (BN <= 128, MT = 1) serve the long-K layers here
        const char* d = getenv("OPB_COMP_DRAIN");
        op.drain = op.bn <= 128 && op.ks == 7 && !(d && atoi(d) == 0);
      }
    }
  }
  std::memset(&op.P, 0, sizeof(op.P));
  ConvParams& P = op.P;
  P.N = a0.N; P.H = a0.H; P.W = a0.W;
  const int tile_w = (op.pair ? 16 : 8) * op.mt;
  P.tiles_x = (a0.W + tile_w - 1) / tile_w;
  if (op.swap) {
    const int rem = a0.W % 16;
    P.pad_edge8 = (rem >= 1 && rem <= 8) ? 1 : 0;
    P.tiles_x = a0.W / 16 + (rem ? 1 : 0);
  }
  P.tiles_y = (a0.H + 15) / 16;
  if (op.pair && op.mt == 1) {   // pair kernel: 8-column units paired along the linear unit order (no padding block per row)
    const char* e = getenv("OPB_PAIR_UNITS");
    const int units_x = (a0.W + 7) / 8;
    if (!(e && atoi(e) == 0) && ((static_cast<long long>(P.N) * P.tiles_y * units_x) % 2) == 0) {
      P.tiles_x = units_x;
      P.pair_units = 1;
    }
  }
  P.n_blocks = per_problem_cout_pad / op.bn;
  P.n_problems = s.n_problems;
  P.b_tap_stride = w0.k_per_tap;
  if (op.swap && op.ks == 7) {
    // OPB_SWAP_CLUSTER=2: clusters of two CTAs sharing every weight tile (multicast TMA); both CTAs of a cluster must be
    // on the same (problem, channel block), i.e. an even number of pixel tiles per block.  OFF by default: measured on a
    // B200 (profiles/r02_swap_cluster_ab.txt) it is 5 % slower in fp16 and within noise in compensated precision -- the
    // L2 already serves the 148 CTAs' identical weight requests at ~75 % of its throughput cap, and the lockstep costs more
    // than the halved request count saves.  Kept as a measured variant (bit-identical results; emulation-tested).
    const char* e = getenv("OPB_SWAP_CLUSTER");
    const int want = e ? atoi(e) : 0;
    const int m_tiles = P.N * P.tiles_y * P.tiles_x;
    if (want == 2 && m_tiles % 2 == 0 && m_tiles * P.n_blocks * P.n_problems >= 2 && ctx->num_sms >= 2) op.cluster = 2;
    const char* e7 = getenv("OPB_SWAP7");
    op.swap7 = !(e7 && atoi(e7) == 0);
  }
  const int chunks = w0.cin_pad / 64;
  int np = 0;
  for (int i = 0; i < chunks; ++i) {
    P.a_off[np] = i * 64; P.b_off[np] = i * 64; ++np;
    if (split) {
      P.a_off[np] = a0.C + i * 64; P.b_off[np] = i * 64; ++np;             // lo * Whi
      P.a_off[np] = i * 64; P.b_off[np] = w0.cin_pad + i * 64; ++np;        // hi * Wlo
    }
    if (comp) {   // odd pairs: the 128-byte 8-bit-float correction row of chunk i (addressed as 64 halves)
      P.a_off[np] = a0.C + i * 64; P.b_off[np] = w0.cin_pad + i * 64; ++np;
    }
  }
  P.comp = comp ? 1 : 0;
  {  // two-level accumulation granularity of the swap / pair DRAIN kernels: steps (chunk pair x filter column) per TMEM
     // buffer.  Default 4 (112 chained MMAs for 7x7): measured the best speed / accuracy trade (profiles/r02_precision_ladder.txt);
     // OPB_DRAIN_SEG overrides.
    const char* e = getenv("OPB_DRAIN_SEG");
    P.drain_seg = std::max(1, e ? atoi(e) : 4);
  }
  if (np > kMaxPairs) OPB_FAIL(ctx, OPB_ERR_UNSUPPORTED, "too many K chunk pairs");
  P.n_pairs = np;
  for (int p = 0; p < s.n_problems; ++p) {
    const PackedW& w = ctx->packed.at(s.wkey[p]);
    if (w.ks != op.ks || w.cout_pad != per_problem_cout_pad || w.k_per_tap != w0.k_per_tap)
      OPB_FAIL(ctx, OPB_ERR_ARG, "grouped problems must share a shape");
    if ((split || comp) && s.in[p]->C != a0.C) OPB_FAIL(ctx, OPB_ERR_ARG, "grouped problems must share the lo-plane offset");
    int rc = make_act_map(ctx, &op.tmA[p], *s.in[p], s.in_coff[p], op.ks);
    if (rc) return rc;
    if (op.swap) {
      rc = make_act_map(ctx, &op.tmP16[p], *s.in[p], s.in_coff[p], op.ks, 16);
      if (rc) return rc;
    }
    rc = make_w_map(ctx, &op.tmB[p], w, (op.pair || op.cluster == 2) ? op.bn / 2 : op.bn);
    if (rc) return rc;
    ConvProblem& pr = P.prob[p];
    pr.out = s.out[p] ? s.out[p]->p : nullptr;
    pr.out32 = s.out32[p];
    pr.bias = w.bias;
    pr.out_cstride = s.out[p] ? s.out[p]->Ctot : 0;
    pr.out_coff = s.out_coff[p];
    pr.out_lo_off = ((split || comp) && s.out[p]) ? s.out[p]->C : 0;
    pr.cout_valid = s.cout_valid[p];
    pr.relu = s.relu;
    pr.pool = s.pool;
    pr.acc_scale = w.acc_scale;
  }
  if (s.n_problems == 1) { op.tmA[1] = op.tmA[0]; op.tmB[1] = op.tmB[0]; op.tmP16[1] = op.tmP16[0]; P.prob[1] = P.prob[0]; }
  const int total_tiles = P.n_problems * P.n_blocks * P.N * P.tiles_y * P.tiles_x / (P.pair_units ? 2 : 1);
  op.grid = op.pair ? 2 * std::min(total_tiles, ctx->num_sms / 2) : std::min(total_tiles, ctx->num_sms);
  if (op.cluster == 2) op.grid = 2 * std::min(total_tiles / 2, ctx->num_sms / 2);
  {  // swap7: longest-processing-time-first tile lists per CTA (OPB_SWAP7_LPT=0: round-robin).  Cost of a tile = the
     // N of its MMAs: rows computed (16, or the even-rounded rest of the last tile row) x 16 or 8 pixels.
    const char* e = getenv("OPB_SWAP7_LPT");
    if (op.swap && op.ks == 7 && op.swap7 && op.cluster != 2 && !(e && atoi(e) == 0) && total_tiles > op.grid) {
      const int m_tiles = P.N * P.tiles_y * P.tiles_x;
      std::vector<std::pair<int, int>> tiles(total_tiles);        // (cost, tile)
      for (int t = 0; t < total_tiles; ++t) {
        const int rem = (t % m_tiles) % (P.tiles_y * P.tiles_x);
        const int ty = rem / P.tiles_x, tx = rem % P.tiles_x;
        const int rows = std::min(16, (P.H - ty * 16 + 1) & ~1);
        const bool narrow = P.pad_edge8 && tx == P.tiles_x - 1;
        tiles[t] = {rows * (narrow ? 8 : 16), t};
      }
      std::stable_sort(tiles.begin(), tiles.end(), [](const std::pair<int, int>& a, const std::pair<int, int>& b) { return a.first > b.first; });
      std::vector<std::vector<int>> lists(op.grid);
      std::vector<long long> load(op.grid, 0);
      // least-loaded CTA first; ties -> lowest index (a heap keyed by (load, index))
      std::priority_queue<std::pair<long long, int>, std::vector<std::pair<long long, int>>, std::greater<std::pair<long long, int>>> pq;
      for (int c = 0; c < op.grid; ++c) pq.push({0, c});
      for (const auto& tc : tiles) {
        auto top = pq.top(); pq.pop();
        lists[top.second].push_back(tc.second);
        pq.push({top.first + tc.first, top.second});
      }
      size_t len = 0;
      for (auto& l : lists) len = std::max(len, l.size());
      std::vector<int> flat(static_cast<size_t>(op.grid) * len, -1);
      for (int c = 0; c < op.grid; ++c) {
        std::sort(lists[c].begin(), lists[c].end());             // natural order inside a CTA (problem, image, row, column)
        std::copy(lists[c].begin(), lists[c].end(), flat.begin() + static_cast<size_t>(c) * len);
      }
      int* d_sched = nullptr;
      int rc = dev_alloc(ctx, &d_sched, flat.size(), ch->allocs, false);
      if (rc) return rc;
      OPB_CUDA(ctx, cudaMemcpyAsync(d_sched, flat.data(), flat.size() * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
      OPB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));          // `flat` dies here
      op.P.sched = d_sched;
      op.P.sched_len = static_cast<int>(len);
    }
  }
  ch->ops.push_back(op);
  return OPB_OK;
}

int alloc_act(opb_ctx* ctx, Chain* ch, Act* a, int N, int H, int W, int C) {
  a->N = N; a->H = H; a->W = W; a->C = C;
  a->Ctot = C * (ctx->precision == OPB_PRECISION_FAST ? 1 : 2);   // parity: [hi | lo] fp16; compensated: [hi fp16 | 2C correction bytes]
  return dev_alloc(ctx, &a->p, a->bytes() / sizeof(__half), ch->allocs, true);
}

int build_chain_keypoint(opb_ctx* ctx, Chain* ch, int N, int H, int W);

// Fused Mconv6 (1x1 128->128 + ReLU) -> Mconv7 (1x1 128->C, C <= 48) of one stage (csrc/conv_mlp2.cuh): fast precision by
// default, compensated precision on request.
// in: 128 channels at in_coff[p] of `in`; out: channel slice out_coff[p] of `out` (+ optional planar fp32 copy).
bool mlp2_enabled(const opb_ctx* ctx) {
  const char* e = getenv("OPB_NO_MLP2");
  if (e && atoi(e)) return false;
  if (ctx->precision == OPB_PRECISION_FAST) return true;
  // compensated precision: built and bit-identical (conv_mlp2_kernel<true>), but its 216 KB of operand + correction tiles
  // allow one CTA per SM, whose load / GEMM / epilogue phases then run back to back: measured 1.30 ms per pass vs
  // 0.38 + 0.76 ms for the two separate launches (profiles/r02_mlp2_comp_ab.txt) -> opt-in only (OPB_MLP2_COMP=1).
  const char* c = getenv("OPB_MLP2_COMP");
  return ctx->precision == OPB_PRECISION_COMP && c && atoi(c);
}

int add_mlp2(opb_ctx* ctx, Chain* ch, const std::string& tag, int n_problems, const Act& in, const int in_coff[2],
             const std::string w1[2], const std::string w2[2], const Act& out, const int out_coff[2],
             const int cout_valid[2], float* const out32[2]) {
  Op op;
  op.kind = OP_MLP2;
  op.tag = tag;
  std::memset(&op.M, 0, sizeof(op.M));
  Mlp2Params& M = op.M;
  M.N = in.N; M.H = in.H; M.W = in.W;
  M.tiles_x = (in.W + 7) / 8;
  M.tiles_y = (in.H + 15) / 16;
  M.n_problems = n_problems;
  if (in.H < 16 || in.W < 8) OPB_FAIL(ctx, OPB_ERR_UNSUPPORTED, "feature map smaller than one TMA box (16 x 8)");
  for (int p = 0; p < n_problems; ++p) {
    const PackedW& a = ctx->packed.at(w1[p]);
    const PackedW& b = ctx->packed.at(w2[p]);
    const bool comp = ctx->precision == OPB_PRECISION_COMP;
    const int kpt = comp ? 256 : 128;      // compensated precision: 128 fp16 values + 2 x 128 correction bytes per weight row
    if (a.ks != 1 || b.ks != 1 || a.cin_pad != 128 || a.cout_pad != 128 || b.cin_pad != 128 || b.cout_pad != kMlp2N2 ||
        a.k_per_tap != kpt || b.k_per_tap != kpt)
      OPB_FAIL(ctx, OPB_ERR_ARG, "fused 1x1 pair needs 128 -> 128 -> <= 48 channels");
    int rc = make_act_map(ctx, &op.tmA[p], in, in_coff[p], 1);
    if (rc) return rc;
    if ((rc = make_w_map(ctx, &op.tmB[p], a, 128))) return rc;
    if ((rc = make_w_map(ctx, &op.tmP16[p], b, kMlp2N2))) return rc;
    M.bias1[p] = a.bias;
    M.scale1[p] = a.acc_scale;
    M.corr_off = comp ? in.C : 0;          // relative to the (in_coff-shifted) tensor map, like ConvParams::a_off
    M.w_corr_off = comp ? 128 : 0;
    ConvProblem& pr = M.prob[p];
    pr.out = out.p;
    pr.out32 = out32[p];
    pr.bias = b.bias;
    pr.out_cstride = out.Ctot;
    pr.out_coff = out_coff[p];
    pr.out_lo_off = comp ? out.C : 0;
    pr.cout_valid = cout_valid[p];
    pr.relu = 0;
    pr.pool = 0;
    pr.acc_scale = b.acc_scale;
  }
  if (n_problems == 1) { op.tmA[1] = op.tmA[0]; op.tmB[1] = op.tmB[0]; op.tmP16[1] = op.tmP16[0]; M.prob[1] = M.prob[0]; M.bias1[1] = M.bias1[0]; M.scale1[1] = M.scale1[0]; }
  const int m_tiles = M.N * M.tiles_y * M.tiles_x;
  // two CTAs per SM in total (fast: 112 KB each); one in compensated precision (216 KB)
  const int per_sm = (ctx->precision == OPB_PRECISION_COMP) ? 1 : 2;
  const int per_problem = std::min(m_tiles, std::max(1, per_sm * ctx->num_sms / n_problems));
  op.grid = per_problem * n_problems;
  ch->ops.push_back(op);
  return OPB_OK;
}

int build_chain(opb_ctx* ctx, Chain* ch, int N, int H, int W) {
  if (ctx->kp_out) return build_chain_keypoint(ctx, ch, N, H, W);
  ch->N = N; ch->H = H; ch->W = W;
  const bool split = ctx->precision != OPB_PRECISION_FAST;   // two planes per activation tensor (parity: lo; compensated: correction bytes)
  const int h8 = H / 8, w8 = W / 8;
  int rc;
#define RC(x) do { rc = (x); if (rc) return rc; } while (0)
  RC(dev_alloc(ctx, &ch->img_u8, static_cast<size_t>(N) * H * W * 3, ch->allocs, false));
  RC(dev_alloc(ctx, &ch->img_f32, static_cast<size_t>(N) * H * W * 3, ch->allocs, false));
  RC(dev_alloc(ctx, &ch->paf_lo, static_cast<size_t>(N) * 38 * h8 * w8, ch->allocs, true));
  RC(dev_alloc(ctx, &ch->heat_lo, static_cast<size_t>(N) * 19 * h8 * w8, ch->allocs, true));
  // activation buffers (kept alive for the lifetime of the chain; 180 GB of HBM make reuse
  // games unnecessary at batch 32: ~4.5 GB fast, ~9 GB parity)
  Act B0, B1, P1, B2, B3, P2, B4, B5, P3, B6, B7, B8, CAT, SA, SB, S512;   // ops keep raw pointers only
  RC(alloc_act(ctx, ch, &B0, N, H, W, 64));
  RC(alloc_act(ctx, ch, &B1, N, H, W, 64));
  RC(alloc_act(ctx, ch, &P1, N, H / 2, W / 2, 64));
  RC(alloc_act(ctx, ch, &B2, N, H / 2, W / 2, 128));
  RC(alloc_act(ctx, ch, &B3, N, H / 2, W / 2, 128));
  RC(alloc_act(ctx, ch, &P2, N, H / 4, W / 4, 128));
  RC(alloc_act(ctx, ch, &B4, N, H / 4, W / 4, 256));
  RC(alloc_act(ctx, ch, &B5, N, H / 4, W / 4, 256));
  RC(alloc_act(ctx, ch, &P3, N, h8, w8, 256));
  RC(alloc_act(ctx, ch, &B6, N, h8, w8, 512));
  RC(alloc_act(ctx, ch, &B7, N, h8, w8, 512));
  RC(alloc_act(ctx, ch, &B8, N, h8, w8, 256));
  RC(alloc_act(ctx, ch, &CAT, N, h8, w8, 192));
  RC(alloc_act(ctx, ch, &SA, N, h8, w8, 256));
  RC(alloc_act(ctx, ch, &SB, N, h8, w8, 256));
  RC(alloc_act(ctx, ch, &S512, N, h8, w8, 1024));

  int first_rc = OPB_OK;
  auto first = [&]() {
    Op op; op.kind = OP_FIRST; op.tag = "conv1_1"; op.out = B0.p; op.N = N; op.H = H; op.W = W; op.C = 1;
    op.cstride = B0.Ctot; op.lo_off = split ? B0.C : 0;
    first_rc = make_act_map(ctx, &op.tmA[0], B0, 0, 1);   // output tensor map of the tensor-core conv1_1 kernels (TMA store)
    ch->ops.push_back(op);
  };
  auto pool = [&](const char* tag, const Act& in, const Act& out) {
    Op op; op.kind = OP_POOL; op.tag = tag; op.in = in.p; op.out = out.p; op.N = N; op.H = in.H; op.W = in.W;
    op.C = in.Ctot /* hi and lo planes are pooled as one channel range in fast mode */; op.cstride = in.Ctot;
    op.lo_off = split ? in.C : 0;
    if (split) op.C = in.C;
    ch->ops.push_back(op);
  };
  auto conv1 = [&](const std::string& layer, const Act& in, const Act& out, int out_coff, int cout,
                   int fuse_pool = 0) -> int {
    ConvSpec s{};
    s.in[0] = &in; s.in_coff[0] = 0; s.wkey[0] = layer; s.out[0] = &out; s.out_coff[0] = out_coff;
    s.cout_valid[0] = cout; s.out32[0] = nullptr; s.n_problems = 1; s.relu = 1; s.pool = fuse_pool;
    return add_conv(ctx, ch, layer, s);
  };
  const bool fuse = ctx->precision == OPB_PRECISION_COMP ||   // (the stand-alone pool kernel has no compensated variant)
                    !(getenv("OPB_NO_POOL_FUSION") && atoi(getenv("OPB_NO_POOL_FUSION")));   // debug knob
  auto conv2 = [&](const std::string& tag, const std::string& l1, const std::string& l2, const Act& in, int ic1,
                   int ic2, const Act& out, int oc1, int oc2, int cv1, int cv2, int relu, float* o32a,
                   float* o32b) -> int {
    ConvSpec s{};
    s.in[0] = &in; s.in[1] = &in; s.in_coff[0] = ic1; s.in_coff[1] = ic2; s.wkey[0] = l1; s.wkey[1] = l2;
    s.out[0] = &out; s.out[1] = &out; s.out_coff[0] = oc1; s.out_coff[1] = oc2; s.cout_valid[0] = cv1;
    s.cout_valid[1] = cv2; s.out32[0] = o32a; s.out32[1] = o32b; s.n_problems = 2; s.relu = relu;
    return add_conv(ctx, ch, tag, s);
  };

  first();
  if (first_rc) return first_rc;
  // F.max_pooling_2d(2,2) (models/CocoPoseNet.py:138,141,146) is fused into the producing conv's epilogue
  if (fuse) { RC(conv1("conv1_2", B0, P1, 0, 64, 1)); } else { RC(conv1("conv1_2", B0, B1, 0, 64)); pool("pool1", B1, P1); }
  RC(conv1("conv2_1", P1, B2, 0, 128));
  if (fuse) { RC(conv1("conv2_2", B2, P2, 0, 128, 1)); } else { RC(conv1("conv2_2", B2, B3, 0, 128)); pool("pool2", B3, P2); }
  RC(conv1("conv3_1", P2, B4, 0, 256));
  RC(conv1("conv3_2", B4, B5, 0, 256));
  RC(conv1("conv3_3", B5, B4, 0, 256));
  if (fuse) { RC(conv1("conv3_4", B4, P3, 0, 256, 1)); } else { RC(conv1("conv3_4", B4, B5, 0, 256)); pool("pool3", B5, P3); }
  RC(conv1("conv4_1", P3, B6, 0, 512));
  RC(conv1("conv4_2", B6, B7, 0, 512));
  RC(conv1("conv4_3_CPM", B7, B8, 0, 256));
  RC(conv1("conv4_4_CPM", B8, CAT, 0, 128));
  // stage 1 (models/CocoPoseNet.py:154-165): both branches as 2-problem grouped launches
  RC(conv2("conv5_1", "conv5_1_CPM_L1", "conv5_1_CPM_L2", CAT, 0, 0, SA, 0, 128, 128, 128, 1, nullptr, nullptr));
  RC(conv2("conv5_2", "conv5_2_CPM_L1", "conv5_2_CPM_L2", SA, 0, 128, SB, 0, 128, 128, 128, 1, nullptr, nullptr));
  RC(conv2("conv5_3", "conv5_3_CPM_L1", "conv5_3_CPM_L2", SB, 0, 128, SA, 0, 128, 128, 128, 1, nullptr, nullptr));
  RC(conv2("conv5_4", "conv5_4_CPM_L1", "conv5_4_CPM_L2", SA, 0, 128, S512, 0, 512, 512, 512, 1, nullptr, nullptr));
  RC(conv2("conv5_5", "conv5_5_CPM_L1", "conv5_5_CPM_L2", S512, 0, 512, CAT, 128, 166, 38, 19, 0, nullptr, nullptr));
  for (int st = 2; st <= 6; ++st) {
    const std::string S = "_stage" + std::to_string(st);
    {  // Mconv1: both branches read the same concat tensor -> one N=256 GEMM (:168-169,176)
      ConvSpec s{};
      s.in[0] = &CAT; s.in_coff[0] = 0; s.wkey[0] = "Mconv1" + S + "_fused"; s.out[0] = &SA; s.out_coff[0] = 0;
      s.cout_valid[0] = 256; s.n_problems = 1; s.relu = 1;
      RC(add_conv(ctx, ch, "Mconv1", s));
    }
    RC(conv2("Mconv7x7", "Mconv2" + S + "_L1", "Mconv2" + S + "_L2", SA, 0, 128, SB, 0, 128, 128, 128, 1, nullptr, nullptr));
    RC(conv2("Mconv7x7", "Mconv3" + S + "_L1", "Mconv3" + S + "_L2", SB, 0, 128, SA, 0, 128, 128, 128, 1, nullptr, nullptr));
    RC(conv2("Mconv7x7", "Mconv4" + S + "_L1", "Mconv4" + S + "_L2", SA, 0, 128, SB, 0, 128, 128, 128, 1, nullptr, nullptr));
    RC(conv2("Mconv7x7", "Mconv5" + S + "_L1", "Mconv5" + S + "_L2", SB, 0, 128, SA, 0, 128, 128, 128, 1, nullptr, nullptr));
    if (mlp2_enabled(ctx)) {   // Mconv6 + Mconv7 of both branches in one launch; the 128-channel intermediate stays on chip
      const int ic[2] = {0, 128}, oc[2] = {128, 166}, cv[2] = {38, 19};
      const std::string w1[2] = {"Mconv6" + S + "_L1", "Mconv6" + S + "_L2"}, w2[2] = {"Mconv7" + S + "_L1", "Mconv7" + S + "_L2"};
      float* const o32[2] = {st == 6 ? ch->paf_lo : nullptr, st == 6 ? ch->heat_lo : nullptr};
      RC(add_mlp2(ctx, ch, "Mconv6+7", 2, SA, ic, w1, w2, CAT, oc, cv, o32));
    } else {
      RC(conv2("Mconv6", "Mconv6" + S + "_L1", "Mconv6" + S + "_L2", SA, 0, 128, SB, 0, 128, 128, 128, 1, nullptr, nullptr));
      RC(conv2("Mconv7", "Mconv7" + S + "_L1", "Mconv7" + S + "_L2", SB, 0, 128, CAT, 128, 166, 38, 19, 0,
               st == 6 ? ch->paf_lo : nullptr, st == 6 ? ch->heat_lo : nullptr));
    }
  }
#undef RC
  return OPB_OK;
}

// FaceNet / HandNet (models/FaceNet.py:78-161, models/HandNet.py): one branch, VGG front to conv5_2, conv5_3_CPM -> 128
// features, stage 1 = two 1x1 convs, stages 2-6 on concat(previous maps, features).  Device concat layout:
// [features 0..127 | maps 128..128+kp_out-1 | 0 pad] (the Mconv1 weights are permuted to match).
int build_chain_keypoint(opb_ctx* ctx, Chain* ch, int N, int H, int W) {
  ch->N = N; ch->H = H; ch->W = W;
  const bool split = ctx->precision != OPB_PRECISION_FAST;
  const int h8 = H / 8, w8 = W / 8, KC = ctx->kp_out;
  int rc;
#define RC(x) do { rc = (x); if (rc) return rc; } while (0)
  RC(dev_alloc(ctx, &ch->img_u8, static_cast<size_t>(N) * H * W * 3, ch->allocs, false));
  RC(dev_alloc(ctx, &ch->img_f32, static_cast<size_t>(N) * H * W * 3, ch->allocs, false));
  RC(dev_alloc(ctx, &ch->paf_lo, 64, ch->allocs, true));
  RC(dev_alloc(ctx, &ch->heat_lo, static_cast<size_t>(N) * KC * h8 * w8, ch->allocs, true));
  Act B0, P1, B2, P2, B4, B5, P3, B6, B7, CAT, SA, SB, S512;
  RC(alloc_act(ctx, ch, &B0, N, H, W, 64));
  RC(alloc_act(ctx, ch, &P1, N, H / 2, W / 2, 64));
  RC(alloc_act(ctx, ch, &B2, N, H / 2, W / 2, 128));
  RC(alloc_act(ctx, ch, &P2, N, H / 4, W / 4, 128));
  RC(alloc_act(ctx, ch, &B4, N, H / 4, W / 4, 256));
  RC(alloc_act(ctx, ch, &B5, N, H / 4, W / 4, 256));
  RC(alloc_act(ctx, ch, &P3, N, h8, w8, 256));
  RC(alloc_act(ctx, ch, &B6, N, h8, w8, 512));
  RC(alloc_act(ctx, ch, &B7, N, h8, w8, 512));
  RC(alloc_act(ctx, ch, &CAT, N, h8, w8, round_up(128 + KC, 64)));
  RC(alloc_act(ctx, ch, &SA, N, h8, w8, 128));
  RC(alloc_act(ctx, ch, &SB, N, h8, w8, 128));
  RC(alloc_act(ctx, ch, &S512, N, h8, w8, 512));
  {
    Op op; op.kind = OP_FIRST; op.tag = "conv1_1"; op.out = B0.p; op.N = N; op.H = H; op.W = W; op.C = 1;
    op.cstride = B0.Ctot; op.lo_off = split ? B0.C : 0;
    RC(make_act_map(ctx, &op.tmA[0], B0, 0, 1));
    ch->ops.push_back(op);
  }
  auto conv = [&](const std::string& layer, const Act& in, const Act& out, int out_coff, int cout, int relu = 1,
                  int fuse_pool = 0, float* o32 = nullptr) -> int {
    ConvSpec s{};
    s.in[0] = &in; s.in_coff[0] = 0; s.wkey[0] = layer; s.out[0] = &out; s.out_coff[0] = out_coff;
    s.cout_valid[0] = cout; s.out32[0] = o32; s.n_problems = 1; s.relu = relu; s.pool = fuse_pool;
    return add_conv(ctx, ch, layer.rfind("Mconv", 0) == 0 ? layer.substr(0, 6) : layer, s);
  };
  RC(conv("conv1_2", B0, P1, 0, 64, 1, 1));      // max-pools (models/FaceNet.py:83,86,91) fused into the producers
  RC(conv("conv2_1", P1, B2, 0, 128));
  RC(conv("conv2_2", B2, P2, 0, 128, 1, 1));
  RC(conv("conv3_1", P2, B4, 0, 256));
  RC(conv("conv3_2", B4, B5, 0, 256));
  RC(conv("conv3_3", B5, B4, 0, 256));
  RC(conv("conv3_4", B4, P3, 0, 256, 1, 1));
  RC(conv("conv4_1", P3, B6, 0, 512));
  RC(conv("conv4_2", B6, B7, 0, 512));
  RC(conv("conv4_3", B7, B6, 0, 512));
  RC(conv("conv4_4", B6, B7, 0, 512));
  RC(conv("conv5_1", B7, B6, 0, 512));
  RC(conv("conv5_2", B6, B7, 0, 512));
  RC(conv("conv5_3_CPM", B7, CAT, 0, 128));
  RC(conv("conv6_1_CPM", CAT, S512, 0, 512));
  RC(conv("conv6_2_CPM", S512, CAT, 128, KC, 0));
  for (int st = 2; st <= 6; ++st) {
    const std::string S = "_stage" + std::to_string(st);
    RC(conv("Mconv1" + S, CAT, SA, 0, 128));
    RC(conv("Mconv2" + S, SA, SB, 0, 128));
    RC(conv("Mconv3" + S, SB, SA, 0, 128));
    RC(conv("Mconv4" + S, SA, SB, 0, 128));
    RC(conv("Mconv5" + S, SB, SA, 0, 128));
    if (mlp2_enabled(ctx) && KC <= kMlp2N2) {     // HandNet (22 maps); FaceNet's 71 maps keep the two launches
      const int ic[2] = {0, 0}, oc[2] = {128, 128}, cv[2] = {KC, KC};
      const std::string w1[2] = {"Mconv6" + S, "Mconv6" + S}, w2[2] = {"Mconv7" + S, "Mconv7" + S};
      float* const o32[2] = {st == 6 ? ch->heat_lo : nullptr, nullptr};
      RC(add_mlp2(ctx, ch, "Mconv6+7", 1, SA, ic, w1, w2, CAT, oc, cv, o32));
    } else {
      RC(conv("Mconv6" + S, SA, SB, 0, 128));
      RC(conv("Mconv7" + S, SB, CAT, 128, KC, 0, 0, st == 6 ? ch->heat_lo : nullptr));
    }
  }
#undef RC
  return OPB_OK;
}

long long shape_key(int n, int h, int w) { return (static_cast<long long>(n) << 40) | (static_cast<long long>(h) << 20) | w; }
// streaming slot 1 owns its own activations / workspaces so that the two slots can run on two streams
long long slot_key(const opb_ctx* ctx, int n, int h, int w) { return shape_key(n, h, w) | (static_cast<long long>(ctx->cur_slot) << 62); }

int get_chain(opb_ctx* ctx, int n, int h, int w, Chain** out) {
  if (ctx->precision < 0) OPB_FAIL(ctx, OPB_ERR_STATE, "opb_finalize_weights has not been called");
  if (n <= 0 || h <= 0 || w <= 0 || (h % 8) || (w % 8)) OPB_FAIL(ctx, OPB_ERR_ARG, "H and W must be positive multiples of 8");
  const long long key = slot_key(ctx, n, h, w);
  auto it = ctx->chains.find(key);
  if (it != ctx->chains.end()) { *out = it->second; ctx->last_chain = it->second; return OPB_OK; }
  // keep at most a few cached shapes (the precise path cycles through 4)
  if (ctx->chains.size() >= 10) {
    cudaDeviceSynchronize();   // both streaming slots may still be running on their chains
    for (auto& kv : ctx->chains) { free_all(kv.second->allocs); delete kv.second; }
    ctx->chains.clear();
    ctx->cache_epoch++;
    ctx->last_chain = nullptr;
  }
  Chain* ch = new Chain();
  int rc = build_chain(ctx, ch, n, h, w);
  if (rc) { free_all(ch->allocs); delete ch; return rc; }
  ctx->chains[key] = ch;
  ctx->last_chain = ch;
  *out = ch;
  return OPB_OK;
}

int run_chain(opb_ctx* ctx, Chain* ch, bool u8_input) {
  for (Op& op : ch->ops) {
    if (op.kind == OP_FIRST) op.C = u8_input ? 1 : 0;
    int rc = launch_op(ctx, ch, op);
    if (rc) return rc;
    prof_mark(ctx, op.tag);
  }
  return OPB_OK;
}

// ------------------------------------------------------------------ post-process
int get_post(opb_ctx* ctx, int n, int H, int W, PostWs** out) {
  const long long key = slot_key(ctx, n, H, W);
  auto it = ctx->posts.find(key);
  if (it != ctx->posts.end()) { *out = it->second; ctx->last_post = it->second; return OPB_OK; }
  if (ctx->posts.size() >= 6) {
    cudaDeviceSynchronize();
    for (auto& kv : ctx->posts) { free_all(kv.second->allocs); delete kv.second; }
    ctx->posts.clear();
    ctx->cache_epoch++;
    ctx->last_post = nullptr;
  }
  PostWs* ws = new PostWs();
  ws->N = n; ws->H = H; ws->W = W;
  const opb_params& p = ctx->prm;
  int rc = 0;
#define RC(x) do { rc = (x); if (rc) { free_all(ws->allocs); delete ws; return rc; } } while (0)
  RC(dev_alloc(ctx, &ws->pafs, static_cast<size_t>(n) * 38 * H * W, ws->allocs, false));
  RC(dev_alloc(ctx, &ws->heat, static_cast<size_t>(n) * 19 * H * W, ws->allocs, false));
  RC(dev_alloc(ctx, &ws->keys, static_cast<size_t>(n) * p.max_peaks, ws->allocs));
  RC(dev_alloc(ctx, &ws->tile_max, static_cast<size_t>(n) * 18 * ((H + PK_CELL - 1) / PK_CELL) * ((W + PK_CELL - 1) / PK_CELL), ws->allocs));
  RC(dev_alloc(ctx, &ws->peak_counts, n + 1, ws->allocs));     // [n] counts + the peak kernel's work counter
  RC(dev_alloc(ctx, &ws->peaks, static_cast<size_t>(n) * p.max_peaks, ws->allocs));
  RC(dev_alloc(ctx, &ws->idx_list, static_cast<size_t>(n) * p.max_peaks, ws->allocs));
  RC(dev_alloc(ctx, &ws->type_start, static_cast<size_t>(n) * 19, ws->allocs));
  RC(dev_alloc(ctx, &ws->status, n, ws->allocs));
  RC(dev_alloc(ctx, &ws->cands, static_cast<size_t>(n) * 19 * p.max_candidates, ws->allocs, false));
  RC(dev_alloc(ctx, &ws->cands_alt, static_cast<size_t>(n) * 19 * p.max_candidates, ws->allocs, false));
  RC(dev_alloc(ctx, &ws->cand_counts, static_cast<size_t>(n) * 19, ws->allocs));
  RC(dev_alloc(ctx, &ws->conns, static_cast<size_t>(n) * 19 * ctx->conn_cap, ws->allocs, false));
  RC(dev_alloc(ctx, &ws->conn_counts, static_cast<size_t>(n) * 19, ws->allocs));
  RC(dev_alloc(ctx, &ws->subsets_out, static_cast<size_t>(n) * p.max_persons * 20, ws->allocs, false));
  {  // ONE contiguous record block [n headers | n x max_persons persons]: the payload of opb_allgather_results
    static_assert(sizeof(ImageHeader) % 16 == 0, "persons must stay 16-byte aligned behind the headers");
    uint8_t* rec = nullptr;
    RC(dev_alloc(ctx, &rec, static_cast<size_t>(n) * (sizeof(ImageHeader) + sizeof(PersonOut) * p.max_persons), ws->allocs));
    ws->headers = reinterpret_cast<ImageHeader*>(rec);
    ws->persons = reinterpret_cast<PersonOut*>(rec + static_cast<size_t>(n) * sizeof(ImageHeader));
  }
#undef RC
  ctx->posts[key] = ws;
  ctx->last_post = ws;
  *out = ws;
  return OPB_OK;
}

int launch_upsample(opb_ctx* ctx, const float* in, int planes, int h, int w, float* out, int H, int W) {
  const int ppb = 19;
  dim3 block(32, 8);
  const bool v4 = (W % 4 == 0) && ((reinterpret_cast<uintptr_t>(out) & 15) == 0);
  dim3 grid(v4 ? (W + 127) / 128 : (W + 31) / 32, (H + 7) / 8, (planes + ppb - 1) / ppb);
  if (grid.z > 65535) OPB_FAIL(ctx, OPB_ERR_ARG, "too many planes");
  if (v4) upsample_bilinear_ac_v4_kernel<<<grid, block, 0, ctx->stream>>>(in, planes, h, w, out, H, W, ppb);
  else upsample_bilinear_ac_kernel<<<grid, block, 0, ctx->stream>>>(in, planes, h, w, out, H, W, ppb);
  ctx->launches++;
  OPB_CUDA(ctx, cudaGetLastError());
  return OPB_OK;
}

// One axis of the combined (align-corners bilinear upsample, then Gaussian with scipy's 'reflect' border) operator of
// csrc/peaks_sep.cuh: rec[i] = {w0..w5, first input index (int bits), 0}.  false if some output depends on more than
// PKS_TAPS inputs or the first indices are not non-decreasing (the kernel's sliding window needs both).
bool build_sep_axis(int n_in, int n_out, const GaussTaps& taps, std::vector<float>& rec) {
  if (n_in < PKS_TAPS || n_out < 1) return false;
  const int R = taps.radius;
  const double step = (n_out > 1) ? static_cast<double>(n_in - 1) / static_cast<double>(n_out - 1) : 0.0;
  rec.assign(static_cast<size_t>(n_out) * 8, 0.f);
  std::vector<double> c(n_in);
  int prev_base = 0;
  for (int i = 0; i < n_out; ++i) {
    std::fill(c.begin(), c.end(), 0.0);
    for (int j = -R; j <= R; ++j) {
      int ii = i + j;
      while (ii < 0 || ii >= n_out) { if (ii < 0) ii = -ii - 1; if (ii >= n_out) ii = 2 * n_out - 1 - ii; }
      const double u = (n_out == 1) ? 0.0 : (ii == n_out - 1) ? static_cast<double>(n_in - 1) : ii * step;
      int k = static_cast<int>(std::floor(u));
      k = std::max(0, std::min(k, n_in - 2));
      c[k] += taps.w[j + R] * (static_cast<double>(k + 1) - u);
      c[k + 1] += taps.w[j + R] * (u - static_cast<double>(k));
    }
    int lo = 0, hi = n_in - 1;
    while (lo < n_in - 1 && c[lo] == 0.0) ++lo;
    while (hi > lo && c[hi] == 0.0) --hi;
    if (hi - lo + 1 > PKS_TAPS) return false;
    int base = std::max(0, std::min(lo, n_in - PKS_TAPS));
    base = std::max(base, prev_base);                    // keep the window monotone (it still has to cover [lo, hi])
    if (base > lo || base + PKS_TAPS - 1 < hi) return false;
    prev_base = base;
    for (int k = 0; k < PKS_TAPS; ++k) rec[static_cast<size_t>(i) * 8 + k] = static_cast<float>(c[base + k]);
    std::memcpy(&rec[static_cast<size_t>(i) * 8 + 6], &base, sizeof(int));
  }
  return true;
}

// (re)builds the operator records of workspace `ws` for low-resolution size (h_lo, w_lo); *ok = usable
int ensure_sep_axes(opb_ctx* ctx, PostWs* ws, int h_lo, int w_lo, bool* ok) {
  if (ws->sep_h == h_lo && ws->sep_w == w_lo) { *ok = true; return OPB_OK; }
  if (ws->sep_h == -h_lo - 1 && ws->sep_w == -w_lo - 1) { *ok = false; return OPB_OK; }
  std::vector<float> ry, rx;
  const bool good = ctx->taps.radius == PK_R_FAST && ws->H <= 4096 && build_sep_axis(h_lo, ws->H, ctx->taps, ry) &&
                    build_sep_axis(w_lo, ws->W, ctx->taps, rx) &&
                    smooth_nms_sep_smem_bytes(ws->H, PKS_MAX_WARPS) <= 200 * 1024;
  if (!good) { ws->sep_h = -h_lo - 1; ws->sep_w = -w_lo - 1; *ok = false; return OPB_OK; }
  if (!ws->sep_wy) {
    int rc = dev_alloc(ctx, &ws->sep_wy, static_cast<size_t>(ws->H) * 8, ws->allocs, false);
    if (rc) return rc;
    if ((rc = dev_alloc(ctx, &ws->sep_wx, static_cast<size_t>(ws->W) * 8, ws->allocs, false))) return rc;
  }
  OPB_CUDA(ctx, cudaMemcpyAsync(ws->sep_wy, ry.data(), ry.size() * 4, cudaMemcpyHostToDevice, ctx->stream));
  OPB_CUDA(ctx, cudaMemcpyAsync(ws->sep_wx, rx.data(), rx.size() * 4, cudaMemcpyHostToDevice, ctx->stream));
  OPB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));   // the host vectors die here
  ws->sep_h = h_lo; ws->sep_w = w_lo;
  *ok = true;
  return OPB_OK;
}

// heat: [n][c_total][H][W]; fills ws->peaks / idx_list / type_start / peak_counts.
// h_lo > 0: `heat` is the network-resolution map [n][c_total][h_lo][w_lo] and the peak kernel interpolates its tiles
// from it (smooth_nms_lowres_kernel): the same peaks as upsampling to (H, W) first, without the full-resolution map.
// heat_full != nullptr (with h_lo > 0): the materialised maps are read as usual and only the tile-skip bound comes from the
// low-resolution maps (smooth_nms_loskip_kernel).
int launch_peaks(opb_ctx* ctx, PostWs* ws, const float* heat, int n, int c_total, int H, int W, int h_lo = 0,
                 int w_lo = 0, const float* heat_full = nullptr) {
  const opb_params& p = ctx->prm;
  OPB_CUDA(ctx, cudaMemsetAsync(ws->peak_counts, 0, sizeof(int) * (n + 1), ctx->stream));
  OPB_CUDA(ctx, cudaMemsetAsync(ws->status, 0, sizeof(int) * n, ctx->stream));
  const int c_use = c_total - 1;   // background channel dropped, pose_detector.py:78
  const size_t smem = smooth_nms_smem_bytes(ctx->taps.radius);
  // function attributes are per device: key the one-time flags by device like the conv launchers do
  static bool attr1_d[64] = {}, attr2_d[64] = {}, attr3_d[64] = {}, attr4_d[64] = {};
  bool &attr1 = attr1_d[ctx->device & 63], &attr2 = attr2_d[ctx->device & 63], &attr3 = attr3_d[ctx->device & 63],
       &attr4 = attr4_d[ctx->device & 63];
  if (!attr1) {
    OPB_CUDA(ctx, cudaFuncSetAttribute(smooth_nms_kernel<PK_R_FAST>, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024));
    OPB_CUDA(ctx, cudaFuncSetAttribute(smooth_nms_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024));
    attr1 = true;
  }
  dim3 grid((W + PK_TX - 1) / PK_TX, (H + PK_TY - 1) / PK_TY, n * c_use);
  if (grid.z > 65535) OPB_FAIL(ctx, OPB_ERR_ARG, "batch too large for the peaks grid");
  if (h_lo > 0) {
    if (!attr3) {
      OPB_CUDA(ctx, cudaFuncSetAttribute(smooth_nms_lowres_kernel<PK_R_FAST>, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024));
      OPB_CUDA(ctx, cudaFuncSetAttribute(smooth_nms_lowres_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024));
      OPB_CUDA(ctx, cudaFuncSetAttribute(smooth_nms_loskip_kernel<PK_R_FAST>, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024));
      OPB_CUDA(ctx, cudaFuncSetAttribute(smooth_nms_loskip_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024));
      attr3 = true;
    }
    if (h_lo < 2 || w_lo < 2) OPB_FAIL(ctx, OPB_ERR_ARG, "low-resolution maps need at least 2 x 2 samples");
    bool sep = false;
    if (!heat_full && ctx->fused_peaks == 3 && H == ws->H && W == ws->W) {   // separable-operator candidate search (peaks_sep.cuh)
      int rc = ensure_sep_axes(ctx, ws, h_lo, w_lo, &sep);
      if (rc) return rc;
    }
    if (sep) {
      // one block per plane; its warps pull 30-column x 32-row cells from a shared counter (no lockstep between warps)
      const int n_cells = ((W + 29) / 30) * ((H + PKS_SEG - 1) / PKS_SEG);
      const int nw = std::max(1, std::min(PKS_MAX_WARPS, n_cells));
      static bool attr5_d[64] = {};
      if (!attr5_d[ctx->device & 63]) {
        OPB_CUDA(ctx, cudaFuncSetAttribute(smooth_nms_sep_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
        attr5_d[ctx->device & 63] = true;
      }
      // persistent blocks (as many as fit: registers / 75 KB of shared memory allow 3 per SM); warps pull (plane, cell)
      // items from a global counter, so there is no tail of half-empty waves
      const long long n_items = static_cast<long long>(n) * c_use * n_cells;
      dim3 gs(static_cast<unsigned>(std::min<long long>((n_items + nw - 1) / nw, 3LL * ctx->num_sms)), 1, 1);
      SepAxes axes{ws->sep_wy, ws->sep_wx};
      smooth_nms_sep_kernel<<<gs, nw * 32, smooth_nms_sep_smem_bytes(H, nw), ctx->stream>>>(
          heat, c_total, c_use, n * c_use, h_lo, w_lo, H, W, ctx->taps, static_cast<float>(p.heatmap_peak_thresh), axes, ws->keys,
          ws->peak_counts, p.max_peaks, ws->peak_counts + n);
    } else if (heat_full && ctx->peaks_v2 && ctx->taps.radius == PK_R_FAST) {   // + both smoothing passes on all threads
      if (!attr4) {
        OPB_CUDA(ctx, cudaFuncSetAttribute(smooth_nms_loskip_kernel_v2<PK_R_FAST>, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024));
        attr4 = true;
      }
      smooth_nms_loskip_kernel_v2<PK_R_FAST><<<grid, PK_THREADS, smem, ctx->stream>>>(
          heat_full, heat, c_total, c_use, h_lo, w_lo, H, W, ctx->taps, static_cast<float>(p.heatmap_peak_thresh),
          ws->keys, ws->peak_counts, p.max_peaks);
    } else if (heat_full) {   // materialised maps, tile-skip bound from the low-resolution maps (no cell_max pass)
      if (ctx->taps.radius == PK_R_FAST)
        smooth_nms_loskip_kernel<PK_R_FAST><<<grid, PK_THREADS, smem, ctx->stream>>>(
            heat_full, heat, c_total, c_use, h_lo, w_lo, H, W, ctx->taps, static_cast<float>(p.heatmap_peak_thresh),
            ws->keys, ws->peak_counts, p.max_peaks);
      else
        smooth_nms_loskip_kernel<0><<<grid, PK_THREADS, smem, ctx->stream>>>(
            heat_full, heat, c_total, c_use, h_lo, w_lo, H, W, ctx->taps, static_cast<float>(p.heatmap_peak_thresh),
            ws->keys, ws->peak_counts, p.max_peaks);
    } else if (ctx->taps.radius == PK_R_FAST)
      smooth_nms_lowres_kernel<PK_R_FAST><<<grid, PK_THREADS, smem, ctx->stream>>>(
          heat, c_total, c_use, h_lo, w_lo, H, W, ctx->taps, static_cast<float>(p.heatmap_peak_thresh), ws->keys,
          ws->peak_counts, p.max_peaks);
    else
      smooth_nms_lowres_kernel<0><<<grid, PK_THREADS, smem, ctx->stream>>>(
          heat, c_total, c_use, h_lo, w_lo, H, W, ctx->taps, static_cast<float>(p.heatmap_peak_thresh), ws->keys,
          ws->peak_counts, p.max_peaks);
  } else {
  cell_max_kernel<<<grid, 256, 0, ctx->stream>>>(heat, c_total, c_use, H, W, ws->tile_max, (H + PK_CELL - 1) / PK_CELL,
                                                 (W + PK_CELL - 1) / PK_CELL);
  ctx->launches++;
  prof_mark(ctx, "tile_max");
  if (ctx->taps.radius == PK_R_FAST)
    smooth_nms_kernel<PK_R_FAST><<<grid, PK_THREADS, smem, ctx->stream>>>(heat, c_total, c_use, H, W, ctx->taps,
                                                                   static_cast<float>(p.heatmap_peak_thresh), ws->keys,
                                                                   ws->peak_counts, p.max_peaks, ws->tile_max);
  else
    smooth_nms_kernel<0><<<grid, PK_THREADS, smem, ctx->stream>>>(heat, c_total, c_use, H, W, ctx->taps,
                                                           static_cast<float>(p.heatmap_peak_thresh), ws->keys,
                                                           ws->peak_counts, p.max_peaks, ws->tile_max);
  }
  ctx->launches++;
  OPB_CUDA(ctx, cudaGetLastError());
  prof_mark(ctx, "smooth_nms");
  int npow = 1;
  while (npow < p.max_peaks) npow <<= 1;
  const size_t smem2 = static_cast<size_t>(npow) * 8;
  if (!attr2) {
    OPB_CUDA(ctx, cudaFuncSetAttribute(sort_peaks_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    attr2 = true;
  }
  sort_peaks_kernel<<<n, 1024, smem2, ctx->stream>>>(ws->keys, ws->peak_counts, p.max_peaks, H, W, 18, ws->peaks,
                                                     ws->idx_list, ws->type_start, ws->status);
  ctx->launches++;
  OPB_CUDA(ctx, cudaGetLastError());
  return OPB_OK;
}

// h_lo > 0: `pafs` is the network-resolution map [n][38][h_lo][w_lo]; the line integrals sample it on demand
// (paf_candidates_lowres_kernel) at the positions of the (H, W) map the reference upsamples to.
int launch_connections(opb_ctx* ctx, PostWs* ws, const float* pafs, int n, int H, int W, double img_len, int h_lo = 0,
                       int w_lo = 0) {
  const opb_params& p = ctx->prm;
  OPB_CUDA(ctx, cudaMemsetAsync(ws->cand_counts, 0, sizeof(int) * n * 19, ctx->stream));
  dim3 g1(8, 19, n);
  if (h_lo > 0) {
    if (h_lo < 2 || w_lo < 2) OPB_FAIL(ctx, OPB_ERR_ARG, "low-resolution maps need at least 2 x 2 samples");
    paf_candidates_lowres_kernel<<<g1, 128, 0, ctx->stream>>>(pafs, h_lo, w_lo, H, W, ws->peaks, ws->idx_list,
                                                              ws->type_start, p.max_peaks, 18, ctx->pc, img_len,
                                                              ws->cands, ws->cand_counts, p.max_candidates);
  } else {
  paf_candidates_kernel<<<g1, 128, 0, ctx->stream>>>(pafs, H, W, ws->peaks, ws->idx_list, ws->type_start,
                                                     p.max_peaks, 18, ctx->pc, img_len, ws->cands, ws->cand_counts,
                                                     p.max_candidates);
  }
  ctx->launches++;
  OPB_CUDA(ctx, cudaGetLastError());
  prof_mark(ctx, "paf_candidates");
  dim3 g2(19, n);
  limb_assign_kernel<<<g2, kAssignThreads, 0, ctx->stream>>>(ws->peaks, ws->idx_list, ws->type_start, p.max_peaks, 18,
                                                             ctx->pc, ws->cands, ws->cands_alt, ws->cand_counts,
                                                             p.max_candidates, ws->conns, ws->conn_counts, ctx->conn_cap,
                                                             ws->status);
  ctx->launches++;
  OPB_CUDA(ctx, cudaGetLastError());
  return OPB_OK;
}

int launch_group(opb_ctx* ctx, PostWs* ws, int n, bool with_counts) {
  // peak ids fit int16 (max_peaks <= 16384); the subset table takes 52 B of shared memory per row
  const size_t table_bytes = group_smem_bytes(ctx->prm.max_persons, ctx->prm.max_peaks);
  if (table_bytes > 48 * 1024)
    OPB_CUDA(ctx, cudaFuncSetAttribute(group_persons_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       static_cast<int>(table_bytes)));
  group_persons_kernel<<<n, 32, table_bytes, ctx->stream>>>(
      ws->peaks, with_counts ? ws->peak_counts : nullptr, ctx->prm.max_peaks, ctx->pc, ws->conns, ws->conn_counts,
      ctx->conn_cap, ctx->prm.max_persons, ws->status, ws->headers, ws->persons, ws->subsets_out);
  ctx->launches++;
  OPB_CUDA(ctx, cudaGetLastError());
  return OPB_OK;
}

int copy_in(opb_ctx* ctx, void* dst, const void* src, size_t bytes, int loc) {
  OPB_CUDA(ctx, cudaMemcpyAsync(dst, src, bytes, loc == OPB_HOST ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToDevice,
                                ctx->stream));
  return OPB_OK;
}
int copy_out(opb_ctx* ctx, void* dst, const void* src, size_t bytes, int loc) {
  OPB_CUDA(ctx, cudaMemcpyAsync(dst, src, bytes, loc == OPB_HOST ? cudaMemcpyDeviceToHost : cudaMemcpyDeviceToDevice,
                                ctx->stream));
  return OPB_OK;
}

// host peak table [n,5] float64 -> device PeakD + per-type stable index lists
int upload_peaks(opb_ctx* ctx, PostWs* ws, const double* peaks, int n_peaks) {
  if (n_peaks > ctx->prm.max_peaks) OPB_FAIL(ctx, OPB_ERR_CAPACITY, "peak table larger than opb_params.max_peaks");
  std::vector<PeakD> pk(n_peaks);
  std::vector<int> idx(n_peaks), ts(19, 0);
  std::vector<int> cnt(19, 0);
  for (int i = 0; i < n_peaks; ++i) {
    pk[i].type = static_cast<int>(peaks[i * 5 + 0]);
    pk[i].x = peaks[i * 5 + 1];
    pk[i].y = peaks[i * 5 + 2];
    pk[i].score = static_cast<float>(peaks[i * 5 + 3]);
    if (pk[i].type < 0 || pk[i].type >= 18) OPB_FAIL(ctx, OPB_ERR_ARG, "peak type out of range");
    cnt[pk[i].type + 1]++;
  }
  for (int t = 1; t < 19; ++t) ts[t] = ts[t - 1] + cnt[t];
  std::vector<int> fill(ts.begin(), ts.end());
  for (int i = 0; i < n_peaks; ++i) idx[fill[pk[i].type]++] = i;
  OPB_CUDA(ctx, cudaMemcpyAsync(ws->peaks, pk.data(), sizeof(PeakD) * n_peaks, cudaMemcpyHostToDevice, ctx->stream));
  OPB_CUDA(ctx, cudaMemcpyAsync(ws->idx_list, idx.data(), sizeof(int) * n_peaks, cudaMemcpyHostToDevice, ctx->stream));
  OPB_CUDA(ctx, cudaMemcpyAsync(ws->type_start, ts.data(), sizeof(int) * 19, cudaMemcpyHostToDevice, ctx->stream));
  OPB_CUDA(ctx, cudaMemcpyAsync(ws->peak_counts, &n_peaks, sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
  OPB_CUDA(ctx, cudaMemsetAsync(ws->status, 0, sizeof(int), ctx->stream));
  OPB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return OPB_OK;
}

}  // namespace

// ====================================================================== C ABI
extern "C" {

int opb_version(void) { return 1; }

const char* opb_last_error(const opb_ctx* ctx) { return ctx ? ctx->err.c_str() : g_create_error.c_str(); }

int opb_create(opb_ctx** out, int device, const opb_params* params) {
  if (!out || !params) { g_create_error = "null argument"; return OPB_ERR_ARG; }
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0) {
    g_create_error = std::string("no CUDA device: ") + cudaGetErrorString(e) + " (libopb has no CPU fallback)";
    return OPB_ERR_CUDA;
  }
  if (device < 0) device = 0;   // reference: device<0 means CPU; here it means GPU 0 (no CPU path)
  if (device >= ndev) { g_create_error = "device id out of range"; return OPB_ERR_ARG; }
  cudaDeviceProp prop;
  cudaGetDeviceProperties(&prop, device);
  if (prop.major != 10) {
    g_create_error = "libopb is built for sm_100a (B200) only; found sm_" + std::to_string(prop.major * 10 + prop.minor);
    return OPB_ERR_UNSUPPORTED;
  }
  if (params->n_integ_points != 10 || params->gauss_radius < 1 || params->gauss_radius > PK_R_MAX ||
      params->max_peaks < 32 || params->max_peaks > 16384 || params->max_candidates < 32 || params->max_persons < 1 || params->max_persons > 4096) {
    g_create_error = "unsupported opb_params (n_integ_points must be 10, gauss_radius 1..16, max_peaks 32..16384, max_persons 1..4096)";
    return OPB_ERR_ARG;
  }
  opb_ctx* ctx = new opb_ctx();
  ctx->device = device;
  ctx->num_sms = prop.multiProcessorCount;
  ctx->prm = *params;
  cudaSetDevice(device);
  if (cudaStreamCreateWithFlags(&ctx->own_stream, cudaStreamNonBlocking) != cudaSuccess) {
    g_create_error = "cudaStreamCreate failed";
    delete ctx;
    return OPB_ERR_CUDA;
  }
  ctx->stream = ctx->own_stream;
  void* fn = nullptr;
  cudaDriverEntryPointQueryResult qres;
  e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres);
  if (e != cudaSuccess || !fn) {
    g_create_error = "cuTensorMapEncodeTiled driver entry point not found";
    delete ctx;
    return OPB_ERR_CUDA;
  }
  ctx->encode = reinterpret_cast<EncodeTiledFn>(fn);
  std::memset(&ctx->pc, 0, sizeof(ctx->pc));
  for (int l = 0; l < 19; ++l) { ctx->pc.limbs[l][0] = params->limbs[l][0]; ctx->pc.limbs[l][1] = params->limbs[l][1]; }
  ctx->pc.inner_product_thresh = params->inner_product_thresh;
  ctx->pc.limb_length_ratio = params->limb_length_ratio;
  ctx->pc.length_penalty_value = params->length_penalty_value;
  ctx->pc.n_subset_limbs_thresh = params->n_subset_limbs_thresh;
  ctx->pc.subset_score_thresh = params->subset_score_thresh;
  ctx->pc.n_integ_points_thresh = params->n_integ_points_thresh;
  ctx->taps.radius = params->gauss_radius;
  for (int i = 0; i < 2 * params->gauss_radius + 1; ++i) ctx->taps.w[i] = params->gauss_taps[i];
  ctx->conn_cap = kAssignMaxType;
  ctx->profile = getenv("OPB_PROFILE") && atoi(getenv("OPB_PROFILE")) > 0;
  if (const char* g = getenv("OPB_GRAPH")) ctx->use_graphs = atoi(g);
  if (const char* g = getenv("OPB_TWO_STREAMS")) ctx->two_streams = atoi(g);
  if (const char* g = getenv("OPB_FUSED_PEAKS")) ctx->fused_peaks = atoi(g);
  if (const char* g = getenv("OPB_PAF_LOWRES")) ctx->paf_lowres = atoi(g);
  if (const char* g = getenv("OPB_PEAKS_V2")) ctx->peaks_v2 = atoi(g);
  *out = ctx;
  return OPB_OK;
}

void opb_destroy(opb_ctx* ctx) {
  if (!ctx) return;
  cudaSetDevice(ctx->device);
  cudaDeviceSynchronize();
  for (auto& kv : ctx->chains) { free_all(kv.second->allocs); delete kv.second; }
  for (auto& kv : ctx->posts) { free_all(kv.second->allocs); delete kv.second; }
  free_all(ctx->weight_allocs);
  if (ctx->ingest_buf) cudaFree(ctx->ingest_buf);
  if (ctx->precise_mid) cudaFree(ctx->precise_mid);
  if (ctx->ov_buf) cudaFree(ctx->ov_buf);
  if (ctx->kp_ws) {
    cudaFree(ctx->kp_ws->up); cudaFree(ctx->kp_ws->tmp); cudaFree(ctx->kp_ws->res); cudaFreeHost(ctx->kp_ws->h_res);
    cudaFreeHost(ctx->kp_ws->h_stage);
    delete ctx->kp_ws;
  }
  for (auto& sl : ctx->slots) {
    if (sl.d_frames) cudaFree(sl.d_frames);
    if (sl.h_frames) cudaFreeHost(sl.h_frames);
    if (sl.h_result) cudaFreeHost(sl.h_result);
    if (sl.gexec) cudaGraphExecDestroy(sl.gexec);
    if (sl.h2d_done) cudaEventDestroy(sl.h2d_done);
    if (sl.done) cudaEventDestroy(sl.done);
  }
  if (ctx->copy_stream) cudaStreamDestroy(ctx->copy_stream);
  if (ctx->stream_b) cudaStreamDestroy(ctx->stream_b);
  if (ctx->own_stream) cudaStreamDestroy(ctx->own_stream);
  delete ctx;
}

int opb_set_stream(opb_ctx* ctx, void* cuda_stream) {
  if (!ctx) return OPB_ERR_ARG;
  ctx->stream = cuda_stream ? static_cast<cudaStream_t>(cuda_stream) : ctx->own_stream;
  return OPB_OK;
}

int opb_synchronize(opb_ctx* ctx) {
  if (!ctx) return OPB_ERR_ARG;
  OPB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  if (ctx->stream_b) OPB_CUDA(ctx, cudaStreamSynchronize(ctx->stream_b));   // streaming slot 1
  return OPB_OK;
}

int64_t opb_launch_count(const opb_ctx* ctx) { return ctx ? ctx->launches : 0; }

int opb_load_weights(opb_ctx* ctx, const char* layer, const float* W, const int64_t shape[4], const float* b) {
  if (!ctx || !layer || !W || !shape || !b) return OPB_ERR_ARG;
  if (shape[2] != shape[3] || (shape[2] != 1 && shape[2] != 3 && shape[2] != 7))
    OPB_FAIL(ctx, OPB_ERR_ARG, std::string("unsupported kernel shape for layer ") + layer);
  HostLayer L;
  L.cout = static_cast<int>(shape[0]);
  L.cin = static_cast<int>(shape[1]);
  L.ks = static_cast<int>(shape[2]);
  const size_t n = static_cast<size_t>(L.cout) * L.cin * L.ks * L.ks;
  L.W.assign(W, W + n);
  L.b.assign(b, b + L.cout);
  ctx->host_layers[layer] = std::move(L);
  return OPB_OK;
}

int opb_finalize_weights(opb_ctx* ctx, int precision_mode) {
  if (!ctx) return OPB_ERR_ARG;
  if (precision_mode != OPB_PRECISION_FAST && precision_mode != OPB_PRECISION_PARITY && precision_mode != OPB_PRECISION_COMP)
    OPB_FAIL(ctx, OPB_ERR_ARG, "bad precision mode");
  cudaSetDevice(ctx->device);
  // drop everything derived from older weights
  OPB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  for (auto& kv : ctx->chains) { free_all(kv.second->allocs); delete kv.second; }
  ctx->chains.clear();
  ctx->cache_epoch++;
  ctx->last_chain = nullptr;
  free_all(ctx->weight_allocs);
  ctx->packed.clear();
  ctx->precision = precision_mode;
  const int split = precision_mode;   // pack_weights' precision argument
  int rc;
  // conv1_1: [27][64] fp32, k = (r*3+s)*3 + c
  {
    auto it = ctx->host_layers.find("conv1_1");
    if (it == ctx->host_layers.end()) OPB_FAIL(ctx, OPB_ERR_STATE, "weights for layer conv1_1 were not loaded");
    const HostLayer& L = it->second;
    if (L.cin != 3 || L.cout != 64 || L.ks != 3) OPB_FAIL(ctx, OPB_ERR_ARG, "conv1_1 must be 3->64, 3x3");
    std::vector<float> wt(27 * 64);
    for (int o = 0; o < 64; ++o)
      for (int c = 0; c < 3; ++c)
        for (int t = 0; t < 9; ++t) wt[(t * 3 + c) * 64 + o] = L.W[(static_cast<size_t>(o) * 3 + c) * 9 + t];
    std::vector<__half> wh(64 * 32, __float2half(0.f));
    for (int o = 0; o < 64; ++o)
      for (int c = 0; c < 3; ++c)
        for (int t = 0; t < 9; ++t) wh[o * 32 + t * 3 + c] = __float2half_rn(L.W[(static_cast<size_t>(o) * 3 + c) * 9 + t]);
    if ((rc = dev_alloc(ctx, &ctx->w_first_h, wh.size(), ctx->weight_allocs, false))) return rc;
    OPB_CUDA(ctx, cudaMemcpyAsync(ctx->w_first_h, wh.data(), wh.size() * 2, cudaMemcpyHostToDevice, ctx->stream));
    {  // exact tensor-core conv1_1 (csrc/conv_first.cuh: conv_first_tcx_kernel): k < 27: W/255, k = 27 + tap: -0.5 * sum_c W
      std::vector<double> wx(64 * 36);
      const double denom = ctx->host_layers.count("conv6_2_CPM") ? 256.0 : 255.0;   // face / hand nets: /256 (face_detector.py:32)
      double mx = 0.0;
      for (int o = 0; o < 64; ++o)
        for (int t = 0; t < 9; ++t) {
          double sum = 0.0;
          for (int c = 0; c < 3; ++c) {
            const double w = L.W[(static_cast<size_t>(o) * 3 + c) * 9 + t];
            wx[o * 36 + t * 3 + c] = w / denom;
            sum += w;
          }
          wx[o * 36 + 27 + t] = -0.5 * sum;
        }
      for (double v : wx) mx = std::max(mx, std::fabs(v));
      int S = 0;
      if (mx > 0.0 && std::isfinite(mx)) S = std::max(-60, std::min(60, static_cast<int>(std::floor(std::log2(16384.0 / mx)))));
      std::vector<__half> whx(2 * 64 * 64, __float2half(0.f));
      for (int o = 0; o < 64; ++o)
        for (int k = 0; k < 36; ++k) {
          const double v = std::ldexp(wx[o * 36 + k], S);
          const __half hi = __float2half_rn(static_cast<float>(v));
          whx[o * 64 + k] = hi;
          whx[64 * 64 + o * 64 + k] = __float2half_rn(static_cast<float>(v - static_cast<double>(__half2float(hi))));
        }
      ctx->first_x_scale = std::ldexp(1.f, -S);
      if ((rc = dev_alloc(ctx, &ctx->w_first_x, whx.size(), ctx->weight_allocs, false))) return rc;
      OPB_CUDA(ctx, cudaMemcpyAsync(ctx->w_first_x, whx.data(), whx.size() * 2, cudaMemcpyHostToDevice, ctx->stream));
    }
    OPB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    if ((rc = dev_alloc(ctx, &ctx->w_first, wt.size(), ctx->weight_allocs, false))) return rc;
    if ((rc = dev_alloc(ctx, &ctx->b_first, 64, ctx->weight_allocs, false))) return rc;
    OPB_CUDA(ctx, cudaMemcpyAsync(ctx->w_first, wt.data(), wt.size() * 4, cudaMemcpyHostToDevice, ctx->stream));
    OPB_CUDA(ctx, cudaMemcpyAsync(ctx->b_first, L.b.data(), 64 * 4, cudaMemcpyHostToDevice, ctx->stream));
    OPB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  }
  auto simple = [&](const std::string& name, int cin, int cout, int ks) -> int {
    return pack_weights(ctx, name, {{name, cout}}, identity_map(cin, round_up(cin, 64)), ks, split);
  };
  ctx->kp_out = 0;
  ctx->u8_denom = 255.f;
  if (ctx->host_layers.count("conv6_2_CPM")) {
    // FaceNet / HandNet (models/FaceNet.py:10-76): 52 layers, single branch; uint8 input is /256 - 0.5
    const int KC = ctx->host_layers.at("conv6_2_CPM").cout;
    if (KC < 2 || KC > 128) OPB_FAIL(ctx, OPB_ERR_ARG, "conv6_2_CPM must have 2..128 output channels");
    const int kc_pad = KC <= 48 ? 48 : KC <= 64 ? 64 : 128;
    const struct { const char* n; int cin, cout; } vgg[] = {
        {"conv1_2", 64, 64},   {"conv2_1", 64, 128},  {"conv2_2", 128, 128}, {"conv3_1", 128, 256}, {"conv3_2", 256, 256},
        {"conv3_3", 256, 256}, {"conv3_4", 256, 256}, {"conv4_1", 256, 512}, {"conv4_2", 512, 512}, {"conv4_3", 512, 512},
        {"conv4_4", 512, 512}, {"conv5_1", 512, 512}, {"conv5_2", 512, 512}, {"conv5_3_CPM", 512, 128}};
    for (auto& b : vgg)
      if ((rc = simple(b.n, b.cin, b.cout, 3))) return rc;
    if ((rc = simple("conv6_1_CPM", 128, 512, 1))) return rc;
    if ((rc = pack_weights(ctx, "conv6_2_CPM", {{"conv6_2_CPM", kc_pad}}, identity_map(512, 512), 1, split))) return rc;
    // device concat [features 0..127 | maps 128..128+KC-1]; reference order is (h, feature_map) (models/FaceNet.py:108)
    std::vector<int> cat_map(round_up(128 + KC, 64), -1);
    for (int d = 0; d < 128; ++d) cat_map[d] = KC + d;
    for (int d = 0; d < KC; ++d) cat_map[128 + d] = d;
    for (int st = 2; st <= 6; ++st) {
      const std::string S = "_stage" + std::to_string(st);
      if ((rc = pack_weights(ctx, "Mconv1" + S, {{"Mconv1" + S, 128}}, cat_map, 7, split))) return rc;
      for (int i = 2; i <= 5; ++i)
        if ((rc = simple("Mconv" + std::to_string(i) + S, 128, 128, 7))) return rc;
      if ((rc = simple("Mconv6" + S, 128, 128, 1))) return rc;
      if ((rc = pack_weights(ctx, "Mconv7" + S, {{"Mconv7" + S, kc_pad}}, identity_map(128, 128), 1, split))) return rc;
    }
    ctx->kp_out = KC;
    ctx->u8_denom = 256.f;
    return OPB_OK;
  }
  const struct { const char* n; int cin, cout; } backbone[] = {
      {"conv1_2", 64, 64},    {"conv2_1", 64, 128},   {"conv2_2", 128, 128},     {"conv3_1", 128, 256},
      {"conv3_2", 256, 256},  {"conv3_3", 256, 256},  {"conv3_4", 256, 256},     {"conv4_1", 256, 512},
      {"conv4_2", 512, 512},  {"conv4_3_CPM", 512, 256}, {"conv4_4_CPM", 256, 128}};
  for (auto& b : backbone)
    if ((rc = simple(b.n, b.cin, b.cout, 3))) return rc;
  for (const char* br : {"L1", "L2"}) {
    const std::string B(br);
    for (int i = 1; i <= 3; ++i)
      if ((rc = simple("conv5_" + std::to_string(i) + "_CPM_" + B, 128, 128, 3))) return rc;
    if ((rc = simple("conv5_4_CPM_" + B, 128, 512, 1))) return rc;
    if ((rc = pack_weights(ctx, "conv5_5_CPM_" + B, {{"conv5_5_CPM_" + B, 48}}, identity_map(512, 512), 1, split)))
      return rc;
  }
  // concat order on the device: [feature_map 0..127 | PAF 128..165 | heat 166..184 | 0 x 7];
  // reference order is (h1[38], h2[19], feature_map[128]) (models/CocoPoseNet.py:168)
  std::vector<int> cat_map(192, -1);
  for (int d = 0; d < 128; ++d) cat_map[d] = 57 + d;
  for (int d = 0; d < 38; ++d) cat_map[128 + d] = d;
  for (int d = 0; d < 19; ++d) cat_map[166 + d] = 38 + d;
  for (int st = 2; st <= 6; ++st) {
    const std::string S = "_stage" + std::to_string(st);
    if ((rc = pack_weights(ctx, "Mconv1" + S + "_fused", {{"Mconv1" + S + "_L1", 128}, {"Mconv1" + S + "_L2", 128}},
                           cat_map, 7, split)))
      return rc;
    for (const char* br : {"L1", "L2"}) {
      const std::string B = std::string("_") + br;
      for (int i = 2; i <= 5; ++i)
        if ((rc = simple("Mconv" + std::to_string(i) + S + B, 128, 128, 7))) return rc;
      if ((rc = simple("Mconv6" + S + B, 128, 128, 1))) return rc;
      if ((rc = pack_weights(ctx, "Mconv7" + S + B, {{"Mconv7" + S + B, 48}}, identity_map(128, 128), 1, split)))
        return rc;
    }
  }
  return OPB_OK;
}

int opb_forward(opb_ctx* ctx, const void* x, int x_format, int x_loc, int n, int h, int w, float* paf_out,
                float* heat_out, int out_loc) {
  if (!ctx || !x) return OPB_ERR_ARG;
  cudaSetDevice(ctx->device);
  Chain* ch = nullptr;
  int rc = get_chain(ctx, n, h, w, &ch);
  if (rc) return rc;
  const size_t px = static_cast<size_t>(n) * h * w * 3;
  ch->img_u8_src = nullptr;
  if (x_format == OPB_U8_NHWC_BGR) {
    if ((rc = copy_in(ctx, ch->img_u8, x, px, x_loc))) return rc;
  } else if (x_format == OPB_F32_NCHW) {
    if ((rc = copy_in(ctx, ch->img_f32, x, px * 4, x_loc))) return rc;
  } else {
    OPB_FAIL(ctx, OPB_ERR_ARG, "bad x_format");
  }
  if ((rc = run_chain(ctx, ch, x_format == OPB_U8_NHWC_BGR))) return rc;
  const size_t lo = static_cast<size_t>(n) * (h / 8) * (w / 8);
  if (paf_out && !ctx->kp_out && (rc = copy_out(ctx, paf_out, ch->paf_lo, lo * 38 * 4, out_loc))) return rc;
  if (heat_out && (rc = copy_out(ctx, heat_out, ch->heat_lo, lo * (ctx->kp_out ? ctx->kp_out : 19) * 4, out_loc))) return rc;
  OPB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return OPB_OK;
}

int opb_upsample(opb_ctx* ctx, int mode, const float* in, int in_loc, int planes, int h, int w, float* out,
                 int out_loc, int out_h, int out_w) {
  if (!ctx || !in || !out || planes <= 0) return OPB_ERR_ARG;
  cudaSetDevice(ctx->device);
  std::vector<void*> tmp;
  const float* d_in = in;
  float* d_out = out;
  int rc;
  if (in_loc == OPB_HOST) {
    float* t;
    if ((rc = dev_alloc(ctx, &t, static_cast<size_t>(planes) * h * w, tmp, false))) { free_all(tmp); return rc; }
    if ((rc = copy_in(ctx, t, in, static_cast<size_t>(planes) * h * w * 4, OPB_HOST))) { free_all(tmp); return rc; }
    d_in = t;
  }
  if (out_loc == OPB_HOST) {
    if ((rc = dev_alloc(ctx, &d_out, static_cast<size_t>(planes) * out_h * out_w, tmp, false))) { free_all(tmp); return rc; }
  }
  if (mode == OPB_UPSAMPLE_BILINEAR_AC) {
    if (h < 2 || w < 2) { free_all(tmp); OPB_FAIL(ctx, OPB_ERR_ARG, "bilinear upsample needs h, w >= 2"); }
    rc = launch_upsample(ctx, d_in, planes, h, w, d_out, out_h, out_w);
  } else if (mode == OPB_UPSAMPLE_BICUBIC) {
    dim3 grid((out_w + 31) / 32, (out_h + 7) / 8, std::min(planes, 64)), block(32, 8);
    resize_cubic_kernel<<<grid, block, 0, ctx->stream>>>(d_in, planes, h, w, d_out, out_h, out_w, out_h, out_w, 0, 0.f);
    ctx->launches++;
    rc = OPB_OK;
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) { ctx->err = cudaGetErrorString(e); rc = OPB_ERR_CUDA; }
  } else {
    ctx->err = "bad upsample mode";
    rc = OPB_ERR_ARG;
  }
  if (!rc && out_loc == OPB_HOST) rc = copy_out(ctx, out, d_out, static_cast<size_t>(planes) * out_h * out_w * 4, OPB_HOST);
  cudaError_t e = cudaStreamSynchronize(ctx->stream);
  if (!rc && e != cudaSuccess) { ctx->err = cudaGetErrorString(e); rc = OPB_ERR_CUDA; }
  free_all(tmp);
  return rc;
}

int opb_peaks(opb_ctx* ctx, const float* heat, int heat_loc, int c_plus_1, int h, int w, double* peaks_out,
              int peaks_cap, int* n_peaks) {
  if (!ctx || !heat || !peaks_out || !n_peaks) return OPB_ERR_ARG;
  if (c_plus_1 != 19) OPB_FAIL(ctx, OPB_ERR_ARG, "heatmaps must have 19 channels (18 joints + background)");
  cudaSetDevice(ctx->device);
  PostWs* ws;
  int rc = get_post(ctx, 1, h, w, &ws);
  if (rc) return rc;
  const float* d_heat = heat;
  if (heat_loc == OPB_HOST) {
    if ((rc = copy_in(ctx, ws->heat, heat, static_cast<size_t>(19) * h * w * 4, OPB_HOST))) return rc;
    d_heat = ws->heat;
  }
  if ((rc = launch_peaks(ctx, ws, d_heat, 1, 19, h, w))) return rc;
  int cnt = 0, st = 0;
  OPB_CUDA(ctx, cudaMemcpyAsync(&cnt, ws->peak_counts, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
  OPB_CUDA(ctx, cudaMemcpyAsync(&st, ws->status, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
  OPB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  if (st) OPB_FAIL(ctx, OPB_ERR_CAPACITY, "more peaks than opb_params.max_peaks");
  if (cnt > peaks_cap) OPB_FAIL(ctx, OPB_ERR_CAPACITY, "peaks_out too small");
  std::vector<PeakD> pk(cnt);
  if (cnt) {
    OPB_CUDA(ctx, cudaMemcpyAsync(pk.data(), ws->peaks, sizeof(PeakD) * cnt, cudaMemcpyDeviceToHost, ctx->stream));
    OPB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  }
  for (int i = 0; i < cnt; ++i) {
    peaks_out[i * 5 + 0] = pk[i].type;
    peaks_out[i * 5 + 1] = pk[i].x;
    peaks_out[i * 5 + 2] = pk[i].y;
    peaks_out[i * 5 + 3] = static_cast<double>(pk[i].score);
    peaks_out[i * 5 + 4] = i;
  }
  *n_peaks = cnt;
  return OPB_OK;
}

static int download_connections(opb_ctx* ctx, PostWs* ws, int img, double* conn_out, int conn_cap, int* conn_counts) {
  std::vector<int> cc(19);
  OPB_CUDA(ctx, cudaMemcpyAsync(cc.data(), ws->conn_counts + img * 19, sizeof(int) * 19, cudaMemcpyDeviceToHost,
                                ctx->stream));
  std::vector<Connection> all(static_cast<size_t>(19) * ctx->conn_cap);
  OPB_CUDA(ctx, cudaMemcpyAsync(all.data(), ws->conns + static_cast<size_t>(img) * 19 * ctx->conn_cap,
                                sizeof(Connection) * all.size(), cudaMemcpyDeviceToHost, ctx->stream));
  OPB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  int o = 0;
  for (int l = 0; l < 19; ++l) {
    conn_counts[l] = cc[l];
    for (int k = 0; k < cc[l]; ++k) {
      if (o >= conn_cap) OPB_FAIL(ctx, OPB_ERR_CAPACITY, "conn_out too small");
      const Connection& c = all[static_cast<size_t>(l) * ctx->conn_cap + k];
      conn_out[o * 3 + 0] = c.id_a;
      conn_out[o * 3 + 1] = c.id_b;
      conn_out[o * 3 + 2] = c.score;
      ++o;
    }
  }
  return OPB_OK;
}

int opb_connections(opb_ctx* ctx, const float* paf, int paf_loc, int h, int w, const double* peaks, int n_peaks,
                    double img_len, double* conn_out, int conn_cap, int* conn_counts) {
  if (!ctx || !paf || !conn_out || !conn_counts || (n_peaks > 0 && !peaks)) return OPB_ERR_ARG;
  cudaSetDevice(ctx->device);
  PostWs* ws;
  int rc = get_post(ctx, 1, h, w, &ws);
  if (rc) return rc;
  const float* d_paf = paf;
  if (paf_loc == OPB_HOST) {
    if ((rc = copy_in(ctx, ws->pafs, paf, static_cast<size_t>(38) * h * w * 4, OPB_HOST))) return rc;
    d_paf = ws->pafs;
  }
  if ((rc = upload_peaks(ctx, ws, peaks, n_peaks))) return rc;
  if ((rc = launch_connections(ctx, ws, d_paf, 1, h, w, img_len))) return rc;
  int st = 0;
  OPB_CUDA(ctx, cudaMemcpyAsync(&st, ws->status, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
  OPB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  if (st) OPB_FAIL(ctx, OPB_ERR_CAPACITY, "candidate / per-type capacity exceeded (status " + std::to_string(st) +
                                              "); raise opb_params.max_candidates");
  return download_connections(ctx, ws, 0, conn_out, conn_cap, conn_counts);
}

int opb_candidates(opb_ctx* ctx, const float* paf, int h, int w, const double* cand_a, int n_a, const double* cand_b,
                   int n_b, double img_len, double* out, int out_cap, int* n_out) {
  if (!ctx || !paf || !out || !n_out || (n_a > 0 && !cand_a) || (n_b > 0 && !cand_b)) return OPB_ERR_ARG;
  cudaSetDevice(ctx->device);
  PostWs* ws;
  int rc = get_post(ctx, 1, h, w, &ws);
  if (rc) return rc;
  *n_out = 0;
  if (n_a == 0 || n_b == 0) return OPB_OK;
  // limb 0 of the table joins joint types limbs[0][0] -> limbs[0][1]; its PAF channels are 0 and 1
  const int ja = ctx->pc.limbs[0][0], jb = ctx->pc.limbs[0][1];
  std::vector<double> pk(static_cast<size_t>(n_a + n_b) * 5);
  for (int i = 0; i < n_a + n_b; ++i) {
    const double* src = (i < n_a) ? cand_a + i * 4 : cand_b + (i - n_a) * 4;
    pk[i * 5 + 0] = (i < n_a) ? ja : jb;
    pk[i * 5 + 1] = src[0]; pk[i * 5 + 2] = src[1]; pk[i * 5 + 3] = src[2]; pk[i * 5 + 4] = i;
  }
  if ((rc = upload_peaks(ctx, ws, pk.data(), n_a + n_b))) return rc;
  OPB_CUDA(ctx, cudaMemsetAsync(ws->pafs, 0, sizeof(float) * 38 * static_cast<size_t>(h) * w, ctx->stream));
  if ((rc = copy_in(ctx, ws->pafs, paf, sizeof(float) * 2 * static_cast<size_t>(h) * w, OPB_HOST))) return rc;
  OPB_CUDA(ctx, cudaMemsetAsync(ws->cand_counts, 0, sizeof(int) * 19, ctx->stream));
  dim3 g1(8, 1, 1);
  paf_candidates_kernel<<<g1, 128, 0, ctx->stream>>>(ws->pafs, h, w, ws->peaks, ws->idx_list, ws->type_start,
                                                     ctx->prm.max_peaks, 18, ctx->pc, img_len, ws->cands,
                                                     ws->cand_counts, ctx->prm.max_candidates);
  ctx->launches++;
  OPB_CUDA(ctx, cudaGetLastError());
  int cnt = 0;
  OPB_CUDA(ctx, cudaMemcpyAsync(&cnt, ws->cand_counts, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
  OPB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  if (cnt > ctx->prm.max_candidates) OPB_FAIL(ctx, OPB_ERR_CAPACITY, "more candidates than opb_params.max_candidates");
  if (cnt > out_cap) OPB_FAIL(ctx, OPB_ERR_CAPACITY, "out too small");
  std::vector<Candidate> cd(cnt);
  if (cnt) {
    OPB_CUDA(ctx, cudaMemcpyAsync(cd.data(), ws->cands, sizeof(Candidate) * cnt, cudaMemcpyDeviceToHost, ctx->stream));
    OPB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  }
  // presentation order only (the scores were computed on the device): descending score, ties in
  // generation order (a-major, b-minor) = Python's stable sorted(..., reverse=True)
  std::sort(cd.begin(), cd.end(), [](const Candidate& x, const Candidate& y) {
    return x.score > y.score || (x.score == y.score && x.pair < y.pair);
  });
  for (int i = 0; i < cnt; ++i) {
    const int a = cd[i].pair / n_b, b = cd[i].pair % n_b;
    out[i * 3 + 0] = static_cast<double>(static_cast<int>(cand_a[a * 4 + 3]));
    out[i * 3 + 1] = static_cast<double>(static_cast<int>(cand_b[b * 4 + 3]));
    out[i * 3 + 2] = cd[i].score;
  }
  *n_out = cnt;
  return OPB_OK;
}

int opb_group(opb_ctx* ctx, const double* conns, const int* conn_counts, const double* peaks, int n_peaks,
              double* subsets_out, int subsets_cap, int* n_subsets) {
  if (!ctx || !conn_counts || !subsets_out || !n_subsets || (n_peaks > 0 && !peaks)) return OPB_ERR_ARG;
  cudaSetDevice(ctx->device);
  PostWs* ws;
  int rc = get_post(ctx, 1, 8, 8, &ws);
  if (rc) return rc;
  if ((rc = upload_peaks(ctx, ws, peaks, n_peaks))) return rc;
  std::vector<Connection> all(static_cast<size_t>(19) * ctx->conn_cap);
  int o = 0;
  for (int l = 0; l < 19; ++l) {
    if (conn_counts[l] > ctx->conn_cap) OPB_FAIL(ctx, OPB_ERR_CAPACITY, "too many connections for one limb");
    for (int k = 0; k < conn_counts[l]; ++k, ++o) {
      Connection& c = all[static_cast<size_t>(l) * ctx->conn_cap + k];
      c.id_a = static_cast<int>(conns[o * 3 + 0]);
      c.id_b = static_cast<int>(conns[o * 3 + 1]);
      c.score = conns[o * 3 + 2];
      if (c.id_a < 0 || c.id_a >= n_peaks || c.id_b < 0 || c.id_b >= n_peaks) OPB_FAIL(ctx, OPB_ERR_ARG, "connection id out of range");
    }
  }
  OPB_CUDA(ctx, cudaMemcpyAsync(ws->conns, all.data(), sizeof(Connection) * all.size(), cudaMemcpyHostToDevice, ctx->stream));
  OPB_CUDA(ctx, cudaMemcpyAsync(ws->conn_counts, conn_counts, sizeof(int) * 19, cudaMemcpyHostToDevice, ctx->stream));
  if ((rc = launch_group(ctx, ws, 1, true))) return rc;
  ImageHeader hd;
  OPB_CUDA(ctx, cudaMemcpyAsync(&hd, ws->headers, sizeof(hd), cudaMemcpyDeviceToHost, ctx->stream));
  OPB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  if (hd.status == OPB_ERR_INDEX) OPB_FAIL(ctx, OPB_ERR_INDEX, "list assignment index out of range");
  if (hd.status) OPB_FAIL(ctx, OPB_ERR_CAPACITY, "more live subsets than opb_params.max_persons");
  if (hd.n_persons > subsets_cap) OPB_FAIL(ctx, OPB_ERR_CAPACITY, "subsets_out too small");
  if (hd.n_persons) {
    OPB_CUDA(ctx, cudaMemcpyAsync(subsets_out, ws->subsets_out, sizeof(double) * 20 * hd.n_persons,
                                  cudaMemcpyDeviceToHost, ctx->stream));
    OPB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  }
  *n_subsets = hd.n_persons;
  return OPB_OK;
}

// upsample + peaks + connections + grouping of n images' network outputs (device pointers, [n][38|19][h8][w8]):
// pose_detector.py:501-512.  OPB_PAF_LOWRES / OPB_FUSED_PEAKS skip the materialised full-resolution PAFs / heat maps.
static int run_postprocess(opb_ctx* ctx, PostWs* ws, int n, int h8, int w8, int map_h, int map_w, double img_len,
                           const float* paf_lo, const float* heat_lo) {
  int rc;
  ws->last_paf_lo = paf_lo; ws->last_heat_lo = heat_lo; ws->last_img_len = img_len;
  ws->last_h8 = h8; ws->last_w8 = w8;
  if (!ctx->paf_lowres) {
    if ((rc = launch_upsample(ctx, paf_lo, n * 38, h8, w8, ws->pafs, map_h, map_w))) return rc;
    prof_mark(ctx, "upsample_paf");
  }
  if (ctx->fused_peaks == 1 || ctx->fused_peaks == 3) {
    if ((rc = launch_peaks(ctx, ws, heat_lo, n, 19, map_h, map_w, h8, w8))) return rc;
  } else if (ctx->fused_peaks == 2) {
    if ((rc = launch_upsample(ctx, heat_lo, n * 19, h8, w8, ws->heat, map_h, map_w))) return rc;
    prof_mark(ctx, "upsample_heat");
    if ((rc = launch_peaks(ctx, ws, heat_lo, n, 19, map_h, map_w, h8, w8, ws->heat))) return rc;
  } else {
    if ((rc = launch_upsample(ctx, heat_lo, n * 19, h8, w8, ws->heat, map_h, map_w))) return rc;
    prof_mark(ctx, "upsample_heat");
    if ((rc = launch_peaks(ctx, ws, ws->heat, n, 19, map_h, map_w))) return rc;
  }
  prof_mark(ctx, "peaks");
  if (ctx->paf_lowres) rc = launch_connections(ctx, ws, paf_lo, n, map_h, map_w, img_len, h8, w8);
  else rc = launch_connections(ctx, ws, ws->pafs, n, map_h, map_w, img_len);
  if (rc) return rc;
  prof_mark(ctx, "connections");
  if ((rc = launch_group(ctx, ws, n, true))) return rc;
  prof_mark(ctx, "group");
  return OPB_OK;
}

// conv chain + upsample + peaks + connections + grouping for the frames ch->img_u8_src points at (all on ctx->stream,
// no host synchronisation): the device-resident body of PoseDetector.__call__ (pose_detector.py:495-512)
static int run_pipeline(opb_ctx* ctx, Chain* ch, PostWs* ws, int n, int h, int w, int map_h, int map_w, double img_len,
                        const float* inject_paf, const float* inject_heat) {
  int rc;
  if (ctx->kp_out) OPB_FAIL(ctx, OPB_ERR_STATE, "this context holds a face / hand net: use opb_keypoints_detect");
  if ((rc = run_chain(ctx, ch, true))) return rc;
  return run_postprocess(ctx, ws, n, h / 8, w / 8, map_h, map_w, img_len, inject_paf ? inject_paf : ch->paf_lo,
                         inject_heat ? inject_heat : ch->heat_lo);
}

int opb_detect_batch(opb_ctx* ctx, const uint8_t* imgs, int imgs_loc, int n, int h, int w, int map_h, int map_w,
                     double img_len, const float* inject_paf, const float* inject_heat, opb_image_header* headers_out,
                     opb_person* persons_out, int out_loc) {
  if (!ctx || !imgs || !headers_out || !persons_out) return OPB_ERR_ARG;
  cudaSetDevice(ctx->device);
  Chain* ch = nullptr;
  PostWs* ws = nullptr;
  int rc;
  if ((rc = get_chain(ctx, n, h, w, &ch))) return rc;
  if ((rc = get_post(ctx, n, map_h, map_w, &ws))) return rc;
  prof_mark(ctx, "begin");
  if (imgs_loc == OPB_DEVICE) {
    ch->img_u8_src = imgs;            // frames already resident in HBM: conv1_1 reads them in place
  } else {
    ch->img_u8_src = nullptr;
    if ((rc = copy_in(ctx, ch->img_u8, imgs, static_cast<size_t>(n) * h * w * 3, imgs_loc))) return rc;
  }
  prof_mark(ctx, "copy_in");
  if ((rc = run_pipeline(ctx, ch, ws, n, h, w, map_h, map_w, img_len, inject_paf, inject_heat))) return rc;
  if ((rc = copy_out(ctx, headers_out, ws->headers, sizeof(ImageHeader) * n, out_loc))) return rc;
  if ((rc = copy_out(ctx, persons_out, ws->persons, sizeof(PersonOut) * n * ctx->prm.max_persons, out_loc))) return rc;
  prof_mark(ctx, "copy_out");
  OPB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  prof_report(ctx);
  return OPB_OK;
}

int opb_postprocess_batch(opb_ctx* ctx, const float* paf_lo, const float* heat_lo, int maps_loc, int n, int h8, int w8,
                          int map_h, int map_w, double img_len, opb_image_header* headers_out, opb_person* persons_out,
                          int out_loc) {
  if (!ctx || !paf_lo || !heat_lo || !headers_out || !persons_out || n <= 0 || h8 < 2 || w8 < 2 || map_h <= 0 || map_w <= 0)
    return OPB_ERR_ARG;
  cudaSetDevice(ctx->device);
  PostWs* ws = nullptr;
  int rc;
  if ((rc = get_post(ctx, n, map_h, map_w, &ws))) return rc;
  const size_t plane = static_cast<size_t>(h8) * w8;
  if (maps_loc == OPB_HOST) {
    if (ws->lo_cap < static_cast<size_t>(n) * 57 * plane) {   // grows only; earlier blocks stay owned by the workspace
      if ((rc = dev_alloc(ctx, &ws->lo_stage, static_cast<size_t>(n) * 57 * plane, ws->allocs, false))) return rc;
      ws->lo_cap = static_cast<size_t>(n) * 57 * plane;
    }
    if ((rc = copy_in(ctx, ws->lo_stage, paf_lo, sizeof(float) * n * 38 * plane, OPB_HOST))) return rc;
    if ((rc = copy_in(ctx, ws->lo_stage + n * 38 * plane, heat_lo, sizeof(float) * n * 19 * plane, OPB_HOST))) return rc;
    paf_lo = ws->lo_stage;
    heat_lo = ws->lo_stage + n * 38 * plane;
  }
  if ((rc = run_postprocess(ctx, ws, n, h8, w8, map_h, map_w, img_len, paf_lo, heat_lo))) return rc;
  if ((rc = copy_out(ctx, headers_out, ws->headers, sizeof(ImageHeader) * n, out_loc))) return rc;
  if ((rc = copy_out(ctx, persons_out, ws->persons, sizeof(PersonOut) * n * ctx->prm.max_persons, out_loc))) return rc;
  OPB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return OPB_OK;
}

int opb_get_image_detail(opb_ctx* ctx, int img, double* peaks_out, int peaks_cap, int* n_peaks, double* conn_out,
                         int conn_cap, int* conn_counts, double* subsets_out, int subsets_cap, int* n_subsets) {
  if (!ctx) return OPB_ERR_ARG;
  PostWs* ws = ctx->last_post;
  if (!ws || img < 0 || img >= ws->N) OPB_FAIL(ctx, OPB_ERR_STATE, "no post-process result for that image");
  cudaSetDevice(ctx->device);
  ImageHeader hd;
  OPB_CUDA(ctx, cudaMemcpyAsync(&hd, ws->headers + img, sizeof(hd), cudaMemcpyDeviceToHost, ctx->stream));
  OPB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  if (n_peaks) *n_peaks = hd.n_peaks;
  if (peaks_out) {
    if (hd.n_peaks > peaks_cap) OPB_FAIL(ctx, OPB_ERR_CAPACITY, "peaks_out too small");
    std::vector<PeakD> pk(hd.n_peaks);
    if (hd.n_peaks) {
      OPB_CUDA(ctx, cudaMemcpyAsync(pk.data(), ws->peaks + static_cast<size_t>(img) * ctx->prm.max_peaks,
                                    sizeof(PeakD) * hd.n_peaks, cudaMemcpyDeviceToHost, ctx->stream));
      OPB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    }
    for (int i = 0; i < hd.n_peaks; ++i) {
      peaks_out[i * 5 + 0] = pk[i].type; peaks_out[i * 5 + 1] = pk[i].x; peaks_out[i * 5 + 2] = pk[i].y;
      peaks_out[i * 5 + 3] = static_cast<double>(pk[i].score); peaks_out[i * 5 + 4] = i;
    }
  }
  if (conn_out && conn_counts) {
    int rc = download_connections(ctx, ws, img, conn_out, conn_cap, conn_counts);
    if (rc) return rc;
  }
  if (n_subsets) *n_subsets = hd.n_persons;
  if (subsets_out) {
    if (hd.n_persons > subsets_cap) OPB_FAIL(ctx, OPB_ERR_CAPACITY, "subsets_out too small");
    if (hd.n_persons) {
      OPB_CUDA(ctx, cudaMemcpyAsync(subsets_out, ws->subsets_out + static_cast<size_t>(img) * ctx->prm.max_persons * 20,
                                    sizeof(double) * 20 * hd.n_persons, cudaMemcpyDeviceToHost, ctx->stream));
      OPB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    }
  }
  return OPB_OK;
}

int opb_precise_begin(opb_ctx* ctx, int orig_h, int orig_w) {
  if (!ctx || orig_h <= 0 || orig_w <= 0) return OPB_ERR_ARG;
  cudaSetDevice(ctx->device);
  PostWs* ws;
  return get_post(ctx, 1, orig_h, orig_w, &ws);
}

static int ensure_ingest(opb_ctx* ctx, size_t bytes);
static int launch_resize_u8(opb_ctx* ctx, const uint8_t* d_src, int n, int h0, int w0, uint8_t* d_dst, int h, int w,
                            bool cubic = false);

// forward + both cubic resizes + accumulate for the padded frame already in ch->img_u8 (:447-467)
static int precise_accumulate(opb_ctx* ctx, PostWs* ws, Chain* ch, int ph, int pw, int pad_h, int pad_w, int scale_index,
                              int n_scales) {
  int rc;
  ch->img_u8_src = nullptr;
  if ((rc = run_chain(ctx, ch, true))) return rc;
  const int h8 = ph / 8, w8 = pw / 8;
  const int ch_h = ph - pad_h, ch_w = pw - pad_w;   // crop after the x8 resize (:462,:466)
  const size_t need = static_cast<size_t>(38) * ch_h * ch_w;
  if (ctx->precise_mid_cap < need) {                 // x8 intermediate, kept across scales and calls
    if (ctx->precise_mid) { OPB_CUDA(ctx, cudaStreamSynchronize(ctx->stream)); cudaFree(ctx->precise_mid); ctx->precise_mid = nullptr; }
    OPB_CUDA(ctx, cudaMalloc(reinterpret_cast<void**>(&ctx->precise_mid), need * sizeof(float)));
    ctx->precise_mid_cap = need;
  }
  float* mid = ctx->precise_mid;
  const float scale = (scale_index == n_scales - 1) ? static_cast<float>(n_scales) : 0.f;   // divisor of the last pass (0 = none)
  for (int which = 0; which < 2; ++which) {
    const int C = which ? 19 : 38;
    const float* lo = which ? ch->heat_lo : ch->paf_lo;
    float* acc = which ? ws->heat : ws->pafs;
    dim3 block(32, 8);
    dim3 g1((ch_w + 31) / 32, (ch_h + 7) / 8, C);
    resize_cubic_kernel<<<g1, block, 0, ctx->stream>>>(lo, C, h8, w8, mid, ph, pw, ch_h, ch_w, 0, 0.f);
    dim3 g2((ws->W + 31) / 32, (ws->H + 7) / 8, C);
    resize_cubic_kernel<<<g2, block, 0, ctx->stream>>>(mid, C, ch_h, ch_w, acc, ws->H, ws->W, ws->H, ws->W,
                                                       scale_index > 0 ? 1 : 0, scale);
    ctx->launches += 2;
  }
  OPB_CUDA(ctx, cudaGetLastError());
  return OPB_OK;
}

int opb_precise_add_scale(opb_ctx* ctx, const uint8_t* img, int img_loc, int ph, int pw, int pad_h, int pad_w,
                          int scale_index, int n_scales) {
  if (!ctx || !img) return OPB_ERR_ARG;
  PostWs* ws = ctx->last_post;
  if (!ws || ws->N != 1) OPB_FAIL(ctx, OPB_ERR_STATE, "opb_precise_begin was not called");
  cudaSetDevice(ctx->device);
  Chain* ch = nullptr;
  int rc = get_chain(ctx, 1, ph, pw, &ch);
  if (rc) return rc;
  if ((rc = copy_in(ctx, ch->img_u8, img, static_cast<size_t>(ph) * pw * 3, img_loc))) return rc;
  return precise_accumulate(ctx, ws, ch, ph, pw, pad_h, pad_w, scale_index, n_scales);
}

int opb_precise_add_scale_unpadded(opb_ctx* ctx, const uint8_t* img, int img_loc, int h, int w, int stride,
                                   const uint8_t pad_value[3], int scale_index, int n_scales) {
  if (!ctx || !img || !pad_value || h <= 0 || w <= 0 || stride <= 0) return OPB_ERR_ARG;
  PostWs* ws = ctx->last_post;
  if (!ws || ws->N != 1) OPB_FAIL(ctx, OPB_ERR_STATE, "opb_precise_begin was not called");
  cudaSetDevice(ctx->device);
  const int pad_h = (stride - h % stride) % stride, pad_w = (stride - w % stride) % stride;     // :50-51
  const int ph = h + pad_h, pw = w + pad_w;
  Chain* ch = nullptr;
  int rc = get_chain(ctx, 1, ph, pw, &ch);
  if (rc) return rc;
  const size_t in_b = static_cast<size_t>(h) * w * 3;
  const uint8_t* d_src = img;
  if (img_loc == OPB_HOST) {
    if ((rc = ensure_ingest(ctx, in_b + 512))) return rc;
    if ((rc = copy_in(ctx, ctx->ingest_buf, img, in_b, OPB_HOST))) return rc;
    d_src = ctx->ingest_buf;
  }
  dim3 block(32, 8), grid((pw + 31) / 32, (ph + 7) / 8);
  pad_image_u8_kernel<<<grid, block, 0, ctx->stream>>>(d_src, h, w, ch->img_u8, ph, pw, pad_value[0], pad_value[1],
                                                       pad_value[2]);
  ctx->launches++;
  OPB_CUDA(ctx, cudaGetLastError());
  return precise_accumulate(ctx, ws, ch, ph, pw, pad_h, pad_w, scale_index, n_scales);
}

int opb_precise_add_scale_orig(opb_ctx* ctx, const uint8_t* orig, int img_loc, int orig_h, int orig_w, int h, int w,
                               int stride, const uint8_t pad_value[3], int scale_index, int n_scales) {
  if (!ctx || !orig || !pad_value || orig_h <= 0 || orig_w <= 0 || h <= 0 || w <= 0 || stride <= 0) return OPB_ERR_ARG;
  PostWs* ws = ctx->last_post;
  if (!ws || ws->N != 1) OPB_FAIL(ctx, OPB_ERR_STATE, "opb_precise_begin was not called");
  cudaSetDevice(ctx->device);
  const size_t in_b = static_cast<size_t>(orig_h) * orig_w * 3, mid_b = static_cast<size_t>(h) * w * 3;
  const size_t mid_off = (in_b + 255) & ~size_t(255);
  int rc = ensure_ingest(ctx, mid_off + mid_b + 512);
  if (rc) return rc;
  const uint8_t* d_src = orig;
  if (img_loc == OPB_HOST) {
    if ((rc = copy_in(ctx, ctx->ingest_buf, orig, in_b, OPB_HOST))) return rc;
    d_src = ctx->ingest_buf;
  }
  uint8_t* d_mid = ctx->ingest_buf + mid_off;
  if ((rc = launch_resize_u8(ctx, d_src, 1, orig_h, orig_w, d_mid, h, w, true))) return rc;   // :443
  return opb_precise_add_scale_unpadded(ctx, d_mid, OPB_DEVICE, h, w, stride, pad_value, scale_index, n_scales);
}

int opb_precise_finish(opb_ctx* ctx, double img_len, opb_image_header* header_out, opb_person* persons_out,
                       int out_loc) {
  if (!ctx || !header_out || !persons_out) return OPB_ERR_ARG;
  PostWs* ws = ctx->last_post;
  if (!ws || ws->N != 1) OPB_FAIL(ctx, OPB_ERR_STATE, "opb_precise_begin was not called");
  cudaSetDevice(ctx->device);
  int rc;
  if ((rc = launch_peaks(ctx, ws, ws->heat, 1, 19, ws->H, ws->W))) return rc;
  if ((rc = launch_connections(ctx, ws, ws->pafs, 1, ws->H, ws->W, img_len))) return rc;
  if ((rc = launch_group(ctx, ws, 1, true))) return rc;
  if ((rc = copy_out(ctx, header_out, ws->headers, sizeof(ImageHeader), out_loc))) return rc;
  if ((rc = copy_out(ctx, persons_out, ws->persons, sizeof(PersonOut) * ctx->prm.max_persons, out_loc))) return rc;
  OPB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return OPB_OK;
}

int opb_download_maps(opb_ctx* ctx, float* pafs_out, float* heat_out, int out_loc) {
  if (!ctx) return OPB_ERR_ARG;
  PostWs* ws = ctx->last_post;
  if (!ws) OPB_FAIL(ctx, OPB_ERR_STATE, "no post-process workspace");
  cudaSetDevice(ctx->device);
  int rc;
  const size_t plane = static_cast<size_t>(ws->H) * ws->W * 4;
  if (pafs_out && (rc = copy_out(ctx, pafs_out, ws->pafs, plane * 38, out_loc))) return rc;
  if (heat_out && (rc = copy_out(ctx, heat_out, ws->heat, plane * 19, out_loc))) return rc;
  OPB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return OPB_OK;
}

// ---- draw_person_pose on the device (pose_detector.py:520-553; csrc/overlay.cuh) -------------------------------
static OverlayTables overlay_tables(const opb_ctx* ctx) {
  // limb_colors / joint_colors of pose_detector.py:523-535, written into channels 0,1,2 as given
  static const uint8_t kLimb[OV_LIMBS][3] = {
      {0, 255, 0}, {0, 255, 85}, {0, 255, 170}, {0, 255, 255}, {0, 170, 255}, {0, 85, 255}, {255, 0, 0},
      {255, 85, 0}, {255, 170, 0}, {255, 255, 0}, {255, 0, 85}, {170, 255, 0}, {85, 255, 0}, {170, 0, 255},
      {0, 0, 255}, {0, 0, 255}, {255, 0, 255}, {170, 0, 255}, {255, 0, 170}};
  static const uint8_t kJoint[OV_JOINTS][3] = {
      {255, 0, 0}, {255, 85, 0}, {255, 170, 0}, {255, 255, 0}, {170, 255, 0}, {85, 255, 0}, {0, 255, 0},
      {0, 255, 85}, {0, 255, 170}, {0, 255, 255}, {0, 170, 255}, {0, 85, 255}, {0, 0, 255}, {85, 0, 255},
      {170, 0, 255}, {255, 0, 255}, {255, 0, 170}, {255, 0, 85}};
  OverlayTables tb;
  for (int l = 0; l < OV_LIMBS; ++l) {
    tb.limb_a[l] = ctx->prm.limbs[l][0];
    tb.limb_b[l] = ctx->prm.limbs[l][1];
    for (int c = 0; c < 3; ++c) tb.limb_color[l][c] = kLimb[l][c];
  }
  for (int j = 0; j < OV_JOINTS; ++j)
    for (int c = 0; c < 3; ++c) tb.joint_color[j][c] = kJoint[j][c];
  return tb;
}

// poses: device int [n_poses][18][3] when from_records == nullptr; otherwise the records of one image are converted first
static int overlay_run(opb_ctx* ctx, const uint8_t* img, int img_loc, int h, int w, const int32_t* host_poses, int n_poses,
                       const PersonOut* d_records, double sx, double sy, uint8_t* out, int out_loc) {
  cudaSetDevice(ctx->device);
  const size_t px = static_cast<size_t>(h) * w, img_b = (px * 3 + 255) & ~size_t(255);
  const size_t prio_b = (px * 4 + 255) & ~size_t(255), poses_b = (static_cast<size_t>(n_poses > 0 ? n_poses : 1) * OV_JOINTS * 3 * 4 + 255) & ~size_t(255);
  const size_t need = 2 * img_b + prio_b + poses_b + 256;
  if (ctx->ov_bytes < need) {
    if (ctx->ov_buf) { cudaStreamSynchronize(ctx->stream); cudaFree(ctx->ov_buf); ctx->ov_buf = nullptr; ctx->ov_bytes = 0; }
    OPB_CUDA(ctx, cudaMalloc(reinterpret_cast<void**>(&ctx->ov_buf), need));
    ctx->ov_bytes = need;
  }
  uint8_t* d_in = ctx->ov_buf;
  uint8_t* d_out = ctx->ov_buf + img_b;
  unsigned int* d_prio = reinterpret_cast<unsigned int*>(ctx->ov_buf + 2 * img_b);
  int* d_poses = reinterpret_cast<int*>(ctx->ov_buf + 2 * img_b + prio_b);
  int* d_bad = reinterpret_cast<int*>(ctx->ov_buf + 2 * img_b + prio_b + poses_b);
  int rc;
  const uint8_t* d_src = img;
  if (img_loc == OPB_HOST) {
    if ((rc = copy_in(ctx, d_in, img, px * 3, OPB_HOST))) return rc;
    d_src = d_in;
  }
  uint8_t* d_dst = (out_loc == OPB_HOST) ? d_out : out;
  OPB_CUDA(ctx, cudaMemsetAsync(d_prio, 0, px * 4, ctx->stream));
  OPB_CUDA(ctx, cudaMemsetAsync(d_bad, 0, 4, ctx->stream));
  const OverlayTables tb = overlay_tables(ctx);
  if (n_poses > 0) {
    if (d_records) {
      const int* base = reinterpret_cast<const int*>(d_records);
      const int stride = static_cast<int>(sizeof(PersonOut) / 4), off_id = 4, off_x = 4 + OPB_N_JOINTS, off_y = 4 + 2 * OPB_N_JOINTS;
      overlay_poses_from_records_kernel<<<(n_poses * OV_JOINTS + 127) / 128, 128, 0, ctx->stream>>>(
          base + off_x, base + off_y, base + off_id, stride, n_poses, sx, sy, d_poses);
      ctx->launches++;
    } else {
      if ((rc = copy_in(ctx, d_poses, host_poses, static_cast<size_t>(n_poses) * OV_JOINTS * 3 * 4, OPB_HOST))) return rc;
    }
    const int n_prim = n_poses * (OV_LIMBS + OV_JOINTS);
    overlay_raster_kernel<<<(n_prim + 63) / 64, 64, 0, ctx->stream>>>(d_poses, n_poses, tb, d_prio, h, w, d_bad);
    ctx->launches++;
  }
  overlay_paint_kernel<<<static_cast<unsigned>((px + 255) / 256), 256, 0, ctx->stream>>>(d_src, d_prio, static_cast<int>(px), n_poses, tb, d_dst);
  ctx->launches++;
  OPB_CUDA(ctx, cudaGetLastError());
  int bad = 0;
  OPB_CUDA(ctx, cudaMemcpyAsync(&bad, d_bad, 4, cudaMemcpyDeviceToHost, ctx->stream));
  if (out_loc == OPB_HOST && (rc = copy_out(ctx, out, d_dst, px * 3, OPB_HOST))) return rc;
  OPB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  if (bad) OPB_FAIL(ctx, OPB_ERR_ARG, "draw_person_pose: a joint lies outside the image");
  return OPB_OK;
}

int opb_draw_person_pose(opb_ctx* ctx, const uint8_t* img, int img_loc, int h, int w, const int32_t* poses, int n_poses,
                         uint8_t* out, int out_loc) {
  if (!ctx || !img || !out || h <= 0 || w <= 0 || n_poses < 0 || (n_poses > 0 && !poses)) return OPB_ERR_ARG;
  return overlay_run(ctx, img, img_loc, h, w, poses, n_poses, nullptr, 1.0, 1.0, out, out_loc);
}

int opb_draw_last_result(opb_ctx* ctx, int image_index, const uint8_t* img, int img_loc, int h, int w, double sx, double sy,
                         uint8_t* out, int out_loc) {
  if (!ctx || !img || !out || h <= 0 || w <= 0) return OPB_ERR_ARG;
  PostWs* ws = ctx->last_post;
  if (!ws || image_index < 0 || image_index >= ws->N) OPB_FAIL(ctx, OPB_ERR_STATE, "no result for that image");
  cudaSetDevice(ctx->device);
  ImageHeader hd;
  OPB_CUDA(ctx, cudaMemcpyAsync(&hd, ws->headers + image_index, sizeof(hd), cudaMemcpyDeviceToHost, ctx->stream));
  OPB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  if (hd.status != 0) OPB_FAIL(ctx, hd.status, "the image's result carries an error status");
  return overlay_run(ctx, img, img_loc, h, w, nullptr, hd.n_persons,
                     ws->persons + static_cast<size_t>(image_index) * ctx->prm.max_persons, sx, sy, out, out_loc);
}

static int launch_resize_u8(opb_ctx* ctx, const uint8_t* d_src, int n, int h0, int w0, uint8_t* d_dst, int h, int w,
                            bool cubic) {
  if (h0 == h && w0 == w) {
    OPB_CUDA(ctx, cudaMemcpyAsync(d_dst, d_src, static_cast<size_t>(n) * h * w * 3, cudaMemcpyDeviceToDevice, ctx->stream));
    return OPB_OK;
  }
  const double sx = 1.0 / (static_cast<double>(w) / w0), sy = 1.0 / (static_cast<double>(h) / h0);
  dim3 grid((w + 31) / 32, (h + 7) / 8, n), block(32, 8);
  if (cubic) resize_cubic_u8_kernel<<<grid, block, 0, ctx->stream>>>(d_src, h0, w0, d_dst, h, w, sx, sy);
  else resize_linear_u8_kernel<<<grid, block, 0, ctx->stream>>>(d_src, h0, w0, d_dst, h, w, sx, sy);
  ctx->launches++;
  OPB_CUDA(ctx, cudaGetLastError());
  return OPB_OK;
}

static int ensure_ingest(opb_ctx* ctx, size_t bytes) {
  if (ctx->ingest_bytes >= bytes) return OPB_OK;
  if (ctx->ingest_buf) { cudaStreamSynchronize(ctx->stream); cudaFree(ctx->ingest_buf); ctx->ingest_buf = nullptr; }
  OPB_CUDA(ctx, cudaMalloc(reinterpret_cast<void**>(&ctx->ingest_buf), bytes));
  ctx->ingest_bytes = bytes;
  return OPB_OK;
}

static int resize_u8_entry(opb_ctx* ctx, const uint8_t* src, int src_loc, int n, int h0, int w0, uint8_t* dst,
                           int dst_loc, int h, int w, bool cubic);

int opb_resize_linear_u8(opb_ctx* ctx, const uint8_t* src, int src_loc, int n, int h0, int w0, uint8_t* dst,
                         int dst_loc, int h, int w) {
  return resize_u8_entry(ctx, src, src_loc, n, h0, w0, dst, dst_loc, h, w, false);
}

int opb_resize_cubic_u8(opb_ctx* ctx, const uint8_t* src, int src_loc, int n, int h0, int w0, uint8_t* dst,
                        int dst_loc, int h, int w) {
  return resize_u8_entry(ctx, src, src_loc, n, h0, w0, dst, dst_loc, h, w, true);
}

static int resize_u8_entry(opb_ctx* ctx, const uint8_t* src, int src_loc, int n, int h0, int w0, uint8_t* dst,
                           int dst_loc, int h, int w, bool cubic) {
  if (!ctx || !src || !dst || n <= 0 || h0 <= 0 || w0 <= 0 || h <= 0 || w <= 0) return OPB_ERR_ARG;
  cudaSetDevice(ctx->device);
  const size_t in_b = static_cast<size_t>(n) * h0 * w0 * 3, out_b = static_cast<size_t>(n) * h * w * 3;
  int rc = ensure_ingest(ctx, in_b + out_b + 512);
  if (rc) return rc;
  const uint8_t* d_src = src;
  if (src_loc == OPB_HOST) {
    if ((rc = copy_in(ctx, ctx->ingest_buf, src, in_b, OPB_HOST))) return rc;
    d_src = ctx->ingest_buf;
  }
  uint8_t* d_dst = (dst_loc == OPB_HOST) ? ctx->ingest_buf + ((in_b + 255) & ~size_t(255)) : dst;
  if ((rc = launch_resize_u8(ctx, d_src, n, h0, w0, d_dst, h, w, cubic))) return rc;
  if (dst_loc == OPB_HOST && (rc = copy_out(ctx, dst, d_dst, out_b, OPB_HOST))) return rc;
  OPB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return OPB_OK;
}

int opb_detect_image(opb_ctx* ctx, const uint8_t* img, int img_loc, int orig_h, int orig_w, int in_h, int in_w,
                     int map_h, int map_w, double img_len, opb_image_header* header_out, opb_person* persons_out,
                     int out_loc) {
  if (!ctx || !img || !header_out || !persons_out) return OPB_ERR_ARG;
  cudaSetDevice(ctx->device);
  Chain* ch = nullptr;
  int rc = get_chain(ctx, 1, in_h, in_w, &ch);
  if (rc) return rc;
  const size_t in_b = static_cast<size_t>(orig_h) * orig_w * 3;
  const uint8_t* d_src = img;
  if (img_loc == OPB_HOST) {
    if ((rc = ensure_ingest(ctx, in_b + 512))) return rc;
    if ((rc = copy_in(ctx, ctx->ingest_buf, img, in_b, OPB_HOST))) return rc;
    d_src = ctx->ingest_buf;
  }
  if ((rc = launch_resize_u8(ctx, d_src, 1, orig_h, orig_w, ch->img_u8, in_h, in_w))) return rc;
  // frames are now resident at network-input size: reuse the batch path in place
  return opb_detect_batch(ctx, ch->img_u8, OPB_DEVICE, 1, in_h, in_w, map_h, map_w, img_len, nullptr, nullptr, header_out,
                          persons_out, out_loc);
}

int opb_stream_submit(opb_ctx* ctx, const uint8_t* frames, int frames_loc, int n, int orig_h, int orig_w, int in_h, int in_w,
                      int map_h, int map_w, double img_len, const float* inject_paf, const float* inject_heat, int slot) {
  if (!ctx || !frames || n <= 0 || slot < 0 || slot > 1) return OPB_ERR_ARG;
  cudaSetDevice(ctx->device);
  auto& sl = ctx->slots[slot];
  if (sl.busy) OPB_FAIL(ctx, OPB_ERR_ARG, "opb_stream_submit: slot still holds an uncollected batch");
  Chain* ch = nullptr;
  PostWs* ws = nullptr;
  int rc;
  if (slot == 1 && ctx->two_streams && !ctx->stream_b)
    OPB_CUDA(ctx, cudaStreamCreateWithFlags(&ctx->stream_b, cudaStreamNonBlocking));
  // slot 1 runs on its own stream with its own activations, so the tail / launch gaps of one slot's kernels are
  // filled by the other slot's; everything below launches on ctx->stream, which is swapped for the call
  struct SlotScope {
    opb_ctx* c; cudaStream_t saved; int saved_slot;
    SlotScope(opb_ctx* c_, int slot_) : c(c_), saved(c_->stream), saved_slot(c_->cur_slot) {
      if (slot_ == 1 && c->two_streams) { c->stream = c->stream_b; c->cur_slot = 1; }
    }
    ~SlotScope() { c->stream = saved; c->cur_slot = saved_slot; }
  } scope(ctx, slot);
  if ((rc = get_chain(ctx, n, in_h, in_w, &ch))) return rc;
  if ((rc = get_post(ctx, n, map_h, map_w, &ws))) return rc;
  if (!ctx->copy_stream) OPB_CUDA(ctx, cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking));
  if (!sl.done) {
    OPB_CUDA(ctx, cudaEventCreateWithFlags(&sl.h2d_done, cudaEventDisableTiming));
    OPB_CUDA(ctx, cudaEventCreateWithFlags(&sl.done, cudaEventDisableTiming));
  }
  const size_t in_b = static_cast<size_t>(n) * orig_h * orig_w * 3;
  const size_t res_b = n * (sizeof(ImageHeader) + sizeof(PersonOut) * static_cast<size_t>(ctx->prm.max_persons));
  const bool resident = frames_loc == OPB_DEVICE;   // frames already in HBM: used in place, no upload
  if (!resident && sl.d_bytes < in_b) {
    if (sl.d_frames) { OPB_CUDA(ctx, cudaStreamSynchronize(ctx->stream)); cudaFree(sl.d_frames); sl.d_frames = nullptr; }
    OPB_CUDA(ctx, cudaMalloc(reinterpret_cast<void**>(&sl.d_frames), in_b));
    sl.d_bytes = in_b;
  }
  if (sl.r_bytes < res_b) {
    if (sl.h_result) cudaFreeHost(sl.h_result);
    OPB_CUDA(ctx, cudaMallocHost(reinterpret_cast<void**>(&sl.h_result), res_b));
    sl.r_bytes = res_b;
  }
  // pageable caller memory goes through the slot's pinned staging buffer so the H2D copy is truly asynchronous
  const uint8_t* h_src = frames;
  cudaPointerAttributes at{};
  const bool pinned = resident || (cudaPointerGetAttributes(&at, frames) == cudaSuccess && at.type == cudaMemoryTypeHost);
  cudaGetLastError();
  if (!pinned) {
    if (sl.h_bytes < in_b) {
      if (sl.h_frames) cudaFreeHost(sl.h_frames);
      OPB_CUDA(ctx, cudaMallocHost(reinterpret_cast<void**>(&sl.h_frames), in_b));
      sl.h_bytes = in_b;
    }
    memcpy(sl.h_frames, frames, in_b);
    h_src = sl.h_frames;
  }
  // the slot's previous batch was collected (sl.done reached), so its device frames are free to overwrite
  const uint8_t* d_frames = resident ? frames : sl.d_frames;
  if (!resident) {
    OPB_CUDA(ctx, cudaMemcpyAsync(sl.d_frames, h_src, in_b, cudaMemcpyHostToDevice, ctx->copy_stream));
    OPB_CUDA(ctx, cudaEventRecord(sl.h2d_done, ctx->copy_stream));
    OPB_CUDA(ctx, cudaStreamWaitEvent(ctx->stream, sl.h2d_done, 0));
  }
  // everything between the upload and the `done` event: [resize] + pipeline + record download
  auto body = [&]() -> int {
    int r;
    if (orig_h == in_h && orig_w == in_w) {
      ch->img_u8_src = d_frames;
    } else {
      if ((r = launch_resize_u8(ctx, d_frames, n, orig_h, orig_w, ch->img_u8, in_h, in_w))) return r;
      ch->img_u8_src = nullptr;
    }
    if ((r = run_pipeline(ctx, ch, ws, n, in_h, in_w, map_h, map_w, img_len, inject_paf, inject_heat))) return r;
    if ((r = copy_out(ctx, sl.h_result, ws->headers, sizeof(ImageHeader) * n, OPB_HOST))) return r;
    return copy_out(ctx, sl.h_result + sizeof(ImageHeader) * n, ws->persons,
                    sizeof(PersonOut) * n * static_cast<size_t>(ctx->prm.max_persons), OPB_HOST);
  };
  const opb_ctx::StreamSlot::Key key{n, orig_h, orig_w, in_h, in_w, map_h, map_w, img_len, inject_paf, inject_heat,
                                     d_frames, sl.h_result, ch, ws, ctx->cache_epoch};
  const bool graphs = ctx->use_graphs && !ctx->profile;
  if (!(key == sl.key)) {
    if (sl.gexec) { cudaGraphExecDestroy(sl.gexec); sl.gexec = nullptr; }
    sl.key = key;
    sl.key_seen = 0;
  }
  if (graphs && sl.gexec) {
    OPB_CUDA(ctx, cudaGraphLaunch(sl.gexec, ctx->stream));
    ctx->launches += sl.graph_launches;
  } else if (graphs && sl.key_seen >= 1) {
    // second submit of this combination: capture the launch sequence, then run it as a graph
    const int64_t l0 = ctx->launches;
    OPB_CUDA(ctx, cudaStreamBeginCapture(ctx->stream, cudaStreamCaptureModeRelaxed));
    rc = body();
    cudaGraph_t graph = nullptr;
    const cudaError_t ce = cudaStreamEndCapture(ctx->stream, &graph);
    if (rc) { if (graph) cudaGraphDestroy(graph); return rc; }
    if (ce != cudaSuccess || !graph) OPB_FAIL(ctx, OPB_ERR_CUDA, std::string("stream capture failed: ") + cudaGetErrorString(ce));
    const cudaError_t ie = cudaGraphInstantiate(&sl.gexec, graph, 0);
    cudaGraphDestroy(graph);
    if (ie != cudaSuccess) { sl.gexec = nullptr; OPB_FAIL(ctx, OPB_ERR_CUDA, std::string("cudaGraphInstantiate: ") + cudaGetErrorString(ie)); }
    sl.graph_launches = ctx->launches - l0;
    OPB_CUDA(ctx, cudaGraphLaunch(sl.gexec, ctx->stream));
  } else {
    if ((rc = body())) return rc;
  }
  sl.key_seen++;
  OPB_CUDA(ctx, cudaEventRecord(sl.done, ctx->stream));
  sl.n = n;
  sl.post = ws;
  sl.busy = true;
  return OPB_OK;
}

// ---- the one collective of the path (SURVEY.md 8e): all-gather of the fixed-size result records --------------------
// NCCL is resolved at run time from the library the process already carries (torch loads libnccl.so.2; a stand-alone
// C program links or preloads it): no link-time dependency, and a box without NCCL can still use everything else.
namespace {
struct NcclApi {
  int (*GetUniqueId)(void*) = nullptr;
  int (*CommInitRank)(void**, int, OpbNcclId, int) = nullptr;
  int (*CommDestroy)(void*) = nullptr;
  int (*AllGather)(const void*, void*, size_t, int, void*, cudaStream_t) = nullptr;
  const char* (*GetErrorString)(int) = nullptr;
  bool ok = false;
  std::string why;
};
NcclApi& nccl_api() {
  static NcclApi api;
  static bool tried = false;
  if (tried) return api;
  tried = true;
  void* h = nullptr;
  const char* names[] = {getenv("OPB_NCCL_LIB"), "libnccl.so.2", "libnccl.so"};
  for (const char* n : names) {
    if (!n || !*n) continue;
    h = dlopen(n, RTLD_NOW | RTLD_GLOBAL);
    if (h) break;
  }
  if (!h) { api.why = "libnccl.so.2 not found (set OPB_NCCL_LIB)"; return api; }
  api.GetUniqueId = reinterpret_cast<int (*)(void*)>(dlsym(h, "ncclGetUniqueId"));
  api.CommInitRank = reinterpret_cast<int (*)(void**, int, OpbNcclId, int)>(dlsym(h, "ncclCommInitRank"));
  api.CommDestroy = reinterpret_cast<int (*)(void*)>(dlsym(h, "ncclCommDestroy"));
  api.AllGather = reinterpret_cast<int (*)(const void*, void*, size_t, int, void*, cudaStream_t)>(dlsym(h, "ncclAllGather"));
  api.GetErrorString = reinterpret_cast<const char* (*)(int)>(dlsym(h, "ncclGetErrorString"));
  api.ok = api.GetUniqueId && api.CommInitRank && api.CommDestroy && api.AllGather;
  if (!api.ok) api.why = "libnccl lacks ncclGetUniqueId / ncclCommInitRank / ncclCommDestroy / ncclAllGather";
  return api;
}
}  // namespace

int opb_nccl_unique_id(uint8_t id_out[128]) {
  if (!id_out) return OPB_ERR_ARG;
  NcclApi& a = nccl_api();
  if (!a.ok) { g_create_error = a.why; return OPB_ERR_UNSUPPORTED; }
  OpbNcclId id;
  const int r = a.GetUniqueId(&id);
  if (r) { g_create_error = std::string("ncclGetUniqueId: ") + (a.GetErrorString ? a.GetErrorString(r) : "error"); return OPB_ERR_CUDA; }
  std::memcpy(id_out, id.internal, 128);
  return OPB_OK;
}

int opb_nccl_comm_init(opb_ctx* ctx, void** comm_out, int world, int rank, const uint8_t id[128]) {
  if (!ctx || !comm_out || !id || world < 1 || rank < 0 || rank >= world) return OPB_ERR_ARG;
  NcclApi& a = nccl_api();
  if (!a.ok) OPB_FAIL(ctx, OPB_ERR_UNSUPPORTED, a.why);
  cudaSetDevice(ctx->device);
  OpbNcclId uid;
  std::memcpy(uid.internal, id, 128);
  void* comm = nullptr;
  const int r = a.CommInitRank(&comm, world, uid, rank);
  if (r) OPB_FAIL(ctx, OPB_ERR_CUDA, std::string("ncclCommInitRank: ") + (a.GetErrorString ? a.GetErrorString(r) : "error"));
  *comm_out = comm;
  return OPB_OK;
}

int opb_nccl_comm_destroy(void* comm) {
  NcclApi& a = nccl_api();
  if (!a.ok || !comm) return OPB_ERR_ARG;
  return a.CommDestroy(comm) ? OPB_ERR_CUDA : OPB_OK;
}

size_t opb_record_block_bytes(const opb_ctx* ctx, int n) {
  return ctx ? static_cast<size_t>(n) * (sizeof(ImageHeader) + sizeof(PersonOut) * static_cast<size_t>(ctx->prm.max_persons)) : 0;
}

int opb_allgather_results(opb_ctx* ctx, void* nccl_comm, int slot, void* gathered_dev) {
  if (!ctx || !nccl_comm || !gathered_dev || slot < 0 || slot > 1) return OPB_ERR_ARG;
  NcclApi& a = nccl_api();
  if (!a.ok) OPB_FAIL(ctx, OPB_ERR_UNSUPPORTED, a.why);
  cudaSetDevice(ctx->device);
  auto& sl = ctx->slots[slot];
  if (!sl.busy || !sl.post) OPB_FAIL(ctx, OPB_ERR_STATE, "opb_allgather_results: nothing submitted on this slot");
  cudaStream_t st = (slot == 1 && ctx->two_streams && ctx->stream_b) ? ctx->stream_b : ctx->stream;
  const PostWs* ws = static_cast<const PostWs*>(sl.post);
  // device-resident [headers | persons] of the slot's batch -> every rank's block, in rank order; no host hop
  const int r = a.AllGather(ws->headers, gathered_dev, opb_record_block_bytes(ctx, sl.n), 1 /* ncclUint8 */, nccl_comm, st);
  if (r) OPB_FAIL(ctx, OPB_ERR_CUDA, std::string("ncclAllGather: ") + (a.GetErrorString ? a.GetErrorString(r) : "error"));
  ctx->launches++;
  OPB_CUDA(ctx, cudaEventRecord(sl.done, st));       // opb_stream_collect / opb_stream_join now also cover the collective
  return OPB_OK;
}

int opb_stream_join(opb_ctx* ctx) {
  if (!ctx) return OPB_ERR_ARG;
  cudaSetDevice(ctx->device);
  for (auto& sl : ctx->slots)
    if (sl.busy && sl.done) OPB_CUDA(ctx, cudaStreamWaitEvent(ctx->stream, sl.done, 0));
  return OPB_OK;
}

int opb_stream_collect(opb_ctx* ctx, int slot, opb_image_header* headers_out, opb_person* persons_out) {
  if (!ctx || slot < 0 || slot > 1 || !headers_out || !persons_out) return OPB_ERR_ARG;
  cudaSetDevice(ctx->device);
  auto& sl = ctx->slots[slot];
  if (!sl.busy) OPB_FAIL(ctx, OPB_ERR_ARG, "opb_stream_collect: nothing submitted on this slot");
  OPB_CUDA(ctx, cudaEventSynchronize(sl.done));
  sl.busy = false;
  memcpy(headers_out, sl.h_result, sizeof(ImageHeader) * sl.n);
  memcpy(persons_out, sl.h_result + sizeof(ImageHeader) * sl.n, sizeof(PersonOut) * sl.n * static_cast<size_t>(ctx->prm.max_persons));
  return OPB_OK;
}

// Face / hand nets on ragged batches: n crops of different sizes share one upload, one resize launch, one forward of
// the chain for the next batch size in kKpBuckets, and one launch per post-process stage.
static const int kKpBuckets[] = {1, 2, 4, 8, 16, 32};
static const int kKpMaxCrops = 32;   // larger batches run in chunks of this many crops
static const int kKpUpsamplePlanes = 19;   // planes per block of upsample_bilinear_ac_ragged_kernel

static int kp_bucket(int n) {
  for (int b : kKpBuckets)
    if (b >= n) return b;
  return kKpMaxCrops;
}

static size_t align256(size_t v) { return (v + 255) & ~size_t(255); }

static int kp_workspace(opb_ctx* ctx, size_t floats, int records, size_t stage_bytes, KpWs** out) {
  if (!ctx->kp_ws) ctx->kp_ws = new KpWs();
  KpWs* ws = ctx->kp_ws;
  if (ws->cap < floats || ws->records < records) {
    OPB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    cudaFree(ws->up); cudaFree(ws->tmp); cudaFree(ws->res); cudaFreeHost(ws->h_res);
    ws->up = ws->tmp = nullptr; ws->res = nullptr; ws->h_res = nullptr; ws->cap = 0; ws->records = 0;
    OPB_CUDA(ctx, cudaMalloc(reinterpret_cast<void**>(&ws->up), floats * 4));
    OPB_CUDA(ctx, cudaMalloc(reinterpret_cast<void**>(&ws->tmp), floats * 4));
    OPB_CUDA(ctx, cudaMalloc(reinterpret_cast<void**>(&ws->res), sizeof(ChannelMax) * records));
    OPB_CUDA(ctx, cudaMallocHost(reinterpret_cast<void**>(&ws->h_res), sizeof(ChannelMax) * records));
    ws->cap = floats; ws->records = records;
  }
  if (ws->stage_cap < stage_bytes) {
    OPB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    cudaFreeHost(ws->h_stage);
    ws->h_stage = nullptr; ws->stage_cap = 0;
    OPB_CUDA(ctx, cudaMallocHost(reinterpret_cast<void**>(&ws->h_stage), stage_bytes));
    ws->stage_cap = stage_bytes;
  }
  *out = ws;
  return OPB_OK;
}

// Appends a crop of h x w maps to a ragged table: its place in the packed maps and its first block in the upsample
// and per-plane launches.
static void kp_add_crop(RaggedMaps& t, int h, int w, int mirror, int planes, long long& floats, int& blk_up,
                        int& blk_plane) {
  t.off = floats; t.h = h; t.w = w; t.mirror = mirror ? 1 : 0; t.pad_ = 0;
  t.tiles_x = (w + 31) / 32;
  t.tiles = t.tiles_x * ((h + 7) / 8);
  t.blk_up = blk_up; t.blk_plane = blk_plane;
  floats += static_cast<long long>(planes) * h * w;
  blk_up += t.tiles * ((planes + kKpUpsamplePlanes - 1) / kKpUpsamplePlanes);
  blk_plane += t.tiles * planes;
}

// Smooths ws->up (both passes) and takes the per-plane maximum of every crop of `tab` (d_tab: its device copy), then
// one copy of all records to the host and one synchronise.  out [n][planes][3], valid [n][planes].
static int kp_peaks(opb_ctx* ctx, KpWs* ws, int n, int planes, const RaggedMaps* tab, const RaggedMaps* d_tab,
                    int blk_plane, double thresh, double* out, int32_t* valid) {
  const dim3 block(32, 8);
  gauss_pass_ragged_kernel<0><<<blk_plane, block, 0, ctx->stream>>>(ws->up, ws->tmp, d_tab, n, ctx->taps);
  gauss_pass_ragged_kernel<1><<<blk_plane, block, 0, ctx->stream>>>(ws->tmp, ws->up, d_tab, n, ctx->taps);
  channel_argmax_ragged_kernel<<<n * planes, 256, 0, ctx->stream>>>(ws->up, d_tab, planes, ws->res);
  ctx->launches += 3;
  OPB_CUDA(ctx, cudaGetLastError());
  OPB_CUDA(ctx, cudaMemcpyAsync(ws->h_res, ws->res, sizeof(ChannelMax) * n * planes, cudaMemcpyDeviceToHost, ctx->stream));
  OPB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  const float th = static_cast<float>(thresh);      // `max_value > thresh` with a float32 max_value compares in float32
  for (int i = 0; i < n; ++i) {
    const int W = tab[i].w;
    for (int c = i * planes; c < (i + 1) * planes; ++c) {
      const ChannelMax& r = ws->h_res[c];
      valid[c] = r.value > th ? 1 : 0;
      // np.array(np.where(g == m)).flatten() = [y0..yk-1, x0..xk-1]; the reference reads [1] as x and [0] as y
      const int y0 = r.key0 / W, x0 = r.key0 - y0 * W;
      out[c * 3 + 0] = r.count >= 2 ? static_cast<double>(r.key1 / W) : static_cast<double>(x0);
      out[c * 3 + 1] = static_cast<double>(y0);
      out[c * 3 + 2] = static_cast<double>(r.value);
    }
  }
  return OPB_OK;
}

// One chunk of at most kKpMaxCrops crops (arguments checked by the caller).
static int kp_detect_chunk(opb_ctx* ctx, const uint8_t* imgs, int imgs_loc, int n, const int32_t* dims,
                           const int32_t* mirror, int net, double thresh, double* out, int32_t* valid, float* maps_out) {
  const int planes = ctx->kp_out - 1;              // the last channel is background (face_detector.py:59)
  const int bucket = kp_bucket(n), lo = net / 8;
  Chain* ch = nullptr;
  int rc = get_chain(ctx, bucket, net, net, &ch);
  if (rc) return rc;
  std::vector<RaggedCrop> rz(n);
  std::vector<RaggedMaps> tab(n);
  size_t crop_bytes = 0;
  long long floats = 0;
  int blk_up = 0, blk_plane = 0;
  for (int i = 0; i < n; ++i) {
    const int h = dims[2 * i], w = dims[2 * i + 1];
    rz[i].src_off = static_cast<long long>(crop_bytes);
    rz[i].h0 = h; rz[i].w0 = w;
    rz[i].scale_x = 1.0 / (static_cast<double>(net) / w);   // cv2::resize: scale = 1 / (dsize / ssize)
    rz[i].scale_y = 1.0 / (static_cast<double>(net) / h);
    crop_bytes += static_cast<size_t>(h) * w * 3;
    kp_add_crop(tab[i], h, w, mirror[i], planes, floats, blk_up, blk_plane);
  }
  // one upload: [resize table | post-process table | crops (host input only)]
  const size_t off_tab = align256(sizeof(RaggedCrop) * n), off_img = align256(off_tab + sizeof(RaggedMaps) * n);
  const size_t up_bytes = imgs_loc == OPB_HOST ? off_img + crop_bytes : off_tab + sizeof(RaggedMaps) * n;
  KpWs* ws = nullptr;
  if ((rc = kp_workspace(ctx, static_cast<size_t>(floats), n * planes, up_bytes, &ws))) return rc;
  if ((rc = ensure_ingest(ctx, up_bytes))) return rc;
  memcpy(ws->h_stage, rz.data(), sizeof(RaggedCrop) * n);
  memcpy(ws->h_stage + off_tab, tab.data(), sizeof(RaggedMaps) * n);
  if (imgs_loc == OPB_HOST) memcpy(ws->h_stage + off_img, imgs, crop_bytes);
  OPB_CUDA(ctx, cudaMemcpyAsync(ctx->ingest_buf, ws->h_stage, up_bytes, cudaMemcpyHostToDevice, ctx->stream));
  const uint8_t* d_src = imgs_loc == OPB_HOST ? ctx->ingest_buf + off_img : imgs;
  const RaggedCrop* d_rz = reinterpret_cast<const RaggedCrop*>(ctx->ingest_buf);
  const RaggedMaps* d_tab = reinterpret_cast<const RaggedMaps*>(ctx->ingest_buf + off_tab);
  // slots past the last crop are zeroed; the network computes every image of the batch independently, and nothing
  // after it reads those slots
  const size_t slot_bytes = static_cast<size_t>(net) * net * 3;
  if (bucket > n) OPB_CUDA(ctx, cudaMemsetAsync(ch->img_u8 + n * slot_bytes, 0, (bucket - n) * slot_bytes, ctx->stream));
  // cv2.resize(crop, (368, 368)) (face_detector.py:31) of every crop, bit-exact uint8 INTER_LINEAR
  resize_linear_u8_ragged_kernel<<<dim3((net + 31) / 32, (net + 7) / 8, n), dim3(32, 8), 0, ctx->stream>>>(
      d_src, d_rz, ch->img_u8, net, net);
  ctx->launches++;
  OPB_CUDA(ctx, cudaGetLastError());
  ch->img_u8_src = nullptr;
  if ((rc = run_chain(ctx, ch, true))) return rc;
  // F.resize_images(hs[-1], (crop_h, crop_w)) (face_detector.py:38) of every crop
  upsample_bilinear_ac_ragged_kernel<<<blk_up, dim3(32, 8), 0, ctx->stream>>>(
      ch->heat_lo, static_cast<long long>(ctx->kp_out) * lo * lo, planes, lo, lo, d_tab, n, ws->up, kKpUpsamplePlanes);
  ctx->launches++;
  OPB_CUDA(ctx, cudaGetLastError());
  if (maps_out && (rc = copy_out(ctx, maps_out, ws->up, static_cast<size_t>(floats) * 4, OPB_HOST))) return rc;
  return kp_peaks(ctx, ws, n, planes, tab.data(), d_tab, blk_plane, thresh, out, valid);
}

int opb_keypoints_from_heatmaps(opb_ctx* ctx, const float* heat, int heat_loc, int planes, int h, int w, int mirror,
                                double thresh, double* out, int32_t* valid) {
  if (!ctx || !heat || !out || !valid || planes <= 0 || h <= 0 || w <= 0) return OPB_ERR_ARG;
  cudaSetDevice(ctx->device);
  RaggedMaps tab;
  long long floats = 0;
  int blk_up = 0, blk_plane = 0;
  kp_add_crop(tab, h, w, mirror, planes, floats, blk_up, blk_plane);
  KpWs* ws = nullptr;
  int rc = kp_workspace(ctx, static_cast<size_t>(floats), planes, sizeof(tab), &ws);
  if (rc) return rc;
  if ((rc = ensure_ingest(ctx, sizeof(tab)))) return rc;
  memcpy(ws->h_stage, &tab, sizeof(tab));
  OPB_CUDA(ctx, cudaMemcpyAsync(ctx->ingest_buf, ws->h_stage, sizeof(tab), cudaMemcpyHostToDevice, ctx->stream));
  if ((rc = copy_in(ctx, ws->up, heat, static_cast<size_t>(floats) * 4, heat_loc))) return rc;
  return kp_peaks(ctx, ws, 1, planes, &tab, reinterpret_cast<const RaggedMaps*>(ctx->ingest_buf), blk_plane, thresh,
                  out, valid);
}

int opb_keypoints_detect_batch(opb_ctx* ctx, const uint8_t* imgs, int imgs_loc, int n, const int32_t* dims,
                               const int32_t* mirror, int net_size, double thresh, double* out, int32_t* valid,
                               float* maps_out) {
  if (!ctx) return OPB_ERR_ARG;
  if (n < 0) OPB_FAIL(ctx, OPB_ERR_ARG, "opb_keypoints_detect_batch: n = " + std::to_string(n) + " < 0");
  if (!ctx->kp_out) OPB_FAIL(ctx, OPB_ERR_STATE, "this context holds the pose net: load FaceNet / HandNet weights first");
  if (n == 0) return OPB_OK;
  if (!imgs || !dims || !mirror || !out || !valid) OPB_FAIL(ctx, OPB_ERR_ARG, "opb_keypoints_detect_batch: null argument");
  if (net_size <= 0 || net_size % 8) OPB_FAIL(ctx, OPB_ERR_ARG, "net_size must be a positive multiple of 8");
  for (int i = 0; i < n; ++i)
    if (dims[2 * i] <= 0 || dims[2 * i + 1] <= 0)
      OPB_FAIL(ctx, OPB_ERR_ARG, "crop " + std::to_string(i) + " has size " + std::to_string(dims[2 * i]) + "x" +
                                     std::to_string(dims[2 * i + 1]));
  cudaSetDevice(ctx->device);
  const int planes = ctx->kp_out - 1;
  for (int c0 = 0; c0 < n; c0 += kKpMaxCrops) {
    const int m = std::min(n - c0, kKpMaxCrops);
    int rc = kp_detect_chunk(ctx, imgs, imgs_loc, m, dims + 2 * c0, mirror + c0, net_size, thresh,
                             out + static_cast<size_t>(c0) * planes * 3, valid + static_cast<size_t>(c0) * planes,
                             maps_out);
    if (rc) return rc;
    for (int i = c0; i < c0 + m; ++i) {
      const size_t px = static_cast<size_t>(dims[2 * i]) * dims[2 * i + 1];
      imgs += px * 3;
      if (maps_out) maps_out += px * planes;
    }
  }
  return OPB_OK;
}

int opb_keypoints_detect(opb_ctx* ctx, const uint8_t* img, int img_loc, int img_h, int img_w, int net_size, int mirror,
                         double thresh, double* out, int32_t* valid, float* maps_out) {
  if (!ctx || !img || !out || !valid || img_h <= 0 || img_w <= 0) return OPB_ERR_ARG;
  const int32_t dims[2] = {img_h, img_w}, mir[1] = {mirror};
  return opb_keypoints_detect_batch(ctx, img, img_loc, 1, dims, mir, net_size, thresh, out, valid, maps_out);
}

void* opb_device_buffer(opb_ctx* ctx, int which) {
  if (!ctx) return nullptr;
  Chain* ch = ctx->last_chain;
  PostWs* ws = ctx->last_post;
  switch (which) {
    case 0: return ch ? ch->paf_lo : nullptr;
    case 1: return ch ? ch->heat_lo : nullptr;
    case 2: return ws ? ws->pafs : nullptr;
    case 3: return ws ? ws->heat : nullptr;
    case 4: return ws ? ws->headers : nullptr;
    case 5: return ws ? ws->persons : nullptr;
    case 6: return ws ? ws->peaks : nullptr;
    case 7: return ch ? ch->img_u8 : nullptr;
    default: return nullptr;
  }
}

int opb_time_stage(opb_ctx* ctx, const char* stage, int reps, float* ms) {
  if (!ctx || !stage || !ms || reps <= 0) return OPB_ERR_ARG;
  cudaSetDevice(ctx->device);
  Chain* ch = ctx->last_chain;
  PostWs* ws = ctx->last_post;
  const std::string s(stage);
  cudaEvent_t e0, e1;
  OPB_CUDA(ctx, cudaEventCreate(&e0));
  OPB_CUDA(ctx, cudaEventCreate(&e1));
  int rc = OPB_OK;
  int n_launch = 0;
  auto run_once = [&]() -> int {
    if (s == "upsample_paf" || s == "upsample_heat" || s == "peaks" || s == "paf_integral" || s == "limb_assign" ||
        s == "group") {
      if (!ws || (!ch && !ws->last_paf_lo)) { ctx->err = "no cached pipeline to time"; return OPB_ERR_STATE; }
      const int n = ws->N, h8 = ws->last_h8 ? ws->last_h8 : ch->H / 8, w8 = ws->last_w8 ? ws->last_w8 : ch->W / 8;
      const float* plo = ws->last_paf_lo ? ws->last_paf_lo : ch->paf_lo;     // same maps as the last batch
      const float* hlo = ws->last_heat_lo ? ws->last_heat_lo : ch->heat_lo;
      const double ilen = ws->last_img_len > 0 ? ws->last_img_len : ws->W;
      if (s == "upsample_paf") { ++n_launch; return launch_upsample(ctx, plo, n * 38, h8, w8, ws->pafs, ws->H, ws->W); }
      if (s == "upsample_heat") { ++n_launch; return launch_upsample(ctx, hlo, n * 19, h8, w8, ws->heat, ws->H, ws->W); }
      if (s == "peaks") {
        if (ctx->fused_peaks == 1 || ctx->fused_peaks == 3) { n_launch += 2; return launch_peaks(ctx, ws, hlo, n, 19, ws->H, ws->W, h8, w8); }
        if (ctx->fused_peaks == 2) { n_launch += 2; return launch_peaks(ctx, ws, hlo, n, 19, ws->H, ws->W, h8, w8, ws->heat); }
        n_launch += 3;
        return launch_peaks(ctx, ws, ws->heat, n, 19, ws->H, ws->W);
      }
      if (s == "paf_integral") {
        n_launch += 2;
        if (ctx->paf_lowres) return launch_connections(ctx, ws, plo, n, ws->H, ws->W, ilen, h8, w8);
        return launch_connections(ctx, ws, ws->pafs, n, ws->H, ws->W, ilen);
      }
      if (s == "limb_assign") {
        ++n_launch;
        dim3 g2(19, n);
        limb_assign_kernel<<<g2, kAssignThreads, 0, ctx->stream>>>(ws->peaks, ws->idx_list, ws->type_start,
                                                                   ctx->prm.max_peaks, 18, ctx->pc, ws->cands, ws->cands_alt,
                                                                   ws->cand_counts, ctx->prm.max_candidates, ws->conns,
                                                                   ws->conn_counts, ctx->conn_cap, ws->status);
        return OPB_OK;
      }
      ++n_launch;
      return launch_group(ctx, ws, n, true);
    }
    if (!ch) { ctx->err = "no cached conv chain to time"; return OPB_ERR_STATE; }
    bool any = false;
    for (Op& op : ch->ops) {
      if (s == "conv_chain" || op.tag == s) {
        any = true;
        ++n_launch;
        int r = launch_op(ctx, ch, op);
        if (r) return r;
      }
    }
    if (!any) { ctx->err = "unknown stage " + s; return OPB_ERR_ARG; }
    return OPB_OK;
  };
  rc = run_once();  // warm-up
  if (!rc) {
    n_launch = 0;
    cudaEventRecord(e0, ctx->stream);
    for (int i = 0; i < reps && !rc; ++i) rc = run_once();
    cudaEventRecord(e1, ctx->stream);
    cudaError_t e = cudaEventSynchronize(e1);
    if (e != cudaSuccess && !rc) { ctx->err = cudaGetErrorString(e); rc = OPB_ERR_CUDA; }
    float t = 0.f;
    cudaEventElapsedTime(&t, e0, e1);
    *ms = t / reps;
  }
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  return rc;
}

int opb_test_conv(opb_ctx* ctx, const float* x, int n, int h, int w, int cin, const float* W, const float* b, int cout,
                  int ksize, int relu, int precision_mode, float* y) {
  if (!ctx || !x || !W || !b || !y) return OPB_ERR_ARG;
  cudaSetDevice(ctx->device);
  const bool split = precision_mode == OPB_PRECISION_PARITY, comp = precision_mode == OPB_PRECISION_COMP;
  const int saved_precision = ctx->precision;
  ctx->precision = precision_mode;
  const int pool = (relu >> 1) & 1;   // bit 1 of `relu`: fuse the 2x2 max-pool (y is then [N,H/2,W/2,Cout])
  relu &= 1;
  if (pool && ((h | w) & 1)) { ctx->precision = saved_precision; OPB_FAIL(ctx, OPB_ERR_ARG, "pooled test conv needs even H, W"); }
  const int oh = pool ? h / 2 : h, ow = pool ? w / 2 : w;
  Chain tmp;
  int rc = OPB_OK;
  const int cin_pad = round_up(cin, 64);
  const int cout_pad = cout <= 48 ? 48 : round_up(cout, 64);
  if (cout_pad > 256 && cout_pad % 256) { ctx->precision = saved_precision; OPB_FAIL(ctx, OPB_ERR_ARG, "test conv: cout must be <=256 or a multiple of 256"); }
  HostLayer L;
  L.cin = cin; L.cout = cout; L.ks = ksize;
  L.W.assign(W, W + static_cast<size_t>(cout) * cin * ksize * ksize);
  L.b.assign(b, b + cout);
  ctx->host_layers["__test__"] = L;
  Act in, out;
  std::vector<__half> hx;
  std::vector<__half> hy;
  do {
    if ((rc = pack_weights(ctx, "__test__", {{"__test__", cout_pad}}, identity_map(cin, cin_pad), ksize, precision_mode))) break;
    if ((rc = alloc_act(ctx, &tmp, &in, n, h, w, cin_pad))) break;
    // (the correction plane of the compensated precision is laid out in whole 64-channel chunks)
    if ((rc = alloc_act(ctx, &tmp, &out, n, oh, ow, comp ? round_up(cout_pad, 64) : cout_pad))) break;
    hx.assign(static_cast<size_t>(n) * h * w * in.Ctot, __float2half(0.f));
    for (size_t pix = 0; pix < static_cast<size_t>(n) * h * w; ++pix)
      for (int c = 0; c < cin; ++c) {
        const float v = x[pix * cin + c];
        const __half hi = __float2half_rn(v);
        hx[pix * in.Ctot + c] = hi;
        if (split) hx[pix * in.Ctot + in.C + c] = __float2half_rn(v - __half2float(hi));
        if (comp) {
          uint8_t* cb = reinterpret_cast<uint8_t*>(&hx[pix * in.Ctot + in.C]) + comp_byte_off(c);
          cb[0] = f32_to_act8((v - __half2float(hi)) * kCompLoScale);
          cb[64] = f32_to_act8(v);
        }
      }
    cudaError_t e = cudaMemcpyAsync(in.p, hx.data(), hx.size() * 2, cudaMemcpyHostToDevice, ctx->stream);
    if (e != cudaSuccess) { ctx->err = cudaGetErrorString(e); rc = OPB_ERR_CUDA; break; }
    ConvSpec s{};
    s.in[0] = &in; s.in_coff[0] = 0; s.wkey[0] = "__test__"; s.out[0] = &out; s.out_coff[0] = 0;
    s.cout_valid[0] = cout; s.n_problems = 1; s.relu = relu; s.pool = pool;
    if ((rc = add_conv(ctx, &tmp, "__test__", s))) break;
    if ((rc = launch_op(ctx, &tmp, tmp.ops[0]))) break;
    hy.resize(static_cast<size_t>(n) * oh * ow * out.Ctot);
    e = cudaMemcpyAsync(hy.data(), out.p, hy.size() * 2, cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    if (e != cudaSuccess) { ctx->err = std::string("test conv: ") + cudaGetErrorString(e); rc = OPB_ERR_CUDA; break; }
    for (size_t pix = 0; pix < static_cast<size_t>(n) * oh * ow; ++pix)
      for (int c = 0; c < cout; ++c) {
        float v = __half2float(hy[pix * out.Ctot + c]);
        if (split) v += __half2float(hy[pix * out.Ctot + out.C + c]);
        if (comp)   // hi + the 8-bit-float lo
          v += act8_to_f32(reinterpret_cast<const uint8_t*>(&hy[pix * out.Ctot + out.C])[comp_byte_off(c)]) / kCompLoScale;
        y[pix * cout + c] = v;
      }
  } while (0);
  cudaStreamSynchronize(ctx->stream);
  free_all(tmp.allocs);
  ctx->host_layers.erase("__test__");
  ctx->packed.erase("__test__");
  ctx->precision = saved_precision;
  return rc;
}

}  // extern "C"
