// libdavo_b200.so -- C ABI (include/davo_b200.h) over the sm_100a kernels.
// Host side: variant config -> layer plans (K-step tables, TF32 weight packing,
// TMA tensor maps) -> per-micro-batch launch sequence.
#include "../../include/davo_b200.h"

#include <cuda.h>
#include <cuda_runtime.h>
#include <atomic>

#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <cctype>
#include <sched.h>
#if defined(__SSE2__)
#include <emmintrin.h>
#endif

#include <condition_variable>
#include <functional>
#include <climits>
#include <map>
#include <set>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "conv_cm.cuh"
#include "conv_pm.cuh"
#include "frontend.cuh"
#include "features.cuh"
#include "comm.cuh"
#include "trajectory.cuh"
#include "odometry_many.cuh"
#include "odometry_state.cuh"
#include "bn.cuh"
#include "jpeg.cuh"
#include "host_convert.h"

using namespace davo;

namespace {

thread_local std::string g_create_error;

// A few host threads for the one CPU pass of the host-buffer entry point (label floats -> bytes).
class HostPool {
 public:
  explicit HostPool(int n) {
    for (int i = 0; i < n; ++i) workers_.emplace_back([this, i] { loop(i); });
  }
  ~HostPool() {
    { std::lock_guard<std::mutex> g(m_); stop_ = true; ++epoch_; }
    cv_.notify_all();
    for (auto& t : workers_) t.join();
  }
  int size() const { return (int)workers_.size() + 1; }
  // fn(part, parts) on every worker and on the calling thread; returns when all are done
  void run(const std::function<void(int, int)>& fn) {
    {
      std::lock_guard<std::mutex> g(m_);
      fn_ = &fn; pending_ = (int)workers_.size(); ++epoch_;
    }
    cv_.notify_all();
    fn((int)workers_.size(), size());
    std::unique_lock<std::mutex> g(m_);
    done_.wait(g, [this] { return pending_ == 0; });
  }
 private:
  void loop(int id) {
    unsigned long seen = 0;
    for (;;) {
      const std::function<void(int, int)>* fn;
      {
        std::unique_lock<std::mutex> g(m_);
        cv_.wait(g, [&] { return epoch_ != seen; });
        seen = epoch_;
        if (stop_) return;
        fn = fn_;
      }
      (*fn)(id, size());
      {
        std::lock_guard<std::mutex> g(m_);
        if (--pending_ == 0) done_.notify_one();
      }
    }
  }
  std::vector<std::thread> workers_;
  std::mutex m_;
  std::condition_variable cv_, done_;
  const std::function<void(int, int)>* fn_ = nullptr;
  int pending_ = 0;
  unsigned long epoch_ = 0;
  bool stop_ = false;
};

struct HostTensor {
  std::vector<int64_t> shape;
  std::vector<float> data;
};

// TF 'SAME' (asymmetric) padding: out = ceil(in / stride), pad_before = total / 2.
struct SamePad { int out, before, after; };
SamePad same_pad(int in, int k, int stride, int dil) {
  SamePad s;
  s.out = (in + stride - 1) / stride;
  int eff = (k - 1) * dil + 1;
  int total = (s.out - 1) * stride + eff - in;
  if (total < 0) total = 0;
  s.before = total / 2;
  s.after = total - s.before;
  return s;
}

float host_round_tf32(float x) {   // cvt.rna.tf32.f32
  uint32_t u;
  memcpy(&u, &x, 4);
  if ((u & 0x7F800000u) == 0x7F800000u) return x;
  u = (u + 0x1000u) & 0xFFFFE000u;
  memcpy(&x, &u, 4);
  return x;
}

// The TF32 neighbour of x on the other side of the exact value (x_hat = RN result).
float tf32_other_neighbour(float x, float x_hat) {
  if (x_hat == x) return x_hat;
  uint32_t u;
  memcpy(&u, &x_hat, 4);
  const bool away = fabsf(x_hat) > fabsf(x);      // RN went away from zero -> step towards zero
  if (away) u -= 0x2000u;
  else if ((u & 0x7FFFFFFFu) == 0) { float t = ldexpf(1.0f, -126); u = 0; memcpy(&u, &t, 4); if (x < 0) u |= 0x80000000u; }
  else u += 0x2000u;
  float r;
  memcpy(&r, &u, 4);
  return r;
}

int floordiv(int a, int b) { return (a >= 0) ? a / b : -((-a + b - 1) / b); }
int posmod(int a, int b) { return a - floordiv(a, b) * b; }

struct Layer {
  const char* name;
  int k, stride, dil;
  int Hin, Win, Cin_total;     // input tensor
  int Cin_g, groups;           // channels reduced per group
  int BN;                      // output channels per group (= MMA N)
  int Hout, Wout, out_stride;
  // Buffer pitches (rows x columns actually allocated): odd maps are padded to even with a zero
  // row / column that is never written, so that the stride-2 view [H/2][2][W/2][2C] exists (the
  // non-dilated nets go down to 4x13, 2x7, 1x4 maps).  Equal to the map size everywhere else.
  int Hin_p = 0, Win_p = 0, Hout_p = 0, Wout_p = 0;
  bool pitched_out() const { return Hout_p != Hout || Wout_p != Wout; }
  int pad_t, pad_l;
  int epi;
  int tiles_h, tiles_w;
  // device
  float* d_in = nullptr;
  float* d_out = nullptr;
  float* d_wpack = nullptr;    // [groups][n_ksteps][BN][32]
  float* d_bias = nullptr;     // [groups*BN]
  float* d_whwio[2] = {nullptr, nullptr};   // unpacked HWIO per group (direct debug path)
  int cmap[16];
  int use_cmap = 0;
  int Cin_w = 0;               // weight input channels (HWIO 'I')
  int orient = 0;              // 0: pixels on the MMA M axis (conv_pm), 1: channels on M (conv_cm)
  int npix = 128;              // output pixels per tile: 128 = 16x8 (pm, or cm on short maps), 256 = 32x8
  int m_blocks = 1;            // cm: 128-channel blocks per group
  bool cm_staged = false;      // cm: store epilogue through shared memory + TMA tile stores
  bool cm_cluster = false;     // cm: 2-CTA clusters, each weight slab fetched once and multicast
  bool b_resident = false;     // pm: all weight slabs stay in shared memory
  bool cin_shared = false;     // grouped layer whose groups all read the same input channels (cin_group_off = 0)
  int strips = -1;             // halo patches cut into one vertical strip per filter column: -1 = decided by plan_layer
                               // (and recorded here); a latency twin takes its big plan's choice so that both accumulate
                               // every output element in the same tap order (bit-identical results at any batch size)
  int wide_G = 0;              // pm, column-widened: output pixels per M row (0 = off)
  int wide_tw = 0;             //   runs per tile row (tile = 128/wide_tw rows x wide_tw runs)
  bool fused_front = false;    // cnv1, widened, 8-channel input: planned with the staging area of the fused front end (conv_pm.cuh: FUSED)
  int pc2w[16];                // input tensor channel -> HWIO input channel of the weights, -1: none (cnv1: packed input)
  int smem_bytes = 0;
  float* d_beta = nullptr;     // -batch_norm: BatchNorm/beta of this layer [out_stride] (bn.cuh)
  CUtensorMap tmA, tmB;          // activation (patch) map, weight map
  CUtensorMap tmO;               // pm store epilogue: output tiles (TMA store)
  CUtensorMap tmB64;             // cm clusters: weight map with a 64-row box (half a slab per CTA)
  pm::ConvParams prm_pm;
  cm::ConvParams prm_cm;
};

}  // namespace

struct davo_ctx {
  davo_config cfg;
  int device = 0;
  int num_sms = 148;
  std::string err;
  std::map<std::string, HostTensor> weights;
  bool finalized = false;
  uint64_t weights_digest = 0;      // of the values davo_finalize_weights was given (weights_digest_of)
  int mb = 0;                       // frame pairs per micro-batch
  int packed_c = 16;                // channels per pixel of the packed PoseNN input (8 or 16)
  int conv_impl = 0;                // 0 tcgen05 (product), 1 direct fp32 (debug cross-check)
  bool fuse_front = false;          // cnv1 builds its operand from the raw inputs: pack8_kernel is not launched (conv_pm.cuh: FUSED)
  FrontParams fp_cur;               // the front-end parameters of the pass being launched (the fused cnv1 takes them)
  bool compensated_rounding = true; // TF32 weight rounding directions chosen so tap sums cancel
  bool pdl = true;                  // programmatic dependent launch of every kernel of a pass
  std::vector<Layer> layers;        // cnv1..cnv7
  // Latency plans (BASELINE configs[0], batch 1): the channels-on-M layers re-planned with 128-pixel tiles (16 x 8)
  // instead of 256.  A 256-pixel tile costs 128 cycles per MMA, a 128-pixel one 64: when the big tiling cannot fill
  // the SMs anyway (few units), half-size tiles halve the layer's critical path at no cost.  Same buffers, own
  // weight pack and tensor maps.  layers_small[i].npix == 0: layer i has no such plan.
  std::vector<Layer> layers_small;
  // device buffers
  std::vector<void*> allocs;
  unsigned int* d_poolcnt = nullptr;
  float *d_pool = nullptr, *d_attw = nullptr, *d_packed = nullptr, *d_sum7 = nullptr;
  float *d_sew = nullptr, *d_staticw = nullptr, *d_wpred = nullptr, *d_bpred = nullptr;
  float* d_c7tmp = nullptr;         // direct path only
  // -se_insert: excitation of cnv5 per branch (frontend.cuh: se5_*)
  float *d_se5w = nullptr, *d_se5part = nullptr, *d_se5scale = nullptr, *d_se5out = nullptr;
  unsigned int* d_se5cnt = nullptr;
  int nparts7 = 0;
  int nbr = 2;                      // pose branches: 2 (rotation, translation: decouple nets) or 1 (couple nets)
  bool unit_sample = false;         // non-shared nets: one evaluation per sample on (tgt, src0, src1)
  int max_units() const { return unit_sample ? cfg.max_batch : 2 * cfg.max_batch; }
  // host-buffer entry point staging
  static constexpr int kStage = 3;  // staging buffers: copy of chunk i+2 never waits for compute of chunk i
  uint8_t* s_img[kStage] = {};
  float *s_flow[kStage] = {}, *s_seg[kStage] = {}, *s_depth[kStage] = {}, *s_pose = nullptr;
  // Labels cross PCIe as bytes: converted on the CPU into pinned staging (h_seg8), copied to s_seg8.
  uint8_t *h_seg8[kStage] = {}, *s_seg8[kStage] = {};
  cudaEvent_t ev_seg8[kStage] = {};  // h_seg8[i] has been read by its copy
  // The flow crosses PCIe as binary16 (host_convert.cpp; frontend.cuh: flow_q): h_flow16 -> s_flow16,
  // [chunk][2 planes][H][W][2] halves.  ev_seg8[i] covers both pinned staging buffers of slot i.
  uint16_t *h_flow16[kStage] = {}, *s_flow16[kStage] = {};
  bool host_flow16 = true;
  int numa_node = -1, numa_cpus = 0;      // davo_bind_host_numa
  nvjpegHandle_t jpeg_handle = nullptr;   // davo_decode_jpeg_batch (jpeg.cuh)
  nvjpegJpegState_t jpeg_state = nullptr;
  int* d_pipe = nullptr;                  // front_pipeline_kernel: work counter, exit counter, launch counter, [mb] ready flags
  double* d_bn_part = nullptr;            // -batch_norm scratch: partial sums, means, reciprocal deviations (bn.cuh)
  float *d_bn_mean = nullptr, *d_bn_rstd = nullptr;
  void* d_traj_scratch = nullptr;         // davo_compose_trajectory / davo_kitti_errors: relative motions, distances, segments
  size_t traj_scratch_bytes = 0;
  float flow16_frac = 0.75f;              // share of a chunk's samples (of a push's flow entries) converted on the CPU (the
                                          // rest keeps the copy engine busy)
  HostPool* pool = nullptr;
  bool host_seg8 = true;
  int s_chunk = 0;                  // samples per staging buffer
  cudaStream_t copy_stream = nullptr;
  cudaEvent_t ev_copied[kStage] = {}, ev_consumed[kStage] = {}, ev_start = nullptr;
  static constexpr int kTickets = 8;      // asynchronous host calls whose completion can still be waited for by name
  cudaEvent_t ev_host_done[kTickets] = {};
  long long host_tickets = 0, host_calls = 0;
  long long last_h2d = 0, last_d2h = 0;
  // last forward
  int last_launches = 0;
  int last_npairs_mb = 0;
  InputView last_in{};              // inputs of the last forward's last micro-batch (davo_profile_layers runs on them)
  float* last_pose = nullptr; int last_B = 0; int last_pairs = 0;
  // davo_forward_sequence_host: the frames of a call (images, labels, depth) staged at their final place, so that a
  // frame shared by two chunks crosses PCIe once; two sets, so that a call's copies can run under the previous call
  uint8_t* q_img[2] = {}; uint8_t* q_seg8[2] = {}; float *q_seg[2] = {}, *q_depth[2] = {};
  cudaEvent_t ev_q_done[2] = {};    // the call that last used set i has finished reading it
  long long q_calls = 0;
  // odometry pushes: one stacked-triplet staging batch of max_batch samples (input_view.cuh: stacked_view) and
  // its poses, allocated by the first push of any kind; the per-call session and sample descriptors and the attention
  // unit table and rows go from a pinned ring slot to its device twin in one copy, and a slot is refilled once the call
  // that used it has finished
  uint8_t *m_img = nullptr, *m_lab = nullptr;
  float *m_depth = nullptr, *m_flow = nullptr, *m_pose = nullptr;
  static constexpr int kManyRing = 4;
  void *m_hdesc[kManyRing] = {}, *m_ddesc[kManyRing] = {};
  size_t m_desc_cap[kManyRing] = {};
  cudaEvent_t m_ev[kManyRing] = {};
  long long m_calls = 0;
  // host sessions' pushes: two arrivals sets (device; pinned byte labels and binary16 flow entries), the caller's
  // frames and flow entries of a call at the indices the stage kernel reads them; set i is refilled once the stage and
  // carry kernels of the call that last used it have finished (a_done[i]), so that the copies of call t+1 run under the
  // forward of call t
  uint8_t* a_dev[2] = {}; uint8_t* a_pin[2] = {};
  size_t a_dev_cap[2] = {}, a_pin_cap[2] = {};
  cudaEvent_t a_copied[2] = {}, a_done[2] = {};
  long long a_calls = 0;
  float* m_hpose = nullptr;           // the pose rows of each session's push, [max_batch,2,6], copied to the host from here
  // davo_odometry_save_many / load_many: a staging area laid out as the caller's blobs (a chunk of them at a time), and
  // the call's blob descriptors, headers and checksum accumulators in one pinned area and its device twin; grown on
  // demand, used by one synchronous call at a time
  uint8_t* b_stage = nullptr;
  size_t b_stage_cap = 0;
  void *b_hdesc = nullptr, *b_ddesc = nullptr;
  size_t b_desc_cap = 0;
  std::map<std::pair<const void*, int>, int> max_clusters;   // by (kernel, dynamic shared memory)
  float depth_thres = 0.f;          // -se_flow_on_depthseg_seplayers: the variable se_flow/depth_threshold
  // mode='feature' (features.cuh)
  float* d_wheel = nullptr;         // Middlebury colour wheel / 255
  unsigned int* d_maxrad = nullptr; // largest flow magnitude per source frame
  // attention outputs of odometry pushes (features.cuh: attention_out_kernel).  While a push that asked for them runs
  // its forward, att_units / att_rows are the device unit table of the forward being launched and its destination
  // rows (in the call's m_ddesc slot); NULL otherwise.  Host sessions' maps and weights are written to att_stage and
  // copied back on the caller's stream.
  const int4* att_units = nullptr;
  const AttRow* att_rows = nullptr;
  float* att_stage = nullptr;
  size_t att_stage_cap = 0;
  // pose all-gather (comm.cuh): the handle's own communicator, if davo_comm_create made one
  davo_comm::Comm comm = nullptr;
  int comm_rank = 0, comm_world = 1;
};

namespace {

int fail(davo_ctx* c, int code, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  if (c) c->err = buf; else g_create_error = buf;
  return code;
}

#define CU_OK(call)                                                                      \
  do {                                                                                   \
    cudaError_t e_ = (call);                                                             \
    if (e_ != cudaSuccess)                                                               \
      return fail(ctx, DAVO_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), \
                  __FILE__, __LINE__);                                                   \
  } while (0)

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*,
                                  const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                  const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  }
  return fn;
}

// Every kernel of a pass goes through here: programmatic dependent launch (ptx.cuh: pdl_wait), and
// a 2-CTA cluster where the kernel wants one.
template <class... KArgs, class... Args>
int launch_k(davo_ctx* ctx, void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st,
             bool cluster2, Args&&... args) {
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof cfg);
  cudaLaunchAttribute attr[2];
  int na = 0;
  if (ctx->pdl) {
    attr[na].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[na].val.programmaticStreamSerializationAllowed = 1;
    ++na;
  }
  if (cluster2) {
    attr[na].id = cudaLaunchAttributeClusterDimension;
    attr[na].val.clusterDim.x = 2; attr[na].val.clusterDim.y = 1; attr[na].val.clusterDim.z = 1;
    ++na;
  }
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
  cfg.attrs = attr; cfg.numAttrs = na;
  CU_OK(cudaLaunchKernelEx(&cfg, kern, std::forward<Args>(args)...));
  return 0;
}

// Opt the kernel in to `bytes` of dynamic shared memory on this context's device (once per size).  The attribute
// belongs to the kernel on the device, not to a handle, so what has been raised is kept per (device, kernel) for the
// whole process and only ever raised: two handles on one device must not lower it under each other's launches.
std::mutex g_smem_mutex;
std::map<std::pair<int, const void*>, int> g_smem_attr;
template <class K>
int ensure_smem(davo_ctx* ctx, K kern, int bytes) {
  std::lock_guard<std::mutex> lk(g_smem_mutex);
  int& have = g_smem_attr[std::make_pair(ctx->device, reinterpret_cast<const void*>(kern))];
  if (have < bytes) {
    CU_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
    have = bytes;
  }
  return 0;
}

int dev_alloc(davo_ctx* ctx, void** p, size_t bytes) {
  CU_OK(cudaMalloc(p, bytes));
  CU_OK(cudaMemset(*p, 0, bytes));
  ctx->allocs.push_back(*p);
  return 0;
}

const HostTensor* find_w(davo_ctx* ctx, const std::string& name) {
  auto it = ctx->weights.find(name);
  return it == ctx->weights.end() ? nullptr : &it->second;
}

// 64-bit digest of every variable in name order: its name, shape and float32 bits (davo_odometry_move compares two
// handles' weights with it).  Each step, h = f(h ^ word) with f a bijection, so a single differing word changes it.
uint64_t weights_digest_of(const std::map<std::string, HostTensor>& weights) {
  uint64_t h = 0xcbf29ce484222325ull;
  auto mix = [&h](uint64_t x) { h ^= x; h *= 0x100000001b3ull; h ^= h >> 32; };
  for (const auto& kv : weights) {
    mix(kv.first.size());
    for (unsigned char ch : kv.first) mix(ch);
    mix(kv.second.shape.size());
    for (int64_t d : kv.second.shape) mix((uint64_t)d);
    const std::vector<float>& v = kv.second.data;
    for (size_t i = 0; i < v.size(); ++i) {
      uint32_t u;
      memcpy(&u, &v[i], 4);
      mix(u);
    }
  }
  return h;
}

bool shape_is(const HostTensor* t, std::initializer_list<int64_t> s) {
  if (!t || t->shape.size() != s.size()) return false;
  size_t i = 0;
  for (int64_t v : s) if (t->shape[i++] != v) return false;
  return true;
}

// ------------------------------------------------------------ weight rounding --
// tcgen05.mma.kind::tf32 multiplies by W_hat = tf32(W).  Round-to-nearest leaves, for every
// (input channel k, output channel n), a sum over the filter taps S[k][n] = sum_t (W_hat - W)[t]
// that is a random walk of ~sqrt(taps) half-ulps.  After a ReLU every input channel has a
// positive spatial mean, so S becomes an offset of the layer's output that is the same for
// every pixel and every sample: the one rounding error that survives the final spatial mean
// and then accumulates along a composed trajectory (DESIGN.md section 5).  Both TF32
// neighbours of W are within one ulp of it, so the rounding DIRECTION of each weight is chosen
// to make the tap sums cancel:
//     minimise  sum_regions frac_r * S_r^2  +  lambda * sum_t e_t^2
// A region is a set of output pixels that see the same subset of taps (zero padding removes
// whole tap rows / columns near the border -- with dilation 8 on a 32-row map, for half of the
// pixels).  Greedy descent over single direction changes, starting from round-to-nearest.
struct TapRegion { uint64_t mask; double frac; };

std::vector<TapRegion> tap_regions(const Layer& L) {
  std::map<uint32_t, int> rows, cols;
  for (int o = 0; o < L.Hout; ++o) {
    uint32_t m = 0;
    for (int t = 0; t < L.k; ++t) { const int i = o * L.stride + t * L.dil - L.pad_t; if (i >= 0 && i < L.Hin) m |= 1u << t; }
    rows[m]++;
  }
  for (int o = 0; o < L.Wout; ++o) {
    uint32_t m = 0;
    for (int t = 0; t < L.k; ++t) { const int i = o * L.stride + t * L.dil - L.pad_l; if (i >= 0 && i < L.Win) m |= 1u << t; }
    cols[m]++;
  }
  std::vector<TapRegion> out;
  for (auto& r : rows)
    for (auto& c : cols) {
      uint64_t mask = 0;
      for (int ty = 0; ty < L.k; ++ty)
        for (int tx = 0; tx < L.k; ++tx)
          if ((r.first >> ty & 1u) && (c.first >> tx & 1u)) mask |= 1ull << (ty * L.k + tx);
      if (mask) out.push_back(TapRegion{mask, (double)r.second * c.second / ((double)L.Hout * L.Wout)});
    }
  return out;
}

// Returns the TF32 weights, HWIO per group: [g][ty][tx][ci][n].
template <class GetW>
std::vector<float> round_weights_tf32(const Layer& L, GetW getw, bool compensate) {
  const int T = L.k * L.k;
  std::vector<float> out((size_t)L.groups * T * L.Cin_w * L.BN);
  auto at = [&](int g, int t, int ci, int n) -> float& { return out[(((size_t)g * T + t) * L.Cin_w + ci) * L.BN + n]; };
  const std::vector<TapRegion> regions = tap_regions(L);
  const int R = (int)regions.size();
  const double lambda = 0.05;
  std::vector<double> e0(T), e1(T), S(R);
  std::vector<float> w0(T), w1(T);
  std::vector<char> flip(T);
  for (int g = 0; g < L.groups; ++g)
    for (int ci = 0; ci < L.Cin_w; ++ci)
      for (int n = 0; n < L.BN; ++n) {
        for (int t = 0; t < T; ++t) {
          const float w = getw(g, t / L.k, t % L.k, ci, n);
          w0[t] = host_round_tf32(w);
          w1[t] = tf32_other_neighbour(w, w0[t]);
          e0[t] = (double)w0[t] - (double)w;
          e1[t] = (double)w1[t] - (double)w;
          flip[t] = 0;
        }
        if (compensate) {
          for (int r = 0; r < R; ++r) {
            double a = 0.0;
            for (int t = 0; t < T; ++t) if (regions[r].mask >> t & 1ull) a += e0[t];
            S[r] = a;
          }
          for (int iter = 0; iter < 4 * T; ++iter) {
            int best = -1;
            double best_dj = -1e-30;
            for (int t = 0; t < T; ++t) {
              if (w1[t] == w0[t]) continue;
              const double cur = flip[t] ? e1[t] : e0[t], alt = flip[t] ? e0[t] : e1[t];
              const double d = alt - cur;
              double dj = lambda * (alt * alt - cur * cur);
              for (int r = 0; r < R; ++r)
                if (regions[r].mask >> t & 1ull) dj += regions[r].frac * ((S[r] + d) * (S[r] + d) - S[r] * S[r]);
              if (dj < best_dj) { best_dj = dj; best = t; }
            }
            if (best < 0) break;
            const double d = flip[best] ? e0[best] - e1[best] : e1[best] - e0[best];
            for (int r = 0; r < R; ++r) if (regions[r].mask >> best & 1ull) S[r] += d;
            flip[best] ^= 1;
          }
        }
        for (int t = 0; t < T; ++t) at(g, t, ci, n) = flip[t] ? w1[t] : w0[t];
      }
  return out;
}

// Output map of the pixels-on-M store epilogue: one box = 32 floats x tile_w units x (32 / tile_w)
// rows, where a unit is an output pixel (inner = all its channels) or, for the column-widened
// layers, a run of G pixels (inner = G * Cout floats).
int encode_output_map(davo_ctx* ctx, Layer& L, int inner, int units_w, int tile_w) {
  EncodeTiledFn enc = get_encode_fn();
  if (!enc) return fail(ctx, DAVO_ERR_CUDA, "cuTensorMapEncodeTiled entry point not found");
  // units per allocated row: the pitch, in the same units (pixels, or runs of Wout / units_w pixels)
  const cuuint64_t units_p = (cuuint64_t)units_w * L.Wout_p / L.Wout;
  const cuuint64_t dims[4] = {(cuuint64_t)inner, (cuuint64_t)units_w, (cuuint64_t)L.Hout, (cuuint64_t)ctx->mb};
  const cuuint64_t strides[3] = {(cuuint64_t)inner * 4, (cuuint64_t)inner * units_p * 4,
                                 (cuuint64_t)inner * units_p * L.Hout_p * 4};
  const cuuint32_t box[4] = {32, (cuuint32_t)tile_w, (cuuint32_t)(32 / tile_w), 1};
  const cuuint32_t es[4] = {1, 1, 1, 1};
  CUresult r = enc(&L.tmO, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, L.d_out, dims, strides, box, es,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                   CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(ctx, DAVO_ERR_CUDA, "%s: cuTensorMapEncodeTiled(output) -> %d", L.name, (int)r);
  return 0;
}

// ---------------------------------------------------------------- layer plan --
// Builds the patch / tap tables and packs weights for one conv layer.
// getw(g, ty, tx, ci, n): HWIO weight of group g (ci = weight input channel).
template <class GetW>
int plan_layer(davo_ctx* ctx, Layer& L, GetW getw, const std::vector<float>& bias_host) {
  // One entry of a tap's 32-wide reduction slab: (ty, tx, ci) or ci = -1 (zero weight).
  struct Ent { int ty, tx, ci; };
  struct Tap { int par, colkey, slab, dh, dw, c; std::vector<Ent> e; };
  std::vector<Tap> taps;
  const bool strided = L.stride == 2;
  if (L.stride != 1 && L.stride != 2) return fail(ctx, DAVO_ERR_ARG, "%s: stride %d unsupported", L.name, L.stride);
  if (strided && (L.dil != 1 || (L.Hin_p & 1) || (L.Win_p & 1)))
    return fail(ctx, DAVO_ERR_ARG, "%s: stride-2 layer needs dilation 1 and an even input pitch", L.name);
  const bool pair_slab = strided && L.Cin_total == 16;
  if (!pair_slab && (L.Cin_g % 32) != 0)
    return fail(ctx, DAVO_ERR_ARG, "%s: %d input channels per group is not a multiple of 32", L.name, L.Cin_g);
  // Full 2-D halo patch unless it would not leave room for a 3-deep ring: then one
  // vertical strip per filter column (cnv5: dilation 8).
  const int TR = L.npix / kTileW;                 // tile rows
  const int full_hp = TR + (L.k - 1) * L.dil, full_wp = kTileW + (L.k - 1) * L.dil;
  const bool strips = L.strips >= 0 ? L.strips != 0 : (!strided && (size_t)full_hp * full_wp * kSlabBytes > 64 * 1024);
  L.strips = strips ? 1 : 0;
  for (int ty = 0; ty < L.k; ++ty) {
    const int dy = ty * L.dil - L.pad_t;
    const int dh = strided ? floordiv(dy, 2) : dy;
    const int par = strided ? posmod(dy, 2) : 0;
    if (pair_slab) {
      // one tap = two horizontally adjacent input pixels x 16 channels
      const int dx_lo = -L.pad_l, dx_hi = L.k - 1 - L.pad_l;
      for (int w2 = floordiv(dx_lo, 2); w2 <= floordiv(dx_hi, 2); ++w2) {
        Tap t{par, 0, 0, dh, w2, 0, std::vector<Ent>(32)};
        for (int kk = 0; kk < 32; ++kk) {
          const int wp = kk / 16;
          const int ch = kk % 16;
          const int tx = 2 * w2 + wp + L.pad_l;
          const int ci = (tx >= 0 && tx < L.k) ? L.pc2w[ch] : -1;
          t.e[kk] = Ent{ty, tx, ci};
        }
        taps.push_back(t);
      }
    } else {
      for (int tx = 0; tx < L.k; ++tx) {
        const int dx = tx * L.dil - L.pad_l;
        const int dw = strided ? floordiv(dx, 2) : dx;
        const int wp = strided ? posmod(dx, 2) : 0;
        for (int sl = 0; sl < L.Cin_g / 32; ++sl) {
          Tap t{par, strided ? wp : (strips ? tx : 0), sl, dh, dw, wp * L.Cin_total + sl * 32, std::vector<Ent>(32)};
          for (int kk = 0; kk < 32; ++kk) t.e[kk] = Ent{ty, tx, sl * 32 + kk};
          taps.push_back(t);
        }
      }
    }
  }
  // group taps into patches: key (slab, par, colkey); origin = min offsets over the group
  struct Patch { int par, colkey, slab, c, dh0, dw0, dh1, dw1; std::vector<int> idx; };
  std::vector<Patch> patches;
  for (int i = 0; i < (int)taps.size(); ++i) {
    const Tap& t = taps[i];
    Patch* pp = nullptr;
    for (Patch& q : patches) if (q.par == t.par && q.colkey == t.colkey && q.slab == t.slab) pp = &q;
    if (!pp) { patches.push_back(Patch{t.par, t.colkey, t.slab, t.c, t.dh, t.dw, t.dh, t.dw, {}}); pp = &patches.back(); }
    pp->dh0 = std::min(pp->dh0, t.dh); pp->dh1 = std::max(pp->dh1, t.dh);
    pp->dw0 = std::min(pp->dw0, t.dw); pp->dw1 = std::max(pp->dw1, t.dw);
    pp->idx.push_back(i);
  }
  int Hp = 0, Wp = 0;
  for (const Patch& q : patches) {
    Hp = std::max(Hp, TR + q.dh1 - q.dh0);
    Wp = std::max(Wp, kTileW + q.dw1 - q.dw0);
  }
  const int nt = (int)taps.size(), np = (int)patches.size();
  if (nt > kMaxTaps || np > kMaxPatches)
    return fail(ctx, DAVO_ERR_ARG, "%s: %d taps / %d patches exceed the tables", L.name, nt, np);
  // Patch / tap tables (same for both orientations).  Weight slabs are packed in patch-major
  // tap order, which is also the issue order.
  PatchDesc pdesc[kMaxPatches];
  TapDesc tdesc[kMaxTaps];
  memset(pdesc, 0, sizeof pdesc);
  memset(tdesc, 0, sizeof tdesc);
  std::vector<int> order;
  for (int pi = 0; pi < np; ++pi) {
    const Patch& q = patches[pi];
    PatchDesc& d = pdesc[pi];
    d.c = (int16_t)q.c; d.dw = (int8_t)q.dw0; d.par = (int8_t)q.par; d.dh = (int8_t)q.dh0;
    d.ntaps = (uint8_t)q.idx.size(); d.tap0 = (uint16_t)order.size();
    for (int i : q.idx) {
      TapDesc& td = tdesc[order.size()];
      td.a_off = (uint16_t)((taps[i].dh - q.dh0) * Wp + (taps[i].dw - q.dw0));
      td.b_idx = (uint16_t)order.size();
      order.push_back(i);
    }
  }
  const int patch_bytes = Hp * Wp * kSlabBytes;
  const int patch_stage = (patch_bytes + 1023) & ~1023;
  const std::vector<float> wr = round_weights_tf32(L, getw, ctx->compensated_rounding);
  auto wq = [&](int g, int ty, int tx, int ci, int n) {
    return wr[((((size_t)g * L.k + ty) * L.k + tx) * L.Cin_w + ci) * L.BN + n];
  };
  // ---- weights: TF32-rounded, K-major 32-float slabs ----
  //   pm: [g][tap][Cout][32]                      (Cout = MMA N)
  //   cm: [g][m-block][tap][128][32], zero rows beyond the real channels (128 = MMA M)
  const int MB = L.m_blocks;
  const int rows_per_slab = L.orient == 0 ? L.BN : cm::kBlockM;
  const size_t n_slabs = (size_t)L.groups * (L.orient == 0 ? 1 : MB) * nt;
  std::vector<float> pack(n_slabs * rows_per_slab * 32, 0.f);
  for (int g = 0; g < L.groups; ++g)
    for (int mb = 0; mb < (L.orient == 0 ? 1 : MB); ++mb)
      for (int k = 0; k < nt; ++k)
        for (int m = 0; m < rows_per_slab; ++m) {
          const int n = mb * cm::kBlockM + m;
          if (n >= L.BN) continue;
          const size_t slab = L.orient == 0 ? (size_t)g * nt + k : ((size_t)g * MB + mb) * nt + k;
          for (int kk = 0; kk < 32; ++kk) {
            const Ent& e = taps[order[k]].e[kk];
            if (e.ci >= 0)
              pack[(slab * rows_per_slab + m) * 32 + kk] = wq(g, e.ty, e.tx, e.ci, n);
          }
        }
  if (int rc = dev_alloc(ctx, (void**)&L.d_wpack, pack.size() * 4)) return rc;
  CU_OK(cudaMemcpy(L.d_wpack, pack.data(), pack.size() * 4, cudaMemcpyHostToDevice));
  if (int rc = dev_alloc(ctx, (void**)&L.d_bias, bias_host.size() * 4)) return rc;
  CU_OK(cudaMemcpy(L.d_bias, bias_host.data(), bias_host.size() * 4, cudaMemcpyHostToDevice));
  // unpacked HWIO copies for the direct cross-check path
  for (int g = 0; g < L.groups; ++g) {
    std::vector<float> hw((size_t)L.k * L.k * L.Cin_w * L.BN);
    for (int ty = 0; ty < L.k; ++ty)
      for (int tx = 0; tx < L.k; ++tx)
        for (int ci = 0; ci < L.Cin_w; ++ci)
          for (int n = 0; n < L.BN; ++n)
            hw[(((size_t)ty * L.k + tx) * L.Cin_w + ci) * L.BN + n] = wq(g, ty, tx, ci, n);
    if (int rc = dev_alloc(ctx, (void**)&L.d_whwio[g], hw.size() * 4)) return rc;
    CU_OK(cudaMemcpy(L.d_whwio[g], hw.data(), hw.size() * 4, cudaMemcpyHostToDevice));
  }
  // ---- kernel parameters and shared-memory plan ----
  int p_stages = 0, w_stages = 0;
  if (L.orient == 0) {
    pm::ConvParams& P = L.prm_pm;
    memset(&P, 0, sizeof P);
    P.tiles_w = L.tiles_w; P.tiles_h = L.tiles_h; P.groups = L.groups;
    P.Hout = L.Hout; P.Wout = L.Wout; P.out_stride = L.out_stride;
    P.cin_group_off = L.cin_shared ? 0 : L.Cin_g;
    P.n_patches = np; P.n_taps = nt; P.patch_w = Wp;
    P.patch_bytes = patch_bytes; P.patch_stage_bytes = patch_stage;
    P.bias = L.d_bias;
    memcpy(P.patches, pdesc, sizeof pdesc);
    memcpy(P.taps, tdesc, sizeof tdesc);
    const int bbytes = L.BN * kSlabBytes;
    const int fixed = 1024 /*alignment*/ + kBarrierBytes + pm::kBiasSmemBytes + pm::kEpiStageBytes;
    const int avail = kSmemBudget - fixed;
    const int resident_bytes = L.groups * nt * bbytes;
    L.b_resident = L.groups == 1 && resident_bytes + 2 * patch_stage <= avail && resident_bytes <= 100 * 1024;
    if (L.b_resident) {
      P.p_stages = std::min(kMaxStages, (avail - resident_bytes) / patch_stage);
      P.b_stages = 0;
      L.smem_bytes = fixed + resident_bytes + P.p_stages * patch_stage;
    } else {
      P.p_stages = 3;
      if ((avail - 3 * patch_stage) / bbytes < 4) P.p_stages = 2;
      P.b_stages = std::min(kMaxStages, (avail - P.p_stages * patch_stage) / bbytes);
      if (P.b_stages < 2) return fail(ctx, DAVO_ERR_ARG, "%s: shared-memory plan does not fit", L.name);
      L.smem_bytes = fixed + P.b_stages * bbytes + P.p_stages * patch_stage;
    }
    p_stages = P.p_stages; w_stages = P.b_stages;
  } else {
    cm::ConvParams& P = L.prm_cm;
    memset(&P, 0, sizeof P);
    P.tiles_w = L.tiles_w; P.tiles_h = L.tiles_h; P.groups = L.groups; P.m_blocks = MB;
    P.Hout = L.Hout; P.Wout = L.Wout; P.out_stride = L.out_stride; P.cout_g = L.BN;
    P.cin_group_off = L.cin_shared ? 0 : L.Cin_g;
    P.n_patches = np; P.n_taps = nt; P.patch_w = Wp;
    P.patch_bytes = patch_bytes; P.patch_stage_bytes = patch_stage;
    P.bias = L.d_bias;
    memcpy(P.patches, pdesc, sizeof pdesc);
    memcpy(P.taps, tdesc, sizeof tdesc);
    // Short main loops (cnv4: 18 taps) are epilogue-bound with direct stores: stage them.
    const char* stg_env = getenv("DAVO_B200_CM_STAGED");     // debug: "0" / "1" for every cm layer
    L.cm_staged = L.epi == EPI_STORE_RELU && (stg_env ? !strcmp(stg_env, "1") : nt <= 18);
    const int fixed = 1024 /*alignment*/ + kBarrierBytes + (L.cm_staged ? cm::kEpiWarps * 4096 : 0);
    const int avail = kSmemBudget - fixed;
    P.p_stages = patch_stage <= 40 * 1024 ? 3 : 2;
    if (const char* e = getenv("DAVO_B200_CM_PSTAGES")) P.p_stages = std::max(2, atoi(e));   // experiment knob
    // A third patch stage pays when at least five weight stages remain (cnv5: P3 W5, 0.610 -> 0.589 ms).
    if (!getenv("DAVO_B200_CM_PSTAGES") && P.p_stages == 2 && (avail - 3 * patch_stage) / cm::kWBytes >= 5) P.p_stages = 3;
    if (P.p_stages >= 3 && (avail - P.p_stages * patch_stage) / cm::kWBytes < 4) P.p_stages = 2;
    P.w_stages = std::min(kMaxStages, (avail - P.p_stages * patch_stage) / cm::kWBytes);
    if (P.w_stages < 2) return fail(ctx, DAVO_ERR_ARG, "%s: shared-memory plan does not fit", L.name);
    L.smem_bytes = fixed + P.w_stages * cm::kWBytes + P.p_stages * patch_stage;
    p_stages = P.p_stages; w_stages = P.w_stages;
  }
  if (p_stages < 2) return fail(ctx, DAVO_ERR_ARG, "%s: patch ring does not fit", L.name);
  // ---- tensor maps ----
  EncodeTiledFn enc = get_encode_fn();
  if (!enc) return fail(ctx, DAVO_ERR_CUDA, "cuTensorMapEncodeTiled entry point not found");
  {
    // extents: the real map (out-of-bounds = 'SAME' zeros); the strided view takes the even pitch,
    // whose extra row / column is zero memory.  Strides: the pitch.
    const cuuint64_t C = L.Cin_total, H = L.Hin, W = L.Win, Hq = L.Hin_p, Wq = L.Win_p, N = ctx->mb;
    cuuint64_t dims[5], strides[4];
    if (strided) {
      dims[0] = 2 * C; dims[1] = Wq / 2; dims[2] = 2; dims[3] = Hq / 2; dims[4] = N;
      strides[0] = 2 * C * 4; strides[1] = Wq * C * 4; strides[2] = 2 * Wq * C * 4; strides[3] = Hq * Wq * C * 4;
    } else {
      dims[0] = C; dims[1] = W; dims[2] = 1; dims[3] = H; dims[4] = N;
      strides[0] = C * 4; strides[1] = Wq * C * 4; strides[2] = Wq * C * 4; strides[3] = Hq * Wq * C * 4;
    }
    const cuuint32_t box[5] = {32, (cuuint32_t)Wp, 1, (cuuint32_t)Hp, 1};
    const cuuint32_t es[5] = {1, 1, 1, 1, 1};
    CUresult r = enc(&L.tmA, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 5, L.d_in, dims, strides, box, es,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                     CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(ctx, DAVO_ERR_CUDA, "%s: cuTensorMapEncodeTiled(activation) -> %d", L.name, (int)r);
  }
  {
    cuuint64_t dims[2] = {32, (cuuint64_t)n_slabs * rows_per_slab};
    cuuint64_t strides[1] = {128};
    const cuuint32_t box[2] = {32, (cuuint32_t)rows_per_slab};
    const cuuint32_t es[2] = {1, 1};
    CUresult r = enc(&L.tmB, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, L.d_wpack, dims, strides, box, es,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                     CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(ctx, DAVO_ERR_CUDA, "%s: cuTensorMapEncodeTiled(weights) -> %d", L.name, (int)r);
    L.tmB64 = L.tmB;
    const char* cl_env = getenv("DAVO_B200_CLUSTER");            // debug: "0" switches the clusters off
    L.cm_cluster = L.orient == 1 && (L.epi == EPI_STORE_RELU || getenv("DAVO_B200_CNV7_CM")) && !(cl_env && !strcmp(cl_env, "0"));
    if (L.cm_cluster) {
      const cuuint32_t box64[2] = {32, (cuuint32_t)(rows_per_slab / 2)};
      r = enc(&L.tmB64, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, L.d_wpack, dims, strides, box64, es,
              CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
              CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
      if (r != CUDA_SUCCESS) return fail(ctx, DAVO_ERR_CUDA, "%s: cuTensorMapEncodeTiled(weights, half slab) -> %d", L.name, (int)r);
    }
  }
  L.tmO = L.tmA;
  if (L.pitched_out() && L.epi == EPI_STORE_RELU && !(L.orient == 0 && L.BN >= 32))
    return fail(ctx, DAVO_ERR_ARG, "%s: an odd-sized output map needs the TMA-store epilogue (pixels-on-M, >= 32 channels)", L.name);
  if ((L.orient == 1 && L.cm_staged) || (L.orient == 0 && L.epi == EPI_STORE_RELU && L.BN >= 32))
    if (int rc = encode_output_map(ctx, L, L.out_stride, L.Wout, kTileW)) return rc;
  if (getenv("DAVO_B200_VERBOSE"))
    fprintf(stderr, "[davo_b200] %s: %s, tile %dx8 px, %d m-block(s), patch %dx%d (%d B) x%d, %d taps, weights %s, rings P%d W%d, smem %d\n",
            L.name, L.orient == 0 ? "pixels-on-M" : "channels-on-M", TR, MB, Hp, Wp, patch_bytes, np, nt,
            L.b_resident ? "resident" : "streamed", p_stages, w_stages, L.smem_bytes);
  return 0;
}

// ----------------------------------------------------------- widened layer plan --
// Column-widened plan of a thin stride-2 layer whose input has 16 channels (cnv1, cnv2):
// one M row = a run of G adjacent output pixels, N = G * Cout (conv_pm.cuh, WIDE).
//   output pixel g of a run reads input pixel 2g + tx - pad_l (relative to the run's first
//   input pixel 2G*j); pixel pair c = floor(.. / 2), wp = .. mod 2, and with d = c - g the
//   filter column is tx = 2d + wp + pad_l.  Weight block of filter row ty:
//   R[ty] = [W[d_max]; ...; W[d_min]], W[d] = Cout rows x 32 (two pixels x 16 channels).
//   Pair c feeds g in [c - d_max, c - d_min] (clipped to the run): rows
//   (d_max - c + g_lo) * Cout.. of R[ty], accumulator columns g_lo * Cout...
template <class GetW>
int plan_layer_wide(davo_ctx* ctx, Layer& L, GetW getw, const std::vector<float>& bias_host) {
  const int G = L.wide_G, TWc = L.wide_tw, THr = 128 / TWc, Co = L.BN, NW = G * Co;
  if (NW != 128) return fail(ctx, DAVO_ERR_ARG, "%s: the widened kernel is built for N = 128 (got %d)", L.name, NW);
  // S input pixels x C channels make one 32-float slab (C = 16: S = 2; cnv1's 8-channel input: S = 4).
  // Output pixel g of a run reads input pixel u = 2g + tx - pad_l (relative to the run's first
  // input pixel); slab c = floor(u / S), wp = u mod S.  With d = (S/2) c - g the filter column is
  // tx = 2d + wp + pad_l, so the weights of (c, g) depend on d only.
  const int C = L.Cin_total, S = 32 / C, half = S / 2, slabs_per_run = 2 * G / S;
  const int d_min = -floordiv(L.pad_l + S - 1, 2), d_max = floordiv(L.k - 1 - L.pad_l, 2), nd = d_max - d_min + 1;
  const int c_min = floordiv(-L.pad_l, S), c_max = floordiv(2 * (G - 1) + L.k - 1 - L.pad_l, S);
  const std::vector<float> wr = round_weights_tf32(L, getw, ctx->compensated_rounding);
  auto wq = [&](int ty, int tx, int ci, int n) { return wr[(((size_t)ty * L.k + tx) * L.Cin_w + ci) * Co + n]; };
  // ---- weights: [ty][d_max..d_min][Cout][32] ----
  const int box_rows = nd * Co;
  std::vector<float> pack((size_t)L.k * box_rows * 32, 0.f);
  for (int ty = 0; ty < L.k; ++ty)
    for (int b = 0; b < nd; ++b)
      for (int n = 0; n < Co; ++n)
        for (int kk = 0; kk < 32; ++kk) {
          const int tx = 2 * (d_max - b) + kk / C + L.pad_l, ci = L.pc2w[kk % C];
          if (tx >= 0 && tx < L.k && ci >= 0) pack[(((size_t)ty * nd + b) * Co + n) * 32 + kk] = wq(ty, tx, ci, n);
        }
  if (int rc = dev_alloc(ctx, (void**)&L.d_wpack, pack.size() * 4)) return rc;
  CU_OK(cudaMemcpy(L.d_wpack, pack.data(), pack.size() * 4, cudaMemcpyHostToDevice));
  std::vector<float> bias_rep((size_t)NW);
  for (int i = 0; i < NW; ++i) bias_rep[i] = bias_host[i % Co];
  if (int rc = dev_alloc(ctx, (void**)&L.d_bias, bias_rep.size() * 4)) return rc;
  CU_OK(cudaMemcpy(L.d_bias, bias_rep.data(), bias_rep.size() * 4, cudaMemcpyHostToDevice));
  {
    std::vector<float> hw((size_t)L.k * L.k * L.Cin_w * Co);
    for (int ty = 0; ty < L.k; ++ty)
      for (int tx = 0; tx < L.k; ++tx)
        for (int ci = 0; ci < L.Cin_w; ++ci)
          for (int n = 0; n < Co; ++n) hw[(((size_t)ty * L.k + tx) * L.Cin_w + ci) * Co + n] = wq(ty, tx, ci, n);
    if (int rc = dev_alloc(ctx, (void**)&L.d_whwio[0], hw.size() * 4)) return rc;
    CU_OK(cudaMemcpy(L.d_whwio[0], hw.data(), hw.size() * 4, cudaMemcpyHostToDevice));
  }
  // ---- patches (one per slab position and row parity) and taps ----
  auto g_lo_of = [&](int c) { return std::max(half * c - d_max, 0); };
  auto g_hi_of = [&](int c) { return std::min(half * c - d_min, G - 1); };
  // The tile's first MMAs must OVERWRITE the accumulator.  Cover the run with column windows
  // that do not overlap: slab positions whose windows reach furthest, each cut to start where
  // the previous one ended; what is cut off is issued as an extra accumulating tap.
  struct Cover { int c, from; };
  std::vector<Cover> cover;
  for (int s0 = 0; s0 < G;) {
    int best = c_min - 1;
    for (int c = c_min; c <= c_max; ++c)
      if (g_lo_of(c) <= s0 && s0 <= g_hi_of(c) && (best < c_min || g_hi_of(c) > g_hi_of(best))) best = c;
    if (best < c_min) return fail(ctx, DAVO_ERR_ARG, "%s: widened plan cannot cover the run", L.name);
    cover.push_back(Cover{best, s0});
    s0 = g_hi_of(best) + 1;
  }
  const int par0 = posmod(-L.pad_t, 2);
  struct P2 { int c, par, from; };                 // from >= 0: cover patch, fresh columns start there
  std::vector<P2> plist;
  for (const Cover& cv : cover) plist.push_back(P2{cv.c, par0, cv.from});
  for (int par = 0; par < 2; ++par)
    for (int c = c_min; c <= c_max; ++c) {
      bool seen = false;
      for (const P2& q : plist) seen |= (q.c == c && q.par == par);
      if (!seen) plist.push_back(P2{c, par, -1});
    }
  int dh_lo[2] = {1 << 20, 1 << 20}, dh_hi[2] = {-(1 << 20), -(1 << 20)};
  for (int ty = 0; ty < L.k; ++ty) {
    const int dy = ty - L.pad_t, par = posmod(dy, 2), dh = floordiv(dy, 2);
    dh_lo[par] = std::min(dh_lo[par], dh); dh_hi[par] = std::max(dh_hi[par], dh);
  }
  const int Hp = THr + std::max(dh_hi[0] - dh_lo[0], dh_hi[1] - dh_lo[1]), Wp = TWc;
  PatchDesc pdesc[kMaxPatches];
  TapDesc tdesc[kMaxTaps];
  memset(pdesc, 0, sizeof pdesc);
  memset(tdesc, 0, sizeof tdesc);
  int np = 0, nt = 0;
  for (const P2& q : plist) {
    if (np >= kMaxPatches) return fail(ctx, DAVO_ERR_ARG, "%s: too many patches for the widened plan", L.name);
    PatchDesc& d = pdesc[np];
    d.c = (int16_t)(32 * posmod(q.c, slabs_per_run)); d.dw = (int8_t)floordiv(q.c, slabs_per_run); d.par = (int8_t)q.par;
    d.dh = (int8_t)dh_lo[q.par]; d.tap0 = (uint16_t)nt;
    const int g_lo = g_lo_of(q.c), g_hi = g_hi_of(q.c);
    int n_here = 0;
    auto emit = [&](int ty, int ga, int gb, int fresh) {
      TapDesc& t = tdesc[nt++];
      t.a_off = (uint16_t)((floordiv(ty - L.pad_t, 2) - dh_lo[q.par]) * Wp);
      t.b_idx = (uint16_t)ty;
      t.n16 = (uint8_t)((gb - ga + 1) * Co / 16);
      t.dcol16 = (uint8_t)(ga * Co / 16);
      t.brow8 = (uint8_t)((d_max - half * q.c + ga) * Co / 8);
      t.fresh = (uint8_t)fresh;
      ++n_here;
    };
    for (int ty = 0; ty < L.k; ++ty) {
      if (posmod(ty - L.pad_t, 2) != q.par) continue;
      if (nt + 2 > kMaxTaps) return fail(ctx, DAVO_ERR_ARG, "%s: too many taps for the widened plan", L.name);
      if (q.from >= 0 && n_here == 0) {
        emit(ty, q.from, g_hi, 1);
        if (g_lo < q.from) emit(ty, g_lo, q.from - 1, 0);
      } else {
        emit(ty, g_lo, g_hi, 0);
      }
    }
    d.ntaps = (uint8_t)n_here;
    ++np;
  }
  const int patch_bytes = Hp * Wp * kSlabBytes;
  const int patch_stage = (patch_bytes + 1023) & ~1023;
  pm::ConvParams& P = L.prm_pm;
  memset(&P, 0, sizeof P);
  P.tiles_w = L.tiles_w; P.tiles_h = L.tiles_h; P.groups = 1;
  P.Hout = L.Hout; P.Wout = L.Wout; P.out_stride = L.out_stride;
  P.cin_group_off = 0;
  P.n_patches = np; P.n_taps = nt; P.patch_w = Wp;
  P.patch_bytes = patch_bytes; P.patch_stage_bytes = patch_stage;
  P.bias = L.d_bias;
  P.tile_h = THr; P.tile_w = TWc; P.run_px = G; P.b_boxes = L.k; P.b_box_rows = box_rows;
  memcpy(P.patches, pdesc, sizeof pdesc);
  memcpy(P.taps, tdesc, sizeof tdesc);
  const int fixed = 1024 /*alignment*/ + kBarrierBytes + pm::kBiasSmemBytes + pm::kEpiStageBytes;
  const int resident_bytes = L.k * box_rows * kSlabBytes;
  L.b_resident = true;
  int raw_bytes = 0;
  if (L.fused_front) {
    // the staging area of the fused front end (conv_pm.cuh: FusedGeo): Hp rows x raw_px pixels of flow, target and
    // source bytes and labels.  Needs the patch list in two halves, one per row parity, each with one dh.
    pm::FusedGeo& g = P.fg;
    bool ok = S == 4 && np % 2 == 0 && np >= 2;
    g.half_patches = np / 2;
    for (int i = 0; ok && i < np; ++i) {
      const PatchDesc& a = pdesc[(i / g.half_patches) * g.half_patches];
      ok = pdesc[i].par == a.par && pdesc[i].dh == a.dh;
    }
    ok = ok && pdesc[0].par != pdesc[g.half_patches].par;
    int x_lo = 1 << 20, x_hi = -(1 << 20);
    for (int i = 0; i < np; ++i)
      for (int j = 0; j < TWc; ++j) {
        const int x = 2 * G * (j + pdesc[i].dw) + (pdesc[i].c >> 5) * S;
        x_lo = std::min(x_lo, x); x_hi = std::max(x_hi, x + S);
      }
    g.x_lo = x_lo; g.raw_px = x_hi - x_lo;
    ok = ok && (g.raw_px % 4) == 0 && (x_lo % 4) == 0 && g.raw_px <= 160 && g.half_patches * Hp * Wp <= pm::kFusedItems * pm::kFusedThreads;
    const int NF = g.raw_px / 2, NT = g.raw_px * 3 / 4, NL = g.raw_px / 4;
    g.flow_pitch = NF + 1;
    g.off_tgt = Hp * g.flow_pitch * 16;
    g.off_src = g.off_tgt + Hp * NT * 4;
    g.off_lab_s = g.off_src + Hp * NT * 4;
    g.off_lab_t = g.off_lab_s + Hp * NL * 4;                 // labels are staged as bytes
    g.raw_bytes = (g.off_lab_t + (ctx->cfg.att_tgt_ones ? 0 : Hp * NL * 4) + 15) & ~15;
    raw_bytes = 2 * g.raw_bytes - pm::kEpiStageBytes / 2;    // two staging areas; the fused kernel's epilogue gives back half of its buffers
    if (!ok || (kSmemBudget - fixed - resident_bytes - raw_bytes) / patch_stage < 3) {
      L.fused_front = false;                     // the plain widened plan (pack8_kernel feeds it)
      raw_bytes = 0;
      memset(&g, 0, sizeof g);
    }
  }
  P.p_stages = std::min(kMaxStages, (kSmemBudget - fixed - resident_bytes - raw_bytes) / patch_stage);
  P.b_stages = 0;
  if (P.p_stages < 2) return fail(ctx, DAVO_ERR_ARG, "%s: widened plan does not fit shared memory", L.name);
  L.smem_bytes = fixed + resident_bytes + P.p_stages * patch_stage + raw_bytes;
  if (L.fused_front)      // behind the ring, the resident weights, the epilogue staging, the barriers and the bias table
    P.fg.raw_off = P.p_stages * patch_stage + resident_bytes + pm::kEpiStageBytes / 2 + kBarrierBytes + pm::kBiasSmemBytes;
  EncodeTiledFn enc = get_encode_fn();
  if (!enc) return fail(ctx, DAVO_ERR_CUDA, "cuTensorMapEncodeTiled entry point not found");
  {
    const cuuint64_t H = L.Hin, W = L.Win, N = ctx->mb;
    const cuuint64_t dims[5] = {(cuuint64_t)2 * G * C, W / (2 * G), 2, H / 2, N};
    const cuuint64_t strides[4] = {(cuuint64_t)2 * G * C * 4, W * C * 4, 2 * W * C * 4, H * W * C * 4};
    const cuuint32_t box[5] = {32, (cuuint32_t)Wp, 1, (cuuint32_t)Hp, 1};
    const cuuint32_t es[5] = {1, 1, 1, 1, 1};
    CUresult r = enc(&L.tmA, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 5, L.d_in, dims, strides, box, es,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                     CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(ctx, DAVO_ERR_CUDA, "%s: cuTensorMapEncodeTiled(activation) -> %d", L.name, (int)r);
  }
  {
    const cuuint64_t dims[2] = {32, (cuuint64_t)L.k * box_rows};
    const cuuint64_t strides[1] = {128};
    const cuuint32_t box[2] = {32, (cuuint32_t)box_rows};
    const cuuint32_t es[2] = {1, 1};
    CUresult r = enc(&L.tmB, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, L.d_wpack, dims, strides, box, es,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                     CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(ctx, DAVO_ERR_CUDA, "%s: cuTensorMapEncodeTiled(weights) -> %d", L.name, (int)r);
  }
  if (int rc = encode_output_map(ctx, L, NW, L.Wout / G, TWc)) return rc;
  if (getenv("DAVO_B200_VERBOSE"))
    fprintf(stderr, "[davo_b200] %s: pixels-on-M widened x%d (N=%d, %d-pixel slabs), tile %dx%d runs, patch %dx%d (%d B) x%d, %d taps, weights resident %d B, ring P%d, smem %d%s\n",
            L.name, G, NW, S, THr, TWc, Hp, Wp, patch_bytes, np, nt, resident_bytes, P.p_stages, L.smem_bytes,
            L.fused_front ? (", fused front end: staging " + std::to_string(raw_bytes) + " B, " + std::to_string(P.fg.raw_px) + " pixels per row from " + std::to_string(P.fg.x_lo)).c_str() : "");
  return 0;
}

template <int BN, int EPI, bool RES>
int launch_pm_t(davo_ctx* ctx, const Layer& L, int npairs, cudaStream_t st) {
  if (int rc = ensure_smem(ctx, pm::conv_tc_kernel<BN, EPI, RES>, L.smem_bytes)) return rc;
  pm::ConvParams P = L.prm_pm;
  P.raw = ctx->cfg.batch_norm ? 1 : 0;
  P.num_tiles = npairs * L.groups * L.tiles_h * L.tiles_w;
  P.out = L.d_out;
  P.sum_out = ctx->d_sum7;
  const int grid = P.num_tiles < ctx->num_sms ? P.num_tiles : ctx->num_sms;
  return launch_k(ctx, pm::conv_tc_kernel<BN, EPI, RES>, dim3(grid), dim3(kConvThreads), L.smem_bytes, st, false,
                  L.tmA, L.tmB, L.tmO, P);
}

int launch_pm_wide(davo_ctx* ctx, const Layer& L, int npairs, cudaStream_t st) {
  pm::ConvParams P = L.prm_pm;
  P.raw = ctx->cfg.batch_norm ? 1 : 0;
  P.num_tiles = npairs * L.tiles_h * L.tiles_w;
  P.out = L.d_out;
  const int grid = P.num_tiles < ctx->num_sms ? P.num_tiles : ctx->num_sms;
  if (L.fused_front && ctx->fuse_front && ctx->conv_impl == 0) {      // cnv1 with the front end inside (no packed input in memory)
    auto* kern = pm::conv_tc_kernel<128, EPI_STORE_RELU, true, true, true>;
    if (int rc = ensure_smem(ctx, kern, L.smem_bytes)) return rc;
    P.front = ctx->fp_cur;
    return launch_k(ctx, kern, dim3(grid), dim3(kConvThreads + pm::kFusedThreads), L.smem_bytes, st, false, L.tmA, L.tmB, L.tmO, P);
  }
  auto* kern = pm::conv_tc_kernel<128, EPI_STORE_RELU, true, true>;
  if (int rc = ensure_smem(ctx, kern, L.smem_bytes)) return rc;
  return launch_k(ctx, kern, dim3(grid), dim3(kConvThreads), L.smem_bytes, st, false, L.tmA, L.tmB, L.tmO, P);
}

template <int BN, int EPI>
int launch_pm_r(davo_ctx* ctx, const Layer& L, int npairs, cudaStream_t st) {
  return L.b_resident ? launch_pm_t<BN, EPI, true>(ctx, L, npairs, st)
                      : launch_pm_t<BN, EPI, false>(ctx, L, npairs, st);
}

template <int NPIX, int EPI, bool STAGED = false>
int launch_cm_t(davo_ctx* ctx, const Layer& L, int npairs, cudaStream_t st) {
  if (int rc = ensure_smem(ctx, cm::conv_tc_kernel<NPIX, EPI, STAGED>, L.smem_bytes)) return rc;
  cm::ConvParams P = L.prm_cm;
  P.raw = ctx->cfg.batch_norm ? 1 : 0;
  P.num_tiles = npairs * L.groups * L.tiles_h * L.tiles_w * L.m_blocks;
  P.out = L.d_out;
  P.sum_out = ctx->d_sum7;
  const int grid = P.num_tiles < ctx->num_sms ? P.num_tiles : ctx->num_sms;
  return launch_k(ctx, cm::conv_tc_kernel<NPIX, EPI, STAGED>, dim3(grid), dim3(cm::kThreads), L.smem_bytes, st, false,
                  L.tmA, L.tmB, L.tmO, P);
}

// 2-CTA clusters, weights multicast (conv_cm.cuh: CLUSTER).
template <int NPIX, bool STAGED, int EPI = EPI_STORE_RELU>
int launch_cm_cluster(davo_ctx* ctx, const Layer& L, int npairs, cudaStream_t st) {
  auto* kern = cm::conv_tc_kernel<NPIX, EPI, STAGED, true>;
  if (int rc = ensure_smem(ctx, kern, L.smem_bytes)) return rc;
  int& max_clusters = ctx->max_clusters[std::make_pair(reinterpret_cast<const void*>(kern), L.smem_bytes)];
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof cfg);
  cudaLaunchAttribute attr;
  attr.id = cudaLaunchAttributeClusterDimension;
  attr.val.clusterDim.x = 2; attr.val.clusterDim.y = 1; attr.val.clusterDim.z = 1;
  cfg.blockDim = dim3(cm::kThreads); cfg.dynamicSmemBytes = L.smem_bytes; cfg.stream = st;
  cfg.attrs = &attr; cfg.numAttrs = 1;
  if (max_clusters == 0) {
    cfg.gridDim = dim3(ctx->num_sms & ~1);
    CU_OK(cudaOccupancyMaxActiveClusters(&max_clusters, kern, &cfg));
    if (max_clusters <= 0) return fail(ctx, DAVO_ERR_CUDA, "%s: no 2-CTA cluster fits", L.name);
    if (getenv("DAVO_B200_VERBOSE")) fprintf(stderr, "[davo_b200] %s: %d active 2-CTA clusters\n", L.name, max_clusters);
  }
  cm::ConvParams P = L.prm_cm;
  P.raw = ctx->cfg.batch_norm ? 1 : 0;
  P.num_pixel_tiles = npairs * L.tiles_h * L.tiles_w;
  P.num_tiles = ((P.num_pixel_tiles + 1) / 2) * L.groups * L.m_blocks;
  P.out = L.d_out;
  P.sum_out = ctx->d_sum7;
  const int clusters = P.num_tiles < max_clusters ? P.num_tiles : max_clusters;
  return launch_k(ctx, kern, dim3(2 * clusters), dim3(cm::kThreads), L.smem_bytes, st, true, L.tmA, L.tmB64, L.tmO, P);
}

int launch_conv(davo_ctx* ctx, const Layer& L, int npairs, cudaStream_t st) {
  if (L.orient == 1 && L.cm_cluster) {
    if (L.epi == EPI_SUM_RELU)
      return L.npix == 256 ? launch_cm_cluster<256, false, EPI_SUM_RELU>(ctx, L, npairs, st)
                           : launch_cm_cluster<128, false, EPI_SUM_RELU>(ctx, L, npairs, st);
    if (L.cm_staged)
      return L.npix == 256 ? launch_cm_cluster<256, true>(ctx, L, npairs, st) : launch_cm_cluster<128, true>(ctx, L, npairs, st);
    return L.npix == 256 ? launch_cm_cluster<256, false>(ctx, L, npairs, st) : launch_cm_cluster<128, false>(ctx, L, npairs, st);
  }
  if (L.orient == 1) {
    if (L.epi == EPI_SUM_RELU)
      return L.npix == 256 ? launch_cm_t<256, EPI_SUM_RELU>(ctx, L, npairs, st)
                           : launch_cm_t<128, EPI_SUM_RELU>(ctx, L, npairs, st);
    if (L.cm_staged)
      return L.npix == 256 ? launch_cm_t<256, EPI_STORE_RELU, true>(ctx, L, npairs, st)
                           : launch_cm_t<128, EPI_STORE_RELU, true>(ctx, L, npairs, st);
    return L.npix == 256 ? launch_cm_t<256, EPI_STORE_RELU>(ctx, L, npairs, st)
                         : launch_cm_t<128, EPI_STORE_RELU>(ctx, L, npairs, st);
  }
  if (L.wide_G) return launch_pm_wide(ctx, L, npairs, st);
  if (L.epi == EPI_SUM_RELU) {
    if (L.BN == 256) return launch_pm_t<256, EPI_SUM_RELU, false>(ctx, L, npairs, st);
    return fail(ctx, DAVO_ERR_ARG, "%s: pixels-on-M sum epilogue is built for 256 channels only", L.name);
  }
  switch (L.BN) {
    case 16: return launch_pm_r<16, EPI_STORE_RELU>(ctx, L, npairs, st);
    case 32: return launch_pm_r<32, EPI_STORE_RELU>(ctx, L, npairs, st);
    case 64: return launch_pm_r<64, EPI_STORE_RELU>(ctx, L, npairs, st);
    case 128: return launch_pm_r<128, EPI_STORE_RELU>(ctx, L, npairs, st);
    case 256: return launch_pm_t<256, EPI_STORE_RELU, false>(ctx, L, npairs, st);
  }
  return fail(ctx, DAVO_ERR_ARG, "%s: %d output channels have no kernel instance", L.name, L.BN);
}

int launch_conv_direct(davo_ctx* ctx, const Layer& L, int npairs, cudaStream_t st) {
  if (L.pitched_out() || L.Hin_p != L.Hin || L.Win_p != L.Win)
    return fail(ctx, DAVO_ERR_ARG, "%s: the direct cross-check path does not handle padded pitches", L.name);
  for (int g = 0; g < L.groups; ++g) {
    DirectConvParams p;
    memset(&p, 0, sizeof p);
    p.npairs = npairs; p.Hin = L.Hin; p.Win = L.Win; p.Cin_total = L.Cin_total;
    p.cin_off = L.cin_shared ? 0 : g * L.Cin_g; p.Cin = L.Cin_w;
    p.Hout = L.Hout; p.Wout = L.Wout; p.Cout = L.BN;
    p.kh = p.kw = L.k; p.stride = L.stride; p.dil = L.dil; p.pad_t = L.pad_t; p.pad_l = L.pad_l;
    p.relu = 1;
    p.use_cmap = L.use_cmap;
    for (int i = 0; i < 16; ++i) p.cmap[i] = L.cmap[i];
    p.in = L.d_in; p.w = L.d_whwio[g]; p.bias = L.d_bias + g * L.BN;
    if (L.epi == EPI_SUM_RELU) {
      p.out = ctx->d_c7tmp; p.out_stride = L.groups * L.BN; p.cout_off = g * L.BN; p.round_out = 0;
    } else {
      p.out = L.d_out; p.out_stride = L.out_stride; p.cout_off = g * L.BN; p.round_out = 1;
    }
    const long long total = (long long)npairs * L.Hout * L.Wout * L.BN;
    conv_direct_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(p);
    CU_OK(cudaGetLastError());
  }
  return 0;
}

__global__ void sum7_direct_kernel(const float* in, int hw, int nparts, float* out) {
  // in [n][hw][nbr*256] -> out [n][nbr][nparts][256]; row 0 holds the sum, the rest zeros.
  const int n = blockIdx.x, br = blockIdx.y, nbr = gridDim.y, c = threadIdx.x;
  float a = 0.f;
  for (int i = 0; i < hw; ++i) a += in[((size_t)n * hw + i) * nbr * 256 + br * 256 + c];
  float* o = out + ((size_t)(n * nbr + br) * nparts) * 256 + c;
  o[0] = a;
  for (int i = 1; i < nparts; ++i) o[(size_t)i * 256] = 0.f;
}

// Blocks per frame pair of pack8_kernel (a block covers 1024 pixels per iteration; 52 cover the frame in one).
// A full pass runs best with 13 blocks x 4 iterations (the per-block prologue is paid once per 4096 pixels:
// front end 0.168 -> 0.161 ms per 256 pairs, tools/front_probe.py); small passes need the blocks to fill the GPU.
int pack8_blocks(int npairs) {
  static const int forced = [] { const char* e = getenv("DAVO_B200_PACK8_BLOCKS"); return e ? std::max(1, atoi(e)) : 0; }();
  if (forced) return forced;
  return npairs >= 64 ? kPack8Blocks / 4 : kPack8Blocks;
}

int launch_front(davo_ctx* ctx, int pair_mode, int pair0, int npairs, const InputView& in, cudaStream_t st, int* launches) {
  const davo_config& c = ctx->cfg;
  FrontParams fp;
  memset(&fp, 0, sizeof fp);
  fp.H = c.H; fp.W = c.W; fp.pair0 = pair0; fp.npairs = npairs; fp.pair_mode = pair_mode;
  fp.unit_sample = ctx->unit_sample ? 1 : 0;
  fp.packed_c = ctx->packed_c;
  fp.in_mode = c.in_mode; fp.att_src = c.att_src; fp.att_tgt_ones = c.att_tgt_ones;
  fp.mask_rgb = c.mask_mode != 0;
  fp.mask_flow = c.mask_mode == 2;
  fp.se_act = c.se_act; fp.flow_abs = c.flow_abs; fp.flow_norm = c.flow_norm;
  fp.in = in; fp.depth_norm = c.depth_norm;
  fp.flow_f16 = c.flow_f16;
  fp.se_w = ctx->d_sew; fp.static_w = ctx->d_staticw;
  fp.pool_part = ctx->d_pool; fp.pool_count = ctx->d_poolcnt; fp.att_w = ctx->d_attw; fp.packed = ctx->d_packed;
  if (c.att_src == 1 || c.att_src >= 3) {
    static const int se_dims[7][2] = {{0, 0}, {2, 8}, {0, 0}, {19, 19}, {3, 8}, {1, 8}, {21, 19}};
    fp.se_in = se_dims[c.att_src][0]; fp.se_hid = c.se_hidden > 0 ? c.se_hidden : se_dims[c.att_src][1];
    fp.se_out = kNumClasses;
    fp.pixel_map = c.pixel_map;
    fp.depth_split = c.depth_split; fp.depth_thres = ctx->depth_thres;
    if (c.pixel_map == 2) fp.se_in = 3;                    // depth term, SE flow x, SE flow y
    if (c.pixel_map) fp.se_hid = fp.se_out = fp.se_in;     // se_block(..., ratio=1): channel -> channel -> channel
    fp.pool_2x2 = c.se_pool == 1 ? 1 : 0;
    if (fp.pool_2x2 && c.att_src == 1) fp.se_in = 8;
    const int src_frames = ctx->unit_sample ? 2 : 1;
    // Experiment, off by default (DAVO_B200_FRONT_PIPE=1): pool + pack in ONE launch (frontend.cuh: front_pipeline_kernel)
    // for se_flow with global pooling and the 8-channel layout.  Same bits, but measured slower than the two kernels
    // (0.237 vs 0.186 ms per 256 pairs, 21 vs 10 us for one sample: profiles/r2_experiment_front_pipeline.log).
    static const bool pipe_on = [] { const char* e = getenv("DAVO_B200_FRONT_PIPE"); return e && !strcmp(e, "1"); }();
    if (pipe_on && !ctx->fuse_front && c.att_src == 1 && c.se_pool == 0 && !c.depth_split && !c.pixel_map && c.att_tgt_ones && !ctx->unit_sample &&
        ctx->packed_c == 8 && ctx->d_pipe) {
      FrontPipe q;
      q.next = ctx->d_pipe; q.done = ctx->d_pipe + 1; q.launches = reinterpret_cast<unsigned int*>(ctx->d_pipe + 2);
      q.ready = reinterpret_cast<unsigned int*>(ctx->d_pipe + 4);
      const int work = (npairs + kPipeLook) * (kPoolSplits + kPipePack);
      const int grid = std::min(work, ctx->num_sms * 4);
      if (int rc = launch_k(ctx, front_pipeline_kernel, dim3(grid), dim3(256), 0, st, false, fp, q)) return rc;
      ++*launches;
      ctx->fp_cur = fp;
      return 0;
    }
    if (c.se_pool >= 2) {                         // mode='spp': out_pool_size [2,1] / [2] / [8,6,4]
      static const int sizes[3][4] = {{2, 2, 1, 0}, {1, 2, 0, 0}, {3, 8, 6, 4}};
      const int* sz = sizes[c.se_pool - 2];
      fp.spp_levels = sz[0];
      for (int i = 0; i < sz[0]; ++i) fp.spp_n[i] = sz[1 + i];
    }
    if ((c.att_src == 3 || c.att_src == 6) && c.se_pool != 0) {   // cell-wise class frequencies of the label map (+ flow means)
      if (int rc = launch_k(ctx, se_segcells_kernel, dim3(npairs, src_frames + (c.att_tgt_ones ? 0 : 1)), dim3(256), 0, st, false, fp))
        return rc;
    } else if (c.att_src == 1 && c.se_pool >= 2) {
      if (int rc = launch_k(ctx, se_spp_kernel, dim3(npairs, src_frames), dim3(256), 0, st, false, fp)) return rc;
    } else if (int rc = launch_k(ctx, se_pool_kernel, dim3(kPoolSplits, npairs, c.depth_split ? 2 * src_frames : src_frames + (c.att_tgt_ones ? 0 : 1)),
                                 dim3(256), 0, st, false, fp)) {
      return rc;
    }
    ++*launches;
  }
  ctx->fp_cur = fp;
  if (ctx->fuse_front && ctx->conv_impl == 0 && ctx->layers[0].fused_front) return 0;     // cnv1 builds its own operand
  if (int rc = ctx->unit_sample ? launch_k(ctx, pack_sample_kernel, dim3(kPackBlocksPerPair, npairs), dim3(256), 0, st, false, fp)
             : ctx->packed_c == 8 ? launch_k(ctx, pack8_kernel, dim3(pack8_blocks(npairs), npairs), dim3(256), 0, st, false, fp)
                                  : launch_k(ctx, pack_kernel, dim3(kPackBlocksPerPair, npairs), dim3(256), 0, st, false, fp))
    return rc;
  ++*launches;
  return 0;
}

int launch_head(davo_ctx* ctx, int pair_mode, int pair0, int npairs, float* pose_out, cudaStream_t st, int* launches) {
  const Layer& L7 = ctx->layers.back();
  HeadParams hp;
  hp.pair0 = pair0; hp.npairs = npairs; hp.pair_mode = pair_mode; hp.nparts = ctx->nparts7; hp.nbr = ctx->nbr;
  hp.nsrc = ctx->unit_sample ? 2 : 1;
  hp.inv_hw = 1.0f / (float)(L7.Hout * L7.Wout);
  hp.sums = ctx->d_sum7; hp.wpred = ctx->d_wpred; hp.bpred = ctx->d_bpred; hp.pose_out = pose_out;
  if (int rc = launch_k(ctx, head_kernel, dim3(npairs), dim3(256), 0, st, false, hp)) return rc;
  ++*launches;
  return 0;
}

// The plan of layer `li` for a pass of `npairs` units: the latency twin (128-pixel tiles: twice as many, half as long)
// when the 256-pixel tiling would leave SMs idle.
Layer& pick_layer(davo_ctx* ctx, size_t li, int npairs) {
  Layer& B = ctx->layers[li];
  if (li < ctx->layers_small.size() && ctx->layers_small[li].npix != 0) {
    const long tiles_big = (long)npairs * B.groups * B.tiles_h * B.tiles_w * B.m_blocks;
    if (tiles_big < ctx->num_sms) return ctx->layers_small[li];
  }
  return B;
}

// Width of a weight row of the attention outputs: what davo_get_intermediate("att_weights:<k>") returns (19 class
// weights, or the excitation of a per-pixel source: 3 rgb, 1 depth term, 3 depth term and SE flow, 21 labels and SE flow)
int att_width(const davo_config& c) {
  return !c.pixel_map ? kNumClasses : c.pixel_map == 2 ? 3 : c.att_src == 4 ? 3 : c.att_src == 5 ? 1 : kNumClasses + 2;
}

int run_microbatch(davo_ctx* ctx, int pair_mode, int pair0, int npairs, const InputView& in, float* pose_out,
                   cudaStream_t st, int* launches) {
  if (int rc = launch_front(ctx, pair_mode, pair0, npairs, in, st, launches)) return rc;
  if (ctx->att_units) {          // an odometry push asked for each posed frame's attention: att_w holds this pass's tables
    AttentionOutParams ap;
    ap.fp = ctx->fp_cur; ap.units = ctx->att_units; ap.rows = ctx->att_rows; ap.width = att_width(ctx->cfg);
    const int groups = ctx->cfg.H * ctx->cfg.W / 4;
    attention_out_kernel<<<dim3((groups + 255) / 256, npairs), 256, 0, st>>>(ap);
    CU_OK(cudaGetLastError());
    ++*launches;
  }
  for (size_t li = 0; li < ctx->layers.size(); ++li) {
    Layer& L = pick_layer(ctx, li, npairs);
    const int pse = ctx->cfg.posenn_se;
    auto se5 = [&](int skipadd) -> int {
      Se5Params sp;
      memset(&sp, 0, sizeof sp);
      // the cnv5 map with its pitch (the stride-2 nets store 4x13 as 4x14: the extra column is zeros and stays zeros)
      sp.npairs = npairs; sp.hw = ctx->layers[5].Hin_p * ctx->layers[5].Win_p; sp.nbr = ctx->nbr; sp.stack = pse == 1; sp.skipadd = skipadd;
      sp.inv_n = 1.0f / (float)(ctx->layers[5].Hin * ctx->layers[5].Win);
      sp.cnv5 = ctx->layers[4].d_out; sp.cnv6 = ctx->layers[5].d_out; sp.w = ctx->d_se5w; sp.part = ctx->d_se5part; sp.count = ctx->d_se5cnt;
      sp.scale = ctx->d_se5scale; sp.out = ctx->d_se5out;
      if (int rc = launch_k(ctx, se5_excite_kernel, dim3(kSe5Splits, npairs), dim3(256), 0, st, false, sp)) return rc;
      const long long total = (long long)npairs * sp.hw * 64;
      if (int rc = launch_k(ctx, se5_scale_kernel, dim3((unsigned)((total + 255) / 256)), dim3(256), 0, st, false, sp)) return rc;
      *launches += 2;
      return 0;
    };
    if (li == 5 && (pse == 1 || pse == 3)) {       // -se_insert: excite cnv5 per branch in front of cnv6; -se_replace: instead of it
      if (int rc = se5(0)) return rc;
      if (pse == 3) continue;                      // cnv6 := se_block(cnv5): there is no cnv6 convolution (posenn.py:234-236)
    }
    int rc = ctx->conv_impl == 0 ? launch_conv(ctx, L, npairs, st) : launch_conv_direct(ctx, L, npairs, st);
    if (rc) return rc;
    *launches += (ctx->conv_impl == 0) ? 1 : L.groups;
    if (ctx->cfg.batch_norm) {                     // the conv wrote plain sums: normalise with this call's batch statistics
      BnParams bp;
      memset(&bp, 0, sizeof bp);
      bp.units = npairs; bp.pair0 = pair0; bp.pair_mode = pair_mode;
      bp.ngroups = (!ctx->unit_sample && pair_mode == DAVO_PAIRS_ALL) ? 2 : 1;
      bp.H = L.Hout; bp.W = L.Wout; bp.Hp = L.Hout_p; bp.Wp = L.Wout_p; bp.C = L.out_stride;
      bp.x = L.d_out; bp.beta = L.d_beta; bp.part = ctx->d_bn_part; bp.mean = ctx->d_bn_mean; bp.rstd = ctx->d_bn_rstd;
      bp.sum_out = ctx->d_sum7;
      if (int rc2 = launch_k(ctx, bn_stats_kernel, dim3(kBnSplits, bp.ngroups), dim3(256), 0, st, false, bp)) return rc2;
      if (int rc2 = launch_k(ctx, bn_finalize_kernel, dim3(bp.ngroups), dim3(256), 0, st, false, bp)) return rc2;
      if (li + 1 == ctx->layers.size()) {
        if (int rc2 = launch_k(ctx, bn_apply_sum_kernel, dim3(npairs), dim3(256), 0, st, false, bp)) return rc2;
      } else {
        const long long total = (long long)npairs * L.Hout * L.Wout * (L.out_stride / 4);
        if (int rc2 = launch_k(ctx, bn_apply_kernel, dim3((unsigned)((total + 255) / 256)), dim3(256), 0, st, false, bp)) return rc2;
      }
      *launches += 3;
    }
    if (li == 5 && pse == 2)                       // -se_skipadd: cnv6 := relu(cnv5 + se_block(cnv6)) (posenn.py:229-233);
      if (int rc2 = se5(1)) return rc2;            // under -batch_norm the block sees the normalised, activated cnv6
  }
  const Layer& L7 = ctx->layers.back();
  if (ctx->conv_impl != 0) {
    sum7_direct_kernel<<<dim3(npairs, ctx->nbr), 256, 0, st>>>(ctx->d_c7tmp, L7.Hout * L7.Wout, ctx->nparts7, ctx->d_sum7);
    CU_OK(cudaGetLastError());
    ++*launches;
  }
  return launch_head(ctx, pair_mode, pair0, npairs, pose_out, st, launches);
}

constexpr int kUnitsAreSamples = 3;     // pair_of_slot mode of the non-shared nets
int pairs_selected(int pairs, int B) {
  return pairs == DAVO_PAIRS_ALL ? 2 * B : (pairs == DAVO_PAIRS_TRAJECTORY || pairs == kUnitsAreSamples) ? B : B + 1;
}

}  // namespace

// =============================================================== C ABI ========

extern "C" const char* davo_build_info(void) {
  return "davo_b200 sm_100a tcgen05/TMA, nvcc " __DATE__;
}

extern "C" int davo_config_bytes(void) { return (int)sizeof(davo_config); }

// include/davo_b200.h: davo_bind_host_numa.  sysfs only; no libnuma in the image.
extern "C" int davo_bind_host_numa(davo_ctx* ctx) {
  if (!ctx) return -1;
  char bus[32] = {0};
  if (cudaDeviceGetPCIBusId(bus, sizeof bus, ctx->device) != cudaSuccess) return -1;
  for (char* c = bus; *c; ++c) *c = (char)tolower(*c);
  char path[128];
  snprintf(path, sizeof path, "/sys/bus/pci/devices/%s/numa_node", bus);
  int node = -1;
  if (FILE* f = fopen(path, "r")) { if (fscanf(f, "%d", &node) != 1) node = -1; fclose(f); }
  if (node < 0) return -1;
  snprintf(path, sizeof path, "/sys/devices/system/node/node%d/cpulist", node);
  FILE* f = fopen(path, "r");
  if (!f) return -1;
  char list[1024] = {0};
  const bool got = fgets(list, sizeof list, f) != nullptr;
  fclose(f);
  if (!got) return -1;
  cpu_set_t allowed, want;
  CPU_ZERO(&want);
  if (sched_getaffinity(0, sizeof allowed, &allowed) != 0) return -1;
  int n = 0;
  for (char* tok = strtok(list, ",\n"); tok; tok = strtok(nullptr, ",\n")) {
    int a = 0, b = 0;
    const int k = sscanf(tok, "%d-%d", &a, &b);
    if (k < 1) continue;
    if (k == 1) b = a;
    for (int c = a; c <= b && c < CPU_SETSIZE; ++c)
      if (CPU_ISSET(c, &allowed)) { CPU_SET(c, &want); ++n; }      // never outside what the container allows
  }
  if (n == 0 || sched_setaffinity(0, sizeof want, &want) != 0) return -1;
  ctx->numa_node = node; ctx->numa_cpus = n;
  return node;
}

extern "C" const char* davo_last_error(const davo_ctx* ctx) {
  return ctx ? ctx->err.c_str() : g_create_error.c_str();
}

extern "C" int davo_create(const davo_config* cfg, int device, davo_ctx** out) {
  davo_ctx* ctx = nullptr;   // errors before allocation go to the thread-local slot
  if (!cfg || !out) return fail(nullptr, DAVO_ERR_ARG, "davo_create: null argument");
  *out = nullptr;
  if (cfg->posenn < 0 || cfg->posenn > 5)
    return fail(nullptr, DAVO_ERR_ARG, "davo_create: PoseNN kind %d unknown (0..5, posenn.py:12-378)", cfg->posenn);
  if (cfg->posenn_se < 0 || cfg->posenn_se > 3)
    return fail(nullptr, DAVO_ERR_ARG, "davo_create: PoseNN-internal SE mode %d unknown (1 insert, 2 skipadd, 3 replace)", cfg->posenn_se);
  if (cfg->batch_norm != 0 && cfg->batch_norm != 1)
    return fail(nullptr, DAVO_ERR_ARG, "davo_create: batch_norm is 0 or 1");
  if (cfg->posenn_se == 2 && cfg->cnv6_out != 256)
    return fail(nullptr, DAVO_ERR_ARG, "davo_create: -se_skipadd adds cnv5 (256 channels) to se_block(cnv6): cnv6 width must be 256, got %d", cfg->cnv6_out);
  if (cfg->H <= 0 || cfg->W <= 0 || (cfg->H % 8) || (cfg->W % 8))
    return fail(nullptr, DAVO_ERR_ARG, "davo_create: H and W must be positive multiples of 8 (got %dx%d)", cfg->H, cfg->W);
  if (cfg->max_batch <= 0) return fail(nullptr, DAVO_ERR_ARG, "davo_create: max_batch must be positive");
  if (cfg->cnv6_out != 256 && cfg->cnv6_out != 128 && cfg->cnv6_out != 64 && cfg->cnv6_out != 32)
    return fail(nullptr, DAVO_ERR_ARG, "davo_create: cnv6 width %d unsupported (32, 64, 128 or 256)", cfg->cnv6_out);
  if (cfg->in_mode != 0 && cfg->in_mode != 1) return fail(nullptr, DAVO_ERR_ARG, "davo_create: bad in_mode");
  if (cfg->att_src < 0 || cfg->att_src > 6) return fail(nullptr, DAVO_ERR_ARG, "davo_create: bad att_src");
  if (cfg->se_pool < 0 || cfg->se_pool > 4 || cfg->se_hidden < 0 || cfg->se_hidden > 19 ||
      (cfg->se_pool != 0 && cfg->att_src != 1 && cfg->att_src != 3 && !(cfg->att_src == 6 && cfg->pixel_map == 1 && cfg->se_pool == 2)))
    return fail(nullptr, DAVO_ERR_ARG, "davo_create: bad se_pool / se_hidden");
  if (cfg->se_pool >= 2 && (cfg->H > cfg->W || (cfg->att_src == 1 && !cfg->att_tgt_ones)))
    return fail(nullptr, DAVO_ERR_ARG, "davo_create: the pyramid pooling is built for H <= W (and, on the flow, a target map of ones)");
  if (cfg->depth_split != 0 && (cfg->depth_split != 1 || cfg->att_src != 1 || cfg->se_pool != 0 || !cfg->att_tgt_ones))
    return fail(nullptr, DAVO_ERR_ARG, "davo_create: depth_split needs att_src 1 with global pooling and a target map of ones");
  if (cfg->pixel_map != 0 && (cfg->pixel_map < 1 || cfg->pixel_map > 2 || (cfg->pixel_map == 2 && cfg->att_src != 5) ||
                              cfg->att_src < 4 || cfg->att_src > 6 || (cfg->se_pool != 0 && cfg->att_src != 6)))
    return fail(nullptr, DAVO_ERR_ARG, "davo_create: per-pixel maps are built for att_src 4..6 and global pooling");
  if (cfg->att_src == 5 && ((cfg->H * cfg->W) % 4) != 0) return fail(nullptr, DAVO_ERR_ARG, "davo_create: se_depth needs H*W % 4 == 0");
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0)
    return fail(nullptr, DAVO_ERR_CUDA, "davo_create: no CUDA device (%s); there is no CPU fallback", cudaGetErrorString(e));
  if (device < 0 || device >= ndev) return fail(nullptr, DAVO_ERR_ARG, "davo_create: device %d out of range", device);
  cudaDeviceProp prop;
  e = cudaGetDeviceProperties(&prop, device);
  if (e != cudaSuccess) return fail(nullptr, DAVO_ERR_CUDA, "cudaGetDeviceProperties: %s", cudaGetErrorString(e));
  if (prop.major != 10)
    return fail(nullptr, DAVO_ERR_CUDA, "davo_create: device is sm_%d%d; this library is sm_100a only", prop.major, prop.minor);
  e = cudaSetDevice(device);
  if (e != cudaSuccess) return fail(nullptr, DAVO_ERR_CUDA, "cudaSetDevice: %s", cudaGetErrorString(e));
  ctx = new davo_ctx();
  ctx->cfg = *cfg;
  ctx->device = device;
  ctx->num_sms = prop.multiProcessorCount;
  // Frame pairs per pass of the conv stack.  Large passes amortise launch, prologue and the last
  // partial wave of every layer (measured: 62 k pairs/s at 34, 73 k at 256); 256 pairs keep the
  // workspace at 3.6 GB.
  int mb = cfg->micro_batch > 0 ? cfg->micro_batch : 256;
  ctx->unit_sample = cfg->posenn >= 2;
  if (mb > ctx->max_units()) mb = ctx->max_units();
  ctx->mb = mb;
  if (const char* e = getenv("DAVO_B200_HOST_SEG8")) ctx->host_seg8 = strcmp(e, "0") != 0;   // "0": labels cross PCIe as floats
  ctx->host_flow16 = cfg->flow_f16 != 0;        // the binary16 transport exists only where the flow is defined as binary16
  if (const char* e = getenv("DAVO_B200_HOST_FLOW16")) ctx->host_flow16 = ctx->host_flow16 && strcmp(e, "0") != 0;   // "0": flow crosses PCIe as float32
  if (const char* e = getenv("DAVO_B200_HOST_FLOW16_FRAC")) ctx->flow16_frac = std::max(0.0f, std::min(1.0f, (float)atof(e)));
  if (const char* e = getenv("DAVO_B200_PDL")) ctx->pdl = strcmp(e, "0") != 0;               // "0": plain stream order
  if (const char* cr = getenv("DAVO_B200_WEIGHT_ROUNDING"))     // "nearest": plain round-to-nearest
    ctx->compensated_rounding = strcmp(cr, "nearest") != 0;
  *out = ctx;
  return 0;
}

static void destroy_sessions_of(davo_ctx* ctx);

extern "C" void davo_destroy(davo_ctx* ctx) {
  if (!ctx) return;
  destroy_sessions_of(ctx);
  cudaSetDevice(ctx->device);
  for (void* p : ctx->allocs) cudaFree(p);
  if (ctx->d_traj_scratch) cudaFree(ctx->d_traj_scratch);
  if (ctx->jpeg_state) davo_jpeg::api().StateDestroy(ctx->jpeg_state);
  if (ctx->jpeg_handle) davo_jpeg::api().Destroy(ctx->jpeg_handle);
  for (int i = 0; i < davo_ctx::kStage; ++i) {
    if (ctx->s_img[i]) cudaFree(ctx->s_img[i]);
    if (ctx->s_flow[i]) cudaFree(ctx->s_flow[i]);
    if (ctx->s_seg[i]) cudaFree(ctx->s_seg[i]);
    if (ctx->s_depth[i]) cudaFree(ctx->s_depth[i]);
    if (ctx->s_seg8[i]) cudaFree(ctx->s_seg8[i]);
    if (ctx->s_flow16[i]) cudaFree(ctx->s_flow16[i]);
    if (ctx->h_flow16[i]) cudaFreeHost(ctx->h_flow16[i]);
    if (ctx->h_seg8[i]) cudaFreeHost(ctx->h_seg8[i]);
    if (ctx->ev_seg8[i]) cudaEventDestroy(ctx->ev_seg8[i]);
    if (ctx->ev_copied[i]) cudaEventDestroy(ctx->ev_copied[i]);
    if (ctx->ev_consumed[i]) cudaEventDestroy(ctx->ev_consumed[i]);
  }
  cudaFree(ctx->m_img); cudaFree(ctx->m_lab); cudaFree(ctx->m_depth); cudaFree(ctx->m_flow); cudaFree(ctx->m_pose);
  for (int i = 0; i < davo_ctx::kManyRing; ++i) {
    if (ctx->m_hdesc[i]) cudaFreeHost(ctx->m_hdesc[i]);
    if (ctx->m_ddesc[i]) cudaFree(ctx->m_ddesc[i]);
    if (ctx->m_ev[i]) cudaEventDestroy(ctx->m_ev[i]);
  }
  for (int i = 0; i < 2; ++i) {
    if (ctx->q_img[i]) cudaFree(ctx->q_img[i]);
    if (ctx->q_seg8[i]) cudaFree(ctx->q_seg8[i]);
    if (ctx->q_seg[i]) cudaFree(ctx->q_seg[i]);
    if (ctx->q_depth[i]) cudaFree(ctx->q_depth[i]);
    if (ctx->ev_q_done[i]) cudaEventDestroy(ctx->ev_q_done[i]);
    if (ctx->a_dev[i]) cudaFree(ctx->a_dev[i]);
    if (ctx->a_pin[i]) cudaFreeHost(ctx->a_pin[i]);
    if (ctx->a_copied[i]) cudaEventDestroy(ctx->a_copied[i]);
    if (ctx->a_done[i]) cudaEventDestroy(ctx->a_done[i]);
  }
  cudaFree(ctx->m_hpose);
  cudaFree(ctx->att_stage);
  cudaFree(ctx->b_stage); cudaFree(ctx->b_ddesc);
  if (ctx->b_hdesc) cudaFreeHost(ctx->b_hdesc);
  delete ctx->pool;
  if (ctx->comm) davo_comm::api().CommDestroy(ctx->comm);
  if (ctx->s_pose) cudaFree(ctx->s_pose);
  if (ctx->ev_start) cudaEventDestroy(ctx->ev_start);
  for (cudaEvent_t& ev : ctx->ev_host_done) if (ev) cudaEventDestroy(ev);
  if (ctx->copy_stream) cudaStreamDestroy(ctx->copy_stream);
  delete ctx;
}

extern "C" int davo_set_weight(davo_ctx* ctx, const char* name, const float* host,
                               const int64_t* shape, int rank) {
  if (!ctx) return DAVO_ERR_ARG;
  if (!name || !host || (!shape && rank > 0) || rank < 0 || rank > 4) return fail(ctx, DAVO_ERR_ARG, "davo_set_weight: bad argument");   // rank 0: a scalar variable
  if (ctx->finalized) return fail(ctx, DAVO_ERR_STATE, "davo_set_weight: weights already finalized");
  HostTensor t;
  size_t n = 1;
  for (int i = 0; i < rank; ++i) { t.shape.push_back(shape[i]); n *= (size_t)shape[i]; }
  t.data.assign(host, host + n);
  ctx->weights[name] = std::move(t);
  return 0;
}

extern "C" int davo_finalize_weights(davo_ctx* ctx) {
  if (!ctx) return DAVO_ERR_ARG;
  if (ctx->finalized) return fail(ctx, DAVO_ERR_STATE, "davo_finalize_weights: already finalized");
  CU_OK(cudaSetDevice(ctx->device));
  const davo_config& c = ctx->cfg;
  const int mb = ctx->mb;
  const std::string P = "pose_exp_net/";
  const int c6 = c.cnv6_out;
  // cnv1 input channels of the reference: (rgb [+ flow]) x (tgt + sources), posenn.py:21, 198
  const int cin1 = (c.in_mode == 1 ? 5 : 3) * (1 + (c.posenn >= 2 ? 2 : 1));
  int Hq = c.H, Wq = c.W;                          // pitch of the running activation

  // ---- activation geometry (TF SAME) ----
  struct Geo { int k, stride, dil; };
  // dilated nets (posenn.py:12-254): cnv3-5 dilated 2/4/8, cnv6 dilated 2; the original nets
  // (couple_net_v0 / decouple_net_v0, posenn.py:257-378): stride 2 all the way down
  const bool dilated = c.posenn <= 3;
  const Geo geo_dil[7] = {{7, 2, 1}, {5, 2, 1}, {3, 1, 2}, {3, 1, 4}, {3, 1, 8}, {3, 1, 2}, {3, 2, 1}};
  const Geo geo_v0[7] = {{7, 2, 1}, {5, 2, 1}, {3, 2, 1}, {3, 2, 1}, {3, 2, 1}, {3, 2, 1}, {3, 2, 1}};
  // -se_skipadd in the original nets: there, and only there, cnv6 runs at stride 1 (posenn.py:292, 355), so that
  // cnv5 + se_block(cnv6) add maps of one size
  const Geo geo_v0_skip[7] = {{7, 2, 1}, {5, 2, 1}, {3, 2, 1}, {3, 2, 1}, {3, 2, 1}, {3, 1, 1}, {3, 2, 1}};
  const Geo* geo = dilated ? geo_dil : (c.posenn_se == 2 ? geo_v0_skip : geo_v0);
  // couple nets (posenn.py:133-187): one branch, pred 256 -> 6; decouple nets: rotation | translation
  const int nbr = (c.posenn == 1 || c.posenn == 3 || c.posenn == 4) ? 1 : 2;
  // two 256-wide cnv6 branches (-cnv6_256, which -se_skipadd requires) on a map too short for the channels-on-M plan
  // (the stride-2 nets; a dilated net on a frame under 128 rows): the branches run as groups of one pixels-on-M layer
  // that all read the SAME input -- a fused N = 512 accumulator does not exist there
  const int h_cnv3_in = same_pad(same_pad(c.H, 7, 2, 1).out, 5, 2, 1).out;
  const bool skip_grouped = c.cnv6_out == 256 && nbr == 2 && c.posenn_se != 1 && c.posenn_se != 3 && !(dilated && h_cnv3_in >= 32);
  const int nsrc = ctx->unit_sample ? 2 : 1;      // poses per evaluation (num_source, posenn.py:19, 76, 140, 196)
  ctx->nbr = nbr;
  const int cout_total[7] = {16, 32, 64, 128, 256, nbr * c6, nbr * 256};
  const int bn[7] = {16, 32, 64, 128, 256, ((c.posenn_se == 1 || skip_grouped) ? 1 : nbr) * c6, 256};
  const int groups[7] = {1, 1, 1, 1, 1, (c.posenn_se == 1 || skip_grouped) ? nbr : 1, nbr};
  // -se_insert: cnv6 reads two differently scaled copies of cnv5 (one per branch): a grouped layer
  const bool se5 = c.posenn_se == 1;
  // -se_replace: cnv6 IS the excited cnv5 (256 channels per branch); cnv7 reads the scaled copies directly
  const bool rep = c.posenn_se == 3;
  // -se_skipadd: cnv6 (256 channels per branch, one N = nbr*256 GEMM) feeds an SE block and is added to cnv5; cnv7
  // reads relu(cnv5 + se_block(cnv6)) from the same per-branch buffer -se_replace uses
  const bool skip = c.posenn_se == 2;
  const int c7in = rep ? 256 : c6;
  // Packed PoseNN input (frontend.cuh: pack_kernel): 8 channels per pixel when the width allows the
  // column-widened cnv1 plan (runs of 16 input pixels), else the 16-channel layout of the plain plan.
  const char* wide_env0 = getenv("DAVO_B200_WIDE");
  // (the per-pixel attention maps are computed by the 16-channel pack_kernel only)
  ctx->packed_c = (!ctx->unit_sample && !c.pixel_map && !c.depth_split && (c.W % 16) == 0 && !(wide_env0 && !strcmp(wide_env0, "0"))) ? 8 : 16;
  const int cin_total[7] = {ctx->packed_c, 16, 32, 64, 128, se5 ? nbr * 256 : 256, nbr * c7in};   // skip: c6 == 256, so cnv7 reads nbr*256 as well
  const int cin_g[7] = {ctx->packed_c, 16, 32, 64, 128, 256, c7in};
  const int cin_w[7] = {cin1, 16, 32, 64, 128, 256, c7in};
  const char* names[7] = {"cnv1", "cnv2", "cnv3", "cnv4", "cnv5", "cnv6", "cnv7"};
  ctx->layers.resize(7);
  int H = c.H, W = c.W;
  for (int i = 0; i < 7; ++i) {
    Layer& L = ctx->layers[i];
    L.name = names[i];
    L.k = geo[i].k; L.stride = geo[i].stride; L.dil = geo[i].dil;
    L.Hin = H; L.Win = W; L.Hin_p = Hq; L.Win_p = Wq;
    L.Cin_total = cin_total[i]; L.Cin_g = cin_g[i]; L.groups = groups[i];
    L.Cin_w = cin_w[i];
    L.BN = bn[i];
    L.cin_shared = i == 5 && skip_grouped;
    SamePad ph = same_pad(H, L.k, L.stride, L.dil), pw = same_pad(W, L.k, L.stride, L.dil);
    L.Hout = ph.out; L.Wout = pw.out; L.pad_t = ph.before; L.pad_l = pw.before;
    L.Hout_p = L.Hout + (L.Hout & 1); L.Wout_p = L.Wout + (L.Wout & 1);      // even pitches: the stride-2 consumer views rows and columns in pairs (a 1-row map too)
    if (i == 6 && !c.batch_norm) { L.Hout_p = L.Hout; L.Wout_p = L.Wout; }      // cnv7 is never stored ...
    L.out_stride = cout_total[i];
    L.epi = (i == 6 && !c.batch_norm) ? EPI_SUM_RELU : EPI_STORE_RELU;   // ... except under -batch_norm, whose statistics need the whole map
    // Orientation (measured, DESIGN.md 4.1): channels-on-M for the wide stride-1 layers whose
    // maps are tall enough for a 32-row tile; pixels-on-M for thin layers and the summed cnv7.
    const char* force = getenv("DAVO_B200_ORIENT");          // debug: "pm" or "cm" for every layer
    L.orient = (L.stride == 1 && L.BN >= 128 && L.Hout >= 32) ? 1 : 0;
    if (force && !strcmp(force, "pm")) L.orient = 0;
    if (force && !strcmp(force, "cm")) L.orient = 1;
    if (L.orient == 0 && L.epi == EPI_SUM_RELU && L.BN != 256) L.orient = 1;
    // cnv7 channels-on-M (experiment knob, DESIGN.md 8): 128-pixel tiles, 2-CTA clusters sharing the weight slabs
    if (const char* e7 = getenv("DAVO_B200_CNV7_CM")) if (i == 6 && !strcmp(e7, "1") && L.epi == EPI_SUM_RELU) L.orient = 1;
    L.npix = (L.orient == 1 && L.Hout > 16) ? 256 : 128;
    L.m_blocks = L.orient == 1 ? (L.BN + cm::kBlockM - 1) / cm::kBlockM : 1;
    L.tiles_h = (L.Hout + L.npix / kTileW - 1) / (L.npix / kTileW);
    L.tiles_w = (L.Wout + kTileW - 1) / kTileW;
    // Thin stride-2 layers: runs of G output pixels on one M row, N = G * Cout = 128 (conv_pm.cuh, WIDE).
    const char* wide_env = getenv("DAVO_B200_WIDE");          // debug: "0" switches the widened plan off
    const int G = 128 / L.BN;
    if (L.orient == 0 && L.stride == 2 && (L.Cin_total == 16 || L.Cin_total == 8) && L.groups == 1 && L.BN <= 32 &&
        (L.Win % (2 * G)) == 0 &&
        L.epi == EPI_STORE_RELU && !(wide_env && !strcmp(wide_env, "0"))) {
      const int runs = L.Wout / G;
      long best = -1;
      for (int tw = 2; tw <= 8; tw *= 2) {
        const long tiles = (long)((L.Hout + 128 / tw - 1) / (128 / tw)) * ((runs + tw - 1) / tw);
        if (best < 0 || tiles < best) { best = tiles; L.wide_tw = tw; }
      }
      L.wide_G = G;
      // Experiment (DAVO_B200_FUSED_FRONT=1): cnv1 builds its operand from the raw inputs (conv_pm.cuh: FUSED)
      if (const char* ef = getenv("DAVO_B200_FUSED_FRONT"))
        if (!strcmp(ef, "1") && i == 0 && ctx->packed_c == 8 && L.Cin_total == 8) { L.fused_front = true; ctx->fuse_front = true; }
      L.tiles_h = (L.Hout + 128 / L.wide_tw - 1) / (128 / L.wide_tw);
      L.tiles_w = (runs + L.wide_tw - 1) / L.wide_tw;
    }
    for (int j = 0; j < 16; ++j) { L.cmap[j] = j; L.pc2w[j] = j < L.Cin_w ? j : -1; }
    if (!(i == 5 && c.posenn_se == 3)) {             // -se_replace: there is no cnv6 (cnv6 := se_block(cnv5)): cnv7 reads cnv5's map
      H = L.Hout; W = L.Wout; Hq = L.Hout_p; Wq = L.Wout_p;
    }
  }
  {
    // cnv1 reads the packed input.  The reference's cnv1 sees [tgt rgb, tgt flow (zeros), src rgb,
    // src flow] (v1: 10 channels) or [tgt rgb, src rgb] (v0: 6).  Packed layouts:
    //   8 channels:  tgt rgb, src rgb, src flow            (the all-zero target flow is not stored)
    //   16 channels: tgt rgb, 0 0, src rgb, src flow, 6 x TF32 residuals (ignored: measured to
    //                make no difference once the weights are rounded with compensation, DESIGN.md 5)
    Layer& L = ctx->layers[0];
    if (L.wide_G == 0 && ctx->packed_c == 8)
      return fail(ctx, DAVO_ERR_ARG, "cnv1: 8-channel packed input needs the widened plan");
    for (int j = 0; j < 16; ++j) L.pc2w[j] = -1;
    const int per_frame = c.in_mode == 1 ? 5 : 3;           // reference channels per frame: rgb [+ flow]
    if (ctx->unit_sample) {
      // pack_sample_kernel: 0-2 tgt rgb, 3-5 src0 rgb, 6-7 src0 flow, 8-10 src1 rgb, 11-12 src1 flow
      for (int j = 0; j < 3; ++j) {
        L.pc2w[j] = j;
        L.pc2w[3 + j] = per_frame + j;
        L.pc2w[8 + j] = 2 * per_frame + j;
      }
      if (c.in_mode == 1)
        for (int j = 0; j < 2; ++j) { L.pc2w[6 + j] = per_frame + 3 + j; L.pc2w[11 + j] = 2 * per_frame + 3 + j; }
    } else {
      const int rgb_src = ctx->packed_c == 8 ? 3 : 5, flow_src = ctx->packed_c == 8 ? 6 : 8;
      for (int j = 0; j < 3; ++j) {
        L.pc2w[j] = j;                                        // tgt rgb
        L.pc2w[rgb_src + j] = per_frame + j;                  // src rgb
      }
      if (c.in_mode == 1) { L.pc2w[flow_src] = 8; L.pc2w[flow_src + 1] = 9; }
    }
    L.use_cmap = 1;                                         // direct cross-check path: weight channel -> packed channel
    for (int ci = 0; ci < L.Cin_w; ++ci) {
      L.cmap[ci] = 0;
      bool found = false;
      for (int j = 0; j < 16; ++j) if (L.pc2w[j] == ci) { L.cmap[ci] = j; found = true; }
      if (!found) L.cmap[ci] = -1;                          // the target's zero flow: no packed channel
    }
  }

  // ---- workspace ----
  if (int rc = dev_alloc(ctx, (void**)&ctx->d_pool, (size_t)mb * kAttFrames * kPoolSplits * kPoolDim * 4)) return rc;
  if (int rc = dev_alloc(ctx, (void**)&ctx->d_poolcnt, (size_t)mb * kAttFrames * 4)) return rc;
  if (int rc = dev_alloc(ctx, (void**)&ctx->d_attw, (size_t)mb * kAttFrames * kAttStride * 4)) return rc;
  if (int rc = dev_alloc(ctx, (void**)&ctx->d_packed, (size_t)mb * c.H * c.W * ctx->packed_c * 4)) return rc;
  if (int rc = dev_alloc(ctx, (void**)&ctx->d_pipe, (size_t)(4 + mb) * 4)) return rc;
  CU_OK(cudaMemset(ctx->d_pipe, 0, (size_t)(4 + mb) * 4));
  float* prev = ctx->d_packed;
  for (int i = 0; i < 7; ++i) {
    Layer& L = ctx->layers[i];
    if (i == 5 && (se5 || rep || skip)) {
      const size_t hw5 = (size_t)L.Hin_p * L.Win_p;
      if (int rc = dev_alloc(ctx, (void**)&ctx->d_se5part, (size_t)mb * kSe5Splits * 256 * (skip ? nbr : 1) * 4)) return rc;
      if (int rc = dev_alloc(ctx, (void**)&ctx->d_se5cnt, (size_t)mb * 4)) return rc;
      if (int rc = dev_alloc(ctx, (void**)&ctx->d_se5scale, (size_t)mb * 2 * 256 * 4)) return rc;
      if (int rc = dev_alloc(ctx, (void**)&ctx->d_se5out, (size_t)mb * hw5 * nbr * 256 * 4)) return rc;
      if (!skip) prev = ctx->d_se5out;          // skip: cnv6 still reads cnv5; cnv7 reads d_se5out (below)
    }
    L.d_in = (i == 6 && skip) ? ctx->d_se5out : prev;
    if (i == 5 && rep) continue;                   // no cnv6 convolution and no buffer: cnv7 reads d_se5out
    if (i < 6 || c.batch_norm) {
      if (int rc = dev_alloc(ctx, (void**)&L.d_out, (size_t)mb * L.Hout_p * L.Wout_p * L.out_stride * 4)) return rc;
      prev = L.d_out;
    }
  }
  {
    const Layer& L7 = ctx->layers[6];
    ctx->nparts7 = c.batch_norm ? 1 : L7.tiles_h * L7.tiles_w * (L7.orient == 0 ? 4 : 1);    // bn_apply_sum_kernel writes one row per unit
    if (c.batch_norm) {
      if (int rc = dev_alloc(ctx, (void**)&ctx->d_bn_part, (size_t)2 * kBnSplits * 2 * kBnMaxC * sizeof(double))) return rc;
      if (int rc = dev_alloc(ctx, (void**)&ctx->d_bn_mean, (size_t)2 * kBnMaxC * 4)) return rc;
      if (int rc = dev_alloc(ctx, (void**)&ctx->d_bn_rstd, (size_t)2 * kBnMaxC * 4)) return rc;
    }
    if (int rc = dev_alloc(ctx, (void**)&ctx->d_sum7, (size_t)mb * nbr * ctx->nparts7 * 256 * 4)) return rc;
  }

  // ---- weights ----
  // -batch_norm: slim creates <scope>/BatchNorm/beta instead of <scope>/biases for every conv but pred (posenn.py:206, 240).
  // The beta vector is handed back through `b` (the callers assemble it per output channel exactly like a bias) and
  // ends up in Layer::d_beta; the conv itself then runs with a zero bias (plan_layer_bn below).
  auto need_conv = [&](const std::string& scope, int k, int ci, int co, const HostTensor** w, const HostTensor** b) -> int {
    const bool bn_layer = c.batch_norm && scope.size() >= 4 && scope.compare(scope.size() - 4, 4, "pred") != 0;
    *w = find_w(ctx, P + scope + "/weights");
    *b = find_w(ctx, P + scope + (bn_layer ? "/BatchNorm/beta" : "/biases"));
    if (!*w || !*b) return fail(ctx, DAVO_ERR_WEIGHT, "missing variable %s%s/{weights,%s}", P.c_str(), scope.c_str(), bn_layer ? "BatchNorm/beta" : "biases");
    if (!shape_is(*w, {k, k, ci, co}) || !shape_is(*b, {co}))
      return fail(ctx, DAVO_ERR_WEIGHT, "variable %s%s has the wrong shape (want [%d,%d,%d,%d])", P.c_str(), scope.c_str(), k, k, ci, co);
    return 0;
  };
  // -batch_norm: the per-channel vector the callers assembled is beta, kept for bn.cuh; the conv adds nothing
  auto bias_or_beta = [&](Layer& L, const std::vector<float>& v, std::vector<float>* out) -> int {
    *out = v;
    if (!c.batch_norm) return 0;
    if (int rc = dev_alloc(ctx, (void**)&L.d_beta, v.size() * 4)) return rc;
    CU_OK(cudaMemcpy(L.d_beta, v.data(), v.size() * 4, cudaMemcpyHostToDevice));
    std::fill(out->begin(), out->end(), 0.f);
    return 0;
  };
  // plan a layer and, for the channels-on-M layers with 256-pixel tiles, its latency twin with 128-pixel tiles
  ctx->layers_small.assign(7, Layer());
  for (Layer& Ls : ctx->layers_small) Ls.npix = 0;
  const char* small_env = getenv("DAVO_B200_SMALL_TILES");          // debug: "0" never uses the latency plans
  auto plan_both = [&](int idx, auto getw, const std::vector<float>& bias) -> int {
    Layer& L = ctx->layers[idx];
    if (int rc = L.wide_G ? plan_layer_wide(ctx, L, getw, bias) : plan_layer(ctx, L, getw, bias)) return rc;
    if (L.orient == 1 && L.npix == 256 && L.epi == EPI_STORE_RELU && !(small_env && !strcmp(small_env, "0"))) {
      Layer Ls = L;
      Ls.npix = 128;
      Ls.tiles_h = (Ls.Hout + Ls.npix / kTileW - 1) / (Ls.npix / kTileW);
      Ls.d_wpack = nullptr; Ls.d_bias = nullptr; Ls.d_whwio[0] = Ls.d_whwio[1] = nullptr;
      if (int rc = plan_layer(ctx, Ls, getw, bias)) return rc;
      ctx->layers_small[idx] = Ls;
    }
    return 0;
  };
  for (int i = 0; i < 5; ++i) {
    Layer& L = ctx->layers[i];
    const HostTensor *w, *b;
    if (int rc = need_conv(names[i], L.k, L.Cin_w, L.BN, &w, &b)) return rc;
    const int Ci = L.Cin_w, Co = L.BN, K = L.k;
    auto getw = [&](int, int ty, int tx, int ci, int n) { return w->data[(((size_t)ty * K + tx) * Ci + ci) * Co + n]; };
    std::vector<float> bias;
    if (int rc = bias_or_beta(L, b->data, &bias)) return rc;
    if (int rc = plan_both(i, getw, bias)) return rc;
  }
  const char* brs[2] = {"rotation", "translation"};
  // variable scope of branch g under pose_exp_net/: pose/rotation/, pose/translation/ (decouple) or pose/ (couple)
  auto branch_scope = [&](int g) { return nbr == 2 ? std::string("pose/") + brs[g] + "/" : std::string("pose/"); };
  if (!rep) {
    Layer& L = ctx->layers[5];
    const HostTensor *w[2], *b[2];
    for (int g = 0; g < nbr; ++g)
      if (int rc = need_conv(branch_scope(g) + "cnv6", 3, 256, c6, &w[g], &b[g])) return rc;
    std::vector<float> bias0(nbr * c6), bias;
    for (int n = 0; n < nbr * c6; ++n) bias0[n] = b[n / c6]->data[n % c6];
    if (int rc = bias_or_beta(L, bias0, &bias)) return rc;
    if (se5 || skip_grouped) {      // two groups: branch g convolves its own scaled copy of cnv5 (skip_grouped: the same cnv5)
      auto getw = [&](int g, int ty, int tx, int ci, int n) {
        return w[g]->data[(((size_t)ty * 3 + tx) * 256 + ci) * c6 + n];
      };
      if (int rc = plan_both(5, getw, bias)) return rc;
    } else {        // one N = 2*c6 GEMM: rotation | translation
      auto getw = [&](int, int ty, int tx, int ci, int n) {
        const HostTensor* t = w[n / c6];
        return t->data[(((size_t)ty * 3 + tx) * 256 + ci) * c6 + (n % c6)];
      };
      if (int rc = plan_both(5, getw, bias)) return rc;
    }
  }
  if (se5 || rep || skip) {
    // reference nets/posenn.py:227 / :232, :236: variables pose/<branch>/cnv5_se_attention/{bottleneck_fc,recover_fc}
    // (-se_insert) or pose/<branch>/cnv6_se_attention/... (-se_skipadd, -se_replace)
    std::vector<float> sw;
    for (int g = 0; g < nbr; ++g) {
      const std::string S = P + branch_scope(g) + ((rep || skip) ? "cnv6_se_attention/" : "cnv5_se_attention/");
      const HostTensor* w1 = find_w(ctx, S + "bottleneck_fc/kernel");
      const HostTensor* b1 = find_w(ctx, S + "bottleneck_fc/bias");
      const HostTensor* w2 = find_w(ctx, S + "recover_fc/kernel");
      const HostTensor* b2 = find_w(ctx, S + "recover_fc/bias");
      if (!shape_is(w1, {256, 32}) || !shape_is(b1, {32}) || !shape_is(w2, {32, 256}) || !shape_is(b2, {256}))
        return fail(ctx, DAVO_ERR_WEIGHT, "missing or mis-shaped %s{bottleneck_fc,recover_fc}/{kernel,bias}", S.c_str());
      sw.insert(sw.end(), w1->data.begin(), w1->data.end());
      sw.insert(sw.end(), b1->data.begin(), b1->data.end());
      sw.insert(sw.end(), w2->data.begin(), w2->data.end());
      sw.insert(sw.end(), b2->data.begin(), b2->data.end());
    }
    if (int rc = dev_alloc(ctx, (void**)&ctx->d_se5w, sw.size() * 4)) return rc;
    CU_OK(cudaMemcpy(ctx->d_se5w, sw.data(), sw.size() * 4, cudaMemcpyHostToDevice));
  }
  {
    Layer& L = ctx->layers[6];
    const HostTensor *w[2], *b[2];
    for (int g = 0; g < nbr; ++g)
      if (int rc = need_conv(branch_scope(g) + "cnv7", 3, c7in, 256, &w[g], &b[g])) return rc;
    auto getw = [&](int g, int ty, int tx, int ci, int n) {
      return w[g]->data[(((size_t)ty * 3 + tx) * c7in + ci) * 256 + n];
    };
    std::vector<float> bias0(nbr * 256), bias;
    for (int n = 0; n < nbr * 256; ++n) bias0[n] = b[n / 256]->data[n % 256];
    if (int rc = bias_or_beta(L, bias0, &bias)) return rc;
    if (int rc = plan_layer(ctx, L, getw, bias)) return rc;
    if (int rc = dev_alloc(ctx, (void**)&ctx->d_c7tmp, (size_t)mb * L.Hout * L.Wout * nbr * 256 * 4)) return rc;
  }
  {
    // pred: [256, 3*num_source] per branch (decouple, posenn.py:117, 240) or [256, 6*num_source]
    // (couple, :58, 181); stored [br][256][per]
    const int per = 6 * nsrc / nbr;
    std::vector<float> wp(256 * 6 * nsrc), bp(6 * nsrc);
    for (int g = 0; g < nbr; ++g) {
      const HostTensor *w, *b;
      if (int rc = need_conv(branch_scope(g) + "pred", 1, 256, per, &w, &b)) return rc;
      for (int i = 0; i < 256 * per; ++i) wp[g * 256 * per + i] = w->data[i];
      for (int j = 0; j < per; ++j) bp[g * per + j] = b->data[j];
    }
    if (int rc = dev_alloc(ctx, (void**)&ctx->d_wpred, wp.size() * 4)) return rc;
    if (int rc = dev_alloc(ctx, (void**)&ctx->d_bpred, bp.size() * 4)) return rc;
    CU_OK(cudaMemcpy(ctx->d_wpred, wp.data(), wp.size() * 4, cudaMemcpyHostToDevice));
    CU_OK(cudaMemcpy(ctx->d_bpred, bp.data(), bp.size() * 4, cudaMemcpyHostToDevice));
  }
  if (int rc = dev_alloc(ctx, (void**)&ctx->d_sew, (kSegCellsMaxDim * 19 + 19 + 19 * 19 + 19) * 4)) return rc;
  if (int rc = dev_alloc(ctx, (void**)&ctx->d_staticw, kNumClasses * 4)) return rc;
  if (c.att_src == 1 || c.att_src >= 3) {
    // se(flow|rgb, [8,19]) (attention_module.py:54-103) or se_block(seg_19, ratio=1) (:9-52)
    const std::string S = P + (c.att_src == 1 ? "se_flow/" : c.att_src == 3 ? (c.se_pool >= 2 ? "se_spp_seg/" : "se_seg/") : c.att_src == 4 ? "se_rgb/" : c.att_src == 5 ? (c.pixel_map == 2 ? (c.depth_norm == 2 ? "se_dispflow/" : "se_depthflow/") : c.depth_norm == 2 ? "se_disp/" : "se_depth/") : (c.se_pool >= 2 ? "se_spp_segflow/" : "se_segflow/"));
    static const int spp_dim[5] = {2, 8, 10, 8, kSppMaxDim};      // pooled vector of se_flow by se_pool: gp, gp2x2, spp [2,1], [2], [8,6,4]
    static const int cells[5] = {1, 4, 5, 4, 116};                // pooled cells by se_pool
    const int din = c.att_src == 1 ? spp_dim[c.se_pool] : c.att_src == 3 ? 19 * cells[c.se_pool] : c.att_src == 4 ? 3 : c.att_src == 5 ? (c.pixel_map == 2 ? 3 : 1) : 21 * cells[c.se_pool];
    const int chan = c.att_src == 6 ? 21 : din;             // channels of the SE input (the pooled vector may be several cells of them)
    const int dh = c.pixel_map ? chan : c.se_hidden > 0 ? c.se_hidden : ((c.att_src == 3 || c.att_src == 6) ? 19 : 8);
    const int dout = c.pixel_map ? chan : 19;
    // depth_split: the two SEs "se_flow_near", "se_flow_far" (davo.py:1150) one after the other, and the threshold
    std::vector<std::string> scopes = {S};
    if (c.depth_split) scopes = {P + "se_flow_near/", P + "se_flow_far/"};
    std::vector<float> se;
    for (const std::string& sc : scopes) {
      const HostTensor* w1 = find_w(ctx, sc + "bottleneck_fc/kernel");
      const HostTensor* b1 = find_w(ctx, sc + "bottleneck_fc/bias");
      const HostTensor* w2 = find_w(ctx, sc + "recover_fc/kernel");
      const HostTensor* b2 = find_w(ctx, sc + "recover_fc/bias");
      if (!shape_is(w1, {din, dh}) || !shape_is(b1, {dh}) || !shape_is(w2, {dh, dout}) || !shape_is(b2, {dout}))
        return fail(ctx, DAVO_ERR_WEIGHT, "missing or mis-shaped %s{bottleneck_fc,recover_fc}/{kernel,bias}", sc.c_str());
      se.insert(se.end(), w1->data.begin(), w1->data.end());
      se.insert(se.end(), b1->data.begin(), b1->data.end());
      se.insert(se.end(), w2->data.begin(), w2->data.end());
      se.insert(se.end(), b2->data.begin(), b2->data.end());
    }
    if (c.depth_split) {
      const HostTensor* th = find_w(ctx, P + "se_flow/depth_threshold");
      if (!th || th->data.size() != 1) return fail(ctx, DAVO_ERR_WEIGHT, "missing scalar variable %sse_flow/depth_threshold", P.c_str());
      ctx->depth_thres = th->data[0];
    }
    CU_OK(cudaMemcpy(ctx->d_sew, se.data(), se.size() * 4, cudaMemcpyHostToDevice));
  } else if (c.att_src == 2) {
    // reference posenn.py:380-394 -- variable is double-scoped by davo.py:1392 inside :1114
    const HostTensor* sw = find_w(ctx, P + "pose_exp_net/seg_channel_weight/weight");
    if (!shape_is(sw, {19}))
      return fail(ctx, DAVO_ERR_WEIGHT, "missing or mis-shaped %spose_exp_net/seg_channel_weight/weight", P.c_str());
    std::vector<float> s(19);
    for (int i = 0; i < 19; ++i) s[i] = 1.0f / (1.0f + expf(-sw->data[i]));
    CU_OK(cudaMemcpy(ctx->d_staticw, s.data(), 19 * 4, cudaMemcpyHostToDevice));
  }
  CU_OK(cudaDeviceSynchronize());
  ctx->weights_digest = weights_digest_of(ctx->weights);
  ctx->finalized = true;
  return 0;
}

extern "C" int davo_forward(davo_ctx* ctx, int B, const uint8_t* img, const float* flow,
                            const float* seg, const float* depth, float* pose_out, void* stream) {
  return davo_forward_pairs(ctx, B, DAVO_PAIRS_ALL, img, flow, seg, depth, pose_out, stream);
}

// The passes of a device-buffer forward of B samples, on either input layout.  `who` names the entry point in errors.
static int forward_device(davo_ctx* ctx, const char* who, int B, int pairs, const InputView& in, float* pose_out, void* stream) {
  CU_OK(cudaSetDevice(ctx->device));
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  if (ctx->cfg.batch_norm && !ctx->unit_sample && pairs != DAVO_PAIRS_ALL)
    return fail(ctx, DAVO_ERR_ARG, "%s: -batch_norm normalises with the statistics of a whole PoseNN call: every pair must be computed (DAVO_PAIRS_ALL)", who);
  if (ctx->unit_sample) pairs = kUnitsAreSamples;        // both poses come out of one evaluation
  int launches = 0;
  const int total = pairs_selected(pairs, B);
  if (ctx->cfg.batch_norm && total > ctx->mb)
    return fail(ctx, DAVO_ERR_ARG, "%s: -batch_norm needs the whole batch in one pass (%d units > micro_batch %d)", who, total, ctx->mb);
  int last_n = 0;
  if (pairs == DAVO_PAIRS_TRAJECTORY || pairs == DAVO_PAIRS_TRAJECTORY_FIRST)
    CU_OK(cudaMemsetAsync(pose_out, 0, (size_t)B * 12 * sizeof(float), st));
  for (int p0 = 0; p0 < total; p0 += ctx->mb) {
    const int n = (total - p0) < ctx->mb ? (total - p0) : ctx->mb;
    if (int rc = run_microbatch(ctx, pairs, p0, n, in, pose_out, st, &launches)) return rc;
    last_n = n;
  }
  ctx->last_launches = launches;
  ctx->last_npairs_mb = last_n;
  ctx->last_in = in; ctx->last_pose = pose_out; ctx->last_B = B;
  ctx->last_pairs = pairs;
  return 0;
}

extern "C" int davo_forward_pairs(davo_ctx* ctx, int B, int pairs, const uint8_t* img, const float* flow,
                                  const float* seg, const float* depth, float* pose_out, void* stream) {
  if (!ctx) return DAVO_ERR_ARG;
  if (pairs < DAVO_PAIRS_ALL || pairs > DAVO_PAIRS_TRAJECTORY_FIRST)
    return fail(ctx, DAVO_ERR_ARG, "davo_forward: pair selection %d unknown", pairs);
  if ((ctx->cfg.att_src == 5 || ctx->cfg.depth_split) && !depth) return fail(ctx, DAVO_ERR_ARG, "davo_forward: this variant reads input_depth; got NULL");
  if (!ctx->finalized) return fail(ctx, DAVO_ERR_STATE, "davo_forward: weights not finalized");
  if (B <= 0 || B > ctx->cfg.max_batch) return fail(ctx, DAVO_ERR_ARG, "davo_forward: B=%d outside 1..%d", B, ctx->cfg.max_batch);
  if (!img || !pose_out || (ctx->cfg.att_src != 0 && !seg) || ((ctx->cfg.in_mode == 1 || ctx->cfg.att_src == 1 || ctx->cfg.att_src == 6 || ctx->cfg.pixel_map == 2) && !flow))
    return fail(ctx, DAVO_ERR_ARG, "davo_forward: null input buffer");
  return forward_device(ctx, "davo_forward", B, pairs, triplet_view(ctx->cfg.H, ctx->cfg.W, img, flow, seg, nullptr, depth, nullptr, 0),
                        pose_out, stream);
}

namespace {

// What a sequence call of n frames reads (include/davo_b200.h: davo_forward_sequence).  Sample s computes the pair
// tgt -> src1 always and tgt -> src0 when k0(s); a frame is read as the target of sample f - 1, as src1 of f - 2 and as
// src0 of f.
struct SeqReads {
  bool flow = false, labels = false, tgt_labels = false, depth = false;
  int pairs = 0;                  // the selection as the passes run it (kUnitsAreSamples for the non-shared nets)
  bool k0(int s) const { return pairs == DAVO_PAIRS_ALL || pairs == kUnitsAreSamples || (pairs == DAVO_PAIRS_TRAJECTORY_FIRST && s == 0); }
  bool fwd(int s) const { return flow && k0(s); }                              // flow_fwd[s]
  bool img(int f, int n) const {                                               // image (and depth) of frame f
    return (f >= 1 && f - 1 < n - 2) || (f >= 2) || (f < n - 2 && k0(f));
  }
  bool lab(int f, int n) const {
    if (!labels) return false;
    return f >= 2 || (f < n - 2 && k0(f)) || (tgt_labels && f >= 1 && f - 1 < n - 2);
  }
};
SeqReads seq_reads(const davo_ctx* ctx, int pairs) {
  const davo_config& c = ctx->cfg;
  SeqReads r;
  r.pairs = ctx->unit_sample ? kUnitsAreSamples : pairs;
  r.flow = c.in_mode == 1 || c.att_src == 1 || c.att_src == 6 || c.pixel_map == 2;
  r.labels = c.att_src != 0 && (!c.pixel_map || c.att_src == 6);     // the per-pixel rgb / depth sources gather no class weight
  r.tgt_labels = r.labels && !c.att_tgt_ones;
  r.depth = c.att_src == 5 || c.depth_split;
  return r;
}

// Argument checks shared by the two sequence entry points.
int check_sequence(davo_ctx* ctx, const char* who, int n_frames, int pairs, const void* img, const void* flow_fwd,
                   const void* flow_bwd, const void* seg, const void* depth, const void* pose_out) {
  if (pairs < DAVO_PAIRS_ALL || pairs > DAVO_PAIRS_TRAJECTORY_FIRST) return fail(ctx, DAVO_ERR_ARG, "%s: pair selection %d unknown", who, pairs);
  if (!ctx->finalized) return fail(ctx, DAVO_ERR_STATE, "%s: weights not finalized", who);
  if (n_frames < 3) return fail(ctx, DAVO_ERR_ARG, "%s: n_frames=%d: a sample needs 3 frames", who, n_frames);
  if (n_frames - 2 > ctx->cfg.max_batch)
    return fail(ctx, DAVO_ERR_ARG, "%s: n_frames=%d is %d samples, more than max_batch %d", who, n_frames, n_frames - 2, ctx->cfg.max_batch);
  const SeqReads r = seq_reads(ctx, pairs);
  const davo_config& c = ctx->cfg;
  struct { const void* p; bool needed; const char* name; } in[] = {
      {img, true, "img"}, {pose_out, true, "pose_out"}, {seg, c.att_src != 0, "seg"}, {depth, r.depth, "depth"},
      {flow_bwd, r.flow, "flow_bwd"}, {flow_fwd, r.flow && r.k0(0), "flow_fwd"}};
  for (const auto& x : in) {
    if (x.needed && !x.p) return fail(ctx, DAVO_ERR_ARG, "%s: %s is NULL; this variant and pair selection read it", who, x.name);
    if (x.p && (reinterpret_cast<uintptr_t>(x.p) & 15)) return fail(ctx, DAVO_ERR_ARG, "%s: %s is not 16-byte aligned", who, x.name);
  }
  return 0;
}

}  // namespace

namespace {
// The view of a device-buffer sequence call.  Plane 1 of sample s is flow_bwd[s + 1]; a flow_fwd nobody reads stands in
// as flow_bwd, so that a front end re-run over every pair (davo_profile_layers) still reads mapped memory.
InputView sequence_device_view(const davo_ctx* ctx, const uint8_t* img, const float* flow_fwd, const float* flow_bwd,
                               const float* seg, const float* depth) {
  const davo_config& c = ctx->cfg;
  const size_t hw = (size_t)c.H * c.W;
  const float* bwd1 = flow_bwd ? flow_bwd + 2 * hw : nullptr;
  return sequence_view(c.H, c.W, img, flow_fwd ? flow_fwd : flow_bwd, bwd1, seg, nullptr, depth, nullptr, nullptr, 0);
}
}  // namespace

extern "C" int davo_forward_sequence(davo_ctx* ctx, int n_frames, int pairs, const uint8_t* img, const float* flow_fwd,
                                     const float* flow_bwd, const float* seg, const float* depth, float* pose_out, void* stream) {
  if (!ctx) return DAVO_ERR_ARG;
  if (int rc = check_sequence(ctx, "davo_forward_sequence", n_frames, pairs, img, flow_fwd, flow_bwd, seg, depth, pose_out)) return rc;
  return forward_device(ctx, "davo_forward_sequence", n_frames - 2, pairs,
                        sequence_device_view(ctx, img, flow_fwd, flow_bwd, seg, depth), pose_out, stream);
}

// Host-buffer entry point: the batch is cut into micro-batch chunks; chunk i+1 is copied
// host->device on a private copy stream while chunk i computes (two staging buffers), and only
// the planes the graph reads are copied: flow[:,0:2] (davo.py:978-982) and, when the target
// map is forced to ones, seg[:,0] and seg[:,2] (davo.py:1000-1004).
extern "C" int davo_forward_host(davo_ctx* ctx, int B, const uint8_t* img, const float* flow,
                                 const float* seg, const float* depth, float* pose_out, void* stream) {
  return davo_forward_host_pairs(ctx, B, DAVO_PAIRS_ALL, img, flow, seg, depth, pose_out, stream);
}

// flow16 / seg8 non-NULL: the caller already holds the compact forms (davo_forward_host_compact) -- the two flow
// planes the graph reads as binary16 [B][2][H][W][2], the labels as bytes [B][3][H][W] -- and they are copied
// straight from the caller's memory: no CPU pass at all.
static int forward_host_impl(davo_ctx* ctx, int B, int pairs, const uint8_t* img, const float* flow,
                             const float* seg, const float* depth, float* pose_out, void* stream,
                             const uint16_t* flow16, const uint8_t* seg8, long long* ticket = nullptr);

extern "C" int davo_forward_host_pairs(davo_ctx* ctx, int B, int pairs, const uint8_t* img, const float* flow,
                                       const float* seg, const float* depth, float* pose_out, void* stream) {
  return forward_host_impl(ctx, B, pairs, img, flow, seg, depth, pose_out, stream, nullptr, nullptr);
}

// Asynchronous forms (include/davo_b200.h): everything is queued, nothing is waited for; *ticket names the call.
extern "C" int davo_forward_host_pairs_async(davo_ctx* ctx, int B, int pairs, const uint8_t* img, const float* flow,
                                             const float* seg, const float* depth, float* pose_out, void* stream,
                                             long long* ticket) {
  if (!ticket) return fail(ctx, DAVO_ERR_ARG, "davo_forward_host_pairs_async: null ticket");
  return forward_host_impl(ctx, B, pairs, img, flow, seg, depth, pose_out, stream, nullptr, nullptr, ticket);
}

extern "C" int davo_host_wait(davo_ctx* ctx, long long ticket) {
  if (!ctx) return DAVO_ERR_ARG;
  if (ticket <= 0 || ticket > ctx->host_tickets) return fail(ctx, DAVO_ERR_ARG, "davo_host_wait: ticket %lld was never issued", ticket);
  CU_OK(cudaSetDevice(ctx->device));
  // the ring holds the last kTickets calls; an older ticket's slot now belongs to a later call on the same stream,
  // whose completion implies the older one's
  CU_OK(cudaEventSynchronize(ctx->ev_host_done[ticket % davo_ctx::kTickets]));
  return 0;
}

extern "C" int davo_forward_host_compact(davo_ctx* ctx, int B, int pairs, const uint8_t* img, const uint16_t* flow_f16,
                                         const uint8_t* seg_u8, const float* depth, float* pose_out, void* stream) {
  if (!ctx) return DAVO_ERR_ARG;
  const davo_config& c = ctx->cfg;
  const bool uses_flow = (c.in_mode == 1 || c.att_src == 1 || c.att_src == 6 || c.pixel_map == 2);
  if ((uses_flow && !flow_f16) || (c.att_src != 0 && !seg_u8))
    return fail(ctx, DAVO_ERR_ARG, "davo_forward_host_compact: null input buffer");
  // the float pointers only serve as "present" flags and are never dereferenced when the compact forms are given
  return forward_host_impl(ctx, B, pairs, img, reinterpret_cast<const float*>(flow_f16), reinterpret_cast<const float*>(seg_u8),
                           depth, pose_out, stream, uses_flow ? flow_f16 : nullptr, c.att_src != 0 ? seg_u8 : nullptr);
}

extern "C" int davo_forward_host_compact_async(davo_ctx* ctx, int B, int pairs, const uint8_t* img, const uint16_t* flow_f16,
                                               const uint8_t* seg_u8, const float* depth, float* pose_out, void* stream,
                                               long long* ticket) {
  if (!ctx) return DAVO_ERR_ARG;
  if (!ticket) return fail(ctx, DAVO_ERR_ARG, "davo_forward_host_compact_async: null ticket");
  const davo_config& c = ctx->cfg;
  const bool uses_flow = (c.in_mode == 1 || c.att_src == 1 || c.att_src == 6 || c.pixel_map == 2);
  if ((uses_flow && !flow_f16) || (c.att_src != 0 && !seg_u8))
    return fail(ctx, DAVO_ERR_ARG, "davo_forward_host_compact_async: null input buffer");
  return forward_host_impl(ctx, B, pairs, img, reinterpret_cast<const float*>(flow_f16), reinterpret_cast<const float*>(seg_u8),
                           depth, pose_out, stream, uses_flow ? flow_f16 : nullptr, c.att_src != 0 ? seg_u8 : nullptr, ticket);
}

namespace {

// Staging of the host entry points: kStage chunk slots of `cs` samples, pinned buffers for the CPU narrowing, the
// private copy stream.  Allocated by the first host call; returns the chunk size, or an error code (< 0).
int host_setup(davo_ctx* ctx, const char* who) {
  const davo_config& c = ctx->cfg;
  const size_t hw = (size_t)c.H * c.W;
  const size_t n_img = hw * 9, n_flow = hw * 8, n_seg = hw * 3;   // elements per sample
  const bool uses_flow = (c.in_mode == 1 || c.att_src == 1 || c.att_src == 6 || c.pixel_map == 2);
  // Host inputs arrive over PCIe more slowly than the stack computes, so what matters is how soon
  // compute can start behind the copy: chunks of 16 samples (8 chunks per 128-sample batch).
  const int ups = ctx->unit_sample ? 1 : 2;                        // units of a pass per sample
  int cs = std::max(1, std::min(ctx->mb / ups, 16));               // samples per chunk
  if (const char* e = getenv("DAVO_B200_HOST_CHUNK"))              // experiment knob
    cs = std::max(1, std::min(atoi(e), std::max(1, ctx->mb / ups)));
  if (ctx->s_img[0] && ctx->s_chunk != cs) return fail(ctx, DAVO_ERR_STATE, "%s: chunk size changed", who);
  if (ctx->s_img[0]) return cs;
  ctx->s_chunk = cs;
  // A slot also holds a sequence chunk: its cs + 2 frames, cs flow_fwd and cs flow_bwd entries take less room than cs
  // triplets (davo_forward_sequence_host).
  for (int i = 0; i < davo_ctx::kStage; ++i) {
    CU_OK(cudaMalloc((void**)&ctx->s_img[i], n_img * cs));
    CU_OK(cudaMalloc((void**)&ctx->s_flow[i], n_flow * 4 * cs));
    CU_OK(cudaMalloc((void**)&ctx->s_seg[i], n_seg * 4 * cs));
    CU_OK(cudaMemset(ctx->s_flow[i], 0, n_flow * 4 * cs));
    CU_OK(cudaMemset(ctx->s_seg[i], 0, n_seg * 4 * cs));
    if (c.att_src == 5 || c.depth_split) CU_OK(cudaMalloc((void**)&ctx->s_depth[i], n_seg * 4 * cs));
    if (c.att_src != 0) {
      CU_OK(cudaMalloc((void**)&ctx->s_seg8[i], n_seg * cs));
      if (ctx->host_seg8) CU_OK(cudaHostAlloc((void**)&ctx->h_seg8[i], n_seg * cs, cudaHostAllocDefault));
    }
    if (uses_flow) {
      CU_OK(cudaMalloc((void**)&ctx->s_flow16[i], n_flow / 2 * sizeof(uint16_t) * cs));
      if (ctx->host_flow16) CU_OK(cudaHostAlloc((void**)&ctx->h_flow16[i], n_flow / 2 * sizeof(uint16_t) * cs, cudaHostAllocDefault));
    }
    CU_OK(cudaEventCreateWithFlags(&ctx->ev_seg8[i], cudaEventDisableTiming));
    CU_OK(cudaEventCreateWithFlags(&ctx->ev_copied[i], cudaEventDisableTiming));
    CU_OK(cudaEventCreateWithFlags(&ctx->ev_consumed[i], cudaEventDisableTiming));
  }
  CU_OK(cudaMalloc((void**)&ctx->s_pose, (size_t)12 * 4 * c.max_batch));
  if ((ctx->host_seg8 && c.att_src != 0) || (ctx->host_flow16 && uses_flow)) {
    // conversion threads: the host's hardware threads shared among the ranks of the box (torchrun sets
    // LOCAL_WORLD_SIZE), at most 16: one thread streams ~9 GB/s and a chunk is ~30 MB of traffic
    int ranks_here = 1;
    if (const char* e = getenv("LOCAL_WORLD_SIZE")) ranks_here = std::max(1, atoi(e));
    int nthreads = std::max(2, std::min(16, (int)std::thread::hardware_concurrency() / ranks_here));
    if (const char* e = getenv("DAVO_B200_HOST_THREADS")) nthreads = std::max(1, std::min(atoi(e), 32));
    // Narrowing the flow only pays when this process has the host's cores and memory system to
    // itself: with 16 threads it is +10 % on one GPU; with the 4 threads per rank of an 8-GPU box
    // (32 host threads) it costs 35 % (profiles/r1_e2e_n8_flow_transport.log), and ranks that share
    // a host share its memory bandwidth too, which the conversion doubles.  So: a single rank with
    // >= 16 threads, unless an explicit fraction says otherwise.
    if ((nthreads < 16 || ranks_here > 1) && !getenv("DAVO_B200_HOST_FLOW16_FRAC")) ctx->flow16_frac = 0.0f;
    ctx->pool = new HostPool(nthreads - 1);
  }
  CU_OK(cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking));
  CU_OK(cudaEventCreateWithFlags(&ctx->ev_start, cudaEventDisableTiming));
  return cs;
}

// The copy stream must not run ahead of work already queued on the caller's stream.  (Staging buffers are protected
// by their own events, so consecutive calls may overlap: the copies of call k+1 run under the compute of call k.  Only
// the first use of the copy stream is ordered behind the caller's stream.)
int host_order_first_call(davo_ctx* ctx, cudaStream_t st) {
  if (ctx->host_calls++ == 0) {
    CU_OK(cudaEventRecord(ctx->ev_start, st));
    CU_OK(cudaStreamWaitEvent(ctx->copy_stream, ctx->ev_start, 0));
  }
  return 0;
}

// One piece of CPU narrowing: n float32 flow values -> binary16, or n float labels -> bytes.
struct NarrowJob { const float* src; void* dst; size_t n; bool flow; };

// Runs the jobs on the handle's thread pool (flow jobs first); returns false when some flow value has no finite half.
bool host_narrow(davo_ctx* ctx, const std::vector<NarrowJob>& jobs) {
  std::atomic<int> flow_bad{0};
  ctx->pool->run([&](int part, int parts) {
    // Work units are pieces of a plane: `sub` pieces per plane so that every thread gets a few
    // long contiguous streams (a label plane costs half a flow plane: 4 bytes read per pixel vs 8).
    const size_t sub = jobs.size() >= (size_t)4 * parts ? 1 : (size_t)parts;
    const size_t units = jobs.size() * sub;
    for (size_t u = part; u < units; u += parts) {
      const NarrowJob& jb = jobs[u / sub];
      const size_t piece = u % sub, n = jb.n;
      const size_t beg = (n * piece / sub) & ~(size_t)15, end = piece + 1 == sub ? n : ((n * (piece + 1) / sub) & ~(size_t)15);
      if (jb.flow) {
        if (!davo_host::flows_to_half(jb.src + beg, static_cast<uint16_t*>(jb.dst) + beg, end - beg))
          flow_bad.store(1, std::memory_order_relaxed);
      } else {
        davo_host::labels_to_bytes(jb.src + beg, static_cast<uint8_t*>(jb.dst) + beg, end - beg);
      }
    }
  });
  return flow_bad.load() == 0;
}

// The end of a host call whose copies back are queued on st: blocking, or the asynchronous form's ticket.
int host_done(davo_ctx* ctx, cudaStream_t st, long long* ticket) {
  if (ticket) {
    const long long t = ++ctx->host_tickets;
    cudaEvent_t& ev = ctx->ev_host_done[t % davo_ctx::kTickets];
    if (!ev) CU_OK(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
    CU_OK(cudaEventRecord(ev, st));
    *ticket = t;
  } else {
    CU_OK(cudaStreamSynchronize(st));
  }
  return 0;
}

// Poses of a host call back to the caller's memory; blocking, or the asynchronous form's ticket.
int host_finish(davo_ctx* ctx, int B, float* pose_out, cudaStream_t st, long long* ticket) {
  if (B > 0) CU_OK(cudaMemcpyAsync(pose_out, ctx->s_pose, (size_t)12 * 4 * B, cudaMemcpyDeviceToHost, st));
  if (int rc = host_done(ctx, st, ticket)) return rc;
  ctx->last_d2h = (long long)12 * 4 * B;
  return 0;
}

// The passes of one chunk: `chunk_pairs` over its `ns` samples, poses to s_pose from sample s0 on.
int host_run_chunk(davo_ctx* ctx, int chunk_pairs, int s0, int ns, const InputView& in, cudaStream_t st, int* launches,
                   int* last_n) {
  const int np_chunk = pairs_selected(chunk_pairs, ns);
  const bool copy_only = getenv("DAVO_B200_HOST_COPY_ONLY") != nullptr;   // measurement: the copies alone (bench.py e2e.copy_only)
  for (int q0 = 0; q0 < np_chunk && !copy_only; q0 += ctx->mb)
    if (int rc = run_microbatch(ctx, chunk_pairs, q0, std::min(ctx->mb, np_chunk - q0), in, ctx->s_pose + (size_t)12 * s0, st, launches))
      return rc;
  *last_n = np_chunk;
  return 0;
}

}  // namespace

static int forward_host_impl(davo_ctx* ctx, int B, int pairs, const uint8_t* img, const float* flow,
                             const float* seg, const float* depth, float* pose_out, void* stream,
                             const uint16_t* flow16_in, const uint8_t* seg8_in, long long* ticket) {
  if (!ctx) return DAVO_ERR_ARG;
  if (pairs < DAVO_PAIRS_ALL || pairs > DAVO_PAIRS_TRAJECTORY_FIRST)
    return fail(ctx, DAVO_ERR_ARG, "davo_forward_host: pair selection %d unknown", pairs);
  if ((ctx->cfg.att_src == 5 || ctx->cfg.depth_split) && !depth) return fail(ctx, DAVO_ERR_ARG, "davo_forward_host: this variant reads input_depth; got NULL");
  if (!ctx->finalized) return fail(ctx, DAVO_ERR_STATE, "davo_forward_host: weights not finalized");
  if (B <= 0 || B > ctx->cfg.max_batch) return fail(ctx, DAVO_ERR_ARG, "davo_forward_host: B=%d outside 1..%d", B, ctx->cfg.max_batch);
  if (ctx->cfg.batch_norm)
    return fail(ctx, DAVO_ERR_ARG, "davo_forward_host: -batch_norm needs the whole batch in one pass; the chunked host entry point does not take it (copy the batch to the device and call davo_forward)");
  const davo_config& c = ctx->cfg;
  if (!img || !pose_out || (c.att_src != 0 && !seg) || ((c.in_mode == 1 || c.att_src == 1 || c.att_src == 6 || c.pixel_map == 2) && !flow))
    return fail(ctx, DAVO_ERR_ARG, "davo_forward_host: null input buffer");
  CU_OK(cudaSetDevice(ctx->device));
  const size_t hw = (size_t)c.H * c.W;
  const size_t n_img = hw * 9, n_flow = hw * 8, n_seg = hw * 3;   // elements per sample
  const bool uses_flow = (c.in_mode == 1 || c.att_src == 1 || c.att_src == 6 || c.pixel_map == 2);
  const int cs = host_setup(ctx, "davo_forward_host");
  if (cs < 0) return cs;
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  cudaStream_t cp = ctx->copy_stream;
  if (int rc = host_order_first_call(ctx, st)) return rc;
  const bool need_flow = uses_flow;
  const bool need_seg = c.att_src != 0;
  const bool seg_tgt = need_seg && !c.att_tgt_ones;
  size_t h2d = 0;
  int launches = 0, last_n = 0, chunk = 0;
  if (ctx->unit_sample) pairs = kUnitsAreSamples;
  if (pairs == DAVO_PAIRS_TRAJECTORY || pairs == DAVO_PAIRS_TRAJECTORY_FIRST)
    CU_OK(cudaMemsetAsync(ctx->s_pose, 0, (size_t)B * 12 * sizeof(float), st));
  // With byte labels the copy of a chunk (0.36 ms per 16 samples) and its compute (0.43 ms per 32
  // pairs) are nearly balanced, so equal chunks are best: tapering the last ones (tried) only adds
  // passes that are too small to fill the GPU.
  int ns = 0, last_ns = 0;
  InputView in{};
  for (int s0 = 0; s0 < B; s0 += ns, ++chunk) {
    ns = std::min(cs, B - s0);
    last_ns = ns;
    const int buf = chunk % davo_ctx::kStage;
    CU_OK(cudaStreamWaitEvent(cp, ctx->ev_consumed[buf], 0));       // whoever read this staging slot last (this call or the one before) is done
    CU_OK(cudaMemcpyAsync(ctx->s_img[buf], img + n_img * s0, n_img * ns, cudaMemcpyHostToDevice, cp));
    h2d += n_img * ns;
    // Labels are small integers held in floats, and the flow is read with 11 significant bits
    // (frontend.cuh: flow_q): a few CPU threads convert the planes the graph reads to bytes /
    // binary16 in pinned staging while the DMA engine moves the previous chunk, and a quarter /
    // half of the bytes cross PCIe.  The pinned buffers are reused every kStage chunks: wait for
    // their copies first.
    // The CPU conversion streams ~64 GB/s on this class of host and would become the bottleneck if it
    // took every flow plane, while the copy engine has bandwidth to spare: the first n16 samples of a
    // chunk cross as binary16 and the rest as float32 (flow16_frac; both read through flow_q, so the
    // split does not change a bit of the result).
    const bool conv_seg = need_seg && ctx->host_seg8 && !seg8_in;
    int n16 = (need_flow && ctx->host_flow16 && !flow16_in) ? std::min(ns, (int)std::lround(ctx->flow16_frac * ns)) : 0;
    const bool conv_flow = n16 > 0;
    const int planes[3] = {0, 2, 1};
    const int npl = seg_tgt ? 3 : 2;
    bool flow_ok = true;
    if (conv_seg || conv_flow) {
      CU_OK(cudaEventSynchronize(ctx->ev_seg8[buf]));              // the pinned staging of this slot has been copied out (no-op before its first use)
      std::vector<NarrowJob> jobs;
      const size_t fl = hw * 2;                                    // floats per flow plane
      for (int j = 0; conv_flow && j < 2 * n16; ++j)
        jobs.push_back({flow + n_flow * s0 + (j / 2) * n_flow + (j % 2) * fl, ctx->h_flow16[buf] + j * fl, fl, true});
      for (int jl = 0; conv_seg && jl < ns * npl; ++jl) {
        const size_t off = ((size_t)(jl / npl) * 3 + planes[jl % npl]) * hw;
        jobs.push_back({seg + n_seg * s0 + off, ctx->h_seg8[buf] + off, hw, false});
      }
      flow_ok = host_narrow(ctx, jobs);
    }
    if (conv_flow && !flow_ok) n16 = 0;                            // a value with no finite half: the whole chunk as float32
    if (flow16_in && need_flow) n16 = ns;                         // the caller's binary16 planes, as they are
    if (n16 > 0) {
      CU_OK(cudaMemcpyAsync(ctx->s_flow16[buf], flow16_in ? flow16_in + hw * 4 * (size_t)s0 : ctx->h_flow16[buf],
                            hw * 4 * sizeof(uint16_t) * n16, cudaMemcpyHostToDevice, cp));
      h2d += hw * 4 * sizeof(uint16_t) * n16;
    }
    if (need_flow && n16 < ns) {
      CU_OK(cudaMemcpy2DAsync(ctx->s_flow[buf] + n_flow * n16, n_flow * 4, flow + n_flow * (s0 + n16), n_flow * 4, n_flow * 2,
                              ns - n16, cudaMemcpyHostToDevice, cp));
      h2d += n_flow * 2 * (ns - n16);
    }
    const uint8_t* seg8_dev = nullptr;
    if (conv_seg || (seg8_in && need_seg)) {
      const uint8_t* dst = seg8_in ? seg8_in + n_seg * (size_t)s0 : ctx->h_seg8[buf];
      if (seg_tgt) {
        CU_OK(cudaMemcpyAsync(ctx->s_seg8[buf], dst, n_seg * ns, cudaMemcpyHostToDevice, cp));
        h2d += n_seg * ns;
      } else {
        for (int pl = 0; pl < 3; pl += 2)
          CU_OK(cudaMemcpy2DAsync(ctx->s_seg8[buf] + hw * pl, n_seg, dst + hw * pl, n_seg, hw, ns, cudaMemcpyHostToDevice, cp));
        h2d += hw * 2 * ns;
      }
      seg8_dev = ctx->s_seg8[buf];
    } else if (need_seg) {
      if (seg_tgt) {
        CU_OK(cudaMemcpyAsync(ctx->s_seg[buf], seg + n_seg * s0, n_seg * 4 * ns, cudaMemcpyHostToDevice, cp));
        h2d += n_seg * 4 * ns;
      } else {
        for (int pl = 0; pl < 3; pl += 2)
          CU_OK(cudaMemcpy2DAsync(ctx->s_seg[buf] + hw * pl, n_seg * 4, seg + n_seg * s0 + hw * pl, n_seg * 4,
                                  hw * 4, ns, cudaMemcpyHostToDevice, cp));
        h2d += hw * 4 * 2 * ns;
      }
    }
    if (c.att_src == 5 || c.depth_split) {       // depth sources: all three planes (the frame's and the target's are read)
      CU_OK(cudaMemcpyAsync(ctx->s_depth[buf], depth + n_seg * s0, n_seg * 4 * ns, cudaMemcpyHostToDevice, cp));
      h2d += n_seg * 4 * ns;
    }
    if (conv_seg || conv_flow) CU_OK(cudaEventRecord(ctx->ev_seg8[buf], cp));   // pinned staging of this slot has been read
    CU_OK(cudaEventRecord(ctx->ev_copied[buf], cp));
    CU_OK(cudaStreamWaitEvent(st, ctx->ev_copied[buf], 0));
    in = triplet_view(c.H, c.W, ctx->s_img[buf], ctx->s_flow[buf], seg8_dev ? nullptr : ctx->s_seg[buf], seg8_dev,
                      ctx->s_depth[buf], n16 > 0 ? ctx->s_flow16[buf] : nullptr, n16);
    // a chunk is a batch of its own: only the first one may hold the first sample's tgt->src0
    const int chunk_pairs = (pairs == DAVO_PAIRS_TRAJECTORY_FIRST && s0 > 0) ? DAVO_PAIRS_TRAJECTORY : pairs;
    if (int rc = host_run_chunk(ctx, chunk_pairs, s0, ns, in, st, &launches, &last_n)) return rc;
    CU_OK(cudaEventRecord(ctx->ev_consumed[buf], st));
  }
  if (int rc = host_finish(ctx, B, pose_out, st, ticket)) return rc;
  ctx->last_launches = launches;
  ctx->last_npairs_mb = last_n;
  ctx->last_h2d = (long long)h2d;
  ctx->last_in = in;
  ctx->last_pose = ctx->s_pose; ctx->last_B = last_ns;
  ctx->last_pairs = (pairs == DAVO_PAIRS_TRAJECTORY_FIRST && chunk > 1) ? DAVO_PAIRS_TRAJECTORY : pairs;
  return 0;
}

// An online odometry session (include/davo_b200.h: davo_odometry_*).  A push of k frames computes the samples of a
// virtual sequence: the session's last `head` (<= 2) frames, then the k new ones.  Virtual frame v is global frame
// g0 + v, and every sample of that push is new.  The carried state lives in the session's own buffers; the frames of a
// push are staged in the handle's buffers (odometry_push_many_impl).
struct davo_odometry {
  davo_ctx* ctx = nullptr;
  int max_push = 0, pairs = DAVO_PAIRS_TRAJECTORY;
  bool host = true;
  long long pushed = 0, posed = 0;               // frames pushed; frames whose absolute pose has been written
  // carried state: the last two frames (labels as bytes in host sessions with byte labels, else as floats), the last
  // flow_fwd entry when a later sample reads it, the last absolute pose
  uint8_t* c_img = nullptr; uint8_t* c_seg8 = nullptr; float *c_seg = nullptr, *c_depth = nullptr, *c_fwd = nullptr;
  double* d_P = nullptr;
  Mat4 *d_rel = nullptr, *d_traj = nullptr;      // this push's relative motions; a host push's absolute poses
  int head() const { return (int)std::min<long long>(pushed, 2); }
};

namespace {

std::mutex g_odo_mutex;
std::set<davo_odometry*> g_odo_live;             // sessions not yet destroyed (a push on any other pointer is refused)

// ---- each posed frame's attention (include/davo_b200.h: davo_odometry_attention) ----
// Row r of a push's outputs is the frame of traj_out[r]: with sample 0 of the stream, frame 0 (src0 of sample 0) and
// frame 1 (its target), then frame s+2, src1 of sample s.  attention_out_kernel writes the rows through a unit table:
// the only code that knows how the staging of a push orders its units.

// Where view sample b's frames go: the row of its src1 frame, and whether it opens its stream (its src0 and target then
// take the two rows before), or row -1 when no frame of it has a row.
struct AttSample { int row; bool opens; };

// The unit table of a forward over `nsel` selection slots of pair mode `mode` (pair_of_slot; kUnitsAreSamples for the
// non-shared nets): unit -> (row of its target, src0, src1 frame or -1, view sample).  A pair unit tgt -> src1 places
// src1; the unit tgt -> src0 of a sample that opens its stream places src0 and the target, whose maps it masks; a
// sample unit places all three.
template <class F>
void att_unit_table(std::vector<int4>& out, int mode, int nsel, F sample_of) {
  for (int q = 0; q < nsel; ++q) {
    int b = 0, k = 0;
    pair_of_slot(mode, q, &b, &k);
    const AttSample a = sample_of(b);
    int4 e = make_int4(-1, -1, -1, b);
    if (a.row >= 0) {
      const bool sample_unit = mode == kUnitsAreSamples;
      if (sample_unit || k == 1) e.z = a.row;
      if (a.opens && (sample_unit || k == 0)) { e.y = a.row - 2; e.x = a.row - 1; }
    }
    out.push_back(e);
  }
}

// The unit table in use while a forward is launched; cleared on every way out.
struct AttScope {
  davo_ctx* ctx;
  AttScope(davo_ctx* c, const int4* units, const AttRow* rows) : ctx(c) { ctx->att_units = units; ctx->att_rows = rows; }
  ~AttScope() { ctx->att_units = nullptr; ctx->att_rows = nullptr; }
};

constexpr size_t kAttWeightFloats = 2 * kAttStride;      // a frame's weight rows

// Device staging of host sessions' maps and weights for `n_rows` rows: maps [n_rows][H][W], then weights
// [n_rows][2][kAttStride].  Grown on demand, after the work that may still write or read it.
int att_stage(davo_ctx* ctx, size_t n_rows, float** maps, float** weights) {
  const size_t hw = (size_t)ctx->cfg.H * ctx->cfg.W, need = n_rows * (hw + kAttWeightFloats);
  if (ctx->att_stage_cap < need) {
    if (ctx->att_stage) {
      CU_OK(cudaDeviceSynchronize());
      CU_OK(cudaFree(ctx->att_stage));
      ctx->att_stage = nullptr;
    }
    const size_t cap = std::max(need, 2 * ctx->att_stage_cap);
    ctx->att_stage_cap = 0;
    CU_OK(cudaMalloc((void**)&ctx->att_stage, cap * sizeof(float)));
    ctx->att_stage_cap = cap;
  }
  *maps = ctx->att_stage;
  *weights = ctx->att_stage + n_rows * hw;
  return 0;
}

// An input's name in a push's messages: `name[idx]` for entry idx of a batched push, `name` for a single push (-1)
struct EntryName {
  char s[48];
  EntryName(const char* name, int idx) {
    if (idx >= 0) snprintf(s, sizeof s, "%s[%d]", name, idx);
    else snprintf(s, sizeof s, "%s", name);
  }
};

// A session's attention entry where `n_rows` rows are due: map / weights each NULL (not written) or 16-byte aligned,
// not both NULL.
int att_check(davo_ctx* ctx, const char* who, const davo_odometry_attention& a, int n_rows, int idx) {
  const EntryName name("att", idx);
  if (n_rows > 0 && !a.map && !a.weights)
    return fail(ctx, DAVO_ERR_ARG, "%s: %s has neither map nor weights; %d row(s) are due", who, name.s, n_rows);
  if ((reinterpret_cast<uintptr_t>(a.map) | reinterpret_cast<uintptr_t>(a.weights)) & 15)
    return fail(ctx, DAVO_ERR_ARG, "%s: %s.%s is not 16-byte aligned", who, name.s,
                (reinterpret_cast<uintptr_t>(a.map) & 15) ? "map" : "weights");
  return 0;
}

// Row pointers of `n` rows from the start of a session's (or the staging's) map and weight buffers
void att_rows_of(std::vector<AttRow>& rows, float* map, float* weights, int n, size_t hw) {
  for (int r = 0; r < n; ++r)
    rows.push_back({map ? map + hw * r : nullptr, weights ? weights + kAttWeightFloats * r : nullptr});
}

}  // namespace

// Host-buffer sequence entry point (include/davo_b200.h: davo_forward_sequence_host).  The samples are cut into the
// chunks of the triplet entry point.  Flow entries belong to one sample each and go through the chunk slots like the
// triplet flow planes.  Frames (images, labels, depth) are shared by up to three samples, so they are staged at their
// final place in one of two per-call frame sets: a chunk copies the frames that the call reads and that no earlier
// chunk copied, and the chunk's passes read the set through a sequence view.  Every copied frame or flow crosses PCIe
// once; those that no computed pair reads are not copied.
static int forward_sequence_host_impl(davo_ctx* ctx, int n_frames, int pairs, const uint8_t* img, const float* flow_fwd,
                                      const float* flow_bwd, const float* seg, const float* depth, float* pose_out,
                                      void* stream, long long* ticket) {
  const char* who = ticket ? "davo_forward_sequence_host_async" : "davo_forward_sequence_host";
  if (int rc = check_sequence(ctx, who, n_frames, pairs, img, flow_fwd, flow_bwd, seg, depth, pose_out)) return rc;
  if (ctx->cfg.batch_norm)
    return fail(ctx, DAVO_ERR_ARG, "%s: -batch_norm needs the whole batch in one pass; the chunked host entry point does not take it (copy the frames to the device and call davo_forward_sequence)", who);
  const davo_config& c = ctx->cfg;
  CU_OK(cudaSetDevice(ctx->device));
  const SeqReads r = seq_reads(ctx, pairs);
  pairs = r.pairs;
  const int B = n_frames - 2;
  const size_t hw = (size_t)c.H * c.W, fl = hw * 2;               // pixels per frame, floats per flow entry
  const int cs = host_setup(ctx, who);
  if (cs < 0) return cs;
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  cudaStream_t cp = ctx->copy_stream;
  if (int rc = host_order_first_call(ctx, st)) return rc;
  const bool seg8 = r.labels && ctx->host_seg8;
  const int set = (int)(ctx->q_calls++ & 1);
  if (!ctx->q_img[set]) {
    const size_t nf = (size_t)c.max_batch + 2;
    CU_OK(cudaMalloc((void**)&ctx->q_img[set], nf * hw * 3));
    if (c.att_src != 0 && ctx->host_seg8) CU_OK(cudaMalloc((void**)&ctx->q_seg8[set], nf * hw));
    if (c.att_src != 0 && !ctx->host_seg8) CU_OK(cudaMalloc((void**)&ctx->q_seg[set], nf * hw * 4));
    if (r.depth) CU_OK(cudaMalloc((void**)&ctx->q_depth[set], nf * hw * 4));
    CU_OK(cudaEventCreateWithFlags(&ctx->ev_q_done[set], cudaEventDisableTiming));
  } else {
    CU_OK(cudaStreamWaitEvent(cp, ctx->ev_q_done[set], 0));         // the call before the previous one has read this set
  }
  size_t h2d = 0;
  int launches = 0, last_n = 0, chunk = 0, ns = 0, last_ns = 0;
  int staged = 0;                                                  // frames [0, staged) are on the device (or never read)
  if (pairs == DAVO_PAIRS_TRAJECTORY || pairs == DAVO_PAIRS_TRAJECTORY_FIRST)
    CU_OK(cudaMemsetAsync(ctx->s_pose, 0, (size_t)B * 12 * sizeof(float), st));
  // copies runs of consecutive frames in [f0, f1) that `read` selects: copy(first frame, frame count)
  auto runs = [](int f0, int f1, auto read, auto copy) -> int {
    for (int f = f0; f < f1;) {
      if (!read(f)) { ++f; continue; }
      int e = f;
      while (e < f1 && read(e)) ++e;
      if (int rc = copy(f, e - f)) return rc;
      f = e;
    }
    return 0;
  };
  InputView in{};
  for (int s0 = 0; s0 < B; s0 += ns, ++chunk) {
    ns = std::min(cs, B - s0);
    last_ns = ns;
    const int buf = chunk % davo_ctx::kStage;
    const int f0 = staged, f1 = s0 + ns + 2;                       // frames this chunk stages
    CU_OK(cudaStreamWaitEvent(cp, ctx->ev_consumed[buf], 0));       // whoever read this staging slot last is done
    auto img_rd = [&](int f) { return r.img(f, n_frames); };
    auto lab_rd = [&](int f) { return r.lab(f, n_frames); };
    auto dep_rd = [&](int f) { return r.depth && r.img(f, n_frames); };
    if (int rc = runs(f0, f1, img_rd, [&](int f, int n) -> int {
          CU_OK(cudaMemcpyAsync(ctx->q_img[set] + hw * 3 * f, img + hw * 3 * f, hw * 3 * n, cudaMemcpyHostToDevice, cp));
          h2d += hw * 3 * n;
          return 0;
        })) return rc;
    if (int rc = runs(f0, f1, dep_rd, [&](int f, int n) -> int {
          CU_OK(cudaMemcpyAsync(ctx->q_depth[set] + hw * f, depth + hw * f, hw * 4 * n, cudaMemcpyHostToDevice, cp));
          h2d += hw * 4 * n;
          return 0;
        })) return rc;
    // flow entries of the chunk: flow_fwd[s0 + i] at slot entry i, flow_bwd[s0 + 1 + i] at slot entry cs + i
    const int nfwd = r.fwd(s0) ? (r.k0(s0 + ns - 1) ? ns : 1) : 0;    // fwd entries read: all, the first one (FIRST), none
    const bool need_bwd = r.flow;
    int n16 = (r.flow && ctx->host_flow16) ? std::min(ns, (int)std::lround(ctx->flow16_frac * ns)) : 0;
    const bool conv_flow = n16 > 0;
    bool flow_ok = true;
    if (seg8 || conv_flow) {
      CU_OK(cudaEventSynchronize(ctx->ev_seg8[buf]));              // the pinned staging of this slot has been copied out
      std::vector<NarrowJob> jobs;
      uint16_t* h16 = ctx->h_flow16[buf];
      for (int i = 0; conv_flow && i < n16; ++i) {
        if (i < nfwd) jobs.push_back({flow_fwd + fl * (s0 + i), h16 + fl * i, fl, true});
        jobs.push_back({flow_bwd + fl * (s0 + 1 + i), h16 + fl * (cs + i), fl, true});
      }
      for (int f = f0; seg8 && f < f1; ++f)                         // pinned label staging: frame f at f - f0
        if (lab_rd(f)) jobs.push_back({seg + hw * f, ctx->h_seg8[buf] + hw * (f - f0), hw, false});
      flow_ok = host_narrow(ctx, jobs);
    }
    if (conv_flow && !flow_ok) n16 = 0;                            // a value with no finite half: the whole chunk as float32
    const int n16_fwd = std::min(n16, nfwd);
    if (n16 > 0) {
      uint16_t* d16 = ctx->s_flow16[buf];
      const uint16_t* h16 = ctx->h_flow16[buf];
      if (n16_fwd > 0) CU_OK(cudaMemcpyAsync(d16, h16, fl * 2 * n16_fwd, cudaMemcpyHostToDevice, cp));
      CU_OK(cudaMemcpyAsync(d16 + fl * cs, h16 + fl * cs, fl * 2 * n16, cudaMemcpyHostToDevice, cp));
      h2d += fl * 2 * (n16_fwd + n16);
    }
    float* dflow = ctx->s_flow[buf];
    if (nfwd > n16_fwd) {
      CU_OK(cudaMemcpyAsync(dflow + fl * n16_fwd, flow_fwd + fl * (s0 + n16_fwd), fl * 4 * (nfwd - n16_fwd), cudaMemcpyHostToDevice, cp));
      h2d += fl * 4 * (nfwd - n16_fwd);
    }
    if (need_bwd && ns > n16) {
      CU_OK(cudaMemcpyAsync(dflow + fl * (cs + n16), flow_bwd + fl * (s0 + 1 + n16), fl * 4 * (ns - n16), cudaMemcpyHostToDevice, cp));
      h2d += fl * 4 * (ns - n16);
    }
    if (seg8) {
      if (int rc = runs(f0, f1, lab_rd, [&](int f, int n) -> int {
            CU_OK(cudaMemcpyAsync(ctx->q_seg8[set] + hw * f, ctx->h_seg8[buf] + hw * (f - f0), hw * n, cudaMemcpyHostToDevice, cp));
            h2d += hw * n;
            return 0;
          })) return rc;
    } else if (r.labels) {
      if (int rc = runs(f0, f1, lab_rd, [&](int f, int n) -> int {
            CU_OK(cudaMemcpyAsync(ctx->q_seg[set] + hw * f, seg + hw * f, hw * 4 * n, cudaMemcpyHostToDevice, cp));
            h2d += hw * 4 * n;
            return 0;
          })) return rc;
    }
    staged = f1;
    if (seg8 || conv_flow) CU_OK(cudaEventRecord(ctx->ev_seg8[buf], cp));   // pinned staging of this slot has been read
    CU_OK(cudaEventRecord(ctx->ev_copied[buf], cp));
    CU_OK(cudaStreamWaitEvent(st, ctx->ev_copied[buf], 0));
    // the chunk's view: sample 0 is sequence sample s0; a flow_fwd the chunk does not read stands in as its flow_bwd
    // (davo_profile_layers re-runs every pair of the last chunk)
    in = sequence_view(c.H, c.W, ctx->q_img[set] + hw * 3 * s0, nfwd ? dflow : dflow + fl * cs, dflow + fl * cs,
                       seg8 ? nullptr : (ctx->q_seg[set] ? ctx->q_seg[set] + hw * s0 : nullptr),
                       seg8 ? ctx->q_seg8[set] + hw * s0 : nullptr, ctx->q_depth[set] ? ctx->q_depth[set] + hw * s0 : nullptr,
                       n16 > 0 ? (n16_fwd > 0 ? ctx->s_flow16[buf] : ctx->s_flow16[buf] + fl * cs) : nullptr,
                       n16 > 0 ? ctx->s_flow16[buf] + fl * cs : nullptr, n16);
    const int chunk_pairs = (pairs == DAVO_PAIRS_TRAJECTORY_FIRST && s0 > 0) ? DAVO_PAIRS_TRAJECTORY : pairs;
    if (int rc = host_run_chunk(ctx, chunk_pairs, s0, ns, in, st, &launches, &last_n)) return rc;
    CU_OK(cudaEventRecord(ctx->ev_consumed[buf], st));
  }
  CU_OK(cudaEventRecord(ctx->ev_q_done[set], st));
  if (int rc = host_finish(ctx, B, pose_out, st, ticket)) return rc;
  ctx->last_launches = launches;
  ctx->last_npairs_mb = last_n;
  ctx->last_h2d = (long long)h2d;
  ctx->last_in = in;
  ctx->last_pose = ctx->s_pose; ctx->last_B = last_ns;
  ctx->last_pairs = (pairs == DAVO_PAIRS_TRAJECTORY_FIRST && chunk > 1) ? DAVO_PAIRS_TRAJECTORY : pairs;
  return 0;
}

extern "C" int davo_forward_sequence_host(davo_ctx* ctx, int n_frames, int pairs, const uint8_t* img, const float* flow_fwd,
                                          const float* flow_bwd, const float* seg, const float* depth, float* pose_out,
                                          void* stream, long long* ticket) {
  if (!ctx) return DAVO_ERR_ARG;
  return forward_sequence_host_impl(ctx, n_frames, pairs, img, flow_fwd, flow_bwd, seg, depth, pose_out, stream, ticket);
}

// ---- online odometry sessions (include/davo_b200.h: davo_odometry_*) ----
static void odometry_free(davo_odometry* o) {
  cudaSetDevice(o->ctx->device);
  cudaFree(o->c_img); cudaFree(o->c_seg8); cudaFree(o->c_seg); cudaFree(o->c_depth); cudaFree(o->c_fwd);
  cudaFree(o->d_P); cudaFree(o->d_rel); cudaFree(o->d_traj);
  delete o;
}

// A session's buffers on its handle's device (o->ctx): the carried state, the relative motions, a host session's
// absolute poses.
static int odometry_alloc(davo_odometry* o) {
  davo_ctx* ctx = o->ctx;
  CU_OK(cudaSetDevice(ctx->device));
  const davo_config& c = ctx->cfg;
  const SeqReads r = seq_reads(ctx, o->pairs);
  const size_t hw = (size_t)c.H * c.W;
  const bool seg8 = o->host && ctx->host_seg8;                     // the form the session carries its labels in
  auto alloc = [&](void** p, size_t bytes) -> int {
    CU_OK(cudaMalloc(p, bytes));
    return 0;
  };
  int rc = alloc((void**)&o->c_img, hw * 3 * 2);
  if (!rc && c.att_src != 0) rc = seg8 ? alloc((void**)&o->c_seg8, hw * 2) : alloc((void**)&o->c_seg, hw * 4 * 2);
  if (!rc && r.depth) rc = alloc((void**)&o->c_depth, hw * 4 * 2);
  if (!rc && r.flow) rc = alloc((void**)&o->c_fwd, hw * 2 * 4);
  if (!rc) rc = alloc((void**)&o->d_P, 16 * sizeof(double));
  if (!rc) rc = alloc((void**)&o->d_rel, (size_t)(o->max_push + 1) * sizeof(Mat4));
  if (!rc && o->host) rc = alloc((void**)&o->d_traj, (size_t)(o->max_push + 2) * sizeof(Mat4));
  return rc;
}

extern "C" int davo_odometry_create(davo_ctx* ctx, int max_push, int pairs, int host_inputs, davo_odometry** out) {
  if (!ctx) return DAVO_ERR_ARG;
  const char* who = "davo_odometry_create";
  if (!out) return fail(ctx, DAVO_ERR_ARG, "%s: out is NULL", who);
  *out = nullptr;
  if (!ctx->finalized) return fail(ctx, DAVO_ERR_STATE, "%s: weights not finalized", who);
  if (ctx->cfg.batch_norm)
    return fail(ctx, DAVO_ERR_ARG, "%s: -batch_norm normalises with the statistics of the samples that share a call, so its poses depend on how the stream is cut into pushes; a session does not take it", who);
  if (pairs != DAVO_PAIRS_TRAJECTORY && pairs != DAVO_PAIRS_ALL)
    return fail(ctx, DAVO_ERR_ARG, "%s: pairs %d: a session takes DAVO_PAIRS_TRAJECTORY or DAVO_PAIRS_ALL", who, pairs);
  if (max_push < 1 || max_push > ctx->cfg.max_batch)
    return fail(ctx, DAVO_ERR_ARG, "%s: max_push=%d outside 1..max_batch %d", who, max_push, ctx->cfg.max_batch);
  davo_odometry* o = new davo_odometry;
  o->ctx = ctx; o->max_push = max_push; o->pairs = pairs; o->host = host_inputs != 0;
  if (int rc = odometry_alloc(o)) { odometry_free(o); return rc; }
  {
    std::lock_guard<std::mutex> lk(g_odo_mutex);
    g_odo_live.insert(o);
  }
  *out = o;
  return 0;
}

namespace {

// Host sessions' pushes: each session's new frames, label planes, depth planes and flow entries that some computed pair
// of its stream reads, now or in a later push, copied on the copy stream into one of the two arrivals sets.  Session
// i's part of the set holds its caller frame u and caller flow entry u at index u, so that the stage and carry kernels
// read it as they read a device session's buffers; ds[i]'s caller pointers are replaced by pointers into the set.
// Labels are narrowed to bytes on the CPU for all sessions in one pool pass into the set's pinned area (float labels
// with DAVO_B200_HOST_SEG8=0); the label planes of consecutive sessions sit back to back there and on the device, so
// one copy sends them all, except where a plane no pair reads (global frame 1 in trajectory mode when the target's
// labels are not read) breaks the run.  With the binary16 transport (host_flow16), the first flow16_frac of the flow
// entries the call sends (rounded up) are narrowed in the same pass, cross PCIe as binary16 in one copy with their
// destination table, and odo_widen_kernel writes them into the set's float32 flow areas; a call with a value that has
// no finite binary16 sends those entries as float32.  The front end reads the flow through flow_q, which rounds it to
// binary16 when flow_f16 = 1, so either way the bits are the same.
int many_host_arrivals(davo_ctx* ctx, int n, davo_odometry* const* sessions, OdoManySession* ds,
                       cudaStream_t st, int set, size_t* h2d_out) {
  const davo_config& c = ctx->cfg;
  const SeqReads rv = seq_reads(ctx, DAVO_PAIRS_ALL);
  const size_t hw = (size_t)c.H * c.W, fl = hw * 2;
  const bool seg8 = rv.labels && ctx->host_seg8;
  cudaStream_t cp = ctx->copy_stream;
  // flow_fwd entry u is read as plane 0 of sample u + fe when that sample computes both pairs, or carried; flow_bwd
  // entry u as plane 1 of sample u + fe - 1, for every sample
  auto fwd_rd = [](const OdoManySession& d, int u) { return u + d.fe < d.na || u == d.carry_fwd; };
  // the set's regions: session i's k[i] frames (or flow entries) at its running offset in each; ne flow entries sent
  size_t kt = 0, ne = 0;
  for (int i = 0; i < n; ++i) {
    kt += (size_t)ds[i].k;
    for (int u = 0; rv.flow && u < ds[i].k; ++u) ne += fwd_rd(ds[i], u);
    if (rv.flow) ne += (size_t)ds[i].ns;
  }
  // the first ceil(flow16_frac * ne) of them go as binary16
  const size_t n16 = rv.flow && ctx->host_flow16 ? std::min(ne, (size_t)std::ceil(ctx->flow16_frac * ne)) : 0;
  auto up = [](size_t b) { return (b + 255) & ~(size_t)255; };
  const size_t b_img = up(kt * hw * 3), b_lab = seg8 ? up(kt * hw) : 0, b_seg = rv.labels && !seg8 ? up(kt * hw * 4) : 0;
  const size_t b_dep = rv.depth ? up(kt * hw * 4) : 0, b_fl = rv.flow ? up(kt * fl * 4) : 0;
  const size_t b_16 = n16 * (fl * 2 + sizeof(int));                 // binary16 entries, then their destinations
  const size_t total = b_img + b_lab + b_seg + b_dep + 2 * b_fl + b_16, pinned = b_lab + b_16;
  cudaEvent_t& done = ctx->a_done[set];
  if (!done) {
    CU_OK(cudaEventCreateWithFlags(&done, cudaEventDisableTiming));
    CU_OK(cudaEventCreateWithFlags(&ctx->a_copied[set], cudaEventDisableTiming));
  }
  if (ctx->a_dev_cap[set] < total || ctx->a_pin_cap[set] < pinned) {
    CU_OK(cudaEventSynchronize(done));                             // the call that last used the set has read it
    if (ctx->a_dev_cap[set] < total) {
      const size_t cap = std::max(total, 2 * ctx->a_dev_cap[set]);
      if (ctx->a_dev[set]) { CU_OK(cudaFree(ctx->a_dev[set])); ctx->a_dev[set] = nullptr; }
      ctx->a_dev_cap[set] = 0;
      CU_OK(cudaMalloc((void**)&ctx->a_dev[set], cap));
      ctx->a_dev_cap[set] = cap;
    }
    if (ctx->a_pin_cap[set] < pinned) {
      const size_t cap = std::max(pinned, 2 * ctx->a_pin_cap[set]);
      if (ctx->a_pin[set]) { CU_OK(cudaFreeHost(ctx->a_pin[set])); ctx->a_pin[set] = nullptr; }
      ctx->a_pin_cap[set] = 0;
      CU_OK(cudaHostAlloc((void**)&ctx->a_pin[set], cap, cudaHostAllocDefault));
      ctx->a_pin_cap[set] = cap;
    }
  }
  uint8_t* a_img = ctx->a_dev[set];
  uint8_t* a_lab = a_img + b_img;
  float* a_seg = reinterpret_cast<float*>(a_lab + b_lab);
  float* a_dep = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(a_seg) + b_seg);
  float* a_fwd = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(a_dep) + b_dep);
  float* a_bwd = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(a_fwd) + b_fl);
  uint8_t* a_16 = reinterpret_cast<uint8_t*>(a_bwd) + b_fl;
  uint16_t* h16 = reinterpret_cast<uint16_t*>(ctx->a_pin[set] + b_lab);
  int* h16_dst = reinterpret_cast<int*>(h16 + n16 * fl);              // entry j's destination: fwd entry e < kt, else bwd e - kt
  CU_OK(cudaStreamWaitEvent(cp, done, 0));                         // the device part of the set is free
  size_t h2d = 0;
  auto h2d_copy = [&](void* dst, const void* src, size_t bytes) -> int {
    CU_OK(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, cp));
    h2d += bytes;
    return 0;
  };
  // copies runs of consecutive indices in [0, m) that `read` selects: copy(first index, count)
  auto runs = [](int m, auto read, auto copy) -> int {
    for (int u = 0; u < m;) {
      if (!read(u)) { ++u; continue; }
      int e = u;
      while (e < m && read(e)) ++e;
      if (int rc = copy(u, e - u)) return rc;
      u = e;
    }
    return 0;
  };
  std::vector<NarrowJob> jobs;
  std::vector<std::pair<size_t, size_t>> lab_runs;                  // byte label planes read: [begin, end) in the area
  std::vector<std::pair<int, const float*>> e16;                    // the entries narrowed: destination, source
  auto flow_at = [&](size_t e) { return e < kt ? a_fwd + e * fl : a_bwd + (e - kt) * fl; };
  // m flow entries from src to the set's entries e on (fwd e < kt, else bwd e - kt): the call's first n16 as binary16
  auto send_flow = [&](size_t e, const float* src, int m) -> int {
    for (; m > 0 && e16.size() < n16; --m, ++e, src += fl) {
      jobs.push_back({src, h16 + e16.size() * fl, fl, true});
      e16.push_back({(int)e, src});
    }
    return m > 0 ? h2d_copy(flow_at(e), src, fl * 4 * m) : 0;
  };
  size_t off = 0;
  for (int i = 0; i < n; off += (size_t)ds[i].k, ++i) {
    OdoManySession& d = ds[i];
    const davo_odometry* o = sessions[i];
    const int head = d.head, k = d.k;
    const long long g0 = o->pushed - head;
    const SeqReads rg = seq_reads(ctx, o->pairs == DAVO_PAIRS_ALL ? DAVO_PAIRS_ALL : DAVO_PAIRS_TRAJECTORY_FIRST);
    auto glob = [&](int u) { return (int)std::min<long long>(g0 + head + u, 2); };   // caller frame u: virtual head + u
    auto img_rd = [&](int u) { return rg.img(glob(u), INT_MAX); };
    auto lab_rd = [&](int u) { return rg.lab(glob(u), INT_MAX); };
    const uint8_t* img = d.img;
    const float *seg = d.seg, *depth = d.depth, *fwd = d.fwd, *bwd = d.bwd;
    uint8_t* ai = a_img + off * hw * 3;
    d.img = ai;
    if (int rc = runs(k, img_rd, [&](int u, int m) { return h2d_copy(ai + u * hw * 3, img + u * hw * 3, hw * 3 * m); }))
      return rc;
    if (rv.depth) {
      float* ad = a_dep + off * hw;
      d.depth = ad;
      if (int rc = runs(k, img_rd, [&](int u, int m) { return h2d_copy(ad + u * hw, depth + u * hw, hw * 4 * m); })) return rc;
    }
    d.seg = nullptr;
    d.c_seg = nullptr;
    if (seg8) {
      d.seg8 = a_lab + off * hw;
      d.c_seg8 = o->c_seg8;
      for (int u = 0; u < k; ++u) {
        if (!lab_rd(u)) continue;
        const size_t b = (off + u) * hw;
        jobs.push_back({seg + u * hw, ctx->a_pin[set] + b, hw, false});
        if (!lab_runs.empty() && lab_runs.back().second == b) lab_runs.back().second = b + hw;
        else lab_runs.push_back({b, b + hw});
      }
    } else if (rv.labels) {
      float* as = a_seg + off * hw;
      d.seg = as;
      d.c_seg = o->c_seg;
      if (int rc = runs(k, lab_rd, [&](int u, int m) { return h2d_copy(as + u * hw, seg + u * hw, hw * 4 * m); })) return rc;
    }
    if (rv.flow) {
      d.fwd = a_fwd + off * fl;
      d.bwd = a_bwd + off * fl;
      if (int rc = runs(k, [&](int u) { return fwd_rd(d, u); },
                        [&](int u, int m) { return send_flow(off + u, fwd + u * fl, m); })) return rc;
      if (d.ns > 0)
        if (int rc = send_flow(kt + off + 1 - d.fe, bwd + (1 - d.fe) * fl, d.ns)) return rc;
    }
  }
  if (!jobs.empty()) {
    CU_OK(cudaEventSynchronize(done));                             // the pinned area has been copied out by that call
    const bool flow_ok = host_narrow(ctx, jobs);
    for (const auto& r : lab_runs)
      if (int rc = h2d_copy(a_lab + r.first, ctx->a_pin[set] + r.first, r.second - r.first)) return rc;
    if (!e16.empty() && flow_ok) {
      for (size_t j = 0; j < e16.size(); ++j) h16_dst[j] = e16[j].first;
      CU_OK(cudaMemcpyAsync(a_16, h16, b_16, cudaMemcpyHostToDevice, cp));
      h2d += n16 * fl * 2;                                         // the flow's bytes (descriptors are not counted)
      const int ny = (int)std::min<size_t>(n16, 65535);
      odo_widen_kernel<<<dim3(std::max(1, 4 * 148 / ny), ny), 256, 0, cp>>>(
          reinterpret_cast<const uint16_t*>(a_16), reinterpret_cast<const int*>(a_16 + n16 * fl * 2), (int)n16,
          a_fwd, a_bwd, (long long)kt, (long long)fl);
      CU_OK(cudaGetLastError());
    } else {
      for (const auto& x : e16)                                    // a value with no finite binary16: as float32
        if (int rc = h2d_copy(flow_at(x.first), x.second, fl * 4)) return rc;
    }
  }
  CU_OK(cudaEventRecord(ctx->a_copied[set], cp));
  CU_OK(cudaStreamWaitEvent(st, ctx->a_copied[set], 0));
  *h2d_out = h2d;
  return 0;
}

}  // namespace

// A push (include/davo_b200.h: davo_odometry_push, davo_odometry_push_many, davo_odometry_push_many_host): entry i is
// the push of sessions[i], k[i] new frames, and all of them share one forward; a single push is the call with n = 1.
// The samples are staged as stacked triplets, those that compute both pairs (all-mode sessions, sample 0 of a
// trajectory session that opens its sequence, every sample of the non-shared nets) first, so that the forward is one
// DAVO_PAIRS_TRAJECTORY_FIRST call when only the first sample computes both pairs, else at most one DAVO_PAIRS_ALL and
// one DAVO_PAIRS_TRAJECTORY call.  A pair's result does not depend on which pairs share its pass, so every pose is
// the bits of the session's push alone; the trajectory is chained by one code for every push (traj_chain).  Launches:
// stage, carry, the forward's, compose -- none per session.  Host sessions (`host`) first copy what the call reads
// into an arrivals set (many_host_arrivals); their pose rows and absolute poses go back to the caller's host buffers
// at the end.  `single`: the messages name the inputs of davo_odometry_push, without an index.
static int odometry_push_many_impl(bool host, int n, davo_odometry* const* sessions, const int* k, const uint8_t* const* img,
                                   const float* const* flow_fwd, const float* const* flow_bwd,
                                   const float* const* seg, const float* const* depth, float* const* pose_out,
                                   double* const* traj_out, const davo_odometry_attention* att, int* n_samples,
                                   int* n_traj, void* stream, long long* ticket, const char* who, bool single = false) {
  if (n < 1) return fail(nullptr, DAVO_ERR_ARG, "%s: n=%d: at least one session", who, n);
  if (!sessions) return fail(nullptr, DAVO_ERR_ARG, "%s: sessions is NULL", who);
  {
    std::lock_guard<std::mutex> lk(g_odo_mutex);
    for (int i = 0; i < n; ++i)
      if (!sessions[i] || !g_odo_live.count(sessions[i]))
        return fail(nullptr, DAVO_ERR_ARG, "%s: %s is NULL or was destroyed", who,
                    single ? "the session" : EntryName("sessions", i).s);
  }
  davo_ctx* ctx = sessions[0]->ctx;
  const davo_config& c = ctx->cfg;
  if (n > 65535) return fail(ctx, DAVO_ERR_ARG, "%s: n=%d sessions, more than 65535", who, n);
  if (!k) return fail(ctx, DAVO_ERR_ARG, "%s: k is NULL", who);
  if (!img) return fail(ctx, DAVO_ERR_ARG, "%s: img is NULL", who);
  std::set<const davo_odometry*> seen;
  for (int i = 0; i < n; ++i) {
    const davo_odometry* o = sessions[i];
    if (!seen.insert(o).second) return fail(ctx, DAVO_ERR_ARG, "%s: sessions[%d] is given twice", who, i);
    if (o->ctx != ctx) return fail(ctx, DAVO_ERR_ARG, "%s: sessions[%d] belongs to another handle than sessions[0]", who, i);
    if (o->host && !host) return fail(ctx, DAVO_ERR_ARG, "%s: sessions[%d] is a host session; a batched push takes device sessions", who, i);
    if (!o->host && host)
      return fail(ctx, DAVO_ERR_ARG, "%s: sessions[%d] is a device session; davo_odometry_push_many takes it", who, i);
  }
  const SeqReads rv = seq_reads(ctx, DAVO_PAIRS_ALL);                      // what the variant reads at all
  const size_t hw = (size_t)c.H * c.W;
  std::vector<OdoManySession> ds(n);
  int B = 0, nA = 0;
  for (int i = 0; i < n; ++i) {
    davo_odometry* o = sessions[i];
    const int idx = single ? -1 : i;
    if (k[i] < 1 || k[i] > o->max_push)
      return fail(ctx, DAVO_ERR_ARG, "%s: %s=%d new frames outside 1..max_push %d", who, EntryName("k", idx).s, k[i], o->max_push);
    const long long f0 = o->pushed;
    const int head = o->head(), fe = head == 2 ? 1 : 0, nn = head + k[i], ns = std::max(0, nn - 2);
    const long long g0 = f0 - head;
    const int first = g0 == 0 && ns > 0;
    // what the stream reads of this push's flow entries: flow_fwd global entry e is read by sample e (as its plane 0)
    // now or later, flow_bwd entry e by sample e - 1 (plane 1), which is computed now when it exists
    const SeqReads rg = seq_reads(ctx, o->pairs == DAVO_PAIRS_ALL ? DAVO_PAIRS_ALL : DAVO_PAIRS_TRAJECTORY_FIRST);
    const long long e0 = std::max(f0 - 1, 0LL), e1 = f0 + k[i] - 1;
    const bool fwd_read = rg.flow && e1 > e0 && rg.k0((int)std::min(e0, 2LL));
    const bool bwd_read = rg.flow && ns > 0;
    auto at = [&](auto* const* a) { return a ? a[i] : nullptr; };
    OdoManySession& d = ds[i];
    d.img = img[i]; d.seg = at(seg); d.depth = at(depth); d.fwd = at(flow_fwd); d.bwd = at(flow_bwd);
    d.pose_out = at(pose_out); d.traj_out = reinterpret_cast<Mat4*>(at(traj_out));
    struct { const void* p; bool needed; const char* name; } in[] = {
        {d.img, true, "img"}, {d.pose_out, ns > 0, "pose_out"}, {d.traj_out, ns + 2 * first > 0, "traj_out"},
        {d.seg, c.att_src != 0, "seg"}, {d.depth, rg.depth, "depth"}, {d.bwd, bwd_read, "flow_bwd"},
        {d.fwd, fwd_read, "flow_fwd"}};
    for (const auto& x : in) {
      if (x.needed && !x.p)
        return fail(ctx, DAVO_ERR_ARG, "%s: %s is NULL; this variant and pair selection read it", who, EntryName(x.name, idx).s);
      if (x.p && (reinterpret_cast<uintptr_t>(x.p) & 15))
        return fail(ctx, DAVO_ERR_ARG, "%s: %s is not 16-byte aligned", who, EntryName(x.name, idx).s);
    }
    d.c_img = o->c_img; d.c_seg = o->c_seg; d.c_depth = rv.depth ? o->c_depth : nullptr; d.c_fwd = o->c_fwd;
    d.P = o->d_P; d.rel = o->d_rel;
    d.head = head; d.fe = fe; d.k = k[i]; d.ns = ns; d.first = first;
    d.na = (ctx->unit_sample || o->pairs == DAVO_PAIRS_ALL) ? ns : first;
    const int e = nn - 2;                                                 // the last flow_fwd entry, read by a later sample
    d.carry_fwd = e >= fe && rg.fwd((int)std::min(g0 + e, 2LL)) ? e - fe : -1;
    if (att)
      if (int rc = att_check(ctx, who, att[i], ns + 2 * first, idx)) return rc;
    B += ns;
    nA += d.na;
  }
  if (B > c.max_batch) return fail(ctx, DAVO_ERR_ARG, "%s: %d samples in all, more than max_batch %d", who, B, c.max_batch);
  std::vector<int2> smp(B);                                               // staging order: both-pair samples first
  for (int i = 0, a = 0, t = nA; i < n; ++i) {
    OdoManySession& d = ds[i];
    d.ba = a; d.bt = t;
    for (int s = 0; s < d.ns; ++s) smp[s < d.na ? a++ : t++] = make_int2(i, s);
  }
  // the forwards over the staging batch: one pass when only staging sample 0 computes both pairs (the opening push of a
  // trajectory session; the non-shared nets stage every sample as both-pair, nA == B)
  struct Pass { int mode, b0, nb; };
  std::vector<Pass> passes;
  if (nA == 1 && B > 1) {
    passes.push_back({DAVO_PAIRS_TRAJECTORY_FIRST, 0, B});
  } else {
    if (nA > 0) passes.push_back({DAVO_PAIRS_ALL, 0, nA});
    if (B > nA) passes.push_back({DAVO_PAIRS_TRAJECTORY, nA, B - nA});
  }
  CU_OK(cudaSetDevice(ctx->device));
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  if (!ctx->m_img) {                                                      // the staging batch, once per handle
    const size_t mb = (size_t)c.max_batch;
    CU_OK(cudaMalloc((void**)&ctx->m_img, mb * hw * 9));
    if (rv.labels) CU_OK(cudaMalloc((void**)&ctx->m_lab, mb * hw * 3));
    if (rv.depth) CU_OK(cudaMalloc((void**)&ctx->m_depth, mb * hw * 3 * 4));
    if (rv.flow) CU_OK(cudaMalloc((void**)&ctx->m_flow, mb * hw * 4 * 4));
    CU_OK(cudaMalloc((void**)&ctx->m_pose, mb * 12 * 4));
  }
  size_t h2d = 0;
  int set = 0;
  if (host) {
    if (int rc = host_setup(ctx, who); rc < 0) return rc;
    if (int rc = host_order_first_call(ctx, st)) return rc;
    if (!ctx->m_hpose) CU_OK(cudaMalloc((void**)&ctx->m_hpose, (size_t)c.max_batch * 12 * 4));
    for (int i = 0, s = 0; i < n; s += ds[i].ns, ++i) {                   // device results, copied back at the end
      ds[i].pose_out = ctx->m_hpose + (size_t)12 * s;
      ds[i].traj_out = sessions[i]->d_traj;
    }
    set = (int)(ctx->a_calls++ & 1);
    if (int rc = many_host_arrivals(ctx, n, sessions, ds.data(), st, set, &h2d)) return rc;
  }
  // each posed frame's attention: session i's rows from rb[i] on, one unit table per pass; host sessions' rows are
  // staged on the device
  std::vector<int> rb(n + 1, 0);
  for (int i = 0; i < n; ++i) rb[i + 1] = rb[i] + ds[i].ns + 2 * ds[i].first;
  const bool want_att = att && B > 0;
  float *att_maps = nullptr, *att_wts = nullptr;
  std::vector<int4> units;
  std::vector<AttRow> rows;
  std::vector<size_t> unit0;                                              // each pass's first unit
  if (want_att) {
    if (host)
      if (int rc = att_stage(ctx, (size_t)rb[n], &att_maps, &att_wts)) return rc;
    for (int i = 0; i < n; ++i) {
      const int nt = rb[i + 1] - rb[i];
      if (host) att_rows_of(rows, att[i].map ? att_maps + hw * rb[i] : nullptr,
                            att[i].weights ? att_wts + kAttWeightFloats * rb[i] : nullptr, nt, hw);
      else att_rows_of(rows, att[i].map, att[i].weights, nt, hw);
    }
    for (const Pass& p : passes) {
      const int mode = ctx->unit_sample ? kUnitsAreSamples : p.mode;
      unit0.push_back(units.size());
      att_unit_table(units, mode, pairs_selected(mode, p.nb), [&](int b) {
        const int2 m = smp[p.b0 + b];
        const OdoManySession& d = ds[m.x];
        return AttSample{rb[m.x] + m.y + 2 * d.first, d.first && m.y == 0};
      });
    }
  }
  // the descriptors (sessions, staging samples, unit table, rows): one copy from a pinned ring slot, refilled only
  // after the call that last used it has finished
  const int slot = (int)(ctx->m_calls++ % davo_ctx::kManyRing);
  auto up16 = [](size_t b) { return (b + 15) & ~(size_t)15; };
  const size_t o_smp = up16(sizeof(OdoManySession) * n), o_units = up16(o_smp + sizeof(int2) * B);
  const size_t o_rows = o_units + sizeof(int4) * units.size(), bytes = o_rows + sizeof(AttRow) * rows.size();
  if (ctx->m_ev[slot]) CU_OK(cudaEventSynchronize(ctx->m_ev[slot]));
  else CU_OK(cudaEventCreateWithFlags(&ctx->m_ev[slot], cudaEventDisableTiming));
  if (ctx->m_desc_cap[slot] < bytes) {
    const size_t cap = std::max<size_t>(bytes, 2 * ctx->m_desc_cap[slot]);
    if (ctx->m_hdesc[slot]) { CU_OK(cudaFreeHost(ctx->m_hdesc[slot])); ctx->m_hdesc[slot] = nullptr; }
    if (ctx->m_ddesc[slot]) { CU_OK(cudaFree(ctx->m_ddesc[slot])); ctx->m_ddesc[slot] = nullptr; }
    ctx->m_desc_cap[slot] = 0;
    CU_OK(cudaHostAlloc(&ctx->m_hdesc[slot], cap, cudaHostAllocDefault));
    CU_OK(cudaMalloc(&ctx->m_ddesc[slot], cap));
    ctx->m_desc_cap[slot] = cap;
  }
  uint8_t* h = static_cast<uint8_t*>(ctx->m_hdesc[slot]);
  memcpy(h, ds.data(), sizeof(OdoManySession) * n);
  if (B) memcpy(h + o_smp, smp.data(), sizeof(int2) * B);
  if (!units.empty()) memcpy(h + o_units, units.data(), sizeof(int4) * units.size());
  if (!rows.empty()) memcpy(h + o_rows, rows.data(), sizeof(AttRow) * rows.size());
  CU_OK(cudaMemcpyAsync(ctx->m_ddesc[slot], h, bytes, cudaMemcpyHostToDevice, st));
  const uint8_t* dd = static_cast<const uint8_t*>(ctx->m_ddesc[slot]);
  const OdoManySession* dsess = reinterpret_cast<const OdoManySession*>(dd);
  constexpr int kCopyBlocks = 4 * 148;                                     // blocks of a copy launch, over its rows
  if (B > 0) {
    OdoStageParams sp;
    sp.sess = dsess;
    sp.smp = reinterpret_cast<const int2*>(dd + o_smp);
    sp.hw = (long long)hw; sp.na = nA;
    sp.flow = rv.flow; sp.labels = rv.labels; sp.tgt_labels = rv.tgt_labels; sp.depth = rv.depth;
    sp.lab8 = host && ctx->host_seg8;
    sp.img = ctx->m_img; sp.lab = ctx->m_lab; sp.dep = ctx->m_depth; sp.fl = ctx->m_flow;
    odo_stage_kernel<<<dim3(std::min(32, std::max(1, kCopyBlocks / B)), B), 256, 0, st>>>(sp);
    CU_OK(cudaGetLastError());
  }
  // a separate launch: the stage kernel reads the carried frames this one overwrites
  odo_carry_kernel<<<dim3(std::min(16, std::max(1, kCopyBlocks / n)), n), 256, 0, st>>>(dsess, (long long)hw, rv.depth);
  CU_OK(cudaGetLastError());
  if (host) {
    // the arrivals set is free again; the next call's copies also wait for this point, which measured faster for host
    // pushes of 128 frames than letting them start under this call's staging (DESIGN section 8.5)
    CU_OK(cudaEventRecord(ctx->a_done[set], st));
    CU_OK(cudaStreamWaitEvent(ctx->copy_stream, ctx->a_done[set], 0));
  }
  if (B > 0) {
    for (size_t q = 0; q < passes.size(); ++q) {
      const Pass& p = passes[q];
      const size_t b0 = (size_t)p.b0;
      const InputView v = stacked_view(c.H, c.W, ctx->m_img + hw * 9 * b0, ctx->m_flow ? ctx->m_flow + hw * 4 * b0 : nullptr,
                                       ctx->m_lab ? ctx->m_lab + hw * 3 * b0 : nullptr,
                                       ctx->m_depth ? ctx->m_depth + hw * 3 * b0 : nullptr);
      AttScope scope(ctx, want_att ? reinterpret_cast<const int4*>(dd + o_units) + unit0[q] : nullptr,
                     want_att ? reinterpret_cast<const AttRow*>(dd + o_rows) : nullptr);
      if (int rc = forward_device(ctx, who, p.nb, p.mode, v, ctx->m_pose + 12 * b0, st)) return rc;
    }
    odo_compose_many_kernel<<<(n + 3) / 4, 128, 0, st>>>(dsess, n, ctx->m_pose);
    CU_OK(cudaGetLastError());
  }
  CU_OK(cudaEventRecord(ctx->m_ev[slot], st));
  if (host) {                                                             // each session's results to its host buffers
    long long d2h = 0;
    for (int i = 0; i < n; ++i) {
      const size_t np = (size_t)12 * 4 * ds[i].ns, nt = (size_t)16 * 8 * (ds[i].ns + 2 * ds[i].first);
      if (np) CU_OK(cudaMemcpyAsync(pose_out[i], ds[i].pose_out, np, cudaMemcpyDeviceToHost, st));
      if (nt) CU_OK(cudaMemcpyAsync(traj_out[i], ds[i].traj_out, nt, cudaMemcpyDeviceToHost, st));
      d2h += (long long)(np + nt);
      const int na = rb[i + 1] - rb[i];
      if (want_att && na > 0) {
        const size_t mb = hw * 4 * na, wb = kAttWeightFloats * 4 * na;
        if (att[i].map) CU_OK(cudaMemcpyAsync(att[i].map, att_maps + hw * rb[i], mb, cudaMemcpyDeviceToHost, st));
        if (att[i].weights) CU_OK(cudaMemcpyAsync(att[i].weights, att_wts + kAttWeightFloats * rb[i], wb, cudaMemcpyDeviceToHost, st));
        d2h += (att[i].map ? (long long)mb : 0) + (att[i].weights ? (long long)wb : 0);
      }
    }
    if (int rc = host_done(ctx, st, ticket)) return rc;
    ctx->last_h2d = (long long)h2d;
    ctx->last_d2h = d2h;
  }
  for (int i = 0; i < n; ++i) {                                           // host bookkeeping, once all is enqueued
    const int nt = ds[i].ns + 2 * ds[i].first;
    sessions[i]->pushed += k[i];
    sessions[i]->posed += nt;
    if (n_samples) n_samples[i] = ds[i].ns;
    if (n_traj) n_traj[i] = nt;
  }
  return 0;
}

// The single push: the push of one session, with the messages of the single form.  Only host sessions take a ticket.
static int odometry_push_one(const char* who, davo_odometry* o, int k, const uint8_t* img, const float* flow_fwd,
                             const float* flow_bwd, const float* seg, const float* depth, float* pose_out,
                             double* traj_out, const davo_odometry_attention* att, int* n_samples, int* n_traj,
                             void* stream, long long* ticket) {
  bool host;
  {
    std::lock_guard<std::mutex> lk(g_odo_mutex);
    if (!o || !g_odo_live.count(o)) return fail(nullptr, DAVO_ERR_ARG, "%s: the session is NULL or was destroyed", who);
    host = o->host;
  }
  if (ticket && !host) return fail(o->ctx, DAVO_ERR_ARG, "%s: ticket: a device session runs on the caller's stream; only host sessions take a ticket", who);
  return odometry_push_many_impl(host, 1, &o, &k, &img, &flow_fwd, &flow_bwd, &seg, &depth, &pose_out, &traj_out, att,
                                 n_samples, n_traj, stream, ticket, who, true);
}

extern "C" int davo_odometry_push(davo_odometry* o, int k, const uint8_t* img, const float* flow_fwd, const float* flow_bwd,
                                  const float* seg, const float* depth, float* pose_out, double* traj_out, int* n_samples,
                                  int* n_traj, void* stream, long long* ticket) {
  return odometry_push_one("davo_odometry_push", o, k, img, flow_fwd, flow_bwd, seg, depth, pose_out, traj_out, nullptr,
                           n_samples, n_traj, stream, ticket);
}

extern "C" int davo_odometry_push_attention(davo_odometry* o, int k, const uint8_t* img, const float* flow_fwd,
                                            const float* flow_bwd, const float* seg, const float* depth, float* pose_out,
                                            double* traj_out, const davo_odometry_attention* att, int* n_samples,
                                            int* n_traj, void* stream, long long* ticket) {
  return odometry_push_one("davo_odometry_push_attention", o, k, img, flow_fwd, flow_bwd, seg, depth, pose_out,
                           traj_out, att, n_samples, n_traj, stream, ticket);
}

extern "C" int davo_odometry_push_many(int n, davo_odometry* const* sessions, const int* k, const uint8_t* const* img,
                                       const float* const* flow_fwd, const float* const* flow_bwd,
                                       const float* const* seg, const float* const* depth, float* const* pose_out,
                                       double* const* traj_out, int* n_samples, int* n_traj, void* stream) {
  return odometry_push_many_impl(false, n, sessions, k, img, flow_fwd, flow_bwd, seg, depth, pose_out, traj_out, nullptr,
                                 n_samples, n_traj, stream, nullptr, "davo_odometry_push_many");
}

extern "C" int davo_odometry_push_many_host(int n, davo_odometry* const* sessions, const int* k, const uint8_t* const* img,
                                            const float* const* flow_fwd, const float* const* flow_bwd,
                                            const float* const* seg, const float* const* depth, float* const* pose_out,
                                            double* const* traj_out, int* n_samples, int* n_traj, void* stream,
                                            long long* ticket) {
  return odometry_push_many_impl(true, n, sessions, k, img, flow_fwd, flow_bwd, seg, depth, pose_out, traj_out, nullptr,
                                 n_samples, n_traj, stream, ticket, "davo_odometry_push_many_host");
}

extern "C" int davo_odometry_push_many_attention(int n, davo_odometry* const* sessions, const int* k,
                                                 const uint8_t* const* img, const float* const* flow_fwd,
                                                 const float* const* flow_bwd, const float* const* seg,
                                                 const float* const* depth, float* const* pose_out,
                                                 double* const* traj_out, const davo_odometry_attention* att,
                                                 int* n_samples, int* n_traj, void* stream) {
  return odometry_push_many_impl(false, n, sessions, k, img, flow_fwd, flow_bwd, seg, depth, pose_out, traj_out, att,
                                 n_samples, n_traj, stream, nullptr, "davo_odometry_push_many_attention");
}

extern "C" int davo_odometry_push_many_host_attention(int n, davo_odometry* const* sessions, const int* k,
                                                      const uint8_t* const* img, const float* const* flow_fwd,
                                                      const float* const* flow_bwd, const float* const* seg,
                                                      const float* const* depth, float* const* pose_out,
                                                      double* const* traj_out, const davo_odometry_attention* att,
                                                      int* n_samples, int* n_traj, void* stream, long long* ticket) {
  return odometry_push_many_impl(true, n, sessions, k, img, flow_fwd, flow_bwd, seg, depth, pose_out, traj_out, att,
                                 n_samples, n_traj, stream, ticket, "davo_odometry_push_many_host_attention");
}

extern "C" int davo_odometry_reset(davo_odometry* o) {
  std::lock_guard<std::mutex> lk(g_odo_mutex);
  if (!o || !g_odo_live.count(o)) return fail(nullptr, DAVO_ERR_ARG, "davo_odometry_reset: the session is NULL or was destroyed");
  o->pushed = 0; o->posed = 0;
  return 0;
}

extern "C" int davo_odometry_frames(const davo_odometry* o, long long* pushed, long long* posed) {
  std::lock_guard<std::mutex> lk(g_odo_mutex);
  if (!o || !g_odo_live.count(const_cast<davo_odometry*>(o)))
    return fail(nullptr, DAVO_ERR_ARG, "davo_odometry_frames: the session is NULL or was destroyed");
  if (pushed) *pushed = o->pushed;
  if (posed) *posed = o->posed;
  return 0;
}

extern "C" void davo_odometry_destroy(davo_odometry* o) {
  {
    std::lock_guard<std::mutex> lk(g_odo_mutex);
    if (!o || !g_odo_live.erase(o)) return;
  }
  cudaSetDevice(o->ctx->device);
  cudaDeviceSynchronize();                                         // work still queued may read the session's buffers
  odometry_free(o);
}

namespace {

// Every davo_config field but max_batch, in the order of davo_config: what two handles must agree on for one to
// continue the other's sessions (davo_odometry_move, davo_odometry_load).  A saved blob's header stores them so.
const struct { const char* name; int32_t davo_config::*f; } kSessionConfig[] = {
    {"H", &davo_config::H}, {"W", &davo_config::W}, {"posenn", &davo_config::posenn},
    {"cnv6_out", &davo_config::cnv6_out}, {"in_mode", &davo_config::in_mode}, {"att_src", &davo_config::att_src},
    {"att_tgt_ones", &davo_config::att_tgt_ones}, {"mask_mode", &davo_config::mask_mode},
    {"se_act", &davo_config::se_act}, {"flow_abs", &davo_config::flow_abs}, {"flow_norm", &davo_config::flow_norm},
    {"posenn_se", &davo_config::posenn_se}, {"micro_batch", &davo_config::micro_batch},
    {"depth_norm", &davo_config::depth_norm}, {"se_pool", &davo_config::se_pool},
    {"se_hidden", &davo_config::se_hidden}, {"pixel_map", &davo_config::pixel_map},
    {"depth_split", &davo_config::depth_split}, {"flow_f16", &davo_config::flow_f16},
    {"batch_norm", &davo_config::batch_norm}};
constexpr int kSessionConfigFields = sizeof kSessionConfig / sizeof kSessionConfig[0];
static_assert(kSessionConfigFields + 1 == sizeof(davo_config) / sizeof(int32_t), "a davo_config field is missing");

// the form a session of this kind holds its labels in on this handle: 0 none, 1 bytes, 2 float32
int label_form(const davo_ctx* ctx, bool host) { return ctx->cfg.att_src == 0 ? 0 : host && ctx->host_seg8 ? 1 : 2; }

// What a session carries from one push to the next, decided here alone: davo_odometry_move, _save and _load copy
// exactly these sections.  They are the last min(pushed, 2) frames' images, labels (in the form the session holds
// them) and depth planes, the flow_fwd entry a later sample reads (global entry pushed - 2, there when the push that
// ended at frame `pushed` kept it) and the last absolute pose.  The sizes follow from the handle's configuration, the
// session's kind and its counts, so they hold for a session whose buffers are not allocated yet; p[] are its buffers.
// Per-push buffers are not state: a push writes them before it reads them.
enum { kSecImg, kSecSeg8, kSecSeg, kSecDepth, kSecFwd, kSecPose };
struct Carried {
  void* p[kOdoSections];
  size_t bytes[kOdoSections];
};

Carried carried_state(const davo_odometry* o) {
  const davo_ctx* ctx = o->ctx;
  const size_t hw = (size_t)ctx->cfg.H * ctx->cfg.W, head = (size_t)o->head();
  const SeqReads r = seq_reads(ctx, o->pairs);                       // what odometry_alloc allocates
  const SeqReads rg = seq_reads(ctx, o->pairs == DAVO_PAIRS_ALL ? DAVO_PAIRS_ALL : DAVO_PAIRS_TRAJECTORY_FIRST);
  const int lf = label_form(ctx, o->host);
  const bool fwd = r.flow && o->pushed >= 2 && rg.fwd((int)std::min(o->pushed - 2, 2LL));
  return {{o->c_img, o->c_seg8, o->c_seg, o->c_depth, o->c_fwd, o->d_P},
          {hw * 3 * head, lf == 1 ? hw * head : 0, lf == 2 ? hw * 4 * head : 0, r.depth ? hw * 4 * head : 0,
           fwd ? hw * 2 * 4 : 0, o->posed > 0 ? 16 * sizeof(double) : 0}};
}

// The header of a saved session (include/davo_b200.h: davo_odometry_save), format version 1, little-endian, no padding.
struct OdoBlobHeader {
  char magic[8];                                 // "DAVOSESS"
  uint32_t version, header_bytes;
  uint64_t total_bytes;
  int32_t config[kSessionConfigFields];          // kSessionConfig
  uint64_t weights_digest;                       // weights_digest_of
  int32_t weight_rounding, conv_impl;            // 1 compensated, 0 nearest (DAVO_B200_WEIGHT_ROUNDING); davo_ctx::conv_impl
  int32_t host, label_form;
  int32_t pairs, max_push;
  int64_t pushed, posed;
  int32_t carried_frames, carried_fwd, carried_pose, reserved;
  uint64_t section_off[kOdoSections], section_bytes[kOdoSections];
  uint64_t checksum;                             // odometry_state.cuh, over the blob with this field zero
};
static_assert(sizeof(OdoBlobHeader) == 272 && offsetof(OdoBlobHeader, checksum) == 264, "the documented header layout");
constexpr uint32_t kOdoBlobVersion = 1;

// the header of session o's blob, checksum zero; sections back to back after it, each 16-byte aligned
OdoBlobHeader blob_header(const davo_odometry* o, const Carried& cs) {
  const davo_ctx* ctx = o->ctx;
  OdoBlobHeader h;
  memset(&h, 0, sizeof h);
  memcpy(h.magic, "DAVOSESS", 8);
  h.version = kOdoBlobVersion;
  h.header_bytes = sizeof h;
  for (int i = 0; i < kSessionConfigFields; ++i) h.config[i] = ctx->cfg.*kSessionConfig[i].f;
  h.weights_digest = ctx->weights_digest;
  h.weight_rounding = ctx->compensated_rounding;
  h.conv_impl = ctx->conv_impl;
  h.host = o->host;
  h.label_form = label_form(ctx, o->host);
  h.pairs = o->pairs;
  h.max_push = o->max_push;
  h.pushed = o->pushed;
  h.posed = o->posed;
  h.carried_frames = o->head();
  h.carried_fwd = cs.bytes[kSecFwd] != 0;
  h.carried_pose = cs.bytes[kSecPose] != 0;
  uint64_t at = sizeof h;
  for (int j = 0; j < kOdoSections; ++j) {
    h.section_off[j] = at;
    h.section_bytes[j] = cs.bytes[j];
    at += (cs.bytes[j] + 15) & ~(uint64_t)15;
  }
  h.total_bytes = at;
  return h;
}

// The descriptor area of a save or load call: n OdoBlob, n headers (save), n checksum accumulators, n block counters.
struct BlobArea {
  size_t headers, sums, done, bytes;
};
BlobArea blob_area(int n) {
  auto up = [](size_t b) { return (b + 15) & ~(size_t)15; };
  BlobArea a;
  a.headers = up(sizeof(OdoBlob) * n);
  a.sums = a.headers + sizeof(OdoBlobHeader) * n;
  a.done = a.sums + 8 * (size_t)n;
  a.bytes = up(a.done + 4 * (size_t)n);
  return a;
}

// Consecutive blobs [first, end) staged together: at most kBlobChunk bytes (a larger blob alone) and one grid's rows.
// *stage: the staging bytes the largest chunk needs.
constexpr size_t kBlobChunk = (size_t)256 << 20;
std::vector<std::pair<int, int>> blob_chunks(int n, const int64_t* offsets, size_t* stage) {
  std::vector<std::pair<int, int>> ch;
  *stage = 0;
  for (int i = 0; i < n;) {
    int e = i + 1;
    while (e < n && e - i < 65535 && (size_t)(offsets[e + 1] - offsets[i]) <= kBlobChunk) ++e;
    ch.push_back({i, e});
    *stage = std::max(*stage, (size_t)(offsets[e] - offsets[i]));
    i = e;
  }
  return ch;
}

// the handle's staging and descriptor areas at least this large (the calls using them are synchronous)
int blob_buffers(davo_ctx* ctx, size_t stage, size_t desc) {
  if (ctx->b_stage_cap < stage) {
    if (ctx->b_stage) { CU_OK(cudaFree(ctx->b_stage)); ctx->b_stage = nullptr; }
    ctx->b_stage_cap = 0;
    CU_OK(cudaMalloc((void**)&ctx->b_stage, stage));
    ctx->b_stage_cap = stage;
  }
  if (ctx->b_desc_cap < desc) {
    const size_t cap = std::max(desc, 2 * ctx->b_desc_cap);
    if (ctx->b_hdesc) { CU_OK(cudaFreeHost(ctx->b_hdesc)); ctx->b_hdesc = nullptr; }
    if (ctx->b_ddesc) { CU_OK(cudaFree(ctx->b_ddesc)); ctx->b_ddesc = nullptr; }
    ctx->b_desc_cap = 0;
    CU_OK(cudaHostAlloc(&ctx->b_hdesc, cap, cudaHostAllocDefault));
    CU_OK(cudaMalloc(&ctx->b_ddesc, cap));
    ctx->b_desc_cap = cap;
  }
  return 0;
}

dim3 blob_grid(int rows) { return dim3(std::min(32, std::max(1, 4 * 148 / rows)), rows); }

// "sessions[i]: " / "blob i: " for the _many forms, nothing for the single ones
std::string at_index(bool many, const char* what, int i) {
  return many ? std::string(what) + "[" + std::to_string(i) + "]: " : std::string();
}

}  // namespace

// Re-homes a session (include/davo_b200.h: davo_odometry_move).  A push reads of the session only the counts and the
// carried state, and a pose does not depend on the handle that computes it (same configuration and weights: a
// pair's result does not depend on which pairs share its pass, so not on max_batch either); so the carried state,
// copied as it is onto buffers allocated as davo_odometry_create allocates them on dst, continues the stream with the
// same bits.  The new buffers are allocated first, so a failure leaves the session where it was.
extern "C" int davo_odometry_move(davo_odometry* o, davo_ctx* dst) {
  const char* who = "davo_odometry_move";
  {
    std::lock_guard<std::mutex> lk(g_odo_mutex);
    if (!o || !g_odo_live.count(o)) return fail(nullptr, DAVO_ERR_ARG, "%s: the session is NULL or was destroyed", who);
  }
  davo_ctx* ctx = o->ctx;
  if (!dst) return fail(ctx, DAVO_ERR_ARG, "%s: dst is NULL", who);
  if (dst == ctx) return 0;
  const davo_config &a = ctx->cfg, &b = dst->cfg;
  for (const auto& x : kSessionConfig)
    if (a.*x.f != b.*x.f)
      return fail(ctx, DAVO_ERR_ARG, "%s: dst's davo_config differs in %s (%d here, %d on dst); only max_batch may differ",
                  who, x.name, a.*x.f, b.*x.f);
  if (o->max_push > b.max_batch)
    return fail(ctx, DAVO_ERR_ARG, "%s: the session's max_push %d is more than dst's max_batch %d", who, o->max_push, b.max_batch);
  if (!ctx->finalized || !dst->finalized)
    return fail(ctx, DAVO_ERR_ARG, "%s: weights not finalized on the %s handle", who, ctx->finalized ? "dst" : "session's");
  if (ctx->weights_digest != dst->weights_digest)
    return fail(ctx, DAVO_ERR_ARG, "%s: the two handles hold different weights", who);
  // settings fixed at davo_create from the environment that change what a push computes or how a session holds it
  if (ctx->compensated_rounding != dst->compensated_rounding || ctx->conv_impl != dst->conv_impl)
    return fail(ctx, DAVO_ERR_ARG, "%s: the two handles round the weights (DAVO_B200_WEIGHT_ROUNDING) or run the convolutions differently", who);
  if (label_form(ctx, o->host) != label_form(dst, o->host))
    return fail(ctx, DAVO_ERR_ARG, "%s: the two handles hold a host session's labels in different forms (DAVO_B200_HOST_SEG8)", who);
  davo_odometry* t = new davo_odometry;
  t->ctx = dst; t->max_push = o->max_push; t->pairs = o->pairs; t->host = o->host;
  if (int rc = odometry_alloc(t)) {
    ctx->err = dst->err;
    odometry_free(t);
    return rc;
  }
  const Carried from = carried_state(o), to = carried_state(t);
  auto copy = [&]() -> int {
    // as davo_odometry_destroy: work still queued on the source device may read or write the carried state
    CU_OK(cudaSetDevice(ctx->device));
    CU_OK(cudaDeviceSynchronize());
    for (int j = 0; j < kOdoSections; ++j)                        // peer access is not needed, and is not enabled
      if (from.bytes[j]) CU_OK(cudaMemcpyPeerAsync(to.p[j], dst->device, from.p[j], ctx->device, from.bytes[j], 0));
    CU_OK(cudaStreamSynchronize(0));
    return 0;
  };
  if (int rc = copy()) {
    odometry_free(t);
    return rc;
  }
  t->pushed = o->pushed; t->posed = o->posed;
  {
    std::lock_guard<std::mutex> lk(g_odo_mutex);
    std::swap(*o, *t);                                             // t: the old buffers, on the source handle
  }
  odometry_free(t);
  return 0;
}

// Saves sessions (include/davo_b200.h: davo_odometry_save_many): after the device has finished the work queued on it,
// odo_save_kernel stages every blob as the caller's buffer lays them out, chunk by chunk, and each chunk goes to the
// caller's buffer in one copy.  The sessions are only read.
static int odometry_save_impl(const char* who, bool many, int n, davo_odometry* const* sessions, void* buf,
                              int64_t capacity, int64_t* offsets) {
  if (n < 1) return fail(nullptr, DAVO_ERR_ARG, "%s: n=%d: at least one session", who, n);
  if (!sessions) return fail(nullptr, DAVO_ERR_ARG, "%s: sessions is NULL", who);
  {
    std::lock_guard<std::mutex> lk(g_odo_mutex);
    for (int i = 0; i < n; ++i)
      if (!sessions[i] || !g_odo_live.count(sessions[i]))
        return fail(nullptr, DAVO_ERR_ARG, "%s: %sthe session is NULL or was destroyed", who, at_index(many, "sessions", i).c_str());
  }
  davo_ctx* ctx = sessions[0]->ctx;
  if (!offsets) return fail(ctx, DAVO_ERR_ARG, "%s: %s is NULL", who, many ? "offsets" : "bytes");
  for (int i = 1; i < n; ++i)
    if (sessions[i]->ctx != ctx)
      return fail(ctx, DAVO_ERR_ARG, "%s: sessions[%d] belongs to another handle than sessions[0]", who, i);
  std::vector<Carried> cs(n);
  std::vector<OdoBlobHeader> hd(n);
  offsets[0] = 0;
  for (int i = 0; i < n; ++i) {
    cs[i] = carried_state(sessions[i]);
    hd[i] = blob_header(sessions[i], cs[i]);
    offsets[i + 1] = offsets[i] + (int64_t)hd[i].total_bytes;
  }
  if (!buf || capacity < offsets[n])
    return fail(ctx, DAVO_ERR_ARG, "%s: capacity %lld bytes%s; the blobs take %lld (%s)", who, (long long)capacity,
                buf ? "" : " (buf is NULL)", (long long)offsets[n], many ? "offsets[n]" : "*bytes");
  CU_OK(cudaSetDevice(ctx->device));
  CU_OK(cudaDeviceSynchronize());          // as davo_odometry_move: queued pushes and host tickets write the carried state
  size_t stage = 0;
  const auto chunks = blob_chunks(n, offsets, &stage);
  const BlobArea A = blob_area(n);
  if (int rc = blob_buffers(ctx, stage, A.bytes)) return rc;
  uint8_t* h = static_cast<uint8_t*>(ctx->b_hdesc);
  uint8_t* dd = static_cast<uint8_t*>(ctx->b_ddesc);
  memset(h, 0, A.bytes);
  OdoBlob* hb = reinterpret_cast<OdoBlob*>(h);
  for (const auto& ch : chunks)
    for (int i = ch.first; i < ch.second; ++i) {
      OdoBlob& b = hb[i];
      b.blob = ctx->b_stage + (offsets[i] - offsets[ch.first]);
      memcpy(h + A.headers + sizeof(OdoBlobHeader) * i, &hd[i], sizeof(OdoBlobHeader));
      b.header = dd + A.headers + sizeof(OdoBlobHeader) * i;
      for (int j = 0; j < kOdoSections; ++j) {
        b.sec[j] = static_cast<uint8_t*>(cs[i].p[j]);
        b.off[j] = hd[i].section_off[j];
        b.bytes[j] = cs[i].bytes[j];
      }
      b.sum = reinterpret_cast<unsigned long long*>(dd + A.sums) + i;
      b.done = reinterpret_cast<unsigned int*>(dd + A.done) + i;
    }
  cudaStream_t st = 0;
  CU_OK(cudaMemcpyAsync(dd, h, A.bytes, cudaMemcpyHostToDevice, st));
  int launches = 0;
  for (const auto& ch : chunks) {
    odo_save_kernel<<<blob_grid(ch.second - ch.first), 256, 0, st>>>(reinterpret_cast<const OdoBlob*>(dd) + ch.first,
                                                                     (unsigned)sizeof(OdoBlobHeader));
    CU_OK(cudaGetLastError());
    ++launches;
    CU_OK(cudaMemcpyAsync(static_cast<uint8_t*>(buf) + offsets[ch.first], ctx->b_stage,
                          (size_t)(offsets[ch.second] - offsets[ch.first]), cudaMemcpyDeviceToHost, st));
  }
  CU_OK(cudaStreamSynchronize(st));
  ctx->last_launches = launches;
  ctx->last_h2d = (long long)A.bytes;
  ctx->last_d2h = (long long)offsets[n];
  return 0;
}

// Loads sessions (include/davo_b200.h: davo_odometry_load_many): every header is checked on the host first, against a
// session of its kind and counts on dst (blob_header), so a blob whose fields disagree with each other or with dst is
// refused before anything is allocated.  Then the sessions are allocated, each chunk of blobs goes to the staging area
// in one copy, odo_load_kernel scatters the sections and sums the blobs, and the sessions are handed out only when
// every sum equals its stored checksum.
static int odometry_load_impl(const char* who, bool many, davo_ctx* dst, int n, const void* buf, const int64_t* offsets,
                              davo_odometry** out) {
  if (!dst) return fail(nullptr, DAVO_ERR_ARG, "%s: dst is NULL", who);
  davo_ctx* ctx = dst;                                             // CU_OK reports on it
  if (n < 1) return fail(dst, DAVO_ERR_ARG, "%s: n=%d: at least one blob", who, n);
  if (!buf) return fail(dst, DAVO_ERR_ARG, "%s: buf is NULL", who);
  if (!offsets) return fail(dst, DAVO_ERR_ARG, "%s: %s is NULL", who, many ? "offsets" : "bytes");
  if (!out) return fail(dst, DAVO_ERR_ARG, "%s: out is NULL", who);
  if (!dst->finalized) return fail(dst, DAVO_ERR_ARG, "%s: weights not finalized on dst", who);
  if (dst->cfg.batch_norm) return fail(dst, DAVO_ERR_ARG, "%s: -batch_norm: a session does not take it (davo_odometry_create)", who);
  const uint8_t* base = static_cast<const uint8_t*>(buf);
  std::vector<OdoBlobHeader> hd(n);
  for (int i = 0; i < n; ++i) {
    const std::string at = at_index(many, "blob", i);
    const char* p = at.c_str();
    const int64_t size = offsets[i + 1] - offsets[i];
    if (offsets[i] < 0 || size < (int64_t)sizeof(OdoBlobHeader))
      return fail(dst, DAVO_ERR_ARG, "%s: %s%lld bytes at offset %lld: shorter than the %d-byte header (truncated?)", who, p,
                  (long long)size, (long long)offsets[i], (int)sizeof(OdoBlobHeader));
    OdoBlobHeader& h = hd[i];
    memcpy(&h, base + offsets[i], sizeof h);
    if (memcmp(h.magic, "DAVOSESS", 8) != 0)
      return fail(dst, DAVO_ERR_ARG, "%s: %snot a saved odometry session (bad magic)", who, p);
    if (h.version != kOdoBlobVersion || h.header_bytes != sizeof h)
      return fail(dst, DAVO_ERR_ARG, "%s: %sformat version %u with a %u-byte header; this library reads version %u (%d bytes)",
                  who, p, h.version, h.header_bytes, kOdoBlobVersion, (int)sizeof h);
    if (h.total_bytes != (uint64_t)size)
      return fail(dst, DAVO_ERR_ARG, "%s: %sthe blob is %lld bytes, its header says %llu (truncated or cut wrongly)", who, p,
                  (long long)size, (unsigned long long)h.total_bytes);
    for (int f = 0; f < kSessionConfigFields; ++f)
      if (h.config[f] != dst->cfg.*kSessionConfig[f].f)
        return fail(dst, DAVO_ERR_ARG, "%s: %sdst's davo_config differs in %s (%d in the blob, %d on dst); only max_batch may differ",
                    who, p, kSessionConfig[f].name, h.config[f], dst->cfg.*kSessionConfig[f].f);
    if (h.weights_digest != dst->weights_digest)
      return fail(dst, DAVO_ERR_ARG, "%s: %sthe blob was saved from different weights than dst holds", who, p);
    if (h.weight_rounding != (int32_t)dst->compensated_rounding || h.conv_impl != dst->conv_impl)
      return fail(dst, DAVO_ERR_ARG, "%s: %sthe blob's handle rounded the weights (DAVO_B200_WEIGHT_ROUNDING) or ran the convolutions differently than dst", who, p);
    if ((h.host != 0 && h.host != 1) || (h.pairs != DAVO_PAIRS_TRAJECTORY && h.pairs != DAVO_PAIRS_ALL) || h.max_push < 1 ||
        h.pushed < 0 || h.posed < 0)
      return fail(dst, DAVO_ERR_ARG, "%s: %sthe header's session kind or counts are out of range", who, p);
    if (h.label_form != label_form(dst, h.host))
      return fail(dst, DAVO_ERR_ARG, "%s: %sthe blob holds a host session's labels in another form (%d) than dst does (%d) (DAVO_B200_HOST_SEG8)",
                  who, p, h.label_form, label_form(dst, h.host));
    if (h.max_push > dst->cfg.max_batch)
      return fail(dst, DAVO_ERR_ARG, "%s: %sthe session's max_push %d is more than dst's max_batch %d", who, p, h.max_push,
                  dst->cfg.max_batch);
    davo_odometry s;                                               // its kind and counts on dst, no buffers
    s.ctx = dst; s.max_push = h.max_push; s.pairs = h.pairs; s.host = h.host; s.pushed = h.pushed; s.posed = h.posed;
    OdoBlobHeader want = blob_header(&s, carried_state(&s));
    want.checksum = h.checksum;
    if (memcmp(&want, &h, sizeof h) != 0)
      return fail(dst, DAVO_ERR_ARG, "%s: %sthe header's carried sections disagree with its counts", who, p);
  }
  CU_OK(cudaSetDevice(dst->device));
  std::vector<davo_odometry*> made;
  auto drop = [&]() {
    for (davo_odometry* o : made) odometry_free(o);
  };
  std::vector<Carried> cs(n);
  for (int i = 0; i < n; ++i) {
    davo_odometry* t = new davo_odometry;
    t->ctx = dst; t->max_push = hd[i].max_push; t->pairs = hd[i].pairs; t->host = hd[i].host;
    made.push_back(t);
    if (int rc = odometry_alloc(t)) { drop(); return rc; }
    t->pushed = hd[i].pushed; t->posed = hd[i].posed;
    cs[i] = carried_state(t);
  }
  size_t stage = 0;
  const auto chunks = blob_chunks(n, offsets, &stage);
  const BlobArea A = blob_area(n);
  cudaStream_t st = 0;
  int launches = 0;
  auto run = [&]() -> int {
    if (int rc = blob_buffers(dst, stage, A.bytes)) return rc;
    uint8_t* h = static_cast<uint8_t*>(dst->b_hdesc);
    uint8_t* dd = static_cast<uint8_t*>(dst->b_ddesc);
    memset(h, 0, A.bytes);
    OdoBlob* hb = reinterpret_cast<OdoBlob*>(h);
    for (const auto& ch : chunks)
      for (int i = ch.first; i < ch.second; ++i) {
        OdoBlob& b = hb[i];
        b.blob = dst->b_stage + (offsets[i] - offsets[ch.first]);
        for (int j = 0; j < kOdoSections; ++j) {
          b.sec[j] = static_cast<uint8_t*>(cs[i].p[j]);
          b.off[j] = hd[i].section_off[j];
          b.bytes[j] = cs[i].bytes[j];
        }
        b.sum = reinterpret_cast<unsigned long long*>(dd + A.sums) + i;
      }
    CU_OK(cudaMemcpyAsync(dd, h, A.bytes, cudaMemcpyHostToDevice, st));
    for (const auto& ch : chunks) {
      CU_OK(cudaMemcpyAsync(dst->b_stage, base + offsets[ch.first], (size_t)(offsets[ch.second] - offsets[ch.first]),
                            cudaMemcpyHostToDevice, st));
      odo_load_kernel<<<blob_grid(ch.second - ch.first), 256, 0, st>>>(reinterpret_cast<const OdoBlob*>(dd) + ch.first,
                                                                       (unsigned)sizeof(OdoBlobHeader));
      CU_OK(cudaGetLastError());
      ++launches;
    }
    CU_OK(cudaMemcpyAsync(h + A.sums, dd + A.sums, 8 * (size_t)n, cudaMemcpyDeviceToHost, st));
    CU_OK(cudaStreamSynchronize(st));
    const unsigned long long* sum = reinterpret_cast<const unsigned long long*>(h + A.sums);
    for (int i = 0; i < n; ++i)
      if (sum[i] != hd[i].checksum)
        return fail(dst, DAVO_ERR_ARG, "%s: %schecksum mismatch: the blob is corrupt", who, at_index(many, "blob", i).c_str());
    return 0;
  };
  if (int rc = run()) {
    drop();
    return rc;
  }
  {
    std::lock_guard<std::mutex> lk(g_odo_mutex);
    for (davo_odometry* o : made) g_odo_live.insert(o);
  }
  for (int i = 0; i < n; ++i) out[i] = made[i];
  dst->last_launches = launches;
  dst->last_h2d = (long long)(A.bytes + (offsets[n] - offsets[0]));
  dst->last_d2h = 8LL * n;
  return 0;
}

extern "C" int davo_odometry_state_bytes(const davo_odometry* o, int64_t* bytes) {
  std::lock_guard<std::mutex> lk(g_odo_mutex);
  if (!o || !g_odo_live.count(const_cast<davo_odometry*>(o)))
    return fail(nullptr, DAVO_ERR_ARG, "davo_odometry_state_bytes: the session is NULL or was destroyed");
  if (!bytes) return fail(o->ctx, DAVO_ERR_ARG, "davo_odometry_state_bytes: bytes is NULL");
  *bytes = (int64_t)blob_header(o, carried_state(o)).total_bytes;
  return 0;
}

extern "C" int davo_odometry_save(davo_odometry* o, void* buf, int64_t capacity, int64_t* bytes) {
  int64_t off[2] = {0, 0};
  const int rc = odometry_save_impl("davo_odometry_save", false, 1, &o, buf, capacity, bytes ? off : nullptr);
  if (bytes) *bytes = off[1];
  return rc;
}

extern "C" int davo_odometry_save_many(int n, davo_odometry* const* sessions, void* buf, int64_t capacity, int64_t* offsets) {
  return odometry_save_impl("davo_odometry_save_many", true, n, sessions, buf, capacity, offsets);
}

extern "C" int davo_odometry_load(davo_ctx* dst, const void* buf, int64_t bytes, davo_odometry** out) {
  const int64_t off[2] = {0, bytes};
  return odometry_load_impl("davo_odometry_load", false, dst, 1, buf, off, out);
}

extern "C" int davo_odometry_load_many(davo_ctx* dst, int n, const void* buf, const int64_t* offsets, davo_odometry** out) {
  return odometry_load_impl("davo_odometry_load_many", true, dst, n, buf, offsets, out);
}

// davo_destroy: the handle's sessions go with it
static void destroy_sessions_of(davo_ctx* ctx) {
  std::vector<davo_odometry*> mine;
  {
    std::lock_guard<std::mutex> lk(g_odo_mutex);
    for (davo_odometry* o : g_odo_live) if (o->ctx == ctx) mine.push_back(o);
  }
  for (davo_odometry* o : mine) davo_odometry_destroy(o);
}

extern "C" int davo_last_host_copy_bytes(const davo_ctx* ctx, long long* h2d, long long* d2h) {
  if (!ctx || !h2d || !d2h) return DAVO_ERR_ARG;
  *h2d = ctx->last_h2d;
  *d2h = ctx->last_d2h;
  return 0;
}

extern "C" int davo_last_launch_count(const davo_ctx* ctx) { return ctx ? ctx->last_launches : 0; }

extern "C" int davo_get_intermediate(davo_ctx* ctx, const char* name, int pair, float* out,
                                     int64_t cap, int64_t* n_out) {
  if (!ctx || !name || !out || !n_out) return DAVO_ERR_ARG;
  if (!ctx->finalized || ctx->last_npairs_mb == 0) return fail(ctx, DAVO_ERR_STATE, "davo_get_intermediate: no forward has run");
  if (pair < 0 || pair >= ctx->last_npairs_mb) return fail(ctx, DAVO_ERR_ARG, "davo_get_intermediate: pair %d not in the last micro-batch (0..%d)", pair, ctx->last_npairs_mb - 1);
  CU_OK(cudaSetDevice(ctx->device));
  CU_OK(cudaDeviceSynchronize());
  const davo_config& c = ctx->cfg;
  const float* src = nullptr;
  int64_t n = 0;
  std::string s(name);
  // A caller whose buffer is too small learns the size it needs from *n_out.
  auto too_small = [&](int64_t need) {
    *n_out = need;
    return fail(ctx, DAVO_ERR_ARG, "davo_get_intermediate: buffer too small (%lld < %lld)", (long long)cap, (long long)need);
  };
  // the fused cnv1 never writes the packed input: pack8_kernel, the same arithmetic (frontend.cuh: pack8_quad), on the last pass's inputs
  auto materialise_packed = [&]() -> int {
    if (ctx->fuse_front && ctx->conv_impl == 0 && ctx->layers[0].fused_front) {
      if (int rc = launch_k(ctx, pack8_kernel, dim3(pack8_blocks(ctx->fp_cur.npairs), ctx->fp_cur.npairs), dim3(256), 0, (cudaStream_t)0, false, ctx->fp_cur)) return rc;
      CU_OK(cudaDeviceSynchronize());
    }
    return 0;
  };
  const size_t colon = s.find(':');
  const std::string lname = s.substr(0, colon), part = colon == std::string::npos ? "" : s.substr(colon + 1);
  int li = -1;
  for (int i = 0; i < (int)ctx->layers.size(); ++i) if (lname == ctx->layers[i].name) li = i;
  if (s == "att_weights") {
    n = kNumClasses;
    if (cap < n) return too_small(n);
    if (c.att_src == 1 || c.att_src >= 3) src = ctx->d_attw + (size_t)pair * kAttFrames * kAttStride;
    else if (c.att_src == 2) src = ctx->d_staticw;
    else { for (int i = 0; i < n; ++i) out[i] = 1.0f; *n_out = n; return 0; }
  }
  else if (lname == "att_weights") {
    // slot <k> of the unit's attention weights, laid out as unit_frame / pack_sample_kernel read them (frontend.cuh):
    // the slots the SE kernels write, or the static table for every frame that has a map; anything else is refused
    const int slot = (part.size() == 1 && part[0] >= '0' && part[0] <= '9') ? part[0] - '0' : -1;
    const int src_frames = ctx->unit_sample ? 2 : 1;
    const int nslots = c.att_src == 0 ? 0 : c.depth_split ? 2 * src_frames : src_frames + (c.att_tgt_ones ? 0 : 1);
    if (slot < 0 || slot >= nslots)
      return fail(ctx, DAVO_ERR_ARG, "davo_get_intermediate: %s: this variant computes %d attention-weight slot(s) per unit (%s)",
                  name, nslots, ctx->unit_sample ? "0 src0, 1 src1, 2 target; depth split: 0/1 src0 near/far, 2/3 src1 near/far"
                                                 : "0 source, 1 target or, under the depth split, the far table");
    // width: 19 class weights, or the excitation of a per-pixel source (its SE input channels)
    n = !c.pixel_map ? kNumClasses : c.pixel_map == 2 ? 3 : c.att_src == 4 ? 3 : c.att_src == 5 ? 1 : kNumClasses + 2;
    if (cap < n) return too_small(n);
    src = c.att_src == 2 ? ctx->d_staticw : ctx->d_attw + ((size_t)pair * kAttFrames + slot) * kAttStride;
  }
  else if (s == "packed") {
    n = (int64_t)c.H * c.W * ctx->packed_c; src = ctx->d_packed + (size_t)pair * n;
    if (int rc = materialise_packed()) return rc;
  }
  else if (s == "se5_scale") {
    if (!ctx->d_se5scale) return fail(ctx, DAVO_ERR_ARG, "davo_get_intermediate: se5_scale: this variant has no SE block on cnv5 / cnv6");
    n = (int64_t)ctx->nbr * 256; src = ctx->d_se5scale + (size_t)pair * n;
  }
  else if (s == "cnv7_sum") {
    // reduce the deterministic partials on the host
    const int np = ctx->nparts7;
    const int nbr = ctx->nbr;
    std::vector<float> tmp((size_t)nbr * np * 256);
    CU_OK(cudaMemcpy(tmp.data(), ctx->d_sum7 + (size_t)pair * nbr * np * 256, tmp.size() * 4, cudaMemcpyDeviceToHost));
    if (cap < nbr * 256) return too_small(nbr * 256);
    for (int br = 0; br < nbr; ++br)
      for (int ch = 0; ch < 256; ++ch) {
        float a = 0.f;
        for (int i = 0; i < np; ++i) a += tmp[((size_t)br * np + i) * 256 + ch];
        out[br * 256 + ch] = a;
      }
    *n_out = nbr * 256;
    return 0;
  } else if (li >= 0) {
    const Layer& L = ctx->layers[li];
    const bool rep6 = li == 5 && c.posenn_se == 3;          // -se_replace: no cnv6 convolution
    if (part.empty() || part == "pitched") {
      // the map [Hout][Wout][C] with the pad row / column of an odd map removed, or the whole [Hout_p][Wout_p][C] buffer
      if (!L.d_out) return fail(ctx, DAVO_ERR_ARG, "davo_get_intermediate: %s is not stored by this variant", L.name);
      const int64_t per = (int64_t)L.Hout_p * L.Wout_p * L.out_stride;
      if (part == "pitched" || !L.pitched_out()) { n = per; src = L.d_out + (size_t)pair * per; }
      else {
        n = (int64_t)L.Hout * L.Wout * L.out_stride;
        if (cap < n) return too_small(n);
        const size_t row = (size_t)L.Wout * L.out_stride * 4;
        CU_OK(cudaMemcpy2D(out, row, L.d_out + (size_t)pair * per, (size_t)L.Wout_p * L.out_stride * 4, row, L.Hout, cudaMemcpyDeviceToHost));
        *n_out = n;
        return 0;
      }
    } else if (part == "in") {
      // what the layer's kernel reads: [Hin_p][Win_p][Cin_total] (cnv1: the packed input; d_se5out under the SE variants)
      if (rep6) return fail(ctx, DAVO_ERR_ARG, "davo_get_intermediate: %s is not computed by this variant", L.name);
      n = (int64_t)L.Hin_p * L.Win_p * L.Cin_total; src = L.d_in + (size_t)pair * n;
      if (li == 0)
        if (int rc = materialise_packed()) return rc;
    } else if (part == "b") {
      // the bias the weight pack was built with (-batch_norm: beta; the conv itself adds nothing)
      if (rep6) return fail(ctx, DAVO_ERR_ARG, "davo_get_intermediate: %s is not computed by this variant", L.name);
      n = (int64_t)L.groups * L.BN; src = c.batch_norm ? L.d_beta : L.d_bias;
    } else if (part.size() >= 2 && part[0] == 'w' && part.find_first_not_of("0123456789", 1) == std::string::npos) {
      // TF32 weights of group g as the pack was built from them (round_weights_tf32), HWIO over the input tensor's
      // channels of that group: [k][k][Cin_g][BN], zero for an input channel no weight reads (cnv1's packed layout)
      const int g = atoi(part.c_str() + 1);
      if (rep6) return fail(ctx, DAVO_ERR_ARG, "davo_get_intermediate: %s is not computed by this variant", L.name);
      if (g >= L.groups) return fail(ctx, DAVO_ERR_ARG, "davo_get_intermediate: %s has %d group(s)", L.name, L.groups);
      const int T = L.k * L.k;
      n = (int64_t)T * L.Cin_g * L.BN;
      if (cap < n) return too_small(n);
      std::vector<float> hw((size_t)T * L.Cin_w * L.BN);
      CU_OK(cudaMemcpy(hw.data(), L.d_whwio[g], hw.size() * 4, cudaMemcpyDeviceToHost));
      for (int t = 0; t < T; ++t)
        for (int j = 0; j < L.Cin_g; ++j) {
          const int ci = li == 0 ? L.pc2w[j] : j;
          for (int o = 0; o < L.BN; ++o) out[((size_t)t * L.Cin_g + j) * L.BN + o] = ci >= 0 ? hw[((size_t)t * L.Cin_w + ci) * L.BN + o] : 0.f;
        }
      *n_out = n;
      return 0;
    } else if (part == "plan") {
      // the plan the last pass ran for this layer (its latency twin included)
      if (rep6) return fail(ctx, DAVO_ERR_ARG, "davo_get_intermediate: %s is not computed by this variant", L.name);
      const Layer& P = pick_layer(ctx, (size_t)li, ctx->last_npairs_mb);
      const float v[] = {(float)P.orient, (float)P.npix, (float)P.wide_G, (float)P.wide_tw, (float)P.cm_staged,
                         (float)P.cm_cluster, (float)P.strips, (float)P.m_blocks, (float)P.groups, (float)(c.batch_norm ? 1 : 0),
                         (float)P.epi, (float)P.BN, (float)P.b_resident, (float)P.fused_front};
      n = (int64_t)(sizeof v / sizeof v[0]);
      if (cap < n) return too_small(n);
      for (int i = 0; i < n; ++i) out[i] = v[i];
      *n_out = n;
      return 0;
    }
  }
  if (!src) return fail(ctx, DAVO_ERR_ARG, "davo_get_intermediate: unknown name '%s'", name);
  if (cap < n) return too_small(n);
  CU_OK(cudaMemcpy(out, src, (size_t)n * 4, cudaMemcpyDeviceToHost));
  *n_out = n;
  return 0;
}

#ifdef DAVO_TIMING
// Debug build only: run layer `layer` once and return the per-CTA stall counters (8 x 148).
extern "C" int davo_debug_layer_timing(davo_ctx* ctx, int layer, long long* out, void* stream) {
  if (!ctx || layer < 0 || layer > 6 || !out) return DAVO_ERR_ARG;
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const int npairs = std::min(ctx->last_B * (ctx->unit_sample ? 1 : 2), ctx->mb);
  Layer& L = pick_layer(ctx, (size_t)layer, npairs);     // the plan a forward of this size runs (latency twin included)
  if (int rc = launch_conv(ctx, L, npairs, st)) return rc;
  if (int rc = launch_conv(ctx, L, npairs, st)) return rc;
  CU_OK(cudaStreamSynchronize(st));
  CU_OK(cudaMemcpyFromSymbol(out, davo::g_conv_timing, sizeof(long long) * 148 * 8));
  return 0;
}
#endif

extern "C" int davo_debug_set_conv_impl(davo_ctx* ctx, int impl) {
  if (!ctx || impl < 0 || impl > 1) return DAVO_ERR_ARG;
  ctx->conv_impl = impl;
  return 0;
}

extern "C" int davo_profile_layers(davo_ctx* ctx, int iters, float* ms_out, int* npairs_out,
                                   void* stream) {
  if (!ctx || !ms_out || iters <= 0) return DAVO_ERR_ARG;
  if (!ctx->finalized || ctx->last_npairs_mb == 0) return fail(ctx, DAVO_ERR_STATE, "davo_profile_layers: run a forward first");
  CU_OK(cudaSetDevice(ctx->device));
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const int npairs = std::min(ctx->last_B * (ctx->unit_sample ? 1 : 2), ctx->mb);
  if (npairs_out) *npairs_out = npairs;
  cudaEvent_t e0, e1;
  CU_OK(cudaEventCreate(&e0));
  CU_OK(cudaEventCreate(&e1));
  int dummy = 0;
  auto timed = [&](auto&& fn, float* ms_dst) -> int {
    if (int rc = fn()) return rc;   // warm
    CU_OK(cudaEventRecord(e0, st));
    for (int it = 0; it < iters; ++it)
      if (int rc = fn()) return rc;
    CU_OK(cudaEventRecord(e1, st));
    CU_OK(cudaEventSynchronize(e1));
    float ms = 0.f;
    CU_OK(cudaEventElapsedTime(&ms, e0, e1));
    *ms_dst = ms / iters;
    return 0;
  };
  if (int rc = timed([&] { return launch_front(ctx, ctx->unit_sample ? kUnitsAreSamples : 0, 0, npairs, ctx->last_in, st, &dummy); }, &ms_out[0])) return rc;
  for (int i = 0; i < 7; ++i) {
    const Layer& L = pick_layer(ctx, i, npairs);
    if (i == 5 && ctx->cfg.posenn_se == 3) { ms_out[1 + i] = 0.f; continue; }      // -se_replace has no cnv6 convolution
    if (int rc = timed([&] { return launch_conv(ctx, L, npairs, st); }, &ms_out[1 + i])) return rc;
  }
  if (int rc = timed([&] { return launch_head(ctx, ctx->unit_sample ? kUnitsAreSamples : 0, 0, npairs, ctx->last_pose, st, &dummy); }, &ms_out[8])) return rc;
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  return 0;
}

// ---------------------------------------------------------------------------------------------
// Pose all-gather over NCCL (SURVEY.md 8e).  Ranks hold equal, padded blocks of [n_local, 2, 6]
// poses (davo_b200/parallel.py: padded_indices); rank r's block lands at all[r * n_local].
// ---------------------------------------------------------------------------------------------
extern "C" int davo_comm_unique_id(void* id128) {
  if (!id128) return fail(nullptr, DAVO_ERR_ARG, "davo_comm_unique_id: null argument");
  const davo_comm::Api& n = davo_comm::api();
  if (!n.why.empty()) return fail(nullptr, DAVO_ERR_STATE, "davo_comm_unique_id: %s", n.why.c_str());
  davo_comm::UniqueId id;
  const int r = n.GetUniqueId(&id);
  if (r != davo_comm::kNcclSuccess) return fail(nullptr, DAVO_ERR_CUDA, "ncclGetUniqueId: %s", n.GetErrorString(r));
  std::memcpy(id128, &id, sizeof id);
  return 0;
}

extern "C" int davo_comm_create(davo_ctx* ctx, const void* id128, int rank, int world) {
  if (!ctx) return DAVO_ERR_ARG;
  if (!id128 || world < 1 || rank < 0 || rank >= world) return fail(ctx, DAVO_ERR_ARG, "davo_comm_create: bad argument (rank %d of %d)", rank, world);
  if (ctx->comm) return fail(ctx, DAVO_ERR_STATE, "davo_comm_create: the handle already has a communicator");
  const davo_comm::Api& n = davo_comm::api();
  if (!n.why.empty()) return fail(ctx, DAVO_ERR_STATE, "davo_comm_create: %s", n.why.c_str());
  CU_OK(cudaSetDevice(ctx->device));
  davo_comm::UniqueId id;
  std::memcpy(&id, id128, sizeof id);
  const int r = n.CommInitRank(&ctx->comm, world, id, rank);
  if (r != davo_comm::kNcclSuccess) {
    ctx->comm = nullptr;
    return fail(ctx, DAVO_ERR_CUDA, "ncclCommInitRank(rank %d of %d): %s", rank, world, n.GetErrorString(r));
  }
  ctx->comm_rank = rank;
  ctx->comm_world = world;
  return 0;
}

extern "C" int davo_comm_world(const davo_ctx* ctx, int* rank, int* world) {
  if (!ctx) return DAVO_ERR_ARG;
  if (rank) *rank = ctx->comm_rank;
  if (world) *world = ctx->comm ? ctx->comm_world : 1;
  return 0;
}

extern "C" int davo_allgather_poses(davo_ctx* ctx, void* nccl_comm, const float* local, int n_local,
                                    float* all, void* stream) {
  if (!ctx) return DAVO_ERR_ARG;
  if (!local || !all || n_local < 0) return fail(ctx, DAVO_ERR_ARG, "davo_allgather_poses: bad argument");
  davo_comm::Comm comm = nccl_comm ? nccl_comm : ctx->comm;
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const size_t count = static_cast<size_t>(n_local) * 2 * 6;
  if (!comm) {
    // no communicator: a world of one, the gather is a copy
    CU_OK(cudaSetDevice(ctx->device));
    if (all != local && count) CU_OK(cudaMemcpyAsync(all, local, count * sizeof(float), cudaMemcpyDeviceToDevice, st));
    return 0;
  }
  const davo_comm::Api& n = davo_comm::api();
  if (!n.why.empty()) return fail(ctx, DAVO_ERR_STATE, "davo_allgather_poses: %s", n.why.c_str());
  CU_OK(cudaSetDevice(ctx->device));
  const int r = n.AllGather(local, all, count, davo_comm::kNcclFloat, comm, st);
  if (r != davo_comm::kNcclSuccess) return fail(ctx, DAVO_ERR_CUDA, "ncclAllGather: %s", n.GetErrorString(r));
  return 0;
}

// ---------------------------------------------------------------------------------------------
// mode='feature' (davo.py:1553-1564): the pass, then the visualisation tensors (features.cuh)
// ---------------------------------------------------------------------------------------------
namespace {
// utils/flow_utils.py:546-593: six colour ramps of 15, 6, 4, 11, 13 and 6 steps; stored / 255 the way
// compute_color reads it (a float64 division cast to float32, flow_utils.py:488-490)
void middlebury_wheel(float (*wheel)[3]) {
  const int seg[6] = {15, 6, 4, 11, 13, 6};
  const int fixed[6] = {0, 1, 1, 2, 2, 0};       // channel held at 255
  const int ramp[6] = {1, 0, 2, 1, 0, 2};        // channel that moves
  const bool rising[6] = {true, false, true, false, true, false};
  int col = 0;
  for (int s = 0; s < 6; ++s)
    for (int i = 0; i < seg[s]; ++i, ++col) {
      double v[3] = {0.0, 0.0, 0.0};
      const double step = std::floor(255.0 * i / seg[s]);
      v[fixed[s]] = 255.0;
      v[ramp[s]] = rising[s] ? step : 255.0 - step;
      for (int ch = 0; ch < 3; ++ch) wheel[col][ch] = (float)(v[ch] / 255.0);
    }
}
}  // namespace

namespace {
// The output table's checks of mode='feature' on B samples (davo_forward_features, davo_forward_sequence_features).
int features_check(davo_ctx* ctx, const char* who, const char* samples, int B, const davo_features* out, bool flow, bool seg) {
  if (!out) return fail(ctx, DAVO_ERR_ARG, "%s: null output table", who);
  const int units = ctx->unit_sample ? B : 2 * B;
  if (ctx->finalized && units > ctx->mb)
    return fail(ctx, DAVO_ERR_ARG, "%s: %s needs %d units, one pass holds %d", who, samples, units, ctx->mb);
  if ((out->flow_color) && !flow) return fail(ctx, DAVO_ERR_ARG, "%s: flow colouring needs input_flow", who);
  if ((out->seg_19 || out->seg_color) && !seg) return fail(ctx, DAVO_ERR_ARG, "%s: label outputs need input_seglabel", who);
  return 0;
}

// The feature outputs of the one pass that just ran over the B samples of `in` (either layout).
int features_outputs(davo_ctx* ctx, int B, const InputView& in, const davo_features* out, void* stream) {
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const davo_config& c = ctx->cfg;
  if (!ctx->d_wheel) {
    float wheel[kWheelCols][3];
    middlebury_wheel(wheel);
    void* p = nullptr;
    CU_OK(cudaMalloc(&p, sizeof wheel + 2 * sizeof(unsigned int)));
    ctx->allocs.push_back(p);
    ctx->d_wheel = static_cast<float*>(p);
    ctx->d_maxrad = reinterpret_cast<unsigned int*>(ctx->d_wheel + kWheelCols * 3);
    CU_OK(cudaMemcpy(ctx->d_wheel, wheel, sizeof wheel, cudaMemcpyHostToDevice));
  }
  FeatureParams fp;
  memset(&fp, 0, sizeof fp);
  fp.B = B; fp.H = c.H; fp.W = c.W;
  fp.unit_sample = ctx->unit_sample ? 1 : 0; fp.att_src = c.att_src; fp.att_tgt_ones = c.att_tgt_ones;
  fp.mask_rgb = c.mask_mode != 0;
  // what frame_attention reads: the variant's flags and the flow / depth planes of this batch
  fp.fp.H = c.H; fp.fp.W = c.W; fp.fp.att_src = c.att_src; fp.fp.pixel_map = c.pixel_map; fp.fp.depth_norm = c.depth_norm;
  fp.fp.depth_split = c.depth_split; fp.fp.depth_thres = ctx->depth_thres; fp.fp.flow_abs = c.flow_abs; fp.fp.flow_norm = c.flow_norm;
  fp.fp.in = in; fp.fp.flow_f16 = c.flow_f16;
  fp.att_w = ctx->d_attw; fp.static_w = ctx->d_staticw;
  fp.wheel = ctx->d_wheel; fp.maxrad = ctx->d_maxrad;
  fp.image = out->image; fp.attention = out->attention; fp.masked_image = out->masked_image;
  fp.seg_19 = out->seg_19; fp.seg_color = out->seg_color; fp.flow_color = out->flow_color;
  int launches = ctx->last_launches;
  if (fp.image || fp.attention || fp.masked_image || fp.seg_19 || fp.seg_color) {
    const int groups = c.H * c.W / 4;
    feature_frames_kernel<<<dim3((groups + 255) / 256, B, 3), 256, 0, st>>>(fp);
    CU_OK(cudaGetLastError());
    ++launches;
  }
  if (fp.flow_color) {
    CU_OK(cudaMemsetAsync(ctx->d_maxrad, 0, 2 * sizeof(unsigned int), st));
    const int blocks = std::min(ctx->num_sms * 4, (B * c.H * c.W + 255) / 256);
    flow_maxrad_kernel<<<dim3(blocks, 2), 256, 0, st>>>(fp);
    flow_color_kernel<<<dim3(blocks, 2), 256, 0, st>>>(fp);
    CU_OK(cudaGetLastError());
    launches += 2;
  }
  if (out->cnv6_rot || out->cnv6_trans) {
    const Layer& L6 = ctx->layers[5];
    ResizeParams rp;
    rp.B = B; rp.H = c.H; rp.W = c.W;
    const bool rep = c.posenn_se == 3 || c.posenn_se == 2;   // -se_replace: "cnv6" is the excited cnv5, 256 channels per branch;
                                                             // -se_skipadd: relu(cnv5 + se_block(cnv6)), same buffer and geometry
    rp.h = rep ? L6.Hin : L6.Hout; rp.w = rep ? L6.Win : L6.Wout; rp.hp = rep ? L6.Hin_p : L6.Hout_p; rp.wp = rep ? L6.Win_p : L6.Wout_p;
    rp.C = rep ? 256 : c.cnv6_out; rp.cstride = rep ? ctx->nbr * 256 : L6.out_stride;
    rp.unit_mul = ctx->unit_sample ? 1 : 2; rp.unit_add = ctx->unit_sample ? 0 : 1;
    rp.src = rep ? ctx->d_se5out : L6.d_out;
    const size_t total = (size_t)B * c.H * c.W * (rp.C / 4);
    const int blocks = (int)std::min<size_t>((size_t)ctx->num_sms * 8, (total + 255) / 256);
    float* dsts[2] = {out->cnv6_rot, out->cnv6_trans};
    for (int br = 0; br < 2; ++br) {
      if (!dsts[br]) continue;
      rp.coff = (ctx->nbr == 2 && br == 1) ? rp.C : 0;            // couple nets return (cnv6, cnv6), posenn.py:66, 187, 311
      rp.dst = dsts[br];
      resize_bilinear_kernel<<<blocks, 256, 0, st>>>(rp);
      CU_OK(cudaGetLastError());
      ++launches;
    }
  }
  ctx->last_launches = launches;
  return 0;
}
}  // namespace

extern "C" int davo_forward_features(davo_ctx* ctx, int B, const uint8_t* img, const float* flow,
                                     const float* seg, const float* depth, float* pose_out,
                                     const davo_features* out, void* stream) {
  if (!ctx) return DAVO_ERR_ARG;
  char samples[32];
  snprintf(samples, sizeof samples, "B=%d", B);
  if (int rc = features_check(ctx, "davo_forward_features", samples, B, out, flow != nullptr, seg != nullptr)) return rc;
  if (int rc = davo_forward_pairs(ctx, B, DAVO_PAIRS_ALL, img, flow, seg, depth, pose_out, stream)) return rc;
  return features_outputs(ctx, B, triplet_view(ctx->cfg.H, ctx->cfg.W, img, flow, seg, nullptr, depth, nullptr, 0), out, stream);
}

extern "C" int davo_forward_sequence_features(davo_ctx* ctx, int n_frames, const uint8_t* img, const float* flow_fwd,
                                              const float* flow_bwd, const float* seg, const float* depth, float* pose_out,
                                              const davo_features* out, void* stream) {
  if (!ctx) return DAVO_ERR_ARG;
  const char* who = "davo_forward_sequence_features";
  if (int rc = check_sequence(ctx, who, n_frames, DAVO_PAIRS_ALL, img, flow_fwd, flow_bwd, seg, depth, pose_out)) return rc;
  const int B = n_frames - 2;
  char samples[64];
  snprintf(samples, sizeof samples, "n_frames=%d (B=%d samples)", n_frames, B);
  if (int rc = features_check(ctx, who, samples, B, out, flow_fwd && flow_bwd, seg != nullptr)) return rc;
  const InputView in = sequence_device_view(ctx, img, flow_fwd, flow_bwd, seg, depth);
  if (int rc = forward_device(ctx, who, B, DAVO_PAIRS_ALL, in, pose_out, stream)) return rc;
  return features_outputs(ctx, B, in, out, stream);
}

// Test hook (no GPU needed): the CPU float32 -> binary16 conversion of the host entry point.
// ---- on-device trajectory composition and KITTI evaluation (include/davo_b200.h; csrc/trajectory.cuh) ----
static int traj_scratch(davo_ctx* ctx, size_t bytes) {
  if (ctx->traj_scratch_bytes >= bytes) return 0;
  if (ctx->d_traj_scratch) cudaFree(ctx->d_traj_scratch);
  ctx->d_traj_scratch = nullptr; ctx->traj_scratch_bytes = 0;
  CU_OK(cudaMalloc(&ctx->d_traj_scratch, bytes));
  ctx->traj_scratch_bytes = bytes;
  return 0;
}

extern "C" int davo_compose_trajectory(davo_ctx* ctx, const float* poses, int n, double* traj, void* stream) {
  if (!ctx) return DAVO_ERR_ARG;
  if (!poses || !traj || n < 1) return fail(ctx, DAVO_ERR_ARG, "davo_compose_trajectory: null buffer or no samples");
  CU_OK(cudaSetDevice(ctx->device));
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const int m = n + 1;                                   // relative motions
  if (int rc = traj_scratch(ctx, (size_t)m * sizeof(Mat4))) return rc;
  Mat4* rel = reinterpret_cast<Mat4*>(ctx->d_traj_scratch);
  pose_rel_kernel<<<(m + 127) / 128, 128, 0, st>>>(poses, n, rel);
  CU_OK(cudaGetLastError());
  const int threads = 256, chunk = (m + threads - 1) / threads;
  traj_scan_kernel<<<1, threads, threads * 16 * sizeof(double), st>>>(rel, m, chunk, reinterpret_cast<Mat4*>(traj));
  CU_OK(cudaGetLastError());
  return 0;
}

extern "C" int davo_kitti_errors(davo_ctx* ctx, const double* gt, const double* res, int n, davo_kitti_segment* seg,
                                 float* stats_host, void* stream) {
  if (!ctx) return DAVO_ERR_ARG;
  if (!gt || !res || n < 1 || !stats_host) return fail(ctx, DAVO_ERR_ARG, "davo_kitti_errors: null buffer or no frames");
  static_assert(sizeof(davo_kitti_segment) == sizeof(KittiSeg), "segment layouts differ");
  CU_OK(cudaSetDevice(ctx->device));
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const int n_first = (n + kKittiStep - 1) / kKittiStep, count = n_first * kKittiLengths;
  const size_t off_seg = ((size_t)n * sizeof(float) + 255) & ~(size_t)255, off_stats = off_seg + (size_t)count * sizeof(KittiSeg);
  if (int rc = traj_scratch(ctx, off_stats + 64)) return rc;
  uint8_t* base = reinterpret_cast<uint8_t*>(ctx->d_traj_scratch);
  float* dist = reinterpret_cast<float*>(base);
  KittiSeg* segs = seg ? reinterpret_cast<KittiSeg*>(seg) : reinterpret_cast<KittiSeg*>(base + off_seg);
  float* stats = reinterpret_cast<float*>(base + off_stats);
  kitti_dist_kernel<<<1, 32, 0, st>>>(reinterpret_cast<const Mat4*>(gt), n, dist);
  kitti_segments_kernel<<<(count + 127) / 128, 128, 0, st>>>(reinterpret_cast<const Mat4*>(gt), reinterpret_cast<const Mat4*>(res), dist, n, n_first, segs);
  kitti_stats_kernel<<<1, 32, 0, st>>>(segs, count, stats);
  CU_OK(cudaGetLastError());
  CU_OK(cudaMemcpyAsync(stats_host, stats, 3 * sizeof(float), cudaMemcpyDeviceToHost, st));
  CU_OK(cudaStreamSynchronize(st));
  return 0;
}

// ---- nvJPEG decode into the frame tensor (include/davo_b200.h; csrc/jpeg.cuh) ----
extern "C" int davo_decode_jpeg_batch(davo_ctx* ctx, const uint8_t* const* jpeg, const int64_t* nbytes, int n, uint8_t* img_dev,
                                      void* stream) {
  if (!ctx) return DAVO_ERR_ARG;
  if (!jpeg || !nbytes || !img_dev || n < 1) return fail(ctx, DAVO_ERR_ARG, "davo_decode_jpeg_batch: null buffer or no images");
  const davo_jpeg::Api& j = davo_jpeg::api();
  if (!j.why.empty()) return fail(ctx, DAVO_ERR_STATE, "davo_decode_jpeg_batch: %s", j.why.c_str());
  CU_OK(cudaSetDevice(ctx->device));
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  if (!ctx->jpeg_handle) {
    if (j.CreateSimple(&ctx->jpeg_handle) != NVJPEG_STATUS_SUCCESS) return fail(ctx, DAVO_ERR_CUDA, "nvjpegCreateSimple failed");
    if (j.StateCreate(ctx->jpeg_handle, &ctx->jpeg_state) != NVJPEG_STATUS_SUCCESS) return fail(ctx, DAVO_ERR_CUDA, "nvjpegJpegStateCreate failed");
  }
  const int H = ctx->cfg.H, W3 = 3 * ctx->cfg.W;
  for (int i = 0; i < n; ++i) {
    int comps = 0, ws[NVJPEG_MAX_COMPONENT], hs[NVJPEG_MAX_COMPONENT];
    nvjpegChromaSubsampling_t sub;
    if (j.GetImageInfo(ctx->jpeg_handle, jpeg[i], (size_t)nbytes[i], &comps, &sub, ws, hs) != NVJPEG_STATUS_SUCCESS)
      return fail(ctx, DAVO_ERR_ARG, "davo_decode_jpeg_batch: image %d is not a JPEG nvJPEG can parse", i);
    if (ws[0] != W3 || hs[0] != H)
      return fail(ctx, DAVO_ERR_ARG, "davo_decode_jpeg_batch: image %d is %dx%d, the frame triple must be %dx%d", i, hs[0], ws[0], H, W3);
    nvjpegImage_t out;
    memset(&out, 0, sizeof out);
    out.channel[0] = img_dev + (size_t)i * H * W3 * 3;
    out.pitch[0] = (size_t)W3 * 3;
    const nvjpegStatus_t rc = j.Decode(ctx->jpeg_handle, ctx->jpeg_state, jpeg[i], (size_t)nbytes[i], NVJPEG_OUTPUT_RGBI, &out, st);
    if (rc != NVJPEG_STATUS_SUCCESS) return fail(ctx, DAVO_ERR_CUDA, "nvjpegDecode(image %d) -> %d", i, (int)rc);
  }
  CU_OK(cudaStreamSynchronize(st));
  return 0;
}

extern "C" int davo_debug_labels_to_bytes(const float* src, uint8_t* dst, long long n, int portable) {
  if (!src || !dst || n < 0) return DAVO_ERR_ARG;
  if (portable) davo_host::labels_to_bytes_portable(src, dst, (size_t)n);
  else davo_host::labels_to_bytes(src, dst, (size_t)n);
  return 0;
}

extern "C" int davo_debug_flows_to_half(const float* src, uint16_t* dst, long long n, int portable) {
  if (!src || !dst || n < 0) return DAVO_ERR_ARG;
  const bool ok = portable ? davo_host::flows_to_half_portable(src, dst, (size_t)n) : davo_host::flows_to_half(src, dst, (size_t)n);
  return ok ? 0 : 1;
}
