// libb200sac: C-ABI implementation (see include/b200sac.h) -- host orchestration of the
// sm_100a SAC gradient step.  One handle = R independent learners of one shape stepped
// together; one step = a fixed list of grouped launches captured once into a CUDA graph.
#include <cuda_runtime.h>
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <functional>
#include <map>
#include <mutex>
#include <new>
#include <random>
#include <string>
#include <tuple>
#include <unordered_set>
#include <vector>

#include "../../include/b200sac.h"
#include "gemm_simt.cuh"
#include "gemm_thin.cuh"
#include "gemm_tc.cuh"
#include "sac_kernels.cuh"
#include "care_kernels.cuh"
#include "chain.cuh"
#include "chain2.cuh"

using namespace bsac;

// ------------------------------------------------------------------------------------------
// errors
// ------------------------------------------------------------------------------------------
static thread_local char g_err[512] = "";
static int fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}
#define CU(call)                                                                                     \
  do {                                                                                               \
    cudaError_t e__ = (call);                                                                        \
    if (e__ != cudaSuccess)                                                                          \
      return fail(B200SAC_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e__), __FILE__, __LINE__); \
  } while (0)

extern "C" const char* b200sac_last_error(void) { return g_err; }
extern "C" const char* b200sac_version(void) { return "b200sac 0.1 (sm_100a)"; }

// ------------------------------------------------------------------------------------------
// layout
// ------------------------------------------------------------------------------------------
struct LayerOff { int64_t w, b; int in, out; int ld; };   // ld = row pitch of the weight matrix (>= in)
struct Layout {
  std::vector<b200sac_tensor_desc> descs;
  std::vector<LayerOff> actor, q[2], qt[2];
  // CARE: the critic's state encoder (the target's sits at + target_delta with the same relative layout)
  std::vector<LayerOff> mix, trunk, ctx;      // mix: w = [K][out][in], b = [K][out]
  std::vector<LayerOff> cenc;                 // CARE(O): the trainable context encoder (header + mlp), no target copy
  int64_t cse_begin = 0, off_emb = 0, cenc_begin = 0, cenc_n = 0;
  int in_w = 0;                               // width of the state part of the MLP inputs
  int64_t off_alpha = 0, arena = 0, trainable = 0;
  int64_t actor_begin = 0, actor_n = 0, critic_begin = 0, critic_n = 0, target_delta = 0;
};

static int64_t pad4(int64_t x) { return (x + 3) & ~int64_t(3); }

static int check_cfg(const b200sac_cfg* c) {
  if (!c) return fail(B200SAC_ERR_INVALID, "cfg is NULL");
  if (c->state_dim < 1 || c->act_dim < 1 || c->act_dim > kMaxAct)
    return fail(B200SAC_ERR_INVALID, "state_dim >= 1 and 1 <= act_dim <= %d required", kMaxAct);
  if (c->num_tasks < 0 || c->num_tasks > 64) return fail(B200SAC_ERR_INVALID, "0 <= num_tasks <= 64 required");
  if (c->n_actor_hidden < 1 || c->n_actor_hidden > B200SAC_MAX_HIDDEN || c->n_critic_hidden < 1 ||
      c->n_critic_hidden > B200SAC_MAX_HIDDEN)
    return fail(B200SAC_ERR_INVALID, "1..%d hidden layers required", B200SAC_MAX_HIDDEN);
  for (int i = 0; i < c->n_actor_hidden; ++i)
    if (c->actor_hidden[i] < 1) return fail(B200SAC_ERR_INVALID, "actor_hidden[%d] < 1", i);
  for (int i = 0; i < c->n_critic_hidden; ++i)
    if (c->critic_hidden[i] < 1) return fail(B200SAC_ERR_INVALID, "critic_hidden[%d] < 1", i);
  if (c->batch < 1 || c->batch > 2048) return fail(B200SAC_ERR_INVALID, "1 <= batch <= 2048 required");
  if (c->num_tasks > 0 && c->batch % c->num_tasks != 0)
    return fail(B200SAC_ERR_INVALID, "batch must be a multiple of num_tasks");
  if (c->replicas < 1 || c->replicas > 4096) return fail(B200SAC_ERR_INVALID, "1 <= replicas <= 4096 required");
  if (c->precision != 0 && c->precision != 1) return fail(B200SAC_ERR_INVALID, "precision must be 0 (fp32 FFMA) or 1 (3xTF32 tcgen05)");
  if (c->care != 0 && c->care != 1 && c->care != 2) return fail(B200SAC_ERR_INVALID, "care must be 0, 1 (CARE(M)) or 2 (CARE(O))");
  if (c->care == 2) {
    if (c->emb_dim < 1 || c->emb_dim > 256) return fail(B200SAC_ERR_INVALID, "1 <= emb_dim <= 256 required for CARE(O)");
    if (c->emb_dim != c->ctx_out)
      return fail(B200SAC_ERR_INVALID, "CARE(O): the attention trunk reads the context code, so embedding_dim_contextEnc (%d) must equal output_dim_contextEnc (%d) (state_encoder.py:120-122)", c->emb_dim, c->ctx_out);
    if (c->n_ctx_hidden + 3 > kCareMaxLayers) return fail(B200SAC_ERR_INVALID, "too many context-encoder layers");
  }
  if (c->care) {
    if (c->num_tasks < 1) return fail(B200SAC_ERR_INVALID, "CARE needs num_tasks >= 1 (one-hot task id in the observation)");
    if (c->num_encoders < 1 || c->num_encoders > 32) return fail(B200SAC_ERR_INVALID, "1 <= num_encoders <= 32 required");
    if (c->n_mix_hidden < 1 || c->n_mix_hidden > B200SAC_MAX_HIDDEN || c->n_ctx_hidden < 0 || c->n_ctx_hidden > B200SAC_MAX_HIDDEN)
      return fail(B200SAC_ERR_INVALID, "bad number of encoder hidden layers");
    if (c->mix_out < 1 || c->mix_out > 512 || c->ctx_out < 1 || c->ctx_out > 512 || c->ctx_in < 1 || c->ctx_in > 2048)
      return fail(B200SAC_ERR_INVALID, "encoder widths out of range (mix_out, ctx_out <= 512, ctx_in <= 2048)");
    for (int i = 0; i < c->n_mix_hidden; ++i)
      if (c->mix_hidden[i] < 1 || c->mix_hidden[i] > 512) return fail(B200SAC_ERR_INVALID, "mix_hidden[%d] out of range", i);
    for (int i = 0; i < c->n_ctx_hidden; ++i)
      if (c->ctx_hidden[i] < 1 || c->ctx_hidden[i] > 512) return fail(B200SAC_ERR_INVALID, "ctx_hidden[%d] out of range", i);
    if (c->num_encoders + c->ctx_out > 64 * 8) return fail(B200SAC_ERR_INVALID, "num_encoders + ctx_out too large");
  }
  return 0;
}

static void build_layout(const b200sac_cfg* c, Layout& L) {
  const int obs = c->state_dim + c->num_tasks;
  L.in_w = c->care ? (c->ctx_out + c->mix_out) : obs;
  int64_t off = 0;
  auto add = [&](const char* name, int rows, int cols, int trainable, int opt, int pitch = 0) {
    b200sac_tensor_desc d;
    memset(&d, 0, sizeof(d));
    snprintf(d.name, sizeof(d.name), "%s", name);
    if (pitch < cols) pitch = cols;
    d.offset = off; d.rows = rows; d.cols = cols; d.trainable = trainable; d.opt = opt; d.pitch = pitch;
    L.descs.push_back(d);
    int64_t o = off;
    off = pad4(off + (int64_t)rows * pitch);
    return o;
  };
  char nm[48];
  auto add_net = [&](const char* net, std::vector<LayerOff>* v, int in0, const int* hid, int nh, int out, int tr, int opt,
                     bool pad_first = false) {
    int in = in0;
    for (int i = 0; i <= nh; ++i) {
      int o = (i < nh) ? hid[i] : out;
      LayerOff lo;
      lo.in = in; lo.out = o;
      lo.ld = (i == 0 && pad_first) ? (int)pad4(in) : in;     // first layer: TMA-addressable rows (16-B pitch)
      snprintf(nm, sizeof(nm), "%s.%d.weight", net, i);
      lo.w = add(nm, o, in, tr, opt, lo.ld);
      snprintf(nm, sizeof(nm), "%s.%d.bias", net, i);
      lo.b = add(nm, o, 1, tr, opt);
      if (v) v->push_back(lo);
      in = o;
    }
  };
  // state encoder block: mixture layers ([K][out][in] | [K][out]), attention trunk, context MLP
  auto add_encoder = [&](const char* pre, bool record, int tr, int opt) {
    int in = c->state_dim;
    for (int l = 0; l <= c->n_mix_hidden; ++l) {
      int o = (l < c->n_mix_hidden) ? c->mix_hidden[l] : c->mix_out;
      LayerOff lo;
      lo.in = in; lo.out = o; lo.ld = in;
      snprintf(nm, sizeof(nm), "%s.mix.%d.W", pre, l);
      lo.w = add(nm, c->num_encoders * o, in, tr, opt);
      snprintf(nm, sizeof(nm), "%s.mix.%d.b", pre, l);
      lo.b = add(nm, c->num_encoders * o, 1, tr, opt);
      if (record) L.mix.push_back(lo);
      in = o;
    }
    char pfx[24];
    snprintf(pfx, sizeof(pfx), "%s.trunk", pre);
    add_net(pfx, record ? &L.trunk : nullptr, c->care == 2 ? c->emb_dim : c->ctx_in, c->mix_hidden, c->n_mix_hidden,
            c->num_encoders, tr, opt);
    if (c->care == 1) {          // CARE(M): mlp_context lives inside every state encoder
      snprintf(pfx, sizeof(pfx), "%s.ctx", pre);
      add_net(pfx, record ? &L.ctx : nullptr, c->ctx_in, c->ctx_hidden, c->n_ctx_hidden, c->ctx_out, tr, opt);
    }
  };
  L.actor_begin = off;
  add_net("actor", &L.actor, L.in_w, c->actor_hidden, c->n_actor_hidden, 2 * c->act_dim, 1, 1, true);
  L.actor_n = off - L.actor_begin;
  L.critic_begin = off;
  add_net("q1", &L.q[0], L.in_w + c->act_dim, c->critic_hidden, c->n_critic_hidden, 1, 1, 0, true);
  add_net("q2", &L.q[1], L.in_w + c->act_dim, c->critic_hidden, c->n_critic_hidden, 1, 1, 0, true);
  L.cse_begin = off;
  if (c->care) add_encoder("cse", true, 1, 0);
  L.critic_n = off - L.critic_begin;
  L.off_alpha = add("log_alpha", c->num_tasks > 0 ? c->num_tasks : 1, 1, 1, 2);
  if (c->care == 2) {            // context encoder: Linear(ctx_in, 2e) ReLU Linear(2e, e) ReLU + mlp e -> ctx_hidden -> ctx_out
    L.cenc_begin = off;
    int hid[B200SAC_MAX_HIDDEN + 2];
    int nh = 0;
    hid[nh++] = 2 * c->emb_dim;
    hid[nh++] = c->emb_dim;
    for (int i = 0; i < c->n_ctx_hidden; ++i) hid[nh++] = c->ctx_hidden[i];
    add_net("cenc", &L.cenc, c->ctx_in, hid, nh, c->ctx_out, 1, 3);
    L.cenc_n = off - L.cenc_begin;
  }
  L.trainable = off;
  int64_t tb = off;
  add_net("q1_target", &L.qt[0], L.in_w + c->act_dim, c->critic_hidden, c->n_critic_hidden, 1, 0, -1, true);
  add_net("q2_target", &L.qt[1], L.in_w + c->act_dim, c->critic_hidden, c->n_critic_hidden, 1, 0, -1, true);
  if (c->care) add_encoder("tse", false, 0, -1);
  L.target_delta = tb - L.critic_begin;
  if (c->care) L.off_emb = add("embedding", c->num_tasks, c->ctx_in, 0, -1);
  L.arena = off;
}

extern "C" int b200sac_layout(const b200sac_cfg* cfg, b200sac_tensor_desc* out, int32_t cap, int32_t* n,
                              int64_t* arena_floats, int64_t* trainable_floats) {
  if (int rc = check_cfg(cfg)) return rc;
  Layout L;
  build_layout(cfg, L);
  if (n) *n = (int32_t)L.descs.size();
  if (arena_floats) *arena_floats = L.arena;
  if (trainable_floats) *trainable_floats = L.trainable;
  if (out)
    for (int i = 0; i < (int)L.descs.size() && i < cap; ++i) out[i] = L.descs[i];
  return 0;
}

// ------------------------------------------------------------------------------------------
// handle
// ------------------------------------------------------------------------------------------
struct Buf {           // [R][n] fp32 (or int32) slab slice
  float* p = nullptr;
  long long rs = 0;    // replica stride in floats
};

enum LaunchKind { L_POLICY_DOUT, L_CARE_TAB, L_CARE_MIXFWD, L_CARE_MIX, L_CARE_MIXBWD, L_CARE_TABRED, L_CARE_TABWG, L_GEMM_BIG, L_GEMM_SMALL, L_GEMM_THIN, L_GEMM_TC, L_POLICY, L_CHEADS, L_AQHEADS, L_HEADBWD, L_ADAM, L_CHAIN, L_WGRAD, L_CHAIN2 };

struct Launch {
  LaunchKind kind;
  dim3 grid, block;
  size_t smem = 0;
  int branch = 0;        // 1: may run on the fork stream, concurrently with the launches that follow it on the main stream
  bool join = false;     // the main stream waits for the fork stream before this launch
  // payloads (only the one matching `kind` is used)
  const GemmProb* probs = nullptr; int G = 0;
  GemmGroup grp;
  const TcProb* tprobs = nullptr;
  int bn = 64;
  PolicyDoutArgs pdo;
  CareTabArgs ctab;
  CareMixArgs cmix;
  CareMixFwdArgs cmf;
  CareMixBwdArgs cmixb;
  CareTabReduceArgs ctred;
  CareTabWgradArgs ctwg;
  PolicyHeadArgs pol;
  CriticHeadArgs ch;
  ActorQHeadArgs aq;
  HeadBwdArgs hb;
  AdamArgs ad;
  ChainArgs chain;
  Chain2Args chain2;
  WgradArgs wg;
  const char* label = nullptr;
};

struct GraphKey {
  int variant;
  const void* p[9];
  bool operator<(const GraphKey& o) const {
    if (variant != o.variant) return variant < o.variant;
    return memcmp(p, o.p, sizeof(p)) < 0;
  }
};

struct b200sac_replay;

struct b200sac {
  b200sac_cfg cfg;
  int device = 0;
  Layout L;
  StepConst K;
  int R = 1;
  // arenas
  float *params = nullptr, *adam_m = nullptr, *adam_v = nullptr, *grads = nullptr;
  Counters* cnt = nullptr;
  float* losses = nullptr;        // [kLossSlots][R][4]
  long long host_steps = 0;       // steps enqueued so far
  // work slab
  float* slab = nullptr;
  size_t slab_floats = 0;
  Buf XA, XQ, XT, XP, r, d, tid, eps, pout, psave, act_out, logp, logstd, y, q, dq, lq, dqa, la, qmin, dxP,
      dout_dbg, dact_dbg, qt, qp, alpha;
  bool stamping = false;          // true while b200sac_graph_timeline runs on this handle (one unforked step per graph)
  bool fused = false;             // layer-chained plan (chain.cuh): every hidden width <= 256, exact-fp32 mode, no CARE
  PolicyHeadArgs pol;             // the policy head's arguments (also used by b200sac_act)
  // CARE
  Buf XS, careTab[3], careDtab, careDatt, mixZ[3], mixDZ;     // instances: 0 = critic's (old) on [s';s], 1 = target's on s', 2 = critic's (new) on s
  std::vector<Buf> mixH[3], mixDH;                             // per mixture hidden layer: [K][rows][pitch]
  CareNet care_trunk, care_ctx;
  int care_row_w = 0, care_off_att = 0, care_off_ctx = 0;
  std::vector<Buf> hA, dhA;       // per actor hidden layer
  std::vector<Buf> hQ, hT, hP, dhQ;   // per critic hidden layer, [2][B][H]
  GemmProb* d_probs = nullptr;
  std::vector<GemmProb> h_probs;
  TcProb* d_tprobs = nullptr;
  std::vector<TcProb> h_tprobs;
  std::vector<Launch> plan;
  IngestOut ing;
  int use_eps_buf_idx = -1;       // index of the policy launch in plan (its use_eps_buf flag varies)
  // split-K weight gradients: slices 1..gslices-1 of the gradient arena, [slice-1][R][trainable] (slice 0 = grads)
  float* grads_x = nullptr;
  int gslices = 1;
  unsigned long long act_calls = 0;     // b200sac_act invocations (noise stream selector)
  // graphs
  std::map<GraphKey, cudaGraphExec_t> graphs;
  // host staging for step_host / pinned replay
  float* stage_h[2] = {nullptr, nullptr};
  float* stage_d[2] = {nullptr, nullptr};
  size_t stage_floats = 0;
  int row_w = 0, row_stride = 0;
  cudaStream_t side = nullptr;
  cudaStream_t fork = nullptr;    // capture-time fork for the next step's index sampling (multi-step graphs)
  cudaEvent_t ev_ingested = nullptr, ev_sampled = nullptr, ev_fork_src = nullptr, ev_fork_done = nullptr;
  cudaStream_t own = nullptr;     // used when the caller hands us the legacy default stream (not capturable)
  cudaEvent_t ev_in = nullptr, ev_out = nullptr;
  cudaEvent_t ev_copied[2] = {nullptr, nullptr}, ev_consumed[2] = {nullptr, nullptr};
  int stage_slot = 0;
  bool stage_used[2] = {false, false};
  int prefetch_slot = -1;         // host-ring step_sampled: minibatch already drawn, gathered and in flight (H2D)
  b200sac_replay* prefetch_rb = nullptr;
  // publication path (b200sac_publish_*): device snapshot -> pinned host, on its own stream
  // two snapshot slots: the caller may build the published blob from snapshot k while snapshot k+1 (begun after the next
  // step was enqueued) is still landing
  cudaStream_t pub = nullptr;
  cudaEvent_t ev_pub_snap[2] = {nullptr, nullptr}, ev_pub_done[2] = {nullptr, nullptr};
  float* pub_d[2] = {nullptr, nullptr};   // device snapshots (consistent: taken in stream order between two steps)
  float* pub_h[2] = {nullptr, nullptr};   // pinned host copies handed to the caller
  int64_t pub_cap = 0, pub_n[2] = {0, 0};
  int pub_head = 0, pub_pending = 0;      // next slot to fill; snapshots begun and not yet collected (<= 2)
  // blob publication (b200sac_blob_*): the published byte string is assembled ON THE DEVICE (constant bytes + float payloads
  // gathered from the arena by a kernel) and crosses PCIe as one copy; the host never touches individual tensors
  uint8_t* blob_d[2] = {nullptr, nullptr};
  uint8_t* blob_h[2] = {nullptr, nullptr};
  int* blob_src = nullptr;                // [blob_nf] arena index of payload float j
  int* blob_dst = nullptr;                // [blob_nf] byte offset of payload float j inside the image
  int64_t blob_bytes = 0, blob_nf = 0;
  int blob_replica = 0, blob_head = 0, blob_pending = 0;
  cudaEvent_t ev_blob_snap[2] = {nullptr, nullptr}, ev_blob_done[2] = {nullptr, nullptr};
  CUtensorMap* d_wmaps = nullptr; // layer-chained plan: 2-D maps of the weight-gradient operands, [R][maps per learner]
  CUtensorMap* d_cmaps = nullptr; // layer-chained plan: 2-D tensor maps of the forward weight matrices, [R][maps per learner]
  long long* chain_dbg = nullptr; // B200SAC_CHAIN_DBG=1: [plan launches][CH_DBG_SLOTS] clock64 timelines of the chain kernels
  float* split_d = nullptr;       // b200sac_step: handle-owned copy of the caller's minibatch arrays (stable graph pointers)
  float* loss_h = nullptr;        // mapped pinned loss ring [kLossSlots][R][4], written by the tail kernels
  float* loss_h_dev = nullptr;    // its device-side address
};

struct b200sac_replay {
  b200sac* h = nullptr;
  int where = 0;
  long long cap = 0, cap_per_task = 0;
  int Teff = 1;
  float* rows = nullptr;          // [R][cap][row_stride] device or pinned host
  long long rs_rows = 0;
  std::vector<long long> fill, head;   // [R][Teff]
  long long* d_fill = nullptr;    // device copy (device ring)
  int* d_idx = nullptr;           // [R][B]
  unsigned long long seed = 0;
  std::mt19937_64 rng;
  std::mutex mu;
  cudaEvent_t ev_gather = nullptr;   // device ring: recorded after the last enqueued gather (pushes wait for it under `mu`)
  bool gather_pending = false;
};

static size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

static Buf carve(size_t& cursor, size_t n_per_rep, int R) {
  Buf b;
  size_t n = align_up(n_per_rep, 64);
  b.rs = (long long)n;
  b.p = (float*)(uintptr_t)(cursor * sizeof(float));   // offset for now; rebased after allocation
  cursor += n * (size_t)R;
  return b;
}

static void rebase(Buf& b, float* base) { b.p = base + (size_t)(uintptr_t)b.p / sizeof(float); }

static int destroy_impl(b200sac* h) {
  if (!h) return 0;
  cudaSetDevice(h->device);
  for (auto& kv : h->graphs) cudaGraphExecDestroy(kv.second);
  cudaFree(h->params); cudaFree(h->adam_m); cudaFree(h->adam_v); cudaFree(h->grads); cudaFree(h->grads_x);
  cudaFree(h->cnt); cudaFree(h->losses); cudaFree(h->slab); cudaFree(h->d_probs); cudaFree(h->d_tprobs);
  for (int i = 0; i < 2; ++i) {
    if (h->stage_h[i]) cudaFreeHost(h->stage_h[i]);
    cudaFree(h->stage_d[i]);
    if (h->ev_copied[i]) cudaEventDestroy(h->ev_copied[i]);
    if (h->ev_consumed[i]) cudaEventDestroy(h->ev_consumed[i]);
  }
  if (h->loss_h) cudaFreeHost(h->loss_h);
  if (h->pub) { cudaStreamSynchronize(h->pub); cudaStreamDestroy(h->pub); }
  for (int i = 0; i < 2; ++i) {
    if (h->ev_pub_snap[i]) cudaEventDestroy(h->ev_pub_snap[i]);
    if (h->ev_pub_done[i]) cudaEventDestroy(h->ev_pub_done[i]);
    cudaFree(h->pub_d[i]);
    if (h->pub_h[i]) cudaFreeHost(h->pub_h[i]);
    if (h->ev_blob_snap[i]) cudaEventDestroy(h->ev_blob_snap[i]);
    if (h->ev_blob_done[i]) cudaEventDestroy(h->ev_blob_done[i]);
    cudaFree(h->blob_d[i]);
    if (h->blob_h[i]) cudaFreeHost(h->blob_h[i]);
  }
  cudaFree(h->blob_src);
  cudaFree(h->blob_dst);
  cudaFree(h->split_d);
  cudaFree(h->chain_dbg);
  cudaFree(h->d_cmaps);
  cudaFree(h->d_wmaps);
  if (h->side) cudaStreamDestroy(h->side);
  if (h->fork) cudaStreamDestroy(h->fork);
  if (h->ev_ingested) cudaEventDestroy(h->ev_ingested);
  if (h->ev_sampled) cudaEventDestroy(h->ev_sampled);
  if (h->ev_fork_src) cudaEventDestroy(h->ev_fork_src);
  if (h->ev_fork_done) cudaEventDestroy(h->ev_fork_done);
  if (h->own) cudaStreamDestroy(h->own);
  if (h->ev_in) cudaEventDestroy(h->ev_in);
  if (h->ev_out) cudaEventDestroy(h->ev_out);
  delete h;
  return 0;
}

// ---- TMA tensor maps (driver entry point resolved at run time: no link-time libcuda dependency) ----
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn get_encode_tiled() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
      fn = (EncodeTiledFn)p;
  }
  return fn;
}

// 2-D fp32 row-major [outer][inner] (pitch in floats), box {32 floats = 128 B, box_outer rows}, SWIZZLE_128B, zero OOB fill
static int make_map(CUtensorMap* tm, const float* ptr, long long inner, long long outer, long long pitch, int box_outer,
                    bool mn_major = false, bool dense = false) {
  EncodeTiledFn enc = get_encode_tiled();
  if (!enc) return fail(B200SAC_ERR_CUDA, "cuTensorMapEncodeTiled not available from the driver");
  cuuint64_t dims[2] = {(cuuint64_t)inner, (cuuint64_t)outer};
  cuuint64_t strides[1] = {(cuuint64_t)pitch * sizeof(float)};
  cuuint32_t box[2] = {32u, (cuuint32_t)box_outer};
  cuuint32_t estr[2] = {1u, 1u};
  CUresult r = enc(tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, (void*)ptr, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   dense ? CU_TENSOR_MAP_SWIZZLE_NONE : (mn_major ? CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B : CU_TENSOR_MAP_SWIZZLE_128B),
                   CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(B200SAC_ERR_CUDA, "cuTensorMapEncodeTiled failed (%d) inner=%lld outer=%lld pitch=%lld", (int)r, inner, outer, pitch);
  return 0;
}

static bool tc_eligible(const GemmProb& p) {
  auto al16 = [](const void* q) { return ((uintptr_t)q & 15) == 0; };
  if (p.lda % 4 || p.ldb % 4 || !al16(p.A) || !al16(p.B) || (p.rsA % 4) || (p.rsB % 4)) return false;
  return p.M >= 32 && p.N >= 32 && p.K >= 32;
}

// Tile variants of the tcgen05 GEMM (gemm_tc.cuh): 128x64 paired, 128x128 unpaired / paired (N = 256 MMAs), 128x160.
typedef void (*TcKernel)(const TcProb*);
static bool tc_pair128() { const char* e = getenv("B200SAC_TC_PAIR128"); return !(e && e[0] == '0'); }
static TcKernel tc_kernel(int bn) {
  if (bn == 160) return gemm_tc_kernel<160, false>;
  if (bn == 128) return tc_pair128() ? (TcKernel)gemm_tc_kernel<128, true> : (TcKernel)gemm_tc_kernel<128, false>;
  return gemm_tc_kernel<64, true>;
}
static size_t tc_smem(int bn) {
  return bn == 160 ? TcCfg<160, false>::kSmemBytes : (bn == 128 ? TcCfg<128, false>::kSmemBytes : TcCfg<64, true>::kSmemBytes);
}
static cudaError_t tc_set_attrs() {
  cudaError_t e = cudaFuncSetAttribute(gemm_tc_kernel<64, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, TcCfg<64, true>::kSmemBytes);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(gemm_tc_kernel<128, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, TcCfg<128, false>::kSmemBytes);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(gemm_tc_kernel<128, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, TcCfg<128, true>::kSmemBytes);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(gemm_tc_kernel<160, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, TcCfg<160, false>::kSmemBytes);
  return e;
}
// Modelled cycles of one launch group with `bn`-wide tiles (measured constants, scripts/tc_timeline.py): a tile costs a
// ~2.5k-cycle prologue, 4 k steps per 32-wide k chunk at 210 (64, paired) / 276 (128, paired) / 315 (128) / 366 (160)
// cycles of MMA issue each, and ~1.5k cycles of epilogue per pair of 32-column blocks; tiles beyond 148 x R wait for a
// second wave.  The plan builder takes the cheapest width.
static double tc_group_cost(const std::vector<GemmProb>& v, int bn, int R) {
  long long tiles = 0;
  int nk = 1;
  for (auto& p : v) {
    tiles += (long long)((p.M + TC_BM - 1) / TC_BM) * ((p.N + bn - 1) / bn);
    nk = std::max(nk, (p.K + TC_BK - 1) / TC_BK);
  }
  const double kstep = bn == 64 ? 210.0 : (bn == 160 ? 366.0 : (tc_pair128() ? 276.0 : 315.0));
  const double tile = 2500.0 + nk * 4 * kstep + 1500.0 * ((bn / 32 + 1) / 2);
  const long long waves = (tiles * R + 147) / 148;
  return (double)waves * tile;
}
static int tc_pick_bn(const std::vector<GemmProb>& v, int R) {
  if (const char* e = getenv("B200SAC_TC_BN")) { const int b = atoi(e); return b == 128 ? 128 : (b == 160 ? 160 : 64); }
  int maxN = 0;
  for (auto& p : v) maxN = std::max(maxN, p.N);
  if (getenv("B200SAC_TC_OLDRULE")) {             // round-1 rule: 128 when the group still fills most of the GPU with 128x128 tiles
    long long c128 = 0;
    for (auto& p : v) c128 += (long long)((p.M + TC_BM - 1) / TC_BM) * ((p.N + 127) / 128);
    return (maxN >= 256 && c128 * R >= 96) ? 128 : 64;
  }
  const bool no160 = getenv("B200SAC_TC_NO160") != nullptr;
  int best = 64;
  double cost = tc_group_cost(v, 64, R);
  for (int bn : {128, 160}) {
    if (bn == 160 && no160) continue;
    if (maxN < 2 * bn - 64) continue;             // a lone, mostly empty wide tile is never better than 64-wide ones
    const double c = tc_group_cost(v, bn, R);
    if (c < cost) { cost = c; best = bn; }
  }
  return best;
}

constexpr int kSplitK = 4, kSplitKMin = 512;     // weight gradients with K >= 512 rows are computed in 4 K slices

static int make_tc_prob(const GemmProb& p, int rep, TcProb& t, int bn = 64) {
  memset(&t, 0, sizeof(t));
  const float* A = p.A + (long long)rep * p.rsA;
  const float* B = p.B + (long long)rep * p.rsB;
  t.M = p.M; t.N = p.N; t.K = p.K; t.mode = p.mode; t.relu = p.relu; t.ldc = p.ldc; t.ldmask = p.ldmask;
  t.bias = p.bias ? p.bias + (long long)rep * p.rsBias : nullptr;
  t.mask = p.mask ? p.mask + (long long)rep * p.rsMask : nullptr;
  t.C = p.C + (long long)rep * p.rsC;
  t.C2 = p.C2 ? p.C2 + (long long)rep * p.rsC2 : nullptr;
  if (p.mode == GEMM_FWD) {            // A[M][K], B[N][K]: both K-major
    t.a_mn = 0; t.b_mn = 0;
    if (int rc = make_map(&t.tmA, A, p.K, p.M, p.lda, TC_BM)) return rc;
    if (int rc = make_map(&t.tmB, B, p.K, p.N, p.ldb, bn)) return rc;
  } else if (p.mode == GEMM_DGRAD) {   // A = dY[M][K] K-major, B = W[K][N] MN-major
    t.a_mn = 0; t.b_mn = 1;
    if (int rc = make_map(&t.tmA, A, p.K, p.M, p.lda, TC_BM)) return rc;
    if (int rc = make_map(&t.tmB, B, p.N, p.K, p.ldb, TC_BK, true)) return rc;
  } else {                             // WGRAD: A = dY[K][M], B = X[K][N]: both MN-major
    t.a_mn = 1; t.b_mn = 1;
    if (int rc = make_map(&t.tmA, A, p.M, p.K, p.lda, TC_BK, true)) return rc;
    if (int rc = make_map(&t.tmB, B, p.N, p.K, p.ldb, TC_BK, true)) return rc;
  }
  // output map for the bulk-store epilogue: [M][N] fp32, row pitch ldc, boxes of 32 x 32
  if ((p.ldc % 4) == 0 && (((uintptr_t)t.C) & 15) == 0 && getenv("B200SAC_TC_NO_TMA_STORE") == nullptr) {
    if (int rc = make_map(&t.tmC, t.C, p.N, p.M, p.ldc, 32)) return rc;
    t.c_tma = 1;
  }
  return 0;
}

// ------------------------------------------------------------------------------------------
// Layer-chained plan (chain.cuh): 10 launches per step instead of one per layer.
//   A   forward  {actor on [s';s], Q1, Q2 on (s,a)}  -> policy head / scalar heads
//   B   forward  {Qt1, Qt2 on (s',a')}               -> scalar heads
//   C   backward {Q1, Q2}: y, dQ from the per-row scalars, input-gradient chain   -> wgrad -> adam_critic+polyak
//   D1  forward  {Q1, Q2 on (s,a~)} with the updated critics
//   D2  backward {Q1, Q2}: min routing, input-gradient chain down to d(action)
//   E   backward {actor}: d(mu|log_std), input-gradient chain                     -> wgrad -> adam_actor+alpha
// Eligible: exact-fp32 mode, no CARE, every hidden width a multiple of 4 and <= 256, obs+act <= 252.
// ------------------------------------------------------------------------------------------
static bool fused_eligible(const b200sac_cfg& c) {
  if (c.precision != 0 || c.care) return false;
  if (const char* e = getenv("B200SAC_FUSE")) if (e[0] == '0') return false;
  for (int i = 0; i < c.n_actor_hidden; ++i) if (c.actor_hidden[i] % 4 || c.actor_hidden[i] > CH_MAXW) return false;
  for (int i = 0; i < c.n_critic_hidden; ++i) if (c.critic_hidden[i] % 4 || c.critic_hidden[i] > CH_MAXW) return false;
  if (c.state_dim + c.num_tasks + c.act_dim > CH_MAXW - 4) return false;
  return true;
}

static int build_plan_fused(b200sac* h, const std::function<void(int, int)>& adam) {
  const b200sac_cfg& c = h->cfg;
  const Layout& L = h->L;
  const int B = c.batch, R = h->R, A = c.act_dim;
  const int La = c.n_actor_hidden, Lc = c.n_critic_hidden;
  const long long rsP = L.arena, rsG = L.trainable;
  auto W = [&](int64_t off) { return h->params + off; };
  auto Gp = [&](int64_t off) { return h->grads + off; };
  const int Hc = c.critic_hidden[Lc - 1], Ha = c.actor_hidden[La - 1];

  ChainRows rw;
  memset(&rw, 0, sizeof(rw));
  rw.r = h->r.p; rw.d = h->d.p; rw.tid = (const int*)h->tid.p; rw.rsR = h->r.rs;
  rw.logp = h->logp.p; rw.rsLogp = h->logp.rs;
  rw.log_alpha = W(L.off_alpha);
  rw.alpha = h->alpha.p; rw.rsAlpha = h->alpha.rs;
  rw.qt = h->qt.p; rw.q = h->q.p; rw.qp = h->qp.p;
  rw.y = h->y.p; rw.dq = h->dq.p; rw.lq = h->lq.p; rw.dqa = h->dqa.p; rw.la = h->la.p; rw.qmin = h->qmin.p; rw.rsY = h->y.rs;
  rw.dxP = h->dxP.p; rw.rsDxNet = (long long)B * h->K.ldx; rw.rsDxRep = h->dxP.rs; rw.lddx = h->K.ldx;
  rw.psave = h->psave.p + (long long)B * A * kSaveW; rw.rsSave = h->psave.rs;
  rw.dout_dbg = h->dout_dbg.p; rw.dact_dbg = h->dact_dbg.p; rw.rsDbg = h->dout_dbg.rs;

  struct WMap { const float* p; long long rs; int ld, cols; };
  std::vector<WMap> wmaps;                 // weight-gradient operands [B rows][cols] that get a tensor map
  struct FMap { int64_t off; int K, N, ld; };
  std::vector<FMap> fmaps;                 // forward weight matrices that need a tensor map (one per chained forward stage)
  auto new_chain = [&](const char* label, int early_weights = 1) {
    Launch l;
    l.kind = L_CHAIN;
    l.label = label;
    memset(&l.chain, 0, sizeof(l.chain));
    l.chain.early_weights = (early_weights && getenv("B200SAC_NO_EARLY_WEIGHTS") == nullptr) ? 1 : 0;
    l.chain.rsP = rsP;
    l.chain.pol = h->pol;
    l.chain.rw = rw;
    l.block = dim3(CH_BLOCK);
    l.smem = CH_SMEM_BYTES;
    return l;
  };
  if (getenv("B200SAC_CHAIN_DBG")) {
    CU(cudaMalloc(&h->chain_dbg, sizeof(long long) * CH_DBG_SLOTS * 16));
    CU(cudaMemset(h->chain_dbg, 0, sizeof(long long) * CH_DBG_SLOTS * 16));
  }
  auto finish_chain = [&](Launch& l) {
    if (h->chain_dbg && h->plan.size() < 16) l.chain.dbg = h->chain_dbg + h->plan.size() * CH_DBG_SLOTS;
    // rows per CTA: every CTA streams the whole weight matrices whatever its row count, so fewer rows per CTA only pay
    // while the launch still fits the GPU: 8 rows when that already gives >= 96 CTAs, else 4 (twice the CTAs, half the math each)
    long long total = 0;
    for (int j = 0; j < l.chain.njobs; ++j) total += l.chain.job[j].rows;
    l.bn = 8;                                      // (bn is reused as "rows per CTA" for chain launches)
    for (int rows = 4; rows >= 2; rows >>= 1)      // the fewest rows per CTA whose launch still fits one wave of 148 CTAs
      if ((total + rows - 1) / rows * R <= 148) l.bn = rows;
    if (const char* e = getenv("B200SAC_CHAIN_ROWS")) { const int v = atoi(e); l.bn = (v == 2 || v == 4) ? v : 8; }
    int maxb = 1;
    for (int j = 0; j < l.chain.njobs; ++j) {
      const int nb = (l.chain.job[j].rows + l.bn - 1) / l.bn;
      maxb = nb > maxb ? nb : maxb;
    }
    l.grid = dim3(maxb, l.chain.njobs, R);
    h->plan.push_back(l);
  };
  // forward job of one MLP: input rows X, per-layer stores `store[l]` (+ net offset), head
  auto fwd_job = [&](ChainJob& J, const std::vector<LayerOff>& net, int nh, const float* X, long long rsX, int ldx, int K0, int rows,
                     const std::vector<Buf>* store, int net_idx, int rows_per_net) {
    memset(&J, 0, sizeof(J));
    J.kind = CJ_FWD; J.rows = rows; J.nstages = nh; J.net = net_idx;
    J.X = X; J.rsX = rsX; J.ldx = ldx; J.K0 = K0;
    for (int l = 0; l < nh; ++l) {
      const LayerOff& lo = net[l];
      ChainStage& S = J.st[l];
      S.W = W(lo.w); S.bias = W(lo.b); S.ldw = lo.ld; S.K = lo.in; S.N = lo.out;
      S.tm_idx = (int)fmaps.size();
      fmaps.push_back(FMap{lo.w, lo.in, lo.out, lo.ld});
      if (store) { S.out = (*store)[l].p + (long long)net_idx * rows_per_net * lo.out; S.rsOut = (*store)[l].rs; S.ldo = lo.out; }
    }
    const LayerOff& hd = net[nh];
    J.Wh = W(hd.w); J.bh = W(hd.b); J.NO = hd.out; J.Hh = hd.in;
  };
  // backward job of one MLP (input-gradient chain): gate activations acts[l], stores dstore[l] (nullable)
  auto bwd_job = [&](ChainJob& J, int kind, const std::vector<LayerOff>& net, int nh, int rows, const std::vector<Buf>& acts,
                     long long act_row_off /* rows to skip in acts */, const std::vector<Buf>* dstore, int net_idx) {
    memset(&J, 0, sizeof(J));
    J.kind = kind; J.rows = rows; J.nstages = nh - 1; J.net = net_idx;
    const LayerOff& hd = net[nh];
    J.Wh = W(hd.w); J.bh = W(hd.b); J.NO = hd.out; J.Hh = hd.in;
    const int Hl = net[nh - 1].out;
    J.hlast = acts[nh - 1].p + ((long long)net_idx * rows + act_row_off) * Hl; J.rsHlast = acts[nh - 1].rs; J.ldh = Hl;
    if (dstore) { J.dylast = (*dstore)[nh - 1].p + (long long)net_idx * rows * Hl; J.rsDy = (*dstore)[nh - 1].rs; J.lddy = Hl; }
    for (int s = 0; s + 1 < nh; ++s) {
      const int l = nh - 1 - s;                    // dh_{l-1} = (dh_l W_l) * [h_{l-1} > 0]
      const LayerOff& lo = net[l];
      ChainStage& S = J.st[s];
      S.W = W(lo.w); S.ldw = lo.ld; S.K = lo.out; S.N = lo.in;
      S.mask = acts[l - 1].p + ((long long)net_idx * rows + act_row_off) * lo.in; S.rsMask = acts[l - 1].rs; S.ldmask = lo.in;
      if (dstore) { S.out = (*dstore)[l - 1].p + (long long)net_idx * rows * lo.in; S.rsOut = (*dstore)[l - 1].rs; S.ldo = lo.in; }
    }
  };
  // weight-gradient launch of a group of networks
  struct WNet { const std::vector<LayerOff>* net; int nh; const std::vector<Buf>* dstore; const std::vector<Buf>* acts; long long act_row_off;
                const float* X; long long rsX; int ldx; const float* dout; long long rsDout; int lddout; int net_idx; };
  const bool fuse_adam = getenv("B200SAC_NO_FUSED_ADAM") == nullptr;
  auto wgrad_launch = [&](const std::vector<WNet>& nets, const char* label, int which) -> int {
    Launch l;
    l.kind = L_WGRAD;
    l.label = label;
    memset(&l.wg, 0, sizeof(l.wg));
    l.wg.M = B; l.wg.rsG = rsG;
    if (fuse_adam) {                             // the CTA that reduces a gradient tile applies Adam (+ Polyak) to it
      WgradAdam& O = l.wg.adam;
      O.enabled = 1; O.which = which;
      O.params = h->params; O.m = h->adam_m; O.v = h->adam_v; O.grads = h->grads;
      O.rsP = rsP; O.rsM = rsG;
      O.target_delta = which == 0 ? L.target_delta : 0;
      O.lr = which == 0 ? c.lr_critic : c.lr_actor;
      O.cnt = h->cnt;
    }
    int tiles = 0;
    auto add = [&](const float* Ap, long long rsA, int lda, const float* Bp, long long rsB, int ldb, int64_t offW, int ldc, int64_t offB,
                   int Kout, int Nin) -> int {
      if (l.wg.njobs >= WG_MAXJOBS) return fail(B200SAC_ERR_INVALID, "too many weight-gradient jobs in one launch");
      WgradJob& J = l.wg.job[l.wg.njobs++];
      J.A = Ap; J.rsA = rsA; J.lda = lda; J.B = Bp; J.rsB = rsB; J.ldb = ldb;
      J.C = Gp(offW); J.C2 = Gp(offB); J.ldc = ldc; J.Kout = Kout; J.Nin = Nin;
      J.tile0 = tiles; J.tn = (Nin + WG_T - 1) / WG_T;
      J.shape = Kout <= 4 ? WG_KTHIN : (Nin <= 16 ? WG_NTHIN : WG_FULL);
      tiles += J.tn * ((Kout + WG_T - 1) / WG_T);
      // operands a tensor map can address (16-byte row pitch and base) arrive by TMA, the others are staged by the threads
      auto tmable = [&](const float* p_, long long rs_, int ld_) { return (ld_ % 4) == 0 && (((uintptr_t)p_) & 15) == 0 && (rs_ % 4) == 0; };
      J.tmA_idx = J.tmB_idx = -1;
      if (tmable(Ap, rsA, lda)) { J.tmA_idx = (int)wmaps.size(); wmaps.push_back(WMap{Ap, rsA, lda, Kout}); }
      if (tmable(Bp, rsB, ldb)) { J.tmB_idx = (int)wmaps.size(); wmaps.push_back(WMap{Bp, rsB, ldb, Nin}); }
      return 0;
    };
    for (const WNet& n : nets) {
      const std::vector<LayerOff>& net = *n.net;
      for (int lyr = n.nh - 1; lyr >= 0; --lyr) {      // biggest layers first
        const LayerOff& lo = net[lyr];
        const Buf& db = (*n.dstore)[lyr];
        const float* Ap = db.p + (long long)n.net_idx * B * lo.out;
        const float* Bp; long long rsB; int ldb;
        if (lyr == 0) { Bp = n.X; rsB = n.rsX; ldb = n.ldx; }
        else {
          const Buf& ab = (*n.acts)[lyr - 1];
          Bp = ab.p + ((long long)n.net_idx * B + n.act_row_off) * lo.in; rsB = ab.rs; ldb = lo.in;   // (actor: [s';s], skip the s' half)
        }
        if (int rc = add(Ap, db.rs, lo.out, Bp, rsB, ldb, lo.w, lo.ld, lo.b, lo.out, lo.in)) return rc;
      }
      const LayerOff& hd = net[n.nh];
      const Buf& ab = (*n.acts)[n.nh - 1];
      const float* Bp = ab.p + ((long long)n.net_idx * B + n.act_row_off) * hd.in;
      if (int rc = add(n.dout, n.rsDout, n.lddout, Bp, ab.rs, hd.in, hd.w, hd.in, hd.b, hd.out, hd.in)) return rc;
    }
    l.grid = dim3(tiles, R);
    l.block = dim3(WG_THREADS);
    l.smem = WG_SMEM_BYTES;
    if (h->chain_dbg && h->plan.size() < 16) l.wg.dbg = h->chain_dbg + h->plan.size() * CH_DBG_SLOTS;
    h->plan.push_back(l);
    return 0;
  };

  // ---- A: actor over [s';s], Q1/Q2 over (s,a) ----------------------------------------------------------------------
  {
    Launch l = new_chain("chain_fwd{actor,q1,q2}");
    l.chain.njobs = 3;
    fwd_job(l.chain.job[0], L.actor, La, h->XA.p, h->XA.rs, h->K.ldxa, h->K.in_w, 2 * B, &h->hA, 0, 0);
    l.chain.job[0].head = CH_HEAD_POLICY;
    for (int net = 0; net < 2; ++net) {
      ChainJob& J = l.chain.job[1 + net];
      fwd_job(J, L.q[net], Lc, h->XQ.p, h->XQ.rs, h->K.ldx, h->K.xw, B, &h->hQ, net, B);
      J.head = CH_HEAD_SCALAR; J.qout = h->q.p + (long long)net * B; J.rsQ = h->q.rs;
    }
    h->use_eps_buf_idx = (int)h->plan.size();
    finish_chain(l);
  }
  // Twin forward + backward in one clustered launch (chain2.cuh) when the critic is shallow enough for its stage tables
  const bool pair = Lc <= C2_MAXL && getenv("B200SAC_NO_CLUSTER") == nullptr;
  auto pair_launch = [&](const char* label, int kind, int early, const std::vector<LayerOff>* fnet /* [2] */, const float* X, long long rsX,
                         const std::vector<Buf>* fstore, const Buf& qf, const std::vector<Buf>& acts, const std::vector<Buf>* dstore,
                         bool tail) {
    Launch l;
    l.kind = L_CHAIN2;
    l.label = label;
    memset(&l.chain2, 0, sizeof(l.chain2));
    Chain2Args& P = l.chain2;
    P.kind = kind; P.rsP = rsP; P.rw = rw;
    P.early_weights = (early && getenv("B200SAC_NO_EARLY_WEIGHTS") == nullptr) ? 1 : 0;
    for (int net = 0; net < 2; ++net) {
      Chain2Job& J = P.job[net];
      J.rows = B; J.nfwd = Lc; J.nbwd = Lc - 1; J.net = net;
      J.X = X; J.rsX = rsX; J.ldx = h->K.ldx; J.K0 = h->K.xw;
      for (int lyr = 0; lyr < Lc; ++lyr) {
        const LayerOff& lo = fnet[net][lyr];
        ChainStage& S = J.fst[lyr];
        S.W = W(lo.w); S.bias = W(lo.b); S.ldw = lo.ld; S.K = lo.in; S.N = lo.out;
        S.tm_idx = (int)fmaps.size();
        fmaps.push_back(FMap{lo.w, lo.in, lo.out, lo.ld});
        if (fstore) { S.out = (*fstore)[lyr].p + (long long)net * B * lo.out; S.rsOut = (*fstore)[lyr].rs; S.ldo = lo.out; }
      }
      const LayerOff& fh = fnet[net][Lc];
      J.Whf = W(fh.w); J.bhf = W(fh.b); J.Hhf = fh.in;
      J.qf_out = qf.p + (long long)net * B; J.rsQf = qf.rs;
      // backward through the LOCAL twin
      const std::vector<LayerOff>& bn = L.q[net];
      const int Hl = bn[Lc - 1].out;
      J.hlast = acts[Lc - 1].p + (long long)net * B * Hl; J.rsHlast = acts[Lc - 1].rs; J.ldh = Hl;
      if (dstore) { J.dylast = (*dstore)[Lc - 1].p + (long long)net * B * Hl; J.rsDy = (*dstore)[Lc - 1].rs; J.lddy = Hl; }
      J.Whb = W(bn[Lc].w); J.Hhb = bn[Lc].in;
      for (int sidx = 0; sidx + 1 < Lc; ++sidx) {
        const int lyr = Lc - 1 - sidx;
        const LayerOff& lo = bn[lyr];
        ChainStage& S = J.bst[sidx];
        S.W = W(lo.w); S.ldw = lo.ld; S.K = lo.out; S.N = lo.in;
        S.mask = acts[lyr - 1].p + (long long)net * B * lo.in; S.rsMask = acts[lyr - 1].rs; S.ldmask = lo.in;
        if (dstore) { S.out = (*dstore)[lyr - 1].p + (long long)net * B * lo.in; S.rsOut = (*dstore)[lyr - 1].rs; S.ldo = lo.in; }
      }
      if (tail) {
        const LayerOff& lo = bn[0];
        J.W0 = W(lo.w); J.ldw0 = lo.ld; J.col0 = h->K.in_w; J.nact = A; J.H0 = lo.out;
        J.dx = h->dxP.p + (long long)net * B * h->K.ldx; J.rsDx = h->dxP.rs; J.lddx = h->K.ldx;
      }
    }
    if (h->chain_dbg && h->plan.size() < 16) P.dbg = h->chain_dbg + h->plan.size() * CH_DBG_SLOTS;
    l.bn = 8;
    for (int rows = 4; rows >= 2; rows >>= 1)
      if ((long long)2 * ((B + rows - 1) / rows) * R <= 148) l.bn = rows;
    if (const char* e = getenv("B200SAC_CHAIN_ROWS")) { const int v = atoi(e); l.bn = (v == 2 || v == 4) ? v : 8; }
    l.grid = dim3((B + l.bn - 1) / l.bn, 2, R);
    l.block = dim3(CH_BLOCK);
    l.smem = C2_SMEM_BYTES;
    h->plan.push_back(l);
  };
  // ---- B + C: target critics over (s', a'), TD target, critic backward (one clustered launch), weight gradients, Adam ----
  if (pair) {
    pair_launch("chain2{qt->y->bwd q}", C2_CRITIC, 1, L.qt, h->XT.p, h->XT.rs, nullptr, h->qt, h->hQ, &h->dhQ, false);
  } else {
    {
      Launch l = new_chain("chain_fwd{qt1,qt2}");
      l.chain.njobs = 2;
      for (int net = 0; net < 2; ++net) {
        ChainJob& J = l.chain.job[net];
        fwd_job(J, L.qt[net], Lc, h->XT.p, h->XT.rs, h->K.ldx, h->K.xw, B, nullptr, net, B);
        J.head = CH_HEAD_SCALAR; J.qout = h->qt.p + (long long)net * B; J.rsQ = h->qt.rs;
      }
      finish_chain(l);
    }
    Launch l = new_chain("chain_bwd{q1,q2}");
    l.chain.njobs = 2;
    for (int net = 0; net < 2; ++net) bwd_job(l.chain.job[net], CJ_BWD_CRITIC, L.q[net], Lc, B, h->hQ, 0, &h->dhQ, net);
    finish_chain(l);
  }
  {
    std::vector<WNet> nets;
    for (int net = 0; net < 2; ++net)
      nets.push_back(WNet{&L.q[net], Lc, &h->dhQ, &h->hQ, 0, h->XQ.p, h->XQ.rs, h->K.ldx, h->dq.p + (long long)net * B, h->dq.rs, 1, net});
    if (int rc = wgrad_launch(nets, fuse_adam ? "wgrad+adam+polyak{q1,q2}" : "wgrad{q1,q2}", 0)) return rc;
    if (!fuse_adam) adam(0, 0);
  }
  // ---- D: actor pass through the updated critics ------------------------------------------------------------------------
  {
    if (pair) {
      // (the launch right before this one is the critic Adam: no weight request before the dependency wait)
      pair_launch("chain2{q(s,a~)->min->bwd->d(action)}", C2_ACTORQ, 0, L.q, h->XP.p, h->XP.rs, &h->hP, h->qp, h->hP, nullptr, true);
    } else {
      // (the launch right before this one is the critic Adam: no weight request before the dependency wait)
      Launch l = new_chain("chain_fwd{q1,q2}(s,a~)", 0);
      l.chain.njobs = 2;
      for (int net = 0; net < 2; ++net) {
        ChainJob& J = l.chain.job[net];
        fwd_job(J, L.q[net], Lc, h->XP.p, h->XP.rs, h->K.ldx, h->K.xw, B, &h->hP, net, B);
        J.head = CH_HEAD_SCALAR; J.qout = h->qp.p + (long long)net * B; J.rsQ = h->qp.rs;
      }
      finish_chain(l);
      Launch l2 = new_chain("chain_bwd{q1,q2}->d(action)");
      l2.chain.njobs = 2;
      for (int net = 0; net < 2; ++net) {
        ChainJob& J = l2.chain.job[net];
        bwd_job(J, CJ_BWD_ACTORQ, L.q[net], Lc, B, h->hP, 0, nullptr, net);
        const LayerOff& lo = L.q[net][0];
        J.head = CH_TAIL_DACTION;
        J.W0 = W(lo.w); J.ldw0 = lo.ld; J.col0 = h->K.in_w; J.nact = A; J.H0 = lo.out;
        J.dx = h->dxP.p + (long long)net * B * h->K.ldx; J.rsDx = h->dxP.rs; J.lddx = h->K.ldx;
      }
      finish_chain(l2);
    }
    // actor loss / entropy / temperature gradient + its Adam step need only what D produced (the step's alpha is the
    // snapshot taken at ingest): they run on the fork stream beside the policy backward instead of trailing the actor Adam
    adam(1, fuse_adam ? 3 : 2);
  }
  // ---- E: policy backward, weight gradients, Adam + temperature ------------------------------------------------------------
  {
    Launch l = new_chain("chain_bwd{actor}");
    l.chain.njobs = 1;
    bwd_job(l.chain.job[0], CJ_BWD_POLICY, L.actor, La, B, h->hA, B, &h->dhA, 0);
    finish_chain(l);
    std::vector<WNet> nets;
    nets.push_back(WNet{&L.actor, La, &h->dhA, &h->hA, (long long)B, h->XA.p + (long long)B * h->K.ldxa, h->XA.rs, h->K.ldxa,
                        h->dout_dbg.p, h->dout_dbg.rs, 2 * A, 0});
    if (int rc = wgrad_launch(nets, fuse_adam ? "wgrad+adam{actor}" : "wgrad{actor}", 1)) return rc;
    if (!fuse_adam) adam(1, 1);
  }
  (void)Hc; (void)Ha;
  {  // tensor maps [R][n]: W [N][K] row-major (pitch ld), box {32 k, N rows}, SWIZZLE_128B, OOB k zero-filled
    const int n = (int)fmaps.size();
    std::vector<CUtensorMap> maps((size_t)R * n);
    for (int rep = 0; rep < R; ++rep)
      for (int i = 0; i < n; ++i)
        if (int rc = make_map(&maps[(size_t)rep * n + i], h->params + (long long)rep * rsP + fmaps[i].off, fmaps[i].K, fmaps[i].N,
                              fmaps[i].ld, fmaps[i].N))
          return rc;
    CU(cudaMalloc(&h->d_cmaps, maps.size() * sizeof(CUtensorMap)));
    CU(cudaMemcpy(h->d_cmaps, maps.data(), maps.size() * sizeof(CUtensorMap), cudaMemcpyHostToDevice));
    for (auto& l : h->plan) {
      if (l.kind == L_CHAIN)
        for (int j = 0; j < l.chain.njobs; ++j)
          if (l.chain.job[j].kind == CJ_FWD)
            for (int st = 0; st < l.chain.job[j].nstages; ++st) {
              ChainStage& S = l.chain.job[j].st[st];
              S.tm = h->d_cmaps + S.tm_idx;
              S.rsTm = n;
            }
      if (l.kind == L_CHAIN2)
        for (int j = 0; j < 2; ++j)
          for (int st = 0; st < l.chain2.job[j].nfwd; ++st) {
            ChainStage& S = l.chain2.job[j].fst[st];
            S.tm = h->d_cmaps + S.tm_idx;
            S.rsTm = n;
          }
    }
  }
  CU(cudaFuncSetAttribute(chain2_kernel<8>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)C2_SMEM_BYTES));
  CU(cudaFuncSetAttribute(chain2_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)C2_SMEM_BYTES));
  CU(cudaFuncSetAttribute(chain2_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)C2_SMEM_BYTES));
  {  // weight-gradient operand maps [R][n]: [B rows][cols] row-major, box {32 cols, 256 rows}, dense
    const int n = (int)wmaps.size();
    std::vector<CUtensorMap> maps((size_t)R * n);
    for (int rep = 0; rep < R; ++rep)
      for (int i = 0; i < n; ++i)
        if (int rc = make_map(&maps[(size_t)rep * n + i], wmaps[i].p + (long long)rep * wmaps[i].rs, wmaps[i].cols, B, wmaps[i].ld, WG_ROWS,
                              false, true))
          return rc;
    if (n > 0) {
      CU(cudaMalloc(&h->d_wmaps, maps.size() * sizeof(CUtensorMap)));
      CU(cudaMemcpy(h->d_wmaps, maps.data(), maps.size() * sizeof(CUtensorMap), cudaMemcpyHostToDevice));
    }
    for (auto& l : h->plan)
      if (l.kind == L_WGRAD)
        for (int j = 0; j < l.wg.njobs; ++j) {
          WgradJob& J = l.wg.job[j];
          J.tmA = J.tmA_idx >= 0 ? h->d_wmaps + J.tmA_idx : nullptr;
          J.tmB = J.tmB_idx >= 0 ? h->d_wmaps + J.tmB_idx : nullptr;
          J.rsTm = n;
        }
  }
  CU(cudaFuncSetAttribute(chain_kernel<true, 8>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)CH_SMEM_BYTES));
  CU(cudaFuncSetAttribute(chain_kernel<false, 8>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)CH_SMEM_BYTES));
  CU(cudaFuncSetAttribute(chain_kernel<true, 4>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)CH_SMEM_BYTES));
  CU(cudaFuncSetAttribute(chain_kernel<false, 4>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)CH_SMEM_BYTES));
  CU(cudaFuncSetAttribute(chain_kernel<true, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)CH_SMEM_BYTES));
  CU(cudaFuncSetAttribute(chain_kernel<false, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)CH_SMEM_BYTES));
  CU(cudaFuncSetAttribute(wgrad_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)WG_SMEM_BYTES));
  return 0;
}

// Build the launch list of one gradient step (everything after the ingest kernel).
static int build_plan(b200sac* h) {
  const b200sac_cfg& c = h->cfg;
  const Layout& L = h->L;
  const int B = c.batch, R = h->R, A = c.act_dim;
  const int La = c.n_actor_hidden, Lc = c.n_critic_hidden;
  const long long rsP = L.arena, rsG = L.trainable;
  std::vector<std::vector<GemmProb>> groups;
  struct Pending { int group; };
  auto W = [&](int64_t off) { return h->params + off; };
  auto Gp = [&](int64_t off) { return h->grads + off; };

  int plan_rc = 0;
  int cur_branch = 0;            // branch tag given to the launches gemm_launch creates
  // FFMA back-end, plain SAC nets: a layer's weight gradient only feeds Adam, while its input gradient heads the rest of the
  // backward chain.  The weight-gradient launch goes to the fork stream and the chain continues at once (the kernels hold
  // <= 2 CTAs per SM, so both fit); Adam joins.  (tcgen05 tiles own a whole SM each: grouping is better there.)
  const bool use_fork = (c.precision == 0) && !c.care && getenv("B200SAC_NO_FORK") == nullptr;
  std::function<void(std::vector<GemmProb>)> gemm_launch_ref;
  auto gemm_launch = [&](std::vector<GemmProb> ps_in) {
    // Split-K for the weight gradients: K = batch (1024 / 1280) is the long dimension and M x N = out x in gives only a
    // handful of tiles, so one CTA would walk 32-40 k chunks alone (measured 26-32 us per launch at the 400-wide shapes).
    // WGRAD operands are both [K][*] row-major, so a K slice is just a row offset: slice s of a problem becomes its own
    // problem writing gradient slice s; Adam adds the slices in index order (deterministic, no atomics).
    auto expand = [&](int Smax, std::vector<GemmProb>& out) {
      for (auto& p : ps_in) {
        const int S = (p.mode == GEMM_WGRAD && p.K >= kSplitKMin && h->gslices > 1) ? Smax : 1;
        if (S == 1) { out.push_back(p); continue; }
        const int len = (((p.K + S - 1) / S) + 31) & ~31;
        const long long coff = p.C - h->grads, c2off = p.C2 ? p.C2 - h->grads : 0;
        if (coff < 0 || coff >= L.trainable) { plan_rc = fail(B200SAC_ERR_INVALID, "internal: split-K output outside the gradient arena"); out.push_back(p); continue; }
        for (int sidx = 0; sidx < S; ++sidx) {
          const int kb = sidx * len;
          if (kb >= p.K) break;
          GemmProb q = p;
          q.A = p.A + (long long)kb * p.lda; q.B = p.B + (long long)kb * p.ldb;
          q.K = (p.K - kb < len) ? p.K - kb : len;
          if (sidx > 0) {
            float* base = h->grads_x + (long long)(sidx - 1) * R * L.trainable;
            q.C = base + coff;
            if (p.C2) q.C2 = base + c2off;
          }
          out.push_back(q);
        }
      }
    };
    // tcgen05 tiles hold one CTA per SM: take the split factor (and with it the tile width) whose launch is cheapest under
    // tc_group_cost's model -- a finer split shortens the k loop but a second wave of CTAs costs a whole tile time; the FFMA
    // engine (several CTAs per SM) always takes the finest.
    auto tc_only = [&](const std::vector<GemmProb>& v) {
      std::vector<GemmProb> o;
      for (auto& p : v) if (tc_eligible(p)) o.push_back(p);
      return o;
    };
    std::vector<GemmProb> ps;
    {
      int S = kSplitK;
      if (c.precision == 1) {
        double best = 1e300;
        for (int s_ = kSplitK; s_ >= 1; s_ >>= 1) {
          std::vector<GemmProb> trial;
          expand(s_, trial);
          const std::vector<GemmProb> o = tc_only(trial);
          if (o.empty()) { S = s_; break; }
          if (getenv("B200SAC_TC_OLDRULE")) {          // round-1 rule: the finest split that fits one wave
            const int bn = tc_pick_bn(o, R);
            long long ct = 0;
            for (auto& p : o) ct += (long long)((p.M + TC_BM - 1) / TC_BM) * ((p.N + bn - 1) / bn);
            S = s_;
            if (ct * R <= 148) break;
            continue;
          }
          const double cost = tc_group_cost(o, tc_pick_bn(o, R), R);
          if (cost < best) { best = cost; S = s_; }
        }
      }
      expand(S, ps);
    }
    if (c.precision == 1) {
      std::vector<GemmProb> tc, rest;
      for (auto& p : ps) (tc_eligible(p) ? tc : rest).push_back(p);
      if (!tc.empty()) {
        Launch l;
        int maxM = 0, maxN = 0;
        for (auto& p : tc) { maxM = p.M > maxM ? p.M : maxM; maxN = p.N > maxN ? p.N : maxN; }
        const int bn = tc_pick_bn(tc, R);          // tile width: the cheapest of 64 / 128 / 160 under tc_group_cost's model
        if (getenv("B200SAC_PLAN_DBG")) {
          long long tiles = 0;
          for (auto& p : tc) tiles += (long long)((p.M + TC_BM - 1) / TC_BM) * ((p.N + bn - 1) / bn);
          fprintf(stderr, "[plan] launch %zu: tcgen05 bn=%d problems=%zu tiles=%lld:", h->plan.size(), bn, tc.size(), tiles);
          for (auto& p : tc) fprintf(stderr, " %s%dx%dx%d", p.mode == GEMM_FWD ? "F" : (p.mode == GEMM_DGRAD ? "D" : "W"), p.M, p.N, p.K);
          fprintf(stderr, "\n");
        }
        l.kind = L_GEMM_TC;
        l.branch = cur_branch;
        l.bn = bn;
        l.grid = dim3((maxN + bn - 1) / bn, (maxM + TC_BM - 1) / TC_BM, (unsigned)(tc.size() * R));
        l.block = dim3(TC_THREADS);
        l.smem = tc_smem(bn);
        l.G = (int)tc.size();
        l.tprobs = (const TcProb*)(uintptr_t)h->h_tprobs.size();
        l.probs = (const GemmProb*)(uintptr_t)h->h_probs.size();   // keep the SIMT descriptors too (labels)
        for (int rep = 0; rep < R; ++rep)
          for (auto& p : tc) {
            TcProb t;
            if (int rc = make_tc_prob(p, rep, t, bn)) plan_rc = rc;
            h->h_tprobs.push_back(t);
          }
        for (auto& p : tc) h->h_probs.push_back(p);
        h->plan.push_back(l);
      }
      if (rest.empty()) return;
      ps = rest;
    }
    if (ps.size() > GS_MAXG) {            // more problems than one parameter block holds: several launches
      std::vector<GemmProb> head(ps.begin(), ps.begin() + GS_MAXG), tail(ps.begin() + GS_MAXG, ps.end());
      gemm_launch_ref(head);
      gemm_launch_ref(tail);
      return;
    }
    Launch l;
    int maxM = 0, maxN = 0;
    bool thin = getenv("B200SAC_NO_THIN") == nullptr;
    for (auto& p : ps) { maxM = p.M > maxM ? p.M : maxM; maxN = p.N > maxN ? p.N : maxN; thin = thin && gemm_is_thin(p); }
    l.kind = L_GEMM_SMALL;
    l.branch = cur_branch;
    l.grid = dim3((maxN + GS_T - 1) / GS_T, (maxM + GS_T - 1) / GS_T, (unsigned)(ps.size() * R));
    l.block = dim3(GS_THREADS);
    if (thin) {        // input-layer weight / input gradients (N = obs+act <= 16): gemm_thin.cuh
      int rows = 1;
      for (auto& p : ps) {
        const int per = p.mode == GEMM_WGRAD ? GT_ROWS_WGRAD : GT_ROWS_DGRAD, r = (p.M + per - 1) / per;
        rows = r > rows ? r : rows;
      }
      l.kind = L_GEMM_THIN;
      l.grid = dim3(1, rows, (unsigned)(ps.size() * R));
      l.block = dim3(GT_THREADS);
    }
    l.G = (int)ps.size();
    if (ps.size() > GS_MAXG) plan_rc = fail(B200SAC_ERR_INVALID, "internal: more than %d problems in one GEMM group", GS_MAXG);
    memset(&l.grp, 0, sizeof(l.grp));
    l.grp.G = l.G;
    for (size_t i = 0; i < ps.size() && i < GS_MAXG; ++i) l.grp.p[i] = ps[i];
    l.probs = (const GemmProb*)(uintptr_t)h->h_probs.size();   // index for now; rebased later
    for (auto& p : ps) h->h_probs.push_back(p);
    h->plan.push_back(l);
  };
  gemm_launch_ref = gemm_launch;

  // ---- CARE helpers ------------------------------------------------------------------------
  const int Kenc = c.num_encoders, nmix = c.care ? (int)L.mix.size() : 0;
  auto pitch = [](int w) { return (w + 3) & ~3; };
  // mixture-of-encoders forward of encoder instance `inst` (0: critic's on XS rows [row0, row0+rows) into the
  // instance-0 buffers at the same rows; 1: target's; 2: critic's after its Adam step)
  auto care_tables = [&](std::vector<int> insts) {
    Launch l;
    l.kind = L_CARE_TAB;
    CareTabArgs& P = l.ctab;
    memset(&P, 0, sizeof(P));
    P.params = h->params; P.rsP = rsP; P.emb_off = L.off_emb;
    P.trunk = h->care_trunk; P.ctx = h->care_ctx;
    P.T = c.num_tasks; P.K = Kenc; P.row_w = h->care_row_w; P.off_att = h->care_off_att;
    P.original = c.care == 2 ? 1 : 0;
    for (size_t i = 0; i < insts.size(); ++i) {
      P.inst_delta[i] = insts[i] == 1 ? L.target_delta : 0;
      P.tab[i] = h->careTab[insts[i]].p;
    }
    P.rsTab = h->careTab[0].rs;
    l.grid = dim3(c.num_tasks, (unsigned)insts.size(), R);
    l.block = dim3(512);
    h->plan.push_back(l);
  };
  auto care_mixture_fwd = [&](std::vector<std::tuple<int, int, int>> jobs /* (inst, xs_row0, rows) */) {
    for (int l = 0; l < nmix; ++l) {
      std::vector<GemmProb> ps;
      for (auto& jb : jobs) {
        const int inst = std::get<0>(jb), row0 = std::get<1>(jb), rows = std::get<2>(jb);
        const int rows_buf = inst == 0 ? 2 * B : B;             // rows held by the instance's buffers
        const int out_row0 = inst == 0 ? row0 : 0;
        const LayerOff& lo = L.mix[l];
        const long long delta = inst == 1 ? L.target_delta : 0;
        const bool last = (l == nmix - 1);
        const Buf& ob = last ? h->mixZ[inst] : h->mixH[inst][l];
        for (int k = 0; k < Kenc; ++k) {
          GemmProb p;
          memset(&p, 0, sizeof(p));
          if (l == 0) { p.A = h->XS.p + (long long)row0 * h->K.obs; p.rsA = h->XS.rs; p.lda = h->K.obs; }
          else {
            const Buf& ib = h->mixH[inst][l - 1];
            p.A = ib.p + ((long long)k * rows_buf + out_row0) * pitch(lo.in); p.rsA = ib.rs; p.lda = pitch(lo.in);
          }
          p.B = W(delta + lo.w + (long long)k * lo.out * lo.in); p.rsB = rsP; p.ldb = lo.in;
          p.bias = W(delta + lo.b + (long long)k * lo.out); p.rsBias = rsP;
          p.C = ob.p + ((long long)k * rows_buf + out_row0) * pitch(lo.out); p.rsC = ob.rs; p.ldc = pitch(lo.out);
          p.M = rows; p.N = lo.out; p.K = lo.in; p.mode = GEMM_FWD; p.relu = last ? 0 : 1;
          ps.push_back(p);
        }
      }
      gemm_launch(ps);
    }
  };
  auto care_mix = [&](int inst, int rows, float* d1, long long rs1, int ld1, float* d2, long long rs2, int ld2, int off2) {
    Launch l;
    l.kind = L_CARE_MIX;
    CareMixArgs& P = l.cmix;
    memset(&P, 0, sizeof(P));
    const int rows_buf = inst == 0 ? 2 * B : B;
    P.Z = h->mixZ[inst].p; P.rsZ = h->mixZ[inst].rs; P.kstride = (long long)rows_buf * pitch(c.mix_out); P.ldz = pitch(c.mix_out);
    P.tab = h->careTab[inst].p; P.rsTab = h->careTab[inst].rs; P.row_w = h->care_row_w; P.off_att = h->care_off_att;
    P.off_ctx = h->care_off_ctx;
    P.tid = (const int*)h->tid.p; P.rsR = h->r.rs;
    P.rows = rows; P.B = B; P.K = Kenc; P.mo = c.mix_out; P.co = c.ctx_out;
    P.dst1 = d1; P.rsD1 = rs1; P.ld1 = ld1; P.dst2 = d2; P.rsD2 = rs2; P.ld2 = ld2; P.row_off2 = off2;
    l.grid = dim3((rows + 7) / 8, R);
    l.block = dim3(256);
    h->plan.push_back(l);
  };
  // mixture layers + attention mix of up to three encoder instances in ONE launch (care_mixfwd_kernel: all mixture weights of
  // an instance resident in shared memory); falls back to the grouped-GEMM path when the weights do not fit
  struct EncJob { int inst, xs_row0, rows; float* d1; long long rs1; int ld1; float* d2; long long rs2; int ld2; int off2; };
  auto care_encode = [&](std::vector<EncJob> jobs) {
    CareMixFwdArgs A;
    memset(&A, 0, sizeof(A));
    A.njobs = (int)jobs.size(); A.nl = nmix; A.K = Kenc; A.B = B;
    if (const char* e = getenv("B200SAC_CMF_SKIP")) A.dbg_skip = atoi(e);
    A.params = h->params; A.rsP = rsP;
    A.XS = h->XS.p; A.rsXS = h->XS.rs; A.ldx = h->K.obs;
    A.tid = (const int*)h->tid.p; A.rsR = h->r.rs;
    A.row_w = h->care_row_w; A.off_att = h->care_off_att; A.off_ctx = h->care_off_ctx; A.mo = c.mix_out; A.co = c.ctx_out;
    bool ok = nmix >= 1 && nmix <= CMF_MAXL && (int)jobs.size() <= CMF_MAXJOBS && getenv("B200SAC_NO_CARE_FUSED") == nullptr;
    for (int l = 0; ok && l < nmix; ++l) {
      A.w_off[l] = L.mix[l].w; A.b_off[l] = L.mix[l].b; A.in[l] = L.mix[l].in; A.out[l] = L.mix[l].out;
      A.maxw = std::max(A.maxw, L.mix[l].out);
    }
    int cta = 0;
    for (size_t i = 0; ok && i < jobs.size(); ++i) {
      const EncJob& e = jobs[i];
      CareMixFwdJob& J = A.job[i];
      const int rows_buf = e.inst == 0 ? 2 * B : B;
      J.inst_delta = e.inst == 1 ? L.target_delta : 0;
      J.rows = e.rows; J.xs_row0 = e.xs_row0; J.out_row0 = e.inst == 0 ? e.xs_row0 : 0; J.rows_buf = rows_buf;
      J.cta0 = cta; cta += (e.rows + CMF_ROWS - 1) / CMF_ROWS;
      J.tab = h->careTab[e.inst].p; J.rsTab = h->careTab[e.inst].rs;
      for (int l = 0; l < nmix; ++l) {
        const Buf& ob = (l == nmix - 1) ? h->mixZ[e.inst] : h->mixH[e.inst][l];
        J.H[l] = ob.p; J.rsH[l] = ob.rs;
      }
      J.dst1 = e.d1; J.rsD1 = e.rs1; J.ld1 = e.ld1; J.dst2 = e.d2; J.rsD2 = e.rs2; J.ld2 = e.ld2; J.row_off2 = e.off2;
    }
    const size_t smem = ok ? care_mixfwd_smem_floats(A) * sizeof(float) : 0;
    if (ok && smem <= 225 * 1024 &&
        cudaFuncSetAttribute(care_mixfwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 225 * 1024) == cudaSuccess) {
      Launch l;
      l.kind = L_CARE_MIXFWD;
      l.cmf = A;
      l.grid = dim3(cta, R);
      l.block = dim3(CMF_THREADS);
      l.smem = smem;
      h->plan.push_back(l);
      return;
    }
    std::vector<std::tuple<int, int, int>> mj;
    for (auto& e : jobs) mj.push_back(std::make_tuple(e.inst, e.xs_row0, e.rows));
    care_mixture_fwd(mj);
    for (auto& e : jobs) care_mix(e.inst, e.rows, e.d1, e.rs1, e.ld1, e.d2, e.rs2, e.ld2, e.off2);
  };
  if (c.care) {
    // encoded states of [s'; s] with the critic's (== actor's, tied) encoder and of s' with the target's
    care_tables({0, 1});
    care_encode({EncJob{0, 0, 2 * B, h->XA.p, h->XA.rs, h->K.ldxa, h->XQ.p, h->XQ.rs, h->K.ldx, B},
                 EncJob{1, 0, B, h->XT.p, h->XT.rs, h->K.ldx, nullptr, 0, 0, 0}});
  }

  auto fwd = [&](const float* Ain, long long rsA, int M, const LayerOff& lo, bool target_or_local_params, float* out,
                 long long rsOut) {
    (void)target_or_local_params;
    GemmProb p;
    memset(&p, 0, sizeof(p));
    p.A = Ain; p.rsA = rsA; p.lda = lo.ld;
    p.B = W(lo.w); p.rsB = rsP; p.ldb = lo.ld;
    p.bias = W(lo.b); p.rsBias = rsP;
    p.C = out; p.rsC = rsOut; p.ldc = lo.out;
    p.M = M; p.N = lo.out; p.K = lo.in; p.mode = GEMM_FWD; p.relu = 1;
    return p;
  };
  auto wgrad = [&](const float* dZ, long long rsdZ, const float* X, long long rsX, const LayerOff& lo) {
    GemmProb p;
    memset(&p, 0, sizeof(p));
    p.A = dZ; p.rsA = rsdZ; p.lda = lo.out;
    p.B = X; p.rsB = rsX; p.ldb = lo.ld;
    p.C = Gp(lo.w); p.rsC = rsG; p.ldc = lo.ld;
    p.C2 = Gp(lo.b); p.rsC2 = rsG;
    p.M = lo.out; p.N = lo.in; p.K = B; p.mode = GEMM_WGRAD;
    return p;
  };
  auto dgrad = [&](const float* dZ, long long rsdZ, const LayerOff& lo, const float* mask, long long rsMask, float* out,
                   long long rsOut) {
    GemmProb p;
    memset(&p, 0, sizeof(p));
    p.A = dZ; p.rsA = rsdZ; p.lda = lo.out;
    p.B = W(lo.w); p.rsB = rsP; p.ldb = lo.ld;
    p.mask = mask; p.rsMask = rsMask; p.ldmask = lo.ld;
    p.C = out; p.rsC = rsOut; p.ldc = lo.ld;
    p.M = B; p.N = lo.in; p.K = lo.out; p.mode = GEMM_DGRAD;
    return p;
  };
  auto netp = [&](const Buf& b, int net, int H) { return b.p + (long long)net * B * H; };

  {  // policy head arguments (the generic plan's policy_head launch, the chained forward kernel and b200sac_act share them)
    PolicyHeadArgs& P = h->pol;
    memset(&P, 0, sizeof(P));
    const LayerOff& lo = L.actor[La];
    P.h = h->hA[La - 1].p; P.rsH = h->hA[La - 1].rs; P.ldh = lo.in;
    P.W = W(lo.w); P.b = W(lo.b); P.rsP = rsP;
    P.eps = h->eps.p; P.rsEps = h->eps.rs; P.use_eps_buf = 0;
    P.pout = h->pout.p; P.rsPout = h->pout.rs;
    P.psave = h->psave.p; P.rsSave = h->psave.rs;
    P.XT = h->XT.p; P.XP = h->XP.p; P.rsX = h->XT.rs;
    P.act_out = h->act_out.p; P.rsAct = h->act_out.rs;
    P.logp = h->logp.p; P.rsLogp = h->logp.rs;
    P.logstd_sum = h->logstd.p;
    P.cnt = h->cnt;
  }
  // mode 0: parameter update + the tail job (last CTA); 1: parameter update only; 2 / 3: the tail job alone, on the fork
  // stream (3: + the critic-loss reduction, for plans whose critic Adam is fused into the weight-gradient launch)
  auto adam = [&](int which, int mode) {
    Launch l;
    l.kind = L_ADAM;
    AdamArgs& P = l.ad;
    memset(&P, 0, sizeof(P));
    const int64_t beg = which == 0 ? L.critic_begin : (which == 1 ? L.actor_begin : L.cenc_begin);
    const int64_t n = which == 0 ? L.critic_n : (which == 1 ? L.actor_n : L.cenc_n);
    P.p = h->params + beg; P.m = h->adam_m + beg; P.v = h->adam_v + beg; P.g = h->grads + beg;
    P.rsP = rsP; P.rsM = rsG; P.n = n;
    P.gx = h->grads_x ? h->grads_x + beg : nullptr; P.xs = (long long)R * L.trainable; P.nx = h->gslices - 1;
    P.target_delta = which == 0 ? L.target_delta : 0;
    P.tau2_begin = (which == 0 && c.care) ? (L.cse_begin - L.critic_begin) : (long long)1 << 60;
    P.tau2 = (float)c.tau_se; P.one_minus_tau2 = (float)(1.0 - c.tau_se);
    P.which = which == 2 ? 4 : which;                    // counter slot: 0 critic, 1 actor, 4 context encoder
    P.lr = which == 0 ? c.lr_critic : (which == 1 ? c.lr_actor : c.lr_ctx);
    P.cnt = h->cnt;
    P.tail = which == 0 ? TAIL_CRITIC_LOSS : (which == 1 ? TAIL_ALPHA_AND_LOSSES : TAIL_NONE);
    if (mode == 1) P.tail = TAIL_NONE;
    if (mode == 3) P.tail = TAIL_ALL;              // forked tail that also reduces the critic loss (no critic Adam launch)
    P.lq = h->lq.p; P.la = h->la.p; P.rsY = h->y.rs;
    P.logp_cur = h->logp.p + B; P.logstd_sum = h->logstd.p + B; P.rsLogp = h->logp.rs;
    P.tid = (const int*)h->tid.p; P.rsR = h->r.rs;
    P.log_alpha = h->params + L.off_alpha;
    P.m_alpha = h->adam_m + L.off_alpha; P.v_alpha = h->adam_v + L.off_alpha; P.g_alpha = h->grads + L.off_alpha;
    P.losses = h->losses; P.losses_host = h->loss_h_dev; P.R = R;
    int nb = (int)((n + 256 * 4 - 1) / (256 * 4));
    if (nb < 1) nb = 1;
    if (nb > 592) nb = 592;
    l.grid = dim3(nb + (P.tail != TAIL_NONE ? 1 : 0), R);
    l.block = dim3(256);
    l.join = true;                 // every gradient of the slice must have landed, including the forked weight gradients
    if (mode == 2 || mode == 3) { l.grid = dim3(1, R); l.join = false; l.branch = 1; }
    h->plan.push_back(l);
  };
  if (h->fused) {
    if (int rc = build_plan_fused(h, adam)) return rc;
  } else {
  // ---- Phase A: actor over [s2; s] and Q1,Q2 over (s,a), layer by layer -----------------
  for (int l = 0; l < (La > Lc ? La : Lc); ++l) {
    std::vector<GemmProb> ps;
    if (l < La) {
      const LayerOff& lo = L.actor[l];
      ps.push_back(fwd(l == 0 ? h->XA.p : h->hA[l - 1].p, l == 0 ? h->XA.rs : h->hA[l - 1].rs, 2 * B, lo, true,
                       h->hA[l].p, h->hA[l].rs));
    }
    if (l < Lc)
      for (int net = 0; net < 2; ++net) {
        const LayerOff& lo = L.q[net][l];
        ps.push_back(fwd(l == 0 ? h->XQ.p : netp(h->hQ[l - 1], net, lo.in), l == 0 ? h->XQ.rs : h->hQ[l - 1].rs, B, lo,
                         true, netp(h->hQ[l], net, lo.out), h->hQ[l].rs));
      }
    if (use_fork && La == Lc) {
      // Q1,Q2 on (s,a) are not needed before critic_heads, while the actor's output heads the policy_head -> target-critic
      // chain: the critics' layer goes to the fork stream (joined at critic_heads), the actor's stays on the main stream.
      cur_branch = 1; gemm_launch(std::vector<GemmProb>(ps.begin() + 1, ps.end())); cur_branch = 0;
      gemm_launch(std::vector<GemmProb>(ps.begin(), ps.begin() + 1));
    } else {
      gemm_launch(ps);
    }
  }
  {  // policy head
    Launch l;
    l.kind = L_POLICY;
    l.grid = dim3((2 * B + 7) / 8, R);
    l.block = dim3(256);
    l.pol = h->pol;
    h->use_eps_buf_idx = (int)h->plan.size();
    h->plan.push_back(l);
  }
  // ---- Phase B: target critics over (s2, a') ---------------------------------------------
  for (int l = 0; l < Lc; ++l) {
    std::vector<GemmProb> ps;
    for (int net = 0; net < 2; ++net) {
      const LayerOff& lo = L.qt[net][l];
      ps.push_back(fwd(l == 0 ? h->XT.p : netp(h->hT[l - 1], net, lo.in), l == 0 ? h->XT.rs : h->hT[l - 1].rs, B, lo,
                       true, netp(h->hT[l], net, lo.out), h->hT[l].rs));
    }
    gemm_launch(ps);
  }
  const int Hc = c.critic_hidden[Lc - 1], Ha = c.actor_hidden[La - 1];
  {  // critic heads: y, Q1, Q2, dQ
    Launch l;
    l.kind = L_CHEADS;
    l.join = true;                 // needs Q1,Q2 on (s,a), which may have run on the fork stream
    l.grid = dim3((B + 7) / 8, R);
    l.block = dim3(256);
    CriticHeadArgs& P = l.ch;
    memset(&P, 0, sizeof(P));
    P.hT = h->hT[Lc - 1].p; P.hQ = h->hQ[Lc - 1].p; P.rsHnet = (long long)B * Hc; P.rsHrep = h->hT[Lc - 1].rs; P.ldh = Hc;
    for (int net = 0; net < 2; ++net) {
      P.Wt[net] = W(L.qt[net][Lc].w); P.bt[net] = W(L.qt[net][Lc].b);
      P.Wq[net] = W(L.q[net][Lc].w); P.bq[net] = W(L.q[net][Lc].b);
    }
    P.rsP = rsP;
    P.r = h->r.p; P.d = h->d.p; P.tid = (const int*)h->tid.p; P.rsR = h->r.rs;
    P.logp = h->logp.p; P.rsLogp = h->logp.rs;
    P.log_alpha = W(L.off_alpha);
    P.y = h->y.p; P.q = h->q.p; P.dq = h->dq.p; P.lq = h->lq.p; P.rsY = h->y.rs;
    h->plan.push_back(l);
  }
  auto head_bwd = [&](bool policy, bool want_wgrad) {
    Launch l;
    l.kind = L_HEADBWD;
    HeadBwdArgs& P = l.hb;
    memset(&P, 0, sizeof(P));
    P.M = B;
    P.rsP = rsP; P.rsG = rsG;
    if (!policy) {
      P.NO = 1; P.Kdim = Hc; P.nets = 2;
      for (int net = 0; net < 2; ++net) {
        P.W[net] = W(L.q[net][Lc].w);
        P.dW[net] = want_wgrad ? Gp(L.q[net][Lc].w) : nullptr;
        P.db[net] = want_wgrad ? Gp(L.q[net][Lc].b) : nullptr;
      }
      const Buf& hb = want_wgrad ? h->hQ[Lc - 1] : h->hP[Lc - 1];
      const Buf& dq = want_wgrad ? h->dq : h->dqa;
      P.dout = dq.p; P.rsDoutNet = B; P.rsDoutRep = 2 * h->y.rs;
      P.h = hb.p; P.rsHnet = (long long)B * Hc; P.rsHrep = hb.rs; P.ldh = Hc;
      P.dh = h->dhQ[Lc - 1].p; P.rsDhNet = (long long)B * Hc; P.rsDhRep = h->dhQ[Lc - 1].rs; P.lddh = Hc;
    } else {
      const bool split = (long long)B * A > 2048;      // large batch: one tiny kernel computes d(mu|log_std) for all rows
      if (split) {
        Launch pl;
        pl.kind = L_POLICY_DOUT;
        PolicyDoutArgs& Q = pl.pdo;
        memset(&Q, 0, sizeof(Q));
        Q.dx = h->dxP.p; Q.rsDxNet = (long long)B * h->K.ldx; Q.rsDxRep = h->dxP.rs; Q.lddx = h->K.ldx;
        Q.psave = h->psave.p + (long long)B * A * kSaveW; Q.rsSave = h->psave.rs;
        Q.tid = (const int*)h->tid.p; Q.rsR = h->r.rs;
        Q.log_alpha = W(L.off_alpha); Q.rsP = rsP;
        Q.dout = h->dout_dbg.p; Q.dact = h->dact_dbg.p; Q.rsDout = h->dout_dbg.rs;
        Q.M = B;
        pl.grid = dim3((B * A + 255) / 256, R);
        pl.block = dim3(256);
        h->plan.push_back(pl);
      }
      P.NO = 2 * A; P.Kdim = Ha; P.nets = 1; P.policy_mode = split ? 0 : 1;
      if (split) { P.dout = h->dout_dbg.p; P.rsDoutNet = 0; P.rsDoutRep = h->dout_dbg.rs; }
      const LayerOff& lo = L.actor[La];
      P.W[0] = W(lo.w); P.dW[0] = Gp(lo.w); P.db[0] = Gp(lo.b);
      P.h = h->hA[La - 1].p + (long long)B * Ha; P.rsHrep = h->hA[La - 1].rs; P.ldh = Ha;   // rows B..2B-1 (= s half)
      P.dh = h->dhA[La - 1].p; P.rsDhRep = h->dhA[La - 1].rs; P.lddh = Ha;
      P.dx = h->dxP.p; P.rsDxNet = (long long)B * h->K.ldx; P.rsDxRep = h->dxP.rs; P.lddx = h->K.ldx;
      P.psave = h->psave.p + (long long)B * A * kSaveW; P.rsSave = h->psave.rs;
      P.tid = (const int*)h->tid.p; P.rsR = h->r.rs;
      P.log_alpha = W(L.off_alpha);
      P.dout_dbg = h->dout_dbg.p; P.dact_dbg = h->dact_dbg.p; P.rsDbg = h->dout_dbg.rs;
    }
    // large batches: rows cut into slices (4x the CTAs, a quarter of the serial row loop each); slice s >= 1 leaves its
    // partial head-weight gradient in gradient slice s, exactly like the split-K GEMM weight gradients
    P.row_slices = h->gslices;
    P.xs = (long long)R * L.trainable;
    for (int net = 0; net < P.nets; ++net)
      if (P.dW[net] && h->grads_x) { P.dWx[net] = h->grads_x + (P.dW[net] - h->grads); P.dbx[net] = h->grads_x + (P.db[net] - h->grads); }
    const int rows_per = (B + P.row_slices - 1) / P.row_slices;
    // 128-bit column mapping when every row pitch / tensor offset involved is a multiple of 4 floats (l.bn = 4 marks it)
    // -- for the scalar critic heads; the policy head (NO = 2 x act outputs, one network) would be left with 28 CTAs and
    // measured slower (12.6 vs 8.7 us at B = 1 024)
    const bool wide = P.NO == 1 && (P.Kdim % 4) == 0 && (P.ldh % 4) == 0 && (P.lddh % 4) == 0 && getenv("B200SAC_HEADBWD_NARROW") == nullptr;
    l.bn = wide ? 4 : 1;
    const int cols = wide ? kHb4Cols : kHbCols;
    l.grid = dim3(((P.Kdim + cols - 1) / cols) * ((B + rows_per - 1) / rows_per), P.nets, R);
    l.block = dim3(256);
    l.smem = ((size_t)pad4((int64_t)rows_per * P.NO) + (wide ? 1024 : 256) * (size_t)P.NO) * sizeof(float);   // (head_bwd4 aligns its reduction tiles)
    h->plan.push_back(l);
  };
  // ---- Phase C: critic backward + Adam/Polyak ----------------------------------------------
  head_bwd(false, true);
  for (int l = Lc - 1; l >= 0; --l) {
    std::vector<GemmProb> ps;
    for (int net = 0; net < 2; ++net) {
      const LayerOff& lo = L.q[net][l];
      const float* X = l == 0 ? h->XQ.p : netp(h->hQ[l - 1], net, lo.in);
      const long long rsX = l == 0 ? h->XQ.rs : h->hQ[l - 1].rs;
      ps.push_back(wgrad(netp(h->dhQ[l], net, lo.out), h->dhQ[l].rs, X, rsX, lo));
    }
    if (l > 0)
      for (int net = 0; net < 2; ++net) {
        const LayerOff& lo = L.q[net][l];
        ps.push_back(dgrad(netp(h->dhQ[l], net, lo.out), h->dhQ[l].rs, lo, netp(h->hQ[l - 1], net, lo.in), h->hQ[l - 1].rs,
                           netp(h->dhQ[l - 1], net, lo.in), h->dhQ[l - 1].rs));
      }
    else if (c.care)     // the critic loss also trains the critic's state encoder: need d(loss)/d(encoded state)
      for (int net = 0; net < 2; ++net) {
        const LayerOff& lo = L.q[net][0];
        ps.push_back(dgrad(netp(h->dhQ[0], net, lo.out), h->dhQ[0].rs, lo, nullptr, 0,
                           h->dxP.p + (long long)net * B * h->K.ldx, h->dxP.rs));
      }
    if (use_fork && l > 0) {        // ps = {wgrad q1, wgrad q2, dgrad q1, dgrad q2}
      cur_branch = 1; gemm_launch(std::vector<GemmProb>(ps.begin(), ps.begin() + 2)); cur_branch = 0;
      gemm_launch(std::vector<GemmProb>(ps.begin() + 2, ps.end()));
    } else {
      gemm_launch(ps);
    }
  }
  if (c.care) {
    {  // backward of the attention mix: dZk, d(att)
      Launch l;
      l.kind = L_CARE_MIXBWD;
      CareMixBwdArgs& P = l.cmixb;
      memset(&P, 0, sizeof(P));
      P.dx = h->dxP.p; P.rsDxNet = (long long)B * h->K.ldx; P.rsDxRep = h->dxP.rs; P.lddx = h->K.ldx;
      P.Z = h->mixZ[0].p; P.rsZ = h->mixZ[0].rs; P.kstride = (long long)2 * B * pitch(c.mix_out); P.ldz = pitch(c.mix_out);
      P.z_row_off = B;
      P.tab = h->careTab[0].p; P.rsTab = h->careTab[0].rs; P.row_w = h->care_row_w; P.off_att = h->care_off_att;
      P.tid = (const int*)h->tid.p; P.rsR = h->r.rs;
      P.dZ = h->mixDZ.p; P.rsDZ = h->mixDZ.rs; P.dkstride = (long long)B * pitch(c.mix_out); P.lddz = pitch(c.mix_out);
      P.datt = h->careDatt.p; P.rsDatt = h->careDatt.rs;
      P.B = B; P.K = Kenc; P.mo = c.mix_out; P.co = c.ctx_out;
      l.grid = dim3((B + 7) / 8, R);
      l.block = dim3(256);
      h->plan.push_back(l);
    }
    for (int l = nmix - 1; l >= 0; --l) {          // mixture-of-encoders backward, K problems per kind
      std::vector<GemmProb> ps;
      const LayerOff& lo = L.mix[l];
      const Buf& dzb = (l == nmix - 1) ? h->mixDZ : h->mixDH[l];
      for (int k = 0; k < Kenc; ++k) {
        GemmProb p;
        memset(&p, 0, sizeof(p));
        p.A = dzb.p + (long long)k * B * pitch(lo.out); p.rsA = dzb.rs; p.lda = pitch(lo.out);
        if (l == 0) { p.B = h->XS.p + (long long)B * h->K.obs; p.rsB = h->XS.rs; p.ldb = h->K.obs; }
        else {
          const Buf& ib = h->mixH[0][l - 1];
          p.B = ib.p + ((long long)k * 2 * B + B) * pitch(lo.in); p.rsB = ib.rs; p.ldb = pitch(lo.in);
        }
        p.C = Gp(lo.w + (long long)k * lo.out * lo.in); p.rsC = rsG; p.ldc = lo.in;
        p.C2 = Gp(lo.b + (long long)k * lo.out); p.rsC2 = rsG;
        p.M = lo.out; p.N = lo.in; p.K = B; p.mode = GEMM_WGRAD;
        ps.push_back(p);
      }
      if (l > 0)
        for (int k = 0; k < Kenc; ++k) {
          const Buf& ib = h->mixH[0][l - 1];
          GemmProb p;
          memset(&p, 0, sizeof(p));
          p.A = dzb.p + (long long)k * B * pitch(lo.out); p.rsA = dzb.rs; p.lda = pitch(lo.out);
          p.B = W(lo.w + (long long)k * lo.out * lo.in); p.rsB = rsP; p.ldb = lo.in;
          p.mask = ib.p + ((long long)k * 2 * B + B) * pitch(lo.in); p.rsMask = ib.rs; p.ldmask = pitch(lo.in);
          p.C = h->mixDH[l - 1].p + (long long)k * B * pitch(lo.in); p.rsC = h->mixDH[l - 1].rs; p.ldc = pitch(lo.in);
          p.M = B; p.N = lo.in; p.K = lo.out; p.mode = GEMM_DGRAD;
          ps.push_back(p);
        }
      gemm_launch(ps);
    }
    {  // per-task reduction + softmax backward, then the trunk / context-MLP weight gradients
      Launch l;
      l.kind = L_CARE_TABRED;
      CareTabReduceArgs& P = l.ctred;
      memset(&P, 0, sizeof(P));
      P.datt = h->careDatt.p; P.rsDatt = h->careDatt.rs;
      P.dx = h->dxP.p; P.rsDxNet = (long long)B * h->K.ldx; P.rsDxRep = h->dxP.rs; P.lddx = h->K.ldx;
      P.tab = h->careTab[0].p; P.rsTab = h->careTab[0].rs; P.row_w = h->care_row_w; P.off_att = h->care_off_att;
      P.tid = (const int*)h->tid.p; P.rsR = h->r.rs;
      P.dtab = h->careDtab.p; P.rsDtab = h->careDtab.rs;
      P.B = B; P.K = Kenc; P.co = c.ctx_out;
      l.grid = dim3(c.num_tasks, R);
      l.block = dim3(1024);
      h->plan.push_back(l);
      Launch l2;
      l2.kind = L_CARE_TABWG;
      CareTabWgradArgs& Q = l2.ctwg;
      memset(&Q, 0, sizeof(Q));
      Q.params = h->params; Q.rsP = rsP; Q.emb_off = L.off_emb;
      Q.tab = h->careTab[0].p; Q.rsTab = h->careTab[0].rs; Q.row_w = h->care_row_w;
      Q.dtab = h->careDtab.p; Q.rsDtab = h->careDtab.rs;
      Q.grads = h->grads; Q.rsG = rsG;
      Q.trunk = h->care_trunk; Q.ctx = h->care_ctx;
      Q.T = c.num_tasks; Q.K = Kenc; Q.co = c.ctx_out;
      Q.original = c.care == 2 ? 1 : 0; Q.off_ctx = h->care_off_ctx;
      size_t fl = 0;
      for (int j = 0; j < Q.trunk.n; ++j) fl += (size_t)c.num_tasks * Q.trunk.dims[j + 1];
      for (int j = 0; j < Q.ctx.n; ++j) fl += (size_t)c.num_tasks * Q.ctx.dims[j + 1];
      l2.smem = fl * sizeof(float);
      l2.grid = dim3(148, R);
      l2.block = dim3(256);
      h->plan.push_back(l2);
    }
  }
  adam(0, 0);
  if (c.care) {          // encoded states of s with the UPDATED critic encoder for the actor pass (learner.py:336-341)
    care_tables({2});
    care_encode({EncJob{2, B, B, h->XP.p, h->XP.rs, h->K.ldx, nullptr, 0, 0, 0}});
  }
  // ---- Phase D: actor pass through the updated critics ---------------------------------------
  for (int l = 0; l < Lc; ++l) {
    std::vector<GemmProb> ps;
    for (int net = 0; net < 2; ++net) {
      const LayerOff& lo = L.q[net][l];
      ps.push_back(fwd(l == 0 ? h->XP.p : netp(h->hP[l - 1], net, lo.in), l == 0 ? h->XP.rs : h->hP[l - 1].rs, B, lo, true,
                       netp(h->hP[l], net, lo.out), h->hP[l].rs));
    }
    gemm_launch(ps);
  }
  {
    Launch l;
    l.kind = L_AQHEADS;
    l.grid = dim3((B + 7) / 8, R);
    l.block = dim3(256);
    ActorQHeadArgs& P = l.aq;
    memset(&P, 0, sizeof(P));
    P.hP = h->hP[Lc - 1].p; P.rsHnet = (long long)B * Hc; P.rsHrep = h->hP[Lc - 1].rs; P.ldh = Hc;
    for (int net = 0; net < 2; ++net) { P.Wq[net] = W(L.q[net][Lc].w); P.bq[net] = W(L.q[net][Lc].b); }
    P.rsP = rsP;
    P.tid = (const int*)h->tid.p; P.rsR = h->r.rs;
    P.logp = h->logp.p + B; P.rsLogp = h->logp.rs;
    P.log_alpha = W(L.off_alpha);
    P.dqa = h->dqa.p; P.la = h->la.p; P.qmin = h->qmin.p; P.rsY = h->y.rs;
    h->plan.push_back(l);
  }
  head_bwd(false, false);
  for (int l = Lc - 1; l >= 0; --l) {
    std::vector<GemmProb> ps;
    for (int net = 0; net < 2; ++net) {
      const LayerOff& lo = L.q[net][l];
      if (l > 0)
        ps.push_back(dgrad(netp(h->dhQ[l], net, lo.out), h->dhQ[l].rs, lo, netp(h->hP[l - 1], net, lo.in), h->hP[l - 1].rs,
                           netp(h->dhQ[l - 1], net, lo.in), h->dhQ[l - 1].rs));
      else
        ps.push_back(dgrad(netp(h->dhQ[0], net, lo.out), h->dhQ[0].rs, lo, nullptr, 0,
                           h->dxP.p + (long long)net * B * h->K.ldx, h->dxP.rs));
    }
    gemm_launch(ps);
  }
  // ---- Phase E: policy backward + Adam + temperature -----------------------------------------
  head_bwd(true, true);
  for (int l = La - 1; l >= 0; --l) {
    std::vector<GemmProb> ps;
    const LayerOff& lo = L.actor[l];
    const float* X = l == 0 ? h->XA.p + (long long)B * lo.ld : h->hA[l - 1].p + (long long)B * lo.ld;
    const long long rsX = l == 0 ? h->XA.rs : h->hA[l - 1].rs;
    ps.push_back(wgrad(h->dhA[l].p, h->dhA[l].rs, X, rsX, lo));
    if (l > 0)
      ps.push_back(dgrad(h->dhA[l].p, h->dhA[l].rs, lo, h->hA[l - 1].p + (long long)B * lo.ld, h->hA[l - 1].rs,
                         h->dhA[l - 1].p, h->dhA[l - 1].rs));
    if (use_fork && l > 0) {
      cur_branch = 1; gemm_launch(std::vector<GemmProb>(ps.begin(), ps.begin() + 1)); cur_branch = 0;
      gemm_launch(std::vector<GemmProb>(ps.begin() + 1, ps.end()));
    } else {
      gemm_launch(ps);
    }
  }
  adam(1, 0);
  if (c.care == 2) adam(2, 0);        // update(): context_encoder_optimizer.step() (learner.py:399), gradients from the critic loss
  }   // generic (per-layer) plan

  if (plan_rc) return plan_rc;
  // upload problem tables and rebase
  if (!h->h_tprobs.empty()) {
    CU(cudaMalloc(&h->d_tprobs, h->h_tprobs.size() * sizeof(TcProb)));
    CU(cudaMemcpy(h->d_tprobs, h->h_tprobs.data(), h->h_tprobs.size() * sizeof(TcProb), cudaMemcpyHostToDevice));
    CU(tc_set_attrs());
  }
  if (!h->h_probs.empty()) {
    CU(cudaMalloc(&h->d_probs, h->h_probs.size() * sizeof(GemmProb)));
    CU(cudaMemcpy(h->d_probs, h->h_probs.data(), h->h_probs.size() * sizeof(GemmProb), cudaMemcpyHostToDevice));
  }
  for (auto& l : h->plan) {
    if (l.kind == L_GEMM_BIG || l.kind == L_GEMM_SMALL || l.kind == L_GEMM_THIN || l.kind == L_GEMM_TC) l.probs = h->d_probs + (size_t)(uintptr_t)l.probs;
    if (l.kind == L_GEMM_TC) l.tprobs = h->d_tprobs + (size_t)(uintptr_t)l.tprobs;
  }
  size_t max_smem = 0;
  for (auto& l : h->plan)
    if (l.kind == L_HEADBWD && l.smem > max_smem) max_smem = l.smem;
  if (max_smem > 200 * 1024) return fail(B200SAC_ERR_INVALID, "batch * head width too large for head_bwd smem");
  CU(cudaFuncSetAttribute(head_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)max_smem));
  CU(cudaFuncSetAttribute(head_bwd4_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)max_smem));
  return 0;
}

// Launch with programmatic stream serialization (PDL): the kernel may start while its predecessor
// drains; every kernel begins with griddepcontrol.wait (common.cuh::kstamp), so data dependencies hold.
static bool g_use_pdl = true;
template <typename... KArgs, typename... Args>
static cudaError_t launch_k(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args... args) {
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = g_use_pdl ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kern, KArgs(args)...);
}

// the same with a thread-block cluster of (1, 2, 1): the two CTAs with equal blockIdx.x / z are co-scheduled and can read
// each other's shared memory
template <typename... KArgs, typename... Args>
static cudaError_t launch_pair_k(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args... args) {
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
  cudaLaunchAttribute attr[2];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 1; attr[0].val.clusterDim.y = 2; attr[0].val.clusterDim.z = 1;
  attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[1].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = g_use_pdl ? 2 : 1;
  return cudaLaunchKernelEx(&cfg, kern, KArgs(args)...);
}

static int run_plan(b200sac* h, cudaStream_t st, bool use_eps_buf, cudaEvent_t* evs = nullptr, bool allow_fork = false) {
  bool fork_pending = false;
  for (size_t i = 0; i < h->plan.size(); ++i) {
    Launch& l = h->plan[i];
    if (evs) CU(cudaEventRecord(evs[i], st));
    cudaStream_t s = st;
    if (l.join && fork_pending) {                       // e.g. Adam: wait for the forked weight gradients
      CU(cudaStreamWaitEvent(st, h->ev_fork_done, 0));
      fork_pending = false;
    }
    const bool forked = allow_fork && l.branch == 1;
    if (forked) {                                       // runs beside the launches that follow on `st`
      CU(cudaEventRecord(h->ev_fork_src, st));
      CU(cudaStreamWaitEvent(h->fork, h->ev_fork_src, 0));
      s = h->fork;
    }
    switch (l.kind) {
      case L_POLICY_DOUT:
        launch_k(policy_dout_kernel, l.grid, l.block, 0, s, h->K, l.pdo);
        break;
      case L_CARE_TAB:
        launch_k(care_tables_kernel, l.grid, l.block, 0, s, l.ctab);
        break;
      case L_CARE_MIX:
        launch_k(care_mix_kernel, l.grid, l.block, 0, s, l.cmix);
        break;
      case L_CARE_MIXFWD:
        launch_k(care_mixfwd_kernel, l.grid, l.block, l.smem, s, l.cmf);
        break;
      case L_CARE_MIXBWD:
        launch_k(care_mix_bwd_kernel, l.grid, l.block, 0, s, l.cmixb);
        break;
      case L_CARE_TABRED:
        launch_k(care_tab_reduce_kernel, l.grid, l.block, 0, s, l.ctred);
        break;
      case L_CARE_TABWG:
        launch_k(care_tab_wgrad_kernel, l.grid, l.block, l.smem, s, l.ctwg);
        break;
      case L_GEMM_BIG:
      case L_GEMM_SMALL:
        launch_k(gemm_simt_kernel, l.grid, l.block, 0, s, l.grp);
        break;
      case L_GEMM_THIN:
        launch_k(gemm_thin_kernel, l.grid, l.block, 0, s, l.grp);
        break;
      case L_GEMM_TC:
        launch_k(tc_kernel(l.bn), l.grid, l.block, l.smem, s, l.tprobs);
        break;
      case L_POLICY: {
        PolicyHeadArgs P = l.pol;
        P.use_eps_buf = use_eps_buf ? 1 : 0;
        launch_k(policy_head_kernel, l.grid, l.block, 0, s, h->K, P);
        break;
      }
      case L_CHEADS:
        launch_k(critic_heads_kernel, l.grid, l.block, 0, s, h->K, l.ch);
        break;
      case L_AQHEADS:
        launch_k(actor_q_heads_kernel, l.grid, l.block, 0, s, h->K, l.aq);
        break;
      case L_HEADBWD:
        if (l.bn == 4) launch_k(head_bwd4_kernel<1>, l.grid, l.block, l.smem, s, h->K, l.hb);
        else launch_k(head_bwd_kernel, l.grid, l.block, l.smem, s, h->K, l.hb);
        break;
      case L_ADAM:
        launch_k(adam_kernel, l.grid, l.block, 0, s, h->K, l.ad);
        break;
      case L_CHAIN: {
        ChainArgs a = l.chain;
        a.pol.use_eps_buf = use_eps_buf ? 1 : 0;
        const bool f = a.job[0].kind == CJ_FWD;
        if (l.bn == 8) {
          if (f) launch_k(chain_kernel<true, 8>, l.grid, l.block, l.smem, s, a, h->K);
          else launch_k(chain_kernel<false, 8>, l.grid, l.block, l.smem, s, a, h->K);
        } else if (l.bn == 4) {
          if (f) launch_k(chain_kernel<true, 4>, l.grid, l.block, l.smem, s, a, h->K);
          else launch_k(chain_kernel<false, 4>, l.grid, l.block, l.smem, s, a, h->K);
        } else {
          if (f) launch_k(chain_kernel<true, 2>, l.grid, l.block, l.smem, s, a, h->K);
          else launch_k(chain_kernel<false, 2>, l.grid, l.block, l.smem, s, a, h->K);
        }
        break;
      }
      case L_WGRAD:
        launch_k(wgrad_kernel, l.grid, l.block, l.smem, s, l.wg, h->K);
        break;
      case L_CHAIN2:
        if (l.bn == 8) launch_pair_k(chain2_kernel<8>, l.grid, l.block, l.smem, s, l.chain2, h->K);
        else if (l.bn == 4) launch_pair_k(chain2_kernel<4>, l.grid, l.block, l.smem, s, l.chain2, h->K);
        else launch_pair_k(chain2_kernel<2>, l.grid, l.block, l.smem, s, l.chain2, h->K);
        break;
    }
    if (forked) {
      CU(cudaEventRecord(h->ev_fork_done, h->fork));
      fork_pending = true;
    }
  }
  if (fork_pending) CU(cudaStreamWaitEvent(st, h->ev_fork_done, 0));
  if (evs) CU(cudaEventRecord(evs[h->plan.size()], st));
  CU(cudaGetLastError());
  return 0;
}

extern "C" int b200sac_launches_per_step(b200sac_t* h, int32_t* n) {
  if (!h || !n) return fail(B200SAC_ERR_INVALID, "null argument");
  *n = (int32_t)h->plan.size() + 1;   // + ingest (the sampled-device path adds one more: index sampling)
  return 0;
}

extern "C" int b200sac_create(const b200sac_cfg* cfg, int32_t device, uint64_t seed, b200sac_t** out) {
  if (!out) return fail(B200SAC_ERR_INVALID, "out is NULL");
  *out = nullptr;
  if (int rc = check_cfg(cfg)) return rc;
  int ndev = 0;
  CU(cudaGetDeviceCount(&ndev));
  if (device < 0 || device >= ndev) return fail(B200SAC_ERR_INVALID, "device %d out of range (%d visible)", device, ndev);
  CU(cudaSetDevice(device));
  b200sac* h = new (std::nothrow) b200sac();
  if (!h) return fail(B200SAC_ERR_NOMEM, "out of host memory");
  h->cfg = *cfg;
  h->device = device;
  h->R = cfg->replicas;
  // programmatic dependent launch with the exit-time trigger only (see common.cuh::KStamp); B200SAC_PDL=0 turns it off
  if (const char* e = getenv("B200SAC_PDL")) g_use_pdl = (e[0] != '0');      // process-wide switch, read at every create

  build_layout(cfg, h->L);
  const Layout& L = h->L;
  const int B = cfg->batch, R = h->R, A = cfg->act_dim, obs = cfg->state_dim + cfg->num_tasks, xw = L.in_w + A;
  const int in_w = L.in_w;
  StepConst& K = h->K;
  memset(&K, 0, sizeof(K));
  K.B = B; K.obs = obs; K.act = A; K.T = cfg->num_tasks; K.xw = xw; K.in_w = in_w; K.care = cfg->care ? 1 : 0;
  K.ldxa = (int)pad4(in_w); K.ldx = (int)pad4(xw);
  const int ldxa = K.ldxa, ldx = K.ldx;
  K.Ha = cfg->actor_hidden[cfg->n_actor_hidden - 1];
  K.Hc = cfg->critic_hidden[cfg->n_critic_hidden - 1];
  K.gamma = (float)cfg->gamma; K.reward_scale = (float)cfg->reward_scale; K.action_scale = (float)cfg->action_scale;
  K.c_loss = (float)(1.0 / B / (cfg->weighted_loss ? (double)B : 1.0));
  K.inv_B = (float)(1.0 / B);
  K.tau = (float)cfg->tau; K.one_minus_tau = (float)(1.0 - cfg->tau);
  K.hbar = -(float)A;
  K.lr_actor = cfg->lr_actor; K.lr_critic = cfg->lr_critic; K.lr_alpha = cfg->lr_alpha;
  K.beta1 = cfg->beta1; K.beta2 = cfg->beta2; K.adam_eps = cfg->adam_eps;
  K.seed = seed;

#define CUH(call)                                                                                            \
  do {                                                                                                       \
    cudaError_t e__ = (call);                                                                                \
    if (e__ != cudaSuccess) {                                                                                \
      int rc__ = fail(e__ == cudaErrorMemoryAllocation ? B200SAC_ERR_NOMEM : B200SAC_ERR_CUDA, "%s failed: %s", #call, \
                      cudaGetErrorString(e__));                                                              \
      destroy_impl(h);                                                                                       \
      return rc__;                                                                                           \
    }                                                                                                        \
  } while (0)

  CUH(cudaMalloc(&h->params, sizeof(float) * L.arena * R));
  CUH(cudaMalloc(&h->adam_m, sizeof(float) * L.trainable * R));
  CUH(cudaMalloc(&h->adam_v, sizeof(float) * L.trainable * R));
  CUH(cudaMalloc(&h->grads, sizeof(float) * L.trainable * R));
  CUH(cudaMalloc(&h->cnt, sizeof(Counters) * R));
  CUH(cudaMalloc(&h->losses, sizeof(float) * kLossSlots * R * 4));
  CUH(cudaMemset(h->params, 0, sizeof(float) * L.arena * R));
  CUH(cudaMemset(h->adam_m, 0, sizeof(float) * L.trainable * R));
  CUH(cudaMemset(h->adam_v, 0, sizeof(float) * L.trainable * R));
  CUH(cudaMemset(h->grads, 0, sizeof(float) * L.trainable * R));
  h->gslices = (cfg->batch >= kSplitKMin && getenv("B200SAC_NO_SPLITK") == nullptr) ? kSplitK : 1;   // K of every weight gradient = batch
  if (h->gslices > 1) {     // never-written entries of slices >= 1 must read as zero (Adam sums all slices)
    CUH(cudaMalloc(&h->grads_x, sizeof(float) * L.trainable * R * (h->gslices - 1)));
    CUH(cudaMemset(h->grads_x, 0, sizeof(float) * L.trainable * R * (h->gslices - 1)));
  }
  {
    std::vector<Counters> c0((size_t)R);
    for (auto& c : c0) { memset(&c, 0, sizeof(c)); for (int i = 0; i < 5; ++i) c.b1p[i] = c.b2p[i] = 1.0; }
    CUH(cudaMemcpy(h->cnt, c0.data(), sizeof(Counters) * R, cudaMemcpyHostToDevice));
  }
  CUH(cudaMemset(h->losses, 0, sizeof(float) * kLossSlots * R * 4));

  // work slab
  size_t cur = 0;
  const int La = cfg->n_actor_hidden, Lc = cfg->n_critic_hidden;
  h->XA = carve(cur, (size_t)2 * B * ldxa, R);
  h->XQ = carve(cur, (size_t)B * ldx, R);
  h->XT = carve(cur, (size_t)B * ldx, R);
  h->XP = carve(cur, (size_t)B * ldx, R);
  h->XT.rs = h->XP.rs = h->XQ.rs;
  h->r = carve(cur, B, R);
  h->d = carve(cur, B, R);
  h->tid = carve(cur, B, R);
  h->eps = carve(cur, (size_t)2 * B * A, R);
  h->pout = carve(cur, (size_t)2 * B * 2 * A, R);
  h->psave = carve(cur, (size_t)2 * B * A * kSaveW, R);
  h->act_out = carve(cur, (size_t)2 * B * A, R);
  h->logp = carve(cur, (size_t)2 * B, R);
  h->logstd = carve(cur, (size_t)2 * B, R);
  h->y = carve(cur, B, R);
  h->lq = carve(cur, B, R);
  h->la = carve(cur, B, R);
  h->qmin = carve(cur, B, R);
  // q, dq, dqa are [2][B] with replica stride 2 * y.rs
  h->q = carve(cur, (size_t)2 * h->y.rs, R);
  h->dq = carve(cur, (size_t)2 * h->y.rs, R);
  h->dqa = carve(cur, (size_t)2 * h->y.rs, R);
  h->qt = carve(cur, (size_t)2 * h->y.rs, R);
  h->qp = carve(cur, (size_t)2 * h->y.rs, R);
  h->alpha = carve(cur, 64, R);
  h->dxP = carve(cur, (size_t)2 * B * ldx, R);
  h->dout_dbg = carve(cur, (size_t)B * 2 * A, R);
  h->dact_dbg = carve(cur, (size_t)B * 2 * A, R);
  h->dact_dbg.rs = h->dout_dbg.rs;
  for (int l = 0; l < La; ++l) {
    h->hA.push_back(carve(cur, (size_t)2 * B * cfg->actor_hidden[l], R));
    h->dhA.push_back(carve(cur, (size_t)B * cfg->actor_hidden[l], R));
  }
  for (int l = 0; l < Lc; ++l) {
    h->hQ.push_back(carve(cur, (size_t)2 * B * cfg->critic_hidden[l], R));
    h->hT.push_back(carve(cur, (size_t)2 * B * cfg->critic_hidden[l], R));
    h->hP.push_back(carve(cur, (size_t)2 * B * cfg->critic_hidden[l], R));
    h->dhQ.push_back(carve(cur, (size_t)2 * B * cfg->critic_hidden[l], R));
  }
  if (cfg->care) {
    const int Kenc = cfg->num_encoders, T = cfg->num_tasks;
    auto pitch = [](int w) { return (w + 3) & ~3; };
    h->XS = carve(cur, (size_t)2 * B * obs, R);
    // per-task table row: trunk activations per layer, attention, context-MLP activations per layer
    int off = 0;
    CareNet& tr = h->care_trunk;
    CareNet& cx = h->care_ctx;
    memset(&tr, 0, sizeof(tr)); memset(&cx, 0, sizeof(cx));
    const std::vector<LayerOff>& cxl = cfg->care == 2 ? L.cenc : L.ctx;      // CARE(O): the context net is the shared encoder
    tr.n = (int)L.trunk.size(); cx.n = (int)cxl.size();
    tr.dims[0] = cfg->care == 2 ? cfg->emb_dim : cfg->ctx_in;
    cx.dims[0] = cfg->ctx_in;
    for (int j = 0; j < tr.n; ++j) { tr.dims[j + 1] = L.trunk[j].out; tr.w[j] = L.trunk[j].w; tr.b[j] = L.trunk[j].b; tr.act_off[j] = off; off += L.trunk[j].out; }
    h->care_off_att = off; off += Kenc;
    for (int j = 0; j < cx.n; ++j) { cx.dims[j + 1] = cxl[j].out; cx.w[j] = cxl[j].w; cx.b[j] = cxl[j].b; cx.act_off[j] = off; off += cxl[j].out; }
    h->care_off_ctx = cx.act_off[cx.n - 1];
    h->care_row_w = off;
    for (int i = 0; i < 3; ++i) h->careTab[i] = carve(cur, (size_t)T * off, R);
    h->careDtab = carve(cur, (size_t)T * (Kenc + cfg->ctx_out), R);
    h->careDatt = carve(cur, (size_t)B * Kenc, R);
    const int rows_of[3] = {2 * B, B, B};
    for (int i = 0; i < 3; ++i) {
      for (int l = 0; l < cfg->n_mix_hidden; ++l) h->mixH[i].push_back(carve(cur, (size_t)Kenc * rows_of[i] * pitch(cfg->mix_hidden[l]), R));
      h->mixZ[i] = carve(cur, (size_t)Kenc * rows_of[i] * pitch(cfg->mix_out), R);
    }
    for (int l = 0; l < cfg->n_mix_hidden; ++l) h->mixDH.push_back(carve(cur, (size_t)Kenc * B * pitch(cfg->mix_hidden[l]), R));
    h->mixDZ = carve(cur, (size_t)Kenc * B * pitch(cfg->mix_out), R);
  }
  h->slab_floats = cur;
  CUH(cudaMalloc(&h->slab, cur * sizeof(float)));
  CUH(cudaMemset(h->slab, 0, cur * sizeof(float)));
  for (Buf* b : {&h->XA, &h->XQ, &h->XT, &h->XP, &h->r, &h->d, &h->tid, &h->eps, &h->pout, &h->psave, &h->act_out, &h->logp,
                 &h->logstd, &h->y, &h->lq, &h->la, &h->qmin, &h->q, &h->dq, &h->dqa, &h->dxP, &h->dout_dbg, &h->dact_dbg, &h->qt, &h->qp, &h->alpha})
    rebase(*b, h->slab);
  for (auto* v : {&h->hA, &h->dhA, &h->hQ, &h->hT, &h->hP, &h->dhQ})
    for (auto& b : *v) rebase(b, h->slab);
  if (cfg->care) {
    for (Buf* b : {&h->XS, &h->careTab[0], &h->careTab[1], &h->careTab[2], &h->careDtab, &h->careDatt, &h->mixZ[0], &h->mixZ[1],
                   &h->mixZ[2], &h->mixDZ})
      rebase(*b, h->slab);
    for (auto* v : {&h->mixH[0], &h->mixH[1], &h->mixH[2], &h->mixDH})
      for (auto& b : *v) rebase(b, h->slab);
  }
  if (h->q.rs != 2 * h->y.rs || h->dq.rs != 2 * h->y.rs || h->dqa.rs != 2 * h->y.rs || h->qt.rs != 2 * h->y.rs || h->qp.rs != 2 * h->y.rs) {
    destroy_impl(h);
    return fail(B200SAC_ERR_INVALID, "internal: q stride");
  }

  IngestOut& O = h->ing;
  O.XA = h->XA.p; O.XQ = h->XQ.p; O.XT = h->XT.p; O.XP = h->XP.p; O.r = h->r.p; O.d = h->d.p; O.eps = h->eps.p;
  O.tid = (int*)h->tid.p; O.cnt = h->cnt;
  O.rsXA = h->XA.rs; O.rsXQ = h->XQ.rs; O.rsR = h->r.rs; O.rsEps = h->eps.rs;
  O.XS = cfg->care ? h->XS.p : nullptr; O.rsXS = cfg->care ? h->XS.rs : 0;
  O.log_alpha = h->params + L.off_alpha; O.rsP = L.arena; O.alpha = h->alpha.p; O.rsAlpha = h->alpha.rs;
  if (h->d.rs != h->r.rs || h->tid.rs != h->r.rs || h->lq.rs != h->y.rs || h->la.rs != h->y.rs || h->qmin.rs != h->y.rs ||
      h->logstd.rs != h->logp.rs) {
    destroy_impl(h);
    return fail(B200SAC_ERR_INVALID, "internal: stride mismatch");
  }

  // parameter init: Xavier-uniform weights, zero biases, log_alpha = cfg; targets = locals
  {
    int tag = 0;
    for (const auto* net : {&L.actor, &L.q[0], &L.q[1]})
      for (const auto& lo : *net) {
        xavier_kernel<<<dim3(64, R), 256>>>(h->params + lo.w, L.arena, lo.out, lo.in, lo.ld, seed, tag++);
      }
    if (cfg->care) {     // mixture weights ~ N(0,1) (state_encoder.py:146-153); trunk / context MLP Xavier; embedding random
      for (const auto& lo : L.mix) {
        randn_kernel<<<dim3(64, R), 256>>>(h->params + lo.w, L.arena, (long long)cfg->num_encoders * lo.out * lo.in, seed, tag++);
        randn_kernel<<<dim3(8, R), 256>>>(h->params + lo.b, L.arena, (long long)cfg->num_encoders * lo.out, seed, tag++);
      }
      for (const auto* net : {&L.trunk, &L.ctx, &L.cenc})
        for (const auto& lo : *net) xavier_kernel<<<dim3(64, R), 256>>>(h->params + lo.w, L.arena, lo.out, lo.in, lo.ld, seed, tag++);
      randn_kernel<<<dim3(64, R), 256>>>(h->params + L.off_emb, L.arena, (long long)cfg->num_tasks * cfg->ctx_in, seed ^ 0x5EEDull, tag++);
    }
    std::vector<float> la((size_t)(cfg->num_tasks > 0 ? cfg->num_tasks : 1), (float)cfg->log_alpha_init);
    for (int rep = 0; rep < R; ++rep)
      CUH(cudaMemcpy(h->params + (size_t)rep * L.arena + L.off_alpha, la.data(), la.size() * sizeof(float), cudaMemcpyHostToDevice));
    polyak_kernel<<<dim3(128, R), 256>>>(h->params + L.critic_begin, L.arena, L.critic_n, L.target_delta, 1.0f, 0.0f);
    CUH(cudaGetLastError());
  }

  // staging (pinned host <-> device), side stream
  h->row_w = 2 * obs + A + 2;
  h->row_stride = (h->row_w + 31) / 32 * 32;   // 128-byte aligned transition rows
  h->stage_floats = (size_t)R * B * h->row_stride + (size_t)2 * R * B * A;   // rows + eps_next/eps_cur
  for (int i = 0; i < 2; ++i) {
    CUH(cudaMallocHost(&h->stage_h[i], h->stage_floats * sizeof(float)));
    CUH(cudaMalloc(&h->stage_d[i], h->stage_floats * sizeof(float)));
    CUH(cudaEventCreateWithFlags(&h->ev_copied[i], cudaEventDisableTiming));
    CUH(cudaEventCreateWithFlags(&h->ev_consumed[i], cudaEventDisableTiming));
  }
  CUH(cudaHostAlloc(&h->loss_h, sizeof(float) * R * 4 * kLossSlots, cudaHostAllocMapped));
  memset(h->loss_h, 0, sizeof(float) * R * 4 * kLossSlots);
  CUH(cudaHostGetDevicePointer((void**)&h->loss_h_dev, h->loss_h, 0));
  CUH(cudaStreamCreateWithFlags(&h->side, cudaStreamNonBlocking));
  CUH(cudaStreamCreateWithFlags(&h->own, cudaStreamNonBlocking));
  CUH(cudaStreamCreateWithFlags(&h->fork, cudaStreamNonBlocking));
  CUH(cudaEventCreateWithFlags(&h->ev_ingested, cudaEventDisableTiming));
  CUH(cudaEventCreateWithFlags(&h->ev_sampled, cudaEventDisableTiming));
  CUH(cudaEventCreateWithFlags(&h->ev_fork_src, cudaEventDisableTiming));
  CUH(cudaEventCreateWithFlags(&h->ev_fork_done, cudaEventDisableTiming));
  CUH(cudaEventCreateWithFlags(&h->ev_in, cudaEventDisableTiming));
  CUH(cudaEventCreateWithFlags(&h->ev_out, cudaEventDisableTiming));

  h->fused = fused_eligible(*cfg);
  if (int rc = build_plan(h)) {
    destroy_impl(h);
    return rc;
  }
  CUH(cudaDeviceSynchronize());
  *out = h;
  return 0;
}

extern "C" int b200sac_destroy(b200sac_t* h) { return destroy_impl(h); }

static int arena_of(b200sac* h, int which, float** p, int64_t* n) {
  switch (which) {
    case B200SAC_PARAMS: *p = h->params; *n = h->L.arena; return 0;
    case B200SAC_ADAM_M: *p = h->adam_m; *n = h->L.trainable; return 0;
    case B200SAC_ADAM_V: *p = h->adam_v; *n = h->L.trainable; return 0;
    case B200SAC_GRADS: *p = h->grads; *n = h->L.trainable; return 0;
  }
  return fail(B200SAC_ERR_INVALID, "unknown arena %d", which);
}

extern "C" int b200sac_arena_ptr(b200sac_t* h, int32_t which, float** dev_ptr, int64_t* floats_per_replica) {
  if (!h || !dev_ptr || !floats_per_replica) return fail(B200SAC_ERR_INVALID, "null argument");
  return arena_of(h, which, dev_ptr, floats_per_replica);
}

extern "C" int b200sac_export(b200sac_t* h, int32_t which, int32_t replica, float* buf, int64_t n_floats, void* stream) {
  if (!h || !buf) return fail(B200SAC_ERR_INVALID, "null argument");
  float* p; int64_t n;
  if (int rc = arena_of(h, which, &p, &n)) return rc;
  if (replica < 0 || replica >= h->R) return fail(B200SAC_ERR_INVALID, "replica %d out of range", replica);
  if (n_floats != n) return fail(B200SAC_ERR_INVALID, "arena %d holds %lld floats per replica, got %lld", which, (long long)n, (long long)n_floats);
  CU(cudaSetDevice(h->device));
  CU(cudaMemcpyAsync(buf, p + (size_t)replica * n, n * sizeof(float), cudaMemcpyDefault, (cudaStream_t)stream));
  CU(cudaStreamSynchronize((cudaStream_t)stream));
  if (which == B200SAC_GRADS && h->gslices > 1) {       // split-K slices: the gradient is their sum (same order as Adam's)
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, buf) != cudaSuccess || at.type == cudaMemoryTypeDevice) {
      cudaGetLastError();
      return fail(B200SAC_ERR_INVALID, "exporting split-K gradients needs a host buffer");
    }
    std::vector<float> tmp((size_t)n);
    for (int sidx = 1; sidx < h->gslices; ++sidx) {
      CU(cudaMemcpy(tmp.data(), h->grads_x + ((size_t)(sidx - 1) * h->R + replica) * n, n * sizeof(float), cudaMemcpyDeviceToHost));
      for (int64_t i = 0; i < n; ++i) buf[i] += tmp[(size_t)i];
    }
  }
  return 0;
}

// A few floats of one arena (e.g. log_alpha for the logger) without exporting the whole arena.
extern "C" int b200sac_read_range(b200sac_t* h, int32_t which, int32_t replica, int64_t offset, int64_t n_floats, float* out_host,
                                  void* stream) {
  if (!h || !out_host) return fail(B200SAC_ERR_INVALID, "null argument");
  float* p; int64_t n;
  if (int rc = arena_of(h, which, &p, &n)) return rc;
  if (replica < 0 || replica >= h->R) return fail(B200SAC_ERR_INVALID, "replica %d out of range", replica);
  if (offset < 0 || n_floats < 1 || offset + n_floats > n) return fail(B200SAC_ERR_INVALID, "range [%lld, +%lld) outside the arena", (long long)offset, (long long)n_floats);
  CU(cudaSetDevice(h->device));
  CU(cudaMemcpyAsync(out_host, p + (size_t)replica * n + offset, (size_t)n_floats * sizeof(float), cudaMemcpyDeviceToHost, (cudaStream_t)stream));
  CU(cudaStreamSynchronize((cudaStream_t)stream));
  return 0;
}

extern "C" int b200sac_import(b200sac_t* h, int32_t which, int32_t replica, const float* buf, int64_t n_floats, void* stream) {
  if (!h || !buf) return fail(B200SAC_ERR_INVALID, "null argument");
  float* p; int64_t n;
  if (int rc = arena_of(h, which, &p, &n)) return rc;
  if (replica < 0 || replica >= h->R) return fail(B200SAC_ERR_INVALID, "replica %d out of range", replica);
  if (n_floats != n) return fail(B200SAC_ERR_INVALID, "arena %d holds %lld floats per replica, got %lld", which, (long long)n, (long long)n_floats);
  CU(cudaSetDevice(h->device));
  CU(cudaMemcpyAsync(p + (size_t)replica * n, buf, n * sizeof(float), cudaMemcpyDefault, (cudaStream_t)stream));
  CU(cudaStreamSynchronize((cudaStream_t)stream));
  return 0;
}

extern "C" int b200sac_get_steps(b200sac_t* h, int32_t replica, int64_t steps[4]) {
  if (!h || !steps || replica < 0 || replica >= h->R) return fail(B200SAC_ERR_INVALID, "bad argument");
  CU(cudaSetDevice(h->device));
  Counters c;
  CU(cudaMemcpy(&c, h->cnt + replica, sizeof(c), cudaMemcpyDeviceToHost));
  steps[0] = c.v[0]; steps[1] = c.v[1]; steps[2] = c.v[2]; steps[3] = c.v[4];
  return 0;
}

extern "C" int b200sac_set_steps(b200sac_t* h, int32_t replica, const int64_t steps[4]) {
  if (!h || !steps || replica < 0 || replica >= h->R) return fail(B200SAC_ERR_INVALID, "bad argument");
  CU(cudaSetDevice(h->device));
  Counters c;
  CU(cudaMemcpy(&c, h->cnt + replica, sizeof(c), cudaMemcpyDeviceToHost));
  for (int i = 0; i < 4; ++i) {
    const int slot = i == 3 ? 4 : i;
    c.v[slot] = steps[i];
    c.b1p[slot] = pow(h->cfg.beta1, (double)steps[i]);
    c.b2p[slot] = pow(h->cfg.beta2, (double)steps[i]);
  }
  CU(cudaMemcpy(h->cnt + replica, &c, sizeof(c), cudaMemcpyHostToDevice));
  return 0;
}

// The legacy default stream cannot be captured into a graph.  When the caller passes it (NULL,
// which is also torch's default current stream) the step runs on the handle's own stream,
// ordered after everything already queued on the caller's stream, and the caller's stream is
// made to wait for it afterwards -- same ordering semantics, capturable.
struct StreamBridge {
  b200sac* h;
  cudaStream_t user, run;
  bool bridged;
  StreamBridge(b200sac* h_, void* s) : h(h_), user((cudaStream_t)s) {
    bridged = (user == nullptr || user == cudaStreamLegacy || user == cudaStreamPerThread);
    run = bridged ? h->own : user;
  }
  int begin() {
    if (!bridged) return 0;
    CU(cudaEventRecord(h->ev_in, user));
    CU(cudaStreamWaitEvent(run, h->ev_in, 0));
    return 0;
  }
  int end() {
    if (!bridged) return 0;
    CU(cudaEventRecord(h->ev_out, run));
    CU(cudaStreamWaitEvent(user, h->ev_out, 0));
    return 0;
  }
};

// ------------------------------------------------------------------------------------------
// Publication path: Learner.get_parameters() -> pickle -> Redis runs after EVERY update in the reference
// (LunarLander_Distributed_SAC/src/learner.py:272-276,298-299; MT10_Distributed_CARE/src/learner.py:412-417,442-443)
// and costs one synchronous .cpu() per tensor.  Here: a device-to-device snapshot of the requested arena
// ranges is enqueued in stream order (so it is the state after the steps enqueued so far, never a torn
// one), the D2H copy into pinned memory runs on a private stream behind the next steps, and the host
// only blocks in publish_wait.
// ------------------------------------------------------------------------------------------
extern "C" int b200sac_publish_begin(b200sac_t* h, int32_t replica, int32_t n_ranges, const int64_t* offsets, const int64_t* counts,
                                     void* stream) {
  if (!h || !offsets || !counts || n_ranges <= 0) return fail(B200SAC_ERR_INVALID, "bad argument");
  if (replica < 0 || replica >= h->R) return fail(B200SAC_ERR_INVALID, "replica %d out of range", replica);
  int64_t total = 0;
  for (int i = 0; i < n_ranges; ++i) {
    if (offsets[i] < 0 || counts[i] <= 0 || offsets[i] + counts[i] > h->L.arena)
      return fail(B200SAC_ERR_INVALID, "range %d [%lld, +%lld) outside the %lld-float parameter arena", i, (long long)offsets[i],
                  (long long)counts[i], (long long)h->L.arena);
    total += counts[i];
  }
  CU(cudaSetDevice(h->device));
  if (!h->pub) {
    CU(cudaStreamCreateWithFlags(&h->pub, cudaStreamNonBlocking));
    for (int i = 0; i < 2; ++i) {
      CU(cudaEventCreateWithFlags(&h->ev_pub_snap[i], cudaEventDisableTiming));
      CU(cudaEventCreateWithFlags(&h->ev_pub_done[i], cudaEventDisableTiming));
    }
  }
  if (h->pub_pending == 2) {            // both slots hold uncollected snapshots: the older one is superseded
    CU(cudaEventSynchronize(h->ev_pub_done[h->pub_head]));
    h->pub_pending = 1;
  }
  if (total > h->pub_cap) {
    CU(cudaStreamSynchronize(h->pub));
    for (int i = 0; i < 2; ++i) {
      cudaFree(h->pub_d[i]); h->pub_d[i] = nullptr;
      if (h->pub_h[i]) { cudaFreeHost(h->pub_h[i]); h->pub_h[i] = nullptr; }
      CU(cudaMalloc(&h->pub_d[i], (size_t)total * sizeof(float)));
      CU(cudaHostAlloc(&h->pub_h[i], (size_t)total * sizeof(float), cudaHostAllocDefault));
    }
    h->pub_cap = total;
    h->pub_pending = 0;
  }
  const int slot = h->pub_head;
  StreamBridge sb(h, stream);
  if (int rc = sb.begin()) return rc;
  const float* base = h->params + (size_t)replica * h->L.arena;
  int64_t at = 0;
  for (int i = 0; i < n_ranges; ++i) {
    CU(cudaMemcpyAsync(h->pub_d[slot] + at, base + offsets[i], (size_t)counts[i] * sizeof(float), cudaMemcpyDeviceToDevice, sb.run));
    at += counts[i];
  }
  CU(cudaEventRecord(h->ev_pub_snap[slot], sb.run));
  if (int rc = sb.end()) return rc;
  CU(cudaStreamWaitEvent(h->pub, h->ev_pub_snap[slot], 0));
  CU(cudaMemcpyAsync(h->pub_h[slot], h->pub_d[slot], (size_t)total * sizeof(float), cudaMemcpyDeviceToHost, h->pub));
  CU(cudaEventRecord(h->ev_pub_done[slot], h->pub));
  h->pub_n[slot] = total;
  h->pub_head ^= 1;
  h->pub_pending += 1;
  return 0;
}

extern "C" int b200sac_publish_wait(b200sac_t* h, const float** host_ptr, int64_t* n_floats) {
  if (!h || !host_ptr || !n_floats) return fail(B200SAC_ERR_INVALID, "null argument");
  if (h->pub_pending <= 0) return fail(B200SAC_ERR_STATE, "publish_wait without publish_begin");
  CU(cudaSetDevice(h->device));
  const int slot = (h->pub_head + 2 - h->pub_pending) & 1;      // the oldest snapshot not collected yet
  CU(cudaEventSynchronize(h->ev_pub_done[slot]));
  h->pub_pending -= 1;
  *host_ptr = h->pub_h[slot];
  *n_floats = h->pub_n[slot];
  return 0;
}

// ------------------------------------------------------------------------------------------
// Blob publication.  What Learner.run() stores in Redis after every update is ONE byte string: _pickle.dumps of
// {'actor': state_dict} (LunarLander_Distributed_SAC/src/learner.py:272-276,298-299).  Its shape never changes, so the
// caller hands over the byte image once (b200sac_blob_template: constant pickle bytes + where every payload float sits and
// which arena element it is -- pitch padding and the CARE [k][out][in] -> [k][in][out] transposition are just index maps);
// per publication a kernel, in stream order between two steps, gathers the floats into a device copy of the image, one
// D2H copy on the private stream brings it to pinned memory, and the host's only work is handing the bytes on.
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) blob_pack_kernel(const float* __restrict__ params, const int* __restrict__ src,
                                                        const int* __restrict__ dst, uint8_t* __restrict__ img, int n) {
  const int j = blockIdx.x * 256 + threadIdx.x;
  if (j >= n) return;
  const uint32_t v = __float_as_uint(params[src[j]]);
  uint8_t* o = img + dst[j];
  if ((reinterpret_cast<uintptr_t>(o) & 3) == 0) {
    *reinterpret_cast<uint32_t*>(o) = v;
  } else {                                  // pickle payloads start at arbitrary byte offsets
    o[0] = (uint8_t)v; o[1] = (uint8_t)(v >> 8); o[2] = (uint8_t)(v >> 16); o[3] = (uint8_t)(v >> 24);
  }
}

extern "C" int b200sac_blob_template(b200sac_t* h, int32_t replica, const uint8_t* image, int64_t image_bytes, int64_t n_floats,
                                     const int32_t* src_index, const int32_t* dst_byte) {
  if (!h || !image || image_bytes <= 0 || n_floats <= 0 || !src_index || !dst_byte) return fail(B200SAC_ERR_INVALID, "bad argument");
  if (replica < 0 || replica >= h->R) return fail(B200SAC_ERR_INVALID, "replica %d out of range", replica);
  if (n_floats > 0x7fffffffLL || image_bytes > 0x7fffffffLL) return fail(B200SAC_ERR_INVALID, "image too large");
  for (int64_t j = 0; j < n_floats; ++j) {
    if (src_index[j] < 0 || src_index[j] >= h->L.arena) return fail(B200SAC_ERR_INVALID, "payload float %lld reads arena index %d outside [0, %lld)", (long long)j, src_index[j], (long long)h->L.arena);
    if (dst_byte[j] < 0 || (int64_t)dst_byte[j] + 4 > image_bytes) return fail(B200SAC_ERR_INVALID, "payload float %lld lands outside the image", (long long)j);
  }
  CU(cudaSetDevice(h->device));
  if (!h->pub) CU(cudaStreamCreateWithFlags(&h->pub, cudaStreamNonBlocking));
  CU(cudaStreamSynchronize(h->pub));
  for (int i = 0; i < 2; ++i) {
    if (!h->ev_blob_snap[i]) CU(cudaEventCreateWithFlags(&h->ev_blob_snap[i], cudaEventDisableTiming));
    if (!h->ev_blob_done[i]) CU(cudaEventCreateWithFlags(&h->ev_blob_done[i], cudaEventDisableTiming));
    cudaFree(h->blob_d[i]); h->blob_d[i] = nullptr;
    if (h->blob_h[i]) { cudaFreeHost(h->blob_h[i]); h->blob_h[i] = nullptr; }
    CU(cudaMalloc(&h->blob_d[i], (size_t)image_bytes));
    CU(cudaHostAlloc(&h->blob_h[i], (size_t)image_bytes, cudaHostAllocDefault));
    CU(cudaMemcpy(h->blob_d[i], image, (size_t)image_bytes, cudaMemcpyHostToDevice));
  }
  cudaFree(h->blob_src); cudaFree(h->blob_dst); h->blob_src = h->blob_dst = nullptr;
  CU(cudaMalloc(&h->blob_src, (size_t)n_floats * sizeof(int)));
  CU(cudaMalloc(&h->blob_dst, (size_t)n_floats * sizeof(int)));
  CU(cudaMemcpy(h->blob_src, src_index, (size_t)n_floats * sizeof(int), cudaMemcpyHostToDevice));
  CU(cudaMemcpy(h->blob_dst, dst_byte, (size_t)n_floats * sizeof(int), cudaMemcpyHostToDevice));
  h->blob_bytes = image_bytes; h->blob_nf = n_floats; h->blob_replica = replica;
  h->blob_head = 0; h->blob_pending = 0;
  return 0;
}

extern "C" int b200sac_blob_begin(b200sac_t* h, void* stream) {
  if (!h) return fail(B200SAC_ERR_INVALID, "null handle");
  if (h->blob_nf <= 0) return fail(B200SAC_ERR_STATE, "blob_begin without blob_template");
  CU(cudaSetDevice(h->device));
  if (h->blob_pending == 2) {           // both images hold uncollected blobs: the older one is superseded
    CU(cudaEventSynchronize(h->ev_blob_done[h->blob_head]));
    h->blob_pending = 1;
  }
  const int slot = h->blob_head;
  StreamBridge sb(h, stream);
  if (int rc = sb.begin()) return rc;
  // (slot reuse: the D2H of the blob begun two calls ago was collected or superseded above, so image `slot` is idle)
  const float* base = h->params + (size_t)h->blob_replica * h->L.arena;
  blob_pack_kernel<<<(unsigned)((h->blob_nf + 255) / 256), 256, 0, sb.run>>>(base, h->blob_src, h->blob_dst, h->blob_d[slot], (int)h->blob_nf);
  CU(cudaGetLastError());
  CU(cudaEventRecord(h->ev_blob_snap[slot], sb.run));
  if (int rc = sb.end()) return rc;
  CU(cudaStreamWaitEvent(h->pub, h->ev_blob_snap[slot], 0));
  CU(cudaMemcpyAsync(h->blob_h[slot], h->blob_d[slot], (size_t)h->blob_bytes, cudaMemcpyDeviceToHost, h->pub));
  CU(cudaEventRecord(h->ev_blob_done[slot], h->pub));
  h->blob_head ^= 1;
  h->blob_pending += 1;
  return 0;
}

extern "C" int b200sac_blob_wait(b200sac_t* h, const uint8_t** host_ptr, int64_t* n_bytes) {
  if (!h || !host_ptr || !n_bytes) return fail(B200SAC_ERR_INVALID, "null argument");
  if (h->blob_pending <= 0) return fail(B200SAC_ERR_STATE, "blob_wait without blob_begin");
  CU(cudaSetDevice(h->device));
  const int slot = (h->blob_head + 2 - h->blob_pending) & 1;    // the oldest blob not collected yet
  CU(cudaEventSynchronize(h->ev_blob_done[slot]));
  h->blob_pending -= 1;
  *host_ptr = h->blob_h[slot];
  *n_bytes = h->blob_bytes;
  return 0;
}

// ------------------------------------------------------------------------------------------
// step variants.  variant 0: split device arrays; 1: packed rows (dense, staged); 2: replay gather
// ------------------------------------------------------------------------------------------
// variant 2 sampling modes (multi-step graphs): SAMPLE_INLINE = sample on `st` right before the gather (one step per graph);
// SAMPLE_DONE = the indices of this step were already drawn on the fork stream (wait for them); `fork_next` = once this
// step's gather has consumed the index buffer and bumped the step counter, draw the NEXT step's indices on the fork stream
// -- that kernel then overlaps the whole step instead of heading its critical path.
enum { SAMPLE_INLINE = 0, SAMPLE_DONE = 1 };
static int enqueue_body(b200sac* h, cudaStream_t st, int variant, const void* const* p, b200sac_replay* rb,
                        cudaEvent_t* evs = nullptr, int sample_mode = SAMPLE_INLINE, bool fork_next = false) {
  if (evs) CU(cudaEventRecord(evs[0], st));
  const int B = h->cfg.batch, R = h->R;
  dim3 grid((B + 7) / 8, R), block(256);
  if (grid.x > 64) grid.x = 64;
  bool use_eps = false;
  if (variant == 0) {
    use_eps = p[5] != nullptr;
    launch_k(ingest_split_kernel, grid, block, 0, st, h->K, h->ing, (const float*)p[0], (const float*)p[1], (const float*)p[2],
             (const float*)p[3], (const float*)p[4], (const float*)p[5], (const float*)p[6]);
  } else if (variant == 1) {
    const float* rows = (const float*)p[0];
    const float* e = (const float*)p[1];
    use_eps = e != nullptr;
    if (use_eps) {
      // eps staged as [R][B][A] next, then [R][B][A] cur: reuse the split ingest just for the noise
      // (rows carry the transition itself)
    }
    launch_k(ingest_rows_kernel, grid, block, 0, st, h->K, h->ing, rows, (long long)B * h->row_stride, h->row_stride,
             (const int*)nullptr, (long long)0);
    if (use_eps) {
      const size_t n = (size_t)B * h->cfg.act_dim * sizeof(float);
      for (int rep = 0; rep < R; ++rep) {
        CU(cudaMemcpyAsync(h->eps.p + rep * h->eps.rs, e + (size_t)rep * B * h->cfg.act_dim, n, cudaMemcpyDeviceToDevice, st));
        CU(cudaMemcpyAsync(h->eps.p + rep * h->eps.rs + (size_t)B * h->cfg.act_dim,
                           e + (size_t)(R + rep) * B * h->cfg.act_dim, n, cudaMemcpyDeviceToDevice, st));
      }
    }
  } else {
    auto sample_on = [&](cudaStream_t s2) {
      return launch_k(sample_indices_kernel, dim3(R), dim3(B > 256 ? 512 : 256), 0, s2, h->K,   // 98 regs/thread: 512 threads fit
                      (const Counters*)h->cnt, (const long long*)rb->d_fill, rb->cap_per_task, rb->d_idx, (long long)B, rb->seed);
    };
    if (sample_mode == SAMPLE_INLINE) sample_on(st);
    else CU(cudaStreamWaitEvent(st, h->ev_sampled, 0));
    launch_k(ingest_rows_kernel, grid, block, 0, st, h->K, h->ing, (const float*)rb->rows, rb->rs_rows, h->row_stride,
             (const int*)rb->d_idx, (long long)B);
    if (fork_next) {
      CU(cudaEventRecord(h->ev_ingested, st));
      CU(cudaStreamWaitEvent(h->fork, h->ev_ingested, 0));
      sample_on(h->fork);
      CU(cudaEventRecord(h->ev_sampled, h->fork));
    }
  }
  CU(cudaGetLastError());
  return run_plan(h, st, use_eps, evs ? evs + 1 : nullptr, evs == nullptr && !h->stamping);
}

// nsteps > 1 (device-ring sampling only): that many consecutive gradient steps captured in ONE graph, so a pipelined
// run pays the graph-launch gap (~3-4 us between two graph launches on B200) once per graph.  A run of n steps is cut
// greedily into graphs of 8, 4, 2 and 1 steps.
constexpr int kGraphSteps = 8;
static int get_graph(b200sac* h, cudaStream_t st, int variant, const void* const* p, int np, b200sac_replay* rb, int nsteps,
                     cudaGraphExec_t* out) {
  GraphKey key;
  memset(&key, 0, sizeof(key));
  key.variant = variant + 4 * (h->stamping ? 1 : 0) + 16 * (nsteps - 1);      // the timeline run captures unforked graphs
  for (int i = 0; i < np && i < 9; ++i) key.p[i] = p[i];
  if (rb) key.p[8] = rb;
  auto it = h->graphs.find(key);
  if (it == h->graphs.end()) {
    if (h->graphs.size() >= 64) {   // bound the cache: drop everything (pointers churn)
      for (auto& kv : h->graphs) cudaGraphExecDestroy(kv.second);
      h->graphs.clear();
    }
    cudaGraph_t g = nullptr;
    CU(cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal));
    int rc = 0;
    for (int k = 0; k < nsteps && rc == 0; ++k)
      rc = enqueue_body(h, st, variant, p, rb, nullptr, (nsteps > 1 && k > 0) ? SAMPLE_DONE : SAMPLE_INLINE, nsteps > 1 && k + 1 < nsteps);
    cudaError_t e = cudaStreamEndCapture(st, &g);
    if (rc) { if (g) cudaGraphDestroy(g); return rc; }
    if (e != cudaSuccess) return fail(B200SAC_ERR_CUDA, "graph capture failed: %s", cudaGetErrorString(e));
    cudaGraphExec_t ge = nullptr;
    e = cudaGraphInstantiate(&ge, g, 0);
    cudaGraphDestroy(g);
    if (e != cudaSuccess) return fail(B200SAC_ERR_CUDA, "graph instantiate failed: %s", cudaGetErrorString(e));
    if (cudaGraphUpload(ge, st) != cudaSuccess) cudaGetLastError();    // best effort: first launch does not pay the upload
    it = h->graphs.emplace(key, ge).first;
  }
  *out = it->second;
  return 0;
}

static int launch_step(b200sac* h, cudaStream_t st, int variant, const void* const* p, int np, b200sac_replay* rb, int nsteps = 1) {
  cudaGraphExec_t ge = nullptr;
  if (int rc = get_graph(h, st, variant, p, np, rb, nsteps, &ge)) return rc;
  CU(cudaGraphLaunch(ge, st));
  h->host_steps += nsteps;
  return 0;
}

// Capture + instantiate every graph the sampled path can launch (device ring: the 8/4/2/1-step graphs; host ring: the
// staged one-step graphs of both staging slots) without running a step, so that no later call pays graph construction.
extern "C" int b200sac_prepare(b200sac_t* h, b200sac_replay_t* rb, void* stream) {
  if (!h || !rb || rb->h != h) return fail(B200SAC_ERR_INVALID, "bad handle");
  CU(cudaSetDevice(h->device));
  StreamBridge sb(h, stream);
  if (int rc = sb.begin()) return rc;
  cudaGraphExec_t ge = nullptr;
  if (rb->where == 0) {
    const void* p[1] = {rb->rows};
    for (int n = kGraphSteps; n >= 1; n >>= 1)
      if (int rc = get_graph(h, sb.run, 2, p, 1, rb, n, &ge)) return rc;
  } else {
    for (int slot = 0; slot < 2; ++slot) {
      const void* p[2] = {h->stage_d[slot], nullptr};
      if (int rc = get_graph(h, sb.run, 1, p, 2, nullptr, 1, &ge)) return rc;
    }
  }
  if (int rc = sb.end()) return rc;
  CU(cudaStreamSynchronize(sb.run));
  return 0;
}

extern "C" int b200sac_step(b200sac_t* h, const float* s, const float* a, const float* r, const float* s2, const float* d,
                            const float* eps_next, const float* eps_cur, void* stream) {
  if (!h || !s || !a || !r || !s2 || !d) return fail(B200SAC_ERR_INVALID, "null minibatch pointer");
  if ((eps_next == nullptr) != (eps_cur == nullptr)) return fail(B200SAC_ERR_INVALID, "eps_next and eps_cur must both be given or both NULL");
  CU(cudaSetDevice(h->device));
  // The caller's arrays are copied (device to device, in stream order) into handle-owned buffers, so the captured graph
  // sees the same pointers whatever tensors the caller passes: one graph per (with / without injected noise), never a
  // re-capture per call.
  const size_t RB = (size_t)h->R * h->cfg.batch, obs = (size_t)h->K.obs, A = (size_t)h->K.act;
  const size_t n_s = RB * obs, n_a = RB * A, n_1 = RB;
  if (!h->split_d) CU(cudaMalloc(&h->split_d, (2 * n_s + 3 * n_a + 2 * n_1) * sizeof(float)));
  float* ds = h->split_d; float* da = ds + n_s; float* dr = da + n_a; float* ds2 = dr + n_1; float* dd = ds2 + n_s;
  float* de1 = dd + n_1; float* de2 = de1 + n_a;
  StreamBridge sb(h, stream);
  if (int rc = sb.begin()) return rc;
  CU(cudaMemcpyAsync(ds, s, n_s * sizeof(float), cudaMemcpyDefault, sb.run));
  CU(cudaMemcpyAsync(da, a, n_a * sizeof(float), cudaMemcpyDefault, sb.run));
  CU(cudaMemcpyAsync(dr, r, n_1 * sizeof(float), cudaMemcpyDefault, sb.run));
  CU(cudaMemcpyAsync(ds2, s2, n_s * sizeof(float), cudaMemcpyDefault, sb.run));
  CU(cudaMemcpyAsync(dd, d, n_1 * sizeof(float), cudaMemcpyDefault, sb.run));
  if (eps_next) {
    CU(cudaMemcpyAsync(de1, eps_next, n_a * sizeof(float), cudaMemcpyDefault, sb.run));
    CU(cudaMemcpyAsync(de2, eps_cur, n_a * sizeof(float), cudaMemcpyDefault, sb.run));
  }
  const void* p[7] = {ds, da, dr, ds2, dd, eps_next ? de1 : nullptr, eps_next ? de2 : nullptr};
  if (int rc = launch_step(h, sb.run, 0, p, 7, nullptr)) return rc;
  return sb.end();
}

// pack one replica-major minibatch into packed rows in pinned staging
static void pack_rows(const b200sac* h, float* dst, const float* s, const float* a, const float* r, const float* s2,
                      const float* d) {
  const int B = h->cfg.batch, R = h->R, obs = h->K.obs, A = h->K.act, rs = h->row_stride;
  for (long long i = 0; i < (long long)R * B; ++i) {
    float* row = dst + i * rs;
    memcpy(row, s + i * obs, obs * sizeof(float));
    memcpy(row + obs, a + i * A, A * sizeof(float));
    row[obs + A] = r[i];
    memcpy(row + obs + A + 1, s2 + i * obs, obs * sizeof(float));
    row[2 * obs + A + 1] = d[i];
  }
}

// stage slot -> device on the side stream, make `st` wait for it, run the step from the staged rows
static int staged_step(b200sac* h, cudaStream_t st, int slot, bool with_eps) {
  const size_t rows_f = (size_t)h->R * h->cfg.batch * h->row_stride;
  const size_t eps_f = (size_t)2 * h->R * h->cfg.batch * h->cfg.act_dim;
  CU(cudaMemcpyAsync(h->stage_d[slot], h->stage_h[slot], (rows_f + (with_eps ? eps_f : 0)) * sizeof(float),
                     cudaMemcpyHostToDevice, h->side));
  CU(cudaEventRecord(h->ev_copied[slot], h->side));
  CU(cudaStreamWaitEvent(st, h->ev_copied[slot], 0));
  const void* p[2] = {h->stage_d[slot], with_eps ? h->stage_d[slot] + rows_f : nullptr};
  if (int rc = launch_step(h, st, 1, p, 2, nullptr)) return rc;
  CU(cudaEventRecord(h->ev_consumed[slot], st));
  h->stage_used[slot] = true;
  return 0;
}

static int acquire_slot(b200sac* h, int* slot) {
  int s = h->stage_slot;
  if (s == h->prefetch_slot) h->prefetch_slot = -1;          // the slot is being reused: its prefetched batch is void
  h->stage_slot ^= 1;
  if (h->stage_used[s]) {
    CU(cudaEventSynchronize(h->ev_consumed[s]));          // host may overwrite the pinned slot
    CU(cudaStreamWaitEvent(h->side, h->ev_consumed[s], 0));   // and the side stream the device slot
  }
  *slot = s;
  return 0;
}

static int fetch_losses(b200sac* h, cudaStream_t st, int n_last, float* out) {
  if (n_last < 1 || n_last > kLossSlots || n_last > h->host_steps)
    return fail(B200SAC_ERR_INVALID, "n_last=%d out of range (steps so far %lld, ring %d)", n_last, h->host_steps, kLossSlots);
  const size_t per = (size_t)h->R * 4;
  CU(cudaStreamSynchronize(st));       // the tail kernels wrote the mapped host ring directly
  for (int i = 0; i < n_last; ++i) {
    const long long step = h->host_steps - n_last + i;
    const long long slot = step % kLossSlots;
    memcpy(out + (size_t)i * per, h->loss_h + (size_t)slot * per, per * sizeof(float));
  }
  return 0;
}

extern "C" int b200sac_step_host(b200sac_t* h, const float* s, const float* a, const float* r, const float* s2,
                                 const float* d, const float* eps_next, const float* eps_cur, float* out_losses, void* stream) {
  if (!h || !s || !a || !r || !s2 || !d) return fail(B200SAC_ERR_INVALID, "null minibatch pointer");
  if ((eps_next == nullptr) != (eps_cur == nullptr)) return fail(B200SAC_ERR_INVALID, "eps_next and eps_cur must both be given or both NULL");
  CU(cudaSetDevice(h->device));
  StreamBridge sb(h, stream);
  if (int rc = sb.begin()) return rc;
  cudaStream_t st = sb.run;
  int slot;
  if (int rc = acquire_slot(h, &slot)) return rc;
  pack_rows(h, h->stage_h[slot], s, a, r, s2, d);
  if (eps_next) {
    const size_t rows_f = (size_t)h->R * h->cfg.batch * h->row_stride;
    const size_t n = (size_t)h->R * h->cfg.batch * h->cfg.act_dim;
    memcpy(h->stage_h[slot] + rows_f, eps_next, n * sizeof(float));
    memcpy(h->stage_h[slot] + rows_f + n, eps_cur, n * sizeof(float));
  }
  if (int rc = staged_step(h, st, slot, eps_next != nullptr)) return rc;
  if (out_losses)
    if (int rc = fetch_losses(h, st, 1, out_losses)) return rc;
  return sb.end();
}

static const char* launch_name(const Launch& l, const std::vector<GemmProb>& hp, const GemmProb* dbase) {
  switch (l.kind) {
    case L_GEMM_TC: {
      const GemmProb& p0 = hp[(size_t)(l.probs - dbase)];
      const GemmProb& pl = hp[(size_t)(l.probs - dbase) + l.G - 1];
      const bool w = l.bn == 128;
      if (p0.mode == GEMM_FWD) return w ? "gemm_fwd(tcgen05 128x128)" : "gemm_fwd(tcgen05)";
      if (p0.mode == GEMM_WGRAD && pl.mode == GEMM_DGRAD) return w ? "gemm_wgrad+dgrad(tcgen05 128x128)" : "gemm_wgrad+dgrad(tcgen05)";
      if (p0.mode == GEMM_WGRAD) return w ? "gemm_wgrad(tcgen05 128x128)" : "gemm_wgrad(tcgen05)";
      return w ? "gemm_dgrad(tcgen05 128x128)" : "gemm_dgrad(tcgen05)";
    }
    case L_GEMM_BIG:
    case L_GEMM_SMALL: {
      const GemmProb& p0 = hp[(size_t)(l.probs - dbase)];
      const GemmProb& pl = hp[(size_t)(l.probs - dbase) + l.G - 1];
      if (p0.mode == GEMM_FWD) return "gemm_fwd(ffma)";
      if (p0.mode == GEMM_WGRAD && pl.mode == GEMM_DGRAD) return "gemm_wgrad+dgrad(ffma)";
      if (p0.mode == GEMM_WGRAD) return "gemm_wgrad(ffma)";
      return "gemm_dgrad(ffma)";
    }
    case L_GEMM_THIN: {
      const GemmProb& p0 = hp[(size_t)(l.probs - dbase)];
      return p0.mode == GEMM_WGRAD ? "gemm_wgrad(thin)" : "gemm_dgrad(thin)";
    }
    case L_POLICY_DOUT: return "policy_dout";
    case L_CARE_TAB: return "care_tables";
    case L_CARE_MIX: return "care_mix";
    case L_CARE_MIXFWD: return "care_mixture_fwd+mix";
    case L_CARE_MIXBWD: return "care_mix_bwd";
    case L_CARE_TABRED: return "care_tab_reduce";
    case L_CARE_TABWG: return "care_tab_wgrad";
    case L_POLICY: return "policy_head";
    case L_CHEADS: return "critic_heads";
    case L_AQHEADS: return "actor_q_heads";
    case L_HEADBWD: return (l.hb.policy_mode || l.hb.NO > 1) ? "head_bwd(policy)" : "head_bwd(q)";
    case L_CHAIN:
    case L_CHAIN2:
    case L_WGRAD: return l.label ? l.label : "chain";
    case L_ADAM:
      if (l.ad.which == 1 && l.branch == 1) return "alpha+losses(forked)";
      if (l.ad.which == 1 && l.ad.tail == TAIL_NONE) return "adam_actor";
      return l.ad.which == 0 ? "adam_critic+polyak" : (l.ad.which == 1 ? "adam_actor+alpha" : "adam_context_encoder");
  }
  return "?";
}

// Eager (non-graph) run of `iters` sampled steps with a CUDA event between every launch.
// out_ms[i] = mean device time of launch i (i = 0 is sampling + ingest); names are returned as a
// ';'-separated list.  This is what bench.py uses for the per-kernel roofline numbers.
extern "C" int b200sac_profile_step(b200sac_t* h, b200sac_replay_t* rb, int32_t iters, float* out_ms, int32_t cap,
                                    int32_t* n_out, char* names, int32_t names_cap, void* stream) {
  if (!h || !rb || rb->h != h || rb->where != 0 || !out_ms || !n_out) return fail(B200SAC_ERR_INVALID, "profile_step needs a device ring");
  CU(cudaSetDevice(h->device));
  const int n = (int)h->plan.size() + 1;
  *n_out = n;
  if (cap < n) return fail(B200SAC_ERR_INVALID, "need room for %d launches", n);
  StreamBridge sb(h, stream);
  if (int rc = sb.begin()) return rc;
  std::vector<cudaEvent_t> evs((size_t)n + 1);
  for (auto& e : evs) CU(cudaEventCreate(&e));
  std::vector<double> acc((size_t)n, 0.0);
  const void* p[1] = {rb->rows};
  for (int it = 0; it < iters; ++it) {
    if (int rc = enqueue_body(h, sb.run, 2, p, rb, evs.data())) return rc;
    h->host_steps += 1;
    CU(cudaStreamSynchronize(sb.run));
    for (int i = 0; i < n; ++i) {
      float ms = 0.f;
      CU(cudaEventElapsedTime(&ms, evs[i], evs[i + 1]));
      acc[i] += ms;
    }
  }
  for (int i = 0; i < n; ++i) out_ms[i] = (float)(acc[i] / iters);
  for (auto& e : evs) cudaEventDestroy(e);
  if (names && names_cap > 0) {
    std::string s = "sample+ingest";
    for (auto& l : h->plan) { s += ";"; s += launch_name(l, h->h_probs, h->d_probs); }
    snprintf(names, names_cap, "%s", s.c_str());
  }
  return sb.end();
}

// Stand-alone run of one GEMM engine on caller-provided DEVICE arrays (parity tests):
// engine 0 = 32x32-tile FFMA (gemm_simt.cuh), 1 = tcgen05 3xTF32 (gemm_tc.cuh), 2 = thin backward (gemm_thin.cuh).
static int tc_gemm_test_impl(int32_t mode, int32_t M, int32_t N, int32_t K, const float* A, int32_t lda, const float* B, int32_t ldb,
                             const float* bias, const float* mask, int32_t ldmask, float* C, int32_t ldc, float* C2, int32_t relu,
                             void* stream);
extern "C" int b200sac_gemm_test(int32_t engine, int32_t mode, int32_t M, int32_t N, int32_t K, const float* A, int32_t lda,
                                 const float* B, int32_t ldb, const float* bias, const float* mask, int32_t ldmask, float* C,
                                 int32_t ldc, float* C2, int32_t relu, void* stream) {
  if (engine == 1) return tc_gemm_test_impl(mode, M, N, K, A, lda, B, ldb, bias, mask, ldmask, C, ldc, C2, relu, stream);
  if (!A || !B || !C || M < 1 || N < 1 || K < 1 || mode < 0 || mode > 2) return fail(B200SAC_ERR_INVALID, "bad argument");
  GemmGroup grp;
  memset(&grp, 0, sizeof(grp));
  grp.G = 1;
  GemmProb& p = grp.p[0];
  p.A = A; p.B = B; p.bias = bias; p.mask = mask; p.C = C; p.C2 = C2;
  p.M = M; p.N = N; p.K = K; p.lda = lda; p.ldb = ldb; p.ldc = ldc; p.ldmask = ldmask; p.mode = mode; p.relu = relu;
  if (engine == 0) {
    gemm_simt_kernel<<<dim3((N + GS_T - 1) / GS_T, (M + GS_T - 1) / GS_T, 1), GS_THREADS, 0, (cudaStream_t)stream>>>(grp);
  } else if (engine == 2) {
    if (!gemm_is_thin(p)) return fail(B200SAC_ERR_INVALID, "thin engine needs a backward problem with N <= %d", GT_NMAX);
    const int per = mode == GEMM_WGRAD ? GT_ROWS_WGRAD : GT_ROWS_DGRAD;
    gemm_thin_kernel<<<dim3(1, (M + per - 1) / per, 1), GT_THREADS, 0, (cudaStream_t)stream>>>(grp);
  } else {
    return fail(B200SAC_ERR_INVALID, "unknown GEMM engine %d", engine);
  }
  cudaError_t e = cudaGetLastError();
  if (e == cudaSuccess) e = cudaStreamSynchronize((cudaStream_t)stream);
  if (e != cudaSuccess) return fail(B200SAC_ERR_CUDA, "GEMM engine %d failed: %s", engine, cudaGetErrorString(e));
  return 0;
}

extern "C" int b200sac_tc_gemm_test(int32_t mode, int32_t M, int32_t N, int32_t K, const float* A, int32_t lda,
                                    const float* B, int32_t ldb, const float* bias, const float* mask, int32_t ldmask,
                                    float* C, int32_t ldc, float* C2, int32_t relu, void* stream) {
  return tc_gemm_test_impl(mode, M, N, K, A, lda, B, ldb, bias, mask, ldmask, C, ldc, C2, relu, stream);
}

static int tc_gemm_test_impl(int32_t mode, int32_t M, int32_t N, int32_t K, const float* A, int32_t lda,
                                    const float* B, int32_t ldb, const float* bias, const float* mask, int32_t ldmask,
                                    float* C, int32_t ldc, float* C2, int32_t relu, void* stream) {
  if (!A || !B || !C) return fail(B200SAC_ERR_INVALID, "null argument");
  GemmProb p;
  memset(&p, 0, sizeof(p));
  p.A = A; p.B = B; p.bias = bias; p.mask = mask; p.C = C; p.C2 = C2;
  p.M = M; p.N = N; p.K = K; p.lda = lda; p.ldb = ldb; p.ldc = ldc; p.ldmask = ldmask; p.mode = mode; p.relu = relu;
  if (!tc_eligible(p)) return fail(B200SAC_ERR_INVALID, "problem not eligible for the tcgen05 path (need 16-B aligned operands, lda/ldb %% 4 == 0, M,N,K >= 32)");
  int bn = 64;
  if (const char* e = getenv("B200SAC_TC_BN")) { const int b = atoi(e); bn = b == 128 ? 128 : (b == 160 ? 160 : 64); }
  TcProb t;
  if (int rc = make_tc_prob(p, 0, t, bn)) return rc;
  TcProb* d = nullptr;
  CU(cudaMalloc(&d, sizeof(TcProb)));
  CU(cudaMemcpy(d, &t, sizeof(TcProb), cudaMemcpyHostToDevice));
  CU(tc_set_attrs());
  dim3 grid((N + bn - 1) / bn, (M + TC_BM - 1) / TC_BM, 1);
  tc_kernel(bn)<<<grid, TC_THREADS, tc_smem(bn), (cudaStream_t)stream>>>(d);
  cudaError_t e = cudaGetLastError();
  if (e == cudaSuccess) e = cudaStreamSynchronize((cudaStream_t)stream);
  cudaFree(d);
  if (e != cudaSuccess) return fail(B200SAC_ERR_CUDA, "gemm_tc_kernel failed: %s", cudaGetErrorString(e));
  return 0;
}

// clock64() timeline of CTA (0,0) of one warm tcgen05 GEMM launch (see TC_STAMP indices in gemm_tc.cuh).
extern "C" int b200sac_tc_gemm_timeline(int32_t mode, int32_t M, int32_t N, int32_t K, long long* out96) {
  float *A = nullptr, *B = nullptr, *C = nullptr;
  long long* dbg = nullptr;
  const size_t na = (size_t)(mode == GEMM_WGRAD ? K * M : M * K), nb = (size_t)(mode == GEMM_FWD ? N * K : K * N);
  CU(cudaMalloc(&A, na * 4)); CU(cudaMalloc(&B, nb * 4)); CU(cudaMalloc(&C, (size_t)M * N * 4)); CU(cudaMalloc(&dbg, 96 * 8));
  CU(cudaMemset(A, 0, na * 4)); CU(cudaMemset(B, 0, nb * 4)); CU(cudaMemset(dbg, 0, 96 * 8));
  GemmProb p;
  memset(&p, 0, sizeof(p));
  p.A = A; p.B = B; p.C = C; p.M = M; p.N = N; p.K = K; p.mode = mode;
  p.lda = mode == GEMM_WGRAD ? M : K; p.ldb = mode == GEMM_FWD ? K : N; p.ldc = N;
  int bn = 64;
  if (const char* e = getenv("B200SAC_TC_BN")) { const int b = atoi(e); bn = b == 128 ? 128 : (b == 160 ? 160 : 64); }
  TcProb t;
  if (int rc = make_tc_prob(p, 0, t, bn)) return rc;
  t.dbg = dbg;
  TcProb* d = nullptr;
  CU(cudaMalloc(&d, sizeof(TcProb)));
  CU(cudaMemcpy(d, &t, sizeof(TcProb), cudaMemcpyHostToDevice));
  CU(tc_set_attrs());
  dim3 grid((N + bn - 1) / bn, (M + TC_BM - 1) / TC_BM, 1);
  for (int it = 0; it < 3; ++it) tc_kernel(bn)<<<grid, TC_THREADS, tc_smem(bn)>>>(d);
  CU(cudaDeviceSynchronize());
  CU(cudaMemcpy(out96, dbg, 96 * 8, cudaMemcpyDeviceToHost));
  cudaFree(A); cudaFree(B); cudaFree(C); cudaFree(dbg); cudaFree(d);
  return 0;
}

// In-graph timeline: run `iters` sampled steps (graph launches) with kernel-start stamping enabled and
// return the mean start-to-start time (us) of each launch of the step: out_us[0] = sampling kernel, ...,
// out_us[n-1] = last kernel (measured to the next step's first kernel).
extern "C" int b200sac_graph_timeline(b200sac_t* h, b200sac_replay_t* rb, int32_t iters, float* out_us, int32_t cap,
                                      int32_t* n_out, void* stream) {
  if (!h || !rb || rb->h != h || rb->where != 0 || !out_us || !n_out) return fail(B200SAC_ERR_INVALID, "graph_timeline needs a device ring");
  CU(cudaSetDevice(h->device));
  const int n = (int)h->plan.size() + 2;       // sample + ingest + plan
  *n_out = n;
  if (cap < n) return fail(B200SAC_ERR_INVALID, "need room for %d launches", n);
  const int total = n * (iters + 1);
  unsigned long long* dt = nullptr;
  int* di = nullptr;
  CU(cudaMalloc(&dt, sizeof(unsigned long long) * total));
  CU(cudaMalloc(&di, sizeof(int)));
  CU(cudaMemset(di, 0, sizeof(int)));
  StampBuf sb_on = {dt, di, total}, sb_off = {nullptr, nullptr, 0};
  if (int rc = b200sac_step_sampled(h, rb, 5, stream)) return rc;     // warm (graph instantiated)
  CU(cudaDeviceSynchronize());
  CU(cudaMemcpyToSymbol(g_stamp, &sb_on, sizeof(StampBuf)));
  h->stamping = true;
  int rc = b200sac_step_sampled(h, rb, iters + 1, stream);
  h->stamping = false;
  CU(cudaDeviceSynchronize());
  CU(cudaMemcpyToSymbol(g_stamp, &sb_off, sizeof(StampBuf)));
  if (rc) return rc;
  std::vector<unsigned long long> t((size_t)total);
  CU(cudaMemcpy(t.data(), dt, sizeof(unsigned long long) * total, cudaMemcpyDeviceToHost));
  cudaFree(dt); cudaFree(di);
  for (int i = 0; i < n; ++i) {
    double acc = 0;
    for (int it = 0; it < iters; ++it) acc += (double)(t[(size_t)it * n + i + 1] - t[(size_t)it * n + i]);
    out_us[i] = (float)(acc / iters * 1e-3);
  }
  return 0;
}

// Learner.update() in one call: sample + one gradient step + the losses of that step (LL/learner.py:246-264).
extern "C" int b200sac_update(b200sac_t* h, b200sac_replay_t* rb, float* losses_host, void* stream) {
  if (!h || !rb || !losses_host) return fail(B200SAC_ERR_INVALID, "null argument");
  if (int rc = b200sac_step_sampled(h, rb, 1, stream)) return rc;
  CU(cudaSetDevice(h->device));
  return fetch_losses(h, (cudaStream_t)stream, 1, losses_host);
}

extern "C" int b200sac_read_losses(b200sac_t* h, int32_t n_last, float* out_host, void* stream) {
  if (!h || !out_host) return fail(B200SAC_ERR_INVALID, "null argument");
  CU(cudaSetDevice(h->device));
  return fetch_losses(h, (cudaStream_t)stream, n_last, out_host);
}

// ------------------------------------------------------------------------------------------
// Batched policy inference (SURVEY 8(f) rank 4): the actor forward + tanh-Gaussian head the step uses, on n <= 2B
// caller-provided observation rows -- Actor.get_action (LunarLander_Distributed_SAC/src/model.py:67-82; MT: mtobs rows,
// MT10_Distributed_MTSAC/src/model.py:58-73) for many environments at once.  stochastic = 0 gives k*tanh(mu).
// Uses the actor's own work buffers, so it is ordered with the steps on `stream` like any other call of the handle.
// ------------------------------------------------------------------------------------------
// LunarLander's deterministic action: k * mu, no tanh (LunarLander_Distributed_SAC/src/model.py:78-80)
__global__ void act_scaled_mu_kernel(const float* __restrict__ pout, int A, int n, float k, float* __restrict__ act) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= n * A) return;
  act[e] = k * pout[(long long)(e / A) * 2 * A + (e % A)];
}

// task id of n observation rows: argmax of the trailing one-hot (context_encoder.py:101-106), first maximum like torch.argmax
__global__ void act_task_ids_kernel(const float* __restrict__ X, int obs, int T, int n, int* __restrict__ tid) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float* row = X + (long long)i * obs + (obs - T);
  int t = 0;
  float best = row[0];
  for (int q = 1; q < T; ++q)
    if (row[q] > best) { best = row[q]; t = q; }
  tid[i] = t;
}

// CARE actors (MT10_Distributed_CARE/src/player.py:199-209: z = context_encoder(mtobs); actor.get_action(mtobs, z)):
// encode the n observation rows sitting in XS[0..n) of `replica` with the critic's state encoder -- the actor's is its
// hard copy (learner.py:402) -- into XA[0..n): per-task tables, K mixture encoders, attention mix.
static int care_encode_rows(b200sac* h, cudaStream_t st, int replica, int n) {
  const b200sac_cfg& c = h->cfg;
  const Layout& L = h->L;
  const int B = c.batch, Kenc = c.num_encoders, nmix = (int)L.mix.size();
  auto pitch = [](int w) { return (w + 3) & ~3; };
  float* par = h->params + (long long)replica * L.arena;
  float* XS = h->XS.p + (long long)replica * h->XS.rs;
  int* tid = (int*)(h->tid.p + (long long)replica * h->tid.rs);
  act_task_ids_kernel<<<(n + 255) / 256, 256, 0, st>>>(XS, h->K.obs, c.num_tasks, n, tid);
  {
    CareTabArgs P;
    memset(&P, 0, sizeof(P));
    P.params = par; P.rsP = 0; P.emb_off = L.off_emb;
    P.trunk = h->care_trunk; P.ctx = h->care_ctx;
    P.T = c.num_tasks; P.K = Kenc; P.row_w = h->care_row_w; P.off_att = h->care_off_att;
    P.original = c.care == 2 ? 1 : 0;
    P.inst_delta[0] = 0;
    P.tab[0] = h->careTab[0].p + (long long)replica * h->careTab[0].rs; P.rsTab = 0;
    care_tables_kernel<<<dim3(c.num_tasks, 1, 1), 512, 0, st>>>(P);
  }
  for (int l = 0; l < nmix; ++l) {
    const LayerOff& lo = L.mix[l];
    const bool last = (l == nmix - 1);
    const Buf& ob = last ? h->mixZ[0] : h->mixH[0][l];
    GemmGroup grp;
    memset(&grp, 0, sizeof(grp));
    for (int k0 = 0; k0 < Kenc; k0 += GS_MAXG) {
      const int cnt = (Kenc - k0 < GS_MAXG) ? Kenc - k0 : GS_MAXG;
      grp.G = cnt;
      for (int q = 0; q < cnt; ++q) {
        const int k = k0 + q;
        GemmProb& p = grp.p[q];
        memset(&p, 0, sizeof(p));
        if (l == 0) { p.A = XS; p.lda = h->K.obs; }
        else { p.A = h->mixH[0][l - 1].p + (long long)replica * h->mixH[0][l - 1].rs + (long long)k * 2 * B * pitch(lo.in); p.lda = pitch(lo.in); }
        p.B = par + lo.w + (long long)k * lo.out * lo.in; p.ldb = lo.in;
        p.bias = par + lo.b + (long long)k * lo.out;
        p.C = ob.p + (long long)replica * ob.rs + (long long)k * 2 * B * pitch(lo.out); p.ldc = pitch(lo.out);
        p.M = n; p.N = lo.out; p.K = lo.in; p.mode = GEMM_FWD; p.relu = last ? 0 : 1;
      }
      gemm_simt_kernel<<<dim3((lo.out + GS_T - 1) / GS_T, (n + GS_T - 1) / GS_T, cnt), GS_THREADS, 0, st>>>(grp);
    }
  }
  {
    CareMixArgs P;
    memset(&P, 0, sizeof(P));
    P.Z = h->mixZ[0].p + (long long)replica * h->mixZ[0].rs; P.rsZ = 0; P.kstride = (long long)2 * B * pitch(c.mix_out); P.ldz = pitch(c.mix_out);
    P.tab = h->careTab[0].p + (long long)replica * h->careTab[0].rs; P.rsTab = 0; P.row_w = h->care_row_w; P.off_att = h->care_off_att;
    P.off_ctx = h->care_off_ctx;
    P.tid = tid; P.rsR = 0;
    P.rows = n; P.B = B; P.K = Kenc; P.mo = c.mix_out; P.co = c.ctx_out;
    P.dst1 = h->XA.p + (long long)replica * h->XA.rs; P.rsD1 = 0; P.ld1 = h->K.ldxa;
    care_mix_kernel<<<dim3((n + 7) / 8, 1), 256, 0, st>>>(P);
  }
  CU(cudaGetLastError());
  return 0;
}

extern "C" int b200sac_act(b200sac_t* h, int32_t replica, int32_t n, const float* obs, const float* eps, int32_t stochastic,
                           float* actions_out, void* stream) {
  if (!h || !obs || !actions_out) return fail(B200SAC_ERR_INVALID, "null argument");
  if (replica < 0 || replica >= h->R) return fail(B200SAC_ERR_INVALID, "replica %d out of range", replica);
  const b200sac_cfg& c = h->cfg;
  const int B = c.batch, A = c.act_dim, La = c.n_actor_hidden;
  const int nmax = c.care ? B : 2 * B;           // CARE: one task id per row lives in the [batch] task-id buffer
  if (n < 1 || n > nmax) return fail(B200SAC_ERR_INVALID, "n must be in [1, %d] (2*batch; batch for CARE handles), got %d", nmax, n);
  CU(cudaSetDevice(h->device));
  StreamBridge sb(h, stream);
  if (int rc = sb.begin()) return rc;
  cudaStream_t st = sb.run;
  const Layout& L = h->L;
  const int obs_w = h->K.obs;
  float* XA = h->XA.p + (long long)replica * h->XA.rs;
  if (c.care) {
    CU(cudaMemcpyAsync(h->XS.p + (long long)replica * h->XS.rs, obs, (size_t)n * obs_w * sizeof(float), cudaMemcpyDefault, st));
    if (int rc = care_encode_rows(h, st, replica, n)) return rc;
  } else {
    CU(cudaMemcpy2DAsync(XA, (size_t)h->K.ldxa * sizeof(float), obs, (size_t)obs_w * sizeof(float), (size_t)obs_w * sizeof(float),
                         (size_t)n, cudaMemcpyDefault, st));
  }
  for (int l = 0; l < La; ++l) {
    const LayerOff& lo = L.actor[l];
    GemmGroup grp;
    memset(&grp, 0, sizeof(grp));
    grp.G = 1;
    GemmProb& p = grp.p[0];
    p.A = (l == 0 ? XA : h->hA[l - 1].p + (long long)replica * h->hA[l - 1].rs); p.lda = lo.ld;
    p.B = h->params + (long long)replica * L.arena + lo.w; p.ldb = lo.ld;
    p.bias = h->params + (long long)replica * L.arena + lo.b;
    p.C = h->hA[l].p + (long long)replica * h->hA[l].rs; p.ldc = lo.out;
    p.M = n; p.N = lo.out; p.K = lo.in; p.mode = GEMM_FWD; p.relu = 1;
    gemm_simt_kernel<<<dim3((p.N + GS_T - 1) / GS_T, (p.M + GS_T - 1) / GS_T, 1), GS_THREADS, 0, st>>>(grp);
  }
  PolicyHeadArgs P = h->pol;
  P.h += replica * P.rsH; P.W += replica * P.rsP; P.b += replica * P.rsP; P.eps += replica * P.rsEps;
  P.pout += replica * P.rsPout; P.psave += replica * P.rsSave; P.XT += replica * P.rsX; P.XP += replica * P.rsX;
  P.act_out += replica * P.rsAct; P.logp += replica * P.rsLogp; P.logstd_sum += replica * P.rsLogp; P.cnt += replica;
  P.rows = n;
  float* epsb = h->eps.p + (long long)replica * h->eps.rs;
  if (eps != nullptr) {
    CU(cudaMemcpyAsync(epsb, eps, (size_t)n * A * sizeof(float), cudaMemcpyDefault, st));
    P.use_eps_buf = 1;
  } else if (stochastic <= 0) {
    CU(cudaMemsetAsync(epsb, 0, (size_t)n * A * sizeof(float), st));       // u = mu: Actor.get_action(stochastic=False)
    P.use_eps_buf = 1;
  } else {
    P.use_eps_buf = 0;
  }
  StepConst K = h->K;
  K.seed ^= 0x5851F42D4C957F2Dull * (unsigned long long)(++h->act_calls);    // fresh noise per call, not per training step
  policy_head_kernel<<<dim3((n + 7) / 8, 1), 256, 0, st>>>(K, P);
  if (stochastic < 0 && eps == nullptr)          // k * mu instead of k * tanh(mu)
    act_scaled_mu_kernel<<<(n * A + 255) / 256, 256, 0, st>>>(P.pout, A, n, (float)c.action_scale, P.act_out);
  CU(cudaGetLastError());
  CU(cudaMemcpyAsync(actions_out, h->act_out.p + (long long)replica * h->act_out.rs, (size_t)n * A * sizeof(float), cudaMemcpyDefault, st));
  if (int rc = sb.end()) return rc;
  CU(cudaStreamSynchronize((cudaStream_t)stream));
  return 0;
}

extern "C" int b200sac_soft_update(b200sac_t* h, double tau, void* stream) {
  if (!h) return fail(B200SAC_ERR_INVALID, "null handle");
  CU(cudaSetDevice(h->device));
  // CARE: Learner.soft_update is called per module with its own tau; this entry point applies `tau` to the Q
  // functions and, unless tau == 1 (hard copy of everything), state_encoder_tau to the state encoder.
  const bool hard = (tau == 1.0);
  polyak_kernel<<<dim3(128, h->R), 256, 0, (cudaStream_t)stream>>>(
      h->params + h->L.critic_begin, h->L.arena, h->L.critic_n, h->L.target_delta, (float)tau, (float)(1.0 - tau),
      (h->cfg.care && !hard) ? (long long)(h->L.cse_begin - h->L.critic_begin) : -1LL, (float)h->cfg.tau_se,
      (float)(1.0 - h->cfg.tau_se));
  CU(cudaGetLastError());
  return 0;
}

extern "C" int b200sac_debug_read(b200sac_t* h, const char* name, int32_t replica, float* out_host, int64_t cap_floats,
                                  int64_t* n_floats, void* stream) {
  if (!h || !name || !out_host) return fail(B200SAC_ERR_INVALID, "null argument");
  if (replica < 0 || replica >= h->R) return fail(B200SAC_ERR_INVALID, "replica out of range");
  CU(cudaSetDevice(h->device));
  const int B = h->cfg.batch, A = h->cfg.act_dim;
  const float* src = nullptr;
  int64_t n = 0;
  std::string nm(name);
  if (nm == "y") { src = h->y.p + replica * h->y.rs; n = B; }
  else if (nm == "q1") { src = h->q.p + replica * h->q.rs; n = B; }
  else if (nm == "q2") { src = h->q.p + replica * h->q.rs + B; n = B; }
  else if (nm == "a_next") { src = h->act_out.p + replica * h->act_out.rs; n = (int64_t)B * A; }
  else if (nm == "a_cur") { src = h->act_out.p + replica * h->act_out.rs + (int64_t)B * A; n = (int64_t)B * A; }
  else if (nm == "logp_next") { src = h->logp.p + replica * h->logp.rs; n = B; }
  else if (nm == "logp_cur") { src = h->logp.p + replica * h->logp.rs + B; n = B; }
  else if (nm == "r") { src = h->r.p + replica * h->r.rs; n = B; }
  else if (nm == "d") { src = h->d.p + replica * h->d.rs; n = B; }
  else if (nm == "qmin") { src = h->qmin.p + replica * h->qmin.rs; n = B; }
  else if (nm == "q_pi") { src = h->qp.p + replica * 2 * h->y.rs; n = 2 * B; }        // [2][B]: Q1, Q2 at (s, a~) (actor pass)
  else if (nm == "dq_pi") { src = h->dqa.p + replica * 2 * h->y.rs; n = 2 * B; }      // [2][B]: d(actor loss)/dQk -- the min routing
  else if (nm == "d_action") { src = h->dact_dbg.p + replica * h->dact_dbg.rs; n = (int64_t)B * A; }
  else if (nm == "d_head") { src = h->dout_dbg.p + replica * h->dout_dbg.rs; n = (int64_t)B * 2 * A; }
  else if (nm == "psave") { src = h->psave.p + replica * h->psave.rs; n = (int64_t)2 * B * A * kSaveW; }   // [2B][A][8]: std, diff, tanh, act, jac, EPS, mask, logp_j
  else if (nm == "chain_dbg") {
    if (!h->chain_dbg) return fail(B200SAC_ERR_INVALID, "chain_dbg needs B200SAC_CHAIN_DBG=1 at create time");
    src = reinterpret_cast<const float*>(h->chain_dbg); n = 2 * CH_DBG_SLOTS * 16;     // int64 stamps viewed as float pairs
  }
  else {
    // hidden activations (the ReLU masks of the step): "hA.<l>" [2B][H] rows [s';s]; "hQ.<l>" / "hT.<l>" / "hP.<l>" [2][B][H]
    // (critic update pass / target pass -- not kept by the layer-chained plan -- / actor pass); CARE mixture encoders
    // "mixH.<inst>.<l>" [K][rows][pitch4(H)], inst 0 = critic's on [s';s] (rows 2B), 1 = target's on s', 2 = updated critic's on s
    int l = -1, inst = -1;
    char kind[8] = "";
    const Buf* b = nullptr;
    if (sscanf(name, "mixH.%d.%d", &inst, &l) == 2) {
      if (!h->cfg.care || inst < 0 || inst > 2 || l < 0 || l >= (int)h->mixH[inst].size()) return fail(B200SAC_ERR_INVALID, "no such tensor '%s'", name);
      b = &h->mixH[inst][l];
      const int rows = inst == 0 ? 2 * B : B, pw = (h->cfg.mix_hidden[l] + 3) & ~3;
      n = (int64_t)h->cfg.num_encoders * rows * pw;
    } else if (sscanf(name, "h%1[AQTP].%d", kind, &l) == 2) {
      const std::vector<Buf>& v = kind[0] == 'A' ? h->hA : (kind[0] == 'Q' ? h->hQ : (kind[0] == 'T' ? h->hT : h->hP));
      if (l < 0 || l >= (int)v.size()) return fail(B200SAC_ERR_INVALID, "no such tensor '%s'", name);
      b = &v[l];
      n = (int64_t)2 * B * (kind[0] == 'A' ? h->cfg.actor_hidden[l] : h->cfg.critic_hidden[l]);
    } else {
      return fail(B200SAC_ERR_INVALID, "unknown debug tensor '%s'", name);
    }
    src = b->p + replica * b->rs;
  }
  if (n_floats) *n_floats = n;
  if (cap_floats < n) return fail(B200SAC_ERR_INVALID, "buffer too small: need %lld floats", (long long)n);
  CU(cudaMemcpyAsync(out_host, src, n * sizeof(float), cudaMemcpyDeviceToHost, (cudaStream_t)stream));
  CU(cudaStreamSynchronize((cudaStream_t)stream));
  return 0;
}

// ------------------------------------------------------------------------------------------
// replay ring
// ------------------------------------------------------------------------------------------
extern "C" int b200sac_replay_create(b200sac_t* h, int64_t capacity, int32_t where, uint64_t seed, b200sac_replay_t** out) {
  if (!h || !out) return fail(B200SAC_ERR_INVALID, "null argument");
  *out = nullptr;
  if (where != 0 && where != 1) return fail(B200SAC_ERR_INVALID, "where must be 0 (device) or 1 (pinned host)");
  const int Teff = h->cfg.num_tasks > 0 ? h->cfg.num_tasks : 1;
  if (capacity / Teff < 4LL * (h->cfg.batch / Teff))
    return fail(B200SAC_ERR_INVALID, "capacity %lld too small for batch %d", (long long)capacity, h->cfg.batch);
  if ((long long)capacity > 0x7fffffffLL) return fail(B200SAC_ERR_INVALID, "capacity must fit in int32");
  CU(cudaSetDevice(h->device));
  b200sac_replay* rb = new (std::nothrow) b200sac_replay();
  if (!rb) return fail(B200SAC_ERR_NOMEM, "out of host memory");
  rb->h = h; rb->where = where; rb->Teff = Teff;
  rb->cap_per_task = capacity / Teff;
  rb->cap = rb->cap_per_task * Teff;
  rb->rs_rows = rb->cap * h->row_stride;
  rb->seed = seed;
  rb->rng.seed(seed);
  rb->fill.assign((size_t)h->R * Teff, 0);
  rb->head.assign((size_t)h->R * Teff, 0);
  const size_t bytes = (size_t)h->R * rb->rs_rows * sizeof(float);
  cudaError_t e = where == 0 ? cudaMalloc(&rb->rows, bytes) : cudaMallocHost(&rb->rows, bytes);
  if (e != cudaSuccess) { delete rb; return fail(B200SAC_ERR_NOMEM, "replay allocation of %zu bytes failed: %s", bytes, cudaGetErrorString(e)); }
  if (where == 0) {
    if (cudaMalloc(&rb->d_fill, sizeof(long long) * h->R * Teff) != cudaSuccess ||
        cudaMalloc(&rb->d_idx, sizeof(int) * h->R * h->cfg.batch) != cudaSuccess ||
        cudaMemset(rb->d_fill, 0, sizeof(long long) * h->R * Teff) != cudaSuccess ||
        cudaEventCreateWithFlags(&rb->ev_gather, cudaEventDisableTiming) != cudaSuccess) {
      cudaFree(rb->rows); cudaFree(rb->d_fill); cudaFree(rb->d_idx);
      delete rb;
      return fail(B200SAC_ERR_NOMEM, "replay index allocation failed");
    }
  }
  *out = rb;
  return 0;
}

extern "C" int b200sac_replay_destroy(b200sac_replay_t* rb) {
  if (!rb) return 0;
  cudaSetDevice(rb->h->device);
  // graphs that captured this ring's pointers must go
  if (rb->h->prefetch_rb == rb) { rb->h->prefetch_slot = -1; rb->h->prefetch_rb = nullptr; }
  for (auto it = rb->h->graphs.begin(); it != rb->h->graphs.end();) {
    if (it->first.p[8] == rb) { cudaGraphExecDestroy(it->second); it = rb->h->graphs.erase(it); }
    else ++it;
  }
  if (rb->where == 0) cudaFree(rb->rows); else cudaFreeHost(rb->rows);
  cudaFree(rb->d_fill); cudaFree(rb->d_idx);
  if (rb->ev_gather) cudaEventDestroy(rb->ev_gather);
  delete rb;
  return 0;
}

extern "C" int b200sac_replay_push(b200sac_replay_t* rb, int32_t replica, int64_t n, const float* s, const float* a,
                                   const float* r, const float* s2, const float* d) {
  if (!rb || !s || !a || !r || !s2 || !d) return fail(B200SAC_ERR_INVALID, "null argument");
  b200sac* h = rb->h;
  if (replica < 0 || replica >= h->R) return fail(B200SAC_ERR_INVALID, "replica out of range");
  CU(cudaSetDevice(h->device));
  const int obs = h->K.obs, A = h->K.act, T = h->cfg.num_tasks, rs = h->row_stride;
  // pack the rows, bucketed by task, then copy each bucket as at most two contiguous runs (ring wrap)
  std::vector<std::vector<float>> bucket((size_t)rb->Teff);
  std::vector<float> row((size_t)rs, 0.f);
  for (int64_t i = 0; i < n; ++i) {
    memcpy(row.data(), s + i * obs, obs * sizeof(float));
    memcpy(row.data() + obs, a + i * A, A * sizeof(float));
    row[obs + A] = r[i];
    memcpy(row.data() + obs + A + 1, s2 + i * obs, obs * sizeof(float));
    row[2 * obs + A + 1] = d[i];
    int task = 0;
    if (T > 0) {
      float best = row[obs - T];
      for (int q = 1; q < T; ++q)
        if (row[obs - T + q] > best) { best = row[obs - T + q]; task = q; }
    }
    bucket[(size_t)task].insert(bucket[(size_t)task].end(), row.begin(), row.end());
  }
  std::lock_guard<std::mutex> lk(rb->mu);
  // Device ring: the gathers of every step enqueued so far must have read their rows before a wrapped ring overwrites
  // them (a torn transition otherwise); step_sampled enqueues under the same mutex, so none can slip in while we copy.
  if (rb->where == 0 && rb->gather_pending) { CU(cudaEventSynchronize(rb->ev_gather)); rb->gather_pending = false; }
  for (int task = 0; task < rb->Teff; ++task) {
    const float* src = bucket[(size_t)task].data();
    long long cnt = (long long)(bucket[(size_t)task].size() / (size_t)rs);
    if (cnt > rb->cap_per_task) {                  // more than a full ring: only the newest cap rows survive (deque maxlen)
      src += (size_t)(cnt - rb->cap_per_task) * rs;
      cnt = rb->cap_per_task;
    }
    long long& hd = rb->head[(size_t)replica * rb->Teff + task];
    long long& fl = rb->fill[(size_t)replica * rb->Teff + task];
    long long done = 0;
    while (done < cnt) {
      const long long run = std::min(cnt - done, rb->cap_per_task - hd);
      float* dst = rb->rows + (size_t)replica * rb->rs_rows + ((size_t)task * rb->cap_per_task + hd) * rs;
      if (rb->where == 0) CU(cudaMemcpy(dst, src + (size_t)done * rs, (size_t)run * rs * sizeof(float), cudaMemcpyHostToDevice));
      else memcpy(dst, src + (size_t)done * rs, (size_t)run * rs * sizeof(float));
      hd = (hd + run) % rb->cap_per_task;
      fl = std::min(fl + run, rb->cap_per_task);
      done += run;
    }
  }
  if (rb->where == 0)
    CU(cudaMemcpy(rb->d_fill + (size_t)replica * rb->Teff, rb->fill.data() + (size_t)replica * rb->Teff,
                  sizeof(long long) * rb->Teff, cudaMemcpyHostToDevice));
  return 0;
}

extern "C" int b200sac_replay_fill_synthetic(b200sac_replay_t* rb, int64_t n, uint64_t seed, void* stream) {
  if (!rb) return fail(B200SAC_ERR_INVALID, "null argument");
  b200sac* h = rb->h;
  CU(cudaSetDevice(h->device));
  long long per = n / rb->Teff;
  if (per > rb->cap_per_task) per = rb->cap_per_task;
  if (per < 1) return fail(B200SAC_ERR_INVALID, "n too small");
  cudaStream_t st = (cudaStream_t)stream;
  float* dev_rows = rb->rows;
  float* tmp = nullptr;
  if (rb->where == 1) {   // generate on the device, copy down into the pinned ring
    CU(cudaMalloc(&tmp, (size_t)h->R * rb->rs_rows * sizeof(float)));
    dev_rows = tmp;
  }
  CU(cudaMemsetAsync(dev_rows, 0, (size_t)h->R * rb->rs_rows * sizeof(float), st));
  fill_synthetic_kernel<<<dim3(592, h->R), 256, 0, st>>>(dev_rows, rb->rs_rows, h->row_stride, per, rb->cap_per_task,
                                                        h->cfg.state_dim, h->cfg.act_dim, h->cfg.num_tasks, seed);
  CU(cudaGetLastError());
  if (rb->where == 1) {
    CU(cudaMemcpyAsync(rb->rows, tmp, (size_t)h->R * rb->rs_rows * sizeof(float), cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    CU(cudaFree(tmp));
  }
  std::lock_guard<std::mutex> lk(rb->mu);
  for (auto& f : rb->fill) f = per;
  for (auto& hd : rb->head) hd = per % rb->cap_per_task;
  if (rb->where == 0)
    CU(cudaMemcpyAsync(rb->d_fill, rb->fill.data(), sizeof(long long) * rb->fill.size(), cudaMemcpyHostToDevice, st));
  CU(cudaStreamSynchronize(st));
  return 0;
}

extern "C" int b200sac_replay_size(b200sac_replay_t* rb, int32_t replica, int64_t* n) {
  if (!rb || !n || replica < 0 || replica >= rb->h->R) return fail(B200SAC_ERR_INVALID, "bad argument");
  std::lock_guard<std::mutex> lk(rb->mu);
  long long mn = rb->fill[(size_t)replica * rb->Teff];
  for (int t = 1; t < rb->Teff; ++t) mn = std::min(mn, rb->fill[(size_t)replica * rb->Teff + t]);
  *n = rb->Teff > 1 ? mn : rb->fill[(size_t)replica * rb->Teff];
  return 0;
}

// host-side index draw: uniform without replacement, per task (random.sample semantics)
static int host_draw(b200sac_replay* rb, int replica, std::vector<long long>& idx) {
  const int B = rb->h->cfg.batch, per = B / rb->Teff;
  idx.clear();
  for (int t = 0; t < rb->Teff; ++t) {
    const long long n = rb->fill[(size_t)replica * rb->Teff + t];
    if (n < per) return fail(B200SAC_ERR_STATE, "replay holds %lld transitions for task %d, need %d", n, t, per);
    std::unordered_set<long long> seen;
    while ((int)seen.size() < per) {
      const long long v = (long long)(rb->rng() % (unsigned long long)n);
      if (seen.insert(v).second) idx.push_back((long long)t * rb->cap_per_task + v);
    }
  }
  if (rb->Teff > 1) std::shuffle(idx.begin(), idx.end(), rb->rng);   // MS/replay_buffers.py:83-84
  return 0;
}

extern "C" int b200sac_replay_sample(b200sac_replay_t* rb, int32_t replica, float* s, float* a, float* r, float* s2,
                                     float* d, int64_t* idx_out) {
  if (!rb || !s || !a || !r || !s2 || !d) return fail(B200SAC_ERR_INVALID, "null argument");
  b200sac* h = rb->h;
  if (replica < 0 || replica >= h->R) return fail(B200SAC_ERR_INVALID, "replica out of range");
  CU(cudaSetDevice(h->device));
  const int B = h->cfg.batch, obs = h->K.obs, A = h->K.act, rs = h->row_stride;
  std::vector<long long> idx;
  std::vector<float> row((size_t)rs);
  std::lock_guard<std::mutex> lk(rb->mu);
  if (int rc = host_draw(rb, replica, idx)) return rc;
  for (int i = 0; i < B; ++i) {
    const float* src = rb->rows + (size_t)replica * rb->rs_rows + (size_t)idx[i] * rs;
    if (rb->where == 0) { CU(cudaMemcpy(row.data(), src, rs * sizeof(float), cudaMemcpyDeviceToHost)); src = row.data(); }
    memcpy(s + (size_t)i * obs, src, obs * sizeof(float));
    memcpy(a + (size_t)i * A, src + obs, A * sizeof(float));
    r[i] = src[obs + A];
    memcpy(s2 + (size_t)i * obs, src + obs + A + 1, obs * sizeof(float));
    d[i] = src[2 * obs + A + 1];
    if (idx_out) idx_out[i] = idx[i];
  }
  return 0;
}

extern "C" int b200sac_step_sampled(b200sac_t* h, b200sac_replay_t* rb, int32_t n_steps, void* stream) {
  if (!h || !rb || rb->h != h) return fail(B200SAC_ERR_INVALID, "bad handle");
  if (n_steps < 1) return fail(B200SAC_ERR_INVALID, "n_steps < 1");
  CU(cudaSetDevice(h->device));
  StreamBridge sb(h, stream);
  if (int rc = sb.begin()) return rc;
  cudaStream_t st = sb.run;
  const int B = h->cfg.batch, per = B / rb->Teff;
  {
    std::lock_guard<std::mutex> lk(rb->mu);
    for (auto f : rb->fill)
      if (f < 4LL * per)
        return fail(B200SAC_ERR_STATE, "replay not ready: a ring holds %lld transitions, need >= %d (4 x per-task batch)", f, 4 * per);
  }
  if (rb->where == 0) {
    std::lock_guard<std::mutex> lk(rb->mu);           // ordered against b200sac_replay_push (see there)
    const void* p[1] = {rb->rows};
    int i = 0;
    if (!h->stamping)                           // (the in-graph timeline wants one step per graph)
      for (int n = kGraphSteps; n > 1; n >>= 1)
        for (; i + n <= n_steps; i += n)
          if (int rc = launch_step(h, st, 2, p, 1, rb, n)) return rc;
    for (; i < n_steps; ++i)
      if (int rc = launch_step(h, st, 2, p, 1, rb)) return rc;
    CU(cudaEventRecord(rb->ev_gather, st));
    rb->gather_pending = true;
    return sb.end();
  }
  // pinned-host ring: draw + gather on the host into the pinned slot, H2D on the side stream.  The NEXT
  // minibatch is prepared right after the current step has been launched, so host sampling, the gather and
  // the copy overlap the GPU step (the reference samples at the start of update(); here the draw for step k+1
  // happens while step k runs -- the same RNG sequence, the ring contents as of that moment).
  std::vector<long long> idx;
  const int rs = h->row_stride;
  const size_t rows_bytes = (size_t)h->R * B * rs * sizeof(float);
  auto prepare = [&](int* slot_out) -> int {
    int slot;
    if (int rc = acquire_slot(h, &slot)) return rc;
    {
      std::lock_guard<std::mutex> lk(rb->mu);
      for (int rep = 0; rep < h->R; ++rep) {
        if (int rc = host_draw(rb, rep, idx)) return rc;
        float* dst = h->stage_h[slot] + (size_t)rep * B * rs;
        const float* base = rb->rows + (size_t)rep * rb->rs_rows;
        for (int j = 0; j < B; ++j) memcpy(dst + (size_t)j * rs, base + (size_t)idx[j] * rs, rs * sizeof(float));
      }
    }
    CU(cudaMemcpyAsync(h->stage_d[slot], h->stage_h[slot], rows_bytes, cudaMemcpyHostToDevice, h->side));
    CU(cudaEventRecord(h->ev_copied[slot], h->side));
    *slot_out = slot;
    return 0;
  };
  if (h->prefetch_slot >= 0 && h->prefetch_rb != rb) h->prefetch_slot = -1;     // belongs to another ring: drop it
  for (int i = 0; i < n_steps; ++i) {
    int slot = h->prefetch_slot;
    if (slot < 0)
      if (int rc = prepare(&slot)) return rc;
    h->prefetch_slot = -1;
    CU(cudaStreamWaitEvent(st, h->ev_copied[slot], 0));
    const void* p[2] = {h->stage_d[slot], nullptr};
    if (int rc = launch_step(h, st, 1, p, 2, nullptr)) return rc;
    CU(cudaEventRecord(h->ev_consumed[slot], st));
    h->stage_used[slot] = true;
    int next;
    if (int rc = prepare(&next)) return rc;      // overlaps the step just launched
    h->prefetch_slot = next;
    h->prefetch_rb = rb;
  }
  return sb.end();
}
