// tcs_api.cu — the C ABI (include/tcs.h): handle, weights, workspace, the score network pass,
// the three samplers (Heun ODE, Euler-Maruyama SDE, DPM-Solver++(2M)) and their CUDA-graph replay.  No PyTorch types, no CPU fallback.
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <memory>
#include <string>
#include <vector>

#include "attn_tc.cuh"
#include "conv_tc.cuh"
#include "kernels.cuh"

namespace tcs {

static thread_local std::string g_err;
void set_error(const std::string& m) { g_err = m; }
int fail(int code, const std::string& m) {
  g_err = m;
  return code;
}

// ------------------------------------------------------------------------------------------
// host-side schedule in the reference's fp32 arithmetic (VPSDE :287-298, time grid :482-483)
// ------------------------------------------------------------------------------------------
static void time_grid_host(int steps, double t_end, float* ts) {
  // torch.linspace(0, 1, steps+1) (fp32): start + step*i for the first half, end - step*(n-1-i) after
  const int n = steps + 1;
  const float step = n > 1 ? (1.0f - 0.0f) / static_cast<float>(n - 1) : 0.f;
  const int halfway = n / 2;
  const float te = static_cast<float>(t_end);
  const float ome = static_cast<float>(1.0 - t_end);
  for (int i = 0; i < n; ++i) {
    const float u = i < halfway ? 0.0f + step * static_cast<float>(i) : 1.0f - step * static_cast<float>(n - i - 1);
    const float om = 1.0f - u;
    const float sq = om * om;
    ts[i] = te + ome * sq;
  }
}
struct Sched {
  double bmin, bmax;
  float beta(float t) const { return static_cast<float>(bmin) + t * static_cast<float>(bmax - bmin); }
  float int_beta(float t) const {
    return static_cast<float>(bmin) * t + static_cast<float>(0.5 * (bmax - bmin)) * (t * t);
  }
  float alpha(float t) const { return expf(-0.5f * int_beta(t)); }
  float sigma(float t) const {
    const float a = alpha(t);
    const float v = 1.0f - a * a;
    return sqrtf(v < 1e-8f ? 1e-8f : v);
  }
};

// DPM-Solver++(2M) schedule: times uniform in log-SNR lambda = log alpha - log sigma from t = 1 to t_end (endpoints pinned),
// stored as fp32 like time_grid_host; the coefficients of step i are computed in double from those fp32 times and rounded
// to fp32 once.  Step 0 is first order, and so is the last step when steps < 15 (the "lower order final" rule).
static void dpm_schedule_host(int steps, double t_end, double bmin, double bmax, float* ts, DpmCoef* k) {
  const double d = bmax - bmin;
  auto alpha = [&](double t) { return exp(-0.5 * (bmin * t + 0.5 * d * (t * t))); };
  auto sigma = [&](double t) { const double a = alpha(t); return sqrt(fmax(1.0 - a * a, 1e-8)); };
  auto lambda = [&](double t) { return log(alpha(t)) - log(sigma(t)); };
  const double l_start = lambda(1.0), l_end = lambda(t_end);
  ts[0] = 1.0f;
  for (int i = 1; i < steps; ++i) {
    const double l = l_start + (static_cast<double>(i) / steps) * (l_end - l_start);
    const double ib = log1p(exp(-2.0 * l));   // int_0^t beta = -2 log alpha, and alpha^2 = 1 / (1 + exp(-2 lambda))
    ts[i] = static_cast<float>(d > 0.0 ? (-bmin + sqrt(bmin * bmin + 2.0 * d * ib)) / d : ib / bmin);
  }
  if (steps >= 1) ts[steps] = static_cast<float>(t_end);
  double h_prev = 0.0;
  for (int i = 0; i < steps; ++i) {
    const double t0 = ts[i], t1 = ts[i + 1];
    const double h = lambda(t1) - lambda(t0);
    DpmCoef c;
    c.a = static_cast<float>(sigma(t1) / sigma(t0));
    c.m = static_cast<float>(alpha(t1) * -expm1(-h));
    if (i == 0 || (i == steps - 1 && steps < 15)) {
      c.c0 = 1.0f; c.c1 = 0.0f;
    } else {
      const double r = h_prev / h;
      c.c0 = static_cast<float>(1.0 + 1.0 / (2.0 * r));
      c.c1 = static_cast<float>(-1.0 / (2.0 * r));
    }
    k[i] = c;
    h_prev = h;
  }
}


enum ConvId { C_D1B, C_DS1, C_D2A, C_D2B, C_DS2, C_MA, C_MB, C_QKV, C_PROJ, C_US2, C_U2A, C_U2B, C_US1, C_U1A, C_U1B, C_COUNT };
struct ConvSpec { const char* key; int cin0, cin1, cout, k, stride, res; };
static const ConvSpec kConv[C_COUNT] = {
    {"down1.net.3", 96, 0, 96, 3, 1, 64},  {"ds1", 96, 0, 96, 4, 2, 32},       {"down2.net.0", 96, 0, 192, 3, 1, 32},
    {"down2.net.3", 192, 0, 192, 3, 1, 32}, {"ds2", 192, 0, 192, 4, 2, 16},     {"mid.net.0", 192, 0, 192, 3, 1, 16},
    {"mid.net.3", 192, 0, 192, 3, 1, 16},   {"attn.qkv", 192, 0, 576, 1, 1, 16}, {"attn.proj", 192, 0, 192, 1, 1, 16},
    {"us2_conv", 192, 0, 192, 3, 1, 32},    {"up2.net.0", 192, 192, 96, 3, 1, 32}, {"up2.net.3", 96, 0, 96, 3, 1, 32},
    {"us1_conv", 96, 0, 96, 3, 1, 64},      {"up1.net.0", 96, 96, 96, 3, 1, 64}, {"up1.net.3", 96, 0, 96, 3, 1, 64}};

static ConvGeom geom_of(int id, int B, int in_pad) {
  const ConvSpec& s = kConv[id];
  ConvGeom g;
  g.B = B; g.H = g.W = s.res; g.ksize = s.k; g.stride = s.stride;
  g.nsrc = s.cin1 ? 2 : 1;
  g.csrc[0] = s.cin0; g.csrc[1] = s.cin1 ? s.cin1 : s.cin0;
  g.in_pad[0] = g.in_pad[1] = in_pad;
  g.ntot = s.cout;
  return g;
}

// layer taps exported by tcs_debug_layer, in execution order
static const char* kTapNames[] = {
    "down1.net.0.raw", "down1.net.0.act", "down1.net.3.raw", "down1.net.3.act", "ds1",
    "down2.net.0.raw", "down2.net.0.act", "down2.net.3.raw", "down2.net.3.act", "ds2",
    "mid.net.0.raw", "mid.net.0.act", "mid.net.3.raw", "mid.net.3.act", "attn.qkv", "attn.y", "attn",
    "us2.up", "us2_conv", "up2.net.0.raw", "up2.net.0.act", "up2.net.3.raw", "up2.net.3.act",
    "us1.up", "us1_conv", "up1.net.0.raw", "up1.net.0.act", "up1.net.3.raw", "up1.net.3.act", "eps"};
constexpr int kNumTaps = sizeof(kTapNames) / sizeof(kTapNames[0]);

struct TapRequest {
  int id = -1;          // which tap (-1: none)
  float* out = nullptr; // device fp32 destination
  int64_t capacity = 0;
  int64_t written = 0;
};

}  // namespace tcs

using namespace tcs;

struct tcs_handle {
  tcs_config cfg;
  int sm_count = 148;
  bool bf16 = false, use_tc = false, fuse_gn = false, fuse_first = true;
  bool fuse_attn = false;   // the attention block as one tcgen05 kernel (attn_tc.cu); TCS_FUSE_ATTN=0 keeps the four launches
  DevBuf attn_wpack;
  bool fuse_ups = false;    // us1_conv / us2_conv read the half-resolution tensor, the bilinear x2 upsample is blended inside the conv (TCS_FUSE_UPS=0: stand-alone kernel)
  ConvTcPlan plan_us[2];    // [us2_conv, us1_conv] with ConvGeom::ups
  bool split3 = false;   // precision fp32 on the tcgen05 engine: conv operands as bf16 (hi, lo) pairs (kernels_split.cu)
  size_t esz = 4;
  cudaStream_t stream = nullptr;   // internal stream all work runs on
  cudaEvent_t ev_in = nullptr, ev_out = nullptr;
  int64_t launches = 0;
  cudaEvent_t prof_ev[2 * 16] = {};   // tcs_score_profiled: begin/end per conv id
  bool profiling = false;

  std::map<std::string, HostTensor> host_w;
  bool finalized = false;
  DevBuf arena;                           // fp32 weights, device
  std::map<std::string, const float*> dw;  // key -> device pointer
  EmbedWeights ew{};
  const float *d_w9 = nullptr, *d_wout = nullptr;
  float out_bias = 0.f;
  DevBuf wpack[C_COUNT];                  // packed conv weights for the active engine

  // workspace (sized for `chunk` images)
  int chunk = 0;
  DevBuf raw64, raw32, raw16, partials, gnstats;
  DevBuf p64_h1, p64_a, p64_b;
  DevBuf p32_96a, p32_96b, p32_192a, p32_192h2, p32_192b;
  DevBuf p16_a, p16_b, p16_c, qkv, atty;
  DevBuf split_s;                         // bf16x3 mode: split copy of the fp32 tensor the next conv reads
  ConvTcPlan plan[C_COUNT];
  ConvTcPlan plan_eps, plan_eps_pair;     // 96 -> 1 output conv on the tensor pipe (N padded to 16)
  DevBuf wpack_out;
  const float* d_bias16 = nullptr;
  bool tc_out = false, eps_kxn = true;

  // per-call state
  DevBuf cvec, tvec, tvals, coef, dpm_coef, x, xpred, d0, eps, step_ctr, ycat_tmp, ycont_tmp;
  DevBuf status;                          // device status word (bit 0: fp16 stash range exceeded in a fused GroupNorm layer)
  void* pinned = nullptr; size_t pinned_bytes = 0;
  cudaEvent_t ev_pinned = nullptr;

  // graph cache.  The captured kernels hold the device pointers of the per-call buffers below, so the key carries the
  // workspace generation: DevBuf::ensure bumps ws_gen whenever one of them is re-allocated (by tcs_sample with more
  // steps / samples, or by tcs_score / tcs_debug_layer in between), which forces a re-capture.
  cudaGraphExec_t gexec = nullptr;
  uint64_t ws_gen = 0;
  struct GKey { int n = -1, dup, sampler; const void *noise, *teps, *tx; float guidance; uint64_t seed, gidx, gen; } gkey;
  int64_t graph_kernels = 0;

  tcs_handle() {
    for (DevBuf* b : {&cvec, &tvec, &tvals, &coef, &dpm_coef, &x, &xpred, &d0, &eps, &step_ctr}) b->gen = &ws_gen;
  }

  ~tcs_handle() {
    if (gexec) cudaGraphExecDestroy(gexec);
    if (pinned) cudaFreeHost(pinned);
    if (ev_in) cudaEventDestroy(ev_in);
    if (ev_out) cudaEventDestroy(ev_out);
    if (ev_pinned) cudaEventDestroy(ev_pinned);
    for (cudaEvent_t e : prof_ev) if (e) cudaEventDestroy(e);
    if (stream) cudaStreamDestroy(stream);
  }
};

namespace tcs {

// expected state dict: key -> shape (SURVEY 8a-W)
static std::vector<std::pair<std::string, std::vector<int64_t>>> expected_weights(const tcs_config& c) {
  std::vector<std::pair<std::string, std::vector<int64_t>>> v;
  const int64_t e = c.emb_dim, b = c.base_ch, cin = 1 + c.cond_ch + c.time_ch;
  auto lin = [&](const std::string& k, int64_t i, int64_t o) { v.push_back({k + ".weight", {o, i}}); v.push_back({k + ".bias", {o}}); };
  auto conv = [&](const std::string& k, int64_t i, int64_t o, int64_t ks) { v.push_back({k + ".weight", {o, i, ks, ks}}); v.push_back({k + ".bias", {o}}); };
  auto gn = [&](const std::string& k, int64_t ch) { v.push_back({k + ".weight", {ch}}); v.push_back({k + ".bias", {ch}}); };
  auto block = [&](const std::string& k, int64_t i, int64_t o) { conv(k + ".net.0", i, o, 3); gn(k + ".net.1", o); conv(k + ".net.3", o, o, 3); gn(k + ".net.4", o); };
  v.push_back({"cond_emb.cat_emb.weight", {c.n_types + 1, e}});
  lin("cond_emb.cont_mlp.0", c.y_cont_dim, e); lin("cond_emb.cont_mlp.2", e, e); lin("cond_emb.out.1", 2 * e, e);
  lin("time_mlp.0", e, e); lin("time_mlp.2", e, e);
  lin("to_cond_map", e, c.cond_ch); lin("to_time_map", e, c.time_ch);
  block("down1", cin, b); conv("ds1", b, b, 4); block("down2", b, 2 * b); conv("ds2", 2 * b, 2 * b, 4);
  block("mid", 2 * b, 2 * b); gn("attn.norm", 2 * b); conv("attn.qkv", 2 * b, 6 * b, 1); conv("attn.proj", 2 * b, 2 * b, 1);
  conv("us2_conv", 2 * b, 2 * b, 3); block("up2", 4 * b, b); conv("us1_conv", b, b, 3); block("up1", 2 * b, b);
  conv("out", b, 1, 3);
  return v;
}

static int enter(tcs_handle* h, cudaStream_t user) {
  TCS_CUDA(cudaSetDevice(h->cfg.device));
  TCS_CUDA(cudaEventRecord(h->ev_in, user));
  TCS_CUDA(cudaStreamWaitEvent(h->stream, h->ev_in, 0));
  return TCS_OK;
}
static int leave(tcs_handle* h, cudaStream_t user) {
  TCS_CUDA(cudaEventRecord(h->ev_out, h->stream));
  TCS_CUDA(cudaStreamWaitEvent(user, h->ev_out, 0));
  return TCS_OK;
}

static int ensure_pinned(tcs_handle* h, size_t bytes) {
  if (h->pinned_bytes >= bytes) {
    TCS_CUDA(cudaEventSynchronize(h->ev_pinned));  // previous upload out of the staging buffer finished
    return TCS_OK;
  }
  TCS_CUDA(cudaEventSynchronize(h->ev_pinned));
  if (h->pinned) cudaFreeHost(h->pinned);
  h->pinned = nullptr; h->pinned_bytes = 0;
  TCS_CUDA(cudaMallocHost(&h->pinned, bytes));
  h->pinned_bytes = bytes;
  return TCS_OK;
}

// ------------------------------------------------------------------------------------------
// workspace + plans
// ------------------------------------------------------------------------------------------
static int alloc_workspace(tcs_handle* h) {
  const size_t MB = h->chunk, e = h->esz;
  TCS_CHECK(h->raw64.ensure(MB * 4096 * 96 * 4));
  TCS_CHECK(h->raw32.ensure(MB * 1024 * 192 * 4));
  TCS_CHECK(h->raw16.ensure(MB * 256 * 192 * 4));
  TCS_CHECK(h->partials.ensure(MB * 128 * 16 * 4));
  TCS_CHECK(h->gnstats.ensure(MB * 8 * 8));
  const size_t P64 = MB * 66 * 66 * 96 * e, P32a = MB * 34 * 34 * 96 * e, P32b = MB * 34 * 34 * 192 * e,
               P16 = MB * 18 * 18 * 192 * e;
  TCS_CHECK(h->p64_h1.ensure(P64)); TCS_CHECK(h->p64_a.ensure(P64)); TCS_CHECK(h->p64_b.ensure(P64));
  TCS_CHECK(h->p32_96a.ensure(P32a)); TCS_CHECK(h->p32_96b.ensure(P32a));
  TCS_CHECK(h->p32_192a.ensure(P32b)); TCS_CHECK(h->p32_192h2.ensure(P32b)); TCS_CHECK(h->p32_192b.ensure(P32b));
  TCS_CHECK(h->p16_a.ensure(P16)); TCS_CHECK(h->p16_b.ensure(P16)); TCS_CHECK(h->p16_c.ensure(P16));
  TCS_CHECK(h->qkv.ensure(MB * 256 * 576 * e));
  TCS_CHECK(h->atty.ensure(MB * 256 * 192 * e));
  if (h->split3) TCS_CHECK(h->split_s.ensure(P64));
  return TCS_OK;
}

// (source buffers, destination, epilogue) of every GEMM conv, shared by both engines
struct ConvWiring { const void *s0, *s1; void* out; int epi; const void* residual; int ldo; int in_pad;
                    const char* gn; void* act; };  // gn: GroupNorm that follows (or null); act: its padded output
static ConvWiring wiring(tcs_handle* h, int id) {
  ConvWiring w{};
  switch (id) {
    case C_D1B: w = {h->p64_a.p, nullptr, h->raw64.p, EPI_RAW_STATS, nullptr, 96, 1, "down1.net.4", h->p64_h1.p}; break;
    case C_DS1: w = {h->p64_h1.p, nullptr, h->p32_96a.p, EPI_PADDED, nullptr, 96, 1, nullptr, nullptr}; break;
    case C_D2A: w = {h->p32_96a.p, nullptr, h->raw32.p, EPI_RAW_STATS, nullptr, 192, 1, "down2.net.1", h->p32_192a.p}; break;
    case C_D2B: w = {h->p32_192a.p, nullptr, h->raw32.p, EPI_RAW_STATS, nullptr, 192, 1, "down2.net.4", h->p32_192h2.p}; break;
    case C_DS2: w = {h->p32_192h2.p, nullptr, h->p16_a.p, EPI_PADDED, nullptr, 192, 1, nullptr, nullptr}; break;
    case C_MA: w = {h->p16_a.p, nullptr, h->raw16.p, EPI_RAW_STATS, nullptr, 192, 1, "mid.net.1", h->p16_b.p}; break;
    case C_MB: w = {h->p16_b.p, nullptr, h->raw16.p, EPI_RAW_STATS, nullptr, 192, 1, "mid.net.4", h->p16_a.p}; break;
    case C_QKV: w = {h->p16_b.p, nullptr, h->qkv.p, EPI_PLAIN, nullptr, 576, 1, nullptr, nullptr}; break;
    case C_PROJ: w = {h->atty.p, nullptr, h->p16_c.p, EPI_PADDED, h->p16_a.p, 192, 0, nullptr, nullptr}; break;
    case C_US2: w = {h->p32_192a.p, nullptr, h->p32_192b.p, EPI_PADDED, nullptr, 192, 1, nullptr, nullptr}; break;
    case C_U2A: w = {h->p32_192b.p, h->p32_192h2.p, h->raw32.p, EPI_RAW_STATS, nullptr, 96, 1, "up2.net.1", h->p32_96a.p}; break;
    case C_U2B: w = {h->p32_96a.p, nullptr, h->raw32.p, EPI_RAW_STATS, nullptr, 96, 1, "up2.net.4", h->p32_96b.p}; break;
    case C_US1: w = {h->p64_a.p, nullptr, h->p64_b.p, EPI_PADDED, nullptr, 96, 1, nullptr, nullptr}; break;
    case C_U1A: w = {h->p64_b.p, h->p64_h1.p, h->raw64.p, EPI_RAW_STATS, nullptr, 96, 1, "up1.net.1", h->p64_a.p}; break;
    default: w = {h->p64_a.p, nullptr, h->raw64.p, EPI_RAW_STATS, nullptr, 96, 1, "up1.net.4", h->p64_b.p}; break;  // C_U1B
  }
  if (h->fuse_gn && w.gn) {   // conv + GroupNorm + SiLU in one kernel: the padded activation is the output
    w.out = w.act;
    w.epi = EPI_GN_FUSED;
  }
  return w;
}

static int slots_of(tcs_handle* h, int id) {
  const int r = kConv[id].res;
  return h->use_tc ? tc_slots(r, r) : simt_slots(r, r);
}

// ---- bf16x3 mode: (split source tensors, raw fp32 destination) of every conv ---------------------------------------
// A split tensor lives in a buffer sized for the fp32 tensor it replaces: hi plane first, lo plane `lo` elements later
// (= the element count of the full-chunk tensor, so the planes never move with the size of a pass).
struct SplitSrc { const void* p; size_t lo; };
struct SplitWiring { SplitSrc s0, s1; float* raw; int ldo; int in_pad; };
static size_t padded_elems(const tcs_handle* h, int res, int C) { return static_cast<size_t>(h->chunk) * (res + 2) * (res + 2) * C; }
static SplitWiring split_wiring(tcs_handle* h, int id) {
  const SplitSrc S64{h->split_s.p, padded_elems(h, 64, 96)}, S32{h->split_s.p, padded_elems(h, 32, 192)},
      S16{h->split_s.p, padded_elems(h, 16, 192)}, SY{h->split_s.p, static_cast<size_t>(h->chunk) * 256 * 192};
  const SplitSrc h1{h->p64_h1.p, padded_elems(h, 64, 96)}, h2{h->p32_192h2.p, padded_elems(h, 32, 192)};
  const SplitSrc none{nullptr, 0};
  float *r64 = h->raw64.as<float>(), *r32 = h->raw32.as<float>(), *r16 = h->raw16.as<float>();
  switch (id) {
    case C_D1B: return {S64, none, r64, 96, 1};
    case C_DS1: return {h1, none, r32, 96, 1};
    case C_D2A: return {{h->p32_96a.p, padded_elems(h, 32, 96)}, none, r32, 192, 1};
    case C_D2B: return {{h->p32_192a.p, padded_elems(h, 32, 192)}, none, r32, 192, 1};
    case C_DS2: return {h2, none, r16, 192, 1};
    case C_MA: return {{h->p16_c.p, padded_elems(h, 16, 192)}, none, r16, 192, 1};
    case C_MB: return {{h->p16_b.p, padded_elems(h, 16, 192)}, none, r16, 192, 1};
    case C_QKV: return {S16, none, h->qkv.as<float>(), 576, 1};
    case C_PROJ: return {SY, none, r16, 192, 0};
    case C_US2: return {S32, none, r32, 192, 1};
    case C_U2A: return {{h->p32_192b.p, padded_elems(h, 32, 192)}, h2, r32, 96, 1};
    case C_U2B: return {{h->p32_96a.p, padded_elems(h, 32, 96)}, none, r32, 96, 1};
    case C_US1: return {S64, none, r64, 96, 1};
    case C_U1A: return {{h->p64_b.p, padded_elems(h, 64, 96)}, h1, r64, 96, 1};
    default: return {{h->p64_a.p, padded_elems(h, 64, 96)}, none, r64, 96, 1};   // C_U1B
  }
}

static int build_plans(tcs_handle* h) {
  if (!h->use_tc) return TCS_OK;
  if (h->split3) {
    for (int id = 0; id < C_COUNT; ++id) {
      const SplitWiring w = split_wiring(h, id);
      ConvGeom g = geom_of(id, h->chunk, w.in_pad);
      g.split3 = 1;
      EpiArgs ea{};
      ea.bias = h->dw.at(std::string(kConv[id].key) + ".bias");
      ea.out = w.raw; ea.partials = h->partials.as<float>(); ea.ldo = w.ldo; ea.slots = slots_of(h, id);
      auto lo = [](const SplitSrc& s) { return s.p ? static_cast<const void*>(static_cast<const __nv_bfloat16*>(s.p) + s.lo) : nullptr; };
      TCS_CHECK(conv_tc_make_plan(&h->plan[id], g, w.s0.p, w.s1.p, h->wpack[id].as<__nv_bfloat16>(), EPI_RAW_STATS, ea,
                                  h->sm_count, lo(w.s0), lo(w.s1)));
    }
    return TCS_OK;
  }
  {
    const char* e = getenv("TCS_TC_OUT");   // 0 = keep the CUDA-core out conv (A/B switch)
    h->tc_out = !(e && atoi(e) == 0);
    ConvGeom g = geom_of(C_U1B, h->chunk, 1);
    g.ntot = 16;
    g.kx_in_n = h->eps_kxn ? 1 : 0;
    EpiArgs ea{};
    ea.bias = h->d_bias16; ea.out = nullptr; ea.ldo = 1;
    TCS_CHECK(conv_tc_make_plan(&h->plan_eps, g, h->p64_b.p, nullptr, h->wpack_out.as<__nv_bfloat16>(), EPI_EPS, ea, h->sm_count));
    h->plan_eps_pair = h->plan_eps;
    TCS_CHECK(conv_tc_make_pair(&h->plan_eps_pair, h->p64_b.p, h->chunk));
  }
  for (int id = 0; id < C_COUNT; ++id) {
    const ConvWiring w = wiring(h, id);
    const ConvGeom g = geom_of(id, h->chunk, w.in_pad);
    EpiArgs ea{};
    ea.bias = h->dw.at(std::string(kConv[id].key) + ".bias");
    ea.out = w.out; ea.partials = h->partials.as<float>(); ea.residual = w.residual; ea.ldo = w.ldo;
    ea.slots = slots_of(h, id);
    ea.overflow = h->status.as<int>();
    if (w.epi == EPI_GN_FUSED) {
      ea.gamma = h->dw.at(std::string(w.gn) + ".weight");
      ea.beta = h->dw.at(std::string(w.gn) + ".bias");
    }
    TCS_CHECK(conv_tc_make_plan(&h->plan[id], g, w.s0, w.s1, h->wpack[id].as<__nv_bfloat16>(), w.epi, ea, h->sm_count));
  }
  if (h->fuse_ups) {
    const int ids[2] = {C_US2, C_US1};
    const void* lowres[2] = {h->p16_c.p, h->p32_96b.p};
    for (int k = 0; k < 2; ++k) {
      const ConvWiring w = wiring(h, ids[k]);
      ConvGeom g = geom_of(ids[k], h->chunk, w.in_pad);
      g.ups = 1;
      EpiArgs ea{};
      ea.bias = h->dw.at(std::string(kConv[ids[k]].key) + ".bias");
      ea.out = w.out; ea.partials = h->partials.as<float>(); ea.residual = nullptr; ea.ldo = w.ldo;
      ea.slots = slots_of(h, ids[k]);
      ea.overflow = h->status.as<int>();
      const int rc = conv_tc_make_plan(&h->plan_us[k], g, lowres[k], nullptr, h->wpack[ids[k]].as<__nv_bfloat16>(), EPI_PADDED, ea, h->sm_count);
      if (rc == TCS_ERR_UNSUPPORTED) { h->fuse_ups = false; break; }   // e.g. TCS_GEO=0 (A/B switch): the stand-alone upsample kernel runs
      TCS_CHECK(rc);
    }
  }
  // The fused-GroupNorm kernels are launched as CTA pairs WITH the cooperative attribute where the runtime accepts the
  // combination.  Try it once here, outside any stream capture (a refused launch inside a capture would invalidate the
  // captured graph): a full-width grid over a few images of the (uninitialised) workspace.
  for (int id = 0; id < C_COUNT; ++id) {
    if (!h->plan[id].coop_cluster) continue;
    ConvTcPlan pl = h->plan[id];
    const int B = h->chunk < 16 ? h->chunk : 16;
    pl.p.n_mtiles = B * pl.p.tiles_per_img;
    pl.grid = conv_tc_grid(pl, B, h->sm_count);
    const int rc = conv_tc_launch(pl, h->stream);
    const cudaError_t se = cudaStreamSynchronize(h->stream);
    if (rc != TCS_OK || se != cudaSuccess) {
      cudaGetLastError();
      if (se != cudaSuccess && se != cudaErrorCooperativeLaunchTooLarge && se != cudaErrorInvalidValue)
        return fail(TCS_ERR_CUDA, std::string("trial launch of a fused conv failed: ") + cudaGetErrorString(se));
      for (int j = 0; j < C_COUNT; ++j) h->plan[j].coop_cluster = false;
      break;
    }
  }
  TCS_CUDA(cudaMemsetAsync(h->status.p, 0, 4, h->stream));   // the trial launches ran on uninitialised data
  return TCS_OK;
}

template <typename T>
static int run_conv_inner(tcs_handle* h, int id, int B, cudaStream_t st);

template <typename T>
static int run_conv(tcs_handle* h, int id, int B, cudaStream_t st) {
  if (!h->profiling) return run_conv_inner<T>(h, id, B, st);
  TCS_CUDA(cudaEventRecord(h->prof_ev[2 * id], st));
  TCS_CHECK(run_conv_inner<T>(h, id, B, st));
  TCS_CUDA(cudaEventRecord(h->prof_ev[2 * id + 1], st));
  return TCS_OK;
}

template <typename T>
static int run_conv_inner(tcs_handle* h, int id, int B, cudaStream_t st) {
  ++h->launches;
  if (h->use_tc) {
    ConvTcPlan pl = h->plan[id];
    pl.p.n_mtiles = B * pl.p.tiles_per_img;
    pl.grid = conv_tc_grid(pl, B, h->sm_count);
    return conv_tc_launch(pl, st);
  }
  const ConvWiring w = wiring(h, id);
  const ConvGeom g = geom_of(id, B, w.in_pad);
  EpiArgs ea{};
  ea.bias = h->dw.at(std::string(kConv[id].key) + ".bias");
  ea.out = w.out; ea.partials = h->partials.as<float>(); ea.residual = w.residual; ea.ldo = w.ldo;
  ea.slots = slots_of(h, id);
  return launch_conv_simt<T>(g, static_cast<const T*>(w.s0), static_cast<const T*>(w.s1), h->wpack[id].as<float>(),
                             w.epi, ea, st);
}

// ------------------------------------------------------------------------------------------
// one network pass over B = ns*dup images (B <= chunk)
// ------------------------------------------------------------------------------------------
struct PassArgs {
  const float* x;        // [ns,4096]
  const float* cvec;     // [ns*dup,96]
  const float* tvec;     // rows of 96
  int tvec_stride;       // 0: one row for all samples; 1: a row per sample
  const int* step_ptr;   // device step counter or null
  int trow_off;
  int ns, dup;
  float guidance;
  float* eps;            // [ns,4096]
};

template <typename T>
static int forward_chunk(tcs_handle* h, const PassArgs& a, cudaStream_t st, TapRequest* tap) {
  const int B = a.ns * a.dup;
  float* part = h->partials.as<float>();
  auto gnw = [&](const char* k) { return h->dw.at(std::string(k) + ".weight"); };
  auto gnb = [&](const char* k) { return h->dw.at(std::string(k) + ".bias"); };
  int tap_idx = 0;
  // export helper: kind 0 = fp32 plain, 1 = padded T, 2 = plain T
  auto tapout = [&](int kind, const void* p, int H, int W, int C) -> int {
    const int my = tap_idx++;
    if (!tap || tap->id != my) return 0;
    const int64_t cnt = static_cast<int64_t>(B) * H * W * C;
    if (cnt > tap->capacity) return fail(TCS_ERR_BAD_ARGUMENT, "tcs_debug_layer: output buffer too small");
    if (kind == 0) { TCS_CUDA(cudaMemcpyAsync(tap->out, p, cnt * 4, cudaMemcpyDeviceToDevice, st)); }
    else TCS_CHECK(launch_unpad_to_f32<T>(static_cast<const T*>(p), B, H, W, C, kind == 1 ? 1 : 0, tap->out, st));
    tap->written = cnt;
    return 1;
  };
#define TAP(kind, p, H, W, C) { int _r = tapout(kind, p, H, W, C); if (_r != 0) return _r < 0 ? _r : TCS_OK; }
// conv followed by GroupNorm+SiLU: one fused kernel (tcgen05) or conv -> raw fp32 -> gn_apply
#define CONV_GN(cid, raw, res, C)                                                                         \
  {                                                                                                      \
    const ConvWiring _w = wiring(h, cid);                                                                 \
    TCS_CHECK(run_conv<T>(h, cid, B, st));                                                                \
    if (_w.epi == EPI_GN_FUSED) {                                                                        \
      if (tap && tap->id == tap_idx) return fail(TCS_ERR_UNSUPPORTED, "raw conv output does not exist when GroupNorm is fused"); \
      ++tap_idx;                                                                                         \
    } else {                                                                                             \
      TAP(0, raw, res, res, C);                                                                          \
      GN(_w.gn, raw, slots_of(h, cid), res, C, static_cast<T*>(_w.act));                                  \
    }                                                                                                    \
    TAP(1, _w.act, res, res, C);                                                                         \
  }
#define GN(key, raw, slots, res, C, out) \
  { h->launches += 2; TCS_CHECK(launch_gn_apply<T>(raw, 0, part, slots, gnw(key), gnb(key), B, res, res, C, 1, out, h->gnstats.as<float2>(), st)); }

  // ---- down1 -------------------------------------------------------------------------------
  if (h->fuse_first && !(tap && tap->id == 0)) {
    ++h->launches;
    TCS_CHECK(launch_first_conv_gn<T>(a.x, h->d_w9, a.tvec, a.tvec_stride, a.step_ptr, a.trow_off, a.cvec, a.ns, a.dup,
                                      gnw("down1.net.1"), gnb("down1.net.1"), h->p64_a.as<T>(), st));
    ++tap_idx;
  } else {   // unfused variant (also serves the "down1.net.0.raw" debug tap)
    ++h->launches;
    TCS_CHECK(launch_first_conv(a.x, h->d_w9, a.tvec, a.tvec_stride, a.step_ptr, a.trow_off, a.cvec, a.ns, a.dup,
                                h->raw64.as<float>(), part, st));
    TAP(0, h->raw64.p, 64, 64, 96);
    GN("down1.net.1", h->raw64.p, FIRST_CONV_SLOTS, 64, 96, h->p64_a.as<T>());
  }
  TAP(1, h->p64_a.p, 64, 64, 96);
  CONV_GN(C_D1B, h->raw64.p, 64, 96);
  TCS_CHECK(run_conv<T>(h, C_DS1, B, st));
  TAP(1, h->p32_96a.p, 32, 32, 96);
  // ---- down2 -------------------------------------------------------------------------------
  CONV_GN(C_D2A, h->raw32.p, 32, 192);
  CONV_GN(C_D2B, h->raw32.p, 32, 192);
  TCS_CHECK(run_conv<T>(h, C_DS2, B, st));
  TAP(1, h->p16_a.p, 16, 16, 192);
  // ---- mid + attention ---------------------------------------------------------------------
  CONV_GN(C_MA, h->raw16.p, 16, 192);
  CONV_GN(C_MB, h->raw16.p, 16, 192);   // -> p16_a = x_in of the attention block
  if (h->fuse_attn && sizeof(T) == 2 && !(tap && (tap->id == tap_idx || tap->id == tap_idx + 1))) {
    // GroupNorm -> qkv -> softmax(q k^T) v -> proj -> + x_in in ONE tcgen05 kernel (q, k, v and the scores stay on the SM)
    ++h->launches;
    AttnTcParams ap{};
    ap.x = h->p16_a.as<__nv_bfloat16>(); ap.out = h->p16_c.as<__nv_bfloat16>();
    ap.wpack = h->attn_wpack.as<uint8_t>();
    ap.bias_qkv = h->dw.at("attn.qkv.bias"); ap.bias_proj = h->dw.at("attn.proj.bias");
    ap.gamma = gnw("attn.norm"); ap.beta = gnb("attn.norm");
    ap.B = B;
    if (h->profiling) {   // the block is reported in the attn.qkv slot, attn.proj reads 0
      TCS_CUDA(cudaEventRecord(h->prof_ev[2 * C_QKV], st));
    }
    TCS_CHECK(launch_attn_block_tc(ap, h->sm_count, st));
    if (h->profiling) {
      TCS_CUDA(cudaEventRecord(h->prof_ev[2 * C_QKV + 1], st));
      TCS_CUDA(cudaEventRecord(h->prof_ev[2 * C_PROJ], st));
      TCS_CUDA(cudaEventRecord(h->prof_ev[2 * C_PROJ + 1], st));
    }
    tap_idx += 2;
  } else {
    ++h->launches;   // attn.norm: statistics + normalisation of the 16x16x192 image in one kernel
    TCS_CHECK(launch_gn_image16<T>(h->p16_a.as<T>(), B, gnw("attn.norm"), gnb("attn.norm"), h->p16_b.as<T>(), st));
    TCS_CHECK(run_conv<T>(h, C_QKV, B, st));
    TAP(2, h->qkv.p, 16, 16, 576);
    ++h->launches;
    TCS_CHECK(launch_attention<T>(h->qkv.as<T>(), B, h->atty.as<T>(), st));
    TAP(2, h->atty.p, 16, 16, 192);
    TCS_CHECK(run_conv<T>(h, C_PROJ, B, st));   // + residual x_in -> p16_c
  }
  TAP(1, h->p16_c.p, 16, 16, 192);
  // ---- up2 ---------------------------------------------------------------------------------
  // us*_conv: nn.Upsample(x2, bilinear) + 3x3 conv.  Fused: the conv reads the half-resolution tensor and blends the
  // upsampled window in shared memory; the "us?.up" debug taps need the stand-alone upsample kernel.
  auto us_conv = [&](int k, int id) -> int {
    ++h->launches;
    ConvTcPlan pl = h->plan_us[k];
    pl.p.n_mtiles = B * pl.p.tiles_per_img;
    pl.grid = conv_tc_grid(pl, B, h->sm_count);
    if (h->profiling) TCS_CUDA(cudaEventRecord(h->prof_ev[2 * id], st));
    TCS_CHECK(conv_tc_launch(pl, st));
    if (h->profiling) TCS_CUDA(cudaEventRecord(h->prof_ev[2 * id + 1], st));
    return TCS_OK;
  };
  if (h->fuse_ups && sizeof(T) == 2 && !(tap && tap->id == tap_idx)) {
    ++tap_idx;
    TCS_CHECK(us_conv(0, C_US2));
  } else {
    ++h->launches;
    TCS_CHECK(launch_upsample2x<T>(h->p16_c.as<T>(), B, 16, 16, 192, h->p32_192a.as<T>(), st));
    TAP(1, h->p32_192a.p, 32, 32, 192);
    TCS_CHECK(run_conv<T>(h, C_US2, B, st));
  }
  TAP(1, h->p32_192b.p, 32, 32, 192);
  CONV_GN(C_U2A, h->raw32.p, 32, 96);
  CONV_GN(C_U2B, h->raw32.p, 32, 96);
  // ---- up1 ---------------------------------------------------------------------------------
  if (h->fuse_ups && sizeof(T) == 2 && !(tap && tap->id == tap_idx)) {
    ++tap_idx;
    TCS_CHECK(us_conv(1, C_US1));
  } else {
    ++h->launches;
    TCS_CHECK(launch_upsample2x<T>(h->p32_96b.as<T>(), B, 32, 32, 96, h->p64_a.as<T>(), st));
    TAP(1, h->p64_a.p, 64, 64, 96);
    TCS_CHECK(run_conv<T>(h, C_US1, B, st));
  }
  TAP(1, h->p64_b.p, 64, 64, 96);
  CONV_GN(C_U1A, h->raw64.p, 64, 96);
  CONV_GN(C_U1B, h->raw64.p, 64, 96);
  // ---- out conv + CFG combine ------------------------------------------------------------------
  ++h->launches;
  if (h->use_tc && h->tc_out) {
    ConvTcPlan pl = a.dup == 2 ? h->plan_eps_pair : h->plan_eps;
    pl.p.n_mtiles = (a.dup == 2 ? B / 2 : B) * pl.p.tiles_per_img;
    pl.p.guidance = a.guidance;
    pl.p.epi.out = a.eps;
    pl.grid = conv_tc_grid(pl, B, h->sm_count);
    TCS_CHECK(conv_tc_launch(pl, st));
  } else {
    TCS_CHECK(launch_out_conv<T>(h->p64_b.as<T>(), h->d_wout, h->out_bias, a.ns, a.dup, a.guidance, a.eps, st));
  }
  if (tap && tap->id == kNumTaps - 1) {
    const int64_t cnt = static_cast<int64_t>(a.ns) * 4096;
    if (cnt > tap->capacity) return fail(TCS_ERR_BAD_ARGUMENT, "tcs_debug_layer: output buffer too small");
    TCS_CUDA(cudaMemcpyAsync(tap->out, a.eps, cnt * 4, cudaMemcpyDeviceToDevice, st));
    tap->written = cnt;
  }
#undef TAP
#undef GN
#undef CONV_GN
  return TCS_OK;
}

// ------------------------------------------------------------------------------------------
// the same pass in bf16x3 mode: every conv = tcgen05 over split operands -> raw fp32, everything else fp32 FFMA kernels
// ------------------------------------------------------------------------------------------
static int forward_chunk_split3(tcs_handle* h, const PassArgs& a, cudaStream_t st, TapRequest* tap) {
  const int B = a.ns * a.dup;
  float* part = h->partials.as<float>();
  float2* stats = h->gnstats.as<float2>();
  auto gnw = [&](const char* k) { return h->dw.at(std::string(k) + ".weight"); };
  auto gnb = [&](const char* k) { return h->dw.at(std::string(k) + ".bias"); };
  auto bf = [](void* p) { return static_cast<__nv_bfloat16*>(p); };
  int tap_idx = 0;
  // kind 0 = raw fp32 plain, 1 = padded fp32, 2 = plain fp32, 3 = split padded, -1 = not materialised in this mode
  auto tapout = [&](int kind, const void* p, size_t lo, int res, int C) -> int {
    const int my = tap_idx++;
    if (!tap || tap->id != my) return 0;
    if (kind < 0) return fail(TCS_ERR_UNSUPPORTED, "this activation is not materialised in bf16x3 mode");
    const int64_t cnt = static_cast<int64_t>(B) * res * res * C;
    if (cnt > tap->capacity) return fail(TCS_ERR_BAD_ARGUMENT, "tcs_debug_layer: output buffer too small");
    if (kind == 0 || kind == 2) { TCS_CUDA(cudaMemcpyAsync(tap->out, p, cnt * 4, cudaMemcpyDeviceToDevice, st)); }
    else if (kind == 1) TCS_CHECK(launch_unpad_to_f32<float>(static_cast<const float*>(p), B, res, res, C, 1, tap->out, st));
    else TCS_CHECK(launch_unsplit_to_f32(static_cast<const __nv_bfloat16*>(p), lo, B, res, res, C, 1, tap->out, st));
    tap->written = cnt;
    return 1;
  };
#define TAP(kind, p, lo, res, C) { int _r = tapout(kind, p, lo, res, C); if (_r != 0) return _r < 0 ? _r : TCS_OK; }
  auto conv = [&](int id) -> int {
    ++h->launches;
    ConvTcPlan pl = h->plan[id];
    pl.p.n_mtiles = B * pl.p.tiles_per_img;
    pl.grid = conv_tc_grid(pl, B, h->sm_count);
    if (h->profiling) TCS_CUDA(cudaEventRecord(h->prof_ev[2 * id], st));
    TCS_CHECK(conv_tc_launch(pl, st));
    if (h->profiling) TCS_CUDA(cudaEventRecord(h->prof_ev[2 * id + 1], st));
    return TCS_OK;
  };
  // fp32 tensor -> split scratch (the conv that follows reads it)
  auto split_in = [&](const float* src, size_t elems_per_img, size_t lo) -> int {
    ++h->launches;
    return launch_split(src, static_cast<size_t>(B) * elems_per_img, bf(h->split_s.p), lo, st);
  };
  // raw conv output -> GroupNorm + SiLU -> split padded tensor (next consumer is a conv) or fp32 padded (FFMA consumer)
  auto gn_split = [&](const char* key, int id, const float* raw, int res, int C, void* out) -> int {
    h->launches += 2;
    TCS_CHECK(launch_gn_finalize(part, slots_of(h, id), B, res, res, C, stats, st));
    return launch_raw_to_padded(0, raw, stats, gnw(key), gnb(key), nullptr, B, res, res, C, out, padded_elems(h, res, C), st);
  };
  auto gn_f32 = [&](const char* key, int id, const float* raw, int res, int C, float* out) -> int {
    h->launches += 2;
    return launch_gn_apply<float>(raw, 0, part, slots_of(h, id), gnw(key), gnb(key), B, res, res, C, 1, out, stats, st);
  };
  auto pad_split = [&](const float* raw, int res, int C, void* out) -> int {
    ++h->launches;
    return launch_raw_to_padded(1, raw, nullptr, nullptr, nullptr, nullptr, B, res, res, C, out, padded_elems(h, res, C), st);
  };
  float *r64 = h->raw64.as<float>(), *r32 = h->raw32.as<float>(), *r16 = h->raw16.as<float>();
  const size_t E64 = padded_elems(h, 64, 96), E32a = padded_elems(h, 32, 96), E32b = padded_elems(h, 32, 192),
               E16 = padded_elems(h, 16, 192);
  // ---- down1 ---------------------------------------------------------------------------------
  if (!(tap && tap->id == 0)) {
    ++h->launches;
    TCS_CHECK(launch_first_conv_gn<float>(a.x, h->d_w9, a.tvec, a.tvec_stride, a.step_ptr, a.trow_off, a.cvec, a.ns, a.dup,
                                          gnw("down1.net.1"), gnb("down1.net.1"), h->p64_a.as<float>(), st));
    ++tap_idx;
  } else {
    ++h->launches;
    TCS_CHECK(launch_first_conv(a.x, h->d_w9, a.tvec, a.tvec_stride, a.step_ptr, a.trow_off, a.cvec, a.ns, a.dup, r64, part, st));
    TAP(0, r64, 0, 64, 96);
  }
  TAP(1, h->p64_a.p, 0, 64, 96);
  TCS_CHECK(split_in(h->p64_a.as<float>(), 66 * 66 * 96, E64));
  TCS_CHECK(conv(C_D1B));
  TAP(0, r64, 0, 64, 96);
  TCS_CHECK(gn_split("down1.net.4", C_D1B, r64, 64, 96, h->p64_h1.p));
  TAP(3, h->p64_h1.p, E64, 64, 96);
  TCS_CHECK(conv(C_DS1));
  TCS_CHECK(pad_split(r32, 32, 96, h->p32_96a.p));
  TAP(3, h->p32_96a.p, E32a, 32, 96);
  // ---- down2 ---------------------------------------------------------------------------------
  TCS_CHECK(conv(C_D2A));
  TAP(0, r32, 0, 32, 192);
  TCS_CHECK(gn_split("down2.net.1", C_D2A, r32, 32, 192, h->p32_192a.p));
  TAP(3, h->p32_192a.p, E32b, 32, 192);
  TCS_CHECK(conv(C_D2B));
  TAP(0, r32, 0, 32, 192);
  TCS_CHECK(gn_split("down2.net.4", C_D2B, r32, 32, 192, h->p32_192h2.p));
  TAP(3, h->p32_192h2.p, E32b, 32, 192);
  TCS_CHECK(conv(C_DS2));
  TCS_CHECK(pad_split(r16, 16, 192, h->p16_c.p));
  TAP(3, h->p16_c.p, E16, 16, 192);
  // ---- mid + attention -----------------------------------------------------------------------
  TCS_CHECK(conv(C_MA));
  TAP(0, r16, 0, 16, 192);
  TCS_CHECK(gn_split("mid.net.1", C_MA, r16, 16, 192, h->p16_b.p));
  TAP(3, h->p16_b.p, E16, 16, 192);
  TCS_CHECK(conv(C_MB));
  TAP(0, r16, 0, 16, 192);
  TCS_CHECK(gn_f32("mid.net.4", C_MB, r16, 16, 192, h->p16_a.as<float>()));   // x_in of the attention block (fp32)
  TAP(1, h->p16_a.p, 0, 16, 192);
  ++h->launches;
  TCS_CHECK(launch_gn_image16<float>(h->p16_a.as<float>(), B, gnw("attn.norm"), gnb("attn.norm"), h->p16_b.as<float>(), st));
  TCS_CHECK(split_in(h->p16_b.as<float>(), 18 * 18 * 192, E16));
  TCS_CHECK(conv(C_QKV));
  TAP(2, h->qkv.p, 0, 16, 576);
  ++h->launches;
  TCS_CHECK(launch_attention<float>(h->qkv.as<float>(), B, h->atty.as<float>(), st));
  TAP(2, h->atty.p, 0, 16, 192);
  TCS_CHECK(split_in(h->atty.as<float>(), 256 * 192, static_cast<size_t>(h->chunk) * 256 * 192));
  TCS_CHECK(conv(C_PROJ));
  ++h->launches;
  TCS_CHECK(launch_raw_to_padded(2, r16, nullptr, nullptr, nullptr, h->p16_a.as<float>(), B, 16, 16, 192, h->p16_c.p, 0, st));
  TAP(1, h->p16_c.p, 0, 16, 192);
  // ---- up2 -----------------------------------------------------------------------------------
  ++h->launches;
  TCS_CHECK(launch_upsample2x<float>(h->p16_c.as<float>(), B, 16, 16, 192, h->p32_192a.as<float>(), st));
  TAP(1, h->p32_192a.p, 0, 32, 192);
  TCS_CHECK(split_in(h->p32_192a.as<float>(), 34 * 34 * 192, E32b));
  TCS_CHECK(conv(C_US2));
  TCS_CHECK(pad_split(r32, 32, 192, h->p32_192b.p));
  TAP(3, h->p32_192b.p, E32b, 32, 192);
  TCS_CHECK(conv(C_U2A));
  TAP(0, r32, 0, 32, 96);
  TCS_CHECK(gn_split("up2.net.1", C_U2A, r32, 32, 96, h->p32_96a.p));
  TAP(3, h->p32_96a.p, E32a, 32, 96);
  TCS_CHECK(conv(C_U2B));
  TAP(0, r32, 0, 32, 96);
  TCS_CHECK(gn_f32("up2.net.4", C_U2B, r32, 32, 96, h->p32_96b.as<float>()));
  TAP(1, h->p32_96b.p, 0, 32, 96);
  // ---- up1 -----------------------------------------------------------------------------------
  ++h->launches;
  TCS_CHECK(launch_upsample2x<float>(h->p32_96b.as<float>(), B, 32, 32, 96, h->p64_a.as<float>(), st));
  TAP(1, h->p64_a.p, 0, 64, 96);
  TCS_CHECK(split_in(h->p64_a.as<float>(), 66 * 66 * 96, E64));
  TCS_CHECK(conv(C_US1));
  TCS_CHECK(pad_split(r64, 64, 96, h->p64_b.p));
  TAP(3, h->p64_b.p, E64, 64, 96);
  TCS_CHECK(conv(C_U1A));
  TAP(0, r64, 0, 64, 96);
  TCS_CHECK(gn_split("up1.net.1", C_U1A, r64, 64, 96, h->p64_a.p));
  TAP(3, h->p64_a.p, E64, 64, 96);
  TCS_CHECK(conv(C_U1B));
  TAP(0, r64, 0, 64, 96);
  TCS_CHECK(gn_f32("up1.net.4", C_U1B, r64, 64, 96, h->p64_b.as<float>()));
  TAP(1, h->p64_b.p, 0, 64, 96);
  ++h->launches;
  TCS_CHECK(launch_out_conv<float>(h->p64_b.as<float>(), h->d_wout, h->out_bias, a.ns, a.dup, a.guidance, a.eps, st));
  if (tap && tap->id == kNumTaps - 1) {
    const int64_t cnt = static_cast<int64_t>(a.ns) * 4096;
    if (cnt > tap->capacity) return fail(TCS_ERR_BAD_ARGUMENT, "tcs_debug_layer: output buffer too small");
    TCS_CUDA(cudaMemcpyAsync(tap->out, a.eps, cnt * 4, cudaMemcpyDeviceToDevice, st));
    tap->written = cnt;
  }
#undef TAP
  return TCS_OK;
}

static int forward_one(tcs_handle* h, const PassArgs& a, cudaStream_t st, TapRequest* tap) {
  if (h->split3) return forward_chunk_split3(h, a, st, tap);
  if (h->bf16) return forward_chunk<__nv_bfloat16>(h, a, st, tap);
  return forward_chunk<float>(h, a, st, tap);
}

// network over all n samples, chunk by chunk
static int forward_all(tcs_handle* h, const float* x, const float* cvec, const float* tvec, int tvec_stride,
                       const int* step_ptr, int trow_off, int n, int dup, float guidance, float* eps, cudaStream_t st) {
  const int per = h->chunk / dup;  // samples per pass
  for (int i0 = 0; i0 < n; i0 += per) {
    PassArgs a;
    a.ns = (n - i0 < per) ? n - i0 : per;
    a.dup = dup;
    a.x = x + static_cast<size_t>(i0) * 4096;
    a.cvec = cvec + static_cast<size_t>(i0) * dup * 96;
    a.tvec = tvec + (tvec_stride ? static_cast<size_t>(i0) * 96 : 0);
    a.tvec_stride = tvec_stride;
    a.step_ptr = step_ptr; a.trow_off = trow_off;
    a.guidance = guidance;
    a.eps = eps + static_cast<size_t>(i0) * 4096;
    TCS_CHECK(forward_one(h, a, st, nullptr));
  }
  return TCS_OK;
}

// trace copy: dst + (step*mult + add)*stride  <-  src   (step read on the device)
__global__ void __launch_bounds__(256) trace_copy_kernel(float4* __restrict__ dst, const float4* __restrict__ src,
                                                        const int* __restrict__ step_ptr, int mult, int add,
                                                        long long stride_v, long long nv) {
  const long long v = blockIdx.x * 256LL + threadIdx.x;
  if (v >= nv) return;
  const long long row = static_cast<long long>(step_ptr ? *step_ptr : 0) * mult + add;
  dst[row * stride_v + v] = src[v];
}
static int trace_copy(tcs_handle* h, float* dst, const float* src, const int* step_ptr, int mult, int add, int n,
                      cudaStream_t st) {
  if (!dst) return TCS_OK;
  const long long nv = static_cast<long long>(n) * 1024;
  ++h->launches;
  trace_copy_kernel<<<static_cast<unsigned>((nv + 255) / 256), 256, 0, st>>>(
      reinterpret_cast<float4*>(dst), reinterpret_cast<const float4*>(src), step_ptr, mult, add, nv, nv);
  TCS_CUDA(cudaGetLastError());
  return TCS_OK;
}

__global__ void cond_grid_kernel(int n, long long offset, long long n_total, float theta_max, int n_types, int ycd,
                                 long long* y_cat, float* y_cont) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const long long gi = offset + i;
  y_cat[i] = gi % n_types;
  // torch.linspace(0, theta_max, n_total) in fp32
  const float step = n_total > 1 ? (theta_max - 0.0f) / static_cast<float>(n_total - 1) : 0.f;
  const long long halfway = n_total / 2;
  const float th = gi < halfway ? 0.0f + step * static_cast<float>(gi) : theta_max - step * static_cast<float>(n_total - gi - 1);
  for (int k = 0; k < ycd; ++k) y_cont[static_cast<size_t>(i) * ycd + k] = (k == 1) ? th : 0.f;
}

}  // namespace tcs

// ==========================================================================================
// C ABI
// ==========================================================================================
extern "C" {

const char* tcs_last_error(void) { return g_err.c_str(); }
#ifndef TCS_SRC_HASH
#define TCS_SRC_HASH "unknown"
#endif
// build.py passes the SHA-256 of every source and header of the library; __graft_entry__.build() and the tests compare
// it with the tree, so that a prebuilt libtcs.so that does not match the sources is rebuilt / reported, never used silently
const char* tcs_build_info(void) {
  return "libtcs sm_100a: tcgen05 implicit-GEMM conv (bf16, bf16x3) + FFMA conv (fp32), built " __DATE__ " " __TIME__
         " TCS_SRC_HASH=" TCS_SRC_HASH;
}
int64_t tcs_launch_count(const tcs_handle* h) { return h ? h->launches : 0; }
int32_t tcs_check(tcs_handle* h) {
  if (!h) return fail(TCS_ERR_BAD_ARGUMENT, "tcs_check: null handle");
  TCS_CUDA(cudaSetDevice(h->cfg.device));
  int bits = 0;
  TCS_CUDA(cudaMemcpyAsync(&bits, h->status.p, 4, cudaMemcpyDeviceToHost, h->stream));
  TCS_CUDA(cudaStreamSynchronize(h->stream));
  if (bits) TCS_CUDA(cudaMemsetAsync(h->status.p, 0, 4, h->stream));
  return bits & 0x7fffffff;
}
int32_t tcs_launch_mode(const tcs_handle* h) {
  if (!h || !h->finalized || !h->use_tc) return 0;
  const ConvTcPlan& pl = h->plan[C_D1B];
  return (h->fuse_gn ? 1 : 0) | (pl.coop_cluster ? 2 : 0) | (pl.max_ctas << 8);
}
int32_t tcs_nfe(int32_t sampler, int32_t steps) { return sampler == TCS_SAMPLER_ODE ? 2 * steps + 1 : steps + 1; }

void tcs_default_config(tcs_config* c) {
  if (!c) return;
  memset(c, 0, sizeof(*c));
  c->n_types = 4; c->y_cont_dim = 4; c->base_ch = 96; c->emb_dim = 128; c->cond_ch = 8; c->time_ch = 8;
  c->beta_min = 0.1; c->beta_max = 30.0;
  c->precision = TCS_BF16; c->engine = TCS_ENGINE_AUTO; c->device = 0; c->chunk = 0; c->use_graph = 1; c->fuse_gn = 1;
}

int tcs_time_grid_host(int32_t steps, double t_end, float* ts) {
  if (steps < 1 || !ts) return fail(TCS_ERR_BAD_ARGUMENT, "tcs_time_grid_host: steps >= 1 and ts required");
  time_grid_host(steps, t_end, ts);
  return TCS_OK;
}
int tcs_schedule_host(double bmin, double bmax, float t, float* beta, float* alpha, float* sigma) {
  const Sched s{bmin, bmax};
  if (beta) *beta = s.beta(t);
  if (alpha) *alpha = s.alpha(t);
  if (sigma) *sigma = s.sigma(t);
  return TCS_OK;
}
int tcs_dpm_schedule_host(int32_t steps, double t_end, double bmin, double bmax, float* ts, float* coef) {
  if (steps < 1 || !ts || !coef) return fail(TCS_ERR_BAD_ARGUMENT, "tcs_dpm_schedule_host: steps >= 1, ts and coef required");
  if (!(t_end > 0.0 && t_end < 1.0)) return fail(TCS_ERR_BAD_ARGUMENT, "tcs_dpm_schedule_host: t_end must be in (0,1)");
  if (!(bmin > 0.0 && bmax >= bmin)) return fail(TCS_ERR_BAD_ARGUMENT, "tcs_dpm_schedule_host: need 0 < beta_min <= beta_max");
  std::vector<DpmCoef> k(steps);
  dpm_schedule_host(steps, t_end, bmin, bmax, ts, k.data());
  memcpy(coef, k.data(), sizeof(DpmCoef) * steps);
  return TCS_OK;
}

int tcs_create(tcs_handle** out, const tcs_config* cfg) {
  if (!out || !cfg) return fail(TCS_ERR_BAD_ARGUMENT, "tcs_create: null argument");
  *out = nullptr;
  if (cfg->base_ch != 96 || cfg->emb_dim != 128 || cfg->cond_ch != 8 || cfg->time_ch != 8)
    return fail(TCS_ERR_UNSUPPORTED,
                "this build supports base_ch=96, emb_dim=128, cond_ch=8, time_ch=8 only (got " +
                    std::to_string(cfg->base_ch) + "/" + std::to_string(cfg->emb_dim) + "/" +
                    std::to_string(cfg->cond_ch) + "/" + std::to_string(cfg->time_ch) + ")");
  if (cfg->n_types < 1 || cfg->y_cont_dim < 3 || cfg->y_cont_dim > 16)
    return fail(TCS_ERR_BAD_ARGUMENT, "tcs_create: need n_types >= 1 and 3 <= y_cont_dim <= 16 (theta sin/cos uses columns 1,2)");
  if (cfg->precision != TCS_FP32 && cfg->precision != TCS_BF16) return fail(TCS_ERR_BAD_ARGUMENT, "tcs_create: bad precision");
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0)
    return fail(TCS_ERR_CUDA, std::string("no CUDA device: ") + cudaGetErrorString(e) + " (libtcs has no CPU fallback)");
  if (cfg->device < 0 || cfg->device >= ndev) return fail(TCS_ERR_BAD_ARGUMENT, "tcs_create: bad device ordinal");
  TCS_CUDA(cudaSetDevice(cfg->device));
  cudaDeviceProp prop;
  TCS_CUDA(cudaGetDeviceProperties(&prop, cfg->device));
  if (prop.major != 10)
    return fail(TCS_ERR_UNSUPPORTED, std::string("libtcs is built for sm_100a only; device is ") + prop.name);
  std::unique_ptr<tcs_handle> h(new tcs_handle());
  h->cfg = *cfg;
  h->sm_count = prop.multiProcessorCount;
  h->bf16 = cfg->precision == TCS_BF16;
  h->esz = h->bf16 ? 2 : 4;
  int eng = cfg->engine;
  if (eng == TCS_ENGINE_AUTO) eng = h->bf16 ? TCS_ENGINE_TCGEN05 : TCS_ENGINE_SIMT;
  h->use_tc = eng == TCS_ENGINE_TCGEN05;
  h->split3 = h->use_tc && !h->bf16;   // fp32 operands as bf16 hi + lo pairs, three MMAs per product (1e-4 parity mode)
  {
    const char* e = getenv("TCS_FUSE_GN");   // 0 = keep conv -> raw fp32 -> gn_apply (A/B switch)
    h->fuse_gn = h->use_tc && !h->split3 && cfg->fuse_gn != 0 && !(e && atoi(e) == 0);
    h->fuse_first = !(e && atoi(e) == 0);
    const char* eu = getenv("TCS_FUSE_UPS");
    h->fuse_ups = h->use_tc && !h->split3 && !(eu && atoi(eu) == 0);
    const char* ea = getenv("TCS_FUSE_ATTN");
    h->fuse_attn = h->use_tc && !h->split3 && !(ea && atoi(ea) == 0);
  }
  h->chunk = cfg->chunk > 0 ? cfg->chunk : 2048;
  if (h->chunk % 2) h->chunk += 1;
  TCS_CUDA(cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking));
  TCS_CUDA(cudaEventCreateWithFlags(&h->ev_in, cudaEventDisableTiming));
  TCS_CUDA(cudaEventCreateWithFlags(&h->ev_out, cudaEventDisableTiming));
  TCS_CUDA(cudaEventCreateWithFlags(&h->ev_pinned, cudaEventDisableTiming));
  TCS_CHECK(h->step_ctr.ensure(16));
  TCS_CHECK(h->status.ensure(16));
  TCS_CUDA(cudaMemset(h->status.p, 0, 16));
  *out = h.release();
  return TCS_OK;
}

void tcs_destroy(tcs_handle* h) {
  if (!h) return;
  cudaSetDevice(h->cfg.device);
  cudaStreamSynchronize(h->stream);
  delete h;
}

int tcs_set_weight(tcs_handle* h, const char* key, const float* data, const int64_t* shape, int32_t ndim) {
  if (!h || !key || !data || !shape || ndim < 1 || ndim > 4) return fail(TCS_ERR_BAD_ARGUMENT, "tcs_set_weight: bad argument");
  TCS_CUDA(cudaSetDevice(h->cfg.device));
  HostTensor t;
  size_t cnt = 1;
  for (int i = 0; i < ndim; ++i) { t.shape.push_back(shape[i]); cnt *= static_cast<size_t>(shape[i]); }
  t.v.resize(cnt);
  TCS_CUDA(cudaMemcpy(t.v.data(), data, cnt * 4, cudaMemcpyDefault));
  h->host_w[key] = std::move(t);
  h->finalized = false;
  return TCS_OK;
}

int tcs_finalize_weights(tcs_handle* h) {
  if (!h) return fail(TCS_ERR_BAD_ARGUMENT, "tcs_finalize_weights: null handle");
  TCS_CUDA(cudaSetDevice(h->cfg.device));
  const auto exp = expected_weights(h->cfg);
  size_t total = 0;
  for (const auto& kv : exp) {
    auto it = h->host_w.find(kv.first);
    if (it == h->host_w.end()) return fail(TCS_ERR_STATE, "missing state-dict tensor: " + kv.first);
    if (it->second.shape != kv.second) return fail(TCS_ERR_BAD_ARGUMENT, "state-dict tensor has the wrong shape: " + kv.first);
    total += (it->second.v.size() + 63) / 64 * 64;
  }
  if (h->host_w.size() != exp.size()) return fail(TCS_ERR_BAD_ARGUMENT, "unexpected extra state-dict tensors");
  // derived: wsum [96][16], w9 [96][9], wout [9][96]
  const HostTensor& w0 = h->host_w.at("down1.net.0.weight");  // [96,17,3,3]
  std::vector<float> wsum(96 * 16), w9(96 * 9), wout(9 * 96);
  for (int oc = 0; oc < 96; ++oc) {
    for (int k = 0; k < 9; ++k) w9[oc * 9 + k] = w0.v[(oc * 17 + 0) * 9 + k];
    for (int c = 0; c < 16; ++c) {
      float s = 0.f;
      for (int k = 0; k < 9; ++k) s += w0.v[(oc * 17 + 1 + c) * 9 + k];
      wsum[oc * 16 + c] = s;
    }
  }
  const HostTensor& wo = h->host_w.at("out.weight");  // [1,96,3,3]
  for (int c = 0; c < 96; ++c)
    for (int k = 0; k < 9; ++k) wout[k * 96 + c] = wo.v[c * 9 + k];
  h->out_bias = h->host_w.at("out.bias").v[0];
  const size_t extra = 96 * 16 + 96 * 9 + 9 * 96 + 64 + 256;
  TCS_CHECK(h->arena.ensure((total + extra) * 4));
  float* base = h->arena.as<float>();
  size_t off = 0;
  h->dw.clear();
  for (const auto& kv : exp) {
    const HostTensor& t = h->host_w.at(kv.first);
    TCS_CUDA(cudaMemcpy(base + off, t.v.data(), t.v.size() * 4, cudaMemcpyHostToDevice));
    h->dw[kv.first] = base + off;
    off += (t.v.size() + 63) / 64 * 64;
  }
  auto put = [&](const std::vector<float>& v, const float** dst) -> int {
    TCS_CUDA(cudaMemcpy(base + off, v.data(), v.size() * 4, cudaMemcpyHostToDevice));
    *dst = base + off;
    off += (v.size() + 63) / 64 * 64;
    return TCS_OK;
  };
  const float* d_wsum = nullptr;
  std::vector<float> bias16(16, 0.f);
  bias16[0] = h->out_bias;
  TCS_CHECK(put(bias16, &h->d_bias16));
  TCS_CHECK(put(wsum, &d_wsum));
  TCS_CHECK(put(w9, &h->d_w9));
  TCS_CHECK(put(wout, &h->d_wout));
  EmbedWeights& ew = h->ew;
  ew.cat_emb = h->dw.at("cond_emb.cat_emb.weight");
  ew.cm0_w = h->dw.at("cond_emb.cont_mlp.0.weight"); ew.cm0_b = h->dw.at("cond_emb.cont_mlp.0.bias");
  ew.cm2_w = h->dw.at("cond_emb.cont_mlp.2.weight"); ew.cm2_b = h->dw.at("cond_emb.cont_mlp.2.bias");
  ew.co_w = h->dw.at("cond_emb.out.1.weight"); ew.co_b = h->dw.at("cond_emb.out.1.bias");
  ew.tm0_w = h->dw.at("time_mlp.0.weight"); ew.tm0_b = h->dw.at("time_mlp.0.bias");
  ew.tm2_w = h->dw.at("time_mlp.2.weight"); ew.tm2_b = h->dw.at("time_mlp.2.bias");
  ew.tc_w = h->dw.at("to_cond_map.weight"); ew.tc_b = h->dw.at("to_cond_map.bias");
  ew.tt_w = h->dw.at("to_time_map.weight"); ew.tt_b = h->dw.at("to_time_map.bias");
  ew.wsum = d_wsum; ew.b0 = h->dw.at("down1.net.0.bias");
  ew.n_types = h->cfg.n_types; ew.y_cont_dim = h->cfg.y_cont_dim;
  // conv weights for the active engine
  for (int id = 0; id < C_COUNT; ++id) {
    ConvGeom g = geom_of(id, 1, 1);
    g.split3 = h->split3 ? 1 : 0;
    const HostTensor& w = h->host_w.at(std::string(kConv[id].key) + ".weight");
    if (h->use_tc) {
      std::vector<__nv_bfloat16> pk(conv_tc_packed_elems(g));
      conv_tc_pack_weights(g, EPI_PADDED, w.v.data(), pk.data());   // (any epilogue but EPI_EPS: same tile shape)
      TCS_CHECK(h->wpack[id].ensure(pk.size() * 2));
      TCS_CUDA(cudaMemcpy(h->wpack[id].p, pk.data(), pk.size() * 2, cudaMemcpyHostToDevice));
    } else {
      std::vector<float> pk(w.v.size());
      conv_simt_pack_weights(g, w.v.data(), pk.data(), h->bf16);
      TCS_CHECK(h->wpack[id].ensure(pk.size() * 4));
      TCS_CUDA(cudaMemcpy(h->wpack[id].p, pk.data(), pk.size() * 4, cudaMemcpyHostToDevice));
    }
  }
  if (h->use_tc && !h->split3) {   // out conv as a 16-channel GEMM: row 0 = out.weight, rows 1..15 zero
    ConvGeom g = geom_of(C_U1B, 1, 1);
    g.ntot = 16;
    {
      const char* e = getenv("TCS_EPS_KXN");   // 0 = one window per kx tap (A/B switch)
      h->eps_kxn = !(e && atoi(e) == 0);
    }
    g.kx_in_n = h->eps_kxn ? 1 : 0;
    std::vector<float> w16(16 * 96 * 9, 0.f);
    for (int k = 0; k < 96 * 9; ++k) w16[k] = wo.v[k];
    std::vector<__nv_bfloat16> pk(conv_tc_packed_elems(g));
    conv_tc_pack_weights(g, EPI_EPS, w16.data(), pk.data());
    TCS_CHECK(h->wpack_out.ensure(pk.size() * 2));
    TCS_CUDA(cudaMemcpy(h->wpack_out.p, pk.data(), pk.size() * 2, cudaMemcpyHostToDevice));
  }
  if (h->fuse_attn) {
    std::vector<uint8_t> pk(attn_tc_wpack_bytes());
    attn_tc_pack_weights(h->host_w.at("attn.qkv.weight").v.data(), h->host_w.at("attn.proj.weight").v.data(), pk.data());
    TCS_CHECK(h->attn_wpack.ensure(pk.size()));
    TCS_CUDA(cudaMemcpy(h->attn_wpack.p, pk.data(), pk.size(), cudaMemcpyHostToDevice));
  }
  TCS_CHECK(alloc_workspace(h));
  TCS_CHECK(build_plans(h));
  if (h->gexec) { cudaGraphExecDestroy(h->gexec); h->gexec = nullptr; h->gkey.n = -1; }
  h->finalized = true;
  return TCS_OK;
}

static int check_ready(tcs_handle* h, const char* who) {
  if (!h) return fail(TCS_ERR_BAD_ARGUMENT, std::string(who) + ": null handle");
  if (!h->finalized) return fail(TCS_ERR_STATE, std::string(who) + ": call tcs_finalize_weights first");
  return TCS_OK;
}

int tcs_score(tcs_handle* h, const float* x, const float* t, const int64_t* y_cat, const float* y_cont, int32_t n,
              float guidance, float* eps_out, void* stream) {
  TCS_CHECK(check_ready(h, "tcs_score"));
  if (n < 0 || (n > 0 && (!x || !t || !y_cat || !y_cont || !eps_out))) return fail(TCS_ERR_BAD_ARGUMENT, "tcs_score: null tensor");
  if (n == 0) return TCS_OK;
  cudaStream_t user = static_cast<cudaStream_t>(stream);
  TCS_CHECK(enter(h, user));
  const int dup = guidance > 0.f ? 2 : 1;
  TCS_CHECK(h->cvec.ensure(static_cast<size_t>(n) * dup * 96 * 4));
  TCS_CHECK(h->tvec.ensure(static_cast<size_t>(n) * 96 * 4));
  cudaStream_t st = h->stream;
  h->launches += 2;
  TCS_CHECK(launch_cond_embed(h->ew, y_cat, y_cont, n, dup, h->cvec.as<float>(), st));
  TCS_CHECK(launch_time_embed(h->ew, t, n, h->tvec.as<float>(), st));
  TCS_CHECK(forward_all(h, x, h->cvec.as<float>(), h->tvec.as<float>(), 1, nullptr, 0, n, dup, guidance, eps_out, st));
  return leave(h, user);
}

int tcs_score_profiled(tcs_handle* h, const float* x, const float* t, const int64_t* y_cat, const float* y_cont,
                       int32_t n, float guidance, float* eps_out, float* conv_ms, float* total_ms, void* stream) {
  TCS_CHECK(check_ready(h, "tcs_score_profiled"));
  if (!x || !t || !y_cat || !y_cont || !eps_out || !conv_ms || !total_ms || n < 1)
    return fail(TCS_ERR_BAD_ARGUMENT, "tcs_score_profiled: bad argument");
  const int dup = guidance > 0.f ? 2 : 1;
  if (n * dup > h->chunk) return fail(TCS_ERR_BAD_ARGUMENT, "tcs_score_profiled: n exceeds one pass (chunk)");
  cudaStream_t user = static_cast<cudaStream_t>(stream);
  TCS_CHECK(enter(h, user));
  for (cudaEvent_t& e : h->prof_ev)
    if (!e) TCS_CUDA(cudaEventCreate(&e));
  TCS_CHECK(h->cvec.ensure(static_cast<size_t>(n) * dup * 96 * 4));
  TCS_CHECK(h->tvec.ensure(static_cast<size_t>(n) * 96 * 4));
  cudaStream_t st = h->stream;
  TCS_CHECK(launch_cond_embed(h->ew, y_cat, y_cont, n, dup, h->cvec.as<float>(), st));
  TCS_CHECK(launch_time_embed(h->ew, t, n, h->tvec.as<float>(), st));
  PassArgs a;
  a.x = x; a.cvec = h->cvec.as<float>(); a.tvec = h->tvec.as<float>(); a.tvec_stride = 1; a.step_ptr = nullptr;
  a.trow_off = 0; a.ns = n; a.dup = dup; a.guidance = guidance; a.eps = eps_out;
  h->profiling = true;
  cudaError_t e0 = cudaEventRecord(h->prof_ev[30], st);
  int rc = forward_one(h, a, st, nullptr);
  cudaError_t e1 = cudaEventRecord(h->prof_ev[31], st);
  h->profiling = false;
  TCS_CHECK(rc);
  TCS_CUDA(e0);
  TCS_CUDA(e1);
  TCS_CUDA(cudaStreamSynchronize(st));
  for (int id = 0; id < C_COUNT; ++id) TCS_CUDA(cudaEventElapsedTime(conv_ms + id, h->prof_ev[2 * id], h->prof_ev[2 * id + 1]));
  TCS_CUDA(cudaEventElapsedTime(total_ms, h->prof_ev[30], h->prof_ev[31]));
  return leave(h, user);
}

int64_t tcs_debug_layer(tcs_handle* h, const char* name, const float* x, const float* t, const int64_t* y_cat,
                        const float* y_cont, int32_t n, int32_t uncond, float* out, int64_t cap, void* stream) {
  TCS_CHECK(check_ready(h, "tcs_debug_layer"));
  if (!name || !x || !t || !y_cat || !y_cont || !out || n < 1) return fail(TCS_ERR_BAD_ARGUMENT, "tcs_debug_layer: bad argument");
  const int dup = uncond ? 2 : 1;   // uncond=1 runs the doubled batch; rows alternate cond/uncond
  if (n * dup > h->chunk) return fail(TCS_ERR_BAD_ARGUMENT, "tcs_debug_layer: n exceeds the chunk size");
  TapRequest tap;
  for (int i = 0; i < kNumTaps; ++i)
    if (!strcmp(name, kTapNames[i])) tap.id = i;
  if (tap.id < 0) return fail(TCS_ERR_BAD_ARGUMENT, std::string("tcs_debug_layer: unknown layer ") + name);
  tap.out = out; tap.capacity = cap;
  cudaStream_t user = static_cast<cudaStream_t>(stream);
  TCS_CHECK(enter(h, user));
  TCS_CHECK(h->cvec.ensure(static_cast<size_t>(n) * dup * 96 * 4));
  TCS_CHECK(h->tvec.ensure(static_cast<size_t>(n) * 96 * 4));
  TCS_CHECK(h->eps.ensure(static_cast<size_t>(n) * 4096 * 4));
  cudaStream_t st = h->stream;
  TCS_CHECK(launch_cond_embed(h->ew, y_cat, y_cont, n, dup, h->cvec.as<float>(), st));
  TCS_CHECK(launch_time_embed(h->ew, t, n, h->tvec.as<float>(), st));
  PassArgs a;
  a.x = x; a.cvec = h->cvec.as<float>(); a.tvec = h->tvec.as<float>(); a.tvec_stride = 1; a.step_ptr = nullptr;
  a.trow_off = 0; a.ns = n; a.dup = dup; a.guidance = dup == 2 ? 1.5f : 0.f; a.eps = h->eps.as<float>();
  TCS_CHECK(forward_one(h, a, st, &tap));
  TCS_CHECK(leave(h, user));
  return tap.written;
}

int tcs_condition_grid(tcs_handle* h, int32_t n, int64_t offset, int64_t n_total, float theta_max, int64_t* y_cat,
                       float* y_cont, void* stream) {
  if (!h || n < 0 || !y_cat || !y_cont) return fail(TCS_ERR_BAD_ARGUMENT, "tcs_condition_grid: bad argument");
  if (n == 0) return TCS_OK;
  TCS_CUDA(cudaSetDevice(h->cfg.device));
  cond_grid_kernel<<<(n + 127) / 128, 128, 0, static_cast<cudaStream_t>(stream)>>>(
      n, offset, n_total, theta_max, h->cfg.n_types, h->cfg.y_cont_dim, reinterpret_cast<long long*>(y_cat), y_cont);
  TCS_CUDA(cudaGetLastError());
  ++h->launches;
  return TCS_OK;
}

int tcs_sde_update(tcs_handle* h, float* x, const float* eps, const float* noise, int32_t n, float t, float t_next,
                   uint64_t seed, uint64_t gidx0, int32_t step, void* stream) {
  if (!h || !x || !eps || n < 0) return fail(TCS_ERR_BAD_ARGUMENT, "tcs_sde_update: bad argument");
  if (n == 0) return TCS_OK;
  TCS_CUDA(cudaSetDevice(h->cfg.device));
  cudaStream_t user = static_cast<cudaStream_t>(stream);
  TCS_CHECK(enter(h, user));
  const Sched s{h->cfg.beta_min, h->cfg.beta_max};
  TCS_CHECK(h->coef.ensure(sizeof(StepCoef) * 8));
  TCS_CHECK(ensure_pinned(h, sizeof(StepCoef) * 8 + 64));
  StepCoef* c = static_cast<StepCoef*>(h->pinned);
  memset(c, 0, sizeof(StepCoef) * 2);
  c[0].t = t; c[0].beta = s.beta(t); c[0].sigma = s.sigma(t); c[0].alpha = s.alpha(t);
  c[0].dt = t_next - t; c[0].g_sqrt_dt = sqrtf(c[0].beta) * sqrtf(fabsf(c[0].dt));
  int* hs = reinterpret_cast<int*>(c + 2);
  *hs = step;
  TCS_CUDA(cudaMemcpyAsync(h->coef.p, c, sizeof(StepCoef) * 2, cudaMemcpyHostToDevice, h->stream));
  TCS_CUDA(cudaMemcpyAsync(h->step_ctr.p, hs, 4, cudaMemcpyHostToDevice, h->stream));
  TCS_CUDA(cudaEventRecord(h->ev_pinned, h->stream));
  StepArgs a{};
  a.coef = h->coef.as<StepCoef>();
  a.step_ptr = h->step_ctr.as<int>();
  a.row_off = -step;   // row 0 regardless of the step word used for the Philox stream
  a.mode = STEP_SDE; a.x = x; a.eps = eps;
  a.noise = noise; a.noise_step_stride = 0;   // injected noise is for this step only (stride 0)
  a.seed = seed; a.gidx0 = gidx0; a.n = n;
  ++h->launches;
  TCS_CHECK(launch_step(a, h->stream));
  return leave(h, user);
}

int tcs_ode_update(tcs_handle* h, int32_t mode, float* x, float* x_pred, float* d0, const float* eps, int32_t n, float t,
                   float t_next, void* stream) {
  if (!h || !x || !x_pred || !d0 || !eps || n < 0 || mode < STEP_ODE_PREDICT || mode > STEP_FINAL)
    return fail(TCS_ERR_BAD_ARGUMENT, "tcs_ode_update: bad argument");
  if (n == 0) return TCS_OK;
  TCS_CUDA(cudaSetDevice(h->cfg.device));
  cudaStream_t user = static_cast<cudaStream_t>(stream);
  TCS_CHECK(enter(h, user));
  const Sched s{h->cfg.beta_min, h->cfg.beta_max};
  TCS_CHECK(h->coef.ensure(sizeof(StepCoef) * 8));
  TCS_CHECK(ensure_pinned(h, sizeof(StepCoef) * 8 + 64));
  StepCoef* c = static_cast<StepCoef*>(h->pinned);
  memset(c, 0, sizeof(StepCoef) * 2);
  const float tt[2] = {t, t_next};
  for (int i = 0; i < 2; ++i) {   // row 0: schedule at t and dt of the step; row 1: schedule at t_next (the corrector's)
    c[i].t = tt[i]; c[i].beta = s.beta(tt[i]); c[i].sigma = s.sigma(tt[i]); c[i].alpha = s.alpha(tt[i]);
    c[i].dt = i == 0 ? t_next - t : 0.f;
    c[i].g_sqrt_dt = sqrtf(c[i].beta) * sqrtf(fabsf(c[i].dt));
  }
  TCS_CUDA(cudaMemcpyAsync(h->coef.p, c, sizeof(StepCoef) * 2, cudaMemcpyHostToDevice, h->stream));
  TCS_CUDA(cudaEventRecord(h->ev_pinned, h->stream));
  StepArgs a{};
  a.coef = h->coef.as<StepCoef>();
  a.step_ptr = nullptr;
  a.row_off = mode == STEP_ODE_CORRECT ? 1 : 0;
  a.mode = mode; a.x = x; a.x_pred = x_pred; a.d0 = d0; a.eps = eps; a.n = n;
  if (mode == STEP_FINAL) { a.out_img = x_pred; a.out_x0 = d0; }
  ++h->launches;
  TCS_CHECK(launch_step(a, h->stream));
  return leave(h, user);
}

int tcs_dpm_update(tcs_handle* h, float* x, float* x0_prev, const float* eps, int32_t n, float alpha, float sigma, float a,
                   float m, float c0, float c1, void* stream) {
  if (!h || !x || !x0_prev || !eps || n < 0) return fail(TCS_ERR_BAD_ARGUMENT, "tcs_dpm_update: bad argument");
  if (n == 0) return TCS_OK;
  TCS_CUDA(cudaSetDevice(h->cfg.device));
  cudaStream_t user = static_cast<cudaStream_t>(stream);
  TCS_CHECK(enter(h, user));
  TCS_CHECK(h->coef.ensure(sizeof(StepCoef) * 8));
  TCS_CHECK(h->dpm_coef.ensure(sizeof(DpmCoef) * 8));
  TCS_CHECK(ensure_pinned(h, sizeof(StepCoef) * 8 + 64));
  StepCoef* c = static_cast<StepCoef*>(h->pinned);
  memset(c, 0, sizeof(StepCoef));
  c->alpha = alpha; c->sigma = sigma;
  DpmCoef* k = reinterpret_cast<DpmCoef*>(c + 1);
  *k = DpmCoef{a, m, c0, c1};
  TCS_CUDA(cudaMemcpyAsync(h->coef.p, c, sizeof(StepCoef), cudaMemcpyHostToDevice, h->stream));
  TCS_CUDA(cudaMemcpyAsync(h->dpm_coef.p, k, sizeof(DpmCoef), cudaMemcpyHostToDevice, h->stream));
  TCS_CUDA(cudaEventRecord(h->ev_pinned, h->stream));
  StepArgs s{};
  s.coef = h->coef.as<StepCoef>(); s.dpm = h->dpm_coef.as<DpmCoef>();
  s.step_ptr = nullptr; s.row_off = 0;
  s.mode = STEP_DPM2M; s.x = x; s.d0 = x0_prev; s.eps = eps; s.n = n;
  ++h->launches;
  TCS_CHECK(launch_step(s, h->stream));
  return leave(h, user);
}

int tcs_sample(tcs_handle* h, const tcs_sample_args* args, void* stream) {
  TCS_CHECK(check_ready(h, "tcs_sample"));
  if (!args) return fail(TCS_ERR_BAD_ARGUMENT, "tcs_sample: null args");
  const tcs_sample_args& A = *args;
  if (!(A.t_end > 0.0 && A.t_end < 1.0))
    return fail(TCS_ERR_BAD_ARGUMENT, "t_end must be in (0,1), got " + std::to_string(A.t_end));
  if (A.sampler != TCS_SAMPLER_ODE && A.sampler != TCS_SAMPLER_SDE && A.sampler != TCS_SAMPLER_DPMPP_2M)
    return fail(TCS_ERR_BAD_ARGUMENT, "Unknown sampler. Use 'ode', 'sde' or 'dpm++2m'.");
  if (A.sampler == TCS_SAMPLER_DPMPP_2M && A.noise)
    return fail(TCS_ERR_BAD_ARGUMENT, "tcs_sample: the dpm++2m sampler is deterministic; noise must be NULL");
  if (A.n < 0 || A.steps < 0) return fail(TCS_ERR_BAD_ARGUMENT, "tcs_sample: n and steps must be >= 0");
  if (A.n == 0) return TCS_OK;
  if (!A.y_cat || !A.y_cont || !A.x_out) return fail(TCS_ERR_BAD_ARGUMENT, "tcs_sample: y_cat, y_cont and x_out are required");
  const int n = A.n, steps = A.steps;
  const int dup = A.guidance > 0.f ? 2 : 1;
  const bool ode = A.sampler == TCS_SAMPLER_ODE;
  const bool dpm = A.sampler == TCS_SAMPLER_DPMPP_2M;
  const Sched sc = A.beta_max > 0.0 ? Sched{A.beta_min, A.beta_max} : Sched{h->cfg.beta_min, h->cfg.beta_max};
  if (dpm && !(sc.bmin > 0.0 && sc.bmax >= sc.bmin))
    return fail(TCS_ERR_BAD_ARGUMENT, "tcs_sample: the dpm++2m sampler needs 0 < beta_min <= beta_max");
  cudaStream_t user = static_cast<cudaStream_t>(stream);
  TCS_CHECK(enter(h, user));
  cudaStream_t st = h->stream;
  const size_t img = static_cast<size_t>(n) * 4096 * 4;
  TCS_CHECK(h->x.ensure(img)); TCS_CHECK(h->eps.ensure(img));
  if (ode) { TCS_CHECK(h->xpred.ensure(img)); TCS_CHECK(h->d0.ensure(img)); }
  if (dpm) { TCS_CHECK(h->d0.ensure(img)); TCS_CHECK(h->dpm_coef.ensure(sizeof(DpmCoef) * (steps + 1))); }   // d0 = x0_prev
  TCS_CHECK(h->cvec.ensure(static_cast<size_t>(n) * dup * 96 * 4));
  TCS_CHECK(h->tvec.ensure(static_cast<size_t>(steps + 1) * 96 * 4));
  TCS_CHECK(h->tvals.ensure(static_cast<size_t>(steps + 1) * 4));
  TCS_CHECK(h->coef.ensure(sizeof(StepCoef) * (steps + 2)));

  // ---- tables: time grid, schedule coefficients, embeddings --------------------------------------
  const size_t pin_bytes = sizeof(StepCoef) * (steps + 2) + (dpm ? sizeof(DpmCoef) * (steps + 1) : 0) + 4 * (steps + 1) + 64;
  TCS_CHECK(ensure_pinned(h, pin_bytes));
  StepCoef* hc = static_cast<StepCoef*>(h->pinned);
  DpmCoef* hk = reinterpret_cast<DpmCoef*>(hc + steps + 2);
  float* hts = dpm ? reinterpret_cast<float*>(hk + steps + 1) : reinterpret_cast<float*>(hc + steps + 2);
  if (dpm) {
    if (steps >= 1) dpm_schedule_host(steps, A.t_end, sc.bmin, sc.bmax, hts, hk);
    else hts[0] = 1.0f;   // no step: the projection of x_T at t = 1, as for the other samplers
  } else if (steps >= 1) {
    time_grid_host(steps, A.t_end, hts);
  } else {
    hts[0] = static_cast<float>(A.t_end) + static_cast<float>(1.0 - A.t_end);  // linspace(0,1,1) = [0]
  }
  for (int i = 0; i <= steps; ++i) {
    StepCoef c{};
    c.t = hts[i]; c.beta = sc.beta(c.t); c.sigma = sc.sigma(c.t); c.alpha = sc.alpha(c.t);
    c.dt = i < steps ? hts[i + 1] - hts[i] : 0.f;
    c.g_sqrt_dt = sqrtf(c.beta) * sqrtf(fabsf(c.dt));
    hc[i] = c;
  }
  TCS_CUDA(cudaMemcpyAsync(h->coef.p, hc, sizeof(StepCoef) * (steps + 1), cudaMemcpyHostToDevice, st));
  if (dpm && steps >= 1) TCS_CUDA(cudaMemcpyAsync(h->dpm_coef.p, hk, sizeof(DpmCoef) * steps, cudaMemcpyHostToDevice, st));
  TCS_CUDA(cudaMemcpyAsync(h->tvals.p, hts, 4 * (steps + 1), cudaMemcpyHostToDevice, st));
  TCS_CUDA(cudaEventRecord(h->ev_pinned, st));
  TCS_CUDA(cudaMemsetAsync(h->step_ctr.p, 0, 4, st));
  h->launches += 2;
  TCS_CHECK(launch_cond_embed(h->ew, A.y_cat, A.y_cont, n, dup, h->cvec.as<float>(), st));
  TCS_CHECK(launch_time_embed(h->ew, h->tvals.as<float>(), steps + 1, h->tvec.as<float>(), st));
  // ---- initial state -------------------------------------------------------------------------------
  float* x = h->x.as<float>();
  ++h->launches;
  if (A.x_init) TCS_CHECK(launch_copy_f32(x, A.x_init, static_cast<size_t>(n) * 4096, st));
  else TCS_CHECK(launch_philox_normal(x, n, A.seed, A.global_index_offset, st));

  const int* sp = h->step_ctr.as<int>();
  float* eps = h->eps.as<float>();
  const float* cvec = h->cvec.as<float>();
  const float* tvec = h->tvec.as<float>();
  const int epe = ode ? 2 : 1;  // network evaluations per step

  auto step_args = [&](int mode, int row_off) {
    StepArgs a{};
    a.coef = h->coef.as<StepCoef>(); a.dpm = h->dpm_coef.as<DpmCoef>(); a.step_ptr = sp; a.row_off = row_off; a.mode = mode;
    a.x = x; a.x_pred = h->xpred.as<float>(); a.d0 = h->d0.as<float>(); a.eps = eps;
    a.noise = A.noise; a.noise_step_stride = static_cast<long long>(n) * 4096;
    a.seed = A.seed; a.gidx0 = A.global_index_offset; a.n = n;
    return a;
  };
  auto enqueue_step = [&]() -> int {
    if (!ode) {   // SDE and DPM-Solver++(2M): one evaluation per step
      TCS_CHECK(trace_copy(h, A.trace_x, x, sp, 1, 0, n, st));
      TCS_CHECK(forward_all(h, x, cvec, tvec, 0, sp, 0, n, dup, A.guidance, eps, st));
      TCS_CHECK(trace_copy(h, A.trace_eps, eps, sp, 1, 0, n, st));
      ++h->launches;
      TCS_CHECK(launch_step(step_args(dpm ? STEP_DPM2M : STEP_SDE, 0), st));
    } else {
      TCS_CHECK(trace_copy(h, A.trace_x, x, sp, 2, 0, n, st));
      TCS_CHECK(forward_all(h, x, cvec, tvec, 0, sp, 0, n, dup, A.guidance, eps, st));
      TCS_CHECK(trace_copy(h, A.trace_eps, eps, sp, 2, 0, n, st));
      ++h->launches;
      TCS_CHECK(launch_step(step_args(STEP_ODE_PREDICT, 0), st));
      TCS_CHECK(trace_copy(h, A.trace_x, h->xpred.as<float>(), sp, 2, 1, n, st));
      TCS_CHECK(forward_all(h, h->xpred.as<float>(), cvec, tvec, 0, sp, 1, n, dup, A.guidance, eps, st));
      TCS_CHECK(trace_copy(h, A.trace_eps, eps, sp, 2, 1, n, st));
      ++h->launches;
      TCS_CHECK(launch_step(step_args(STEP_ODE_CORRECT, 1), st));
    }
    ++h->launches;
    TCS_CHECK(launch_advance(h->step_ctr.as<int>(), 1, st));
    return TCS_OK;
  };

  if (steps > 0) {
    if (h->cfg.use_graph) {
      tcs_handle::GKey k;
      k.n = n; k.dup = dup; k.sampler = A.sampler; k.noise = A.noise; k.teps = A.trace_eps; k.tx = A.trace_x;
      k.guidance = A.guidance; k.seed = A.seed; k.gidx = A.global_index_offset; k.gen = h->ws_gen;
      const bool same = h->gexec && h->gkey.n == k.n && h->gkey.dup == k.dup && h->gkey.sampler == k.sampler &&
                        h->gkey.noise == k.noise && h->gkey.teps == k.teps && h->gkey.tx == k.tx &&
                        h->gkey.guidance == k.guidance && h->gkey.seed == k.seed && h->gkey.gidx == k.gidx &&
                        h->gkey.gen == k.gen;
      if (!same) {
        if (h->gexec) { cudaGraphExecDestroy(h->gexec); h->gexec = nullptr; }
        const int64_t before = h->launches;
        TCS_CUDA(cudaStreamBeginCapture(st, cudaStreamCaptureModeRelaxed));
        const int rc = enqueue_step();
        cudaGraph_t graph = nullptr;
        const cudaError_t ce = cudaStreamEndCapture(st, &graph);
        if (rc != TCS_OK) { if (graph) cudaGraphDestroy(graph); return rc; }
        if (ce != cudaSuccess) return fail(TCS_ERR_CUDA, std::string("cudaStreamEndCapture: ") + cudaGetErrorString(ce));
        h->graph_kernels = h->launches - before;
        h->launches = before;
        const cudaError_t ie = cudaGraphInstantiate(&h->gexec, graph, 0);
        cudaGraphDestroy(graph);
        if (ie != cudaSuccess) { h->gexec = nullptr; return fail(TCS_ERR_CUDA, std::string("cudaGraphInstantiate: ") + cudaGetErrorString(ie)); }
        h->gkey = k;
      }
      for (int i = 0; i < steps; ++i) TCS_CUDA(cudaGraphLaunch(h->gexec, st));
      h->launches += h->graph_kernels * steps;
    } else {
      for (int i = 0; i < steps; ++i) TCS_CHECK(enqueue_step());
    }
  }
  // ---- final projection from x_{t_end} ----------------------------------------------------------------
  TCS_CHECK(trace_copy(h, A.trace_x, x, sp, epe, 0, n, st));
  TCS_CHECK(forward_all(h, x, cvec, tvec, 0, sp, 0, n, dup, A.guidance, eps, st));
  TCS_CHECK(trace_copy(h, A.trace_eps, eps, sp, epe, 0, n, st));
  StepArgs fa = step_args(STEP_FINAL, 0);
  fa.out_img = A.x_out; fa.out_x0 = A.x0_hat;
  ++h->launches;
  TCS_CHECK(launch_step(fa, st));
  return leave(h, user);
}


}  // extern "C"

template <typename T>
static int debug_conv_t(bool use_tc, const ConvGeom& g, const float* in0, const float* in1, const float* weight,
                        const float* bias, float* out, float* stats, int epi, cudaStream_t st) {
  const int B = g.B, Hin = g.ups ? g.H / 2 : g.H * g.stride, Win = g.ups ? g.W / 2 : g.W * g.stride;   // ups: half-resolution source
  const int pad = g.in_pad[0];
  DevBuf s0, s1, wp, db, dout, part;
  const size_t in_elems0 = static_cast<size_t>(B) * (Hin + 2 * pad) * (Win + 2 * pad) * g.csrc[0];
  TCS_CHECK(s0.ensure(in_elems0 * sizeof(T)));
  TCS_CHECK(launch_pad_from_plain<T>(in0, B, Hin, Win, g.csrc[0], pad, s0.as<T>(), st));
  if (g.nsrc == 2) {
    const size_t in_elems1 = static_cast<size_t>(B) * (Hin + 2 * pad) * (Win + 2 * pad) * g.csrc[1];
    TCS_CHECK(s1.ensure(in_elems1 * sizeof(T)));
    TCS_CHECK(launch_pad_from_plain<T>(in1, B, Hin, Win, g.csrc[1], pad, s1.as<T>(), st));
  }
  int cin = 0;
  for (int s = 0; s < g.nsrc; ++s) cin += g.csrc[s];
  const size_t wcount = static_cast<size_t>(g.ntot) * cin * g.ksize * g.ksize;
  std::vector<float> hw(wcount), hb(g.ntot);
  TCS_CUDA(cudaMemcpy(hw.data(), weight, wcount * 4, cudaMemcpyDefault));
  TCS_CUDA(cudaMemcpy(hb.data(), bias, g.ntot * 4, cudaMemcpyDefault));
  TCS_CHECK(db.ensure(g.ntot * 4));
  TCS_CUDA(cudaMemcpy(db.p, hb.data(), g.ntot * 4, cudaMemcpyHostToDevice));
  const size_t out_px = static_cast<size_t>(B) * g.H * g.W;
  const int slots = use_tc ? tc_slots(g.H, g.W) : simt_slots(g.H, g.W);
  EpiArgs ea{};
  ea.bias = db.as<float>(); ea.ldo = g.ntot; ea.slots = slots; ea.residual = nullptr;
  TCS_CHECK(part.ensure(static_cast<size_t>(B) * slots * 16 * 4));
  ea.partials = part.as<float>();
  if (epi == EPI_RAW_STATS) { ea.out = out; }
  else if (epi == EPI_PADDED) {
    TCS_CHECK(dout.ensure(static_cast<size_t>(B) * (g.H + 2) * (g.W + 2) * g.ntot * sizeof(T)));
    TCS_CUDA(cudaMemsetAsync(dout.p, 0xff, dout.bytes, st));
    ea.out = dout.p;
  } else {
    TCS_CHECK(dout.ensure(out_px * g.ntot * sizeof(T)));
    ea.out = dout.p;
  }
  if (use_tc) {
    std::vector<__nv_bfloat16> pk(conv_tc_packed_elems(g));
    conv_tc_pack_weights(g, epi, hw.data(), pk.data());
    TCS_CHECK(wp.ensure(pk.size() * 2));
    TCS_CUDA(cudaMemcpy(wp.p, pk.data(), pk.size() * 2, cudaMemcpyHostToDevice));
    ConvTcPlan pl;
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    TCS_CHECK(conv_tc_make_plan(&pl, g, s0.p, g.nsrc == 2 ? s1.p : s0.p, wp.as<__nv_bfloat16>(), epi, ea, sms));
    TCS_CHECK(conv_tc_launch(pl, st));
  } else {
    std::vector<float> pk(wcount);
    conv_simt_pack_weights(g, hw.data(), pk.data(), sizeof(T) == 2);
    TCS_CHECK(wp.ensure(wcount * 4));
    TCS_CUDA(cudaMemcpy(wp.p, pk.data(), wcount * 4, cudaMemcpyHostToDevice));
    TCS_CHECK(launch_conv_simt<T>(g, s0.as<T>(), s1.as<T>(), wp.as<float>(), epi, ea, st));
  }
  if (epi == EPI_PADDED) {
    // interior -> out; additionally verify the halo by re-deriving a padded copy and comparing on the host
    TCS_CHECK(launch_unpad_to_f32<T>(dout.as<T>(), B, g.H, g.W, g.ntot, 1, out, st));
    DevBuf ref;
    TCS_CHECK(ref.ensure(dout.bytes));
    TCS_CHECK(launch_pad_from_plain<T>(out, B, g.H, g.W, g.ntot, 1, ref.as<T>(), st));
    TCS_CUDA(cudaStreamSynchronize(st));
    std::vector<uint8_t> a(dout.bytes), b(dout.bytes);
    TCS_CUDA(cudaMemcpy(a.data(), dout.p, dout.bytes, cudaMemcpyDeviceToHost));
    TCS_CUDA(cudaMemcpy(b.data(), ref.p, dout.bytes, cudaMemcpyDeviceToHost));
    if (memcmp(a.data(), b.data(), dout.bytes) != 0)
      return fail(TCS_ERR_STATE, "tcs_debug_conv: circular halo of the padded output is wrong");
  } else if (epi == EPI_PLAIN) {
    TCS_CHECK(launch_unpad_to_f32<T>(dout.as<T>(), B, g.H, g.W, g.ntot, 0, out, st));
  }
  TCS_CUDA(cudaStreamSynchronize(st));
  if (stats && epi == EPI_RAW_STATS) {
    std::vector<float> hp(static_cast<size_t>(B) * slots * 16);
    TCS_CUDA(cudaMemcpy(hp.data(), part.p, hp.size() * 4, cudaMemcpyDeviceToHost));
    std::vector<float> hs(static_cast<size_t>(B) * 16);
    for (int b = 0; b < B; ++b)
      for (int k = 0; k < 16; ++k) {
        double acc = 0;
        for (int s = 0; s < slots; ++s) acc += hp[(static_cast<size_t>(b) * slots + s) * 16 + k];
        hs[b * 16 + k] = static_cast<float>(acc);
      }
    TCS_CUDA(cudaMemcpy(stats, hs.data(), hs.size() * 4, cudaMemcpyDefault));
  }
  return TCS_OK;
}

// one convolution in bf16x3 mode: fp32 inputs -> padded fp32 -> split (hi, lo) -> tcgen05 (K tripled) -> raw fp32 + stats
static int debug_conv_split3(const ConvGeom& g0, const float* in0, const float* in1, const float* weight, const float* bias,
                             float* out, float* stats, int epi, cudaStream_t st) {
  ConvGeom g = g0;
  g.split3 = 1;
  const int B = g.B, Hin = g.H * g.stride, Win = g.W * g.stride, pad = g.in_pad[0];
  DevBuf f32[2], sp[2], wp, db, part;
  const float* ins[2] = {in0, in1};
  size_t elems[2] = {0, 0};
  for (int s = 0; s < g.nsrc; ++s) {
    elems[s] = static_cast<size_t>(B) * (Hin + 2 * pad) * (Win + 2 * pad) * g.csrc[s];
    TCS_CHECK(f32[s].ensure(elems[s] * 4));
    TCS_CHECK(sp[s].ensure(elems[s] * 4));
    TCS_CHECK(launch_pad_from_plain<float>(ins[s], B, Hin, Win, g.csrc[s], pad, f32[s].as<float>(), st));
    TCS_CHECK(launch_split(f32[s].as<float>(), elems[s], sp[s].as<__nv_bfloat16>(), elems[s], st));
  }
  int cin = 0;
  for (int s = 0; s < g.nsrc; ++s) cin += g.csrc[s];
  const size_t wcount = static_cast<size_t>(g.ntot) * cin * g.ksize * g.ksize;
  std::vector<float> hw(wcount), hb(g.ntot);
  TCS_CUDA(cudaMemcpy(hw.data(), weight, wcount * 4, cudaMemcpyDefault));
  TCS_CUDA(cudaMemcpy(hb.data(), bias, g.ntot * 4, cudaMemcpyDefault));
  TCS_CHECK(db.ensure(g.ntot * 4));
  TCS_CUDA(cudaMemcpy(db.p, hb.data(), g.ntot * 4, cudaMemcpyHostToDevice));
  std::vector<__nv_bfloat16> pk(conv_tc_packed_elems(g));
  conv_tc_pack_weights(g, EPI_RAW_STATS, hw.data(), pk.data());
  TCS_CHECK(wp.ensure(pk.size() * 2));
  TCS_CUDA(cudaMemcpy(wp.p, pk.data(), pk.size() * 2, cudaMemcpyHostToDevice));
  const int slots = tc_slots(g.H, g.W);
  TCS_CHECK(part.ensure(static_cast<size_t>(B) * slots * 16 * 4));
  EpiArgs ea{};
  ea.bias = db.as<float>(); ea.ldo = g.ntot; ea.slots = slots; ea.out = out; ea.partials = part.as<float>();
  ConvTcPlan pl;
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  TCS_CHECK(conv_tc_make_plan(&pl, g, sp[0].p, g.nsrc == 2 ? sp[1].p : nullptr, wp.as<__nv_bfloat16>(), EPI_RAW_STATS, ea, sms,
                              sp[0].as<__nv_bfloat16>() + elems[0], g.nsrc == 2 ? sp[1].as<__nv_bfloat16>() + elems[1] : nullptr));
  TCS_CHECK(conv_tc_launch(pl, st));
  TCS_CUDA(cudaStreamSynchronize(st));
  if (stats && epi == EPI_RAW_STATS) {
    std::vector<float> hp(static_cast<size_t>(B) * slots * 16);
    TCS_CUDA(cudaMemcpy(hp.data(), part.p, hp.size() * 4, cudaMemcpyDeviceToHost));
    std::vector<float> hs(static_cast<size_t>(B) * 16);
    for (int b = 0; b < B; ++b)
      for (int k = 0; k < 16; ++k) {
        double acc = 0;
        for (int s = 0; s < slots; ++s) acc += hp[(static_cast<size_t>(b) * slots + s) * 16 + k];
        hs[b * 16 + k] = static_cast<float>(acc);
      }
    TCS_CUDA(cudaMemcpy(stats, hs.data(), hs.size() * 4, cudaMemcpyDefault));
  }
  return TCS_OK;
}

extern "C" {

int tcs_debug_conv(int32_t engine, int32_t precision, int32_t B, int32_t H_out, int32_t W_out, int32_t cin0,
                   int32_t cin1, int32_t cout, int32_t ksize, int32_t stride, const float* in0, const float* in1,
                   const float* weight, const float* bias, float* out, float* stats, int32_t epi, void* stream) {
  if (!in0 || !weight || !bias || !out || B < 1) return fail(TCS_ERR_BAD_ARGUMENT, "tcs_debug_conv: bad argument");
  if (epi < 0 || epi > 2) return fail(TCS_ERR_BAD_ARGUMENT, "tcs_debug_conv: bad epilogue");
  if (H_out != W_out) return fail(TCS_ERR_UNSUPPORTED, "tcs_debug_conv: square outputs only");
  const bool bf16 = precision == TCS_BF16;
  const int eng = engine == TCS_ENGINE_AUTO ? (bf16 ? TCS_ENGINE_TCGEN05 : TCS_ENGINE_SIMT) : engine;
  ConvGeom g;
  g.B = B; g.H = H_out; g.W = W_out; g.ksize = ksize; g.stride = stride;
  g.nsrc = cin1 > 0 ? 2 : 1;
  g.csrc[0] = cin0; g.csrc[1] = cin1 > 0 ? cin1 : cin0;
  g.in_pad[0] = g.in_pad[1] = ksize == 1 ? 0 : 1;
  g.ntot = cout;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  // fp32 on the tcgen05 engine = bf16x3 mode: always the raw fp32 epilogue (its padded / plain forms are separate kernels)
  if (eng == TCS_ENGINE_TCGEN05 && !bf16) return debug_conv_split3(g, in0, in1, weight, bias, out, stats, epi, st);
  if (bf16) return debug_conv_t<__nv_bfloat16>(eng == TCS_ENGINE_TCGEN05, g, in0, in1, weight, bias, out, stats, epi, st);
  return debug_conv_t<float>(false, g, in0, in1, weight, bias, out, stats, epi, st);
}

// 3x3 conv of the bilinear x2 upsample of a half-resolution input, upsample fused into the conv (ConvGeom::ups)
int tcs_debug_conv_ups(int32_t B, int32_t H_out, int32_t W_out, int32_t cin, int32_t cout, const float* in_lowres,
                       const float* weight, const float* bias, float* out, void* stream) {
  if (!in_lowres || !weight || !bias || !out || B < 1) return fail(TCS_ERR_BAD_ARGUMENT, "tcs_debug_conv_ups: bad argument");
  if (H_out != W_out) return fail(TCS_ERR_UNSUPPORTED, "tcs_debug_conv_ups: square outputs only");
  ConvGeom g;
  g.B = B; g.H = H_out; g.W = W_out; g.ksize = 3; g.stride = 1;
  g.nsrc = 1; g.csrc[0] = g.csrc[1] = cin; g.in_pad[0] = g.in_pad[1] = 1; g.ntot = cout;
  g.ups = 1;
  return debug_conv_t<__nv_bfloat16>(true, g, in_lowres, nullptr, weight, bias, out, nullptr, EPI_PADDED,
                                     static_cast<cudaStream_t>(stream));
}

// Host-only: the weight image attn_block_tc_kernel bulk-copies (no device needed; tests check the layout on the CPU).
int64_t tcs_debug_attn_pack(const float* qkv_w, const float* proj_w, uint8_t* out, int64_t capacity) {
  const int64_t need = static_cast<int64_t>(attn_tc_wpack_bytes());
  if (!out) return need;
  if (!qkv_w || !proj_w || capacity < need) return fail(TCS_ERR_BAD_ARGUMENT, "tcs_debug_attn_pack: bad argument");
  attn_tc_pack_weights(qkv_w, proj_w, out);
  return need;
}

// The fused attention block in isolation (halo of the padded output verified like tcs_debug_conv's).
int tcs_debug_attn_block(int32_t B, const float* x, const float* gn_w, const float* gn_b, const float* qkv_w,
                         const float* qkv_b, const float* proj_w, const float* proj_b, float* out, float* dbg,
                         void* stream) {
  if (!x || !gn_w || !gn_b || !qkv_w || !qkv_b || !proj_w || !proj_b || !out || B < 1)
    return fail(TCS_ERR_BAD_ARGUMENT, "tcs_debug_attn_block: bad argument");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  using T = __nv_bfloat16;
  DevBuf din, dout, wp, small;
  const size_t pbytes = static_cast<size_t>(B) * 18 * 18 * 192 * sizeof(T);
  TCS_CHECK(din.ensure(pbytes));
  TCS_CHECK(dout.ensure(pbytes));
  TCS_CUDA(cudaMemsetAsync(dout.p, 0xff, pbytes, st));
  TCS_CHECK(launch_pad_from_plain<T>(x, B, 16, 16, 192, 1, din.as<T>(), st));
  std::vector<float> hq(576 * 192), hp(192 * 192);
  TCS_CUDA(cudaMemcpy(hq.data(), qkv_w, hq.size() * 4, cudaMemcpyDefault));
  TCS_CUDA(cudaMemcpy(hp.data(), proj_w, hp.size() * 4, cudaMemcpyDefault));
  std::vector<uint8_t> pk(attn_tc_wpack_bytes());
  attn_tc_pack_weights(hq.data(), hp.data(), pk.data());
  TCS_CHECK(wp.ensure(pk.size()));
  TCS_CUDA(cudaMemcpy(wp.p, pk.data(), pk.size(), cudaMemcpyHostToDevice));
  TCS_CHECK(small.ensure((576 + 192 * 3) * 4));
  float* sp = small.as<float>();
  TCS_CUDA(cudaMemcpy(sp, qkv_b, 576 * 4, cudaMemcpyDefault));
  TCS_CUDA(cudaMemcpy(sp + 576, proj_b, 192 * 4, cudaMemcpyDefault));
  TCS_CUDA(cudaMemcpy(sp + 768, gn_w, 192 * 4, cudaMemcpyDefault));
  TCS_CUDA(cudaMemcpy(sp + 960, gn_b, 192 * 4, cudaMemcpyDefault));
  AttnTcParams ap{};
  ap.x = din.as<T>(); ap.out = dout.as<T>(); ap.wpack = wp.as<uint8_t>();
  ap.bias_qkv = sp; ap.bias_proj = sp + 576; ap.gamma = sp + 768; ap.beta = sp + 960;
  ap.B = B; ap.dbg = dbg;
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  TCS_CHECK(launch_attn_block_tc(ap, sms, st));
  TCS_CHECK(launch_unpad_to_f32<T>(dout.as<T>(), B, 16, 16, 192, 1, out, st));
  DevBuf ref;
  TCS_CHECK(ref.ensure(pbytes));
  TCS_CHECK(launch_pad_from_plain<T>(out, B, 16, 16, 192, 1, ref.as<T>(), st));
  TCS_CUDA(cudaStreamSynchronize(st));
  std::vector<uint8_t> a(pbytes), b(pbytes);
  TCS_CUDA(cudaMemcpy(a.data(), dout.p, pbytes, cudaMemcpyDeviceToHost));
  TCS_CUDA(cudaMemcpy(b.data(), ref.p, pbytes, cudaMemcpyDeviceToHost));
  if (memcmp(a.data(), b.data(), pbytes) != 0)
    return fail(TCS_ERR_STATE, "tcs_debug_attn_block: circular halo of the padded output is wrong");
  return TCS_OK;
}

}  // extern "C"
