// libamodal_b200.so -- host side of the B200 forward pass of Amodal-Depth-Anything behind the C ABI of
// include/amodal_b200.h: weight packing, workspace, kernel launch sequence. No torch types, no CPU fallback.
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <atomic>
#include <map>
#include <mutex>
#include <set>
#include <stdexcept>
#include <string>
#include <unordered_map>
#include <vector>

#include "../../include/amodal_b200.h"
#include "attention.cuh"
#include "attention2.cuh"
#include "elementwise.cuh"
#include "postproc.cuh"
#include "evalops.cuh"
#include "gemm.cuh"
#include "pack.cuh"
#include "tail_mma.cuh"
#include "tma_host.h"

namespace ada {

static thread_local std::string g_last_error;

struct AdaError : std::runtime_error {
  int code;
  AdaError(int c, const std::string& m) : std::runtime_error(m), code(c) {}
};
#define ADA_CHECK_CUDA(expr)                                                                         \
  do {                                                                                               \
    cudaError_t _e = (expr);                                                                         \
    if (_e != cudaSuccess)                                                                           \
      throw AdaError(ADA_ECUDA, std::string(#expr) + " -> " + cudaGetErrorString(_e));               \
  } while (0)
#define ADA_REQUIRE(cond, msg)                                \
  do {                                                        \
    if (!(cond)) throw AdaError(ADA_EINVAL, std::string(msg)); \
  } while (0)

static inline int round_up(int a, int b) { return (a + b - 1) / b * b; }
// ------------------------------------------------------------------------------------------------ device context
// Everything that CUDA keeps per device (SM count, the opt-in shared-memory size of each kernel) is keyed by the device
// ordinal that is current on the calling thread: one process may drive several GPUs, one handle each (SURVEY.md section 5,
// "one process, 8 streams"), and handles may be driven from different threads.
constexpr int kMaxDevices = 64;
struct DeviceInfo {
  int device = -1;
  int sms = 0;
  bool ok = false;
  std::string why;
};
static DeviceInfo& device_info() {
  static DeviceInfo table[kMaxDevices];
  static std::once_flag once[kMaxDevices];
  static DeviceInfo none;
  static std::once_flag none_once;
  int dev = -1;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess || dev < 0 || dev >= kMaxDevices) {
    cudaGetLastError();
    std::call_once(none_once, [&] { none.why = std::string("no CUDA device: ") + cudaGetErrorString(e); });
    return none;
  }
  std::call_once(once[dev], [&] {
    DeviceInfo& di = table[dev];
    cudaDeviceProp p;
    cudaError_t pe = cudaGetDeviceProperties(&p, dev);
    if (pe != cudaSuccess) {
      cudaGetLastError();
      di.why = std::string("no CUDA device: ") + cudaGetErrorString(pe);
      return;
    }
    if (p.major != 10) {
      di.why = "device is sm_" + std::to_string(p.major) + std::to_string(p.minor) + ", this library is sm_100a only";
      return;
    }
    di.device = dev;
    di.sms = p.multiProcessorCount;
    di.ok = true;
  });
  return table[dev];
}
static void require_device() {
  DeviceInfo& di = device_info();
  if (!di.ok) throw AdaError(ADA_ENODEVICE, di.why);
}
// cudaFuncAttributeMaxDynamicSharedMemorySize is a per-device attribute: `done` is a per-kernel bit mask of the device
// ordinals it has been set on (setting it twice from two racing threads is harmless).
template <typename K>
static void ensure_smem_attr(K kernel, int bytes, std::atomic<uint64_t>& done) {
  const int dev = device_info().device;
  if (dev < 0) throw AdaError(ADA_ENODEVICE, device_info().why);
  const uint64_t bit = 1ull << dev;
  if (done.load(std::memory_order_acquire) & bit) return;
  ADA_CHECK_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
  done.fetch_or(bit, std::memory_order_release);
}

static int env_int(const char* name, int dflt) {
  const char* v = getenv(name);
  return v ? atoi(v) : dflt;
}

// ------------------------------------------------------------------------------------------------ GEMM launcher
// Programmatic dependent launch: GEMM / LayerNorm / attention launches carry the programmatic-stream-serialization
// attribute (their kernels call griddepcontrol.wait after the prologue), so a kernel's prologue overlaps its predecessor's
// tail. Measured (ViT-L 518^2, ms per step off -> on): batch 1 3.74 -> 3.37, 2 4.63 -> 4.36, 4 7.37 -> 7.18, 8 13.13 -> 12.98,
// 16 25.10 -> 25.10, 32 +1 % (early CTAs of the next kernel compete with the draining one). ADA_PDL = 1 / 0 forces it
// on / off; default: on up to 12000 tokens (set per forward).
static thread_local bool g_pdl_now = false;  // per calling thread: handles may be driven from different threads
static bool pdl_enabled() { return g_pdl_now; }
static void pdl_select(long long tokens) {
  static const int v = env_int("ADA_PDL", -1);
  g_pdl_now = (v < 0) ? (tokens <= 12000) : (v != 0);
}
template <typename... KArgs, typename... Args>
static void launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args&&... args) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = pdl_enabled() ? 1 : 0;
  ADA_CHECK_CUDA(cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...));
}

template <int BN, int CG, int EPI>
static void launch_gemm_bn(const CUtensorMap& ta, const CUtensorMap& tb, const CUtensorMap& tc, const CUtensorMap& tc2,
                           const GemmArgs& g, int num_tiles, cudaStream_t st) {
  using Cfg = GemmCfg<BN, CG, EPI>;
  static std::atomic<uint64_t> attr_done{0};
  ensure_smem_attr(gemm_tcgen05_kernel<BN, CG, EPI>, Cfg::kSmemBytes, attr_done);
  const int units = std::min(num_tiles, device_info().sms / CG);  // persistent: one CTA (or CTA pair) per SM (pair)
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(static_cast<unsigned>(units * CG));
  cfg.blockDim = dim3(kGemmThreads);
  cfg.dynamicSmemBytes = Cfg::kSmemBytes;
  cfg.stream = st;
  cudaLaunchAttribute attr[2];
  int na = 0;
  if (CG > 1) {
    attr[na].id = cudaLaunchAttributeClusterDimension;
    attr[na].val.clusterDim.x = CG;
    attr[na].val.clusterDim.y = 1;
    attr[na].val.clusterDim.z = 1;
    ++na;
  }
  if (pdl_enabled()) {
    attr[na].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[na].val.programmaticStreamSerializationAllowed = 1;
    ++na;
  }
  cfg.attrs = attr;
  cfg.numAttrs = na;
  ADA_CHECK_CUDA(cudaLaunchKernelEx(&cfg, gemm_tcgen05_kernel<BN, CG, EPI>, ta, tb, tc, tc2, g));
}

static int pick_bn(int N) {
  // smallest padded N wins; ties go to the wider tile (fewer A re-reads, better smem operand bandwidth)
  int best = 64, best_pad = round_up(N, 64);  // 32 is reserved for the fused tail (EPI_TAIL)
  const int cands[2] = {128, 256};
  for (int c : cands) {
    const int pad = round_up(N, c);
    if (pad <= best_pad + best_pad / 16) {  // allow ~6% padding for a wider tile
      best = c;
      best_pad = pad;
    }
  }
  return best;
}

struct GemmLaunch {
  const void* A = nullptr;   // linear: [M, K] pitch lda. conv: NHWC [batch, H, W, Cin]
  const void* Bw = nullptr;  // [N, K] pitch ldb
  int M = 0, N = 0, K = 0, lda = 0, ldb = 0;
  int a_mode = A_LINEAR;
  int batch = 0, H = 0, W = 0, Cin = 0;  // conv: OUTPUT map size
  int conv_stride = 1, Hin = 0, Win = 0;  // conv: stride 1 or 2 and the input map size (0 = same as output)
  int conv_taps = 9;         // conv: 9 = 3x3, 1 = pointwise on pixel tiles (the k == s transposed convs, EPI_CONVT)
  GemmArgs args{};           // epilogue fields filled by caller
  __nv_bfloat16* out_relu = nullptr;  // EPI_BF16: optional relu(out) copy (second TMA store map)
  int force_bn = 0;
  int force_cg = 0;          // 0 = auto, 1 = single CTA tiles, 2 = CTA pairs (cta_group::2)
};


static thread_local int g_launches = 0;  // counted per forward (host side, single-threaded per handle)

// ---- optional per-launch CUDA-event profiler (bench.py's roofline / breakdown; off in the headline timing loop)
enum ProfClass : int { PC_GEMM_LINEAR = 0, PC_GEMM_CONV, PC_ATTENTION, PC_LAYERNORM, PC_CHANNEL_LN, PC_UPSAMPLE, PC_GATHER, PC_TAIL_GATHER, PC_COUNT };
struct ProfRec {
  int cls;
  double flops, bytes;
  cudaEvent_t a, b;
  int m, n, k, tag;  // shape + (epi | act << 4 | bn << 8) for GEMMs
};
struct Profiler {
  std::vector<ProfRec> recs;
};
static thread_local Profiler* g_prof = nullptr;
struct ProfScope {
  ProfRec* r = nullptr;
  cudaStream_t st;
  ProfScope(int cls, double flops, double bytes, cudaStream_t s) : st(s) {
    if (!g_prof) return;
    ProfRec rec{cls, flops, bytes, nullptr, nullptr, 0, 0, 0, 0};
    cudaEventCreate(&rec.a);
    cudaEventCreate(&rec.b);
    g_prof->recs.push_back(rec);
    r = &g_prof->recs.back();
    cudaEventRecord(r->a, st);
  }
  ~ProfScope() {
    if (r) cudaEventRecord(r->b, st);
  }
};

// Pixel-tile shape of an implicit-GEMM conv launch: 2^lw x 2^lh pixels of 2^lb images (128 A rows per CTA; a CTA pair puts two
// tiles side by side in x). Picks the shape with the fewest padded pixels over (batch, H, W); ties keep the 16 x 8 x 1 default,
// then prefer tiles that span fewer images and more of a row (DRAM locality of the TMA boxes). Every shape accumulates an
// output element over (tap, channel) in the same order, so the choice -- which depends on the batch -- never changes a bit.
struct TileGeo {
  int lw = 4, lh = 3, lb = 0;
  long long padded = 0;  // pixels computed, padding included
};
static TileGeo pick_tile_geo(int B, int H, int W, int cg, bool general) {
  auto cost = [&](int lw, int lh, int lb) {
    const long long tw = (1LL << lw) * cg, th = 1LL << lh, nb = 1LL << lb;
    return ((W + tw - 1) / tw * tw) * ((H + th - 1) / th * th) * ((B + nb - 1) / nb * nb);
  };
  TileGeo best;
  best.padded = cost(4, 3, 0);
  if (!general) return best;
  for (int lw = 5; lw >= 1; --lw)        // 2 .. 32 pixels wide: a warp's 32 accumulator rows are whole tile rows
    for (int lh = 7 - lw; lh >= 0; --lh) {
      const int lb = 7 - lw - lh;
      const long long c = cost(lw, lh, lb);
      if (c < best.padded) {  // strict: earlier candidates (wider, taller, fewer images) win ties
        best.lw = lw;
        best.lh = lh;
        best.lb = lb;
        best.padded = c;
      }
    }
  return best;
}

static void launch_gemm(const GemmLaunch& L, cudaStream_t st) {
  GemmArgs g = L.args;
  g.M = L.M;
  g.N = L.N;
  g.K = L.K;
  g.a_mode = L.a_mode;
  int bn = L.force_bn ? L.force_bn : pick_bn(g.epi == EPI_SWIGLU ? std::max(L.N, 64) : L.N);
  if (!L.force_bn && L.a_mode == A_LINEAR && L.K <= 256 && L.N > 64 && bn < 128) bn = 128;  // store-bound: fewer, wider tiles
  if (g.epi == EPI_TAIL) bn = 32;
  if (g.epi == EPI_BF16_CHLN) {
    ADA_REQUIRE(L.N <= 256 && L.N % 8 == 0 && g.gamma != nullptr && g.aux != nullptr && g.act == ACT_NONE &&
                    g.resid1 == nullptr && g.resid2 == nullptr && L.out_relu == nullptr,
                "EPI_BF16_CHLN: N <= 256, LayerNorm weight (gamma) and bias (aux), no activation / residuals");
    bn = 256;
  }
  if (g.epi == EPI_SWIGLU && bn < 128) bn = 128;
  ADA_REQUIRE(bn == 32 || bn == 64 || bn == 128 || bn == 256, "bad BN");
  ADA_REQUIRE(bn != 32 || g.epi == EPI_TAIL, "BN=32 is only built for the fused tail epilogue");
  ADA_REQUIRE(g.epi != EPI_SWIGLU || L.N % 128 == 0, "SwiGLU needs N % 128 == 0");
  ADA_REQUIRE(L.ldb % 8 == 0, "weight pitch must be a multiple of 8 elements");
  // general pixel-tile shapes: 3x3 convs whose epilogue stores through the 4-D output map (ADA_CONV_GEO=0: 16 x 8 x 1 only)
  static const int conv_geo_env = env_int("ADA_CONV_GEO", 1);
  const bool conv_geo_general = conv_geo_env != 0 && L.a_mode == A_CONV3X3 && L.conv_taps == 9 &&
                                (g.epi == EPI_BF16 || g.epi == EPI_F16 || g.epi == EPI_BF16_CHLN);
  // ---- CTA pairs (cta_group::2) when the problem is big enough to keep 74 pairs busy and pairing wastes little
  int cg = 1;
  {
    static const int cg_env = env_int("ADA_GEMM_CG", 0);
    const int want = L.force_cg ? L.force_cg : cg_env;
    const int tiles_n_ = (L.N + bn - 1) / bn;
    bool ok = (bn == 256 || (want == 2 && bn == 128 && g.epi == EPI_BF16)) && g.epi != EPI_TAIL;  // N=128 pairs are smem-read bound (A 4 KB + B 2 KB / 32 clk)
    if (ok && L.a_mode == A_CONV3X3) {
      const long long pad1 = pick_tile_geo(L.batch, L.H, L.W, 1, conv_geo_general).padded;
      const long long pad2 = pick_tile_geo(L.batch, L.H, L.W, 2, conv_geo_general).padded;
      const long long pairs = pad2 / (2 * kBlockM) * tiles_n_;
      if (want != 2) ok = (pad2 * 100 <= pad1 * 107) && pairs >= 2 * (device_info().sms / 2);
    } else if (ok) {
      const long long pairs = static_cast<long long>((L.M + 2 * kBlockM - 1) / (2 * kBlockM)) * tiles_n_;
      if (want != 2) ok = pairs >= 2 * (device_info().sms / 2);
    }
    if (ok && want != 1) cg = 2;
  }
  // ---- small linear problems: wave quantisation. The rules above pick the widest tile; at M = 5480 (ViT-L, four images:
  // the per-GPU share of the batch-32 configuration on eight GPUs) a [M, 1024] output is 172 128x256 tiles on 148 SMs --
  // two waves, the second one 16 % full (fc2: 846 TFLOP/s, proj: 509). Choose the tile by modelled time = waves x tile
  // width / relative tile efficiency instead (efficiencies from the per-signature timings in profiles/README.md). The
  // accumulation order of an output element does not depend on the tile shape, so results stay bit-identical.
  if (!L.force_bn && !L.force_cg && L.a_mode == A_LINEAR && (epi_is_bf16(g.epi) || g.epi == EPI_SWIGLU) && L.K > 256) {
    static const int tile_model = env_int("ADA_GEMM_TILE_MODEL", 1);
    const int sms = device_info().sms;
    const long long units_now = static_cast<long long>((L.M + kBlockM * cg - 1) / (kBlockM * cg)) * ((L.N + bn - 1) / bn);
    if (tile_model && units_now < 6LL * (sms / cg)) {  // large grids keep the established choice
      struct Cand { int bn, cg; double eff; };
      const Cand cands[4] = {{256, 2, 1.00}, {256, 1, 0.88}, {128, 1, 0.72}, {64, 1, 0.45}};
      double best = 1e30;
      for (const Cand& c : cands) {
        if (g.epi == EPI_SWIGLU && c.bn < 128) continue;
        if (c.bn > 64 && (L.N + c.bn - 1) / c.bn * c.bn > L.N + L.N / 8 + 63) continue;  // too much column padding
        const long long tiles = static_cast<long long>((L.M + kBlockM * c.cg - 1) / (kBlockM * c.cg)) * ((L.N + c.bn - 1) / c.bn);
        const long long units = sms / c.cg;
        const double t = static_cast<double>((tiles + units - 1) / units) * c.bn / c.eff;
        if (t < best * 0.999) {
          best = t;
          bn = c.bn;
          cg = c.cg;
        }
      }
    }
  }
  CUtensorMap ta, tb;
  int tiles_m;
  if (L.a_mode == A_CONV3X3) {
    ADA_REQUIRE(L.Cin % 8 == 0, "conv Cin must be a multiple of 8");
    g.H = L.H;
    g.W = L.W;
    const TileGeo geo = pick_tile_geo(L.batch, L.H, L.W, cg, conv_geo_general);
    g.lw = geo.lw;
    g.lh = geo.lh;
    g.lb = geo.lb;
    const int tw = 1 << geo.lw, th = 1 << geo.lh, nb = 1 << geo.lb;
    g.tiles_x = (L.W + tw * cg - 1) / (tw * cg);
    g.tiles_y = (L.H + th - 1) / th;
    g.tiles_b = (L.batch + nb - 1) / nb;
    g.c_chunks = round_up(L.Cin, kBlockK) / kBlockK;
    g.K = L.conv_taps * g.c_chunks * kBlockK;
    const int sd = L.conv_stride;
    ADA_REQUIRE(sd == 1 || sd == 2, "conv stride is 1 or 2");
    const int Hin = L.Hin ? L.Hin : L.H, Win = L.Win ? L.Win : L.W;
    ADA_REQUIRE((Hin - 1) / sd + 1 == L.H && (Win - 1) / sd + 1 == L.W, "conv input / output size mismatch (k3, pad 1)");
    g.conv_stride = sd;
    g.conv_taps = L.conv_taps;
    ADA_REQUIRE(L.conv_taps == 9 || (L.conv_taps == 1 && sd == 1 && L.Cin % kBlockK == 0), "pointwise pixel-tile mode: stride 1, Cin % 64 == 0");
    uint64_t dims[4] = {static_cast<uint64_t>(L.Cin), static_cast<uint64_t>(Win), static_cast<uint64_t>(Hin),
                        static_cast<uint64_t>(L.batch)};
    uint64_t str[3] = {static_cast<uint64_t>(L.Cin) * 2, static_cast<uint64_t>(Win) * L.Cin * 2,
                       static_cast<uint64_t>(Hin) * Win * L.Cin * 2};
    uint32_t box[4] = {kBlockK, static_cast<uint32_t>(tw * sd), static_cast<uint32_t>(th * sd), static_cast<uint32_t>(nb)};
    uint32_t es[4] = {1, static_cast<uint32_t>(sd), static_cast<uint32_t>(sd), 1};
    ta = make_tmap_bf16(L.A, 4, dims, str, box, es);
    tiles_m = g.tiles_b * g.tiles_x * g.tiles_y;
    ADA_REQUIRE(L.M == L.batch * L.H * L.W, "conv M mismatch");
  } else {
    ADA_REQUIRE(L.lda % 8 == 0, "A pitch must be a multiple of 8 elements");
    ta = make_tmap_2d(L.A, static_cast<uint64_t>(L.K), static_cast<uint64_t>(L.M), static_cast<uint64_t>(L.lda), kBlockK,
                      kBlockM);
    tiles_m = (L.M + kBlockM * cg - 1) / (kBlockM * cg);
  }
  tb = make_tmap_2d(L.Bw, static_cast<uint64_t>(g.K), static_cast<uint64_t>(L.N), static_cast<uint64_t>(L.ldb), kBlockK,
                    static_cast<uint32_t>(bn / cg));
  // output maps for the TMA-store epilogues (dummy = tb otherwise; never dereferenced)
  CUtensorMap tc = tb, tc2 = tb;
  g.has_relu_copy = 0;
#ifdef ADA_BRINGUP
  {
    static const int dbg = env_int("ADA_GEMM_TIMELINE", 0);
    g.debug_timeline = dbg;
  }
#else
  g.debug_timeline = 0;
#endif
  if (g.epi == EPI_BF16 || g.epi == EPI_F16 || g.epi == EPI_SWIGLU || g.epi == EPI_BF16_CHLN) {
    const int n_out = (g.epi == EPI_SWIGLU) ? L.N / 2 : L.N;
    ADA_REQUIRE(g.out_bf16 != nullptr && g.ldo % 8 == 0 && n_out % 8 == 0, "bf16 output needs ldo, N multiples of 8");
    auto make_c = [&](const void* ptr) {
      if (L.a_mode == A_CONV3X3) {
        ADA_REQUIRE(g.ldo == n_out, "conv output must be dense NHWC");
        uint64_t dims[4] = {static_cast<uint64_t>(n_out), static_cast<uint64_t>(L.W), static_cast<uint64_t>(L.H),
                            static_cast<uint64_t>(L.batch)};
        uint64_t str[3] = {static_cast<uint64_t>(n_out) * 2, static_cast<uint64_t>(L.W) * n_out * 2,
                           static_cast<uint64_t>(L.H) * L.W * n_out * 2};
        // one epilogue warp = 32 consecutive accumulator rows = whole tile rows (and whole images of the tile if it is small)
        const int srows = std::min(1 << g.lh, 32 >> g.lw), simgs = std::max(1, 32 >> (g.lw + g.lh));
        uint32_t box[4] = {64, static_cast<uint32_t>(1 << g.lw), static_cast<uint32_t>(srows), static_cast<uint32_t>(simgs)};
        return make_tmap_bf16(ptr, 4, dims, str, box);
      }
      return make_tmap_2d(ptr, static_cast<uint64_t>(n_out), static_cast<uint64_t>(L.M), static_cast<uint64_t>(g.ldo), 64, 32);
    };
    tc = make_c(g.out_bf16);
    if (L.out_relu) {
      tc2 = make_c(L.out_relu);
      g.has_relu_copy = 1;
    }
  }
  if (g.epi == EPI_CONVT && L.a_mode == A_CONV3X3) {
    // pixel-shuffle output [B, H*ks, W*ks, Cout] viewed as (kx*Cout + co, x, ky, y, b) for the TMA-store epilogue
    ADA_REQUIRE(g.out_bf16 != nullptr && g.ks >= 1 && g.cout % 64 == 0 && bn >= 64 && L.N == g.ks * g.ks * g.cout,
                "EPI_CONVT on pixel tiles: Cout % 64 == 0, N = ks * ks * Cout");
    const uint64_t co = static_cast<uint64_t>(g.cout), ks = static_cast<uint64_t>(g.ks), Wd = static_cast<uint64_t>(L.W),
                   Hd = static_cast<uint64_t>(L.H);
    uint64_t dims[5] = {ks * co, Wd, ks, Hd, static_cast<uint64_t>(L.batch)};
    uint64_t str[4] = {ks * co * 2, Wd * ks * co * 2, ks * Wd * ks * co * 2, Hd * ks * Wd * ks * co * 2};
    uint32_t box[5] = {64, static_cast<uint32_t>(kTileW), 1, 2, 1};
    tc = make_tmap_bf16(g.out_bf16, 5, dims, str, box);
  }
  if (g.epi == EPI_RESID_F32) {
    ADA_REQUIRE(L.a_mode == A_LINEAR && g.out_f32 != nullptr && g.ldo % 4 == 0, "RESID_F32: linear A, fp32 in/out, ldo % 4");
    tc = make_tmap_f32_2d(g.out_f32, static_cast<uint64_t>(L.N), static_cast<uint64_t>(L.M), static_cast<uint64_t>(g.ldo), 32, 32);
  }
  const int tiles_n = (L.N + bn - 1) / bn;
  const int num_tiles = tiles_m * tiles_n;
  const double kreal = (L.a_mode == A_CONV3X3) ? static_cast<double>(L.conv_taps) * L.Cin : static_cast<double>(L.K);
  ProfScope prof((L.a_mode == A_CONV3X3 && L.conv_taps == 9) ? PC_GEMM_CONV : PC_GEMM_LINEAR, 2.0 * L.M * static_cast<double>(L.N) * kreal,
                 2.0 * (static_cast<double>(L.M) * kreal + static_cast<double>(L.N) * kreal + static_cast<double>(L.M) * L.N), st);
  if (prof.r) {
    prof.r->m = L.M;
    prof.r->n = L.N;
    prof.r->k = static_cast<int>(kreal);
    prof.r->tag = g.epi | (g.act << 4) | (bn << 8) | (cg << 20);
  }
  // one instantiation per (tile, pairing, epilogue): keeps each kernel's code small (instruction-cache resident)
  // EPI_BF16 is specialised at compile time on (activation, residual adds); the rest of the launcher keeps seeing EPI_BF16
  int epi_t = g.epi;
  if (g.epi == EPI_BF16) {
    const bool resid = g.resid1 != nullptr || g.resid2 != nullptr;
    ADA_REQUIRE(!(resid && g.act == ACT_GELU), "EPI_BF16: GELU and residual adds are not combined on this path");
  }
  if (g.epi == EPI_F16) {
    ADA_REQUIRE(g.act == ACT_NONE && g.resid1 == nullptr && g.resid2 == nullptr && L.out_relu == nullptr,
                "EPI_F16: no activation, residuals or ReLU copy");
  }
  if (g.epi == EPI_BF16) {
    const bool resid = g.resid1 != nullptr || g.resid2 != nullptr;
    epi_t = resid ? EPI_BF16_RESID : (g.act == ACT_GELU) ? EPI_BF16_GELU : (g.act == ACT_RELU) ? EPI_BF16_RELU : EPI_BF16;
  }
#define ADA_GEMM_CASE(BN_, CG_, EPI_)                                      \
  if (bn == BN_ && cg == CG_ && epi_t == EPI_) {                           \
    launch_gemm_bn<BN_, CG_, EPI_>(ta, tb, tc, tc2, g, num_tiles, st);     \
    launched = true;                                                       \
  }
  bool launched = false;
  ADA_GEMM_CASE(64, 1, EPI_BF16)
  ADA_GEMM_CASE(128, 1, EPI_BF16)
  ADA_GEMM_CASE(128, 2, EPI_BF16)
  ADA_GEMM_CASE(256, 1, EPI_BF16)
  ADA_GEMM_CASE(256, 2, EPI_BF16)
  ADA_GEMM_CASE(64, 1, EPI_BF16_GELU)
  ADA_GEMM_CASE(128, 1, EPI_BF16_GELU)
  ADA_GEMM_CASE(128, 2, EPI_BF16_GELU)
  ADA_GEMM_CASE(256, 1, EPI_BF16_GELU)
  ADA_GEMM_CASE(256, 2, EPI_BF16_GELU)
  ADA_GEMM_CASE(64, 1, EPI_BF16_RELU)
  ADA_GEMM_CASE(128, 1, EPI_BF16_RELU)
  ADA_GEMM_CASE(128, 2, EPI_BF16_RELU)
  ADA_GEMM_CASE(256, 1, EPI_BF16_RELU)
  ADA_GEMM_CASE(256, 2, EPI_BF16_RELU)
  ADA_GEMM_CASE(64, 1, EPI_BF16_RESID)
  ADA_GEMM_CASE(128, 1, EPI_BF16_RESID)
  ADA_GEMM_CASE(128, 2, EPI_BF16_RESID)
  ADA_GEMM_CASE(256, 1, EPI_BF16_RESID)
  ADA_GEMM_CASE(256, 2, EPI_BF16_RESID)
  ADA_GEMM_CASE(64, 1, EPI_F16)
  ADA_GEMM_CASE(128, 1, EPI_F16)
  ADA_GEMM_CASE(256, 1, EPI_F16)
  ADA_GEMM_CASE(256, 2, EPI_F16)
  ADA_GEMM_CASE(256, 1, EPI_BF16_CHLN)
  ADA_GEMM_CASE(256, 2, EPI_BF16_CHLN)
  ADA_GEMM_CASE(64, 1, EPI_RESID_F32)
  ADA_GEMM_CASE(128, 1, EPI_RESID_F32)
  ADA_GEMM_CASE(256, 1, EPI_RESID_F32)
  ADA_GEMM_CASE(256, 2, EPI_RESID_F32)
  ADA_GEMM_CASE(128, 1, EPI_SWIGLU)
  ADA_GEMM_CASE(256, 1, EPI_SWIGLU)
  ADA_GEMM_CASE(256, 2, EPI_SWIGLU)
  ADA_GEMM_CASE(64, 1, EPI_EMBED)
  ADA_GEMM_CASE(128, 1, EPI_EMBED)
  ADA_GEMM_CASE(256, 1, EPI_EMBED)
  ADA_GEMM_CASE(256, 2, EPI_EMBED)
  ADA_GEMM_CASE(64, 1, EPI_CONVT)
  ADA_GEMM_CASE(128, 1, EPI_CONVT)
  ADA_GEMM_CASE(256, 1, EPI_CONVT)
  ADA_GEMM_CASE(256, 2, EPI_CONVT)
  ADA_GEMM_CASE(32, 1, EPI_TAIL)
#undef ADA_GEMM_CASE
  if (!launched)
    throw AdaError(ADA_EINVAL, "no GEMM instantiation for BN=" + std::to_string(bn) + " CG=" + std::to_string(cg) +
                                   " epi=" + std::to_string(g.epi));
  ++g_launches;
}

// ------------------------------------------------------------------------------------------------ other launchers
static void launch_layernorm(float* x, const __nv_bfloat16* delta, const __nv_bfloat16* delta2, const float* w, const float* b,
                             __nv_bfloat16* out, int rows, int D, float eps, int n_tok, int drop_cls, int write_x,
                             cudaStream_t st, const float* w2 = nullptr, const float* b2 = nullptr,
                             __nv_bfloat16* out2 = nullptr) {
  const int grid = (rows + 7) / 8;
  ADA_REQUIRE(delta != nullptr || delta2 == nullptr, "layernorm: delta2 without delta");
  ADA_REQUIRE(out2 == nullptr || (w2 != nullptr && b2 != nullptr && !drop_cls && n_tok > 1), "layernorm: second output needs w2 / b2, a full first output and n_tok");
  ProfScope prof(PC_LAYERNORM, 0.0,
                 (6.0 + (delta ? 2.0 : 0.0) + (delta2 ? 2.0 : 0.0) + (delta && write_x ? 4.0 : 0.0) + (out2 ? 2.0 : 0.0)) * rows *
                     static_cast<double>(D), st);
#define ADA_LN_CASE(C)                                                                                                      \
  case C:                                                                                                                   \
    launch_pdl(layernorm_rows_kernel<C>, dim3(grid), dim3(256), 0, st, x, delta, delta2, w, b, out, rows, eps, n_tok, drop_cls, \
               write_x, w2, b2, out2);                                                                                     \
    break;
  switch (D / 128) {
    ADA_LN_CASE(3)
    ADA_LN_CASE(6)
    ADA_LN_CASE(8)
    ADA_LN_CASE(12)
    default: throw AdaError(ADA_EINVAL, "layernorm: embed_dim must be 384/768/1024/1536");
  }
#undef ADA_LN_CASE
  ADA_REQUIRE(D % 128 == 0, "layernorm: D % 128");
  ADA_CHECK_CUDA(cudaGetLastError());
  ++g_launches;
}

template <int EMU, bool STAGGER, int WAITP, bool SPLIT = false>
static void launch_attention_fa(const CUtensorMap& tm, const CUtensorMap& tmo, const FaArgs& fa, cudaStream_t st) {
  static std::atomic<uint64_t> attr_done{0};
  ensure_smem_attr(attention_fa_kernel<EMU, STAGGER, WAITP, SPLIT>, kFaSmemBytes, attr_done);
  const int grid = std::min(fa.total_units, device_info().sms);  // persistent: one CTA per SM
  launch_pdl(attention_fa_kernel<EMU, STAGGER, WAITP, SPLIT>, dim3(grid), dim3(SPLIT ? kFaThreadsSplit : kFaThreads),
             kFaSmemBytes, st, tm, tmo, fa);
}

static void launch_attention(const __nv_bfloat16* qkv, __nv_bfloat16* out, int B, int N, int heads, cudaStream_t st,
                             int force_impl = -1) {
  const int D = heads * 64;
  uint64_t dims[3] = {static_cast<uint64_t>(3 * D), static_cast<uint64_t>(N), static_cast<uint64_t>(B)};
  uint64_t str[2] = {static_cast<uint64_t>(3 * D) * 2, static_cast<uint64_t>(N) * 3 * D * 2};
  uint32_t box[3] = {64, 128, 1};  // Q tile and K/V tiles: 128 tokens x 64 head dims
  static_assert(kAttQ == 128 && kAttKV == 128, "the attention tensor map assumes 128-token tiles");
  CUtensorMap tm = make_tmap_bf16(qkv, 3, dims, str, box);
  uint64_t odims[3] = {static_cast<uint64_t>(D), static_cast<uint64_t>(N), static_cast<uint64_t>(B)};
  uint64_t ostr[2] = {static_cast<uint64_t>(D) * 2, static_cast<uint64_t>(N) * D * 2};
  CUtensorMap tmo = make_tmap_bf16(out, 3, odims, ostr, box);
  AttArgs a;
  a.B = B;
  a.N = N;
  a.heads = heads;
  a.D = D;
  a.scale_log2e = 0.125f * 1.4426950408889634f;
  dim3 grid((N + kAttQ - 1) / kAttQ, heads, B);
  ProfScope prof(PC_ATTENTION, 4.0 * B * heads * static_cast<double>(N) * N * 64.0, 8.0 * B * static_cast<double>(N) * D, st);
  // Two kernels that agree bit for bit (tools/gpu_check.py attention_geo_*). attention.cuh (one 128-query tile per
  // CTA, two CTAs per SM, a score row shared by two threads) is the product path. attention2.cuh (persistent CTAs, 256
  // queries per work unit, one thread per score row, three issuing warps) is selectable with ADA_ATT_IMPL=1 / impl = 1 of
  // ada_op_attention: round-2 measurements (profiles/README.md) put it 3-6 % ahead stand-alone and in the model when ALL
  // its exponentials run on MUFU (10.1-10.4 vs 10.7-10.8 ms per step at batch 32, 16.3 vs 17.4 ms at 1036^2), but level or
  // behind (11.25 vs 10.7 ms) with the 6/16 FMA-pipe split that bit-identity with attention.cuh requires -- and an image
  // must not change with the batch size it is processed in, so the kernel choice may not depend on the grid.
  static const int impl_env = env_int("ADA_ATT_IMPL", -1);
  FaArgs fa;
  fa.B = B;
  fa.N = N;
  fa.heads = heads;
  fa.D = D;
  fa.units_per_seq = ((N + 127) / 128 + 1) / 2;
  fa.total_units = B * heads * fa.units_per_seq;
  fa.scale_log2e = a.scale_log2e;
  const int impl_sel = force_impl >= 0 ? force_impl : impl_env;
  if (impl_sel == 2) {  // attention2.cuh, two threads per score row (the arithmetic of attention.cuh in the persistent frame)
    launch_attention_fa<6, false, 2, true>(tm, tmo, fa, st);
    ADA_CHECK_CUDA(cudaGetLastError());
    ++g_launches;
    return;
  }
  const bool use_fa = impl_sel == 1;
  if (use_fa) {
#ifdef ADA_BRINGUP
    // measurement variants (exponential split MUFU / FMA pipe, group stagger, placement of the P V wait); the sweeps are
    // in profiles/README.md. The product library carries <6, false, 2> only.
    static const int emu = env_int("ADA_ATT_EMU", 6);
    static const int stagger = env_int("ADA_ATT_STAGGER", 0);
    static const int waitp = env_int("ADA_ATT_WAIT", 2);
#define ADA_FA_CASE(E)                                                                                  \
  case E:                                                                                               \
    if (stagger) {                                                                                      \
      if (waitp == 0) launch_attention_fa<E, true, 0>(tm, tmo, fa, st);                                 \
      else if (waitp == 1) launch_attention_fa<E, true, 1>(tm, tmo, fa, st);                            \
      else launch_attention_fa<E, true, 2>(tm, tmo, fa, st);                                            \
    } else {                                                                                            \
      if (waitp == 0) launch_attention_fa<E, false, 0>(tm, tmo, fa, st);                                \
      else if (waitp == 1) launch_attention_fa<E, false, 1>(tm, tmo, fa, st);                           \
      else launch_attention_fa<E, false, 2>(tm, tmo, fa, st);                                           \
    }                                                                                                   \
    break;
    switch (emu) {
      ADA_FA_CASE(0)
      ADA_FA_CASE(4)
      ADA_FA_CASE(6)
      ADA_FA_CASE(-1)
      ADA_FA_CASE(-2)
      default: throw AdaError(ADA_EINVAL, "ADA_ATT_EMU must be one of 0, 4, 6 (-1 / -2: timing skeletons)");
    }
#undef ADA_FA_CASE
#else
    launch_attention_fa<6, false, 2>(tm, tmo, fa, st);
#endif
    ADA_CHECK_CUDA(cudaGetLastError());
    ++g_launches;
    return;
  }
#ifdef ADA_BRINGUP
  // measurement variants of the kernel (attention.cuh: exponential placement, timing skeleton, clock64 timeline) exist only
  // in bring-up builds (-DADA_BRINGUP); the product library carries variant 0 alone.
  static const int variant = env_int("ADA_ATT_VARIANT", 0);
#define ADA_ATT_LAUNCH(V, SMEM)                                                                 \
  do {                                                                                          \
    static std::atomic<uint64_t> done{0};                                                       \
    ensure_smem_attr(attention_tcgen05_kernel<V>, SMEM, done);                                  \
    launch_pdl(attention_tcgen05_kernel<V>, grid, dim3(kAttThreads), SMEM, st, tm, tmo, a);     \
  } while (0)
  switch (variant) {
    case 1: ADA_ATT_LAUNCH(1, kAttSmemBytes); break;
    case 2: ADA_ATT_LAUNCH(2, kAttSmemBytes); break;
    case 3: ADA_ATT_LAUNCH(3, kAttSmemBytes); break;
    case 4: ADA_ATT_LAUNCH(4, kAttSmemBytes); break;
    case 5: ADA_ATT_LAUNCH(5, kAttSmemBytes); break;
    case 10: ADA_ATT_LAUNCH(10, kAttSmemBytes); break;
    default: ADA_ATT_LAUNCH(0, kAttSmemBytes); break;
  }
#undef ADA_ATT_LAUNCH
#else
  static std::atomic<uint64_t> attr_done{0};
  ensure_smem_attr(attention_tcgen05_kernel<0>, kAttSmemBytes, attr_done);
  launch_pdl(attention_tcgen05_kernel<0>, grid, dim3(kAttThreads), kAttSmemBytes, st, tm, tmo, a);
#endif
  ADA_CHECK_CUDA(cudaGetLastError());
  ++g_launches;
}

static void launch_channel_ln_relu(const __nv_bfloat16* in, const float* w, const float* b, __nv_bfloat16* out,
                                   long long pixels, int C, float eps, cudaStream_t st) {
  ADA_REQUIRE(C % 8 == 0 && C <= 1536, "channel LN: C % 8 == 0 and C <= 1536");
  const int sms = device_info().sms;
  ProfScope prof(PC_CHANNEL_LN, 0.0, 4.0 * pixels * static_cast<double>(C), st);
  auto grid_for = [&](int pix_per_warp, int blocks_per_sm) {  // persistent warps walking pixels with a grid stride
    return static_cast<int>(std::min<long long>((pixels + 8 * pix_per_warp - 1) / (8 * pix_per_warp), static_cast<long long>(sms) * blocks_per_sm));
  };
  if (C <= 256)
    channel_ln_relu_kernel<1, true, 4><<<grid_for(4, 8), 256, 0, st>>>(in, w, b, out, pixels, C, eps);
  else if (C <= 512)
    channel_ln_relu_kernel<2, true, 2><<<grid_for(2, 8), 256, 0, st>>>(in, w, b, out, pixels, C, eps);
  else if (C <= 1024)
    channel_ln_relu_kernel<4, false, 1><<<grid_for(1, 8), 256, 0, st>>>(in, w, b, out, pixels, C, eps);
  else
    channel_ln_relu_kernel<6, false, 1><<<grid_for(1, 8), 256, 0, st>>>(in, w, b, out, pixels, C, eps);
  ADA_CHECK_CUDA(cudaGetLastError());
  ++g_launches;
}

static void launch_upsample(const __nv_bfloat16* in, __nv_bfloat16* out, int B, int Hi, int Wi, int Ho, int Wo, int C,
                            cudaStream_t st) {
  ADA_REQUIRE(C % 8 == 0, "upsample: C % 8");
  const long long total = static_cast<long long>(B) * Ho * Wo * (C / 8);
  ProfScope prof(PC_UPSAMPLE, 0.0, 2.0 * B * C * (static_cast<double>(Hi) * Wi + static_cast<double>(Ho) * Wo), st);
  const int groups = C / 8;
  int shift = -1;
  for (int sft = 0; sft < 12; ++sft)
    if ((1 << sft) == groups) shift = sft;
  dim3 grid(static_cast<unsigned>((static_cast<long long>(Wo) * groups + 255) / 256),
            static_cast<unsigned>((Ho + kUpRows - 1) / kUpRows), static_cast<unsigned>(B));
  (void)total;
  upsample_bilinear_kernel<<<grid, 256, 0, st>>>(in, out, Hi, Wi, Ho, Wo, C, shift);
  ADA_CHECK_CUDA(cudaGetLastError());
  ++g_launches;
}

static void launch_tail_gather(const __half* V, const float* bias2, const float* aux, float* out, int B, int Hl,
                               int Wl, int H, int W, int sigmoid, cudaStream_t st) {
  // other geometries can need a low-resolution patch of more than 12 x 12 and trap (tests/test_head_check_cpu.py)
  ADA_REQUIRE(Hl * 14 == H * 8 && Wl * 14 == W * 8, "tail_gather: 8h -> 14h geometry");
  static std::atomic<uint64_t> attr_done{0};
  ensure_smem_attr(tail_gather_kernel, kTailSmemBytes, attr_done);
  dim3 grid((W + kTailTile - 1) / kTailTile, (H + kTailTile - 1) / kTailTile, B);
  // HBM-bound: algorithmic bytes = the tap map read once + the fp32 output (its 36 x 32 FMAs per pixel are not counted)
  ProfScope prof(PC_TAIL_GATHER, 0.0, static_cast<double>(B) * (2.0 * Hl * Wl * kTailCh + 4.0 * H * W), st);
  tail_gather_kernel<<<grid, 256, kTailSmemBytes, st>>>(V, bias2, aux, out, Hl, Wl, H, W, sigmoid);
  ADA_CHECK_CUDA(cudaGetLastError());
  ++g_launches;
}

// Tail on tensor cores (tail_mma.cuh): the fp16 output_conv1 map in, the fp32 result out.
static bool tail_mma_supported(int C, int Hl, int Wl, int H, int W) {
  return C % 32 == 0 && C <= kTmMaxC && Hl * 14 == H * 8 && Wl * 14 == W * 8 && W % kTmTileW == 0;
}
static void launch_tail_mma(const __half* L, const __half* wpk, const float* bias2, const float* aux, float* out, int B,
                            int Hl, int Wl, int H, int W, int C, int sigmoid, cudaStream_t st) {
  ADA_REQUIRE(tail_mma_supported(C, Hl, Wl, H, W), "tail_mma: C % 32 == 0, C <= 128, 8h -> 14h geometry");
  static std::atomic<uint64_t> attr_done{0};
  ensure_smem_attr(tail_mma_kernel, tm_smem_bytes(kTmMaxC), attr_done);
  uint64_t dims[4] = {static_cast<uint64_t>(C), static_cast<uint64_t>(Wl), static_cast<uint64_t>(Hl), static_cast<uint64_t>(B)};
  uint64_t str[3] = {static_cast<uint64_t>(C) * 2, static_cast<uint64_t>(Wl) * C * 2, static_cast<uint64_t>(Hl) * Wl * C * 2};
  uint32_t box[4] = {static_cast<uint32_t>(C), kTmPatchW, kTmPatchH, 1};
  const CUtensorMap tl = make_tmap_bf16(L, 4, dims, str, box, nullptr, false);  // 2-byte elements, dense box
  TailMmaArgs a;
  a.wpk = wpk;
  a.bias2 = bias2;
  a.aux = aux;
  a.out = out;
  a.B = B;
  a.Hl = Hl;
  a.Wl = Wl;
  a.H = H;
  a.W = W;
  a.C = C;
  a.sigmoid = sigmoid;
  a.tiles_x = W / kTmTileW;
  a.tiles_y = (H + kTmTileH - 1) / kTmTileH;
  a.total_tiles = B * a.tiles_x * a.tiles_y;
  ADA_REQUIRE(static_cast<long long>(a.total_tiles) * std::max(a.tiles_x, a.tiles_y) < (1LL << 31), "tail_mma: too many tiles");
  a.magic_x = static_cast<uint32_t>(((1ULL << 32) + a.tiles_x - 1) / a.tiles_x);
  a.magic_y = static_cast<uint32_t>(((1ULL << 32) + a.tiles_y - 1) / a.tiles_y);
  const int grid = std::min(a.total_tiles, device_info().sms);
  // tensor-bound by construction, reported with the conv FLOPs of the layer it replaces (dpt.py:195: 3x3, C -> 32, at H x W)
  ProfScope prof(PC_TAIL_GATHER, 2.0 * B * static_cast<double>(H) * W * 32.0 * 9.0 * C,
                 static_cast<double>(B) * (2.0 * Hl * Wl * C + 4.0 * H * W), st);
  launch_pdl(tail_mma_kernel, dim3(grid), dim3(kTmThreads), static_cast<size_t>(tm_smem_bytes(C)), st, tl, a);
  ADA_CHECK_CUDA(cudaGetLastError());
  ++g_launches;
}

static void launch_patch_gather(const float* rgb, const float* const* guides, const int* guide_ch, int n_guides,
                                __nv_bfloat16* out, int B, int H, int W, int Kpad, int normalize, cudaStream_t st) {
  ADA_REQUIRE(n_guides >= 0 && n_guides <= 3, "at most 3 guide tensors");
  PatchSrc src{};
  src.ptr[0] = rgb;
  src.ch[0] = 3;
  int C = 3;
  for (int i = 0; i < n_guides; ++i) {
    src.ptr[i + 1] = guides[i];
    src.ch[i + 1] = guide_ch[i];
    C += guide_ch[i];
  }
  src.n = n_guides + 1;
  ADA_REQUIRE(C * 196 <= Kpad, "patch gather: Kpad too small");
  ADA_REQUIRE(Kpad % 4 == 0, "patch gather: row pitch must be a multiple of 4 elements");
  const int pw = W / 14, ph = H / 14;
  const int chunks = (pw + kPgPatches - 1) / kPgPatches, npc = (pw + chunks - 1) / chunks;  // even split of a patch row
  const int smem = npc * C * 196 * 2;
  static std::atomic<uint64_t> attr_done{0};
  ensure_smem_attr(patch_gather_kernel, kPgPatches * 8 * 196 * 2, attr_done);
  ADA_REQUIRE(C <= 8, "patch gather: at most 8 input channels");
  ProfScope prof(PC_GATHER, 0.0, 6.0 * B * C * static_cast<double>(H) * W, st);
  const unsigned grid = static_cast<unsigned>(B) * ph * chunks;
  if (normalize)
    patch_gather_kernel<<<grid, 256, smem, st>>>(src, out, B, C, H, W, Kpad, chunks, npc, 0.485f, 0.456f, 0.406f, 0.229f,
                                                 0.224f, 0.225f);
  else  // un-guided model: the caller normalised the image (infer.py:18)
    patch_gather_kernel<<<grid, 256, smem, st>>>(src, out, B, C, H, W, Kpad, chunks, npc, 0.f, 0.f, 0.f, 1.f, 1.f, 1.f);
  ADA_CHECK_CUDA(cudaGetLastError());
  ++g_launches;
}

// ------------------------------------------------------------------------------------------------ weight packing
// Bicubic resampling of the position table, mirroring ATen upsample_bicubic2d (align_corners=False, A=-0.75) called
// with an explicit scale_factor: src = (dst + 0.5) / scale_factor - 0.5, taps clamped to the border.
static void cubic_coeffs(float t, float c[4]) {
  const float A = -0.75f;
  auto c1 = [&](float x) { return ((A + 2.f) * x - (A + 3.f)) * x * x + 1.f; };
  auto c2 = [&](float x) { return ((A * x - 5.f * A) * x + 8.f * A) * x - 4.f * A; };
  c[0] = c2(t + 1.f);
  c[1] = c1(t);
  c[2] = c1(1.f - t);
  c[3] = c2(2.f - t);
}
static void interp_pos_host(const float* pos, int grid, int D, int gh, int gw, float offset, float* out) {
  const double sf_h = static_cast<double>(gh + offset) / grid;  // python float math (dinov2.py:214-219)
  const double sf_w = static_cast<double>(gw + offset) / grid;
  const float rh = static_cast<float>(1.0 / sf_h), rw = static_cast<float>(1.0 / sf_w);
  for (int oy = 0; oy < gh; ++oy) {
    const float fy = rh * (oy + 0.5f) - 0.5f;
    const int iy = static_cast<int>(floorf(fy));
    float cy[4];
    cubic_coeffs(fy - iy, cy);
    for (int ox = 0; ox < gw; ++ox) {
      const float fx = rw * (ox + 0.5f) - 0.5f;
      const int ix = static_cast<int>(floorf(fx));
      float cx[4];
      cubic_coeffs(fx - ix, cx);
      float* o = out + (static_cast<size_t>(oy) * gw + ox) * D;
      for (int d = 0; d < D; ++d) o[d] = 0.f;
      for (int a = 0; a < 4; ++a) {
        const int yy = std::min(std::max(iy - 1 + a, 0), grid - 1);
        float rowacc_w[4];
        for (int b = 0; b < 4; ++b) rowacc_w[b] = cx[b] * cy[a];
        for (int b = 0; b < 4; ++b) {
          const int xx = std::min(std::max(ix - 1 + b, 0), grid - 1);
          const float* p = pos + (static_cast<size_t>(yy) * grid + xx) * D;
          const float wgt = rowacc_w[b];
          for (int d = 0; d < D; ++d) o[d] += wgt * p[d];
        }
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------ model
// One state-dict tensor between ada_set_weight and ada_finalize: fp32, staged where it arrived -- a device copy for device
// sources (no PCIe round trip), a host copy for host sources (works without a device; uploaded by ada_finalize).
struct StagedTensor {
  std::vector<float> host;
  float* dev = nullptr;
  std::vector<int64_t> shape;
  size_t n = 0;
};

struct DevBuf {
  void* p = nullptr;
  size_t bytes = 0;
};

struct BlockW {
  float *ln1w, *ln1b, *ln2w, *ln2b, *bqkv, *bproj, *g1, *g2, *b1, *b2;
  __nv_bfloat16 *wqkv, *wproj, *w1, *w2;
};
struct ConvW {
  __nv_bfloat16* w = nullptr;
  float* b = nullptr;
  int cin = 0, cout = 0, ldw = 0;
};
struct RefineW {
  ConvW rcu1c1, rcu1c2, rcu2c1, rcu2c2;
  __nv_bfloat16* wout = nullptr;
  float* bout = nullptr;
};

}  // namespace ada

using namespace ada;

struct ada_model;
namespace ada { struct Profiler; }
struct ada_model {
  ada_config cfg{};
  int device = -1;  // device ordinal current at ada_create: weights, workspace and every launch live there
  std::map<std::string, std::vector<int64_t>> spec;  // expected state dict: name -> shape (expected_weights)
  std::unordered_map<std::string, StagedTensor> host;  // staged fp32 state dict (released by ada_finalize)
  bool finalized = false;
  bool capture = false;
  bool profile = false;
  ada::Profiler prof;
  std::vector<void*> owned;  // device allocations holding packed weights

  // packed weights
  int kpad = 0, cin_total = 0;
  __nv_bfloat16* w_embed = nullptr;
  std::vector<float> pos_host;      // [1 + grid*grid, D]
  std::vector<float> cls_host;      // [D]
  std::vector<float> embed_bias;    // [D] b_rgb + b_guide
  std::vector<BlockW> blocks;
  float *normw = nullptr, *normb = nullptr;
  __nv_bfloat16* w_proj[4] = {};
  float* b_proj[4] = {};
  __nv_bfloat16* w_rs[4] = {};
  float* b_rs[4] = {};
  ConvW ip[4];
  float *ipln_w[4] = {}, *ipln_b[4] = {};
  ConvW rn[4];
  RefineW ref[5];  // 1..4
  ConvW oc1, oc2;
  __nv_bfloat16* w_tail_taps = nullptr;  // [288, F/2]
  __half* w_tail_mma = nullptr;          // [3][F/16][96][8] fp16 (tail_mma_kernel), null when F/2 is not supported there
  float* tail_aux = nullptr;  // 32 weights + 1 bias of output_conv2.2

  // per-(H,W) position cache on device
  struct PosCache {
    float* posb = nullptr;     // [P, D] pos + embed bias
    float* cls_pos = nullptr;  // [D]
  };
  std::map<std::pair<int, int>, PosCache> pos_cache;

  // workspace
  DevBuf arena;
  int wsB = 0, wsH = 0, wsW = 0;
  std::unordered_map<std::string, std::pair<void*, size_t>> named;  // intermediates (ptr, elements) + dtype by prefix
  std::unordered_map<std::string, int> named_is_f32;
  // buffers
  float* x = nullptr;
  __nv_bfloat16 *xn = nullptr, *qkv = nullptr, *att = nullptr, *hbuf = nullptr, *ybuf = nullptr, *ybuf2 = nullptr, *a_embed = nullptr;
  __nv_bfloat16* tap[4] = {};
  float* tokens_dbg = nullptr;
  __nv_bfloat16 *proj[4] = {}, *rs[4] = {}, *ipb[4] = {}, *rnb[4] = {}, *rnr[4] = {};
  __nv_bfloat16 *t1 = nullptr, *sum = nullptr, *sumr = nullptr, *r2 = nullptr, *ocb = nullptr, *path[5] = {},
                *oc1b = nullptr, *up = nullptr, *vtap = nullptr;
  int last_B = 0, last_H = 0, last_W = 0, last_launches = 0;

  // ---- optional CUDA-graph replay of the forward (ada_set_graph): small batches are launch bound (ViT-L, one image:
  // 220 launches in 4 ms). The graph works on handle-owned staging copies of the inputs / output so that it does not
  // depend on the caller's pointers; it is dropped whenever the workspace is re-planned.
  bool graph_on = false;
  int graph_state = 0;  // 0: nothing, 1: one eager forward done at this shape (allocations, caches), 2: captured
  cudaGraph_t graph = nullptr;
  cudaGraphExec_t graph_exec = nullptr;
  cudaStream_t cap_stream = nullptr;
  float* g_rgb = nullptr;
  float* g_guides[3] = {nullptr, nullptr, nullptr};
  int g_guide_ch[3] = {0, 0, 0};
  int g_nguides = 0;
  float* g_out = nullptr;
  void drop_graph() {
    if (graph_exec) cudaGraphExecDestroy(graph_exec);
    if (graph) cudaGraphDestroy(graph);
    graph_exec = nullptr;
    graph = nullptr;
    if (g_rgb) cudaFree(g_rgb);
    for (float*& p : g_guides) {
      if (p) cudaFree(p);
      p = nullptr;
    }
    if (g_out) cudaFree(g_out);
    g_rgb = g_out = nullptr;
    graph_state = 0;
  }

  void drop_staged() {
    for (auto& kv : host)
      if (kv.second.dev) cudaFree(kv.second.dev);
    host.clear();
  }

  ~ada_model() {
    drop_graph();
    drop_staged();
    if (cap_stream) cudaStreamDestroy(cap_stream);
    for (void* p : owned) cudaFree(p);
    if (arena.p) cudaFree(arena.p);
    for (auto& kv : pos_cache) {
      cudaFree(kv.second.posb);
      cudaFree(kv.second.cls_pos);
    }
  }
};

namespace ada {

template <typename T>
static T* upload(ada_model* m, const void* src, size_t bytes) {
  void* d = nullptr;
  ADA_CHECK_CUDA(cudaMalloc(&d, std::max<size_t>(bytes, 16)));
  ADA_CHECK_CUDA(cudaMemcpy(d, src, bytes, cudaMemcpyHostToDevice));
  m->owned.push_back(d);
  return reinterpret_cast<T*>(d);
}
template <typename T>
static T* dev_alloc(ada_model* m, size_t elems) {
  void* d = nullptr;
  ADA_CHECK_CUDA(cudaMalloc(&d, std::max<size_t>(elems * sizeof(T), 16)));
  m->owned.push_back(d);
  return reinterpret_cast<T*>(d);
}
// staged tensor -> device fp32 pointer (shape checked); host-staged tensors are uploaded on first use
static const float* need(ada_model* m, const std::string& key, std::vector<int64_t> shape) {
  auto it = m->host.find(key);
  if (it == m->host.end()) throw AdaError(ADA_ESTATE, "missing weight: " + key);
  StagedTensor& t = it->second;
  if (t.shape != shape) {
    std::string s = "shape mismatch for " + key + ": got [";
    for (auto v : t.shape) s += std::to_string(v) + ",";
    s += "] expected [";
    for (auto v : shape) s += std::to_string(v) + ",";
    throw AdaError(ADA_EINVAL, s + "]");
  }
  if (!t.dev) {
    ADA_CHECK_CUDA(cudaMalloc(&t.dev, std::max<size_t>(t.n * 4, 16)));
    ADA_CHECK_CUDA(cudaMemcpy(t.dev, t.host.data(), t.n * 4, cudaMemcpyHostToDevice));
    std::vector<float>().swap(t.host);
  }
  return t.dev;
}
static size_t numel_of(const std::vector<int64_t>& shape) {
  size_t n = 1;
  for (auto v : shape) n *= static_cast<size_t>(v);
  return n;
}
// small tensors the host needs (position table, cls token, patch-embed biases)
static std::vector<float> need_host(ada_model* m, const std::string& key, std::vector<int64_t> shape) {
  const float* d = need(m, key, shape);
  std::vector<float> h(numel_of(shape));
  ADA_CHECK_CUDA(cudaMemcpy(h.data(), d, h.size() * 4, cudaMemcpyDeviceToHost));
  return h;
}
static void run_pack(const float* src, const float* src2, __nv_bfloat16* dst, long long n, const PackDesc& d) {
  pack_weights_kernel<<<static_cast<unsigned>((n + 255) / 256), 256>>>(src, src2, dst, n, d);
  ADA_CHECK_CUDA(cudaGetLastError());
}
static float* up_f32(ada_model* m, const std::string& key, std::vector<int64_t> shape) {
  const float* src = need(m, key, shape);
  const size_t n = numel_of(shape);
  float* d = dev_alloc<float>(m, n);
  ADA_CHECK_CUDA(cudaMemcpyAsync(d, src, n * 4, cudaMemcpyDeviceToDevice, nullptr));
  return d;
}
static __nv_bfloat16* up_bf16(ada_model* m, const std::string& key, std::vector<int64_t> shape) {
  const float* src = need(m, key, shape);
  const size_t n = numel_of(shape);
  __nv_bfloat16* d = dev_alloc<__nv_bfloat16>(m, n);
  run_pack(src, nullptr, d, static_cast<long long>(n), PackDesc{PACK_CAST, 0, 0, 0, 0});
  return d;
}
// conv3x3 weight [Cout, Cin, 3, 3] (torch) -> [Cout, 9 * Cpad], K index = tap*Cpad + ci, zero padded channels
static __nv_bfloat16* pack_conv3x3_dev(ada_model* m, const float* src, int cout, int cin) {
  const int Cpad = round_up(cin, kBlockK);
  const long long n = static_cast<long long>(cout) * 9 * Cpad;
  __nv_bfloat16* d = dev_alloc<__nv_bfloat16>(m, n);
  run_pack(src, nullptr, d, n, PackDesc{PACK_CONV3X3, cout, cin, Cpad, 0});
  return d;
}
static ConvW up_conv3x3(ada_model* m, const std::string& prefix, int cout, int cin, bool bias) {
  ConvW c;
  c.w = pack_conv3x3_dev(m, need(m, prefix + ".weight", {cout, cin, 3, 3}), cout, cin);
  c.cin = cin;
  c.cout = cout;
  c.ldw = 9 * round_up(cin, kBlockK);
  c.b = bias ? up_f32(m, prefix + ".bias", {cout}) : nullptr;
  return c;
}

// The reference state dict for this architecture (relative to `encoder.`): name -> shape. SURVEY.md section 8b key template;
// dinov2.py:107-117,188-196 (embeddings), block.py:60-80 (blocks), dpt.py:86-159 (head). ada_set_weight rejects anything
// that is not in this table (ADA_EINVAL), ada_finalize reports every entry that was never set (ADA_ESTATE).
static std::map<std::string, std::vector<int64_t>> expected_weights(const ada_config& c) {
  std::map<std::string, std::vector<int64_t>> w;
  const int64_t D = c.embed_dim, Cg = c.guide_channels, G = c.pos_grid, F = c.features, Hd = c.ffn_hidden;
  const std::string pre = "pretrained.";
  w[pre + "cls_token"] = {1, 1, D};
  w[pre + "pos_embed"] = {1, 1 + G * G, D};
  w[pre + "mask_token"] = {1, D};
  w[pre + "patch_embed.proj.weight"] = {D, 3, 14, 14};
  w[pre + "patch_embed.proj.bias"] = {D};
  if (Cg > 0) {
    w[pre + "patch_embed_guidance.proj.weight"] = {D, Cg, 14, 14};
    w[pre + "patch_embed_guidance.proj.bias"] = {D};
  }
  for (int i = 0; i < c.depth; ++i) {
    const std::string b = pre + "blocks." + std::to_string(i) + ".";
    for (const char* n : {"norm1", "norm2"}) {
      w[b + n + ".weight"] = {D};
      w[b + n + ".bias"] = {D};
    }
    w[b + "attn.qkv.weight"] = {3 * D, D};
    w[b + "attn.qkv.bias"] = {3 * D};
    w[b + "attn.proj.weight"] = {D, D};
    w[b + "attn.proj.bias"] = {D};
    w[b + "ls1.gamma"] = {D};
    w[b + "ls2.gamma"] = {D};
    if (c.ffn_kind == 0) {
      w[b + "mlp.fc1.weight"] = {Hd, D};
      w[b + "mlp.fc1.bias"] = {Hd};
      w[b + "mlp.fc2.weight"] = {D, Hd};
      w[b + "mlp.fc2.bias"] = {D};
    } else {
      w[b + "mlp.w12.weight"] = {2 * Hd, D};
      w[b + "mlp.w12.bias"] = {2 * Hd};
      w[b + "mlp.w3.weight"] = {D, Hd};
      w[b + "mlp.w3.bias"] = {D};
    }
  }
  w[pre + "norm.weight"] = {D};
  w[pre + "norm.bias"] = {D};
  const std::string hd = "depth_head.";
  auto conv = [&](const std::string& name, int64_t co, int64_t ci, int64_t k, bool bias) {
    w[hd + name + ".weight"] = {co, ci, k, k};
    if (bias) w[hd + name + ".bias"] = {co};
  };
  for (int i = 0; i < 4; ++i) {
    const int64_t Ci = c.out_channels[i];
    const std::string si = std::to_string(i);
    conv("projects." + si, Ci, D, 1, true);
    if (i == 0) conv("resize_layers.0", Ci, Ci, 4, true);  // ConvTranspose2d: [Cin, Cout, k, k], Cin == Cout
    if (i == 1) conv("resize_layers.1", Ci, Ci, 2, true);
    if (i == 3) conv("resize_layers.3", Ci, Ci, 3, true);
    if (c.input_projection) {
      conv("input_projection." + si + ".0", Ci, Ci, 3, true);
      w[hd + "input_projection." + si + ".1.weight"] = {Ci};
      w[hd + "input_projection." + si + ".1.bias"] = {Ci};
    }
    conv("scratch.layer" + std::to_string(i + 1) + "_rn", F, Ci, 3, false);
  }
  for (int k = 1; k <= 4; ++k) {
    const std::string r = "scratch.refinenet" + std::to_string(k) + ".";
    conv(r + "out_conv", F, F, 1, true);
    for (const char* u : {"resConfUnit1", "resConfUnit2"})
      for (const char* cv : {"conv1", "conv2"}) conv(r + u + "." + cv, F, F, 3, true);
  }
  conv("scratch.output_conv1", F / 2, F, 3, true);
  conv("scratch.output_conv2.0", 32, F / 2, 3, true);
  conv("scratch.output_conv2.2", 1, 32, 1, true);
  return w;
}

static void finalize_model(ada_model* m) {
  {  // report EVERY missing tensor, not just the first one the packer would trip over
    std::string missing;
    int n_missing = 0;
    for (const auto& kv : m->spec)
      if (!m->host.count(kv.first)) {
        if (n_missing++ < 24) missing += (missing.empty() ? "" : ", ") + kv.first;
      }
    if (n_missing)
      throw AdaError(ADA_ESTATE, "ada_finalize: " + std::to_string(n_missing) + " of " + std::to_string(m->spec.size()) +
                                     " tensors were never set: " + missing + (n_missing > 24 ? ", ..." : ""));
  }
  require_device();
  if (m->device < 0) m->device = device_info().device;
  ADA_REQUIRE(device_info().device == m->device, "ada_finalize: the device that was current at ada_create must be current");
  const ada_config& c = m->cfg;
  const int D = c.embed_dim, Cg = c.guide_channels, G = c.pos_grid;
  const std::string pre = "pretrained.";
  // ---- patch embed: fused (3+Cg)-channel weight, summed biases (dinov2.py:234-240)
  m->cin_total = 3 + Cg;
  m->kpad = round_up(m->cin_total * 196, kBlockK);
  {
    const float* wr = need(m, pre + "patch_embed.proj.weight", {D, 3, 14, 14});
    m->embed_bias = need_host(m, pre + "patch_embed.proj.bias", {D});
    const float* wg = nullptr;
    if (Cg > 0) {
      wg = need(m, pre + "patch_embed_guidance.proj.weight", {D, Cg, 14, 14});
      const std::vector<float> bg = need_host(m, pre + "patch_embed_guidance.proj.bias", {D});
      for (int d = 0; d < D; ++d) m->embed_bias[d] += bg[d];
    }
    const long long n = static_cast<long long>(D) * m->kpad;
    m->w_embed = dev_alloc<__nv_bfloat16>(m, n);
    run_pack(wr, wg, m->w_embed, n, PackDesc{PACK_EMBED, D, Cg, m->kpad, 0});
  }
  m->pos_host = need_host(m, pre + "pos_embed", {1, 1 + G * G, D});
  m->cls_host = need_host(m, pre + "cls_token", {1, 1, D});
  need(m, pre + "mask_token", {1, D});  // dead weight, must exist for strict loading (dinov2.py:188)
  // ---- blocks
  m->blocks.resize(c.depth);
  for (int i = 0; i < c.depth; ++i) {
    const std::string b = pre + "blocks." + std::to_string(i) + ".";
    BlockW& w = m->blocks[i];
    w.ln1w = up_f32(m, b + "norm1.weight", {D});
    w.ln1b = up_f32(m, b + "norm1.bias", {D});
    w.ln2w = up_f32(m, b + "norm2.weight", {D});
    w.ln2b = up_f32(m, b + "norm2.bias", {D});
    w.wqkv = up_bf16(m, b + "attn.qkv.weight", {3 * D, D});
    w.bqkv = up_f32(m, b + "attn.qkv.bias", {3 * D});
    w.wproj = up_bf16(m, b + "attn.proj.weight", {D, D});
    w.bproj = up_f32(m, b + "attn.proj.bias", {D});
    w.g1 = up_f32(m, b + "ls1.gamma", {D});
    w.g2 = up_f32(m, b + "ls2.gamma", {D});
    if (c.ffn_kind == 0) {
      const int Hd = c.ffn_hidden;
      w.w1 = up_bf16(m, b + "mlp.fc1.weight", {Hd, D});
      w.b1 = up_f32(m, b + "mlp.fc1.bias", {Hd});
      w.w2 = up_bf16(m, b + "mlp.fc2.weight", {D, Hd});
      w.b2 = up_f32(m, b + "mlp.fc2.bias", {D});
    } else {
      // SwiGLU: interleave x1 / x2 rows in 32-wide chunks so one accumulator tile holds both halves (swiglu_ffn.py:30-32)
      const int Hd = c.ffn_hidden;
      const float* w12 = need(m, b + "mlp.w12.weight", {2 * Hd, D});
      const float* b12 = need(m, b + "mlp.w12.bias", {2 * Hd});
      const long long n = 2LL * Hd * D;
      w.w1 = dev_alloc<__nv_bfloat16>(m, n);
      run_pack(w12, nullptr, w.w1, n, PackDesc{PACK_SWIGLU, Hd, D, 0, 0});
      w.b1 = dev_alloc<float>(m, 2 * Hd);
      swiglu_bias_kernel<<<(2 * Hd + 255) / 256, 256>>>(b12, w.b1, Hd);
      ADA_CHECK_CUDA(cudaGetLastError());
      w.w2 = up_bf16(m, b + "mlp.w3.weight", {D, Hd});
      w.b2 = up_f32(m, b + "mlp.w3.bias", {D});
    }
  }
  m->normw = up_f32(m, pre + "norm.weight", {D});
  m->normb = up_f32(m, pre + "norm.bias", {D});
  // ---- DPT head
  const std::string hd = "depth_head.";
  const int F = c.features;
  for (int i = 0; i < 4; ++i) {
    const int Ci = c.out_channels[i];
    const std::string si = std::to_string(i);
    m->w_proj[i] = up_bf16(m, hd + "projects." + si + ".weight", {Ci, D, 1, 1});
    m->b_proj[i] = up_f32(m, hd + "projects." + si + ".bias", {Ci});
    if (i == 0 || i == 1) {
      const int ks = (i == 0) ? 4 : 2;
      const float* t = need(m, hd + "resize_layers." + si + ".weight", {Ci, Ci, ks, ks});
      const long long n = static_cast<long long>(ks) * ks * Ci * Ci;
      m->w_rs[i] = dev_alloc<__nv_bfloat16>(m, n);
      run_pack(t, nullptr, m->w_rs[i], n, PackDesc{PACK_CONVT, Ci, Ci, ks, 0});
      m->b_rs[i] = up_f32(m, hd + "resize_layers." + si + ".bias", {Ci});
    } else if (i == 3) {
      ADA_REQUIRE(Ci % kBlockK == 0, "resize_layers.3 expects C % 64 == 0");
      m->w_rs[i] = pack_conv3x3_dev(m, need(m, hd + "resize_layers.3.weight", {Ci, Ci, 3, 3}), Ci, Ci);
      m->b_rs[i] = up_f32(m, hd + "resize_layers.3.bias", {Ci});
    }
    if (c.input_projection) {
      m->ip[i] = up_conv3x3(m, hd + "input_projection." + si + ".0", Ci, Ci, true);
      m->ipln_w[i] = up_f32(m, hd + "input_projection." + si + ".1.weight", {Ci});
      m->ipln_b[i] = up_f32(m, hd + "input_projection." + si + ".1.bias", {Ci});
    }
    m->rn[i] = up_conv3x3(m, hd + "scratch.layer" + std::to_string(i + 1) + "_rn", F, Ci, false);
  }
  for (int k = 1; k <= 4; ++k) {
    const std::string r = hd + "scratch.refinenet" + std::to_string(k) + ".";
    RefineW& w = m->ref[k];
    w.rcu1c1 = up_conv3x3(m, r + "resConfUnit1.conv1", F, F, true);  // dead for refinenet4 (blocks.py:131-133) but loaded
    w.rcu1c2 = up_conv3x3(m, r + "resConfUnit1.conv2", F, F, true);
    w.rcu2c1 = up_conv3x3(m, r + "resConfUnit2.conv1", F, F, true);
    w.rcu2c2 = up_conv3x3(m, r + "resConfUnit2.conv2", F, F, true);
    w.wout = up_bf16(m, r + "out_conv.weight", {F, F, 1, 1});
    w.bout = up_f32(m, r + "out_conv.bias", {F});
  }
  m->oc1 = up_conv3x3(m, hd + "scratch.output_conv1", F / 2, F, true);
  {
    const float* t = need(m, hd + "scratch.output_conv2.0.weight", {32, F / 2, 3, 3});
    const long long n = 288LL * (F / 2);
    m->w_tail_taps = dev_alloc<__nv_bfloat16>(m, n);
    run_pack(t, nullptr, m->w_tail_taps, n, PackDesc{PACK_TAIL, F / 2, 0, 0, 0});
  }
  if ((F / 2) % 32 == 0 && F / 2 <= kTmMaxC) {
    const float* t = need(m, hd + "scratch.output_conv2.0.weight", {32, F / 2, 3, 3});
    const int n = 288 * (F / 2);
    m->w_tail_mma = dev_alloc<__half>(m, n);
    pack_tail_mma_kernel<<<(n + 255) / 256, 256>>>(t, m->w_tail_mma, F / 2);
    ADA_CHECK_CUDA(cudaGetLastError());
  }
  m->oc2 = up_conv3x3(m, hd + "scratch.output_conv2.0", 32, F / 2, true);
  {
    const std::vector<float> w2 = need_host(m, hd + "scratch.output_conv2.2.weight", {1, 32, 1, 1});
    const std::vector<float> b2 = need_host(m, hd + "scratch.output_conv2.2.bias", {1});
    float aux[33];
    for (int i = 0; i < 32; ++i) aux[i] = w2[i];
    aux[32] = b2[0];
    m->tail_aux = upload<float>(m, aux, sizeof(aux));
  }
  ADA_CHECK_CUDA(cudaDeviceSynchronize());  // the pack kernels read the staged tensors released next
  m->drop_staged();
  m->finalized = true;
}

static ada_model::PosCache& get_pos(ada_model* m, int gh, int gw) {
  auto key = std::make_pair(gh, gw);
  auto it = m->pos_cache.find(key);
  if (it != m->pos_cache.end()) return it->second;
  const int D = m->cfg.embed_dim, G = m->cfg.pos_grid;
  if (m->pos_cache.size() >= 16) {  // bounded: a sweep over many resolutions must not grow the cache without limit
    ADA_CHECK_CUDA(cudaDeviceSynchronize());  // an in-flight forward may still read an entry
    for (auto& kv : m->pos_cache) {
      cudaFree(kv.second.posb);
      cudaFree(kv.second.cls_pos);
    }
    m->pos_cache.clear();
  }
  std::vector<float> pp(static_cast<size_t>(gh) * gw * D);
  if (gh == G && gw == G) {  // dinov2.py:203-204: table used as is
    std::copy(m->pos_host.begin() + D, m->pos_host.end(), pp.begin());
  } else {
    interp_pos_host(m->pos_host.data() + D, G, D, gh, gw, m->cfg.interpolate_offset, pp.data());
  }
  for (size_t p = 0; p < static_cast<size_t>(gh) * gw; ++p)
    for (int d = 0; d < D; ++d) pp[p * D + d] += m->embed_bias[d];
  std::vector<float> cp(D);
  for (int d = 0; d < D; ++d) cp[d] = m->cls_host[d] + m->pos_host[d];
  ada_model::PosCache pc;
  ADA_CHECK_CUDA(cudaMalloc(&pc.posb, pp.size() * 4));
  ADA_CHECK_CUDA(cudaMemcpy(pc.posb, pp.data(), pp.size() * 4, cudaMemcpyHostToDevice));
  ADA_CHECK_CUDA(cudaMalloc(&pc.cls_pos, D * 4));
  ADA_CHECK_CUDA(cudaMemcpy(pc.cls_pos, cp.data(), D * 4, cudaMemcpyHostToDevice));
  return m->pos_cache[key] = pc;
}

// ---- workspace: one arena, bump-allocated, rebuilt when a larger (B,H,W) arrives
struct Bump {
  char* base;
  size_t off = 0;
  bool dry;
  template <typename T>
  T* take(size_t elems) {
    off = (off + 1023) & ~static_cast<size_t>(1023);
    T* p = dry ? nullptr : reinterpret_cast<T*>(base + off);
    off += elems * sizeof(T);
    return p;
  }
};

static int down2(int h) { return (h - 1) / 2 + 1; }
// fused tail (tap GEMM at low resolution + gather) needs the 8h -> 14h geometry; ADA_TAIL=0 selects the unfused path
// (upsample + implicit-GEMM conv with the EPI_TAIL epilogue), kept for A/B measurements
static bool tail_fused(int hl, int wl, int H, int W) {
  static const int tail_mode = env_int("ADA_TAIL", 1);
  return tail_mode == 1 && hl * 14 == H * 8 && wl * 14 == W * 8;
}

static size_t plan_workspace(ada_model* m, int B, int H, int W, bool dry, char* base) {
  const ada_config& c = m->cfg;
  const int D = c.embed_dim, F = c.features;
  const int gh = H / 14, gw = W / 14, P = gh * gw, N = P + 1;
  const size_t M = static_cast<size_t>(B) * N, BP = static_cast<size_t>(B) * P;
  Bump b{base, 0, dry};
  m->named.clear();
  m->named_is_f32.clear();
  auto reg = [&](const std::string& n, void* p, size_t elems, int f32) {
    m->named[n] = {p, elems};
    m->named_is_f32[n] = f32;
  };
  m->x = b.take<float>(M * D);
  m->xn = b.take<__nv_bfloat16>(M * D);
  m->qkv = b.take<__nv_bfloat16>(M * 3 * D);
  m->att = b.take<__nv_bfloat16>(M * D);
  m->hbuf = b.take<__nv_bfloat16>(M * c.ffn_hidden);
  m->ybuf = b.take<__nv_bfloat16>(M * D);
  m->ybuf2 = b.take<__nv_bfloat16>(M * D);
  m->a_embed = b.take<__nv_bfloat16>(BP * m->kpad);
  m->tokens_dbg = nullptr;
  if (m->capture) {  // test hook only (ada_set_capture re-plans the workspace)
    m->tokens_dbg = b.take<float>(M * D);
    reg("tokens", m->tokens_dbg, M * D, 1);
  }
  for (int i = 0; i < 4; ++i) {
    m->tap[i] = b.take<__nv_bfloat16>(BP * D);
    reg("tap" + std::to_string(i), m->tap[i], BP * D, 0);
  }
  const int sh[4] = {gh * 4, gh * 2, gh, down2(gh)}, sw[4] = {gw * 4, gw * 2, gw, down2(gw)};
  size_t maxpix = 0;
  for (int i = 0; i < 4; ++i) {
    const size_t pix = static_cast<size_t>(B) * sh[i] * sw[i];
    const int Ci = c.out_channels[i];
    maxpix = std::max(maxpix, pix);
    m->proj[i] = b.take<__nv_bfloat16>(BP * Ci);
    m->rs[i] = (i == 2) ? m->proj[i] : b.take<__nv_bfloat16>(pix * Ci);
    m->ipb[i] = c.input_projection ? b.take<__nv_bfloat16>(pix * Ci) : m->rs[i];  // un-guided head: layer_i = resize output
    m->rnb[i] = b.take<__nv_bfloat16>(pix * F);
    m->rnr[i] = b.take<__nv_bfloat16>(pix * F);
    reg("layer" + std::to_string(i + 1) + "_rn", m->rnb[i], pix * F, 0);
    reg("layer" + std::to_string(i + 1), m->ipb[i], pix * Ci, 0);
  }
  m->t1 = b.take<__nv_bfloat16>(maxpix * F);
  m->sum = b.take<__nv_bfloat16>(maxpix * F);
  m->sumr = b.take<__nv_bfloat16>(maxpix * F);
  m->r2 = b.take<__nv_bfloat16>(maxpix * F);
  m->ocb = b.take<__nv_bfloat16>(maxpix * F);
  // path_k lives at the resolution of level k-1 (path_1: 2x level 1)
  const int ph[5] = {0, sh[0] * 2, sh[0], sh[1], sh[2]}, pw[5] = {0, sw[0] * 2, sw[0], sw[1], sw[2]};
  for (int k = 1; k <= 4; ++k) {
    const size_t pix = static_cast<size_t>(B) * ph[k] * pw[k];
    m->path[k] = b.take<__nv_bfloat16>(pix * F);
    reg("path_" + std::to_string(k), m->path[k], pix * F, 0);
  }
  m->oc1b = b.take<__nv_bfloat16>(static_cast<size_t>(B) * ph[1] * pw[1] * (F / 2));
  // the [B,H,W,F/2] upsampled map only exists on the unfused tail path (ADA_TAIL=0); the default fused tail never
  // materialises it (2.2 GB at ViT-L, batch 32, 518^2)
  m->up = tail_fused(ph[1], pw[1], H, W) ? nullptr : b.take<__nv_bfloat16>(static_cast<size_t>(B) * H * W * (F / 2));
  m->vtap = b.take<__nv_bfloat16>(static_cast<size_t>(B) * ph[1] * pw[1] * 288);
  return b.off + 1024;
}

// Re-plans the arena when (B,H,W) changes. The previous forward may still be running in the OLD layout on `st` (any
// non-blocking stream; a ragged last batch of a streamed run): every re-plan first drains `st`, and the one-off memset of
// the patch matrix' K padding is ordered on `st` as well, so nothing of the new layout is touched before earlier work on
// the caller's stream has finished. A handle is driven from one stream at a time (include/amodal_b200.h). This is the only
// host synchronisation ada_forward ever performs, and only on the first call at a new shape.
static void ensure_workspace(ada_model* m, int B, int H, int W, cudaStream_t st) {
  if (B == m->wsB && H == m->wsH && W == m->wsW) return;
  m->drop_graph();  // a captured graph points into the old workspace layout
  ADA_CHECK_CUDA(cudaStreamSynchronize(st));
  const size_t need_bytes = plan_workspace(m, B, H, W, true, nullptr);
  if (need_bytes > m->arena.bytes) {
    if (m->arena.p) {
      ADA_CHECK_CUDA(cudaDeviceSynchronize());
      ADA_CHECK_CUDA(cudaFree(m->arena.p));
      m->arena.p = nullptr;
      m->arena.bytes = 0;
    }
    ADA_CHECK_CUDA(cudaMalloc(&m->arena.p, need_bytes));
    m->arena.bytes = need_bytes;
  }
  plan_workspace(m, B, H, W, false, static_cast<char*>(m->arena.p));
  // zero the K padding of the patch matrix once (the gather never writes it)
  ADA_CHECK_CUDA(cudaMemsetAsync(m->a_embed, 0, static_cast<size_t>(B) * (H / 14) * (W / 14) * m->kpad * 2, st));
  m->wsB = B;
  m->wsH = H;
  m->wsW = W;
}

// conv3x3 (pad 1, stride 1) over NHWC bf16 through the implicit-GEMM path
static void conv3x3(const __nv_bfloat16* in, int B, int H, int W, const ConvW& cw, int act, const __nv_bfloat16* r1,
                    const __nv_bfloat16* r2, __nv_bfloat16* out, __nv_bfloat16* out_relu, cudaStream_t st, int force_cg = 0,
                    int epi = EPI_BF16) {
  GemmLaunch L;
  L.force_cg = force_cg;
  L.A = in;
  L.Bw = cw.w;
  L.M = B * H * W;
  L.N = cw.cout;
  L.ldb = cw.ldw;
  L.a_mode = A_CONV3X3;
  L.batch = B;
  L.H = H;
  L.W = W;
  L.Cin = cw.cin;
  L.args.epi = epi;
  L.args.act = act;
  L.args.bias = cw.b;
  L.args.resid1 = r1;
  L.args.resid2 = r2;
  L.args.out_bf16 = out;
  L.out_relu = out_relu;
  L.args.ldo = cw.cout;
  launch_gemm(L, st);
}

static void linear(const __nv_bfloat16* A, int M, int K, int lda, const __nv_bfloat16* Wt, int N, int ldb,
                   const GemmArgs& epi, cudaStream_t st) {
  GemmLaunch L;
  L.A = A;
  L.Bw = Wt;
  L.M = M;
  L.N = N;
  L.K = K;
  L.lda = lda;
  L.ldb = ldb;
  L.args = epi;
  launch_gemm(L, st);
}

static void forward_body(ada_model* m, const float* rgb, const float* const* guides, const int* guide_ch, int n_guides,
                         float* out, int B, int H, int W, cudaStream_t st) {
  require_device();
  if (!m->finalized) throw AdaError(ADA_ESTATE, "ada_forward before ada_finalize");
  ADA_REQUIRE(device_info().device == m->device, "ada_forward: the handle was created on device " + std::to_string(m->device) +
                                                     " but device " + std::to_string(device_info().device) + " is current");
  ADA_REQUIRE(B > 0 && H > 0 && W > 0, "B, H, W must be positive");
  ADA_REQUIRE(H % 14 == 0, "Input image height is not a multiple of patch height 14");
  ADA_REQUIRE(W % 14 == 0, "Input image width is not a multiple of patch width 14");
  int cg = 0;
  for (int i = 0; i < n_guides; ++i) cg += guide_ch[i];
  ADA_REQUIRE(cg == m->cfg.guide_channels, "guide channels do not match guide_type");
  const ada_config& c = m->cfg;
  const int D = c.embed_dim, F = c.features, heads = c.num_heads;
  const int gh = H / 14, gw = W / 14, P = gh * gw, N = P + 1;
  const int M = B * N, BP = B * P;
  ensure_workspace(m, B, H, W, st);
  ada_model::PosCache& pc = get_pos(m, gh, gw);
  g_launches = 0;
  pdl_select(static_cast<long long>(M));
  struct ProfGuard {
    ProfGuard(Profiler* p) { g_prof = p; }
    ~ProfGuard() { g_prof = nullptr; }
  } prof_guard(m->profile ? &m->prof : nullptr);

  // ---- tokens: patch gather -> embed GEMM (+bias +pos) ; cls rows     (dav2.py:65-76, dinov2.py:232-246)
  launch_patch_gather(rgb, guides, guide_ch, n_guides, m->a_embed, B, H, W, m->kpad, c.normalize_input, st);
  cls_rows_kernel<<<(B * D + 255) / 256, 256, 0, st>>>(pc.cls_pos, m->x, B, N, D);
  ADA_CHECK_CUDA(cudaGetLastError());
  ++g_launches;
  {
    GemmArgs e{};
    e.epi = EPI_EMBED;
    e.aux = pc.posb;
    e.out_f32 = m->x;
    e.ldo = D;
    e.P = P;
    linear(m->a_embed, BP, m->kpad, m->kpad, m->w_embed, D, m->kpad, e, st);
  }
  if (m->capture)
    ADA_CHECK_CUDA(cudaMemcpyAsync(m->tokens_dbg, m->x, static_cast<size_t>(M) * D * 4, cudaMemcpyDeviceToDevice, st));

  // ---- encoder blocks (block.py:82-107 eval branch). The fp32 stream x is only touched by the LayerNorm kernel:
  //      default: the attention branch leaves gamma1 * (W h + b) in `ybuf` and the MLP branch gamma2 * (...) in `ybuf2`
  //      (bf16); norm2 normalises x + ybuf without storing it, the NEXT block's norm1 (or the tap norm) adds both and
  //      norm1 stores x <- (x + ybuf) + ybuf2 (block.py:105-106): one fp32 write of the stream per block, all of it in the
  //      coalesced LayerNorm kernel.
  //      ADA_RESID_EPI=1: x is instead updated in place by the proj / fc2 GEMM epilogues (EPI_RESID_F32, x tiles staged
  //      through TMA) and the LayerNorm kernels only read x. Measured on the same box (batch 32): LayerNorm 4.4 -> 2.45 ms
  //      but fc2 6.2 -> 7.25 ms and proj 1.9 -> 2.6 ms (the fp32 staging costs pipeline stages and the GEMMs then carry
  //      the stream's HBM traffic): 658 vs 665 img/s, so it stays off.
  static const int resid_epi = env_int("ADA_RESID_EPI", 0);
  int tap_i = 0;
  int pending_tap = -1;  // tap whose LayerNorm rides on the next block's norm1
  const __nv_bfloat16 *pend1 = nullptr, *pend2 = nullptr;  // residual-branch outputs not yet added to x
  for (int i = 0; i < c.depth; ++i) {
    const BlockW& w = m->blocks[i];
    // norm1; if the previous block was tapped, the same pass also emits its tap (shared final norm, cls dropped, NHWC):
    // identical input, identical statistics, only the affine differs (dinov2.py:337-340)
    launch_layernorm(m->x, pend1, pend2, w.ln1w, w.ln1b, m->xn, M, D, 1e-6f, N, 0, pend1 != nullptr, st,
                     pending_tap >= 0 ? m->normw : nullptr, pending_tap >= 0 ? m->normb : nullptr,
                     pending_tap >= 0 ? m->tap[pending_tap] : nullptr);
    pending_tap = -1;
    {
      GemmArgs e{};
      e.epi = EPI_BF16;
      e.bias = w.bqkv;
      e.out_bf16 = m->qkv;
      e.ldo = 3 * D;
      linear(m->xn, M, D, D, w.wqkv, 3 * D, D, e, st);
    }
    launch_attention(m->qkv, m->att, B, N, heads, st);
    {
      GemmArgs e{};
      e.bias = w.bproj;
      e.gamma = w.g1;
      e.ldo = D;
      if (resid_epi) {
        e.epi = EPI_RESID_F32;  // x += gamma1 * (att W^T + b), in place through TMA (block.py:105)
        e.out_f32 = m->x;
      } else {
        e.epi = EPI_BF16;
        e.out_bf16 = m->ybuf;
      }
      linear(m->att, M, D, D, w.wproj, D, D, e, st);
    }
    launch_layernorm(m->x, resid_epi ? nullptr : m->ybuf, nullptr, w.ln2w, w.ln2b, m->xn, M, D, 1e-6f, N, 0, 0, st);
    const int Hd = c.ffn_hidden;
    {
      GemmArgs e{};
      e.bias = w.b1;
      e.out_bf16 = m->hbuf;
      e.ldo = Hd;
      if (c.ffn_kind == 0) {
        e.epi = EPI_BF16;
        e.act = ACT_GELU;
        linear(m->xn, M, D, D, w.w1, Hd, D, e, st);
      } else {
        e.epi = EPI_SWIGLU;
        linear(m->xn, M, D, D, w.w1, 2 * Hd, D, e, st);
      }
    }
    {
      GemmArgs e{};
      e.bias = w.b2;
      e.gamma = w.g2;
      e.ldo = D;
      if (resid_epi) {
        e.epi = EPI_RESID_F32;  // x += gamma2 * (h W^T + b) (block.py:106)
        e.out_f32 = m->x;
      } else {
        e.epi = EPI_BF16;
        e.out_bf16 = m->ybuf2;
      }
      linear(m->hbuf, M, Hd, Hd, w.w2, D, Hd, e, st);
    }
    if (!resid_epi) {
      pend1 = m->ybuf;
      pend2 = m->ybuf2;
    }
    if (tap_i < 4 && i == c.taps[tap_i]) {
      // shared final norm of x (+ both pending branches), cls dropped, NHWC patch map (dinov2.py:337-340). Fused into the
      // next block's norm1 when there is one (and the residual epilogue variant is off: then x is already complete);
      // after the last block it is a pass of its own, and x is not written back.
      if (i + 1 < c.depth && !resid_epi)
        pending_tap = tap_i;
      else
        launch_layernorm(m->x, pend1, pend2, m->normw, m->normb, m->tap[tap_i], M, D, 1e-6f, N, 1, 0, st);
      ++tap_i;
    }
  }
  if (tap_i != 4) throw AdaError(ADA_EINVAL, "taps must be increasing block indices < depth");

  // ---- DPT head (dpt.py:161-197)
  const int sh[4] = {gh * 4, gh * 2, gh, down2(gh)}, sw[4] = {gw * 4, gw * 2, gw, down2(gw)};
  for (int i = 0; i < 4; ++i) {
    const int Ci = c.out_channels[i];
    {  // projects[i]: 1x1 conv D -> C_i (dpt.py:172)
      GemmArgs e{};
      e.epi = EPI_BF16;
      e.bias = m->b_proj[i];
      e.out_bf16 = m->proj[i];
      e.ldo = Ci;
      linear(m->tap[i], BP, D, D, m->w_proj[i], Ci, D, e, st);
    }
    if (i == 0 || i == 1) {  // ConvTranspose k == s (dpt.py:89-100): GEMM + pixel-shuffle scatter
      const int ks = (i == 0) ? 4 : 2;
      GemmArgs e{};
      e.epi = EPI_CONVT;
      e.bias = m->b_rs[i];
      e.out_bf16 = m->rs[i];
      e.H = gh;
      e.W = gw;
      e.ks = ks;
      e.cout = Ci;
      if (Ci % 64 == 0) {  // pixel-tile A operand: the pixel shuffle goes out through TMA boxes
        GemmLaunch L;
        L.A = m->proj[i];
        L.Bw = m->w_rs[i];
        L.M = BP;
        L.N = ks * ks * Ci;
        L.ldb = Ci;
        L.a_mode = A_CONV3X3;
        L.conv_taps = 1;
        L.batch = B;
        L.H = gh;
        L.W = gw;
        L.Cin = Ci;
        L.args = e;
        launch_gemm(L, st);
      } else {
        linear(m->proj[i], BP, Ci, Ci, m->w_rs[i], ks * ks * Ci, Ci, e, st);
      }
    } else if (i == 3) {  // conv 3x3 stride 2 (dpt.py:102-107): implicit GEMM, the tensor map walks the input with stride 2
      GemmLaunch L;
      L.A = m->proj[3];
      L.Bw = m->w_rs[3];
      L.M = B * sh[3] * sw[3];
      L.N = Ci;
      L.ldb = 9 * round_up(Ci, kBlockK);
      L.a_mode = A_CONV3X3;
      L.batch = B;
      L.H = sh[3];
      L.W = sw[3];
      L.Hin = gh;
      L.Win = gw;
      L.conv_stride = 2;
      L.Cin = Ci;
      L.args.epi = EPI_BF16;
      L.args.bias = m->b_rs[3];
      L.args.out_bf16 = m->rs[3];
      L.args.ldo = Ci;
      launch_gemm(L, st);
    }
    if (c.input_projection) {  // input_projection[i]: conv3x3 + channel LN + ReLU (dpt.py:153-159,178-179)
      static const int chln_epi = env_int("ADA_CHLN_EPI", 1);
      if (chln_epi && Ci <= 256) {  // all channels of a pixel in one accumulator tile: LayerNorm + ReLU in the conv epilogue
        GemmLaunch L;
        L.A = m->rs[i];
        L.Bw = m->ip[i].w;
        L.M = B * sh[i] * sw[i];
        L.N = Ci;
        L.ldb = m->ip[i].ldw;
        L.a_mode = A_CONV3X3;
        L.batch = B;
        L.H = sh[i];
        L.W = sw[i];
        L.Cin = Ci;
        L.args.epi = EPI_BF16_CHLN;
        L.args.bias = m->ip[i].b;
        L.args.gamma = m->ipln_w[i];
        L.args.aux = m->ipln_b[i];
        L.args.out_bf16 = m->ipb[i];
        L.args.ldo = Ci;
        launch_gemm(L, st);
      } else {
        conv3x3(m->rs[i], B, sh[i], sw[i], m->ip[i], ACT_NONE, nullptr, nullptr, m->ipb[i], nullptr, st);
        launch_channel_ln_relu(m->ipb[i], m->ipln_w[i], m->ipln_b[i], m->ipb[i], static_cast<long long>(B) * sh[i] * sw[i],
                               Ci, 1e-6f, st);
      }
    }
    // layer{i}_rn: conv3x3 C_i -> F, no bias (blocks.py:20-24); keep x and relu(x) for the residual units
    conv3x3(m->ipb[i], B, sh[i], sw[i], m->rn[i], ACT_NONE, nullptr, nullptr, m->rnb[i], m->rnr[i], st);
  }
  // refinenet4..1 (blocks.py:123-148). out_conv (1x1) commutes with the bilinear resize, so it runs at low resolution.
  const int ph[5] = {0, sh[0] * 2, sh[0], sh[1], sh[2]}, pw[5] = {0, sw[0] * 2, sw[0], sw[1], sw[2]};
  for (int k = 4; k >= 1; --k) {
    const int lv = k - 1;  // pyramid level of this block's input
    const int hh = sh[lv], ww = sw[lv];
    const RefineW& rw = m->ref[k];
    const __nv_bfloat16 *xin, *xin_relu;
    if (k == 4) {
      xin = m->rnb[3];
      xin_relu = m->rnr[3];
    } else {
      // output = path_{k+1} + RCU1(layer_k_rn)
      conv3x3(m->rnr[lv], B, hh, ww, rw.rcu1c1, ACT_RELU, nullptr, nullptr, m->t1, nullptr, st);
      conv3x3(m->t1, B, hh, ww, rw.rcu1c2, ACT_NONE, m->rnb[lv], m->path[k + 1], m->sum, m->sumr, st);
      xin = m->sum;
      xin_relu = m->sumr;
    }
    conv3x3(xin_relu, B, hh, ww, rw.rcu2c1, ACT_RELU, nullptr, nullptr, m->t1, nullptr, st);
    conv3x3(m->t1, B, hh, ww, rw.rcu2c2, ACT_NONE, xin, nullptr, m->r2, nullptr, st);
    {
      GemmArgs e{};
      e.epi = EPI_BF16;
      e.bias = rw.bout;
      e.out_bf16 = m->ocb;
      e.ldo = F;
      linear(m->r2, B * hh * ww, F, F, rw.wout, F, F, e, st);
    }
    launch_upsample(m->ocb, m->path[k], B, hh, ww, ph[k], pw[k], F, st);
  }
  // output_conv1 -> bilinear to (H, W) -> output_conv2 (conv3x3 + ReLU + 1x1 + Sigmoid) (dpt.py:193-195)
  static const int oc1_cg = env_int("ADA_OC1_CG", 0);
  // tail_mma_kernel (upsample + output_conv2 on tensor cores, one kernel) wherever its geometry and channel count allow;
  // ADA_TAIL_MMA=0 selects the older tap-GEMM + gather pair, which also serves F/2 > 128 (ViT-G heads)
  static const int tail_mma_env = env_int("ADA_TAIL_MMA", 1);
  const bool tail_mma = tail_mma_env && m->w_tail_mma != nullptr && tail_mma_supported(F / 2, ph[1], pw[1], H, W) &&
                        tail_fused(ph[1], pw[1], H, W);
  conv3x3(m->path[1], B, ph[1], pw[1], m->oc1, ACT_NONE, nullptr, nullptr, m->oc1b, nullptr, st, oc1_cg,
          tail_mma ? EPI_F16 : EPI_BF16);
  if (tail_mma) {
    launch_tail_mma(reinterpret_cast<const __half*>(m->oc1b), m->w_tail_mma, m->oc2.b, m->tail_aux, out, B, ph[1], pw[1], H, W,
                    F / 2, c.sigmoid, st);
  } else if (tail_fused(ph[1], pw[1], H, W)) {
    GemmArgs e{};
    e.epi = EPI_F16;  // the tap map is stored as fp16 (tail_gather_kernel interpolates it with packed fp16 FMAs)
    e.out_bf16 = m->vtap;
    e.ldo = 288;
    {
      // N = 288: three 128-wide column tiles (auto). Forcing 256 (two tiles, the second mostly padding) measured slower
      // (1.21 vs 0.95 ms at batch 32); ADA_TAIL_BN overrides for experiments.
      static const int tail_bn = env_int("ADA_TAIL_BN", 0);
      GemmLaunch L;
      L.A = m->oc1b;
      L.Bw = m->w_tail_taps;
      L.M = B * ph[1] * pw[1];
      L.N = 288;
      L.K = F / 2;
      L.lda = F / 2;
      L.ldb = F / 2;
      L.args = e;
      L.force_bn = tail_bn;
      launch_gemm(L, st);
    }
    launch_tail_gather(reinterpret_cast<const __half*>(m->vtap), m->oc2.b, m->tail_aux, out, B, ph[1], pw[1], H, W, c.sigmoid, st);
  } else {
    launch_upsample(m->oc1b, m->up, B, ph[1], pw[1], H, W, F / 2, st);
    GemmLaunch L;
    L.A = m->up;
    L.Bw = m->oc2.w;
    L.M = B * H * W;
    L.N = 32;
    L.ldb = m->oc2.ldw;
    L.a_mode = A_CONV3X3;
    L.batch = B;
    L.H = H;
    L.W = W;
    L.Cin = F / 2;
    L.args.epi = EPI_TAIL;
    L.args.bias = m->oc2.b;
    L.args.aux = m->tail_aux;
    L.args.out_f32 = out;
    L.args.sigmoid = c.sigmoid;
    launch_gemm(L, st);
  }
  m->last_B = B;
  m->last_H = H;
  m->last_W = W;
  m->last_launches = g_launches;
}

// ada_forward: eager launches, or (ada_set_graph) replay of a captured graph over staging buffers.
static void forward_impl(ada_model* m, const float* rgb, const float* const* guides, const int* guide_ch, int n_guides,
                         float* out, int B, int H, int W, cudaStream_t st) {
  if (!m->graph_on || m->profile || m->capture) {
    forward_body(m, rgb, guides, guide_ch, n_guides, out, B, H, W, st);
    return;
  }
  const bool same_shape = (B == m->wsB && H == m->wsH && W == m->wsW);
  if (!same_shape || m->graph_state == 0) {  // first forward at this shape runs eagerly: workspace, position cache, attrs
    forward_body(m, rgb, guides, guide_ch, n_guides, out, B, H, W, st);
    m->graph_state = 1;
    return;
  }
  const size_t plane = static_cast<size_t>(B) * H * W * sizeof(float);
  if (m->graph_state == 1) {
    ADA_REQUIRE(n_guides >= 0 && n_guides <= 3, "at most 3 guide tensors");
    // Any failure below (an allocation, the capture, the instantiation) releases everything acquired so far through
    // drop_graph(), so a later call starts from a clean state instead of leaking the staging buffers.
    bool capturing = false;
    try {
      if (!m->cap_stream) ADA_CHECK_CUDA(cudaStreamCreateWithFlags(&m->cap_stream, cudaStreamNonBlocking));
      ADA_CHECK_CUDA(cudaMalloc(&m->g_rgb, 3 * plane));
      ADA_CHECK_CUDA(cudaMalloc(&m->g_out, plane));
      m->g_nguides = n_guides;
      for (int i = 0; i < n_guides; ++i) {
        m->g_guide_ch[i] = guide_ch[i];
        ADA_CHECK_CUDA(cudaMalloc(&m->g_guides[i], guide_ch[i] * plane));
      }
      // capture on a private stream (the caller's may be the legacy default stream, which cannot be captured)
      ADA_CHECK_CUDA(cudaStreamBeginCapture(m->cap_stream, cudaStreamCaptureModeThreadLocal));
      capturing = true;
      forward_body(m, m->g_rgb, m->g_guides, m->g_guide_ch, n_guides, m->g_out, B, H, W, m->cap_stream);
      capturing = false;
      ADA_CHECK_CUDA(cudaStreamEndCapture(m->cap_stream, &m->graph));
      ADA_CHECK_CUDA(cudaGraphInstantiate(&m->graph_exec, m->graph, 0));
    } catch (...) {
      if (capturing) {
        cudaGraph_t dead = nullptr;
        cudaStreamEndCapture(m->cap_stream, &dead);
        if (dead) cudaGraphDestroy(dead);
      }
      cudaGetLastError();
      m->drop_graph();
      throw;
    }
    m->graph_state = 2;
  }
  ADA_REQUIRE(n_guides == m->g_nguides, "guide tensors differ from the captured call");
  for (int i = 0; i < n_guides; ++i) ADA_REQUIRE(guide_ch[i] == m->g_guide_ch[i], "guide channels differ from the captured call");
  ADA_CHECK_CUDA(cudaMemcpyAsync(m->g_rgb, rgb, 3 * plane, cudaMemcpyDeviceToDevice, st));
  for (int i = 0; i < n_guides; ++i)
    ADA_CHECK_CUDA(cudaMemcpyAsync(m->g_guides[i], guides[i], guide_ch[i] * plane, cudaMemcpyDeviceToDevice, st));
  ADA_CHECK_CUDA(cudaGraphLaunch(m->graph_exec, st));
  ADA_CHECK_CUDA(cudaMemcpyAsync(out, m->g_out, plane, cudaMemcpyDeviceToDevice, st));
}

__global__ void bf16_to_f32_kernel(const __nv_bfloat16* in, float* out, long long n) {
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i < n) out[i] = __bfloat162float(in[i]);
}

template <typename F>
static int guarded(F&& f) {
  try {
    f();
    return ADA_OK;
  } catch (const AdaError& e) {
    g_last_error = e.what();
    return e.code;
  } catch (const std::exception& e) {
    g_last_error = e.what();
    return ADA_EINVAL;
  } catch (...) {
    g_last_error = "unknown error";
    return ADA_EINVAL;
  }
}

}  // namespace ada

// =================================================================================================== C ABI
extern "C" {

const char* ada_last_error(void) { return g_last_error.c_str(); }

int ada_debug_timeline(long long* out, int32_t n) {
  return guarded([&] {
    ADA_REQUIRE(out && n > 0 && n <= 512, "bad argument");
#ifdef ADA_BRINGUP
    ADA_CHECK_CUDA(cudaDeviceSynchronize());
    ADA_CHECK_CUDA(cudaMemcpyFromSymbol(out, g_dev_timeline, sizeof(long long) * n));
#else
    throw AdaError(ADA_ESTATE, "ada_debug_timeline: this library was built without -DADA_BRINGUP (no instrumented kernels)");
#endif
  });
}

int ada_device_error(uint32_t out[4]) {
  return guarded([&] { ADA_CHECK_CUDA(cudaMemcpyFromSymbol(out, g_dev_error, 16)); });
}

int ada_create(const ada_config* cfg, ada_handle* out) {
  return guarded([&] {
    ADA_REQUIRE(cfg && out, "null argument");
    ADA_REQUIRE(cfg->embed_dim == cfg->num_heads * 64, "head_dim must be 64");
    ADA_REQUIRE(cfg->embed_dim % 128 == 0, "embed_dim % 128");
    ADA_REQUIRE(cfg->features % 16 == 0 && cfg->features >= 64, "features must be a multiple of 16, >= 64");
    ADA_REQUIRE(cfg->guide_channels >= 0 && cfg->guide_channels <= 5, "guide_channels in [0,5]");
    ADA_REQUIRE(cfg->sigmoid >= 0 && cfg->sigmoid <= 2, "sigmoid (final activation) in {0: none, 1: sigmoid, 2: relu}");
    ADA_REQUIRE((cfg->input_projection | 1) == 1 && (cfg->normalize_input | 1) == 1, "input_projection / normalize_input are flags");
    for (int i = 0; i < 4; ++i) ADA_REQUIRE(cfg->out_channels[i] % 8 == 0, "out_channels % 8");
    ADA_REQUIRE(cfg->depth > 0 && cfg->depth <= 64 && cfg->ffn_hidden % 64 == 0 && cfg->pos_grid > 0, "bad depth / ffn_hidden / pos_grid");
    ADA_REQUIRE(cfg->ffn_kind == 0 || cfg->ffn_kind == 1, "ffn_kind is 0 (Mlp) or 1 (SwiGLU)");
    ada_model* m = new ada_model();
    m->cfg = *cfg;
    m->spec = expected_weights(*cfg);
    if (cudaGetDevice(&m->device) != cudaSuccess) {  // no device: weights can still be staged, finalize / forward will fail
      cudaGetLastError();
      m->device = -1;
    }
    *out = m;
  });
}

int ada_set_weight(ada_handle h, const char* key, const float* data, const int64_t* shape, int32_t ndim) {
  return guarded([&] {
    ADA_REQUIRE(h && key && data && shape && ndim >= 0 && ndim <= 8, "bad argument");
    if (h->finalized) throw AdaError(ADA_ESTATE, "ada_set_weight after ada_finalize");
    auto sp = h->spec.find(key);
    if (sp == h->spec.end())
      throw AdaError(ADA_EINVAL, std::string("ada_set_weight: unknown weight key for this architecture: ") + key);
    StagedTensor t;
    size_t n = 1;
    for (int i = 0; i < ndim; ++i) {
      t.shape.push_back(shape[i]);
      n *= static_cast<size_t>(shape[i]);
    }
    if (t.shape != sp->second) {
      std::string msg = std::string("ada_set_weight: shape mismatch for ") + key + ": got [";
      for (auto v : t.shape) msg += std::to_string(v) + ",";
      msg += "] expected [";
      for (auto v : sp->second) msg += std::to_string(v) + ",";
      throw AdaError(ADA_EINVAL, msg + "]");
    }
    t.n = n;
    cudaPointerAttributes attr;
    bool on_device = false;
    if (cudaPointerGetAttributes(&attr, data) == cudaSuccess) on_device = (attr.type == cudaMemoryTypeDevice);
    cudaGetLastError();
    auto old = h->host.find(key);
    if (old != h->host.end() && old->second.dev) cudaFree(old->second.dev);
    if (on_device) {  // stays on the device: one device-to-device copy, packed by kernels in ada_finalize
      ADA_CHECK_CUDA(cudaMalloc(&t.dev, std::max<size_t>(n * 4, 16)));
      ADA_CHECK_CUDA(cudaMemcpyAsync(t.dev, data, n * 4, cudaMemcpyDeviceToDevice, nullptr));
      ADA_CHECK_CUDA(cudaStreamSynchronize(nullptr));  // the caller may release `data` as soon as this returns
    } else {
      t.host.assign(data, data + n);
    }
    h->host[key] = std::move(t);
  });
}

int ada_finalize(ada_handle h) {
  return guarded([&] {
    ADA_REQUIRE(h, "null handle");
    if (h->finalized) throw AdaError(ADA_ESTATE, "already finalized");
    finalize_model(h);
  });
}

int ada_forward(ada_handle h, const float* rgb, const float* const* guides, const int32_t* guide_ch, int32_t n_guides,
                float* out, int32_t B, int32_t H, int32_t W, void* stream) {
  return guarded([&] {
    ADA_REQUIRE(h && rgb && out, "null argument");
    forward_impl(h, rgb, guides, guide_ch, n_guides, out, B, H, W, static_cast<cudaStream_t>(stream));
  });
}

size_t ada_workspace_bytes(ada_handle h) { return h ? h->arena.bytes : 0; }

int ada_launch_count(ada_handle h, int32_t B, int32_t H, int32_t W) {
  // counted while launching: exact for the shape of the last forward, 0 before the first one
  if (!h) return -1;
  if (h->last_launches > 0 && (B <= 0 || (B == h->last_B && H == h->last_H && W == h->last_W))) return h->last_launches;
  return 0;
}

int ada_set_graph(ada_handle h, int32_t on) {
  if (!h) return ADA_EINVAL;
  h->graph_on = on != 0;
  if (!h->graph_on) h->drop_graph();
  return ADA_OK;
}

int ada_set_capture(ada_handle h, int32_t on) {
  if (!h) return ADA_EINVAL;
  if (h->capture != (on != 0)) h->wsB = 0;  // the "tokens" copy is only planned while capturing: force a re-plan
  h->capture = on != 0;
  return ADA_OK;
}

int ada_read_intermediate(ada_handle h, const char* name, float* dst, int64_t count) {
  return guarded([&] {
    ADA_REQUIRE(h && name && dst, "null argument");
    auto it = h->named.find(name);
    ADA_REQUIRE(it != h->named.end(), std::string("unknown intermediate: ") + name);
    ADA_REQUIRE(static_cast<size_t>(count) == it->second.second,
                std::string(name) + " has " + std::to_string(it->second.second) + " elements");
    cudaPointerAttributes attr;
    bool dst_dev = false;
    if (cudaPointerGetAttributes(&attr, dst) == cudaSuccess) dst_dev = (attr.type == cudaMemoryTypeDevice);
    cudaGetLastError();
    float* tmp = dst;
    if (!dst_dev) ADA_CHECK_CUDA(cudaMalloc(&tmp, count * 4));
    if (h->named_is_f32[name]) {
      ADA_CHECK_CUDA(cudaMemcpy(tmp, it->second.first, count * 4, cudaMemcpyDeviceToDevice));
    } else {
      bf16_to_f32_kernel<<<static_cast<unsigned>((count + 255) / 256), 256>>>(
          static_cast<const __nv_bfloat16*>(it->second.first), tmp, count);
      ADA_CHECK_CUDA(cudaGetLastError());
    }
    ADA_CHECK_CUDA(cudaDeviceSynchronize());
    if (!dst_dev) {
      ADA_CHECK_CUDA(cudaMemcpy(dst, tmp, count * 4, cudaMemcpyDeviceToHost));
      cudaFree(tmp);
    }
  });
}

int ada_set_profile(ada_handle h, int32_t on) {
  if (!h) return ADA_EINVAL;
  h->profile = on != 0;
  return ADA_OK;
}

int ada_profile_records(ada_handle h, int32_t max_recs, int32_t* meta, double* ms) {
  if (!h || !meta || !ms) return ADA_EINVAL;
  if (cudaDeviceSynchronize() != cudaSuccess) return ADA_ECUDA;
  int n = 0;
  for (ProfRec& r : h->prof.recs) {
    if (n >= max_recs) break;
    float t = 0.f;
    if (cudaEventElapsedTime(&t, r.a, r.b) != cudaSuccess) return ADA_ECUDA;
    meta[5 * n + 0] = r.cls;
    meta[5 * n + 1] = r.m;
    meta[5 * n + 2] = r.n;
    meta[5 * n + 3] = r.k;
    meta[5 * n + 4] = r.tag;
    ms[n] = t;
    ++n;
  }
  return n;
}

int ada_profile_read(ada_handle h, int32_t n_classes, double* ms, double* flops, double* bytes, int32_t* launches) {
  return guarded([&] {
    ADA_REQUIRE(h && ms && flops && bytes && launches && n_classes >= PC_COUNT, "bad argument");
    for (int i = 0; i < n_classes; ++i) ms[i] = flops[i] = bytes[i] = 0.0, launches[i] = 0;
    ADA_CHECK_CUDA(cudaDeviceSynchronize());
    for (ProfRec& r : h->prof.recs) {
      float t = 0.f;
      ADA_CHECK_CUDA(cudaEventElapsedTime(&t, r.a, r.b));
      ms[r.cls] += t;
      flops[r.cls] += r.flops;
      bytes[r.cls] += r.bytes;
      launches[r.cls] += 1;
      cudaEventDestroy(r.a);
      cudaEventDestroy(r.b);
    }
    h->prof.recs.clear();
  });
}

void ada_destroy(ada_handle h) { delete h; }

int ada_interp_pos_embed_host(const float* pos_patch, int32_t grid, int32_t D, int32_t gh, int32_t gw, float offset,
                              float* out) {
  return guarded([&] {
    ADA_REQUIRE(pos_patch && out && grid > 0 && D > 0 && gh > 0 && gw > 0, "bad argument");
    interp_pos_host(pos_patch, grid, D, gh, gw, offset, out);
  });
}

int ada_conv_tile_shape(int32_t B, int32_t H, int32_t W, int32_t pair, int64_t out[4]) {
  return guarded([&] {
    ADA_REQUIRE(out && B > 0 && H > 0 && W > 0 && (pair == 1 || pair == 2), "bad argument");
    const TileGeo g = pick_tile_geo(B, H, W, pair, true);
    out[0] = g.lw;
    out[1] = g.lh;
    out[2] = g.lb;
    out[3] = g.padded;
  });
}

// ---- operator level
int ada_op_gemm(const ada_gemm_desc* d, void* stream) {
  return guarded([&] {
    require_device();
    ADA_REQUIRE(d && d->A && d->Bw, "null argument");
    GemmLaunch L;
    L.A = d->A;
    L.Bw = d->Bw;
    L.M = d->M;
    L.N = d->N;
    L.K = d->K;
    L.lda = d->lda;
    L.ldb = d->ldb;
    L.a_mode = d->a_mode;
    L.batch = d->batch;
    L.H = d->H;
    L.W = d->W;
    L.Cin = d->Cin;
    L.force_bn = d->force_bn;
    L.force_cg = d->force_cg;
    if (d->a_mode == A_CONV3X3 && d->conv_taps == 1) L.conv_taps = 1;  // pointwise on pixel tiles (EPI_CONVT through TMA boxes)
    if (d->a_mode == A_CONV3X3 && d->conv_stride == 2) {  // H, W of the descriptor are the INPUT map
      L.conv_stride = 2;
      L.Hin = d->H;
      L.Win = d->W;
      L.H = (d->H - 1) / 2 + 1;
      L.W = (d->W - 1) / 2 + 1;
      L.M = d->batch * L.H * L.W;
    }
    GemmArgs& e = L.args;
    e.epi = d->epi;
    e.act = d->act;
    e.bias = d->bias;
    e.gamma = d->gamma;
    e.out_f32 = d->out_f32;
    e.out_bf16 = static_cast<__nv_bfloat16*>(d->out_bf16);
    L.out_relu = static_cast<__nv_bfloat16*>(d->out_relu);
    e.resid1 = static_cast<const __nv_bfloat16*>(d->resid1);
    e.resid2 = static_cast<const __nv_bfloat16*>(d->resid2);
    e.aux = d->aux;
    e.ldo = d->ldo;
    e.P = d->P;
    e.ks = d->ks;
    e.cout = d->cout;
    e.sigmoid = d->sigmoid;
    if (d->epi == EPI_CONVT) {
      e.H = d->H;
      e.W = d->W;
    }
    launch_gemm(L, static_cast<cudaStream_t>(stream));
  });
}

int ada_op_layernorm(float* x, const void* delta_bf16, const void* delta2_bf16, const float* w, const float* b,
                     void* out_bf16, int32_t rows, int32_t D, float eps, int32_t n_tok, int32_t drop_cls, int32_t write_x,
                     const float* w2, const float* b2, void* out2_bf16, void* stream) {
  return guarded([&] {
    require_device();
    launch_layernorm(x, static_cast<const __nv_bfloat16*>(delta_bf16), static_cast<const __nv_bfloat16*>(delta2_bf16), w, b,
                     static_cast<__nv_bfloat16*>(out_bf16), rows, D, eps, n_tok, drop_cls, write_x,
                     static_cast<cudaStream_t>(stream), w2, b2, static_cast<__nv_bfloat16*>(out2_bf16));
  });
}

// ---- pre/post-processing of infer.py (SURVEY.md section 8 row f2): the single-image entry points launch the batched
// kernels with B = 1 and no descriptor table
int ada_pre_image_nearest(const uint8_t* img_hwc, int32_t H0, int32_t W0, float* out_chw, int32_t H, int32_t W,
                          int32_t normalize, void* stream) {
  return guarded([&] {
    require_device();
    ADA_REQUIRE(img_hwc && out_chw && H0 > 0 && W0 > 0 && H > 0 && W > 0, "bad argument");
    image_nearest_kernel<<<dim3((H * W + 255) / 256, 1), 256, 0, static_cast<cudaStream_t>(stream)>>>(
        img_hwc, nullptr, H0, W0, out_chw, H, W, normalize);
    ADA_CHECK_CUDA(cudaGetLastError());
  });
}

int ada_pre_mask_nearest(const uint8_t* mask, int32_t H0, int32_t W0, float* mask01, float* guide, int32_t H, int32_t W,
                         void* stream) {
  return guarded([&] {
    require_device();
    ADA_REQUIRE(mask && (mask01 || guide) && H0 > 0 && W0 > 0 && H > 0 && W > 0, "bad argument");
    mask_nearest_kernel<<<dim3((H * W + 255) / 256, 1), 256, 0, static_cast<cudaStream_t>(stream)>>>(
        mask, nullptr, H0, W0, mask01, guide, H, W);
    ADA_CHECK_CUDA(cudaGetLastError());
  });
}

static void launch_minmax_normalize(const float* depth, int B, long long n, float* base01, float* obs, void* scratch,
                                    cudaStream_t st) {
  uint32_t* mm = static_cast<uint32_t*>(scratch);
  const int gx = static_cast<int>(std::min<long long>((n + 255) / 256, std::max(1, 148 * 8 / B)));
  minmax_init_kernel<<<1, 256, 0, st>>>(mm, B);
  minmax_kernel<<<dim3(gx, B), 256, 0, st>>>(depth, n, mm);
  normalize_kernel<<<dim3(gx, B), 256, 0, st>>>(depth, n, mm, base01, obs);
  ADA_CHECK_CUDA(cudaGetLastError());
}

int ada_post_minmax_normalize(const float* depth, int64_t n, float* base01, float* obs, void* scratch8, void* stream) {
  return guarded([&] {
    require_device();
    ADA_REQUIRE(depth && (base01 || obs) && scratch8 && n > 0, "bad argument");
    launch_minmax_normalize(depth, 1, n, base01, obs, scratch8, static_cast<cudaStream_t>(stream));
  });
}

int ada_post_blend_seam(const float* raw01, const float* amodal, const float* mask01, float* out, int32_t H, int32_t W,
                        void* stream) {
  return guarded([&] {
    require_device();
    ADA_REQUIRE(raw01 && amodal && mask01 && out && H > 1 && W > 1, "bad argument");
    ADA_REQUIRE(out != raw01 && out != amodal, "blend_seam is not in-place safe");
    blend_seam_kernel<<<dim3((H * W + 255) / 256, 1), 256, 0, static_cast<cudaStream_t>(stream)>>>(raw01, amodal, mask01,
                                                                                                   out, H, W);
    ADA_CHECK_CUDA(cudaGetLastError());
  });
}

static void require_batch(int B, int H, int W) {
  ADA_REQUIRE(B > 0 && B <= 65535, "batch must be in [1, 65535]");
  ADA_REQUIRE(H > 0 && W > 0 && static_cast<long long>(H) * W < (1LL << 31) / 3, "bad output size");
}

int ada_pre_resize_linear_batch(const uint8_t* src, const ada_img_desc* desc, int32_t B, uint8_t* out_hwc, int32_t H,
                                int32_t W, void* stream) {
  return guarded([&] {
    require_device();
    ADA_REQUIRE(src && desc && out_hwc, "bad argument");
    require_batch(B, H, W);
    resize_linear_kernel<<<dim3((H * W + 255) / 256, B), 256, 0, static_cast<cudaStream_t>(stream)>>>(src, desc, out_hwc,
                                                                                                      H, W);
    ADA_CHECK_CUDA(cudaGetLastError());
  });
}

int ada_pre_image_nearest_batch(const uint8_t* src, const ada_img_desc* desc, int32_t B, float* out_chw, int32_t H,
                                int32_t W, int32_t normalize, void* stream) {
  return guarded([&] {
    require_device();
    ADA_REQUIRE(src && desc && out_chw, "bad argument");
    require_batch(B, H, W);
    image_nearest_kernel<<<dim3((H * W + 255) / 256, B), 256, 0, static_cast<cudaStream_t>(stream)>>>(
        src, desc, 0, 0, out_chw, H, W, normalize);
    ADA_CHECK_CUDA(cudaGetLastError());
  });
}

int ada_pre_mask_nearest_batch(const uint8_t* src, const ada_img_desc* desc, int32_t B, float* mask01, float* guide,
                               int32_t H, int32_t W, void* stream) {
  return guarded([&] {
    require_device();
    ADA_REQUIRE(src && desc && (mask01 || guide), "bad argument");
    require_batch(B, H, W);
    mask_nearest_kernel<<<dim3((H * W + 255) / 256, B), 256, 0, static_cast<cudaStream_t>(stream)>>>(
        src, desc, 0, 0, mask01, guide, H, W);
    ADA_CHECK_CUDA(cudaGetLastError());
  });
}

int ada_post_minmax_normalize_batch(const float* depth, int32_t B, int64_t n, float* base01, float* obs, void* scratch,
                                    void* stream) {
  return guarded([&] {
    require_device();
    ADA_REQUIRE(depth && (base01 || obs) && scratch && n > 0, "bad argument");
    ADA_REQUIRE(B > 0 && B <= 65535, "batch must be in [1, 65535]");
    launch_minmax_normalize(depth, B, n, base01, obs, scratch, static_cast<cudaStream_t>(stream));
  });
}

int ada_post_blend_seam_batch(const float* raw01, const float* amodal, const float* mask01, float* out, int32_t B,
                              int32_t H, int32_t W, void* stream) {
  return guarded([&] {
    require_device();
    ADA_REQUIRE(raw01 && amodal && mask01 && out && H > 1 && W > 1, "bad argument");
    ADA_REQUIRE(out != raw01 && out != amodal, "blend_seam is not in-place safe");
    require_batch(B, H, W);
    blend_seam_kernel<<<dim3((H * W + 255) / 256, B), 256, 0, static_cast<cudaStream_t>(stream)>>>(raw01, amodal, mask01,
                                                                                                   out, H, W);
    ADA_CHECK_CUDA(cudaGetLastError());
  });
}

// ---- DepthAnythingV2.infer_image's pre/post-processing over a batch
int ada_pre_resize_cubic_normalize_batch(const uint8_t* src, const ada_img_desc* desc, int32_t B, float* out_chw,
                                         int32_t H, int32_t W, void* stream) {
  return guarded([&] {
    require_device();
    ADA_REQUIRE(src && desc && out_chw, "bad argument");
    require_batch(B, H, W);
    resize_cubic_normalize_kernel<<<dim3((H * W + 255) / 256, B), 256, 0, static_cast<cudaStream_t>(stream)>>>(
        src, desc, out_chw, H, W);
    ADA_CHECK_CUDA(cudaGetLastError());
  });
}

int ada_post_upsample_restore_batch(const float* depth, int32_t B, int32_t H, int32_t W, const ada_img_desc* out_desc,
                                    float* out, void* stream) {
  return guarded([&] {
    require_device();
    ADA_REQUIRE(depth && out_desc && out, "bad argument");
    require_batch(B, H, W);
    // the output sizes are on the device: a fixed grid of ~8 blocks per SM over the batch, striding over each image
    const int gx = std::max(1, 148 * 8 / B);
    upsample_restore_kernel<<<dim3(gx, B), 256, 0, static_cast<cudaStream_t>(stream)>>>(depth, H, W, out_desc, out);
    ADA_CHECK_CUDA(cudaGetLastError());
  });
}

// ---- per-sample evaluation post-ops of the validation loop (SURVEY.md section 8 row f3): ada_eval_sample launches the
// batched kernel with B = 1 and no descriptor table
static void launch_eval(const float* pred, const uint8_t* src, const ada_eval_desc* desc, const EvalSample& one, int B,
                        double* out, cudaStream_t st) {
  eval_batch_kernel<<<dim3(kEvalCluster, B), kEvalThreads, 0, st>>>(pred, src, desc, one, out);
  ADA_CHECK_CUDA(cudaGetLastError());
}

int ada_eval_sample(const float* pred, int32_t h, int32_t w, const float* depth_gt, const float* depth_obs,
                    const uint8_t* visible_mask, const uint8_t* object_mask, int32_t H, int32_t W, double* out24,
                    double* scratch26, void* stream) {
  return guarded([&] {
    require_device();
    ADA_REQUIRE(pred && depth_gt && depth_obs && visible_mask && object_mask && out24 && scratch26, "bad argument");
    ADA_REQUIRE(h > 0 && w > 0 && H > 0 && W > 0 && static_cast<long long>(H) * W < (1LL << 31), "bad size");
    const EvalSample one{pred, h, w, depth_gt, depth_obs, visible_mask, object_mask, H, W};
    launch_eval(nullptr, nullptr, nullptr, one, 1, out24, static_cast<cudaStream_t>(stream));
  });
}

int ada_eval_batch(const float* pred, const uint8_t* src, const ada_eval_desc* desc, int32_t B, double* out, void* stream) {
  return guarded([&] {
    require_device();
    ADA_REQUIRE(pred && src && desc && out, "bad argument");
    ADA_REQUIRE(B > 0 && B <= 65535, "batch must be in [1, 65535]");
    launch_eval(pred, src, desc, EvalSample{}, B, out, static_cast<cudaStream_t>(stream));
  });
}

int ada_eval_accumulate(const double* rows, int32_t B, const int32_t* bucket, int32_t n_buckets, double* acc, void* stream) {
  return guarded([&] {
    require_device();
    ADA_REQUIRE(rows && acc, "bad argument");
    ADA_REQUIRE(B > 0 && B <= 65535, "batch must be in [1, 65535]");
    ADA_REQUIRE(n_buckets >= 0 && n_buckets <= 65535, "n_buckets must be in [0, 65535]");
    eval_accumulate_kernel<<<1, 256, 0, static_cast<cudaStream_t>(stream)>>>(rows, B, bucket, n_buckets, acc);
    ADA_CHECK_CUDA(cudaGetLastError());
  });
}

int ada_op_attention(const void* qkv_bf16, void* out_bf16, int32_t B, int32_t N, int32_t heads, int32_t impl, void* stream) {
  return guarded([&] {
    require_device();
    ADA_REQUIRE(qkv_bf16 && out_bf16 && B > 0 && N > 0 && heads > 0 && impl >= -1 && impl <= 2, "bad argument");
    launch_attention(static_cast<const __nv_bfloat16*>(qkv_bf16), static_cast<__nv_bfloat16*>(out_bf16), B, N, heads,
                     static_cast<cudaStream_t>(stream), impl);
  });
}

int ada_op_channel_ln_relu(const void* in_bf16, const float* w, const float* b, void* out_bf16, int64_t pixels, int32_t C,
                           float eps, void* stream) {
  return guarded([&] {
    require_device();
    launch_channel_ln_relu(static_cast<const __nv_bfloat16*>(in_bf16), w, b, static_cast<__nv_bfloat16*>(out_bf16), pixels,
                           C, eps, static_cast<cudaStream_t>(stream));
  });
}

int ada_op_upsample(const void* in_bf16, void* out_bf16, int32_t B, int32_t Hi, int32_t Wi, int32_t Ho, int32_t Wo,
                    int32_t C, void* stream) {
  return guarded([&] {
    require_device();
    launch_upsample(static_cast<const __nv_bfloat16*>(in_bf16), static_cast<__nv_bfloat16*>(out_bf16), B, Hi, Wi, Ho, Wo, C,
                    static_cast<cudaStream_t>(stream));
  });
}

int ada_op_patch_gather(const float* rgb, const float* const* guides, const int32_t* guide_ch, int32_t n_guides,
                        void* out_bf16, int32_t B, int32_t H, int32_t W, int32_t Kpad, void* stream) {
  return guarded([&] {
    require_device();
    launch_patch_gather(rgb, guides, guide_ch, n_guides, static_cast<__nv_bfloat16*>(out_bf16), B, H, W, Kpad, 1,
                        static_cast<cudaStream_t>(stream));
  });
}

int ada_op_tail_gather(const void* v_f16, const float* bias2, const float* aux, float* out, int32_t B, int32_t Hl, int32_t Wl,
                       int32_t H, int32_t W, int32_t sigmoid, void* stream) {
  return guarded([&] {
    require_device();
    launch_tail_gather(static_cast<const __half*>(v_f16), bias2, aux, out, B, Hl, Wl, H, W, sigmoid,
                       static_cast<cudaStream_t>(stream));
  });
}

int ada_op_tail_mma(const void* l_f16, const void* wpk_f16, const float* bias2, const float* aux, float* out, int32_t B,
                    int32_t Hl, int32_t Wl, int32_t H, int32_t W, int32_t C, int32_t sigmoid, void* stream) {
  return guarded([&] {
    require_device();
    launch_tail_mma(static_cast<const __half*>(l_f16), static_cast<const __half*>(wpk_f16), bias2, aux, out, B, Hl, Wl, H, W,
                    C, sigmoid, static_cast<cudaStream_t>(stream));
  });
}

int ada_pack_tail_mma(const float* w_host, int32_t C, void* dst_f16) {
  return guarded([&] {
    require_device();
    ADA_REQUIRE(w_host && dst_f16 && C % 32 == 0 && C <= kTmMaxC, "ada_pack_tail_mma: C % 32 == 0, C <= 128");
    float* tmp = nullptr;
    const size_t n = static_cast<size_t>(288) * C;
    ADA_CHECK_CUDA(cudaMalloc(&tmp, n * 4));
    cudaError_t e = cudaMemcpy(tmp, w_host, n * 4, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) {
      pack_tail_mma_kernel<<<static_cast<unsigned>((n + 255) / 256), 256>>>(tmp, static_cast<__half*>(dst_f16), C);
      e = cudaGetLastError();
      if (e == cudaSuccess) e = cudaDeviceSynchronize();
    }
    cudaFree(tmp);
    ADA_CHECK_CUDA(e);
  });
}

// Weight packers for the operator-level tests: host fp32 in, device bf16 out -- through the same device kernels
// (csrc/pack.cuh) ada_finalize uses.
static void pack_from_host(const float* w_host, size_t n_in, void* dst, long long n_out, const PackDesc& d) {
  require_device();
  ADA_REQUIRE(w_host && dst, "null argument");
  float* tmp = nullptr;
  ADA_CHECK_CUDA(cudaMalloc(&tmp, n_in * 4));
  cudaError_t e = cudaMemcpy(tmp, w_host, n_in * 4, cudaMemcpyHostToDevice);
  if (e == cudaSuccess) {
    pack_weights_kernel<<<static_cast<unsigned>((n_out + 255) / 256), 256>>>(tmp, nullptr, static_cast<__nv_bfloat16*>(dst), n_out, d);
    e = cudaGetLastError();
    if (e == cudaSuccess) e = cudaDeviceSynchronize();
  }
  cudaFree(tmp);
  ADA_CHECK_CUDA(e);
}

int ada_pack_tail_taps(const float* w_host, int32_t Cm, void* dst) {
  return guarded([&] {
    pack_from_host(w_host, static_cast<size_t>(32) * Cm * 9, dst, 288LL * Cm, PackDesc{PACK_TAIL, Cm, 0, 0, 0});
  });
}

int ada_pack_conv3x3(const float* w_host, int32_t Cout, int32_t Cin, void* dst) {
  return guarded([&] {
    const int Cpad = round_up(Cin, kBlockK);
    pack_from_host(w_host, static_cast<size_t>(Cout) * Cin * 9, dst, static_cast<long long>(Cout) * 9 * Cpad,
                   PackDesc{PACK_CONV3X3, Cout, Cin, Cpad, 0});
  });
}

int ada_pack_convT(const float* w_host, int32_t Cin, int32_t Cout, int32_t ks, void* dst) {
  return guarded([&] {
    pack_from_host(w_host, static_cast<size_t>(Cin) * Cout * ks * ks, dst, static_cast<long long>(ks) * ks * Cout * Cin,
                   PackDesc{PACK_CONVT, Cin, Cout, ks, 0});
  });
}

}  // extern "C"
