// libovg C ABI (include/ovg.h): argument validation, TMA descriptor cache, kernel launches.
#include <atomic>
#include <climits>
#include <cstdlib>
#include <mutex>
#include <string>
#include <unordered_map>
#include <vector>

#include <cudaTypedefs.h>

#include "../../include/ovg.h"
#include "attn.cuh"
#include "camera.cuh"
#include "elem.cuh"
#include "gemm.cuh"
#include "post.cuh"
#include "tail.cuh"
#include "pre.cuh"

namespace {

thread_local std::string g_err;
std::atomic<long long> g_launches{0};

int fail(int code, const std::string& msg) {
  g_err = msg;
  return code;
}

#define OVG_REQUIRE(cond, msg)                                                           \
  do {                                                                                   \
    if (!(cond)) return fail(OVG_E_INVALID, std::string(__func__) + ": " + (msg));        \
  } while (0)

#define OVG_CUDA(expr)                                                                   \
  do {                                                                                   \
    cudaError_t e__ = (expr);                                                            \
    if (e__ != cudaSuccess)                                                              \
      return fail(OVG_E_CUDA, std::string(__func__) + ": " #expr ": " + cudaGetErrorString(e__)); \
  } while (0)

int post_launch(const char* what) {
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return fail(OVG_E_CUDA, std::string(what) + ": launch failed: " + cudaGetErrorString(e));
  g_launches.fetch_add(1, std::memory_order_relaxed);
  return OVG_OK;
}

// ------------------------------------------------------------------------------ tensor maps
PFN_cuTensorMapEncodeTiled_v12000 get_encode() {
  static PFN_cuTensorMapEncodeTiled_v12000 fn = [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess) p = nullptr;
    return reinterpret_cast<PFN_cuTensorMapEncodeTiled_v12000>(p);
  }();
  return fn;
}

struct MapKey {
  const void* ptr;
  unsigned long long d0, d1, d2, ld, box1;   // box1 also carries (kind << 32) for output maps
  bool operator==(const MapKey& o) const {
    return ptr == o.ptr && d0 == o.d0 && d1 == o.d1 && d2 == o.d2 && ld == o.ld && box1 == o.box1;
  }
};
struct MapKeyHash {
  size_t operator()(const MapKey& k) const {
    size_t h = std::hash<const void*>()(k.ptr);
    for (unsigned long long v : {k.d0, k.d1, k.d2, k.ld, k.box1}) h = h * 1000003u ^ std::hash<unsigned long long>()(v);
    return h;
  }
};
std::mutex g_map_mu;
std::unordered_map<MapKey, CUtensorMap, MapKeyHash> g_maps;

// bf16 tensor [d2][d1][d0] (d0 contiguous, row stride ld elements, d2 stride d1*ld), box = [64, box1, 1], 128B swizzle.
// d2 == 0 -> rank 2.
int get_map(const void* ptr, unsigned long long d0, unsigned long long d1, unsigned long long d2,
            unsigned long long ld, unsigned box1, CUtensorMap* out) {
  MapKey key{ptr, d0, d1, d2, ld, box1};
  {
    std::lock_guard<std::mutex> g(g_map_mu);
    auto it = g_maps.find(key);
    if (it != g_maps.end()) {
      *out = it->second;
      return OVG_OK;
    }
  }
  auto enc = get_encode();
  if (!enc) return fail(OVG_E_CUDA, "cuTensorMapEncodeTiled entry point not available");
  if ((reinterpret_cast<uintptr_t>(ptr) & 15) || ((ld * 2) & 15))
    return fail(OVG_E_INVALID, "TMA operand must be 16-byte aligned with a 16-byte multiple row stride");
  cuuint64_t gdim[3] = {d0, d1, d2 ? d2 : 1};
  cuuint64_t gstr[2] = {ld * 2, d1 * ld * 2};
  cuuint32_t box[3] = {64, box1, 1};
  cuuint32_t estr[3] = {1, 1, 1};
  CUtensorMap m;
  CUresult r = enc(&m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, d2 ? 3 : 2, const_cast<void*>(ptr), gdim, gstr, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(OVG_E_CUDA, "cuTensorMapEncodeTiled failed (" + std::to_string(int(r)) + ")");
  {
    std::lock_guard<std::mutex> g(g_map_mu);
    if (g_maps.size() > 8192) g_maps.clear();
    g_maps.emplace(key, m);
  }
  *out = m;
  return OVG_OK;
}

// Output map for the staged epilogue: [rows, cols] row-major (row stride ld elements), box 32 cols x 32 rows;
// bf16 -> 64 B inner box, SWIZZLE_64B; fp32 -> 128 B inner box, SWIZZLE_128B.
int get_out_map(const void* ptr, bool f32, unsigned long long cols, unsigned long long rows, unsigned long long ld,
                CUtensorMap* out) {
  MapKey key{ptr, cols, rows, 0, ld, (f32 ? 2ull : 1ull) << 32};
  {
    std::lock_guard<std::mutex> g(g_map_mu);
    auto it = g_maps.find(key);
    if (it != g_maps.end()) {
      *out = it->second;
      return OVG_OK;
    }
  }
  auto enc = get_encode();
  if (!enc) return fail(OVG_E_CUDA, "cuTensorMapEncodeTiled entry point not available");
  const unsigned esz = f32 ? 4 : 2;
  if ((reinterpret_cast<uintptr_t>(ptr) & 15) || ((ld * esz) & 15))
    return fail(OVG_E_INVALID, "TMA store target must be 16-byte aligned with a 16-byte multiple row stride");
  cuuint64_t gdim[2] = {cols, rows};
  cuuint64_t gstr[1] = {ld * esz};
  cuuint32_t box[2] = {32, 32};
  cuuint32_t estr[2] = {1, 1};
  CUtensorMap m;
  CUresult r = enc(&m, f32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(ptr),
                   gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   f32 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(OVG_E_CUDA, "cuTensorMapEncodeTiled(out) failed (" + std::to_string(int(r)) + ")");
  {
    std::lock_guard<std::mutex> g(g_map_mu);
    g_maps.emplace(key, m);
  }
  *out = m;
  return OVG_OK;
}

// Function attributes and the SM count are per device: one process may drive several GPUs (or several host threads).
constexpr int kMaxDevices = 64;
int current_device() {
  int dev = 0;
  cudaGetDevice(&dev);
  return dev >= 0 && dev < kMaxDevices ? dev : 0;
}
int num_sms() {
  static std::atomic<int> n[kMaxDevices];
  const int dev = current_device();
  int v = n[dev].load(std::memory_order_relaxed);
  if (v == 0) {
    cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev);
    n[dev].store(v, std::memory_order_relaxed);
  }
  return v;
}
// true exactly until `mark_done` has been called for (slot, current device); setting an attribute twice is harmless
struct PerDeviceOnce {
  std::atomic<bool> done[kMaxDevices];
  bool needed() { return !done[current_device()].load(std::memory_order_acquire); }
  void mark_done() { done[current_device()].store(true, std::memory_order_release); }
};

template <int BN, int EPI>
int launch_gemm(const CUtensorMap& ta, const CUtensorMap& tb, const ovg::GemmParams& p, cudaStream_t st) {
  using Cfg = ovg::GemmCfg<BN>;
  static PerDeviceOnce once;
  auto kern = ovg::gemm_kernel<BN, EPI>;
  if (once.needed()) {
    OVG_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM_BYTES));
    once.mark_done();
  }
  const int tiles = ((p.M + 127) / 128) * ((p.N + BN - 1) / BN);
  const int grid = tiles < num_sms() ? tiles : num_sms();
  kern<<<grid, ovg::GEMM_THREADS, Cfg::SMEM_BYTES, st>>>(ta, tb, p);
  return post_launch("ovg_gemm");
}

template <int BN, int EPI>
int launch_gemm2(const CUtensorMap& ta, const CUtensorMap& tb, const CUtensorMap& tbh, const CUtensorMap (&to)[3],
                 ovg::GemmParams& p, cudaStream_t st) {
  using Cfg = ovg::Gemm2Cfg<BN>;
  static PerDeviceOnce once;
  auto kern = ovg::gemm2_kernel<BN, EPI>;
  if (once.needed()) {
    OVG_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM_BYTES));
    once.mark_done();
  }
  const int tiles = ((p.M + 255) / 256) * ((p.N + BN - 1) / BN);
  const int pairs = num_sms() / 2;
  const int grid = 2 * (tiles < pairs ? tiles : pairs);
  // last partial wave as half tiles when both halves of every leftover tile find a free cluster (gemm.cuh)
  const int tail = tiles > pairs ? tiles % pairs : 0;
#ifndef OVG_GEMM_SPLIT_TAIL
#define OVG_GEMM_SPLIT_TAIL 1
#endif
  p.split_tail = (OVG_GEMM_SPLIT_TAIL && BN == 256 && tail > 0 && 2 * tail <= pairs) ? 1 : 0;
  kern<<<grid, ovg::GEMM_THREADS, Cfg::SMEM_BYTES, st>>>(ta, tb, tbh, to[0], to[1], to[2], p);
  return post_launch("ovg_gemm(2sm)");
}

template <int EPI>
int dispatch_bn(int bn, const CUtensorMap& ta, const CUtensorMap& tb, const ovg::GemmParams& p, cudaStream_t st) {
  switch (bn) {
    case 256: return launch_gemm<256, EPI>(ta, tb, p, st);
    case 128: return launch_gemm<128, EPI>(ta, tb, p, st);
    case 64: return launch_gemm<64, EPI>(ta, tb, p, st);
    default: return fail(OVG_E_INVALID, "ovg_gemm: unsupported block_n");
  }
}

}  // namespace

long long* g_attn_prof = nullptr;   // set through ovg_debug_set_attn_profile (profiling builds)
long long* g_tail_prof = nullptr;   // ovg_debug_set_tail_profile: clock64 stamps of the fused DPT tail (csrc/tail.cuh)

extern "C" {

void ovg_debug_set_attn_profile(long long* buf) { g_attn_prof = buf; }
void ovg_debug_set_tail_profile(long long* buf) { g_tail_prof = buf; }

int ovg_version(void) { return 3; }
const char* ovg_last_error(void) { return g_err.c_str(); }
long long ovg_launch_count(void) { return g_launches.load(); }

int ovg_device_check(void) {
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return fail(OVG_E_NODEVICE, "no CUDA device");
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, dev) != cudaSuccess) return fail(OVG_E_NODEVICE, "cannot query device");
  if (prop.major != 10)
    return fail(OVG_E_NODEVICE, std::string("libovg requires sm_100 (B200); found sm_") + std::to_string(prop.major) +
                                    std::to_string(prop.minor));
  return OVG_OK;
}

int ovg_gemm(const ovg_gemm_args* a, void* stream) {
  OVG_REQUIRE(a && a->a && a->b, "null operand");
  OVG_REQUIRE(a->m > 0 && a->n > 0 && a->a_cols > 0 && a->a_rows > 0, "empty problem");
  OVG_REQUIRE(a->num_taps >= 1 && a->num_taps <= 9, "num_taps must be in [1,9]");
  OVG_REQUIRE(a->a_cols % 8 == 0, "a_cols must be a multiple of 8");
  OVG_REQUIRE(a->num_taps == 1 || a->a_cols % 64 == 0, "multi-tap GEMM needs a_cols % 64 == 0");
  OVG_REQUIRE(a->n % 32 == 0, "n must be a multiple of 32");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);

  ovg::GemmParams p{};
  p.M = a->m;
  p.N = a->n;
  p.kc_blocks = (a->a_cols + 63) / 64;
  p.k_blocks = p.kc_blocks * a->num_taps;
  for (int i = 0; i < 9; ++i) p.tap_off[i] = i < a->num_taps ? a->tap_off[i] : 0;
  p.bias = a->bias;
  p.act = a->act;
  p.out = a->out;
  p.ldo = a->ldo;
  p.table = a->table;
  p.table_rows = a->table_rows > 0 ? a->table_rows : 1;
  p.f16 = (a->f16 && (a->epi == OVG_EPI_BF16 || a->epi == OVG_EPI_HEADTAIL)) ? 1 : 0;
  p.skip1 = reinterpret_cast<const __nv_bfloat16*>(a->skip1);
  p.skip2 = reinterpret_cast<const __nv_bfloat16*>(a->skip2);
  p.rowmap = a->rowmap;
  p.gh = a->gh;
  p.gw = a->gw;
  p.ps = a->ps;
  p.cout = a->cout;
  p.gamma = a->gamma;
  p.row_index = a->row_index;
  p.q_out = reinterpret_cast<__nv_bfloat16*>(a->q_out);
  p.k_out = reinterpret_cast<__nv_bfloat16*>(a->k_out);
  p.v_out = reinterpret_cast<__nv_bfloat16*>(a->v_out);
  p.C = a->C;
  p.ntok = a->ntok;
  p.T = a->T;
  p.nspecial = a->nspecial;
  p.wp = a->wp;
  p.maxpos = a->maxpos;
  p.qn_w = a->qn_w;
  p.qn_b = a->qn_b;
  p.kn_w = a->kn_w;
  p.kn_b = a->kn_b;
  p.rope_cos = a->rope_cos;
  p.rope_sin = a->rope_sin;
  p.qscale = a->qscale;
  p.qk_norm = a->qk_norm;
  p.rope = a->rope;
  p.w2 = a->w2;
  p.b2 = a->b2;
  p.outc = a->outc;
  p.head_act = a->head_act;
  p.preds = a->preds;
  p.conf = a->conf;
  p.n_peers = a->epi == OVG_EPI_QKV ? a->n_peers : 0;
  p.peer_ntok = a->peer_ntok;
  p.peer_tok_off = a->peer_tok_off;
  OVG_REQUIRE(p.n_peers >= 0 && p.n_peers <= 8, "at most 8 peers");
  for (int i = 0; i < p.n_peers; ++i) {
    OVG_REQUIRE(a->k_peers[i] && a->v_peers[i], "null peer buffer");
    p.k_peer[i] = reinterpret_cast<__nv_bfloat16*>(a->k_peers[i]);
    p.v_peer[i] = reinterpret_cast<__nv_bfloat16*>(a->v_peers[i]);
  }
  if (p.n_peers > 0) OVG_REQUIRE(a->peer_ntok >= a->ntok && a->peer_tok_off >= 0 && a->peer_tok_off + a->ntok <= a->peer_ntok,
                                 "peer token window");

  int bn = a->block_n;
  if (a->epi == OVG_EPI_HEADTAIL) {
    OVG_REQUIRE(a->n == 32, "HEADTAIL epilogue needs n == 32");
    OVG_REQUIRE(a->w2 && a->b2 && a->bias && a->preds && a->conf && a->outc >= 2 && a->outc <= 4, "HEADTAIL args");
    OVG_REQUIRE(a->rowmap == OVG_ROWS_PAD, "HEADTAIL runs on the zero-bordered grid");
    bn = 32;
  } else if (bn == 0) {
    bn = a->n >= 256 ? 256 : (a->n >= 128 ? 128 : 64);
    if (a->epi != OVG_EPI_QKV && bn == 256) {
      // prefer 128-wide tiles when 256-wide ones leave a badly quantised last wave
      const long long mt = (a->m + 127) / 128;
      const long long t256 = mt * ((a->n + 255) / 256), t128 = mt * ((a->n + 127) / 128);
      const int sms = num_sms();
      const double e256 = double(t256) / double(((t256 + sms - 1) / sms) * sms);
      const double e128 = double(t128) / double(((t128 + sms - 1) / sms) * sms);
      if (e128 > e256 + 0.08) bn = 128;
    }
  }
  if (a->epi == OVG_EPI_QKV) {
    OVG_REQUIRE(a->q_out && a->bias && ((a->k_out && a->v_out) || a->n_peers > 0), "QKV args");
    if (a->qk_norm) OVG_REQUIRE(a->qn_w && a->qn_b && a->kn_w && a->kn_b, "QKV q/k norm weights");
    if (a->rope) OVG_REQUIRE(a->rope_cos && a->rope_sin && a->maxpos > 0 && a->maxpos <= OVG_ROPE_MAX_POSITIONS && a->wp > 0,
                             "QKV rope table (maxpos <= " + std::to_string(OVG_ROPE_MAX_POSITIONS) + ")");
    else p.maxpos = 0;
    OVG_REQUIRE(a->C % 64 == 0 && a->n == 3 * a->C && a->ntok > 0 && a->T > 0, "QKV geometry");
    if (p.wp <= 0) p.wp = 1;
    OVG_REQUIRE(a->m % a->ntok == 0, "m must be a multiple of ntok");
    if (bn < 64) bn = 64;
  } else if (a->epi == OVG_EPI_RESID) {
    OVG_REQUIRE(a->out && a->gamma && a->bias, "RESID needs out, gamma, bias");
  } else if (a->epi == OVG_EPI_BF16) {
    OVG_REQUIRE(a->out, "BF16 epilogue needs out");
    OVG_REQUIRE((reinterpret_cast<uintptr_t>(a->bias) & 15) == 0 && (reinterpret_cast<uintptr_t>(a->table) & 15) == 0 &&
                    (a->table == nullptr || a->n % 4 == 0),
                "bias / table must be 16-byte aligned");
    if (a->rowmap == OVG_ROWS_PIXSHUF)
      OVG_REQUIRE(a->ps > 0 && a->cout % 32 == 0 && a->n == a->ps * a->ps * a->cout, "PIXSHUF geometry");
    if (a->rowmap != OVG_ROWS_IDENT) OVG_REQUIRE(a->gh > 0 && a->gw > 0, "row map needs gh, gw");
  }

  // RoPE grids larger than the epilogue's smem table: the QKV kernels that read cos / sin from global memory
  const bool gtab = a->epi == OVG_EPI_QKV && p.maxpos > ovg::GEMM_QKV_SMEM_POS;
  CUtensorMap ta, tb;
  int rc = get_map(a->a, a->a_cols, a->a_rows, 0, a->lda, 128, &ta);
  if (rc) return rc;
  const unsigned long long ktot = static_cast<unsigned long long>(a->a_cols) * a->num_taps;
  // block_n 512 / 384 select the CTA-pair kernels (256 x 256 / 256 x 128 tile per 2-SM cluster).  They stage 33% fewer
  // L2->SM bytes per FLOP than the single-CTA tiles, which is what bounds these GEMMs; auto-selected for large problems.
  const bool pair = (a->block_n == 512 || a->block_n == 384) ||
                    (a->block_n == 0 && a->epi != OVG_EPI_HEADTAIL && a->n >= 128 && a->m >= 1024);
  if (pair) {
    OVG_REQUIRE(a->epi != OVG_EPI_HEADTAIL, "pair kernel has no HEADTAIL epilogue");
    const int pbn = (a->block_n == 384 || (a->block_n == 0 && a->n < 256)) ? 128 : 256;
    rc = get_map(a->b, ktot, a->n, 0, a->ldb, pbn / 2, &tb);
    if (rc) return rc;
    CUtensorMap tbh;
    rc = get_map(a->b, ktot, a->n, 0, a->ldb, pbn / 4, &tbh);     // half tiles of the last wave: N/4 rows of B per CTA
    if (rc) return rc;
    // staged epilogue (smem -> TMA store / fp32 reduce-add) whenever output rows are the GEMM rows
    CUtensorMap to[3] = {ta, ta, ta};
    const bool stage_ok = (a->epi == OVG_EPI_RESID && !a->row_index) ||
                          (a->epi == OVG_EPI_BF16 && (a->rowmap == OVG_ROWS_IDENT || a->rowmap == OVG_ROWS_PAD));
    if (stage_ok) {
      rc = get_out_map(a->out, a->epi == OVG_EPI_RESID, a->n, a->m, a->ldo, &to[0]);
      if (rc) return rc;
      p.staged = 1;
    } else if (a->epi == OVG_EPI_QKV && a->n_peers == 0) {
      // head-major q / k / v [batch * heads, ntok, 64]: one 32-token x 64 box per bulk store
      const unsigned long long bh = static_cast<unsigned long long>(a->m / a->ntok) * (a->C / 64);
      const void* outs[3] = {a->q_out, a->k_out, a->v_out};
      for (int i = 0; i < 3; ++i) {
        rc = get_map(outs[i], 64, a->ntok, bh, 64, 32, &to[i]);
        if (rc) return rc;
      }
      p.staged = 1;
    }
    if (pbn == 256) {
      switch (a->epi) {
        case OVG_EPI_BF16: return launch_gemm2<256, ovg::EPI_BF16>(ta, tb, tbh, to, p, st);
        case OVG_EPI_RESID: return launch_gemm2<256, ovg::EPI_RESID>(ta, tb, tbh, to, p, st);
        case OVG_EPI_QKV:
          return gtab ? launch_gemm2<256, ovg::EPI_QKV_GTAB>(ta, tb, tbh, to, p, st) : launch_gemm2<256, ovg::EPI_QKV>(ta, tb, tbh, to, p, st);
        default: return fail(OVG_E_INVALID, "ovg_gemm: unknown epilogue");
      }
    }
    switch (a->epi) {
      case OVG_EPI_BF16: return launch_gemm2<128, ovg::EPI_BF16>(ta, tb, tbh, to, p, st);
      case OVG_EPI_RESID: return launch_gemm2<128, ovg::EPI_RESID>(ta, tb, tbh, to, p, st);
      case OVG_EPI_QKV:
        return gtab ? launch_gemm2<128, ovg::EPI_QKV_GTAB>(ta, tb, tbh, to, p, st) : launch_gemm2<128, ovg::EPI_QKV>(ta, tb, tbh, to, p, st);
      default: return fail(OVG_E_INVALID, "ovg_gemm: unknown epilogue");
    }
  }
  rc = get_map(a->b, ktot, a->n, 0, a->ldb, bn, &tb);
  if (rc) return rc;

  switch (a->epi) {
    case OVG_EPI_BF16: return dispatch_bn<ovg::EPI_BF16>(bn, ta, tb, p, st);
    case OVG_EPI_RESID: return dispatch_bn<ovg::EPI_RESID>(bn, ta, tb, p, st);
    case OVG_EPI_QKV: return gtab ? dispatch_bn<ovg::EPI_QKV_GTAB>(bn, ta, tb, p, st) : dispatch_bn<ovg::EPI_QKV>(bn, ta, tb, p, st);
    case OVG_EPI_HEADTAIL: {
      // row-shift kernel: 3x3 taps in row-major order over a 128-channel map ((ky, kx) -> tap_off = (ky-1)*pitch + kx-1)
      bool shape_ok = a->num_taps == 9 && a->a_cols == 128 && a->n == 32;
      for (int ky = 0; ky < 3 && shape_ok; ++ky)
        shape_ok = a->tap_off[ky * 3 + 1] - a->tap_off[ky * 3] == 1 && a->tap_off[ky * 3 + 2] - a->tap_off[ky * 3 + 1] == 1;
      if (!shape_ok) return launch_gemm<32, ovg::EPI_HEADTAIL>(ta, tb, p, st);
      CUtensorMap ta136, tb32;
      rc = get_map(a->a, a->a_cols, a->a_rows, 0, a->lda, ovg::HT_A_ROWS, &ta136);
      if (rc) return rc;
      rc = get_map(a->b, ktot, a->n, 0, a->ldb, 32, &tb32);
      if (rc) return rc;
      static PerDeviceOnce once;
      if (once.needed()) {
        OVG_CUDA(cudaFuncSetAttribute(ovg::headtail_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, ovg::HT_SMEM_BYTES));
        once.mark_done();
      }
      const int tiles = (p.M + ovg::GEMM_BM - 1) / ovg::GEMM_BM;
      const int grid = tiles < num_sms() ? tiles : num_sms();
      ovg::headtail_kernel<<<grid, ovg::GEMM_THREADS, ovg::HT_SMEM_BYTES, st>>>(ta136, tb32, p);
      return post_launch("ovg_gemm(headtail)");
    }
    default: return fail(OVG_E_INVALID, "ovg_gemm: unknown epilogue");
  }
}

long long ovg_attention_scratch_bytes(void) { return 4LL * 2 * num_sms() * 128 * (64 * 4 + 8) + 256; }   // <= 4 parts of < one wave of tiles

int ovg_attention_kv_ws(const void* q, const void* k, const void* v, void* out, int batch, int heads, int nq, int nkv,
                        void* scratch, long long scratch_bytes, void* stream) {
  OVG_REQUIRE(q && k && v && out, "null operand");
  OVG_REQUIRE(batch > 0 && heads > 0 && nq > 0 && nkv > 0, "empty problem");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  CUtensorMap tq, tk, tv;
  const unsigned long long bh = static_cast<unsigned long long>(batch) * heads;
  int rc = get_map(q, 64, nq, bh, 64, 128, &tq);
  if (rc) return rc;
  rc = get_map(k, 64, nkv, bh, 64, 128, &tk);
  if (rc) return rc;
  rc = get_map(v, 64, nkv, bh, 64, 128, &tv);
  if (rc) return rc;
  static PerDeviceOnce once;
  if (once.needed()) {
    OVG_CUDA(cudaFuncSetAttribute(ovg::attn1_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, ovg::ATT1_SMEM_BYTES));
    OVG_CUDA(cudaFuncSetAttribute(ovg::attn1_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, 100));
    once.mark_done();
  }
  const int q_tiles = (nq + 127) / 128;
  const long long tiles = static_cast<long long>(q_tiles) * heads * batch;
  OVG_REQUIRE(tiles < (1LL << 28), "too many tiles");
  ovg::AttnParams p{nq, nkv, heads, heads * 64, reinterpret_cast<__nv_bfloat16*>(out), g_attn_prof, q_tiles, static_cast<int>(tiles),
                    static_cast<int>(tiles), 1, nullptr, nullptr};
#ifndef OVG_ATT_PERSISTENT
#define OVG_ATT_PERSISTENT 1    // 0: always one CTA per work item (A/B builds)
#endif
#ifndef OVG_ATT_SPLIT_TAIL
#define OVG_ATT_SPLIT_TAIL 1    // 0: never split the tiles of the last wave over the keys (A/B builds)
#endif
  // Short sequences (frame / DINOv2 attention: 11 KV tiles per item): two resident CTAs per SM walk the items, so barrier /
  // TMEM set-up is paid once and the next item's Q, K, V stream in under the current item's tail (0.1126 -> 0.1085 ms at
  // 8 x 16 x 1374).  Long sequences keep one CTA per item: the hardware's dynamic CTA placement balances the 4.65 "waves" of
  // the global attention better than a static round robin (0.619 vs 0.649 ms), profiles/r02_attn_ab.jsonl.
  const int resident = 2 * num_sms();
  const int kv_tiles = (nkv + 127) / 128;
  const bool persistent = OVG_ATT_PERSISTENT && tiles > resident && kv_tiles <= 16;
  // Long sequences: the tiles of the last, partly empty wave are cut into 2-4 KV ranges (one CTA each, issued after the whole
  // tiles) whose partial (O, reference, row sum) a small kernel merges: 1 376 tiles on 296 slots cost 4.67 instead of 5 waves.
  int parts = 1;
  const int tail = static_cast<int>(tiles % resident);
  if (OVG_ATT_SPLIT_TAIL && !persistent && scratch && tiles > resident && tail > 0 && kv_tiles >= 24) {
    double best = 1.0;
    for (int c = 2; c <= 4; ++c) {
      const double cost = static_cast<double>((static_cast<long long>(tail) * c + resident - 1) / resident) / c + 0.04;   // + merge
      if (cost < best - 0.1) {
        best = cost;
        parts = c;
      }
    }
    if (parts > 1) {
      const long long need = static_cast<long long>(tail) * parts * 128 * (64 * 4 + 8);
      if (need > scratch_bytes - 256 || (reinterpret_cast<uintptr_t>(scratch) & 15)) parts = 1;
    }
  }
  if (parts > 1) {
    p.n_full = static_cast<int>(tiles) - tail;
    p.parts = parts;
    p.items = p.n_full + tail * parts;
    p.part_o = static_cast<float*>(scratch);
    p.part_ml = reinterpret_cast<float2*>(p.part_o + static_cast<long long>(tail) * parts * 128 * 64);
  }
  const int grid1 = persistent ? resident : p.items;
  ovg::attn1_kernel<<<grid1, ovg::ATT1_THREADS, ovg::ATT1_SMEM_BYTES, st>>>(tq, tk, tv, p);
  rc = post_launch("ovg_attention");
  if (rc || parts <= 1) return rc;
  ovg::attn_merge_kernel<<<tail, 128, 0, st>>>(p);
  return post_launch("ovg_attention(merge)");
}

int ovg_attention_kv(const void* q, const void* k, const void* v, void* out, int batch, int heads, int nq, int nkv,
                     void* stream) {
  return ovg_attention_kv_ws(q, k, v, out, batch, heads, nq, nkv, nullptr, 0, stream);
}

int ovg_attention(const void* q, const void* k, const void* v, void* out, int batch, int heads, int n, void* stream) {
  return ovg_attention_kv(q, k, v, out, batch, heads, n, n, stream);
}

int ovg_layernorm(const void* in, int in_is_bf16, long long ld_in, void* out, int out_is_f32, long long ld_out, int rows,
                  int C, const float* w, const float* b, float eps, int grp_out, int grp_in, int grp_off, void* stream) {
  OVG_REQUIRE(in && out && rows > 0, "null operand");
  OVG_REQUIRE(out_is_f32 >= 0 && out_is_f32 <= 2, "output type: 0 bf16, 1 fp32, 2 fp16");
  OVG_REQUIRE((w == nullptr) == (b == nullptr), "affine needs both weight and bias");
  OVG_REQUIRE(C % 128 == 0 && C <= 2048, "C must be a multiple of 128, <= 2048");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  ovg::LnParams p{in, in_is_bf16, ld_in, out, out_is_f32, ld_out, rows, C, w, b, eps,
                  grp_out, grp_in, grp_off};
  constexpr int ln_threads = 256;     // 8 rows per block
#ifndef OVG_LN_PERSIST
#define OVG_LN_PERSIST 2
#endif
  constexpr int ln_persist = OVG_LN_PERSIST;       // persistent grid: blocks per SM
  OVG_REQUIRE((reinterpret_cast<uintptr_t>(w) & 15) == 0 && (reinterpret_cast<uintptr_t>(b) & 15) == 0, "w / b must be 16-byte aligned");
  const int rpb = ln_threads / 32;
  int blocks = (rows + rpb - 1) / rpb;
  if (blocks > num_sms() * ln_persist) blocks = num_sms() * ln_persist;
  switch (C / 32) {
#define OVG_LN_CASE(V) \
  case V: ovg::layernorm_kernel<V><<<blocks, ln_threads, 0, st>>>(p); break;
    OVG_LN_CASE(4) OVG_LN_CASE(8) OVG_LN_CASE(12) OVG_LN_CASE(16) OVG_LN_CASE(20) OVG_LN_CASE(24) OVG_LN_CASE(28)
    OVG_LN_CASE(32) OVG_LN_CASE(36) OVG_LN_CASE(40) OVG_LN_CASE(44) OVG_LN_CASE(48) OVG_LN_CASE(52) OVG_LN_CASE(56)
    OVG_LN_CASE(60) OVG_LN_CASE(64)
#undef OVG_LN_CASE
    default: return fail(OVG_E_INVALID, "ovg_layernorm: unsupported C");
  }
  return post_launch("ovg_layernorm");
}

int ovg_assemble_tokens(float* x, const float* patch, const float* cam_tok, const float* reg_tok, const float* inj0,
                        const float* placeholder, const int* has_depth, int K, int S, int T, int R, int C, int view_base,
                        void* stream) {
  OVG_REQUIRE(x && patch && cam_tok && reg_tok && inj0 && placeholder && has_depth, "null operand");
  OVG_REQUIRE(K > 0 && S > 0 && K % S == 0 && T > R + 1 && C % 4 == 0, "bad geometry");
  ovg::AssembleParams p{x, patch, cam_tok, reg_tok, inj0, placeholder, has_depth, K, S, T, R, C, view_base};
  const int threads = C / 4 < 256 ? ((C / 4 + 31) / 32) * 32 : 256;
  ovg::assemble_tokens_kernel<<<K * T, threads, 0, reinterpret_cast<cudaStream_t>(stream)>>>(p);
  return post_launch("ovg_assemble_tokens");
}

int ovg_peer_barrier(int* const* flag_peers, int* epoch_counter, int rank, int world, void* stream) {
  OVG_REQUIRE(flag_peers && epoch_counter && world >= 1 && world <= 8 && rank >= 0 && rank < world, "bad arguments");
  ovg::PeerBarrierParams p{};
  for (int i = 0; i < world; ++i) {
    OVG_REQUIRE(flag_peers[i], "null flag array");
    p.flags[i] = flag_peers[i];
  }
  p.epoch = epoch_counter; p.rank = rank; p.world = world;
  ovg::peer_barrier_kernel<<<1, 32, 0, reinterpret_cast<cudaStream_t>(stream)>>>(p);
  return post_launch("ovg_peer_barrier");
}

int ovg_inject_snapshot(float* x, const float* inj, void* slot, float* cam_out, int K, int T, int C, int coff,
                        void* stream) {
  OVG_REQUIRE(x && K > 0 && T > 0 && C % 4 == 0, "bad arguments");
  OVG_REQUIRE(coff == 0 || coff == C, "coff must be 0 or C");
  ovg::InjectParams p{x, inj, reinterpret_cast<__nv_bfloat16*>(slot), cam_out, K, T, C, coff};
  const int threads = C / 4 < 256 ? ((C / 4 + 31) / 32) * 32 : 256;
  ovg::inject_snapshot_kernel<<<slot ? K * T : K, threads, 0, reinterpret_cast<cudaStream_t>(stream)>>>(p);
  return post_launch("ovg_inject_snapshot");
}

int ovg_depth_im2col2(const float* depth, const float* mask, const int* idx_stats, int n_stats, const int* idx_cols, int n_cols,
                      double* scratch, void* cols, int ldc, int B, int S, int H, int W, int patch, void* stream) {
  OVG_REQUIRE(depth && mask && idx_stats && scratch && (n_cols == 0 || (idx_cols && cols)), "null operand");
  OVG_REQUIRE(B > 0 && n_stats > 0 && n_stats <= S && n_cols >= 0 && n_cols <= S && H % patch == 0 && W % patch == 0 &&
                  patch % 2 == 0, "bad geometry");
  OVG_REQUIRE(ldc >= 2 * patch * patch && ldc % 2 == 0, "ldc too small / odd");
  OVG_REQUIRE((reinterpret_cast<uintptr_t>(depth) & 7) == 0 && (reinterpret_cast<uintptr_t>(mask) & 7) == 0 &&
                  (reinterpret_cast<uintptr_t>(cols) & 3) == 0, "depth / mask must be 8-byte aligned");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  ovg::DepthParams ps{depth, mask, idx_stats, scratch, reinterpret_cast<__nv_bfloat16*>(cols), ldc, B, S, n_stats, H, W, patch};
  ovg::depth_stats_kernel<<<dim3(ovg::DEPTH_NCHUNK, B), 256, 0, st>>>(ps);
  int rc = post_launch("ovg_depth_im2col(stats)");
  if (rc) return rc;
  ovg::depth_scale_kernel<<<B, 256, 0, st>>>(ps);
  rc = post_launch("ovg_depth_im2col(scale)");
  if (rc || n_cols == 0) return rc;
  ovg::DepthParams pc = ps;
  pc.idx = idx_cols;
  pc.Sd = n_cols;
  if (patch == 14) ovg::depth_im2col_kernel<14><<<B * n_cols * (H / patch), 256, 0, st>>>(pc);
  else ovg::depth_im2col_kernel<0><<<B * n_cols * (H / patch), 256, 0, st>>>(pc);
  return post_launch("ovg_depth_im2col");
}

int ovg_depth_im2col(const float* depth, const float* mask, const int* idx, double* scratch, void* cols, int ldc,
                     int B, int S, int Sd, int H, int W, int patch, void* stream) {
  OVG_REQUIRE(Sd > 0, "bad geometry");
  return ovg_depth_im2col2(depth, mask, idx, Sd, idx, Sd, scratch, cols, ldc, B, S, H, W, patch, stream);
}

int ovg_image_im2col(const float* images, const float* mean3, const float* std3, void* cols, int ldc, int K, int H, int W,
                     int patch, void* stream) {
  OVG_REQUIRE(images && mean3 && std3 && cols, "null operand");
  OVG_REQUIRE(K > 0 && H % patch == 0 && W % patch == 0 && patch % 2 == 0 && ldc >= 3 * patch * patch && ldc % 8 == 0,
              "bad geometry");
  OVG_REQUIRE((reinterpret_cast<uintptr_t>(images) & 7) == 0, "images must be 8-byte aligned");
  ovg::ImageColParams p{images, reinterpret_cast<__nv_bfloat16*>(cols), ldc, K, H, W, patch, {}, {}};
  for (int c = 0; c < 3; ++c) {
    p.mean[c] = mean3[c];
    p.istd[c] = 1.0f / std3[c];
  }
  if (patch == 14) ovg::image_im2col_kernel<14><<<K * (H / patch), 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(p);
  else ovg::image_im2col_kernel<0><<<K * (H / patch), 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(p);
  return post_launch("ovg_image_im2col");
}

int ovg_im2col3x3s2(const void* src, void* dst, int F, int h, int w, int C, void* stream) {
  OVG_REQUIRE(src && dst && F > 0 && h > 0 && w > 0 && C % 8 == 0, "bad arguments");
  const int oh = (h - 1) / 2 + 1, ow = (w - 1) / 2 + 1;
  ovg::Im2colParams p{reinterpret_cast<const __nv_bfloat16*>(src), reinterpret_cast<__nv_bfloat16*>(dst), F, h, w, C, oh, ow};
  const int threads = C / 8 < 128 ? ((C / 8 + 31) / 32) * 32 : 128;
  ovg::im2col3x3s2_kernel<<<dim3(F * oh * ow, 9), threads, 0, reinterpret_cast<cudaStream_t>(stream)>>>(p);
  return post_launch("ovg_im2col3x3s2");
}

int ovg_upsample_bilinear(const void* src, void* dst, const float* tx, const float* ty, int F, int h, int w, int H, int W,
                          int C, int f16, void* stream) {
  OVG_REQUIRE(src && dst && F > 0 && h > 0 && w > 0 && H > 0 && W > 0 && C % 16 == 0, "bad arguments");
  OVG_REQUIRE((tx == nullptr) == (ty == nullptr), "position tables come as a pair");
  OVG_REQUIRE(F <= 65535 && H + 2 <= 65535, "grid too large");
  ovg::UpsampleParams p{reinterpret_cast<const __nv_bfloat16*>(src), reinterpret_cast<__nv_bfloat16*>(dst), tx, ty,
                        F, h, w, H, W, C,
                        H > 1 ? static_cast<float>(h - 1) / static_cast<float>(H - 1) : 0.f,
                        W > 1 ? static_cast<float>(w - 1) / static_cast<float>(W - 1) : 0.f, f16 ? 1 : 0};
  const size_t row_smem = static_cast<size_t>(w) * 32 * sizeof(float);
  if (C % 32 == 0 && row_smem <= 48 * 1024 && C / 32 <= 65535) {
    dim3 grid(H + 2, F, C / 32);
    ovg::upsample_rows_kernel<<<grid, 256, row_smem, reinterpret_cast<cudaStream_t>(stream)>>>(p);
    return post_launch("ovg_upsample_bilinear");
  }
  const int per_row = (W + 2) * (C / 8);
  dim3 grid((per_row + 255) / 256, H + 2, F);
  ovg::upsample_bilinear_kernel<<<grid, 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(p);
  return post_launch("ovg_upsample_bilinear");
}

int ovg_dpt_tail_supported(int h, int w, int H, int W, int C) {
  if (C != 128 || h < 2 || w < 2 || H < h || W < w) return 0;
  const float sx = W > 1 ? static_cast<float>(w - 1) / static_cast<float>(W - 1) : 0.f;
  const int span = static_cast<int>(sx * 129.0f) + 3;           // source pixels under 130 output pixels
  return span <= ovg::FT_VBUF_PX ? 1 : 0;
}

long long ovg_dpt_tail_scratch_bytes(int H, int W) { return (H > 0 && W > 0) ? 3LL * (H + W) * 32 * 4 : -1; }

int ovg_dpt_tail(const void* src, const float* tx, const float* ty, const void* w3x3, const float* bias, const float* w2,
                 const float* b2, int outc, int head_act, float* preds, float* conf, int F, int h, int w, int H, int W, int f16,
                 void* scratch, void* stream) {
  OVG_REQUIRE(src && w3x3 && bias && w2 && b2 && preds && conf, "null argument");
  OVG_REQUIRE((tx == nullptr) == (ty == nullptr), "position tables come as a pair");
  OVG_REQUIRE(tx == nullptr || (scratch && (reinterpret_cast<uintptr_t>(scratch) & 15) == 0),
              "position embedding needs 16-byte aligned scratch (ovg_dpt_tail_scratch_bytes)");
  OVG_REQUIRE(H >= 2 && W >= 2, "image too small");
  OVG_REQUIRE(F > 0 && outc >= 2 && outc <= 4, "bad arguments");
  OVG_REQUIRE(ovg_dpt_tail_supported(h, w, H, W, 128), "unsupported geometry (ovg_dpt_tail_supported)");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  CUtensorMap tb;
  int rc = get_map(w3x3, 9 * 128, 32, 0, 9 * 128, 32, &tb);
  if (rc) return rc;
  ovg::TailParams p{};
  p.src = reinterpret_cast<const uint16_t*>(src);
  if (tx) {
    float* gx = static_cast<float*>(scratch);
    float* gy = gx + 3LL * W * 32;
    ovg::TailTableParams tp{tx, ty, reinterpret_cast<const uint16_t*>(w3x3), gx, gy, H, W, f16 ? 1 : 0};
    ovg::tail_tables_kernel<<<dim3(W > H ? W : H, 2), 96, 0, st>>>(tp);
    rc = post_launch("ovg_dpt_tail(tables)");
    if (rc) return rc;
    p.gx = gx; p.gy = gy;
  }
  p.bias = bias; p.w2 = w2; p.b2 = b2; p.preds = preds; p.conf = conf;
  p.F = F; p.h = h; p.w = w; p.H = H; p.W = W;
  p.sy = H > 1 ? static_cast<float>(h - 1) / static_cast<float>(H - 1) : 0.f;
  p.sx = W > 1 ? static_cast<float>(w - 1) / static_cast<float>(W - 1) : 0.f;
  p.outc = outc; p.head_act = head_act; p.f16 = f16 ? 1 : 0;
  p.n_strips = (W + 127) / 128;
  // segments of rows per (frame, strip): about three work items per SM, each paying two halo rows
  const int sms = num_sms();
  int segs = (3 * sms + F * p.n_strips - 1) / (F * p.n_strips);
  if (segs < 1) segs = 1;
  if (segs > H) segs = H;
  p.seg_rows = (H + segs - 1) / segs;
  if (p.seg_rows < 8 && H >= 8) p.seg_rows = 8;
  p.n_segs = (H + p.seg_rows - 1) / p.seg_rows;
  p.n_items = F * p.n_strips * p.n_segs;
  p.prof = g_tail_prof;
  static PerDeviceOnce once;
  if (once.needed()) {
    OVG_CUDA(cudaFuncSetAttribute(ovg::fusedtail_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, ovg::FT_SMEM_BYTES));
    OVG_CUDA(cudaFuncSetAttribute(ovg::fusedtail_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, ovg::FT_SMEM_BYTES));
    once.mark_done();
  }
  const int grid = p.n_items < sms ? p.n_items : sms;
  if (p.f16) ovg::fusedtail_kernel<true><<<grid, ovg::FT_THREADS, ovg::FT_SMEM_BYTES, st>>>(tb, p);
  else ovg::fusedtail_kernel<false><<<grid, ovg::FT_THREADS, ovg::FT_SMEM_BYTES, st>>>(tb, p);
  return post_launch("ovg_dpt_tail");
}

int ovg_preprocess_image(const unsigned char* src, int h, int w, int nw, int nh, int crop, int fh, const int* hmin, const int* hcnt,
                         const int* hk, int hksize, const int* vmin, const int* vcnt, const int* vk, int vksize,
                         unsigned char* tmp, float* out, void* stream) {
  OVG_REQUIRE(src && out && h > 0 && w > 0 && nw > 0 && nh > 0 && crop >= 0 && fh > 0 && crop + fh <= nh, "bad geometry");
  OVG_REQUIRE(w == nw || (hmin && hcnt && hk && hksize > 0 && tmp), "horizontal pass needs its tap table and a temporary");
  OVG_REQUIRE(h == nh || (vmin && vcnt && vk && vksize > 0), "vertical pass needs its tap table");
  OVG_REQUIRE(h <= 65535 && fh <= 65535, "image too tall");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const unsigned char* mid = src;
  if (w != nw) {
    ovg::ResizeParams ph{src, tmp, nullptr, hmin, hcnt, hk, hksize, h, w, nw, 0, 0, 0};
    ovg::resize_h_u8_kernel<<<dim3((nw + 127) / 128, h), 128, 0, st>>>(ph);
    int rc = post_launch("ovg_preprocess_image(horizontal)");
    if (rc) return rc;
    mid = tmp;
  }
  ovg::ResizeParams pv{mid, nullptr, out, vmin, vcnt, vk, vksize, h, w, nw, crop, fh, h == nh ? 1 : 0};
  ovg::resize_v_u8_f32_kernel<<<dim3((nw + 127) / 128, fh), 128, 0, st>>>(pv);
  return post_launch("ovg_preprocess_image");
}

int ovg_preprocess_depth(const float* src, long long row_stride, long long col_stride, const int* sy, const int* sx, int crop,
                         int fh, int nw, float max_depth, float* depth, float* mask, void* stream) {
  OVG_REQUIRE(src && sy && sx && depth && mask && fh > 0 && nw > 0 && crop >= 0 && fh <= 65535, "bad arguments");
  ovg::DepthNearestParams p{src, row_stride, col_stride, sy, sx, depth, mask, crop, fh, nw, max_depth};
  ovg::depth_nearest_kernel<<<dim3((nw + 255) / 256, fh), 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(p);
  return post_launch("ovg_preprocess_depth");
}

int ovg_prepare_cameras(const float* c2w, const float* kin, const float* geom, const int* has, float* w2c, float* kout, int K,
                        void* stream) {
  OVG_REQUIRE(c2w && kin && geom && has && w2c && kout && K > 0, "bad arguments");
  ovg::CameraPrepParams p{c2w, kin, geom, has, w2c, kout, K};
  ovg::camera_prepare_kernel<<<(K + 63) / 64, 64, 0, reinterpret_cast<cudaStream_t>(stream)>>>(p);
  return post_launch("ovg_prepare_cameras");
}

int ovg_pose_decode(const float* pose_enc, float* extrinsic, float* intrinsic, float* cam2world, int K, int H, int W,
                    void* stream) {
  OVG_REQUIRE(pose_enc && extrinsic && K > 0 && H > 0 && W > 0, "bad arguments");
  ovg::PoseDecodeParams p{pose_enc, extrinsic, intrinsic, cam2world, K, static_cast<float>(H), static_cast<float>(W)};
  ovg::pose_decode_kernel<<<(K + 127) / 128, 128, 0, reinterpret_cast<cudaStream_t>(stream)>>>(p);
  return post_launch("ovg_pose_decode");
}

int ovg_unproject_depth(const float* depth, const float* intrinsic, const float* cam2world, float* world, int K, int H, int W,
                        void* stream) {
  OVG_REQUIRE(depth && intrinsic && cam2world && world && K > 0 && H > 0 && W > 0, "bad arguments");
  OVG_REQUIRE(K <= 65535, "too many frames");
  OVG_REQUIRE((reinterpret_cast<uintptr_t>(depth) & 15) == 0 && (reinterpret_cast<uintptr_t>(world) & 15) == 0,
              "depth / world must be 16-byte aligned");
  ovg::UnprojectParams p{depth, intrinsic, cam2world, world, K, H, W};
  const long long nq = (static_cast<long long>(H) * W + 3) / 4;
  int bx = static_cast<int>((nq + 255) / 256);
  const int cap = (num_sms() * 8 + K - 1) / K;       // ~8 blocks per SM over all frames, grid-stride inside
  if (bx > cap) bx = cap > 0 ? cap : 1;
  ovg::unproject_kernel<<<dim3(bx, K), 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(p);
  return post_launch("ovg_unproject_depth");
}

int ovg_conf_percentile_mask(const float* conf, long long n, float percent, float floor_, void* workspace,
                             unsigned char* mask, float* threshold_out, unsigned long long* count_out, void* stream) {
  OVG_REQUIRE(conf && workspace && mask && threshold_out && n > 0, "bad arguments");
  OVG_REQUIRE(percent >= 0.f && percent <= 100.f, "percent must be in [0, 100]");
  OVG_REQUIRE((reinterpret_cast<uintptr_t>(conf) & 15) == 0 && (reinterpret_cast<uintptr_t>(mask) & 3) == 0 &&
                  (reinterpret_cast<uintptr_t>(workspace) & 15) == 0,
              "conf must be 16-byte, mask 4-byte, workspace 16-byte aligned");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  // numpy.percentile(method="linear"): virtual index p/100 * (n - 1), linear interpolation between its two neighbours
  const double vi = static_cast<double>(percent) / 100.0 * static_cast<double>(n - 1);
  const unsigned long long r0 = static_cast<unsigned long long>(vi);
  const unsigned long long r1 = r0 + 1 < static_cast<unsigned long long>(n) ? r0 + 1 : r0;
  const double frac = vi - static_cast<double>(r0);
  // workspace: 6 x u64 state | 512 x u32 histograms | 3 x f32 results       (OVG_PERCENTILE_WORKSPACE_BYTES)
  unsigned long long* state = reinterpret_cast<unsigned long long*>(workspace);
  unsigned int* hist = reinterpret_cast<unsigned int*>(state + 6);
  float* res = reinterpret_cast<float*>(hist + 512);
  ovg::select_init_kernel<<<1, 128, 0, st>>>(state, hist, r0, r1, count_out);
  {
    int rc = post_launch("ovg_conf_percentile_mask(init)");
    if (rc) return rc;
  }
  int blocks = static_cast<int>((n / 4 + 255) / 256);
  if (blocks > num_sms() * 4) blocks = num_sms() * 4;
  if (blocks < 1) blocks = 1;
  for (int pass = 0; pass < 4; ++pass) {
    ovg::SelectParams sp{conf, n, state, hist, pass, res, static_cast<float>(frac)};
    ovg::select_hist_kernel<<<blocks, 256, 0, st>>>(sp);
    int rc = post_launch("ovg_conf_percentile_mask(hist)");
    if (rc) return rc;
    ovg::select_decide_kernel<<<1, 32, 0, st>>>(sp);
    rc = post_launch("ovg_conf_percentile_mask(decide)");
    if (rc) return rc;
  }
  OVG_CUDA(cudaMemcpyAsync(threshold_out, res + 2, sizeof(float), cudaMemcpyDeviceToDevice, st));
  ovg::ConfMaskParams mp{conf, res + 2, mask, n, floor_, count_out};
  ovg::conf_mask_kernel<<<blocks, 256, 0, st>>>(mp);
  return post_launch("ovg_conf_percentile_mask");
}

}  // extern "C"

#include "runtime.inc"
