// Persistent warp-specialised tcgen05 GEMM for sm_100a with fused epilogues.
//
//   D[M,N] = sum_taps A[m + tap_off[t], 0:Kc] * B[n, t*Kc:(t+1)*Kc]^T      (bf16 x bf16 -> fp32 in TMEM)
//
// One kernel serves every dense contraction on the hot path:
//   * aggregator linears  (reference layers/attention.py:52,:75, layers/mlp.py:35-38)  -- 1 tap
//   * DPT 1x1 / transposed convs (heads/dpt_head.py:69-96)                              -- 1 tap
//   * DPT 3x3 convs as 9 row-shifted GEMMs over a zero-bordered ("padded-linear") NHWC
//     layout (heads/dpt_head.py:326-354,:379-399,:115-126)                              -- 9 taps
// Roles: warp0 = TMA producer, warp1 = MMA issuer (+TMEM alloc), warps 2..9 = epilogue.
// Pipelines: smem full/empty ring (TMA<->MMA), 2 TMEM accumulator stages (MMA<->epilogue).
#pragma once
#include "ptx.cuh"

namespace ovg {

// EPI_QKV_GTAB: EPI_QKV for RoPE grids above GEMM_QKV_SMEM_POS positions (cos / sin read from global memory).  A separate
// instantiation, so that the code and register allocation of the EPI_QKV kernels do not change with it.
enum EpiKind { EPI_BF16 = 0, EPI_RESID = 1, EPI_QKV = 2, EPI_HEADTAIL = 3, EPI_QKV_GTAB = 4 };
enum RowMap { RM_IDENT = 0, RM_DENSE2PAD = 1, RM_PAD = 2, RM_PIXSHUF = 3 };

struct GemmParams {
  int M, N;
  int k_blocks;    // total 64-wide K blocks
  int kc_blocks;   // K blocks per tap
  int tap_off[9];  // A row offset of each tap
  // ---- common epilogue
  const float* bias;  // [N] ([cout] for RM_PIXSHUF) or nullptr
  int act;            // 0 none, 1 exact-erf GELU, 2 ReLU
  void* out;
  long long ldo;  // elements
  // ---- EPI_BF16
  const float* table;  // additive fp32 [table_rows][N] indexed by (m % table_rows), or nullptr
  int table_rows;
  int f16;                     // EPI_BF16 / EPI_HEADTAIL: operands, skips and the 16-bit output are IEEE half instead of bf16
  const __nv_bfloat16* skip1;  // optional addends, indexed like `out`
  const __nv_bfloat16* skip2;
  int rowmap;  // RowMap
  int gh, gw;  // source grid (rows are (frame, y, x)); RM_PAD: interior size of the padded domain
  int ps, cout;  // RM_PIXSHUF: stride (= kernel) and output channels
  // ---- EPI_RESID:  out(fp32)[row,n] += gamma[n] * (acc + bias[n]),  row = row_index ? row_index[m] : m
  const float* gamma;
  const int* row_index;
  int split_tail;  // pair kernel, BN = 256: the tiles of the last (partial) wave are issued as two 256 x 128 halves
  int staged;  // 1: epilogue output goes through smem + TMA (store for EPI_BF16, fp32 reduce-add for EPI_RESID)
  // ---- EPI_QKV (layers/attention.py:52-58 fused: bias, q/k LayerNorm(64), 2-D RoPE, head-major bf16)
  __nv_bfloat16* q_out;
  __nv_bfloat16* k_out;
  __nv_bfloat16* v_out;
  int C, ntok, T, nspecial, wp, maxpos;
  const float* qn_w;
  const float* qn_b;
  const float* kn_w;
  const float* kn_b;
  const float* rope_cos;  // [maxpos][16]
  const float* rope_sin;
  float qscale;  // softmax scale * log2(e), folded into q
  int qk_norm;   // 1: LayerNorm(64) on q,k (aggregator blocks); 0: plain (DINOv2 blocks)
  int rope;      // 1: 2-D RoPE on q,k
  // context parallelism: K and V rows of this rank's tokens are stored into every rank's full-length K / V buffer
  // ([batch*heads, peer_ntok, 64], this rank's tokens starting at row peer_tok_off) instead of k_out / v_out
  __nv_bfloat16* k_peer[8];
  __nv_bfloat16* v_peer[8];
  int n_peers;
  int peer_ntok;
  long long peer_tok_off;
  // ---- EPI_HEADTAIL (heads/dpt_head.py:121-126 + heads/head_act.py:61-112): relu, 1x1 32->outc, activation
  const float* w2;  // [outc][32]
  const float* b2;  // [outc]
  int outc;         // 2 (depth) or 4 (points)
  int head_act;     // 0 exp, 1 inverse-log
  float* preds;     // [F,gh,gw,outc-1]
  float* conf;      // [F,gh,gw]
};

constexpr int GEMM_BM = 128;
constexpr int GEMM_BK = 64;
constexpr int GEMM_THREADS = 320;
constexpr int GEMM_A_BYTES = GEMM_BM * GEMM_BK * 2;

// QKV epilogue: rope cos / sin / -sin for up to GEMM_QKV_SMEM_POS positions + q,k LayerNorm affine.  Larger RoPE grids
// (images above 63 patches per side) read cos / sin from the global fp32 tables instead, so this reservation -- and with
// it the pipeline depth of every GEMM -- does not grow with the image size.
constexpr int GEMM_QKV_SMEM_POS = 64;
constexpr int GEMM_QKV_TABLE_BYTES = 3 * GEMM_QKV_SMEM_POS * 18 * 4 + 1024;
template <int BN>
struct GemmCfg {
  static constexpr int B_BYTES = BN * GEMM_BK * 2;
  static constexpr int STAGE_BYTES = GEMM_A_BYTES + B_BYTES;
  static constexpr int STAGES = (BN >= 256) ? 4 : (BN >= 128 ? 6 : 8);
  static constexpr int TMEM_COLS = (2 * BN < 32) ? 32 : 2 * BN;
  static constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + 1024 /*align*/ + 256 /*barriers*/ + GEMM_QKV_TABLE_BYTES;
};

// Exact-erf GELU (nn.GELU() default, reference layers/mlp.py:22,:36) with erf evaluated by Abramowitz-Stegun 7.1.26
// (|abs err| <= 1.5e-7, three orders below the bf16 output resolution): 2 MUFU (rcp, ex2) + FMA-pipe work per element;
// erff() costs ~3x more and made the fc1 epilogue longer than its K = 1024 mainloop.
// Two values at a time on the packed fp32x2 pipes (FFMA2 / FMUL2): ~9 instead of ~16 issue slots per element for the
// scalar form.  The epilogue warps of the fc1 GEMM are issue-bound (2 warps per SM sub-partition, 32 768 GELUs per tile).
__device__ __forceinline__ float2 gelu_erf2(const float2 x) {
  const float2 z = make_float2(fabsf(x.x) * 0.70710678118654752f, fabsf(x.y) * 0.70710678118654752f);
  const float2 d = ffma2(make_float2(0.3275911f, 0.3275911f), z, make_float2(1.0f, 1.0f));
  float2 t;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(t.x) : "f"(d.x));
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(t.y) : "f"(d.y));
  float2 poly = ffma2(make_float2(1.061405429f, 1.061405429f), t, make_float2(-1.453152027f, -1.453152027f));
  poly = ffma2(poly, t, make_float2(1.421413741f, 1.421413741f));
  poly = ffma2(poly, t, make_float2(-0.284496736f, -0.284496736f));
  poly = ffma2(poly, t, make_float2(0.254829592f, 0.254829592f));
  poly = fmul2(poly, t);
  const float2 a = fmul2(fmul2(z, make_float2(-1.4426950408889634f, -1.4426950408889634f)), z);
  float2 e;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e.x) : "f"(a.x));
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e.y) : "f"(a.y));
  // erf_abs = 1 - poly * e;  gelu = 0.5 x (1 + sign(x) erf_abs) = 0.5 x + (0.5 |x|) (1 - poly e)
  const float2 hx = fmul2(x, make_float2(0.5f, 0.5f));
  const float2 hax = fmul2(z, make_float2(0.70710678118654752f, 0.70710678118654752f));   // 0.5 |x|
  const float2 w = ffma2(fmul2(poly, e), make_float2(-1.0f, -1.0f), make_float2(1.0f, 1.0f));
  return ffma2(hax, w, hx);
}

// One 128 x BN accumulator tile: TMEM -> registers -> fused epilogue -> global.  `trow` addresses this warp's TMEM lane
// quarter of the accumulator stage, `m` is this thread's global row, `colhalf` selects which column chunks this warp owns.
template <int BN, int EPI>
__device__ __forceinline__ void epilogue_tile(const GemmParams& p, const uint32_t trow, const int m, const int n0,
                                              const int colhalf, const float* s_rope, uint8_t* stg = nullptr,
                                              const CUtensorMap* tmO = nullptr, const CUtensorMap* tmO2 = nullptr,
                                              const CUtensorMap* tmO3 = nullptr) {
  if constexpr (EPI == EPI_QKV || EPI == EPI_QKV_GTAB) {
    // ---- per-row RoPE position (reference omnivggt_aggregator.py:215-224; layers/rope.py:39-59)
    int py = 0, px = 0;
    {
      const int t = m % p.T;
      if (t >= p.nspecial) {
        const int pp = t - p.nspecial;
        py = pp / p.wp + 1;
        px = pp % p.wp + 1;
      }
    }
    // smem tables (filled at kernel start): [cos | sin | -sin][64 positions][18] (16 frequencies, rows padded to 18
    // floats so that float2 reads stay aligned), then the q / k LayerNorm affine [qw*qscale | qb*qscale | kw | kb][64].
    const float2* cy = reinterpret_cast<const float2*>(s_rope + py * 18);
    const float2* sy = reinterpret_cast<const float2*>(s_rope + 64 * 18 + py * 18);
    const float2* nsy = reinterpret_cast<const float2*>(s_rope + 128 * 18 + py * 18);
    const float2* cx = reinterpret_cast<const float2*>(s_rope + px * 18);
    const float2* sx = reinterpret_cast<const float2*>(s_rope + 64 * 18 + px * 18);
    const float2* nsx = reinterpret_cast<const float2*>(s_rope + 128 * 18 + px * 18);
    const float* s_ln = s_rope + 3 * 64 * 18;
    const long long seq = m / p.ntok;
    const long long tok = m % p.ntok;
    const int heads = p.C >> 6;
    for (int c = colhalf; c < BN / 64; c += 2) {
      const int n = n0 + c * 64;
      uint32_t raw[64];
      tmem_ld32(trow + c * 64, raw);
      tmem_ld32(trow + c * 64 + 32, raw + 32);
      tmem_ld_wait();
      if (n >= p.N || m - static_cast<int>(threadIdx.x & 31) >= p.M) continue;   // warp-uniform
      const long long tok0 = __shfl_sync(0xffffffffu, tok, 0);   // all 32 lanes are converged here
      if (p.staged || m < p.M) {                               // staged: every lane of the warp takes part
        // all arithmetic on packed fp32 pairs (FADD2 / FMUL2 / FFMA2): v2[i] = elements (2i, 2i+1) of this head
        float2 v2[32];
        {
          const float4* b4 = reinterpret_cast<const float4*>(p.bias + n);
#pragma unroll
          for (int i = 0; i < 16; ++i) {
            const float4 b = __ldg(b4 + i);
            v2[2 * i] = fadd2(make_float2(__uint_as_float(raw[4 * i + 0]), __uint_as_float(raw[4 * i + 1])), make_float2(b.x, b.y));
            v2[2 * i + 1] = fadd2(make_float2(__uint_as_float(raw[4 * i + 2]), __uint_as_float(raw[4 * i + 3])), make_float2(b.z, b.w));
          }
        }
        const int which = n / p.C;
        const int h = (n - which * p.C) >> 6;
        if (which < 2 && p.qk_norm) {
          float2 s01 = make_float2(0.f, 0.f), s23 = make_float2(0.f, 0.f);
#pragma unroll
          for (int i = 0; i < 32; i += 2) {
            s01 = fadd2(s01, v2[i]);
            s23 = fadd2(s23, v2[i + 1]);
          }
          const float mean = ((s01.x + s01.y) + (s23.x + s23.y)) * (1.0f / 64.0f);
          const float2 nm = make_float2(-mean, -mean);
          float2 q01 = make_float2(0.f, 0.f), q23 = make_float2(0.f, 0.f);
#pragma unroll
          for (int i = 0; i < 32; i += 2) {
            v2[i] = fadd2(v2[i], nm);
            v2[i + 1] = fadd2(v2[i + 1], nm);
            q01 = ffma2(v2[i], v2[i], q01);
            q23 = ffma2(v2[i + 1], v2[i + 1], q23);
          }
          const float rstd = rsqrtf(((q01.x + q01.y) + (q23.x + q23.y)) * (1.0f / 64.0f) + 1e-5f);
          const float2 rr = make_float2(rstd, rstd);
          const float4* w4 = reinterpret_cast<const float4*>(s_ln + which * 128);        // q: pre-multiplied by qscale
          const float4* b4 = reinterpret_cast<const float4*>(s_ln + which * 128 + 64);
#pragma unroll
          for (int i = 0; i < 16; ++i) {
            const float4 w = w4[i];
            const float4 b = b4[i];
            v2[2 * i] = ffma2(fmul2(v2[2 * i], rr), make_float2(w.x, w.y), make_float2(b.x, b.y));
            v2[2 * i + 1] = ffma2(fmul2(v2[2 * i + 1], rr), make_float2(w.z, w.w), make_float2(b.z, b.w));
          }
        } else if (which == 0) {
          const float2 qs = make_float2(p.qscale, p.qscale);
#pragma unroll
          for (int i = 0; i < 32; ++i) v2[i] = fmul2(v2[i], qs);
        }
        if (EPI == EPI_QKV && which < 2 && p.rope) {
          // rotate (d, d+16) with the row angle and (32+d, 48+d) with the column angle (layers/rope.py:154-188)
#pragma unroll
          for (int k = 0; k < 8; ++k) {
            const float2 a0 = v2[k], b0 = v2[8 + k];
            v2[k] = ffma2(b0, nsy[k], fmul2(a0, cy[k]));
            v2[8 + k] = ffma2(a0, sy[k], fmul2(b0, cy[k]));
            const float2 a1 = v2[16 + k], b1 = v2[24 + k];
            v2[16 + k] = ffma2(b1, nsx[k], fmul2(a1, cx[k]));
            v2[24 + k] = ffma2(a1, sx[k], fmul2(b1, cx[k]));
          }
        } else if (EPI == EPI_QKV_GTAB && which < 2 && p.rope) {
          // more positions than the smem table holds: the same fp32 table entries straight from the global [maxpos][16]
          // tables (L1 / L2 resident: 147 positions are 19 KB), -sin negated in registers -- the same operands and
          // instructions as above, so both paths round identically
          const float2* gcy = reinterpret_cast<const float2*>(p.rope_cos + py * 16);
          const float2* gsy = reinterpret_cast<const float2*>(p.rope_sin + py * 16);
          const float2* gcx = reinterpret_cast<const float2*>(p.rope_cos + px * 16);
          const float2* gsx = reinterpret_cast<const float2*>(p.rope_sin + px * 16);
#pragma unroll
          for (int k = 0; k < 8; ++k) {
            const float2 c0 = __ldg(gcy + k), s0 = __ldg(gsy + k), c1 = __ldg(gcx + k), s1 = __ldg(gsx + k);
            const float2 a0 = v2[k], b0 = v2[8 + k];
            v2[k] = ffma2(b0, make_float2(-s0.x, -s0.y), fmul2(a0, c0));
            v2[8 + k] = ffma2(a0, s0, fmul2(b0, c0));
            const float2 a1 = v2[16 + k], b1 = v2[24 + k];
            v2[16 + k] = ffma2(b1, make_float2(-s1.x, -s1.y), fmul2(a1, c1));
            v2[24 + k] = ffma2(a1, s1, fmul2(b1, c1));
          }
        }
        // 32 rows x 128 B (one head of 32 tokens) -> 128B-swizzled smem tile -> one bulk tensor store into the
        // head-major [batch*heads, ntok, 64] output.  Direct stores (every lane a different 128 B row) kept the LSU
        // busy for ~20% of the kernel.  The few warps whose 32 rows straddle two sequences (or the end of the problem)
        // keep the direct path: a second bulk store at a negative token coordinate faults on sm_100.
        if (p.staged && tok0 + 32 <= p.ntok) {
          const int lane = threadIdx.x & 31;
          if (lane == 0) tma_store_wait_read0();
          __syncwarp();
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            uint4 o;
            o.x = pack_bf16(v2[4 * i + 0].x, v2[4 * i + 0].y);
            o.y = pack_bf16(v2[4 * i + 1].x, v2[4 * i + 1].y);
            o.z = pack_bf16(v2[4 * i + 2].x, v2[4 * i + 2].y);
            o.w = pack_bf16(v2[4 * i + 3].x, v2[4 * i + 3].y);
            *reinterpret_cast<uint4*>(stg + lane * 128 + ((i ^ (lane & 7)) << 4)) = o;
          }
          fence_proxy_async();
          __syncwarp();
          if (lane == 0) {
            const CUtensorMap* tm = which == 0 ? tmO : (which == 1 ? tmO2 : tmO3);
            const int bh = static_cast<int>(seq) * heads + h;     // lane 0: seq / tok of the warp's first row
            tma_store_3d(tm, stg, 0, static_cast<int>(tok), bh);
            tma_store_commit();
          }
          continue;
        }
        if (m >= p.M) continue;
        uint4 o8[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          o8[i].x = pack_bf16(v2[4 * i + 0].x, v2[4 * i + 0].y);
          o8[i].y = pack_bf16(v2[4 * i + 1].x, v2[4 * i + 1].y);
          o8[i].z = pack_bf16(v2[4 * i + 2].x, v2[4 * i + 2].y);
          o8[i].w = pack_bf16(v2[4 * i + 3].x, v2[4 * i + 3].y);
        }
        if (which > 0 && p.n_peers > 0) {
          // one 128-byte row per lane into every rank's buffer: plain stores over NVLink (peer-mapped memory)
          const long long roff = ((seq * heads + h) * p.peer_ntok + p.peer_tok_off + tok) * 64;
          for (int pr = 0; pr < p.n_peers; ++pr) {
            uint4* d4 = reinterpret_cast<uint4*>((which == 1 ? p.k_peer[pr] : p.v_peer[pr]) + roff);
#pragma unroll
            for (int i = 0; i < 8; ++i) d4[i] = o8[i];
          }
          continue;
        }
        uint4* d4 = reinterpret_cast<uint4*>((which == 0 ? p.q_out : (which == 1 ? p.k_out : p.v_out)) +
                                             ((seq * heads + h) * p.ntok + tok) * 64);
#pragma unroll
        for (int i = 0; i < 8; ++i) d4[i] = o8[i];
      }
    }
  } else {
    // ---- row mapping
    bool row_ok = m < p.M;
    bool interior = true;  // RM_PAD: border rows are written as zeros
    long long drow = m;
    int fr = 0, yy = 0, xx = 0;
    if (EPI == EPI_RESID) {
      if (p.row_index && row_ok) drow = p.row_index[m];
    }
    if (EPI == EPI_BF16 || EPI == EPI_HEADTAIL) {
      if (p.rowmap == RM_DENSE2PAD || p.rowmap == RM_PIXSHUF) {
        const int hw = p.gh * p.gw;
        fr = m / hw;
        const int rem = m - fr * hw;
        yy = rem / p.gw;
        xx = rem - yy * p.gw;
        if (p.rowmap == RM_DENSE2PAD)
          drow = (static_cast<long long>(fr) * (p.gh + 2) + (yy + 1)) * (p.gw + 2) + (xx + 1);
      } else if (p.rowmap == RM_PAD) {
        const int pw = p.gw + 2;
        const int pp = (p.gh + 2) * pw;
        fr = m / pp;
        const int rem = m - fr * pp;
        yy = rem / pw;
        xx = rem - yy * pw;
        interior = (yy >= 1 && yy <= p.gh && xx >= 1 && xx <= p.gw);
      }
    }
    for (int c = colhalf; c < BN / 32; c += 2) {
      const int n = n0 + c * 32;
      uint32_t raw[32];
      tmem_ld32(trow + c * 32, raw);
      tmem_ld_wait();
      if (n >= p.N) continue;                       // warp-uniform
      if (!p.staged && !row_ok) continue;           // staged: all lanes take part (TMA clips rows >= M)
      float v[32];
#pragma unroll
      for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(raw[i]);

      if constexpr (EPI == EPI_RESID) {
        if (p.staged) {
          // gamma * (acc + bias) -> swizzled fp32 smem tile [32 rows x 32 cols] of this warp -> TMA reduce-add into x.
          // The SM never reads x: the read-modify-write happens in L2, and the stores leave as whole 128 B rows.
          const int lane = threadIdx.x & 31;
          if (lane == 0) tma_store_wait_read0();      // previous chunk's bulk read of this buffer has finished
          __syncwarp();
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const float4 g = __ldg(reinterpret_cast<const float4*>(p.gamma + n) + i);
            const float4 b = __ldg(reinterpret_cast<const float4*>(p.bias + n) + i);
            const float2 o01 = fmul2(make_float2(g.x, g.y), fadd2(make_float2(v[4 * i + 0], v[4 * i + 1]), make_float2(b.x, b.y)));
            const float2 o23 = fmul2(make_float2(g.z, g.w), fadd2(make_float2(v[4 * i + 2], v[4 * i + 3]), make_float2(b.z, b.w)));
            *reinterpret_cast<float4*>(stg + lane * 128 + ((i ^ (lane & 7)) << 4)) = make_float4(o01.x, o01.y, o23.x, o23.y);
          }
          fence_proxy_async();
          __syncwarp();
          if (lane == 0) {
            tma_reduce_add_2d(tmO, stg, n, m - lane);
            tma_store_commit();
          }
          continue;
        }
        float* x = reinterpret_cast<float*>(p.out) + drow * p.ldo + n;
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          float4 xv = reinterpret_cast<float4*>(x)[i];
          const float4 g = __ldg(reinterpret_cast<const float4*>(p.gamma + n) + i);
          const float4 b = __ldg(reinterpret_cast<const float4*>(p.bias + n) + i);
          xv.x += g.x * (v[4 * i + 0] + b.x);
          xv.y += g.y * (v[4 * i + 1] + b.y);
          xv.z += g.z * (v[4 * i + 2] + b.z);
          xv.w += g.w * (v[4 * i + 3] + b.w);
          reinterpret_cast<float4*>(x)[i] = xv;
        }
      } else if constexpr (EPI == EPI_HEADTAIL) {
        if (!interior) continue;
#pragma unroll
        for (int i = 0; i < 32; ++i) v[i] = fmaxf(v[i] + __ldg(p.bias + i), 0.f);
        const long long pix = (static_cast<long long>(fr) * p.gh + (yy - 1)) * p.gw + (xx - 1);
        for (int o = 0; o < p.outc; ++o) {
          float acc = __ldg(p.b2 + o);
#pragma unroll
          for (int i = 0; i < 32; ++i) acc += __ldg(p.w2 + o * 32 + i) * v[i];
          if (o == p.outc - 1) {
            p.conf[pix] = 1.0f + expf(acc);
          } else {
            const float y = p.head_act == 0 ? expf(acc) : copysignf(expm1f(fabsf(acc)), acc);
            p.preds[pix * (p.outc - 1) + o] = y;
          }
        }
      } else {  // EPI_BF16
        int bn = n;      // bias / channel index
        long long dcol = n;
        if (p.rowmap == RM_PIXSHUF) {
          const int kk = n / p.cout;
          bn = n - kk * p.cout;
          const int ky = kk / p.ps, kx = kk - ky * p.ps;
          const int oh = p.gh * p.ps, ow = p.gw * p.ps;
          drow = (static_cast<long long>(fr) * (oh + 2) + (yy * p.ps + ky + 1)) * (ow + 2) + (xx * p.ps + kx + 1);
          dcol = bn;
        }
        if (p.bias) {
          const float4* b4 = reinterpret_cast<const float4*>(p.bias + bn);
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const float4 b = __ldg(b4 + i);
            const float2 s01 = fadd2(make_float2(v[4 * i + 0], v[4 * i + 1]), make_float2(b.x, b.y));
            const float2 s23 = fadd2(make_float2(v[4 * i + 2], v[4 * i + 3]), make_float2(b.z, b.w));
            v[4 * i + 0] = s01.x; v[4 * i + 1] = s01.y; v[4 * i + 2] = s23.x; v[4 * i + 3] = s23.y;
          }
        }
        if (p.table) {
          const float* t = p.table + static_cast<long long>(m % p.table_rows) * p.N + n;
#pragma unroll
          for (int i = 0; i < 32; ++i) v[i] += __ldg(t + i);
        }
        const long long off = drow * p.ldo + dcol;
        if (p.skip1 && row_ok) {
          const uint4* s4 = reinterpret_cast<const uint4*>(p.skip1 + off);
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const uint4 sv = __ldg(s4 + i);
            const float2 s0 = unpack_h(sv.x, p.f16), s1 = unpack_h(sv.y, p.f16), s2 = unpack_h(sv.z, p.f16), s3 = unpack_h(sv.w, p.f16);
            v[8 * i + 0] += s0.x; v[8 * i + 1] += s0.y;
            v[8 * i + 2] += s1.x; v[8 * i + 3] += s1.y;
            v[8 * i + 4] += s2.x; v[8 * i + 5] += s2.y;
            v[8 * i + 6] += s3.x; v[8 * i + 7] += s3.y;
          }
        }
        if (p.skip2 && row_ok) {
          const uint4* s4 = reinterpret_cast<const uint4*>(p.skip2 + off);
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const uint4 sv = __ldg(s4 + i);
            const float2 s0 = unpack_h(sv.x, p.f16), s1 = unpack_h(sv.y, p.f16), s2 = unpack_h(sv.z, p.f16), s3 = unpack_h(sv.w, p.f16);
            v[8 * i + 0] += s0.x; v[8 * i + 1] += s0.y;
            v[8 * i + 2] += s1.x; v[8 * i + 3] += s1.y;
            v[8 * i + 4] += s2.x; v[8 * i + 5] += s2.y;
            v[8 * i + 6] += s3.x; v[8 * i + 7] += s3.y;
          }
        }
        if (p.act == 1) {
#pragma unroll
          for (int i = 0; i < 32; i += 2) {
            const float2 g = gelu_erf2(make_float2(v[i], v[i + 1]));
            v[i] = g.x;
            v[i + 1] = g.y;
          }
        } else if (p.act == 2) {
#pragma unroll
          for (int i = 0; i < 32; ++i) v[i] = fmaxf(v[i], 0.f);
        }
        if (!interior) {
#pragma unroll
          for (int i = 0; i < 32; ++i) v[i] = 0.f;
        }
        if (p.staged) {
          const int lane = threadIdx.x & 31;
          if (lane == 0) tma_store_wait_read0();
          __syncwarp();
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            uint4 o;
            o.x = pack_h(v[8 * i + 0], v[8 * i + 1], p.f16);
            o.y = pack_h(v[8 * i + 2], v[8 * i + 3], p.f16);
            o.z = pack_h(v[8 * i + 4], v[8 * i + 5], p.f16);
            o.w = pack_h(v[8 * i + 6], v[8 * i + 7], p.f16);
            *reinterpret_cast<uint4*>(stg + lane * 64 + ((i ^ ((lane >> 1) & 3)) << 4)) = o;   // 64B-swizzled tile
          }
          fence_proxy_async();
          __syncwarp();
          if (lane == 0) {
            tma_store_2d(tmO, stg, n, m - lane);
            tma_store_commit();
          }
          continue;
        }
        uint4* d4 = reinterpret_cast<uint4*>(reinterpret_cast<__nv_bfloat16*>(p.out) + off);
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          uint4 o;
          o.x = pack_h(v[8 * i + 0], v[8 * i + 1], p.f16);
          o.y = pack_h(v[8 * i + 2], v[8 * i + 3], p.f16);
          o.z = pack_h(v[8 * i + 4], v[8 * i + 5], p.f16);
          o.w = pack_h(v[8 * i + 6], v[8 * i + 7], p.f16);
          d4[i] = o;
        }
      }
    }
  }
}

template <int BN, int EPI>
__global__ void __launch_bounds__(GEMM_THREADS, 1)
gemm_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, const GemmParams p) {
  using Cfg = GemmCfg<BN>;
  constexpr int STAGES = Cfg::STAGES;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* sA = smem;
  uint8_t* sB = smem + STAGES * GEMM_A_BYTES;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + STAGES * Cfg::STAGE_BYTES);
  uint64_t* full = bars;
  uint64_t* empty = bars + STAGES;
  uint64_t* tfull = bars + 2 * STAGES;
  uint64_t* tempty = bars + 2 * STAGES + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * STAGES + 4);
  float* s_rope = reinterpret_cast<float*>(smem + STAGES * Cfg::STAGE_BYTES + 256);  // [3][64][18] + [4][64]

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int m_tiles = (p.M + GEMM_BM - 1) / GEMM_BM;
  const int n_tiles = (p.N + BN - 1) / BN;
  const int num_tiles = m_tiles * n_tiles;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
    for (int i = 0; i < STAGES; ++i) {
      mbar_init(&full[i], 1);
      mbar_init(&empty[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&tfull[i], 1);
      mbar_init(&tempty[i], 8);
    }
    fence_barrier_init();
  }
  if (warp == 1) {
    tmem_alloc(tmem_slot, Cfg::TMEM_COLS);
    tmem_relinquish();
  }
  if ((EPI == EPI_QKV || EPI == EPI_QKV_GTAB) && warp >= 2) {
    for (int i = threadIdx.x - 64; EPI == EPI_QKV && i < p.maxpos * 16; i += GEMM_THREADS - 64) {   // GTAB: tables stay in global memory
      s_rope[(i >> 4) * 18 + (i & 15)] = p.rope_cos[i];
      s_rope[64 * 18 + (i >> 4) * 18 + (i & 15)] = p.rope_sin[i];
      s_rope[128 * 18 + (i >> 4) * 18 + (i & 15)] = -p.rope_sin[i];
    }
    if (p.qk_norm && threadIdx.x >= 64 && threadIdx.x < 128) {
      float* s_ln = s_rope + 3 * 64 * 18;
      const int i = threadIdx.x - 64;
      s_ln[i] = p.qn_w[i] * p.qscale;          // q is pre-scaled by log2(e)/sqrt(head_dim): fold it into the affine
      s_ln[64 + i] = p.qn_b[i] * p.qscale;
      s_ln[128 + i] = p.kn_w[i];
      s_ln[192 + i] = p.kn_b[i];
    }
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ===================== TMA producer =====================
    if (lane == 0) {
      int s = 0;
      uint32_t ph = 0;
      for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
        const int m0 = (tile / n_tiles) * GEMM_BM;
        const int n0 = (tile % n_tiles) * BN;
        for (int kb = 0; kb < p.k_blocks; ++kb) {
          mbar_wait(&empty[s], ph ^ 1);
          mbar_expect_tx(&full[s], Cfg::STAGE_BYTES);
          const int tap = kb / p.kc_blocks;
          const int c0 = (kb - tap * p.kc_blocks) * GEMM_BK;
          tma_load_2d(sA + s * GEMM_A_BYTES, &tmA, &full[s], c0, m0 + p.tap_off[tap]);
          tma_load_2d(sB + s * Cfg::B_BYTES, &tmB, &full[s], kb * GEMM_BK, n0);
          if (++s == STAGES) {
            s = 0;
            ph ^= 1;
          }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    if (lane == 0) {
      const uint32_t idesc = make_idesc_bf16(GEMM_BM, BN, 0, 0) & ~(p.f16 ? IDESC_BF16_BITS : 0u);
      int s = 0;
      uint32_t ph = 0;
      int as = 0;
      uint32_t aph = 0;
      for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
        mbar_wait(&tempty[as], aph ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + as * BN;
        for (int kb = 0; kb < p.k_blocks; ++kb) {
          mbar_wait(&full[s], ph);
          tc_fence_after();
          const uint64_t adesc = make_sw128_desc(smem_u32(sA + s * GEMM_A_BYTES));
          const uint64_t bdesc = make_sw128_desc(smem_u32(sB + s * Cfg::B_BYTES));
#pragma unroll
          for (int k = 0; k < GEMM_BK / 16; ++k) {
            umma_ss(d_tmem, adesc + 2 * k, bdesc + 2 * k, idesc, (kb | k) != 0 ? 1u : 0u);
          }
          umma_commit(&empty[s]);
          if (++s == STAGES) {
            s = 0;
            ph ^= 1;
          }
        }
        umma_commit(&tfull[as]);
        if (++as == 2) {
          as = 0;
          aph ^= 1;
        }
      }
    }
  } else {
    // ===================== epilogue (8 warps) =====================
    const int e = warp - 2;
    const int quarter = warp & 3;  // TMEM lanes accessible to this warp: 32*(warp%4)..+31
    const int colhalf = e >> 2;
    const int r = quarter * 32 + lane;
    int as = 0;
    uint32_t aph = 0;
    for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
      const int m0 = (tile / n_tiles) * GEMM_BM;
      const int n0 = (tile % n_tiles) * BN;
      const int m = m0 + r;
      mbar_wait(&tfull[as], aph);
      tc_fence_after();
      const uint32_t trow = tmem_base + as * BN + (static_cast<uint32_t>(quarter * 32) << 16);

      epilogue_tile<BN, EPI>(p, trow, m, n0, colhalf, s_rope);
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tempty[as]);
      if (++as == 2) {
        as = 0;
        aph ^= 1;
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, Cfg::TMEM_COLS);
  }
}


// =====================================================================================================================
// CTA-pair variant (cta_group::2): one 256 x 256 output tile per 2-SM cluster.  Each CTA stages its own 128 rows of A and
// 128 of the 256 B rows per K block (32 KB/stage instead of 48 KB for the same FLOPs), which is what matters here: a
// 128 x 256 single-CTA tile needs ~87 FLOP per L2->SM byte and saturates the L2 fabric (~10-12 TB/s) near 1 PFLOP/s;
// the paired tile needs 131 FLOP/B.  The pair leader issues M=256 MMAs that write both CTAs' TMEM; every CTA runs its own
// TMA producer and epilogue (rows [128*rank, 128*rank+128) of the tile).
// ---------------------------------------------------------------------------------------------------------------------
// DPT output tail at full resolution (heads/dpt_head.py:121-126,:255-260): 3x3 conv 128 -> 32 over the zero-bordered NHWC
// map + ReLU + 1x1 conv + activations.  With N = 32 the generic 9-tap path is bound by L2->SM traffic: it re-loads the
// 128 x 64 A tile for every tap (18 loads of 16 KB per 128 output pixels).  Here the three horizontal taps of one kernel
// row read ONE smem block of 136 rows through row-shifted UMMA descriptors (start address + kx * 128 B), so a tile needs 6
// A loads instead of 18, and the 72 KB of weights are loaded once per CTA and stay resident.
constexpr int HT_A_ROWS = 136;
constexpr int HT_A_BYTES = HT_A_ROWS * 128;          // 17 408 = 17 swizzle atoms
constexpr int HT_STAGES = 6;
constexpr int HT_B_TILE = 32 * 128;                  // one [32 x 64] bf16 weight tile
constexpr int HT_B_BYTES = 18 * HT_B_TILE;           // 9 taps x 2 K blocks
constexpr int HT_SMEM_BYTES = HT_STAGES * HT_A_BYTES + HT_B_BYTES + 1024 + 256;

__global__ void __launch_bounds__(GEMM_THREADS, 1)
headtail_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, const GemmParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* sA = smem;
  uint8_t* sB = smem + HT_STAGES * HT_A_BYTES;
  uint64_t* bars = reinterpret_cast<uint64_t*>(sB + HT_B_BYTES);
  uint64_t* full = bars;
  uint64_t* empty = bars + HT_STAGES;
  uint64_t* tfull = bars + 2 * HT_STAGES;
  uint64_t* tempty = tfull + 2;
  uint64_t* bfull = tempty + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bfull + 1);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int num_tiles = (p.M + GEMM_BM - 1) / GEMM_BM;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
    for (int i = 0; i < HT_STAGES; ++i) {
      mbar_init(&full[i], 1);
      mbar_init(&empty[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&tfull[i], 1);
      mbar_init(&tempty[i], 4);
    }
    mbar_init(bfull, 1);
    fence_barrier_init();
  }
  if (warp == 1) {
    tmem_alloc(tmem_slot, 64);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    if (lane == 0) {
      mbar_expect_tx(bfull, HT_B_BYTES);
      for (int t = 0; t < 18; ++t) tma_load_2d(sB + t * HT_B_TILE, &tmB, bfull, t * GEMM_BK, 0);
      int s = 0;
      uint32_t ph = 0;
      for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
        const int m0 = tile * GEMM_BM;
        for (int ky = 0; ky < 3; ++ky) {
          const int row0 = m0 + p.tap_off[ky * 3 + 1] - 1;     // first row the kx = 0 tap reads
          for (int kb = 0; kb < 2; ++kb) {
            mbar_wait(&empty[s], ph ^ 1);
            mbar_expect_tx(&full[s], HT_A_BYTES);
            tma_load_2d(sA + s * HT_A_BYTES, &tmA, &full[s], kb * GEMM_BK, row0);
            if (++s == HT_STAGES) {
              s = 0;
              ph ^= 1;
            }
          }
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      const uint32_t idesc = make_idesc_bf16(GEMM_BM, 32, 0, 0) & ~(p.f16 ? IDESC_BF16_BITS : 0u);
      int s = 0;
      uint32_t ph = 0;
      int as = 0;
      uint32_t aph = 0;
      mbar_wait(bfull, 0);
      for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
        mbar_wait(&tempty[as], aph ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + as * 32;
        for (int ky = 0; ky < 3; ++ky) {
          for (int kb = 0; kb < 2; ++kb) {
            mbar_wait(&full[s], ph);
            tc_fence_after();
            const uint32_t a_atom = smem_u32(sA + s * HT_A_BYTES);
#pragma unroll
            for (int kx = 0; kx < 3; ++kx) {
              const uint64_t adesc = make_sw128_desc_rows(a_atom, kx);
              const uint64_t bdesc = make_sw128_desc(smem_u32(sB + ((ky * 3 + kx) * 2 + kb) * HT_B_TILE));
#pragma unroll
              for (int k = 0; k < GEMM_BK / 16; ++k)
                umma_ss(d_tmem, adesc + 2 * k, bdesc + 2 * k, idesc, (ky | kb | kx | k) != 0 ? 1u : 0u);
            }
            umma_commit(&empty[s]);
            if (++s == HT_STAGES) {
              s = 0;
              ph ^= 1;
            }
          }
        }
        umma_commit(&tfull[as]);
        if (++as == 2) {
          as = 0;
          aph ^= 1;
        }
      }
    }
  } else {
    // The tile is only 32 columns wide, so a column split would leave half of the epilogue warps idle; instead the two
    // warp sets (2-5, 6-9) own one accumulator stage each and take alternate tiles (the per-row 1x1 conv + activations
    // + strided fp32 stores are latency-bound).
    const int quarter = warp & 3;
    const int eset = (warp - 2) >> 2;          // == accumulator stage this warp set serves
    const int r = quarter * 32 + lane;
    uint32_t aph = 0;
    int seq = 0;
    for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x, ++seq) {
      if ((seq & 1) != eset) continue;
      const int m = tile * GEMM_BM + r;
      mbar_wait(&tfull[eset], aph);
      tc_fence_after();
      const uint32_t trow = tmem_base + eset * 32 + (static_cast<uint32_t>(quarter * 32) << 16);
      epilogue_tile<32, EPI_HEADTAIL>(p, trow, m, 0, 0, nullptr);
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tempty[eset]);
      aph ^= 1;
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 64);
  }
}

constexpr int GEMM2_STG_BYTES = 8 * 4096;   // one 32 x 32 fp32 (or bf16) staging tile per epilogue warp; followed by the QKV tables
template <int BN>
struct Gemm2Cfg {
#ifndef OVG_GEMM2_STAGES
#define OVG_GEMM2_STAGES 5
#endif
  static constexpr int STAGES = BN >= 256 ? OVG_GEMM2_STAGES : 7;
  static constexpr int B_BYTES = (BN / 2) * GEMM_BK * 2;       // each CTA stages half of the B rows
  static constexpr int STAGE_BYTES = GEMM_A_BYTES + B_BYTES;
  static constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + 1024 + 256 + 1024 + GEMM2_STG_BYTES + GEMM_QKV_TABLE_BYTES;
};

template <int BN, int EPI>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(GEMM_THREADS, 1)
gemm2_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
             const __grid_constant__ CUtensorMap tmBh, const __grid_constant__ CUtensorMap tmO,
             const __grid_constant__ CUtensorMap tmO2, const __grid_constant__ CUtensorMap tmO3, const GemmParams p) {
  using Cfg2 = Gemm2Cfg<BN>;
  constexpr int STAGES = Cfg2::STAGES;
  constexpr int GEMM2_B_BYTES = Cfg2::B_BYTES;
  constexpr int GEMM2_STAGE_BYTES = Cfg2::STAGE_BYTES;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* sA = smem;
  uint8_t* sB = smem + STAGES * GEMM_A_BYTES;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + STAGES * GEMM2_STAGE_BYTES);
  uint64_t* full = bars;                    // used in the leader only: its arrive.expect_tx covers both CTAs' bytes
  uint64_t* empty = bars + STAGES;          // per CTA: multicast MMA commit
  uint64_t* tfull = bars + 2 * STAGES;      // per CTA: multicast MMA commit
  uint64_t* tempty = bars + 2 * STAGES + 2; // used in the leader only: 8 epilogue warps x 2 CTAs
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * STAGES + 4);
  uint8_t* s_stage = smem + STAGES * GEMM2_STAGE_BYTES + 1024;     // 1024-aligned: swizzled TMA-store tiles
  float* s_rope = reinterpret_cast<float*>(s_stage + GEMM2_STG_BYTES);   // QKV epilogue tables

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const bool leader = rank == 0;
  const int cluster_id = blockIdx.x >> 1;
  const int num_clusters = gridDim.x >> 1;
  const int m_tiles = (p.M + 255) / 256;
  const int n_tiles = (p.N + BN - 1) / BN;
  const int num_tiles = m_tiles * n_tiles;
  // Wave quantisation: with T tiles on G clusters the last wave holds T mod G tiles and the other clusters idle for a
  // whole tile time (proj / fc2 at cfg2: 172 tiles on 74 clusters = 2.32 waves, paid as 3).  When that remainder fits
  // twice into the machine its tiles are issued as two 256 x 128 halves (tmBh: 64 B rows per CTA, N = 128 MMAs, the
  // BN = 128 epilogue), so the tail costs half a tile time.  All three roles walk the same sequence `it`.
  const int full_tiles = (BN == 256 && p.split_tail) ? (num_tiles / num_clusters) * num_clusters : num_tiles;
  const int num_items = full_tiles + 2 * (num_tiles - full_tiles);
#define OVG_GEMM2_ITEM(it)                                                          \
  const bool half_tile = (it) >= full_tiles;                                        \
  const int tile = half_tile ? full_tiles + (((it) - full_tiles) >> 1) : (it);      \
  const int hsel = half_tile ? (((it) - full_tiles) & 1) : 0;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
    if (BN == 256 && p.split_tail) tma_prefetch_desc(&tmBh);
    if (p.staged) {
      tma_prefetch_desc(&tmO);
      if (EPI == EPI_QKV || EPI == EPI_QKV_GTAB) {
        tma_prefetch_desc(&tmO2);
        tma_prefetch_desc(&tmO3);
      }
    }
    for (int i = 0; i < STAGES; ++i) {
      mbar_init(&full[i], 1);
      mbar_init(&empty[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&tfull[i], 1);
      mbar_init(&tempty[i], 16);
    }
    fence_barrier_init();
  }
  if (warp == 1) {
    tmem_alloc_2sm(tmem_slot, 2 * BN);
    tmem_relinquish_2sm();
  }
  if ((EPI == EPI_QKV || EPI == EPI_QKV_GTAB) && warp >= 2) {
    for (int i = threadIdx.x - 64; EPI == EPI_QKV && i < p.maxpos * 16; i += GEMM_THREADS - 64) {   // GTAB: tables stay in global memory
      s_rope[(i >> 4) * 18 + (i & 15)] = p.rope_cos[i];
      s_rope[64 * 18 + (i >> 4) * 18 + (i & 15)] = p.rope_sin[i];
      s_rope[128 * 18 + (i >> 4) * 18 + (i & 15)] = -p.rope_sin[i];
    }
    if (p.qk_norm && threadIdx.x >= 64 && threadIdx.x < 128) {
      float* s_ln = s_rope + 3 * 64 * 18;
      const int i = threadIdx.x - 64;
      s_ln[i] = p.qn_w[i] * p.qscale;          // q is pre-scaled by log2(e)/sqrt(head_dim): fold it into the affine
      s_ln[64 + i] = p.qn_b[i] * p.qscale;
      s_ln[128 + i] = p.kn_w[i];
      s_ln[192 + i] = p.kn_b[i];
    }
  }
  tc_fence_before();
  cluster_sync();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ===================== TMA producer (both CTAs) =====================
    if (lane == 0) {
      int s = 0;
      uint32_t ph = 0;
      for (int it = cluster_id; it < num_items; it += num_clusters) {
        OVG_GEMM2_ITEM(it)
        const int m0 = (tile / n_tiles) * 256 + static_cast<int>(rank) * 128;
        const int n0 = half_tile ? (tile % n_tiles) * BN + hsel * (BN / 2) + static_cast<int>(rank) * (BN / 4)
                                 : (tile % n_tiles) * BN + static_cast<int>(rank) * (BN / 2);
        const uint32_t stage_tx = half_tile ? GEMM_A_BYTES + GEMM2_B_BYTES / 2 : GEMM2_STAGE_BYTES;
        for (int kb = 0; kb < p.k_blocks; ++kb) {
          mbar_wait(&empty[s], ph ^ 1);
          const uint32_t lead_full = mapa_u32(smem_u32(&full[s]), 0);
          // Only the leader arrives; the peer's TMA bytes are accounted for by the leader's expect_tx (the transaction
          // count may go transiently negative, which mbarrier allows).  The peer cannot run a phase ahead: it refills
          // stage s only after the MMA that consumed the previous fill has committed to its empty[s].
          if (leader) mbar_expect_tx(&full[s], 2 * stage_tx);
          const int tap = kb / p.kc_blocks;
          const int c0 = (kb - tap * p.kc_blocks) * GEMM_BK;
          tma_load_2d_2sm(sA + s * GEMM_A_BYTES, &tmA, lead_full, c0, m0 + p.tap_off[tap]);
          tma_load_2d_2sm(sB + s * GEMM2_B_BYTES, half_tile ? &tmBh : &tmB, lead_full, kb * GEMM_BK, n0);
          if (++s == STAGES) {
            s = 0;
            ph ^= 1;
          }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer (pair leader only) =====================
    if (leader && lane == 0) {
      const uint32_t fmt_clear = ~(p.f16 ? IDESC_BF16_BITS : 0u);
      const uint32_t idesc_full = make_idesc_bf16(256, BN, 0, 0) & fmt_clear;
      const uint32_t idesc_half = make_idesc_bf16(256, BN / 2, 0, 0) & fmt_clear;
      int s = 0;
      uint32_t ph = 0;
      int as = 0;
      uint32_t aph = 0;
      for (int it = cluster_id; it < num_items; it += num_clusters) {
        const uint32_t idesc = it >= full_tiles ? idesc_half : idesc_full;
        mbar_wait(&tempty[as], aph ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + as * BN;
        for (int kb = 0; kb < p.k_blocks; ++kb) {
          mbar_wait(&full[s], ph);
          tc_fence_after();
          const uint64_t adesc = make_sw128_desc(smem_u32(sA + s * GEMM_A_BYTES));
          const uint64_t bdesc = make_sw128_desc(smem_u32(sB + s * GEMM2_B_BYTES));
#pragma unroll
          for (int k = 0; k < GEMM_BK / 16; ++k)
            umma_ss_2sm(d_tmem, adesc + 2 * k, bdesc + 2 * k, idesc, (kb | k) != 0 ? 1u : 0u);
          umma_commit_2sm(&empty[s], 3);
          if (++s == STAGES) {
            s = 0;
            ph ^= 1;
          }
        }
        umma_commit_2sm(&tfull[as], 3);
        if (++as == 2) {
          as = 0;
          aph ^= 1;
        }
      }
    }
  } else {
    // ===================== epilogue (8 warps per CTA) =====================
    const int quarter = warp & 3;
    const int colhalf = (warp - 2) >> 2;
    const int r = quarter * 32 + lane;
    int as = 0;
    uint32_t aph = 0;
    for (int it = cluster_id; it < num_items; it += num_clusters) {
      OVG_GEMM2_ITEM(it)
      const int m = (tile / n_tiles) * 256 + static_cast<int>(rank) * 128 + r;
      const int n0 = (tile % n_tiles) * BN + hsel * (BN / 2);
      mbar_wait(&tfull[as], aph);
      tc_fence_after();
      const uint32_t trow = tmem_base + as * BN + (static_cast<uint32_t>(quarter * 32) << 16);
      if (half_tile)
        epilogue_tile<BN / 2, EPI>(p, trow, m, n0, colhalf, s_rope, s_stage + (warp - 2) * 4096, &tmO, &tmO2, &tmO3);
      else
        epilogue_tile<BN, EPI>(p, trow, m, n0, colhalf, s_rope, s_stage + (warp - 2) * 4096, &tmO, &tmO2, &tmO3);
      tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        if (leader) mbar_arrive(&tempty[as]);
        else mbar_arrive_cluster(mapa_u32(smem_u32(&tempty[as]), 0));
      }
      if (++as == 2) {
        as = 0;
        aph ^= 1;
      }
    }
  }
#undef OVG_GEMM2_ITEM
  if (p.staged && warp >= 2 && lane == 0) tma_store_wait_all();   // bulk stores issued by this thread have completed
  tc_fence_before();
  cluster_sync();   // the peer may still signal barriers / read smem of this CTA until both are done
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc_2sm(tmem_base, 2 * BN);
  }
}

}  // namespace ovg
