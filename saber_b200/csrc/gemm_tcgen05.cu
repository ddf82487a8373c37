// saber_b200 — bf16 GEMM on the 5th-gen tensor cores (tcgen05.mma, accumulators in TMEM, operands
// staged by TMA with 128-byte swizzle), persistent, warp-specialised, with fused epilogues:
//
//   STD : out[m,n] = act(alpha * sum_k A[m,k] W[n,k] + bias[n]) + residual[m (mod res_mod), n]
//   LN  : out[m,:] = LayerNorm_N(acc + bias + residual) * gamma + beta            (N <= tile width)
//   UP1 : mask-decoder output_upscaling[0..2]: ConvTranspose2d(256->64,k2,s2) as a GEMM whose epilogue does the
//         pixel shuffle, adds the high-res skip (feat_s1), LayerNorm2d(64) and GELU            (N = 4*64)
//   UP2 : output_upscaling[3..4] + hyper-network product: ConvTranspose2d(64->32,k2,s2), + feat_s0, GELU, then the
//         dot product with the 4 hyper-network vectors of the prompt -> 4 mask logits per output pixel (N = 4*32)
//
// This one kernel carries every Linear / 1x1-conv / im2col'd conv / transposed-conv of the SAM2 path (Hiera
// QKV / proj / MLP, FPN laterals, mask-decoder projections and MLPs). Replaces the cuBLASLt / cuDNN calls made by
// torch inside upstream sam2, reached from REF saber/adapters/sam2/predictor.py:24-26 and automask.py:62
// (SURVEY §8a U1/U3). The fused epilogues remove the fp32 round trips of sam2/modeling/sam/transformer.py
// (norm4 after cross_attn_image_to_token) and mask_decoder.py (output_upscaling, hyper_in @ upscaled_embedding).
//
// Roles (384 threads, 1 CTA / SM): warp0 = TMA producer, warp1 = MMA issuer (one elected lane), warp2 = TMEM
// allocator, warps 4-7 = epilogue set 0, warps 8-11 = epilogue set 1. TMEM holds two accumulator stages; set s
// drains stage s, so two tile epilogues (the bottleneck of the small-K, HBM-bound GEMMs of this model) run
// concurrently and overlap the main loop of the following tiles. Inside an epilogue the TMEM load and the residual
// loads of column chunk c+1 are issued before chunk c is processed.
#include "common.cuh"
#include <stdlib.h>

namespace {

constexpr int BM = 128;
constexpr int BK = 64;  // 64 bf16 = 128 B = one swizzle row
constexpr int CH = 16;  // epilogue column chunk
constexpr int NTHREADS = 384;   // 4 role warps + 8 epilogue warps

enum { EPI_STD = 0, EPI_LN = 1, EPI_UP1 = 2, EPI_UP2 = 3 };

struct GemmParams {
  int M, N, K;
  void* out;
  long long ldo;
  int out_f32;
  const float* bias;
  int act;  // 0 none, 1 gelu(erf), 2 relu, 3 sigmoid
  const void* res;
  long long ldr;
  int res_f32;
  int res_mod;  // 0: residual row = m ; >0: residual row = m % res_mod (broadcast over batch)
  float alpha;
  // fused epilogues
  const float* gamma;
  const float* beta;
  float eps;
  const float* skip;          // UP1: feat_s1 [.., (2h)(2w), 64] fp32 ; UP2: feat_s0 [.., (2h)(2w), 32] fp32
  long long skip_bstride;     // elements between batch entries of skip (0 = shared by all prompts)
  const float* hyper;         // UP2: [B, 4, 32] fp32
  int gh, gw;                 // input token grid of the transposed conv (rows m = (b, y, x), y < gh, x < gw)
  unsigned long long* prof;   // optional (sb_gemm_set_prof): 8 clock counters summed over CTAs, see sb_gemm_set_prof
  // UP1 / UP2 on a device-side prompt list: only the prompts plist[0 .. *pcount) are processed (rows of prompt b are
  // b * gh * gw ...); the other prompts' outputs are left untouched. nullptr = all B prompts.
  const int* plist;
  const int* pcount;
};

template <int BN>
struct Cfg {
  static constexpr int MAX_STAGES = 8;
  static constexpr int A_BYTES = BM * BK * 2;
  static constexpr int B_BYTES = BN * BK * 2;
  static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
  static constexpr int ACC_STRIDE = BN == 192 ? 256 : BN;  // TMEM column distance between the two accumulator stages
  static constexpr int TMEM_COLS = 2 * ACC_STRIDE;         // 128 / 256 / 512: powers of two
};
constexpr int SMEM_MAX = 227 * 1024;
constexpr int BAR_BYTES = 1024;           // barriers + tmem pointer, at the (1024-aligned) start of dynamic smem
constexpr int STG_BYTES = 32 * 128;       // one staging tile: 32 rows x 128 B
constexpr int NEPI_WARPS = 8;
constexpr int VEC_FLOATS = 3 * 256;        // per epilogue set: bias | gamma (or hyper) | beta of the current tile's columns
constexpr int VEC_BYTES = 2 * VEC_FLOATS * 4;

template <int ACT>
__device__ __forceinline__ float apply_act(float x) {
  if (ACT == 1) return sb::gelu_erf(x);
  if (ACT == 2) return fmaxf(x, 0.0f);
  if (ACT == 3) return __fdividef(1.0f, 1.0f + __expf(-x));
  return x;
}
// named barrier among the 4 warps of one epilogue set (ids 1 and 2; 0 is __syncthreads)
__device__ __forceinline__ void set_barrier(int set) {
  asm volatile("bar.sync %0, 128;" ::"r"(set + 1) : "memory");
}
// Cooperative (128 threads of a set) staging of n floats src[0..n) -> dst (zero beyond `valid` / null src); n % 4 == 0.
__device__ __forceinline__ void stage_vec(float* dst, const float* src, int n, int valid, int tid128) {
  for (int c = tid128 * 4; c < n; c += 512) {
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (src != nullptr && c < valid) v = __ldg(reinterpret_cast<const float4*>(src + c));
    *reinterpret_cast<float4*>(dst + c) = v;
  }
}

// ---- per-warp staging tiles (32 rows x RB bytes, RB = 128 or 64), XOR-swizzled in 16-byte chunks so that both the
// "one thread = one row" accesses of the TMEM epilogue and the "8 (4) lanes = one row" coalesced global accesses are
// bank-conflict free. All global traffic of the epilogue goes through them: per-thread-row LDG/STG.128 would cost
// one L1 wavefront per 16 bytes, the cooperative form moves 64-128 bytes per wavefront. -----------------------------
template <int RB>
__device__ __forceinline__ uint32_t swz(int row, int chunk) {
  return RB == 128 ? static_cast<uint32_t>(row * 128 + ((chunk ^ (row & 7)) << 4))
                   : static_cast<uint32_t>(row * 64 + ((chunk ^ ((row >> 1) & 3)) << 4));
}
__device__ __forceinline__ void cp_async16(uint32_t smem_addr, const void* gmem) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_addr), "l"(gmem) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_1() { asm volatile("cp.async.wait_group 1;" ::: "memory"); }
__device__ __forceinline__ uint4 lds128(uint32_t addr) {
  uint4 v;
  asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr));
  return v;
}
__device__ __forceinline__ void sts128(uint32_t addr, uint4 v) {
  asm volatile("st.shared.v4.u32 [%0], {%1,%2,%3,%4};" ::"r"(addr), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}
// staged per-column vectors: float index -> float4 / float2 (warp-uniform address: one broadcast wavefront)
__device__ __forceinline__ float4 ldsf4(uint32_t base, int fidx) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(base + fidx * 4));
  return v;
}
__device__ __forceinline__ float2 ldsf2(uint32_t base, int fidx) {
  float2 v;
  asm volatile("ld.shared.v2.f32 {%0,%1}, [%2];" : "=f"(v.x), "=f"(v.y) : "r"(base + fidx * 4));
  return v;
}

// Asynchronous cooperative gather of 32 rows x `valid` bytes (valid <= RB, multiple of 16) into a staging tile.
// Lane r owns row r: its source is gbase + off16 * 16 bytes (off16 < 0 = row not loaded).
template <int RB>
__device__ __forceinline__ void gather_async(uint32_t stg, const uint8_t* gbase, int off16, int valid, int lane) {
  constexpr int PPR = RB / 16;
#pragma unroll
  for (int t = 0; t < PPR; ++t) {
    const int id = t * 32 + lane;
    const int row = id / PPR, ch = id % PPR;
    const int o = __shfl_sync(0xffffffffu, off16, row);
    if (o >= 0 && ch * 16 < valid) cp_async16(stg + swz<RB>(row, ch), gbase + (static_cast<long long>(o) + ch) * 16);
  }
  cp_async_commit();
}
// Cooperative coalesced store of a staging tile: row r goes to gbase + off16 * 16 bytes (off16 < 0 = skip).
template <int RB>
__device__ __forceinline__ void scatter_store(uint32_t stg, uint8_t* gbase, int off16, int valid, int lane) {
  constexpr int PPR = RB / 16;
#pragma unroll
  for (int t = 0; t < PPR; ++t) {
    const int id = t * 32 + lane;
    const int row = id / PPR, ch = id % PPR;
    const int o = __shfl_sync(0xffffffffu, off16, row);
    if (o >= 0 && ch * 16 < valid) {
      const uint4 v = lds128(stg + swz<RB>(row, ch));
      *reinterpret_cast<uint4*>(gbase + (static_cast<long long>(o) + ch) * 16) = v;
    }
  }
}

// The same for the 32 CONSECUTIVE rows of an epilogue warp (row r at base16 + r * ld16, in 16-byte units; rows >= nrows are
// skipped): addresses are arithmetic instead of a shuffle per 16 bytes, and the store reads all its staging chunks before
// the first global store is issued — SHFL -> LDS -> STG was a serial short-scoreboard chain per 16 bytes, the largest
// stall group of the STD epilogue in the source-level profile (profiles/r02q: ~20 % of its samples).
template <int RB>
__device__ __forceinline__ void gather_async_lin(uint32_t stg, const uint8_t* gbase, int base16, int ld16, int nrows,
                                                 int valid, int lane) {
  constexpr int PPR = RB / 16;
#pragma unroll
  for (int t = 0; t < PPR; ++t) {
    const int id = t * 32 + lane;
    const int row = id / PPR, ch = id % PPR;
    if (row < nrows && ch * 16 < valid)
      cp_async16(stg + swz<RB>(row, ch), gbase + static_cast<long long>(base16 + row * ld16 + ch) * 16);
  }
  cp_async_commit();
}
template <int RB>
__device__ __forceinline__ void scatter_store_lin(uint32_t stg, uint8_t* gbase, int base16, int ld16, int nrows,
                                                  int valid, int lane) {
  constexpr int PPR = RB / 16;
#pragma unroll
  for (int t0 = 0; t0 < PPR; t0 += 4) {
    uint4 v[4];
#pragma unroll
    for (int t = 0; t < 4; ++t) {
      const int id = (t0 + t) * 32 + lane;
      v[t] = lds128(stg + swz<RB>(id / PPR, id % PPR));
    }
#pragma unroll
    for (int t = 0; t < 4; ++t) {
      const int id = (t0 + t) * 32 + lane;
      const int row = id / PPR, ch = id % PPR;
      if (row < nrows && ch * 16 < valid)
        *reinterpret_cast<uint4*>(gbase + static_cast<long long>(base16 + row * ld16 + ch) * 16) = v[t];
    }
  }
}

struct EpiSmem {
  uint32_t out_stg;     // shared-space address of this warp's output staging tile
  uint32_t res0, res1;  // residual / skip staging tiles (res1 == res0 when single-buffered). Two scalars selected with
                        // res_buf(): an array indexed by the group parity was placed in LOCAL memory by the compiler, and the
                        // LDL of its address was the largest stall of the residual epilogues (profiles/r02m: 165 of 987
                        // epilogue samples on one long-scoreboard wait)
  int nres;             // number of distinct residual staging tiles (0, 1 or 2)
  int alias;            // STD: the output of a group is staged IN the residual tile it was computed from (same element
                        // size; a thread reads and writes only its own row's chunks) -> no separate output tile
  uint32_t vec;         // shared-space address of this set's staged vectors: [0,256) bias, [256,512) gamma / hyper,
                        // [512,768) beta. Read with ld.shared (a generic-pointer dereference compiles to LD.E: the
                        // generic-address path, reported by ncu as long-scoreboard stalls in every epilogue)
};

__device__ __forceinline__ uint32_t res_buf(const EpiSmem& es, int i) { return (i & 1) ? es.res1 : es.res0; }

__device__ __forceinline__ void unpack_bf16x8(const uint4 r, float* f) {
  f[0] = sb::bf16_lo(r.x);
  f[1] = sb::bf16_hi(r.x);
  f[2] = sb::bf16_lo(r.y);
  f[3] = sb::bf16_hi(r.y);
  f[4] = sb::bf16_lo(r.z);
  f[5] = sb::bf16_hi(r.z);
  f[6] = sb::bf16_lo(r.w);
  f[7] = sb::bf16_hi(r.w);
}

// Residual of 16 columns (half `h` of the current 32-column group) of this thread's row: staging -> f[16] += residual
template <bool RES_F32>
__device__ __forceinline__ void add_res_from_stg(uint32_t stg, int lane, int h, float* f) {
  if (RES_F32) {
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const uint4 r = lds128(stg + swz<128>(lane, h * 4 + j));
      f[4 * j + 0] += __uint_as_float(r.x);
      f[4 * j + 1] += __uint_as_float(r.y);
      f[4 * j + 2] += __uint_as_float(r.z);
      f[4 * j + 3] += __uint_as_float(r.w);
    }
  } else {
#pragma unroll
    for (int j = 0; j < 2; ++j) {
      float t[8];
      unpack_bf16x8(lds128(stg + swz<64>(lane, h * 2 + j)), t);
#pragma unroll
      for (int e = 0; e < 8; ++e) f[8 * j + e] += t[e];
    }
  }
}

// this thread's 16 results (half `h` of the group) -> output staging (fp32: 128-byte rows, bf16: 64-byte rows)
__device__ __forceinline__ void stage_out(uint32_t stg, int lane, int h, int out_f32, const float* f) {
  if (out_f32) {
#pragma unroll
    for (int j = 0; j < 4; ++j)
      sts128(stg + swz<128>(lane, h * 4 + j), make_uint4(__float_as_uint(f[4 * j]), __float_as_uint(f[4 * j + 1]),
                                                          __float_as_uint(f[4 * j + 2]), __float_as_uint(f[4 * j + 3])));
  } else {
#pragma unroll
    for (int j = 0; j < 2; ++j)
      sts128(stg + swz<64>(lane, h * 2 + j),
             make_uint4(sb::pack_bf16x2(f[8 * j + 0], f[8 * j + 1]), sb::pack_bf16x2(f[8 * j + 2], f[8 * j + 3]),
                        sb::pack_bf16x2(f[8 * j + 4], f[8 * j + 5]), sb::pack_bf16x2(f[8 * j + 6], f[8 * j + 7])));
  }
}

__device__ __forceinline__ void issue_res_gather(const GemmParams& p, uint32_t stg, int res_off16_row, int n0,
                                                 int ncols, int lane) {
  // res_off16_row: 16-byte offset of this lane's residual row start (or < 0); group starts n0 columns in
  if (p.res_f32)
    gather_async<128>(stg, reinterpret_cast<const uint8_t*>(p.res), res_off16_row < 0 ? -1 : res_off16_row + n0 / 4,
                      ncols * 4, lane);
  else
    gather_async<64>(stg, reinterpret_cast<const uint8_t*>(p.res), res_off16_row < 0 ? -1 : res_off16_row + n0 / 8,
                     ncols * 2, lane);
}

// ---- STD / LN epilogue of one 128 x BN tile (this warp: 32 rows). Arithmetic runs on 16-column chunks (TMEM loads
// one chunk ahead), global IO on 32-column groups through the staging tiles.
// LN: two passes over the row (statistics, then normalise); the tile spans the whole row (N <= BN).
template <int BN, bool LN, int ACT>
__device__ __forceinline__ void epilogue_rows(const GemmParams& p, const EpiSmem& es, uint32_t tmem_acc, int m_idx,
                                              int n_idx, int q, int lane, int g_begin = 0, int g_end = BN / 32) {
  const int NG = g_end;  // this warp drains the 32-column groups [g_begin, g_end) of the tile
  const int row = m_idx + q * 32 + lane;
  const bool row_ok = row < p.M;
  const long long rrow = p.res_mod > 0 ? (row % p.res_mod) : row;
  const uint32_t taddr = tmem_acc + (static_cast<uint32_t>(q * 32) << 16);
  const bool has_res = p.res != nullptr;
  // 16-byte offsets of this lane's rows (all pitches are multiples of 16 bytes on this path)
  const int res_off16 = (has_res && row_ok) ? static_cast<int>(rrow * p.ldr / (p.res_f32 ? 4 : 8)) : -1;
  const int out_off16 = row_ok ? static_cast<int>(static_cast<long long>(row) * p.ldo / (p.out_f32 ? 4 : 8)) : -1;
  float sum = 0.f, sumsq = 0.f, shift = 0.f, mean = 0.f, rstd = 0.f;
#pragma unroll 1
  for (int pass = 0; pass < (LN ? 2 : 1); ++pass) {
    if (n_idx + g_begin * 32 >= p.N) break;
    // LN: pass 0 computes acc + bias + residual, accumulates the row statistics and parks the sums back in TMEM
    // (tcgen05.st); pass 1 only re-reads TMEM — the residual stream is gathered once.
    const bool use_res = has_res && !(LN && pass == 1);
    if (use_res)
      issue_res_gather(p, res_buf(es, g_begin & 1), res_off16, n_idx + g_begin * 32, min(32, p.N - n_idx - g_begin * 32), lane);
    uint32_t v[2][CH];
    sb::tmem_ld_32x16(taddr + static_cast<uint32_t>(g_begin * 32), v[0]);
#pragma unroll 1
    for (int g = g_begin; g < NG; ++g) {
      const int n0 = n_idx + g * 32;
      if (n0 >= p.N) break;  // warp-uniform
      const int ncols = min(32, p.N - n0);  // 16 or 32
      if (use_res) {
        const bool more = (n0 + 32 < p.N) && (g + 1 < NG);
        if (es.nres == 2 && more) {  // double-buffered: the next group's gather is in flight while this one is consumed
          issue_res_gather(p, res_buf(es, (g + 1) & 1), res_off16, n0 + 32, min(32, p.N - n0 - 32), lane);
          cp_async_wait_1();
        } else {
          cp_async_wait_all();
        }
        __syncwarp();
      }
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        if (h * CH >= ncols) break;  // warp-uniform
        const int c0 = n0 + h * CH;
        sb::tmem_ld_wait();
        if (c0 + CH < p.N && (g * 2 + h + 1) < 2 * NG)  // next chunk of this tile row
          sb::tmem_ld_32x16(taddr + static_cast<uint32_t>((g * 2 + h + 1) * CH), v[(h + 1) & 1]);
        float f[CH];
        const float2 al2 = sb::splat2(p.alpha);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const float4 b = ldsf4(es.vec, (c0 - n_idx) + 4 * j);  // staged bias (LDS broadcast)
          const float2 v01 = make_float2(__uint_as_float(v[h][4 * j + 0]), __uint_as_float(v[h][4 * j + 1]));
          const float2 v23 = make_float2(__uint_as_float(v[h][4 * j + 2]), __uint_as_float(v[h][4 * j + 3]));
          float2 r01, r23;
          if (!LN) {  // act(alpha * acc + bias); packed fp32 pairs (GELU: 6 packed + 2 MUFU per pair)
            r01 = sb::fma2(v01, al2, make_float2(b.x, b.y));
            r23 = sb::fma2(v23, al2, make_float2(b.z, b.w));
            if (ACT == 1) {
              r01 = sb::gelu_erf2(r01);
              r23 = sb::gelu_erf2(r23);
            } else if (ACT != 0) {
              r01 = make_float2(apply_act<ACT>(r01.x), apply_act<ACT>(r01.y));
              r23 = make_float2(apply_act<ACT>(r23.x), apply_act<ACT>(r23.y));
            }
          } else if (pass == 0) {
            r01 = sb::add2(v01, make_float2(b.x, b.y));
            r23 = sb::add2(v23, make_float2(b.z, b.w));
          } else {
            r01 = v01;
            r23 = v23;
          }
          f[4 * j + 0] = r01.x;
          f[4 * j + 1] = r01.y;
          f[4 * j + 2] = r23.x;
          f[4 * j + 3] = r23.y;
        }
        const uint32_t ostg = (!LN && es.alias) ? res_buf(es, g & 1) : es.out_stg;
        if (use_res) {
          if (p.res_f32)
            add_res_from_stg<true>(res_buf(es, g & 1), lane, h, f);
          else
            add_res_from_stg<false>(res_buf(es, g & 1), lane, h, f);
        }
        if (LN) {
          if (pass == 0) {
            // sums of x - x0 (x0 = the row's first value): sumsq / N - mean^2 in fp32 on the raw values loses the
            // variance of rows whose |mean| is large against their std (rstd off by 2.5e-3 at |mean| / std = 64)
            if (g == g_begin && h == 0) shift = f[0];
            const float2 nsh = sb::splat2(-shift);
            float2 s2 = make_float2(0.f, 0.f), q2 = make_float2(0.f, 0.f);
#pragma unroll
            for (int j = 0; j < CH / 2; ++j) {
              const float2 ff = sb::add2(make_float2(f[2 * j], f[2 * j + 1]), nsh);
              s2 = sb::add2(s2, ff);
              q2 = sb::fma2(ff, ff, q2);
            }
            sum += s2.x + s2.y;
            sumsq += q2.x + q2.y;
            sb::tmem_st_32x16(taddr + static_cast<uint32_t>((g * 2 + h) * CH), reinterpret_cast<const uint32_t*>(f));
            continue;
          }
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const float4 ga = ldsf4(es.vec, 256 + c0 + 4 * j);
            const float4 be = ldsf4(es.vec, 512 + c0 + 4 * j);
            const float2 nm2 = sb::splat2(-mean), rs2 = sb::splat2(rstd);
            const float2 o01 = sb::fma2(sb::add2(make_float2(f[4 * j + 0], f[4 * j + 1]), nm2),
                                        sb::mul2(rs2, make_float2(ga.x, ga.y)), make_float2(be.x, be.y));
            const float2 o23 = sb::fma2(sb::add2(make_float2(f[4 * j + 2], f[4 * j + 3]), nm2),
                                        sb::mul2(rs2, make_float2(ga.z, ga.w)), make_float2(be.z, be.w));
            f[4 * j + 0] = o01.x;
            f[4 * j + 1] = o01.y;
            f[4 * j + 2] = o23.x;
            f[4 * j + 3] = o23.y;
          }
        }
        stage_out(ostg, lane, h, p.out_f32, f);
      }
      __syncwarp();  // residual tile fully consumed, output tile fully written
      const bool alias = !LN && es.alias;
      const uint32_t ostg = alias ? res_buf(es, g & 1) : es.out_stg;
      const bool late_gather = use_res && es.nres != 2 && (n0 + 32 < p.N) && (g + 1 < NG);
      if (late_gather && !alias)
        issue_res_gather(p, res_buf(es, (g + 1) & 1), res_off16, n0 + 32, min(32, p.N - n0 - 32), lane);
      if (!(LN && pass == 0)) {
        if (p.out_f32)
          scatter_store<128>(ostg, reinterpret_cast<uint8_t*>(p.out), out_off16 < 0 ? -1 : out_off16 + n0 / 4,
                             ncols * 4, lane);
        else
          scatter_store<64>(ostg, reinterpret_cast<uint8_t*>(p.out), out_off16 < 0 ? -1 : out_off16 + n0 / 8,
                            ncols * 2, lane);
        __syncwarp();
      }
      if (late_gather && alias)  // single aliased tile: refill only after the staged output has been read back
        issue_res_gather(p, res_buf(es, (g + 1) & 1), res_off16, n0 + 32, min(32, p.N - n0 - 32), lane);
    }
    if (LN && pass == 0) {
      sb::tmem_st_wait();
      const float dmean = sum / static_cast<float>(p.N);
      mean = shift + dmean;
      const float var = fmaxf(sumsq / static_cast<float>(p.N) - dmean * dmean, 0.f);
      rstd = rsqrtf(var + p.eps);
    }
  }
}

// ---- STD epilogue of the 32-column groups [g_begin, g_end) of one 128 x BN tile (this warp: 32 rows), software-
// pipelined ACROSS tiles: while the last group of a tile is processed, the residual gather of this warp's first group
// of its NEXT tile is already in flight (the first gather of a tile used to be an exposed HBM round trip per tile:
// ~1 900 clocks of the ~6 700 a warp spent on its half of a proj tile). `pb` = staging buffer of the first group
// (alternates with the number of groups processed), `issued` = that gather is already in flight. Bias comes from the
// staged vector at es.vec, indexed by (column - vbase).
template <int BN, int ACT>
__device__ __forceinline__ void epilogue_std(const GemmParams& p, const EpiSmem& es, uint32_t tmem_acc, int m_idx,
                                             int n_idx, int q, int lane, int g_begin, int g_end, int vbase, int& pb,
                                             bool& issued, int next_m_idx, int next_n_idx) {
  const int first_n = n_idx + g_begin * 32;
  if (first_n >= p.N) return;  // (never prefetched: the prefetch applies the same test)
  const int row0 = m_idx + q * 32;  // this warp's rows are row0 .. row0 + 31: linear addresses (res_mod % 32 == 0)
  const int nrows = min(32, max(0, p.M - row0));
  const uint32_t taddr = tmem_acc + (static_cast<uint32_t>(q * 32) << 16);
  const bool has_res = p.res != nullptr;
  const int res_e16 = p.res_f32 ? 4 : 8, out_e16 = p.out_f32 ? 4 : 8;  // elements per 16 bytes
  const int ld16r = has_res ? static_cast<int>(p.ldr / res_e16) : 0, ld16o = static_cast<int>(p.ldo / out_e16);
  // 16-byte offsets fit an int: the launch checks M * pitch < 2^35 bytes on this path
  auto res_base16 = [&](int r0) -> int { return (p.res_mod > 0 ? (r0 % p.res_mod) : r0) * ld16r; };
  auto gather = [&](uint32_t stg, int base16, int rows, int n0) {
    const int ncols = min(32, p.N - n0);
    if (p.res_f32)
      gather_async_lin<128>(stg, reinterpret_cast<const uint8_t*>(p.res), base16 + n0 / 4, ld16r, rows, ncols * 4, lane);
    else
      gather_async_lin<64>(stg, reinterpret_cast<const uint8_t*>(p.res), base16 + n0 / 8, ld16r, rows, ncols * 2, lane);
  };
  const int res16 = has_res ? res_base16(row0) : 0;
  const int out16 = row0 * ld16o;
  const int g_last = min(g_end, (p.N - n_idx + 31) / 32);  // exclusive
  if (has_res && !issued) gather(res_buf(es, pb), res16, nrows, first_n);
  issued = false;
  const int next_first_n = next_n_idx + g_begin * 32;
  const bool next_ok = has_res && next_m_idx >= 0 && next_first_n < p.N;
  const int next_row0 = next_m_idx + q * 32;
  const int next_res16 = next_ok ? res_base16(next_row0) : 0;
  const int next_nrows = next_ok ? min(32, max(0, p.M - next_row0)) : 0;
  const bool alias = es.alias != 0;
  uint32_t v[2][CH];
  sb::tmem_ld_32x16(taddr + static_cast<uint32_t>(g_begin * 32), v[0]);
#pragma unroll 1
  for (int g = g_begin; g < g_last; ++g) {
    const int n0 = n_idx + g * 32;
    const int ncols = min(32, p.N - n0);  // 16 or 32
    const int bi = g - g_begin + pb;      // parity = this group's residual buffer
    const bool more = g + 1 < g_last;
    if (has_res) {
      if (es.nres == 2 && more) {  // the next group's gather is in flight while this one is consumed
        gather(res_buf(es, bi + 1), res16, nrows, n0 + 32);
        cp_async_wait_1();
      } else if (es.nres == 2 && next_ok) {  // ... or the first group of the next tile
        gather(res_buf(es, bi + 1), next_res16, next_nrows, next_first_n);
        issued = true;
        cp_async_wait_1();
      } else {
        cp_async_wait_all();
      }
      __syncwarp();
    }
    const uint32_t rstg = res_buf(es, bi);
    const uint32_t ostg = alias ? rstg : es.out_stg;
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      if (h * CH >= ncols) break;  // warp-uniform
      const int c0 = n0 + h * CH;
      sb::tmem_ld_wait();
      if (c0 + CH < p.N && (g * 2 + h + 1) < 2 * g_last)  // next chunk of this tile row
        sb::tmem_ld_32x16(taddr + static_cast<uint32_t>((g * 2 + h + 1) * CH), v[(h + 1) & 1]);
      float f[CH];
      const float2 al2 = sb::splat2(p.alpha);
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float4 b = ldsf4(es.vec, (c0 - vbase) + 4 * j);  // staged bias (LDS broadcast)
        const float2 v01 = make_float2(__uint_as_float(v[h][4 * j + 0]), __uint_as_float(v[h][4 * j + 1]));
        const float2 v23 = make_float2(__uint_as_float(v[h][4 * j + 2]), __uint_as_float(v[h][4 * j + 3]));
        // act(alpha * acc + bias); packed fp32 pairs (GELU: 6 packed + 2 MUFU per pair)
        float2 r01 = sb::fma2(v01, al2, make_float2(b.x, b.y));
        float2 r23 = sb::fma2(v23, al2, make_float2(b.z, b.w));
        if (ACT == 1) {
          r01 = sb::gelu_erf2(r01);
          r23 = sb::gelu_erf2(r23);
        } else if (ACT != 0) {
          r01 = make_float2(apply_act<ACT>(r01.x), apply_act<ACT>(r01.y));
          r23 = make_float2(apply_act<ACT>(r23.x), apply_act<ACT>(r23.y));
        }
        f[4 * j + 0] = r01.x;
        f[4 * j + 1] = r01.y;
        f[4 * j + 2] = r23.x;
        f[4 * j + 3] = r23.y;
      }
      if (has_res) {
        if (p.res_f32)
          add_res_from_stg<true>(rstg, lane, h, f);
        else
          add_res_from_stg<false>(rstg, lane, h, f);
      }
      stage_out(ostg, lane, h, p.out_f32, f);
    }
    __syncwarp();  // residual tile fully consumed, output tile fully written
    if (p.out_f32)
      scatter_store_lin<128>(ostg, reinterpret_cast<uint8_t*>(p.out), out16 + n0 / 4, ld16o, nrows, ncols * 4, lane);
    else
      scatter_store_lin<64>(ostg, reinterpret_cast<uint8_t*>(p.out), out16 + n0 / 8, ld16o, nrows, ncols * 2, lane);
    __syncwarp();
    if (has_res && es.nres != 2) {  // single tile: refill only after the staged output has been read back
      if (more) {
        gather(res_buf(es, bi + 1), res16, nrows, n0 + 32);
      } else if (next_ok) {
        gather(res_buf(es, bi + 1), next_res16, next_nrows, next_first_n);
        issued = true;
      }
    }
  }
  pb = (pb + (g_last - g_begin)) & 1;
}

// ---- scalar fallback for shapes the staged path cannot take (N % 16 != 0 or pitches not multiples of 16 bytes) -----
template <int BN, int ACT>
__device__ __forceinline__ void epilogue_scalar(const GemmParams& p, uint32_t tmem_acc, int m_idx, int n_idx, int q,
                                                int lane, int c_begin = 0, int c_end = BN / CH) {
  const int row = m_idx + q * 32 + lane;
  const bool row_ok = row < p.M;
  const long long rrow = p.res_mod > 0 ? (row % p.res_mod) : row;
  const uint32_t taddr = tmem_acc + (static_cast<uint32_t>(q * 32) << 16);
#pragma unroll 1
  for (int c = c_begin; c < c_end; ++c) {
    const int n0 = n_idx + c * CH;
    if (n0 >= p.N) break;  // warp-uniform
    uint32_t v[CH];
    sb::tmem_ld_32x16(taddr + static_cast<uint32_t>(c * CH), v);
    sb::tmem_ld_wait();
    const int ncols = min(CH, p.N - n0);
#pragma unroll
    for (int j = 0; j < CH; ++j) {
      if (j < ncols && row_ok) {
        float x = __uint_as_float(v[j]) * p.alpha + (p.bias ? __ldg(p.bias + n0 + j) : 0.f);
        x = apply_act<ACT>(x);
        if (p.res) {
          x += p.res_f32 ? reinterpret_cast<const float*>(p.res)[rrow * p.ldr + n0 + j]
                         : __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(p.res)[rrow * p.ldr + n0 + j]);
        }
        if (p.out_f32)
          reinterpret_cast<float*>(p.out)[static_cast<long long>(row) * p.ldo + n0 + j] = x;
        else
          reinterpret_cast<__nv_bfloat16*>(p.out)[static_cast<long long>(row) * p.ldo + n0 + j] = __float2bfloat16(x);
      }
    }
  }
}

// ---- UP1 epilogue: N = 4 groups x 64 channels; row m = (b, y, x) of the gh x gw token grid ---------------
__device__ __forceinline__ void epilogue_up1(const GemmParams& p, const EpiSmem& es, uint32_t tmem_acc, int m_idx,
                                             int q, int lane, int d_begin, int d_end) {
  const int row = m_idx + q * 32 + lane;
  const bool row_ok = row < p.M;
  const uint32_t taddr = tmem_acc + (static_cast<uint32_t>(q * 32) << 16);
  const int x = row % p.gw, y = (row / p.gw) % p.gh;
  const long long b = row / (p.gw * p.gh);
  const uint8_t* skip = reinterpret_cast<const uint8_t*>(p.skip);
#pragma unroll 1
  for (int d = d_begin; d < d_end; ++d) {
    const int oy = 2 * y + (d >> 1), ox = 2 * x + (d & 1);
    const long long pix = static_cast<long long>(oy) * (2 * p.gw) + ox;
    // skip row: 64 fp32 = 256 bytes = 16 x 16 B ; output row: 64 bf16 = 128 bytes = 8 x 16 B
    const int skip_off16 = row_ok ? static_cast<int>((b * p.skip_bstride + pix * 64) / 4) : -1;
    const int out_off16 = row_ok ? static_cast<int>(((b * (2 * p.gh) + oy) * (2 * p.gw) + ox) * 8) : -1;
    float f[64];
    float2 sum2 = make_float2(0.f, 0.f);
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      gather_async<128>(res_buf(es, 0), skip, skip_off16 < 0 ? -1 : skip_off16 + h * 8, 128, lane);
      uint32_t v[32];
      sb::tmem_ld_32x16(taddr + static_cast<uint32_t>(d * 64 + h * 32), v);
      sb::tmem_ld_32x16(taddr + static_cast<uint32_t>(d * 64 + h * 32 + 16), v + 16);
      cp_async_wait_all();
      __syncwarp();
      sb::tmem_ld_wait();
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const uint4 sk = lds128(res_buf(es, 0) + swz<128>(lane, j));
        const float4 bb = ldsf4(es.vec, d * 64 + h * 32 + 4 * j);
        const int e = h * 32 + 4 * j;
        const float2 f01 = sb::add2(
            sb::add2(make_float2(__uint_as_float(v[4 * j + 0]), __uint_as_float(v[4 * j + 1])), make_float2(bb.x, bb.y)),
            make_float2(__uint_as_float(sk.x), __uint_as_float(sk.y)));
        const float2 f23 = sb::add2(
            sb::add2(make_float2(__uint_as_float(v[4 * j + 2]), __uint_as_float(v[4 * j + 3])), make_float2(bb.z, bb.w)),
            make_float2(__uint_as_float(sk.z), __uint_as_float(sk.w)));
        f[e + 0] = f01.x;
        f[e + 1] = f01.y;
        f[e + 2] = f23.x;
        f[e + 3] = f23.y;
        sum2 = sb::add2(sum2, sb::add2(f01, f23));
      }
      __syncwarp();
    }
    const float mean = (sum2.x + sum2.y) * (1.f / 64.f);
    const float2 nmean = sb::splat2(-mean);
    float2 vs2 = make_float2(0.f, 0.f);
#pragma unroll
    for (int j = 0; j < 32; ++j) {
      const float2 dd = sb::add2(make_float2(f[2 * j], f[2 * j + 1]), nmean);
      vs2 = sb::fma2(dd, dd, vs2);
    }
    const float rstd = rsqrtf((vs2.x + vs2.y) * (1.f / 64.f) + p.eps);
    const float2 rs2 = sb::splat2(rstd);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      float2 g[4];
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const float2 ga = ldsf2(es.vec, 256 + 8 * j + 2 * e);
        const float2 be = ldsf2(es.vec, 512 + 8 * j + 2 * e);
        const float2 dd = sb::add2(make_float2(f[8 * j + 2 * e], f[8 * j + 2 * e + 1]), nmean);
        g[e] = sb::gelu_erf2(sb::fma2(dd, sb::mul2(rs2, ga), be));
      }
      sts128(es.out_stg + swz<128>(lane, j), make_uint4(sb::pack_bf16x2(g[0].x, g[0].y), sb::pack_bf16x2(g[1].x, g[1].y),
                                                         sb::pack_bf16x2(g[2].x, g[2].y), sb::pack_bf16x2(g[3].x, g[3].y)));
    }
    __syncwarp();
    scatter_store<128>(es.out_stg, reinterpret_cast<uint8_t*>(p.out), out_off16, 128, lane);
    __syncwarp();
  }
}

// ---- UP2 epilogue: N = 4 groups x 32 channels -> 4 mask logits per output pixel --------------------------
__device__ __forceinline__ void epilogue_up2(const GemmParams& p, const EpiSmem& es, uint32_t tmem_acc, int m_idx,
                                             int q, int lane, int d_begin, int d_end, int hy_off) {
  const int row = m_idx + q * 32 + lane;
  const bool row_ok = row < p.M;
  const uint32_t taddr = tmem_acc + (static_cast<uint32_t>(q * 32) << 16);
  const int x = row % p.gw, y = (row / p.gw) % p.gh;
  const long long b = row / (p.gw * p.gh);
  const int H2 = 2 * p.gh, W2 = 2 * p.gw;
  float* masks = reinterpret_cast<float*>(p.out);
  const uint32_t hy = es.vec + hy_off * 4;  // this tile's prompt: staged hyper-network vectors
  const uint8_t* skip = reinterpret_cast<const uint8_t*>(p.skip);
  // skip row of (d): 32 fp32 = 128 bytes
  auto skip_off = [&](int d) -> int {
    const int oy = 2 * y + (d >> 1), ox = 2 * x + (d & 1);
    return row_ok ? static_cast<int>((b * p.skip_bstride + (static_cast<long long>(oy) * W2 + ox) * 32) / 4) : -1;
  };
  gather_async<128>(res_buf(es, d_begin & 1), skip, skip_off(d_begin), 128, lane);
  float held[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll 1
  for (int d = d_begin; d < d_end; ++d) {
    const int oy = 2 * y + (d >> 1), ox = 2 * x + (d & 1);
    uint32_t v[32];
    sb::tmem_ld_32x16(taddr + static_cast<uint32_t>(d * 32), v);
    sb::tmem_ld_32x16(taddr + static_cast<uint32_t>(d * 32 + CH), v + CH);
    cp_async_wait_all();
    __syncwarp();
    if (d + 1 < d_end) gather_async<128>(res_buf(es, (d + 1) & 1), skip, skip_off(d + 1), 128, lane);
    sb::tmem_ld_wait();
    // packed fp32 pairs throughout: the epilogue is issue-bound (128 GELUs + 512 MACs per row on 8 warps per SM)
    float2 acc2[4] = {make_float2(0.f, 0.f), make_float2(0.f, 0.f), make_float2(0.f, 0.f), make_float2(0.f, 0.f)};
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const float4 bb = ldsf4(es.vec, d * 32 + 4 * j);
      const uint4 sk = lds128(res_buf(es, d & 1) + swz<128>(lane, j));  // skip tile of d (the tile of d + 1 is the other one)
      const float2 g01 = sb::gelu_erf2(sb::add2(
          sb::add2(make_float2(__uint_as_float(v[4 * j + 0]), __uint_as_float(v[4 * j + 1])), make_float2(bb.x, bb.y)),
          make_float2(__uint_as_float(sk.x), __uint_as_float(sk.y))));
      const float2 g23 = sb::gelu_erf2(sb::add2(
          sb::add2(make_float2(__uint_as_float(v[4 * j + 2]), __uint_as_float(v[4 * j + 3])), make_float2(bb.z, bb.w)),
          make_float2(__uint_as_float(sk.z), __uint_as_float(sk.w))));
#pragma unroll
      for (int m = 0; m < 4; ++m) {
        const float4 h = ldsf4(hy, (m * 8 + j) * 4);  // warp-uniform shared-memory address: broadcast
        acc2[m] = sb::fma2(g01, make_float2(h.x, h.y), acc2[m]);
        acc2[m] = sb::fma2(g23, make_float2(h.z, h.w), acc2[m]);
      }
    }
    const float acc[4] = {acc2[0].x + acc2[0].y, acc2[1].x + acc2[1].y, acc2[2].x + acc2[2].y, acc2[3].x + acc2[3].y};
    // d = 2 dy + dx: the two dx of an output row are adjacent pixels -> one 8-byte store per mask (a warp then writes 256
    // contiguous bytes per instruction instead of two half-used 256-byte spans: the LSU data pipe was 59 % busy)
    if ((d & 1) == 0 && d + 1 < d_end) {
#pragma unroll
      for (int m = 0; m < 4; ++m) held[m] = acc[m];
    } else if ((d & 1) == 1 && d - 1 >= d_begin) {
      if (row_ok) {
#pragma unroll
        for (int m = 0; m < 4; ++m)
          *reinterpret_cast<float2*>(masks + ((b * 4 + m) * H2 + oy) * W2 + ox - 1) = make_float2(held[m], acc[m]);
      }
    } else if (row_ok) {
#pragma unroll
      for (int m = 0; m < 4; ++m) masks[((b * 4 + m) * H2 + oy) * W2 + ox] = acc[m];
    }
  }
}

template <int BN, int EPI, int ACT>
__global__ void __launch_bounds__(NTHREADS, 1)
gemm_bf16_tcgen05_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                         const GemmParams p, const int stages, const int res_bufs, const int staged,
                         const int stg_out_bytes, const int stg_res_bytes, const int split, const int vec_all_bytes) {
  using C = Cfg<BN>;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) &
                                             ~static_cast<uintptr_t>(1023));
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem);
  uint64_t* full_bar = bars;
  uint64_t* empty_bar = bars + C::MAX_STAGES;
  uint64_t* tfull_bar = bars + 2 * C::MAX_STAGES;
  uint64_t* tempty_bar = bars + 2 * C::MAX_STAGES + 2;
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(bars + 2 * C::MAX_STAGES + 4);
  uint8_t* sA = smem + BAR_BYTES;
  uint8_t* sB = sA + stages * C::A_BYTES;
  float* sVec = reinterpret_cast<float*>(sA + stages * C::STAGE_BYTES);
  uint8_t* sEpi = reinterpret_cast<uint8_t*>(sVec) + (vec_all_bytes > 0 ? vec_all_bytes : VEC_BYTES);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  const int m_tiles = (p.M + BM - 1) / BM;
  const int n_tiles = (p.N + BN - 1) / BN;
  // up-scaling on a prompt list: tile t -> (listed prompt t / tpp, row block t % tpp); the tile count is read on the device
  const int tpp = ((EPI == EPI_UP1 || EPI == EPI_UP2) && p.plist != nullptr) ? (p.gh * p.gw) / BM : 0;
  const int num_tiles = tpp > 0 ? __ldg(p.pcount) * tpp : m_tiles * n_tiles;
  auto tile_m = [&](int tile) -> int {
    if (tpp > 0) return __ldg(p.plist + tile / tpp) * (p.gh * p.gw) + (tile % tpp) * BM;
    return (tile / n_tiles) * BM;
  };
  const int num_kb = (p.K + BK - 1) / BK;
  const int last_ksteps = ((p.K - (num_kb - 1) * BK) + 15) / 16;

  if (warp == 0 && lane == 0) {
    sb::tma_prefetch_desc(&tmA);
    sb::tma_prefetch_desc(&tmB);
  }
  if (warp == 1 && lane == 0) {
    for (int i = 0; i < stages; ++i) {
      sb::mbar_init(&full_bar[i], 1);
      sb::mbar_init(&empty_bar[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      sb::mbar_init(&tfull_bar[i], 1);
      sb::mbar_init(&tempty_bar[i], split ? 8 : 4);  // one arrive per warp that drains this stage
    }
    sb::fence_barrier_init();
  }
  if (warp == 2) {
    sb::tmem_alloc(tmem_ptr, C::TMEM_COLS);
    sb::tmem_relinquish();
  }
  sb::tc_fence_before();
  __syncthreads();
  sb::tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;

  if (warp == 0) {
    // ===================== TMA producer =====================
    // Lane 0 feeds the operand ring.
    int stage = 0;
    uint32_t phase = 0;
    long long prof_acc = 0;
    for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
      const int m_idx = tile_m(tile);
      const int n_idx = (tile % n_tiles) * BN;
      if (lane == 0) {
        for (int kb = 0; kb < num_kb; ++kb) {
          if (p.prof) {
            const long long t0 = clock64();
            sb::mbar_wait(&empty_bar[stage], phase ^ 1);
            prof_acc += clock64() - t0;
          } else {
            sb::mbar_wait(&empty_bar[stage], phase ^ 1);
          }
          sb::mbar_arrive_expect_tx(&full_bar[stage], C::STAGE_BYTES);
          sb::tma_load_2d(sA + stage * C::A_BYTES, &tmA, &full_bar[stage], kb * BK, m_idx);
          sb::tma_load_2d(sB + stage * C::B_BYTES, &tmB, &full_bar[stage], kb * BK, n_idx);
          if (++stage == stages) {
            stage = 0;
            phase ^= 1;
          }
        }
      }
      __syncwarp();
    }
    if (p.prof && lane == 0) atomicAdd(p.prof + 0, static_cast<unsigned long long>(prof_acc));
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    // warp-converged; one elected lane issues each tcgen05 instruction (inside a divergent `if (lane == 0)` every UMMA is
    // wrapped in an ELECT / BRA.U.ANY loop: ~13 instructions per UMMA, which bounds the BN = 64 / 128 tiles)
    {
      constexpr uint32_t idesc = sb::umma_idesc_bf16(BM, BN);
      int stage = 0;
      uint32_t phase = 0;
      int acc = 0;
      uint32_t acc_phase = 0;
      long long w_full = 0, w_tempty = 0;
      const long long t_begin = p.prof ? clock64() : 0;
      for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
        if (p.prof) {
          const long long t0 = clock64();
          sb::mbar_wait(&tempty_bar[acc], acc_phase ^ 1);
          w_tempty += clock64() - t0;
        } else {
          sb::mbar_wait(&tempty_bar[acc], acc_phase ^ 1);
        }
        sb::tc_fence_after();
        const uint32_t tmem_d = tmem_base + static_cast<uint32_t>(acc * C::ACC_STRIDE);
        for (int kb = 0; kb < num_kb; ++kb) {
          if (p.prof) {
            const long long t0 = clock64();
            sb::mbar_wait(&full_bar[stage], phase);
            w_full += clock64() - t0;
          } else {
            sb::mbar_wait(&full_bar[stage], phase);
          }
          sb::tc_fence_after();
          const uint64_t da = sb::umma_desc_k_sw128(sb::smem_u32(sA + stage * C::A_BYTES));
          const uint64_t db = sb::umma_desc_k_sw128(sb::smem_u32(sB + stage * C::B_BYTES));
          const int ksteps = (kb == num_kb - 1) ? last_ksteps : (BK / 16);
          for (int k = 0; k < ksteps; ++k) {
            // advance 16 bf16 = 32 B along K inside the 128-B swizzle row: +2 in 16-B units
            if (sb::elect_one())
              sb::umma_bf16(tmem_d, da + static_cast<uint64_t>(2 * k), db + static_cast<uint64_t>(2 * k), idesc,
                            static_cast<uint32_t>((kb | k) != 0));
          }
          if (sb::elect_one()) sb::umma_commit(&empty_bar[stage]);  // frees the smem slot when these MMAs retire
          __syncwarp();
          if (++stage == stages) {
            stage = 0;
            phase ^= 1;
          }
        }
        if (sb::elect_one()) sb::umma_commit(&tfull_bar[acc]);  // accumulator ready for the epilogue
        __syncwarp();
        if (++acc == 2) {
          acc = 0;
          acc_phase ^= 1;
        }
      }
      if (p.prof && lane == 0) {
        atomicAdd(p.prof + 1, static_cast<unsigned long long>(w_full));
        atomicAdd(p.prof + 2, static_cast<unsigned long long>(w_tempty));
        atomicAdd(p.prof + 5, static_cast<unsigned long long>(clock64() - t_begin));
        atomicAdd(p.prof + 6, 1ull);
      }
    }
  } else if (warp >= 4) {
    // ===================== epilogue: set s = (warp - 4) / 4 drains accumulator stage s =====================
    const int q = warp & 3;  // TMEM lane quadrant this warp may access
    const int set = (warp - 4) >> 2;
    EpiSmem es;
    {
      // per warp: one output staging tile (32 rows x 128 B, or x 64 B for bf16 output of the STD / LN epilogues) and
      // res_bufs residual tiles (x 64 B for a bf16 residual): the bf16-output GEMMs (QKV, fc1) gain a pipeline stage
      uint8_t* mine = sEpi + (warp - 4) * (stg_out_bytes + res_bufs * stg_res_bytes);
      es.out_stg = sb::smem_u32(mine);
      es.res0 = sb::smem_u32(mine + (res_bufs > 0 ? stg_out_bytes : 0));
      es.res1 = sb::smem_u32(mine + (res_bufs > 1 ? stg_out_bytes + stg_res_bytes : (res_bufs > 0 ? stg_out_bytes : 0)));
      es.nres = res_bufs;
      es.alias = (stg_out_bytes == 0) ? 1 : 0;
      es.vec = sb::smem_u32(sVec + set * VEC_FLOATS);
    }
    const bool vec_all = EPI == EPI_STD && vec_all_bytes > 0;  // the whole bias vector is staged once, for both sets
    float* myvec = vec_all ? sVec : sVec + set * VEC_FLOATS;
    if (vec_all) es.vec = sb::smem_u32(sVec);
    const int tid128 = (warp & 3) * 32 + lane;
    uint32_t acc_phase = 0;
    int it = 0;
    // Per-column vectors that do not change from tile to tile are staged ONCE: the two 128-thread barriers per tile
    // that guarded the re-staging were 1.8 stalled warps per issued instruction in the up-scaling epilogues
    // (profiles/r02f_upscale_ncu_summary.txt). UP2's per-prompt hyper-network vectors are staged per warp (512 B,
    // one LDG.128 + STS.128 per lane, __syncwarp only). STD with several column tiles: the whole bias vector when the
    // launch reserved room for it (vec_all), else this tile's slice per tile.
    const bool const_vec = EPI == EPI_UP1 || EPI == EPI_UP2 || EPI == EPI_LN || (EPI == EPI_STD && n_tiles == 1) || vec_all;
    if (vec_all) {
      const int tid256 = (warp - 4) * 32 + lane;
      const int valid = (p.N + 3) & ~3;
      for (int c = tid256 * 4; c < vec_all_bytes / 4; c += NEPI_WARPS * 128) {
        float4 b4 = make_float4(0.f, 0.f, 0.f, 0.f);
        if (p.bias != nullptr && c < valid) b4 = __ldg(reinterpret_cast<const float4*>(p.bias + c));
        *reinterpret_cast<float4*>(sVec + c) = b4;
      }
      asm volatile("bar.sync 6, %0;" ::"n"(NEPI_WARPS * 32) : "memory");
    } else if (const_vec) {
      if (EPI == EPI_STD) {
        stage_vec(myvec, p.bias, BN, (p.N + 3) & ~3, tid128);
      } else if (EPI == EPI_LN) {
        stage_vec(myvec, p.bias, BN, p.N, tid128);
        stage_vec(myvec + 256, p.gamma, BN, p.N, tid128);
        stage_vec(myvec + 512, p.beta, BN, p.N, tid128);
      } else if (EPI == EPI_UP1) {
        stage_vec(myvec, p.bias, 256, 256, tid128);
        stage_vec(myvec + 256, p.gamma, 64, 64, tid128);
        stage_vec(myvec + 512, p.beta, 64, 64, tid128);
      } else {
        stage_vec(myvec, p.bias, 128, 128, tid128);
      }
      set_barrier(set);
    }
    // diagnostic clock counters live in shared memory (behind the barriers), not in registers: the kernel sits at the
    // 168-register cap of a 384-thread CTA
    unsigned long long* e_cnt = reinterpret_cast<unsigned long long*>(smem + 512) + (warp - 4) * 3;
    if (p.prof && lane == 0) e_cnt[0] = e_cnt[1] = e_cnt[2] = 0ull;
    const int hy_off = 256 + (warp & 3) * 128;  // UP2: this warp's private copy of the prompt's 4 x 32 hyper vector
    // Which warps drain which accumulator (`split`, chosen per launch).
    // split = 0: set s drains stage s, i.e. every other tile; a stage is held for a whole tile epilogue T_e, a set's
    // cycle is T_e + T_m (MMA of its next tile) and the CTA retires a tile every max(T_m, (T_e + T_m) / 2). LN (whole
    // rows) always runs this way.
    // split = 1: BOTH sets drain EVERY tile, set s taking column half s (d-groups 2s, 2s+1 of the transposed
    // convolutions): a stage is held T_e / 2 and its refill overlaps the drain of the other stage -> a tile every
    // max(T_m, T_e / 2), better whenever the main loop is not negligible. Measured clocks per tile before the change
    // (tools/gemm_probe.py, profiles/r02n_gemm_probe.log): QKV T_e 8 946 vs T_m 4 608, fc1 12 043 vs 4 608, proj 11 172
    // vs 2 304 — the main loop was waiting for accumulators 17-28 % of the time.
    const int tile_step = split ? static_cast<int>(gridDim.x) : 2 * static_cast<int>(gridDim.x);
    int pb = 0;           // epilogue_std: residual staging buffer of the next tile's first group
    bool issued = false;  // ... whose gather is already in flight
    for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x, ++it) {
      if (!split && (it & 1) != set) continue;
      const int st = split ? (it & 1) : set;
      if (split) acc_phase = static_cast<uint32_t>((it >> 1) & 1);
      const int m_idx = tile_m(tile);
      const int n_idx = (tile % n_tiles) * BN;
      if (!const_vec) {
        // stage this tile's per-column vectors once per set: every read in the epilogues is a shared-memory broadcast
        // (per-chunk __ldg of bias / gamma / hyper was the epilogue's critical path: ~4x the main loop at K = 576)
        set_barrier(set);  // the previous tile's readers are done
        stage_vec(myvec, p.bias ? p.bias + n_idx : nullptr, BN, ((p.N - n_idx) + 3) & ~3, tid128);
        set_barrier(set);
      } else if (EPI == EPI_UP2) {
        __syncwarp();  // the previous tile's reads of this warp's hyper copy are done
        *reinterpret_cast<float4*>(myvec + hy_off + lane * 4) =
            __ldg(reinterpret_cast<const float4*>(p.hyper + static_cast<long long>(m_idx / (p.gh * p.gw)) * 128 + lane * 4));
        __syncwarp();
      }
      if (p.prof) {
        const long long t0 = clock64();
        sb::mbar_wait(&tfull_bar[st], acc_phase);
        if (lane == 0) {
          const long long t1 = clock64();
          e_cnt[0] += static_cast<unsigned long long>(t1 - t0);
          e_cnt[1] -= static_cast<unsigned long long>(t1);  // + end time below = work clocks
        }
      } else {
        sb::mbar_wait(&tfull_bar[st], acc_phase);
      }
      sb::tc_fence_after();
      const uint32_t tmem_acc = tmem_base + static_cast<uint32_t>(st * C::ACC_STRIDE);
      // column range of this warp: its half of the tile (split) or all of it
      const int part = split ? set : 0, nparts = split ? 2 : 1;
      if (EPI == EPI_STD) {
        constexpr int NG = BN / 32;
        if (staged) {
          const int nt = tile + tile_step;
          const int next_m = nt < num_tiles ? (nt / n_tiles) * BM : -1;
          const int next_n = nt < num_tiles ? (nt % n_tiles) * BN : 0;
          // BN = 64 has two groups: one per half
          epilogue_std<BN, ACT>(p, es, tmem_acc, m_idx, n_idx, q, lane, part * (NG / nparts), (part + 1) * (NG / nparts),
                                vec_all ? 0 : n_idx, pb, issued, next_m, next_n);
        } else {
          epilogue_scalar<BN, ACT>(p, tmem_acc, m_idx, n_idx, q, lane, part * (BN / CH / nparts),
                                   (part + 1) * (BN / CH / nparts));
        }
      } else if (EPI == EPI_LN) {
        epilogue_rows<BN, true, 0>(p, es, tmem_acc, m_idx, 0, q, lane);
      } else if (EPI == EPI_UP1) {
        epilogue_up1(p, es, tmem_acc, m_idx, q, lane, part * (4 / nparts), (part + 1) * (4 / nparts));
      } else {
        epilogue_up2(p, es, tmem_acc, m_idx, q, lane, part * (4 / nparts), (part + 1) * (4 / nparts), hy_off);
      }
      sb::tc_fence_before();
      __syncwarp();
      if (lane == 0) sb::mbar_arrive(&tempty_bar[st]);
      if (p.prof && lane == 0) {
        e_cnt[1] += static_cast<unsigned long long>(clock64());
        e_cnt[2] += 1ull;
      }
      if (!split) acc_phase ^= 1;
    }
    if (p.prof && lane == 0 && q == 0) {
      atomicAdd(p.prof + 3, e_cnt[0]);
      atomicAdd(p.prof + 4, e_cnt[1]);
      atomicAdd(p.prof + 7, e_cnt[2]);
    }
  }

  sb::tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    sb::tc_fence_after();
    sb::tmem_dealloc(tmem_base, C::TMEM_COLS);
  }
}

template <int BN, int EPI, int ACT = 0>
int launch_gemm(const CUtensorMap& tmA, const CUtensorMap& tmB, const GemmParams& p, int num_sms,
                cudaStream_t stream) {
  using C = Cfg<BN>;
  static SbPerDeviceOnce attr_once;
  if (attr_once.need()) {
    SB_CHECK_CUDA(cudaFuncSetAttribute(gemm_bf16_tcgen05_kernel<BN, EPI, ACT>,
                                       cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_MAX));
    attr_once.mark();
  }
  // staged (coalesced) epilogue needs 16-byte-aligned pitches and N % 16 == 0
  int staged = 1;
  if (EPI == EPI_STD) {
    const long long ob = p.ldo * (p.out_f32 ? 4 : 2), rb = p.ldr * (p.res_f32 ? 4 : 2);
    staged = ((p.N & 15) == 0) && (ob % 16 == 0) && (!p.res || rb % 16 == 0) &&
             ((reinterpret_cast<uintptr_t>(p.out) & 15) == 0) && ((reinterpret_cast<uintptr_t>(p.res) & 15) == 0) &&
             (p.res_mod == 0 || (p.res_mod % 32) == 0) &&
             (static_cast<long long>(p.M) * ob < (1ll << 35)) && (!p.res || static_cast<long long>(p.M) * rb < (1ll << 35));
  }
  const bool needs_res = (EPI == EPI_UP1 || EPI == EPI_UP2) || (p.res != nullptr);
  int res_bufs = needs_res ? 2 : 0;
  const int num_kb = (p.K + BK - 1) / BK;
  const bool narrow = EPI == EPI_STD || EPI == EPI_LN;
  const int stg_res_bytes = (narrow && p.res != nullptr && !p.res_f32) ? STG_BYTES / 2 : STG_BYTES;
  // STD with a residual of the output's element size: outputs are staged in place of the residual tile (no output tile)
  const bool alias = EPI == EPI_STD && staged && p.res != nullptr && (p.out_f32 != 0) == (p.res_f32 != 0);
  const int stg_out_bytes = alias ? 0 : ((narrow && !p.out_f32) ? STG_BYTES / 2 : STG_BYTES);
  auto epi_bytes = [&](int rbufs) { return NEPI_WARPS * (stg_out_bytes + rbufs * stg_res_bytes) + VEC_BYTES; };
  auto stages_for = [&](int rbufs) { return (SMEM_MAX - 1024 - BAR_BYTES - epi_bytes(rbufs)) / C::STAGE_BYTES; };
  int stages = stages_for(res_bufs);
  // trade the second residual buffer for a pipeline stage when the ring would be shallow, or when the main loop is long
  // enough (K >= 1152) to hide a one-deep residual prefetch (fc2: the MMA warp waited for operands 25 % of the time
  // with 3 stages)
  if (needs_res && EPI != EPI_UP2 && (stages < 3 || (p.K >= 1152 && stages_for(1) > stages))) {
    res_bufs = 1;
    stages = stages_for(res_bufs);
  }
  if (stages > C::MAX_STAGES) stages = C::MAX_STAGES;
  if (stages > num_kb + 2) stages = num_kb + 2 > 2 ? num_kb + 2 : 2;
  // STD with several column tiles: stage the whole bias vector once when it fits without costing a pipeline stage
  int vec_all_bytes = 0;
  if (EPI == EPI_STD && staged && (p.N + BN - 1) / BN > 1) {
    const int need = ((p.N + 255) / 256) * 1024;  // N floats rounded up to 256 (the staging loop's stride)
    const int extra = need - VEC_BYTES;
    const int have = SMEM_MAX - 1024 - BAR_BYTES - epi_bytes(res_bufs) - stages * C::STAGE_BYTES;
    if (extra <= 0) vec_all_bytes = VEC_BYTES;
    else if (extra <= have) vec_all_bytes = need;
  }
  // Both warp sets on every tile (see the kernel): for UP1 and for STD when the main loop is a visible part of the tile
  // (K >= split_min_k, SB_GEMM_SPLIT_MINK to override for A/B runs)
  static int split_min_k = -1;
  if (split_min_k < 0) {
    const char* e = getenv("SB_GEMM_SPLIT_MINK");
    split_min_k = e ? atoi(e) : 512;
  }
  // UP2 (K = 64: no main loop to hide) stays on the alternating scheme: in the bench's decoder passes the split form
  // was 25 % slower (16.2 vs 12.9 ms per slice, profiles/r02w_gemm_shapes.txt vs r02k), UP1 (K = 256) 9 % faster.
  const int split = (EPI == EPI_UP1 || (EPI == EPI_STD && p.K >= split_min_k)) ? 1 : 0;
  const int smem_bytes = 1024 + BAR_BYTES + stages * C::STAGE_BYTES + epi_bytes(res_bufs) +
                         (vec_all_bytes > VEC_BYTES ? vec_all_bytes - VEC_BYTES : 0);
  const int m_tiles = (p.M + BM - 1) / BM;
  const int n_tiles = (p.N + BN - 1) / BN;
  const int tiles = m_tiles * n_tiles;
  const int grid = tiles < num_sms ? tiles : num_sms;
  gemm_bf16_tcgen05_kernel<BN, EPI, ACT><<<grid, NTHREADS, smem_bytes, stream>>>(tmA, tmB, p, stages, res_bufs, staged,
                                                                                stg_out_bytes, stg_res_bytes, split,
                                                                                vec_all_bytes);
  SB_CHECK_LAUNCH();
  return SB_OK;
}

// =====================================================================================================================
// CTA-pair version (cta_group::2) of the STD GEMM for the large encoder / decoder products.
//
// Why: a single CTA feeding 128 x 256 x 16 UMMAs reads A (4 KB) + B (8 KB) from shared memory every 128 clocks while TMA
// writes the same bytes: ~190 B/clk against a shared-memory pipe of ~128 B/clk, so the one-CTA main loop tops out at
// ~0.73 of the tensor peak (8192^3: 1 200 TFLOP/s vs 1 641 cuBLAS; the fc1 / QKV tiles then also wait for their staging
// traffic). A CTA PAIR computes a 256 x BN tile with ONE tcgen05.mma.cta_group::2 per k-step: each CTA stages its own
// 128 rows of A but only HALF of B (the tensor core reads the other half from the peer's shared memory), which halves
// the B traffic per SM (32 KB / stage and k-block instead of 48 for BN = 256) and doubles the ring depth per byte.
//
// Roles per CTA (384 threads): warp 0 TMA producer (both CTAs; all bytes complete on the LEADER's full barrier),
// warp 1 MMA issuer (leader CTA only; commits are multicast to the empty / accumulator-full barriers of both CTAs),
// warp 2 TMEM allocator (cta_group::2, both CTAs), warps 4-11 epilogue: both warp sets drain every tile (column halves)
// and arrive on the leader's accumulator-empty barrier through the cluster address space.
// Epilogue: TMEM -> registers -> (bias, activation, residual) -> swizzled staging tile -> ONE TMA tensor store per warp and
// 32-column group (cp.async.bulk.tensor...global.shared::cta: UTMASTG) instead of 4-8 LDS + STG per lane; the residual
// is gathered with cp.async into a second tile that is re-filled (next group, or the first group of the warp's next
// tile) as soon as it has been consumed.
template <int BN>
struct Cfg2 {
  static constexpr int MAX_STAGES = 8;
  static constexpr int A_BYTES = BM * BK * 2;
  static constexpr int B_BYTES = (BN / 2) * BK * 2;  // this CTA's half of the B tile
  static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
  static constexpr int ACC_STRIDE = BN == 192 ? 256 : BN;
  static constexpr int TMEM_COLS = 2 * ACC_STRIDE;
};

template <int BN, int ACT>
__device__ __forceinline__ void epilogue2_std(const GemmParams& p, const CUtensorMap* tmOut, uint32_t out_stg0,
                                              uint32_t out_stg1, int& ob, uint32_t res_stg, uint32_t vec,
                                              uint32_t tmem_acc, int m_idx, int n_idx, int q, int lane, int g_begin,
                                              int g_end, int vbase, bool& issued, int next_m_idx, int next_n_idx) {
  const int first_n = n_idx + g_begin * 32;
  if (first_n >= p.N) return;
  const int row0 = m_idx + q * 32;
  const int nrows = min(32, max(0, p.M - row0));
  const uint32_t taddr = tmem_acc + (static_cast<uint32_t>(q * 32) << 16);
  const bool has_res = p.res != nullptr;
  const int ld16r = has_res ? static_cast<int>(p.ldr / (p.res_f32 ? 4 : 8)) : 0;
  auto res_base16 = [&](int r0) -> int { return (p.res_mod > 0 ? (r0 % p.res_mod) : r0) * ld16r; };
  auto gather = [&](int base16, int rows, int n0) {
    const int ncols = min(32, p.N - n0);
    if (p.res_f32)
      gather_async_lin<128>(res_stg, reinterpret_cast<const uint8_t*>(p.res), base16 + n0 / 4, ld16r, rows, ncols * 4, lane);
    else
      gather_async_lin<64>(res_stg, reinterpret_cast<const uint8_t*>(p.res), base16 + n0 / 8, ld16r, rows, ncols * 2, lane);
  };
  const int res16 = has_res ? res_base16(row0) : 0;
  const int g_last = min(g_end, (p.N - n_idx + 31) / 32);  // exclusive
  if (has_res && !issued) gather(res16, nrows, first_n);
  issued = false;
  const int next_first_n = next_n_idx + g_begin * 32;
  const bool next_ok = has_res && next_m_idx >= 0 && next_first_n < p.N;
  const int next_row0 = next_m_idx + q * 32;
  uint32_t v[2][CH];
  sb::tmem_ld_32x16(taddr + static_cast<uint32_t>(g_begin * 32), v[0]);
#pragma unroll 1
  for (int g = g_begin; g < g_last; ++g) {
    const int n0 = n_idx + g * 32;
    const int ncols = min(32, p.N - n0);  // 16 or 32
    if (has_res) cp_async_wait_all();
    // output tiles alternate (when the launch reserved two): the tensor store issued two groups ago has read this one —
    // waiting for the PREVIOUS group's store here was the second largest stall of the epilogue (profiles/r02ze)
    const bool two = out_stg1 != out_stg0;
    const uint32_t out_stg = (two && ob) ? out_stg1 : out_stg0;
    ob ^= 1;
    if (lane == 0) {
      if (two)
        sb::bulk_wait_read<1>();
      else
        sb::bulk_wait_read<0>();
    }
    __syncwarp();
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      if (h * CH >= ncols) break;  // warp-uniform
      const int c0 = n0 + h * CH;
      sb::tmem_ld_wait();
      if (c0 + CH < p.N && (g * 2 + h + 1) < 2 * g_last)  // next chunk of this tile row
        sb::tmem_ld_32x16(taddr + static_cast<uint32_t>((g * 2 + h + 1) * CH), v[(h + 1) & 1]);
      float f[CH];
      const float2 al2 = sb::splat2(p.alpha);
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float4 b = ldsf4(vec, (c0 - vbase) + 4 * j);  // staged bias (LDS broadcast)
        const float2 v01 = make_float2(__uint_as_float(v[h][4 * j + 0]), __uint_as_float(v[h][4 * j + 1]));
        const float2 v23 = make_float2(__uint_as_float(v[h][4 * j + 2]), __uint_as_float(v[h][4 * j + 3]));
        float2 r01 = sb::fma2(v01, al2, make_float2(b.x, b.y));
        float2 r23 = sb::fma2(v23, al2, make_float2(b.z, b.w));
        if (ACT == 1) {
          r01 = sb::gelu_erf2(r01);
          r23 = sb::gelu_erf2(r23);
        } else if (ACT != 0) {
          r01 = make_float2(apply_act<ACT>(r01.x), apply_act<ACT>(r01.y));
          r23 = make_float2(apply_act<ACT>(r23.x), apply_act<ACT>(r23.y));
        }
        f[4 * j + 0] = r01.x;
        f[4 * j + 1] = r01.y;
        f[4 * j + 2] = r23.x;
        f[4 * j + 3] = r23.y;
      }
      if (has_res) {
        if (p.res_f32)
          add_res_from_stg<true>(res_stg, lane, h, f);
        else
          add_res_from_stg<false>(res_stg, lane, h, f);
      }
      stage_out(out_stg, lane, h, p.out_f32, f);
    }
    sb::fence_proxy_async();  // this lane's staging writes -> visible to the TMA (async proxy)
    __syncwarp();             // residual tile consumed, output tile complete
    if (has_res) {            // re-fill the residual tile right away: next group, or this warp's first group of its next tile
      if (g + 1 < g_last) {
        gather(res16, nrows, n0 + 32);
      } else if (next_ok) {
        gather(res_base16(next_row0), min(32, max(0, p.M - next_row0)), next_first_n);
        issued = true;
      }
    }
    if (lane == 0 && nrows > 0) {  // rows >= M and columns >= N are clipped by the tensor map
      sb::tma_store_2d_addr(tmOut, out_stg, n0, row0);
      sb::bulk_commit();
    }
  }
}

template <int BN, int ACT>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(NTHREADS, 1)
gemm2_bf16_tcgen05_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                          const __grid_constant__ CUtensorMap tmOut, const GemmParams p, const int stages,
                          const int stg_out_bytes, const int stg_res_bytes, const int vec_bytes, const int vec_all,
                          const int out_bufs) {
  using C = Cfg2<BN>;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~static_cast<uintptr_t>(1023));
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem);
  uint64_t* full_bar = bars;                          // used in the leader CTA only (both CTAs' bytes land there)
  uint64_t* empty_bar = bars + C::MAX_STAGES;         // per CTA: written by the leader's multicast commits
  uint64_t* tfull_bar = bars + 2 * C::MAX_STAGES;     // per CTA
  uint64_t* tempty_bar = bars + 2 * C::MAX_STAGES + 2;  // leader CTA only: 16 arrivals (8 epilogue warps x 2 CTAs)
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(bars + 2 * C::MAX_STAGES + 4);
  uint8_t* sA = smem + BAR_BYTES;
  uint8_t* sB = sA + stages * C::A_BYTES;
  float* sVec = reinterpret_cast<float*>(sA + stages * C::STAGE_BYTES);
  uint8_t* sEpi = reinterpret_cast<uint8_t*>(sVec) + vec_bytes;

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t rank = sb::cluster_ctarank();
  const bool leader = rank == 0;
  const int num_pairs = static_cast<int>(gridDim.x) >> 1;
  const int pair = static_cast<int>(blockIdx.x) >> 1;

  const int m_tiles = (p.M + 2 * BM - 1) / (2 * BM);
  const int n_tiles = (p.N + BN - 1) / BN;
  const int num_tiles = m_tiles * n_tiles;
  const int num_kb = (p.K + BK - 1) / BK;
  const int last_ksteps = ((p.K - (num_kb - 1) * BK) + 15) / 16;

  if (warp == 0 && lane == 0) {
    sb::tma_prefetch_desc(&tmA);
    sb::tma_prefetch_desc(&tmB);
    sb::tma_prefetch_desc(&tmOut);
  }
  if (warp == 1 && lane == 0) {
    for (int i = 0; i < stages; ++i) {
      sb::mbar_init(&full_bar[i], 1);
      sb::mbar_init(&empty_bar[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      sb::mbar_init(&tfull_bar[i], 1);
      sb::mbar_init(&tempty_bar[i], 2 * NEPI_WARPS);
    }
    sb::fence_barrier_init();
  }
  if (warp == 2) {
    sb::tmem_alloc_2sm(tmem_ptr, C::TMEM_COLS);
    sb::tmem_relinquish_2sm();
  }
  sb::tc_fence_before();
  __syncthreads();
  sb::cluster_sync();  // both CTAs' barriers are initialised before any remote arrive / TMA completion
  sb::tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;

  if (warp == 0) {
    // ===================== TMA producer (both CTAs) =====================
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      for (int tile = pair; tile < num_tiles; tile += num_pairs) {
        const int m_idx = (tile / n_tiles) * (2 * BM) + static_cast<int>(rank) * BM;
        const int n_idx = (tile % n_tiles) * BN + static_cast<int>(rank) * (BN / 2);
        for (int kb = 0; kb < num_kb; ++kb) {
          sb::mbar_wait(&empty_bar[stage], phase ^ 1);
          if (leader) sb::mbar_arrive_expect_tx(&full_bar[stage], 2 * C::STAGE_BYTES);
          const uint32_t bar = sb::mapa_shared(sb::smem_u32(&full_bar[stage]), 0);
          sb::tma_load_2d_2sm(sA + stage * C::A_BYTES, &tmA, bar, kb * BK, m_idx);
          sb::tma_load_2d_2sm(sB + stage * C::B_BYTES, &tmB, bar, kb * BK, n_idx);
          if (++stage == stages) {
            stage = 0;
            phase ^= 1;
          }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer (leader CTA; one elected lane per instruction) =====================
    if (leader) {
      constexpr uint32_t idesc = sb::umma_idesc_bf16(2 * BM, BN);
      int stage = 0;
      uint32_t phase = 0;
      int acc = 0;
      uint32_t acc_phase = 0;
      long long w_full = 0, w_tempty = 0;
      const long long t_begin = p.prof ? clock64() : 0;
      for (int tile = pair; tile < num_tiles; tile += num_pairs) {
        if (p.prof) {
          const long long t0 = clock64();
          sb::mbar_wait(&tempty_bar[acc], acc_phase ^ 1);
          w_tempty += clock64() - t0;
        } else {
          sb::mbar_wait(&tempty_bar[acc], acc_phase ^ 1);
        }
        sb::tc_fence_after();
        const uint32_t tmem_d = tmem_base + static_cast<uint32_t>(acc * C::ACC_STRIDE);
        for (int kb = 0; kb < num_kb; ++kb) {
          if (p.prof) {
            const long long t0 = clock64();
            sb::mbar_wait(&full_bar[stage], phase);
            w_full += clock64() - t0;
          } else {
            sb::mbar_wait(&full_bar[stage], phase);
          }
          sb::tc_fence_after();
          const uint64_t da = sb::umma_desc_k_sw128(sb::smem_u32(sA + stage * C::A_BYTES));
          const uint64_t db = sb::umma_desc_k_sw128(sb::smem_u32(sB + stage * C::B_BYTES));
          const int ksteps = (kb == num_kb - 1) ? last_ksteps : (BK / 16);
          for (int k = 0; k < ksteps; ++k) {
            if (sb::elect_one())
              sb::umma_bf16_2sm(tmem_d, da + static_cast<uint64_t>(2 * k), db + static_cast<uint64_t>(2 * k), idesc,
                                static_cast<uint32_t>((kb | k) != 0));
          }
          if (sb::elect_one()) sb::umma_commit_2sm(&empty_bar[stage], 3);  // frees the slot in BOTH CTAs
          __syncwarp();
          if (++stage == stages) {
            stage = 0;
            phase ^= 1;
          }
        }
        if (sb::elect_one()) sb::umma_commit_2sm(&tfull_bar[acc], 3);  // accumulator ready: both CTAs' epilogues
        __syncwarp();
        if (++acc == 2) {
          acc = 0;
          acc_phase ^= 1;
        }
      }
      if (p.prof && lane == 0) {
        atomicAdd(p.prof + 1, static_cast<unsigned long long>(w_full));
        atomicAdd(p.prof + 2, static_cast<unsigned long long>(w_tempty));
        atomicAdd(p.prof + 5, static_cast<unsigned long long>(clock64() - t_begin));
        atomicAdd(p.prof + 6, 1ull);
      }
    }
  } else if (warp >= 4) {
    // ===================== epilogue: both sets on every tile, set s = column half s =====================
    const int q = warp & 3;
    const int set = (warp - 4) >> 2;
    uint8_t* mine = sEpi + (warp - 4) * (out_bufs * stg_out_bytes + stg_res_bytes);
    const uint32_t out_stg0 = sb::smem_u32(mine);
    const uint32_t out_stg1 = sb::smem_u32(mine + (out_bufs - 1) * stg_out_bytes);
    const uint32_t res_stg = sb::smem_u32(mine + out_bufs * stg_out_bytes);
    int ob = 0;
    const uint32_t vec = sb::smem_u32(sVec);
    {  // bias: the whole vector (vec_all) or, for a single column tile, its BN entries — staged once
      const int tid256 = (warp - 4) * 32 + lane;
      const int valid = (p.N + 3) & ~3;
      for (int c = tid256 * 4; c < vec_bytes / 4; c += NEPI_WARPS * 128) {
        float4 b4 = make_float4(0.f, 0.f, 0.f, 0.f);
        if (p.bias != nullptr && c < valid) b4 = __ldg(reinterpret_cast<const float4*>(p.bias + c));
        *reinterpret_cast<float4*>(sVec + c) = b4;
      }
      asm volatile("bar.sync 6, %0;" ::"n"(NEPI_WARPS * 32) : "memory");
    }
    unsigned long long* e_cnt = reinterpret_cast<unsigned long long*>(smem + 512) + (warp - 4) * 3;
    if (p.prof && lane == 0) e_cnt[0] = e_cnt[1] = e_cnt[2] = 0ull;
    const uint32_t tempty_leader[2] = {sb::mapa_shared(sb::smem_u32(&tempty_bar[0]), 0),
                                       sb::mapa_shared(sb::smem_u32(&tempty_bar[1]), 0)};
    bool issued = false;
    int it = 0;
    constexpr int NG = BN / 32;
    for (int tile = pair; tile < num_tiles; tile += num_pairs, ++it) {
      const int st = it & 1;
      const uint32_t acc_phase = static_cast<uint32_t>((it >> 1) & 1);
      const int m_idx = (tile / n_tiles) * (2 * BM) + static_cast<int>(rank) * BM;
      const int n_idx = (tile % n_tiles) * BN;
      if (p.prof) {
        const long long t0 = clock64();
        sb::mbar_wait(&tfull_bar[st], acc_phase);
        if (lane == 0) {
          const long long t1 = clock64();
          e_cnt[0] += static_cast<unsigned long long>(t1 - t0);
          e_cnt[1] -= static_cast<unsigned long long>(t1);
        }
      } else {
        sb::mbar_wait(&tfull_bar[st], acc_phase);
      }
      sb::tc_fence_after();
      const uint32_t tmem_acc = tmem_base + static_cast<uint32_t>(st * C::ACC_STRIDE);
      const int nt = tile + num_pairs;
      const int next_m = nt < num_tiles ? (nt / n_tiles) * (2 * BM) + static_cast<int>(rank) * BM : -1;
      const int next_n = nt < num_tiles ? (nt % n_tiles) * BN : 0;
      epilogue2_std<BN, ACT>(p, &tmOut, out_stg0, out_stg1, ob, res_stg, vec, tmem_acc, m_idx, n_idx, q, lane, set * (NG / 2),
                             (set + 1) * (NG / 2), vec_all ? 0 : n_idx, issued, next_m, next_n);
      sb::tc_fence_before();
      __syncwarp();
      if (lane == 0) sb::mbar_arrive_cluster(st ? tempty_leader[1] : tempty_leader[0]);
      if (p.prof && lane == 0) {
        e_cnt[1] += static_cast<unsigned long long>(clock64());
        e_cnt[2] += 1ull;
      }
    }
    if (lane == 0) sb::bulk_wait<0>();  // all tensor stores of this warp have completed
    if (p.prof && lane == 0 && q == 0) {
      atomicAdd(p.prof + 3, e_cnt[0]);
      atomicAdd(p.prof + 4, e_cnt[1]);
      atomicAdd(p.prof + 7, e_cnt[2]);
    }
  }

  sb::tc_fence_before();
  __syncthreads();
  sb::cluster_sync();  // the peer may still be reading this CTA's operands / arriving on its barriers until here
  if (warp == 2) {
    sb::tc_fence_after();
    sb::tmem_dealloc_2sm(tmem_base, C::TMEM_COLS);
  }
}

template <int BN, int ACT>
int launch_gemm2(const void* A, long long lda, const void* W, long long ldw, const GemmParams& p, int num_sms,
                 cudaStream_t stream) {
  using C = Cfg2<BN>;
  static SbPerDeviceOnce attr_once;
  if (attr_once.need()) {
    SB_CHECK_CUDA(cudaFuncSetAttribute(gemm2_bf16_tcgen05_kernel<BN, ACT>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       SMEM_MAX));
    attr_once.mark();
  }
  CUtensorMap tmA, tmB, tmOut;
  int rc = sb_make_tmap_2d_bf16(&tmA, A, static_cast<uint64_t>(p.M), static_cast<uint64_t>(p.K), static_cast<uint64_t>(lda), BM, BK);
  if (rc != SB_OK) return rc;
  rc = sb_make_tmap_2d_bf16(&tmB, W, static_cast<uint64_t>(p.N), static_cast<uint64_t>(p.K), static_cast<uint64_t>(ldw), BN / 2, BK);
  if (rc != SB_OK) return rc;
  rc = sb_make_tmap_2d(&tmOut, p.out, p.out_f32 ? 4 : 2, static_cast<uint64_t>(p.M), static_cast<uint64_t>(p.N),
                       static_cast<uint64_t>(p.ldo), 32, 32, p.out_f32 ? 128 : 64);
  if (rc != SB_OK) return rc;
  const int stg_out_bytes = p.out_f32 ? STG_BYTES : STG_BYTES / 2;
  const int stg_res_bytes = p.res == nullptr ? 0 : (p.res_f32 ? STG_BYTES : STG_BYTES / 2);
  const int n_tiles = (p.N + BN - 1) / BN;
  const int out_bufs = p.out_f32 ? 1 : 2;  // bf16 output tiles are 2 KB: two per warp decouple the tensor stores
  const int epi = NEPI_WARPS * (out_bufs * stg_out_bytes + stg_res_bytes);
  // bias staging: all of N when it costs no pipeline stage, else the per-tile slice is not supported here -> caller falls back
  int vec_bytes = n_tiles > 1 ? ((p.N + 255) / 256) * 1024 : 1024;
  const int vec_all = n_tiles > 1 ? 1 : 0;
  int stages = (SMEM_MAX - 1024 - BAR_BYTES - epi - vec_bytes) / C::STAGE_BYTES;
  const int num_kb = (p.K + BK - 1) / BK;
  if (stages > C::MAX_STAGES) stages = C::MAX_STAGES;
  if (stages > num_kb + 2) stages = num_kb + 2 > 2 ? num_kb + 2 : 2;
  SB_REQUIRE(stages >= 2, "sb_gemm_bf16 (CTA pair): no room for the operand ring (N=%d)", p.N);
  const int smem_bytes = 1024 + BAR_BYTES + stages * C::STAGE_BYTES + vec_bytes + epi;
  const int m_tiles = (p.M + 2 * BM - 1) / (2 * BM);
  const int tiles = m_tiles * n_tiles;
  int pairs = num_sms / 2;
  if (pairs > tiles) pairs = tiles;
  gemm2_bf16_tcgen05_kernel<BN, ACT><<<2 * pairs, NTHREADS, smem_bytes, stream>>>(tmA, tmB, tmOut, p, stages, stg_out_bytes,
                                                                                 stg_res_bytes, vec_bytes, vec_all, out_bufs);
  SB_CHECK_LAUNCH();
  return SB_OK;
}

int g_num_sms = 0;
unsigned long long* g_prof = nullptr;  // sb_gemm_set_prof

int ensure_sms() {
  if (g_num_sms == 0) {
    int dev = 0;
    SB_CHECK_CUDA(cudaGetDevice(&dev));
    SB_CHECK_CUDA(cudaDeviceGetAttribute(&g_num_sms, cudaDevAttrMultiProcessorCount, dev));
    // SB_GEMM_SMS: SMs the persistent GEMM kernels may occupy. With concurrent slice workers (one slice encoding while
    // another decodes) the SMs left over keep running the other worker's non-persistent, HBM-bound decoder kernels.
    if (const char* e = getenv("SB_GEMM_SMS")) {
      const int lim = atoi(e);
      if (lim >= 2 && lim < g_num_sms) g_num_sms = lim & ~1;
    }
  }
  return SB_OK;
}

int make_maps(const void* A, long long lda, const void* W, long long ldw, int M, int N, int K, int bn,
              CUtensorMap* tmA, CUtensorMap* tmB) {
  SB_REQUIRE(M > 0 && N > 0 && K > 0, "sb_gemm: empty problem M=%d N=%d K=%d", M, N, K);
  SB_REQUIRE((lda % 8) == 0 && (ldw % 8) == 0, "sb_gemm: lda/ldw must be multiples of 8");
  SB_REQUIRE((reinterpret_cast<uintptr_t>(A) & 15) == 0 && (reinterpret_cast<uintptr_t>(W) & 15) == 0,
             "sb_gemm: A/W must be 16-byte aligned");
  int rc = sb_make_tmap_2d_bf16(tmA, A, static_cast<uint64_t>(M), static_cast<uint64_t>(K),
                                static_cast<uint64_t>(lda), BM, BK);
  if (rc != SB_OK) return rc;
  return sb_make_tmap_2d_bf16(tmB, W, static_cast<uint64_t>(N), static_cast<uint64_t>(K),
                              static_cast<uint64_t>(ldw), static_cast<uint32_t>(bn), BK);
}

}  // namespace

// Diagnostic: when `counters` (device, 8 x u64, zeroed by the caller) is non-null every following sb_gemm_* launch of this
// process adds clock64 totals over its CTAs: [0] producer waiting for a free operand slot, [1] MMA warp waiting for
// operands, [2] MMA warp waiting for a drained accumulator, [3] epilogue set (warp q = 0) waiting for an accumulator,
// [4] epilogue working, [5] MMA-warp clocks from first to last tile, [6] CTAs, [7] tiles drained by the reporting warps.
extern "C" int sb_gemm_set_prof(unsigned long long* counters) {
  g_prof = counters;
  return SB_OK;
}

extern "C" int sb_gemm_bf16(const void* A, long long lda, const void* W, long long ldw, void* out,
                            long long ldo, int M, int N, int K, const float* bias, int act,
                            const void* residual, long long ldr, int res_mod, int flags,
                            float alpha, int force_bn, void* stream_) {
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  SB_REQUIRE(act >= 0 && act <= 3, "sb_gemm_bf16: bad act %d", act);
  if (ensure_sms() != SB_OK) return SB_ERR_CUDA;
  GemmParams p;
  memset(&p, 0, sizeof(p));
  p.M = M;
  p.N = N;
  p.K = K;
  p.out = out;
  p.ldo = ldo;
  p.out_f32 = (flags & 1) ? 1 : 0;
  p.bias = bias;
  p.act = act;
  p.res = residual;
  p.ldr = ldr;
  p.res_f32 = (flags & 2) ? 1 : 0;
  p.res_mod = res_mod;
  p.alpha = alpha;
  p.prof = g_prof;

  // Tile-N choice: minimise waves x tile cost (BN as proxy for per-tile time).
  int bn = force_bn < 0 ? 0 : force_bn;
  if (bn == 0) {
    if (N <= 64) {
      bn = 64;
    } else {
      const long long m_tiles = (M + BM - 1) / BM;
      long long best = -1;
      // 192 divides Hiera-L's 576 / 1152-wide outputs exactly (256 wastes a quarter of the last tile): a candidate for
      // every product with a residual (they all have N in {144, 288, 576, 1152}; profiles/r02u_gemm_tile_ab.log) and for
      // K >= 1152 otherwise.
      static int min_k_192 = -1;
      if (min_k_192 < 0) {
        const char* e = getenv("SB_GEMM_192_MINK");
        min_k_192 = e ? atoi(e) : 1152;
      }
      const int cands[4] = {256, 192, 128, 64};
      for (int i = 0; i < 4; ++i) {
        const int c = cands[i];
        if (c == 192 && K < min_k_192 && residual == nullptr) continue;
        const long long tiles = m_tiles * ((N + c - 1) / c);
        const long long waves = (tiles + g_num_sms - 1) / g_num_sms;
        const long long cost = waves * (c + 24);  // +24: fixed per-tile overhead proxy
        if (best < 0 || cost < best) {
          best = cost;
          bn = c;
        }
      }
    }
  }
  SB_REQUIRE(bn == 64 || bn == 128 || bn == 192 || bn == 256, "sb_gemm_bf16: bad tile N %d", bn);
  // CTA-pair kernel (cta_group::2, TMA-store epilogue) for the large products: 256-row pair tiles
  {
    static int pair_env = -1;  // SB_GEMM_2CTA=0 keeps every product on the single-CTA kernel (A/B measurements)
    if (pair_env < 0) {
      const char* e = getenv("SB_GEMM_2CTA");
      pair_env = (e && atoi(e) == 0) ? 0 : 1;
    }
    const long long ob = ldo * (p.out_f32 ? 4 : 2), rb = ldr * (p.res_f32 ? 4 : 2);
    // Measured per shape (profiles/r02u_gemm_tile_ab.log, cold L2): the pair kernel wins for the bf16-output products
    // without a residual (fc1 +6 %, stage-2 fc1 +9 %), the single-CTA kernel (two residual tiles, outputs staged in
    // place) for the "+ residual" ones (proj +8 %), so a residual keeps the product on the single-CTA kernel unless
    // the pair width is forced.
    const bool ok = pair_env && force_bn <= 0 && (force_bn < 0 || residual == nullptr) && M >= 4096 && N >= 128 && (N % 16) == 0 && (ob % 16) == 0 &&
                    (!residual || rb % 16 == 0) && ((reinterpret_cast<uintptr_t>(out) & 15) == 0) &&
                    ((reinterpret_cast<uintptr_t>(residual) & 15) == 0) && (res_mod == 0 || (res_mod % 32) == 0) &&
                    (static_cast<long long>(M) * ob < (1ll << 35)) && (!residual || static_cast<long long>(M) * rb < (1ll << 35)) &&
                    (lda % 8) == 0 && (ldw % 8) == 0 && ((reinterpret_cast<uintptr_t>(A) | reinterpret_cast<uintptr_t>(W)) & 15) == 0 &&
                    N <= 8192;
    if (ok) {
      int bn2 = force_bn < 0 ? -force_bn : force_bn;  // tests: a negative force_bn selects the pair-tile width
      if (bn2 == 0) {  // pair tiles: waves x (tile cost); 192 divides 576 / 1152 exactly
        const long long m_tiles2 = (M + 2 * BM - 1) / (2 * BM);
        long long best = -1;
        const int cands[3] = {256, 192, 128};
        for (int i = 0; i < 3; ++i) {
          const int c = cands[i];
          const long long tiles = m_tiles2 * ((N + c - 1) / c);
          const long long waves = (tiles + g_num_sms / 2 - 1) / (g_num_sms / 2);
          // bytes staged per k-block and CTA ~ 128 rows of A + c / 2 rows of B: wider tiles re-use A better
          const long long cost = waves * (c + 256);
          if (best < 0 || cost < best) {
            best = cost;
            bn2 = c;
          }
        }
      }
      if (bn2 == 128 || bn2 == 192 || bn2 == 256) {
#define SB_DISPATCH_ACT2(BN_)                                                                 \
  switch (act) {                                                                             \
    case 1: return launch_gemm2<BN_, 1>(A, lda, W, ldw, p, g_num_sms, stream);                \
    case 2: return launch_gemm2<BN_, 2>(A, lda, W, ldw, p, g_num_sms, stream);                \
    case 3: return launch_gemm2<BN_, 3>(A, lda, W, ldw, p, g_num_sms, stream);                \
    default: return launch_gemm2<BN_, 0>(A, lda, W, ldw, p, g_num_sms, stream);               \
  }
        if (bn2 == 256) { SB_DISPATCH_ACT2(256) }
        if (bn2 == 192) { SB_DISPATCH_ACT2(192) }
        SB_DISPATCH_ACT2(128)
#undef SB_DISPATCH_ACT2
      }
    }
  }
  CUtensorMap tmA, tmB;
  int rc = make_maps(A, lda, W, ldw, M, N, K, bn, &tmA, &tmB);
  if (rc != SB_OK) return rc;
#define SB_DISPATCH_ACT(BN_)                                                        \
  switch (act) {                                                                   \
    case 1: return launch_gemm<BN_, EPI_STD, 1>(tmA, tmB, p, g_num_sms, stream);   \
    case 2: return launch_gemm<BN_, EPI_STD, 2>(tmA, tmB, p, g_num_sms, stream);   \
    case 3: return launch_gemm<BN_, EPI_STD, 3>(tmA, tmB, p, g_num_sms, stream);   \
    default: return launch_gemm<BN_, EPI_STD, 0>(tmA, tmB, p, g_num_sms, stream);  \
  }
  if (bn == 256) { SB_DISPATCH_ACT(256) }
  if (bn == 192) { SB_DISPATCH_ACT(192) }
  if (bn == 128) { SB_DISPATCH_ACT(128) }
  SB_DISPATCH_ACT(64)
#undef SB_DISPATCH_ACT
}

// out[M,N] = LayerNorm_N(A @ W^T + bias + residual[m % res_mod or m]) * gamma + beta, N in {64,128,256} x (N%16==0).
// flags: bit0 out fp32 (else bf16), bit1 residual fp32 (else bf16).
extern "C" int sb_gemm_ln(const void* A, long long lda, const void* W, long long ldw, void* out, long long ldo,
                          int M, int N, int K, const float* bias, const void* residual, long long ldr,
                          int res_mod, int flags, const float* gamma, const float* beta, float eps,
                          void* stream_) {
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  SB_REQUIRE(N <= 256 && (N % 16) == 0, "sb_gemm_ln: N must be a multiple of 16 and <= 256 (got %d)", N);
  SB_REQUIRE((ldo % 8) == 0 && (!residual || (ldr % 8) == 0), "sb_gemm_ln: ldo/ldr must be multiples of 8");
  SB_REQUIRE(gamma && beta, "sb_gemm_ln: gamma/beta required");
  if (ensure_sms() != SB_OK) return SB_ERR_CUDA;
  GemmParams p;
  memset(&p, 0, sizeof(p));
  p.M = M;
  p.N = N;
  p.K = K;
  p.out = out;
  p.ldo = ldo;
  p.out_f32 = (flags & 1) ? 1 : 0;
  p.bias = bias;
  p.res = residual;
  p.ldr = ldr;
  p.res_f32 = (flags & 2) ? 1 : 0;
  p.res_mod = res_mod;
  p.alpha = 1.f;
  p.gamma = gamma;
  p.beta = beta;
  p.eps = eps;
  const int bn = N > 128 ? 256 : (N > 64 ? 128 : 64);
  CUtensorMap tmA, tmB;
  int rc = make_maps(A, lda, W, ldw, M, N, K, bn, &tmA, &tmB);
  if (rc != SB_OK) return rc;
  if (bn == 256) return launch_gemm<256, EPI_LN>(tmA, tmB, p, g_num_sms, stream);
  if (bn == 128) return launch_gemm<128, EPI_LN>(tmA, tmB, p, g_num_sms, stream);
  return launch_gemm<64, EPI_LN>(tmA, tmB, p, g_num_sms, stream);
}

// Mask-decoder output_upscaling stage 1: keys [B*gh*gw, 256] bf16 @ W1 [4*64, 256] (+bias[256]) -> pixel shuffle,
// + feat_s1 (fp32 [.., 2gh*2gw, 64], batch stride skip_bstride), LayerNorm2d(64, eps), GELU -> u1 [B*2gh*2gw, 64] bf16.
extern "C" int sb_gemm_upscale1(const void* A, long long lda, const void* W, long long ldw, int B, int gh, int gw,
                                const float* bias, const float* feat_s1, long long skip_bstride,
                                const float* gamma, const float* beta, float eps, void* u1, const int* plist,
                                const int* pcount, void* stream_) {
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  SB_REQUIRE(B > 0 && gh > 0 && gw > 0 && bias && feat_s1 && gamma && beta, "sb_gemm_upscale1: bad arguments");
  if (ensure_sms() != SB_OK) return SB_ERR_CUDA;
  GemmParams p;
  memset(&p, 0, sizeof(p));
  p.M = B * gh * gw;
  p.N = 256;
  p.K = 256;
  p.out = u1;
  p.bias = bias;
  p.alpha = 1.f;
  p.gamma = gamma;
  p.beta = beta;
  p.eps = eps;
  p.skip = feat_s1;
  p.skip_bstride = skip_bstride;
  p.gh = gh;
  p.gw = gw;
  SB_REQUIRE((plist == nullptr) == (pcount == nullptr) && (plist == nullptr || (gh * gw) % BM == 0),
             "sb_gemm_upscale1: prompt list needs its count and gh * gw a multiple of 128");
  p.plist = plist;
  p.pcount = pcount;
  p.prof = g_prof;
  CUtensorMap tmA, tmB;
  int rc = make_maps(A, lda, W, ldw, p.M, 256, 256, 256, &tmA, &tmB);
  if (rc != SB_OK) return rc;
  return launch_gemm<256, EPI_UP1>(tmA, tmB, p, g_num_sms, stream);
}

// Stage 2: u1 [B*gh*gw, 64] bf16 @ W2 [4*32, 64] (+bias[128]) -> pixel shuffle, + feat_s0 (fp32 [.., 2gh*2gw, 32]), GELU,
// dot with hyper [B,4,32] -> masks [B, 4, 2gh, 2gw] fp32. gh*gw must be a multiple of 128 (a tile never spans prompts).
extern "C" int sb_gemm_upscale2(const void* A, long long lda, const void* W, long long ldw, int B, int gh, int gw,
                                const float* bias, const float* feat_s0, long long skip_bstride, const float* hyper,
                                float* masks, const int* plist, const int* pcount, void* stream_) {
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  SB_REQUIRE(B > 0 && gh > 0 && gw > 0 && bias && feat_s0 && hyper, "sb_gemm_upscale2: bad arguments");
  if (ensure_sms() != SB_OK) return SB_ERR_CUDA;
  GemmParams p;
  memset(&p, 0, sizeof(p));
  p.M = B * gh * gw;
  p.N = 128;
  p.K = 64;
  p.out = masks;
  p.bias = bias;
  p.alpha = 1.f;
  p.skip = feat_s0;
  p.skip_bstride = skip_bstride;
  p.hyper = hyper;
  p.gh = gh;
  p.gw = gw;
  SB_REQUIRE((plist == nullptr) == (pcount == nullptr) && (gh * gw) % BM == 0,
             "sb_gemm_upscale2: gh * gw must be a multiple of 128 (and a prompt list needs its count)");
  p.plist = plist;
  p.pcount = pcount;
  p.prof = g_prof;
  CUtensorMap tmA, tmB;
  int rc = make_maps(A, lda, W, ldw, p.M, 128, 64, 128, &tmA, &tmB);
  if (rc != SB_OK) return rc;
  return launch_gemm<128, EPI_UP2>(tmA, tmB, p, g_num_sms, stream);
}
