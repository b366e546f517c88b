// ColBERT late-interaction max-sim for sm_100a.
//
//   score[p] = sum_i qmask[i] * max_j ( dmask[j] ? <q_i, d_j> : -1000 )
//
// Reference arithmetic: matchmaker/models/colbert.py:68-75 (forward), :100-112
// (forward_aggregation), :154-162 (forward_inbatch_aggregation).  Not a port: the reference
// materialises the [B, Lq, Ld] score tensor with cuBLAS bmm and runs four more eager kernels
// over it; here one persistent kernel streams the document token matrices through shared
// memory once and never writes the score matrix.
//
// Kernel `maxsim_tc_kernel` (the hot path; HBM-bound, 2 bytes per document element):
//   * one CTA per SM, persistent over a contiguous range of pairs;
//   * warp 0 (one lane): TMA producer.  A document tile is 128 token rows x dim, fetched as
//     [KBS k-blocks][128 rows][64 halfs] with SWIZZLE_128B by ONE 4-D cp.async.bulk.tensor
//     per stage (rows past Ld are zero-filled by the TMA unit, no HBM traffic); the query
//     matrix ([NPAD rows][dim]) lives in a 2-slot ring and is re-fetched only when the query
//     of consecutive pairs changes;
//   * warp 1 (one lane): tcgen05.mma issuer.  D[128 doc rows x NPAD query cols] (fp32, TMEM)
//     = Doc_tile[128 x dim] * Q[NPAD x dim]^T, kind::f16, UMMA_K = 16; 4 accumulator stages
//     in TMEM so the tensor pipe never waits for the epilogue;
//   * warps 2..5: epilogue.  tcgen05.ld the accumulator (lane = document row, register =
//     query column), apply the document mask (-1000) / tile padding (-inf), column-wise max
//     across the 32 lanes by a shuffle "transpose-reduce" (31 SHFL + 31 FMNMX for 32 columns),
//     running max over the tiles of a pair in registers, cross-warp combine through 2 KB of
//     shared memory, query mask, warp-sum, one fp32 store per pair.
//
// Kernel `maxsim_simt_kernel`: CUDA-core version for every shape of the envelope (fp32 inputs,
// dim % 64 != 0, argmax for backward, query tiles too large for the tensor-core kernels); also the
// in-library cross-check of the tensor-core path.
//
// Envelope of mmb200_maxsim_fwd: 1 <= Lq <= 128, 1 <= dim <= 1024, any Ld >= 1; shapes outside it
// are rejected up front.
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include <algorithm>
#include <vector>

#include "host_util.cuh"
#include "masks.cuh"
#include "maxsim.cuh"
#include "ptx.cuh"

namespace mmb {

// ---------------------------------------------------------------------------------------------
// shared device helpers
// ---------------------------------------------------------------------------------------------
template <typename T>
__device__ __forceinline__ float to_float(T v);
template <>
__device__ __forceinline__ float to_float<float>(float v) { return v; }
template <>
__device__ __forceinline__ float to_float<__half>(__half v) { return __half2float(v); }
template <>
__device__ __forceinline__ float to_float<__nv_bfloat16>(__nv_bfloat16 v) { return __bfloat162float(v); }

__device__ __forceinline__ int64_t pair_query(const MaxsimParams& P, int64_t p) {
  return P.pair_q ? static_cast<int64_t>(P.pair_q[p]) : (p + P.pair_base) / P.docs_per_query;
}
__device__ __forceinline__ int64_t pair_doc(const MaxsimParams& P, int64_t p) {
  return P.pair_d ? static_cast<int64_t>(P.pair_d[p]) : p;
}
__device__ __forceinline__ int64_t pair_dmask_row(const MaxsimParams& P, int64_t p) {
  return P.pair_dmask ? static_cast<int64_t>(P.pair_dmask[p]) : pair_doc(P, p);
}

constexpr float kMaskedScore = -1000.0f;  // colbert.py:69

// ---------------------------------------------------------------------------------------------
// SIMT kernel: one CTA (128 threads) per pair.  Q is staged in shared memory as fp32 with a
// padded row stride, `qrows` query rows per pass (all Lq rows when they fit, else a multiple of
// 32); per pass warp w takes document rows w, w+4, ...; lane l owns the pass's query rows l, l+32,
// ...  Each (query row, document row) dot product is the same fmaf chain over k whatever the pass
// size, so scores and argmax do not depend on how many passes a shape needs.
// ---------------------------------------------------------------------------------------------
constexpr int kSimtThreads = 128;
constexpr int kSimtMaxQPerLane = 4;  // Lq <= 128
constexpr int kMaxsimMaxLq = 32 * kSimtMaxQPerLane;
constexpr int kMaxsimMaxDim = 1024;

template <typename T>
__global__ void __launch_bounds__(kSimtThreads) maxsim_simt_kernel(MaxsimParams P, int qrows) {
  extern __shared__ float smem_f[];
  const int Lq = P.Lq, Ld = P.Ld, dim = P.dim;
  const int qstride = dim + 1;
  float* sq = smem_f;                          // [qrows][dim+1]
  float* smax = sq + (size_t)qrows * qstride;  // [4][Lq]
  int* sarg = reinterpret_cast<int*>(smax + 4 * Lq);  // [4][Lq]
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  for (int64_t p = blockIdx.x; p < P.n_pairs; p += gridDim.x) {
    const int64_t qi = pair_query(P, p), di = pair_doc(P, p), dmi = pair_dmask_row(P, p);
    const T* dptr = static_cast<const T*>(P.d) + di * (int64_t)Ld * dim;
    for (int r0 = 0; r0 < Lq; r0 += qrows) {
      const int nr = min(qrows, Lq - r0);
      const T* qptr = static_cast<const T*>(P.q) + (qi * (int64_t)Lq + r0) * dim;
      __syncthreads();
      for (int e = threadIdx.x; e < nr * dim; e += kSimtThreads) {
        sq[(e / dim) * qstride + (e % dim)] = to_float(qptr[e]);
      }
      __syncthreads();
      float best[kSimtMaxQPerLane];
      int barg[kSimtMaxQPerLane];
#pragma unroll
      for (int t = 0; t < kSimtMaxQPerLane; ++t) { best[t] = -INFINITY; barg[t] = -1; }
      for (int j = warp; j < Ld; j += 4) {
        const bool ok = mask_at(P.d_mask, P.d_mask ? P.mask_dtype : MMB200_MASK_NONE, dmi * (int64_t)Ld + j);
        float acc[kSimtMaxQPerLane] = {0.f, 0.f, 0.f, 0.f};
        if (ok) {
          const T* drow = dptr + (int64_t)j * dim;
          for (int k = 0; k < dim; ++k) {
            const float dv = to_float(drow[k]);
#pragma unroll
            for (int t = 0; t < kSimtMaxQPerLane; ++t) {
              const int i = lane + 32 * t;
              if (i < nr) acc[t] = fmaf(sq[i * qstride + k], dv, acc[t]);
            }
          }
        }
#pragma unroll
        for (int t = 0; t < kSimtMaxQPerLane; ++t) {
          const float v = ok ? acc[t] : kMaskedScore;
          if (v > best[t]) { best[t] = v; barg[t] = ok ? j : -1; }
        }
      }
#pragma unroll
      for (int t = 0; t < kSimtMaxQPerLane; ++t) {
        const int i = lane + 32 * t;
        if (i < nr) { smax[warp * Lq + r0 + i] = best[t]; sarg[warp * Lq + r0 + i] = barg[t]; }
      }
    }
    __syncthreads();
    if (warp == 0) {
      float total = 0.f;
      for (int i = lane; i < Lq; i += 32) {
        float m = smax[i];
        int a = sarg[i];
        for (int w = 1; w < 4; ++w) {
          const float v = smax[w * Lq + i];
          const int aw = sarg[w * Lq + i];
          // first occurrence of the max (lowest j) like a sequential scan
          if (v > m || (v == m && aw >= 0 && (a < 0 || aw < a))) { m = v; a = aw; }
        }
        const bool qok = mask_at(P.q_mask, P.q_mask ? P.mask_dtype : MMB200_MASK_NONE, qi * (int64_t)Lq + i);
        total += qok ? m : 0.f;
        if (P.argmax) P.argmax[p * Lq + i] = qok ? a : -1;
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) total += __shfl_xor_sync(0xffffffffu, total, o);
      if (lane == 0) P.out[p] = total;
    }
  }
}

// ---------------------------------------------------------------------------------------------
// tcgen05 kernel
// ---------------------------------------------------------------------------------------------
constexpr int kTcThreads = 192;        // warp 0 TMA, warp 1 MMA, warps 2-5 epilogue
constexpr int kTileRows = 128;         // UMMA M
constexpr int kKBlockElems = 64;       // 64 x 16-bit = 128 B = one SWIZZLE_128B row
constexpr int kKBlockBytes = kTileRows * 128;  // 16 KB: [128 rows][128 B]
constexpr int kMaxStages = 12;
constexpr int kAccStages = 4;
constexpr int kQSlots = 2;

struct TcShared {  // control block placed after the tile storage
  uint64_t full[kMaxStages];
  uint64_t empty[kMaxStages];
  uint64_t qfull[kQSlots];
  uint64_t qempty[kQSlots];
  uint64_t accfull[kAccStages];
  uint64_t accempty[kAccStages];
  uint32_t tmem_base;
  uint32_t pad;
  float colmax[2][4][128];  // [pair parity][epilogue warp][query column]
};

struct TcLaunch {
  int32_t npad;        // query rows padded to a multiple of 32 (UMMA N, TMEM columns per stage)
  int32_t kblocks;     // dim / 64
  int32_t kbs;         // k-blocks per stage (1 or 2)
  int32_t stages;      // document stages in the ring
  int32_t tiles;       // ceil(Ld / 128)
  int32_t fmt;         // kFmtF16 / kFmtBF16
  int32_t tmem_cols;   // power of two >= kAccStages * npad
  int32_t qslot_bytes; // kblocks * npad * 128
};

// Column-wise max over the 32 lanes of a warp for 32 per-lane values: afterwards lane l holds
// max over lanes of v[l].  Halving exchange: 16+8+4+2+1 shuffles.
__device__ __forceinline__ float warp_transpose_max32(float (&v)[32], int lane) {
#pragma unroll
  for (int i = 0; i < 16; ++i) {
    const bool up = (lane & 16) != 0;
    const float send = up ? v[i] : v[i + 16];
    const float keep = up ? v[i + 16] : v[i];
    v[i] = fmaxf(keep, __shfl_xor_sync(0xffffffffu, send, 16));
  }
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const bool up = (lane & 8) != 0;
    const float send = up ? v[i] : v[i + 8];
    const float keep = up ? v[i + 8] : v[i];
    v[i] = fmaxf(keep, __shfl_xor_sync(0xffffffffu, send, 8));
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const bool up = (lane & 4) != 0;
    const float send = up ? v[i] : v[i + 4];
    const float keep = up ? v[i + 4] : v[i];
    v[i] = fmaxf(keep, __shfl_xor_sync(0xffffffffu, send, 4));
  }
#pragma unroll
  for (int i = 0; i < 2; ++i) {
    const bool up = (lane & 2) != 0;
    const float send = up ? v[i] : v[i + 2];
    const float keep = up ? v[i + 2] : v[i];
    v[i] = fmaxf(keep, __shfl_xor_sync(0xffffffffu, send, 2));
  }
  {
    const bool up = (lane & 1) != 0;
    const float send = up ? v[0] : v[1];
    const float keep = up ? v[1] : v[0];
    v[0] = fmaxf(keep, __shfl_xor_sync(0xffffffffu, send, 1));
  }
  return v[0];
}

template <int KBS>
__global__ void __launch_bounds__(kTcThreads, 1)
maxsim_tc_kernel(const __grid_constant__ CUtensorMap tmap_q, const __grid_constant__ CUtensorMap tmap_d,
                 MaxsimParams P, TcLaunch L) {
  extern __shared__ uint8_t smem_raw[];
  // SWIZZLE_128B tiles need 1024-B alignment
  // 1024-B alignment for SWIZZLE_128B tiles, derived by pointer arithmetic on the __shared__ array so the
  // compiler keeps the shared address space (LDS/STS instead of generic LD/ST)
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  constexpr int kStageBytes = KBS * kKBlockBytes;
  uint8_t* stage_base = smem;
  uint8_t* q_base = smem + (size_t)L.stages * kStageBytes;
  TcShared* S = reinterpret_cast<TcShared*>(q_base + (size_t)kQSlots * L.qslot_bytes);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  // contiguous pair range of this CTA
  const int64_t per = P.n_pairs / gridDim.x, rem = P.n_pairs % gridDim.x;
  const int64_t p_begin = (int64_t)blockIdx.x * per + min((int64_t)blockIdx.x, rem);
  const int64_t p_end = p_begin + per + ((int64_t)blockIdx.x < rem ? 1 : 0);

  if (threadIdx.x == 0) {
    prefetch_tensormap(&tmap_q);
    prefetch_tensormap(&tmap_d);
    for (int s = 0; s < L.stages; ++s) { mbar_init(&S->full[s], 1); mbar_init(&S->empty[s], 1); }
    for (int s = 0; s < kQSlots; ++s) { mbar_init(&S->qfull[s], 1); mbar_init(&S->qempty[s], 1); }
    for (int s = 0; s < kAccStages; ++s) { mbar_init(&S->accfull[s], 1); mbar_init(&S->accempty[s], 4); }
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc(&S->tmem_base, (uint32_t)L.tmem_cols);
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  const uint32_t tmem_base = S->tmem_base;

  const int ksteps = L.kblocks / KBS;

  if (warp == 0) {
    // ------------------------------- TMA producer -------------------------------
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      int64_t prev_q = -1;
      uint32_t qcount = 0;
      for (int64_t p = p_begin; p < p_end; ++p) {
        const int64_t qi = pair_query(P, p), di = pair_doc(P, p);
        if (qi != prev_q) {
          const uint32_t slot = qcount & 1u, use = qcount >> 1;
          mbar_wait(&S->qempty[slot], (use & 1u) ^ 1u);
          mbar_arrive_expect_tx(&S->qfull[slot], (uint32_t)L.qslot_bytes);
          tma_load_4d(&tmap_q, q_base + (size_t)slot * L.qslot_bytes, &S->qfull[slot], 0, 0, 0, (int)qi,
                      kEvictLast);
          ++qcount;
          prev_q = qi;
        }
        for (int t = 0; t < L.tiles; ++t) {
          for (int ks = 0; ks < ksteps; ++ks) {
            mbar_wait(&S->empty[stage], phase ^ 1u);
            mbar_arrive_expect_tx(&S->full[stage], (uint32_t)kStageBytes);
            tma_load_4d(&tmap_d, stage_base + (size_t)stage * kStageBytes, &S->full[stage], 0, t * kTileRows,
                        ks * KBS, (int)di, kEvictFirst);
            if (++stage == L.stages) { stage = 0; phase ^= 1u; }
          }
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------- MMA issuer ---------------------------------
    if (lane == 0) {
      const uint32_t idesc = make_idesc((uint32_t)L.fmt, kTileRows, (uint32_t)L.npad);
      int stage = 0;
      uint32_t phase = 0;
      int acc = 0;
      uint32_t accphase = 0;
      int64_t prev_q = -1;
      uint32_t qcount = 0;
      int cur_slot = 0;
      for (int64_t p = p_begin; p < p_end; ++p) {
        const int64_t qi = pair_query(P, p);
        if (qi != prev_q) {
          if (prev_q >= 0) umma_commit(&S->qempty[cur_slot]);  // all MMAs reading the old Q are done
          cur_slot = (int)(qcount & 1u);
          mbar_wait(&S->qfull[cur_slot], (qcount >> 1) & 1u);
          ++qcount;
          prev_q = qi;
        }
        const uint32_t qaddr = smem_u32(q_base + (size_t)cur_slot * L.qslot_bytes);
        for (int t = 0; t < L.tiles; ++t) {
          mbar_wait(&S->accempty[acc], accphase ^ 1u);
          tc_fence_after_sync();
          const uint32_t tmem_d = tmem_base + (uint32_t)(acc * L.npad);
          for (int ks = 0; ks < ksteps; ++ks) {
            mbar_wait(&S->full[stage], phase);
            tc_fence_after_sync();
            const uint32_t aaddr = smem_u32(stage_base + (size_t)stage * kStageBytes);
#pragma unroll
            for (int kb = 0; kb < KBS; ++kb) {
              const uint32_t a_kb = aaddr + kb * kKBlockBytes;
              const uint32_t b_kb = qaddr + (uint32_t)((ks * KBS + kb) * L.npad * 128);
#pragma unroll
              for (int k = 0; k < 4; ++k) {  // 64 / UMMA_K(16)
                umma_f16(tmem_d, make_sw128_kmajor_desc(a_kb + k * 32), make_sw128_kmajor_desc(b_kb + k * 32),
                         idesc, (uint32_t)((ks | kb | k) != 0));
              }
            }
            umma_commit(&S->empty[stage]);  // smem stage free once these MMAs retire
            if (++stage == L.stages) { stage = 0; phase ^= 1u; }
          }
          umma_commit(&S->accfull[acc]);
          if (++acc == kAccStages) { acc = 0; accphase ^= 1u; }
        }
      }
    }
  } else {
    // ------------------------------- epilogue ------------------------------------
    const int ew = warp - 2;          // 0..3
    const int lq = warp & 3;          // TMEM lane quarter this warp may access
    const int ncol32 = L.npad >> 5;   // 32-column groups
    int acc = 0;
    uint32_t accphase = 0;
    const int dmt = P.d_mask ? P.mask_dtype : MMB200_MASK_NONE;
    const int qmt = P.q_mask ? P.mask_dtype : MMB200_MASK_NONE;
    // Mask words are fetched two tiles ahead and only *tested* when their tile is processed, so the
    // global-load latency hides behind the TMEM loads / shuffles of the tiles in between.
    int64_t fp = p_begin;  // (pair, tile) whose mask word is fetched next
    int ft = 0;
    auto fetch = [&](uint64_t& raw) -> bool {  // returns "row lies inside the document"
      bool in_doc = false;
      raw = 1;
      if (fp < p_end) {
        const int row = ft * kTileRows + lq * 32 + lane;
        in_doc = row < P.Ld;
        if (in_doc && dmt != MMB200_MASK_NONE) raw = mask_raw(P.d_mask, dmt, pair_dmask_row(P, fp) * (int64_t)P.Ld + row);
      }
      if (++ft == L.tiles) { ft = 0; ++fp; }
      return in_doc;
    };
    uint64_t raw0, raw1;
    bool in0 = fetch(raw0);
    bool in1 = fetch(raw1);
    for (int64_t p = p_begin; p < p_end; ++p) {
      const int64_t qi = pair_query(P, p);
      // query-mask words for this lane's columns: fetched now, tested after the pair's tiles
      uint64_t qraw[4];
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        const int col = c * 32 + lane;
        qraw[c] = (c < ncol32 && col < P.Lq) ? (qmt != MMB200_MASK_NONE ? mask_raw(P.q_mask, qmt, qi * (int64_t)P.Lq + col) : 1) : 0;
      }
      float colmax[4] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY};
      for (int t = 0; t < L.tiles; ++t) {
        const bool in_doc = in0;
        const uint64_t raw = raw0;
        in0 = in1;
        raw0 = raw1;
        in1 = fetch(raw1);
        mbar_wait(&S->accfull[acc], accphase);
        tc_fence_after_sync();
        const bool tok_ok = mask_test(raw, dmt);
        const uint32_t taddr = tmem_base + ((uint32_t)(lq * 32) << 16) + (uint32_t)(acc * L.npad);
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          if (c < ncol32) {
            uint32_t r[32];
            tmem_ld_32x32b_x32(taddr + c * 32, r);
            tmem_ld_wait();
            float v[32];
#pragma unroll
            for (int j = 0; j < 32; ++j) {
              v[j] = in_doc ? (tok_ok ? __uint_as_float(r[j]) : kMaskedScore) : -INFINITY;
            }
            colmax[c] = fmaxf(colmax[c], warp_transpose_max32(v, lane));
          }
        }
        tc_fence_before_sync();
        __syncwarp();
        if (lane == 0) mbar_arrive(&S->accempty[acc]);
        if (++acc == kAccStages) { acc = 0; accphase ^= 1u; }
      }
      const int buf = (int)((p - p_begin) & 1);
#pragma unroll
      for (int c = 0; c < 4; ++c)
        if (c < ncol32) S->colmax[buf][ew][c * 32 + lane] = colmax[c];
      named_bar_sync(1, 128);
      if (ew == (int)((p - p_begin) & 3)) {  // rotate the final reduction over the 4 warps
        float total = 0.f;
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          if (c < ncol32) {
            const int col = c * 32 + lane;
            float m = fmaxf(fmaxf(S->colmax[buf][0][col], S->colmax[buf][1][col]),
                            fmaxf(S->colmax[buf][2][col], S->colmax[buf][3][col]));
            total += mask_test(qraw[c], qmt) ? m : 0.f;
          }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) total += __shfl_xor_sync(0xffffffffu, total, o);
        if (lane == 0) P.out[p] = total;
      }
    }
  }

  tc_fence_before_sync();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after_sync();
    tmem_dealloc(tmem_base, (uint32_t)L.tmem_cols);
  }
}

// ---------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------
// Launch geometry of maxsim_tc_kernel; L.stages < 2 means the two query slots leave no room for a
// double-buffered document ring in shared memory.
static TcLaunch tc_plan(const MaxsimParams& P, int dtype, const DeviceInfo& dev, size_t* smem_bytes) {
  TcLaunch L;
  L.npad = ((P.Lq + 31) / 32) * 32;
  L.kblocks = P.dim / 64;
  L.kbs = (L.kblocks % 2 == 0) ? 2 : 1;
  L.tiles = (P.Ld + kTileRows - 1) / kTileRows;
  L.fmt = dtype == MMB200_F16 ? kFmtF16 : kFmtBF16;
  L.qslot_bytes = L.kblocks * L.npad * 128;
  int tc = kAccStages * L.npad;
  L.tmem_cols = 32;
  while (L.tmem_cols < tc) L.tmem_cols <<= 1;
  const int stage_bytes = L.kbs * kKBlockBytes;
  const int fixed = kQSlots * L.qslot_bytes + (int)sizeof(TcShared) + 1024 /* alignment slack */;
  const int budget = dev.max_smem_optin - fixed;
  L.stages = budget < 0 ? 0 : std::min(kMaxStages, budget / stage_bytes);
  *smem_bytes = (size_t)L.stages * stage_bytes + fixed;
  return L;
}

static bool tc_supported(const MaxsimParams& P, int dtype, const DeviceInfo& dev, std::string* why) {
  if (dtype != MMB200_F16 && dtype != MMB200_BF16) { *why = "tcgen05 path needs f16/bf16 inputs"; return false; }
  if (P.dim % 64 != 0 || P.dim < 64 || P.dim > 1024) { *why = "tcgen05 path needs dim % 64 == 0, 64 <= dim <= 1024"; return false; }
  if (P.Lq < 1 || P.Lq > 128) { *why = "tcgen05 path needs 1 <= Lq <= 128"; return false; }
  if (P.Ld < 1) { *why = "Ld < 1"; return false; }
  if (P.argmax) { *why = "argmax output is produced by the SIMT kernel"; return false; }
  if ((reinterpret_cast<uintptr_t>(P.q) | reinterpret_cast<uintptr_t>(P.d)) & 15) { *why = "q/d must be 16-byte aligned"; return false; }
  size_t smem_bytes;
  if (tc_plan(P, dtype, dev, &smem_bytes).stages < 2) {
    *why = "tcgen05 path: the query tile (2 x dim/64 x round32(Lq) x 128 B) leaves no room for two document stages in shared memory";
    return false;
  }
  return true;
}

// Only called for shapes that tc_supported() accepts.
static int launch_tc(const MaxsimParams& P, int dtype, const DeviceInfo& dev, cudaStream_t stream) {
  size_t smem_bytes;
  const TcLaunch L = tc_plan(P, dtype, dev, &smem_bytes);

  const CUtensorMapDataType tdt = dtype == MMB200_F16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16;
  CUtensorMap tq, td;
  {
    const uint64_t dims[4] = {64, (uint64_t)P.Lq, (uint64_t)L.kblocks, (uint64_t)P.n_q};
    const uint64_t strides[3] = {(uint64_t)P.dim * 2, 128, (uint64_t)P.Lq * P.dim * 2};
    const uint32_t box[4] = {64, (uint32_t)L.npad, (uint32_t)L.kblocks, 1};
    if (int rc = encode_tensor_map(&tq, tdt, 4, P.q, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_128B,
                                   CU_TENSOR_MAP_L2_PROMOTION_L2_128B))
      return rc;
  }
  {
    const uint64_t dims[4] = {64, (uint64_t)P.Ld, (uint64_t)L.kblocks, (uint64_t)P.n_d};
    const uint64_t strides[3] = {(uint64_t)P.dim * 2, 128, (uint64_t)P.Ld * P.dim * 2};
    const uint32_t box[4] = {64, (uint32_t)kTileRows, (uint32_t)L.kbs, 1};
    if (int rc = encode_tensor_map(&td, tdt, 4, P.d, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_128B,
                                   CU_TENSOR_MAP_L2_PROMOTION_L2_256B))
      return rc;
  }
  const int grid = (int)std::min<int64_t>(dev.sm_count, P.n_pairs);
  if (L.kbs == 2) {
    MMB_CHECK_CUDA(cudaFuncSetAttribute(maxsim_tc_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_bytes));
    maxsim_tc_kernel<2><<<grid, kTcThreads, smem_bytes, stream>>>(tq, td, P, L);
  } else {
    MMB_CHECK_CUDA(cudaFuncSetAttribute(maxsim_tc_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_bytes));
    maxsim_tc_kernel<1><<<grid, kTcThreads, smem_bytes, stream>>>(tq, td, P, L);
  }
  MMB_CHECK_CUDA(cudaGetLastError());
  return MMB200_OK;
}

static int launch_simt(const MaxsimParams& P, int dtype, const DeviceInfo& dev, cudaStream_t stream) {
  // shared memory: qrows staged query rows of dim+1 floats + the per-warp [4][Lq] max and argmax
  const size_t row_bytes = (size_t)(P.dim + 1) * sizeof(float), fixed = 8 * (size_t)P.Lq * sizeof(float);
  int qrows = P.Lq;
  if (fixed + (size_t)qrows * row_bytes > (size_t)dev.max_smem_optin)
    qrows = (int)(((size_t)dev.max_smem_optin - fixed) / row_bytes) / 32 * 32;
  MMB_REQUIRE(qrows >= 1, "SIMT max-sim: 32 query rows of this dim do not fit in shared memory");
  const size_t smem_bytes = fixed + (size_t)qrows * row_bytes;
  const int grid = (int)std::min<int64_t>((int64_t)dev.sm_count * 8, P.n_pairs);
#define MMB_LAUNCH_SIMT(T)                                                                                  \
  do {                                                                                                      \
    MMB_CHECK_CUDA(cudaFuncSetAttribute(maxsim_simt_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, \
                                        (int)smem_bytes));                                                  \
    maxsim_simt_kernel<T><<<grid, kSimtThreads, smem_bytes, stream>>>(P, qrows);                           \
  } while (0)
  if (dtype == MMB200_F16) MMB_LAUNCH_SIMT(__half);
  else if (dtype == MMB200_BF16) MMB_LAUNCH_SIMT(__nv_bfloat16);
  else MMB_LAUNCH_SIMT(float);
#undef MMB_LAUNCH_SIMT
  MMB_CHECK_CUDA(cudaGetLastError());
  return MMB200_OK;
}

int maxsim_fwd_device(const MaxsimParams& P, int dtype, int impl, cudaStream_t stream) {
  MMB_REQUIRE(P.q && P.d && P.out, "q, d, out must be non-null");
  MMB_REQUIRE(dtype_size(dtype) != 0, "unknown dtype");
  MMB_REQUIRE(P.n_pairs >= 0 && P.n_q > 0 && P.n_d > 0, "bad counts");
  MMB_REQUIRE(P.Lq > 0 && P.Ld > 0 && P.dim > 0, "bad shape");
  MMB_REQUIRE(P.Lq <= kMaxsimMaxLq && P.dim <= kMaxsimMaxDim, "max-sim supports 1 <= Lq <= 128 and 1 <= dim <= 1024");
  MMB_REQUIRE(P.docs_per_query >= 1, "docs_per_query must be >= 1");
  if ((P.q_mask || P.d_mask)) MMB_REQUIRE(mask_dtype_size(P.mask_dtype) != 0, "unknown mask dtype");
  if (!P.pair_q) MMB_REQUIRE((P.pair_base + P.n_pairs + P.docs_per_query - 1) / P.docs_per_query <= P.n_q, "n_pairs / docs_per_query exceeds n_q");
  if (!P.pair_d) MMB_REQUIRE(P.n_pairs <= P.n_d, "n_pairs exceeds n_d");
  if (P.n_pairs == 0) return MMB200_OK;
  DeviceInfo dev;
  if (int rc = current_device_info(&dev)) return rc;
  if (!is_sm100(dev)) {
    set_error("matchmaker_b200 kernels are built for sm_100a only; device is sm_" + std::to_string(dev.cc_major) +
              std::to_string(dev.cc_minor));
    return MMB200_ERR_UNSUPPORTED;
  }
  if (impl == MMB200_IMPL_TCGEN05_RAGGED) {
    // skip-padding variant: fetch only rows up to each document's last unmasked row
    MMB_REQUIRE(P.pair_dmask == nullptr, "ragged fetch is incompatible with pair_dmask");
    int32_t* rows = nullptr;
    MMB_CHECK_CUDA(cudaMallocAsync(reinterpret_cast<void**>(&rows), (size_t)P.n_d * sizeof(int32_t), stream));
    int rc = maxsim_rows_needed_launch(P.d_mask, P.mask_dtype, rows, P.n_d, P.Ld, stream);
    bool handled = false;
    if (rc == MMB200_OK) {
      MaxsimParams R = P;
      R.rows_needed = rows;
      rc = maxsim_qm_launch(R, dtype, dev, stream, &handled);
    }
    cudaFreeAsync(rows, stream);
    if (rc == MMB200_OK && !handled) { set_error("ragged max-sim: shape outside the queries-on-M kernel (Lq <= 32, dim 64/128, f16/bf16)"); rc = MMB200_ERR_UNSUPPORTED; }
    return rc;
  }
  if (impl == MMB200_IMPL_AUTO || impl == MMB200_IMPL_TCGEN05) {
    bool handled = false;
    const int rc = maxsim_qm_launch(P, dtype, dev, stream, &handled);
    if (handled || rc != MMB200_OK) return rc;
  }
  std::string why;
  const bool tc_ok = tc_supported(P, dtype, dev, &why);
  if ((impl == MMB200_IMPL_TCGEN05 || impl == MMB200_IMPL_TCGEN05_DOCM) && !tc_ok) {
    set_error(why);
    return MMB200_ERR_UNSUPPORTED;
  }
  if (impl == MMB200_IMPL_SIMT || !tc_ok) return launch_simt(P, dtype, dev, stream);
  return launch_tc(P, dtype, dev, stream);
}

}  // namespace mmb

extern "C" int mmb200_maxsim_fwd(const void* q, const void* d, const void* q_mask, const void* d_mask,
                                 const int32_t* pair_q, const int32_t* pair_d, const int32_t* pair_dmask,
                                 float* out, int32_t* argmax, int64_t n_q, int64_t n_d, int64_t n_pairs, int32_t docs_per_query, int32_t Lq,
                                 int32_t Ld, int32_t dim, int32_t dtype, int32_t mask_dtype, int32_t impl,
                                 void* stream) {
  mmb::MaxsimParams P;
  P.q = q; P.d = d; P.q_mask = q_mask; P.d_mask = d_mask; P.pair_q = pair_q; P.pair_d = pair_d; P.pair_dmask = pair_dmask; P.rows_needed = nullptr;
  P.out = out; P.argmax = argmax; P.n_q = n_q; P.n_d = n_d; P.n_pairs = n_pairs;
  P.pair_base = 0;
  P.docs_per_query = docs_per_query; P.Lq = Lq; P.Ld = Ld; P.dim = dim; P.mask_dtype = mask_dtype;
  return mmb::maxsim_fwd_device(P, dtype, impl, static_cast<cudaStream_t>(stream));
}
