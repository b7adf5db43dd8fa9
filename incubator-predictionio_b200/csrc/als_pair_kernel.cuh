// als_pair_kernel.cuh -- rank 33..64 half-step, second generation: every warp is an independent worker that
// accumulates the Gramians of TWO destination rows one after the other on the warp-level tensor-core path (mma.sync
// m16n8k16 FP16 with f32 accumulate, three passes hi*hi + lo*hi + hi*lo on an fp16 hi/lo split scaled by a power of two
// per 16-rating chunk = fp32-class products) and then solves both normal equations at once with the lockstep Cholesky
// of als_lockstep.cuh (16 lanes per matrix).
//
// Differences to the round-1 kernel (als_mma_kernel.cuh: four warps per CTA, one row each):
//   * no CTA-wide barrier: a warp stages its own sixteen gathered rows per chunk (cp.async, 2-deep ring, 72-float row
//     stride so that the fragment LDS.32 are conflict-free) and synchronises with __syncwarp only; warps of unrelated
//     rows no longer wait for each other;
//   * the right-hand side is accumulated from the fragment values (32 FMA per 16-rating chunk, quad-reduced once per
//     row) instead of a second pass over the staged rows;
//   * the solve costs ~1.8 k instead of ~6.4 k warp instructions per row and its 64-step pivot chain is shared by
//     the two matrices;
//   * work-list mode: an item may be a PART of a long row; its partial normal equation goes to global memory in the
//     slot layout and als_finish_pair_kernel adds the parts of a row in fixed order and solves.  Cutting rows above
//     1024 ratings into 512-rating parts is a two-level summation: the per-chunk round-to-nearest accumulation stays
//     short, which keeps the kernel inside the 1e-4 parity bound on rows of thousands of ratings (round 1: 1.1e-4).
// Per-row arithmetic depends on the row alone (sharded runs stay bit-identical).
//
// Replaces, per destination row: NormalEquation.add + CholeskySolver.solve of Spark 2.4 ml.recommendation.ALS
// (SURVEY.md section 8(c) items 5-6), reached from examples/scala-parallel-recommendation/.../ALSAlgorithm.scala:76-86.
#pragma once
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "als_kernels.cuh"
#include "als_lockstep.cuh"

namespace pio {
namespace pr {

constexpr int KP = 64;
constexpr int CH = 16;                    // ratings per chunk = K of one m16n8k16 mma
constexpr int RSTR = 72;                  // floats per staged source row (64 + 8 pad)
constexpr int NSTAGE = 2;
constexpr int STAGE = CH * RSTR;          // floats per stage
constexpr int NTILE = 20;                 // 16x8 accumulator tiles covering the lower triangle of 64x64
using LL = LsLayout<KP>;
constexpr int SLOT_STRIDE = LL::STRIDE;   // 2096 floats: the second matrix starts 16 banks further
constexpr int VSTR = 80;                  // per-matrix stride of the small vectors (== 16 mod 32)
constexpr int PART_FLOATS = LL::SIZE + KP;   // one partial normal equation in global memory: slot + right-hand side
// per-warp shared memory (floats): two slots, b of matrix 1, pivot lines, b of matrix 0, rating ring.  The staging ring
// starts at slot 1 and runs on into b of matrix 1 and the pivot lines: all three are dead while a row accumulates (b of
// the row is written after the ring dies, the solve comes after both rows); b of matrix 0 is live during the second row.
constexpr int W_BVEC1 = 2 * SLOT_STRIDE;
constexpr int W_COL = W_BVEC1 + VSTR;
constexpr int W_BVEC0 = W_COL + 2 * VSTR;
constexpr int W_MVAL = W_BVEC0 + VSTR;
constexpr int W_FLOATS = W_MVAL + NSTAGE * CH;
static_assert(SLOT_STRIDE + NSTAGE * STAGE <= W_BVEC0, "the staging ring must end before b of matrix 0");
static_assert((W_BVEC0 - W_BVEC1) % 32 == 16, "the b vectors of the two matrices start 16 banks apart");
constexpr size_t smem_bytes(int warps) { return sizeof(float) * (size_t)W_FLOATS * warps; }
__device__ __forceinline__ float* bvec_of(float* smem, int h) { return smem + (h ? W_BVEC1 : W_BVEC0); }

__device__ __forceinline__ void mma_f16(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile(
      "mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};\n"
      : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}

// First mma of a chain: C = 0 as an immediate (no registers to clear)
__device__ __forceinline__ void mma_f16_z(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile(
      "mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%10,%10,%10,%10};\n"
      : "=f"(d[0]), "=f"(d[1]), "=f"(d[2]), "=f"(d[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1), "f"(0.f));
}

// hi/lo split of two values into packed fp16 pairs: hi = v rounded to fp16, lo = (v - hi) rounded to fp16 (v - hi is
// exact in fp32).  |v - hi| <= 2^-11 |v|; the dropped lo*lo term is 2^-22.  Caller keeps |v| < 2^15 (no overflow).
__device__ __forceinline__ void split_f16x2(float a, float b, uint32_t& hi, uint32_t& lo) {
  const __half2 h = __floats2half2_rn(a, b);
  const float2 hf = __half22float2(h);
  const __half2 l = __floats2half2_rn(__fsub_rn(a, hf.x), __fsub_rn(b, hf.y));
  hi = *reinterpret_cast<const uint32_t*>(&h);
  lo = *reinterpret_cast<const uint32_t*>(&l);
}

// Accumulates sum c1 y y^T (lower triangle, slot layout) and b of ratings [beg, end) into `slot` / `bv`.
template <bool IMPLICIT>
__device__ __forceinline__ void accumulate_row(const SolveParams& p, long long beg, long long end, float* ring,
                                               float* mval, float* slot, float* bv) {
  const int lane = threadIdx.x & 31;
  const int g = lane >> 2, t = lane & 3;
  const int nchunks = (int)((end - beg + CH - 1) / CH);
  const int prow = lane >> 4, psl = lane & 15;     // staging: piece j of this lane = (staged row 2 j + prow, 16-byte slot psl)

  // metadata of rating (lane & 15) of a chunk; the staging takes the index of each of its rows from the owning lane
  int nidx;
  float nval;
  auto prefetch_meta = [&](int c) {
    const long long e = beg + (long long)c * CH + (lane & (CH - 1));
    const bool in = c < nchunks && e < end;
    nidx = in ? __ldg(p.idx + e) : -1;
    nval = in ? __ldg(p.val + e) : 0.f;
  };
  auto issue = [&](int c) {   // uses the metadata prefetched for chunk c; rows past the end are zero-filled
    if (c < nchunks) {
      float* sbuf = ring + (c % NSTAGE) * STAGE;
#pragma unroll
      for (int j = 0; j < CH / 2; ++j) {
        const int src = __shfl_sync(0xffffffffu, nidx, 2 * j + prow);
        float4* d4 = reinterpret_cast<float4*>(sbuf + (2 * j + prow) * RSTR + psl * 4);
        if (src >= 0) cp_async16(d4, p.src + (size_t)src * KP + psl * 4);
        else *d4 = make_float4(0.f, 0.f, 0.f, 0.f);
      }
      if (lane < CH) mval[(c % NSTAGE) * CH + lane] = nval;
    }
    cp_async_commit();
  };

  float acc[NTILE][4];
#pragma unroll
  for (int i = 0; i < NTILE; ++i)
#pragma unroll
    for (int e = 0; e < 4; ++e) acc[i][e] = 0.f;
  float pb[4][2];             // right-hand side partials: columns 16 i + 8 h + g over the ratings t + 4 q of the chunks
#pragma unroll
  for (int i = 0; i < 4; ++i) pb[i][0] = pb[i][1] = 0.f;

  prefetch_meta(0);
  issue(0);
  prefetch_meta(1);

#pragma unroll 1
  for (int c = 0; c < nchunks; ++c) {
    cp_async_wait<0>();
    __syncwarp();
    issue(c + 1);
    prefetch_meta(c + 2);
    const float* X = ring + (c % NSTAGE) * STAGE;
    const float* mv = mval + (c % NSTAGE) * CH;
    // This lane's ratings are the staged rows t + 4 q, q = 0..3.  Fragment k index 2 t + q holds row t + 4 q for q < 2
    // and k = 2 t + 8 + (q - 2) holds row t + 4 q for q >= 2: the four rows of a lane quad lie 8 banks apart at the
    // 72-float stride (conflict-free LDS); the sum over k does not care which rating sits in which k slot.
    float sc[4], wb[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const float r = mv[t + 4 * q];
      sc[q] = 1.f;
      wb[q] = r;
      if (IMPLICIT) {
        const float c1 = p.alpha * fabsf(r);
        sc[q] = sqrtf(c1);
        wb[q] = r > 0.f ? 1.f + c1 : 0.f;
      }
    }
    // y[i][q][h] = X[t + 4 q][16 i + 8 h + g]; the right-hand side takes the unscaled values
    float y[4][4][2];
    float rmax[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int q = 0; q < 4; ++q)
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          y[i][q][h] = X[(t + 4 * q) * RSTR + 16 * i + 8 * h + g];
          pb[i][h] = fmaf(wb[q], y[i][q][h], pb[i][h]);
          rmax[q] = fmaxf(rmax[q], fabsf(y[i][q][h]));
        }
    // Chunk scale 2^e from the largest |sqrt(c1) y| of the chunk (rounding is monotonic, so max|y| * sqrt(c1) is that
    // value exactly): the scaled maximum lies in [2^14, 2^15), below the fp16 maximum, and lo stays a normal fp16
    // number down to 2^-18 of it.  e depends on the chunk's own data only; |e| <= 63 keeps 2^-2e a normal float.
    float mx = 0.f;
#pragma unroll
    for (int q = 0; q < 4; ++q) mx = fmaxf(mx, IMPLICIT ? rmax[q] * sc[q] : rmax[q]);
    const unsigned mb = __reduce_max_sync(0xffffffffu, __float_as_uint(mx));   // mx >= 0: the bit patterns order alike
    int e = mb ? 141 - (int)(mb >> 23) : 0;                                     // 141 = 127 + 14
    e = min(max(e, -63), 63);
    const float s = __int_as_float((127 + e) << 23), s2 = __int_as_float((127 - 2 * e) << 23);
    // fragments of m-tile i: reg h + 2 kk packs the rows q = 2 kk, 2 kk + 1 of column 16 i + 8 h + g.  The same
    // registers are the A fragment of m-tile i and the B fragments of n-tiles 2i ({0, 2}) and 2i+1 ({1, 3}).
    uint32_t hi[4][4], lo[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int h = 0; h < 2; ++h)
#pragma unroll
        for (int kk = 0; kk < 2; ++kk) {
          const int q0 = 2 * kk, q1 = 2 * kk + 1;
          split_f16x2(y[i][q0][h] * (IMPLICIT ? sc[q0] * s : s), y[i][q1][h] * (IMPLICIT ? sc[q1] * s : s),
                      hi[i][h + 2 * kk], lo[i][h + 2 * kk]);
        }
    // D(16i.., 8j..) += A_i B_j for the tiles on or below the diagonal: j <= 2i+1.  The tensor core adds with
    // truncation: only the 48 products of one chunk are summed inside it (small terms first), the running sum over
    // the chunks is a round-to-nearest FFMA in registers that also undoes the chunk scale (exactly: a power of two).
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int bi = j >> 1, be = j & 1;
#pragma unroll
      for (int i = bi; i < 4; ++i) {
        const int tile = i * (i + 1) + j;               // tiles of m-tile i start at sum_{i' < i} (2 i' + 2) = i (i + 1)
        float d[4];
        mma_f16_z(d, lo[i], hi[bi][be], hi[bi][be + 2]);
        mma_f16(d, hi[i], lo[bi][be], lo[bi][be + 2]);
        mma_f16(d, hi[i], hi[bi][be], hi[bi][be + 2]);
#pragma unroll
        for (int q = 0; q < 4; ++q) acc[tile][q] = fmaf(d[q], s2, acc[tile][q]);
      }
    }
  }
  cp_async_wait<0>();
  __syncwarp();   // the ring is dead from here on
  // ---- right-hand side: reduce over the four lanes of a quad (fixed order), lane t == 0 stores -------------------------
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int e = 0; e < 2; ++e) {
      float v = pb[i][e];
      v += __shfl_xor_sync(0xffffffffu, v, 1);
      v += __shfl_xor_sync(0xffffffffu, v, 2);
      if (t == 0) bv[16 * i + 8 * e + g] = v;
    }
  // ---- accumulators -> slot layout ----------------------------------------------------------------------------------------
  {
    int tile = 0;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
#pragma unroll
      for (int j = 0; j <= 2 * i + 1; ++j, ++tile) {
        const int cb = j >> 1;
        const int cc = 8 * (j & 1) + 2 * t;           // column inside the 16-wide block (even)
        if (cb < i) {
          // off-diagonal block: two 8-byte stores (rows g and g + 8 of the block)
          *reinterpret_cast<float2*>(slot + LL::offd(i, cb, g, cc)) = make_float2(acc[tile][0], acc[tile][1]);
          *reinterpret_cast<float2*>(slot + LL::offd(i, cb, g + 8, cc)) = make_float2(acc[tile][2], acc[tile][3]);
        } else {
          // diagonal block: packed triangle, keep c <= r
          if (cc <= g) slot[LL::diag(i, g, cc)] = acc[tile][0];
          if (cc + 1 <= g) slot[LL::diag(i, g, cc + 1)] = acc[tile][1];
          if (cc <= g + 8) slot[LL::diag(i, g + 8, cc)] = acc[tile][2];
          if (cc + 1 <= g + 8) slot[LL::diag(i, g + 8, cc + 1)] = acc[tile][3];
        }
      }
    }
  }
  __syncwarp();
}

// identity system for the unused half of the last warp
__device__ __forceinline__ void fill_identity(float* slot, float* bv) {
  const int lane = threadIdx.x & 31;
  for (int o = lane; o < LL::SIZE; o += 32) slot[o] = 0.f;
  __syncwarp();
  for (int r = lane; r < KP; r += 32) {
    slot[LL::at(r, r)] = 1.f;
    bv[r] = 0.f;
  }
  __syncwarp();
}

// WARPS independent workers per CTA.  The only CTA-wide synchronisation is one barrier before the solve: the warps of
// a CTA then walk the (fully unrolled, ~80 KB) lockstep solver together, so that an SM's instruction cache holds a few
// positions of that code instead of twelve (ncu, one-warp CTAs: "no instruction" was the first stall reason of the
// user half-step, 1.7 per issued instruction).
template <bool IMPLICIT, int WARPS>
__global__ void __launch_bounds__(32 * WARPS, 12 / WARPS) als_solve_pair_kernel(const SolveParams p, int n_items) {
  extern __shared__ __align__(16) float smem_all[];
  const int warp = threadIdx.x >> 5;
  float* smem = smem_all + warp * W_FLOATS;
  float* slot0 = smem;
  float* slot1 = smem + SLOT_STRIDE;
  float* ring = slot1;                  // dead whenever slot 1 is written
  float* colbuf = smem + W_COL;         // [2][VSTR]
  float* mval = smem + W_MVAL;          // [NSTAGE][CH]
  const int lane = threadIdx.x & 31;
  const int grp = lane >> 4;
  const int npairs = (n_items + 1) >> 1;

#pragma unroll 1
  for (int base = blockIdx.x * WARPS; base < npairs; base += gridDim.x * WARPS) {
    const int pair = base + warp;
    int row0 = -1, row1 = -1;
    if (pair < npairs) {
#pragma unroll 1
      for (int h = 0; h < 2; ++h) {
        const int item = 2 * pair + h;
        float* slot = h ? slot1 : slot0;
        float* bv = bvec_of(smem, h);
        if (item >= n_items) {
          fill_identity(slot, bv);
          continue;
        }
        long long beg, end;
        if (p.partial) {
          beg = p.wl_beg[item];
          end = p.wl_end[item];
        } else {
          const int r = p.row_begin + item;
          beg = p.ptr[r];
          end = p.ptr[r + 1];
          if (h) row1 = r;
          else row0 = r;
        }
        accumulate_row<IMPLICIT>(p, beg, end, ring, mval, slot, bv);
        if (p.partial) {
          // part of a long row: emit the partial normal equation (slot layout + b); als_finish_pair_kernel sums and solves
          float* out = p.partial + (size_t)item * PART_FLOATS;
          for (int o = lane; o < LL::SIZE / 4; o += 32)
            reinterpret_cast<float4*>(out)[o] = reinterpret_cast<const float4*>(slot)[o];
          for (int o = lane; o < KP; o += 32) out[LL::SIZE + o] = bv[o];
          __syncwarp();
        }
      }
    }
    if (p.partial) continue;
    if (WARPS > 1) __syncthreads();
    if (pair < npairs) {
      const int myrow = grp ? row1 : row0;
      const int rr = myrow < 0 ? p.row_begin : myrow;
      chol_lockstep<KP, IMPLICIT>(grp ? slot1 : slot0, bvec_of(smem, grp), p.yty, p.lambda * p.nreg[rr], p.k,
                                  colbuf + grp * VSTR, p.dst + (size_t)(p.dst_row_offset + rr) * KP, myrow >= 0, p.fail);
      __syncwarp();
    }
  }
}

// Finish kernel for rows that were cut into parts: one warp per two rows; fixed-order sum of the partial normal
// equations (float4 lanes over the slot), then the lockstep solve.
template <bool IMPLICIT>
__global__ void __launch_bounds__(32, 12) als_finish_pair_kernel(const SolveParams p, const int* __restrict__ row_part_ptr,
                                                                  int n_rows) {
  extern __shared__ __align__(16) float smem[];
  float* colbuf = smem + W_COL;
  const int lane = threadIdx.x & 31;
  const int grp = lane >> 4;
  const int npairs = (n_rows + 1) >> 1;
#pragma unroll 1
  for (int pair = blockIdx.x; pair < npairs; pair += gridDim.x) {
#pragma unroll 1
    for (int h = 0; h < 2; ++h) {
      const int r = 2 * pair + h;
      float* slot = smem + h * SLOT_STRIDE;
      float* bv = bvec_of(smem, h);
      if (r >= n_rows) {
        fill_identity(slot, bv);
        continue;
      }
      const int p0 = row_part_ptr[r], p1 = row_part_ptr[r + 1];
      for (int o = lane; o < PART_FLOATS / 4; o += 32) {
        float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
        for (int q = p0; q < p1; ++q) {
          const float4 v = __ldg(reinterpret_cast<const float4*>(p.partial + (size_t)q * PART_FLOATS) + o);
          s.x += v.x; s.y += v.y; s.z += v.z; s.w += v.w;
        }
        if (o < LL::SIZE / 4) reinterpret_cast<float4*>(slot)[o] = s;
        else reinterpret_cast<float4*>(bv)[o - LL::SIZE / 4] = s;
      }
      __syncwarp();
    }
    const int myrow = 2 * pair + grp;
    const bool valid = myrow < n_rows;
    const int rr = valid ? myrow : 0;
    chol_lockstep<KP, IMPLICIT>(smem + grp * SLOT_STRIDE, bvec_of(smem, grp), p.yty, p.lambda * p.nreg[rr], p.k,
                                colbuf + grp * VSTR, p.dst + (size_t)(p.dst_row_offset + rr) * KP, valid, p.fail);
    __syncwarp();
  }
}

}  // namespace pr
}  // namespace pio
