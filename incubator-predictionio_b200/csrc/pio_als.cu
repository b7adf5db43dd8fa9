// pio_als.cu -- C-ABI implementation (see include/pio_als.h for the reference interfaces each
// entry point replaces).  Host orchestration only; all arithmetic is in the CUDA kernels of
// als_kernels.cuh / sort_scan.cuh / topk.cuh.  No CPU fallback: without a usable sm_100 device
// every computing entry point returns PIO_ALS_ERR_CUDA.
#include "../../include/pio_als.h"

#include <cuda_runtime.h>
#include <dlfcn.h>
#include <math.h>
#include <nccl.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <chrono>
#include <deque>
#include <exception>
#include <mutex>
#include <string>
#include <vector>

#include "als_kernels.cuh"
#include "als_mma_kernel.cuh"
#include "als_pair_kernel.cuh"
// the tcgen05 half-step kernel; the header is parametrised by the role partition of its sixteen warps.  Measured at C2:
// 2 gather + 5 converter warps + 2 solve teams (below) beats 1 + 2 + 3 teams on long rows AND on short rows (user side
// 38 ms vs 86 ms: two converter warps cannot feed the MMAs), so only this partition is instantiated.
#define TC_NS tc
#define TC_NTEAM 2
#define TC_NCONV 5
#define TC_NGATHER 2
#define TC_NSTAGE 7
#define TC_NRAW 7
#include "als_tc_kernel.cuh"
#undef TC_NS
#undef TC_NTEAM
#undef TC_NCONV
#undef TC_NGATHER
#undef TC_NSTAGE
#undef TC_NRAW
#include "sort_scan.cuh"
#include "topk.cuh"
#include "ids_encode.cuh"
#include "cooc.cuh"

namespace pio {

constexpr int HEAVY_T = 4096;     // rows with more ratings than this are cut into parts (als_finish_kernel solves them)
constexpr int HEAVY_T_TC = 8192;  // same threshold when the tensor-core path handles the shorter rows
constexpr int TC_TILE_ROWS = 1 << 20;  // split mode: rows whose normal equations are buffered at once (9.1 KB per row)
constexpr int PART = 2016;        // ratings per part (multiple of every CH and of the tensor-core stage size 24)
constexpr int PAIR_SEG_T = 1024;  // pair kernel (als_pair_kernel.cuh): rows with more ratings than this are cut into parts ...
constexpr int PAIR_PART = 512;    // ... of this many ratings: two-level summation keeps long rows inside the parity bound

static thread_local std::string g_create_error;

static int ceil_log2(uint64_t n) {
  int b = 0;
  while (b < 63 && (1ull << b) < n) ++b;
  return b < 1 ? 1 : b;
}
static int pad_rank(int k) { return k <= 16 ? 16 : k <= 32 ? 32 : k <= 64 ? 64 : 128; }

// ---------------------------------------------------------------------------------------------
// NCCL through dlopen: the library has no link-time NCCL dependency and shares whichever libnccl
// the host process already loaded (torch's bundled one under torchrun, the system one under a JVM).
// ---------------------------------------------------------------------------------------------
struct NcclApi {
  void* lib = nullptr;
  ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
  ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
  ncclResult_t (*AllGather)(const void*, void*, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*AllReduce)(const void*, void*, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*Send)(const void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*Recv)(void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*GroupStart)() = nullptr;
  ncclResult_t (*GroupEnd)() = nullptr;
  ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
  const char* (*GetErrorString)(ncclResult_t) = nullptr;
  bool ok = false;
};
static NcclApi& nccl_api() {
  static NcclApi api;
  static std::once_flag once;
  std::call_once(once, [] {
    void* lib = dlopen("libnccl.so.2", RTLD_NOW | RTLD_NOLOAD | RTLD_GLOBAL);
    if (!lib) lib = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
    if (!lib) lib = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
    if (!lib) return;
    api.lib = lib;
    api.GetUniqueId = (decltype(api.GetUniqueId))dlsym(lib, "ncclGetUniqueId");
    api.CommInitRank = (decltype(api.CommInitRank))dlsym(lib, "ncclCommInitRank");
    api.AllGather = (decltype(api.AllGather))dlsym(lib, "ncclAllGather");
    api.AllReduce = (decltype(api.AllReduce))dlsym(lib, "ncclAllReduce");
    api.Send = (decltype(api.Send))dlsym(lib, "ncclSend");
    api.Recv = (decltype(api.Recv))dlsym(lib, "ncclRecv");
    api.GroupStart = (decltype(api.GroupStart))dlsym(lib, "ncclGroupStart");
    api.GroupEnd = (decltype(api.GroupEnd))dlsym(lib, "ncclGroupEnd");
    api.CommDestroy = (decltype(api.CommDestroy))dlsym(lib, "ncclCommDestroy");
    api.GetErrorString = (decltype(api.GetErrorString))dlsym(lib, "ncclGetErrorString");
    api.ok = api.GetUniqueId && api.CommInitRank && api.AllGather && api.CommDestroy && api.AllReduce && api.Send &&
             api.Recv && api.GroupStart && api.GroupEnd;
  });
  return api;
}

// ---------------------------------------------------------------------------------------------
// small kernels of the ingest / model plumbing
// ---------------------------------------------------------------------------------------------
__global__ void validate_coo_kernel(const int* u, const int* i, long long n, int nu, int ni, int* bad) {
  const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (e < n && (u[e] < 0 || u[e] >= nu || i[e] < 0 || i[e] >= ni)) atomicAdd(bad, 1);
}
__global__ void make_keys_ext_kernel(const int* u, const int* i, long long n, int bits_i, uint64_t* keys,
                                     uint32_t* pay) {
  const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (e < n) {
    keys[e] = ((uint64_t)(uint32_t)u[e] << bits_i) | (uint64_t)(uint32_t)i[e];
    pay[e] = (uint32_t)e;
  }
}
__global__ void head_flags_kernel(const uint64_t* keys, long long n, uint32_t* flag) {
  const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (e < n) flag[e] = (e == 0 || keys[e] != keys[e - 1]) ? 1u : 0u;
}
// one thread per run head: fold the run in event order (sum) or pick the latest event (keep-last)
__global__ void dedup_compact_kernel(const uint64_t* keys, const uint32_t* pay, const uint32_t* pos,
                                     long long n, int bits_i, const float* rating, const long long* ts,
                                     int mode, int* ou, int* oi, float* orr) {
  const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= n) return;
  const uint64_t key = keys[e];
  if (e > 0 && keys[e - 1] == key) return;
  float acc;
  if (mode == PIO_ALS_DEDUP_SUM) {
    acc = 0.f;
    for (long long t = e; t < n && keys[t] == key; ++t) acc += rating[pay[t]];
  } else {
    long long best_t = ts ? ts[pay[e]] : 0;
    uint32_t best_p = pay[e];
    for (long long t = e + 1; t < n && keys[t] == key; ++t) {
      const uint32_t pp = pay[t];
      const long long tt = ts ? ts[pp] : 0;
      if (tt >= best_t) { best_t = tt; best_p = pp; }  // payload order == event order (stable sort)
    }
    acc = rating[best_p];
  }
  const uint32_t o = pos[e];
  ou[o] = (int)(key >> bits_i);
  oi[o] = (int)(key & ((1ull << bits_i) - 1ull));
  orr[o] = acc;
}
__global__ void degree_kernel(const int* u, const int* i, const float* r, long long n, uint32_t* du,
                              uint32_t* di, uint32_t* pu, uint32_t* pi) {
  const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= n) return;
  atomicAdd(&du[u[e]], 1u);
  atomicAdd(&di[i[e]], 1u);
  if (r[e] > 0.f) {
    atomicAdd(&pu[u[e]], 1u);
    atomicAdd(&pi[i[e]], 1u);
  }
}
__global__ void degree_keys_kernel(const uint32_t* deg, int n, uint64_t* keys, uint32_t* pay) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r < n) {
    keys[r] = (uint64_t)(0xFFFFFFFFu - deg[r]);
    pay[r] = (uint32_t)r;
  }
}
// sorted position p -> internal id: rows are dealt to ranks in snake order so every rank gets
// the same number of rows and a near-equal share of the ratings; a rank's rows stay
// degree-descending.
__global__ void assign_internal_kernel(const uint32_t* order, int n, int W, int R, int* perm, int* inv, int* rpos,
                                       int* p2i) {
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= n) return;
  const int row = (int)order[p];
  const int blk = p / W, pos = p % W;
  const int rk = (blk & 1) ? (W - 1 - pos) : pos;
  const int internal = rk * R + blk;
  perm[row] = internal;
  inv[internal] = row;
  rpos[row] = p;       // degree-rank position: independent of the number of GPUs
  p2i[p] = internal;
}
// sharded ingest: destination rank of every event (by user residue for the dedup pass, by row owner for the CSR passes)
__global__ void dest_mod_kernel(const int* u, long long n, int W, uint64_t* keys, uint32_t* pay) {
  const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (e < n) {
    keys[e] = (uint64_t)((uint32_t)u[e] % (uint32_t)W);
    pay[e] = (uint32_t)e;
  }
}
__global__ void dest_owner_kernel(const int* rowext, long long n, const int* perm, int R, uint64_t* keys, uint32_t* pay) {
  const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (e < n) {
    keys[e] = (uint64_t)(perm[rowext[e]] / R);
    pay[e] = (uint32_t)e;
  }
}
template <class T>
__global__ void gather_by_index_kernel(const T* in, const uint32_t* idx, long long n, T* out) {
  const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (e < n) out[e] = in[idx[e]];
}
__global__ void fill_int_kernel(int* a, long long n, int v) {
  const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (e < n) a[e] = v;
}
// key = (internal row, degree-rank position of the column): inside a row the ratings are ordered by a
// quantity that does not depend on the sharding, so the fp32 summation order -- and hence every bit of the
// result -- is the same on 1, 2, 4 or 8 GPUs.
__global__ void make_keys_int_kernel(const int* rowext, const int* colext, long long n, const int* perm_row,
                                     const int* rpos_col, int bits_col, uint64_t* keys, uint32_t* pay) {
  const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (e < n) {
    keys[e] = ((uint64_t)(uint32_t)perm_row[rowext[e]] << bits_col) | (uint64_t)(uint32_t)rpos_col[colext[e]];
    pay[e] = (uint32_t)e;
  }
}
__global__ void build_ptr_kernel(const uint64_t* keys, long long n, int bits_col, int n_rows, long long* ptr) {
  const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= n) return;
  const int r = (int)(keys[e] >> bits_col);
  const int rp = e == 0 ? -1 : (int)(keys[e - 1] >> bits_col);
  for (int rr = rp + 1; rr <= r; ++rr) ptr[rr] = e;
  if (e == n - 1)
    for (int rr = r + 1; rr <= n_rows; ++rr) ptr[rr] = n;
}
__global__ void extract_csr_kernel(const uint64_t* keys, const uint32_t* pay, const float* rating, long long b,
                                   long long cnt, int bits_col, const int* p2i_col, int* idx, float* val) {
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= cnt) return;
  idx[t] = p2i_col[(int)(keys[b + t] & ((1ull << bits_col) - 1ull))];
  val[t] = rating[pay[b + t]];
}
__global__ void local_rows_kernel(const long long* ptr_full, int row0, int R, long long base, const int* inv,
                                  const uint32_t* deg, const uint32_t* npos, int implicit, long long* ptr,
                                  float* nreg, int* counts /* [0]=active [1]=heavy */, int heavy_t) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r > R) return;
  ptr[r] = ptr_full[row0 + r] - base;
  if (r == R) return;
  const int ext = inv[row0 + r];
  float nr = 0.f;
  if (ext >= 0) {
    const uint32_t d = deg[ext];
    nr = implicit ? (float)npos[ext] : (float)d;
    if (d > 0) atomicAdd(&counts[0], 1);
    if (d > (uint32_t)heavy_t) atomicAdd(&counts[1], 1);
  }
  nreg[r] = nr;
}
__global__ void scatter_init_kernel(const float* ext_f, int n, int k, int kp, const int* perm, const uint32_t* deg,
                                    float* F) {
  const long long o = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (o >= (long long)n * kp) return;
  const int r = (int)(o / kp), c = (int)(o % kp);
  float v = 0.f;
  if (c < k && deg[r] > 0) v = ext_f[(size_t)r * k + c];
  F[(size_t)perm[r] * kp + c] = v;
}
__device__ __forceinline__ uint64_t splitmix64_dev(uint64_t x) {
  x += 0x9E3779B97F4A7C15ull;
  uint64_t z = x;
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  return z ^ (z >> 31);
}
// unit-norm Gaussian rows from the counter hash (mirrors synth.py synth_init_factors)
__global__ void hash_init_kernel(int n, int k, int kp, uint64_t seed, int side, const int* perm,
                                 const uint32_t* deg, float* F) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= n) return;
  float* row = F + (size_t)perm[r] * kp;
  if (deg[r] == 0) {
    for (int c = 0; c < kp; ++c) row[c] = 0.f;
    return;
  }
  const uint64_t s = seed ^ 0xA5A5A5A55A5A5A5Aull;
  double nrm = 0.0;
  for (int c = 0; c < k; ++c) {
    const uint64_t ctr = ((uint64_t)r * (uint64_t)k + (uint64_t)c) * 2ull + ((uint64_t)side << 62);
    const uint64_t h1 = splitmix64_dev(s ^ ctr), h2 = splitmix64_dev(s ^ (ctr + 1ull));
    const double u1 = ((double)(h1 >> 11) + 1.0) * (1.0 / 9007199254740992.0);
    const double u2 = (double)(h2 >> 11) * (1.0 / 9007199254740992.0);
    const float g = (float)(sqrt(-2.0 * log(u1)) * cos(2.0 * 3.14159265358979323846 * u2));
    row[c] = g;
    nrm += (double)g * (double)g;
  }
  float nf = (float)sqrt(nrm);
  if (nf == 0.f) nf = 1.f;
  for (int c = 0; c < k; ++c) row[c] = row[c] / nf;
  for (int c = k; c < kp; ++c) row[c] = 0.f;
}
__global__ void gather_factors_kernel(const float* F, int n, int k, int kp, const int* perm, float* out) {
  const long long o = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (o >= (long long)n * k) return;
  const int r = (int)(o / k), c = (int)(o % k);
  out[o] = F[(size_t)perm[r] * kp + c];
}
__global__ void has_kernel(const uint32_t* deg, int n, uint8_t* has) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r < n) has[r] = deg[r] > 0 ? 1 : 0;
}
// internal row -> external id if the row owns a factor, else -1 (candidate table for top-k)
__global__ void cand_ext_kernel(const int* inv, const uint32_t* deg, int n_internal, int* out) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= n_internal) return;
  const int ext = inv[r];
  out[r] = (ext >= 0 && deg[ext] > 0) ? ext : -1;
}
__global__ void gather_rows_kernel(const float* F, int kp, const int* rows_ext, int n, const int* perm,
                                   const uint32_t* deg, int n_ext, float* out, uint8_t* valid) {
  const int q = blockIdx.x;
  const int r = rows_ext[q];
  const bool ok = r >= 0 && r < n_ext && deg[r] > 0;
  for (int c = threadIdx.x; c < kp; c += blockDim.x) out[(size_t)q * kp + c] = ok ? F[(size_t)perm[r] * kp + c] : 0.f;
  if (threadIdx.x == 0 && valid) valid[q] = ok ? 1 : 0;
  (void)n;
}
// low-latency serving: the (few) row ids travel in the kernel parameters, no host-to-device copy
struct IdList {
  int v[40];
};
__global__ void gather_rows_ids_kernel(const float* F, int kp, IdList ids, const int* perm, const uint32_t* deg, int n_ext,
                                       float* out, uint8_t* valid) {
  const int q = blockIdx.x;
  const int r = ids.v[q];
  const bool ok = r >= 0 && r < n_ext && deg[r] > 0;
  for (int c = threadIdx.x; c < kp; c += blockDim.x) out[(size_t)q * kp + c] = ok ? F[(size_t)perm[r] * kp + c] : 0.f;
  if (threadIdx.x == 0 && valid) valid[q] = ok ? 1 : 0;
}
__global__ void copy_rows_kernel(const float* src, int kp, const int* rows, float* out) {
  const int v = blockIdx.x;
  for (int c = threadIdx.x; c < kp; c += blockDim.x) out[(size_t)v * kp + c] = src[(size_t)rows[v] * kp + c];
}
__global__ void synth_kernel(int nu, int ni, long long n, uint64_t seed, int implicit, long long start, int* u,
                             int* it, float* r) {
  const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= n) return;
  const uint64_t base = (uint64_t)(start + e) * 4ull;
  const uint64_t h1 = splitmix64_dev(seed ^ (base + 1ull));
  const uint64_t h2 = splitmix64_dev(seed ^ (base + 2ull));
  const uint64_t h3 = splitmix64_dev(seed ^ (base + 3ull));
  u[e] = (int)(h1 % (uint64_t)nu);
  const double uu = (double)(h2 >> 11) * (1.0 / 9007199254740992.0);
  long long item = (long long)floor(__dmul_rn(__dmul_rn((double)ni, uu), uu));
  if (item > ni - 1) item = ni - 1;
  it[e] = (int)item;
  if (implicit) {
    int tz = h3 == 0 ? 64 : __ffsll((long long)h3) - 1;
    if (tz > 9) tz = 9;
    r[e] = (float)(1 + tz);
  } else {
    r[e] = (float)(1 + (int)(h3 % 5ull));
  }
}

// ---------------------------------------------------------------------------------------------
// handle
// ---------------------------------------------------------------------------------------------
struct Side {
  int n = 0;           // external rows
  int R = 0;           // rows owned per rank
  int n_internal = 0;  // world * R
  int bits = 1;        // bits of an internal id
  int* perm = nullptr;       // [n] external row -> internal id
  int* inv = nullptr;        // [n_internal]
  int* rpos = nullptr;       // [n] external row -> degree-rank position
  int* p2i = nullptr;        // [n] degree-rank position -> internal id
  uint32_t* deg = nullptr;   // [n]
  uint32_t* npos = nullptr;  // [n]
  long long* ptr = nullptr;  // [R+1]
  int* idx = nullptr;
  float* val = nullptr;
  long long nnz_local = 0;
  float* nreg = nullptr;     // [R]
  float* F = nullptr;        // [n_internal][KP]
  int* cand_ext = nullptr;   // [n_internal]
  int n_active = 0, n_heavy = 0;
  bool use_tc = false;       // this side's short rows go through the tensor-core kernel (decided from GLOBAL counts: every rank agrees)
  int heavy_t = 0;           // rows with more ratings than this are cut into parts
  int part_len = 0;          // ratings per part
  bool use_pair = false;     // rows and parts of this side run on the pair kernel (rank 33..64, mma.sync + lockstep solve)
  // parts of the n_heavy longest local rows
  long long* part_beg = nullptr;
  long long* part_end = nullptr;
  int* row_part_ptr = nullptr;   // [n_heavy + 1]
  float* partial = nullptr;      // [n_parts][SLOT + KP]
  int n_parts = 0;
  std::vector<int> h_row_part_ptr;   // host copy (rank 65..128 walks its rows in tiles)
};

enum EvKind { EV_SOLVE = 0, EV_GRAM = 1, EV_COMM = 2, EV_SOLVE_USER = 3, EV_NKIND = 4 };   // EV_SOLVE = item half-step
struct EvPair {
  cudaEvent_t a, b;
  int kind;
};

}  // namespace pio

using namespace pio;

struct pio_als_handle {
  pio_als_config cfg;
  int KP = 0;
  cudaStream_t stream = nullptr;
  Side U, I;
  float* yty = nullptr;
  double* gram_partial = nullptr;
  double* gram_gsum = nullptr;   // [GRAM_GROUPS][KP*KP] class sums of the YtY partials (slot order, GramMap)
  const Side* gram_side = nullptr;   // the side whose YtY currently sits in `yty` (nullptr: none / stale)
  cudaEvent_t ev_gram = nullptr;
  int gram_blocks = 0;
  int* d_fail = nullptr;
  int* d_counts = nullptr;
  long long* d_timing = nullptr;  // PIO_ALS_TC_TIMING=1: per-warp cycle counters of the last tensor-core launch
  float* d_dbg = nullptr;     // PIO_ALS_TC_DEBUG=1: A/b dump of the last tensor-core half-step
  size_t dbg_rows = 0;
  bool use_tc = false;        // rank in 33..64 and PIO_ALS_TC != 0
  bool use_mma = true;        // PIO_ALS_MMA=0: FP32 kernel instead of the mma.sync kernels for rank 33..64
  bool use_pair = true;       // PIO_ALS_MMA=1: round-1 one-warp-per-row mma.sync kernel instead of the pair kernel
  int pair_seg_t = PAIR_SEG_T, pair_part = PAIR_PART;   // PIO_ALS_SEG_T / PIO_ALS_PART
  int pair_warps = 4;         // PIO_ALS_PAIR_WARPS: warps per CTA of the pair kernel (1, 2, 4, 6 or 12)
  // half-step pipeline (pair-kernel sides): long rows (parts + finish) run on `aux` next to the whole rows on `stream`;
  // the destination rows are cut into n_pieces local ranges and the all-gather of a finished range runs on `comm_st`
  // while the next range is solved (world_size > 1)
  cudaStream_t aux = nullptr, comm_st = nullptr;
  cudaEvent_t ev_start = nullptr, ev_heavy = nullptr, ev_piece[8] = {}, ev_comm = nullptr;
  int n_pieces = 1;           // PIO_ALS_PIECES (1..8); default 4 when world_size > 1
  bool pieces_done = false;   // the last launch_solve recorded ev_piece[] / ev_heavy (pair path)
  // low-latency serving (few queries, topk <= 128): a persistent device arena and a mapped pinned host arena -- no
  // allocation, no staging copies, results written by the merge kernel straight into host memory
  bool trace_on = false;      // PIO_ALS_INGEST_TRACE
  std::chrono::steady_clock::time_point t_prev;
  unsigned char* srv_dev = nullptr;
  size_t srv_dev_cap = 0;
  unsigned char* srv_host = nullptr;       // cudaHostAlloc(mapped)
  unsigned char* srv_host_dev = nullptr;   // its device address
  size_t srv_host_cap = 0;
  unsigned* srv_counter = nullptr;         // arrival counter of score_one_kernel (zero between calls)
  unsigned srv_seq = 0;                    // sequence number of the last fused single-query call
  bool serve_fused = true;                 // PIO_ALS_SERVE_FUSED=0: single queries take the three-launch path
  bool score_blocked = true;               // PIO_ALS_SCORE_BLOCKED=0: batched recommend on the one-item-per-thread kernel
  bool serve_trace = false;                // PIO_ALS_SERVE_TRACE=1: per-phase device timestamps of every fused call on stderr
  bool tc_split = false;      // PIO_ALS_TC_SPLIT=1: the tensor-core kernel only accumulates, a second kernel solves (measured: no gain)
  float* tc_out = nullptr;    // split mode: normal equations of one tile of rows ([rows][ASLOT + KP])
  size_t tc_out_rows = 0;
  double tc_min_deg = 0.0;    // PIO_ALS_TC_MIN_DEG: only sides whose rows average at least this many ratings use it
  bool have_ratings = false, have_init = false, trained = false;
  ncclComm_t comm = nullptr;
  std::string err;
  pio_als_stats st{};
  double phase_ms[8] = {0, 0, 0, 0, 0, 0, 0, 0};  // pio_als_get_phase_ms
  std::deque<EvPair> ev_pool;  // deque: references stay valid while the pool grows
  size_t ev_used = 0;
  std::mutex mu;
  int sm_count = 0;
};

namespace pio {

static int fail(pio_als_handle* h, int code, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  if (h) h->err = buf;
  else g_create_error = buf;
  return code;
}
// PIO_ALS_INGEST_TRACE=1: wall-clock milliseconds per ingest phase (stream drained at every mark) on stderr
static void tmark(pio_als_handle* h, const char* what) {
  if (!h->trace_on) return;
  cudaStreamSynchronize(h->stream);
  const auto now = std::chrono::steady_clock::now();
  fprintf(stderr, "[pio_als ingest r%d] %-34s %8.3f ms\n", h->cfg.world_rank, what,
          std::chrono::duration<double, std::milli>(now - h->t_prev).count());
  h->t_prev = now;
}
#define CK(h, call)                                                                              \
  do {                                                                                           \
    cudaError_t e_ = (call);                                                                     \
    if (e_ != cudaSuccess)                                                                       \
      return fail(h, PIO_ALS_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), \
                  __FILE__, __LINE__);                                                           \
  } while (0)
#define LAUNCHED(h) (++(h)->st.kernel_launches)

static inline unsigned nblk(long long n, int t) { return (unsigned)((n + t - 1) / t); }

template <class T>
static cudaError_t dalloc(pio_als_handle* h, T** p, size_t n) {
  return cudaMallocAsync((void**)p, (n ? n : 1) * sizeof(T), h->stream);
}
template <class T>
static void dfree(pio_als_handle* h, T*& p) {
  if (p) cudaFreeAsync((void*)p, h->stream);
  p = nullptr;
}

// Device temporaries of one API call: released (stream-ordered) on every exit path, including the early error returns
// of CK().
struct Scratch {
  pio_als_handle* h;
  std::vector<void*> ptrs;
  explicit Scratch(pio_als_handle* h_) : h(h_) {}
  Scratch(const Scratch&) = delete;
  Scratch& operator=(const Scratch&) = delete;
  template <class T>
  cudaError_t alloc(T** p, size_t n) {
    const cudaError_t e = dalloc(h, p, n);
    if (e == cudaSuccess) ptrs.push_back((void*)*p);
    return e;
  }
  ~Scratch() {
    for (void* q : ptrs) cudaFreeAsync(q, h->stream);
  }
};

static void free_side(pio_als_handle* h, Side& s, bool keep_factors) {
  dfree(h, s.perm); dfree(h, s.inv); dfree(h, s.rpos); dfree(h, s.p2i); dfree(h, s.deg); dfree(h, s.npos); dfree(h, s.ptr);
  dfree(h, s.idx); dfree(h, s.val); dfree(h, s.nreg); dfree(h, s.cand_ext);
  dfree(h, s.part_beg); dfree(h, s.part_end); dfree(h, s.row_part_ptr); dfree(h, s.partial);
  s.n_parts = 0;
  s.h_row_part_ptr.clear();
  if (!keep_factors) dfree(h, s.F);
}

static EvPair& next_ev(pio_als_handle* h, int kind) {
  if (h->ev_used == h->ev_pool.size()) {
    EvPair p;
    cudaEventCreate(&p.a);
    cudaEventCreate(&p.b);
    p.kind = kind;
    h->ev_pool.push_back(p);
  }
  EvPair& p = h->ev_pool[h->ev_used++];
  p.kind = kind;
  return p;
}

// ---- ingest ---------------------------------------------------------------------------------
static int build_side(pio_als_handle* h, Side& row, const Side& col, const int* rowext, const int* colext,
                      const float* rating, long long nnz, long long nnz_global) {
  // nnz ratings are present on this rank (all of them in replicated mode, those of the rows it owns in sharded mode);
  // nnz_global = ratings after dedup over all ranks (kernel choice must agree on every rank)
  cudaStream_t st = h->stream;
  const int W = h->cfg.world_size, rk = h->cfg.world_rank;
  Scratch tmp(h);
  uint64_t *ka = nullptr, *kb = nullptr;
  uint32_t *va = nullptr, *vb = nullptr;
  CK(h, tmp.alloc(&ka, (size_t)nnz));
  CK(h, tmp.alloc(&kb, (size_t)nnz));
  CK(h, tmp.alloc(&va, (size_t)nnz));
  CK(h, tmp.alloc(&vb, (size_t)nnz));
  bool in_b = false;
  if (nnz > 0) {
    make_keys_int_kernel<<<nblk(nnz, 256), 256, 0, st>>>(rowext, colext, nnz, row.perm, col.rpos, col.bits, ka, va);
    LAUNCHED(h);
    CK(h, radix_sort_pairs(ka, va, kb, vb, (size_t)nnz, row.bits + col.bits, st, &in_b, &h->st.kernel_launches));
  }
  tmark(h, "  side: keys + radix sort");
  const uint64_t* ks = in_b ? kb : ka;
  const uint32_t* vs = in_b ? vb : va;
  long long* ptr_full = nullptr;
  CK(h, tmp.alloc(&ptr_full, (size_t)row.n_internal + 1));
  CK(h, cudaMemsetAsync(ptr_full, 0, sizeof(long long) * ((size_t)row.n_internal + 1), st));
  if (nnz > 0) {
    build_ptr_kernel<<<nblk(nnz, 256), 256, 0, st>>>(ks, nnz, col.bits, row.n_internal, ptr_full);
    LAUNCHED(h);
  }
  long long be[2];
  CK(h, cudaMemcpyAsync(&be[0], ptr_full + (size_t)rk * row.R, sizeof(long long), cudaMemcpyDeviceToHost, st));
  CK(h, cudaMemcpyAsync(&be[1], ptr_full + (size_t)(rk + 1) * row.R, sizeof(long long), cudaMemcpyDeviceToHost, st));
  CK(h, cudaStreamSynchronize(st));
  row.nnz_local = be[1] - be[0];
  if (row.nnz_local >= (1ll << 31))
    return fail(h, PIO_ALS_ERR_ARG, "more than 2^31-1 ratings on one GPU (%lld); use more GPUs", row.nnz_local);
  CK(h, dalloc(h, &row.idx, (size_t)row.nnz_local));
  CK(h, dalloc(h, &row.val, (size_t)row.nnz_local));
  CK(h, dalloc(h, &row.ptr, (size_t)row.R + 1));
  CK(h, dalloc(h, &row.nreg, (size_t)row.R));
  if (row.nnz_local > 0) {
    extract_csr_kernel<<<nblk(row.nnz_local, 256), 256, 0, st>>>(ks, vs, rating, be[0], row.nnz_local, col.bits,
                                                                 col.p2i, row.idx, row.val);
    LAUNCHED(h);
  }
  tmark(h, "  side: ptr + extract csr");
  CK(h, cudaMemsetAsync(h->d_counts, 0, 2 * sizeof(int), st));
  // kernel choice from global numbers only (ratings after dedup / rows of this side), so that every rank of a sharded
  // run and the single-GPU run take the same path for the same row
  row.use_tc = h->use_tc && h->KP == 64 && row.n > 0 && (double)nnz_global / (double)row.n >= h->tc_min_deg;
  row.use_pair = !row.use_tc && h->KP == 64 && h->use_mma && h->use_pair;
  // one warp (mma kernels) or one accumulator slot (tcgen05 kernel) carries a whole row.  Pair kernel: rows up to 1024
  // ratings stay whole, longer rows become 512-rating parts of the same kernel (two-level summation); round-1 mma /
  // tcgen05 kernels: rows up to 8192 ratings whole, longer rows as 2016-rating parts on the FP32 kernel; FP32 kernel
  // (other ranks): cut at 4096
  // rank 65..128: every row is a work-list row (FP32 Gramian kernel -> partial normal equations -> lockstep finish kernel)
  row.heavy_t = h->KP == 128 ? 0 : row.use_pair ? h->pair_seg_t : (row.use_tc || (h->KP == 64 && h->use_mma)) ? HEAVY_T_TC : HEAVY_T;
  row.part_len = row.use_pair ? h->pair_part : PART;
  local_rows_kernel<<<nblk(row.R + 1, 256), 256, 0, st>>>(ptr_full, rk * row.R, row.R, be[0], row.inv, row.deg,
                                                           row.npos, h->cfg.implicit_prefs, row.ptr, row.nreg,
                                                           h->d_counts, row.heavy_t);
  LAUNCHED(h);
  int counts[2];
  CK(h, cudaMemcpyAsync(counts, h->d_counts, sizeof counts, cudaMemcpyDeviceToHost, st));
  CK(h, cudaStreamSynchronize(st));
  row.n_active = counts[0];
  row.n_heavy = counts[1];
  tmark(h, "  side: local rows");
  if (row.n_heavy > 0) {
    // cut the heavy rows (local rows [0, n_heavy), longest first) into parts of part_len ratings
    std::vector<long long> hp((size_t)row.n_heavy + 1);
    CK(h, cudaMemcpyAsync(hp.data(), row.ptr, sizeof(long long) * hp.size(), cudaMemcpyDeviceToHost, st));
    CK(h, cudaStreamSynchronize(st));
    std::vector<long long> pb, pe;
    std::vector<int> rpp((size_t)row.n_heavy + 1);
    for (int r = 0; r < row.n_heavy; ++r) {
      rpp[r] = (int)pb.size();
      for (long long b = hp[r]; b < hp[r + 1]; b += row.part_len) {
        pb.push_back(b);
        pe.push_back(b + row.part_len < hp[r + 1] ? b + row.part_len : hp[r + 1]);
      }
    }
    rpp[row.n_heavy] = (int)pb.size();
    row.n_parts = (int)pb.size();
    row.h_row_part_ptr = rpp;
    tmark(h, "  side: parts of long rows");
    CK(h, dalloc(h, &row.part_beg, pb.size()));
    CK(h, dalloc(h, &row.part_end, pe.size()));
    CK(h, dalloc(h, &row.row_part_ptr, rpp.size()));
    CK(h, cudaMemcpyAsync(row.part_beg, pb.data(), sizeof(long long) * pb.size(), cudaMemcpyHostToDevice, st));
    CK(h, cudaMemcpyAsync(row.part_end, pe.data(), sizeof(long long) * pe.size(), cudaMemcpyHostToDevice, st));
    CK(h, cudaMemcpyAsync(row.row_part_ptr, rpp.data(), sizeof(int) * rpp.size(), cudaMemcpyHostToDevice, st));
    CK(h, cudaStreamSynchronize(st));
  }
  (void)W;
  return PIO_ALS_OK;
}

static int rank_rows(pio_als_handle* h, Side& s) {
  cudaStream_t st = h->stream;
  Scratch tmp(h);
  uint64_t *ka = nullptr, *kb = nullptr;
  uint32_t *va = nullptr, *vb = nullptr;
  CK(h, tmp.alloc(&ka, (size_t)s.n));
  CK(h, tmp.alloc(&kb, (size_t)s.n));
  CK(h, tmp.alloc(&va, (size_t)s.n));
  CK(h, tmp.alloc(&vb, (size_t)s.n));
  degree_keys_kernel<<<nblk(s.n, 256), 256, 0, st>>>(s.deg, s.n, ka, va);
  LAUNCHED(h);
  bool in_b = false;
  CK(h, radix_sort_pairs(ka, va, kb, vb, (size_t)s.n, 32, st, &in_b, &h->st.kernel_launches));
  fill_int_kernel<<<nblk(s.n_internal, 256), 256, 0, st>>>(s.inv, s.n_internal, -1);
  LAUNCHED(h);
  assign_internal_kernel<<<nblk(s.n, 256), 256, 0, st>>>(in_b ? vb : va, s.n, h->cfg.world_size, s.R, s.perm, s.inv,
                                                         s.rpos, s.p2i);
  LAUNCHED(h);
  return PIO_ALS_OK;
}

// ---- sharded ingest: all-to-all exchange of event arrays ------------------------------------------------------------
// The n events on this rank go to the ranks named by the sort keys (destination rank, payload = event index; built by the
// caller in ka/va).  Events keep their order per destination and arrive concatenated in source-rank order, so a global
// event order (rank r's slice precedes rank r + 1's) survives.  The received arrays are allocated in `keep`.
struct XArr {
  const void* in;
  void** out;
  size_t elem;
};
static int exchange_events(pio_als_handle* h, Scratch& keep, uint64_t* ka, uint32_t* va, uint64_t* kb, uint32_t* vb,
                           long long n, XArr* arrs, int na, long long* n_out) {
  cudaStream_t st = h->stream;
  NcclApi& nc = nccl_api();
  const int W = h->cfg.world_size, me = h->cfg.world_rank;
  Scratch tmp(h);
  bool in_b = false;
  if (n > 0) CK(h, radix_sort_pairs(ka, va, kb, vb, (size_t)n, ceil_log2((uint64_t)W), st, &in_b, &h->st.kernel_launches));
  const uint64_t* ks = in_b ? kb : ka;
  const uint32_t* vs = in_b ? vb : va;
  long long *d_off = nullptr, *d_cnt = nullptr, *d_all = nullptr;
  CK(h, tmp.alloc(&d_off, (size_t)W + 1));
  CK(h, tmp.alloc(&d_cnt, (size_t)W));
  CK(h, tmp.alloc(&d_all, (size_t)W * W));
  CK(h, cudaMemsetAsync(d_off, 0, sizeof(long long) * (W + 1), st));
  if (n > 0) {
    build_ptr_kernel<<<nblk(n, 256), 256, 0, st>>>(ks, n, 0, W, d_off);
    LAUNCHED(h);
  }
  std::vector<long long> off(W + 1), all((size_t)W * W);
  CK(h, cudaMemcpyAsync(off.data(), d_off, sizeof(long long) * (W + 1), cudaMemcpyDeviceToHost, st));
  CK(h, cudaStreamSynchronize(st));
  std::vector<long long> cnt(W);
  for (int p = 0; p < W; ++p) cnt[p] = off[p + 1] - off[p];
  CK(h, cudaMemcpyAsync(d_cnt, cnt.data(), sizeof(long long) * W, cudaMemcpyHostToDevice, st));
  if (nc.AllGather(d_cnt, d_all, (size_t)W, ncclInt64, h->comm, st) != ncclSuccess)
    return fail(h, PIO_ALS_ERR_COMM, "ncclAllGather (exchange counts) failed");
  CK(h, cudaMemcpyAsync(all.data(), d_all, sizeof(long long) * W * W, cudaMemcpyDeviceToHost, st));
  CK(h, cudaStreamSynchronize(st));
  tmark(h, "  exchange: sort by rank + counts");
  std::vector<long long> roff(W + 1, 0);
  for (int src = 0; src < W; ++src) roff[src + 1] = roff[src] + all[(size_t)src * W + me];
  const long long nrecv = roff[W];
  if (nrecv >= (1ll << 32)) return fail(h, PIO_ALS_ERR_ARG, "more than 2^32-1 events on one rank after the exchange");
  // gather every array into destination order, then ONE grouped send/recv for all arrays and peers
  std::vector<unsigned char*> sendbufs(na, nullptr), recvbufs(na, nullptr);
  for (int a = 0; a < na; ++a) {
    if (!arrs[a].in) { *arrs[a].out = nullptr; continue; }
    CK(h, tmp.alloc(&sendbufs[a], (size_t)(n > 0 ? n : 1) * arrs[a].elem));
    CK(h, keep.alloc(&recvbufs[a], (size_t)(nrecv > 0 ? nrecv : 1) * arrs[a].elem));
    if (n > 0) {
      if (arrs[a].elem == 4)
        gather_by_index_kernel<uint32_t><<<nblk(n, 256), 256, 0, st>>>((const uint32_t*)arrs[a].in, vs, n, (uint32_t*)sendbufs[a]);
      else
        gather_by_index_kernel<uint64_t><<<nblk(n, 256), 256, 0, st>>>((const uint64_t*)arrs[a].in, vs, n, (uint64_t*)sendbufs[a]);
      LAUNCHED(h);
    }
    *arrs[a].out = recvbufs[a];
  }
  if (nc.GroupStart() != ncclSuccess) return fail(h, PIO_ALS_ERR_COMM, "ncclGroupStart failed");
  for (int a = 0; a < na; ++a) {
    if (!arrs[a].in) continue;
    for (int p = 0; p < W; ++p) {
      const long long sc = cnt[p], rc_ = all[(size_t)p * W + me];
      if (sc > 0 && nc.Send(sendbufs[a] + (size_t)off[p] * arrs[a].elem, (size_t)sc * arrs[a].elem, ncclInt8, p, h->comm, st) != ncclSuccess)
        return fail(h, PIO_ALS_ERR_COMM, "ncclSend failed");
      if (rc_ > 0 && nc.Recv(recvbufs[a] + (size_t)roff[p] * arrs[a].elem, (size_t)rc_ * arrs[a].elem, ncclInt8, p, h->comm, st) != ncclSuccess)
        return fail(h, PIO_ALS_ERR_COMM, "ncclRecv failed");
    }
  }
  if (nc.GroupEnd() != ncclSuccess) return fail(h, PIO_ALS_ERR_COMM, "ncclGroupEnd failed");
  CK(h, cudaStreamSynchronize(st));
  tmark(h, "  exchange: gather + send/recv");
  *n_out = nrecv;
  return PIO_ALS_OK;
}

// sharded == false: the arrays hold ALL events (every rank passes the same COO and keeps the rows it owns).
// sharded == true (world_size > 1): the arrays hold this rank's slice of the events; ratings are routed to the owners of
// their user row and of their item row by NCCL send/recv, degrees are all-reduced; no rank ever holds the full COO.
static int ingest_device(pio_als_handle* h, const int* d_user, const int* d_item, const float* d_rating,
                         long long nnz, int dedup, const long long* d_ts, bool sharded) {
  cudaStream_t st = h->stream;
  const int W = h->cfg.world_size;
  sharded = sharded && W > 1;
  if (nnz <= 0 && !sharded)
    return fail(h, PIO_ALS_ERR_ARG, "ratings cannot be empty (the templates require(!ratings.take(1).isEmpty))");
  if (nnz < 0) return fail(h, PIO_ALS_ERR_ARG, "nnz < 0");
  if (nnz >= (1ll << 32)) return fail(h, PIO_ALS_ERR_ARG, "nnz must be < 2^32 per call");
  if (dedup < 0 || dedup > 2) return fail(h, PIO_ALS_ERR_ARG, "bad dedup_mode %d", dedup);
  free_side(h, h->U, true);
  free_side(h, h->I, true);
  h->have_ratings = false;
  Side& U = h->U;
  Side& I = h->I;
  U.n = h->cfg.n_users;
  I.n = h->cfg.n_items;
  U.R = (U.n + W - 1) / W;
  I.R = (I.n + W - 1) / W;
  U.n_internal = U.R * W;
  I.n_internal = I.R * W;
  U.bits = ceil_log2((uint64_t)U.n_internal);
  I.bits = ceil_log2((uint64_t)I.n_internal);

  h->trace_on = getenv("PIO_ALS_INGEST_TRACE") != nullptr;
  h->t_prev = std::chrono::steady_clock::now();
  auto mark = [&](const char* what) { tmark(h, what); };
  CK(h, cudaMemsetAsync(h->d_fail, 0, sizeof(int), st));
  if (nnz > 0) {
    validate_coo_kernel<<<nblk(nnz, 256), 256, 0, st>>>(d_user, d_item, nnz, U.n, I.n, h->d_fail);
    LAUNCHED(h);
  }
  int bad = 0;
  CK(h, cudaMemcpyAsync(&bad, h->d_fail, sizeof(int), cudaMemcpyDeviceToHost, st));
  CK(h, cudaStreamSynchronize(st));
  if (bad) return fail(h, PIO_ALS_ERR_ARG, "%d ratings have a user/item index out of range", bad);

  mark("validate");
  Scratch tmp(h);   // everything temporary: released on every exit path, including the CK() early returns
  // 0. sharded + dedup: first bring all events of a user to one rank (user mod W), keeping the event order
  const int* su = d_user;
  const int* si = d_item;
  const float* sr = d_rating;
  const long long* sts = d_ts;
  long long ns = nnz;
  if (sharded && dedup != PIO_ALS_DEDUP_NONE) {
    Scratch xs(h);
    uint64_t *ka = nullptr, *kb = nullptr;
    uint32_t *va = nullptr, *vb = nullptr;
    CK(h, xs.alloc(&ka, (size_t)nnz)); CK(h, xs.alloc(&kb, (size_t)nnz));
    CK(h, xs.alloc(&va, (size_t)nnz)); CK(h, xs.alloc(&vb, (size_t)nnz));
    if (nnz > 0) {
      dest_mod_kernel<<<nblk(nnz, 256), 256, 0, st>>>(d_user, nnz, W, ka, va);
      LAUNCHED(h);
    }
    void *xu = nullptr, *xi = nullptr, *xr = nullptr, *xt = nullptr;
    XArr arrs[4] = {{d_user, &xu, 4}, {d_item, &xi, 4}, {d_rating, &xr, 4},
                    {dedup == PIO_ALS_DEDUP_KEEP_LAST ? (const void*)d_ts : nullptr, &xt, 8}};
    int rc = exchange_events(h, tmp, ka, va, kb, vb, nnz, arrs, 4, &ns);
    if (rc) return rc;
    su = (const int*)xu; si = (const int*)xi; sr = (const float*)xr; sts = (const long long*)xt;
  }

  mark("exchange by user residue");
  // 1. optional dedup of repeated (user,item) pairs (all copies of a pair are on this rank)
  const int* cu = su;
  const int* ci = si;
  const float* cr = sr;
  long long n2 = ns;
  if (dedup != PIO_ALS_DEDUP_NONE && ns > 0) {
    Scratch ds(h);
    uint64_t *ka = nullptr, *kb = nullptr;
    uint32_t *va = nullptr, *vb = nullptr;
    CK(h, ds.alloc(&ka, (size_t)ns)); CK(h, ds.alloc(&kb, (size_t)ns));
    CK(h, ds.alloc(&va, (size_t)ns)); CK(h, ds.alloc(&vb, (size_t)ns));
    const int bu = ceil_log2((uint64_t)U.n), bi = ceil_log2((uint64_t)I.n);
    make_keys_ext_kernel<<<nblk(ns, 256), 256, 0, st>>>(su, si, ns, bi, ka, va);
    LAUNCHED(h);
    bool in_b = false;
    CK(h, radix_sort_pairs(ka, va, kb, vb, (size_t)ns, bu + bi, st, &in_b, &h->st.kernel_launches));
    const uint64_t* ks = in_b ? kb : ka;
    const uint32_t* vs = in_b ? vb : va;
    uint32_t* flag = nullptr;
    CK(h, ds.alloc(&flag, (size_t)ns));
    head_flags_kernel<<<nblk(ns, 256), 256, 0, st>>>(ks, ns, flag);
    LAUNCHED(h);
    uint32_t last_flag = 0, last_pos = 0;
    CK(h, cudaMemcpyAsync(&last_flag, flag + ns - 1, sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
    CK(h, scan_exclusive_u32(flag, flag, (size_t)ns, st, &h->st.kernel_launches));
    CK(h, cudaMemcpyAsync(&last_pos, flag + ns - 1, sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
    CK(h, cudaStreamSynchronize(st));
    n2 = (long long)last_pos + last_flag;
    int *du_ = nullptr, *di_ = nullptr;
    float* dr_ = nullptr;
    CK(h, tmp.alloc(&du_, (size_t)n2));
    CK(h, tmp.alloc(&di_, (size_t)n2));
    CK(h, tmp.alloc(&dr_, (size_t)n2));
    dedup_compact_kernel<<<nblk(ns, 256), 256, 0, st>>>(ks, vs, flag, ns, bi, sr, sts, dedup, du_, di_, dr_);
    LAUNCHED(h);
    cu = du_;
    ci = di_;
    cr = dr_;
  }

  mark("dedup");
  // 2. degrees, positive-rating counts (sharded: summed over the ranks)
  for (Side* s : {&U, &I}) {
    CK(h, dalloc(h, &s->deg, (size_t)s->n));
    CK(h, dalloc(h, &s->npos, (size_t)s->n));
    CK(h, dalloc(h, &s->perm, (size_t)s->n));
    CK(h, dalloc(h, &s->inv, (size_t)s->n_internal));
    CK(h, dalloc(h, &s->rpos, (size_t)s->n));
    CK(h, dalloc(h, &s->p2i, (size_t)s->n));
    CK(h, cudaMemsetAsync(s->deg, 0, sizeof(uint32_t) * s->n, st));
    CK(h, cudaMemsetAsync(s->npos, 0, sizeof(uint32_t) * s->n, st));
  }
  if (n2 > 0) {
    degree_kernel<<<nblk(n2, 256), 256, 0, st>>>(cu, ci, cr, n2, U.deg, I.deg, U.npos, I.npos);
    LAUNCHED(h);
  }
  long long n2_global = n2;
  if (sharded) {
    NcclApi& nc = nccl_api();   // only multi-GPU jobs touch NCCL (a single-GPU process must not load libnccl at all)
    long long* d_n = nullptr;
    CK(h, tmp.alloc(&d_n, 1));
    CK(h, cudaMemcpyAsync(d_n, &n2, sizeof(long long), cudaMemcpyHostToDevice, st));
    if (nc.GroupStart() != ncclSuccess) return fail(h, PIO_ALS_ERR_COMM, "ncclGroupStart failed");   // one launch for the five
    for (Side* s : {&U, &I}) {
      if (nc.AllReduce(s->deg, s->deg, (size_t)s->n, ncclUint32, ncclSum, h->comm, st) != ncclSuccess ||
          nc.AllReduce(s->npos, s->npos, (size_t)s->n, ncclUint32, ncclSum, h->comm, st) != ncclSuccess)
        return fail(h, PIO_ALS_ERR_COMM, "ncclAllReduce (degrees) failed");
    }
    if (nc.AllReduce(d_n, d_n, 1, ncclInt64, ncclSum, h->comm, st) != ncclSuccess)
      return fail(h, PIO_ALS_ERR_COMM, "ncclAllReduce (nnz) failed");
    if (nc.GroupEnd() != ncclSuccess) return fail(h, PIO_ALS_ERR_COMM, "ncclGroupEnd failed");
    CK(h, cudaMemcpyAsync(&n2_global, d_n, sizeof(long long), cudaMemcpyDeviceToHost, st));
    CK(h, cudaStreamSynchronize(st));
    if (n2_global <= 0)
      return fail(h, PIO_ALS_ERR_ARG, "ratings cannot be empty (the templates require(!ratings.take(1).isEmpty))");
  }
  h->st.nnz = n2_global;

  mark("degrees (+ all-reduce)");
  // 3. renumber rows: degree-descending, dealt to ranks (the same on every rank)
  int rc = rank_rows(h, U);
  if (rc) return rc;
  rc = rank_rows(h, I);
  if (rc) return rc;

  mark("rank rows");
  // 4. the two CSR orientations in internal numbering (only this rank's rows are kept)
  if (!sharded) {
    rc = build_side(h, U, I, cu, ci, cr, n2, n2_global);
    if (rc) return rc;
    mark("build user side");
    rc = build_side(h, I, U, ci, cu, cr, n2, n2_global);
    if (rc) return rc;
    mark("build item side");
  } else {
    struct { Side* row; Side* col; const int* rowext; const int* colext; } jobs[2] = {{&U, &I, cu, ci}, {&I, &U, ci, cu}};
    for (auto& j : jobs) {
      Scratch xs(h), recv(h);
      uint64_t *ka = nullptr, *kb = nullptr;
      uint32_t *va = nullptr, *vb = nullptr;
      CK(h, xs.alloc(&ka, (size_t)n2)); CK(h, xs.alloc(&kb, (size_t)n2));
      CK(h, xs.alloc(&va, (size_t)n2)); CK(h, xs.alloc(&vb, (size_t)n2));
      if (n2 > 0) {
        dest_owner_kernel<<<nblk(n2, 256), 256, 0, st>>>(j.rowext, n2, j.row->perm, j.row->R, ka, va);
        LAUNCHED(h);
      }
      void *xrow = nullptr, *xcol = nullptr, *xr = nullptr;
      XArr arrs[3] = {{j.rowext, &xrow, 4}, {j.colext, &xcol, 4}, {cr, &xr, 4}};
      long long ne = 0;
      rc = exchange_events(h, recv, ka, va, kb, vb, n2, arrs, 3, &ne);
      if (rc) return rc;
      mark("exchange by row owner");
      rc = build_side(h, *j.row, *j.col, (const int*)xrow, (const int*)xcol, (const float*)xr, ne, n2_global);
      if (rc) return rc;
      mark("build side");
    }
  }

  // 5. factor matrices (zero: rows without ratings must stay zero) and candidate tables
  for (Side* s : {&U, &I}) {
    if (!s->F) {
      CK(h, dalloc(h, &s->F, (size_t)s->n_internal * h->KP));
      h->have_init = false;
    }
    CK(h, dalloc(h, &s->cand_ext, (size_t)s->n_internal));
    cand_ext_kernel<<<nblk(s->n_internal, 256), 256, 0, st>>>(s->inv, s->deg, s->n_internal, s->cand_ext);
    LAUNCHED(h);
  }
  h->have_init = false;
  CK(h, cudaStreamSynchronize(st));
  mark("factor buffers");
  h->st.n_users_active = U.n_active;
  h->st.n_items_active = I.n_active;
  if (W > 1) {
    // n_active per rank is local; the global counts are not needed by the library
    h->st.n_users_active = -1;
    h->st.n_items_active = -1;
  }
  h->have_ratings = true;
  h->trained = false;
  return PIO_ALS_OK;
}

static int init_hash(pio_als_handle* h) {
  cudaStream_t st = h->stream;
  CK(h, cudaMemsetAsync(h->U.F, 0, sizeof(float) * (size_t)h->U.n_internal * h->KP, st));
  CK(h, cudaMemsetAsync(h->I.F, 0, sizeof(float) * (size_t)h->I.n_internal * h->KP, st));
  hash_init_kernel<<<nblk(h->U.n, 128), 128, 0, st>>>(h->U.n, h->cfg.rank, h->KP, (uint64_t)h->cfg.seed, 0, h->U.perm,
                                                      h->U.deg, h->U.F);
  LAUNCHED(h);
  hash_init_kernel<<<nblk(h->I.n, 128), 128, 0, st>>>(h->I.n, h->cfg.rank, h->KP, (uint64_t)h->cfg.seed, 1, h->I.perm,
                                                      h->I.deg, h->I.F);
  LAUNCHED(h);
  h->have_init = true;
  return PIO_ALS_OK;
}

// ---- solve dispatch ---------------------------------------------------------------------------
template <class Cfg, bool IMPLICIT>
static cudaError_t launch_solve_one(pio_als_handle* h, const SolveParams& p, int grid, cudaStream_t st) {
  static bool attr_set[64] = {};
  int dev = h->cfg.device;
  auto kern = als_solve_kernel<Cfg, IMPLICIT>;
  const size_t smem = Cfg::smem_bytes();
  if (dev < 64 && !attr_set[dev]) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    attr_set[dev] = true;
  }
  kern<<<grid, Cfg::NT, smem, st>>>(p);
  LAUNCHED(h);
  ++h->st.solve_launches;
  return cudaGetLastError();
}

// Gramians on tcgen05 (als_tc_kernel.cuh): persistent, one CTA per SM, rows assigned statically.  A = role partition.
// Split mode (PIO_ALS_TC_SPLIT=1, off by default): the kernel only accumulates and stores the normal equations of a
// tile of rows; a second kernel solves them with every warp of the SM.  Measured at C2: item side 15.0 vs 15.4 ms fused,
// user side 39.7 vs 38.2 ms fused (the one-warp 64x64 Cholesky is latency-bound, ~50-70 k cycles per row, so twelve
// solver warps per SM at 168 registers do not beat the fused ones overlapped with the MMAs).
template <class A>
static cudaError_t launch_tc(pio_als_handle* h, Side& dst, const SolveParams& p, bool imp, int nlight) {
  cudaError_t e = cudaSuccess;
  static bool attr_set[64] = {};
  if (h->cfg.device < 64 && !attr_set[h->cfg.device]) {
    if ((e = cudaFuncSetAttribute(A::kernel(true), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)A::kSmem)) != cudaSuccess) return e;
    if ((e = cudaFuncSetAttribute(A::kernel(false), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)A::kSmem)) != cudaSuccess) return e;
    if ((e = cudaFuncSetAttribute(A::solver(true), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)A::kSolveSmem)) != cudaSuccess) return e;
    if ((e = cudaFuncSetAttribute(A::solver(false), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)A::kSolveSmem)) != cudaSuccess) return e;
    attr_set[h->cfg.device] = true;
  }
  typename A::Params tp;
  tp.dbg = nullptr;
  tp.timing = nullptr;
  tp.out = nullptr;
  tp.out_row0 = 0;
  if (getenv("PIO_ALS_TC_TIMING")) {
    if (!h->d_timing && (e = cudaMalloc((void**)&h->d_timing, (size_t)h->sm_count * 16 * 8 * sizeof(long long))) != cudaSuccess) return e;
    cudaMemsetAsync(h->d_timing, 0, (size_t)h->sm_count * 16 * 8 * sizeof(long long), h->stream);
    tp.timing = h->d_timing;
  }
  if (getenv("PIO_ALS_TC_DEBUG")) {
    if (h->dbg_rows < (size_t)dst.R) {
      if (h->d_dbg) cudaFree(h->d_dbg);
      if ((e = cudaMalloc((void**)&h->d_dbg, (size_t)dst.R * A::kRowFloats * sizeof(float))) != cudaSuccess) return e;
      h->dbg_rows = dst.R;
    }
    cudaMemsetAsync(h->d_dbg, 0, (size_t)dst.R * A::kRowFloats * sizeof(float), h->stream);
    tp.dbg = h->d_dbg;
  }
  const int tile = h->tc_split ? TC_TILE_ROWS : nlight;
  if (h->tc_split) {
    const size_t need = (size_t)(nlight < tile ? nlight : tile);
    if (h->tc_out_rows < need) {
      if (h->tc_out) cudaFree(h->tc_out);
      h->tc_out = nullptr;
      h->tc_out_rows = 0;
      if ((e = cudaMalloc((void**)&h->tc_out, need * A::kRowFloats * sizeof(float))) != cudaSuccess) return e;
      h->tc_out_rows = need;
    }
  }
  for (int t0 = p.row_begin; t0 < p.row_end; t0 += tile) {
    SolveParams q = p;
    q.row_begin = t0;
    q.row_end = t0 + tile < p.row_end ? t0 + tile : p.row_end;
    const int nrows = q.row_end - q.row_begin;
    tp.sp = q;
    tp.out = h->tc_split ? h->tc_out : nullptr;
    tp.out_row0 = t0;
    int grid = (nrows + A::kPerCta - 1) / A::kPerCta;
    if (grid > h->sm_count) grid = h->sm_count;
    A::kernel(imp)<<<grid, A::kThreads, A::kSmem, h->stream>>>(tp);
    LAUNCHED(h);
    ++h->st.solve_launches;
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
    if (h->tc_split) {
      int sgrid = (nrows + A::kSolveWarps - 1) / A::kSolveWarps;
      if (sgrid > 4 * h->sm_count) sgrid = 4 * h->sm_count;
      A::solver(imp)<<<sgrid, A::kSolveWarps * 32, A::kSolveSmem, h->stream>>>(q, h->tc_out, t0);
      LAUNCHED(h);
      ++h->st.solve_launches;
      if ((e = cudaGetLastError()) != cudaSuccess) return e;
    }
  }
  return e;
}

template <int WARPS>
static cudaError_t launch_pair_w(pio_als_handle* h, Side& dst, const SolveParams& p0, bool imp) {
  cudaError_t e = cudaSuccess;
  static bool attr_set[64] = {};
  const size_t smem = pr::smem_bytes(WARPS), fsmem = pr::smem_bytes(1);
  if (h->cfg.device < 64 && !attr_set[h->cfg.device]) {
    struct { const void* f; size_t sm; } ks[4] = {{(const void*)pr::als_solve_pair_kernel<true, WARPS>, smem},
                                                 {(const void*)pr::als_solve_pair_kernel<false, WARPS>, smem},
                                                 {(const void*)pr::als_finish_pair_kernel<true>, fsmem},
                                                 {(const void*)pr::als_finish_pair_kernel<false>, fsmem}};
    for (auto& kf : ks) {
      if ((e = cudaFuncSetAttribute(kf.f, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kf.sm)) != cudaSuccess) return e;
      if ((e = cudaFuncSetAttribute(kf.f, cudaFuncAttributePreferredSharedMemoryCarveout, 100)) != cudaSuccess) return e;
    }
    attr_set[h->cfg.device] = true;
  }
  const int max_ctas = (12 / WARPS) * h->sm_count;
  auto grid_for = [&](int items) {
    const int npairs = (items + 1) / 2;
    const int g = (npairs + WARPS - 1) / WARPS;
    return g < max_ctas ? g : max_ctas;
  };
  auto sk = imp ? pr::als_solve_pair_kernel<true, WARPS> : pr::als_solve_pair_kernel<false, WARPS>;
  cudaEventRecord(h->ev_start, h->stream);
  if (dst.n_heavy > 0) {
    // long rows on the auxiliary stream: parts, then the finish kernel.  Launched first: the kernels are persistent
    // (one full wave), so the CTAs of the whole-row launch below move in as the part CTAs retire and the finish
    // kernel overlaps the whole-row kernel instead of waiting behind it.
    if (!dst.partial) {
      if ((e = cudaMallocAsync((void**)&dst.partial, sizeof(float) * (size_t)dst.n_parts * pr::PART_FLOATS, h->stream)) != cudaSuccess) return e;
      cudaEventRecord(h->ev_start, h->stream);
    }
    cudaStreamWaitEvent(h->aux, h->ev_start, 0);
    SolveParams pp = p0;
    pp.wl_beg = dst.part_beg;
    pp.wl_end = dst.part_end;
    pp.partial = dst.partial;
    pp.n_items = dst.n_parts;
    pp.row_begin = 0;
    pp.row_end = dst.n_heavy;
    sk<<<grid_for(dst.n_parts), 32 * WARPS, smem, h->aux>>>(pp, dst.n_parts);
    LAUNCHED(h);
    ++h->st.solve_launches;
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
    auto fk = imp ? pr::als_finish_pair_kernel<true> : pr::als_finish_pair_kernel<false>;
    int fgrid = (dst.n_heavy + 1) / 2;
    if (fgrid > 12 * h->sm_count) fgrid = 12 * h->sm_count;
    fk<<<fgrid, 32, fsmem, h->aux>>>(pp, dst.row_part_ptr, dst.n_heavy);
    LAUNCHED(h);
    ++h->st.solve_launches;
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
  }
  cudaEventRecord(h->ev_heavy, h->aux);
  // whole rows, one launch per piece of the local row range (the all-gather of a piece starts when its rows are done)
  const int C = h->n_pieces;
  for (int c = 0; c < C; ++c) {
    const long long plo = (long long)dst.R * c / C, phi = (long long)dst.R * (c + 1) / C;
    const int lo = plo > dst.n_heavy ? (int)plo : dst.n_heavy;
    const int hi = phi < dst.n_active ? (int)phi : dst.n_active;
    if (hi > lo) {
      SolveParams p = p0;
      p.row_begin = lo;
      p.row_end = hi;
      sk<<<grid_for(hi - lo), 32 * WARPS, smem, h->stream>>>(p, hi - lo);
      LAUNCHED(h);
      ++h->st.solve_launches;
      if ((e = cudaGetLastError()) != cudaSuccess) return e;
    }
    cudaEventRecord(h->ev_piece[c], h->stream);
  }
  cudaStreamWaitEvent(h->stream, h->ev_heavy, 0);   // the half-step ends when both streams are done
  h->pieces_done = true;
  return e;
}

// Rank 33..64, pair kernel (als_pair_kernel.cuh): persistent CTAs of pair_warps independent warps, twelve warps per
// SM.  Long rows first (their 512-rating parts as work items, then the finish kernel), then the rows that stay whole.
static cudaError_t launch_pair(pio_als_handle* h, Side& dst, const SolveParams& p0, bool imp) {
  switch (h->pair_warps) {
    case 1: return launch_pair_w<1>(h, dst, p0, imp);
    case 2: return launch_pair_w<2>(h, dst, p0, imp);
    case 6: return launch_pair_w<6>(h, dst, p0, imp);
    case 12: return launch_pair_w<12>(h, dst, p0, imp);
    default: return launch_pair_w<4>(h, dst, p0, imp);
  }
}

template <class Cfg>
static cudaError_t launch_solve_cfg(pio_als_handle* h, Side& dst, const Side& src) {
  SolveParams p;
  p.ptr = dst.ptr;
  p.idx = dst.idx;
  p.val = dst.val;
  p.src = src.F;
  p.dst = dst.F;
  p.yty = h->yty;
  p.nreg = dst.nreg;
  p.fail = h->d_fail;
  p.lambda = (float)h->cfg.lambda;
  p.alpha = (float)h->cfg.alpha;
  p.k = h->cfg.rank;
  p.dst_row_offset = h->cfg.world_rank * dst.R;
  const bool imp = h->cfg.implicit_prefs != 0;
  cudaError_t e = cudaSuccess;
  p.wl_beg = nullptr;
  p.wl_end = nullptr;
  p.partial = nullptr;
  p.n_items = 0;
  if (dst.use_pair && Cfg::KP == 64) return launch_pair(h, dst, p, imp);
  if (Cfg::LS_PARTIAL) {
    // rank 65..128: rows in tiles; per tile one Gramian launch over the tile's parts and one lockstep finish launch
    constexpr int TILE_ROWS = 32768;
    const int nrows = dst.n_heavy;   // == n_active (heavy_t = 0)
    if (nrows == 0) return cudaSuccess;
    const std::vector<int>& rpp = dst.h_row_part_ptr;
    if (!dst.partial) {
      int mx = 0;
      for (int r0 = 0; r0 < nrows; r0 += TILE_ROWS) {
        const int r1 = r0 + TILE_ROWS < nrows ? r0 + TILE_ROWS : nrows;
        mx = rpp[r1] - rpp[r0] > mx ? rpp[r1] - rpp[r0] : mx;
      }
      if ((e = cudaMallocAsync((void**)&dst.partial, sizeof(float) * (size_t)mx * Cfg::PART_FLOATS, h->stream)) != cudaSuccess) return e;
    }
    static bool fattr[64] = {};
    const size_t fsmem = sizeof(float) * (size_t)FIN128_FLOATS * FIN128_WARPS;
    if (h->cfg.device < 64 && !fattr[h->cfg.device]) {
      if ((e = cudaFuncSetAttribute(als_finish_ls128_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)fsmem)) != cudaSuccess) return e;
      if ((e = cudaFuncSetAttribute(als_finish_ls128_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)fsmem)) != cudaSuccess) return e;
      fattr[h->cfg.device] = true;
    }
    for (int r0 = 0; r0 < nrows; r0 += TILE_ROWS) {
      const int r1 = r0 + TILE_ROWS < nrows ? r0 + TILE_ROWS : nrows;
      const int part0 = rpp[r0], np = rpp[r1] - rpp[r0];
      SolveParams pp = p;
      pp.wl_beg = dst.part_beg + part0;
      pp.wl_end = dst.part_end + part0;
      pp.partial = dst.partial;
      pp.n_items = np;
      pp.row_begin = 0;
      pp.row_end = nrows;
      const int grid = (np + Cfg::NG - 1) / Cfg::NG;
      e = imp ? launch_solve_one<Cfg, true>(h, pp, grid, h->stream) : launch_solve_one<Cfg, false>(h, pp, grid, h->stream);
      if (e != cudaSuccess) return e;
      int fgrid = (r1 - r0 + FIN128_WARPS - 1) / FIN128_WARPS;
      if (fgrid > h->sm_count) fgrid = h->sm_count;
      if (imp) als_finish_ls128_kernel<true><<<fgrid, 32 * FIN128_WARPS, fsmem, h->stream>>>(pp, dst.row_part_ptr, r0, r1 - r0, part0);
      else als_finish_ls128_kernel<false><<<fgrid, 32 * FIN128_WARPS, fsmem, h->stream>>>(pp, dst.row_part_ptr, r0, r1 - r0, part0);
      LAUNCHED(h);
      ++h->st.solve_launches;
      if ((e = cudaGetLastError()) != cudaSuccess) return e;
    }
    return e;
  }
  // very long rows: their parts run as ordinary light batch items that emit partial normal equations
  if (dst.n_heavy > 0) {
    if (!dst.partial) {
      if ((e = cudaMallocAsync((void**)&dst.partial, sizeof(float) * (size_t)dst.n_parts * (Cfg::SLOT + Cfg::KP), h->stream)) != cudaSuccess) return e;
    }
    SolveParams pp = p;
    pp.wl_beg = dst.part_beg;
    pp.wl_end = dst.part_end;
    pp.partial = dst.partial;
    pp.n_items = dst.n_parts;
    pp.row_begin = 0;
    pp.row_end = dst.n_heavy;
    const int grid = (dst.n_parts + Cfg::NG - 1) / Cfg::NG;
    e = imp ? launch_solve_one<Cfg, true>(h, pp, grid, h->stream) : launch_solve_one<Cfg, false>(h, pp, grid, h->stream);
    if (e != cudaSuccess) return e;
    // finish: sum the parts of every heavy row in fixed order, then Cholesky
    {
      static bool fattr[64] = {};
      const size_t fsmem = sizeof(float) * 4 * (Cfg::SLOT + 4 * Cfg::KP);
      auto fk = imp ? als_finish_kernel<Cfg, true> : als_finish_kernel<Cfg, false>;
      if (h->cfg.device < 64 && !fattr[h->cfg.device]) {
        if ((e = cudaFuncSetAttribute(als_finish_kernel<Cfg, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)fsmem)) != cudaSuccess) return e;
        if ((e = cudaFuncSetAttribute(als_finish_kernel<Cfg, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)fsmem)) != cudaSuccess) return e;
        fattr[h->cfg.device] = true;
      }
      const int fgrid = Cfg::WARP_CHOL ? (dst.n_heavy + 3) / 4 : dst.n_heavy;
      fk<<<fgrid, Cfg::WARP_CHOL ? 128 : Cfg::NT, fsmem, h->stream>>>(pp, dst.row_part_ptr, dst.n_heavy);
      LAUNCHED(h);
      ++h->st.solve_launches;
      if ((e = cudaGetLastError()) != cudaSuccess) return e;
    }
  }
  const int nlight = dst.n_active - dst.n_heavy;
  if (nlight > 0) {
    p.row_begin = dst.n_heavy;
    p.row_end = dst.n_active;
    if (dst.use_tc && Cfg::KP == 64) {
      e = launch_tc<tc::Api>(h, dst, p, imp, nlight);
      if (e != cudaSuccess) return e;
    } else if (Cfg::KP == 64 && h->use_mma) {
      // short rows of rank 33..64: one warp per row, mma.sync Gramian (als_mma_kernel.cuh)
      static bool mattr[64] = {};
      auto mk = imp ? mm::als_solve_mma_kernel<true> : mm::als_solve_mma_kernel<false>;
      if (h->cfg.device < 64 && !mattr[h->cfg.device]) {
        if ((e = cudaFuncSetAttribute(mm::als_solve_mma_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)mm::SMEM_BYTES)) != cudaSuccess) return e;
        if ((e = cudaFuncSetAttribute(mm::als_solve_mma_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)mm::SMEM_BYTES)) != cudaSuccess) return e;
        mattr[h->cfg.device] = true;
      }
      const int grid = (nlight + mm::WARPS - 1) / mm::WARPS;
      mk<<<grid, mm::NT, mm::SMEM_BYTES, h->stream>>>(p);
      LAUNCHED(h);
      ++h->st.solve_launches;
      if ((e = cudaGetLastError()) != cudaSuccess) return e;
    } else {
      const int grid = (nlight + Cfg::NG - 1) / Cfg::NG;
      e = imp ? launch_solve_one<Cfg, true>(h, p, grid, h->stream) : launch_solve_one<Cfg, false>(h, p, grid, h->stream);
      if (e != cudaSuccess) return e;
    }
  }
  return e;
}

using Cfg16 = SolveCfg<16, 4, 25, 8>;
using Cfg32 = SolveCfg<32, 8, 25, 4>;
using Cfg64 = SolveCfg<64, 8, 7, 8>;
using Cfg128 = SolveCfg<128, 8, 2, 9>;

static cudaError_t launch_solve(pio_als_handle* h, Side& dst, const Side& src) {
  switch (h->KP) {
    case 16: return launch_solve_cfg<Cfg16>(h, dst, src);
    case 32: return launch_solve_cfg<Cfg32>(h, dst, src);
    case 64: return launch_solve_cfg<Cfg64>(h, dst, src);
    default: return launch_solve_cfg<Cfg128>(h, dst, src);
  }
}

// YtY (implicit feedback): als_kernels.cuh GramMap.  gram_sharded(): every rank owns whole classes (world size 2, 4, 8).
static bool gram_sharded(const pio_als_handle* h) { return h->cfg.world_size > 1 && GRAM_GROUPS % h->cfg.world_size == 0; }
static void gram_layout(const pio_als_handle* h, GramMap& m, int& my_groups, int& slot0) {
  const bool shard = gram_sharded(h);
  const int W = shard ? h->cfg.world_size : 1, me = shard ? h->cfg.world_rank : 0;
  my_groups = GRAM_GROUPS / W;
  slot0 = me * my_groups;
  int seen[GRAM_GROUPS] = {}, mine = 0;
  for (int g = 0; g < GRAM_GROUPS; ++g) {
    const int blk = g / W, pos = g % W;
    const int owner = (blk & 1) ? (W - 1 - pos) : pos;      // assign_internal_kernel's dealing, positions 0 .. 7
    m.slot_of[g] = owner * my_groups + seen[owner]++;
    if (owner == me) m.cls[mine++] = g;
  }
  for (int lg = mine; lg < GRAM_GROUPS; ++lg) m.cls[lg] = 0;
}
// phase A: block partials and slot sums of this rank's classes (sharded: from its own rows only)
static int gram_local(pio_als_handle* h, const Side& s) {
  GramMap m;
  int my_groups, slot0;
  gram_layout(h, m, my_groups, slot0);
  const int bpg = h->gram_blocks / GRAM_GROUPS, n = h->KP * h->KP, grid = my_groups * bpg;
  switch (h->KP) {
    case 16: gram_partial_kernel<16><<<grid, GRAM_THREADS, 0, h->stream>>>(s.F, s.p2i, s.n, h->gram_partial, slot0, bpg, m); break;
    case 32: gram_partial_kernel<32><<<grid, GRAM_THREADS, 0, h->stream>>>(s.F, s.p2i, s.n, h->gram_partial, slot0, bpg, m); break;
    case 64: gram_partial_kernel<64><<<grid, GRAM_THREADS, 0, h->stream>>>(s.F, s.p2i, s.n, h->gram_partial, slot0, bpg, m); break;
    default: gram_partial_kernel<128><<<grid, GRAM_THREADS, 0, h->stream>>>(s.F, s.p2i, s.n, h->gram_partial, slot0, bpg, m); break;
  }
  LAUNCHED(h);
  gram_group_kernel<<<dim3(nblk(n, 128), my_groups), 128, 0, h->stream>>>(h->gram_partial, bpg, n, slot0, h->gram_gsum);
  LAUNCHED(h);
  CK(h, cudaGetLastError());
  return PIO_ALS_OK;
}
// phase B: (sharded) all-gather of the slot sums on `comm_stream`, then the class sums in class order on the main stream
static int gram_exchange(pio_als_handle* h, cudaStream_t comm_stream) {
  if (!gram_sharded(h)) return PIO_ALS_OK;
  const int n = h->KP * h->KP, my_groups = GRAM_GROUPS / h->cfg.world_size;
  const size_t cnt = (size_t)my_groups * n;
  if (nccl_api().AllGather(h->gram_gsum + (size_t)h->cfg.world_rank * cnt, h->gram_gsum, cnt, ncclDouble, h->comm, comm_stream) !=
      ncclSuccess)
    return fail(h, PIO_ALS_ERR_COMM, "ncclAllGather (YtY class sums) failed");
  return PIO_ALS_OK;
}
static int gram_reduce(pio_als_handle* h, const Side& s) {
  GramMap m;
  int my_groups, slot0;
  gram_layout(h, m, my_groups, slot0);
  const int n = h->KP * h->KP;
  gram_reduce_kernel<<<nblk(n, 256), 256, 0, h->stream>>>(h->gram_gsum, n, h->yty, m);
  LAUNCHED(h);
  CK(h, cudaGetLastError());
  h->gram_side = &s;
  return PIO_ALS_OK;
}

// One half-iteration: dst := argmin given src.  `more` = another half-step follows in this run: then YtY of the fresh dst
// factors is prepared here -- on 2 / 4 / 8 GPUs from the rank's own rows while the last pieces of the factor all-gather
// are still in flight, its 8 x KP^2 doubles exchanged on the communication stream right behind them.
static int half_step(pio_als_handle* h, Side& dst, const Side& src, bool more) {
  cudaStream_t st = h->stream;
  const bool implicit = h->cfg.implicit_prefs != 0;
  if (implicit && h->gram_side != &src) {     // first half-step of a run, or the factors were set from outside
    const EvPair e = next_ev(h, EV_GRAM);
    cudaEventRecord(e.a, st);
    int grc = gram_local(h, src);
    if (!grc) grc = gram_exchange(h, st);
    if (!grc) grc = gram_reduce(h, src);
    if (grc) return grc;
    cudaEventRecord(e.b, st);
  }
  {
    const EvPair e = next_ev(h, &dst == &h->U ? EV_SOLVE_USER : EV_SOLVE);
    cudaEventRecord(e.a, st);
    h->pieces_done = false;
    if (h->gram_side == &dst) h->gram_side = nullptr;
    CK(h, launch_solve(h, dst, src));
    cudaEventRecord(e.b, st);
  }
  const bool prep = implicit && more;
  bool gram_pending = false;      // class sums computed, exchange + reduce still to do
  if (h->cfg.world_size > 1) {
    NcclApi& nc = nccl_api();
    const int W = h->cfg.world_size, me = h->cfg.world_rank;
    const EvPair e = next_ev(h, EV_COMM);
    if (h->pieces_done && h->n_pieces > 1) {
      // all-gather piece by piece on the communication stream: piece c = local rows [R c / C, R (c + 1) / C) of every
      // rank, exchanged as soon as its rows are solved (grouped send/recv: NVSwitch gives every pair full bandwidth)
      cudaStream_t sc = h->comm_st;
      const int C = h->n_pieces;
      bool first = true;
      for (int c = 0; c < C; ++c) {
        const long long lo = (long long)dst.R * c / C, hi = (long long)dst.R * (c + 1) / C;
        if (hi <= lo) continue;
        cudaStreamWaitEvent(sc, h->ev_piece[c], 0);
        if (lo < dst.n_heavy) cudaStreamWaitEvent(sc, h->ev_heavy, 0);
        if (first) { cudaEventRecord(e.a, st); first = false; }   // comm time reported = what is NOT hidden behind the solve
        const size_t cnt = (size_t)(hi - lo) * h->KP;
        if (nc.GroupStart() != ncclSuccess) return fail(h, PIO_ALS_ERR_COMM, "ncclGroupStart failed");
        for (int p = 0; p < W; ++p) {
          if (p == me) continue;
          if (nc.Send(dst.F + ((size_t)me * dst.R + lo) * h->KP, cnt, ncclFloat, p, h->comm, sc) != ncclSuccess ||
              nc.Recv(dst.F + ((size_t)p * dst.R + lo) * h->KP, cnt, ncclFloat, p, h->comm, sc) != ncclSuccess)
            return fail(h, PIO_ALS_ERR_COMM, "ncclSend/ncclRecv (factor pieces) failed");
        }
        if (nc.GroupEnd() != ncclSuccess) return fail(h, PIO_ALS_ERR_COMM, "ncclGroupEnd failed");
      }
      if (prep && gram_sharded(h)) {
        // the rank's own rows are final on the main stream once the heavy-row finish has joined it
        if (dst.n_heavy > 0) cudaStreamWaitEvent(st, h->ev_heavy, 0);
        const EvPair g = next_ev(h, EV_GRAM);
        cudaEventRecord(g.a, st);
        const int grc = gram_local(h, dst);
        if (grc) return grc;
        cudaEventRecord(g.b, st);
        cudaEventRecord(h->ev_gram, st);
        cudaStreamWaitEvent(sc, h->ev_gram, 0);
        const int xrc = gram_exchange(h, sc);
        if (xrc) return xrc;
        gram_pending = true;
      }
      cudaEventRecord(e.b, sc);
      cudaEventRecord(h->ev_comm, sc);
      cudaStreamWaitEvent(st, h->ev_comm, 0);
    } else {
      cudaEventRecord(e.a, st);
      const size_t cnt = (size_t)dst.R * h->KP;
      ncclResult_t r = nc.AllGather(dst.F + (size_t)me * cnt, dst.F, cnt, ncclFloat, h->comm, st);
      if (r != ncclSuccess)
        return fail(h, PIO_ALS_ERR_COMM, "ncclAllGather failed: %s", nc.GetErrorString ? nc.GetErrorString(r) : "?");
      cudaEventRecord(e.b, st);
    }
  }
  if (prep) {
    const EvPair e = next_ev(h, EV_GRAM);
    cudaEventRecord(e.a, st);
    int grc = PIO_ALS_OK;
    if (!gram_pending) {
      grc = gram_local(h, dst);
      if (!grc) grc = gram_exchange(h, st);
    }
    if (!grc) grc = gram_reduce(h, dst);
    if (grc) return grc;
    cudaEventRecord(e.b, st);
  }
  return PIO_ALS_OK;
}

}  // namespace pio

// =============================================================================================
// C ABI
// =============================================================================================
extern "C" {

int pio_als_abi_version(void) { return PIO_ALS_ABI_VERSION; }

int pio_als_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) return PIO_ALS_ERR_CUDA;
  int ok = 0;
  for (int d = 0; d < n; ++d) {
    cudaDeviceProp pr;
    if (cudaGetDeviceProperties(&pr, d) == cudaSuccess && pr.major == 10) ++ok;
  }
  return ok;
}

int pio_als_nccl_unique_id(uint8_t out_id[128]) {
  NcclApi& a = nccl_api();
  if (!a.ok) return fail(nullptr, PIO_ALS_ERR_COMM, "libnccl.so.2 not loadable");
  ncclUniqueId id;
  if (a.GetUniqueId(&id) != ncclSuccess) return fail(nullptr, PIO_ALS_ERR_COMM, "ncclGetUniqueId failed");
  static_assert(sizeof(ncclUniqueId) == 128, "ncclUniqueId size");
  memcpy(out_id, &id, 128);
  return PIO_ALS_OK;
}

const char* pio_als_last_error(const pio_als_handle* h) { return h ? h->err.c_str() : g_create_error.c_str(); }

static int create_common(pio_als_handle* h) {
  int ndev = 0;
  cudaError_t ce = cudaGetDeviceCount(&ndev);
  if (ce != cudaSuccess || ndev == 0)
    return fail(nullptr, PIO_ALS_ERR_CUDA, "no CUDA device available (%s); this library has no CPU fallback",
                cudaGetErrorString(ce));
  if (h->cfg.device < 0 || h->cfg.device >= ndev) return fail(nullptr, PIO_ALS_ERR_ARG, "bad device %d", h->cfg.device);
  cudaDeviceProp pr;
  if (cudaGetDeviceProperties(&pr, h->cfg.device) != cudaSuccess) return fail(nullptr, PIO_ALS_ERR_CUDA, "cudaGetDeviceProperties");
  if (pr.major != 10)
    return fail(nullptr, PIO_ALS_ERR_CUDA, "device %d is sm_%d%d; this library is built for sm_100a (B200) only",
                h->cfg.device, pr.major, pr.minor);
  h->sm_count = pr.multiProcessorCount;
  h->st.sm_count = pr.multiProcessorCount;
  if (cudaSetDevice(h->cfg.device) != cudaSuccess) return fail(nullptr, PIO_ALS_ERR_CUDA, "cudaSetDevice");
  if (cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking) != cudaSuccess)
    return fail(nullptr, PIO_ALS_ERR_CUDA, "cudaStreamCreate");
  // keep freed blocks in the pool (ingest allocates and frees multi-GB scratch repeatedly)
  cudaMemPool_t pool;
  if (cudaDeviceGetDefaultMemPool(&pool, h->cfg.device) == cudaSuccess) {
    uint64_t thr = UINT64_MAX;
    cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &thr);
  }
  h->KP = pad_rank(h->cfg.rank);
  // the communication stream gets the highest priority: its few NCCL CTAs must not queue behind a grid that fills the
  // SMs (the YtY class sums run on the main stream next to the last pieces of the factor exchange)
  int prio_lo = 0, prio_hi = 0;
  cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi);
  if (cudaStreamCreateWithFlags(&h->aux, cudaStreamNonBlocking) != cudaSuccess ||
      cudaStreamCreateWithPriority(&h->comm_st, cudaStreamNonBlocking, prio_hi) != cudaSuccess)
    return fail(nullptr, PIO_ALS_ERR_CUDA, "cudaStreamCreate");
  {
    cudaEvent_t* evs[5] = {&h->ev_start, &h->ev_heavy, &h->ev_comm, &h->ev_gram, nullptr};
    for (int i = 0; evs[i]; ++i)
      if (cudaEventCreateWithFlags(evs[i], cudaEventDisableTiming) != cudaSuccess) return fail(nullptr, PIO_ALS_ERR_CUDA, "cudaEventCreate");
    for (int i = 0; i < 8; ++i)
      if (cudaEventCreateWithFlags(&h->ev_piece[i], cudaEventDisableTiming) != cudaSuccess) return fail(nullptr, PIO_ALS_ERR_CUDA, "cudaEventCreate");
    h->n_pieces = h->cfg.world_size > 1 ? 4 : 1;
    if (const char* v = getenv("PIO_ALS_SERVE_FUSED")) h->serve_fused = atoi(v) != 0;
    if (const char* v = getenv("PIO_ALS_SERVE_TRACE")) h->serve_trace = atoi(v) != 0;
    if (const char* v = getenv("PIO_ALS_SCORE_BLOCKED")) h->score_blocked = atoi(v) != 0;
    if (const char* v = getenv("PIO_ALS_PIECES")) {
      const int n = atoi(v);
      if (n >= 1 && n <= 8) h->n_pieces = n;
    }
  }
  {
    // Rank 33..64 kernel selection.  Default: the pair kernel (als_pair_kernel.cuh: mma.sync split-FP16 Gramian, two rows per
    // warp, lockstep Cholesky) for every side -- measured at C2 it is the fastest on both sides (user half-step 18.7 ms,
    // item half-step 12.9 ms vs 17.1 ms for the tcgen05 kernel) and, with rows above 1024 ratings summed in two
    // levels, inside the parity bound on long rows.  PIO_ALS_TC=1: the tcgen05 Gramian kernel (als_tc_kernel.cuh) for
    // every side (PIO_ALS_TC_MIN_DEG=n: only sides averaging >= n ratings per row); PIO_ALS_MMA=1: the round-1
    // one-warp-per-row mma.sync kernel; PIO_ALS_MMA=0: the FP32 CUDA-core kernel.
    const char* env = getenv("PIO_ALS_TC");
    h->use_tc = h->KP == 64 && env && env[0] == '1';
    h->tc_min_deg = 0.0;
    if (const char* md = getenv("PIO_ALS_TC_MIN_DEG")) h->tc_min_deg = atof(md);
    if (const char* sp = getenv("PIO_ALS_TC_SPLIT")) h->tc_split = sp[0] == '1';
    if (const char* mm_ = getenv("PIO_ALS_MMA")) {
      h->use_mma = mm_[0] != '0';
      h->use_pair = mm_[0] != '1';
    }
    if (const char* v = getenv("PIO_ALS_PAIR_WARPS")) h->pair_warps = atoi(v);
    if (const char* v = getenv("PIO_ALS_SEG_T")) h->pair_seg_t = atoi(v) > 0 ? atoi(v) : PAIR_SEG_T;
    if (const char* v = getenv("PIO_ALS_PART")) h->pair_part = atoi(v) >= 8 ? (atoi(v) + 7) / 8 * 8 : PAIR_PART;
  }
  h->gram_blocks = GRAM_GROUPS * h->sm_count;   // a sharded run gives every rank whole groups: one CTA per SM at 8 GPUs
  if (cudaMallocAsync((void**)&h->yty, sizeof(float) * h->KP * h->KP, h->stream) != cudaSuccess ||
      cudaMallocAsync((void**)&h->gram_partial, sizeof(double) * (size_t)h->gram_blocks * h->KP * h->KP, h->stream) != cudaSuccess ||
      cudaMallocAsync((void**)&h->gram_gsum, sizeof(double) * (size_t)GRAM_GROUPS * h->KP * h->KP, h->stream) != cudaSuccess ||
      cudaMallocAsync((void**)&h->d_fail, sizeof(int), h->stream) != cudaSuccess ||
      cudaMallocAsync((void**)&h->d_counts, 4 * sizeof(int), h->stream) != cudaSuccess)
    return fail(nullptr, PIO_ALS_ERR_CUDA, "device allocation failed");
  cudaMemsetAsync(h->yty, 0, sizeof(float) * h->KP * h->KP, h->stream);
  cudaMemsetAsync(h->d_fail, 0, sizeof(int), h->stream);
  return PIO_ALS_OK;
}

int pio_als_create(const pio_als_config* cfg, pio_als_handle** out) {
  if (!cfg || !out) return fail(nullptr, PIO_ALS_ERR_ARG, "null argument");
  *out = nullptr;
  if (cfg->abi_version != PIO_ALS_ABI_VERSION) return fail(nullptr, PIO_ALS_ERR_ARG, "abi_version mismatch");
  if (cfg->rank < 1 || cfg->rank > 128) return fail(nullptr, PIO_ALS_ERR_ARG, "rank must be in 1..128 (got %d)", cfg->rank);
  if (cfg->n_users < 1 || cfg->n_items < 1) return fail(nullptr, PIO_ALS_ERR_ARG, "n_users and n_items must be >= 1");
  if (cfg->world_size < 1 || cfg->world_rank < 0 || cfg->world_rank >= cfg->world_size)
    return fail(nullptr, PIO_ALS_ERR_ARG, "bad world_size/world_rank");
  if (!(cfg->lambda >= 0.0)) return fail(nullptr, PIO_ALS_ERR_ARG, "lambda must be >= 0");
  pio_als_handle* h = new pio_als_handle();
  h->cfg = *cfg;
  int rc = create_common(h);
  if (rc == PIO_ALS_OK && cfg->world_size > 1) {
    NcclApi& a = nccl_api();
    if (!a.ok) rc = fail(nullptr, PIO_ALS_ERR_COMM, "libnccl.so.2 not loadable");
    else {
      ncclUniqueId id;
      memcpy(&id, cfg->nccl_id, 128);
      ncclResult_t r = a.CommInitRank(&h->comm, cfg->world_size, id, cfg->world_rank);
      if (r != ncclSuccess) rc = fail(nullptr, PIO_ALS_ERR_COMM, "ncclCommInitRank failed: %s", a.GetErrorString ? a.GetErrorString(r) : "?");
    }
  }
  if (rc != PIO_ALS_OK) {
    pio_als_destroy(h);
    return rc;
  }
  *out = h;
  return PIO_ALS_OK;
}

void pio_als_destroy(pio_als_handle* h) {
  if (!h) return;
  if (h->stream) {
    cudaSetDevice(h->cfg.device);
    free_side(h, h->U, false);
    free_side(h, h->I, false);
    dfree(h, h->yty);
    dfree(h, h->gram_partial);
    dfree(h, h->gram_gsum);
    dfree(h, h->d_fail);
    dfree(h, h->d_counts);
    cudaStreamSynchronize(h->stream);
    if (h->tc_out) cudaFree(h->tc_out);
    if (h->d_dbg) cudaFree(h->d_dbg);
    if (h->d_timing) cudaFree(h->d_timing);
    for (auto& e : h->ev_pool) {
      cudaEventDestroy(e.a);
      cudaEventDestroy(e.b);
    }
    if (h->comm) nccl_api().CommDestroy(h->comm);
    if (h->ev_start) cudaEventDestroy(h->ev_start);
    if (h->ev_heavy) cudaEventDestroy(h->ev_heavy);
    if (h->ev_comm) cudaEventDestroy(h->ev_comm);
    if (h->ev_gram) cudaEventDestroy(h->ev_gram);
    for (int i = 0; i < 8; ++i)
      if (h->ev_piece[i]) cudaEventDestroy(h->ev_piece[i]);
    if (h->srv_dev) cudaFree(h->srv_dev);
    if (h->srv_host) cudaFreeHost(h->srv_host);
    if (h->srv_counter) cudaFree(h->srv_counter);
    if (h->aux) cudaStreamDestroy(h->aux);
    if (h->comm_st) cudaStreamDestroy(h->comm_st);
    cudaStreamDestroy(h->stream);
  }
  delete h;
}

static int set_ratings_impl(pio_als_handle* h, const int32_t* user, const int32_t* item, const float* rating, int64_t nnz,
                            int dedup_mode, const int64_t* ts, bool on_device, bool sharded) {
  if (!h) return PIO_ALS_ERR_ARG;
  const bool may_be_empty = sharded && h->cfg.world_size > 1;   // a rank's slice may be empty, the union may not
  if (nnz < 0 || (nnz == 0 && !may_be_empty))
    return fail(h, PIO_ALS_ERR_ARG, "ratings cannot be empty (the templates require(!ratings.take(1).isEmpty))");
  if (nnz > 0 && (!user || !item || !rating)) return fail(h, PIO_ALS_ERR_ARG, "null rating arrays");
  std::lock_guard<std::mutex> lk(h->mu);
  CK(h, cudaSetDevice(h->cfg.device));
  cudaStream_t st = h->stream;
  cudaEvent_t a, b;
  cudaEventCreate(&a);
  cudaEventCreate(&b);
  cudaEventRecord(a, st);
  int rc;
  {
    Scratch tmp(h);
    const int *du = user, *di = item;
    const float* dr = rating;
    const long long* dts = (const long long*)ts;
    auto stage = [&]() -> int {
      if (on_device || nnz == 0) return PIO_ALS_OK;
      int *tu = nullptr, *ti = nullptr;
      float* tr = nullptr;
      long long* tt = nullptr;
      CK(h, tmp.alloc(&tu, (size_t)nnz));
      CK(h, tmp.alloc(&ti, (size_t)nnz));
      CK(h, tmp.alloc(&tr, (size_t)nnz));
      CK(h, cudaMemcpyAsync(tu, user, sizeof(int) * nnz, cudaMemcpyHostToDevice, st));
      CK(h, cudaMemcpyAsync(ti, item, sizeof(int) * nnz, cudaMemcpyHostToDevice, st));
      CK(h, cudaMemcpyAsync(tr, rating, sizeof(float) * nnz, cudaMemcpyHostToDevice, st));
      if (ts && dedup_mode == PIO_ALS_DEDUP_KEEP_LAST) {
        CK(h, tmp.alloc(&tt, (size_t)nnz));
        CK(h, cudaMemcpyAsync(tt, ts, sizeof(long long) * nnz, cudaMemcpyHostToDevice, st));
      }
      du = tu; di = ti; dr = tr; dts = tt;
      return PIO_ALS_OK;
    };
    rc = stage();
    if (rc == PIO_ALS_OK) rc = ingest_device(h, du, di, dr, nnz, dedup_mode, dts, sharded);
  }
  cudaEventRecord(b, st);
  cudaEventSynchronize(b);
  float ms = 0;
  cudaEventElapsedTime(&ms, a, b);
  h->st.last_ingest_ms = ms;
  cudaEventDestroy(a);
  cudaEventDestroy(b);
  return rc;
}

int pio_als_set_ratings_coo_device(pio_als_handle* h, const int32_t* d_user, const int32_t* d_item,
                                   const float* d_rating, int64_t nnz, int dedup_mode, const int64_t* d_ts) {
  return set_ratings_impl(h, d_user, d_item, d_rating, nnz, dedup_mode, d_ts, true, false);
}

int pio_als_set_ratings_coo(pio_als_handle* h, const int32_t* user, const int32_t* item, const float* rating,
                            int64_t nnz, int dedup_mode, const int64_t* ts) {
  return set_ratings_impl(h, user, item, rating, nnz, dedup_mode, ts, false, false);
}

int pio_als_set_ratings_coo_sharded(pio_als_handle* h, const int32_t* user, const int32_t* item, const float* rating,
                                    int64_t nnz_local, int dedup_mode, const int64_t* ts) {
  return set_ratings_impl(h, user, item, rating, nnz_local, dedup_mode, ts, false, true);
}

int pio_als_set_ratings_coo_sharded_device(pio_als_handle* h, const int32_t* d_user, const int32_t* d_item,
                                           const float* d_rating, int64_t nnz_local, int dedup_mode, const int64_t* d_ts) {
  return set_ratings_impl(h, d_user, d_item, d_rating, nnz_local, dedup_mode, d_ts, true, true);
}

int pio_als_set_init(pio_als_handle* h, const float* user_factors, const float* item_factors) {
  if (!h) return PIO_ALS_ERR_ARG;
  std::lock_guard<std::mutex> lk(h->mu);
  if (!h->have_ratings) return fail(h, PIO_ALS_ERR_STATE, "set_init before set_ratings");
  if (!user_factors) return fail(h, PIO_ALS_ERR_ARG, "user_factors is null");
  CK(h, cudaSetDevice(h->cfg.device));
  cudaStream_t st = h->stream;
  const int k = h->cfg.rank;
  struct { Side* s; const float* f; } jobs[2] = {{&h->U, user_factors}, {&h->I, item_factors}};
  for (auto& j : jobs) {
    CK(h, cudaMemsetAsync(j.s->F, 0, sizeof(float) * (size_t)j.s->n_internal * h->KP, st));
    if (!j.f) continue;
    float* tmp = nullptr;
    CK(h, dalloc(h, &tmp, (size_t)j.s->n * k));
    CK(h, cudaMemcpyAsync(tmp, j.f, sizeof(float) * (size_t)j.s->n * k, cudaMemcpyHostToDevice, st));
    scatter_init_kernel<<<nblk((long long)j.s->n * h->KP, 256), 256, 0, st>>>(tmp, j.s->n, k, h->KP, j.s->perm, j.s->deg, j.s->F);
    LAUNCHED(h);
    dfree(h, tmp);
  }
  CK(h, cudaStreamSynchronize(st));
  h->have_init = true;
  return PIO_ALS_OK;
}

int pio_als_run(pio_als_handle* h, int n_iters) {
  if (!h) return PIO_ALS_ERR_ARG;
  std::lock_guard<std::mutex> lk(h->mu);
  if (!h->have_ratings) return fail(h, PIO_ALS_ERR_STATE, "run before set_ratings");
  if (n_iters < 0) return fail(h, PIO_ALS_ERR_ARG, "n_iters < 0");
  CK(h, cudaSetDevice(h->cfg.device));
  if (!h->have_init) {
    if (h->cfg.init_mode == PIO_ALS_INIT_HASH) {
      int rc = init_hash(h);
      if (rc) return rc;
    } else {
      return fail(h, PIO_ALS_ERR_STATE, "no initial factors: call pio_als_set_init or use PIO_ALS_INIT_HASH");
    }
  }
  cudaStream_t st = h->stream;
  h->ev_used = 0;
  CK(h, cudaMemsetAsync(h->d_fail, 0, sizeof(int), st));
  EvPair& tot = next_ev(h, -1);
  cudaEventRecord(tot.a, st);
  h->gram_side = nullptr;      // the factors may have been replaced since the last run
  for (int it = 0; it < n_iters; ++it) {
    int rc = half_step(h, h->I, h->U, true);                  // item factors from user factors
    if (rc) return rc;
    rc = half_step(h, h->U, h->I, it + 1 < n_iters);          // user factors from item factors
    if (rc) return rc;
  }
  cudaEventRecord(tot.b, st);
  int nfail = 0;
  CK(h, cudaMemcpyAsync(&nfail, h->d_fail, sizeof(int), cudaMemcpyDeviceToHost, st));
  CK(h, cudaStreamSynchronize(st));
  double ms[EV_NKIND] = {0, 0, 0, 0};
  float t = 0;
  for (size_t i = 0; i < h->ev_used; ++i) {
    EvPair& e = h->ev_pool[i];
    cudaEventElapsedTime(&t, e.a, e.b);
    if (e.kind >= 0) ms[e.kind] += t;
    else h->st.last_run_ms = t;
  }
  h->st.last_solve_ms = ms[EV_SOLVE] + ms[EV_SOLVE_USER];
  h->phase_ms[0] = ms[EV_SOLVE];
  h->phase_ms[1] = ms[EV_SOLVE_USER];
  h->phase_ms[2] = ms[EV_GRAM];
  h->phase_ms[3] = ms[EV_COMM];
  h->phase_ms[6] = (double)n_iters;
  h->st.last_gram_ms = ms[EV_GRAM];
  h->st.last_comm_ms = ms[EV_COMM];
  h->trained = true;
  if (nfail)
    return fail(h, PIO_ALS_ERR_NUMERIC, "%d normal equations were not positive definite (MLlib: dppsv info != 0)", nfail);
  return PIO_ALS_OK;
}

int pio_als_get_phase_ms(pio_als_handle* h, double out[8]) {
  if (!h || !out) return PIO_ALS_ERR_ARG;
  std::lock_guard<std::mutex> lk(h->mu);
  for (int i = 0; i < 8; ++i) out[i] = h->phase_ms[i];
  // kernel of the rows below the heavy-row threshold: 0 = FP32 (als_solve_kernel), 1 = tcgen05, 2 = mma.sync
  const bool mma = h->KP == 64 && h->use_mma;
  out[4] = h->I.use_tc ? 1.0 : h->I.use_pair ? 3.0 : (mma ? 2.0 : 0.0);
  out[5] = h->U.use_tc ? 1.0 : h->U.use_pair ? 3.0 : (mma ? 2.0 : 0.0);
  return PIO_ALS_OK;
}

int pio_als_get_factors(pio_als_handle* h, float* user_out, float* item_out, uint8_t* user_has, uint8_t* item_has) {
  if (!h) return PIO_ALS_ERR_ARG;
  std::lock_guard<std::mutex> lk(h->mu);
  if (!h->have_ratings && !h->trained) return fail(h, PIO_ALS_ERR_STATE, "no model");
  CK(h, cudaSetDevice(h->cfg.device));
  cudaStream_t st = h->stream;
  const int k = h->cfg.rank;
  struct { Side* s; float* f; uint8_t* has; } jobs[2] = {{&h->U, user_out, user_has}, {&h->I, item_out, item_has}};
  for (auto& j : jobs) {
    if (j.f) {
      float* tmp = nullptr;
      CK(h, dalloc(h, &tmp, (size_t)j.s->n * k));
      gather_factors_kernel<<<nblk((long long)j.s->n * k, 256), 256, 0, st>>>(j.s->F, j.s->n, k, h->KP, j.s->perm, tmp);
      LAUNCHED(h);
      CK(h, cudaMemcpyAsync(j.f, tmp, sizeof(float) * (size_t)j.s->n * k, cudaMemcpyDeviceToHost, st));
      dfree(h, tmp);
    }
    if (j.has) {
      uint8_t* tmp = nullptr;
      CK(h, dalloc(h, &tmp, (size_t)j.s->n));
      has_kernel<<<nblk(j.s->n, 256), 256, 0, st>>>(j.s->deg, j.s->n, tmp);
      LAUNCHED(h);
      CK(h, cudaMemcpyAsync(j.has, tmp, (size_t)j.s->n, cudaMemcpyDeviceToHost, st));
      dfree(h, tmp);
    }
  }
  CK(h, cudaStreamSynchronize(st));
  return PIO_ALS_OK;
}

int pio_als_train(pio_als_handle* h, const int32_t* user, const int32_t* item, const float* rating, int64_t nnz,
                  int dedup_mode, const int64_t* ts, const float* user_init, const float* item_init, int n_iters,
                  float* user_out, float* item_out, uint8_t* user_has, uint8_t* item_has) {
  int rc = pio_als_set_ratings_coo(h, user, item, rating, nnz, dedup_mode, ts);
  if (rc) return rc;
  if (user_init) {
    rc = pio_als_set_init(h, user_init, item_init);
    if (rc) return rc;
  }
  rc = pio_als_run(h, n_iters);
  if (rc) return rc;
  return pio_als_get_factors(h, user_out, item_out, user_has, item_has);
}

namespace pio {
static int serve_reserve(pio_als_handle* h, size_t dev_bytes, size_t host_bytes) {
  if (h->srv_dev_cap < dev_bytes) {
    CK(h, cudaStreamSynchronize(h->stream));
    if (h->srv_dev) cudaFree(h->srv_dev);
    h->srv_dev = nullptr;
    h->srv_dev_cap = 0;
    CK(h, cudaMalloc((void**)&h->srv_dev, dev_bytes));
    h->srv_dev_cap = dev_bytes;
  }
  if (h->srv_host_cap < host_bytes) {
    CK(h, cudaStreamSynchronize(h->stream));
    if (h->srv_host) cudaFreeHost(h->srv_host);
    h->srv_host = nullptr;
    h->srv_host_cap = 0;
    CK(h, cudaHostAlloc((void**)&h->srv_host, host_bytes, cudaHostAllocMapped));
    CK(h, cudaHostGetDevicePointer((void**)&h->srv_host_dev, h->srv_host, 0));
    h->srv_host_cap = host_bytes;
  }
  return PIO_ALS_OK;
}
static inline size_t al256(size_t x) { return (x + 255) & ~(size_t)255; }

extern "C++" {
template <int KPT>
static int launch_dot_blocked_kp(pio_als_handle* h, dim3 grid, size_t smem, const float* d_xq, const uint8_t* d_valid, int nq,
                                 const uint8_t* d_mask, const double* d_weight, int topk, ScoreIdx* d_cand) {
  static size_t attr_smem[64] = {};
  if (h->cfg.device < 64 && attr_smem[h->cfg.device] < smem) {
    CK(h, cudaFuncSetAttribute(score_dot_blocked_kernel<KPT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    attr_smem[h->cfg.device] = smem;
  }
  score_dot_blocked_kernel<KPT><<<grid, 32 * DB_WARPS, smem, h->stream>>>(h->I.F, h->I.n_internal, d_xq, d_valid, nq,
                                                                         h->I.cand_ext, d_mask, d_weight, topk, d_cand);
  return PIO_ALS_OK;
}
}  // extern "C++"
extern "C++" {
template <int KPT>
static int launch_cos_blocked_kp(pio_als_handle* h, dim3 grid, size_t smem, const float* d_qf, const int* d_bq0, const int* d_bv0,
                                 int n_bins, const int* d_vq, const long long* d_qptr, const int* d_qid, const uint8_t* d_mask,
                                 const double* d_weight, int keep, int topk, ScoreIdx* d_cand) {
  static size_t attr_smem[64] = {};
  if (h->cfg.device < 64 && attr_smem[h->cfg.device] < smem) {
    CK(h, cudaFuncSetAttribute(score_cos_blocked_kernel<KPT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    attr_smem[h->cfg.device] = smem;
  }
  score_cos_blocked_kernel<KPT><<<grid, 32 * DB_WARPS, smem, h->stream>>>(h->I.F, h->I.n_internal, h->cfg.rank, d_qf, d_bq0, d_bv0,
                                                                         n_bins, d_vq, d_qptr, d_qid, h->I.cand_ext, d_mask,
                                                                         d_weight, keep, topk, d_cand);
  return PIO_ALS_OK;
}
}  // extern "C++"
static int launch_cos_blocked(pio_als_handle* h, dim3 grid, size_t smem, const float* d_qf, const int* d_bq0, const int* d_bv0,
                              int n_bins, const int* d_vq, const long long* d_qptr, const int* d_qid, const uint8_t* d_mask,
                              const double* d_weight, int keep, int topk, ScoreIdx* d_cand) {
  if (h->KP == 16)
    return launch_cos_blocked_kp<16>(h, grid, smem, d_qf, d_bq0, d_bv0, n_bins, d_vq, d_qptr, d_qid, d_mask, d_weight, keep, topk, d_cand);
  if (h->KP == 32)
    return launch_cos_blocked_kp<32>(h, grid, smem, d_qf, d_bq0, d_bv0, n_bins, d_vq, d_qptr, d_qid, d_mask, d_weight, keep, topk, d_cand);
  return launch_cos_blocked_kp<64>(h, grid, smem, d_qf, d_bq0, d_bv0, n_bins, d_vq, d_qptr, d_qid, d_mask, d_weight, keep, topk, d_cand);
}
static int launch_dot_blocked(pio_als_handle* h, dim3 grid, size_t smem, const float* d_xq, const uint8_t* d_valid, int nq,
                              const uint8_t* d_mask, const double* d_weight, int topk, ScoreIdx* d_cand) {
  if (h->KP == 16) return launch_dot_blocked_kp<16>(h, grid, smem, d_xq, d_valid, nq, d_mask, d_weight, topk, d_cand);
  if (h->KP == 32) return launch_dot_blocked_kp<32>(h, grid, smem, d_xq, d_valid, nq, d_mask, d_weight, topk, d_cand);
  return launch_dot_blocked_kp<64>(h, grid, smem, d_xq, d_valid, nq, d_mask, d_weight, topk, d_cand);
}

// recommend for n <= SB_QB users and topk <= TK_MAXK: three launches and one synchronisation
static int recommend_small(pio_als_handle* h, const int32_t* users, int n, int topk, const uint8_t* item_mask,
                           const double* item_weight, int32_t* out_items, float* out_scores, int32_t* out_count) {
  cudaStream_t st = h->stream;
  const int KP = h->KP;
  const int ntiles = (h->I.n_internal + SB_THREADS - 1) / SB_THREADS;
  int gx = 2 * h->sm_count;
  if (gx > (ntiles + 7) / 8) gx = (ntiles + 7) / 8;
  if (gx < 1) gx = 1;
  const size_t o_xq = 0, o_valid = al256(o_xq + sizeof(float) * SB_QB * KP), o_cand = al256(o_valid + SB_QB),
               o_mask = al256(o_cand + sizeof(ScoreIdx) * (size_t)SB_QB * gx * topk),
               o_w = al256(o_mask + (item_mask ? (size_t)h->I.n : 0)),
               dev_bytes = al256(o_w + (item_weight ? sizeof(double) * (size_t)h->I.n : 0));
  const size_t ho_i = 0, ho_s = al256(sizeof(int) * (size_t)SB_QB * topk), ho_c = ho_s + al256(sizeof(float) * (size_t)SB_QB * topk),
               host_bytes = ho_c + al256(sizeof(int) * SB_QB);
  int rc = serve_reserve(h, dev_bytes, host_bytes);
  if (rc) return rc;
  float* d_xq = (float*)(h->srv_dev + o_xq);
  uint8_t* d_valid = h->srv_dev + o_valid;
  ScoreIdx* d_cand = (ScoreIdx*)(h->srv_dev + o_cand);
  uint8_t* d_mask = item_mask ? h->srv_dev + o_mask : nullptr;
  double* d_weight = item_weight ? (double*)(h->srv_dev + o_w) : nullptr;
  if (item_mask) CK(h, cudaMemcpyAsync(d_mask, item_mask, (size_t)h->I.n, cudaMemcpyHostToDevice, st));
  if (item_weight) CK(h, cudaMemcpyAsync(d_weight, item_weight, sizeof(double) * (size_t)h->I.n, cudaMemcpyHostToDevice, st));
  const size_t sb_smem = sizeof(double) * (size_t)KP * SB_QB + sb_tile_bytes(KP) + (sizeof(double) + sizeof(int)) * (size_t)SB_QB * topk;
  {
    static size_t attr_smem[64] = {};
    if (h->cfg.device < 64 && attr_smem[h->cfg.device] < sb_smem) {
      CK(h, cudaFuncSetAttribute(score_dot_topk_batched_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sb_smem));
      attr_smem[h->cfg.device] = sb_smem;
    }
  }
  IdList ids;
  for (int q = 0; q < n; ++q) ids.v[q] = users[q];
  gather_rows_ids_kernel<<<n, 64, 0, st>>>(h->U.F, KP, ids, h->U.perm, h->U.deg, h->U.n, d_xq, d_valid);
  LAUNCHED(h);
  score_dot_topk_batched_kernel<<<dim3(gx, 1), SB_THREADS, sb_smem, st>>>(h->I.F, h->I.n_internal, KP, d_xq, d_valid, n,
                                                                         h->I.cand_ext, d_mask, d_weight, nullptr, topk, d_cand);
  LAUNCHED(h);
  int* m_oi = (int*)(h->srv_host_dev + ho_i);
  float* m_os = (float*)(h->srv_host_dev + ho_s);
  int* m_oc = (int*)(h->srv_host_dev + ho_c);
  topk_merge_kernel<<<n, TK_THREADS, 0, st>>>(d_cand, gx * topk, topk, topk, 0, m_oi, m_os, m_oc, nullptr);
  LAUNCHED(h);
  CK(h, cudaStreamSynchronize(st));
  memcpy(out_items, h->srv_host + ho_i, sizeof(int) * (size_t)n * topk);
  memcpy(out_scores, h->srv_host + ho_s, sizeof(float) * (size_t)n * topk);
  if (out_count) memcpy(out_count, h->srv_host + ho_c, sizeof(int) * (size_t)n);
  return PIO_ALS_OK;
}

// one similar() query with nq <= SM_NV items and topk <= TK_MAXK: query items without a factor enter as zero vectors (their
// cosine terms are exactly 0, like the reference skipping them), so no host round trip is needed to compact the query
static int similar_small(pio_als_handle* h, const int32_t* query_items, int nq, int topk, const uint8_t* item_mask,
                         const double* item_weight, int flags, int32_t* out_items, float* out_scores, int32_t* out_count) {
  cudaStream_t st = h->stream;
  const int KP = h->KP, k = h->cfg.rank;
  const int ntiles = (h->I.n_internal + SB_THREADS - 1) / SB_THREADS;
  int gx = 2 * h->sm_count;
  if (gx > (ntiles + 7) / 8) gx = (ntiles + 7) / 8;
  if (gx < 1) gx = 1;
  const size_t o_qf = 0, o_cand = al256(sizeof(float) * SM_NV * KP), o_mask = al256(o_cand + sizeof(ScoreIdx) * (size_t)gx * topk),
               o_w = al256(o_mask + (item_mask ? (size_t)h->I.n : 0)),
               dev_bytes = al256(o_w + (item_weight ? sizeof(double) * (size_t)h->I.n : 0));
  // mapped host arena: results, then the tiny query description the kernel reads over PCIe
  const size_t ho_i = 0, ho_s = al256(sizeof(int) * (size_t)topk), ho_c = ho_s + al256(sizeof(float) * (size_t)topk),
               ho_g = ho_c + 256, ho_vq = ho_g + 256, ho_qp = ho_vq + 256, ho_qid = ho_qp + 256, host_bytes = ho_qid + 256;
  int rc = serve_reserve(h, dev_bytes, host_bytes);
  if (rc) return rc;
  float* d_qf = (float*)(h->srv_dev + o_qf);
  ScoreIdx* d_cand = (ScoreIdx*)(h->srv_dev + o_cand);
  uint8_t* d_mask = item_mask ? h->srv_dev + o_mask : nullptr;
  double* d_weight = item_weight ? (double*)(h->srv_dev + o_w) : nullptr;
  if (item_mask) CK(h, cudaMemcpyAsync(d_mask, item_mask, (size_t)h->I.n, cudaMemcpyHostToDevice, st));
  if (item_weight) CK(h, cudaMemcpyAsync(d_weight, item_weight, sizeof(double) * (size_t)h->I.n, cudaMemcpyHostToDevice, st));
  int* hg = (int*)(h->srv_host + ho_g);
  int* hvq = (int*)(h->srv_host + ho_vq);
  long long* hqp = (long long*)(h->srv_host + ho_qp);
  int* hqid = (int*)(h->srv_host + ho_qid);
  hg[0] = 0; hg[1] = nq;
  hqp[0] = 0; hqp[1] = nq;
  IdList ids;
  for (int q = 0; q < nq; ++q) { ids.v[q] = query_items[q]; hvq[q] = 0; hqid[q] = query_items[q]; }
  const size_t smem = sizeof(double) * ((size_t)KP * SM_NV + SM_NV) + sb_tile_bytes(KP) +
                      (sizeof(double) + sizeof(int)) * (size_t)SM_QG * topk + sizeof(int) * (SM_NV + SM_QG * SM_QIDS) + 16;
  {
    static size_t attr_smem[64] = {};
    if (h->cfg.device < 64 && attr_smem[h->cfg.device] < smem) {
      CK(h, cudaFuncSetAttribute(score_cos_topk_multi_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      attr_smem[h->cfg.device] = smem;
    }
  }
  gather_rows_ids_kernel<<<nq, 64, 0, st>>>(h->I.F, KP, ids, h->I.perm, h->I.deg, h->I.n, d_qf, nullptr);
  LAUNCHED(h);
  score_cos_topk_multi_kernel<<<dim3(gx, 1), SB_THREADS, smem, st>>>(
      h->I.F, h->I.n_internal, KP, k, d_qf, (const int*)(h->srv_host_dev + ho_g), (const int*)(h->srv_host_dev + ho_vq),
      (const long long*)(h->srv_host_dev + ho_qp), (const int*)(h->srv_host_dev + ho_qid), 1, h->I.cand_ext, d_mask, d_weight,
      nullptr, (flags & PIO_ALS_SIM_KEEP_QUERY_ITEMS) ? 1 : 0, topk, d_cand);
  LAUNCHED(h);
  topk_merge_kernel<<<1, TK_THREADS, 0, st>>>(d_cand, gx * topk, topk, topk, 0, (int*)(h->srv_host_dev + ho_i),
                                              (float*)(h->srv_host_dev + ho_s), (int*)(h->srv_host_dev + ho_c), nullptr);
  LAUNCHED(h);
  CK(h, cudaStreamSynchronize(st));
  memcpy(out_items, h->srv_host + ho_i, sizeof(int) * (size_t)topk);
  memcpy(out_scores, h->srv_host + ho_s, sizeof(float) * (size_t)topk);
  if (out_count) *out_count = *(int*)(h->srv_host + ho_c);
  return PIO_ALS_OK;
}

// ONE query in ONE launch (score_one_kernel): recommend for one user (cos = false, ids[0] = the user) or similar for
// nq <= S1_MAXNV query items.  The host waits on a sequence flag in the mapped arena instead of a stream synchronisation.
extern "C++" {
template <bool COS, int NVP, int KPT>
static void launch_score_one_kp(pio_als_handle* h, int gx, size_t smem, const Side& q, const OneQuery& qry, const uint8_t* d_mask,
                                const double* d_weight, int keep, int topk, ScoreIdx* d_cand, int* m_oi, float* m_os, int* m_oc,
                                unsigned* m_flag, unsigned seq, unsigned long long* m_trace) {
  static size_t attr_smem[64] = {};
  if (h->cfg.device < 64 && attr_smem[h->cfg.device] < smem) {
    cudaFuncSetAttribute(score_one_kernel<COS, NVP, KPT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    attr_smem[h->cfg.device] = smem;
  }
  unsigned long long* g_thr = reinterpret_cast<unsigned long long*>(h->srv_counter + 2);
  score_one_kernel<COS, NVP, KPT><<<gx, S1_THREADS, smem, h->stream>>>(
      h->I.F, h->I.n_internal, h->cfg.rank, q.F, q.perm, q.deg, q.n, qry, h->I.cand_ext, d_mask, d_weight, keep, topk, d_cand,
      h->srv_counter, g_thr, m_oi, m_os, m_oc, m_flag, seq, m_trace);
}
template <bool COS, int NVP>
static void launch_score_one(pio_als_handle* h, int gx, size_t smem, const Side& q, const OneQuery& qry, const uint8_t* d_mask,
                             const double* d_weight, int keep, int topk, ScoreIdx* d_cand, int* m_oi, float* m_os, int* m_oc,
                             unsigned* m_flag, unsigned seq, unsigned long long* m_trace) {
  if (h->KP == 16) launch_score_one_kp<COS, NVP, 16>(h, gx, smem, q, qry, d_mask, d_weight, keep, topk, d_cand, m_oi, m_os, m_oc, m_flag, seq, m_trace);
  else if (h->KP == 32) launch_score_one_kp<COS, NVP, 32>(h, gx, smem, q, qry, d_mask, d_weight, keep, topk, d_cand, m_oi, m_os, m_oc, m_flag, seq, m_trace);
  else launch_score_one_kp<COS, NVP, 64>(h, gx, smem, q, qry, d_mask, d_weight, keep, topk, d_cand, m_oi, m_os, m_oc, m_flag, seq, m_trace);
}
}  // extern "C++"

static bool serve_one_ok(const pio_als_handle* h, int nq, int topk) {
  return h->serve_fused && h->KP <= 64 && topk <= TK_MAXK && nq >= 1 && nq <= S1_MAXNV;
}

static int serve_one(pio_als_handle* h, bool cos, const int32_t* ids, int nq, int topk, const uint8_t* item_mask,
                     const double* item_weight, int flags, int32_t* out_items, float* out_scores, int32_t* out_count) {
  cudaStream_t st = h->stream;
  const int KP = h->KP;
  const int ntiles = (h->I.n_internal + S1_THREADS - 1) / S1_THREADS;
  int gx = h->sm_count < ntiles ? h->sm_count : ntiles;
  if (gx > S1_THREADS) gx = S1_THREADS;   // the list merge reads one list head per thread
  if (gx < 1) gx = 1;
  const int nvp = !cos ? 1 : nq <= 1 ? 1 : nq <= 2 ? 2 : nq <= 4 ? 4 : 8;
  const size_t o_cand = 0, o_mask = al256(sizeof(ScoreIdx) * (size_t)gx * topk),
               o_w = al256(o_mask + (item_mask ? (size_t)h->I.n : 0)),
               dev_bytes = al256(o_w + (item_weight ? sizeof(double) * (size_t)h->I.n : 0));
  const size_t ho_i = 0, ho_s = al256(sizeof(int) * (size_t)topk), ho_c = ho_s + al256(sizeof(float) * (size_t)topk),
               ho_flag = ho_c + 256, ho_trace = ho_flag + 256, host_bytes = ho_trace + 256;
  const bool fresh_host = h->srv_host_cap < host_bytes;
  int rc = serve_reserve(h, dev_bytes, host_bytes);
  if (rc) return rc;
  if (fresh_host) memset(h->srv_host, 0, h->srv_host_cap);
  if (!h->srv_counter) {
    CK(h, cudaMalloc((void**)&h->srv_counter, 256));
    CK(h, cudaMemsetAsync(h->srv_counter, 0, 256, st));
  }
  ScoreIdx* d_cand = (ScoreIdx*)(h->srv_dev + o_cand);
  uint8_t* d_mask = item_mask ? h->srv_dev + o_mask : nullptr;
  double* d_weight = item_weight ? (double*)(h->srv_dev + o_w) : nullptr;
  if (item_mask) CK(h, cudaMemcpyAsync(d_mask, item_mask, (size_t)h->I.n, cudaMemcpyHostToDevice, st));
  if (item_weight) CK(h, cudaMemcpyAsync(d_weight, item_weight, sizeof(double) * (size_t)h->I.n, cudaMemcpyHostToDevice, st));
  OneQuery qry;
  qry.nq = nq;
  for (int t = 0; t < S1_MAXNV; ++t) qry.ids[t] = t < nq ? ids[t] : -1;
  const unsigned seq = ++h->srv_seq ? h->srv_seq : ++h->srv_seq;   // never 0: a fresh arena reads 0
  volatile unsigned* flag = (volatile unsigned*)(h->srv_host + ho_flag);
  int* m_oi = (int*)(h->srv_host_dev + ho_i);
  float* m_os = (float*)(h->srv_host_dev + ho_s);
  int* m_oc = (int*)(h->srv_host_dev + ho_c);
  unsigned* m_flag = (unsigned*)(h->srv_host_dev + ho_flag);
  const size_t smem = s1_smem_bytes(KP, nvp, topk);
  const int keep = (flags & PIO_ALS_SIM_KEEP_QUERY_ITEMS) ? 1 : 0;
  const Side& q = cos ? h->I : h->U;
  unsigned long long* m_trace = h->serve_trace ? (unsigned long long*)(h->srv_host_dev + ho_trace) : nullptr;
  const auto t_call = std::chrono::steady_clock::now();
#define PIO_S1(C, N) launch_score_one<C, N>(h, gx, smem, q, qry, d_mask, d_weight, keep, topk, d_cand, m_oi, m_os, m_oc, m_flag, seq, m_trace)
  if (!cos) PIO_S1(false, 1);
  else if (nvp == 1) PIO_S1(true, 1);
  else if (nvp == 2) PIO_S1(true, 2);
  else if (nvp == 4) PIO_S1(true, 4);
  else PIO_S1(true, 8);
#undef PIO_S1
  LAUNCHED(h);
  CK(h, cudaGetLastError());
  for (unsigned spins = 1; *flag != seq; ++spins) {
    if ((spins & 0x3FFFu) == 0) {   // a faulted kernel never writes the flag: ask the stream now and then
      const cudaError_t e = cudaStreamQuery(st);
      if (e != cudaErrorNotReady) {
        if (e != cudaSuccess) CK(h, e);
        if (*flag != seq) return fail(h, PIO_ALS_ERR_CUDA, "single-query kernel finished without publishing its result");
      }
    }
#if defined(__x86_64__)
    __builtin_ia32_pause();
#endif
  }
  __atomic_thread_fence(__ATOMIC_ACQUIRE);
  if (h->serve_trace) {
    const unsigned long long* t = (const unsigned long long*)(h->srv_host + ho_trace);
    const double host_us = std::chrono::duration<double, std::micro>(std::chrono::steady_clock::now() - t_call).count();
    fprintf(stderr, "pio serve trace: host launch->flag %.1f us; publishing CTA: query lookup %.1f us, first step %.1f us, rest of the scan "
            "%.1f us, cta merge + arrival %.1f us, list merge %.1f us, system fence %.1f us\n", host_us, (t[5] - t[0]) * 1e-3,
            (t[6] - t[5]) * 1e-3, (t[1] - t[6]) * 1e-3, (t[2] - t[1]) * 1e-3, (t[3] - t[2]) * 1e-3, (t[4] - t[3]) * 1e-3);
  }
  memcpy(out_items, h->srv_host + ho_i, sizeof(int) * (size_t)topk);
  memcpy(out_scores, h->srv_host + ho_s, sizeof(float) * (size_t)topk);
  if (out_count) *out_count = *(int*)(h->srv_host + ho_c);
  return PIO_ALS_OK;
}
}  // namespace pio

// Scoring passes: at most TK_MAXK results per pass; a query asking for more runs further passes, each bounded by the last
// result of the one before (topk.cuh below_bound).
int pio_als_recommend(pio_als_handle* h, const int32_t* users, int n, int topk, const uint8_t* item_mask,
                      const double* item_weight, int32_t* out_items, float* out_scores, int32_t* out_count) {
  if (!h) return PIO_ALS_ERR_ARG;
  if (n < 0 || topk < 1) return fail(h, PIO_ALS_ERR_ARG, "topk must be >= 1 and n >= 0");
  if (n == 0) return PIO_ALS_OK;
  if (!users || !out_items || !out_scores) return fail(h, PIO_ALS_ERR_ARG, "null argument");
  std::lock_guard<std::mutex> lk(h->mu);
  if (!h->U.F || !h->I.F || !h->I.cand_ext) return fail(h, PIO_ALS_ERR_STATE, "no model");
  CK(h, cudaSetDevice(h->cfg.device));
  if (n == 1 && serve_one_ok(h, 1, topk))   // the serving case: one query, one launch
    return serve_one(h, false, users, 1, topk, item_mask, item_weight, 0, out_items, out_scores, out_count);
  if (n <= SB_QB && topk <= TK_MAXK)   // a few queries
    return recommend_small(h, users, n, topk, item_mask, item_weight, out_items, out_scores, out_count);
  cudaStream_t st = h->stream;
  const int KP = h->KP;
  Scratch tmp(h);
  int* d_users = nullptr;
  float* d_xq = nullptr;
  uint8_t *d_valid = nullptr, *d_mask = nullptr;
  double* d_weight = nullptr;
  ScoreIdx *d_cand = nullptr, *d_bound = nullptr;
  int *d_oi = nullptr, *d_oc = nullptr;
  float* d_os = nullptr;
  const int pass_max = topk < TK_MAXK ? topk : TK_MAXK;
  // batched scoring: groups of SB_QB queries share every staged item tile; GX persistent CTAs per group
  const int ngroups = (n + SB_QB - 1) / SB_QB;
  const int ntiles = (h->I.n_internal + SB_THREADS - 1) / SB_THREADS;
  int gx = (2 * h->sm_count + ngroups - 1) / ngroups;
  if (gx > (ntiles + 7) / 8) gx = (ntiles + 7) / 8;   // at least eight tiles per CTA: the pools must warm up
  if (gx < 1) gx = 1;
  const size_t sb_smem = sizeof(double) * (size_t)KP * SB_QB + sb_tile_bytes(KP) +
                         (sizeof(double) + sizeof(int)) * (size_t)SB_QB * pass_max;
  {
    static size_t attr_smem[64] = {};
    if (h->cfg.device < 64 && attr_smem[h->cfg.device] < sb_smem) {
      CK(h, cudaFuncSetAttribute(score_dot_topk_batched_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sb_smem));
      attr_smem[h->cfg.device] = sb_smem;
    }
  }
  // blocked kernel (two items x 16 queries per thread, independent warps): rank <= 64, topk <= DB_MAXK
  const bool blocked = h->score_blocked && KP <= 64 && topk <= DB_MAXK;
  if (blocked) {
    const int nsteps = (h->I.n_internal + DB_RINGS * DB_ROWS - 1) / (DB_RINGS * DB_ROWS);
    gx = (h->sm_count + ngroups - 1) / ngroups;
    if (gx > (nsteps + 7) / 8) gx = (nsteps + 7) / 8;   // at least eight steps per warp: the pools must warm up
    if (gx < 1) gx = 1;
  }
  const int lists = blocked ? gx * DB_RINGS : gx;        // candidate lists per query
  CK(h, tmp.alloc(&d_users, (size_t)n));
  CK(h, tmp.alloc(&d_xq, (size_t)n * KP));
  CK(h, tmp.alloc(&d_valid, (size_t)n));
  CK(h, tmp.alloc(&d_cand, (size_t)n * lists * pass_max));
  CK(h, tmp.alloc(&d_oi, (size_t)n * topk));
  CK(h, tmp.alloc(&d_os, (size_t)n * topk));
  CK(h, tmp.alloc(&d_oc, (size_t)n));
  CK(h, cudaMemcpyAsync(d_users, users, sizeof(int) * n, cudaMemcpyHostToDevice, st));
  if (item_mask) {
    CK(h, tmp.alloc(&d_mask, (size_t)h->I.n));
    CK(h, cudaMemcpyAsync(d_mask, item_mask, (size_t)h->I.n, cudaMemcpyHostToDevice, st));
  }
  if (item_weight) {
    CK(h, tmp.alloc(&d_weight, (size_t)h->I.n));
    CK(h, cudaMemcpyAsync(d_weight, item_weight, sizeof(double) * (size_t)h->I.n, cudaMemcpyHostToDevice, st));
  }
  if (topk > TK_MAXK) CK(h, tmp.alloc(&d_bound, (size_t)n));
  gather_rows_kernel<<<n, 64, 0, st>>>(h->U.F, KP, d_users, n, h->U.perm, h->U.deg, h->U.n, d_xq, d_valid);
  LAUNCHED(h);
  for (int done = 0; done < topk; done += TK_MAXK) {
    const int pk = topk - done < TK_MAXK ? topk - done : TK_MAXK;
    // grid.y is limited to 65535 query groups per launch
    for (int g0 = 0; g0 < ngroups; g0 += 32768) {
      const int ng = ngroups - g0 < 32768 ? ngroups - g0 : 32768;
      const int q0 = g0 * SB_QB;
      const int nq = n - q0 < ng * SB_QB ? n - q0 : ng * SB_QB;
      if (blocked) {
        const size_t smem = db_smem_bytes(KP, pk);
        const int brc = launch_dot_blocked(h, dim3(gx, ng), smem, d_xq + (size_t)q0 * KP, d_valid + q0, nq, d_mask, d_weight, pk,
                                           d_cand + (size_t)q0 * lists * pk);
        if (brc) return brc;
      } else {
        score_dot_topk_batched_kernel<<<dim3(gx, ng), SB_THREADS, sb_smem, st>>>(
            h->I.F, h->I.n_internal, KP, d_xq + (size_t)q0 * KP, d_valid + q0, nq, h->I.cand_ext, d_mask, d_weight,
            (done > 0) ? d_bound + q0 : nullptr, pk, d_cand + (size_t)q0 * lists * pk);
      }
      LAUNCHED(h);
    }
    // the candidate lists of a query are [lists][pk] entries, stored with stride pk
    topk_merge_kernel<<<n, TK_THREADS, 0, st>>>(d_cand, lists * pk, pk, topk, done, d_oi, d_os, d_oc, d_bound);
    LAUNCHED(h);
  }
  CK(h, cudaMemcpyAsync(out_items, d_oi, sizeof(int) * (size_t)n * topk, cudaMemcpyDeviceToHost, st));
  CK(h, cudaMemcpyAsync(out_scores, d_os, sizeof(float) * (size_t)n * topk, cudaMemcpyDeviceToHost, st));
  if (out_count) CK(h, cudaMemcpyAsync(out_count, d_oc, sizeof(int) * (size_t)n, cudaMemcpyDeviceToHost, st));
  CK(h, cudaStreamSynchronize(st));
  return PIO_ALS_OK;
}

namespace pio {
// one similar() query with mask / weights already on the device; results to HOST out arrays (topk entries)
static int similar_one(pio_als_handle* h, const int32_t* query_items, int nq, int topk, const uint8_t* d_mask,
                       const double* d_weight, int flags, int32_t* out_items, float* out_scores, int32_t* out_count) {
  for (int t = 0; t < topk; ++t) { out_items[t] = -1; out_scores[t] = 0.f; }
  if (out_count) *out_count = 0;
  if (nq == 0) return PIO_ALS_OK;
  cudaStream_t st = h->stream;
  const int KP = h->KP, k = h->cfg.rank;
  const int keep_query = (flags & PIO_ALS_SIM_KEEP_QUERY_ITEMS) ? 1 : 0;
  Scratch tmp(h);
  int* d_q = nullptr;
  float* d_qf = nullptr;
  uint8_t* d_valid = nullptr;
  CK(h, tmp.alloc(&d_q, (size_t)nq));
  CK(h, tmp.alloc(&d_qf, (size_t)nq * KP));
  CK(h, tmp.alloc(&d_valid, (size_t)nq));
  CK(h, cudaMemcpyAsync(d_q, query_items, sizeof(int) * nq, cudaMemcpyHostToDevice, st));
  gather_rows_kernel<<<nq, 64, 0, st>>>(h->I.F, KP, d_q, nq, h->I.perm, h->I.deg, h->I.n, d_qf, d_valid);
  LAUNCHED(h);
  std::vector<uint8_t> valid(nq);
  CK(h, cudaMemcpyAsync(valid.data(), d_valid, (size_t)nq, cudaMemcpyDeviceToHost, st));
  CK(h, cudaStreamSynchronize(st));
  // compact the query vectors that own a factor (order preserved); all query ids stay excluded
  std::vector<int> keep;
  for (int q = 0; q < nq; ++q)
    if (valid[q]) keep.push_back(q);
  if (keep.empty()) return PIO_ALS_OK;
  float* d_qc = nullptr;
  CK(h, tmp.alloc(&d_qc, keep.size() * (size_t)KP));
  for (size_t j = 0; j < keep.size(); ++j)
    CK(h, cudaMemcpyAsync(d_qc + j * KP, d_qf + (size_t)keep[j] * KP, sizeof(float) * KP, cudaMemcpyDeviceToDevice, st));
  const int pass_max = topk < TK_MAXK ? topk : TK_MAXK;
  // batched kernel (query vectors resident in shared memory) unless the query is too large for it
  const int nqv = (int)keep.size();
  const int nqp = (nqv + SC_G - 1) / SC_G * SC_G;
  constexpr int SC_WARPS = SB_THREADS / 32;   // one candidate pool per warp
  const size_t sc_smem = sizeof(double) * ((size_t)KP * nqp + nqp) + sizeof(float) * (size_t)SB_THREADS * (KP + 4) +
                         (sizeof(double) + sizeof(int)) * (size_t)SC_WARPS * pass_max + sizeof(int) * (size_t)nq + 16;
  const bool batched = sc_smem <= 100 * 1024;
  int ntiles = (h->I.n_internal + TK_TILE - 1) / TK_TILE;
  if (batched) {
    const int nt = (h->I.n_internal + SB_THREADS - 1) / SB_THREADS;
    ntiles = 2 * h->sm_count < (nt + 7) / 8 ? 2 * h->sm_count : (nt + 7) / 8;   // = CTAs (>= 8 tiles each)
    static size_t attr_smem[64] = {};
    if (h->cfg.device < 64 && attr_smem[h->cfg.device] < sc_smem) {
      CK(h, cudaFuncSetAttribute(score_cos_topk_batched_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sc_smem));
      attr_smem[h->cfg.device] = sc_smem;
    }
  }
  ScoreIdx *d_cand = nullptr, *d_bound = nullptr;
  int *d_oi = nullptr, *d_oc = nullptr;
  float* d_os = nullptr;
  const int npools = batched ? ntiles * SC_WARPS : ntiles;   // candidate lists of pass_k entries left for the merge
  CK(h, tmp.alloc(&d_cand, (size_t)npools * pass_max));
  CK(h, tmp.alloc(&d_oi, (size_t)topk));
  CK(h, tmp.alloc(&d_os, (size_t)topk));
  CK(h, tmp.alloc(&d_oc, 1));
  if (topk > TK_MAXK) CK(h, tmp.alloc(&d_bound, 1));
  for (int done = 0; done < topk; done += TK_MAXK) {
    const int pk = topk - done < TK_MAXK ? topk - done : TK_MAXK;
    const ScoreIdx* bnd = done > 0 ? d_bound : nullptr;
    if (batched)
      score_cos_topk_batched_kernel<<<ntiles, SB_THREADS, sc_smem, st>>>(h->I.F, h->I.n_internal, KP, k, d_qc, d_q, nq, nqv,
                                                                         h->I.cand_ext, d_mask, d_weight, bnd, keep_query, pk,
                                                                         d_cand);
    else
      score_cos_topk_kernel<<<ntiles, TK_THREADS, 0, st>>>(h->I.F, h->I.n_internal, KP, k, d_qc, d_q, nq, nqv, h->I.cand_ext,
                                                           d_mask, d_weight, bnd, keep_query, pk, d_cand);
    LAUNCHED(h);
    topk_merge_kernel<<<1, TK_THREADS, 0, st>>>(d_cand, npools * pk, pk, topk, done, d_oi, d_os, d_oc, d_bound);
    LAUNCHED(h);
  }
  CK(h, cudaMemcpyAsync(out_items, d_oi, sizeof(int) * topk, cudaMemcpyDeviceToHost, st));
  CK(h, cudaMemcpyAsync(out_scores, d_os, sizeof(float) * topk, cudaMemcpyDeviceToHost, st));
  int cnt = 0;
  CK(h, cudaMemcpyAsync(&cnt, d_oc, sizeof(int), cudaMemcpyDeviceToHost, st));
  CK(h, cudaStreamSynchronize(st));
  if (out_count) *out_count = cnt;
  return PIO_ALS_OK;
}
}  // namespace pio

int pio_als_similar_batch(pio_als_handle* h, const int64_t* q_ptr, const int32_t* q_items, int n_queries, int topk,
                          const uint8_t* item_mask, const double* item_weight, int flags, int32_t* out_items,
                          float* out_scores, int32_t* out_count) {
  if (!h) return PIO_ALS_ERR_ARG;
  if (n_queries < 0 || topk < 1) return fail(h, PIO_ALS_ERR_ARG, "topk must be >= 1 and n_queries >= 0");
  if (n_queries == 0) return PIO_ALS_OK;
  if (!q_ptr || !out_items || !out_scores) return fail(h, PIO_ALS_ERR_ARG, "null argument");
  for (int j = 0; j < n_queries; ++j)
    if (q_ptr[j + 1] < q_ptr[j] || (q_ptr[j + 1] > q_ptr[j] && !q_items))
      return fail(h, PIO_ALS_ERR_ARG, "q_ptr must be non-decreasing offsets into q_items");
  std::lock_guard<std::mutex> lk(h->mu);
  if (!h->I.F || !h->I.cand_ext) return fail(h, PIO_ALS_ERR_STATE, "no model");
  CK(h, cudaSetDevice(h->cfg.device));
  if (n_queries == 1 && serve_one_ok(h, (int)std::min<long long>(q_ptr[1] - q_ptr[0], 1 << 20), topk))   // the serving case
    return serve_one(h, true, q_items + q_ptr[0], (int)(q_ptr[1] - q_ptr[0]), topk, item_mask, item_weight, flags, out_items,
                     out_scores, out_count);
  if (n_queries == 1 && q_ptr[1] - q_ptr[0] >= 1 && q_ptr[1] - q_ptr[0] <= SM_NV && topk <= TK_MAXK)
    return similar_small(h, q_items + q_ptr[0], (int)(q_ptr[1] - q_ptr[0]), topk, item_mask, item_weight, flags, out_items,
                         out_scores, out_count);
  Scratch tmp(h);
  uint8_t* d_mask = nullptr;
  double* d_weight = nullptr;
  if (item_mask) {
    CK(h, tmp.alloc(&d_mask, (size_t)h->I.n));
    CK(h, cudaMemcpyAsync(d_mask, item_mask, (size_t)h->I.n, cudaMemcpyHostToDevice, h->stream));
  }
  if (item_weight) {
    CK(h, tmp.alloc(&d_weight, (size_t)h->I.n));
    CK(h, cudaMemcpyAsync(d_weight, item_weight, sizeof(double) * (size_t)h->I.n, cudaMemcpyHostToDevice, h->stream));
  }
  cudaStream_t st = h->stream;
  const int KP = h->KP, k = h->cfg.rank;
  const long long total = q_ptr[n_queries] - q_ptr[0];
  bool fast = n_queries > 1 && total > 0 && total < (1ll << 31);
  std::vector<int> gvec0, vq, vsrc;
  if (fast) {
    // all query item vectors in one gather; which of them own a factor decides the vector list of every query
    int* d_qid = nullptr;
    float* d_qf_all = nullptr;
    uint8_t* d_valid = nullptr;
    CK(h, tmp.alloc(&d_qid, (size_t)total));
    CK(h, tmp.alloc(&d_qf_all, (size_t)total * KP));
    CK(h, tmp.alloc(&d_valid, (size_t)total));
    CK(h, cudaMemcpyAsync(d_qid, q_items + q_ptr[0], sizeof(int) * total, cudaMemcpyHostToDevice, st));
    gather_rows_kernel<<<(unsigned)total, 64, 0, st>>>(h->I.F, KP, d_qid, (int)total, h->I.perm, h->I.deg, h->I.n, d_qf_all, d_valid);
    LAUNCHED(h);
    std::vector<uint8_t> valid((size_t)total);
    CK(h, cudaMemcpyAsync(valid.data(), d_valid, (size_t)total, cudaMemcpyDeviceToHost, st));
    CK(h, cudaStreamSynchronize(st));
    // blocked kernel: bins of <= CB_QPW consecutive queries and <= DB_QW query vectors per warp (rank <= 64, topk <= DB_MAXK)
    if (h->score_blocked && KP <= 64 && topk <= DB_MAXK) {
      std::vector<int> bin_q0, bin_v0, bvq, bvsrc;
      bool ok = true;
      int bq = 0, bv = 0;      // queries / vectors in the open bin
      bin_q0.push_back(0);
      bin_v0.push_back(0);
      for (int j = 0; j < n_queries && ok; ++j) {
        int nvq = 0;
        for (long long t = q_ptr[j]; t < q_ptr[j + 1]; ++t) nvq += valid[(size_t)(t - q_ptr[0])] ? 1 : 0;
        if (nvq > DB_QW) { ok = false; break; }
        if (bq == CB_QPW || bv + nvq > DB_QW) {
          bin_q0.push_back(j);
          bin_v0.push_back((int)bvsrc.size());
          bq = bv = 0;
        }
        for (long long t = q_ptr[j]; t < q_ptr[j + 1]; ++t)
          if (valid[(size_t)(t - q_ptr[0])]) {
            bvsrc.push_back((int)(t - q_ptr[0]));
            bvq.push_back(j);
          }
        ++bq;
        bv += nvq;
      }
      if (ok) {
        bin_q0.push_back(n_queries);
        bin_v0.push_back((int)bvsrc.size());
        const int n_bins = (int)bin_q0.size() - 1, nvec = (int)bvsrc.size();
        const int ngroups = (n_bins + DB_WPR - 1) / DB_WPR;
        int *d_bq0 = nullptr, *d_bv0 = nullptr, *d_vq = nullptr, *d_vsrc = nullptr, *d_oi = nullptr, *d_oc = nullptr;
        long long* d_qptr = nullptr;
        float *d_qfc = nullptr, *d_os = nullptr;
        ScoreIdx* d_cand = nullptr;
        std::vector<long long> rel((size_t)n_queries + 1);
        for (int j = 0; j <= n_queries; ++j) rel[j] = q_ptr[j] - q_ptr[0];
        CK(h, tmp.alloc(&d_bq0, bin_q0.size()));
        CK(h, tmp.alloc(&d_bv0, bin_v0.size()));
        CK(h, tmp.alloc(&d_vq, (size_t)(nvec > 0 ? nvec : 1)));
        CK(h, tmp.alloc(&d_vsrc, (size_t)(nvec > 0 ? nvec : 1)));
        CK(h, tmp.alloc(&d_qptr, rel.size()));
        CK(h, tmp.alloc(&d_qfc, (size_t)(nvec > 0 ? nvec : 1) * KP));
        CK(h, cudaMemcpyAsync(d_bq0, bin_q0.data(), sizeof(int) * bin_q0.size(), cudaMemcpyHostToDevice, st));
        CK(h, cudaMemcpyAsync(d_bv0, bin_v0.data(), sizeof(int) * bin_v0.size(), cudaMemcpyHostToDevice, st));
        CK(h, cudaMemcpyAsync(d_qptr, rel.data(), sizeof(long long) * rel.size(), cudaMemcpyHostToDevice, st));
        if (nvec > 0) {
          CK(h, cudaMemcpyAsync(d_vq, bvq.data(), sizeof(int) * nvec, cudaMemcpyHostToDevice, st));
          CK(h, cudaMemcpyAsync(d_vsrc, bvsrc.data(), sizeof(int) * nvec, cudaMemcpyHostToDevice, st));
          copy_rows_kernel<<<nvec, 64, 0, st>>>(d_qf_all, KP, d_vsrc, d_qfc);
          LAUNCHED(h);
        }
        const int nsteps = (h->I.n_internal + DB_RINGS * DB_ROWS - 1) / (DB_RINGS * DB_ROWS);
        int gx = (h->sm_count + ngroups - 1) / ngroups;
        if (gx > (nsteps + 7) / 8) gx = (nsteps + 7) / 8;
        if (gx < 1) gx = 1;
        const int lists = gx * DB_RINGS;
        CK(h, tmp.alloc(&d_cand, (size_t)n_queries * lists * topk));
        CK(h, tmp.alloc(&d_oi, (size_t)n_queries * topk));
        CK(h, tmp.alloc(&d_os, (size_t)n_queries * topk));
        CK(h, tmp.alloc(&d_oc, (size_t)n_queries));
        const int keep_query = (flags & PIO_ALS_SIM_KEEP_QUERY_ITEMS) ? 1 : 0;
        const size_t smem = db_smem_bytes(KP, topk);
        for (int g0 = 0; g0 < ngroups; g0 += 32768) {
          const int ng = ngroups - g0 < 32768 ? ngroups - g0 : 32768;
          const int brc = launch_cos_blocked(h, dim3(gx, ng), smem, d_qfc, d_bq0 + (size_t)g0 * DB_WPR, d_bv0 + (size_t)g0 * DB_WPR,
                                             n_bins - g0 * DB_WPR, d_vq, d_qptr, d_qid, d_mask, d_weight, keep_query, topk, d_cand);
          if (brc) return brc;
          LAUNCHED(h);
        }
        topk_merge_kernel<<<n_queries, TK_THREADS, 0, st>>>(d_cand, lists * topk, topk, topk, 0, d_oi, d_os, d_oc, nullptr);
        LAUNCHED(h);
        CK(h, cudaMemcpyAsync(out_items, d_oi, sizeof(int) * (size_t)n_queries * topk, cudaMemcpyDeviceToHost, st));
        CK(h, cudaMemcpyAsync(out_scores, d_os, sizeof(float) * (size_t)n_queries * topk, cudaMemcpyDeviceToHost, st));
        if (out_count) CK(h, cudaMemcpyAsync(out_count, d_oc, sizeof(int) * (size_t)n_queries, cudaMemcpyDeviceToHost, st));
        CK(h, cudaStreamSynchronize(st));
        return PIO_ALS_OK;
      }
    }
    const int ngroups = (n_queries + SM_QG - 1) / SM_QG;
    gvec0.assign((size_t)ngroups + 1, 0);
    for (int g = 0; g < ngroups && fast; ++g) {
      gvec0[g] = (int)vsrc.size();
      for (int j = g * SM_QG; j < (g + 1) * SM_QG && j < n_queries; ++j)
        for (long long t = q_ptr[j]; t < q_ptr[j + 1]; ++t)
          if (valid[(size_t)(t - q_ptr[0])]) {
            vsrc.push_back((int)(t - q_ptr[0]));
            vq.push_back(j - g * SM_QG);
          }
      if ((int)vsrc.size() - gvec0[g] > SM_NV) fast = false;   // a group with too many query vectors: one query at a time
    }
    gvec0[ngroups] = (int)vsrc.size();
    if (fast) {
      const int nvec = (int)vsrc.size();
      int *d_gvec0 = nullptr, *d_vq = nullptr, *d_vsrc = nullptr, *d_oi = nullptr, *d_oc = nullptr;
      long long* d_qptr = nullptr;
      float *d_qfc = nullptr, *d_os = nullptr;
      ScoreIdx *d_cand = nullptr, *d_bound = nullptr;
      std::vector<long long> rel((size_t)n_queries + 1);
      for (int j = 0; j <= n_queries; ++j) rel[j] = q_ptr[j] - q_ptr[0];
      CK(h, tmp.alloc(&d_gvec0, gvec0.size()));
      CK(h, tmp.alloc(&d_vq, (size_t)(nvec > 0 ? nvec : 1)));
      CK(h, tmp.alloc(&d_vsrc, (size_t)(nvec > 0 ? nvec : 1)));
      CK(h, tmp.alloc(&d_qptr, rel.size()));
      CK(h, tmp.alloc(&d_qfc, (size_t)(nvec > 0 ? nvec : 1) * KP));
      CK(h, cudaMemcpyAsync(d_gvec0, gvec0.data(), sizeof(int) * gvec0.size(), cudaMemcpyHostToDevice, st));
      CK(h, cudaMemcpyAsync(d_qptr, rel.data(), sizeof(long long) * rel.size(), cudaMemcpyHostToDevice, st));
      if (nvec > 0) {
        CK(h, cudaMemcpyAsync(d_vq, vq.data(), sizeof(int) * nvec, cudaMemcpyHostToDevice, st));
        CK(h, cudaMemcpyAsync(d_vsrc, vsrc.data(), sizeof(int) * nvec, cudaMemcpyHostToDevice, st));
        copy_rows_kernel<<<nvec, 64, 0, st>>>(d_qf_all, KP, d_vsrc, d_qfc);
        LAUNCHED(h);
      }
      const int pass_max = topk < TK_MAXK ? topk : TK_MAXK;
      const int ntiles = (h->I.n_internal + SB_THREADS - 1) / SB_THREADS;
      int gx = (2 * h->sm_count + ngroups - 1) / ngroups;
      if (gx > (ntiles + 7) / 8) gx = (ntiles + 7) / 8;
      if (gx < 1) gx = 1;
      const size_t smem = sizeof(double) * ((size_t)KP * SM_NV + SM_NV) + sb_tile_bytes(KP) +
                          (sizeof(double) + sizeof(int)) * (size_t)SM_QG * pass_max + sizeof(int) * (SM_NV + SM_QG * SM_QIDS) + 16;
      {
        static size_t attr_smem[64] = {};
        if (h->cfg.device < 64 && attr_smem[h->cfg.device] < smem) {
          CK(h, cudaFuncSetAttribute(score_cos_topk_multi_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
          attr_smem[h->cfg.device] = smem;
        }
      }
      CK(h, tmp.alloc(&d_cand, (size_t)n_queries * gx * pass_max));
      CK(h, tmp.alloc(&d_oi, (size_t)n_queries * topk));
      CK(h, tmp.alloc(&d_os, (size_t)n_queries * topk));
      CK(h, tmp.alloc(&d_oc, (size_t)n_queries));
      if (topk > TK_MAXK) CK(h, tmp.alloc(&d_bound, (size_t)n_queries));
      const int keep_query = (flags & PIO_ALS_SIM_KEEP_QUERY_ITEMS) ? 1 : 0;
      for (int done = 0; done < topk; done += TK_MAXK) {
        const int pk = topk - done < TK_MAXK ? topk - done : TK_MAXK;
        for (int g0 = 0; g0 < ngroups; g0 += 32768) {
          const int ng = ngroups - g0 < 32768 ? ngroups - g0 : 32768;
          const int qa = g0 * SM_QG;
          const int nq = n_queries - qa < ng * SM_QG ? n_queries - qa : ng * SM_QG;
          score_cos_topk_multi_kernel<<<dim3(gx, ng), SB_THREADS, smem, st>>>(
              h->I.F, h->I.n_internal, KP, k, d_qfc, d_gvec0 + g0, d_vq, d_qptr + qa, d_qid, nq, h->I.cand_ext, d_mask,
              d_weight, done > 0 ? d_bound + qa : nullptr, keep_query, pk, d_cand + (size_t)qa * gx * pk);
          LAUNCHED(h);
        }
        topk_merge_kernel<<<n_queries, TK_THREADS, 0, st>>>(d_cand, gx * pk, pk, topk, done, d_oi, d_os, d_oc, d_bound);
        LAUNCHED(h);
      }
      CK(h, cudaMemcpyAsync(out_items, d_oi, sizeof(int) * (size_t)n_queries * topk, cudaMemcpyDeviceToHost, st));
      CK(h, cudaMemcpyAsync(out_scores, d_os, sizeof(float) * (size_t)n_queries * topk, cudaMemcpyDeviceToHost, st));
      if (out_count) CK(h, cudaMemcpyAsync(out_count, d_oc, sizeof(int) * (size_t)n_queries, cudaMemcpyDeviceToHost, st));
      CK(h, cudaStreamSynchronize(st));
      return PIO_ALS_OK;
    }
  }
  for (int j = 0; j < n_queries; ++j) {
    int32_t cnt = 0;
    const int rc = similar_one(h, q_items + q_ptr[j], (int)(q_ptr[j + 1] - q_ptr[j]), topk, d_mask, d_weight, flags,
                               out_items + (size_t)j * topk, out_scores + (size_t)j * topk, &cnt);
    if (rc) return rc;
    if (out_count) out_count[j] = cnt;
  }
  CK(h, cudaStreamSynchronize(h->stream));
  return PIO_ALS_OK;
}

int pio_als_similar(pio_als_handle* h, const int32_t* query_items, int nq, int topk, const uint8_t* item_mask,
                    const double* item_weight, int flags, int32_t* out_items, float* out_scores, int32_t* out_count) {
  if (!h) return PIO_ALS_ERR_ARG;
  if (nq < 0) return fail(h, PIO_ALS_ERR_ARG, "nq < 0");
  const int64_t ptr[2] = {0, nq};
  return pio_als_similar_batch(h, ptr, query_items, 1, topk, item_mask, item_weight, flags, out_items, out_scores, out_count);
}

// ---- persistence ------------------------------------------------------------------------------
struct ModelHeader {
  char magic[8];
  int32_t version, rank, implicit_prefs, n_users, n_items, reserved;
  double lambda, alpha;
};

int pio_als_save(pio_als_handle* h, const char* path) {
  if (!h || !path) return PIO_ALS_ERR_ARG;
  try {
    const size_t nu = h->cfg.n_users, ni = h->cfg.n_items, k = h->cfg.rank;
    std::vector<float> uf(nu * k), itf(ni * k);
    std::vector<uint8_t> uh(nu), ih(ni);
    int rc = pio_als_get_factors(h, uf.data(), itf.data(), uh.data(), ih.data());
    if (rc) return rc;
    FILE* f = fopen(path, "wb");
    if (!f) return fail(h, PIO_ALS_ERR_IO, "cannot open %s for writing", path);
    ModelHeader hd{};
    memcpy(hd.magic, "PIOALS01", 8);
    hd.version = 1;
    hd.rank = h->cfg.rank;
    hd.implicit_prefs = h->cfg.implicit_prefs;
    hd.n_users = h->cfg.n_users;
    hd.n_items = h->cfg.n_items;
    hd.lambda = h->cfg.lambda;
    hd.alpha = h->cfg.alpha;
    bool ok = fwrite(&hd, sizeof hd, 1, f) == 1 && fwrite(uh.data(), 1, nu, f) == nu && fwrite(ih.data(), 1, ni, f) == ni &&
              fwrite(uf.data(), sizeof(float), nu * k, f) == nu * k && fwrite(itf.data(), sizeof(float), ni * k, f) == ni * k;
    ok = (fclose(f) == 0) && ok;
    return ok ? PIO_ALS_OK : fail(h, PIO_ALS_ERR_IO, "short write to %s", path);
  } catch (const std::exception& e) {   // bad_alloc etc. must not cross the C boundary
    return fail(h, PIO_ALS_ERR_IO, "pio_als_save: %s", e.what());
  }
}

__global__ void load_side_kernel(const uint8_t* has, int n, int* perm, int* inv, uint32_t* deg, uint32_t* npos) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= n) return;
  perm[r] = r;
  inv[r] = r;
  deg[r] = (!has || has[r]) ? 1u : 0u;
  npos[r] = deg[r];
}

int pio_als_model_import(const pio_als_config* cfg_in, const float* user_factors, const float* item_factors,
                         const uint8_t* user_has, const uint8_t* item_has, pio_als_handle** out) {
  if (!cfg_in || !out) return fail(nullptr, PIO_ALS_ERR_ARG, "null argument");
  *out = nullptr;
  if (!item_factors) return fail(nullptr, PIO_ALS_ERR_ARG, "item_factors is null");
  pio_als_config cfg = *cfg_in;
  cfg.world_size = 1;
  cfg.world_rank = 0;
  const bool item_only = cfg.n_users == 0 && !user_factors;
  if (item_only) cfg.n_users = 1;   // an item-only model (similarproduct) carries one factor-less placeholder user
  else if (!user_factors) return fail(nullptr, PIO_ALS_ERR_ARG, "user_factors is null but n_users > 0");
  pio_als_handle* h = nullptr;
  int rc = pio_als_create(&cfg, &h);
  if (rc) return rc;
  cudaStream_t st = h->stream;
  const size_t k = (size_t)cfg.rank;
  const uint8_t zero = 0;
  struct { Side* s; size_t n; const uint8_t* has; const float* fac; } jobs[2] = {
      {&h->U, (size_t)cfg.n_users, item_only ? &zero : user_has, user_factors}, {&h->I, (size_t)cfg.n_items, item_has, item_factors}};
  auto body = [&]() -> int {
    for (auto& j : jobs) {
      Side& s = *j.s;
      s.n = (int)j.n;
      s.R = s.n;
      s.n_internal = s.n;
      s.bits = ceil_log2((uint64_t)s.n);
      CK(h, dalloc(h, &s.perm, j.n)); CK(h, dalloc(h, &s.inv, j.n)); CK(h, dalloc(h, &s.deg, j.n));
      CK(h, dalloc(h, &s.npos, j.n)); CK(h, dalloc(h, &s.cand_ext, j.n));
      CK(h, dalloc(h, &s.F, j.n * (size_t)h->KP));
      Scratch tmp(h);
      uint8_t* dh = nullptr;
      float* dfac = nullptr;
      if (j.has) {
        CK(h, tmp.alloc(&dh, j.n));
        CK(h, cudaMemcpyAsync(dh, j.has, j.n, cudaMemcpyHostToDevice, st));
      }
      load_side_kernel<<<nblk(s.n, 256), 256, 0, st>>>(dh, s.n, s.perm, s.inv, s.deg, s.npos);
      LAUNCHED(h);
      if (j.fac) {
        CK(h, tmp.alloc(&dfac, j.n * k));
        CK(h, cudaMemcpyAsync(dfac, j.fac, sizeof(float) * j.n * k, cudaMemcpyHostToDevice, st));
        scatter_init_kernel<<<nblk((long long)s.n * h->KP, 256), 256, 0, st>>>(dfac, s.n, (int)k, h->KP, s.perm, s.deg, s.F);
        LAUNCHED(h);
      } else {
        CK(h, cudaMemsetAsync(s.F, 0, sizeof(float) * j.n * (size_t)h->KP, st));
      }
      cand_ext_kernel<<<nblk(s.n, 256), 256, 0, st>>>(s.inv, s.deg, s.n, s.cand_ext);
      LAUNCHED(h);
      CK(h, cudaStreamSynchronize(st));   // the host sources may go away after this call
    }
    return PIO_ALS_OK;
  };
  rc = body();
  if (rc) {
    g_create_error = h->err;
    pio_als_destroy(h);
    return rc;
  }
  h->trained = true;
  *out = h;
  return PIO_ALS_OK;
}

int pio_als_load(const char* path, int device, pio_als_handle** out) {
  if (!path || !out) return fail(nullptr, PIO_ALS_ERR_ARG, "null argument");
  *out = nullptr;
  FILE* f = fopen(path, "rb");
  if (!f) return fail(nullptr, PIO_ALS_ERR_IO, "cannot open %s", path);
  ModelHeader hd;
  if (fread(&hd, sizeof hd, 1, f) != 1 || memcmp(hd.magic, "PIOALS01", 8) != 0 || hd.version != 1) {
    fclose(f);
    return fail(nullptr, PIO_ALS_ERR_IO, "%s is not a PIOALS01 model file", path);
  }
  // a corrupt header must not turn into a huge allocation: check the fields and the file size first
  if (hd.rank < 1 || hd.rank > 128 || hd.n_users < 1 || hd.n_items < 1) {
    fclose(f);
    return fail(nullptr, PIO_ALS_ERR_IO, "%s: corrupt header (rank %d, %d users, %d items)", path, hd.rank, hd.n_users, hd.n_items);
  }
  const size_t nu = hd.n_users, ni = hd.n_items, k = hd.rank;
  const long long expect = (long long)sizeof hd + (long long)(nu + ni) + (long long)sizeof(float) * (long long)((nu + ni) * k);
  if (fseek(f, 0, SEEK_END) != 0 || ftell(f) != expect || fseek(f, (long)sizeof hd, SEEK_SET) != 0) {
    fclose(f);
    return fail(nullptr, PIO_ALS_ERR_IO, "%s is truncated or has trailing bytes (expected %lld bytes)", path, expect);
  }
  try {
    std::vector<float> uf(nu * k), itf(ni * k);
    std::vector<uint8_t> uh(nu), ih(ni);
    bool ok = fread(uh.data(), 1, nu, f) == nu && fread(ih.data(), 1, ni, f) == ni &&
              fread(uf.data(), sizeof(float), nu * k, f) == nu * k && fread(itf.data(), sizeof(float), ni * k, f) == ni * k;
    fclose(f);
    f = nullptr;
    if (!ok) return fail(nullptr, PIO_ALS_ERR_IO, "%s is truncated", path);
    pio_als_config cfg{};
    cfg.abi_version = PIO_ALS_ABI_VERSION;
    cfg.rank = hd.rank;
    cfg.implicit_prefs = hd.implicit_prefs;
    cfg.n_users = hd.n_users;
    cfg.n_items = hd.n_items;
    cfg.device = device;
    cfg.world_size = 1;
    cfg.lambda = hd.lambda;
    cfg.alpha = hd.alpha;
    return pio_als_model_import(&cfg, uf.data(), itf.data(), uh.data(), ih.data(), out);
  } catch (const std::exception& e) {
    if (f) fclose(f);
    return fail(nullptr, PIO_ALS_ERR_IO, "pio_als_load: %s", e.what());
  }
}

/* debug only (not in pio_als.h): copies the A/b dump of the last tensor-core half-step (rows in internal order) */
__attribute__((visibility("default"))) int pio_als_debug_dump(pio_als_handle* h, float* out, long long n_floats) {
  if (!h || !h->d_dbg) return PIO_ALS_ERR_STATE;
  cudaStreamSynchronize(h->stream);
  size_t n = h->dbg_rows * (tc::ASLOT + tc::KP);
  if ((size_t)n_floats < n) n = (size_t)n_floats;
  return cudaMemcpy(out, h->d_dbg, n * sizeof(float), cudaMemcpyDeviceToHost) == cudaSuccess ? PIO_ALS_OK : PIO_ALS_ERR_CUDA;
}

__attribute__((visibility("default"))) int pio_als_debug_timing(pio_als_handle* h, long long* out, long long n) {
  if (!h || !h->d_timing) return PIO_ALS_ERR_STATE;
  cudaStreamSynchronize(h->stream);
  size_t m = (size_t)h->sm_count * 16 * 8;
  if ((size_t)n < m) m = (size_t)n;
  return cudaMemcpy(out, h->d_timing, m * sizeof(long long), cudaMemcpyDeviceToHost) == cudaSuccess ? PIO_ALS_OK : PIO_ALS_ERR_CUDA;
}

#define CK0(call)                                                                                         \
  do {                                                                                                    \
    cudaError_t e_ = (call);                                                                              \
    if (e_ != cudaSuccess) return fail(nullptr, PIO_ALS_ERR_CUDA, "%s failed: %s", #call, cudaGetErrorString(e_)); \
  } while (0)

/* debug only (not in pio_als.h): the lockstep Cholesky of als_lockstep.cuh on n dense SPD systems (A: n x N x N
 * row-major, b: n x N; HOST buffers), N = 64 or 128; x = (A + ridge I)^-1 b.  reps > 1 repeats fill + solve for timing
 * (ms_out = device time of the launch).  Used by tests/test_gpu_lockstep.py and tools/bench_solver.py. */
extern "C++" {
template <int N>
__global__ void __launch_bounds__(32) lockstep_probe_kernel(const float* __restrict__ A, const float* __restrict__ b, int n,
                                                            float ridge, float* __restrict__ x, int reps, int* fail) {
  using LL = LsLayout<N>;
  constexpr int LANES = N / 4, NM = 32 / LANES;
  extern __shared__ __align__(16) float sm[];
  float* bvec = sm + NM * LL::STRIDE;
  float* colbuf = bvec + NM * 80 + (N > 64 ? N : 0);
  const int lane = threadIdx.x & 31, grp = lane / LANES;
  for (int base = blockIdx.x * NM; base < n; base += gridDim.x * NM) {
    for (int rep = 0; rep < reps; ++rep) {
      for (int m = 0; m < NM; ++m) {
        const int mi = base + m;
        float* slot = sm + m * LL::STRIDE;
        for (int o = lane; o < N * N; o += 32) {
          const int r = o / N, c = o % N;
          if (c <= r) slot[LL::at(r, c)] = mi < n ? A[(size_t)mi * N * N + o] : (r == c ? 1.f : 0.f);
        }
        for (int o = lane; o < N; o += 32) bvec[m * (N > 64 ? N : 80) + o] = mi < n ? b[(size_t)mi * N + o] : 0.f;
      }
      __syncwarp();
      const int mine = base + grp;
      chol_lockstep<N, false>(sm + grp * LL::STRIDE, bvec + grp * (N > 64 ? N : 80), nullptr, ridge, N, colbuf + grp * 80,
                              x + (size_t)(mine < n ? mine : 0) * N, mine < n, fail);
      __syncwarp();
    }
  }
}
}  // extern "C++"

__attribute__((visibility("default"))) int pio_als_debug_lockstep(int device, int N, int n, const float* A, const float* b,
                                                                  float ridge, float* x, int reps, float* ms_out,
                                                                  int* fail_out) {
  if ((N != 64 && N != 128) || n < 1 || !A || !b || !x) return PIO_ALS_ERR_ARG;
  CK0(cudaSetDevice(device));
  float *dA = nullptr, *db = nullptr, *dx = nullptr;
  int* dfail = nullptr;
  CK0(cudaMalloc((void**)&dA, sizeof(float) * (size_t)n * N * N));
  CK0(cudaMalloc((void**)&db, sizeof(float) * (size_t)n * N));
  CK0(cudaMalloc((void**)&dx, sizeof(float) * (size_t)n * N));
  CK0(cudaMalloc((void**)&dfail, sizeof(int)));
  CK0(cudaMemset(dfail, 0, sizeof(int)));
  CK0(cudaMemcpy(dA, A, sizeof(float) * (size_t)n * N * N, cudaMemcpyHostToDevice));
  CK0(cudaMemcpy(db, b, sizeof(float) * (size_t)n * N, cudaMemcpyHostToDevice));
  const int nm = N == 64 ? 2 : 1;
  const size_t smem = sizeof(float) * (size_t)(nm * (N == 64 ? LsLayout<64>::STRIDE : LsLayout<128>::STRIDE) + 2 * 80 + 2 * 80 + 256);
  cudaDeviceProp pr_;
  CK0(cudaGetDeviceProperties(&pr_, device));
  int grid = (n + nm - 1) / nm;
  const int cap = pr_.multiProcessorCount * (N == 64 ? 12 : 6);
  if (grid > cap) grid = cap;
  cudaEvent_t e0, e1;
  cudaEventCreate(&e0);
  cudaEventCreate(&e1);
  if (N == 64) {
    CK0(cudaFuncSetAttribute(lockstep_probe_kernel<64>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    CK0(cudaFuncSetAttribute(lockstep_probe_kernel<64>, cudaFuncAttributePreferredSharedMemoryCarveout, 100));
    cudaEventRecord(e0);
    lockstep_probe_kernel<64><<<grid, 32, smem>>>(dA, db, n, ridge, dx, reps < 1 ? 1 : reps, dfail);
  } else {
    CK0(cudaFuncSetAttribute(lockstep_probe_kernel<128>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    CK0(cudaFuncSetAttribute(lockstep_probe_kernel<128>, cudaFuncAttributePreferredSharedMemoryCarveout, 100));
    cudaEventRecord(e0);
    lockstep_probe_kernel<128><<<grid, 32, smem>>>(dA, db, n, ridge, dx, reps < 1 ? 1 : reps, dfail);
  }
  cudaEventRecord(e1);
  CK0(cudaDeviceSynchronize());
  float ms = 0.f;
  cudaEventElapsedTime(&ms, e0, e1);
  if (ms_out) *ms_out = ms;
  CK0(cudaMemcpy(x, dx, sizeof(float) * (size_t)n * N, cudaMemcpyDeviceToHost));
  if (fail_out) CK0(cudaMemcpy(fail_out, dfail, sizeof(int), cudaMemcpyDeviceToHost));
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  cudaFree(dA); cudaFree(db); cudaFree(dx); cudaFree(dfail);
  return PIO_ALS_OK;
}

int pio_als_get_stats(const pio_als_handle* h, pio_als_stats* out) {
  if (!h || !out) return PIO_ALS_ERR_ARG;
  *out = h->st;
  return PIO_ALS_OK;
}

int pio_als_synth_ratings_device(int device, int32_t n_users, int32_t n_items, int64_t nnz, int64_t seed, int implicit,
                                 int64_t start, int32_t* d_user, int32_t* d_item, float* d_rating) {
  if (cudaSetDevice(device) != cudaSuccess) return fail(nullptr, PIO_ALS_ERR_CUDA, "cudaSetDevice(%d) failed", device);
  if (nnz <= 0) return PIO_ALS_OK;
  synth_kernel<<<nblk(nnz, 256), 256>>>(n_users, n_items, nnz, (uint64_t)seed, implicit, start, d_user, d_item, d_rating);
  cudaError_t e = cudaDeviceSynchronize();
  if (e != cudaSuccess) return fail(nullptr, PIO_ALS_ERR_CUDA, "synth kernel: %s", cudaGetErrorString(e));
  return PIO_ALS_OK;
}

// ---- string ids -> dense indices (BiMap.stringInt) ---------------------------------------------------------------------
int pio_ids_encode(int device, const uint8_t* bytes, const int64_t* offsets, int64_t n, int32_t* out_index,
                   int64_t* out_first, int32_t* out_n_unique) {
  if (n < 0 || !offsets || !out_index || !out_n_unique || (n > 0 && !bytes && offsets[n] > offsets[0]))
    return fail(nullptr, PIO_ALS_ERR_ARG, "bad pio_ids_encode arguments");
  *out_n_unique = 0;
  if (n == 0) return PIO_ALS_OK;
  if (n >= (1ll << 32)) return fail(nullptr, PIO_ALS_ERR_ARG, "n must be < 2^32");
  if (offsets[0] != 0) return fail(nullptr, PIO_ALS_ERR_ARG, "offsets[0] must be 0");
  CK0(cudaSetDevice(device));
  const size_t nb = (size_t)offsets[n];
  uint8_t* d_bytes = nullptr;
  long long *d_off = nullptr, *d_first = nullptr;
  uint64_t *ka = nullptr, *kb = nullptr;
  uint32_t *va = nullptr, *vb = nullptr, *f1 = nullptr, *f2 = nullptr, *run_start = nullptr, *head = nullptr, *ishead = nullptr,
           *firstpos = nullptr, *isfirst = nullptr;
  int* d_out = nullptr;
  std::vector<void*> owned;
  auto A = [&](void** p, size_t bytes_) -> cudaError_t {
    cudaError_t e = cudaMalloc(p, bytes_ ? bytes_ : 1);
    if (e == cudaSuccess) owned.push_back(*p);
    return e;
  };
  struct Guard { std::vector<void*>& v; ~Guard() { for (void* q : v) cudaFree(q); } } guard{owned};
  CK0(A((void**)&d_bytes, nb));
  CK0(A((void**)&d_off, sizeof(long long) * (n + 1)));
  CK0(A((void**)&ka, 8 * (size_t)n)); CK0(A((void**)&kb, 8 * (size_t)n));
  CK0(A((void**)&va, 4 * (size_t)n)); CK0(A((void**)&vb, 4 * (size_t)n));
  CK0(A((void**)&f1, 4 * (size_t)n)); CK0(A((void**)&f2, 4 * (size_t)n));
  CK0(A((void**)&run_start, 4 * (size_t)n)); CK0(A((void**)&head, 4 * (size_t)n)); CK0(A((void**)&ishead, 4 * (size_t)n));
  CK0(A((void**)&firstpos, 4 * (size_t)n)); CK0(A((void**)&isfirst, 4 * (size_t)n));
  CK0(A((void**)&d_out, 4 * (size_t)n));
  CK0(A((void**)&d_first, 8 * (size_t)n));
  cudaStream_t st = 0;
  CK0(cudaMemcpyAsync(d_bytes, bytes, nb, cudaMemcpyHostToDevice, st));
  CK0(cudaMemcpyAsync(d_off, offsets, sizeof(long long) * (n + 1), cudaMemcpyHostToDevice, st));
  uint64_t mask = ~0ull;
  if (const char* hb = getenv("PIO_IDS_HASH_BITS")) {   // tests: a short hash makes different strings collide on purpose
    const int b = atoi(hb);
    if (b >= 1 && b < 64) mask = (1ull << b) - 1ull;
  }
  ids_hash_kernel<<<nblk(n, 256), 256, 0, st>>>(d_bytes, d_off, n, ka, va, mask);
  bool in_b = false;
  CK0(radix_sort_pairs(ka, va, kb, vb, (size_t)n, 64, st, &in_b, nullptr));
  const uint64_t* ks = in_b ? kb : ka;
  const uint32_t* vs = in_b ? vb : va;
  ids_runflag_kernel<<<nblk(n, 256), 256, 0, st>>>(ks, n, f1);
  CK0(scan_exclusive_u32(f1, f1, (size_t)n, st, nullptr));                 // f1 = run ids
  ids_runstart_kernel<<<nblk(n, 256), 256, 0, st>>>(ks, f1, n, run_start);
  ids_head_kernel<<<nblk(n, 256), 256, 0, st>>>(ks, vs, f1, run_start, d_bytes, d_off, n, head, ishead);
  uint32_t last_flag = 0, last_ex = 0;
  CK0(cudaMemcpyAsync(&last_flag, ishead + n - 1, 4, cudaMemcpyDeviceToHost, st));
  CK0(scan_exclusive_u32(ishead, f2, (size_t)n, st, nullptr));             // f2 = group ids (valid at heads)
  CK0(cudaMemcpyAsync(&last_ex, f2 + n - 1, 4, cudaMemcpyDeviceToHost, st));
  CK0(cudaMemsetAsync(isfirst, 0, 4 * (size_t)n, st));
  ids_firstpos_kernel<<<nblk(n, 256), 256, 0, st>>>(vs, ishead, f2, n, firstpos, isfirst);
  CK0(scan_exclusive_u32(isfirst, isfirst, (size_t)n, st, nullptr));       // ids by first occurrence
  ids_assign_kernel<<<nblk(n, 256), 256, 0, st>>>(vs, head, isfirst, n, d_out, out_first ? d_first : nullptr);
  CK0(cudaMemcpyAsync(out_index, d_out, 4 * (size_t)n, cudaMemcpyDeviceToHost, st));
  CK0(cudaStreamSynchronize(st));
  const int64_t nuniq = (int64_t)last_ex + last_flag;
  if (out_first) CK0(cudaMemcpy(out_first, d_first, 8 * (size_t)nuniq, cudaMemcpyDeviceToHost));
  *out_n_unique = (int32_t)nuniq;
  return PIO_ALS_OK;
}

// ---- item co-occurrence (similarproduct CooccurrenceAlgorithm) ------------------------------------------------------------
int pio_cooc_train(int device, const int32_t* user, const int32_t* item, int64_t n, int32_t n_users, int32_t n_items,
                   int topn, int32_t* out_item, int32_t* out_count, int32_t* out_n) {
  if (!user || !item || !out_item || !out_count || !out_n || n < 1 || n_users < 1 || n_items < 1 || topn < 1)
    return fail(nullptr, PIO_ALS_ERR_ARG, "bad pio_cooc_train arguments");
  if (n >= (1ll << 32)) return fail(nullptr, PIO_ALS_ERR_ARG, "n must be < 2^32");
  for (int64_t e = 0; e < n; ++e)
    if (user[e] < 0 || user[e] >= n_users || item[e] < 0 || item[e] >= n_items)
      return fail(nullptr, PIO_ALS_ERR_ARG, "event %lld has a user/item index out of range", (long long)e);
  CK0(cudaSetDevice(device));
  const int bits_u = ceil_log2((uint64_t)n_users), bits_i = ceil_log2((uint64_t)n_items);
  if (2 * bits_i > 40) return fail(nullptr, PIO_ALS_ERR_ARG, "n_items too large for the pair keys (max 2^20 items)");
  const int bits_c = 64 - 2 * bits_i > 32 ? 32 : 64 - 2 * bits_i;
  std::vector<void*> owned;
  auto A = [&](void** p, size_t bytes_) -> cudaError_t {
    cudaError_t e = cudaMalloc(p, bytes_ ? bytes_ : 1);
    if (e == cudaSuccess) owned.push_back(*p);
    return e;
  };
  struct Guard { std::vector<void*>& v; ~Guard() { for (void* q : v) cudaFree(q); } } guard{owned};
  cudaStream_t st = 0;
  int *du = nullptr, *di = nullptr;
  uint64_t *ka = nullptr, *kb = nullptr, *dk = nullptr;
  uint32_t *va = nullptr, *vb = nullptr, *flag = nullptr, *rank = nullptr;
  CK0(A((void**)&du, 4 * (size_t)n)); CK0(A((void**)&di, 4 * (size_t)n));
  CK0(A((void**)&ka, 8 * (size_t)n)); CK0(A((void**)&kb, 8 * (size_t)n));
  CK0(A((void**)&va, 4 * (size_t)n)); CK0(A((void**)&vb, 4 * (size_t)n));
  CK0(A((void**)&flag, 4 * (size_t)n)); CK0(A((void**)&dk, 8 * (size_t)n)); CK0(A((void**)&rank, 4 * (size_t)n));
  CK0(cudaMemcpyAsync(du, user, 4 * (size_t)n, cudaMemcpyHostToDevice, st));
  CK0(cudaMemcpyAsync(di, item, 4 * (size_t)n, cudaMemcpyHostToDevice, st));
  // 1. distinct (user, item), sorted by user then item
  cooc_keys_kernel<<<nblk(n, 256), 256, 0, st>>>(du, di, n, bits_i, ka, va);
  bool in_b = false;
  CK0(radix_sort_pairs(ka, va, kb, vb, (size_t)n, bits_u + bits_i, st, &in_b, nullptr));
  const uint64_t* ks = in_b ? kb : ka;
  cooc_head_kernel<<<nblk(n, 256), 256, 0, st>>>(ks, n, flag);
  uint32_t lf = 0, lp = 0;
  CK0(cudaMemcpyAsync(&lf, flag + n - 1, 4, cudaMemcpyDeviceToHost, st));
  uint32_t* pos = in_b ? va : vb;   // the payload buffer that is free now
  CK0(scan_exclusive_u32(flag, pos, (size_t)n, st, nullptr));
  CK0(cudaMemcpyAsync(&lp, pos + n - 1, 4, cudaMemcpyDeviceToHost, st));
  CK0(cudaStreamSynchronize(st));
  const long long m = (long long)lp + lf;
  cooc_compact_kernel<<<nblk(n, 256), 256, 0, st>>>(ks, flag, pos, n, dk);
  // 2. pairs (item1 < item2) per user
  cooc_rank_kernel<<<nblk(m, 256), 256, 0, st>>>(dk, m, bits_i, rank);
  uint32_t* off = flag;
  CK0(scan_exclusive_u32(rank, off, (size_t)m, st, nullptr));
  uint32_t lr = 0, lo = 0;
  CK0(cudaMemcpyAsync(&lr, rank + m - 1, 4, cudaMemcpyDeviceToHost, st));
  CK0(cudaMemcpyAsync(&lo, off + m - 1, 4, cudaMemcpyDeviceToHost, st));
  CK0(cudaStreamSynchronize(st));
  const long long np = (long long)lo + lr;
  if (np >= (1ll << 31)) return fail(nullptr, PIO_ALS_ERR_ARG, "more than 2^31-1 co-occurrence pairs (%lld)", np);
  std::vector<int> h_item((size_t)n_items * topn, -1), h_cnt((size_t)n_items * topn, 0), h_n((size_t)n_items, 0);
  if (np > 0) {
    uint64_t *pk = nullptr, *pk2 = nullptr, *rk = nullptr, *rk2 = nullptr;
    uint32_t *pp = nullptr, *pp2 = nullptr, *pf = nullptr, *ppos = nullptr, *rp = nullptr, *rp2 = nullptr;
    CK0(A((void**)&pk, 8 * (size_t)np)); CK0(A((void**)&pk2, 8 * (size_t)np));
    CK0(A((void**)&pp, 4 * (size_t)np)); CK0(A((void**)&pp2, 4 * (size_t)np));
    CK0(A((void**)&pf, 4 * (size_t)np)); CK0(A((void**)&ppos, 4 * (size_t)np));
    cooc_pairs_kernel<<<nblk(m, 256), 256, 0, st>>>(dk, rank, off, m, bits_i, pk, pp);
    bool pb_ = false;
    CK0(radix_sort_pairs(pk, pp, pk2, pp2, (size_t)np, 2 * bits_i, st, &pb_, nullptr));
    const uint64_t* pks = pb_ ? pk2 : pk;
    cooc_head_kernel<<<nblk(np, 256), 256, 0, st>>>(pks, np, pf);
    uint32_t cf = 0, cp = 0;
    CK0(cudaMemcpyAsync(&cf, pf + np - 1, 4, cudaMemcpyDeviceToHost, st));
    CK0(scan_exclusive_u32(pf, ppos, (size_t)np, st, nullptr));
    CK0(cudaMemcpyAsync(&cp, ppos + np - 1, 4, cudaMemcpyDeviceToHost, st));
    CK0(cudaStreamSynchronize(st));
    const long long C = (long long)cp + cf, n2 = 2 * C;
    // 3. both directions, ranked per item by (count desc, other item asc)
    CK0(A((void**)&rk, 8 * (size_t)n2)); CK0(A((void**)&rk2, 8 * (size_t)n2));
    CK0(A((void**)&rp, 4 * (size_t)n2)); CK0(A((void**)&rp2, 4 * (size_t)n2));
    cooc_runs_kernel<<<nblk(np, 256), 256, 0, st>>>(pks, pf, ppos, np, bits_i, bits_c, rk, rp);
    bool rb = false;
    CK0(radix_sort_pairs(rk, rp, rk2, rp2, (size_t)n2, 2 * bits_i + bits_c, st, &rb, nullptr));
    int *d_oi = nullptr, *d_oc = nullptr, *d_on = nullptr;
    CK0(A((void**)&d_oi, 4 * (size_t)n_items * topn)); CK0(A((void**)&d_oc, 4 * (size_t)n_items * topn));
    CK0(A((void**)&d_on, 4 * (size_t)n_items));
    CK0(cudaMemsetAsync(d_oi, 0xff, 4 * (size_t)n_items * topn, st));
    CK0(cudaMemsetAsync(d_oc, 0, 4 * (size_t)n_items * topn, st));
    CK0(cudaMemsetAsync(d_on, 0, 4 * (size_t)n_items, st));
    cooc_take_kernel<<<nblk(n2, 256), 256, 0, st>>>(rb ? rk2 : rk, rb ? rp2 : rp, n2, bits_i, bits_c, topn, d_oi, d_oc, d_on);
    CK0(cudaMemcpyAsync(h_item.data(), d_oi, 4 * h_item.size(), cudaMemcpyDeviceToHost, st));
    CK0(cudaMemcpyAsync(h_cnt.data(), d_oc, 4 * h_cnt.size(), cudaMemcpyDeviceToHost, st));
    CK0(cudaMemcpyAsync(h_n.data(), d_on, 4 * h_n.size(), cudaMemcpyDeviceToHost, st));
    CK0(cudaStreamSynchronize(st));
  }
  memcpy(out_item, h_item.data(), 4 * h_item.size());
  memcpy(out_count, h_cnt.data(), 4 * h_cnt.size());
  memcpy(out_n, h_n.data(), 4 * h_n.size());
  return PIO_ALS_OK;
}

// ---- NaiveBayes ---------------------------------------------------------------------------------
int pio_nb_train(int device, const int32_t* label, const float* x, int64_t n, int n_feat, int n_class, double lambda,
                 double* pi, double* theta) {
  if (!label || !x || !pi || !theta || n <= 0 || n_feat < 1 || n_class < 1)
    return fail(nullptr, PIO_ALS_ERR_ARG, "bad NaiveBayes arguments");
  const int width = n_class * (n_feat + 1);
  if ((size_t)width * 8 * sizeof(double) > 200 * 1024) return fail(nullptr, PIO_ALS_ERR_ARG, "n_class*(n_feat+1) too large");
  CK0(cudaSetDevice(device));
  for (int64_t r = 0; r < n; ++r)
    if (label[r] < 0 || label[r] >= n_class) return fail(nullptr, PIO_ALS_ERR_ARG, "label out of range at row %lld", (long long)r);
  int* dl = nullptr;
  float* dx = nullptr;
  double *dp = nullptr, *dout = nullptr;
  const int nb = 296;
  CK0(cudaMalloc((void**)&dl, sizeof(int) * n));
  CK0(cudaMalloc((void**)&dx, sizeof(float) * n * n_feat));
  CK0(cudaMalloc((void**)&dp, sizeof(double) * (size_t)nb * width));
  CK0(cudaMalloc((void**)&dout, sizeof(double) * width));
  CK0(cudaMemcpy(dl, label, sizeof(int) * n, cudaMemcpyHostToDevice));
  CK0(cudaMemcpy(dx, x, sizeof(float) * n * n_feat, cudaMemcpyHostToDevice));
  const size_t smem = sizeof(double) * 8 * width;
  CK0(cudaFuncSetAttribute(nb_partial_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  nb_partial_kernel<<<nb, 256, smem>>>(dl, dx, n, n_feat, n_class, dp);
  nb_reduce_kernel<<<nblk(width, 128), 128>>>(dp, nb, width, dout);
  std::vector<double> acc(width);
  CK0(cudaMemcpy(acc.data(), dout, sizeof(double) * width, cudaMemcpyDeviceToHost));
  cudaFree(dl); cudaFree(dx); cudaFree(dp); cudaFree(dout);
  // MLlib multinomial: pi_c = log(n_c + l) - log(N + C l); theta_cj = log(s_cj + l) - log(sum_j s_cj + F l)
  const double logden = log((double)n + n_class * lambda);
  for (int c = 0; c < n_class; ++c) {
    pi[c] = log(acc[c * (n_feat + 1) + n_feat] + lambda) - logden;
    double tot = 0;
    for (int j = 0; j < n_feat; ++j) tot += acc[c * (n_feat + 1) + j];
    const double lt = log(tot + n_feat * lambda);
    for (int j = 0; j < n_feat; ++j) theta[c * n_feat + j] = log(acc[c * (n_feat + 1) + j] + lambda) - lt;
  }
  return PIO_ALS_OK;
}

int pio_nb_predict(int device, const float* x, int64_t n, int n_feat, int n_class, const double* pi, const double* theta,
                   int32_t* out_label) {
  if (!x || !pi || !theta || !out_label || n <= 0) return fail(nullptr, PIO_ALS_ERR_ARG, "bad NaiveBayes arguments");
  CK0(cudaSetDevice(device));
  float* dx = nullptr;
  double *dpi = nullptr, *dth = nullptr;
  int* dout = nullptr;
  CK0(cudaMalloc((void**)&dx, sizeof(float) * n * n_feat));
  CK0(cudaMalloc((void**)&dpi, sizeof(double) * n_class));
  CK0(cudaMalloc((void**)&dth, sizeof(double) * n_class * n_feat));
  CK0(cudaMalloc((void**)&dout, sizeof(int) * n));
  CK0(cudaMemcpy(dx, x, sizeof(float) * n * n_feat, cudaMemcpyHostToDevice));
  CK0(cudaMemcpy(dpi, pi, sizeof(double) * n_class, cudaMemcpyHostToDevice));
  CK0(cudaMemcpy(dth, theta, sizeof(double) * n_class * n_feat, cudaMemcpyHostToDevice));
  nb_predict_kernel<<<nblk(n, 256), 256>>>(dx, n, n_feat, n_class, dpi, dth, dout);
  CK0(cudaMemcpy(out_label, dout, sizeof(int) * n, cudaMemcpyDeviceToHost));
  cudaFree(dx); cudaFree(dpi); cudaFree(dth); cudaFree(dout);
  return PIO_ALS_OK;
}

}  // extern "C"
