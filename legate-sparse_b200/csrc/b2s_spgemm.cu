// b2s_spgemm.cu — CSR x CSR -> CSR SpGEMM for sm_100a (hash-based expand / sort / compress).
//
// Replaces SpGEMMCSRxCSRxCSRGPU (reference src/sparse/array/csr/spgemm_csr_csr_csr.cu:64-487,
// two cuSPARSE SpGEMM algorithms) and mirrors the reference's two-task CPU shape
// (NNZ task spgemm_csr_csr_csr.cc:62-87, numeric task :134-158): symbolic → scan → numeric.
//
// Rows of A are binned by their work (upper bound = intermediate products for the symbolic
// pass, exact nnz(C_i) for the numeric pass):
//   class 1  <=  128 entries : one WARP per row, 256-slot hash table in shared memory; the lanes
//                              are split into groups of 8/16/32 so that several short B rows are
//                              expanded at once; the finished row is compacted and only
//                              pow2ceil(nnz) entries are sorted (in registers when <= 32)
//   class 2  <= 1024 entries : one 128-thread CTA per row, 2048-slot table
//   class 3  <= 4096 entries : one 512-thread CTA per row, 8192-slot table
//   class 4  larger          : persistent 1024-thread CTAs, each owning a DENSE accumulator
//                              (ncolsB values + a bitmap) in HBM — Gustavson's dense workspace,
//                              the same structure the reference's CPU task uses
//                              (spgemm_csr_csr_csr.cc:104-131), affordable with 180 GB of HBM3e.
// Hash tables use linear probing with atomicCAS on the key and atomicAdd on the value; each
// finished row is bitonic-sorted by column in shared memory, so C has sorted indices like the
// cuSPARSE path of the reference (the reference's CPU path emits first-touch order).
#include "b2s_common.cuh"

namespace b2s {

constexpr int kT1 = 256, kT2 = 2048, kT3 = 8192;
constexpr int64_t kCap1 = 128, kCap2 = 1024, kCap3 = 4096;
constexpr int kScanBlock = 1024;

// ------------------------------------------------------------------ atomics on value types
__device__ __forceinline__ void vatomic_add(float* a, float v)   { atomicAdd(a, v); }
__device__ __forceinline__ void vatomic_add(double* a, double v) { atomicAdd(a, v); }
__device__ __forceinline__ void vatomic_add(c64* a, c64 v)   { atomicAdd(&a->re, v.re); atomicAdd(&a->im, v.im); }
__device__ __forceinline__ void vatomic_add(c128* a, c128 v) { atomicAdd(&a->re, v.re); atomicAdd(&a->im, v.im); }

template <typename I> struct key_traits;
template <> struct key_traits<int32_t> {
  using U = unsigned int;
  static constexpr int32_t EMPTY = -1;
  __device__ static int32_t cas(int32_t* a, int32_t cmp, int32_t v) {
    return (int32_t)atomicCAS((unsigned int*)a, (unsigned int)cmp, (unsigned int)v);
  }
};
template <> struct key_traits<int64_t> {
  using U = unsigned long long;
  static constexpr int64_t EMPTY = -1;
  __device__ static int64_t cas(int64_t* a, int64_t cmp, int64_t v) {
    return (int64_t)atomicCAS((unsigned long long*)a, (unsigned long long)cmp, (unsigned long long)v);
  }
};

template <int TABLE, typename I>
__device__ __forceinline__ uint32_t hash_slot(I key) {
  constexpr int LOG = (TABLE == 256) ? 8 : (TABLE == 2048) ? 11 : 13;
  static_assert(TABLE == 256 || TABLE == 2048 || TABLE == 8192, "unsupported hash table size");
  uint32_t k = (uint32_t)key ^ (uint32_t)((uint64_t)key >> 32);
  return (k * 0x9E3779B1u) >> (32 - LOG);
}

// insert key; returns true when the key was new
template <int TABLE, typename I>
__device__ __forceinline__ bool hash_insert(I* keys, I key, uint32_t& slot_out) {
  uint32_t h = hash_slot<TABLE, I>(key);
  while (true) {
    I old = reinterpret_cast<volatile I*>(keys)[h];
    if (old == key) { slot_out = h; return false; }
    if (old == key_traits<I>::EMPTY) {
      old = key_traits<I>::cas(&keys[h], key_traits<I>::EMPTY, key);
      if (old == key_traits<I>::EMPTY) { slot_out = h; return true; }
      if (old == key) { slot_out = h; return false; }
    }
    h = (h + 1) & (TABLE - 1);
  }
}

// ------------------------------------------------------------------ workspace
struct SpgemmWs {
  int64_t* counters;   // [16]: 0 products, 1..4 class counts, 5 dense-row cursor, 6 max count
  int64_t* work;       // [nrows] per-row work estimate / nnz
  int32_t* list[5];    // row lists per class (1..4), each [nrows]
  int64_t* blocksum;   // [ceil(nrows/kScanBlock)+1]
};

static SpgemmWs carve_ws(void* ws, int64_t nrows) {
  SpgemmWs w;
  uintptr_t b = ((uintptr_t)ws + 255) & ~(uintptr_t)255;
  w.counters = (int64_t*)b;           b += 16 * 8;
  w.work = (int64_t*)b;               b += (size_t)nrows * 8;
  for (int c = 1; c <= 4; ++c) { w.list[c] = (int32_t*)b; b += (size_t)nrows * 4; }
  w.list[0] = nullptr;
  b = (b + 15) & ~(uintptr_t)15;
  w.blocksum = (int64_t*)b;
  return w;
}

// ------------------------------------------------------------------ analysis kernels
template <typename I>
__global__ void row_products_kernel(int64_t nrows, const int64_t* __restrict__ a_ptr,
                                    const I* __restrict__ a_col, const int64_t* __restrict__ b_ptr,
                                    int64_t* __restrict__ work, int64_t* counters) {
  constexpr int L = 8;
  int64_t g = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) / L;
  int gl = threadIdx.x & (L - 1);
  int64_t total = ((int64_t)gridDim.x * blockDim.x) / L;
  int64_t nr_round = ceil_div(nrows, total) * total;
  int64_t mysum = 0;
  for (int64_t r = g; r < nr_round; r += total) {
    int64_t s = 0;
    if (r < nrows) {
      for (int64_t p = a_ptr[r] + gl; p < a_ptr[r + 1]; p += L) {
        int64_t k = (int64_t)a_col[p];
        s += b_ptr[k + 1] - b_ptr[k];
      }
    }
#pragma unroll
    for (int o = L >> 1; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (r < nrows && gl == 0) { work[r] = s; mysum += s; }
  }
  for (int o = 16; o > 0; o >>= 1) mysum += __shfl_xor_sync(0xffffffffu, mysum, o);
  if ((threadIdx.x & 31) == 0 && mysum) atomicAdd((unsigned long long*)&counters[0], (unsigned long long)mysum);
}

__global__ void row_nnz_from_indptr_kernel(int64_t nrows, const int64_t* __restrict__ c_ptr,
                                           int64_t* __restrict__ work) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < nrows) work[i] = c_ptr[i + 1] - c_ptr[i];
}

__device__ __forceinline__ int class_of(int64_t w) {
  return w <= 0 ? 0 : (w <= kCap1 ? 1 : (w <= kCap2 ? 2 : (w <= kCap3 ? 3 : 4)));
}

__global__ void classify_kernel(int64_t nrows, const int64_t* __restrict__ work, int64_t* counters,
                                int32_t* l1, int32_t* l2, int32_t* l3, int32_t* l4) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  int cls = (i < nrows) ? class_of(work[i]) : 0;
  int lane = threadIdx.x & 31;
  int32_t* lists[5] = {nullptr, l1, l2, l3, l4};
#pragma unroll
  for (int c = 1; c <= 4; ++c) {
    unsigned m = __ballot_sync(0xffffffffu, cls == c);
    if (m == 0) continue;
    int leader = __ffs(m) - 1;
    long long base = 0;
    if (lane == leader) base = (long long)atomicAdd((unsigned long long*)&counters[c], (unsigned long long)__popc(m));
    base = __shfl_sync(0xffffffffu, base, leader);
    if (cls == c) lists[c][base + __popc(m & ((1u << lane) - 1))] = (int32_t)i;
  }
}

// ------------------------------------------------------------------ scan (c_indptr)
__global__ void scan_block_kernel(int64_t n, const int64_t* in, int64_t* out_incl /* may alias in */,
                                  int64_t* __restrict__ blocksum) {
  __shared__ int64_t wtot[32];
  int64_t i = (int64_t)blockIdx.x * kScanBlock + threadIdx.x;
  int64_t v = i < n ? in[i] : 0;
  int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  for (int o = 1; o < 32; o <<= 1) {
    int64_t t = __shfl_up_sync(0xffffffffu, v, o);
    if (lane >= o) v += t;
  }
  if (lane == 31) wtot[w] = v;
  __syncthreads();
  if (w == 0) {
    int64_t t = wtot[lane];
    for (int o = 1; o < 32; o <<= 1) {
      int64_t u = __shfl_up_sync(0xffffffffu, t, o);
      if (lane >= o) t += u;
    }
    wtot[lane] = t;
  }
  __syncthreads();
  if (w > 0) v += wtot[w - 1];
  if (i < n) out_incl[i] = v;
  if (threadIdx.x == kScanBlock - 1) blocksum[blockIdx.x] = v;
}

__global__ void scan_sums_kernel(int64_t nb, int64_t* blocksum) {
  // single thread block; sequential over chunks of 1024 (nb is small: nrows/1024)
  __shared__ int64_t wtot[32];
  __shared__ int64_t carry;
  if (threadIdx.x == 0) carry = 0;
  __syncthreads();
  for (int64_t base = 0; base < nb; base += kScanBlock) {
    int64_t i = base + threadIdx.x;
    int64_t v = i < nb ? blocksum[i] : 0;
    int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    for (int o = 1; o < 32; o <<= 1) {
      int64_t t = __shfl_up_sync(0xffffffffu, v, o);
      if (lane >= o) v += t;
    }
    if (lane == 31) wtot[w] = v;
    __syncthreads();
    if (w == 0) {
      int64_t t = wtot[lane];
      for (int o = 1; o < 32; o <<= 1) {
        int64_t u = __shfl_up_sync(0xffffffffu, t, o);
        if (lane >= o) t += u;
      }
      wtot[lane] = t;
    }
    __syncthreads();
    if (w > 0) v += wtot[w - 1];
    v += carry;
    if (i < nb) blocksum[i] = v;  // inclusive
    __syncthreads();
    if (threadIdx.x == kScanBlock - 1) carry = v;
    __syncthreads();
  }
}

__global__ void scan_add_kernel(int64_t n, int64_t* __restrict__ out_incl, const int64_t* __restrict__ blocksum,
                                int64_t* __restrict__ first) {
  int64_t i = (int64_t)blockIdx.x * kScanBlock + threadIdx.x;
  if (i == 0) first[0] = 0;
  if (i < n && blockIdx.x > 0) out_incl[i] += blocksum[blockIdx.x - 1];
}

// v[0..n) → inclusive prefix sums in place, first[0] = 0 (first is normally v-1: an indptr).
// blocksum: scratch of ceil(n/1024)+1 int64.  Shared with the column-block splitter.
int scan_inclusive_i64(int64_t n, int64_t* v, int64_t* first, int64_t* blocksum, cudaStream_t st) {
  int64_t nb = ceil_div(n > 0 ? n : 1, kScanBlock);
  scan_block_kernel<<<(unsigned)nb, kScanBlock, 0, st>>>(n, v, v, blocksum);
  B2S_CHECK_LAUNCH();
  if (nb > 1) {
    scan_sums_kernel<<<1, kScanBlock, 0, st>>>(nb, blocksum);
    B2S_CHECK_LAUNCH();
  }
  scan_add_kernel<<<(unsigned)nb, kScanBlock, 0, st>>>(n, v, blocksum, first);
  B2S_CHECK_LAUNCH();
  return B2S_OK;
}

// ------------------------------------------------------------------ hash kernels (symbolic)
// One group (warp when WARP_ROWS>1, else the CTA) per row.
template <typename I, int TABLE, int THREADS, bool WARP_PER_ROW>
__global__ void __launch_bounds__(THREADS)
sym_hash_kernel(int64_t nlist, const int32_t* __restrict__ list, const int64_t* __restrict__ a_ptr,
                const I* __restrict__ a_col, const int64_t* __restrict__ b_ptr,
                const I* __restrict__ b_col, int64_t* __restrict__ row_nnz, int gs) {
  constexpr int GROUPS = WARP_PER_ROW ? THREADS / 32 : 1;
  constexpr int GT = WARP_PER_ROW ? 32 : THREADS;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  I* keys = reinterpret_cast<I*>(smem_raw);
  __shared__ int cnt[GROUPS];
  const int grp = WARP_PER_ROW ? (threadIdx.x >> 5) : 0;
  const int gt = WARP_PER_ROW ? (threadIdx.x & 31) : threadIdx.x;
  const int64_t li = (int64_t)blockIdx.x * GROUPS + grp;
  I* mykeys = keys + grp * TABLE;
  for (int i = gt; i < TABLE; i += GT) mykeys[i] = key_traits<I>::EMPTY;
  if (gt == 0) cnt[grp] = 0;
  if (WARP_PER_ROW) __syncwarp(); else __syncthreads();
  int local = 0;
  int64_t row = -1;
  if (li < nlist) {
    row = list[li];
    // warp rows: `gs` lanes per A entry (32/gs entries in flight); CTA rows: one warp per A entry
    const int lane = WARP_PER_ROW ? (threadIdx.x & (gs - 1)) : (threadIdx.x & 31);
    const int step = WARP_PER_ROW ? gs : 32;
    const int sub = WARP_PER_ROW ? ((threadIdx.x & 31) / gs) : (threadIdx.x >> 5);
    const int nsub = WARP_PER_ROW ? 32 / gs : THREADS / 32;
    for (int64_t pa = a_ptr[row] + sub; pa < a_ptr[row + 1]; pa += nsub) {
      int64_t k = (int64_t)a_col[pa];
      for (int64_t pb = b_ptr[k] + lane; pb < b_ptr[k + 1]; pb += step) {
        uint32_t s;
        if (hash_insert<TABLE, I>(mykeys, b_col[pb], s)) ++local;
      }
    }
  }
  for (int o = 16; o > 0; o >>= 1) local += __shfl_xor_sync(0xffffffffu, local, o);
  if (WARP_PER_ROW) {
    if (gt == 0 && row >= 0) row_nnz[row] = local;
  } else {
    if ((threadIdx.x & 31) == 0 && local) atomicAdd(&cnt[0], local);
    __syncthreads();
    if (threadIdx.x == 0 && row >= 0) row_nnz[row] = cnt[0];
  }
}

// ------------------------------------------------------------------ hash kernels (numeric)
template <typename I, typename V, int N, int GT, bool WARP>
__device__ __forceinline__ void bitonic_sort_kv(I* keys, V* vals, int gt) {
  using U = typename key_traits<I>::U;
  for (int k = 2; k <= N; k <<= 1) {
    for (int j = k >> 1; j > 0; j >>= 1) {
      for (int i = gt; i < N; i += GT) {
        int ixj = i ^ j;
        if (ixj > i) {
          U a = (U)keys[i], b = (U)keys[ixj];
          bool up = ((i & k) == 0);
          if ((a > b) == up) {
            keys[i] = (I)b; keys[ixj] = (I)a;
            V t = vals[i]; vals[i] = vals[ixj]; vals[ixj] = t;
          }
        }
      }
      if (WARP) __syncwarp(); else __syncthreads();
    }
  }
}

template <typename V, typename I, int TABLE, int THREADS, bool WARP_PER_ROW>
__global__ void __launch_bounds__(THREADS)
num_hash_kernel(int64_t nlist, const int32_t* __restrict__ list, const int64_t* __restrict__ a_ptr,
                const I* __restrict__ a_col, const V* __restrict__ a_val,
                const int64_t* __restrict__ b_ptr, const I* __restrict__ b_col,
                const V* __restrict__ b_val, const int64_t* __restrict__ c_ptr, I* __restrict__ c_col,
                V* __restrict__ c_val, int gs) {
  constexpr int GROUPS = WARP_PER_ROW ? THREADS / 32 : 1;
  constexpr int GT = WARP_PER_ROW ? 32 : THREADS;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  V* vals_all = reinterpret_cast<V*>(smem_raw);
  I* keys_all = reinterpret_cast<I*>(smem_raw + sizeof(V) * GROUPS * TABLE);
  const int grp = WARP_PER_ROW ? (threadIdx.x >> 5) : 0;
  const int gt = WARP_PER_ROW ? (threadIdx.x & 31) : threadIdx.x;
  const int64_t li = (int64_t)blockIdx.x * GROUPS + grp;
  I* keys = keys_all + grp * TABLE;
  V* vals = vals_all + grp * TABLE;
  for (int i = gt; i < TABLE; i += GT) { keys[i] = key_traits<I>::EMPTY; vals[i] = zero_of<V>(); }
  if (WARP_PER_ROW) __syncwarp(); else __syncthreads();
  int64_t row = -1;
  if (li < nlist) {
    row = list[li];
    const int lane = WARP_PER_ROW ? (threadIdx.x & (gs - 1)) : (threadIdx.x & 31);
    const int step = WARP_PER_ROW ? gs : 32;
    const int sub = WARP_PER_ROW ? ((threadIdx.x & 31) / gs) : (threadIdx.x >> 5);
    const int nsub = WARP_PER_ROW ? 32 / gs : THREADS / 32;
    for (int64_t pa = a_ptr[row] + sub; pa < a_ptr[row + 1]; pa += nsub) {
      int64_t k = (int64_t)a_col[pa];
      V av = a_val[pa];
      for (int64_t pb = b_ptr[k] + lane; pb < b_ptr[k + 1]; pb += step) {
        uint32_t s;
        hash_insert<TABLE, I>(keys, b_col[pb], s);
        vatomic_add(&vals[s], vmul(av, b_val[pb]));
      }
    }
  }
  if (WARP_PER_ROW) __syncwarp(); else __syncthreads();
  if constexpr (WARP_PER_ROW) {
    // ---- in-place compaction of the occupied slots to the front (32 slots per step) ----
    using U = typename key_traits<I>::U;
    const int lane = threadIdx.x & 31;
    int n = 0;
#pragma unroll 1
    for (int b0 = 0; b0 < TABLE; b0 += 32) {
      const I kk = keys[b0 + lane];
      const V vv = vals[b0 + lane];
      const bool valid = kk != key_traits<I>::EMPTY;
      const unsigned m = __ballot_sync(0xffffffffu, valid);
      __syncwarp();                      // everybody has read its slot before anyone overwrites
      if (valid) {
        const int pos = n + __popc(m & ((1u << lane) - 1));
        keys[pos] = kk;
        vals[pos] = vv;
      }
      n += __popc(m);
      __syncwarp();
    }
    if (row >= 0) {
      const int64_t o = c_ptr[row];
      if (n <= 32) {
        // ---- register bitonic sort of <= 32 (key,val) pairs by shuffles ----
        U key = lane < n ? (U)keys[lane] : ~(U)0;
        V val = lane < n ? vals[lane] : zero_of<V>();
#pragma unroll
        for (int k = 2; k <= 32; k <<= 1) {
#pragma unroll
          for (int j = k >> 1; j > 0; j >>= 1) {
            const U okey = __shfl_xor_sync(0xffffffffu, key, j);
            const V oval = vshfl_xor(val, j);
            const bool up = ((lane & k) == 0);
            const bool lower = ((lane & j) == 0);
            const bool take_other = (lower == up) ? (okey < key) : (okey > key);
            if (take_other) { key = okey; val = oval; }
          }
        }
        if (lane < n) { c_col[o + lane] = (I)key; c_val[o + lane] = val; }
      } else {
        // ---- shared-memory bitonic over pow2ceil(n) entries ----
        int mpow = 64;
        while (mpow < n) mpow <<= 1;
        for (int i = n + lane; i < mpow; i += 32) { keys[i] = key_traits<I>::EMPTY; vals[i] = zero_of<V>(); }
        __syncwarp();
        for (int k = 2; k <= mpow; k <<= 1) {
          for (int j = k >> 1; j > 0; j >>= 1) {
            for (int i = lane; i < mpow; i += 32) {
              const int ixj = i ^ j;
              if (ixj > i) {
                const U a = (U)keys[i], b = (U)keys[ixj];
                const bool up = ((i & k) == 0);
                if ((a > b) == up) {
                  keys[i] = (I)b; keys[ixj] = (I)a;
                  const V t = vals[i]; vals[i] = vals[ixj]; vals[ixj] = t;
                }
              }
            }
            __syncwarp();
          }
        }
        for (int i = lane; i < n; i += 32) { c_col[o + i] = keys[i]; c_val[o + i] = vals[i]; }
      }
    }
  } else {
    bitonic_sort_kv<I, V, TABLE, GT, WARP_PER_ROW>(keys, vals, gt);
    if (row >= 0) {
      int64_t o = c_ptr[row];
      int64_t n = c_ptr[row + 1] - o;
      for (int64_t i = gt; i < n; i += GT) { c_col[o + i] = keys[i]; c_val[o + i] = vals[i]; }
    }
  }
}

// ------------------------------------------------------------------ dense-accumulator kernels
constexpr int kDenseThreads = 1024;

__device__ __forceinline__ int block_excl_scan_1024(int v, int* total, int* wtot /*[32]*/) {
  int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  int incl = v;
  for (int o = 1; o < 32; o <<= 1) {
    int t = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += t;
  }
  if (lane == 31) wtot[w] = incl;
  __syncthreads();
  if (w == 0) {
    int t = wtot[lane];
    for (int o = 1; o < 32; o <<= 1) {
      int u = __shfl_up_sync(0xffffffffu, t, o);
      if (lane >= o) t += u;
    }
    wtot[lane] = t;
  }
  __syncthreads();
  int base = w > 0 ? wtot[w - 1] : 0;
  *total = wtot[31];
  __syncthreads();
  return base + incl - v;
}

template <typename V, typename I, bool NUMERIC>
__global__ void __launch_bounds__(kDenseThreads)
dense_row_kernel(int64_t nlist, const int32_t* __restrict__ list, int64_t ncolsB,
                 const int64_t* __restrict__ a_ptr, const I* __restrict__ a_col,
                 const V* __restrict__ a_val, const int64_t* __restrict__ b_ptr,
                 const I* __restrict__ b_col, const V* __restrict__ b_val, unsigned* bitmaps,
                 V* dense, int64_t* cursor, int64_t* __restrict__ row_nnz /*symbolic out*/,
                 const int64_t* __restrict__ c_ptr, I* __restrict__ c_col, V* __restrict__ c_val) {
  const int64_t nwords = (ncolsB + 31) / 32;
  unsigned* bm = bitmaps + (int64_t)blockIdx.x * nwords;
  V* acc = NUMERIC ? dense + (int64_t)blockIdx.x * ncolsB : nullptr;
  __shared__ int64_t s_row;
  __shared__ int wtot[32];
  __shared__ long long s_wmin, s_wmax;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  constexpr int NW = kDenseThreads / 32;
  while (true) {
    if (threadIdx.x == 0) {
      int64_t li = (int64_t)atomicAdd((unsigned long long*)cursor, 1ull);
      s_row = li < nlist ? (int64_t)list[li] : -1;
      s_wmin = LLONG_MAX; s_wmax = -1;
    }
    __syncthreads();
    const int64_t row = s_row;
    if (row < 0) break;
    long long wmin = LLONG_MAX, wmax = -1;
    for (int64_t pa = a_ptr[row] + warp; pa < a_ptr[row + 1]; pa += NW) {
      int64_t k = (int64_t)a_col[pa];
      V av = NUMERIC ? a_val[pa] : zero_of<V>();
      for (int64_t pb = b_ptr[k] + lane; pb < b_ptr[k + 1]; pb += 32) {
        int64_t j = (int64_t)b_col[pb];
        long long w = j >> 5;
        unsigned bit = 1u << (j & 31);
        if (!(__ldcg(&bm[w]) & bit)) atomicOr(&bm[w], bit);
        if (NUMERIC) vatomic_add(&acc[j], vmul(av, b_val[pb]));
        wmin = w < wmin ? w : wmin; wmax = w > wmax ? w : wmax;
      }
    }
    for (int o = 16; o > 0; o >>= 1) {
      long long a = __shfl_xor_sync(0xffffffffu, wmin, o), b = __shfl_xor_sync(0xffffffffu, wmax, o);
      wmin = a < wmin ? a : wmin; wmax = b > wmax ? b : wmax;
    }
    if (lane == 0 && wmax >= 0) { atomicMin(&s_wmin, wmin); atomicMax(&s_wmax, wmax); }
    __syncthreads();
    __threadfence_block();
    const long long lo = s_wmin, hi = s_wmax;
    int64_t out = NUMERIC ? c_ptr[row] : 0;
    int64_t running = 0;
    if (hi >= 0) {
      for (long long base = lo; base <= hi; base += kDenseThreads) {
        long long w = base + threadIdx.x;
        unsigned bits = (w <= hi) ? __ldcg(&bm[w]) : 0u;
        int c = __popc(bits);
        int total;
        int pos = block_excl_scan_1024(c, &total, wtot);
        if (NUMERIC) {
          int64_t o = out + running + pos;
          while (bits) {
            int b = __ffs(bits) - 1;
            bits &= bits - 1;
            int64_t j = w * 32 + b;
            c_col[o] = (I)j;
            c_val[o] = ld_cg(&acc[j]);
            acc[j] = zero_of<V>();
            ++o;
          }
        }
        if (w <= hi && c) bm[w] = 0u;
        running += total;
      }
    }
    if (!NUMERIC && threadIdx.x == 0) row_nnz[row] = running;
    __syncthreads();
  }
}

// ------------------------------------------------------------------ host side
// lanes per A entry in the warp-per-row kernels: short B rows → several B rows expanded at once
static int lane_group_size(int64_t nnzB, int64_t nrowsB) {
  double avg = nrowsB > 0 ? (double)nnzB / (double)nrowsB : 32.0;
  return avg <= 12.0 ? 8 : (avg <= 24.0 ? 16 : 32);
}

static int64_t ws_bytes(int64_t nrows) {
  return 256 + 16 * 8 + nrows * 8 + 4 * nrows * 4 + 16 + (ceil_div(nrows > 0 ? nrows : 1, kScanBlock) + 1) * 8 + 256;
}

struct ClassCounts { int64_t n[5]; int64_t products; };

static int analyse(SpgemmWs& W, int64_t nrows, cudaStream_t st, ClassCounts* out) {
  classify_kernel<<<(unsigned)ceil_div(nrows, 256), 256, 0, st>>>(nrows, W.work, W.counters, W.list[1],
                                                                 W.list[2], W.list[3], W.list[4]);
  B2S_CHECK_LAUNCH();
  int64_t h[8];
  B2S_CUDA_TRY(cudaMemcpyAsync(h, W.counters, sizeof(h), cudaMemcpyDeviceToHost, st));
  B2S_CUDA_TRY(cudaStreamSynchronize(st));
  out->products = h[0];
  for (int c = 1; c <= 4; ++c) out->n[c] = h[c];
  return B2S_OK;
}

struct DenseScratch {
  unsigned* bitmaps = nullptr;
  void* dense = nullptr;
  int64_t nctas = 0;
};

static int alloc_dense(int64_t nD, int64_t ncolsB, size_t vbytes, bool numeric, cudaStream_t st,
                       DenseScratch* D) {
  if (nD <= 0) return B2S_OK;
  int64_t nwords = (ncolsB + 31) / 32;
  size_t per = (size_t)nwords * 4 + (numeric ? (size_t)ncolsB * vbytes : 0);
  size_t freeb = 0, totalb = 0;
  B2S_CUDA_TRY(cudaMemGetInfo(&freeb, &totalb));
  int64_t nctas = nD < kNumSMs * 2 ? nD : kNumSMs * 2;
  while (nctas > 1 && (size_t)nctas * per > freeb / 2) nctas /= 2;
  if ((size_t)nctas * per > freeb) {
    set_error("SpGEMM dense accumulators need %zu bytes, only %zu free", (size_t)nctas * per, freeb);
    return B2S_ERR_WORKSPACE;
  }
  D->nctas = nctas;
  B2S_CUDA_TRY(cudaMallocAsync((void**)&D->bitmaps, (size_t)nctas * nwords * 4, st));
  B2S_CUDA_TRY(cudaMemsetAsync(D->bitmaps, 0, (size_t)nctas * nwords * 4, st));
  if (numeric) {
    B2S_CUDA_TRY(cudaMallocAsync(&D->dense, (size_t)nctas * ncolsB * vbytes, st));
    B2S_CUDA_TRY(cudaMemsetAsync(D->dense, 0, (size_t)nctas * ncolsB * vbytes, st));
  }
  return B2S_OK;
}

static void free_dense(DenseScratch* D, cudaStream_t st) {
  if (D->bitmaps) cudaFreeAsync(D->bitmaps, st);
  if (D->dense) cudaFreeAsync(D->dense, st);
  D->bitmaps = nullptr; D->dense = nullptr;
}

template <typename I, int TABLE, int THREADS, bool WARP>
static int launch_sym_hash(int64_t n, const int32_t* list, const int64_t* a_ptr, const I* a_col,
                           const int64_t* b_ptr, const I* b_col, int64_t* row_nnz, int gs, cudaStream_t st) {
  constexpr int GROUPS = WARP ? THREADS / 32 : 1;
  size_t smem = sizeof(I) * (size_t)GROUPS * TABLE;
  auto kern = sym_hash_kernel<I, TABLE, THREADS, WARP>;
  static bool attr = false;
  if (!attr && smem > 48 * 1024) {
    B2S_CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    attr = true;
  }
  kern<<<(unsigned)ceil_div(n, GROUPS), THREADS, smem, st>>>(n, list, a_ptr, a_col, b_ptr, b_col, row_nnz, gs);
  B2S_CHECK_LAUNCH();
  return B2S_OK;
}

template <typename I>
static int symbolic_typed(int64_t nrowsA, int64_t ncolsB, const int64_t* a_ptr, const I* a_col,
                          const int64_t* b_ptr, const I* b_col, int64_t* c_ptr, void* workspace,
                          int64_t* out_nnzC, int64_t* out_products, int gs, cudaStream_t st) {
  SpgemmWs W = carve_ws(workspace, nrowsA);
  B2S_CUDA_TRY(cudaMemsetAsync(W.counters, 0, 16 * 8, st));
  if (nrowsA == 0) {
    // an empty row block still has c_indptr[0] = nnz(C) = 0 (the caller may have allocated it uninitialised)
    B2S_CUDA_TRY(cudaMemsetAsync(c_ptr, 0, sizeof(int64_t), st));
    if (out_nnzC) *out_nnzC = 0;
    if (out_products) *out_products = 0;
    return B2S_OK;
  }
  {
    int64_t blocks = ceil_div(nrowsA * 8, 256);
    int64_t cap = (int64_t)kNumSMs * 16;
    if (blocks > cap) blocks = cap;
    row_products_kernel<I><<<(unsigned)blocks, 256, 0, st>>>(nrowsA, a_ptr, a_col, b_ptr, W.work, W.counters);
    B2S_CHECK_LAUNCH();
  }
  ClassCounts cc;
  int rc = analyse(W, nrowsA, st, &cc);
  if (rc) return rc;
  // row_nnz is written into c_ptr+1 (then scanned in place); rows of class 0 need zeros
  int64_t* row_nnz = c_ptr + 1;
  B2S_CUDA_TRY(cudaMemsetAsync(c_ptr, 0, (size_t)(nrowsA + 1) * 8, st));
  // NB: kernels index row_nnz[row]
  if (cc.n[1] > 0) {
    rc = launch_sym_hash<I, kT1, 256, true>(cc.n[1], W.list[1], a_ptr, a_col, b_ptr, b_col, row_nnz, gs, st);
    if (rc) return rc;
  }
  if (cc.n[2] > 0) {
    rc = launch_sym_hash<I, kT2, 128, false>(cc.n[2], W.list[2], a_ptr, a_col, b_ptr, b_col, row_nnz, gs, st);
    if (rc) return rc;
  }
  if (cc.n[3] > 0) {
    rc = launch_sym_hash<I, kT3, 512, false>(cc.n[3], W.list[3], a_ptr, a_col, b_ptr, b_col, row_nnz, gs, st);
    if (rc) return rc;
  }
  DenseScratch D;
  if (cc.n[4] > 0) {
    rc = alloc_dense(cc.n[4], ncolsB, 0, false, st, &D);
    if (rc) return rc;
    dense_row_kernel<double, I, false><<<(unsigned)D.nctas, kDenseThreads, 0, st>>>(
        cc.n[4], W.list[4], ncolsB, a_ptr, a_col, nullptr, b_ptr, b_col, nullptr, D.bitmaps, nullptr,
        &W.counters[5], row_nnz, nullptr, nullptr, nullptr);
    B2S_CHECK_LAUNCH();
  }
  // inclusive scan of row_nnz in place → c_ptr[1..nrows]; c_ptr[0] = 0
  { int rc2 = scan_inclusive_i64(nrowsA, row_nnz, c_ptr, W.blocksum, st); if (rc2) return rc2; }
  int64_t nnzC = 0;
  B2S_CUDA_TRY(cudaMemcpyAsync(&nnzC, c_ptr + nrowsA, 8, cudaMemcpyDeviceToHost, st));
  free_dense(&D, st);
  B2S_CUDA_TRY(cudaStreamSynchronize(st));
  if (out_nnzC) *out_nnzC = nnzC;
  if (out_products) *out_products = cc.products;
  return B2S_OK;
}

template <typename V, typename I, int TABLE, int THREADS, bool WARP>
static int launch_num_hash(int64_t n, const int32_t* list, const int64_t* a_ptr, const I* a_col,
                           const V* a_val, const int64_t* b_ptr, const I* b_col, const V* b_val,
                           const int64_t* c_ptr, I* c_col, V* c_val, int gs, cudaStream_t st) {
  constexpr int GROUPS = WARP ? THREADS / 32 : 1;
  size_t smem = (sizeof(V) + sizeof(I)) * (size_t)GROUPS * TABLE;
  auto kern = num_hash_kernel<V, I, TABLE, THREADS, WARP>;
  static bool attr = false;
  if (!attr && smem > 48 * 1024) {
    B2S_CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    attr = true;
  }
  kern<<<(unsigned)ceil_div(n, GROUPS), THREADS, smem, st>>>(n, list, a_ptr, a_col, a_val, b_ptr, b_col,
                                                            b_val, c_ptr, c_col, c_val, gs);
  B2S_CHECK_LAUNCH();
  return B2S_OK;
}

template <typename V, typename I>
static int numeric_typed(int64_t nrowsA, int64_t ncolsB, const int64_t* a_ptr, const I* a_col,
                         const V* a_val, const int64_t* b_ptr, const I* b_col, const V* b_val,
                         const int64_t* c_ptr, I* c_col, V* c_val, void* workspace, int gs,
                         cudaStream_t st) {
  if (nrowsA == 0) return B2S_OK;
  SpgemmWs W = carve_ws(workspace, nrowsA);
  B2S_CUDA_TRY(cudaMemsetAsync(W.counters, 0, 16 * 8, st));
  row_nnz_from_indptr_kernel<<<(unsigned)ceil_div(nrowsA, 256), 256, 0, st>>>(nrowsA, c_ptr, W.work);
  B2S_CHECK_LAUNCH();
  ClassCounts cc;
  int rc = analyse(W, nrowsA, st, &cc);
  if (rc) return rc;
  if (cc.n[1] > 0) {
    rc = launch_num_hash<V, I, kT1, 256, true>(cc.n[1], W.list[1], a_ptr, a_col, a_val, b_ptr, b_col, b_val,
                                               c_ptr, c_col, c_val, gs, st);
    if (rc) return rc;
  }
  if (cc.n[2] > 0) {
    rc = launch_num_hash<V, I, kT2, 128, false>(cc.n[2], W.list[2], a_ptr, a_col, a_val, b_ptr, b_col, b_val,
                                                c_ptr, c_col, c_val, gs, st);
    if (rc) return rc;
  }
  if (cc.n[3] > 0) {
    rc = launch_num_hash<V, I, kT3, 512, false>(cc.n[3], W.list[3], a_ptr, a_col, a_val, b_ptr, b_col, b_val,
                                                c_ptr, c_col, c_val, gs, st);
    if (rc) return rc;
  }
  if (cc.n[4] > 0) {
    DenseScratch D;
    rc = alloc_dense(cc.n[4], ncolsB, sizeof(V), true, st, &D);
    if (rc) return rc;
    dense_row_kernel<V, I, true><<<(unsigned)D.nctas, kDenseThreads, 0, st>>>(
        cc.n[4], W.list[4], ncolsB, a_ptr, a_col, a_val, b_ptr, b_col, b_val, D.bitmaps, (V*)D.dense,
        &W.counters[5], nullptr, c_ptr, c_col, c_val);
    B2S_CHECK_LAUNCH();
    free_dense(&D, st);
  }
  return B2S_OK;
}

}  // namespace b2s

using namespace b2s;

extern "C" int64_t b2s_spgemm_workspace_bytes(int64_t nrowsA, int64_t nnzA, int64_t ncolsB) {
  (void)nnzA; (void)ncolsB;
  if (nrowsA < 0) return -1;
  return ws_bytes(nrowsA);
}

extern "C" int b2s_spgemm_symbolic(b2s_itype it, int64_t nrowsA, int64_t ncolsA, int64_t ncolsB,
                                   const int64_t* a_indptr, const void* a_indices, int64_t nnzA,
                                   const int64_t* b_indptr, const void* b_indices, int64_t nnzB,
                                   int64_t* c_indptr, void* workspace, int64_t workspace_bytes,
                                   int64_t* out_nnzC, int64_t* out_products, b2s_stream_t stream) {
  B2S_REQUIRE(nrowsA >= 0 && ncolsA >= 0 && ncolsB >= 0 && nnzA >= 0 && nnzB >= 0, "negative size");
  B2S_REQUIRE(nrowsA < INT32_MAX, "row block too large for 32-bit row lists");
  B2S_REQUIRE(c_indptr && workspace, "null c_indptr/workspace");
  B2S_REQUIRE(nrowsA == 0 || a_indptr, "null a_indptr");
  B2S_REQUIRE(ncolsA == 0 || b_indptr, "null b_indptr");
  if (workspace_bytes < ws_bytes(nrowsA)) {
    set_error("spgemm workspace too small: %lld < %lld", (long long)workspace_bytes, (long long)ws_bytes(nrowsA));
    return B2S_ERR_WORKSPACE;
  }
  cudaStream_t st = (cudaStream_t)stream;
  B2S_DISPATCH_IT(it, I,
    return symbolic_typed<I>(nrowsA, ncolsB, a_indptr, (const I*)a_indices, b_indptr, (const I*)b_indices,
                             c_indptr, workspace, out_nnzC, out_products, lane_group_size(nnzB, ncolsA), st));
  return B2S_ERR_ARG;
}

extern "C" int b2s_spgemm_numeric(b2s_dtype vt, b2s_itype it, int64_t nrowsA, int64_t ncolsA,
                                  int64_t ncolsB, const int64_t* a_indptr, const void* a_indices,
                                  const void* a_data, int64_t nnzA, const int64_t* b_indptr,
                                  const void* b_indices, const void* b_data, int64_t nnzB,
                                  const int64_t* c_indptr, void* c_indices, void* c_data,
                                  void* workspace, int64_t workspace_bytes, b2s_stream_t stream) {
  B2S_REQUIRE(nrowsA >= 0 && ncolsA >= 0 && ncolsB >= 0 && nnzA >= 0 && nnzB >= 0, "negative size");
  B2S_REQUIRE(nrowsA < INT32_MAX, "row block too large for 32-bit row lists");
  B2S_REQUIRE(c_indptr && workspace, "null c_indptr/workspace");
  if (workspace_bytes < ws_bytes(nrowsA)) {
    set_error("spgemm workspace too small: %lld < %lld", (long long)workspace_bytes, (long long)ws_bytes(nrowsA));
    return B2S_ERR_WORKSPACE;
  }
  cudaStream_t st = (cudaStream_t)stream;
  B2S_DISPATCH_VT(vt, V, B2S_DISPATCH_IT(it, I,
    return numeric_typed<V, I>(nrowsA, ncolsB, a_indptr, (const I*)a_indices, (const V*)a_data, b_indptr,
                               (const I*)b_indices, (const V*)b_data, c_indptr, (I*)c_indices,
                               (V*)c_data, workspace, lane_group_size(nnzB, ncolsA), st)));
  return B2S_ERR_ARG;
}
