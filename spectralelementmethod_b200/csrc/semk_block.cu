// semk_block.cu -- block-vector kernels of the block eigensolver (eigen.py, LOBPCG).
//
// A block of m vectors of length n is stored as rows X + i*ldx, i < m (ldx >= n).  The two
// kernels here are the only passes over whole blocks a LOBPCG iteration makes besides the
// operator applies:
//   Gram    : G[i*k + j] = sum_t X[i][t] w[t] Y[j][t]      (all m*k inner products at once)
//   combine : Y[j] = beta Y[j] + sum_i C[i*k + j] X[i]      (a block times a small matrix)
// Both stage a chunk of rows of every vector in shared memory and form a register-tiled
// product from there, so X, Y and w are each read from memory once per call.  The m*k dots
// of the Gram kernel would otherwise take about m passes of semk_multi_dot_f64 over Y.
//
// Determinism: every CTA of the Gram kernel owns a fixed range of t and accumulates it in a
// fixed order; the per-CTA partial matrices are summed by the CTA that arrives last in CTA
// order (the pattern of semk_finish_reduction, semk_common.cuh).  No atomics on values, so
// the result is bitwise reproducible for a given (n, m, k).
#include "semk_common.cuh"

namespace {

constexpr int kBlkThreads = 256;       // a 16 x 16 thread grid
constexpr int kBlkMax = 96;            // m, k <= 96 (LOBPCG with block size <= 32: 3 x 32)
constexpr int kGramRows = 32;          // rows of t staged per chunk (Gram)
constexpr int kGramMaxBlocks = 148 * 2;
constexpr int kCombRows = 64;          // rows of t staged per chunk (combine)
constexpr int kCombMaxBlocks = 148 * 4;
constexpr int kCombLoads = kBlkMax * kCombRows / kBlkThreads;   // per thread, <= 24

// Padded row length (in doubles) of a staged [rows][m] tile; it covers the 16-wide column
// blocks of the DFMA kernel.  DFMA: odd, so that the 32 lanes staging 32 rows of one column
// store to 16 distinct bank pairs (two wavefronts, the minimum for 256 bytes).  DMMA: 8 mod 16,
// so that the four k-rows an m8n8k4 fragment reads fall into distinct halves of the banks.
__host__ __device__ inline int gram_ld(int m, bool mma) {
  return ((m + 15) & ~15) + (mma ? 8 : 1);
}

inline int gram_blocks(int64_t n) {
  // fixed per-CTA ranges: a whole number of chunks each, at most kGramMaxBlocks CTAs
  const int64_t chunks = (n + kGramRows - 1) / kGramRows;
  const int64_t nb = chunks < kGramMaxBlocks ? chunks : kGramMaxBlocks;
  return (int)(nb < 1 ? 1 : nb);
}

// Stage rows [t0, t0 + kGramRows) of one block (times w if given): S[t][i], zero past r1.  All
// loads of a thread are issued before its first shared-memory store, so staging a block costs
// one memory latency, not one per element.
constexpr int kGramLoads = kBlkMax * kGramRows / kBlkThreads;   // per thread, <= 12
__device__ __forceinline__ void gram_stage(int64_t t0, int64_t r1, int m, const double *__restrict__ X,
                                           int64_t ldx, const double *__restrict__ w, double *S,
                                           int lds) {
  double v[kGramLoads];
  const int t = threadIdx.x % kGramRows;    // the same row for every q: kBlkThreads % 32 == 0
  const int64_t g = t0 + t;
#pragma unroll
  for (int q = 0; q < kGramLoads; ++q) {
    const int e = threadIdx.x + q * kBlkThreads;
    v[q] = (e < m * kGramRows && g < r1) ? __ldcs(X + (int64_t)(e / kGramRows) * ldx + g) : 0.0;
  }
  const double wt = (w && g < r1) ? __ldg(w + g) : 1.0;
#pragma unroll
  for (int q = 0; q < kGramLoads; ++q) {
    const int e = threadIdx.x + q * kBlkThreads;
    if (e < m * kGramRows) S[t * lds + e / kGramRows] = v[q] * wt;
  }
}

// partials layout: one 64-bit arrival counter, one spare double (16-byte alignment), then the
// per-CTA partial matrices [CTA][m * k].  The counter sits at the front, so one buffer sized for
// the largest m * k serves every smaller call too.
constexpr int kGramHeader = 2;

// Last-arriving CTA: G[e] = sum over CTAs b (in order) of the partial matrices' entry e.
__device__ __forceinline__ void gram_finish(int mk, double *__restrict__ partials,
                                            double *__restrict__ G) {
  __shared__ bool is_last;
  unsigned long long *counter = reinterpret_cast<unsigned long long *>(partials);
  partials += kGramHeader;
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    const unsigned long long t = atomicAdd(counter, 1ull);
    is_last = (t == (unsigned long long)gridDim.x - 1ull);
  }
  __syncthreads();
  if (!is_last) return;
  __threadfence();
  for (int e = threadIdx.x; e < mk; e += kBlkThreads) {
    double s = 0.0;
    for (int b = 0; b < (int)gridDim.x; ++b) s += __ldcg(partials + (int64_t)b * mk + e);
    G[e] = s;
  }
  if (threadIdx.x == 0) *counter = 0ull;
}

// DFMA inner product: thread (ty, tx) of the 16 x 16 grid owns G[ty + 16 r][tx + 16 c],
// r < ceil(m / 16), c < ceil(k / 16) -- up to 6 x 6 accumulators.
__global__ void __launch_bounds__(kBlkThreads, 2)
    block_gram_kernel(int64_t n, int64_t rows_per_cta, int m, const double *__restrict__ X,
                      int64_t ldx, int k, const double *__restrict__ Y, int64_t ldy,
                      const double *__restrict__ w, double *__restrict__ G,
                      double *__restrict__ partials) {
  extern __shared__ double smem[];
  const int ldxs = gram_ld(m, false), ldys = gram_ld(k, false);
  double *Xs = smem, *Ys = smem + kGramRows * ldxs;
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  const int rm = (m + 15) >> 4, rk = (k + 15) >> 4;
  double acc[6][6];
#pragma unroll
  for (int r = 0; r < 6; ++r)
#pragma unroll
    for (int c = 0; c < 6; ++c) acc[r][c] = 0.0;
  const int64_t r0 = (int64_t)blockIdx.x * rows_per_cta;
  const int64_t r1 = r0 + rows_per_cta < n ? r0 + rows_per_cta : n;
  for (int64_t t0 = r0; t0 < r1; t0 += kGramRows) {
    __syncthreads();
    gram_stage(t0, r1, m, X, ldx, w, Xs, ldxs);
    gram_stage(t0, r1, k, Y, ldy, nullptr, Ys, ldys);
    __syncthreads();
#pragma unroll 4
    for (int t = 0; t < kGramRows; ++t) {
      double a[6], b[6];
#pragma unroll
      for (int r = 0; r < 6; ++r) a[r] = (r < rm) ? Xs[t * ldxs + ty + 16 * r] : 0.0;
#pragma unroll
      for (int c = 0; c < 6; ++c) b[c] = (c < rk) ? Ys[t * ldys + tx + 16 * c] : 0.0;
#pragma unroll
      for (int r = 0; r < 6; ++r)
#pragma unroll
        for (int c = 0; c < 6; ++c)
          if (r < rm && c < rk) acc[r][c] = fma(a[r], b[c], acc[r][c]);
    }
  }
  const int mk = m * k;
  double *mine = partials + kGramHeader + (int64_t)blockIdx.x * mk;
#pragma unroll
  for (int r = 0; r < 6; ++r)
#pragma unroll
    for (int c = 0; c < 6; ++c) {
      const int i = ty + 16 * r, j = tx + 16 * c;
      if (r < rm && c < rk && i < m && j < k) mine[i * k + j] = acc[r][c];
    }
  gram_finish(mk, partials, G);
}

// The same product on the FP64 tensor-core path (mma.sync m8n8k4, SASS DMMA): warp q owns the
// 8 x 8 output tiles q, q + 8, ... of the ceil(m/8) x ceil(k/8) grid (at most 18 at 96 x 96).
constexpr int kMmaMaxTiles = 18;

__global__ void __launch_bounds__(kBlkThreads, 2)
    block_gram_mma_kernel(int64_t n, int64_t rows_per_cta, int m, const double *__restrict__ X,
                          int64_t ldx, int k, const double *__restrict__ Y, int64_t ldy,
                          const double *__restrict__ w, double *__restrict__ G,
                          double *__restrict__ partials) {
  extern __shared__ double smem[];
  const int ldxs = gram_ld(m, true), ldys = gram_ld(k, true);
  double *Xs = smem, *Ys = smem + kGramRows * ldxs;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int tm = (m + 7) >> 3, tk = (k + 7) >> 3, ntile = tm * tk;
  const int g = lane >> 2, q4 = lane & 3;
  double acc[kMmaMaxTiles][2];
#pragma unroll
  for (int q = 0; q < kMmaMaxTiles; ++q) acc[q][0] = acc[q][1] = 0.0;
  const int64_t r0 = (int64_t)blockIdx.x * rows_per_cta;
  const int64_t r1 = r0 + rows_per_cta < n ? r0 + rows_per_cta : n;
  for (int64_t t0 = r0; t0 < r1; t0 += kGramRows) {
    __syncthreads();
    gram_stage(t0, r1, m, X, ldx, w, Xs, ldxs);
    gram_stage(t0, r1, k, Y, ldy, nullptr, Ys, ldys);
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < kGramRows; kk += 4) {
#pragma unroll
      for (int q = 0; q < kMmaMaxTiles; ++q) {
        const int tile = warp + 8 * q;
        if (tile < ntile) {
          const int ti = tile / tk, tj = tile % tk;
          // A[i][t] = Xs[t][i] (row g, column q4); B[t][j] = Ys[t][j] (row q4, column g)
          const double a = Xs[(kk + q4) * ldxs + ti * 8 + g];
          const double b = Ys[(kk + q4) * ldys + tj * 8 + g];
          asm volatile(
              "mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0, %1}, {%2}, {%3}, {%0, %1};"
              : "+d"(acc[q][0]), "+d"(acc[q][1])
              : "d"(a), "d"(b));
        }
      }
    }
  }
  const int mk = m * k;
  double *mine = partials + kGramHeader + (int64_t)blockIdx.x * mk;
#pragma unroll
  for (int q = 0; q < kMmaMaxTiles; ++q) {
    const int tile = warp + 8 * q;
    if (tile < ntile) {
      const int ti = tile / tk, tj = tile % tk;
      const int i = ti * 8 + g;
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const int j = tj * 8 + 2 * q4 + h;
        if (i < m && j < k) mine[i * k + j] = acc[q][h];
      }
    }
  }
  gram_finish(mk, partials, G);
}

// Y[j] = beta Y[j] + sum_i C[i*k + j] X[i]: per chunk of kCombRows rows, X is staged as
// Xs[i][t] and thread (ty, tx) forms Y[ty + 16 c][t0 + tx + 16 a], a < 4, c < ceil(k / 16).
__global__ void __launch_bounds__(kBlkThreads)
    block_combine_kernel(int64_t n, int m, const double *__restrict__ X, int64_t ldx, int k,
                         const double *__restrict__ C, double beta, double *__restrict__ Y,
                         int64_t ldy) {
  extern __shared__ double smem[];
  double *Cs = smem;                          // [m][k]
  double *Xs = smem + m * k;                  // [m][kCombRows]
  for (int e = threadIdx.x; e < m * k; e += kBlkThreads) Cs[e] = C[e];
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  const int rk = (k + 15) >> 4;
  const int64_t nchunk = (n + kCombRows - 1) / kCombRows;
  for (int64_t ch = blockIdx.x; ch < nchunk; ch += gridDim.x) {
    const int64_t t0 = ch * kCombRows;
    __syncthreads();
    double v[kCombLoads];                     // all loads first: one latency per chunk
    const int64_t g = t0 + threadIdx.x % kCombRows;
#pragma unroll
    for (int q = 0; q < kCombLoads; ++q) {
      const int e = threadIdx.x + q * kBlkThreads;
      v[q] = (e < m * kCombRows && g < n) ? __ldcs(X + (int64_t)(e / kCombRows) * ldx + g) : 0.0;
    }
#pragma unroll
    for (int q = 0; q < kCombLoads; ++q) {
      const int e = threadIdx.x + q * kBlkThreads;
      if (e < m * kCombRows) Xs[e] = v[q];
    }
    __syncthreads();
    double acc[6][4];
#pragma unroll
    for (int c = 0; c < 6; ++c)
#pragma unroll
      for (int a = 0; a < 4; ++a) acc[c][a] = 0.0;
    for (int i = 0; i < m; ++i) {
      double x[4], cv[6];
#pragma unroll
      for (int a = 0; a < 4; ++a) x[a] = Xs[i * kCombRows + tx + 16 * a];
#pragma unroll
      for (int c = 0; c < 6; ++c) cv[c] = (c < rk && ty + 16 * c < k) ? Cs[i * k + ty + 16 * c] : 0.0;
#pragma unroll
      for (int c = 0; c < 6; ++c)
        if (c < rk)
#pragma unroll
          for (int a = 0; a < 4; ++a) acc[c][a] = fma(cv[c], x[a], acc[c][a]);
    }
#pragma unroll
    for (int c = 0; c < 6; ++c) {
      const int j = ty + 16 * c;
      if (c >= rk || j >= k) continue;
#pragma unroll
      for (int a = 0; a < 4; ++a) {
        const int64_t g = t0 + tx + 16 * a;
        if (g >= n) continue;
        double *yp = Y + (int64_t)j * ldy + g;
        // beta == 0 does not read Y (it may hold anything, NaN included)
        *yp = (beta != 0.0) ? fma(beta, *yp, acc[c][a]) : acc[c][a];
      }
    }
  }
}

// One launch of the Gram kernel: DFMA (block_gram_kernel) or DMMA (block_gram_mma_kernel)
// inner products on the same staging, CTA ranges and reduction.
int gram_launch(bool mma, const char *name, int64_t n, int m, const double *X, int64_t ldx, int k,
                const double *Y, int64_t ldy, const double *w, double *G, double *partials,
                void *stream) {
  SEMK_REQUIRE(n > 0 && m >= 1 && m <= kBlkMax && k >= 1 && k <= kBlkMax,
               std::string(name) + ": need n > 0 and 1 <= m, k <= 96");
  SEMK_REQUIRE(ldx >= n && ldy >= n, std::string(name) + ": strides must be >= n");
  SEMK_REQUIRE(X && Y && G && partials, std::string(name) + ": null pointer");
  const int nb = gram_blocks(n);
  const int64_t chunks = (n + kGramRows - 1) / kGramRows;
  const int64_t rows_per_cta = ((chunks + nb - 1) / nb) * kGramRows;
  const int blocks = (int)((n + rows_per_cta - 1) / rows_per_cta);
  const size_t smem = sizeof(double) * kGramRows * (size_t)(gram_ld(m, mma) + gram_ld(k, mma));
  cudaStream_t st = semk_stream(stream);
  auto kernel = mma ? block_gram_mma_kernel : block_gram_kernel;
  SEMK_CUDA_CHECK(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       (int)smem));
  kernel<<<blocks, kBlkThreads, smem, st>>>(n, rows_per_cta, m, X, ldx, k, Y, ldy, w, G, partials);
  SEMK_LAUNCH_CHECK(mma ? "block_gram_mma_kernel" : "block_gram_kernel");
  return SEMK_OK;
}

// The inner product semk_block_gram_f64 uses: DMMA, 15 % faster than DFMA at m = k = 48 on a B200
// (DESIGN.md section 7).
constexpr bool kGramDefaultMma = true;

}  // namespace

extern "C" int64_t semk_block_gram_partials_len(int m, int k) {
  if (m < 1 || k < 1 || m > kBlkMax || k > kBlkMax) return -1;
  // the arrival counter (zeroed by the caller once; every call leaves it at zero), then
  // kGramMaxBlocks partial matrices
  return kGramHeader + (int64_t)kGramMaxBlocks * m * k;
}

extern "C" int semk_block_gram_f64(int64_t n, int m, const double *X, int64_t ldx, int k,
                                   const double *Y, int64_t ldy, const double *w, double *G,
                                   double *partials, void *stream) {
  return gram_launch(kGramDefaultMma, "semk_block_gram_f64", n, m, X, ldx, k, Y, ldy, w, G,
                     partials, stream);
}

extern "C" int semk_block_gram_dfma_f64(int64_t n, int m, const double *X, int64_t ldx, int k,
                                        const double *Y, int64_t ldy, const double *w, double *G,
                                        double *partials, void *stream) {
  return gram_launch(false, "semk_block_gram_dfma_f64", n, m, X, ldx, k, Y, ldy, w, G, partials,
                     stream);
}

extern "C" int semk_block_gram_dmma_f64(int64_t n, int m, const double *X, int64_t ldx, int k,
                                        const double *Y, int64_t ldy, const double *w, double *G,
                                        double *partials, void *stream) {
  return gram_launch(true, "semk_block_gram_dmma_f64", n, m, X, ldx, k, Y, ldy, w, G, partials,
                     stream);
}

extern "C" int semk_block_combine_f64(int64_t n, int m, const double *X, int64_t ldx, int k,
                                      const double *C, double beta, double *Y, int64_t ldy,
                                      void *stream) {
  SEMK_REQUIRE(n > 0 && m >= 1 && m <= kBlkMax && k >= 1 && k <= kBlkMax,
               "semk_block_combine_f64: need n > 0 and 1 <= m, k <= 96");
  SEMK_REQUIRE(ldx >= n && ldy >= n, "semk_block_combine_f64: strides must be >= n");
  SEMK_REQUIRE(X && C && Y, "semk_block_combine_f64: null pointer");
  const int64_t nchunk = (n + kCombRows - 1) / kCombRows;
  const int blocks = (int)(nchunk < kCombMaxBlocks ? nchunk : kCombMaxBlocks);
  const size_t smem = sizeof(double) * (size_t)m * (k + kCombRows);
  SEMK_CUDA_CHECK(cudaFuncSetAttribute(block_combine_kernel,
                                       cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  block_combine_kernel<<<blocks, kBlkThreads, smem, semk_stream(stream)>>>(n, m, X, ldx, k, C,
                                                                           beta, Y, ldy);
  SEMK_LAUNCH_CHECK("block_combine_kernel");
  return SEMK_OK;
}
