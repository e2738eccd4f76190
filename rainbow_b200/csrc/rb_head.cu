// rb_head.cu -- fused factorised-noise dueling head for small learner batches (sm_100a).
//
// Replaces, for batch <= 64 rows, the reference's per-forward weight composition + four F.linear calls
// (model.py:42-46 NoisyLinear.forward, model.py:73-75 DQN.forward head) and their autograd backward:
//
//   h_s = relu(x W1_s^T + b1_s),  z_s = h_s W2_s^T + b2_s      for the two streams s in {value, advantage}
//   W   = mu + sigma * (eps_out (outer) eps_in),  b = b_mu + b_sigma * eps_out         (model.py:39-44)
//
// The noisy weights are composed ON THE FLY from the factor vectors while the mu/sigma tiles are staged
// into shared memory, so neither weight_epsilon (13.6 MB per net) nor a composed W temporary ever
// exists in HBM, and the skinny (M = 32/64) fp32 GEMMs run on every SM through split-K instead of
// cuBLAS's 64x64 tiles (8 CTAs).  fp32 FMA throughout (the reference computes in fp32); these GEMMs
// are weight-bandwidth bound at this batch size, not tensor-core work.
//
// Kernels: k_head_fc<MT,LAYER> (forward, split-K partials), k_head_logits (bias + dueling combine),
//          k_head_wgrad2 / k_head_dh (layer-2 backward), k_head_bwd1 (layer-1 dW + dx, CTA-pair cluster
//          reducing dx over distributed shared memory), k_noise_factors (Philox factor vectors).

#include <cooperative_groups.h>
#include <cuda_runtime.h>
#include <math_constants.h>
#include <stdint.h>
#include <stdio.h>

#include "rainbow_b200.h"
#include "rb_internal.cuh"

namespace cg = cooperative_groups;

namespace {

constexpr int HT = 128;  // threads per CTA
constexpr int NT = 64;   // output-column tile
constexpr int KT = 32;   // reduction tile
constexpr int LDB = NT + 4;
constexpr int FC_T = 256;  // threads of the forward GEMM kernels

struct HeadDesc {  // device pointers; stream 0 = value, 1 = advantage.  Noise pointers may be null (eval mode).
  const float* w1_mu[2]; const float* w1_sig[2]; const float* b1_mu[2]; const float* b1_sig[2];
  const float* w2_mu[2]; const float* w2_sig[2]; const float* b2_mu[2]; const float* b2_sig[2];
  const float* ei1[2]; const float* eo1[2]; const float* ei2[2]; const float* eo2[2];
  int K1, H, Z, A;
};

struct HeadGrads {  // where the parameter gradients are written (overwritten, not accumulated)
  float* w1_mu[2]; float* w1_sig[2]; float* b1_mu[2]; float* b1_sig[2];
  float* w2_mu[2]; float* w2_sig[2]; float* b2_mu[2]; float* b2_sig[2];
};

HeadDesc to_desc(const rb_head_params* p) {
  HeadDesc d;
  for (int s = 0; s < 2; ++s) {
    d.w1_mu[s] = p->w1_mu[s]; d.w1_sig[s] = p->w1_sigma[s]; d.b1_mu[s] = p->b1_mu[s]; d.b1_sig[s] = p->b1_sigma[s];
    d.w2_mu[s] = p->w2_mu[s]; d.w2_sig[s] = p->w2_sigma[s]; d.b2_mu[s] = p->b2_mu[s]; d.b2_sig[s] = p->b2_sigma[s];
    d.ei1[s] = p->eps_in1[s]; d.eo1[s] = p->eps_out1[s]; d.ei2[s] = p->eps_in2[s]; d.eo2[s] = p->eps_out2[s];
  }
  d.K1 = p->conv_features; d.H = p->hidden; d.Z = p->atoms; d.A = p->actions;
  return d;
}

__device__ __forceinline__ int n2_of(const HeadDesc& d, int s) { return s == 0 ? d.Z : d.A * d.Z; }
__device__ __forceinline__ int col2_of(const HeadDesc& d, int s) { return s == 0 ? 0 : d.Z; }

constexpr int FC_STAGES = 3;

__device__ __forceinline__ void cp_async16_zfill(void* smem, const void* gmem, bool valid) {
  const unsigned sa = (unsigned)__cvta_generic_to_shared(smem);
  const int bytes = valid ? 16 : 0;   // src-size 0: the 16 destination bytes are zero-filled
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;\n" ::"r"(sa), "l"(gmem), "r"(bytes));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;\n" ::"n"(N) : "memory"); }

// ------------------------------------------------------------------------------------------------
// Forward: C[m][n] (partial over a K slice) = sum_k A[m][k] * W[n][k],  W composed while staging.
// grid = (n tiles over both streams, k slices, m tiles), block = 128, micro tile (MT/8) x 4.
// LAYER 1: A = x (two row blocks), N per stream = H, K = K1; result h[m][s*H + n] = relu(sum + b1).
// LAYER 2: A = h, N = Z | A*Z, K = H; result z[m][col2(s) + n] = sum + b2.
// Split-K: every CTA writes its partial tile part[ks][m][col]; the LAST CTA of an output tile to arrive
// (atomic ticket, self-resetting) sums the slices in fixed order s = 0..S-1 (deterministic), applies the
// bias (composed b_mu + b_sigma*eps_out) / ReLU epilogue and writes the final tile.
// ------------------------------------------------------------------------------------------------
template <int MT, int LAYER>
__global__ void __launch_bounds__(FC_T, 2)
k_head_fc(const __grid_constant__ HeadDesc d, const float* __restrict__ x_lo, int m_lo, const float* __restrict__ x_hi,
          int M, float* __restrict__ part, float* __restrict__ out, int* __restrict__ tickets, int kslice) {
  // 256 threads = 16 (ty) x 16 (tx).  Thread (ty, tx) owns rows m0 + ty + 16*i (i < TM) and columns n0 + tx + 16*j
  // (j < 4): with the raw tiles kept [row][k] (k contiguous, row stride 36 floats) both operands are read as
  // conflict-free float4 along k, so no transposed copy of the tiles is ever made.
  constexpr int TM = MT / 16;

  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  const int K = (LAYER == 1) ? d.K1 : d.H;
  const int N0 = (LAYER == 1) ? d.H : d.Z;
  const int tiles0 = (N0 + NT - 1) / NT;
  const int s = ((int)blockIdx.x < tiles0) ? 0 : 1;
  const int n0 = (s == 0 ? (int)blockIdx.x : (int)blockIdx.x - tiles0) * NT;
  const int Ns = (LAYER == 1) ? d.H : n2_of(d, s);
  const int ncols = (LAYER == 1) ? 2 * d.H : d.Z + d.A * d.Z;
  const int colbase = (LAYER == 1) ? s * d.H : col2_of(d, s);
  const int k_begin = blockIdx.y * kslice, k_end = min(K, k_begin + kslice);
  const int m0 = blockIdx.z * MT;
  const float* __restrict__ mu = (LAYER == 1) ? d.w1_mu[s] : d.w2_mu[s];
  const float* __restrict__ sg = (LAYER == 1) ? d.w1_sig[s] : d.w2_sig[s];
  const float* __restrict__ ei = (LAYER == 1) ? d.ei1[s] : d.ei2[s];
  const float* __restrict__ eo = (LAYER == 1) ? d.eo1[s] : d.eo2[s];

  float acc[TM][4];
#pragma unroll
  for (int i = 0; i < TM; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.0f;

  // ---- 3-stage cp.async pipeline: raw tiles (A, mu, sigma; k contiguous) land in shared memory two tiles ahead of
  // the one being multiplied; the noisy weights are composed in place and both operands are consumed straight from the raw tiles ----
  constexpr int A_PER = MT * (KT / 4) / FC_T;  // 16-byte chunks per thread for the A tile (1 or 2)
  constexpr int B_PER = NT * (KT / 4) / FC_T;  // 2
  constexpr int LDR = KT + 4;                  // raw row stride (floats): 144 B, keeps 16-byte alignment
  constexpr int STAGE = (MT + 2 * NT) * LDR;   // floats per stage
  extern __shared__ __align__(16) float fc_raw[];
  auto Araw = [&](int st) { return fc_raw + (size_t)st * STAGE; };
  auto Mraw = [&](int st) { return fc_raw + (size_t)st * STAGE + MT * LDR; };
  auto Sraw = [&](int st) { return fc_raw + (size_t)st * STAGE + (MT + NT) * LDR; };

  auto issue_tile = [&](int k0, int st) {
    if (k0 < k_end) {
#pragma unroll
      for (int j = 0; j < A_PER; ++j) {
        const int idx = tid + j * FC_T, row = idx >> 3, kk = (idx & 7) * 4, k = k0 + kk, m = m0 + row;
        const bool ok = (m < M && k < k_end);
        const float* src = x_lo;
        if (ok) {
          if (LAYER == 1) src = ((m < m_lo) ? x_lo + (size_t)m * K : x_hi + (size_t)(m - m_lo) * K) + k;
          else src = x_lo + (size_t)m * (2 * d.H) + s * d.H + k;   // x_lo = h [M][2H] from the layer-1 launch
        }
        cp_async16_zfill(Araw(st) + row * LDR + kk, src, ok);
      }
#pragma unroll
      for (int j = 0; j < B_PER; ++j) {
        const int idx = tid + j * FC_T, row = idx >> 3, kk = (idx & 7) * 4, k = k0 + kk, n = n0 + row;
        const bool ok = (n < Ns && k < k_end);
        cp_async16_zfill(Mraw(st) + row * LDR + kk, ok ? mu + (size_t)n * K + k : mu, ok);
        if (ei) cp_async16_zfill(Sraw(st) + row * LDR + kk, ok ? sg + (size_t)n * K + k : sg, ok);
      }
    }
    cp_async_commit();   // always commit (possibly empty) so the group accounting stays uniform
  };
  auto compose_tile = [&](int k0, int st) {   // W = mu + sigma * (eps_out[n] * eps_in[k]) in place   (model.py:39,43)
#pragma unroll
    for (int j = 0; j < B_PER; ++j) {
      const int idx = tid + j * FC_T, row = idx >> 3, kk = (idx & 7) * 4, k = k0 + kk, n = n0 + row;
      if (n < Ns && k < k_end) {
        float4 w = *reinterpret_cast<const float4*>(Mraw(st) + row * LDR + kk);
        const float4 sg4 = *reinterpret_cast<const float4*>(Sraw(st) + row * LDR + kk);
        const float e = __ldg(eo + n);
        const float4 e4 = __ldg(reinterpret_cast<const float4*>(ei + k));
        w.x = fmaf(sg4.x, e * e4.x, w.x); w.y = fmaf(sg4.y, e * e4.y, w.y);
        w.z = fmaf(sg4.z, e * e4.z, w.z); w.w = fmaf(sg4.w, e * e4.w, w.w);
        *reinterpret_cast<float4*>(Mraw(st) + row * LDR + kk) = w;
      }
    }
  };

  issue_tile(k_begin, 0);
  issue_tile(k_begin + KT, 1);
  int stage = 0;
  for (int k0 = k_begin; k0 < k_end; k0 += KT) {
    cp_async_wait<FC_STAGES - 2>();   // this thread's copies of tile k0 have landed ...
    __syncthreads();                  // ... and everybody else's; everybody is also done with the previous tile
    issue_tile(k0 + 2 * KT, (stage + 2) % FC_STAGES);   // overwrites the stage the previous tile used
    if (ei) {
      compose_tile(k0, stage);
      __syncthreads();
    }
    const float* At = Araw(stage) + ty * LDR;
    const float* Bt = Mraw(stage) + tx * LDR;
#pragma unroll
    for (int k4 = 0; k4 < KT; k4 += 4) {
      float4 a[TM], b[4];
#pragma unroll
      for (int i = 0; i < TM; ++i) a[i] = *reinterpret_cast<const float4*>(At + i * 16 * LDR + k4);
#pragma unroll
      for (int j = 0; j < 4; ++j) b[j] = *reinterpret_cast<const float4*>(Bt + j * 16 * LDR + k4);
#pragma unroll
      for (int i = 0; i < TM; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          acc[i][j] = fmaf(a[i].x, b[j].x, acc[i][j]);
          acc[i][j] = fmaf(a[i].y, b[j].y, acc[i][j]);
          acc[i][j] = fmaf(a[i].z, b[j].z, acc[i][j]);
          acc[i][j] = fmaf(a[i].w, b[j].w, acc[i][j]);
        }
    }
    stage = (stage + 1) % FC_STAGES;
  }
  cp_async_wait<0>();
  const int S = gridDim.y;
  if (S > 1) {
#pragma unroll
    for (int i = 0; i < TM; ++i) {
      const int m = m0 + ty + 16 * i;
      if (m >= M) continue;
      float* dst = part + ((size_t)blockIdx.y * M + m) * ncols + colbase;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int n = n0 + tx + 16 * j;
        if (n < Ns) __stcg(dst + n, acc[i][j]);
      }
    }
    // ---- split-K semaphore: the last slice to arrive finishes the tile ----
    __shared__ int s_last;
    __threadfence();
    __syncthreads();
    if (tid == 0) {
      int* t = tickets + blockIdx.z * gridDim.x + blockIdx.x;
      const int ticket = atomicAdd(t, 1);
      s_last = (ticket == S - 1);
      if (s_last) *t = 0;  // leave the counter ready for the next launch
    }
    __syncthreads();
    if (!s_last) return;
    __threadfence();
    // ---- cooperative, vectorised reduction of the S partial tiles + epilogue (bias, ReLU for layer 1) ----
    const float* __restrict__ bmu_t = (LAYER == 1) ? d.b1_mu[s] : d.b2_mu[s];
    const float* __restrict__ bsg_t = (LAYER == 1) ? d.b1_sig[s] : d.b2_sig[s];
    const size_t slice = (size_t)M * ncols;
    // All loads of a batch are issued before any is consumed (fully unrolled, constant trip counts): the tail costs a
    // couple of memory round trips instead of one per output element.
    if (LAYER == 1) {  // ncols = 2H and colbase + n0 are multiples of 4: float4 path
      constexpr int IT = MT * (NT / 4) / FC_T;  // float4 outputs per thread (2 or 4)
      float4 a4[IT];
      const float* src[IT];
      bool ok[IT];
#pragma unroll
      for (int it = 0; it < IT; ++it) {
        const int idx = tid + it * FC_T, row = idx / (NT / 4), c = (idx % (NT / 4)) * 4, m = m0 + row, n = n0 + c;
        ok[it] = (m < M && n < Ns);
        src[it] = part + (size_t)(ok[it] ? m : m0) * ncols + colbase + (ok[it] ? n : n0);
        a4[it] = make_float4(0.f, 0.f, 0.f, 0.f);
      }
      for (int sp0 = 0; sp0 < S; sp0 += 4) {
        float4 pv[IT][4];
#pragma unroll
        for (int it = 0; it < IT; ++it)
#pragma unroll
          for (int u = 0; u < 4; ++u)
            pv[it][u] = (sp0 + u < S) ? __ldcg(reinterpret_cast<const float4*>(src[it] + (size_t)(sp0 + u) * slice))
                                      : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int it = 0; it < IT; ++it)
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            a4[it].x += pv[it][u].x; a4[it].y += pv[it][u].y; a4[it].z += pv[it][u].z; a4[it].w += pv[it][u].w;
          }
      }
#pragma unroll
      for (int it = 0; it < IT; ++it) {
        if (!ok[it]) continue;
        const int idx = tid + it * FC_T, row = idx / (NT / 4), c = (idx % (NT / 4)) * 4, m = m0 + row, n = n0 + c;
        float4 bv = __ldg(reinterpret_cast<const float4*>(bmu_t + n));
        if (eo) {
          const float4 bs = __ldg(reinterpret_cast<const float4*>(bsg_t + n));
          const float4 e4 = __ldg(reinterpret_cast<const float4*>(eo + n));
          bv.x = fmaf(bs.x, e4.x, bv.x); bv.y = fmaf(bs.y, e4.y, bv.y); bv.z = fmaf(bs.z, e4.z, bv.z); bv.w = fmaf(bs.w, e4.w, bv.w);
        }
        float4 r4;
        r4.x = fmaxf(a4[it].x + bv.x, 0.f); r4.y = fmaxf(a4[it].y + bv.y, 0.f);
        r4.z = fmaxf(a4[it].z + bv.z, 0.f); r4.w = fmaxf(a4[it].w + bv.w, 0.f);
        *reinterpret_cast<float4*>(out + (size_t)m * ncols + colbase + n) = r4;
      }
    } else {
      constexpr int IT = MT * NT / FC_T;  // scalar outputs per thread (8 or 16), handled 8 at a time
#pragma unroll 1
      for (int h0 = 0; h0 < IT; h0 += 8) {
        float a1[8];
#pragma unroll
        for (int it = 0; it < 8; ++it) a1[it] = 0.0f;
        for (int sp0 = 0; sp0 < S; sp0 += 4) {
          float pv[8][4];
#pragma unroll
          for (int it = 0; it < 8; ++it) {
            const int idx = tid + (h0 + it) * FC_T, row = idx / NT, c = idx % NT, m = m0 + row, n = n0 + c;
            const bool okk = (m < M && n < Ns);
            const float* sp = part + (size_t)(okk ? m : m0) * ncols + colbase + (okk ? n : n0);
#pragma unroll
            for (int u = 0; u < 4; ++u) pv[it][u] = (okk && sp0 + u < S) ? __ldcg(sp + (size_t)(sp0 + u) * slice) : 0.0f;
          }
#pragma unroll
          for (int it = 0; it < 8; ++it)
#pragma unroll
            for (int u = 0; u < 4; ++u) a1[it] += pv[it][u];
        }
#pragma unroll
        for (int it = 0; it < 8; ++it) {
          const int idx = tid + (h0 + it) * FC_T, row = idx / NT, c = idx % NT, m = m0 + row, n = n0 + c;
          if (m >= M || n >= Ns) continue;
          float bv = __ldg(bmu_t + n);
          if (eo) bv = fmaf(__ldg(bsg_t + n), __ldg(eo + n), bv);
          out[(size_t)m * ncols + colbase + n] = a1[it] + bv;
        }
      }
    }
    return;
  }
  // ---- no split (S == 1): epilogue straight from the accumulators ----
  const float* __restrict__ bmu = (LAYER == 1) ? d.b1_mu[s] : d.b2_mu[s];
  const float* __restrict__ bsg = (LAYER == 1) ? d.b1_sig[s] : d.b2_sig[s];
  float bias[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const int n = n0 + tx + 16 * j;
    bias[j] = 0.0f;
    if (n < Ns) {
      bias[j] = __ldg(bmu + n);
      if (eo) bias[j] = fmaf(__ldg(bsg + n), __ldg(eo + n), bias[j]);
    }
  }
#pragma unroll
  for (int i = 0; i < TM; ++i) {
    const int m = m0 + ty + 16 * i;
    if (m >= M) continue;
    float* dst = out + (size_t)m * ncols + colbase;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int n = n0 + tx + 16 * j;
      if (n < Ns) {
        const float v = acc[i][j] + bias[j];
        dst[n] = (LAYER == 1) ? fmaxf(v, 0.0f) : v;
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------
// Layer 2 forward in ONE pass (no split-K, no tickets): z[m][col(s) + n] = sum_k h[m][s*H + k] * W2_s[n][k] + b2_s[n].
// The layer is tiny (357 x 512 weights per stream pair, 11.7 MFLOP at 64 rows) and purely latency bound, so the kernel is
// organised around the number of dependent memory round trips: grid = one CTA per group of F2_ROWS weight rows (90 CTAs for
// 51 atoms x (1 + 6 actions)) x 64-row batch tiles; the CTA's h slab [rows][H] arrives as one 1-D TMA bulk copy per batch
// row (cp.async.bulk + mbarrier: a single memory latency for 128 KB) while all threads compose the CTA's F2_ROWS noisy weight
// rows; thread (m, n) then runs one H-long dot product from shared memory (row stride H + 4 floats: conflict-free float4).
// ------------------------------------------------------------------------------------------------
constexpr int F2_ROWS = 4;
constexpr int F2_T = 256;
constexpr int F2_MT = F2_T / F2_ROWS;   // 64 batch rows per CTA

__device__ __forceinline__ uint32_t f2_smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__global__ void __launch_bounds__(F2_T)
k_head_fc2(const __grid_constant__ HeadDesc d, const float* __restrict__ h, int M, float* __restrict__ z) {
  extern __shared__ __align__(16) float f2_smem[];
  const int H = d.H, LD = H + 4;
  float* hs = f2_smem;                          // [F2_MT][LD]
  float* ws = f2_smem + (size_t)F2_MT * LD;     // [F2_ROWS][LD]
  __shared__ __align__(8) uint64_t bar;
  const int tid = threadIdx.x;
  const int groups0 = (d.Z + F2_ROWS - 1) / F2_ROWS;
  const int s = ((int)blockIdx.x < groups0) ? 0 : 1;
  const int r0 = (s == 0 ? (int)blockIdx.x : (int)blockIdx.x - groups0) * F2_ROWS;
  const int Ns = n2_of(d, s), colbase = col2_of(d, s), ncols = d.Z + d.A * d.Z;
  const int m0 = blockIdx.y * F2_MT, mrows = min(F2_MT, M - m0);
  const uint32_t bar_a = f2_smem_u32(&bar);
  if (tid == 0) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar_a) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  if (tid == 0) {   // the whole activation slab in flight at once
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar_a), "r"((uint32_t)(mrows * H * 4)) : "memory");
    for (int r = 0; r < mrows; ++r)
      asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                   ::"r"(f2_smem_u32(hs + (size_t)r * LD)), "l"(h + (size_t)(m0 + r) * (2 * H) + s * H), "r"((uint32_t)(H * 4)), "r"(bar_a)
                   : "memory");
  }
  {  // W2 rows of this CTA, composed: W = mu + sigma * (eps_out[n] * eps_in[k])   (model.py:39,43)
    const float* __restrict__ mu = d.w2_mu[s];
    const float* __restrict__ sg = d.w2_sig[s];
    const float* ei = d.ei2[s];
    const float* eo = d.eo2[s];
    const int per_row = H >> 2;
    for (int idx = tid; idx < F2_ROWS * per_row; idx += F2_T) {
      const int n = idx / per_row, k4 = (idx - n * per_row) << 2, row = r0 + n;
      float4 w = make_float4(0.f, 0.f, 0.f, 0.f);
      if (row < Ns) {
        w = __ldg(reinterpret_cast<const float4*>(mu + (size_t)row * H + k4));
        if (ei) {
          const float4 s4 = __ldg(reinterpret_cast<const float4*>(sg + (size_t)row * H + k4));
          const float4 e4 = __ldg(reinterpret_cast<const float4*>(ei + k4));
          const float e = __ldg(eo + row);
          w.x = fmaf(s4.x, e * e4.x, w.x); w.y = fmaf(s4.y, e * e4.y, w.y);
          w.z = fmaf(s4.z, e * e4.z, w.z); w.w = fmaf(s4.w, e * e4.w, w.w);
        }
      }
      *reinterpret_cast<float4*>(ws + (size_t)n * LD + k4) = w;
    }
  }
  __syncthreads();
  {  // every thread waits for the bulk copies (phase 0 of the barrier)
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "F2WAIT_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], 0;\n\t"
        "@p bra F2DONE_%=;\n\t"
        "bra F2WAIT_%=;\n\t"
        "F2DONE_%=:\n\t"
        "}\n" ::"r"(bar_a) : "memory");
  }
  const int m = tid / F2_ROWS, n = tid % F2_ROWS, row = r0 + n;
  if (m < mrows && row < Ns) {
    const float* hr = hs + (size_t)m * LD;
    const float* wr = ws + (size_t)n * LD;
    float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;   // four independent chains
#pragma unroll 8
    for (int k = 0; k < H; k += 4) {
      const float4 a = *reinterpret_cast<const float4*>(hr + k);
      const float4 b = *reinterpret_cast<const float4*>(wr + k);
      a0 = fmaf(a.x, b.x, a0); a1 = fmaf(a.y, b.y, a1); a2 = fmaf(a.z, b.z, a2); a3 = fmaf(a.w, b.w, a3);
    }
    float bv = __ldg(d.b2_mu[s] + row);
    if (d.eo2[s]) bv = fmaf(__ldg(d.b2_sig[s] + row), __ldg(d.eo2[s] + row), bv);
    z[(size_t)(m0 + m) * ncols + colbase + row] = ((a0 + a1) + (a2 + a3)) + bv;
  }
}

// q[m][a][z] = zv[z] + za[a][z] - mean_a za[.][z]  (model.py:73-75) from the head output z[m][Z + A*Z].
__global__ void __launch_bounds__(128)
k_head_logits(int Z, int A, const float* __restrict__ z, float* __restrict__ q) {
  const int m = blockIdx.x;
  const float* zr = z + (size_t)m * (Z + A * Z);
  for (int c = threadIdx.x; c < Z; c += blockDim.x) {
    float mean = 0.0f;
    for (int a = 0; a < A; ++a) mean += __ldg(zr + Z + a * Z + c);
    mean = mean / (float)A;
    const float zv = __ldg(zr + c);
    for (int a = 0; a < A; ++a) q[((size_t)m * A + a) * Z + c] = zv + __ldg(zr + Z + a * Z + c) - mean;
  }
}

// ------------------------------------------------------------------------------------------------
// Layer-2 backward, weight gradients: g[o][k] = sum_m dz[m][col(o)] * h[m][s*H + k]   (both operands are
// "reduction-major", so tiles are staged without transposition); g_sigma = g * eps_out[o]*eps_in[k].
// grid = (o tiles over both streams, H / 64), micro tile 8 (o) x 4 (k), reduction over m in chunks of 32.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(HT)
k_head_wgrad2(const __grid_constant__ HeadDesc d, const __grid_constant__ HeadGrads g, const float* __restrict__ dz,
              const float* __restrict__ h, int B) {
  __shared__ __align__(16) float Ds[32][LDB];  // dz chunk [m][o]
  __shared__ __align__(16) float Hs[32][LDB];  // h chunk  [m][k]
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  const int tiles0 = (d.Z + NT - 1) / NT;
  const int s = ((int)blockIdx.x < tiles0) ? 0 : 1;
  const int o0 = (s == 0 ? (int)blockIdx.x : (int)blockIdx.x - tiles0) * NT;
  const int Ns = n2_of(d, s), colbase = col2_of(d, s), ncols = d.Z + d.A * d.Z;
  const int k0 = blockIdx.y * NT;
  float acc[8][4];
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.0f;
  float bsum = 0.0f;  // bias gradient, threads 0..63 of the k-tile-0 CTAs
  for (int mb = 0; mb < B; mb += 32) {
    for (int idx = tid; idx < 32 * NT; idx += HT) {
      const int mm = idx / NT, c = idx % NT, m = mb + mm;
      Ds[mm][c] = (m < B && o0 + c < Ns) ? __ldg(dz + (size_t)m * ncols + colbase + o0 + c) : 0.0f;
      Hs[mm][c] = (m < B && k0 + c < d.H) ? __ldg(h + (size_t)m * (2 * d.H) + s * d.H + k0 + c) : 0.0f;
    }
    __syncthreads();
#pragma unroll 8
    for (int mm = 0; mm < 32; ++mm) {
      const float4 a0 = *reinterpret_cast<const float4*>(&Ds[mm][ty * 8]);
      const float4 a1 = *reinterpret_cast<const float4*>(&Ds[mm][ty * 8 + 4]);
      const float4 b = *reinterpret_cast<const float4*>(&Hs[mm][tx * 4]);
      const float a[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        acc[i][0] = fmaf(a[i], b.x, acc[i][0]); acc[i][1] = fmaf(a[i], b.y, acc[i][1]);
        acc[i][2] = fmaf(a[i], b.z, acc[i][2]); acc[i][3] = fmaf(a[i], b.w, acc[i][3]);
      }
    }
    if (blockIdx.y == 0 && tid < NT)
      for (int mm = 0; mm < 32; ++mm) bsum += Ds[mm][tid];
    __syncthreads();
  }
  const float* ei = d.ei2[s];
  const float* eo = d.eo2[s];
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int o = o0 + ty * 8 + i;
    if (o >= Ns) continue;
    const float e = eo ? __ldg(eo + o) : 0.0f;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int k = k0 + tx * 4 + j;
      if (k >= d.H) continue;
      g.w2_mu[s][(size_t)o * d.H + k] = acc[i][j];
      g.w2_sig[s][(size_t)o * d.H + k] = ei ? acc[i][j] * (e * __ldg(ei + k)) : 0.0f;
    }
  }
  if (blockIdx.y == 0 && tid < NT && o0 + tid < Ns) {
    g.b2_mu[s][o0 + tid] = bsum;
    g.b2_sig[s][o0 + tid] = eo ? bsum * __ldg(eo + o0 + tid) : 0.0f;
  }
}

// Layer-2 backward, input gradient with the ReLU mask of layer 1 folded in:
// dh[m][s*H + k] = (h > 0) * sum_o dz[m][col(o)] * W2_s[o][k].   B <= 32 rows.
// The layer is tiny (1.5 MB of weights) and sits on the critical path between the loss and the layer-1 backward, so the
// kernel is organised around ONE memory round trip: grid = 2 streams x H/8 CTAs; a CTA stages the stream's whole dz block
// [32][Ns] and its 8-column slab of W2 (mu and sigma rows, 32 contiguous bytes each) with cp.async, all in flight at once,
// composes the noisy weights in place, and thread (m, k) runs one Ns-long dot product out of shared memory.
// Writes dh [B][2H] and its transpose dhT [2H][32] (rows past B zero) for k_head_bwd1.
constexpr int DH_KB = 8;    // hidden units per CTA
constexpr int DH_T = 256;   // 32 batch rows x 8 hidden units

// the dz block [32][ld_dz] plus the mu and sigma slabs [Ns][DH_KB] of the wider stream
int head_dh_ld(int Z, int A) { return (A * Z > Z ? A * Z : Z) | 1; }   // odd row stride: the 32 rows of a column hit 32 different banks
size_t head_dh_smem(int Z, int A) {
  const int ns_max = A * Z > Z ? A * Z : Z;
  return ((size_t)32 * head_dh_ld(Z, A) + 2 * (size_t)((ns_max + 3) & ~3) * DH_KB) * sizeof(float);
}

__device__ __forceinline__ void cp_async16(void* smem, const void* gmem) {
  unsigned sa = (unsigned)__cvta_generic_to_shared(smem);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(sa), "l"(gmem));
}
__device__ __forceinline__ void cp_async4(void* smem, const void* gmem) {
  unsigned sa = (unsigned)__cvta_generic_to_shared(smem);
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;\n" ::"r"(sa), "l"(gmem));
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.commit_group;\ncp.async.wait_group 0;\n" ::: "memory"); }

__global__ void __launch_bounds__(DH_T)
k_head_dh(const __grid_constant__ HeadDesc d, const float* __restrict__ dz, const float* __restrict__ h, int B,
          float* __restrict__ dh, float* __restrict__ dhT, int ld_dz) {
  extern __shared__ __align__(16) float smem_dh[];
  const int s = blockIdx.y, k0 = blockIdx.x * DH_KB;
  const int Ns = n2_of(d, s), colbase = col2_of(d, s), ncols = d.Z + d.A * d.Z, H = d.H;
  float* Dz = smem_dh;                                  // [32][ld_dz]   dz block of this stream
  float* Wm = Dz + 32 * ld_dz;                          // [Ns][DH_KB]   mu slab, composed in place
  float* Wsg = Wm + (size_t)((Ns + 3) & ~3) * DH_KB;    // [Ns][DH_KB]   sigma slab
  const int tid = threadIdx.x;
  const float* ei = d.ei2[s];
  const float* eo = d.eo2[s];
  // dz rows start at arbitrary 4-byte offsets (colbase = Z for the advantage stream): 4-byte cp.async
  for (int idx = tid; idx < B * Ns; idx += DH_T) {
    const int m = idx / Ns, o = idx - m * Ns;
    cp_async4(Dz + m * ld_dz + o, dz + (size_t)m * ncols + colbase + o);
  }
  for (int idx = tid; idx < Ns * 2; idx += DH_T) {      // two 16-byte chunks per weight row and tensor
    const int o = idx >> 1, c = (idx & 1) * 4;
    cp_async16(Wm + o * DH_KB + c, d.w2_mu[s] + (size_t)o * H + k0 + c);
    if (ei) cp_async16(Wsg + o * DH_KB + c, d.w2_sig[s] + (size_t)o * H + k0 + c);
  }
  const int m = tid >> 3, k = tid & 7;
  const float hv = (m < B) ? __ldg(h + (size_t)m * (2 * H) + s * H + k0 + k) : 0.0f;
  // noise factors of this thread's weight chunks, requested while the copies are still in flight
  constexpr int DH_MAXI = 8;
  float4 ek_r = make_float4(0.f, 0.f, 0.f, 0.f);
  float eo_r[DH_MAXI];
  if (ei) {
    ek_r = __ldg(reinterpret_cast<const float4*>(ei + k0 + (tid & 1) * 4));   // idx & 1 == tid & 1 (DH_T is even)
#pragma unroll
    for (int u = 0; u < DH_MAXI; ++u) {
      const int idx = tid + u * DH_T;
      eo_r[u] = (idx < Ns * 2) ? __ldg(eo + (idx >> 1)) : 0.0f;
    }
  }
  cp_async_wait_all();
  __syncthreads();
  if (ei) {  // W2 = mu + sigma * (eps_out[o] * eps_in[k]) in place
    for (int idx = tid, u = 0; idx < Ns * 2; idx += DH_T, ++u) {
      const int o = idx >> 1, c = (idx & 1) * 4;
      float4 w = *reinterpret_cast<const float4*>(Wm + o * DH_KB + c);
      const float4 sg = *reinterpret_cast<const float4*>(Wsg + o * DH_KB + c);
      const float4 ek = ek_r;
      float e = 0.0f;
      if (u < DH_MAXI) {
#pragma unroll
        for (int q = 0; q < DH_MAXI; ++q)
          if (q == u) e = eo_r[q];
      } else {
        e = __ldg(eo + o);
      }
      w.x = fmaf(sg.x, e * ek.x, w.x); w.y = fmaf(sg.y, e * ek.y, w.y);
      w.z = fmaf(sg.z, e * ek.z, w.z); w.w = fmaf(sg.w, e * ek.w, w.w);
      *reinterpret_cast<float4*>(Wm + o * DH_KB + c) = w;
    }
    __syncthreads();
  }
  float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
  if (m < B) {
    const float* dr = Dz + m * ld_dz;
    int o = 0;
    for (; o + 3 < Ns; o += 4) {
      a0 = fmaf(dr[o], Wm[o * DH_KB + k], a0);
      a1 = fmaf(dr[o + 1], Wm[(o + 1) * DH_KB + k], a1);
      a2 = fmaf(dr[o + 2], Wm[(o + 2) * DH_KB + k], a2);
      a3 = fmaf(dr[o + 3], Wm[(o + 3) * DH_KB + k], a3);
    }
    for (; o < Ns; ++o) a0 = fmaf(dr[o], Wm[o * DH_KB + k], a0);
  }
  const float v = (m < B && hv > 0.f) ? ((a0 + a1) + (a2 + a3)) : 0.0f;
  if (m < B) dh[(size_t)m * (2 * H) + s * H + k0 + k] = v;
  dhT[(size_t)(s * H + k0 + k) * 32 + m] = v;
}

// ------------------------------------------------------------------------------------------------
// Layer-1 backward for B <= 32 rows: one pass over W1 produces BOTH the weight gradients
//   g[o][k] = sum_m dh[m][o] * x[m][k]            (written straight into the flat gradient buffer)
// and the input gradient  dx[m][k] = sum_s sum_o dh[m][s*H+o] * W1_s[o][k].
// grid = (K1/32, 2 streams x 2 halves of the stream's rows) launched as clusters of 4 CTAs along y: three CTAs
// hand their dx partial to rank 0 through distributed shared memory (fixed rank order -> deterministic).
// 256 threads: warps 0-3 compute the weight-gradient tile of the current 32-row chunk of W1 while warps
// 4-7 accumulate the input gradient from the same staged tiles, both as error-compensated TF32 products on the warp-level
// tensor-core path (mma.sync.m16n8k8, three MMAs per product: fp32-equivalent results) -- the FFMA version of this kernel
// was instruction-issue bound (12.2 M warp instructions, FMA pipe 30 % busy: r02b ncu).  The chunks (raw mu / sigma rows, the dh chunk in both
// orientations -- k_head_dh writes dh [m][2H] and its transpose dhT [2H][32], so nothing is transposed through shared
// memory here) arrive through a 3-stage cp.async ring, two chunks ahead of the one being consumed: the eight dependent
// memory latencies of the old single-stage register prefetch collapse into one plus streaming.
// ------------------------------------------------------------------------------------------------
constexpr int B1_K = 32;   // k columns per CTA
constexpr int B1_O = 32;   // rows of W1 per chunk
constexpr int B1_T = 256;  // threads

constexpr int B1_STAGES = 3;                 // cp.async ring: two chunks in flight ahead of the one being consumed (3 CTAs per SM: one wave)
// Row strides (floats) chosen for the mma.m16n8k8 fragment loads: "A" tiles (rows indexed by lane / 4, columns by lane % 4)
// want a stride = 4 (mod 32), "B" tiles (rows by lane % 4, columns by lane / 4) a stride = 8 (mod 32): both conflict free.
constexpr int B1_LDW = B1_K + 8;             // W mu / sigma chunks [o][k]   (B operand of the dx product)
constexpr int B1_LDD = B1_K + 4;             // dh chunks [m][o] and [o][m]  (A operands)
constexpr int B1_STAGE = 2 * 32 * B1_LDW + 2 * 32 * B1_LDD;   // floats per stage: W mu (composed in place) | W sigma | dh | dhT

// ---- error-compensated TF32 on the warp-level tensor-core path (mma.sync.m16n8k8): fp32-equivalent products -------------
// hi = the value with its low 13 mantissa bits cleared (a TF32 number), lo = value - hi (exact);
// D += Alo*Bhi + Ahi*Blo + Ahi*Bhi, fp32 accumulation (the dropped lo*lo term is 2^-22 relative).
__device__ __forceinline__ void tf32_split(float v, uint32_t& hi, uint32_t& lo) {
  hi = __float_as_uint(v) & 0xFFFFE000u;
  lo = __float_as_uint(__fsub_rn(v, __uint_as_float(hi)));
}
__device__ __forceinline__ void mma_tf32(float (&c)[4], const uint32_t (&a)[4], const uint32_t (&b)[2]) {
  asm volatile("mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b[0]), "r"(b[1]));
}
// one 16 x 8 output block, K = 8: A block at `a` (row stride lda, rows = M index, columns = K index), B fragments given
__device__ __forceinline__ void mma3_block(float (&c)[4], const float* a, int lda, const uint32_t (&bhi)[2], const uint32_t (&blo)[2],
                                           int gid, int tig) {
  uint32_t ahi[4], alo[4];
  tf32_split(a[gid * lda + tig], ahi[0], alo[0]);
  tf32_split(a[(gid + 8) * lda + tig], ahi[1], alo[1]);
  tf32_split(a[gid * lda + tig + 4], ahi[2], alo[2]);
  tf32_split(a[(gid + 8) * lda + tig + 4], ahi[3], alo[3]);
  mma_tf32(c, alo, bhi);
  mma_tf32(c, ahi, blo);
  mma_tf32(c, ahi, bhi);
}

__global__ void __cluster_dims__(1, 4, 1) __launch_bounds__(B1_T)
k_head_bwd1(const __grid_constant__ HeadDesc d, const __grid_constant__ HeadGrads g, const float* __restrict__ x,
            const float* __restrict__ dh, const float* __restrict__ dhT, int B, float* __restrict__ dx, int relu_mask_x) {
  extern __shared__ __align__(16) float b1_ring[];     // [B1_STAGES][B1_STAGE]
  __shared__ __align__(16) float Xs[32][B1_K + 8];    // x slice [m][k]  (B operand of the weight-gradient product)
  __shared__ __align__(16) float Red[32][B1_K + 4];   // dx partial handed over the cluster
  __shared__ float EoAll[512];                         // eps_out of every row this CTA walks (H / 2 <= 512), fetched once
  cg::cluster_group cluster = cg::this_cluster();
  const int tid = threadIdx.x;
  // warps 0-3: weight-gradient tile [32 o][32 k] of the current chunk; warps 4-7: input gradient [32 m][32 k].  Warp w of a
  // role owns the 8 columns n0 = 8 w of its role's tile, both 16-row blocks (mma.m16n8k8 fragments: gid = lane / 4, tig = lane % 4)
  const int role = tid >> 7, rt = tid & 127, lane = tid & 31, gid = lane >> 2, tig = lane & 3, n0 = ((tid >> 5) & 3) * 8;
  // cluster of 4 CTAs along y: (stream, half of the stream's W1 rows); rank 0 sums the four dx partials
  const int s = blockIdx.y >> 1, half = blockIdx.y & 1, k0 = blockIdx.x * B1_K, K = d.K1, H = d.H;
  const int o_begin = half * (H / 2), n_chunks = (H / 2) / B1_O;
  const float* __restrict__ mu = d.w1_mu[s];
  const float* __restrict__ sg = d.w1_sig[s];
  const float* ei = d.ei1[s];
  const float* eo = d.eo1[s];
  const int st_r = tid >> 3, st_c = (tid & 7) * 4;   // staging coordinates: one 16-byte chunk of each of the four tiles

  auto Wm = [&](int st) { return b1_ring + (size_t)st * B1_STAGE; };
  auto Wsg = [&](int st) { return b1_ring + (size_t)st * B1_STAGE + 32 * B1_LDW; };
  auto Dm = [&](int st) { return b1_ring + (size_t)st * B1_STAGE + 2 * 32 * B1_LDW; };                 // dh chunk [m][o]
  auto Dt = [&](int st) { return b1_ring + (size_t)st * B1_STAGE + 2 * 32 * B1_LDW + 32 * B1_LDD; };   // dh chunk [o][m]
  auto issue = [&](int c) {   // chunk c of this CTA's rows -> stage c % B1_STAGES (always commits, possibly an empty group)
    if (c < n_chunks) {
      const int st = c % B1_STAGES, ob = o_begin + c * B1_O;
      cp_async16_zfill(Wm(st) + st_r * B1_LDW + st_c, mu + (size_t)(ob + st_r) * K + k0 + st_c, true);
      if (ei) cp_async16_zfill(Wsg(st) + st_r * B1_LDW + st_c, sg + (size_t)(ob + st_r) * K + k0 + st_c, true);
      const bool row_ok = st_r < B;
      cp_async16_zfill(Dm(st) + st_r * B1_LDD + st_c, row_ok ? dh + (size_t)st_r * (2 * H) + s * H + ob + st_c : dh, row_ok);
      cp_async16_zfill(Dt(st) + st_r * B1_LDD + st_c, dhT + (size_t)(s * H + ob + st_r) * 32 + st_c, true);
    }
    cp_async_commit();
  };
  // (a per-chunk __ldg of eps_out inside issue() put one exposed global latency in front of every chunk: r02 ncu, 12 % of
  // the kernel's stall samples on the dependent STS)
  for (int i = tid; i < H / 2; i += B1_T) EoAll[i] = eo ? __ldg(eo + o_begin + i) : 0.0f;

#pragma unroll
  for (int c = 0; c < B1_STAGES - 1; ++c) issue(c);
  {  // x slice: 32 rows x 8 float4 = 256 float4, one per thread
    const int m = tid >> 3, kk = (tid & 7) * 4;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (m < B) v = __ldg(reinterpret_cast<const float4*>(x + (size_t)m * K + k0 + kk));
    *reinterpret_cast<float4*>(&Xs[m][kk]) = v;
  }
  const float ei0 = ei ? __ldg(ei + k0 + n0 + 2 * tig) : 0.0f, ei1v = ei ? __ldg(ei + k0 + n0 + 2 * tig + 1) : 0.0f;
  float4 e4s = make_float4(0.f, 0.f, 0.f, 0.f);
  if (ei) e4s = __ldg(reinterpret_cast<const float4*>(ei + k0 + st_c));

  float acc[2][4];   // input-gradient accumulators (mma C fragments of the two 16-row blocks), kept across the chunks
#pragma unroll
  for (int i = 0; i < 2; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.0f;
  __syncthreads();   // Xs is complete
  // the weight-gradient product's B operand (x slice, K index = batch row) never changes: fragments split once
  uint32_t xhi[4][2], xlo[4][2];
  if (role == 0) {
#pragma unroll
    for (int ks = 0; ks < 4; ++ks) {
      tf32_split(Xs[8 * ks + tig][n0 + gid], xhi[ks][0], xlo[ks][0]);
      tf32_split(Xs[8 * ks + tig + 4][n0 + gid], xhi[ks][1], xlo[ks][1]);
    }
  }

  for (int c = 0; c < n_chunks; ++c) {
    const int st = c % B1_STAGES, ob = o_begin + c * B1_O;
    cp_async_wait<B1_STAGES - 2>();   // this thread's copies of chunk c have landed ...
    __syncthreads();                  // ... and everybody else's; everybody is also done with chunk c - 1
    issue(c + B1_STAGES - 1);         // overwrites the stage chunk c - 1 used
    if (ei) {                         // W = mu + sigma * (eps_out[o] * eps_in[k]) in place   (model.py:39,43)
      float4 w = *reinterpret_cast<const float4*>(Wm(st) + st_r * B1_LDW + st_c);
      const float4 sg4 = *reinterpret_cast<const float4*>(Wsg(st) + st_r * B1_LDW + st_c);
      const float e = EoAll[c * B1_O + st_r];
      w.x = fmaf(sg4.x, e * e4s.x, w.x); w.y = fmaf(sg4.y, e * e4s.y, w.y);
      w.z = fmaf(sg4.z, e * e4s.z, w.z); w.w = fmaf(sg4.w, e * e4s.w, w.w);
      *reinterpret_cast<float4*>(Wm(st) + st_r * B1_LDW + st_c) = w;
      __syncthreads();
    }
    if (role == 0) {
      // ---- weight gradient tile [32 o][32 k] = dhT chunk [o][m] x x slice [m][k]: reduction over the batch rows ----
      const float* DsT = Dt(st);
#pragma unroll
      for (int mb = 0; mb < 2; ++mb) {
        float ga[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
        for (int ks = 0; ks < 4; ++ks) mma3_block(ga, DsT + (16 * mb) * B1_LDD + 8 * ks, B1_LDD, xhi[ks], xlo[ks], gid, tig);
#pragma unroll
        for (int hrow = 0; hrow < 2; ++hrow) {   // C fragment: rows gid and gid + 8, columns 2 tig and 2 tig + 1
          const int ol = 16 * mb + gid + 8 * hrow;
          const size_t off = (size_t)(ob + ol) * K + k0 + n0 + 2 * tig;
          const float g0 = ga[2 * hrow], g1 = ga[2 * hrow + 1];
          __stcs(reinterpret_cast<float2*>(g.w1_mu[s] + off), make_float2(g0, g1));
          const float e = EoAll[c * B1_O + ol];
          __stcs(reinterpret_cast<float2*>(g.w1_sig[s] + off), make_float2(g0 * (e * ei0), g1 * (e * ei1v)));
        }
      }
      if (blockIdx.x == 0 && rt < B1_O) {  // bias gradients of this chunk's rows
        const float* Ds = Dm(st);
        float bs = 0.0f;
        for (int m = 0; m < 32; ++m) bs += Ds[m * B1_LDD + rt];
        g.b1_mu[s][ob + rt] = bs;
        g.b1_sig[s][ob + rt] = bs * EoAll[c * B1_O + rt];
      }
    } else {
      // ---- input gradient [32 m][32 k] += dh chunk [m][o] x composed W chunk [o][k]: reduction over the chunk's rows ----
      const float* Ds = Dm(st);
      const float* Ws = Wm(st);
#pragma unroll
      for (int ks = 0; ks < 4; ++ks) {
        uint32_t whi[2], wlo[2];
        tf32_split(Ws[(8 * ks + tig) * B1_LDW + n0 + gid], whi[0], wlo[0]);
        tf32_split(Ws[(8 * ks + tig + 4) * B1_LDW + n0 + gid], whi[1], wlo[1]);
#pragma unroll
        for (int mb = 0; mb < 2; ++mb) mma3_block(acc[mb], Ds + (16 * mb) * B1_LDD + 8 * ks, B1_LDD, whi, wlo, gid, tig);
      }
    }
  }
  cp_async_wait<0>();
  // ---- dx = sum of the four partials (fixed rank order), over distributed shared memory ----
  const unsigned rank = cluster.block_rank();
  if (rank != 0 && role == 1) {
#pragma unroll
    for (int mb = 0; mb < 2; ++mb)
#pragma unroll
      for (int hrow = 0; hrow < 2; ++hrow)
        *reinterpret_cast<float2*>(&Red[16 * mb + gid + 8 * hrow][n0 + 2 * tig]) = make_float2(acc[mb][2 * hrow], acc[mb][2 * hrow + 1]);
  }
  cluster.sync();
  if (rank == 0 && role == 1) {
#pragma unroll
    for (int r = 1; r < 4; ++r) {
      const float* remote = cluster.map_shared_rank(&Red[0][0], r);
#pragma unroll
      for (int mb = 0; mb < 2; ++mb)
#pragma unroll
        for (int hrow = 0; hrow < 2; ++hrow) {
          const float2 v = *reinterpret_cast<const float2*>(remote + (16 * mb + gid + 8 * hrow) * (B1_K + 4) + n0 + 2 * tig);
          acc[mb][2 * hrow] += v.x;
          acc[mb][2 * hrow + 1] += v.y;
        }
    }
#pragma unroll
    for (int mb = 0; mb < 2; ++mb)
#pragma unroll
      for (int hrow = 0; hrow < 2; ++hrow) {
        const int m = 16 * mb + gid + 8 * hrow;
        if (m < B) {
          float2 o2 = make_float2(acc[mb][2 * hrow], acc[mb][2 * hrow + 1]);
          if (relu_mask_x) {  // x = relu(conv output): fold that ReLU's backward in (x > 0 <=> pre-activation > 0)
            const float2 xv = *reinterpret_cast<const float2*>(&Xs[m][n0 + 2 * tig]);
            o2.x = xv.x > 0.f ? o2.x : 0.f;
            o2.y = xv.y > 0.f ? o2.y : 0.f;
          }
          *reinterpret_cast<float2*>(dx + (size_t)m * K + k0 + n0 + 2 * tig) = o2;
        }
      }
  }
  cluster.sync();  // remote shared memory must outlive the reads above
}

// ------------------------------------------------------------------------------------------------
// Factor vectors f(eps_in), f(eps_out) of every NoisyLinear of a net: one CTA, same Philox indexing as
// k_noisy_resample (normal g of stream `which` for draw `ctr`), so factors + outer product == K6.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(1024)
k_noise_factors(float* __restrict__ f_in, int n_in, float* __restrict__ f_out, int n_out, const float* __restrict__ x_in,
                const float* __restrict__ x_out, uint64_t seed, unsigned long long* rng_counter) {
  const unsigned long long ctr = rng_counter ? *rng_counter : 0ull;
  for (int which = 0; which < 2; ++which) {
    float* dst = which ? f_out : f_in;
    const float* src = which ? x_out : x_in;
    const int n = which ? n_out : n_in;
    if (src) {
      for (int i = threadIdx.x; i < n; i += blockDim.x) dst[i] = rbi::scale_noise(__ldg(src + i));
    } else {
      for (int blk = threadIdx.x; blk * 4 < n; blk += blockDim.x) {
        float4 z = rbi::normal4(seed, ctr, (uint32_t)which, (uint32_t)blk);
        float zz[4] = {z.x, z.y, z.z, z.w};
#pragma unroll
        for (int q = 0; q < 4; ++q)
          if (blk * 4 + q < n) dst[blk * 4 + q] = rbi::scale_noise(zz[q]);
      }
    }
  }
  __syncthreads();
  if (threadIdx.x == 0 && rng_counter && !x_in) *rng_counter = ctr + 1ull;
}

// Conv bias gradient: out[c] = sum over (batch, pixels) of g[b][c][hw].  One CTA per channel, fixed-order tree
// reduction (deterministic); replaces a library reduction that runs this shape on 4 CTAs.
__global__ void __launch_bounds__(256)
k_bias_grad(const float* __restrict__ g, int B, int C, int HW, float* __restrict__ out) {
  __shared__ float s_red[8];
  const int c = blockIdx.x;
  float acc = 0.0f;
  for (int i = threadIdx.x; i < B * HW; i += 256) {
    const int b = i / HW, p = i - b * HW;
    acc += __ldg(g + ((size_t)b * C + c) * HW + p);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    float t = 0.0f;
    for (int w = 0; w < 8; ++w) t += s_red[w];
    out[c] = t;
  }
}

// ------------------------------------------------------------------------------------------------
// Weight gradient of the FIRST conv layer (no data gradient follows it, so in the hand-scheduled backward this is the one
// library launch left alone on the critical path: cuDNN's wgrad_alg0_engine takes 31 us for 105 MFLOP at batch 32):
//   dW[oc][ic][ky][kx] = sum_{b,y,x} g[b][oc][y][x] * in[b][ic][y*S + ky][x*S + kx]            (fp32 FMA, fixed order)
// grid = (bands of output rows, B): a CTA stages its slab of the input (the rows its band touches, all channels) and of g
// in shared memory with every load in flight at once, thread (oc group, kernel row (ic, ky)) accumulates a 4 x KW register
// tile over the band's positions, and the per-CTA partial tiles are summed in CTA order by k_conv_wgrad_reduce
// (deterministic; the partials stay in L2).
// ------------------------------------------------------------------------------------------------
constexpr int CW_OCT = 4;   // output channels per thread

template <int KW>
__global__ void __launch_bounds__(256)
k_conv_wgrad_first(const float* __restrict__ g, const float* __restrict__ in, int IC, int IH, int IW, int OC, int OH, int OW,
                   int S, int RB, float* __restrict__ part) {
  extern __shared__ __align__(16) float cw_smem[];
  const int band = blockIdx.x, b = blockIdx.y, tid = threadIdx.x, nthr = blockDim.x;
  const int y0 = band * RB, rows = min(RB, OH - y0);          // output rows [y0, y0 + rows)
  const int in_rows = (RB - 1) * S + KW;                       // input rows a full band touches (square kernel)
  const int xs_ld = in_rows * IW;                              // floats per channel slab
  float* xs = cw_smem;                                         // [IC][in_rows][IW]
  float* gs = cw_smem + (size_t)IC * xs_ld;                    // [OC][RB * OW]
  const int have_rows = min(in_rows, IH - y0 * S);
  const int n_w = OC * IC * KW * KW;
  // both slabs are contiguous per channel in global memory; cp.async keeps every 16-byte chunk in flight at once
  const bool al = (IW % 4 == 0) && (OW % 4 == 0) && ((((uintptr_t)g | (uintptr_t)in) & 15) == 0);
  if (al) {
    const int xc = have_rows * IW / 4, gc = rows * OW / 4;
    for (int i = tid; i < IC * xc; i += nthr) {
      const int ic = i / xc, c = i - ic * xc;
      cp_async16(xs + ic * xs_ld + 4 * c, in + ((size_t)(b * IC + ic) * IH + (size_t)y0 * S) * IW + 4 * c);
    }
    for (int i = tid; i < OC * gc; i += nthr) {
      const int oc = i / gc, c = i - oc * gc;
      cp_async16(gs + oc * (RB * OW) + 4 * c, g + ((size_t)(b * OC + oc) * OH + y0) * OW + 4 * c);
    }
    cp_async_wait_all();
  } else {
    for (int ic = 0; ic < IC; ++ic) {
      const float* src = in + ((size_t)(b * IC + ic) * IH + (size_t)y0 * S) * IW;
      for (int i = tid; i < have_rows * IW; i += nthr) xs[ic * xs_ld + i] = __ldg(src + i);
    }
    for (int oc = 0; oc < OC; ++oc) {
      const float* src = g + ((size_t)(b * OC + oc) * OH + y0) * OW;
      for (int i = tid; i < rows * OW; i += nthr) gs[oc * (RB * OW) + i] = __ldg(src + i);
    }
  }
  __syncthreads();
  float* dst = part + (size_t)(b * gridDim.x + band) * (size_t)(n_w + OC);
  const bool vec = (S % 4 == 0) && (IW % 4 == 0);
  const int krows = IC * KW;                                    // kernel rows (ic, ky)
  const int kr = tid % krows, og = tid / krows;                 // this thread: kernel row kr, channels og*4 .. og*4+3
  const int ic = kr / KW, ky = kr % KW;
  float acc[CW_OCT][KW];
#pragma unroll
  for (int i = 0; i < CW_OCT; ++i)
#pragma unroll
    for (int j = 0; j < KW; ++j) acc[i][j] = 0.0f;
  if (og * CW_OCT < OC) {
    for (int yy = 0; yy < rows; ++yy) {
      const float* xrow = xs + ic * xs_ld + (yy * S + ky) * IW;
      const float* grow = gs + (og * CW_OCT) * (RB * OW) + yy * OW;
      for (int xx = 0; xx < OW; ++xx) {
        float xv[KW], gv[CW_OCT];
        if ((KW % 4 == 0) && vec) {   // 16-byte aligned kernel rows (stride and row pitch multiples of 4 floats)
#pragma unroll
          for (int j = 0; j < KW; j += 4) {
            const float4 v = *reinterpret_cast<const float4*>(xrow + xx * S + j);
            xv[j] = v.x; xv[j + 1] = v.y; xv[j + 2] = v.z; xv[j + 3] = v.w;
          }
        } else {
#pragma unroll
          for (int j = 0; j < KW; ++j) xv[j] = xrow[xx * S + j];
        }
#pragma unroll
        for (int i = 0; i < CW_OCT; ++i) gv[i] = grow[i * (RB * OW) + xx];
#pragma unroll
        for (int i = 0; i < CW_OCT; ++i)
#pragma unroll
          for (int j = 0; j < KW; ++j) acc[i][j] = fmaf(gv[i], xv[j], acc[i][j]);
      }
    }
#pragma unroll
    for (int i = 0; i < CW_OCT; ++i) {
      const int oc = og * CW_OCT + i;
      if (oc < OC) {
#pragma unroll
        for (int j = 0; j < KW; ++j) dst[((size_t)(oc * IC + ic) * KW + ky) * KW + j] = acc[i][j];
      }
    }
  }
  // bias gradient partial of this slab (sum of g over the band's positions), appended to the partial row
  for (int oc = tid; oc < OC; oc += nthr) {
    float bsum = 0.0f;
    for (int i = 0; i < rows * OW; ++i) bsum += gs[oc * (RB * OW) + i];
    dst[n_w + oc] = bsum;
  }
}

// out[j] = sum over the n_part per-CTA partials, in CTA order (quarters of the partials summed side by side, then combined
// in quarter order: deterministic).  64 outputs per CTA, every load of a thread in flight at once.
constexpr int CWR_J = 64;

__global__ void __launch_bounds__(4 * CWR_J)
k_conv_wgrad_reduce(const float* __restrict__ part, int n_part, int n_w, int n_b, float* __restrict__ out_w,
                    float* __restrict__ out_b) {
  __shared__ float s_q[4][CWR_J];
  const int jl = threadIdx.x % CWR_J, q = threadIdx.x / CWR_J, j = blockIdx.x * CWR_J + jl, n = n_w + n_b;
  const int per = (n_part + 3) / 4, p_lo = q * per, p_hi = min(n_part, p_lo + per);
  float acc = 0.0f;
  if (j < n) {
    for (int p0 = p_lo; p0 < p_hi; p0 += 32) {
      float v[32];
#pragma unroll
      for (int u = 0; u < 32; ++u) v[u] = (p0 + u < p_hi) ? __ldcg(part + (size_t)(p0 + u) * n + j) : 0.0f;
#pragma unroll
      for (int u = 0; u < 32; ++u) acc += v[u];
    }
  }
  s_q[q][jl] = acc;
  __syncthreads();
  if (q == 0 && j < n) {
    const float t = ((s_q[0][jl] + s_q[1][jl]) + s_q[2][jl]) + s_q[3][jl];
    if (j < n_w) out_w[j] = t;
    else if (out_b) out_b[j - n_w] = t;
  }
}

// ------------------------------------------------------------------------------------------------
// Conv body forward, one layer: y[b][oc][oy][ox] = relu(bias[oc] + sum_{ic,ky,kx} W[oc][ic][ky][kx] * x[b][ic][oy*S+ky][ox*S+kx])
// (model.py:55-63, no padding, square kernel) as an implicit GEMM on the warp-level tensor-core path with an error-
// compensated TF32 product (three MMAs per product as in k_head_bwd1; fp32-equivalent results, see tf32_split_rn below):
// D[oc][p] = W[oc][k] x X[k][p], k = (ic, ky, kx).
// grid = (bands of output rows, OC / 32, samples): a CTA owns 32 output channels of one band of one sample.  It stages the
// input rows its band touches (all channels) and its 32 weight rows in shared memory with every copy in flight at once,
// then warp work units (2 n8 pixel tiles x both m16 channel tiles, one slice of the k steps) run mma.sync.m16n8k8 with the
// A operand (W) split into hi / lo once per k step and reused over the unit's two pixel tiles, and the B operand gathered
// from the staged input through a per-k offset table.  The k slices of a pixel group land in separate shared buffers that
// the epilogue sums in slice order (deterministic, no atomics), then adds the bias, applies the ReLU and writes the band's
// rows coalesced.  These layers are latency bound at 32 / 64 rows, not arithmetic bound: the tiling exists to put a few
// hundred CTAs on the machine, each with a short serial chain.
// ------------------------------------------------------------------------------------------------
// Numerics: tf32_split's truncated hi leaves lo with up to 13 significant bits, which the MMA truncates to TF32 again
// (2^-21 relative per product), and one accumulator chained through ~100 MMAs adds the tensor core's inexact internal
// accumulation step after step: measured 3.8e-6 max error on conv 0 against 0.9e-6 for cuDNN's fp32 kernel.  Here hi is
// rounded to nearest (|lo| <= 2^-12 |v|, so lo's own TF32 truncation costs <= 2^-23) and each k step's three MMAs start from
// zero and are added to the fp32 accumulator with an IEEE add.
__device__ __forceinline__ void tf32_split_rn(float v, uint32_t& hi, uint32_t& lo) {
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(hi) : "f"(v));
  lo = __float_as_uint(__fsub_rn(v, __uint_as_float(hi)));
}

constexpr int CF_T = 256;           // threads per CTA
constexpr int CF_WARPS = CF_T / 32;
constexpr int CF_OC = 32;           // output channels per CTA (two m16 tiles)
constexpr int CF_MAX_BAND = 5;      // output rows per band at most

struct ConvFwdCfg {
  int OH, OW, RB, bands, in_rows, npx, groups, ksplit, kdim, kpad, nk, ldw, ldr, slab;
  size_t smem;
};

ConvFwdCfg conv_fwd_cfg(int IC, int IH, int IW, int K, int S) {
  ConvFwdCfg c;
  c.OH = (IH - K) / S + 1;
  c.OW = (IW - K) / S + 1;
  const int nb = (c.OH + CF_MAX_BAND - 1) / CF_MAX_BAND;
  c.RB = (c.OH + nb - 1) / nb;                          // balanced bands: 20 -> 4 x 5, 9 -> 5 + 4, 7 -> 4 + 3, 16 -> 4 x 4
  c.bands = (c.OH + c.RB - 1) / c.RB;
  c.in_rows = (c.RB - 1) * S + K;
  c.npx = c.RB * c.OW;                                  // pixels of a full band
  c.groups = ((c.npx + 7) / 8 + 1) / 2;                 // warp units along the pixels: two n8 tiles each
  c.kdim = IC * K * K;
  c.kpad = (c.kdim + 7) & ~7;
  c.nk = c.kpad / 8;
  c.ksplit = CF_WARPS / c.groups;
  if (c.ksplit < 1) c.ksplit = 1;
  if (c.ksplit > c.nk) c.ksplit = c.nk;
  c.ldw = ((c.kpad + 31) & ~31) + 4;                    // = 4 (mod 32): conflict-free A fragment loads
  c.ldr = c.groups * 16 + 4;                            // partial buffer row stride (pixels)
  c.slab = (IC * c.in_rows * IW + 3) & ~3;
  c.smem = ((size_t)c.slab + (size_t)CF_OC * c.ldw + (size_t)c.ksplit * CF_OC * c.ldr + (size_t)c.kpad) * sizeof(float);
  return c;
}

template <int K, int S>
__global__ void __launch_bounds__(CF_T)
k_conv_fwd(const float* __restrict__ x, const float* __restrict__ w, const float* __restrict__ bias, int IC, int IH, int IW,
           int OC, const ConvFwdCfg c, float* __restrict__ y) {
  extern __shared__ __align__(16) float cf_smem[];
  float* xs = cf_smem;                                            // [IC][in_rows][IW]   input rows of the band
  float* ws = xs + c.slab;                                        // [32][ldw]           weight rows of the CTA's channels
  float* red = ws + (size_t)CF_OC * c.ldw;                        // [ksplit][32][ldr]   partial tiles of the k slices
  int* koff = reinterpret_cast<int*>(red + (size_t)c.ksplit * CF_OC * c.ldr);   // [kpad]  slab offset of k = (ic, ky, kx)
  const int tid = threadIdx.x, band = blockIdx.x, oc0 = blockIdx.y * CF_OC, b = blockIdx.z;
  const int y0 = band * c.RB, rows = min(c.RB, c.OH - y0), npx = rows * c.OW;
  const int have_rows = min(c.in_rows, IH - y0 * S);
  const int xs_ld = c.in_rows * IW;

  // ---- staging: input slab and weight rows, all copies in flight at once ----
  const float* xsrc = x + ((size_t)b * IC * IH + (size_t)y0 * S) * IW;
  const int chunk = have_rows * IW;                               // contiguous floats per channel
  if ((IW & 3) == 0 && ((uintptr_t)x & 15) == 0) {
    const int q = chunk >> 2;
    for (int i = tid; i < IC * q; i += CF_T) {
      const int ic = i / q, j = i - ic * q;
      cp_async16(xs + ic * xs_ld + 4 * j, xsrc + (size_t)ic * IH * IW + 4 * j);
    }
  } else {
    for (int i = tid; i < IC * chunk; i += CF_T) {
      const int ic = i / chunk, j = i - ic * chunk;
      cp_async4(xs + ic * xs_ld + j, xsrc + (size_t)ic * IH * IW + j);
    }
  }
  const float* wsrc = w + (size_t)oc0 * c.kdim;
  if ((c.kdim & 3) == 0 && ((uintptr_t)w & 15) == 0) {
    const int q = c.kdim >> 2;
    for (int i = tid; i < CF_OC * q; i += CF_T) {
      const int r = i / q, j = i - r * q;
      cp_async16(ws + r * c.ldw + 4 * j, wsrc + (size_t)r * c.kdim + 4 * j);
    }
  } else {
    for (int i = tid; i < CF_OC * c.kdim; i += CF_T) {
      const int r = i / c.kdim, j = i - r * c.kdim;
      cp_async4(ws + r * c.ldw + j, wsrc + (size_t)r * c.kdim + j);
    }
  }
  // k padding (kdim % 8 != 0): zero weights, offset 0 (any finite staged value times zero)
  for (int i = tid; i < CF_OC * (c.kpad - c.kdim); i += CF_T) {
    const int r = i / (c.kpad - c.kdim), j = c.kdim + i % (c.kpad - c.kdim);
    ws[r * c.ldw + j] = 0.0f;
  }
  for (int k = tid; k < c.kpad; k += CF_T) {
    const int ic = k / (K * K), r = k - ic * (K * K), ky = r / K, kx = r - ky * K;
    koff[k] = (k < c.kdim) ? ic * xs_ld + ky * IW + kx : 0;
  }
  cp_async_wait_all();
  __syncthreads();

  // ---- products: warp unit u = (pixel group u % groups, k slice u / groups) ----
  const int warp = tid >> 5, lane = tid & 31, gid = lane >> 2, tig = lane & 3;
  const int units = c.groups * c.ksplit, per = (c.nk + c.ksplit - 1) / c.ksplit;
  for (int u = warp; u < units; u += CF_WARPS) {
    const int grp = u % c.groups, ks = u / c.groups;
    float acc[2][2][4];   // [m tile][n tile][C fragment]
#pragma unroll
    for (int i = 0; i < 2; ++i)
#pragma unroll
      for (int j = 0; j < 2; ++j)
#pragma unroll
        for (int q = 0; q < 4; ++q) acc[i][j][q] = 0.0f;
    int poff[2];
#pragma unroll
    for (int j = 0; j < 2; ++j) {   // B fragment column (pixel) of this lane in pixel tile j; pixels past the band read offset 0
      const int p = grp * 16 + 8 * j + gid;
      const int oy = p / c.OW, ox = p - oy * c.OW;
      poff[j] = (p < npx) ? oy * S * IW + ox * S : 0;
    }
    const int s_begin = ks * per, s_end = min(c.nk, s_begin + per);
    for (int s = s_begin; s < s_end; ++s) {
      const int k0 = 8 * s;
      uint32_t ahi[2][4], alo[2][4];
#pragma unroll
      for (int i = 0; i < 2; ++i) {
        const float* a = ws + (16 * i) * c.ldw + k0;
        tf32_split_rn(a[gid * c.ldw + tig], ahi[i][0], alo[i][0]);
        tf32_split_rn(a[(gid + 8) * c.ldw + tig], ahi[i][1], alo[i][1]);
        tf32_split_rn(a[gid * c.ldw + tig + 4], ahi[i][2], alo[i][2]);
        tf32_split_rn(a[(gid + 8) * c.ldw + tig + 4], ahi[i][3], alo[i][3]);
      }
      const int ko0 = koff[k0 + tig], ko1 = koff[k0 + tig + 4];
#pragma unroll
      for (int j = 0; j < 2; ++j) {
        uint32_t bhi[2], blo[2];
        tf32_split_rn(xs[ko0 + poff[j]], bhi[0], blo[0]);
        tf32_split_rn(xs[ko1 + poff[j]], bhi[1], blo[1]);
#pragma unroll
        for (int i = 0; i < 2; ++i) {   // D = Alo*Bhi + Ahi*Blo + Ahi*Bhi (the order of mma3_block), then acc += D
          float d[4] = {0.0f, 0.0f, 0.0f, 0.0f};
          mma_tf32(d, alo[i], bhi);
          mma_tf32(d, ahi[i], blo);
          mma_tf32(d, ahi[i], bhi);
#pragma unroll
          for (int q = 0; q < 4; ++q) acc[i][j][q] += d[q];
        }
      }
    }
    float* dst = red + (size_t)ks * CF_OC * c.ldr + grp * 16;
#pragma unroll
    for (int i = 0; i < 2; ++i)
#pragma unroll
      for (int j = 0; j < 2; ++j)
#pragma unroll
        for (int h = 0; h < 2; ++h)   // C fragment: channel rows gid, gid + 8; pixel columns 2 tig, 2 tig + 1
          *reinterpret_cast<float2*>(dst + (16 * i + gid + 8 * h) * c.ldr + 8 * j + 2 * tig) =
              make_float2(acc[i][j][2 * h], acc[i][j][2 * h + 1]);
  }
  __syncthreads();
  // ---- epilogue: k slices summed in order, bias, ReLU; one output channel's band is contiguous in y ----
  const size_t ohw = (size_t)c.OH * c.OW;
  float* yb = y + ((size_t)b * OC + oc0) * ohw + (size_t)y0 * c.OW;
  for (int i = tid; i < CF_OC * npx; i += CF_T) {
    const int oc = i / npx, p = i - oc * npx;
    float v = red[oc * c.ldr + p];
    for (int ks = 1; ks < c.ksplit; ++ks) v += red[((size_t)ks * CF_OC + oc) * c.ldr + p];
    yb[(size_t)oc * ohw + p] = fmaxf(v + __ldg(bias + oc0 + oc), 0.0f);
  }
}

int head_check(const rb_head_params* p, const char* who) {
  if (!p) return rbi::fail(RB_ERR_INVAL, who);
  for (int s = 0; s < 2; ++s)
    if (!p->w1_mu[s] || !p->w1_sigma[s] || !p->b1_mu[s] || !p->b1_sigma[s] || !p->w2_mu[s] || !p->w2_sigma[s] ||
        !p->b2_mu[s] || !p->b2_sigma[s])
      return rbi::fail(RB_ERR_INVAL, who);
  const bool noisy = p->eps_in1[0] != nullptr;
  for (int s = 0; s < 2; ++s)
    if ((p->eps_in1[s] != nullptr) != noisy || (p->eps_out1[s] != nullptr) != noisy || (p->eps_in2[s] != nullptr) != noisy ||
        (p->eps_out2[s] != nullptr) != noisy)
      return rbi::fail(RB_ERR_INVAL, "rb_head: give all eight noise factor vectors or none");
  if (p->conv_features <= 0 || p->hidden <= 0 || p->atoms <= 1 || p->actions <= 0) return rbi::fail(RB_ERR_INVAL, who);
  for (int s = 0; s < 2; ++s) {  // float4 accesses
    const uintptr_t bits = (uintptr_t)p->w1_mu[s] | (uintptr_t)p->w1_sigma[s] | (uintptr_t)p->b1_mu[s] | (uintptr_t)p->b1_sigma[s] |
                           (uintptr_t)p->w2_mu[s] | (uintptr_t)p->w2_sigma[s] | (uintptr_t)p->eps_in1[s] |
                           (uintptr_t)p->eps_out1[s] | (uintptr_t)p->eps_in2[s];
    if (bits & 15) return rbi::fail(RB_ERR_INVAL, "rb_head: weight / bias / factor pointers must be 16-byte aligned");
  }
  return RB_OK;
}

// Every shape limit of the head kernels, in one place: nullptr if a forward over `rows` rows (and, with `with_backward`,
// the backward over a batch of `rows`) launches, else why not.  rb_head_forward / rb_head_backward refuse exactly these
// shapes, and rb_head_supported lets a caller route them to the library path before it launches anything.
const char* head_limit(int K1, int H, int Z, int A, int rows, bool with_backward) {
  if (K1 % 32 || H % 64) return "rb_head: conv_features % 32 == 0 and hidden % 64 == 0 required";
  if (Z > RB_MAX_ATOMS) return "rb_head: atoms exceeds RB_MAX_ATOMS";
  // forward: one split-K ticket per (row tile, column tile) of each layer, 2048 tickets per layer
  const int MT = (rows > 32) ? 64 : 32;
  const int mt = (rows + MT - 1) / MT;
  const int tiles1 = 2 * H / NT, tiles2 = (Z + NT - 1) / NT + (A * Z + NT - 1) / NT;
  if (mt > 65535 || mt * tiles1 > 2048 || mt * tiles2 > 2048) return "rb_head_forward: too many rows for this head shape";
  if (!with_backward) return nullptr;
  if (rows > 32) return "rb_head_backward: 1 <= B <= 32 required (larger batches use the library GEMM path)";
  if (head_dh_smem(Z, A) > 200 * 1024) return "rb_head_backward: actions * atoms too large for the dh kernel";
  if (H > 1024) return "rb_head_backward: hidden <= 1024 required";
  return nullptr;
}

void head_splits(int K1, int H, int* s1, int* s2, int* ks1, int* ks2) {
  // aim for about two resident CTAs per SM (148 SMs) for layer 1 (N tiles = 2H/64), slices are multiples of the 32-wide k tile
  const int ntiles1 = 2 * H / NT;
  int want = (296 + ntiles1 - 1) / ntiles1;
  const int kt1 = (K1 + KT - 1) / KT;
  if (want > kt1) want = kt1;
  if (want > 16) want = 16;
  if (want < 1) want = 1;
  int per = (kt1 + want - 1) / want;
  *ks1 = per * KT;
  *s1 = (kt1 + per - 1) / per;
  const int kt2 = H / KT;
  int w2 = kt2 < 4 ? kt2 : 4;
  int per2 = (kt2 + w2 - 1) / w2;
  *ks2 = per2 * KT;
  *s2 = (kt2 + per2 - 1) / per2;
}

}  // namespace

extern "C" {

int rb_head_splits(int conv_features, int hidden, int* s1, int* s2) {
  if (!s1 || !s2 || conv_features <= 0 || hidden <= 0) return rbi::fail(RB_ERR_INVAL, "rb_head_splits: bad argument");
  int a, b;
  head_splits(conv_features, hidden, s1, s2, &a, &b);
  int s_tc, per;
  rbi::head_fc1_tc_splits(conv_features, hidden, &s_tc, &per);   // part1 must hold whichever layer-1 kernel runs
  if (s_tc > *s1) *s1 = s_tc;
  return RB_OK;
}

int rb_head_ticket_count(void) { return 4096; }

int rb_head_supported(int conv_features, int hidden, int atoms, int actions, int rows, int with_backward) {
  if (conv_features <= 0 || hidden <= 0 || atoms <= 1 || actions <= 0 || rows <= 0)
    return rbi::fail(RB_ERR_INVAL, "rb_head_supported: bad argument");
  return head_limit(conv_features, hidden, atoms, actions, rows, with_backward != 0) ? RB_ERR_RANGE : RB_OK;
}

static int g_head_debug = 0;   // bit 0: skip the layer-1 launch, bit 1: skip the layer-2 launch (timing probes only); bit 2: FFMA layer 1; bit 3: split-K layer 2
int rb_head_debug(int flags) {
  g_head_debug = flags;
  return RB_OK;
}

int rb_head_forward(const rb_head_params* p, const float* x_lo, int m_lo, const float* x_hi, int m_hi, float* part1, float* part2,
                    int32_t* tickets, float* h, float* z, rb_stream_t stream) {
  int rc = head_check(p, "rb_head_forward: null pointer or bad size");
  if (rc != RB_OK) return rc;
  const int M = m_lo + m_hi;
  if (!x_lo || m_lo <= 0 || m_hi < 0 || (m_hi > 0 && !x_hi) || !part1 || !part2 || !tickets || !h || !z)
    return rbi::fail(RB_ERR_INVAL, "rb_head_forward: bad argument");
  const HeadDesc d = to_desc(p);
  if (const char* why = head_limit(d.K1, d.H, d.Z, d.A, M, false)) return rbi::fail(RB_ERR_RANGE, why);
  int s1, s2, ks1, ks2;
  head_splits(d.K1, d.H, &s1, &s2, &ks1, &ks2);
  cudaStream_t st = (cudaStream_t)stream;
  const int MT = (M > 32) ? 64 : 32;
  const int mt = (M + MT - 1) / MT;
  const int tiles1 = 2 * d.H / NT, tiles2 = (d.Z + NT - 1) / NT + (d.A * d.Z + NT - 1) / NT;
  const size_t smem64 = (size_t)FC_STAGES * (64 + 2 * NT) * (KT + 4) * sizeof(float);
  const size_t smem32 = (size_t)FC_STAGES * (32 + 2 * NT) * (KT + 4) * sizeof(float);
  rc = rbi::ensure_dynamic_smem(k_head_fc<64, 1>, smem64, "rb_head_forward");
  if (rc == RB_OK) rc = rbi::ensure_dynamic_smem(k_head_fc<64, 2>, smem64, "rb_head_forward");
  if (rc == RB_OK) rc = rbi::ensure_dynamic_smem(k_head_fc<32, 1>, smem32, "rb_head_forward");
  if (rc == RB_OK) rc = rbi::ensure_dynamic_smem(k_head_fc<32, 2>, smem32, "rb_head_forward");
  if (rc != RB_OK) return rc;
  if (!(g_head_debug & 1)) {
    if (!(g_head_debug & 4) && rbi::head_fc1_tc_ok(d.K1, d.H, m_lo, m_hi)) {   // tensor cores: TMA + tcgen05.mma (3xTF32), then the fixed-order reduction
      rc = rbi::head_fc1_tc(d.w1_mu, d.w1_sig, d.b1_mu, d.b1_sig, d.ei1, d.eo1, d.K1, d.H, x_lo, m_lo, x_hi, m_hi, part1, h, st);
      if (rc != RB_OK) return rc;
    } else {
      dim3 grid(tiles1, s1, mt);
      rbi::ProfScope prof_(RB_K_HEAD_FC1, st);
      if (MT == 64) k_head_fc<64, 1><<<grid, FC_T, smem64, st>>>(d, x_lo, m_lo, x_hi, M, part1, h, tickets, ks1);
      else k_head_fc<32, 1><<<grid, FC_T, smem32, st>>>(d, x_lo, m_lo, x_hi, M, part1, h, tickets, ks1);
    }
  }
  rc = rbi::check_launch("rb_head_forward(fc1)");
  if (rc != RB_OK) return rc;
  if (!(g_head_debug & 2)) {
    const size_t smem_f2 = (size_t)(F2_MT + F2_ROWS) * (d.H + 4) * sizeof(float);
    rbi::ProfScope prof_(RB_K_HEAD_FC2, st);
    if (smem_f2 <= 200 * 1024 && d.H % 4 == 0 && !(g_head_debug & 8)) {   // single pass, no split-K (the usual shapes)
      rc = rbi::ensure_dynamic_smem(k_head_fc2, smem_f2, "rb_head_forward(fc2)");
      if (rc != RB_OK) return rc;
      dim3 grid((d.Z + F2_ROWS - 1) / F2_ROWS + (d.A * d.Z + F2_ROWS - 1) / F2_ROWS, (M + F2_MT - 1) / F2_MT);
      k_head_fc2<<<grid, F2_T, smem_f2, st>>>(d, h, M, z);
    } else {
      dim3 grid(tiles2, s2, mt);
      if (MT == 64) k_head_fc<64, 2><<<grid, FC_T, smem64, st>>>(d, h, M, nullptr, M, part2, z, tickets + 2048, ks2);
      else k_head_fc<32, 2><<<grid, FC_T, smem32, st>>>(d, h, M, nullptr, M, part2, z, tickets + 2048, ks2);
    }
  }
  return rbi::check_launch("rb_head_forward(fc2)");
}

int rb_head_logits(const float* z, int M, int actions, int atoms, float* q, rb_stream_t stream) {
  if (!z || !q || M <= 0 || actions <= 0 || atoms <= 0) return rbi::fail(RB_ERR_INVAL, "rb_head_logits: bad argument");
  {
    rbi::ProfScope prof_(RB_K_HEAD_LOGITS, (cudaStream_t)stream);
    k_head_logits<<<M, 128, 0, (cudaStream_t)stream>>>(atoms, actions, z, q);
  }
  return rbi::check_launch("rb_head_logits");
}

int rb_head_backward(const rb_head_params* p, const rb_head_grads* gr, const float* x, const float* h, const float* dz, int B,
                     float* dh_scratch, float* dx, int relu_mask_x, int parts, rb_stream_t stream) {
  int rc = head_check(p, "rb_head_backward: null pointer or bad size");
  if ((parts & 7) == 0) return rbi::fail(RB_ERR_INVAL, "rb_head_backward: parts must select at least one of RB_HEAD_BWD_*");
  if (rc != RB_OK) return rc;
  if (!gr || !x || !h || !dz || !dh_scratch || !dx) return rbi::fail(RB_ERR_INVAL, "rb_head_backward: null pointer");
  if (B <= 0) return rbi::fail(RB_ERR_RANGE, "rb_head_backward: 1 <= B <= 32 required");
  // the whole backward's limits, whichever parts this call enqueues: a shape never gets its layer-2 gradient on one stream
  // and a refusal of the dh / layer-1 launches on the other
  if (const char* why = head_limit(p->conv_features, p->hidden, p->atoms, p->actions, B, true)) return rbi::fail(RB_ERR_RANGE, why);
  HeadGrads g;
  for (int s = 0; s < 2; ++s) {
    if (!gr->w1_mu[s] || !gr->w1_sigma[s] || !gr->b1_mu[s] || !gr->b1_sigma[s] || !gr->w2_mu[s] || !gr->w2_sigma[s] ||
        !gr->b2_mu[s] || !gr->b2_sigma[s])
      return rbi::fail(RB_ERR_INVAL, "rb_head_backward: null gradient pointer");
    g.w1_mu[s] = gr->w1_mu[s]; g.w1_sig[s] = gr->w1_sigma[s]; g.b1_mu[s] = gr->b1_mu[s]; g.b1_sig[s] = gr->b1_sigma[s];
    g.w2_mu[s] = gr->w2_mu[s]; g.w2_sig[s] = gr->w2_sigma[s]; g.b2_mu[s] = gr->b2_mu[s]; g.b2_sig[s] = gr->b2_sigma[s];
  }
  const HeadDesc d = to_desc(p);
  cudaStream_t st = (cudaStream_t)stream;
  if (parts & RB_HEAD_BWD_WGRAD2) {
    const int tiles = (d.Z + NT - 1) / NT + (d.A * d.Z + NT - 1) / NT;
    dim3 grid(tiles, d.H / NT);
    rbi::ProfScope prof_(RB_K_HEAD_WGRAD2, st);
    k_head_wgrad2<<<grid, HT, 0, st>>>(d, g, dz, h, B);
  }
  rc = rbi::check_launch("rb_head_backward(wgrad2)");
  if (rc != RB_OK) return rc;
  if (parts & RB_HEAD_BWD_DH) {
    const int ld_dz = head_dh_ld(d.Z, d.A);
    const size_t smem = head_dh_smem(d.Z, d.A);
    rc = rbi::ensure_dynamic_smem(k_head_dh, smem, "rb_head_backward");
    if (rc != RB_OK) return rc;
    dim3 grid(d.H / DH_KB, 2);
    rbi::ProfScope prof_(RB_K_HEAD_DH, st);
    k_head_dh<<<grid, DH_T, smem, st>>>(d, dz, h, B, dh_scratch, dh_scratch + (size_t)B * 2 * d.H, ld_dz);
  }
  rc = rbi::check_launch("rb_head_backward(dh)");
  if (rc != RB_OK) return rc;
  if (parts & RB_HEAD_BWD_LAYER1) {
    dim3 grid(d.K1 / B1_K, 4);
    rbi::ProfScope prof_(RB_K_HEAD_BWD1, st);
    const size_t smem_b1 = (size_t)B1_STAGES * B1_STAGE * sizeof(float);
    rc = rbi::ensure_dynamic_smem(k_head_bwd1, smem_b1, "rb_head_backward");
    if (rc != RB_OK) return rc;
    k_head_bwd1<<<grid, B1_T, smem_b1, st>>>(d, g, x, dh_scratch, dh_scratch + (size_t)B * 2 * d.H, B, dx, relu_mask_x);
  }
  return rbi::check_launch("rb_head_backward(bwd1)");
}

int rb_bias_grad(const float* grad_out, int B, int C, int HW, float* out, rb_stream_t stream) {
  if (!grad_out || !out || B <= 0 || C <= 0 || HW <= 0) return rbi::fail(RB_ERR_INVAL, "rb_bias_grad: bad argument");
  {
    rbi::ProfScope prof_(RB_K_BIAS_GRAD, (cudaStream_t)stream);
    k_bias_grad<<<C, 256, 0, (cudaStream_t)stream>>>(grad_out, B, C, HW, out);
  }
  return rbi::check_launch("rb_bias_grad");
}

static int conv_wgrad_band_rows(int OH) { return OH >= 16 ? (OH + 7) / 8 : OH; }   // ~8 bands of output rows per sample

int rb_conv_wgrad_scratch_elems(int B, int IC, int IH, int OC, int K, int stride) {
  if (B <= 0 || IC <= 0 || OC <= 0 || K <= 0 || stride <= 0 || IH < K) return 0;
  const int OH = (IH - K) / stride + 1, RB = conv_wgrad_band_rows(OH), bands = (OH + RB - 1) / RB;
  return B * bands * (OC * IC * K * K + OC);
}

int rb_conv_wgrad(const float* grad_out, const float* input, int B, int IC, int IH, int IW, int OC, int K, int stride,
                  float* partials, float* out, float* bias_out, rb_stream_t stream) {
  if (!grad_out || !input || !partials || !out) return rbi::fail(RB_ERR_INVAL, "rb_conv_wgrad: null pointer");
  if (B <= 0 || IC <= 0 || OC <= 0 || stride <= 0 || IH < K || IW < K) return rbi::fail(RB_ERR_INVAL, "rb_conv_wgrad: bad shape");
  if (K != 8 && K != 5 && K != 4 && K != 3) return rbi::fail(RB_ERR_RANGE, "rb_conv_wgrad: kernel sizes 3, 4, 5 and 8 are instantiated");
  const int OH = (IH - K) / stride + 1, OW = (IW - K) / stride + 1;
  const int RB = conv_wgrad_band_rows(OH), bands = (OH + RB - 1) / RB;
  const int threads = IC * K * ((OC + CW_OCT - 1) / CW_OCT);
  if (threads > 256 || B > 65535) return rbi::fail(RB_ERR_RANGE, "rb_conv_wgrad: IC * K * ceil(OC / 4) must not exceed 256 threads");
  const size_t smem = ((size_t)IC * ((RB - 1) * stride + K) * IW + (size_t)OC * RB * OW) * sizeof(float);
  if (smem > 200 * 1024) return rbi::fail(RB_ERR_RANGE, "rb_conv_wgrad: slab does not fit in shared memory");
  cudaStream_t st = (cudaStream_t)stream;
  dim3 grid(bands, B);
  int rc = RB_OK;
  {
    rbi::ProfScope prof_(RB_K_CONV_WGRAD, st);
#define RB_CW_LAUNCH(KW_)                                                                                              \
  rc = rbi::ensure_dynamic_smem(k_conv_wgrad_first<KW_>, smem, "rb_conv_wgrad");                                       \
  if (rc == RB_OK) k_conv_wgrad_first<KW_><<<grid, threads, smem, st>>>(grad_out, input, IC, IH, IW, OC, OH, OW, stride, RB, partials);
    if (K == 8) { RB_CW_LAUNCH(8) } else if (K == 5) { RB_CW_LAUNCH(5) } else if (K == 4) { RB_CW_LAUNCH(4) } else { RB_CW_LAUNCH(3) }
#undef RB_CW_LAUNCH
    if (rc != RB_OK) return rc;
    const int n_w = OC * IC * K * K;
    k_conv_wgrad_reduce<<<(n_w + OC + CWR_J - 1) / CWR_J, 4 * CWR_J, 0, st>>>(partials, B * bands, n_w, OC, out, bias_out);
  }
  return rbi::check_launch("rb_conv_wgrad");
}

int rb_conv_forward(const float* input, const float* weight, const float* bias, int B, int IC, int IH, int IW, int OC, int K,
                    int stride, float* out, rb_stream_t stream) {
  if (!input || !weight || !bias || !out) return rbi::fail(RB_ERR_INVAL, "rb_conv_forward: null pointer");
  if (B <= 0 || IC <= 0 || OC <= 0 || K <= 0 || stride <= 0 || IH < K || IW < K) return rbi::fail(RB_ERR_INVAL, "rb_conv_forward: bad shape");
  const bool inst = (K == 8 && stride == 4) || (K == 4 && stride == 2) || (K == 3 && stride == 1) || (K == 5 && stride == 5);
  if (!inst) return rbi::fail(RB_ERR_RANGE, "rb_conv_forward: (kernel, stride) in {(8,4), (4,2), (3,1), (5,5)} are instantiated");
  if (OC % CF_OC) return rbi::fail(RB_ERR_RANGE, "rb_conv_forward: out_channels % 32 == 0 required");
  const ConvFwdCfg c = conv_fwd_cfg(IC, IH, IW, K, stride);
  if (c.smem > 200 * 1024) return rbi::fail(RB_ERR_RANGE, "rb_conv_forward: input band and weight rows do not fit in shared memory");
  if (B > 65535) return rbi::fail(RB_ERR_RANGE, "rb_conv_forward: at most 65535 rows");
  cudaStream_t st = (cudaStream_t)stream;
  dim3 grid(c.bands, OC / CF_OC, B);
  int rc = RB_OK;
  {
    rbi::ProfScope prof_(RB_K_CONV_FWD, st);
#define RB_CF_LAUNCH(K_, S_)                                                                                           \
  rc = rbi::ensure_dynamic_smem(k_conv_fwd<K_, S_>, c.smem, "rb_conv_forward");                                       \
  if (rc == RB_OK) k_conv_fwd<K_, S_><<<grid, CF_T, c.smem, st>>>(input, weight, bias, IC, IH, IW, OC, c, out);
    if (K == 8) { RB_CF_LAUNCH(8, 4) } else if (K == 4) { RB_CF_LAUNCH(4, 2) } else if (K == 3) { RB_CF_LAUNCH(3, 1) } else { RB_CF_LAUNCH(5, 5) }
#undef RB_CF_LAUNCH
  }
  if (rc != RB_OK) return rc;
  return rbi::check_launch("rb_conv_forward");
}

int rb_noise_factors(float* f_in, int n_in, float* f_out, int n_out, const float* x_in, const float* x_out, uint64_t seed,
                     uint64_t* rng_counter, rb_stream_t stream) {
  if (!f_in || !f_out || n_in <= 0 || n_out <= 0) return rbi::fail(RB_ERR_INVAL, "rb_noise_factors: bad argument");
  if ((x_in == nullptr) != (x_out == nullptr)) return rbi::fail(RB_ERR_INVAL, "rb_noise_factors: give both x_in and x_out or neither");
  if (!x_in && !rng_counter) return rbi::fail(RB_ERR_INVAL, "rb_noise_factors: need injected normals or rng_counter");
  {
    rbi::ProfScope prof_(RB_K_NOISE_FACTORS, (cudaStream_t)stream);
    k_noise_factors<<<1, 1024, 0, (cudaStream_t)stream>>>(f_in, n_in, f_out, n_out, x_in, x_out, seed, (unsigned long long*)rng_counter);
  }
  return rbi::check_launch("rb_noise_factors");
}

}  // extern "C"
