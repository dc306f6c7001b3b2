// HBM-bound kernels of the step: mini-batch load/cast/transpose (K1), output layer + loss + its
// backward (K3/K4), fused multi-tensor optimizer (K7), gradient accumulation.
#pragma once
#include "common.cuh"
#include "ptx.cuh"

namespace sb {

// Where the current mini-batch lives (HBM-resident training set or the H2D staging area).
// Written by set_batch_kernel right before the captured step graph runs, so the graph itself
// never changes (res/ssgd_monitor.py:272-276 builds the same feed_dict from x_batch[i]).
struct BatchDesc {
  const float* X;  // [rows, F] row-major fp32
  const float* y;  // [rows]
  const float* w;  // [rows]
  float lr_t;      // Adam: lr * sqrt(1-b2^t)/(1-b1^t); others: lr
  float gscale;    // 1/world (and 1/n_accumulated for the epoch-sync schedule)
  unsigned int epoch;  // exchange round (flag value of the peer-memory all-reduce)
  int row0;            // first row of the batch inside the bf16 HBM-resident set (TMA row-coordinate offset)
  float2* hist;        // nullable: slot of this step in the pinned-host loss history (loss sum, n_nz), written by the step's tail
  const int* idx;      // sparse (wide+deep) steps: the batch's index rows [rows, n_cat] - staged, or inside the resident set
};

// nz_prefix != nullptr (bf16 resident set): the batch is consumed by TMA straight from the resident set, there is no
// load kernel, so this kernel also publishes n_nz = #{w != 0 in the batch} from the prefix counts built at load time
// and clears the loss accumulator.
static __global__ void set_batch_kernel(BatchDesc* d, const float* X, const float* y, const float* w, float lr_t, float gscale,
                                        unsigned int epoch = 0, int row0 = 0, const int* nz_prefix = nullptr, int rows = 0,
                                        float* scal = nullptr, float2* hist = nullptr, const int* idx = nullptr) {
  d->X = X; d->y = y; d->w = w; d->lr_t = lr_t; d->gscale = gscale; d->epoch = epoch; d->row0 = row0; d->hist = hist; d->idx = idx;
  if (nz_prefix != nullptr) {
    scal[1] = static_cast<float>(nz_prefix[row0 + rows] - nz_prefix[row0]);  // SCAL_NNZ
    scal[0] = 0.f;                                                           // SCAL_LOSS_SUM
  }
}

// Split-precision modes: the value whose bf16 rounding is part `part` of x (part 0: x itself; part k: x minus the first k
// parts).  x = bf16(r_0) + bf16(r_1) + ... with r_0 = x, r_{k+1} = r_k - bf16(r_k).
__device__ __forceinline__ float bf16_residual(float x, int part) {
  for (int i = 0; i < part; ++i) x -= __bfloat162float(__float2bfloat16_rn(x));
  return x;
}

// step scalars (device): [0] = sum_i w_i * per-row loss, [1] = n_nz (count of non-zero weights)
enum { SCAL_LOSS_SUM = 0, SCAL_NNZ = 1, SCAL_COUNT = 4 };

// ------------------------------------------------------------------------------------------------
// K1 mini-batch load.  fp32 rows of the current batch -> the operand buffer of the layer-0 GEMMs:
// (bf16 mode) row-major bf16 [rows, ldF] - the SAME buffer feeds the forward GEMM (K-major) and the dW
// GEMM (MN-major), so no transposed copy exists; (fp32 mode) fp32 copy into the batch buffer.
// HBM-bound: each thread moves 8 consecutive columns (2 x 16 B loads -> one 16 B store).
// Block 0 additionally counts the non-zero sample weights of the batch (n_nz of
// SUM_BY_NONZERO_WEIGHTS, res/ssgd_monitor.py:129).
// ------------------------------------------------------------------------------------------------
template <bool BF16>
__global__ void __launch_bounds__(256)
load_batch_kernel(const BatchDesc* __restrict__ desc, int rows, int F, __nv_bfloat16* __restrict__ Xb, int ldF,
                  float* __restrict__ Xf, float* __restrict__ scal, float* __restrict__ zero_buf, long long zero_n,
                  int np = 1, long long part_stride = 0) {
  pdl_wait();
  pdl_launch_dependents();
  // the step's gradient buffer is accumulated with atomics: clear it here (replaces a memset node in the graph)
  for (long long i = blockIdx.x * 256ll + threadIdx.x; i < zero_n; i += gridDim.x * 256ll) zero_buf[i] = 0.f;
  const float* __restrict__ X = desc->X;
  const int groups = ldF >> 3;  // 8-column groups per row (ldF is a multiple of 8)
  const long long total = static_cast<long long>(rows) * groups;
  const bool vec = ((F & 7) == 0) && ((reinterpret_cast<uintptr_t>(X) & 15) == 0);
  for (long long u = blockIdx.x * 256ll + threadIdx.x; u < total; u += gridDim.x * 256ll) {
    const int r = static_cast<int>(u / groups), c = static_cast<int>(u % groups) * 8;
    float v[8];
    if (vec) {
      const float4 a = __ldg(reinterpret_cast<const float4*>(X + static_cast<size_t>(r) * F + c));
      const float4 b = __ldg(reinterpret_cast<const float4*>(X + static_cast<size_t>(r) * F + c + 4));
      v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
    } else {
#pragma unroll
      for (int j = 0; j < 8; ++j) v[j] = (c + j < F) ? __ldg(X + static_cast<size_t>(r) * F + c + j) : 0.f;
    }
    if constexpr (BF16) {
      for (int part = 0; part < np; ++part) {      // np > 1: split-precision parts (bf16_residual)
        uint4 o;
        o.x = pack_bf16x2(bf16_residual(v[0], part), bf16_residual(v[1], part));
        o.y = pack_bf16x2(bf16_residual(v[2], part), bf16_residual(v[3], part));
        o.z = pack_bf16x2(bf16_residual(v[4], part), bf16_residual(v[5], part));
        o.w = pack_bf16x2(bf16_residual(v[6], part), bf16_residual(v[7], part));
        *reinterpret_cast<uint4*>(Xb + part * part_stride + static_cast<size_t>(r) * ldF + c) = o;
      }
    } else {
      if (vec) {
        *reinterpret_cast<float4*>(Xf + static_cast<size_t>(r) * F + c) = make_float4(v[0], v[1], v[2], v[3]);
        *reinterpret_cast<float4*>(Xf + static_cast<size_t>(r) * F + c + 4) = make_float4(v[4], v[5], v[6], v[7]);
      } else {
#pragma unroll
        for (int j = 0; j < 8; ++j)
          if (c + j < F) Xf[static_cast<size_t>(r) * F + c + j] = v[j];
      }
    }
  }
  if (blockIdx.x == 0) {
    const float* __restrict__ w = desc->w;
    float cnt = 0.f;
    for (int i = threadIdx.x; i < rows; i += 256) cnt += (__ldg(w + i) != 0.f) ? 1.f : 0.f;
    cnt = warp_sum(cnt);
    __shared__ float part[8];
    if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = cnt;
    __syncthreads();
    if (threadIdx.x == 0) {
      float t = 0.f;
      for (int i = 0; i < 8; ++i) t += part[i];
      scal[SCAL_NNZ] = t;
      scal[SCAL_LOSS_SUM] = 0.f;
    }
  }
}

// ------------------------------------------------------------------------------------------------
// K3+K4 (+ output-layer backward): y_hat = sigmoid(A_L w_o + b_o); loss = sum w (y_hat-y)^2 / n_nz
// (res/ssgd_monitor.py:121,129) or the sigmoid-CE variant; d z_hat; then the rank-1 backward
//   dZ_L[r,j] = dz_r * w_o[j] * act'(A_L[r,j])     (row-major, bf16 or fp32)
//   dw_o[j] += sum_r dz_r A_L[r,j],  db_o += sum_r dz_r,  db_L[j] += sum_r dZ_L[r,j]
// out = 1 is GEMV-class: CUDA cores, one pass over A_L.  Each block owns 32 rows.
// ------------------------------------------------------------------------------------------------
struct OutLayerParams {
  int rows, H, ldA;          // A_L is [rows, ldA] with H valid columns
  const void* A;             // bf16 or fp32
  const float* wo;           // [H]
  const float* bo;           // [1]
  const BatchDesc* desc;     // y, w
  float* scal;               // SCAL_*
  int loss, act;             // sb_loss, activation of hidden layer L
  int do_bwd;                // 0: forward (+loss) only
  int do_loss;               // 0: scores only (no y / w access)
  float* yhat;               // nullable [rows]
  void* dZ; int ld_dZ;       // [rows, ld_dZ] bf16 or fp32
  float* g_wo; float* g_bo; float* g_bL;  // gradient slots (atomic accumulate)
  unsigned long long* trace;              // debug timeline (nullable): [0] entry, [2] deps resolved (block 0), [10] last exit
  int np;                                 // bf16 parts per value of A / dZ (split-precision modes; 0 or 1 = plain)
  long long a_ps, dz_ps;                  // element stride between parts
};

// in-graph kernel span for the step timeline: begin = block 0's stamp after griddepcontrol.wait, end = atomicMax over blocks
__device__ __forceinline__ void trace_begin(unsigned long long* trace, bool entry) {
  if (trace != nullptr && blockIdx.x == 0 && threadIdx.x == 0) trace[entry ? 0 : 2] = globaltimer_ns();
}
__device__ __forceinline__ void trace_end(unsigned long long* trace) {
  if (trace != nullptr && threadIdx.x == 0) atomicMax(trace + 10, static_cast<unsigned long long>(globaltimer_ns()));
}

template <typename T> __device__ __forceinline__ float ld_as_float(const T* p);
template <> __device__ __forceinline__ float ld_as_float<float>(const float* p) { return __ldg(p); }
template <> __device__ __forceinline__ float ld_as_float<__nv_bfloat16>(const __nv_bfloat16* p) { return __bfloat162float(*p); }
template <typename T> __device__ __forceinline__ void st_from_float(T* p, float v);
template <> __device__ __forceinline__ void st_from_float<float>(float* p, float v) { *p = v; }
template <> __device__ __forceinline__ void st_from_float<__nv_bfloat16>(__nv_bfloat16* p, float v) { *p = __float2bfloat16_rn(v); }

template <typename T>
__global__ void __launch_bounds__(256)
out_layer_kernel(const OutLayerParams p) {
  trace_begin(p.trace, true);
  pdl_wait();
  pdl_launch_dependents();
  trace_begin(p.trace, false);
  __shared__ float dz_row[32];
  __shared__ float blk_red[8];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int r0 = blockIdx.x * 32;
  const T* __restrict__ A = reinterpret_cast<const T*>(p.A);
  const float bo = __ldg(p.bo);
  const float nnz = p.do_loss ? p.scal[SCAL_NNZ] : 1.f;
  const float inv_nnz = nnz > 0.f ? 1.f / nnz : 0.f;

  // ---- phase 1: one warp per row (4 rows per warp) ----
  float loss_part = 0.f;
  for (int i = 0; i < 4; ++i) {
    const int rl = warp * 4 + i, r = r0 + rl;
    float z = 0.f;
    if (r < p.rows) {
      const T* ar = A + static_cast<size_t>(r) * p.ldA;
      for (int j = lane; j < p.H; j += 32) {
        float a = ld_as_float<T>(ar + j);
        for (int part = 1; part < p.np; ++part) a += ld_as_float<T>(ar + part * p.a_ps + j);
        z = fmaf(a, __ldg(p.wo + j), z);
      }
    }
    z = warp_sum(z) + bo;
    if (lane == 0) {
      float dz = 0.f;
      if (r < p.rows) {
        const float yh = sigmoidf_stable(z);
        if (p.yhat) p.yhat[r] = yh;
        if (p.do_loss) {
          const float y = __ldg(p.desc->y + r), w = __ldg(p.desc->w + r);
          if (p.loss == SB_LOSS_MSE) {
            const float d = yh - y;
            loss_part += w * d * d;
            dz = 2.f * w * d * yh * (1.f - yh) * inv_nnz;
          } else {
            loss_part += w * (fmaxf(z, 0.f) - z * y + log1pf(expf(-fabsf(z))));
            dz = w * (yh - y) * inv_nnz;
          }
        }
      }
      dz_row[rl] = dz;
    }
  }
  if (p.do_loss) {
    if (lane == 0) blk_red[warp] = loss_part;
    __syncthreads();
    if (tid == 0) {
      float s = 0.f;
      for (int i = 0; i < 8; ++i) s += blk_red[i];
      atomicAdd(p.scal + SCAL_LOSS_SUM, s);
    }
  }
  if (!p.do_bwd) { trace_end(p.trace); return; }
  __syncthreads();

  // ---- phase 2: rank-1 backward over column chunks of 128 ----
  float dbo = 0.f;
  if (tid < 32) {
    dbo = warp_sum(dz_row[tid]);
    if (tid == 0) atomicAdd(p.g_bo, dbo);
  }
  T* __restrict__ dZ = reinterpret_cast<T*>(p.dZ);
  for (int c0 = 0; c0 < p.H; c0 += 128) {
    const int cl = tid & 127, j = c0 + cl;  // column handled by this thread
    const int rh = tid >> 7;                // row half: rows rh*16 .. rh*16+15
    float s_dw = 0.f, s_db = 0.f;
    const float woj = (j < p.H) ? __ldg(p.wo + j) : 0.f;
    for (int i = 0; i < 16; ++i) {
      const int rl = rh * 16 + i, r = r0 + rl;
      float g = 0.f;
      if (r < p.rows && j < p.H) {
        float a = ld_as_float<T>(A + static_cast<size_t>(r) * p.ldA + j);
        for (int part = 1; part < p.np; ++part) a += ld_as_float<T>(A + part * p.a_ps + static_cast<size_t>(r) * p.ldA + j);
        const float dz = dz_row[rl];
        g = dz * woj * act_grad_from_out(a, p.act);
        s_dw = fmaf(dz, a, s_dw);
        s_db += g;
        st_from_float<T>(dZ + static_cast<size_t>(r) * p.ld_dZ + j, g);
        for (int part = 1; part < p.np; ++part)
          st_from_float<T>(dZ + part * p.dz_ps + static_cast<size_t>(r) * p.ld_dZ + j, bf16_residual(g, part));
      }
    }
    if (j < p.H) {
      atomicAdd(p.g_wo + j, s_dw);
      atomicAdd(p.g_bL + j, s_db);
    }
  }
  trace_end(p.trace);
}

// bf16 variant of the kernel above for H <= 256 * NCH: ONE pass over A_L.  A warp owns whole rows (rows w, w+8, ... of
// the block's slice); lane i owns columns [256 c + 8 i, +8) of every 256-column chunk c of every row, moved with 16-byte
// loads / stores.  Because the lane <-> column mapping is the same for every row, the row's dot product is one xor-shuffle
// reduction and the dw_o / db_L column sums stay in registers over all rows of the warp; a block reduces them through
// shared memory and issues ONE atomic per column (the 32-rows-per-block kernel above read A_L twice with 2-byte
// accesses and took 20 us at cfg2 sizes, scripts/step_timeline.py).
template <int NCH>
__global__ void __launch_bounds__(256)
out_layer_rows_kernel(const OutLayerParams p, int rows_per_block) {
  trace_begin(p.trace, true);
  pdl_wait();
  pdl_launch_dependents();
  trace_begin(p.trace, false);
  __shared__ float red[2][8][256];
  __shared__ float red_s[2][8];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const __nv_bfloat16* __restrict__ A = reinterpret_cast<const __nv_bfloat16*>(p.A);
  __nv_bfloat16* __restrict__ dZ = reinterpret_cast<__nv_bfloat16*>(p.dZ);
  const float bo = __ldg(p.bo);
  const float nnz = p.do_loss ? p.scal[SCAL_NNZ] : 1.f;
  const float inv_nnz = nnz > 0.f ? 1.f / nnz : 0.f;
  float wo[NCH][8], s_dw[NCH][8], s_db[NCH][8];
#pragma unroll
  for (int c = 0; c < NCH; ++c)
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      const int j = c * 256 + lane * 8 + k;
      wo[c][k] = (j < p.H) ? __ldg(p.wo + j) : 0.f;
      s_dw[c][k] = 0.f; s_db[c][k] = 0.f;
    }
  float loss_part = 0.f, dz_sum = 0.f;
  const int r_begin = blockIdx.x * rows_per_block;
  const int r_end = min(p.rows, r_begin + rows_per_block);
  for (int r = r_begin + warp; r < r_end; r += 8) {
    float a[NCH][8];
    float z = 0.f;
#pragma unroll
    for (int c = 0; c < NCH; ++c) {
      const int col0 = c * 256 + lane * 8;
      uint4 raw = make_uint4(0, 0, 0, 0);
      if (col0 < p.ldA && col0 < p.H) raw = *reinterpret_cast<const uint4*>(A + static_cast<size_t>(r) * p.ldA + col0);
      const __nv_bfloat16* h = reinterpret_cast<const __nv_bfloat16*>(&raw);
#pragma unroll
      for (int k = 0; k < 8; ++k) a[c][k] = (col0 + k < p.H) ? __bfloat162float(h[k]) : 0.f;   // pad columns of A_L hold act(0), not 0
      for (int part = 1; part < p.np; ++part) {       // split-precision modes: add the lower parts
        uint4 lo = make_uint4(0, 0, 0, 0);
        if (col0 < p.ldA && col0 < p.H) lo = *reinterpret_cast<const uint4*>(A + part * p.a_ps + static_cast<size_t>(r) * p.ldA + col0);
        const __nv_bfloat16* hl = reinterpret_cast<const __nv_bfloat16*>(&lo);
#pragma unroll
        for (int k = 0; k < 8; ++k) a[c][k] += (col0 + k < p.H) ? __bfloat162float(hl[k]) : 0.f;
      }
#pragma unroll
      for (int k = 0; k < 8; ++k) z = fmaf(a[c][k], wo[c][k], z);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) z += __shfl_xor_sync(0xffffffffu, z, o);
    z += bo;
    const float yh = sigmoidf_stable(z);
    if (p.yhat && lane == 0) p.yhat[r] = yh;
    float dz = 0.f;
    if (p.do_loss) {
      const float y = __ldg(p.desc->y + r), w = __ldg(p.desc->w + r);
      if (p.loss == SB_LOSS_MSE) {
        const float d = yh - y;
        loss_part += w * d * d;
        dz = 2.f * w * d * yh * (1.f - yh) * inv_nnz;
      } else {
        loss_part += w * (fmaxf(z, 0.f) - z * y + log1pf(expf(-fabsf(z))));
        dz = w * (yh - y) * inv_nnz;
      }
    }
    if (p.do_bwd) {
      dz_sum += dz;
#pragma unroll
      for (int c = 0; c < NCH; ++c) {
        const int col0 = c * 256 + lane * 8;
        float g[8];
#pragma unroll
        for (int k = 0; k < 8; ++k) {
          g[k] = dz * wo[c][k] * act_grad_from_out(a[c][k], p.act);   // wo = 0 beyond H -> g = 0 in pad columns
          s_db[c][k] += g[k];
          s_dw[c][k] = fmaf(dz, a[c][k], s_dw[c][k]);
        }
        if (col0 < p.ld_dZ && col0 < p.H) {
          const int np = p.np > 1 ? p.np : 1;
          for (int part = 0; part < np; ++part) {
            uint4 o;
            o.x = pack_bf16x2(bf16_residual(g[0], part), bf16_residual(g[1], part));
            o.y = pack_bf16x2(bf16_residual(g[2], part), bf16_residual(g[3], part));
            o.z = pack_bf16x2(bf16_residual(g[4], part), bf16_residual(g[5], part));
            o.w = pack_bf16x2(bf16_residual(g[6], part), bf16_residual(g[7], part));
            *reinterpret_cast<uint4*>(dZ + part * p.dz_ps + static_cast<size_t>(r) * p.ld_dZ + col0) = o;
          }
        }
      }
    }
  }
  // block reduction: scalars first, then one 256-column chunk at a time
  if (lane == 0) { red_s[0][warp] = loss_part; red_s[1][warp] = dz_sum; }
  __syncthreads();
  if (tid == 0) {
    float l = 0.f, d = 0.f;
    for (int i = 0; i < 8; ++i) { l += red_s[0][i]; d += red_s[1][i]; }
    if (p.do_loss) atomicAdd(p.scal + SCAL_LOSS_SUM, l);
    if (p.do_bwd) atomicAdd(p.g_bo, d);
  }
  if (!p.do_bwd) { trace_end(p.trace); return; }
#pragma unroll
  for (int c = 0; c < NCH; ++c) {
    if (c * 256 >= p.H) break;
    __syncthreads();
#pragma unroll
    for (int k = 0; k < 8; ++k) { red[0][warp][lane * 8 + k] = s_dw[c][k]; red[1][warp][lane * 8 + k] = s_db[c][k]; }
    __syncthreads();
    const int j = c * 256 + tid;
    if (j < p.H) {
      float dw = 0.f, db = 0.f;
#pragma unroll
      for (int i = 0; i < 8; ++i) { dw += red[0][i][tid]; db += red[1][i][tid]; }
      atomicAdd(p.g_wo + j, dw);
      atomicAdd(p.g_bL + j, db);
    }
  }
  trace_end(p.trace);
}

// ------------------------------------------------------------------------------------------------
// K7 fused multi-tensor optimizer over the flat parameter vector (TF 1.x kernel forms: ApplyAdadelta
// res/ssgd_monitor.py:138, ApplyAdam res/ssgd.py:57, ApplyGradientDescent res/ssgd_monitor_bk.py:81,
// ApplyMomentum).  Reads the (all-reduced) gradient once, updates fp32 master weights + state, and in
// bf16 mode refreshes the bf16 shadow of every hidden-layer weight matrix in the same pass.
// ------------------------------------------------------------------------------------------------
struct OptHyper {
  int kind;
  float rho, eps, beta1, beta2, momentum;
};

__device__ __forceinline__ float opt_update(const OptHyper& h, float lr_t, float theta, float g, float& s1, float& s2) {
  switch (h.kind) {
    case SB_OPT_SGD:
      return theta - lr_t * g;
    case SB_OPT_MOMENTUM:
      s1 = s1 * h.momentum + g;
      return theta - lr_t * s1;
    case SB_OPT_ADAM:
      s1 = s1 + (g - s1) * (1.f - h.beta1);
      s2 = s2 + (g * g - s2) * (1.f - h.beta2);
      return theta - lr_t * s1 / (sqrtf(s2) + h.eps);
    default: {  // SB_OPT_ADADELTA
      s1 = s1 * h.rho + g * g * (1.f - h.rho);
      const float upd = sqrtf(s2 + h.eps) / sqrtf(s1 + h.eps) * g;
      s2 = s2 * h.rho + upd * upd * (1.f - h.rho);
      return theta - upd * lr_t;
    }
  }
}

// One work item per block: a run of <= 1024 consecutive parameters.  Runs that lie inside a hidden-layer
// weight matrix also refresh its bf16 shadow W [in, ld_out] (row-major, the layout both the forward GEMM
// (MN-major B operand) and the dA GEMM (K-major B operand) consume).
struct OptWork {
  long long off;          // flat offset of the first element of the run
  int count;              // elements in this run (<= 1024)
  int out_dim;            // > 0: run lies in a weight matrix with this many columns
  long long mat_off;      // flat offset of that matrix
  __nv_bfloat16* Wn;      // shadow base (nullptr: no shadow)
  int ld_out;
  int np;                 // bf16 parts of the shadow (split-precision modes; 1 = plain)
  long long part_stride;  // elements between parts
};

// store 4 / 1 updated weights into the bf16 shadow (all of its parts)
__device__ __forceinline__ void shadow_store4(const OptWork& wk, long long at, const float4& t) {
  for (int part = 0; part < wk.np; ++part) {
    uint2 o;
    o.x = pack_bf16x2(bf16_residual(t.x, part), bf16_residual(t.y, part));
    o.y = pack_bf16x2(bf16_residual(t.z, part), bf16_residual(t.w, part));
    *reinterpret_cast<uint2*>(wk.Wn + part * wk.part_stride + at) = o;
  }
}
__device__ __forceinline__ void shadow_store1(const OptWork& wk, long long at, float t) {
  for (int part = 0; part < wk.np; ++part) wk.Wn[part * wk.part_stride + at] = __float2bfloat16_rn(bf16_residual(t, part));
}

static __global__ void __launch_bounds__(256)
optimizer_kernel(const OptWork* __restrict__ work, const BatchDesc* __restrict__ desc, OptHyper h,
                 float* __restrict__ theta, const float* __restrict__ grad, float* __restrict__ s1, float* __restrict__ s2,
                 const float* __restrict__ scal = nullptr, float* __restrict__ host_scal = nullptr,
                 unsigned long long* __restrict__ trace = nullptr) {
  if (trace != nullptr && blockIdx.x == 0 && threadIdx.x == 0) trace[0] = globaltimer_ns();   // debug timeline: entry
  pdl_wait();
  pdl_launch_dependents();
  if (trace != nullptr && blockIdx.x == 0 && threadIdx.x == 0) trace[2] = globaltimer_ns();   // dependencies resolved
  // last kernel of a step: publish the step scalars (loss sum, n_nz) straight into mapped pinned host memory - a posted
  // PCIe write off the critical path instead of a D2H copy node between two steps (measured: -8.7 us per cfg1 step)
  if (host_scal != nullptr && blockIdx.x == 0 && threadIdx.x < SCAL_COUNT) {
    host_scal[threadIdx.x] = scal[threadIdx.x];
    if (threadIdx.x == 0 && desc->hist != nullptr) *desc->hist = make_float2(scal[SCAL_LOSS_SUM], scal[SCAL_NNZ]);   // loss curve
    __threadfence_system();
  }
  const OptWork wk = work[blockIdx.x];
  const float lr_t = desc->lr_t, gs = desc->gscale;
  // HBM-bound: only touch the state streams the optimizer actually has (SGD: none, Momentum: s1, Adam/Adadelta: s1+s2)
  const bool use_s1 = h.kind != SB_OPT_SGD;
  const bool use_s2 = h.kind == SB_OPT_ADAM || h.kind == SB_OPT_ADADELTA;
  if ((wk.off & 3) == 0 && (wk.count & 3) == 0 && (wk.Wn == nullptr || ((wk.out_dim & 3) == 0 && ((wk.off - wk.mat_off) & 3) == 0))) {
    // 16-byte path: one thread = 4 consecutive parameters (a full 1024-run = 256 threads x float4)
    const int e = threadIdx.x * 4;
    if (e < wk.count) {
      const long long idx = wk.off + e;
      const float4 th = *reinterpret_cast<const float4*>(theta + idx);
      const float4 g = *reinterpret_cast<const float4*>(grad + idx);
      float4 a = use_s1 ? *reinterpret_cast<const float4*>(s1 + idx) : make_float4(0.f, 0.f, 0.f, 0.f);
      float4 b = use_s2 ? *reinterpret_cast<const float4*>(s2 + idx) : make_float4(0.f, 0.f, 0.f, 0.f);
      float4 t;
      t.x = opt_update(h, lr_t, th.x, g.x * gs, a.x, b.x);
      t.y = opt_update(h, lr_t, th.y, g.y * gs, a.y, b.y);
      t.z = opt_update(h, lr_t, th.z, g.z * gs, a.z, b.z);
      t.w = opt_update(h, lr_t, th.w, g.w * gs, a.w, b.w);
      *reinterpret_cast<float4*>(theta + idx) = t;
      if (use_s1) *reinterpret_cast<float4*>(s1 + idx) = a;
      if (use_s2) *reinterpret_cast<float4*>(s2 + idx) = b;
      if (wk.Wn != nullptr) {
        const long long m = idx - wk.mat_off;
        const long long r = m / wk.out_dim;     // 4 consecutive elements never straddle a row (out_dim % 4 == 0)
        shadow_store4(wk, r * wk.ld_out + (m - r * wk.out_dim), t);
      }
    }
    trace_end(trace);
    return;
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int e = threadIdx.x + 256 * i;
    if (e < wk.count) {
      const long long idx = wk.off + e;
      float a = use_s1 ? s1[idx] : 0.f, b = use_s2 ? s2[idx] : 0.f;
      const float t = opt_update(h, lr_t, theta[idx], grad[idx] * gs, a, b);
      theta[idx] = t;
      if (use_s1) s1[idx] = a;
      if (use_s2) s2[idx] = b;
      if (wk.Wn != nullptr) {
        const long long m = idx - wk.mat_off;
        const long long r = m / wk.out_dim;
        shadow_store1(wk, r * wk.ld_out + (m - r * wk.out_dim), t);
      }
    }
  }
  trace_end(trace);
}

// Refresh the bf16 shadows from the fp32 master without touching state (after set_params / restore).
static __global__ void __launch_bounds__(256)
shadow_refresh_kernel(const OptWork* __restrict__ work, const float* __restrict__ theta) {
  const OptWork wk = work[blockIdx.x];
  if (wk.Wn == nullptr) return;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int e = threadIdx.x + 256 * i;
    if (e < wk.count) {
      const long long idx = wk.off + e;
      const long long m = idx - wk.mat_off;
      const long long r = m / wk.out_dim;
      shadow_store1(wk, r * wk.ld_out + (m - r * wk.out_dim), theta[idx]);
    }
  }
}

// ------------------------------------------------------------------------------------------------
// Wide+deep first layer (BASELINE config 4; spec + CPU oracle in oracle/wide_deep.py): Shifu's one-hot normalisation turns
// C categorical columns into n_onehot 0/1 columns of the reference's first dense layer (res/ssgd_monitor.py:57-71).  With
// idx[r, c] = the global one-hot column that is 1 for categorical column c of row r (-1 = missing), the one-hot block of
//     Z_0 = [X_dense | X_onehot] W_0 + b_0
// is a gather-sum of rows of W_e = W_0[n_dense:], and its gradient a scatter-add of dZ_0 rows.  Both read the SAME operand
// precision as the dense path (bf16 shadow / its parts, or fp32), so the sparse evaluation equals the dense layer on the
// materialised one-hot matrix up to fp32 summation order.  HBM/L2-bound: one warp per row, 16-byte accesses.
// ------------------------------------------------------------------------------------------------
struct EmbedParams {
  int rows, n_cat, H;              // H = width of hidden layer 0
  const BatchDesc* desc;           // desc->idx = the batch's index rows [rows, n_cat] (read at run time: a captured graph serves
                                   // any batch)
  const __nv_bfloat16* We;         // bf16 modes: shadow rows of W_e [n_onehot, ldW] (part 0); nullptr in fp32 mode
  long long We_ps; int np;         // parts
  const float* We32;               // fp32 mode: master rows [n_onehot, ldW]
  int ldW;
  float* E; int ldE;               // gather: out [rows, ldE] fp32
  const __nv_bfloat16* dZ; long long dZ_ps; int ld_dZ;   // scatter: dZ_0 (bf16 modes) ...
  const float* dZ32;               // ... or fp32
  float* gWe;                      // scatter: gradient rows of W_e [n_onehot, H] fp32 (flat gradient, ld = H)
};

static __global__ void __launch_bounds__(256) embed_gather_kernel(const EmbedParams p) {
  pdl_wait();
  pdl_launch_dependents();
  const int lane = threadIdx.x & 31;
  const int r = blockIdx.x * 8 + (threadIdx.x >> 5);
  if (r >= p.rows) return;
  const int* __restrict__ idx = p.desc->idx + static_cast<size_t>(r) * p.n_cat;
  for (int c0 = lane * 8; c0 < p.H; c0 += 256) {       // 8 columns per lane per pass
    float acc[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) acc[k] = 0.f;
    for (int c = 0; c < p.n_cat; ++c) {
      const int j = __ldg(idx + c);
      if (j < 0) continue;
      if (p.We != nullptr) {
        for (int part = 0; part < p.np; ++part) {
          const __nv_bfloat16* src = p.We + part * p.We_ps + static_cast<size_t>(j) * p.ldW + c0;
          if (c0 + 8 <= p.H && (p.ldW & 7) == 0) {
            const uint4 raw = __ldg(reinterpret_cast<const uint4*>(src));
            const __nv_bfloat16* h = reinterpret_cast<const __nv_bfloat16*>(&raw);
#pragma unroll
            for (int k = 0; k < 8; ++k) acc[k] += __bfloat162float(h[k]);
          } else {
            for (int k = 0; k < 8; ++k)
              if (c0 + k < p.H) acc[k] += __bfloat162float(src[k]);
          }
        }
      } else {
        const float* src = p.We32 + static_cast<size_t>(j) * p.ldW + c0;
        for (int k = 0; k < 8; ++k)
          if (c0 + k < p.H) acc[k] += __ldg(src + k);
      }
    }
    float* dst = p.E + static_cast<size_t>(r) * p.ldE + c0;
    for (int k = 0; k < 8; ++k)
      if (c0 + k < p.H) dst[k] = acc[k];
  }
}

static __global__ void __launch_bounds__(256) embed_scatter_kernel(const EmbedParams p) {
  pdl_wait();
  pdl_launch_dependents();
  const int lane = threadIdx.x & 31;
  const int r = blockIdx.x * 8 + (threadIdx.x >> 5);
  if (r >= p.rows) return;
  const int* __restrict__ idx = p.desc->idx + static_cast<size_t>(r) * p.n_cat;
  for (int c0 = lane * 4; c0 < p.H; c0 += 128) {       // 4 columns per lane per pass -> red.global.add.v4.f32
    float g[4] = {0.f, 0.f, 0.f, 0.f};
    for (int k = 0; k < 4; ++k) {
      if (c0 + k >= p.H) break;
      if (p.dZ != nullptr) {
        for (int part = 0; part < p.np; ++part) g[k] += __bfloat162float(p.dZ[part * p.dZ_ps + static_cast<size_t>(r) * p.ld_dZ + c0 + k]);
      } else {
        g[k] = p.dZ32[static_cast<size_t>(r) * p.ld_dZ + c0 + k];
      }
    }
    for (int c = 0; c < p.n_cat; ++c) {
      const int j = __ldg(idx + c);
      if (j < 0) continue;
      float* dst = p.gWe + static_cast<size_t>(j) * p.H + c0;
      if (c0 + 4 <= p.H && (p.H & 3) == 0 && (reinterpret_cast<uintptr_t>(p.gWe) & 15) == 0) red_add_v4_f32(dst, g[0], g[1], g[2], g[3]);
      else
        for (int k = 0; k < 4; ++k)
          if (c0 + k < p.H) red_add_f32(dst + k, g[k]);
    }
  }
}

// out[0] = min(out[0], p[0..n)), out[1] = max(out[1], p[0..n)): range check of an index matrix already in device memory
static __global__ void __launch_bounds__(256) int_range_kernel(const int* __restrict__ p, long long n, int* __restrict__ out) {
  int lo = 0x7fffffff, hi = -0x7fffffff - 1;
  for (long long i = blockIdx.x * 256ll + threadIdx.x; i < n; i += gridDim.x * 256ll) {
    const int v = __ldg(p + i);
    lo = min(lo, v); hi = max(hi, v);
  }
  for (int o = 16; o > 0; o >>= 1) {
    lo = min(lo, __shfl_xor_sync(0xffffffffu, lo, o));
    hi = max(hi, __shfl_xor_sync(0xffffffffu, hi, o));
  }
  if ((threadIdx.x & 31) == 0) { atomicMin(out, lo); atomicMax(out + 1, hi); }
}

// acc += g  (epoch-sync schedule: ConditionalAccumulator.apply_grad, res/ssgd_monitor.py:136-141)
static __global__ void axpy_kernel(float* __restrict__ acc, const float* __restrict__ g, long long n,
                                   const float* __restrict__ scal = nullptr, float* __restrict__ host_scal = nullptr) {
  const long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
  if (i < n) acc[i] += g[i];
  if (host_scal != nullptr && i < SCAL_COUNT) {   // tail kernel of an accumulate step: publish (loss sum, n_nz) to the host
    host_scal[i] = scal[i];
    __threadfence_system();
  }
}
// p[0..n) = 0, 16 bytes per thread where aligned (clears the step's gradient buffer on the side stream)
static __global__ void __launch_bounds__(256) zero_f32_kernel(float* __restrict__ p, long long n) {
  const long long n4 = ((reinterpret_cast<uintptr_t>(p) & 15) == 0) ? (n >> 2) : 0;
  for (long long i = blockIdx.x * 256ll + threadIdx.x; i < n4; i += gridDim.x * 256ll)
    reinterpret_cast<float4*>(p)[i] = make_float4(0.f, 0.f, 0.f, 0.f);
  for (long long i = n4 * 4 + blockIdx.x * 256ll + threadIdx.x; i < n; i += gridDim.x * 256ll) p[i] = 0.f;
}
static __global__ void scale_kernel(float* __restrict__ g, const BatchDesc* __restrict__ desc, long long n) {
  const long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
  if (i < n) g[i] *= desc->gscale;
}
static __global__ void fill_kernel(float* __restrict__ p, float v, long long n) {
  const long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
  if (i < n) p[i] = v;
}
// f32 -> bf16 with arbitrary leading dims (test hook operand staging)
static __global__ void cast_bf16_kernel(const float* __restrict__ src, int rows, int cols, __nv_bfloat16* __restrict__ dst, int ld,
                                        int np = 1, long long part_stride = 0) {
  const long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
  if (i < static_cast<long long>(rows) * cols) {
    const int r = static_cast<int>(i / cols), c = static_cast<int>(i % cols);
    for (int part = 0; part < np; ++part)
      dst[part * part_stride + static_cast<size_t>(r) * ld + c] = __float2bfloat16_rn(bf16_residual(src[i], part));
  }
}

}  // namespace sb
