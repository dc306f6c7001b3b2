// Device-side network state shared by the trainer and the scorer: parameters, bf16 shadow weights,
// activation workspace, and the enqueue_* routines that put the step's kernels on a stream.
#pragma once
#include <vector>
#include <map>
#include <mutex>
#include <functional>
#include "common.cuh"
#include "gemm_tc.cuh"
#include "gemm_f32.cuh"
#include "kernels.cuh"
#include "nccl_dyn.h"

namespace sb {

struct Layer {
  int in, out, act;
  long long w_off, b_off;              // offsets into the flat parameter vector
  __nv_bfloat16* Wn = nullptr;  // bf16 shadow of W [in, ld_out] (row-major like the fp32 master)
  int ld_in = 0, ld_out = 0;
};

struct Net {
  int device = 0, num_sms = 148;
  cudaStream_t stream = nullptr;
  cudaStream_t side = nullptr;               // dW GEMMs run here, concurrently with the dA chain on `stream`
  std::vector<cudaEvent_t> ev_dz;            // ev_dz[l]: dZ_l is complete on `stream`
  cudaEvent_t ev_join = nullptr;
  cudaStream_t comm = nullptr;               // the peer exchanges of hidden layer 0's dW chunks alternate between
  cudaStream_t comm2 = nullptr;              // these two streams
  // Peer-exchange schedule (world > 1, set by the trainer around enqueue_backward):
  //   dW_0 runs on the main stream in `dw0_chunks` row chunks of W_0, on_dw0_chunk(c) is called behind each (its exchange
  //   goes to a comm stream and overlaps the GEMMs that follow); dW_1 runs on the main stream in front of dW_0 (dw1_first)
  //   or behind it (dw1_last, so that the LAST chunk's exchange is covered too) instead of beside it.
  int dw0_chunks = 1;
  bool dw1_last = false;
  bool dw1_first = false;                    // dW_1 on the main stream IN FRONT of dW_0 (then after_dw1 is called behind it)
  std::function<int()> after_dw1;
  bool dw1_serial_auto = false;              // let enqueue_backward move dW_1 in front of dW_0 when their grids do not fit together
  std::function<int(int /*chunk*/)> on_dw0_chunk;
  int dw0_chunk_rows() const {
    const int c = dw0_chunks > 1 ? dw0_chunks : 1;
    return ((layers[0].in + c - 1) / c + 127) / 128 * 128;
  }
  // resident steps: the layer-0 forward GEMM's epilogue warps clear this buffer (the step's gradient) while they wait for
  // their first accumulator; consumed (and reset) by enqueue_hidden_forward
  float4* zero_buf = nullptr;
  long long zero_n4 = 0;
  // single-GPU step tail: dW_0 stays on the main stream (PDL-chained after the last dA) and the caller enqueues the
  // optimizer per stream instead of joining first
  bool dw0_on_main = false, defer_join = false;
  cudaEvent_t ev_da_done = nullptr;          // the last dA GEMM (last reader of the bf16 weight shadows) is complete
  std::vector<int> work_begin, work_end;     // optimizer work-table range of layer l (0..L)
  int F = 0, L = 0;             // features, hidden layers
  std::vector<Layer> layers;    // L hidden + 1 output (out = 1)
  long long n_params = 0;
  int precision = SB_PREC_FP32, loss = SB_LOSS_MSE;
  // tensor-core modes keep every GEMM operand as `nparts` bf16 arrays (1 = plain bf16; 3 = SB_PREC_FP32_TC; 2 = BF16X2),
  // see GemmTcParams in gemm_tc.cuh.  Part k of a buffer lies k * <buffer>_ps elements behind part 0.
  int nparts = 1;
  bool tc() const { return precision != SB_PREC_FP32; }
  long long Xb_ps = 0;                       // part strides (elements)
  std::vector<long long> A_ps, Wn_ps;        // A_ps[l] also applies to dZ[l]
  long long resident_ps = 0;
  int max_batch = 0, ldB = 0, ldF = 0;
  bool training = false;

  // Parameter arena: ONE allocation [theta fp32 | s1 | s2 (training) | bf16 weight shadows | extra], so that a trainer can
  // export everything the peer-memory exchange touches with a single CUDA-IPC handle (xchg_p2p.cuh).  `arena_extra_bytes`
  // is set by the trainer BEFORE init(): room for its gradient buffer and flag block behind the parameters.
  char* arena = nullptr;
  size_t arena_bytes = 0, arena_extra_bytes = 0;
  size_t s1_off = 0, s2_off = 0, shadow_off = 0, extra_off = 0;   // byte offsets inside the arena (theta at 0)
  float* theta = nullptr;
  float *s1 = nullptr, *s2 = nullptr;      // optimizer state (training only)
  // bf16 workspace
  __nv_bfloat16* Xb = nullptr;             // current batch as bf16 [rows, ldF]
  std::vector<__nv_bfloat16*> A, dZ;       // A_l, dZ_l as bf16 [rows, ld_out_l]
  // fp32 workspace
  float* Xf = nullptr;
  std::vector<float*> Af, dZf;
  float *yhat = nullptr, *scal = nullptr, *ones = nullptr;
  BatchDesc* desc = nullptr;
  float *stX = nullptr, *stY = nullptr, *stW = nullptr;  // H2D staging (device)
  OptWork* work = nullptr;
  int n_work = 0;
  int launches = 0;  // kernels enqueued since last reset (for gpu_launches accounting)
  // SB_STEP_TRACE=1: every GEMM of a step stamps %globaltimer milestones of its CTA 0 into 16 slots (debug timeline)
  unsigned long long* step_trace = nullptr;
  int trace_k = 0;
  std::vector<std::string> trace_names;
  bool trace_on = true;
  int trace_n = 0;                 // kernels of the last traced step
  // name = role (+ layer, + ".chunk"); GEMMs append "@MxNxK" so that a reader needs no knowledge of the launch order
  unsigned long long* next_trace(const char* name, int layer = -1, int M = 0, int N = 0, int K = 0, int chunk = -1) {
    if (!step_trace || !trace_on || trace_k >= 32) return nullptr;
    if (static_cast<int>(trace_names.size()) <= trace_k) trace_names.resize(trace_k + 1);
    std::string nm = name;
    if (layer >= 0) nm += std::to_string(layer);
    if (chunk >= 0) nm += "." + std::to_string(chunk);
    if (M > 0) nm += "@" + std::to_string(M) + "x" + std::to_string(N) + "x" + std::to_string(K);
    trace_names[trace_k] = nm;
    trace_n = trace_k + 1;
    return step_trace + 16 * (trace_k++);
  }
  // optional per-launch CUDA-event timing (sb_trainer_profile_step): one event after every launch
  bool profiling = false;
  std::vector<cudaEvent_t> prof_events;
  std::vector<std::string> prof_names;
  void mark(const char* name) {
    ++launches;
    if (!profiling) return;
    cudaEvent_t e;
    cudaEventCreate(&e);
    cudaEventRecord(e, stream);
    prof_events.push_back(e);
    prof_names.push_back(name);
  }

  std::vector<void*> allocs;
  // cudaLaunchKernelEx wrapper: optional programmatic-stream-serialization attribute
  template <typename... KArgs, typename... Args>
  int launch(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, bool pdl, Args... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at; cfg.numAttrs = pdl ? 1 : 0;
    SB_CUDA(cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...));
    return SB_OK;
  }
  template <typename T> int dalloc(T** p, size_t n) {
    void* q = nullptr;
    SB_CUDA(cudaMalloc(&q, n * sizeof(T) + 256));
    SB_CUDA(cudaMemsetAsync(q, 0, n * sizeof(T) + 256, stream));
    allocs.push_back(q);
    *p = reinterpret_cast<T*>(q);
    return SB_OK;
  }

  int init(const sb_net_desc* d, int device_, bool training_);
  void destroy();
  int refresh_shadows();
  // forward through the hidden layers (A_0 = current batch -> A_L)
  int enqueue_load(int rows, float* zero_buf = nullptr, long long zero_n = 0);
  // grad != nullptr (training step): the last hidden layer's GEMM also runs the output layer, the loss and the output
  // backward in its epilogue when h_L <= 128; *fused_out tells the caller whether enqueue_out is still needed
  int enqueue_hidden_forward(int rows, float* grad = nullptr, bool* fused_out = nullptr);
  // wide+deep first layer (oracle/wide_deep.py): hidden layer 0 = [n_dense numeric columns | n_onehot one-hot columns of
  // n_cat categorical columns]; a SPARSE step feeds (dense block, index matrix) and evaluates the one-hot block as an
  // embedding gather / scatter-add.  F = n_dense + n_onehot, the parameters are those of the dense net.
  int n_dense = 0, n_onehot = 0, n_cat = 0, ldD = 0;
  int* idx = nullptr;                        // [max_batch, n_cat] staged indices
  float* E = nullptr;                        // [max_batch, ld_out_0] embedding sums
  bool sparse_step = false;                  // set while a sparse step is being enqueued
  int set_sparse(int n_dense_, int n_onehot_, int n_cat_);
  int enqueue_embed(int rows, bool scatter, float* grad, cudaStream_t st);
  static constexpr int fuse_out_max = 256;   // widest last hidden layer whose GEMM also runs the output layer (one n-tile)
  // bf16 HBM-resident training set (trainer): when `from_resident` is set while enqueueing, layer 0's GEMMs read their A
  // operand from it by TMA at row offset desc->row0 and no load_batch kernel runs (a sparse step: the set holds the dense
  // block, pitch ldD, and the embedding gather runs in front of the layer-0 forward GEMM)
  const __nv_bfloat16* resident_Xb = nullptr;
  long long resident_rows = 0;
  bool from_resident = false;
  int enqueue_out(int rows, bool do_loss, bool do_bwd, float* yhat_dst, float* grad);
  int enqueue_backward(int rows, float* grad);
};

int validate_desc(const sb_net_desc* d);

}  // namespace sb
