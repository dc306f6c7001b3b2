// extern "C" surface of libshifu_b200.so: trainer, scorer, rendezvous, test hooks.
// See include/shifu_b200.h for the contract and the reference call each entry point replaces.
#include <math.h>
#include <stdlib.h>
#include <string.h>
#include <algorithm>
#include <memory>
#include <random>
#include "net.cuh"
#include "gemm_tc_launch.cuh"
#include "savedmodel.h"
#include "xchg_p2p.cuh"

using namespace sb;

// ================================================================================================
// trainer
// ================================================================================================
enum { G_STEP = 0, G_ACC = 1, G_KINDS = 2 };

struct sb_trainer {
  Net net;
  sb_net_desc desc;
  OptHyper hyper;
  float lr = 0.f;
  int rank = 0, world = 1;
  NcclComm comm = nullptr;
  float *grad = nullptr, *s1 = nullptr, *s2 = nullptr, *acc = nullptr;
  int n_acc = 0;
  float grad_out_scale = 1.f;  // what sb_trainer_get_grads multiplies the raw buffer by
  long long global_step = 0;
  float* h_scal = nullptr;  // pinned + mapped [SCAL_COUNT]: written by the tail kernel of every step
  float* d_hscal = nullptr; // device-side alias of h_scal
  // loss curve: (loss sum, n_nz) of the last HIST update steps, ring indexed by global_step % HIST, pinned + mapped
  enum { HIST = 8192 };
  float2* h_hist = nullptr;
  float2* d_hist = nullptr;
  float2* hist_slot(long long step) { return d_hist ? d_hist + (step % HIST) : nullptr; }
  // HBM-resident training set
  float *dsX = nullptr, *dsY = nullptr, *dsW = nullptr;   // dsX only in fp32 mode
  __nv_bfloat16* dsXb = nullptr;                           // bf16 mode: the set in GEMM-operand form [ds_rows, ldF]
  int* dsP = nullptr;                                      // prefix counts of non-zero weights [ds_rows + 1]
  long long ds_rows = 0;
  // wide+deep set (sb_trainer_load_dataset_sparse): dsX / dsXb hold the dense block (n_dense columns, bf16 pitch ldD),
  // dsI the index matrix [ds_rows, n_cat]; the resident entry points then run sparse steps
  int* dsI = nullptr;
  bool ds_sparse = false;
  std::map<std::pair<int, int>, cudaGraphExec_t> graphs;  // (rows, kind * 2 + from_resident) -> captured step
  std::map<int, int> kernels_per_step;
  // peer-memory exchange (xchg_p2p.cuh): the net's parameter arena [theta | s1 | s2 | shadows | gradient | P2PFlags] is
  // ONE exported allocation; `xch` aliases it
  void* xch = nullptr;
  long long xch_n4 = 0;            // float4 count of the padded gradient
  long long grad_off = 0, flags_off = 0;   // byte offsets of the gradient / flag block inside the arena
  P2PFlags* flags = nullptr;
  P2PPeers* d_peers = nullptr;     // device table of every rank's arena
  std::vector<void*> peer_bases;   // opened IPC mappings (to close)
  bool p2p_ready = false;
  bool peers_share_device = false; // in-process replicas on this device (tests): smaller exchange grids, dW_1 behind dW_0
  bool grad_sharded = false;       // the reduced gradient of the last step lives in slices on its owners (sb_trainer_get_grads gathers)
  bool master_stale = false;       // sharded updates ran since the fp32 master / state were last gathered from their owners
  unsigned int epoch = 0;
  unsigned int* h_err = nullptr;   // pinned + mapped: a peer that never arrived (xchg_p2p.cuh), 0 = none
  unsigned int* d_herr = nullptr;
  unsigned long long xchg_timeout_ns = 300ull * 1000000000ull;
  int xchg_blocks = 0;             // grid cap of the exchange kernels (0 = one block per SM)
  // slot table of the exchange (fixed for the trainer's life: it defines who owns which run): slot 0 = every layer but
  // hidden layer 0, slots 1..x_chunks = row chunks of hidden layer 0 (the last one also carries b_0)
  int x_chunks = 1, x_slots = 2;
  int x_begin[SB_XCHG_SLOTS] = {}, x_end[SB_XCHG_SLOTS] = {};
  cudaEvent_t ev_x[SB_XCHG_SLOTS] = {};   // exchange of slot s complete (recorded on its comm stream)
  cudaEvent_t ev_c[SB_XCHG_SLOTS] = {};   // dW_0 chunk c complete on the main stream / tail of the main stream
  bool ll_ready = false;           // the LL exchange (xchg_ll_kernel) is usable: plain bf16, world > 1, buffers in the arena
  long long llg_off = 0, lls_off = 0;
  int x_sent = 0;                  // (while enqueueing a step) slots whose exchange the dW_0 chunk hook has launched
  // pipelined host-buffer steps (sb_trainer_step_async): second staging slot + copy stream, so the H2D of batch i+1
  // overlaps the compute of batch i
  cudaStream_t copy_stream = nullptr;
  float *st2X = nullptr, *st2Y = nullptr, *st2W = nullptr;
  cudaEvent_t ev_copied[2] = {nullptr, nullptr}, ev_consumed[2] = {nullptr, nullptr};
  unsigned long long async_steps = 0;
  // resident steps: the batch descriptor of step i+1 is written on `prep` while step i still runs (two descriptor /
  // scalar pairs, one captured graph per pair), so set_batch_kernel leaves the critical path (-2.9 us per cfg1 step)
  BatchDesc* descs[2] = {nullptr, nullptr};
  float* scals[2] = {nullptr, nullptr};
  cudaStream_t prep = nullptr;
  cudaEvent_t ev_prep[2] = {nullptr, nullptr}, ev_pos[2] = {nullptr, nullptr};
  unsigned long long prep_steps = 0;
  bool have_pos = false;   // ev_pos[] of the previous step is valid (no other user of the descriptors in between)
  // sb_trainer_run_resident: RUN_S steps per captured graph (kernel -> kernel edges instead of a graph turn-around
  // between steps), two alternating descriptor sets so that the descriptors of chunk i+1 are written while chunk i runs
  enum { RUN_S = 4 };
  BatchDesc* run_descs[2][RUN_S] = {};
  float* run_scals[2][RUN_S] = {};
  cudaEvent_t ev_run_prep[2] = {nullptr, nullptr}, ev_run_done[2] = {nullptr, nullptr};
  bool run_used[2] = {false, false};
  unsigned long long run_chunks = 0;
  std::map<int, cudaGraphExec_t> run_graphs;   // rows * 2 + set
};

static float lr_for_step(const sb_trainer* t, long long step /*1-based*/) {
  if (t->hyper.kind == SB_OPT_ADAM) {
    const double b1 = t->hyper.beta1, b2 = t->hyper.beta2;
    return static_cast<float>(t->lr * sqrt(1.0 - pow(b2, static_cast<double>(step))) / (1.0 - pow(b1, static_cast<double>(step))));
  }
  return t->lr;
}

static int enqueue_allreduce(sb_trainer* t, float* buf) {
  if (t->world <= 1) return SB_OK;
  NcclApi* api = nccl_api();
  SB_CHECK(api && t->comm, SB_ERR_NCCL, "no gradient exchange configured: world = %d but neither an NCCL communicator (nccl_id) nor a "
           "peer table (sb_trainer_set_peer_handles / _pointers) exists", t->world);
  int r = api->AllReduce(buf, buf, static_cast<size_t>(t->net.n_params), NCCL_FLOAT32, NCCL_SUM, t->comm, t->net.stream);
  SB_CHECK(r == 0, SB_ERR_NCCL, "ncclAllReduce failed: %s", api->GetErrorString(r));
  return SB_OK;
}

static int enqueue_optimizer(sb_trainer* t, const float* g, int w0 = 0, int w1 = -1, cudaStream_t st = nullptr,
                             bool publish_scalars = false, bool pdl = false) {
  Net& n = t->net;
  if (w1 < 0) w1 = n.n_work;
  if (!st) st = n.stream;
  if (w1 <= w0) return SB_OK;
  // pdl = false: plain dependency (runs after a stream join / on the comm stream)
  SB_TRY(n.launch(optimizer_kernel, dim3(static_cast<unsigned>(w1 - w0)), dim3(256), 0, st, pdl, n.work + w0, n.desc, t->hyper,
                  n.theta, g, n.s1, n.s2, n.scal, publish_scalars ? t->d_hscal : static_cast<float*>(nullptr),
                  n.next_trace(st == n.stream ? "opt" : "opt_side")));
  n.mark("optimizer");
  return SB_OK;
}

// slots of the sharded exchange: bit 0 = A (every layer but hidden layer 0), bits 1.. = the row chunks of hidden layer 0
enum { XSEG_A = 1 };
static int xseg_all(const sb_trainer* t) { return (1 << t->x_slots) - 1; }

static XchgParams xchg_params(sb_trainer* t) {
  Net& n = t->net;
  XchgParams p;
  memset(&p, 0, sizeof(p));
  p.peers = t->d_peers;
  p.rank = t->rank; p.world = t->world;
  p.s1_off = static_cast<long long>(n.s1_off); p.s2_off = static_cast<long long>(n.s2_off);
  p.grad_off = t->grad_off; p.flags_off = t->flags_off;
  p.work = n.work;
  p.n_slots = t->x_slots;
  for (int sl = 0; sl < t->x_slots; ++sl) { p.slot_begin[sl] = t->x_begin[sl]; p.slot_end[sl] = t->x_end[sl]; }
  p.desc = n.desc;
  p.hyper = t->hyper;
  p.host_err = t->d_herr;
  p.timeout_ns = t->xchg_timeout_ns;
  static const bool fence_sys = getenv("SB_XCHG_FENCE_SYS") != nullptr;
  p.fence_gpu = fence_sys ? 0 : 1;
  return p;
}

// reduce-scatter -> owner update -> all-gather of the operands for the given segments (xchg_p2p.cuh); `g` must be t->grad
static int enqueue_xchg(sb_trainer* t, int slot_mask, cudaStream_t st, bool publish_scalars, bool pdl, bool alone = false) {
  Net& n = t->net;
  XchgParams p = xchg_params(t);
  p.slot_mask = slot_mask;
  p.scal = publish_scalars ? n.scal : nullptr;
  p.host_scal = publish_scalars ? t->d_hscal : nullptr;
  char nm[24];
  if (slot_mask == XSEG_A) snprintf(nm, sizeof(nm), "xchg_A");
  else if ((slot_mask & (slot_mask - 1)) == 0) snprintf(nm, sizeof(nm), "xchg_B%d", __builtin_ctz(slot_mask) - 1);
  else snprintf(nm, sizeof(nm), "xchg");
  p.trace = n.next_trace(nm);
  int runs = 0, all_runs = 0;      // owned runs of the launch (the largest share) / runs of the launch
  for (int sl = 0; sl < t->x_slots; ++sl)
    if ((slot_mask >> sl) & 1) {
      runs += (p.slot_end[sl] - p.slot_begin[sl] + t->world - 1) / t->world;
      all_runs += p.slot_end[sl] - p.slot_begin[sl];
    }
  const int U = t->world <= 2 ? 2 : 1;      // runs per block iteration of the update phase (xchg_update_kernel)
  const int want = std::max((runs + U - 1) / U, (all_runs - runs + 3) / 4);   // ... and 4 per iteration of the gather phase
  // one block per SM and launch: it fits beside a forward GEMM CTA, and two launches fit beside a dW GEMM CTA (xchg_p2p.cuh;
  // with two blocks per SM the chunk exchanges crowded dW_1 out: 15 -> 27 us, measured).  Blocks that find no room wait for
  // GEMM CTAs to leave - those never wait for an exchange, so this cannot deadlock, only be slow.
  // (alone: nothing but other exchange launches runs beside this one - two blocks per SM, all loads of a phase in one round)
  int grid = t->xchg_blocks > 0 ? t->xchg_blocks : (alone ? 2 : 1) * n.num_sms;
  if (t->peers_share_device && grid > 32) grid = 32;    // replicas on ONE device: leave registers to the replica being waited for
  if (grid > want) grid = want;
  if (grid < 1) grid = 1;
  const dim3 g(static_cast<unsigned>(grid)), b(256);
  // Every launch uses the LL protocol (flags inside the data) where it is available.  Measured on 2 x B200, cfg2: LL for every
  // launch 163.8 us/step, only for the launch nothing runs beside 168.2, for none 171.4; an LL launch takes 21-28 us where
  // the flag-and-pull kernel takes 32-47, at the price of 2-4 us on the GEMM beside it (polling, doubled store traffic).
  if (t->ll_ready) {
    LLParams lp;
    lp.x = p; lp.llg_off = t->llg_off; lp.lls_off = t->lls_off; lp.n4 = t->xch_n4;
    if (t->world <= 2) SB_TRY(n.launch(xchg_ll_kernel<2>, g, b, 0, st, pdl, lp));
    else if (t->world <= 4) SB_TRY(n.launch(xchg_ll_kernel<4>, g, b, 0, st, pdl, lp));
    else if (t->world <= 8) SB_TRY(n.launch(xchg_ll_kernel<8>, g, b, 0, st, pdl, lp));
    else SB_TRY(n.launch(xchg_ll_kernel<16>, g, b, 0, st, pdl, lp));
  } else
  if (t->world <= 2) SB_TRY(n.launch(xchg_update_kernel<2>, g, b, 0, st, pdl, p));
  else if (t->world <= 4) SB_TRY(n.launch(xchg_update_kernel<4>, g, b, 0, st, pdl, p));
  else if (t->world <= 8) SB_TRY(n.launch(xchg_update_kernel<8>, g, b, 0, st, pdl, p));
  else SB_TRY(n.launch(xchg_update_kernel<16>, g, b, 0, st, pdl, p));
  n.mark("xchg_update");
  t->master_stale = true;
  t->grad_sharded = true;
  return SB_OK;
}

// before the host reads theta / s1 / s2: pull the runs other ranks own from their owners (no-op unless sharded updates ran)
static int gather_master(sb_trainer* t) {
  if (!t->p2p_ready || !t->master_stale || t->world <= 1) return SB_OK;
  Net& n = t->net;
  SB_CUDA(cudaStreamSynchronize(n.stream));     // my last exchange kernel has seen every peer's done flag
  XchgParams p = xchg_params(t);
  gather_master_kernel<<<n.n_work, 256, 0, n.stream>>>(p, 0);
  SB_CUDA(cudaGetLastError());
  SB_CUDA(cudaStreamSynchronize(n.stream));
  t->master_stale = false;
  return SB_OK;
}

// the body of one step as a sequence of stream operations (captured into a CUDA graph)
static int enqueue_step_body(sb_trainer* t, int rows, int kind, bool resident = false, bool sparse = false) {
  Net& n = t->net;
  struct Scope {
    Net& n;
    ~Scope() {
      n.from_resident = false; n.zero_buf = nullptr; n.dw0_on_main = n.defer_join = false; n.sparse_step = false;
      n.dw0_chunks = 1; n.dw1_last = false; n.on_dw0_chunk = nullptr;
      n.dw1_first = false; n.after_dw1 = nullptr; n.dw1_serial_auto = false;
    }
  } scope{n};
  n.from_resident = resident;
  n.sparse_step = sparse;
  n.trace_k = 0;
  // ---- schedule of the step's tail ----
  // Single GPU, one update per mini-batch: no exchange, so nothing needs ALL gradients at once.  dW_0 runs on the main
  // stream behind the last dA GEMM and is followed (PDL) by the optimizer of layer 0 alone; the side stream updates the
  // other layers right after their dW GEMMs; the two streams only join at the end of the graph.
  const bool split_tail = kind == G_STEP && (t->world == 1 || t->p2p_ready) && !n.profiling && n.side != nullptr && n.tc() &&
                          n.L > 1;
  // Peer exchange (world > 1): one exchange launch costs 20-30 us through NVSwitch however little data it moves (fabric latency,
  // xchg_p2p.cuh) - hidden when a GEMM follows it, exposed in full behind the last GEMM:
  //   main:  ... dA_1 -> dW_1 -> dW_0 chunk 0 -> dW_0 chunk 1 | wait A, B0, B1 | next step
  //   side:  ... dW_2 ...     A ------------->
  //   comm:                             B0 ---------------->    B1 ------>
  // dW_1 runs in front of dW_0: A (every layer but hidden layer 0) and B0 hide behind dW_0's chunks, only B1 - half of layer
  // 0 - runs on an otherwise idle GPU (an exchange kernel beside a GEMM takes 40-47 us, alone ~25; measured, 2 x B200).
  // Replicas that share ONE device (tests) put dW_1 BEHIND dW_0 as cover for B1, and A behind dW_1: with three exchange
  // launches of both replicas waiting beside each other's persistent GEMMs the order above stopped making progress within
  // the exchange timeout.
  const bool xsched = split_tail && t->world > 1;
  const bool order_last = t->peers_share_device;
  if (resident) {
    // no load kernel: the batch is read by TMA from the bf16 resident set; set_batch_kernel already published n_nz.
    // The gradient buffer is first written by the last forward layer's epilogue, so with more than one hidden layer the
    // layer-0 forward GEMM clears it (its epilogue warps idle until their first accumulator completes); a memset node
    // at the head of the chain cost ~3 us per step.  No peer reads it any more: the previous step's main stream waited
    // for every exchange.
    if (n.L > 1) {
      n.zero_buf = reinterpret_cast<float4*>(t->grad);   // cudaMalloc'ed, padded to xch_n4 float4
      n.zero_n4 = t->xch_n4;
    } else {
      SB_CUDA(cudaMemsetAsync(t->grad, 0, sizeof(float) * n.n_params, n.stream));
    }
  } else {
    SB_TRY(n.enqueue_load(rows, t->grad, n.n_params));   // also clears the gradient buffer and the step scalars
  }
  bool fused_out = false;
  SB_TRY(n.enqueue_hidden_forward(rows, t->grad, &fused_out));
  if (!fused_out) SB_TRY(n.enqueue_out(rows, true, true, nullptr, t->grad));
  // (dW_0 on the main stream also when an exchange or the accumulate kernel follows: it is then joined with the side
  // stream as before)
  n.dw0_on_main = !n.profiling && n.side != nullptr && n.tc() && n.L > 1;
  n.defer_join = split_tail;
  cudaStream_t comms[2] = {n.comm2, n.comm};
  if (xsched) {
    // dW_1 leaves the side stream.  (Beside dW_0, like the single-GPU schedule, the chunks of dW_0 shared the SMs with dW_1:
    // 31 + 19 us instead of 18 + 19, measured on 2 x B200.)
    n.dw0_chunks = t->x_chunks;
    n.dw1_last = order_last;
    n.dw1_first = !order_last;
    t->x_sent = 0;
    if (n.dw1_first) {
      n.after_dw1 = [t]() -> int {       // slot A on the side stream, behind dW_1 (main) and the other layers' dW GEMMs (side)
        Net& nn = t->net;
        SB_CUDA(cudaEventRecord(t->ev_c[0], nn.stream));
        SB_CUDA(cudaStreamWaitEvent(nn.side, t->ev_c[0], 0));
        SB_TRY(enqueue_xchg(t, XSEG_A, nn.side, false, false));
        SB_CUDA(cudaEventRecord(t->ev_x[0], nn.side));
        t->x_sent |= XSEG_A;
        return SB_OK;
      };
    }
    n.on_dw0_chunk = [t, comms](int c) -> int {
      Net& nn = t->net;
      cudaStream_t cs = comms[c & 1];
      SB_CUDA(cudaEventRecord(t->ev_c[1 + c], nn.stream));
      SB_CUDA(cudaStreamWaitEvent(cs, t->ev_c[1 + c], 0));
      const bool last = c == t->x_chunks - 1;
      SB_TRY(enqueue_xchg(t, 1 << (1 + c), cs, last, false, last && !nn.dw1_last));   // (the last chunk publishes the step scalars;
                                                                                      //  no GEMM follows it unless dW_1 does)
      SB_CUDA(cudaEventRecord(t->ev_x[1 + c], cs));
      t->x_sent |= 1 << (1 + c);
      return SB_OK;
    };
  }
  if (split_tail && !xsched) {
    // one GPU: dW_1 may move in front of dW_0 (Net::dw1_serial_auto); the side stream's optimizer launch then waits for it
    n.dw1_serial_auto = true;
    n.after_dw1 = [t]() -> int {
      Net& nn = t->net;
      SB_CUDA(cudaEventRecord(t->ev_c[0], nn.stream));
      SB_CUDA(cudaStreamWaitEvent(nn.side, t->ev_c[0], 0));
      return SB_OK;
    };
  }
  SB_TRY(n.enqueue_backward(rows, t->grad));
  if (xsched) {
    // slot A: every gradient but hidden layer 0's - complete behind dW_1 (main stream), the other layers' dW GEMMs (side
    // stream) and the last dA GEMM (the last reader of their weight shadows).  With dW_1 in front of dW_0, after_dw1 has
    // launched it; with dW_1 behind dW_0 it goes to the side stream here.
    if (!(t->x_sent & XSEG_A)) {
      SB_CUDA(cudaEventRecord(t->ev_c[0], n.stream));
      SB_CUDA(cudaStreamWaitEvent(n.side, t->ev_c[0], 0));
      SB_TRY(enqueue_xchg(t, XSEG_A, n.side, false, false));
      SB_CUDA(cudaEventRecord(t->ev_x[0], n.side));
    }
    // whatever follows on the main stream (the next step, which clears the gradient buffer peers read, or the end of the
    // graph) waits for every slot
    for (int c = 0; c < t->x_chunks; ++c)
      if ((t->x_sent >> (1 + c)) & 1) SB_CUDA(cudaStreamWaitEvent(n.stream, t->ev_x[1 + c], 0));
    // (a layer-0 dW that was not cut into the trainer's chunks - wide+deep steps - is exchanged here, behind everything)
    const int missing = (xseg_all(t) & ~XSEG_A) & ~t->x_sent;
    if (missing) SB_TRY(enqueue_xchg(t, missing, n.stream, true, false));
    SB_CUDA(cudaStreamWaitEvent(n.stream, t->ev_x[0], 0));
    return SB_OK;
  }
  if (split_tail) {
    SB_TRY(enqueue_optimizer(t, t->grad, n.work_begin[0], n.work_end[0], n.stream, true, true));
    // the other layers' shadows are read by the dA GEMMs on the main stream: update them only after the last one
    SB_CUDA(cudaStreamWaitEvent(n.side, n.ev_da_done, 0));
    SB_TRY(enqueue_optimizer(t, t->grad, n.work_end[0], n.n_work, n.side));
    SB_CUDA(cudaEventRecord(n.ev_join, n.side));
    SB_CUDA(cudaStreamWaitEvent(n.stream, n.ev_join, 0));
    return SB_OK;
  }
  if (kind == G_STEP) {
    if (t->world > 1 && t->p2p_ready) {
      // (fp32 mode, one hidden layer: no split tail) one launch handles both segments
      SB_TRY(enqueue_xchg(t, xseg_all(t), n.stream, true, false));
    } else {
      SB_TRY(enqueue_allreduce(t, t->grad));
      if (t->world > 1 && n.profiling) { n.mark("allreduce"); --n.launches; }
      SB_TRY(enqueue_optimizer(t, t->grad, 0, -1, nullptr, true, false));
    }
  } else {
    const long long np = n.n_params;
    axpy_kernel<<<static_cast<unsigned>((np + 255) / 256), 256, 0, n.stream>>>(t->acc, t->grad, np, n.scal, t->d_hscal);
    SB_CUDA(cudaGetLastError());
    n.mark("accumulate");
  }
  return SB_OK;
}

static int get_graph(sb_trainer* t, int rows, int kind, bool resident, int pair, cudaGraphExec_t* out, bool sparse = false) {
  auto key = std::make_pair(rows, kind * 8 + (sparse ? 4 : 0) + (resident ? 2 : 0) + pair);
  auto it = t->graphs.find(key);
  if (it != t->graphs.end()) { *out = it->second; return SB_OK; }
  Net& n = t->net;
  n.launches = 0;
  cudaGraph_t g = nullptr;
  SB_CUDA(cudaStreamBeginCapture(n.stream, cudaStreamCaptureModeThreadLocal));
  int s = enqueue_step_body(t, rows, kind, resident, sparse);
  cudaError_t e = cudaStreamEndCapture(n.stream, &g);
  if (s != SB_OK) { if (g) cudaGraphDestroy(g); return s; }
  SB_CHECK(e == cudaSuccess, SB_ERR_CUDA, "cudaStreamEndCapture failed: %s", cudaGetErrorString(e));
  cudaGraphExec_t ge = nullptr;
  SB_CUDA(cudaGraphInstantiate(&ge, g, 0));
  cudaGraphDestroy(g);
  t->graphs[key] = ge;
  if (kind == G_STEP && sparse == t->ds_sparse && (resident || !t->dsXb)) t->kernels_per_step[rows] = n.launches + 1;  // + set_batch_kernel
  *out = ge;
  return SB_OK;
}

// X, y, w (and idx, the index rows of a sparse step) are DEVICE pointers here
static int run_step(sb_trainer* t, const float* X, const float* y, const float* w, int rows, int kind, long long resident_row0 = -1,
                    bool sparse = false, const int* idx = nullptr) {
  Net& n = t->net;
  SB_CHECK(rows > 0 && rows <= n.max_batch, SB_ERR_INVALID, "rows=%d outside (0, max_batch=%d]", rows, n.max_batch);
  SB_CUDA(cudaSetDevice(n.device));
  static const bool no_graph = getenv("SB_NO_GRAPH") != nullptr;
  const bool resident = resident_row0 >= 0 && t->dsXb != nullptr;
  // descriptor / scalar pair of this step: resident graph steps alternate, everything else uses pair 0
  const bool prep = resident && !no_graph;
  const int pair = prep ? static_cast<int>(t->prep_steps & 1) : 0;
  n.desc = t->descs[pair];
  n.scal = t->scals[pair];
  cudaGraphExec_t ge = nullptr;
  if (!no_graph) SB_TRY(get_graph(t, rows, kind, resident, pair, &ge, sparse));
  float lr_t = t->lr, gscale = 1.f / static_cast<float>(t->world);
  if (kind == G_STEP) {
    ++t->global_step;
    lr_t = lr_for_step(t, t->global_step);
  }
  if (kind == G_STEP) ++t->epoch;
  if (prep) {
    // pair `pair` was last read by the step two back and by whatever followed it on the main stream before the previous
    // step's graph: ev_pos[pair ^ 1] (recorded right before that graph) covers both.  First step of a run: join the
    // main stream's current position.
    if (!t->have_pos) SB_CUDA(cudaEventRecord(t->ev_pos[pair ^ 1], n.stream));
    SB_CUDA(cudaStreamWaitEvent(t->prep, t->ev_pos[pair ^ 1], 0));
    set_batch_kernel<<<1, 1, 0, t->prep>>>(n.desc, nullptr, y, w, lr_t, gscale, t->epoch, static_cast<int>(resident_row0), t->dsP, rows, n.scal,
                                           kind == G_STEP ? t->hist_slot(t->global_step) : nullptr, idx);
    SB_CUDA(cudaGetLastError());
    SB_CUDA(cudaEventRecord(t->ev_prep[pair], t->prep));
    SB_CUDA(cudaEventRecord(t->ev_pos[pair], n.stream));
    SB_CUDA(cudaStreamWaitEvent(n.stream, t->ev_prep[pair], 0));
    t->have_pos = true;
    ++t->prep_steps;
  } else {
    t->have_pos = false;
    if (resident)
      set_batch_kernel<<<1, 1, 0, n.stream>>>(n.desc, nullptr, y, w, lr_t, gscale, t->epoch, static_cast<int>(resident_row0), t->dsP, rows, n.scal,
                                               kind == G_STEP ? t->hist_slot(t->global_step) : nullptr, idx);
    else
      set_batch_kernel<<<1, 1, 0, n.stream>>>(n.desc, X, y, w ? w : n.ones, lr_t, gscale, t->epoch, 0, nullptr, 0, nullptr,
                                               kind == G_STEP ? t->hist_slot(t->global_step) : nullptr, idx);
  }
  SB_CUDA(cudaGetLastError());
  if (no_graph) SB_TRY(enqueue_step_body(t, rows, kind, resident, sparse));
  else SB_CUDA(cudaGraphLaunch(ge, n.stream));
  // the step's tail kernel (optimizer / accumulate) wrote (loss sum, n_nz) into h_scal; visible after a stream sync
  if (kind == G_ACC) ++t->n_acc;
  t->grad_out_scale = (kind == G_STEP) ? gscale : 1.f;
  return SB_OK;
}

// an NCCL failure on another rank (peer died, transport error) is reported asynchronously: surface it at every point where
// the host waits for the device instead of hanging in the next collective
static int poll_nccl(sb_trainer* t) {
  if (!t->comm) return SB_OK;
  NcclApi* api = nccl_api();
  if (!api || !api->CommGetAsyncError) return SB_OK;
  int err = 0;
  if (api->CommGetAsyncError(t->comm, &err) == 0 && err != 0)
    return set_error(SB_ERR_NCCL, "NCCL asynchronous error on rank %d: %s", t->rank, api->GetErrorString(err));
  return SB_OK;
}

// a peer that never arrived at the exchange (xchg_p2p.cuh) left a note in mapped host memory
static int poll_xchg(sb_trainer* t) {
  if (!t->h_err) return SB_OK;
  const unsigned int e = *reinterpret_cast<volatile unsigned int*>(t->h_err);
  if (e == 0) return SB_OK;
  return set_error(SB_ERR_NCCL, "gradient exchange timed out on rank %d: rank %u did not reach slot %u of the exchange within %.0f s "
                   "(peer process dead or stuck); this trainer is no longer usable", t->rank, (e - 1) & 15u, (e - 1) >> 4,
                   t->xchg_timeout_ns * 1e-9);
}

static int finish_loss(sb_trainer* t, float* loss_out) {
  SB_CUDA(cudaStreamSynchronize(t->net.stream));
  SB_TRY(poll_nccl(t));
  SB_TRY(poll_xchg(t));
  if (loss_out) {
    const float nnz = t->h_scal[SCAL_NNZ];
    *loss_out = nnz > 0.f ? t->h_scal[SCAL_LOSS_SUM] / nnz : 0.f;
  }
  return SB_OK;
}

// X / y / w of load_dataset, eval_loss and predict may be HOST or DEVICE pointers (unified addressing: the copies use
// cudaMemcpyDefault); the GPU text ingest hands over device arrays so that the parsed set never visits the host
static bool is_device_ptr(const void* p) {
  if (!p) return false;
  cudaPointerAttributes at;
  if (cudaPointerGetAttributes(&at, p) != cudaSuccess) { cudaGetLastError(); return false; }
  return at.type == cudaMemoryTypeDevice;
}

static int stage_host_batch(sb_trainer* t, const float* X, const float* y, const float* w, int rows) {
  Net& n = t->net;
  SB_CHECK(X && y, SB_ERR_INVALID, "X and y must not be null");
  SB_CHECK(rows > 0 && rows <= n.max_batch, SB_ERR_INVALID, "rows=%d outside (0, max_batch=%d]", rows, n.max_batch);
  SB_CUDA(cudaSetDevice(n.device));
  SB_CUDA(cudaMemcpyAsync(n.stX, X, sizeof(float) * rows * static_cast<size_t>(n.F), cudaMemcpyHostToDevice, n.stream));
  SB_CUDA(cudaMemcpyAsync(n.stY, y, sizeof(float) * rows, cudaMemcpyHostToDevice, n.stream));
  if (w) SB_CUDA(cudaMemcpyAsync(n.stW, w, sizeof(float) * rows, cudaMemcpyHostToDevice, n.stream));
  return SB_OK;
}

extern "C" {

const char* sb_version(void) { return "shifu_b200 0.1 (sm_100a)"; }
const char* sb_last_error(void) { return last_error_ref().c_str(); }

int sb_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) return set_error(SB_ERR_CUDA, "cudaGetDeviceCount failed");
  int ok = 0;
  for (int i = 0; i < n; ++i) {
    cudaDeviceProp p;
    if (cudaGetDeviceProperties(&p, i) == cudaSuccess && p.major == 10) ++ok;
  }
  return ok;
}

int sb_host_alloc(void** ptr, uint64_t bytes) {
  SB_CHECK(ptr, SB_ERR_INVALID, "ptr is null");
  SB_CUDA(cudaHostAlloc(ptr, bytes, cudaHostAllocDefault));
  return SB_OK;
}
int sb_host_free(void* ptr) {
  SB_CUDA(cudaFreeHost(ptr));
  return SB_OK;
}

int sb_nccl_unique_id(void* out128) {
  SB_CHECK(out128, SB_ERR_INVALID, "out is null");
  NcclApi* api = nccl_api();
  SB_CHECK(api, SB_ERR_NCCL, "libnccl.so.2 could not be loaded");
  NcclUniqueId id;
  int r = api->GetUniqueId(&id);
  SB_CHECK(r == 0, SB_ERR_NCCL, "ncclGetUniqueId failed: %s", api->GetErrorString(r));
  memcpy(out128, &id, sizeof(id));
  return SB_OK;
}

int sb_trainer_create(const sb_net_desc* desc, int device, const void* nccl_id, int rank, int world, sb_trainer_t** out) {
  SB_CHECK(out, SB_ERR_INVALID, "out is null");
  *out = nullptr;
  SB_TRY(validate_desc(desc));
  SB_CHECK(world >= 1 && rank >= 0 && rank < world, SB_ERR_INVALID, "bad rank/world %d/%d", rank, world);
  // world > 1 without an NCCL id: the ranks live in one process (sb_trainer_set_peer_pointers is then the only exchange)
  std::unique_ptr<sb_trainer> t(new sb_trainer());
  t->desc = *desc;
  t->rank = rank; t->world = world;
  t->lr = desc->learning_rate;
  t->hyper.kind = desc->optimizer;
  t->hyper.rho = desc->rho; t->hyper.eps = desc->epsilon;
  t->hyper.beta1 = desc->beta1; t->hyper.beta2 = desc->beta2; t->hyper.momentum = desc->momentum;
  {
    // parameter count is needed for the size of the gradient buffer that lives behind the parameters in the arena
    long long np = 0; int prev = desc->n_features;
    for (int l = 0; l <= desc->n_hidden; ++l) { const int out = l < desc->n_hidden ? desc->hidden[l] : 1; np += static_cast<long long>(prev) * out + out; prev = out; }
    t->xch_n4 = (np + 3) / 4;
    t->net.arena_extra_bytes = static_cast<size_t>(t->xch_n4) * 16 + sizeof(P2PFlags);
    // LL exchange buffers (xchg_p2p.cuh): gbuf = world regions, sbuf = one, of n4 entries x 32 bytes
    if (world > 1 && desc->precision == SB_PREC_BF16) {
      t->ll_ready = true;
      t->net.arena_extra_bytes += 256 + static_cast<size_t>(world + 1) * static_cast<size_t>(t->xch_n4) * 32;
    }
  }
  int s = t->net.init(desc, device, true);
  if (s != SB_OK) { t->net.destroy(); return s; }
  // see Net::init: no L1 / shared-memory re-partition between the kernels of a step
  cudaFuncSetAttribute(set_batch_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
  cudaFuncSetAttribute(optimizer_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
  cudaFuncSetAttribute(axpy_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
  Net& n = t->net;
  // gradient + exchange flags behind the parameters, in the arena a single IPC handle exports
  t->xch = n.arena;
  t->grad_off = static_cast<long long>(n.extra_off);
  t->flags_off = t->grad_off + t->xch_n4 * 16;
  t->grad = reinterpret_cast<float*>(n.arena + t->grad_off);
  t->flags = reinterpret_cast<P2PFlags*>(n.arena + t->flags_off);
  if (t->ll_ready) {
    t->llg_off = (t->flags_off + static_cast<long long>(sizeof(P2PFlags)) + 255) / 256 * 256;
    t->lls_off = t->llg_off + static_cast<long long>(world) * t->xch_n4 * 32;
    // entries carry the epoch of the exchange that wrote them; epochs start at 1
    if (cudaMemset(n.arena + t->llg_off, 0, static_cast<size_t>(world + 1) * static_cast<size_t>(t->xch_n4) * 32) != cudaSuccess) {
      n.destroy();
      return set_error(SB_ERR_CUDA, "cudaMemset(exchange buffers) failed");
    }
  }
  t->s1 = n.s1; t->s2 = n.s2;
  if ((s = n.dalloc(&t->acc, n.n_params))) { n.destroy(); return s; }
  if (cudaHostAlloc(reinterpret_cast<void**>(&t->h_err), sizeof(unsigned int) * 4, cudaHostAllocMapped) != cudaSuccess ||
      cudaHostGetDevicePointer(reinterpret_cast<void**>(&t->d_herr), t->h_err, 0) != cudaSuccess) {
    n.destroy();
    return set_error(SB_ERR_CUDA, "cudaHostAlloc(exchange error word) failed");
  }
  memset(t->h_err, 0, sizeof(unsigned int) * 4);
  if (const char* e = getenv("SB_XCHG_TIMEOUT_S")) t->xchg_timeout_ns = static_cast<unsigned long long>(atof(e) * 1e9);
  if (const char* e = getenv("SB_XCHG_BLOCKS")) t->xchg_blocks = atoi(e);
  {
    // exchange slots: hidden layer 0 in row chunks of W_0 (128-row multiples; runs are 1024 parameters, so chunk borders fall
    // on run borders when out % 8 == 0), the last chunk also carries b_0; everything else is slot 0
    int chunks = 2;
    if (const char* e = getenv("SB_XCHG_CHUNKS")) chunks = atoi(e);
    if (chunks > SB_XCHG_SLOTS - 2) chunks = SB_XCHG_SLOTS - 2;   // (ev_c[SLOTS - 1] is the touch event)
    const Layer& l0 = n.layers[0];
    if (chunks < 1 || !n.tc() || (l0.out % 8) != 0 || l0.in < 256 * chunks) chunks = 1;
    n.dw0_chunks = chunks;
    const int cr = n.dw0_chunk_rows();
    chunks = (l0.in + cr - 1) / cr;           // (rounding to 128 rows may need fewer chunks)
    n.dw0_chunks = 1;                          // the GEMM is only cut while a step with the peer exchange is enqueued
    t->x_chunks = chunks;
    t->x_slots = 1 + chunks;
    t->x_begin[0] = n.work_end[0]; t->x_end[0] = n.n_work;
    for (int c = 0; c < chunks; ++c) {
      const long long e0 = static_cast<long long>(c) * cr * l0.out, e1 = static_cast<long long>(c + 1) * cr * l0.out;
      t->x_begin[1 + c] = n.work_begin[0] + static_cast<int>(e0 / 1024);
      t->x_end[1 + c] = (c == chunks - 1) ? n.work_end[0] : n.work_begin[0] + static_cast<int>(e1 / 1024);
    }
    for (int i = 0; i < SB_XCHG_SLOTS; ++i) {
      if (cudaEventCreateWithFlags(&t->ev_x[i], cudaEventDisableTiming) != cudaSuccess ||
          cudaEventCreateWithFlags(&t->ev_c[i], cudaEventDisableTiming) != cudaSuccess) {
        n.destroy();
        return set_error(SB_ERR_CUDA, "cudaEventCreate failed");
      }
    }
  }
  if (cudaHostAlloc(reinterpret_cast<void**>(&t->h_scal), sizeof(float) * SCAL_COUNT, cudaHostAllocMapped) != cudaSuccess) {
    n.destroy();
    return set_error(SB_ERR_CUDA, "cudaHostAlloc failed");
  }
  memset(t->h_scal, 0, sizeof(float) * SCAL_COUNT);
  if (cudaHostAlloc(reinterpret_cast<void**>(&t->h_hist), sizeof(float2) * sb_trainer::HIST, cudaHostAllocMapped) != cudaSuccess ||
      cudaHostGetDevicePointer(reinterpret_cast<void**>(&t->d_hist), t->h_hist, 0) != cudaSuccess) {
    n.destroy();
    return set_error(SB_ERR_CUDA, "cudaHostAlloc(loss history) failed");
  }
  memset(t->h_hist, 0, sizeof(float2) * sb_trainer::HIST);
  t->descs[0] = n.desc;
  t->scals[0] = n.scal;
  if ((s = n.dalloc(&t->descs[1], 1)) || (s = n.dalloc(&t->scals[1], SCAL_COUNT))) { n.destroy(); return s; }
  if (cudaStreamCreateWithFlags(&t->prep, cudaStreamNonBlocking) != cudaSuccess) { n.destroy(); return set_error(SB_ERR_CUDA, "cudaStreamCreate failed"); }
  for (int i = 0; i < 2; ++i) {
    if (cudaEventCreateWithFlags(&t->ev_prep[i], cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&t->ev_pos[i], cudaEventDisableTiming) != cudaSuccess) {
      n.destroy();
      return set_error(SB_ERR_CUDA, "cudaEventCreate failed");
    }
  }
  if (cudaHostGetDevicePointer(reinterpret_cast<void**>(&t->d_hscal), t->h_scal, 0) != cudaSuccess) {
    t->net.destroy();
    return set_error(SB_ERR_CUDA, "cudaHostGetDevicePointer failed");
  }
  if (world > 1 && nccl_id != nullptr) {
    NcclApi* api = nccl_api();
    if (!api) { n.destroy(); return set_error(SB_ERR_NCCL, "libnccl.so.2 could not be loaded"); }
    NcclUniqueId id;
    memcpy(&id, nccl_id, sizeof(id));
    int r = api->CommInitRank(&t->comm, world, id, rank);
    if (r != 0) { n.destroy(); return set_error(SB_ERR_NCCL, "ncclCommInitRank failed: %s", api->GetErrorString(r)); }
  }
  SB_CUDA(cudaStreamSynchronize(n.stream));
  *out = t.release();
  return SB_OK;
}

int sb_trainer_ipc_handle(sb_trainer_t* t, void* out64) {
  SB_CHECK(t && out64, SB_ERR_INVALID, "null argument");
  static_assert(sizeof(cudaIpcMemHandle_t) == SB_IPC_HANDLE_BYTES, "IPC handle size");
  SB_CUDA(cudaSetDevice(t->net.device));
  cudaIpcMemHandle_t h;
  SB_CUDA(cudaIpcGetMemHandle(&h, t->xch));
  memcpy(out64, &h, sizeof(h));
  return SB_OK;
}

static void drop_step_graphs(sb_trainer* t) {
  for (auto& kv : t->graphs) cudaGraphExecDestroy(kv.second);   // captured steps carry the exchange they were captured with
  t->graphs.clear();
  for (auto& kv : t->run_graphs) cudaGraphExecDestroy(kv.second);
  t->run_graphs.clear();
}

static void close_peer_mappings(sb_trainer* t) {
  for (void* p : t->peer_bases) cudaIpcCloseMemHandle(p);
  t->peer_bases.clear();
}

// CUDA loads kernels lazily, at their first launch, and that load may synchronise the device: behind an exchange kernel that
// is still spinning for a peer whose work the same host thread has not queued yet (replicas in one process), the load - and
// with it the thread - would never return.  Everything a non-captured path launches around an exchange is loaded up front.
static int preload_exchange_kernels() {
  cudaFuncAttributes a;
  SB_CUDA(cudaFuncGetAttributes(&a, xchg_update_kernel<2>));
  SB_CUDA(cudaFuncGetAttributes(&a, xchg_update_kernel<4>));
  SB_CUDA(cudaFuncGetAttributes(&a, xchg_update_kernel<8>));
  SB_CUDA(cudaFuncGetAttributes(&a, xchg_update_kernel<16>));
  SB_CUDA(cudaFuncGetAttributes(&a, xchg_ll_kernel<2>));
  SB_CUDA(cudaFuncGetAttributes(&a, xchg_ll_kernel<4>));
  SB_CUDA(cudaFuncGetAttributes(&a, xchg_ll_kernel<8>));
  SB_CUDA(cudaFuncGetAttributes(&a, xchg_ll_kernel<16>));
  SB_CUDA(cudaFuncGetAttributes(&a, gather_master_kernel));
  SB_CUDA(cudaFuncGetAttributes(&a, set_batch_kernel));
  SB_CUDA(cudaFuncGetAttributes(&a, scale_kernel));
  SB_CUDA(cudaFuncGetAttributes(&a, zero_f32_kernel));
  SB_CUDA(cudaFuncGetAttributes(&a, axpy_kernel));
  return SB_OK;
}

// peers' exchange allocations -> device table; bases[rank] is ignored (own allocation)
static int install_peer_table(sb_trainer* t, void* const* bases) {
  SB_TRY(preload_exchange_kernels());
  P2PPeers hp;
  memset(&hp, 0, sizeof(hp));
  for (int q = 0; q < t->world; ++q) hp.base[q] = static_cast<char*>((q == t->rank) ? t->xch : bases[q]);
  if (!t->d_peers) SB_CUDA(cudaMalloc(&t->d_peers, sizeof(P2PPeers)));
  SB_CUDA(cudaMemcpy(t->d_peers, &hp, sizeof(hp), cudaMemcpyHostToDevice));
  drop_step_graphs(t);
  t->p2p_ready = true;
  return SB_OK;
}

int sb_trainer_set_peer_handles(sb_trainer_t* t, const void* handles, int32_t n_handles) {
  SB_CHECK(t && handles, SB_ERR_INVALID, "null argument");
  SB_CHECK(n_handles == t->world && t->world <= SB_MAX_RANKS, SB_ERR_INVALID, "expected %d handles (<= %d), got %d", t->world,
           SB_MAX_RANKS, n_handles);
  SB_CUDA(cudaSetDevice(t->net.device));
  SB_CUDA(cudaStreamSynchronize(t->net.stream));
  close_peer_mappings(t);
  t->p2p_ready = false;
  void* bases[SB_MAX_RANKS] = {};
  for (int q = 0; q < t->world; ++q) {
    if (q == t->rank) continue;
    cudaIpcMemHandle_t h;
    memcpy(&h, static_cast<const char*>(handles) + static_cast<size_t>(q) * sizeof(h), sizeof(h));
    cudaError_t e = cudaIpcOpenMemHandle(&bases[q], h, cudaIpcMemLazyEnablePeerAccess);
    if (e != cudaSuccess) {
      cudaGetLastError();
      close_peer_mappings(t);   // all or nothing: a half-mapped table must never be used
      return set_error(SB_ERR_CUDA, "cudaIpcOpenMemHandle(rank %d) failed: %s (no P2P path / separate IPC namespace?)", q,
                       cudaGetErrorString(e));
    }
    t->peer_bases.push_back(bases[q]);
  }
  return install_peer_table(t, bases);
}

int sb_trainer_clear_peer_handles(sb_trainer_t* t) {
  SB_CHECK(t, SB_ERR_INVALID, "null trainer");
  SB_CUDA(cudaSetDevice(t->net.device));
  SB_CUDA(cudaStreamSynchronize(t->net.stream));
  close_peer_mappings(t);
  if (t->p2p_ready) drop_step_graphs(t);
  t->p2p_ready = false;
  return SB_OK;
}

void* sb_trainer_exchange_base(sb_trainer_t* t) { return t ? t->xch : nullptr; }

int sb_trainer_set_peer_pointers(sb_trainer_t* t, void* const* bases, int32_t n) {
  SB_CHECK(t && bases, SB_ERR_INVALID, "null argument");
  SB_CHECK(n == t->world && t->world <= SB_MAX_RANKS, SB_ERR_INVALID, "expected %d pointers (<= %d), got %d", t->world,
           SB_MAX_RANKS, n);
  SB_CUDA(cudaSetDevice(t->net.device));
  SB_CUDA(cudaStreamSynchronize(t->net.stream));
  for (int q = 0; q < t->world; ++q) {
    if (q == t->rank) continue;
    SB_CHECK(bases[q] != nullptr, SB_ERR_INVALID, "pointer of rank %d is null", q);
    cudaPointerAttributes at;
    SB_CUDA(cudaPointerGetAttributes(&at, bases[q]));
    SB_CHECK(at.type == cudaMemoryTypeDevice, SB_ERR_INVALID, "pointer of rank %d is not device memory", q);
    if (at.device == t->net.device) t->peers_share_device = true;
    if (at.device != t->net.device) {
      int can = 0;
      SB_CUDA(cudaDeviceCanAccessPeer(&can, t->net.device, at.device));
      SB_CHECK(can, SB_ERR_CUDA, "device %d cannot access device %d (no P2P path)", t->net.device, at.device);
      cudaError_t e = cudaDeviceEnablePeerAccess(at.device, 0);
      if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) return set_error(SB_ERR_CUDA, "cudaDeviceEnablePeerAccess failed: %s", cudaGetErrorString(e));
      cudaGetLastError();
    }
  }
  close_peer_mappings(t);
  return install_peer_table(t, bases);
}

int sb_trainer_destroy(sb_trainer_t* t) {
  if (!t) return SB_OK;
  cudaSetDevice(t->net.device);
  if (t->net.stream) cudaStreamSynchronize(t->net.stream);
  for (auto& kv : t->graphs) cudaGraphExecDestroy(kv.second);
  for (auto& kv : t->run_graphs) cudaGraphExecDestroy(kv.second);
  for (int i = 0; i < 2; ++i) {
    if (t->ev_run_prep[i]) cudaEventDestroy(t->ev_run_prep[i]);
    if (t->ev_run_done[i]) cudaEventDestroy(t->ev_run_done[i]);
  }
  if (t->comm) { NcclApi* api = nccl_api(); if (api) api->CommDestroy(t->comm); }
  if (t->dsX) cudaFree(t->dsX);
  if (t->dsXb) cudaFree(t->dsXb);
  if (t->dsP) cudaFree(t->dsP);
  if (t->dsI) cudaFree(t->dsI);
  if (t->dsY) cudaFree(t->dsY);
  if (t->dsW) cudaFree(t->dsW);
  if (t->h_scal) cudaFreeHost(t->h_scal);
  if (t->h_err) cudaFreeHost(t->h_err);
  if (t->h_hist) cudaFreeHost(t->h_hist);
  if (t->copy_stream) cudaStreamDestroy(t->copy_stream);
  if (t->prep) { cudaStreamSynchronize(t->prep); cudaStreamDestroy(t->prep); }
  for (int i = 0; i < 2; ++i) {
    if (t->ev_prep[i]) cudaEventDestroy(t->ev_prep[i]);
    if (t->ev_pos[i]) cudaEventDestroy(t->ev_pos[i]);
    if (t->ev_copied[i]) cudaEventDestroy(t->ev_copied[i]);
    if (t->ev_consumed[i]) cudaEventDestroy(t->ev_consumed[i]);
  }
  for (void* p : t->peer_bases) cudaIpcCloseMemHandle(p);
  if (t->d_peers) cudaFree(t->d_peers);
  t->net.destroy();      // frees the arena (= xch)
  delete t;
  return SB_OK;
}

int64_t sb_trainer_param_count(const sb_trainer_t* t) { return t ? t->net.n_params : 0; }

int sb_trainer_set_params(sb_trainer_t* t, const float* flat, int64_t n) {
  SB_CHECK(t && flat, SB_ERR_INVALID, "null argument");
  SB_CHECK(n == t->net.n_params, SB_ERR_INVALID, "expected %lld params, got %lld", (long long)t->net.n_params, (long long)n);
  SB_CUDA(cudaSetDevice(t->net.device));
  SB_CUDA(cudaMemcpyAsync(t->net.theta, flat, sizeof(float) * n, cudaMemcpyHostToDevice, t->net.stream));
  SB_TRY(t->net.refresh_shadows());
  SB_CUDA(cudaStreamSynchronize(t->net.stream));
  return SB_OK;   // (optimizer state is untouched: a sharded trainer keeps each run's state on its owner)
}

int sb_trainer_get_params(sb_trainer_t* t, float* flat, int64_t n) {
  SB_CHECK(t && flat, SB_ERR_INVALID, "null argument");
  SB_CHECK(n == t->net.n_params, SB_ERR_INVALID, "expected %lld params, got %lld", (long long)t->net.n_params, (long long)n);
  SB_CUDA(cudaSetDevice(t->net.device));
  SB_TRY(gather_master(t));
  SB_CUDA(cudaMemcpyAsync(flat, t->net.theta, sizeof(float) * n, cudaMemcpyDeviceToHost, t->net.stream));
  SB_CUDA(cudaStreamSynchronize(t->net.stream));
  return SB_OK;
}

int sb_trainer_init_xavier(sb_trainer_t* t, uint64_t seed) {
  SB_CHECK(t, SB_ERR_INVALID, "null trainer");
  // xavier_initializer() (uniform) on weights and biases, res/ssgd_monitor.py:59-68
  std::vector<float> flat(static_cast<size_t>(t->net.n_params));
  std::mt19937_64 rng(seed);
  for (const Layer& ly : t->net.layers) {
    const double lw = sqrt(6.0 / (ly.in + ly.out)), lb = sqrt(3.0 / ly.out);
    std::uniform_real_distribution<double> uw(-lw, lw), ub(-lb, lb);
    for (long long i = 0; i < static_cast<long long>(ly.in) * ly.out; ++i) flat[ly.w_off + i] = static_cast<float>(uw(rng));
    for (int i = 0; i < ly.out; ++i) flat[ly.b_off + i] = static_cast<float>(ub(rng));
  }
  return sb_trainer_set_params(t, flat.data(), t->net.n_params);
}

int sb_trainer_get_grads(sb_trainer_t* t, float* flat, int64_t n) {
  SB_CHECK(t && flat, SB_ERR_INVALID, "null argument");
  SB_CHECK(n == t->net.n_params, SB_ERR_INVALID, "expected %lld grads, got %lld", (long long)t->net.n_params, (long long)n);
  SB_CUDA(cudaSetDevice(t->net.device));
  if (t->p2p_ready && t->grad_sharded && t->world > 1) {
    // sharded exchange: every owner kept the reduced gradient of its runs; collect them (overwrites this rank's own
    // contributions, which the next step clears anyway)
    SB_CUDA(cudaStreamSynchronize(t->net.stream));
    gather_master_kernel<<<t->net.n_work, 256, 0, t->net.stream>>>(xchg_params(t), 1);
    SB_CUDA(cudaGetLastError());
  }
  SB_CUDA(cudaMemcpyAsync(flat, t->grad, sizeof(float) * n, cudaMemcpyDeviceToHost, t->net.stream));
  SB_CUDA(cudaStreamSynchronize(t->net.stream));
  const float gs = t->grad_out_scale;
  if (gs != 1.f) for (int64_t i = 0; i < n; ++i) flat[i] *= gs;
  return SB_OK;
}

int sb_trainer_step(sb_trainer_t* t, const float* X, const float* y, const float* w, int32_t rows, float* loss_out) {
  SB_CHECK(t, SB_ERR_INVALID, "null trainer");
  SB_TRY(stage_host_batch(t, X, y, w, rows));
  SB_TRY(run_step(t, t->net.stX, t->net.stY, w ? t->net.stW : nullptr, rows, G_STEP));
  return finish_loss(t, loss_out);
}

// ---- wide+deep (BASELINE config 4): hidden layer 0 = [dense | one-hot]; the step feeds (dense block, index matrix) ----
int sb_trainer_set_sparse(sb_trainer_t* t, int32_t n_dense, int32_t n_onehot, int32_t n_cat) {
  SB_CHECK(t, SB_ERR_INVALID, "null trainer");
  const Net& n = t->net;
  SB_CHECK(!t->ds_sparse || (n_dense == n.n_dense && n_onehot == n.n_onehot && n_cat == n.n_cat), SB_ERR_STATE,
           "a wide+deep resident set of another shape is loaded; load a set of the new shape after this call instead");
  return t->net.set_sparse(n_dense, n_onehot, n_cat);
}

static int stage_sparse_batch(Net& n, const float* Xd, const int32_t* idx, const float* y, const float* w, int rows) {
  SB_CHECK(n.n_cat > 0, SB_ERR_STATE, "sb_trainer_set_sparse has not been called");
  SB_CHECK(Xd && idx, SB_ERR_INVALID, "Xd and idx must not be null");
  SB_CHECK(rows > 0 && rows <= n.max_batch, SB_ERR_INVALID, "rows=%d outside (0, max_batch=%d]", rows, n.max_batch);
  for (long long i = 0; i < static_cast<long long>(rows) * n.n_cat; ++i)
    SB_CHECK(idx[i] < n.n_onehot, SB_ERR_INVALID, "idx[%lld] = %d outside [-1, n_onehot=%d)", i, idx[i], n.n_onehot);
  SB_CUDA(cudaSetDevice(n.device));
  SB_CUDA(cudaMemcpyAsync(n.stX, Xd, sizeof(float) * rows * static_cast<size_t>(n.n_dense), cudaMemcpyHostToDevice, n.stream));
  SB_CUDA(cudaMemcpyAsync(n.idx, idx, sizeof(int32_t) * rows * static_cast<size_t>(n.n_cat), cudaMemcpyHostToDevice, n.stream));
  if (y) SB_CUDA(cudaMemcpyAsync(n.stY, y, sizeof(float) * rows, cudaMemcpyHostToDevice, n.stream));
  if (w) SB_CUDA(cudaMemcpyAsync(n.stW, w, sizeof(float) * rows, cudaMemcpyHostToDevice, n.stream));
  return SB_OK;
}

int sb_trainer_step_sparse(sb_trainer_t* t, const float* Xd, const int32_t* idx, const float* y, const float* w, int32_t rows,
                           float* loss_out) {
  SB_CHECK(t && y, SB_ERR_INVALID, "null argument");
  SB_TRY(stage_sparse_batch(t->net, Xd, idx, y, w, rows));
  SB_TRY(run_step(t, t->net.stX, t->net.stY, w ? t->net.stW : nullptr, rows, G_STEP, -1, true, t->net.idx));
  return finish_loss(t, loss_out);
}

// forward (+ loss) over any number of sparse rows in max_batch chunks; out / loss accumulators nullable
static int forward_chunks_sparse(Net& n, const float* Xd, const int32_t* idx, const float* y, const float* w, int64_t rows, float* out,
                                 double* loss_sum, double* nnz) {
  struct Scope { Net& n; ~Scope() { n.sparse_step = false; } } scope{n};
  const bool do_loss = loss_sum != nullptr;
  float h[SCAL_COUNT];
  for (int64_t r0 = 0; r0 < rows; r0 += n.max_batch) {
    const int c = static_cast<int>(rows - r0 < n.max_batch ? rows - r0 : n.max_batch);
    SB_TRY(stage_sparse_batch(n, Xd + r0 * n.n_dense, idx + r0 * n.n_cat, do_loss ? y + r0 : nullptr, (do_loss && w) ? w + r0 : nullptr, c));
    set_batch_kernel<<<1, 1, 0, n.stream>>>(n.desc, n.stX, n.stY, (do_loss && w) ? n.stW : n.ones, 0.f, 1.f, 0, 0, nullptr, 0, nullptr,
                                             nullptr, n.idx);
    n.sparse_step = true;
    SB_TRY(n.enqueue_load(c));
    SB_TRY(n.enqueue_hidden_forward(c));
    n.sparse_step = false;
    SB_TRY(n.enqueue_out(c, do_loss, false, n.yhat, nullptr));
    if (out) SB_CUDA(cudaMemcpyAsync(out + r0, n.yhat, sizeof(float) * c, cudaMemcpyDeviceToHost, n.stream));
    if (do_loss) SB_CUDA(cudaMemcpyAsync(h, n.scal, sizeof(h), cudaMemcpyDeviceToHost, n.stream));
    SB_CUDA(cudaStreamSynchronize(n.stream));
    if (do_loss) { *loss_sum += h[SCAL_LOSS_SUM]; *nnz += h[SCAL_NNZ]; }
  }
  return SB_OK;
}

int sb_trainer_predict_sparse(sb_trainer_t* t, const float* Xd, const int32_t* idx, int64_t rows, float* out) {
  SB_CHECK(t && out, SB_ERR_INVALID, "null argument");
  return forward_chunks_sparse(t->net, Xd, idx, nullptr, nullptr, rows, out, nullptr, nullptr);
}

int sb_trainer_eval_loss_sparse(sb_trainer_t* t, const float* Xd, const int32_t* idx, const float* y, const float* w, int64_t rows,
                                float* loss_out) {
  SB_CHECK(t && y && loss_out && rows > 0, SB_ERR_INVALID, "bad argument");
  double ls = 0, nz = 0;
  SB_TRY(forward_chunks_sparse(t->net, Xd, idx, y, w, rows, nullptr, &ls, &nz));
  *loss_out = nz > 0 ? static_cast<float>(ls / nz) : 0.f;
  return SB_OK;
}

int sb_trainer_step_async(sb_trainer_t* t, const float* X, const float* y, const float* w, int32_t rows) {
  SB_CHECK(t && X && y, SB_ERR_INVALID, "null argument");
  Net& n = t->net;
  SB_CHECK(rows > 0 && rows <= n.max_batch, SB_ERR_INVALID, "rows=%d outside (0, max_batch=%d]", rows, n.max_batch);
  SB_CUDA(cudaSetDevice(n.device));
  if (!t->copy_stream) {
    SB_CUDA(cudaStreamCreateWithFlags(&t->copy_stream, cudaStreamNonBlocking));
    SB_TRY(n.dalloc(&t->st2X, static_cast<size_t>(n.max_batch) * n.F));
    SB_TRY(n.dalloc(&t->st2Y, n.max_batch));
    SB_TRY(n.dalloc(&t->st2W, n.max_batch));
    for (int i = 0; i < 2; ++i) {
      SB_CUDA(cudaEventCreateWithFlags(&t->ev_copied[i], cudaEventDisableTiming));
      SB_CUDA(cudaEventCreateWithFlags(&t->ev_consumed[i], cudaEventDisableTiming));
    }
    SB_CUDA(cudaStreamSynchronize(n.stream));   // the zero-fill of the new staging buffers ran on the main stream
  }
  const int slot = static_cast<int>(t->async_steps & 1);
  float* sx = slot ? t->st2X : n.stX;
  float* sy = slot ? t->st2Y : n.stY;
  float* sw = slot ? t->st2W : n.stW;
  // the slot is free once the step that consumed it two calls ago has finished
  if (t->async_steps >= 2) SB_CUDA(cudaStreamWaitEvent(t->copy_stream, t->ev_consumed[slot], 0));
  SB_CUDA(cudaMemcpyAsync(sx, X, sizeof(float) * rows * static_cast<size_t>(n.F), cudaMemcpyHostToDevice, t->copy_stream));
  SB_CUDA(cudaMemcpyAsync(sy, y, sizeof(float) * rows, cudaMemcpyHostToDevice, t->copy_stream));
  if (w) SB_CUDA(cudaMemcpyAsync(sw, w, sizeof(float) * rows, cudaMemcpyHostToDevice, t->copy_stream));
  SB_CUDA(cudaEventRecord(t->ev_copied[slot], t->copy_stream));
  SB_CUDA(cudaStreamWaitEvent(n.stream, t->ev_copied[slot], 0));
  SB_TRY(run_step(t, sx, sy, w ? sw : nullptr, rows, G_STEP));
  SB_CUDA(cudaEventRecord(t->ev_consumed[slot], n.stream));
  ++t->async_steps;
  return SB_OK;
}

int sb_trainer_accumulate(sb_trainer_t* t, const float* X, const float* y, const float* w, int32_t rows, float* loss_out) {
  SB_CHECK(t, SB_ERR_INVALID, "null trainer");
  SB_TRY(stage_host_batch(t, X, y, w, rows));
  SB_TRY(run_step(t, t->net.stX, t->net.stY, w ? t->net.stW : nullptr, rows, G_ACC));
  return finish_loss(t, loss_out);
}

static int apply_accumulated_impl(sb_trainer_t* t, int64_t total_pushes);

int sb_trainer_apply_accumulated(sb_trainer_t* t) {
  SB_CHECK(t, SB_ERR_INVALID, "null trainer");
  SB_CHECK(t->n_acc > 0, SB_ERR_STATE, "no accumulated gradients");
  return apply_accumulated_impl(t, static_cast<int64_t>(t->world) * t->n_acc);
}

int sb_trainer_apply_accumulated_mean(sb_trainer_t* t, int64_t total_pushes) {
  SB_CHECK(t, SB_ERR_INVALID, "null trainer");
  SB_CHECK(total_pushes > 0, SB_ERR_INVALID, "total_pushes must be > 0");
  return apply_accumulated_impl(t, total_pushes);
}

static int apply_accumulated_impl(sb_trainer_t* t, int64_t total_pushes) {
  Net& n = t->net;
  SB_CUDA(cudaSetDevice(n.device));
  ++t->global_step;
  const float gscale = 1.f / static_cast<float>(total_pushes);
  ++t->epoch;
  set_batch_kernel<<<1, 1, 0, n.stream>>>(n.desc, nullptr, nullptr, nullptr, lr_for_step(t, t->global_step), gscale, t->epoch);
  SB_CUDA(cudaGetLastError());
  // exchange + apply through the (IPC-exported) gradient buffer; it then holds the applied mean for sb_trainer_get_grads
  SB_CUDA(cudaMemcpyAsync(t->grad, t->acc, sizeof(float) * n.n_params, cudaMemcpyDeviceToDevice, n.stream));
  if (t->world > 1 && t->p2p_ready) {
    SB_TRY(enqueue_xchg(t, xseg_all(t), n.stream, false, false));
  } else {
    SB_TRY(enqueue_allreduce(t, t->grad));
    SB_TRY(enqueue_optimizer(t, t->grad));
  }
  const long long np = n.n_params;
  scale_kernel<<<static_cast<unsigned>((np + 255) / 256), 256, 0, n.stream>>>(t->grad, n.desc, np);
  SB_CUDA(cudaGetLastError());
  t->grad_out_scale = 1.f;  // scale_kernel already applied 1/(world * n_acc)
  zero_f32_kernel<<<static_cast<unsigned>((np + 255) / 256), 256, 0, n.stream>>>(t->acc, np);   // (a preloaded kernel, see preload_exchange_kernels)
  SB_CUDA(cudaGetLastError());
  // queued, not waited for (like a step): with a peer exchange inside, a host thread that drives several replicas must be able
  // to queue the update on all of them before any can complete; everything that reads the result synchronises the stream
  t->n_acc = 0;
  return SB_OK;
}

// The resident set: X [n_rows, cols] fp32, cols = F, or (wide+deep, idx != nullptr) the dense block of n_dense columns beside
// the index matrix idx [n_rows, n_cat].  Any of the pointers may be HOST or DEVICE memory.
static int load_resident_set(sb_trainer* t, const float* X, const int32_t* idx, const float* y, const float* w, int64_t n_rows) {
  SB_CHECK(t && X && y, SB_ERR_INVALID, "null argument");
  SB_CHECK(n_rows > 0 && n_rows < (1ll << 31), SB_ERR_INVALID, "n_rows must be in (0, 2^31)");
  Net& n = t->net;
  const bool sparse = idx != nullptr;
  const int cols = sparse ? n.n_dense : n.F, ld = sparse ? n.ldD : n.ldF;
  SB_CUDA(cudaSetDevice(n.device));
  SB_CUDA(cudaStreamSynchronize(n.stream));
  int* dsI = nullptr;
  if (sparse) {
    // copied and range-checked on the device (host and device input alike) before the old set is dropped, so a rejected
    // set leaves the trainer as it was; steps then do no per-index host work
    const long long ni = n_rows * static_cast<long long>(n.n_cat);
    SB_CUDA(cudaMalloc(&dsI, sizeof(int) * ni));
    int* range = nullptr;
    int h[2] = {0x7fffffff, -0x7fffffff - 1};
    cudaError_t e = cudaMalloc(&range, sizeof(h));
    if (e == cudaSuccess) e = cudaMemcpyAsync(dsI, idx, sizeof(int) * ni, cudaMemcpyDefault, n.stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(range, h, sizeof(h), cudaMemcpyHostToDevice, n.stream);
    if (e == cudaSuccess) {
      const long long blocks = std::min<long long>((ni + 255) / 256, static_cast<long long>(n.num_sms) * 8);
      int_range_kernel<<<static_cast<unsigned>(blocks), 256, 0, n.stream>>>(dsI, ni, range);
      e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaMemcpyAsync(h, range, sizeof(h), cudaMemcpyDeviceToHost, n.stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(n.stream);
    if (range) cudaFree(range);
    if (e != cudaSuccess || h[0] < -1 || h[1] >= n.n_onehot) {
      cudaFree(dsI);
      SB_CHECK(e == cudaSuccess, SB_ERR_CUDA, "index matrix copy / range check failed: %s", cudaGetErrorString(e));
      return set_error(SB_ERR_INVALID, "idx holds values in [%d, %d], outside [-1, n_onehot=%d)", h[0], h[1], n.n_onehot);
    }
  }
  drop_step_graphs(t);   // captured steps carry tensor maps of the old set
  if (t->dsX) cudaFree(t->dsX);
  if (t->dsXb) cudaFree(t->dsXb);
  if (t->dsY) cudaFree(t->dsY);
  if (t->dsW) cudaFree(t->dsW);
  if (t->dsP) cudaFree(t->dsP);
  if (t->dsI) cudaFree(t->dsI);
  t->dsX = t->dsY = t->dsW = nullptr; t->dsXb = nullptr; t->dsP = nullptr; t->ds_rows = 0;
  t->dsI = dsI;
  t->ds_sparse = sparse;
  SB_CUDA(cudaMalloc(&t->dsY, sizeof(float) * n_rows));
  SB_CUDA(cudaMalloc(&t->dsW, sizeof(float) * n_rows));
  SB_CUDA(cudaMemcpyAsync(t->dsY, y, sizeof(float) * n_rows, cudaMemcpyDefault, n.stream));
  if (w) {
    SB_CUDA(cudaMemcpyAsync(t->dsW, w, sizeof(float) * n_rows, cudaMemcpyDefault, n.stream));
  } else {
    fill_kernel<<<static_cast<unsigned>((n_rows + 255) / 256), 256, 0, n.stream>>>(t->dsW, 1.f, n_rows);
    SB_CUDA(cudaGetLastError());
  }
  if (n.tc()) {
    // keep the set in HBM in the form the layer-0 GEMMs consume (bf16, row pitch ld; split modes: nparts such arrays):
    // converted once here, read by TMA every step.  Converted through a bounded fp32 window so a 100+ GB set never needs
    // a second full copy.
    const size_t part_elems = static_cast<size_t>(n_rows) * ld;
    SB_CUDA(cudaMalloc(&t->dsXb, sizeof(__nv_bfloat16) * part_elems * n.nparts));
    SB_CUDA(cudaMemsetAsync(t->dsXb, 0, sizeof(__nv_bfloat16) * part_elems * n.nparts, n.stream));
    n.resident_ps = static_cast<long long>(part_elems);
    const int64_t win = 32768;
    float* tmp = nullptr;
    SB_CUDA(cudaMalloc(&tmp, sizeof(float) * static_cast<size_t>(win < n_rows ? win : n_rows) * cols));
    for (int64_t r0 = 0; r0 < n_rows; r0 += win) {
      const int64_t c = n_rows - r0 < win ? n_rows - r0 : win;
      SB_CUDA(cudaMemcpyAsync(tmp, X + r0 * cols, sizeof(float) * c * cols, cudaMemcpyDefault, n.stream));
      cast_bf16_kernel<<<static_cast<unsigned>((c * cols + 255) / 256), 256, 0, n.stream>>>(tmp, static_cast<int>(c), cols,
                                                                                            t->dsXb + r0 * ld, ld, n.nparts,
                                                                                            n.resident_ps);
      SB_CUDA(cudaGetLastError());
      SB_CUDA(cudaStreamSynchronize(n.stream));   // X may be pageable: the window is reused
    }
    cudaFree(tmp);
    std::vector<int> prefix(static_cast<size_t>(n_rows) + 1);
    prefix[0] = 0;
    std::vector<float> w_host;
    const float* wh = w;
    if (is_device_ptr(w)) {      // 4 bytes per row: the only part of a device-resident set the host looks at
      w_host.resize(static_cast<size_t>(n_rows));
      SB_CUDA(cudaMemcpy(w_host.data(), w, sizeof(float) * n_rows, cudaMemcpyDeviceToHost));
      wh = w_host.data();
    }
    for (int64_t i = 0; i < n_rows; ++i) prefix[i + 1] = prefix[i] + ((wh == nullptr || wh[i] != 0.f) ? 1 : 0);
    SB_CUDA(cudaMalloc(&t->dsP, sizeof(int) * (n_rows + 1)));
    SB_CUDA(cudaMemcpyAsync(t->dsP, prefix.data(), sizeof(int) * (n_rows + 1), cudaMemcpyHostToDevice, n.stream));
    SB_CUDA(cudaStreamSynchronize(n.stream));
    n.resident_Xb = t->dsXb;
    n.resident_rows = n_rows;
  } else {
    SB_CUDA(cudaMalloc(&t->dsX, sizeof(float) * n_rows * cols));
    SB_CUDA(cudaMemcpyAsync(t->dsX, X, sizeof(float) * n_rows * cols, cudaMemcpyDefault, n.stream));
  }
  SB_CUDA(cudaStreamSynchronize(n.stream));
  t->ds_rows = n_rows;
  return SB_OK;
}

int sb_trainer_load_dataset(sb_trainer_t* t, const float* X, const float* y, const float* w, int64_t n_rows) {
  return load_resident_set(t, X, nullptr, y, w, n_rows);
}

int sb_trainer_load_dataset_sparse(sb_trainer_t* t, const float* Xd, const int32_t* idx, const float* y, const float* w,
                                   int64_t n_rows) {
  SB_CHECK(t, SB_ERR_INVALID, "null trainer");
  SB_CHECK(t->net.n_cat > 0, SB_ERR_STATE, "sb_trainer_set_sparse has not been called");
  SB_CHECK(idx, SB_ERR_INVALID, "idx must not be null");
  return load_resident_set(t, Xd, idx, y, w, n_rows);
}

// fp32 rows / index rows of the resident set from `row` on (nullptr where the set has none)
static const float* ds_x(const sb_trainer* t, long long row) {
  return t->dsX ? t->dsX + row * (t->ds_sparse ? t->net.n_dense : t->net.F) : nullptr;
}
static const int* ds_idx(const sb_trainer* t, long long row) { return t->dsI ? t->dsI + row * t->net.n_cat : nullptr; }

static int resident_step(sb_trainer_t* t, int64_t row_offset, int32_t rows, int kind) {
  SB_CHECK(t, SB_ERR_INVALID, "null trainer");
  SB_CHECK(t->ds_rows > 0, SB_ERR_STATE, "no resident dataset loaded");
  SB_CHECK(row_offset >= 0 && rows > 0 && row_offset + rows <= t->ds_rows, SB_ERR_INVALID,
           "rows [%lld, %lld) outside the resident set of %lld rows", (long long)row_offset, (long long)(row_offset + rows),
           (long long)t->ds_rows);
  return run_step(t, ds_x(t, row_offset), t->dsY + row_offset, t->dsW + row_offset, rows, kind, row_offset, t->ds_sparse,
                  ds_idx(t, row_offset));
}

// RUN_S consecutive steps as ONE graph over descriptor set `set`
static int get_run_graph(sb_trainer* t, int rows, int set, cudaGraphExec_t* out) {
  const int key = rows * 2 + set;
  auto it = t->run_graphs.find(key);
  if (it != t->run_graphs.end()) { *out = it->second; return SB_OK; }
  Net& n = t->net;
  BatchDesc* d0 = n.desc; float* s0 = n.scal;
  cudaGraph_t g = nullptr;
  SB_CUDA(cudaStreamBeginCapture(n.stream, cudaStreamCaptureModeThreadLocal));
  int s = SB_OK;
  for (int k = 0; k < sb_trainer::RUN_S && s == SB_OK; ++k) {
    n.desc = t->run_descs[set][k];
    n.scal = t->run_scals[set][k];
    // (SB_STEP_TRACE: the trace holds one step; an interior one is traced, with steps of the same graph on both sides of
    // it like most steps of a run)
    n.trace_on = (k == 1);
    s = enqueue_step_body(t, rows, G_STEP, true, t->ds_sparse);
  }
  n.trace_on = true;
  n.desc = d0; n.scal = s0;
  cudaError_t e = cudaStreamEndCapture(n.stream, &g);
  if (s != SB_OK) { if (g) cudaGraphDestroy(g); return s; }
  SB_CHECK(e == cudaSuccess, SB_ERR_CUDA, "cudaStreamEndCapture failed: %s", cudaGetErrorString(e));
  cudaGraphExec_t ge = nullptr;
  SB_CUDA(cudaGraphInstantiate(&ge, g, 0));
  cudaGraphDestroy(g);
  t->run_graphs[key] = ge;
  *out = ge;
  return SB_OK;
}

int sb_trainer_run_resident(sb_trainer_t* t, const int64_t* row_offsets, int32_t n_steps, int32_t rows) {
  SB_CHECK(t && row_offsets, SB_ERR_INVALID, "null argument");
  SB_CHECK(n_steps >= 0, SB_ERR_INVALID, "n_steps must be >= 0");
  SB_CHECK(t->ds_rows > 0, SB_ERR_STATE, "no resident dataset loaded");
  Net& n = t->net;
  SB_CHECK(rows > 0 && rows <= n.max_batch, SB_ERR_INVALID, "rows=%d outside (0, max_batch=%d]", rows, n.max_batch);
  for (int i = 0; i < n_steps; ++i)
    SB_CHECK(row_offsets[i] >= 0 && row_offsets[i] + rows <= t->ds_rows, SB_ERR_INVALID,
             "step %d: rows [%lld, %lld) outside the resident set of %lld rows", i, (long long)row_offsets[i],
             (long long)(row_offsets[i] + rows), (long long)t->ds_rows);
  constexpr int S = sb_trainer::RUN_S;
  static const bool no_graph = getenv("SB_NO_GRAPH") != nullptr;
  static const bool no_multi = getenv("SB_NO_MULTI_STEP") != nullptr;
  int i = 0;
  if (t->dsXb != nullptr && !no_graph && !no_multi) {
    SB_CUDA(cudaSetDevice(n.device));
    if (t->run_descs[0][0] == nullptr) {
      for (int set = 0; set < 2; ++set) {
        for (int k = 0; k < S; ++k) {
          SB_TRY(n.dalloc(&t->run_descs[set][k], 1));
          SB_TRY(n.dalloc(&t->run_scals[set][k], SCAL_COUNT));
        }
        SB_CUDA(cudaEventCreateWithFlags(&t->ev_run_prep[set], cudaEventDisableTiming));
        SB_CUDA(cudaEventCreateWithFlags(&t->ev_run_done[set], cudaEventDisableTiming));
      }
      SB_CUDA(cudaStreamSynchronize(n.stream));   // the zero-fill of the new descriptors ran on the main stream
    }
    const float gscale = 1.f / static_cast<float>(t->world);
    for (; i + S <= n_steps; i += S) {
      const int set = static_cast<int>(t->run_chunks & 1);
      cudaGraphExec_t ge = nullptr;
      SB_TRY(get_run_graph(t, rows, set, &ge));
      // this set was last read by the chunk two launches back
      if (t->run_used[set]) SB_CUDA(cudaStreamWaitEvent(t->prep, t->ev_run_done[set], 0));
      for (int k = 0; k < S; ++k) {
        const long long off = row_offsets[i + k];
        ++t->global_step;
        ++t->epoch;
        set_batch_kernel<<<1, 1, 0, t->prep>>>(t->run_descs[set][k], nullptr, t->dsY + off, t->dsW + off,
                                               lr_for_step(t, t->global_step), gscale, t->epoch, static_cast<int>(off), t->dsP,
                                               rows, t->run_scals[set][k], t->hist_slot(t->global_step), ds_idx(t, off));
      }
      SB_CUDA(cudaGetLastError());
      SB_CUDA(cudaEventRecord(t->ev_run_prep[set], t->prep));
      SB_CUDA(cudaStreamWaitEvent(n.stream, t->ev_run_prep[set], 0));
      SB_CUDA(cudaGraphLaunch(ge, n.stream));
      SB_CUDA(cudaEventRecord(t->ev_run_done[set], n.stream));
      t->run_used[set] = true;
      ++t->run_chunks;
      t->have_pos = false;          // the single-step descriptor prefetch re-joins the main stream
      t->grad_out_scale = gscale;
    }
  }
  for (; i < n_steps; ++i) SB_TRY(resident_step(t, row_offsets[i], rows, G_STEP));
  return SB_OK;
}

int sb_trainer_step_resident(sb_trainer_t* t, int64_t row_offset, int32_t rows, float* loss_out) {
  SB_TRY(resident_step(t, row_offset, rows, G_STEP));
  return finish_loss(t, loss_out);
}
int sb_trainer_step_resident_async(sb_trainer_t* t, int64_t row_offset, int32_t rows) {
  return resident_step(t, row_offset, rows, G_STEP);
}
int sb_trainer_accumulate_resident(sb_trainer_t* t, int64_t row_offset, int32_t rows, float* loss_out) {
  SB_TRY(resident_step(t, row_offset, rows, G_ACC));
  return finish_loss(t, loss_out);
}
int sb_trainer_loss_resident(sb_trainer_t* t, int64_t row_offset, int32_t rows, float* loss_out) {
  SB_CHECK(t && loss_out, SB_ERR_INVALID, "null argument");
  SB_CHECK(t->ds_rows > 0, SB_ERR_STATE, "no resident dataset loaded");
  Net& n = t->net;
  SB_CHECK(row_offset >= 0 && rows > 0 && rows <= n.max_batch && row_offset + rows <= t->ds_rows, SB_ERR_INVALID,
           "rows [%lld, %lld) outside the resident set of %lld rows", (long long)row_offset, (long long)(row_offset + rows),
           (long long)t->ds_rows);
  SB_CUDA(cudaSetDevice(n.device));
  n.desc = t->descs[0];
  n.scal = t->scals[0];
  t->have_pos = false;
  const bool resident = t->dsXb != nullptr;
  if (resident)
    set_batch_kernel<<<1, 1, 0, n.stream>>>(n.desc, nullptr, t->dsY + row_offset, t->dsW + row_offset, 0.f, 1.f, t->epoch,
                                             static_cast<int>(row_offset), t->dsP, rows, n.scal, nullptr, ds_idx(t, row_offset));
  else
    set_batch_kernel<<<1, 1, 0, n.stream>>>(n.desc, ds_x(t, row_offset), t->dsY + row_offset, t->dsW + row_offset, 0.f, 1.f,
                                             t->epoch, 0, nullptr, 0, nullptr, nullptr, ds_idx(t, row_offset));
  SB_CUDA(cudaGetLastError());
  struct Scope { Net& n; ~Scope() { n.from_resident = false; n.sparse_step = false; } } scope{n};
  n.from_resident = resident;
  n.sparse_step = t->ds_sparse;
  if (!resident) SB_TRY(n.enqueue_load(rows));
  SB_TRY(n.enqueue_hidden_forward(rows));
  SB_TRY(n.enqueue_out(rows, true, false, nullptr, nullptr));
  float h[SCAL_COUNT];
  SB_CUDA(cudaMemcpyAsync(h, n.scal, sizeof(h), cudaMemcpyDeviceToHost, n.stream));
  SB_CUDA(cudaStreamSynchronize(n.stream));
  *loss_out = h[SCAL_NNZ] > 0.f ? h[SCAL_LOSS_SUM] / h[SCAL_NNZ] : 0.f;
  return SB_OK;
}

int sb_trainer_broadcast_state(sb_trainer_t* t, int32_t root) {
  SB_CHECK(t, SB_ERR_INVALID, "null trainer");
  if (t->world <= 1) return SB_OK;
  SB_CHECK(root >= 0 && root < t->world, SB_ERR_INVALID, "root %d outside [0, %d)", root, t->world);
  NcclApi* api = nccl_api();
  SB_CHECK(api && t->comm, SB_ERR_NCCL, "no NCCL communicator");
  Net& n = t->net;
  SB_CUDA(cudaSetDevice(n.device));
  long long* d_step = nullptr;
  SB_CUDA(cudaMalloc(&d_step, sizeof(long long)));
  SB_CUDA(cudaMemcpyAsync(d_step, &t->global_step, sizeof(long long), cudaMemcpyHostToDevice, n.stream));
  int r = api->Broadcast(n.theta, n.theta, static_cast<size_t>(n.n_params), NCCL_FLOAT32, root, t->comm, n.stream);
  if (r == 0) r = api->Broadcast(t->s1, t->s1, static_cast<size_t>(n.n_params), NCCL_FLOAT32, root, t->comm, n.stream);
  if (r == 0) r = api->Broadcast(t->s2, t->s2, static_cast<size_t>(n.n_params), NCCL_FLOAT32, root, t->comm, n.stream);
  if (r == 0) r = api->Broadcast(d_step, d_step, 1, NCCL_INT64, root, t->comm, n.stream);
  if (r != 0) { cudaFree(d_step); return set_error(SB_ERR_NCCL, "ncclBroadcast failed: %s", api->GetErrorString(r)); }
  long long step = 0;
  SB_CUDA(cudaMemcpyAsync(&step, d_step, sizeof(long long), cudaMemcpyDeviceToHost, n.stream));
  SB_TRY(n.refresh_shadows());
  SB_CUDA(cudaStreamSynchronize(n.stream));
  cudaFree(d_step);
  t->global_step = step;
  return poll_nccl(t);
}

int sb_trainer_loss_history(sb_trainer_t* t, int64_t first_step, int32_t n, float* out) {
  SB_CHECK(t && out, SB_ERR_INVALID, "null argument");
  SB_CHECK(n >= 0 && first_step >= 1 && first_step + n - 1 <= t->global_step, SB_ERR_INVALID,
           "steps [%lld, %lld] outside [1, global_step=%lld]", (long long)first_step, (long long)(first_step + n - 1), (long long)t->global_step);
  SB_CHECK(t->global_step - first_step < sb_trainer::HIST, SB_ERR_INVALID, "only the last %d steps are kept", (int)sb_trainer::HIST);
  SB_CUDA(cudaSetDevice(t->net.device));
  SB_CUDA(cudaStreamSynchronize(t->net.stream));
  SB_TRY(poll_nccl(t));
  for (int i = 0; i < n; ++i) {
    const float2 v = t->h_hist[(first_step + i) % sb_trainer::HIST];
    out[i] = v.y > 0.f ? v.x / v.y : 0.f;
  }
  return SB_OK;
}

int sb_trainer_last_loss(sb_trainer_t* t, float* loss_out) {
  SB_CHECK(t && loss_out, SB_ERR_INVALID, "null argument");
  return finish_loss(t, loss_out);
}
int sb_trainer_sync(sb_trainer_t* t) {
  SB_CHECK(t, SB_ERR_INVALID, "null trainer");
  SB_CUDA(cudaStreamSynchronize(t->net.stream));
  SB_TRY(poll_nccl(t));
  SB_TRY(poll_xchg(t));
  return SB_OK;
}
void* sb_trainer_stream(sb_trainer_t* t) { return t ? reinterpret_cast<void*>(t->net.stream) : nullptr; }

int sb_trainer_kernels_per_step(sb_trainer_t* t, int32_t rows) {
  SB_CHECK(t, SB_ERR_INVALID, "null trainer");
  cudaGraphExec_t ge;
  Net& n = t->net;
  BatchDesc* d0 = n.desc; float* s0 = n.scal;
  n.desc = t->descs[0]; n.scal = t->scals[0];      // the graph bakes the pair's pointers
  const int s = get_graph(t, rows, G_STEP, t->dsXb != nullptr, 0, &ge, t->ds_sparse);
  n.desc = d0; n.scal = s0;
  SB_TRY(s);
  return t->kernels_per_step[rows];
}

// One un-captured step over resident rows with a CUDA event after every launch.
// ms[i] = device time between the end of launch i-1 (or the start marker) and the end of launch i.
int sb_trainer_profile_step(sb_trainer_t* t, int64_t row_offset, int32_t rows, char* names, int32_t names_cap, float* ms,
                            int32_t cap, int32_t* n_out) {
  SB_CHECK(t && ms && n_out, SB_ERR_INVALID, "null argument");
  SB_CHECK(t->ds_rows > 0, SB_ERR_STATE, "no resident dataset loaded");
  SB_CHECK(row_offset >= 0 && rows > 0 && rows <= t->net.max_batch && row_offset + rows <= t->ds_rows, SB_ERR_INVALID, "bad row range");
  Net& n = t->net;
  SB_CUDA(cudaSetDevice(n.device));
  ++t->global_step;
  const float gscale = 1.f / static_cast<float>(t->world);
  ++t->epoch;
  const bool resident = t->dsXb != nullptr;
  if (resident)
    set_batch_kernel<<<1, 1, 0, n.stream>>>(n.desc, nullptr, t->dsY + row_offset, t->dsW + row_offset, lr_for_step(t, t->global_step),
                                             gscale, t->epoch, static_cast<int>(row_offset), t->dsP, rows, n.scal, nullptr,
                                             ds_idx(t, row_offset));
  else
    set_batch_kernel<<<1, 1, 0, n.stream>>>(n.desc, ds_x(t, row_offset), t->dsY + row_offset, t->dsW + row_offset,
                                             lr_for_step(t, t->global_step), gscale, t->epoch, 0, nullptr, 0, nullptr, nullptr,
                                             ds_idx(t, row_offset));
  n.profiling = true;
  n.prof_events.clear(); n.prof_names.clear();
  n.launches = 0;
  // the two memsets of the step body run before the start marker so they are not charged to load_batch
  int s = SB_OK;
  {
    n.from_resident = resident;
    n.sparse_step = t->ds_sparse;
    if (resident) s = (cudaMemsetAsync(t->grad, 0, sizeof(float) * n.n_params, n.stream) == cudaSuccess) ? SB_OK : SB_ERR_CUDA;
    n.mark("start"); --n.launches;
    if (!resident) s = n.enqueue_load(rows, t->grad, n.n_params);
    bool fused_out = false;
    if (s == SB_OK) s = n.enqueue_hidden_forward(rows, t->grad, &fused_out);
    if (s == SB_OK && !fused_out) s = n.enqueue_out(rows, true, true, nullptr, t->grad);
    if (s == SB_OK) s = n.enqueue_backward(rows, t->grad);
    if (t->world > 1 && t->p2p_ready) {
      if (s == SB_OK) s = enqueue_xchg(t, xseg_all(t), n.stream, false, false);
    } else {
      if (s == SB_OK) s = enqueue_allreduce(t, t->grad);
      if (s == SB_OK && t->world > 1) { n.mark("allreduce"); --n.launches; }
      if (s == SB_OK) s = enqueue_optimizer(t, t->grad);
    }
  }
  n.profiling = false;
  n.from_resident = false;
  n.sparse_step = false;
  cudaError_t e = cudaStreamSynchronize(n.stream);
  int cnt = 0;
  std::string joined;
  if (s == SB_OK && e == cudaSuccess) {
    for (size_t i = 1; i < n.prof_events.size(); ++i) {
      float v = 0.f;
      cudaEventElapsedTime(&v, n.prof_events[i - 1], n.prof_events[i]);
      if (cnt < cap) ms[cnt] = v;
      if (!joined.empty()) joined += "\n";
      joined += n.prof_names[i];
      ++cnt;
    }
  }
  for (cudaEvent_t ev : n.prof_events) cudaEventDestroy(ev);
  n.prof_events.clear(); n.prof_names.clear();
  SB_TRY(s);
  SB_CHECK(e == cudaSuccess, SB_ERR_CUDA, "profile step failed: %s", cudaGetErrorString(e));
  t->grad_out_scale = gscale;
  *n_out = cnt;
  if (names && names_cap > 0) { strncpy(names, joined.c_str(), names_cap - 1); names[names_cap - 1] = 0; }
  return SB_OK;
}

// forward (+ optional loss) over any number of host rows, in max_batch chunks
static int forward_chunks(Net& n, const float* X, const float* y, const float* w, int64_t rows, bool do_loss,
                          float* out, double* loss_sum, double* nnz) {
  SB_CUDA(cudaSetDevice(n.device));
  float h[SCAL_COUNT];
  for (int64_t r0 = 0; r0 < rows; r0 += n.max_batch) {
    const int c = static_cast<int>(rows - r0 < n.max_batch ? rows - r0 : n.max_batch);
    SB_CUDA(cudaMemcpyAsync(n.stX, X + r0 * n.F, sizeof(float) * c * static_cast<size_t>(n.F), cudaMemcpyDefault, n.stream));
    if (do_loss) {
      SB_CUDA(cudaMemcpyAsync(n.stY, y + r0, sizeof(float) * c, cudaMemcpyDefault, n.stream));
      if (w) SB_CUDA(cudaMemcpyAsync(n.stW, w + r0, sizeof(float) * c, cudaMemcpyDefault, n.stream));
    }
    set_batch_kernel<<<1, 1, 0, n.stream>>>(n.desc, n.stX, n.stY, (do_loss && w) ? n.stW : n.ones, 0.f, 1.f);
    SB_TRY(n.enqueue_load(c));
    SB_TRY(n.enqueue_hidden_forward(c));
    SB_TRY(n.enqueue_out(c, do_loss, false, n.yhat, nullptr));
    if (out) SB_CUDA(cudaMemcpyAsync(out + r0, n.yhat, sizeof(float) * c, cudaMemcpyDefault, n.stream));
    if (do_loss) SB_CUDA(cudaMemcpyAsync(h, n.scal, sizeof(h), cudaMemcpyDeviceToHost, n.stream));
    SB_CUDA(cudaStreamSynchronize(n.stream));
    if (do_loss) { *loss_sum += h[SCAL_LOSS_SUM]; *nnz += h[SCAL_NNZ]; }
  }
  return SB_OK;
}

int sb_trainer_eval_loss(sb_trainer_t* t, const float* X, const float* y, const float* w, int64_t rows, float* loss_out) {
  SB_CHECK(t && X && y && loss_out, SB_ERR_INVALID, "null argument");
  SB_CHECK(rows > 0, SB_ERR_INVALID, "rows must be > 0");
  double ls = 0, nz = 0;
  SB_TRY(forward_chunks(t->net, X, y, w, rows, true, nullptr, &ls, &nz));
  *loss_out = nz > 0 ? static_cast<float>(ls / nz) : 0.f;
  return SB_OK;
}

int sb_trainer_predict(sb_trainer_t* t, const float* X, int64_t rows, float* out) {
  SB_CHECK(t && X && out, SB_ERR_INVALID, "null argument");
  SB_CHECK(rows > 0, SB_ERR_INVALID, "rows must be > 0");
  double ls = 0, nz = 0;
  return forward_chunks(t->net, X, nullptr, nullptr, rows, false, out, &ls, &nz);
}

// ---- checkpoint: flat blob {magic, version, n_params, global_step, optimizer, theta, s1, s2} ----
static const uint64_t CKPT_MAGIC = 0x5348494655423230ull;  // "SHIFUB20"

int sb_trainer_save_checkpoint(sb_trainer_t* t, const char* path) {
  SB_CHECK(t && path, SB_ERR_INVALID, "null argument");
  Net& n = t->net;
  SB_CUDA(cudaSetDevice(n.device));
  SB_TRY(gather_master(t));
  std::vector<float> buf(static_cast<size_t>(n.n_params) * 3);
  SB_CUDA(cudaMemcpyAsync(buf.data(), n.theta, sizeof(float) * n.n_params, cudaMemcpyDeviceToHost, n.stream));
  SB_CUDA(cudaMemcpyAsync(buf.data() + n.n_params, t->s1, sizeof(float) * n.n_params, cudaMemcpyDeviceToHost, n.stream));
  SB_CUDA(cudaMemcpyAsync(buf.data() + 2 * n.n_params, t->s2, sizeof(float) * n.n_params, cudaMemcpyDeviceToHost, n.stream));
  SB_CUDA(cudaStreamSynchronize(n.stream));
  std::string tmp = std::string(path) + ".tmp";
  FILE* f = fopen(tmp.c_str(), "wb");
  SB_CHECK(f, SB_ERR_IO, "cannot open %s for writing", tmp.c_str());
  uint64_t hdr[5] = {CKPT_MAGIC, 1, static_cast<uint64_t>(n.n_params), static_cast<uint64_t>(t->global_step),
                     static_cast<uint64_t>(t->hyper.kind)};
  bool ok = fwrite(hdr, sizeof(hdr), 1, f) == 1 && fwrite(buf.data(), sizeof(float), buf.size(), f) == buf.size();
  ok = (fclose(f) == 0) && ok;
  SB_CHECK(ok, SB_ERR_IO, "short write to %s", tmp.c_str());
  SB_CHECK(rename(tmp.c_str(), path) == 0, SB_ERR_IO, "rename to %s failed", path);
  return SB_OK;
}

int sb_trainer_load_checkpoint(sb_trainer_t* t, const char* path) {
  SB_CHECK(t && path, SB_ERR_INVALID, "null argument");
  Net& n = t->net;
  FILE* f = fopen(path, "rb");
  SB_CHECK(f, SB_ERR_IO, "cannot open %s", path);
  uint64_t hdr[5];
  std::vector<float> buf(static_cast<size_t>(n.n_params) * 3);
  bool ok = fread(hdr, sizeof(hdr), 1, f) == 1;
  ok = ok && hdr[0] == CKPT_MAGIC && hdr[2] == static_cast<uint64_t>(n.n_params);
  ok = ok && fread(buf.data(), sizeof(float), buf.size(), f) == buf.size();
  fclose(f);
  SB_CHECK(ok, SB_ERR_FORMAT, "%s is not a checkpoint of this network", path);
  SB_CHECK(hdr[4] == static_cast<uint64_t>(t->hyper.kind), SB_ERR_FORMAT,
           "%s was written by optimizer %d, this trainer uses optimizer %d: the saved optimizer state does not apply", path,
           static_cast<int>(hdr[4]), t->hyper.kind);
  SB_CUDA(cudaSetDevice(n.device));
  SB_CUDA(cudaMemcpyAsync(n.theta, buf.data(), sizeof(float) * n.n_params, cudaMemcpyHostToDevice, n.stream));
  SB_CUDA(cudaMemcpyAsync(t->s1, buf.data() + n.n_params, sizeof(float) * n.n_params, cudaMemcpyHostToDevice, n.stream));
  SB_CUDA(cudaMemcpyAsync(t->s2, buf.data() + 2 * n.n_params, sizeof(float) * n.n_params, cudaMemcpyHostToDevice, n.stream));
  SB_TRY(n.refresh_shadows());
  SB_CUDA(cudaStreamSynchronize(n.stream));
  t->global_step = static_cast<long long>(hdr[3]);
  return SB_OK;
}

int64_t sb_trainer_global_step(const sb_trainer_t* t) { return t ? t->global_step : 0; }

int sb_trainer_export_savedmodel(sb_trainer_t* t, const char* export_dir) {
  SB_CHECK(t && export_dir, SB_ERR_INVALID, "null argument");
  std::vector<float> flat(static_cast<size_t>(t->net.n_params));
  SB_TRY(sb_trainer_get_params(t, flat.data(), t->net.n_params));
  return sb_savedmodel_write(export_dir, &t->desc, flat.data(), t->net.n_params);
}

// ================================================================================================
// scorer
// ================================================================================================
}  // extern "C"

struct sb_model {
  Net net;
  sb_net_desc desc;
  std::mutex mu;
};

static const int MODEL_CHUNK_ROWS = 16384;        // fp32 parity mode
static const int MODEL_CHUNK_ROWS_BF16 = 65536;   // bf16: bigger GEMMs per launch (workspace ~0.8 GB at 2000 cols)

static int model_from_desc(sb_net_desc d, const float* flat, int64_t n, int device, sb_model_t** out) {
  d.max_batch = d.precision == SB_PREC_FP32 ? MODEL_CHUNK_ROWS : (d.precision == SB_PREC_BF16 ? MODEL_CHUNK_ROWS_BF16 : MODEL_CHUNK_ROWS_BF16 / 2);
  std::unique_ptr<sb_model> m(new sb_model());
  m->desc = d;
  int s = m->net.init(&d, device, false);
  if (s != SB_OK) { m->net.destroy(); return s; }
  if (n != m->net.n_params) {
    m->net.destroy();
    return set_error(SB_ERR_INVALID, "expected %lld params, got %lld", (long long)m->net.n_params, (long long)n);
  }
  Net& net = m->net;
  SB_CUDA(cudaMemcpyAsync(net.theta, flat, sizeof(float) * n, cudaMemcpyHostToDevice, net.stream));
  SB_TRY(net.refresh_shadows());
  SB_CUDA(cudaStreamSynchronize(net.stream));
  *out = m.release();
  return SB_OK;
}

extern "C" {

int sb_model_create(const sb_net_desc* desc, const float* flat_params, int64_t n, int device, sb_model_t** out) {
  SB_CHECK(out && flat_params, SB_ERR_INVALID, "null argument");
  *out = nullptr;
  sb_net_desc d = *desc;
  if (d.max_batch <= 0) d.max_batch = 1;
  SB_TRY(validate_desc(&d));
  return model_from_desc(d, flat_params, n, device, out);
}

int sb_model_load(const char* saved_model_dir, const char* input_name, const char* output_name, const char* tag,
                  int device, int precision, sb_model_t** out) {
  SB_CHECK(out, SB_ERR_INVALID, "out is null");
  *out = nullptr;
  // the null checks mirror TensorflowModel.init (TensorflowModel.java:147-166)
  SB_CHECK(saved_model_dir && saved_model_dir[0], SB_ERR_INVALID, "Model path is null");
  SB_CHECK(input_name && input_name[0], SB_ERR_INVALID, "Input names is null");
  SB_CHECK(output_name && output_name[0], SB_ERR_INVALID, "Output names is null");
  SB_CHECK(tag && tag[0], SB_ERR_INVALID, "Tags is null");
  sb_net_desc d;
  memset(&d, 0, sizeof(d));
  int32_t out_act = SB_ACT_SIGMOID;
  int64_t np = 0;
  SB_TRY(sb_savedmodel_read(saved_model_dir, input_name, output_name, tag, &d, &out_act, nullptr, 0, &np));
  SB_CHECK(out_act == SB_ACT_SIGMOID, SB_ERR_FORMAT, "output layer must be a sigmoid unit");
  std::vector<float> flat(static_cast<size_t>(np));
  SB_TRY(sb_savedmodel_read(saved_model_dir, input_name, output_name, tag, &d, &out_act, flat.data(), np, &np));
  d.precision = precision;
  d.max_batch = 1;
  return model_from_desc(d, flat.data(), np, device, out);
}

int sb_model_destroy(sb_model_t* m) {
  if (!m) return SB_OK;
  cudaSetDevice(m->net.device);
  m->net.destroy();
  delete m;
  return SB_OK;
}

int32_t sb_model_n_features(const sb_model_t* m) { return m ? m->net.F : 0; }
int32_t sb_model_n_layers(const sb_model_t* m) { return m ? m->net.L + 1 : 0; }

int sb_model_score(sb_model_t* m, const float* X, int64_t rows, float* out) {
  SB_CHECK(m, SB_ERR_STATE, "TF model not initialized.");
  SB_CHECK(X && out, SB_ERR_INVALID, "null argument");
  if (rows <= 0) return SB_OK;
  std::lock_guard<std::mutex> lk(m->mu);
  double a = 0, b = 0;
  return forward_chunks(m->net, X, nullptr, nullptr, rows, false, out, &a, &b);
}

int sb_model_score_row_f64(sb_model_t* m, const double* row, int32_t n, double* out) {
  SB_CHECK(m, SB_ERR_STATE, "TF model not initialized.");
  SB_CHECK(row && out, SB_ERR_INVALID, "null argument");
  SB_CHECK(n == m->net.F, SB_ERR_INVALID, "expected %d features, got %d", m->net.F, n);
  std::vector<float> f(static_cast<size_t>(n));
  for (int i = 0; i < n; ++i) f[i] = static_cast<float>(row[i]);  // TensorflowModel.java:64-68
  float r = 0.f;
  SB_TRY(sb_model_score(m, f.data(), 1, &r));
  *out = static_cast<double>(r);
  return SB_OK;
}

int sb_model_score_device(sb_model_t* m, const float* dX, int64_t rows, float* dOut) {
  SB_CHECK(m, SB_ERR_STATE, "TF model not initialized.");
  SB_CHECK(dX && dOut, SB_ERR_INVALID, "null argument");
  std::lock_guard<std::mutex> lk(m->mu);
  Net& n = m->net;
  SB_CUDA(cudaSetDevice(n.device));
  for (int64_t r0 = 0; r0 < rows; r0 += n.max_batch) {
    const int c = static_cast<int>(rows - r0 < n.max_batch ? rows - r0 : n.max_batch);
    set_batch_kernel<<<1, 1, 0, n.stream>>>(n.desc, dX + r0 * n.F, nullptr, n.ones, 0.f, 1.f);
    SB_TRY(n.enqueue_load(c));
    SB_TRY(n.enqueue_hidden_forward(c));
    SB_TRY(n.enqueue_out(c, false, false, dOut + r0, nullptr));
  }
  return SB_OK;
}

int sb_model_sync(sb_model_t* m) {
  SB_CHECK(m, SB_ERR_STATE, "TF model not initialized.");
  SB_CUDA(cudaStreamSynchronize(m->net.stream));
  return SB_OK;
}
void* sb_model_stream(sb_model_t* m) { return m ? reinterpret_cast<void*>(m->net.stream) : nullptr; }

// ================================================================================================
// kernel-level test hook
// ================================================================================================
static int debug_gemm_impl(const float* A, const float* B, float* D, int32_t M, int32_t N, int32_t K, int32_t split_k,
                           int32_t a_mn, int32_t b_mn, int32_t cfg_cg, int32_t cfg_bn, int device, int iters, float* ms_out);

int sb_debug_step_trace(sb_trainer_t* t, uint64_t* stamps, int32_t cap_kernels, char* names, int32_t names_cap, int32_t* n_kernels) {
  SB_CHECK(t && stamps && n_kernels, SB_ERR_INVALID, "null argument");
  Net& n = t->net;
  SB_CHECK(n.step_trace != nullptr, SB_ERR_STATE, "create the trainer with SB_STEP_TRACE=1 in the environment");
  SB_CUDA(cudaSetDevice(n.device));
  SB_CUDA(cudaStreamSynchronize(n.stream));
  const int k = n.trace_n < cap_kernels ? n.trace_n : cap_kernels;
  SB_CUDA(cudaMemcpy(stamps, n.step_trace, sizeof(uint64_t) * 16 * k, cudaMemcpyDeviceToHost));
  *n_kernels = k;
  if (names && names_cap > 0) {
    std::string all;
    for (int i = 0; i < k; ++i) { if (i) all += ','; all += n.trace_names[i]; }
    snprintf(names, names_cap, "%s", all.c_str());
  }
  return SB_OK;
}

int sb_debug_gemm_bf16_cfg(const float* A, const float* B, float* D, int32_t M, int32_t N, int32_t K, int32_t split_k,
                           int32_t a_mn, int32_t b_mn, int32_t cfg_cg, int32_t cfg_bn, int device) {
  return debug_gemm_impl(A, B, D, M, N, K, split_k, a_mn, b_mn, cfg_cg, cfg_bn, device, 0, nullptr);
}
int sb_debug_gemm_bench(const float* A, const float* B, float* D, int32_t M, int32_t N, int32_t K, int32_t split_k,
                        int32_t a_mn, int32_t b_mn, int32_t cfg_cg, int32_t cfg_bn, int device, int32_t iters, float* ms_out) {
  SB_CHECK(iters > 0 && ms_out, SB_ERR_INVALID, "iters / ms_out");
  return debug_gemm_impl(A, B, D, M, N, K, split_k, a_mn, b_mn, cfg_cg, cfg_bn, device, iters, ms_out);
}
}  // extern "C"

static int debug_gemm_impl(const float* A, const float* B, float* D, int32_t M, int32_t N, int32_t K, int32_t split_k,
                           int32_t a_mn, int32_t b_mn, int32_t cfg_cg, int32_t cfg_bn, int device, int iters, float* ms_out) {
  SB_CHECK(cfg_cg == 0 || ((cfg_cg == 1 && (cfg_bn == 64 || cfg_bn == 128)) || (cfg_cg == 2 && (cfg_bn == 128 || cfg_bn == 256))),
           SB_ERR_INVALID, "tile configuration cg=%d bn=%d not instantiated", cfg_cg, cfg_bn);
  SB_CHECK(A && B && D && M > 0 && N > 0 && K > 0, SB_ERR_INVALID, "bad argument");
  SB_CHECK((a_mn == 0 && b_mn == 0) || (a_mn == 0 && b_mn == 1) || (a_mn == 1 && b_mn == 1), SB_ERR_INVALID,
           "layout combination not instantiated (use KK, KM or MM)");
  int n_dev = 0;
  SB_CHECK(cudaGetDeviceCount(&n_dev) == cudaSuccess && n_dev > 0, SB_ERR_CUDA, "no CUDA device available");
  cudaDeviceProp prop;
  SB_CUDA(cudaGetDeviceProperties(&prop, device));
  SB_CHECK(prop.major == 10, SB_ERR_CUDA, "device is sm_%d%d, need sm_100", prop.major, prop.minor);
  SB_CUDA(cudaSetDevice(device));
  // stored shapes: K-major [R, K]; MN-major [K, R]
  const int a_rows = a_mn ? K : M, a_cols = a_mn ? M : K;
  const int b_rows = b_mn ? K : N, b_cols = b_mn ? N : K;
  const int lda = round_up(a_cols, 8), ldb = round_up(b_cols, 8);
  float *dA32 = nullptr, *dB32 = nullptr, *dD = nullptr;
  __nv_bfloat16 *dA = nullptr, *dB = nullptr;
  SB_CUDA(cudaMalloc(&dA32, sizeof(float) * M * K));
  SB_CUDA(cudaMalloc(&dB32, sizeof(float) * N * K));
  SB_CUDA(cudaMalloc(&dD, sizeof(float) * M * N));
  SB_CUDA(cudaMalloc(&dA, sizeof(__nv_bfloat16) * a_rows * lda));
  SB_CUDA(cudaMalloc(&dB, sizeof(__nv_bfloat16) * b_rows * ldb));
  SB_CUDA(cudaMemset(dA, 0, sizeof(__nv_bfloat16) * a_rows * lda));
  SB_CUDA(cudaMemset(dB, 0, sizeof(__nv_bfloat16) * b_rows * ldb));
  SB_CUDA(cudaMemset(dD, 0, sizeof(float) * M * N));
  SB_CUDA(cudaMemcpy(dA32, A, sizeof(float) * M * K, cudaMemcpyHostToDevice));
  SB_CUDA(cudaMemcpy(dB32, B, sizeof(float) * N * K, cudaMemcpyHostToDevice));
  cast_bf16_kernel<<<static_cast<unsigned>((static_cast<long long>(M) * K + 255) / 256), 256>>>(dA32, a_rows, a_cols, dA, lda);
  cast_bf16_kernel<<<static_cast<unsigned>((static_cast<long long>(N) * K + 255) / 256), 256>>>(dB32, b_rows, b_cols, dB, ldb);
  GemmPlan pl = plan_gemm(M, N, K, prop.multiProcessorCount, false);
  if (cfg_cg > 0) {  // explicit tile configuration requested by the test
    pl.cg = cfg_cg; pl.bn = cfg_bn;
    const int tiles = ((M + 128 * pl.cg - 1) / (128 * pl.cg)) * ((N + pl.bn - 1) / pl.bn);
    pl.split_k = 1; pl.kb_per_split = (K + 63) / 64;
    const int slots = prop.multiProcessorCount / pl.cg;
    pl.grid = (tiles < slots ? tiles : slots) * pl.cg;
  }
  {
    const int total_kb = (K + 63) / 64;
    int want = split_k < 1 ? 1 : (split_k > total_kb ? total_kb : split_k);
    pl.kb_per_split = (total_kb + want - 1) / want;
    pl.split_k = (total_kb + pl.kb_per_split - 1) / pl.kb_per_split;
    const int tiles = ((M + 128 * pl.cg - 1) / (128 * pl.cg)) * ((N + pl.bn - 1) / pl.bn);
    const int slots = prop.multiProcessorCount / pl.cg;
    const int work = tiles * pl.split_k;
    pl.grid = (work < slots ? work : slots) * pl.cg;
  }
  TmapSet tms;
  int s = make_tmap_bf16(&tms.a[0], dA, a_rows, a_cols, lda, a_mn ? 64 : 128);
  if (s == SB_OK) s = make_tmap_bf16(&tms.b[0], dB, b_rows, b_cols, ldb, b_mn ? 64 : plan_box_rows_b(pl));
  if (s == SB_OK) {
    GemmTcParams p = {};
    p.M = M; p.N = N; p.K = K;
    p.accum = dD; p.ld_acc = N;
    auto launch = [&]() -> int {
      if (!a_mn && !b_mn) return launch_gemm_tc<EPI_F32, false, false>(pl, tms, p, 0);
      if (!a_mn) return launch_gemm_tc<EPI_F32, false, true>(pl, tms, p, 0);
      return launch_gemm_tc<EPI_F32, true, true>(pl, tms, p, 0);
    };
    if (!a_mn && !b_mn) s = set_gemm_tc_attrs<EPI_F32, false, false>();
    else if (!a_mn) s = set_gemm_tc_attrs<EPI_F32, false, true>();
    else s = set_gemm_tc_attrs<EPI_F32, true, true>();
    if (s == SB_OK) s = launch();
    if (s == SB_OK && iters > 0) {
      // benchmark with the REAL epilogue of the layout's use: KM -> forward (bias + relu -> bf16), KK -> dA
      // (act' * , bf16 store, column sums), MM -> dW (fp32 red.add)
      const int ldn = round_up(N, 8);
      float *d_bias = nullptr, *d_colsum = nullptr;
      __nv_bfloat16 *d_out = nullptr, *d_aux = nullptr;
      cudaMalloc(&d_bias, sizeof(float) * N); cudaMemset(d_bias, 0, sizeof(float) * N);
      cudaMalloc(&d_colsum, sizeof(float) * N); cudaMemset(d_colsum, 0, sizeof(float) * N);
      cudaMalloc(&d_out, sizeof(__nv_bfloat16) * static_cast<size_t>(M) * ldn);
      cudaMalloc(&d_aux, sizeof(__nv_bfloat16) * static_cast<size_t>(M) * ldn);
      cudaMemset(d_aux, 0x3f, sizeof(__nv_bfloat16) * static_cast<size_t>(M) * ldn);
      GemmTcParams q = p;
      q.bias = d_bias; q.act = SB_ACT_RELU; q.out = d_out; q.ld_out = ldn; q.aux = d_aux; q.ld_aux = ldn; q.colsum = d_colsum;
      q.acc_vec4 = (N % 4 == 0) ? 1 : 0;
      if (s == SB_OK) s = make_tmap_bf16(&tms.o, d_out, M, N, ldn, 128);
      if (s == SB_OK) s = make_tmap_bf16(&tms.x, d_aux, M, N, ldn, 128);
      const bool bench_pdl = getenv("SB_BENCH_PDL") != nullptr;
      auto real = [&]() -> int {
        if (!a_mn && !b_mn) return launch_gemm_tc<EPI_DA, false, false>(pl, tms, q, 0, bench_pdl);
        if (!a_mn) return launch_gemm_tc<EPI_FWD, false, true>(pl, tms, q, 0, bench_pdl);
        return launch_gemm_tc<EPI_DW, true, true>(pl, tms, q, 0, bench_pdl);
      };
      if (!a_mn && !b_mn) s = set_gemm_tc_attrs<EPI_DA, false, false>();
      else if (!a_mn) s = set_gemm_tc_attrs<EPI_FWD, false, true>();
      else s = set_gemm_tc_attrs<EPI_DW, true, true>();
      cudaEvent_t e0, e1;
      cudaEventCreate(&e0); cudaEventCreate(&e1);
      for (int i = 0; i < 3 && s == SB_OK; ++i) s = real();
      cudaEventRecord(e0, 0);
      for (int i = 0; i < iters && s == SB_OK; ++i) s = real();
      cudaEventRecord(e1, 0);
      cudaEventSynchronize(e1);
      float ms = 0.f;
      cudaEventElapsedTime(&ms, e0, e1);
      *ms_out = ms / iters;
      cudaEventDestroy(e0); cudaEventDestroy(e1);
      if (getenv("SB_GEMM_TRACE")) {
        // one more launch with %globaltimer stamps from CTA 0 (ns relative to kernel entry), and the host-visible
        // launch-to-completion time of a single isolated launch
        unsigned long long* d_tr = nullptr;
        cudaMalloc(&d_tr, 16 * sizeof(unsigned long long));
        cudaMemset(d_tr, 0, 16 * sizeof(unsigned long long));
        q.trace = d_tr;
        cudaDeviceSynchronize();
        cudaEvent_t t0, t1;
        cudaEventCreate(&t0); cudaEventCreate(&t1);
        cudaEventRecord(t0, 0);
        s = real();
        cudaEventRecord(t1, 0);
        cudaEventSynchronize(t1);
        float one = 0.f;
        cudaEventElapsedTime(&one, t0, t1);
        unsigned long long h[16];
        cudaMemcpy(h, d_tr, sizeof(h), cudaMemcpyDeviceToHost);
        fprintf(stderr, "[trace] M=%d N=%d K=%d cg=%d bn=%d split=%d single-launch %.2f us | ns since entry:", M, N, K, pl.cg, pl.bn,
                pl.split_k, one * 1e3f);
        const char* nm[9] = {"entry", "setup", "deps", "tma0", "land0", "mma_done", "acc_ready", "epi_done", "exit"};
        for (int i = 1; i < 9; ++i) fprintf(stderr, " %s=%lld", nm[i], (long long)(h[i] - h[0]));
        fprintf(stderr, "\n");
        cudaEventDestroy(t0); cudaEventDestroy(t1);
        cudaFree(d_tr);
        q.trace = nullptr;
      }
      cudaFree(d_bias); cudaFree(d_colsum); cudaFree(d_out); cudaFree(d_aux);
    }
  }
  if (s == SB_OK) {
    cudaError_t e = cudaDeviceSynchronize();
    if (e != cudaSuccess) s = set_error(SB_ERR_CUDA, "gemm_tc_kernel failed: %s", cudaGetErrorString(e));
    else if (cudaMemcpy(D, dD, sizeof(float) * M * N, cudaMemcpyDeviceToHost) != cudaSuccess) s = set_error(SB_ERR_CUDA, "D2H failed");
  }
  cudaFree(dA32); cudaFree(dB32); cudaFree(dD); cudaFree(dA); cudaFree(dB);
  return s;
}

extern "C" {

// D[M,N] = A[M,K] B[N,K]^T with every fp32 operand value split into `np` bf16 parts (np = 1: plain bf16)
int sb_debug_gemm_split(const float* A, const float* B, float* D, int32_t M, int32_t N, int32_t K, int32_t np, int device) {
  SB_CHECK(A && B && D && M > 0 && N > 0 && K > 0 && np >= 1 && np <= 3, SB_ERR_INVALID, "bad argument");
  int n_dev = 0;
  SB_CHECK(cudaGetDeviceCount(&n_dev) == cudaSuccess && n_dev > 0, SB_ERR_CUDA, "no CUDA device available");
  cudaDeviceProp prop;
  SB_CUDA(cudaGetDeviceProperties(&prop, device));
  SB_CHECK(prop.major == 10, SB_ERR_CUDA, "device is sm_%d%d, need sm_100", prop.major, prop.minor);
  SB_CUDA(cudaSetDevice(device));
  const int ld = round_up(K, 8);
  const long long a_ps = static_cast<long long>(M) * ld, b_ps = static_cast<long long>(N) * ld;
  float *dA32 = nullptr, *dB32 = nullptr, *dD = nullptr;
  __nv_bfloat16 *dA = nullptr, *dB = nullptr;
  SB_CUDA(cudaMalloc(&dA32, sizeof(float) * M * K));
  SB_CUDA(cudaMalloc(&dB32, sizeof(float) * N * K));
  SB_CUDA(cudaMalloc(&dD, sizeof(float) * M * N));
  SB_CUDA(cudaMalloc(&dA, sizeof(__nv_bfloat16) * a_ps * np));
  SB_CUDA(cudaMalloc(&dB, sizeof(__nv_bfloat16) * b_ps * np));
  SB_CUDA(cudaMemset(dA, 0, sizeof(__nv_bfloat16) * a_ps * np));
  SB_CUDA(cudaMemset(dB, 0, sizeof(__nv_bfloat16) * b_ps * np));
  SB_CUDA(cudaMemset(dD, 0, sizeof(float) * M * N));
  SB_CUDA(cudaMemcpy(dA32, A, sizeof(float) * M * K, cudaMemcpyHostToDevice));
  SB_CUDA(cudaMemcpy(dB32, B, sizeof(float) * N * K, cudaMemcpyHostToDevice));
  cast_bf16_kernel<<<static_cast<unsigned>((static_cast<long long>(M) * K + 255) / 256), 256>>>(dA32, M, K, dA, ld, np, a_ps);
  cast_bf16_kernel<<<static_cast<unsigned>((static_cast<long long>(N) * K + 255) / 256), 256>>>(dB32, N, K, dB, ld, np, b_ps);
  GemmTcParams p = {};
  set_part_pairs(&p, np);
  p.M = M; p.N = N; p.K = K;
  p.accum = dD; p.ld_acc = N;
  const GemmPlan pl = plan_gemm(M, N, round_up(K, 64) * p.n_pairs, prop.multiProcessorCount, false);
  TmapSet tms;
  int s = make_tmaps_bf16(tms.a, dA, a_ps, np, M, K, ld, 128);
  if (s == SB_OK) s = make_tmaps_bf16(tms.b, dB, b_ps, np, N, K, ld, plan_box_rows_b(pl));
  if (s == SB_OK) s = set_gemm_tc_attrs<EPI_F32, false, false>();
  if (s == SB_OK) s = launch_gemm_tc<EPI_F32, false, false>(pl, tms, p, 0);
  if (s == SB_OK) {
    cudaError_t e = cudaDeviceSynchronize();
    if (e != cudaSuccess) s = set_error(SB_ERR_CUDA, "gemm_tc_kernel (split) failed: %s", cudaGetErrorString(e));
    else if (cudaMemcpy(D, dD, sizeof(float) * M * N, cudaMemcpyDeviceToHost) != cudaSuccess) s = set_error(SB_ERR_CUDA, "D2H failed");
  }
  cudaFree(dA32); cudaFree(dB32); cudaFree(dD); cudaFree(dA); cudaFree(dB);
  return s;
}

int sb_debug_gemm_bf16_ex(const float* A, const float* B, float* D, int32_t M, int32_t N, int32_t K, int32_t split_k,
                          int32_t a_mn, int32_t b_mn, int device) {
  return sb_debug_gemm_bf16_cfg(A, B, D, M, N, K, split_k, a_mn, b_mn, 0, 0, device);
}
int sb_debug_gemm_bf16(const float* A, const float* B, float* D, int32_t M, int32_t N, int32_t K, int32_t split_k, int device) {
  return sb_debug_gemm_bf16_cfg(A, B, D, M, N, K, split_k, 0, 0, 0, 0, device);
}

}  // extern "C"
