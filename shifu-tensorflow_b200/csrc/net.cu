// Net: device state + kernel sequencing for the tabular-DNN forward / backward.
// Mirrors generate_from_modelconf + model (res/ssgd_monitor.py:91-144) as a list of fused launches.
#include <stdarg.h>
#include <stdlib.h>
#include <string.h>
#include <algorithm>
#include "net.cuh"
#include "gemm_tc_launch.cuh"

namespace sb {

std::string& last_error_ref() {
  thread_local std::string e;
  return e;
}
int set_error(int code, const char* fmt, ...) {
  char buf[1024];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  last_error_ref() = buf;
  return code;
}

PFN_encodeTiled get_encode_tiled() {
  static PFN_encodeTiled fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<PFN_encodeTiled>(p);
  }
  return fn;
}

int make_tmaps_bf16(CUtensorMap* out3, const void* base, long long part_stride, int np, int rows, int cols, int ld, int box_rows) {
  for (int k = 0; k < (np > 1 ? np : 1); ++k)
    SB_TRY(make_tmap_bf16(out3 + k, static_cast<const __nv_bfloat16*>(base) + k * part_stride, rows, cols, ld, box_rows));
  return SB_OK;
}

void set_part_pairs(GemmTcParams* p, int np) {
  p->np = np > 1 ? np : 1;
  int n = 0;
  // smallest products first: they are added to a still small accumulator
  for (int sum = p->np - 1; sum >= 0; --sum)
    for (int i = 0; i <= sum; ++i) { p->pair_a[n] = static_cast<unsigned char>(i); p->pair_b[n] = static_cast<unsigned char>(sum - i); ++n; }
  p->n_pairs = n;
}

int make_tmap_bf16(CUtensorMap* out, const void* base, int rows, int cols, int ld, int box_rows) {
  PFN_encodeTiled enc = get_encode_tiled();
  SB_CHECK(enc != nullptr, SB_ERR_CUDA, "cuTensorMapEncodeTiled not available from the driver");
  SB_CHECK(rows > 0 && cols > 0 && (ld % 8) == 0 && (reinterpret_cast<uintptr_t>(base) & 15) == 0, SB_ERR_INVALID,
           "tensor map: bad geometry rows=%d cols=%d ld=%d", rows, cols, ld);
  cuuint64_t gdim[2] = {static_cast<cuuint64_t>(cols), static_cast<cuuint64_t>(rows)};
  cuuint64_t gstr[1] = {static_cast<cuuint64_t>(ld) * 2};
  cuuint32_t box[2] = {64u, static_cast<cuuint32_t>(box_rows)};
  cuuint32_t estr[2] = {1u, 1u};
  CUresult r = enc(out, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), gdim, gstr, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  SB_CHECK(r == CUDA_SUCCESS, SB_ERR_CUDA, "cuTensorMapEncodeTiled failed (%d) rows=%d cols=%d ld=%d box_rows=%d",
           static_cast<int>(r), rows, cols, ld, box_rows);
  return SB_OK;
}

// Tile configuration, rules fitted to the on-device sweep in profiles/gemm_sweep_r01.txt (scripts/gemm_sweep.py):
//   - the single-CTA 128x128 tile is L2->SM bandwidth bound (~46 B/cycle/SM with every SM pulling, i.e. ~45 % of the
//     tensor peak); the CTA-pair 256x256 tile (cta_group::2) halves the bytes per flop and reaches ~64 %;
//   - the pair tile only pays when there are enough pair tiles to fill the 74 SM pairs AND the K loop is deep
//     enough (>= 8 k-blocks per tile) to amortise its larger fill / epilogue;
//   - split-K (dW GEMMs, reduction over the batch): fill the machine but keep >= 8 k-blocks per split.
GemmPlan plan_gemm(int M, int N, int K, int num_sms, bool allow_split) {
  const int total_kb = (K + 63) / 64;
  GemmPlan pl = {};
  auto finish = [&](int cg, int bn, int want_split) {
    const int slots = num_sms / cg;
    const int tiles = ((M + 128 * cg - 1) / (128 * cg)) * ((N + bn - 1) / bn);
    if (want_split < 1) want_split = 1;
    if (want_split > total_kb) want_split = total_kb;
    pl.cg = cg; pl.bn = bn;
    pl.kb_per_split = (total_kb + want_split - 1) / want_split;
    pl.split_k = (total_kb + pl.kb_per_split - 1) / pl.kb_per_split;
    const int work = tiles * pl.split_k;
    pl.grid = (work < slots ? work : slots) * cg;
  };
  const int pairs = num_sms / 2;
  const int pair_tiles = ((M + 255) / 256) * ((N + 255) / 256);
  if (N >= 512 && M >= 512) {
    if (!allow_split) {
      if (pair_tiles * 5 >= pairs * 4 && total_kb >= 8) { finish(2, 256, 1); return pl; }
    } else {
      int split = pairs / pair_tiles;
      if (split < 1) split = 1;
      if (pair_tiles * split * 5 >= pairs * 4 && total_kb / split >= 32) { finish(2, 256, split); return pl; }
    }
  }
  const int bn = N <= 64 ? 64 : 128;
  const int tiles = ((M + 127) / 128) * ((N + bn - 1) / bn);
  int split = 1;
  if (allow_split) {
    split = num_sms / tiles;
    const int cap = total_kb / 8;
    if (split > cap) split = cap;
    if (split < 1) split = 1;
  }
  finish(1, bn, split);
  return pl;
}

static inline int pairs_of(int np) { return np == 3 ? 6 : (np == 2 ? 3 : 1); }

int validate_desc(const sb_net_desc* d) {
  SB_CHECK(d != nullptr, SB_ERR_INVALID, "net desc is null");
  SB_CHECK(d->n_features > 0, SB_ERR_INVALID, "n_features must be > 0 (got %d)", d->n_features);
  SB_CHECK(d->n_hidden >= 1 && d->n_hidden <= SB_MAX_HIDDEN, SB_ERR_INVALID, "n_hidden must be in [1,%d] (got %d)",
           SB_MAX_HIDDEN, d->n_hidden);
  for (int l = 0; l < d->n_hidden; ++l) {
    SB_CHECK(d->hidden[l] > 0, SB_ERR_INVALID, "hidden[%d] must be > 0", l);
    SB_CHECK(d->acts[l] >= SB_ACT_NONE && d->acts[l] <= SB_ACT_LEAKYRELU, SB_ERR_INVALID, "acts[%d] invalid", l);
  }
  SB_CHECK(d->max_batch > 0, SB_ERR_INVALID, "max_batch must be > 0");
  SB_CHECK(d->precision >= SB_PREC_FP32 && d->precision <= SB_PREC_BF16X2, SB_ERR_INVALID, "precision invalid");
  SB_CHECK(d->loss == SB_LOSS_MSE || d->loss == SB_LOSS_SIGMOID_CE, SB_ERR_INVALID, "loss invalid");
  SB_CHECK(d->optimizer >= SB_OPT_ADADELTA && d->optimizer <= SB_OPT_MOMENTUM, SB_ERR_INVALID, "optimizer invalid");
  return SB_OK;
}

static int check_device(int device, int* num_sms) {
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  SB_CHECK(e == cudaSuccess && n > 0, SB_ERR_CUDA, "no CUDA device available (%s); this library has no CPU fallback",
           cudaGetErrorString(e));
  SB_CHECK(device >= 0 && device < n, SB_ERR_INVALID, "device %d out of range [0,%d)", device, n);
  cudaDeviceProp prop;
  SB_CUDA(cudaGetDeviceProperties(&prop, device));
  SB_CHECK(prop.major == 10, SB_ERR_CUDA, "device %d is sm_%d%d; this library is built for sm_100a only", device,
           prop.major, prop.minor);
  *num_sms = prop.multiProcessorCount;
  return SB_OK;
}

int Net::init(const sb_net_desc* d, int device_, bool training_) {
  SB_TRY(validate_desc(d));
  SB_TRY(check_device(device_, &num_sms));
  device = device_;
  training = training_;
  const bool want_trace = getenv("SB_STEP_TRACE") != nullptr;
  SB_CUDA(cudaSetDevice(device));
  // the main chain is the critical path: its CTAs are scheduled ahead of the side stream's (dW GEMMs, second optimizer)
  int prio_least = 0, prio_greatest = 0;
  SB_CUDA(cudaDeviceGetStreamPriorityRange(&prio_least, &prio_greatest));
  SB_CUDA(cudaStreamCreateWithPriority(&stream, cudaStreamNonBlocking, prio_greatest));
  if (training_) {
    SB_CUDA(cudaStreamCreateWithPriority(&side, cudaStreamNonBlocking, prio_least));
    ev_dz.resize(d->n_hidden);
    for (auto& e : ev_dz) SB_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    SB_CUDA(cudaEventCreateWithFlags(&ev_join, cudaEventDisableTiming));
    SB_CUDA(cudaEventCreateWithFlags(&ev_da_done, cudaEventDisableTiming));
    SB_CUDA(cudaStreamCreateWithFlags(&comm, cudaStreamNonBlocking));
    SB_CUDA(cudaStreamCreateWithFlags(&comm2, cudaStreamNonBlocking));
  }
  F = d->n_features;
  L = d->n_hidden;
  precision = d->precision;
  nparts = precision == SB_PREC_FP32_TC ? 3 : (precision == SB_PREC_BF16X2 ? 2 : 1);
  loss = d->loss;
  max_batch = d->max_batch;
  ldB = round_up(max_batch, 8);
  ldF = round_up(F, 8);
  layers.resize(L + 1);
  long long off = 0;
  int prev = F;
  for (int l = 0; l <= L; ++l) {
    Layer& ly = layers[l];
    ly.in = prev;
    ly.out = (l < L) ? d->hidden[l] : 1;
    ly.act = (l < L) ? d->acts[l] : SB_ACT_SIGMOID;
    ly.w_off = off; off += static_cast<long long>(ly.in) * ly.out;
    ly.b_off = off; off += ly.out;
    ly.ld_in = round_up(ly.in, 8);
    ly.ld_out = round_up(ly.out, 8);
    prev = ly.out;
  }
  n_params = off;
  const bool bf = tc();
  {
    auto align256 = [](size_t b) { return (b + 255) & ~static_cast<size_t>(255); };
    const size_t vec_bytes = align256(static_cast<size_t>(n_params) * sizeof(float) + 64);
    size_t at = vec_bytes;                       // theta at 0
    if (training) { s1_off = at; at += vec_bytes; s2_off = at; at += vec_bytes; }
    shadow_off = at;
    std::vector<size_t> wn_off(L, 0);
    Wn_ps.assign(L, 0);
    if (bf)
      for (int l = 0; l < L; ++l) {
        const size_t part = align256(static_cast<size_t>(layers[l].in) * layers[l].ld_out * sizeof(__nv_bfloat16));
        wn_off[l] = at; at += part * nparts;
        Wn_ps[l] = static_cast<long long>(part / sizeof(__nv_bfloat16));
      }
    extra_off = at;
    at += align256(arena_extra_bytes);
    arena_bytes = at;
    void* q = nullptr;
    SB_CUDA(cudaMalloc(&q, arena_bytes));
    allocs.push_back(q);
    SB_CUDA(cudaMemsetAsync(q, 0, arena_bytes, stream));
    arena = static_cast<char*>(q);
    theta = reinterpret_cast<float*>(arena);
    if (training) { s1 = reinterpret_cast<float*>(arena + s1_off); s2 = reinterpret_cast<float*>(arena + s2_off); }
    if (bf)
      for (int l = 0; l < L; ++l) layers[l].Wn = reinterpret_cast<__nv_bfloat16*>(arena + wn_off[l]);
  }
  SB_TRY(dalloc(&scal, SCAL_COUNT));
  SB_TRY(dalloc(&desc, 1));
  if (want_trace) SB_TRY(dalloc(&step_trace, 32 * 16));
  SB_TRY(dalloc(&yhat, max_batch));
  SB_TRY(dalloc(&ones, max_batch));
  SB_TRY(dalloc(&stX, static_cast<size_t>(max_batch) * F));
  SB_TRY(dalloc(&stY, max_batch));
  SB_TRY(dalloc(&stW, max_batch));
  fill_kernel<<<(max_batch + 255) / 256, 256, 0, stream>>>(ones, 1.f, max_batch);

  if (bf) {
    Xb_ps = static_cast<long long>(max_batch) * ldF;
    SB_TRY(dalloc(&Xb, static_cast<size_t>(Xb_ps) * nparts));
    A.assign(L, nullptr); dZ.assign(L, nullptr); A_ps.assign(L, 0);
    for (int l = 0; l < L; ++l) {
      Layer& ly = layers[l];
      A_ps[l] = static_cast<long long>(max_batch) * ly.ld_out;
      SB_TRY(dalloc(&A[l], static_cast<size_t>(A_ps[l]) * nparts));
      if (training) SB_TRY(dalloc(&dZ[l], static_cast<size_t>(A_ps[l]) * nparts));
    }
  } else {
    SB_TRY(dalloc(&Xf, static_cast<size_t>(max_batch) * F));
    Af.assign(L, nullptr); dZf.assign(L, nullptr);
    for (int l = 0; l < L; ++l) {
      SB_TRY(dalloc(&Af[l], static_cast<size_t>(max_batch) * layers[l].out));
      if (training) SB_TRY(dalloc(&dZf[l], static_cast<size_t>(max_batch) * layers[l].out));
    }
  }

  // optimizer / shadow-refresh work table: runs of <= 1024 consecutive parameters
  std::vector<OptWork> wk;
  auto add_runs = [&](long long o, long long n, const Layer* mat) {
    for (long long s = 0; s < n; s += 1024) {
      OptWork w = {};
      w.off = o + s; w.count = static_cast<int>(n - s < 1024 ? n - s : 1024);
      w.np = 1;
      if (mat) {
        w.out_dim = mat->out; w.mat_off = mat->w_off; w.Wn = mat->Wn; w.ld_out = mat->ld_out;
        w.np = nparts; w.part_stride = Wn_ps[static_cast<size_t>(mat - layers.data())];
      }
      wk.push_back(w);
    }
  };
  work_begin.assign(L + 1, 0); work_end.assign(L + 1, 0);
  for (int l = 0; l <= L; ++l) {
    Layer& ly = layers[l];
    work_begin[l] = static_cast<int>(wk.size());
    if (bf && l < L) {
      add_runs(ly.w_off, static_cast<long long>(ly.in) * ly.out, &ly);
      add_runs(ly.b_off, ly.out, nullptr);
    } else {
      add_runs(ly.w_off, static_cast<long long>(ly.in) * ly.out + ly.out, nullptr);
    }
    work_end[l] = static_cast<int>(wk.size());
  }
  n_work = static_cast<int>(wk.size());
  SB_TRY(dalloc(&work, wk.size()));
  SB_CUDA(cudaMemcpyAsync(work, wk.data(), wk.size() * sizeof(OptWork), cudaMemcpyHostToDevice, stream));
  SB_CUDA(cudaStreamSynchronize(stream));

  // opt in to > 48 KB dynamic shared memory once, outside of any stream capture
  if (bf) {
    SB_TRY((set_gemm_tc_attrs<EPI_FWD, false, true>()));
    SB_TRY((set_gemm_tc_attrs<EPI_FWD_OUT, false, true>()));
    SB_TRY((set_gemm_tc_attrs<EPI_DA, false, false>()));
    SB_TRY((set_gemm_tc_attrs<EPI_DW, true, true>()));
    // keep the SMs in the GEMMs' shared-memory carve-out for every kernel of the step, so that no launch in the chain
    // has to re-partition L1 / shared memory
    const int co = cudaSharedmemCarveoutMaxShared;
    cudaFuncSetAttribute(load_batch_kernel<true>, cudaFuncAttributePreferredSharedMemoryCarveout, co);
    cudaFuncSetAttribute(out_layer_kernel<__nv_bfloat16>, cudaFuncAttributePreferredSharedMemoryCarveout, co);
  }
  return SB_OK;
}

void Net::destroy() {
  if (stream) cudaStreamSynchronize(stream);
  for (void* p : allocs) cudaFree(p);
  allocs.clear();
  for (cudaEvent_t e : ev_dz) cudaEventDestroy(e);
  ev_dz.clear();
  if (ev_join) cudaEventDestroy(ev_join);
  ev_join = nullptr;
  if (ev_da_done) cudaEventDestroy(ev_da_done);
  ev_da_done = nullptr;
  if (comm) cudaStreamDestroy(comm);
  comm = nullptr;
  if (comm2) cudaStreamDestroy(comm2);
  comm2 = nullptr;
  if (side) cudaStreamDestroy(side);
  side = nullptr;
  if (stream) cudaStreamDestroy(stream);
  stream = nullptr;
}

int Net::set_sparse(int n_dense_, int n_onehot_, int n_cat_) {
  SB_CHECK(n_dense_ >= 1 && n_onehot_ >= 1 && n_cat_ >= 1, SB_ERR_INVALID, "wide+deep needs >= 1 dense, one-hot and categorical column");
  SB_CHECK(n_dense_ + n_onehot_ == F, SB_ERR_INVALID, "n_dense (%d) + n_onehot (%d) must equal n_features (%d): the sparse path evaluates "
           "the SAME first layer", n_dense_, n_onehot_, F);
  SB_CUDA(cudaSetDevice(device));
  n_dense = n_dense_; n_onehot = n_onehot_; n_cat = n_cat_;
  ldD = round_up(n_dense, 8);
  if (!idx) SB_TRY(dalloc(&idx, static_cast<size_t>(max_batch) * n_cat));
  if (!E) SB_TRY(dalloc(&E, static_cast<size_t>(max_batch) * layers[0].ld_out));
  SB_CUDA(cudaStreamSynchronize(stream));
  return SB_OK;
}

int Net::enqueue_embed(int rows, bool scatter, float* grad, cudaStream_t st) {
  const Layer& l0 = layers[0];
  EmbedParams p = {};
  p.rows = rows; p.n_cat = n_cat; p.H = l0.out;
  p.desc = desc;
  p.np = nparts; p.ldW = tc() ? l0.ld_out : l0.out;
  if (tc()) { p.We = l0.Wn + static_cast<size_t>(n_dense) * l0.ld_out; p.We_ps = Wn_ps[0]; }
  else p.We32 = theta + l0.w_off + static_cast<long long>(n_dense) * l0.out;
  p.E = E; p.ldE = l0.ld_out;
  if (scatter) {
    if (tc()) { p.dZ = dZ[0]; p.dZ_ps = A_ps[0]; p.ld_dZ = l0.ld_out; }
    else { p.dZ32 = dZf[0]; p.ld_dZ = l0.out; }
    p.gWe = grad + l0.w_off + static_cast<long long>(n_dense) * l0.out;
    SB_TRY(launch(embed_scatter_kernel, dim3((rows + 7) / 8), dim3(256), 0, st, false, p));
    mark("embed_scatter");
  } else {
    SB_TRY(launch(embed_gather_kernel, dim3((rows + 7) / 8), dim3(256), 0, st, false, p));
    mark("embed_gather");
  }
  return SB_OK;
}

int Net::refresh_shadows() {
  if (!tc()) return SB_OK;
  shadow_refresh_kernel<<<n_work, 256, 0, stream>>>(work, theta);
  SB_CUDA(cudaGetLastError());
  return SB_OK;
}

int Net::enqueue_load(int rows, float* zero_buf, long long zero_n) {
  const int Fx = sparse_step ? n_dense : F;        // a sparse step stages only the dense block
  const int ldx = sparse_step ? ldD : ldF;
  const long long units = static_cast<long long>(rows) * (ldx / 8);
  long long blocks = (units + 255) / 256;
  const long long cap = static_cast<long long>(num_sms) * 16;
  if (blocks > cap) blocks = cap;
  if (blocks < 1) blocks = 1;
  // first kernel of the step: its stream predecessor is set_batch_kernel (a kernel), so PDL applies here too
  if (tc())
    SB_TRY(launch(load_batch_kernel<true>, dim3(static_cast<unsigned>(blocks)), dim3(256), 0, stream, true,
                  static_cast<const BatchDesc*>(desc), rows, Fx, Xb, ldx, static_cast<float*>(nullptr), scal, zero_buf, zero_n,
                  nparts, Xb_ps));
  else
    SB_TRY(launch(load_batch_kernel<false>, dim3(static_cast<unsigned>(blocks)), dim3(256), 0, stream, true,
                  static_cast<const BatchDesc*>(desc), rows, Fx, static_cast<__nv_bfloat16*>(nullptr), ldx, Xf, scal, zero_buf, zero_n,
                  1, 0ll));
  mark("load_batch");
  if (sparse_step) SB_TRY(enqueue_embed(rows, false, nullptr, stream));
  return SB_OK;
}

int Net::enqueue_hidden_forward(int rows, float* grad, bool* fused_out) {
  if (fused_out) *fused_out = false;
  for (int l = 0; l < L; ++l) {
    Layer& ly = layers[l];
    const bool sp0 = (l == 0) && sparse_step;       // wide+deep: contract the dense columns only, add the embedding sums
    if (sp0 && from_resident) SB_TRY(enqueue_embed(rows, false, nullptr, stream));   // (no load kernel launched the gather)
    const int k_in = sp0 ? n_dense : ly.in;
    const int ld_k = sp0 ? ldD : ly.ld_in;
    if (tc()) {
      // Z = A_{l-1}[rows,in] (K-major) x W_l[in,out] (MN-major B operand: n contiguous)
      const GemmPlan pl = plan_gemm(rows, ly.out, round_up(k_in, 64) * pairs_of(nparts), num_sms, false);
      TmapSet tm;
      const bool res0 = (l == 0) && from_resident;
      const __nv_bfloat16* src = (l == 0) ? (res0 ? resident_Xb : Xb) : A[l - 1];
      const long long src_ps = (l == 0) ? (res0 ? resident_ps : Xb_ps) : A_ps[l - 1];
      SB_TRY(make_tmaps_bf16(tm.a, src, src_ps, nparts, res0 ? static_cast<int>(resident_rows) : rows, k_in, ld_k, 128));
      SB_TRY(make_tmaps_bf16(tm.b, ly.Wn, Wn_ps[l], nparts, k_in, ly.out, ly.ld_out, 64));
      GemmTcParams p = {};
      set_part_pairs(&p, nparts);
      p.M = rows; p.N = ly.out; p.K = k_in;
      if (sp0) { p.addend = E; p.ld_add = ly.ld_out; }
      p.bias = theta + ly.b_off; p.act = ly.act;
      p.out = A[l]; p.ld_out = ly.ld_out; p.out_ps = A_ps[l];
      p.a_rows = res0 ? desc : nullptr;
      if (l == L - 1 && grad != nullptr && training && ly.out <= fuse_out_max) {
        // K2 + K3 + K4 + output backward in one kernel: one n-tile must cover the whole layer width
        GemmPlan fp = pl;
        fp.split_k = 1; fp.kb_per_split = ((k_in + 63) / 64) * pairs_of(nparts);
        // (a 256-wide PAIR tile measured slower than GEMM + out_layer kernel in round 1; the single-CTA 128 x 256 tile keeps
        // whole rows of A_L in one CTA's TMEM - 2 x 256 columns, double-buffered - and needs no second kernel)
        if (ly.out <= 64) { fp.cg = 1; fp.bn = 64; }
        else if (ly.out <= 128) { fp.cg = 1; fp.bn = 128; }
        else { fp.cg = 1; fp.bn = 256; }
        const int slots = num_sms / fp.cg;
        const int tiles = (rows + 128 * fp.cg - 1) / (128 * fp.cg);
        fp.grid = (tiles < slots ? tiles : slots) * fp.cg;
        Layer& ol = layers[L];
        p.out = dZ[l];
        p.wo = theta + ol.w_off; p.bo = theta + ol.b_off;
        p.desc = desc; p.scal = scal; p.loss = loss;
        p.g_wo = grad + ol.w_off; p.g_bo = grad + ol.b_off; p.g_bL = grad + ly.b_off;
        p.trace = next_trace("fwd_out", l, rows, ly.out, k_in);
        SB_TRY((launch_gemm_tc<EPI_FWD_OUT, false, true>(fp, tm, p, stream, true)));
        if (fused_out) *fused_out = true;
        mark("gemm_fwd_out");
        continue;
      }
      if (l == 0 && zero_buf != nullptr) {
        p.zero_buf = zero_buf; p.zero_n4 = zero_n4;
        zero_buf = nullptr;
      }
      p.trace = next_trace("fwd", l, rows, ly.out, k_in);
      if (nparts == 1 && p.addend == nullptr)      // plain bf16: the epilogue stores its tiles by TMA
        SB_TRY(make_tmap_bf16(&tm.o, A[l], rows, ly.out, ly.ld_out, 128));
      SB_TRY((launch_gemm_tc<EPI_FWD, false, true>(pl, tm, p, stream, true)));
    } else {
      GemmF32Params p = {};
      p.M = rows; p.N = ly.out; p.K = k_in;
      p.A = (l == 0) ? Xf : Af[l - 1]; p.sAm = k_in; p.sAk = 1;
      if (sp0) { p.addend = E; p.ld_add = ly.ld_out; }
      p.B = theta + ly.w_off; p.sBk = ly.out; p.sBn = 1;
      p.bias = theta + ly.b_off; p.act = ly.act;
      p.out = Af[l]; p.ld_out = ly.out;
      SB_TRY(launch_gemm_f32<EPI_FWD>(p, 1, stream));
    }
    mark("gemm_fwd");
  }
  return SB_OK;
}

int Net::enqueue_out(int rows, bool do_loss, bool do_bwd, float* yhat_dst, float* grad) {
  Layer& hl = layers[L - 1];
  Layer& ol = layers[L];
  OutLayerParams p = {};
  p.rows = rows; p.H = hl.out;
  p.wo = theta + ol.w_off; p.bo = theta + ol.b_off;
  p.desc = desc; p.scal = scal; p.loss = loss; p.act = hl.act;
  p.do_bwd = do_bwd ? 1 : 0; p.do_loss = do_loss ? 1 : 0;
  p.yhat = yhat_dst;
  p.trace = next_trace("out_layer");
  if (do_bwd) {
    p.g_wo = grad + ol.w_off; p.g_bo = grad + ol.b_off; p.g_bL = grad + hl.b_off;
  }
  const int grid = (rows + 31) / 32;
  if (tc()) {
    p.A = A[L - 1]; p.ldA = hl.ld_out;
    p.np = nparts; p.a_ps = A_ps[L - 1]; p.dz_ps = A_ps[L - 1];
    if (do_bwd) { p.dZ = dZ[L - 1]; p.ld_dZ = hl.ld_out; }
    if (hl.out <= 1024) {
      // one-pass kernel: rows per block sized for ~2 blocks per SM, at least one row per warp
      int rpb = (rows + 2 * num_sms - 1) / (2 * num_sms);
      rpb = ((rpb + 7) / 8) * 8;
      if (rpb < 8) rpb = 8;
      const dim3 g((rows + rpb - 1) / rpb);
      if (hl.out <= 256) SB_TRY(launch(out_layer_rows_kernel<1>, g, dim3(256), 0, stream, true, p, rpb));
      else if (hl.out <= 512) SB_TRY(launch(out_layer_rows_kernel<2>, g, dim3(256), 0, stream, true, p, rpb));
      else SB_TRY(launch(out_layer_rows_kernel<4>, g, dim3(256), 0, stream, true, p, rpb));
    } else {
      SB_TRY(launch(out_layer_kernel<__nv_bfloat16>, dim3(grid), dim3(256), 0, stream, true, p));
    }
  } else {
    p.A = Af[L - 1]; p.ldA = hl.out;
    if (do_bwd) { p.dZ = dZf[L - 1]; p.ld_dZ = hl.out; }
    SB_TRY(launch(out_layer_kernel<float>, dim3(grid), dim3(256), 0, stream, true, p));
  }
  SB_CUDA(cudaGetLastError());
  mark("out_layer");
  return SB_OK;
}

int Net::enqueue_backward(int rows, float* grad) {
  // dW_l and dA_l both consume dZ_l and are independent of each other: the dW GEMMs go to the side stream and
  // overlap the dA chain (they are each well under one wave at cfg1 sizes).  Not while profiling (clean times).
  const bool fork = !profiling && side != nullptr && tc();
  // dW_1 (side stream) and dW_0 (main stream) run at the same time, one CTA per SM each.  If their natural grids do not
  // fit the machine together, dW_1's second wave only starts when dW_0's CTAs exit (measured: the side optimizer then
  // finishes 4 us after the main one, scripts/step_timeline.py).  Compare, in k-blocks per CTA, "natural grids, dW_1
  // finishing after dW_0" against "dW_1 on a third of the SMs, dW_0 on the rest" and take the shorter.
  int dw_sms[2] = {num_sms, num_sms};
  // dw1_serial_auto (single-GPU tail): when the natural grids of dW_0 and dW_1 do not fit the machine together, dW_1 runs IN
  // FRONT of dW_0 on the main stream instead of beside it - side by side the two persistent grids take turns on the SMs
  // (cfg2: 47.9 us for both; alone 13.9 + 29.0 us, profiles/ncu_r02_cfg2_launches.txt); small layers (cfg1) stay side by side
  bool dw1_front = dw1_first;
  if (fork && dw0_on_main && L > 1 && !dw1_last && !dw1_first) {
    const int kx = round_up(rows, 64) * pairs_of(nparts);
    const GemmPlan n0 = plan_gemm(layers[0].in, layers[0].out, kx, num_sms, true);
    const GemmPlan n1 = plan_gemm(layers[1].in, layers[1].out, kx, num_sms, true);
    if (n0.grid + n1.grid > num_sms && dw1_serial_auto && n0.cg == 2) {      // (pair tiles = a GEMM of several waves, plan_gemm)
      dw1_front = true;
    } else if (n0.grid + n1.grid > num_sms) {
      const GemmPlan b1 = plan_gemm(layers[1].in, layers[1].out, kx, num_sms / 3, true);
      const GemmPlan b0 = plan_gemm(layers[0].in, layers[0].out, kx, num_sms - b1.grid, true);
      auto waves = [&](const GemmPlan& pl, int M, int N, int sms) {   // k-blocks one CTA works through
        const int tiles = ((M + 128 * pl.cg - 1) / (128 * pl.cg)) * ((N + pl.bn - 1) / pl.bn) * pl.split_k;
        const int slots = sms / pl.cg;
        return ((tiles + slots - 1) / slots) * pl.kb_per_split;
      };
      const int t_nat = waves(n0, layers[0].in, layers[0].out, num_sms) + waves(n1, layers[1].in, layers[1].out, num_sms);
      const int t0 = waves(b0, layers[0].in, layers[0].out, num_sms - b1.grid);
      const int t1 = waves(b1, layers[1].in, layers[1].out, num_sms / 3);
      if ((t0 > t1 ? t0 : t1) < t_nat) { dw_sms[1] = num_sms / 3; dw_sms[0] = num_sms - b1.grid; }
    }
  }
  auto emit_dw_tc = [&](int l, bool force_main) -> int {
        Layer& ly = layers[l];
        const bool xchg_chunks = l == 0 && dw0_chunks >= 1 && on_dw0_chunk && (ly.out % 8 == 0 || dw0_chunks == 1) && !sparse_step;
        const int n_chunks = xchg_chunks ? dw0_chunks : 1;
        // dW_0 has nothing to overlap with (no dA_0): PDL-chained on the main stream right behind the last dA GEMM it
        // starts ~6 us earlier than as a cross-stream launch (measured, scripts/step_timeline.py)
        const bool on_main = !fork || (l == 0 && dw0_on_main && L > 1) || force_main;
        if (!on_main) {
          SB_CUDA(cudaEventRecord(ev_dz[l], stream));
          SB_CUDA(cudaStreamWaitEvent(side, ev_dz[l], 0));
        }
        const bool res0 = (l == 0) && from_resident;
        const bool sp0 = (l == 0) && sparse_step;     // wide+deep: dW of the dense rows by GEMM, of the embedding rows by scatter-add
        const int in_rows = sp0 ? n_dense : ly.in;
        const int ld_k = sp0 ? ldD : ly.ld_in;
        const int chunk_rows = xchg_chunks ? dw0_chunk_rows() : round_up(in_rows, 128);
        const __nv_bfloat16* ap = (l == 0) ? (res0 ? resident_Xb : Xb) : A[l - 1];
        const long long ap_ps = (l == 0) ? (res0 ? resident_ps : Xb_ps) : A_ps[l - 1];
        if (sp0) SB_TRY(enqueue_embed(rows, true, grad, on_main ? stream : side));
        for (int r0 = 0; r0 < in_rows; r0 += chunk_rows) {
          const int r1 = (r0 + chunk_rows < in_rows) ? r0 + chunk_rows : in_rows;
          const GemmPlan pl = plan_gemm(r1 - r0, ly.out, round_up(rows, 64) * pairs_of(nparts), l < 2 ? dw_sms[l] : num_sms, true);
          TmapSet tm;
          // resident set: rows past the batch end are real rows of other batches; the B operand (dZ_l, extent = rows) is
          // zero-filled there, so they contribute nothing
          SB_TRY(make_tmaps_bf16(tm.a, ap + r0, ap_ps, nparts, res0 ? static_cast<int>(resident_rows) : rows, r1 - r0, ld_k, 64));
          SB_TRY(make_tmaps_bf16(tm.b, dZ[l], A_ps[l], nparts, rows, ly.out, ly.ld_out, 64));
          GemmTcParams p = {};
          set_part_pairs(&p, nparts);
          p.M = r1 - r0; p.N = ly.out; p.K = rows;
          p.a_rows = res0 ? desc : nullptr;
          p.accum = grad + ly.w_off + static_cast<long long>(r0) * ly.out; p.ld_acc = ly.out;
          p.acc_vec4 = (ly.out % 4 == 0 && ly.w_off % 4 == 0) ? 1 : 0;
          p.trace = next_trace("dW", l, r1 - r0, ly.out, rows, n_chunks > 1 ? r0 / chunk_rows : -1);
          SB_TRY((launch_gemm_tc<EPI_DW, true, true>(pl, tm, p, on_main ? stream : side, on_main)));
          mark("gemm_dw");
          if (xchg_chunks) SB_TRY(on_dw0_chunk(r0 / chunk_rows));
        }
        return SB_OK;
  };
  for (int l = L - 1; l >= 0; --l) {
    Layer& ly = layers[l];
    if (tc()) {
      // dW_l[in,out] += sum_rows A_{l-1}[rows,in] (MN-major A) * dZ_l[rows,out] (MN-major B), split-K over rows.
      // With the peer exchange, dW_0 is cut into row chunks of W_0 (each a contiguous slice of the flat gradient) so that
      // the exchange of chunk c overlaps the GEMM of chunk c+1.
      const bool dw1_moved = (dw1_last || dw1_front) && L > 1;
      if (dw1_front && l == 0 && L > 1) {         // in front of dW_0 on the main stream: dW_0's last exchange then runs on an idle GPU
        SB_TRY(emit_dw_tc(1, true));
        if (after_dw1) SB_TRY(after_dw1());
      }
      if (!(dw1_moved && l == 1)) SB_TRY(emit_dw_tc(l, false));
      if (dw1_last && !dw1_front && l == 0 && L > 1) SB_TRY(emit_dw_tc(1, true));   // behind dW_0 on the main stream (covers its last exchange)
      if (l > 0) {
        // dZ_{l-1}[rows,in] = (dZ_l[rows,out] (K-major) x W_l[in,out] (K-major B: k = out contiguous)) .* act'(A_{l-1})
        Layer& pl = layers[l - 1];
        const GemmPlan gp = plan_gemm(rows, ly.in, round_up(ly.out, 64) * pairs_of(nparts), num_sms, false);
        TmapSet tm;
        SB_TRY(make_tmaps_bf16(tm.a, dZ[l], A_ps[l], nparts, rows, ly.out, ly.ld_out, 128));
        SB_TRY(make_tmaps_bf16(tm.b, ly.Wn, Wn_ps[l], nparts, ly.in, ly.out, ly.ld_out, plan_box_rows_b(gp)));
        GemmTcParams p = {};
        set_part_pairs(&p, nparts);
        p.M = rows; p.N = ly.in; p.K = ly.out;
        p.act = pl.act;
        p.aux = A[l - 1]; p.ld_aux = pl.ld_out; p.aux_ps = A_ps[l - 1];
        p.out = dZ[l - 1]; p.ld_out = pl.ld_out; p.out_ps = A_ps[l - 1];
        p.colsum = grad + pl.b_off;
        p.trace = next_trace("dA", l, rows, ly.in, ly.out);
        if (nparts == 1) {                           // plain bf16: A_{l-1} in and dZ_{l-1} out move as TMA tiles
          SB_TRY(make_tmap_bf16(&tm.o, dZ[l - 1], rows, ly.in, pl.ld_out, 128));
          SB_TRY(make_tmap_bf16(&tm.x, A[l - 1], rows, ly.in, pl.ld_out, 128));
        }
        SB_TRY((launch_gemm_tc<EPI_DA, false, false>(gp, tm, p, stream, true)));
        mark("gemm_da");
        if (l == 1 && fork && defer_join) SB_CUDA(cudaEventRecord(ev_da_done, stream));
      }
    } else {
      {
        const bool sp0 = (l == 0) && sparse_step;
        const int in_rows = sp0 ? n_dense : ly.in;
        if (sp0) SB_TRY(enqueue_embed(rows, true, grad, stream));
        GemmF32Params p = {};
        p.M = in_rows; p.N = ly.out; p.K = rows;
        p.A = (l == 0) ? Xf : Af[l - 1]; p.sAm = 1; p.sAk = in_rows;
        p.B = dZf[l]; p.sBk = ly.out; p.sBn = 1;
        p.accum = grad + ly.w_off; p.ld_acc = ly.out;
        const int tiles = ((p.M + 63) / 64) * ((p.N + 63) / 64);
        int split = (2 * num_sms) / (tiles > 0 ? tiles : 1);
        const int cap = (rows + 63) / 64;
        if (split > cap) split = cap;
        SB_TRY(launch_gemm_f32<EPI_DW>(p, split, stream));
        mark("gemm_dw");
      }
      if (l > 0) {
        Layer& pl = layers[l - 1];
        GemmF32Params p = {};
        p.M = rows; p.N = ly.in; p.K = ly.out;
        p.A = dZf[l]; p.sAm = ly.out; p.sAk = 1;
        p.B = theta + ly.w_off; p.sBk = 1; p.sBn = ly.out;
        p.act = pl.act;
        p.aux = Af[l - 1]; p.ld_aux = pl.out;
        p.out = dZf[l - 1]; p.ld_out = pl.out;
        p.colsum = grad + pl.b_off;
        SB_TRY(launch_gemm_f32<EPI_DA>(p, 1, stream));
        mark("gemm_da");
      }
    }
  }
  if (fork && !defer_join) {
    SB_CUDA(cudaEventRecord(ev_join, side));
    SB_CUDA(cudaStreamWaitEvent(stream, ev_join, 0));
  }
  return SB_OK;
}

}  // namespace sb
