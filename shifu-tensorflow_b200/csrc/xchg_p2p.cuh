// Sharded gradient exchange + optimizer over NVLink peer memory (CUDA IPC / in-process peers), ONE kernel per launch:
//
//     reduce-scatter (P2P loads)  ->  optimizer on the owned slice only  ->  all-gather of the GEMM operands (P2P stores)
//
// It replaces, on one NVLink/NVSwitch node, what the reference does with parameter servers: every worker pushes its
// gradients to the ConditionalAccumulators on the PS tasks, the mean is applied there ONCE per variable, and every worker
// pulls the new variables (res/ssgd_monitor.py:136-141, 203-206).  Here the "parameter server" of a run of 1024
// parameters is the rank that owns it:
//
//   every rank exports ONE allocation (the parameter arena, net.cuh):  [theta | s1 | s2 | bf16 shadows | gradient | flags]
//   the flat vector is cut into the optimizer's work runs (<= 1024 parameters each); the runs of a SLOT are dealt out to the
//   ranks in equal contiguous shares.  Slot 0 = every layer but hidden layer 0; slots 1..C = row chunks of hidden layer 0
//   (the big one, whose gradient is complete last).  The slot table is fixed for a trainer's life - it defines who owns
//   which run - while a launch may handle any set of slots (the flags of the lowest one synchronise it).
//
//   per launch (flag value = the step's exchange epoch):
//     arrive   "my gradient of these slots is complete": store epoch into arrive[slot][me] of every peer
//              (st.release.sys), every block waits until all peers' words in MY flag block carry it (ld.acquire.sys)
//     owned runs, 256 threads x 4 parameters each:
//              g = sum over ranks (fixed order 0..W-1 -> the same bits wherever it is computed) of the peers' gradients,
//              all W x U 16-byte P2P loads of a thread in flight before the first add;
//              fp32 master + optimizer state of the run are LOCAL (only the owner ever updates them);
//              the result is written LOCALLY: fp32 master, state, and the bf16 weight shadow the GEMMs read.
//     updated  the last block to finish publishes done[slot][me] = epoch to every peer (local stores only: no fabric fence)
//     gather   every block waits for every peer's `updated`, then the runs other ranks own are pulled from their owners by
//              P2P loads: the bf16 shadow (8 B per thread - half the bytes of an fp32 all-gather) or, for runs without a
//              shadow (biases, output layer, fp32 mode), fp32 theta.  A peer's `updated` also says it no longer reads my
//              gradient: on exit all my operands are final and my gradient buffer is free.
//
//   The schedule that hides the launches behind GEMMs lives in capi.cu (enqueue_step_body).
//
// A rank only reads other ranks' gradients of ITS runs and only writes ITS runs of other ranks' operands; the writes
// happen after every rank has arrived, i.e. after every rank's last reader of those operands in this step (the launch is
// stream-ordered behind them).  Non-owners keep a stale fp32 master / state for shadow-backed runs: gather_master_kernel
// refreshes them before anything reads theta on the host side (get_params, checkpoint, export).
//
// A lost peer is reported, not trapped: after `timeout_ns` a waiting block records (slot, missing rank) in mapped host
// memory and every block leaves the kernel; the host turns that into SB_ERR_NCCL at its next wait.
#pragma once
#include "common.cuh"
#include "kernels.cuh"

namespace sb {

#define SB_MAX_RANKS 16
#define SB_XCHG_SLOTS 8                   // slot 0: every layer but hidden layer 0; slots 1..C: row chunks of hidden layer 0

struct P2PFlags {                                     // at arena + flags_off on every rank
  unsigned int arrive[SB_XCHG_SLOTS][SB_MAX_RANKS];   // arrive[slot][q] written by rank q
  unsigned int done[SB_XCHG_SLOTS][SB_MAX_RANKS];     // done[slot][q]   written by rank q
  unsigned int blocks_done[SB_XCHG_SLOTS];            // local: grid-wide completion counter per slot
  unsigned int pad[24];
};

struct P2PPeers {                         // device-resident table, same order on every rank
  char* base[SB_MAX_RANKS];               // arena of every rank (own entry = own arena)
};

struct XchgParams {
  const P2PPeers* peers;
  int rank, world;
  long long s1_off, s2_off, grad_off, flags_off;   // byte offsets inside every arena (theta at 0)
  const OptWork* work;
  int n_slots;
  int slot_begin[SB_XCHG_SLOTS], slot_end[SB_XCHG_SLOTS];   // work-table range of every slot (the same table on every rank:
                                                            // it defines who owns which run, whatever the launch pattern)
  int slot_mask;                          // bit s set: this launch handles slot s (flags of the LOWEST set slot synchronise it)
  const BatchDesc* desc;
  OptHyper hyper;
  const float* scal;                      // step scalars to publish (nullable)
  float* host_scal;
  unsigned int* host_err;                 // mapped pinned: [0] = 0 ok | 1 + 16 * slot + missing rank
  unsigned long long timeout_ns;          // 0 = wait forever
  int fence_gpu;                          // 1 (default): gpu-scope fence before the `updated` flag; SB_XCHG_FENCE_SYS=1 -> 0
  unsigned long long* trace;              // slots: 0 entry, 2 dependencies resolved, 3 every peer arrived (block 0), 4 last block's
                                          // runs done, 5 `updated` published, 6 every peer updated (block 0), 10 exit (gathered)
};

__device__ __forceinline__ void st_release_sys(unsigned int* p, unsigned int v) {
  asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ unsigned int ld_acquire_sys(const unsigned int* p) {
  unsigned int v;
  asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ float4 ld_peer_f4(const float* p) {
  float4 v;
  asm volatile("ld.relaxed.sys.global.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ float ld_peer_f1(const float* p) {
  float v;
  asm volatile("ld.relaxed.sys.global.f32 %0, [%1];" : "=f"(v) : "l"(p) : "memory");
  return v;
}

// first work item of rank r's share of [b, e)
__host__ __device__ inline int xchg_share(int b, int e, int r, int world) {
  return b + static_cast<int>((static_cast<long long>(e - b) * r) / world);
}

// Block-wide wait until slots[q] >= epoch for every q < world.  Returns false after a timeout (error recorded).
__device__ __forceinline__ bool xchg_wait(const unsigned int* slots, int world, unsigned int epoch, const XchgParams& p, int seg,
                                          unsigned int* sh_fail) {
  if (threadIdx.x < 32) {
    const int lane = threadIdx.x;
    bool ok = true;
    if (lane < world) {
      unsigned long long t0 = 0;
      unsigned int spins = 0;
      while (static_cast<int>(ld_acquire_sys(slots + lane) - epoch) < 0) {
        if ((++spins & 0x3FFu) == 0) {
          if (*reinterpret_cast<volatile unsigned int*>(sh_fail)) { ok = false; break; }
          if (p.timeout_ns != 0) {
            const unsigned long long now = globaltimer_ns();
            if (t0 == 0) t0 = now;
            else if (now - t0 > p.timeout_ns) {
              if (p.host_err != nullptr) { atomicCAS(p.host_err, 0u, 1u + 16u * seg + lane); __threadfence_system(); }
              ok = false;
              break;
            }
          }
        }
      }
    }
    if (!__all_sync(0xffffffffu, ok) && lane == 0) *sh_fail = 1u;
  }
  __syncthreads();
  return *reinterpret_cast<volatile unsigned int*>(sh_fail) == 0u;
}

// W = compile-time upper bound of `world`; a block iteration handles U consecutive runs with every load of the iteration in
// flight before the first add.  <= 85 registers per thread: one block (21 k registers) fits beside ANY of the
// persistent GEMM CTAs that may be resident while an exchange runs - the dW GEMMs of the same step (320 threads x 64) -
// so the exchange really overlaps them.
// Measured on 2 x B200 through NVSwitch (scripts/p2p_probe.cu, profiles/p2p_probe_r02.txt): a flag takes 2.7 us one way, a
// P2P load round trip ~5 us, bandwidth 750 GB/s only beyond ~16 MB in flight (4 MB: 14 us).  The chain arrive -> loads ->
// stores + fence -> done therefore costs ~17 us however little data moves: the schedule (capi.cu) hides it behind GEMMs.
template <int W>
static __global__ void __launch_bounds__(256, W <= 8 ? 3 : 2)
xchg_update_kernel(const XchgParams p) {
  constexpr int U = W <= 2 ? 2 : 1;       // runs per block iteration: U x (W + 3) sixteen-byte loads per thread in flight
  __shared__ unsigned int sh_fail;
  __shared__ unsigned int sh_last;
  if (threadIdx.x == 0) sh_fail = 0u;
  trace_begin(p.trace, true);
  pdl_wait();                 // the gradient of these slots is complete (stream order / programmatic dependency)
  trace_begin(p.trace, false);
  __syncthreads();
  const unsigned int epoch = p.desc->epoch;
  char* pb[W];                // every rank's arena (entries >= world alias the own arena and are never used)
#pragma unroll
  for (int q = 0; q < W; ++q) pb[q] = p.peers->base[q < p.world ? q : p.rank];
  char* const my_base = p.peers->base[p.rank];
  float* const theta = reinterpret_cast<float*>(my_base);
  P2PFlags* mine = reinterpret_cast<P2PFlags*>(my_base + p.flags_off);
  if (p.host_scal != nullptr && blockIdx.x == 0 && threadIdx.x < SCAL_COUNT) {
    p.host_scal[threadIdx.x] = p.scal[threadIdx.x];     // loss sum / n_nz of this rank's mini-batch (see optimizer_kernel)
    if (threadIdx.x == 0 && p.desc->hist != nullptr) *p.desc->hist = make_float2(p.scal[SCAL_LOSS_SUM], p.scal[SCAL_NNZ]);
    __threadfence_system();
  }
  const float lr_t = p.desc->lr_t, gs = p.desc->gscale;
  const bool use_s1 = p.hyper.kind != SB_OPT_SGD;
  const bool use_s2 = p.hyper.kind == SB_OPT_ADAM || p.hyper.kind == SB_OPT_ADADELTA;
  float* const s1 = reinterpret_cast<float*>(my_base + p.s1_off);
  float* const s2 = reinterpret_cast<float*>(my_base + p.s2_off);
  float* const my_grad = reinterpret_cast<float*>(my_base + p.grad_off);
  const int sync = __ffs(p.slot_mask) - 1;          // the slot whose flags carry this launch
  auto stamp_max = [&](int slot) { if (p.trace != nullptr && threadIdx.x == 0) atomicMax(p.trace + slot, static_cast<unsigned long long>(globaltimer_ns())); };
  // ---- arrive ----
  if (blockIdx.x == 0 && threadIdx.x < p.world)
    st_release_sys(&reinterpret_cast<P2PFlags*>(p.peers->base[threadIdx.x] + p.flags_off)->arrive[sync][p.rank], epoch);
  bool alive = xchg_wait(mine->arrive[sync], p.world, epoch, p, sync, &sh_fail);
  if (p.trace != nullptr && blockIdx.x == 0 && threadIdx.x == 0) p.trace[3] = globaltimer_ns();
  // ---- owned runs of every slot of the launch ----
  // (every load of an iteration - the peers' gradients, the local master and state - is issued before the first store, so a
  // thread pays the fabric round trip once per iteration; the first version interleaved them run by run and took 20 us for
  // 512 runs beside a GEMM)
  if (alive) {
#pragma unroll 1
    for (int slot = 0; slot < p.n_slots; ++slot) {
      if (!((p.slot_mask >> slot) & 1)) continue;
      const int w0 = xchg_share(p.slot_begin[slot], p.slot_end[slot], p.rank, p.world);
      const int w1 = xchg_share(p.slot_begin[slot], p.slot_end[slot], p.rank + 1, p.world);
#pragma unroll 1
      for (int wb = w0 + static_cast<int>(blockIdx.x) * U; wb < w1; wb += static_cast<int>(gridDim.x) * U) {
        float4 g[U][W], th[U], sa[U], sb[U];
        bool vec[U], on[U];
        const int e = threadIdx.x * 4;
#pragma unroll
        for (int u = 0; u < U; ++u) {
          vec[u] = false; on[u] = false;
          sa[u] = make_float4(0.f, 0.f, 0.f, 0.f); sb[u] = sa[u]; th[u] = sa[u];
          if (wb + u < w1) {
            const OptWork& wk = p.work[wb + u];
            const long long off = wk.off;
            const int cnt = wk.count;
            vec[u] = (off & 3) == 0 && (cnt & 3) == 0 &&
                     (wk.Wn == nullptr || ((wk.out_dim & 3) == 0 && ((off - wk.mat_off) & 3) == 0 && (wk.ld_out & 3) == 0));
            on[u] = vec[u] && e < cnt;
            if (on[u]) {
#pragma unroll
              for (int q = 0; q < W; ++q)
                if (q < p.world) g[u][q] = ld_peer_f4(reinterpret_cast<const float*>(pb[q] + p.grad_off) + off + e);
              th[u] = *reinterpret_cast<const float4*>(theta + off + e);
              if (use_s1) sa[u] = *reinterpret_cast<const float4*>(s1 + off + e);
              if (use_s2) sb[u] = *reinterpret_cast<const float4*>(s2 + off + e);
            }
          }
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
          if (wb + u >= w1) continue;
          const OptWork wk = p.work[wb + u];
          const long long shadow_rel = wk.Wn != nullptr ? reinterpret_cast<char*>(wk.Wn) - my_base : 0;
          if (vec[u]) {
            if (on[u]) {
              float4 acc = g[u][0];               // fixed rank order -> the same bits wherever a sum is computed
#pragma unroll
              for (int q = 1; q < W; ++q)
                if (q < p.world) { acc.x += g[u][q].x; acc.y += g[u][q].y; acc.z += g[u][q].z; acc.w += g[u][q].w; }
              const long long idx = wk.off + e;
              float4 a = sa[u], b = sb[u], t;
              t.x = opt_update(p.hyper, lr_t, th[u].x, acc.x * gs, a.x, b.x);
              t.y = opt_update(p.hyper, lr_t, th[u].y, acc.y * gs, a.y, b.y);
              t.z = opt_update(p.hyper, lr_t, th[u].z, acc.z * gs, a.z, b.z);
              t.w = opt_update(p.hyper, lr_t, th[u].w, acc.w * gs, a.w, b.w);
              *reinterpret_cast<float4*>(theta + idx) = t;
              // the owner keeps the reduced gradient of its runs (nobody else reads this part of my buffer): parity hook
              *reinterpret_cast<float4*>(my_grad + idx) = acc;
              if (use_s1) *reinterpret_cast<float4*>(s1 + idx) = a;
              if (use_s2) *reinterpret_cast<float4*>(s2 + idx) = b;
              if (wk.Wn != nullptr) {
                const long long m = idx - wk.mat_off;
                const long long r = m / wk.out_dim;     // 4 consecutive elements never straddle a row
                const long long rel = shadow_rel + (r * wk.ld_out + (m - r * wk.out_dim)) * 2;
                for (int part = 0; part < wk.np; ++part) {      // split-precision modes: every part of the shadow
                  uint2 o;
                  o.x = pack_bf16x2(bf16_residual(t.x, part), bf16_residual(t.y, part));
                  o.y = pack_bf16x2(bf16_residual(t.z, part), bf16_residual(t.w, part));
                  *reinterpret_cast<uint2*>(my_base + rel + part * wk.part_stride * 2) = o;     // peers pull it in phase 2
                }
              }
            }
          } else {
            // unaligned run (odd widths): scalar path, 4 elements per thread strided by 256
#pragma unroll 1
            for (int i = 0; i < 4; ++i) {
              const int es = threadIdx.x + 256 * i;
              if (es < wk.count) {
                const long long idx = wk.off + es;
                float acc = 0.f;
                for (int q = 0; q < p.world; ++q) acc += ld_peer_f1(reinterpret_cast<const float*>(p.peers->base[q] + p.grad_off) + idx);
                float a = use_s1 ? s1[idx] : 0.f, b = use_s2 ? s2[idx] : 0.f;
                const float t = opt_update(p.hyper, lr_t, theta[idx], acc * gs, a, b);
                theta[idx] = t;
                my_grad[idx] = acc;
                if (use_s1) s1[idx] = a;
                if (use_s2) s2[idx] = b;
                if (wk.Wn != nullptr) {
                  const long long m = idx - wk.mat_off;
                  const long long r = m / wk.out_dim;
                  const long long rel = shadow_rel + (r * wk.ld_out + (m - r * wk.out_dim)) * 2;
                  for (int part = 0; part < wk.np; ++part) {
                    const __nv_bfloat16 hv = __float2bfloat16_rn(bf16_residual(t, part));
                    *reinterpret_cast<__nv_bfloat16*>(my_base + rel + part * wk.part_stride * 2) = hv;
                  }
                }
              }
            }
          }
        }
      }
    }
  }
  stamp_max(4);
  // ---- updated: my owned runs carry the new values (local stores only, so this fence does not wait for the fabric) ----
  // (ONE fence per block, behind the barrier that orders the block's stores before it: a fence per thread serialised the
  // eight warps' MEMBAR.SYS and took 12-14 us on an SM that shares its memory pipeline with a GEMM CTA)
  __syncthreads();
  if (threadIdx.x == 0) {
    // every store of phase 1 went to LOCAL memory, whose point of coherence - this GPU's L2 - also serves the peers' P2P
    // loads, so a gpu-scope fence is enough to order them before the flag: 2 us instead of the 9-11 us MEMBAR.SYS took on an
    // SM that shares its memory pipeline with a GEMM CTA (measured; replicas stay bit-identical, tests/test_multi_gpu.py).
    // fence_gpu = 0 (SB_XCHG_FENCE_SYS=1) uses the sys scope the PTX memory model asks for between devices.
    if (p.fence_gpu) __threadfence(); else __threadfence_system();
    sh_last = (atomicAdd(&mine->blocks_done[sync], 1u) == gridDim.x - 1) ? 1u : 0u;
  }
  __syncthreads();
  if (sh_last) {
    if (threadIdx.x == 0) { mine->blocks_done[sync] = 0; if (p.fence_gpu) __threadfence(); else __threadfence_system(); }
    __syncthreads();
    if (threadIdx.x < p.world)
    {
      unsigned int* f = &reinterpret_cast<P2PFlags*>(p.peers->base[threadIdx.x] + p.flags_off)->done[sync][p.rank];
      if (p.fence_gpu) asm volatile("st.relaxed.sys.global.u32 [%0], %1;" ::"l"(f), "r"(epoch) : "memory");
      else st_release_sys(f, epoch);
    }
  }
  stamp_max(5);
  // ---- all-gather by P2P LOADS: every run somebody else owns is pulled from its owner once that owner has updated ----
  // (a pushed all-gather has to fence its remote stores before it may raise a flag: 12 us per launch on 2 x B200 while the
  // peer's GEMMs kept its L2 busy; a pull needs no fence, and a peer's "updated" flag also tells that it has finished
  // reading MY gradient - on exit my operands are final and my gradient buffer is free)
  if (alive) alive = xchg_wait(mine->done[sync], p.world, epoch, p, sync, &sh_fail);
  if (p.trace != nullptr && blockIdx.x == 0 && threadIdx.x == 0) p.trace[6] = globaltimer_ns();
  if (alive) {
    constexpr int U2 = 4;
#pragma unroll 1
    for (int slot = 0; slot < p.n_slots; ++slot) {
      if (!((p.slot_mask >> slot) & 1)) continue;
      const int sb = p.slot_begin[slot], se = p.slot_end[slot];
      const int w0 = xchg_share(sb, se, p.rank, p.world);
      const int w1 = xchg_share(sb, se, p.rank + 1, p.world);
      const int n_other = (se - sb) - (w1 - w0);
      const int e = threadIdx.x * 4;
#pragma unroll 1
      for (int i0 = static_cast<int>(blockIdx.x) * U2; i0 < n_other; i0 += static_cast<int>(gridDim.x) * U2) {
        uint2 sh[U2];
        float4 th[U2];
        long long dst[U2];          // byte offset inside the arenas (the same on every rank); -1 = nothing to do
        bool is_sh[U2];
#pragma unroll
        for (int u = 0; u < U2; ++u) {
          dst[u] = -1; is_sh[u] = false;
          const int j = i0 + u;
          if (j >= n_other) continue;
          const int w = sb + j + ((sb + j >= w0) ? (w1 - w0) : 0);
          int q = static_cast<int>((static_cast<long long>(w - sb) * p.world) / (se - sb));     // owner of run w: estimate, then fix up
          while (q + 1 < p.world && w >= xchg_share(sb, se, q + 1, p.world)) ++q;
          while (q > 0 && w < xchg_share(sb, se, q, p.world)) --q;
          const OptWork& wk = p.work[w];
          const bool vec = (wk.off & 3) == 0 && (wk.count & 3) == 0 &&
                           (wk.Wn == nullptr || ((wk.out_dim & 3) == 0 && ((wk.off - wk.mat_off) & 3) == 0 && (wk.ld_out & 3) == 0));
          const char* ob = p.peers->base[q];
          if (vec && wk.np == 1) {
            if (e < wk.count) {
              const long long idx = wk.off + e;
              if (wk.Wn != nullptr) {
                const long long m = idx - wk.mat_off;
                const long long r = m / wk.out_dim;
                dst[u] = (reinterpret_cast<char*>(wk.Wn) - my_base) + (r * wk.ld_out + (m - r * wk.out_dim)) * 2;
                is_sh[u] = true;
                asm volatile("ld.relaxed.sys.global.v2.u32 {%0, %1}, [%2];" : "=r"(sh[u].x), "=r"(sh[u].y) : "l"(ob + dst[u]) : "memory");
              } else {
                dst[u] = idx * 4;
                th[u] = ld_peer_f4(reinterpret_cast<const float*>(ob) + idx);
              }
            }
          } else {
            // odd widths / split-precision parts: element by element (parity modes, small layers)
            for (int i = 0; i < 4; ++i) {
              const int es = threadIdx.x + 256 * i;
              if (es >= wk.count) continue;
              const long long idx = wk.off + es;
              if (wk.Wn != nullptr) {
                const long long m = idx - wk.mat_off;
                const long long r = m / wk.out_dim;
                const long long rel = (reinterpret_cast<char*>(wk.Wn) - my_base) + (r * wk.ld_out + (m - r * wk.out_dim)) * 2;
                for (int part = 0; part < wk.np; ++part) {
                  unsigned short hv;
                  asm volatile("ld.relaxed.sys.global.u16 %0, [%1];" : "=h"(hv) : "l"(ob + rel + part * wk.part_stride * 2) : "memory");
                  *reinterpret_cast<unsigned short*>(my_base + rel + part * wk.part_stride * 2) = hv;
                }
              } else {
                theta[idx] = ld_peer_f1(reinterpret_cast<const float*>(ob) + idx);
              }
            }
          }
        }
#pragma unroll
        for (int u = 0; u < U2; ++u) {
          if (dst[u] < 0) continue;
          if (is_sh[u]) *reinterpret_cast<uint2*>(my_base + dst[u]) = sh[u];
          else *reinterpret_cast<float4*>(my_base + dst[u]) = th[u];
        }
      }
    }
  }
  __syncthreads();
  trace_end(p.trace);
}

// ------------------------------------------------------------------------------------------------------------------
// The same exchange with the flags INSIDE the data ("LL" protocol, as in NCCL): no arrive / updated flag, no fence, no
// load round trip - every transfer is a fire-and-forget P2P STORE of 16 bytes {d0, epoch, d1, epoch} (8 data bytes, each
// 8-byte half self-validating), and the receiver polls ITS OWN memory until both halves carry the step's epoch:
//
//   push    my gradient of every run somebody else owns  ->  the owner's  gbuf[me][...]
//   update  owned runs: own gradient + the peers' (polled from gbuf, summed in rank order), optimizer, local master /
//           state / shadow, and the new operand pushed to every peer's  sbuf[...]  (bf16 shadow: one 16-byte store per 4
//           parameters; runs without a shadow: fp32 theta, two stores)
//   gather  runs others own: poll sbuf, unpack into my shadow / theta
//
// The chain is  store latency (2.7 us) + 2 x bytes / bandwidth, twice - about half of the flag-and-pull protocol above,
// whose three fabric round trips cost ~27 us beside a GEMM however little data they moved (profiles/results_r02.md).
// Buffers (arena, behind the flag block): gbuf = world x n4 entries, sbuf = n4 entries of 32 bytes, entry i = parameters
// 4 i .. 4 i + 3 as four 8-byte units {value bits, epoch} (two 16-byte halves in two planes, see the kernel); a shadow
// entry uses the first half {2 x bf16, epoch, 2 x bf16, epoch}.
// Reuse is safe without any handshake: a sender overwrites gbuf / sbuf of step k only after it has left step k's
// exchange of that slot, which it can only do after the receiver has consumed the entry (the receiver's own pushes of
// step k, which the sender waited for, came after it).
struct LLParams {
  XchgParams x;
  long long llg_off, lls_off;     // byte offsets of gbuf / sbuf inside every arena
  long long n4;                   // entries per rank in gbuf
};

__device__ __forceinline__ void ll_store2(char* dst, unsigned int d0, unsigned int d1, unsigned int ep) {
  asm volatile("st.relaxed.sys.global.v4.u32 [%0], {%1, %2, %3, %4};" ::"l"(dst), "r"(d0), "r"(ep), "r"(d1), "r"(ep) : "memory");
}
__device__ __forceinline__ void ll_store1(char* dst, unsigned int d0, unsigned int ep) {
  asm volatile("st.relaxed.sys.global.v2.u32 [%0], {%1, %2};" ::"l"(dst), "r"(d0), "r"(ep) : "memory");
}
// poll one 16-byte LL pair until both halves carry `ep`; false after a timeout / failure elsewhere in the block
__device__ __forceinline__ bool ll_poll2(const char* src, unsigned int ep, unsigned int& d0, unsigned int& d1, const XchgParams& p,
                                         int slot, int from, unsigned int* sh_fail) {
  unsigned int f0, f1, spins = 0;
  unsigned long long t0 = 0;
  for (;;) {
    asm volatile("ld.relaxed.sys.global.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(d0), "=r"(f0), "=r"(d1), "=r"(f1) : "l"(src) : "memory");
    if (f0 == ep && f1 == ep) return true;
    __nanosleep(40);          // (a tight poll loop on every thread takes L2 bandwidth from the GEMM that shares the SM)
    if ((++spins & 0xFFFu) == 0) {
      if (*reinterpret_cast<volatile unsigned int*>(sh_fail)) return false;
      if (p.timeout_ns != 0) {
        const unsigned long long now = globaltimer_ns();
        if (t0 == 0) t0 = now;
        else if (now - t0 > p.timeout_ns) {
          if (p.host_err != nullptr) { atomicCAS(p.host_err, 0u, 1u + 16u * slot + from); __threadfence_system(); }
          *sh_fail = 1u;
          return false;
        }
      }
    }
  }
}
__device__ __forceinline__ bool ll_poll1(const char* src, unsigned int ep, unsigned int& d0, const XchgParams& p, int slot, int from,
                                         unsigned int* sh_fail) {
  unsigned int f0, spins = 0;
  unsigned long long t0 = 0;
  for (;;) {
    asm volatile("ld.relaxed.sys.global.v2.u32 {%0, %1}, [%2];" : "=r"(d0), "=r"(f0) : "l"(src) : "memory");
    if (f0 == ep) return true;
    __nanosleep(40);
    if ((++spins & 0xFFFu) == 0) {
      if (*reinterpret_cast<volatile unsigned int*>(sh_fail)) return false;
      if (p.timeout_ns != 0) {
        const unsigned long long now = globaltimer_ns();
        if (t0 == 0) t0 = now;
        else if (now - t0 > p.timeout_ns) {
          if (p.host_err != nullptr) { atomicCAS(p.host_err, 0u, 1u + 16u * slot + from); __threadfence_system(); }
          *sh_fail = 1u;
          return false;
        }
      }
    }
  }
}

__device__ __forceinline__ bool run_is_vec(const OptWork& wk) {
  return (wk.off & 3) == 0 && (wk.count & 3) == 0 &&
         (wk.Wn == nullptr || ((wk.out_dim & 3) == 0 && ((wk.off - wk.mat_off) & 3) == 0 && (wk.ld_out & 3) == 0));
}
__device__ __forceinline__ int run_owner(int w, int sb, int se, int world) {
  int q = static_cast<int>((static_cast<long long>(w - sb) * world) / (se - sb));
  while (q + 1 < world && w >= xchg_share(sb, se, q + 1, world)) ++q;
  while (q > 0 && w < xchg_share(sb, se, q, world)) --q;
  return q;
}

// plain-bf16 nets only (one shadow part).  One block per SM at most: no block ever waits for another block of its own
// grid, but it does wait for the peers' blocks, which must all be able to become resident beside whatever GEMM is running.
template <int W>
static __global__ void __launch_bounds__(256, W <= 8 ? 3 : 2)
xchg_ll_kernel(const LLParams lp) {
  const XchgParams& p = lp.x;
  __shared__ unsigned int sh_fail;
  if (threadIdx.x == 0) sh_fail = 0u;
  trace_begin(p.trace, true);
  pdl_wait();
  trace_begin(p.trace, false);
  __syncthreads();
  const unsigned int ep = p.desc->epoch;
  char* const my_base = p.peers->base[p.rank];
  float* const theta = reinterpret_cast<float*>(my_base);
  if (p.host_scal != nullptr && blockIdx.x == 0 && threadIdx.x < SCAL_COUNT) {
    p.host_scal[threadIdx.x] = p.scal[threadIdx.x];
    if (threadIdx.x == 0 && p.desc->hist != nullptr) *p.desc->hist = make_float2(p.scal[SCAL_LOSS_SUM], p.scal[SCAL_NNZ]);
    __threadfence_system();
  }
  const float lr_t = p.desc->lr_t, gs = p.desc->gscale;
  const bool use_s1 = p.hyper.kind != SB_OPT_SGD;
  const bool use_s2 = p.hyper.kind == SB_OPT_ADAM || p.hyper.kind == SB_OPT_ADADELTA;
  float* const s1 = reinterpret_cast<float*>(my_base + p.s1_off);
  float* const s2 = reinterpret_cast<float*>(my_base + p.s2_off);
  float* const my_grad = reinterpret_cast<float*>(my_base + p.grad_off);
  // entry i (parameters 4 i .. 4 i + 3) = 16 bytes {p0, ep, p1, ep} at i * 16 in the low plane + 16 bytes {p2, ep, p3, ep} at the
  // same offset in the high plane (n4 * 16 further): a warp's store instruction covers 512 contiguous bytes
  const long long hi_plane = lp.n4 * 16;
  const long long g_stride = lp.n4 * 32;                      // one sender's region of gbuf
  auto unit_off = [&](long long idx) { return ((idx & 2) ? hi_plane : 0ll) + (idx >> 2) * 16 + (idx & 1) * 8; };
  auto stamp_max = [&](int slot) { if (p.trace != nullptr && threadIdx.x == 0) atomicMax(p.trace + slot, static_cast<unsigned long long>(globaltimer_ns())); };
  const int e = threadIdx.x * 4;

  // ---- push: my gradient of the runs other ranks own ----
#pragma unroll 1
  for (int slot = 0; slot < p.n_slots; ++slot) {
    if (!((p.slot_mask >> slot) & 1)) continue;
    const int sb = p.slot_begin[slot], se = p.slot_end[slot];
    const int w0 = xchg_share(sb, se, p.rank, p.world), w1 = xchg_share(sb, se, p.rank + 1, p.world);
    const int n_other = (se - sb) - (w1 - w0);
    constexpr int UP = 4;
#pragma unroll 1
    for (int i0 = static_cast<int>(blockIdx.x) * UP; i0 < n_other; i0 += static_cast<int>(gridDim.x) * UP) {
      float4 g[UP];
      char* dst[UP];
#pragma unroll
      for (int u = 0; u < UP; ++u) {
        dst[u] = nullptr;
        const int j = i0 + u;
        if (j >= n_other) continue;
        const int w = sb + j + ((sb + j >= w0) ? (w1 - w0) : 0);
        const int q = run_owner(w, sb, se, p.world);
        const OptWork& wk = p.work[w];
        char* qb = p.peers->base[q] + lp.llg_off + p.rank * g_stride;
        if (run_is_vec(wk)) {
          if (e < wk.count) {
            g[u] = *reinterpret_cast<const float4*>(my_grad + wk.off + e);
            dst[u] = qb + ((wk.off + e) >> 2) * 16;
          }
        } else {
          for (int i = 0; i < 4; ++i) {
            const int es = threadIdx.x + 256 * i;
            if (es < wk.count) {
              const long long idx = wk.off + es;
              ll_store1(qb + unit_off(idx), __float_as_uint(my_grad[idx]), ep);
            }
          }
        }
      }
#pragma unroll
      for (int u = 0; u < UP; ++u) {
        if (dst[u] == nullptr) continue;
        ll_store2(dst[u], __float_as_uint(g[u].x), __float_as_uint(g[u].y), ep);
        ll_store2(dst[u] + hi_plane, __float_as_uint(g[u].z), __float_as_uint(g[u].w), ep);
      }
    }
  }
  if (p.trace != nullptr && blockIdx.x == 0 && threadIdx.x == 0) p.trace[3] = globaltimer_ns();
  stamp_max(7);

  // ---- update: owned runs ----
  bool alive = true;
#pragma unroll 1
  for (int slot = 0; slot < p.n_slots && alive; ++slot) {
    if (!((p.slot_mask >> slot) & 1)) continue;
    const int sb = p.slot_begin[slot], se = p.slot_end[slot];
    const int w0 = xchg_share(sb, se, p.rank, p.world), w1 = xchg_share(sb, se, p.rank + 1, p.world);
#pragma unroll 1
    for (int w = w0 + static_cast<int>(blockIdx.x); w < w1 && alive; w += static_cast<int>(gridDim.x)) {
      const OptWork wk = p.work[w];
      const long long shadow_rel = wk.Wn != nullptr ? reinterpret_cast<char*>(wk.Wn) - my_base : 0;
      if (run_is_vec(wk)) {
        if (e < wk.count) {
          const long long idx = wk.off + e;
          const float4 own = *reinterpret_cast<const float4*>(my_grad + idx);
          const float4 th = *reinterpret_cast<const float4*>(theta + idx);
          float4 a = use_s1 ? *reinterpret_cast<const float4*>(s1 + idx) : make_float4(0.f, 0.f, 0.f, 0.f);
          float4 b = use_s2 ? *reinterpret_cast<const float4*>(s2 + idx) : make_float4(0.f, 0.f, 0.f, 0.f);
          float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
          const char* src = my_base + lp.llg_off + (idx >> 2) * 16;
          // the peers' entries are polled four ranks at a time with all loads of an attempt in flight together (one L2
          // latency per attempt instead of one per rank), then added in rank order -> the same bits wherever a sum is computed
#pragma unroll
          for (int q0 = 0; q0 < W; q0 += 4) {
            if (q0 >= p.world || !alive) break;
            uint4 lo[4], hi[4];
            unsigned int spins = 0;
            unsigned long long t0 = 0;
            for (;;) {
              bool ok = true;
#pragma unroll
              for (int k = 0; k < 4; ++k) {
                const int q = q0 + k;
                if (q < W && q < p.world && q != p.rank) {
                  asm volatile("ld.relaxed.sys.global.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(lo[k].x), "=r"(lo[k].y), "=r"(lo[k].z), "=r"(lo[k].w) : "l"(src + q * g_stride) : "memory");
                  asm volatile("ld.relaxed.sys.global.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(hi[k].x), "=r"(hi[k].y), "=r"(hi[k].z), "=r"(hi[k].w) : "l"(src + q * g_stride + hi_plane) : "memory");
                }
              }
#pragma unroll
              for (int k = 0; k < 4; ++k) {
                const int q = q0 + k;
                if (q < W && q < p.world && q != p.rank) ok = ok && lo[k].y == ep && lo[k].w == ep && hi[k].y == ep && hi[k].w == ep;
              }
              if (ok) break;
              __nanosleep(40);
              if ((++spins & 0xFFFu) == 0) {
                if (*reinterpret_cast<volatile unsigned int*>(&sh_fail)) { alive = false; break; }
                if (p.timeout_ns != 0) {
                  const unsigned long long now = globaltimer_ns();
                  if (t0 == 0) t0 = now;
                  else if (now - t0 > p.timeout_ns) {
                    int missing = q0;
                    for (int k = 0; k < 4; ++k) {
                      const int q = q0 + k;
                      if (q < W && q < p.world && q != p.rank && !(lo[k].y == ep && lo[k].w == ep && hi[k].y == ep && hi[k].w == ep)) { missing = q; break; }
                    }
                    if (p.host_err != nullptr) { atomicCAS(p.host_err, 0u, 1u + 16u * slot + missing); __threadfence_system(); }
                    sh_fail = 1u;
                    alive = false;
                    break;
                  }
                }
              }
            }
            if (!alive) break;
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              const int q = q0 + k;
              if (q >= W || q >= p.world) break;
              const float4 v = (q == p.rank) ? own
                                             : make_float4(__uint_as_float(lo[k].x), __uint_as_float(lo[k].z), __uint_as_float(hi[k].x), __uint_as_float(hi[k].z));
              if (q == 0) acc = v; else { acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w; }
            }
          }
          if (alive) {
            float4 t;
            t.x = opt_update(p.hyper, lr_t, th.x, acc.x * gs, a.x, b.x);
            t.y = opt_update(p.hyper, lr_t, th.y, acc.y * gs, a.y, b.y);
            t.z = opt_update(p.hyper, lr_t, th.z, acc.z * gs, a.z, b.z);
            t.w = opt_update(p.hyper, lr_t, th.w, acc.w * gs, a.w, b.w);
            *reinterpret_cast<float4*>(theta + idx) = t;
            *reinterpret_cast<float4*>(my_grad + idx) = acc;      // the owner keeps the reduced gradient of its runs (parity hook)
            if (use_s1) *reinterpret_cast<float4*>(s1 + idx) = a;
            if (use_s2) *reinterpret_cast<float4*>(s2 + idx) = b;
            const long long sent = lp.lls_off + (idx >> 2) * 16;
            if (wk.Wn != nullptr) {
              const long long m = idx - wk.mat_off;
              const long long r = m / wk.out_dim;
              uint2 o;
              o.x = pack_bf16x2(t.x, t.y);
              o.y = pack_bf16x2(t.z, t.w);
              *reinterpret_cast<uint2*>(my_base + shadow_rel + (r * wk.ld_out + (m - r * wk.out_dim)) * 2) = o;
#pragma unroll
              for (int q = 0; q < W; ++q)
                if (q < p.world && q != p.rank) ll_store2(p.peers->base[q] + sent, o.x, o.y, ep);
            } else {
#pragma unroll
              for (int q = 0; q < W; ++q)
                if (q < p.world && q != p.rank) {
                  ll_store2(p.peers->base[q] + sent, __float_as_uint(t.x), __float_as_uint(t.y), ep);
                  ll_store2(p.peers->base[q] + sent + hi_plane, __float_as_uint(t.z), __float_as_uint(t.w), ep);
                }
            }
          }
        }
      } else {
#pragma unroll 1
        for (int i = 0; i < 4 && alive; ++i) {
          const int es = threadIdx.x + 256 * i;
          if (es >= wk.count) continue;
          const long long idx = wk.off + es;
          const long long uoff = unit_off(idx);
          float acc = 0.f;
          for (int q = 0; q < p.world; ++q) {
            float v = my_grad[idx];
            if (q != p.rank) {
              unsigned int d0;
              if (!ll_poll1(my_base + lp.llg_off + q * g_stride + uoff, ep, d0, p, slot, q, &sh_fail)) { alive = false; break; }
              v = __uint_as_float(d0);
            }
            acc = (q == 0) ? v : acc + v;
          }
          if (!alive) break;
          float a = use_s1 ? s1[idx] : 0.f, b = use_s2 ? s2[idx] : 0.f;
          const float t = opt_update(p.hyper, lr_t, theta[idx], acc * gs, a, b);
          theta[idx] = t;
          my_grad[idx] = acc;
          if (use_s1) s1[idx] = a;
          if (use_s2) s2[idx] = b;
          unsigned int bits = __float_as_uint(t);
          if (wk.Wn != nullptr) {
            const long long m = idx - wk.mat_off;
            const long long r = m / wk.out_dim;
            const __nv_bfloat16 hv = __float2bfloat16_rn(t);
            *reinterpret_cast<__nv_bfloat16*>(my_base + shadow_rel + (r * wk.ld_out + (m - r * wk.out_dim)) * 2) = hv;
            bits = static_cast<unsigned int>(*reinterpret_cast<const unsigned short*>(&hv));
          }
          for (int q = 0; q < p.world; ++q)
            if (q != p.rank) ll_store1(p.peers->base[q] + lp.lls_off + uoff, bits, ep);
        }
      }
    }
  }
  stamp_max(4);

  // ---- gather: runs other ranks own ----
#pragma unroll 1
  for (int slot = 0; slot < p.n_slots && alive; ++slot) {
    if (!((p.slot_mask >> slot) & 1)) continue;
    const int sb = p.slot_begin[slot], se = p.slot_end[slot];
    const int w0 = xchg_share(sb, se, p.rank, p.world), w1 = xchg_share(sb, se, p.rank + 1, p.world);
    const int n_other = (se - sb) - (w1 - w0);
#pragma unroll 1
    for (int j = static_cast<int>(blockIdx.x); j < n_other && alive; j += static_cast<int>(gridDim.x)) {
      const int w = sb + j + ((sb + j >= w0) ? (w1 - w0) : 0);
      const int q = run_owner(w, sb, se, p.world);
      const OptWork wk = p.work[w];
      const long long shadow_rel = wk.Wn != nullptr ? reinterpret_cast<char*>(wk.Wn) - my_base : 0;
      if (run_is_vec(wk)) {
        if (e < wk.count) {
          const long long idx = wk.off + e;
          const char* src = my_base + lp.lls_off + (idx >> 2) * 16;
          unsigned int d0, d1, d2, d3;
          if (!ll_poll2(src, ep, d0, d1, p, slot, q, &sh_fail)) { alive = false; break; }
          if (wk.Wn != nullptr) {
            const long long m = idx - wk.mat_off;
            const long long r = m / wk.out_dim;
            *reinterpret_cast<uint2*>(my_base + shadow_rel + (r * wk.ld_out + (m - r * wk.out_dim)) * 2) = make_uint2(d0, d1);
          } else {
            if (!ll_poll2(src + hi_plane, ep, d2, d3, p, slot, q, &sh_fail)) { alive = false; break; }
            *reinterpret_cast<float4*>(theta + idx) = make_float4(__uint_as_float(d0), __uint_as_float(d1), __uint_as_float(d2), __uint_as_float(d3));
          }
        }
      } else {
        for (int i = 0; i < 4 && alive; ++i) {
          const int es = threadIdx.x + 256 * i;
          if (es >= wk.count) continue;
          const long long idx = wk.off + es;
          unsigned int d0;
          if (!ll_poll1(my_base + lp.lls_off + unit_off(idx), ep, d0, p, slot, q, &sh_fail)) { alive = false; break; }
          if (wk.Wn != nullptr) {
            const long long m = idx - wk.mat_off;
            const long long r = m / wk.out_dim;
            *reinterpret_cast<unsigned short*>(my_base + shadow_rel + (r * wk.ld_out + (m - r * wk.out_dim)) * 2) = static_cast<unsigned short>(d0);
          } else {
            theta[idx] = __uint_as_float(d0);
          }
        }
      }
    }
  }
  __syncthreads();
  trace_end(p.trace);
}

// Refresh the stale parts of a non-owner's fp32 master and optimizer state from the owners (before the host reads them);
// what = 1: the reduced gradient instead (each owner kept the sum of its runs).
// Every run is pulled from its owner unless this rank owns it.  One block per work item.
static __global__ void __launch_bounds__(256)
gather_master_kernel(const XchgParams p, int what) {
  const int w = blockIdx.x;
  float* const theta = reinterpret_cast<float*>(p.peers->base[p.rank]);
  int owner = -1;
  for (int slot = 0; slot < p.n_slots; ++slot) {
    if (w >= p.slot_begin[slot] && w < p.slot_end[slot]) {
      for (int r = 0; r < p.world; ++r)
        if (w >= xchg_share(p.slot_begin[slot], p.slot_end[slot], r, p.world) && w < xchg_share(p.slot_begin[slot], p.slot_end[slot], r + 1, p.world)) owner = r;
    }
  }
  if (owner < 0 || owner == p.rank) return;
  const OptWork wk = p.work[w];
  char* const my_base = p.peers->base[p.rank];
  const char* ob = p.peers->base[owner];
  for (int e = threadIdx.x; e < wk.count; e += 256) {
    const long long idx = wk.off + e;
    if (what == 1) {
      reinterpret_cast<float*>(my_base + p.grad_off)[idx] = ld_peer_f1(reinterpret_cast<const float*>(ob + p.grad_off) + idx);
      continue;
    }
    theta[idx] = ld_peer_f1(reinterpret_cast<const float*>(ob) + idx);
    reinterpret_cast<float*>(my_base + p.s1_off)[idx] = ld_peer_f1(reinterpret_cast<const float*>(ob + p.s1_off) + idx);
    reinterpret_cast<float*>(my_base + p.s2_off)[idx] = ld_peer_f1(reinterpret_cast<const float*>(ob + p.s2_off) + idx);
  }
}

}  // namespace sb
