// Multi-GPU tail of the ADVI step as ONE kernel over NVLink peer memory (sm_100a):
//     reduce-scatter of the data-term gradients  ->  Adam  ->  all-gather of the updated parameters.
//
// Row-sharded data parallelism (SURVEY.md 8e; the reference carries only an unused tf.distribute
// `strategy` hook, poisson.py:60,72,82-83) leaves every rank with a partial gradient of the 8
// data-touched tensors (v, w, u, s: loc | scale) and identical copies of everything else.  Instead
// of  ncclAllReduce(10.7 MB at C4) -> unpack -> Adam on every rank (every rank repeating the same
// 2.7 M Adam updates), rank r here
//   1. signals "my gradients are final" into every peer's flag page and waits for all peers,
//   2. for ITS 1/world slice of the block: loads the slice of every rank's gradient buffer through the
//      peer mappings (16-byte loads over NVLink / NVSwitch), adds them in rank order 0..world-1 (one fixed
//      order, one owner per element: replicas cannot diverge), applies Adam to its local (params, m, v)
//      -- the moments of an element live on its owner only -- and stores the new parameter value into
//      EVERY rank's parameter buffer,
//   3. applies Adam to the replicated tensors locally (deterministic kernels => bit-identical everywhere;
//      skipped when the step already did it under its data term: spmf_step_args.adam_tail_early),
//   4. folds the per-draw ('z','x') partial sums of all ranks into the loss parts (all ranks, rank order),
//   5. signals "my stores are out" and leaves when every peer has said the same: from then on this
//      rank's parameter buffer is complete and its gradient buffer is free to be overwritten.
// No CTA waits on another CTA of its own grid (only on remote flags), so the grid need not be co-resident.
// Waits are bounded (kSpinLimit): a peer that never arrives makes the kernel give up with status = 1
// instead of hanging the device.
//
// Buffers: gradient + parameter + flag pages are cudaMalloc'ed by spmf_p2p_alloc and mapped into the
// peers with CUDA IPC (one process per GPU); the host exchanges the 64-byte handles once
// (torch.distributed all_gather_object in spmf_b200/parallel.py).
#include <cuda_runtime.h>
#include <stdint.h>
#include <string.h>

#include "../../include/spmf_b200.h"
#include "spmf_model.cuh"

namespace spmf {

#define SPMF_CHECK_LAUNCH()                      \
  do {                                           \
    cudaError_t e__ = cudaGetLastError();        \
    if (e__ != cudaSuccess) return (int)e__;     \
  } while (0)

constexpr long long kSpinLimit = 20000000000LL;     // clock64 ticks (~10 s): give up, do not hang the device
constexpr int kFlagReady = 0, kFlagDone = 32, kFlagCount = 64, kFlagStatus = 65;     // words of a flag page

__device__ __forceinline__ void st_release_sys(unsigned* p, unsigned v) {
  asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ unsigned ld_acquire_sys(const unsigned* p) {
  unsigned v;
  asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
// wrap-safe "flag has reached epoch"
__device__ __forceinline__ bool reached(unsigned flag, unsigned epoch) { return (int)(flag - epoch) >= 0; }

// float4 vectors [v0, v1) of the reduced block (nvec vectors) whose sum, Adam update and moments belong to
// `rank`: ceil(nvec / world) consecutive vectors per rank, in rank order.  The exchange kernel and
// spmf_p2p_owned_range (checkpoints gather the moments by it) both use this one definition.  (`rank` by
// reference: the kernel then reads a.rank where the product needs it, and compiles to the same SASS as with
// the formula written inline.)
__host__ __device__ __forceinline__ void owned_vecs(long long nvec, int world, const int& rank, long long* v0,
                                                   long long* v1) {
  const long long per = (nvec + world - 1) / world;
  *v0 = min(nvec, per * rank);
  *v1 = min(nvec, *v0 + per);
}

struct P2PArgs {
  int world, rank, S, slack;
  unsigned epoch;
  int skip_tail;
  long long n_params, n_block, comm_off;      // floats: whole buffer, reduced block (slack at its end), slack offset
  double w_entropy, w_prior;
  float* grads[SPMF_P2P_MAX_WORLD];
  float* params[SPMF_P2P_MAX_WORLD];
  unsigned* flags[SPMF_P2P_MAX_WORLD];
  double* parts;
  double* loss_out;
  AdamCfg adam;                                 // p = params[rank]
};

// lane q < world of the calling warp: wait until flags[rank][base + q] has reached epoch
__device__ bool wait_all(const P2PArgs& a, int base, int q) {
  bool ok = true;
  if (q < a.world) {
    const unsigned* f = a.flags[a.rank] + base + q;
    const long long t0 = clock64();
    while (!reached(ld_acquire_sys(f), a.epoch)) {
      if (clock64() - t0 > kSpinLimit) { ok = false; break; }
      __nanosleep(64);
    }
  }
  return __all_sync(0xffffffffu, ok);
}

__global__ void __launch_bounds__(256)
p2p_reduce_adam_kernel(const P2PArgs a) {
  __shared__ int s_ok;
  unsigned* myflags = a.flags[a.rank];
  const int W = a.world;
  // ---- 1. my gradients are final (stream order: the backward kernels completed before this launch)
  if (threadIdx.x < 32) {
    if (blockIdx.x == 0 && threadIdx.x < W) {
      __threadfence_system();
      st_release_sys(a.flags[threadIdx.x] + kFlagReady + a.rank, a.epoch);
    }
    const bool ok = wait_all(a, kFlagReady, threadIdx.x);
    if (threadIdx.x == 0) s_ok = ok ? 1 : 0;
  }
  __syncthreads();
  const bool live = s_ok != 0;
  if (!live && threadIdx.x == 0) atomicExch(myflags + kFlagStatus, 1u);

  const long long tid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long nthr = (long long)gridDim.x * blockDim.x;
  if (live) {
    // ---- 2. my slice of the reduced block, 4 floats at a time
    const long long nvec = a.comm_off / 4;                      // (comm_off is a multiple of 4: checked on the host)
    long long v0, v1;
    owned_vecs(nvec, W, a.rank, &v0, &v1);
    for (long long i = v0 + tid; i < v1; i += nthr) {
      float4 g[SPMF_P2P_MAX_WORLD];
#pragma unroll
      for (int q = 0; q < SPMF_P2P_MAX_WORLD; ++q)
        if (q < W) g[q] = __ldcg(reinterpret_cast<const float4*>(a.grads[q]) + i);   // all loads in flight at once
      float4 s = g[0];
#pragma unroll
      for (int q = 1; q < SPMF_P2P_MAX_WORLD; ++q)
        if (q < W) { s.x += g[q].x; s.y += g[q].y; s.z += g[q].z; s.w += g[q].w; }
      float4 p;
      if (a.adam.lr > 0.f) {
        adam_apply(a.adam, 4 * i + 0, s.x);
        adam_apply(a.adam, 4 * i + 1, s.y);
        adam_apply(a.adam, 4 * i + 2, s.z);
        adam_apply(a.adam, 4 * i + 3, s.w);
      }
      p = reinterpret_cast<const float4*>(a.adam.p)[i];
#pragma unroll
      for (int q = 0; q < SPMF_P2P_MAX_WORLD; ++q)
        if (q < W && q != a.rank) reinterpret_cast<float4*>(a.params[q])[i] = p;
    }
    // ---- 3. replicated tensors: local Adam
    if (a.adam.lr > 0.f && !a.skip_tail)
      for (long long i = a.n_block + tid; i < a.n_params; i += nthr) adam_apply(a.adam, i, a.grads[a.rank][i]);
    // ---- 4. loss parts: ('z','x') as (hi, lo) float pairs, summed over the ranks in rank order
    if (blockIdx.x == gridDim.x - 1) {
      __shared__ double sl[64];
      const int s = threadIdx.x;
      double l = 0.0;
      if (s < a.S) {
        double zz = 0.0, xx = 0.0;
        for (int q = 0; q < W; ++q) {
          const float4 c = __ldcg(reinterpret_cast<const float4*>(a.grads[q] + a.comm_off) + s);
          zz += (double)c.x + (double)c.y;
          xx += (double)c.z + (double)c.w;
        }
        double* o = a.parts + (long long)s * NUM_PARTS;
        o[P_Z] = zz;
        o[P_X] = xx;
        double prior = 0.0;
        for (int p = 0; p < P_LOGQ; ++p) prior += o[p];
        l = a.w_entropy * o[P_LOGQ] - a.w_prior * prior - zz - xx;
        o[15] = l;
      }
      if (s < 64) sl[s] = l;
      __syncthreads();
      if (s == 0) {
        double t = 0.0;
        for (int i = 0; i < a.S && i < 64; ++i) t += sl[i];
        *a.loss_out = t / (double)a.S;
      }
    }
  }
  // ---- 5. the last CTA of this rank to get here tells the peers, waits for them, re-arms the slack
  __syncthreads();
  __shared__ int s_last;
  if (threadIdx.x == 0) {
    __threadfence_system();                                      // this CTA's peer stores before the count
    s_last = (atomicAdd(myflags + kFlagCount, 1u) == gridDim.x - 1) ? 1 : 0;
  }
  __syncthreads();
  if (!s_last) return;
  if (threadIdx.x < 32) {
    if (threadIdx.x == 0) {
      __threadfence_system();
      myflags[kFlagCount] = 0u;                                  // re-armed for the next call
    }
    __syncwarp();
    if (threadIdx.x < W) st_release_sys(a.flags[threadIdx.x] + kFlagDone + a.rank, a.epoch);
    const bool ok = wait_all(a, kFlagDone, threadIdx.x);
    if (!ok && threadIdx.x == 0) atomicExch(myflags + kFlagStatus, 1u);
  }
  __syncthreads();
  // every peer has read my gradients: the scalar slack is accumulated into (atomics), so it is zeroed here
  float* slack = a.grads[a.rank] + a.comm_off;
  for (int i = threadIdx.x; i < a.slack; i += blockDim.x) slack[i] = 0.f;
}

}  // namespace spmf

using namespace spmf;

extern "C" {

int spmf_p2p_alloc(long long bytes, void** ptr) {
  if (bytes <= 0 || !ptr) return SPMF_ERR_BAD_ARG;
  cudaError_t e = cudaMalloc(ptr, (size_t)bytes);
  if (e != cudaSuccess) return (int)e;
  e = cudaMemset(*ptr, 0, (size_t)bytes);
  return e == cudaSuccess ? SPMF_OK : (int)e;
}

int spmf_p2p_free(void* ptr) { return ptr ? (int)cudaFree(ptr) : SPMF_OK; }

int spmf_p2p_export(void* ptr, unsigned char* handle64) {
  if (!ptr || !handle64) return SPMF_ERR_BAD_ARG;
  static_assert(sizeof(cudaIpcMemHandle_t) == SPMF_P2P_HANDLE_BYTES, "IPC handle size");
  cudaIpcMemHandle_t h;
  cudaError_t e = cudaIpcGetMemHandle(&h, ptr);
  if (e != cudaSuccess) return (int)e;
  memcpy(handle64, &h, sizeof(h));
  return SPMF_OK;
}

int spmf_p2p_open(const unsigned char* handle64, void** ptr) {
  if (!handle64 || !ptr) return SPMF_ERR_BAD_ARG;
  cudaIpcMemHandle_t h;
  memcpy(&h, handle64, sizeof(h));
  cudaError_t e = cudaIpcOpenMemHandle(ptr, h, cudaIpcMemLazyEnablePeerAccess);
  return e == cudaSuccess ? SPMF_OK : (int)e;
}

int spmf_p2p_close(void* ptr) { return ptr ? (int)cudaIpcCloseMemHandle(ptr) : SPMF_OK; }

long long spmf_p2p_flag_bytes(void) { return 4096; }

int spmf_p2p_owned_range(long long comm_off, int world, int rank, long long* lo, long long* hi) {
  if (comm_off < 0 || (comm_off & 3) || world < 1 || world > SPMF_P2P_MAX_WORLD || rank < 0 || rank >= world || !lo || !hi)
    return SPMF_ERR_BAD_ARG;
  long long v0, v1;
  owned_vecs(comm_off / 4, world, rank, &v0, &v1);
  *lo = 4 * v0;
  *hi = 4 * v1;
  return SPMF_OK;
}

int spmf_p2p_status(const void* flags, void* stream) {
  // host-synchronous read of the give-up flag (diagnostics; not on the step path)
  unsigned v = 0;
  cudaError_t e = cudaMemcpyAsync(&v, (const unsigned*)flags + kFlagStatus, 4, cudaMemcpyDeviceToHost, (cudaStream_t)stream);
  if (e != cudaSuccess) return (int)e;
  e = cudaStreamSynchronize((cudaStream_t)stream);
  if (e != cudaSuccess) return (int)e;
  return v ? SPMF_ERR_PEER_TIMEOUT : SPMF_OK;
}

int spmf_p2p_reduce_adam(const spmf_p2p_args* x, void* stream) {
  if (!x || x->world < 2 || x->world > SPMF_P2P_MAX_WORLD || x->rank < 0 || x->rank >= x->world) return SPMF_ERR_BAD_ARG;
  if (x->S <= 0 || x->S > 64 || x->slack < 4 * x->S || x->comm_off <= 0 || (x->comm_off & 3) ||
      x->n_block != x->comm_off + x->slack || x->n_params < x->n_block || !x->parts || !x->loss_out || !x->adam)
    return SPMF_ERR_BAD_ARG;
  P2PArgs a{};
  a.world = x->world; a.rank = x->rank; a.S = x->S; a.slack = x->slack; a.epoch = x->epoch; a.skip_tail = x->skip_tail;
  a.n_params = x->n_params; a.n_block = x->n_block; a.comm_off = x->comm_off;
  a.w_entropy = x->w_entropy; a.w_prior = x->w_prior;
  for (int q = 0; q < x->world; ++q) {
    if (!x->grads[q] || !x->params[q] || !x->flags[q]) return SPMF_ERR_BAD_ARG;
    if ((reinterpret_cast<uintptr_t>(x->grads[q]) | reinterpret_cast<uintptr_t>(x->params[q])) & 15) return SPMF_ERR_BAD_ARG;
    a.grads[q] = x->grads[q]; a.params[q] = x->params[q]; a.flags[q] = (unsigned*)x->flags[q];
  }
  a.parts = x->parts; a.loss_out = x->loss_out;
  spmf_adam_args ad = *x->adam;
  if (ad.params != x->params[x->rank]) return SPMF_ERR_BAD_ARG;
  a.adam = make_adam_cfg(&ad);
  // enough CTAs to keep a few hundred KB of peer loads in flight per SM; capped so that the tail barrier stays short
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  p2p_reduce_adam_kernel<<<2 * sms, 256, 0, (cudaStream_t)stream>>>(a);
  SPMF_CHECK_LAUNCH();
  return SPMF_OK;
}

}  // extern "C"
