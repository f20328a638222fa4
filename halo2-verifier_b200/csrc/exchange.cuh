// Device-side exchange of a sharded batch (SURVEY.md 8e): one process per GPU, every rank's context owns a WINDOW
// in its HBM that the peers map (CUDA IPC over NVLink / NVSwitch).  No host and no library collective sits in the
// data path: the kernel that packs a shard's per-window sums stores them straight into the ROOT rank's window and
// publishes a sequence number; the root's summing kernel waits for the sequence numbers of all ranks, reads the partials
// in place, runs the pairing checks and stores the verdicts into every rank's window; each rank's last kernel waits
// for them.  A gather (only the root receives data), not an all-gather.  All of it is part of the captured CUDA graph.
//
// Window layout (one cudaMalloc, so one IPC handle):
//   [0, 256)                         XHeader { vseq, ... }     vseq: sequence number of the verdicts below (root -> here)
//   [256, 256 + 8 * XCH_MAX_RANKS)   u64 arrive[rank]          sequence number of the partial rank r stored here
//   [.., + 4 * (max_groups + 4))     u32 verdicts[max_groups] | root_status
//   [partials_off, ...)              partials[rank][max_groups] of H2V_PARTIAL_BYTES
// Ordering: data stores, __threadfence_system(), then st.release.sys of the sequence number; the reader spins with
// ld.acquire.sys.  Every wait has a timeout (globaltimer) and raises a flag instead of hanging the GPU.
#pragma once
#include "curve.cuh"

namespace h2v {

static constexpr u32 XCH_MAX_RANKS = 128;  // k_sum_partials adds at most 128 partials
static constexpr u32 XCH_HDR_BYTES = 256;
static constexpr u32 XCH_PARTIAL_BYTES = 12320;  // == H2V_PARTIAL_BYTES (static_assert in kernels.cu)

struct XHeader {
  u64 vseq;  // written by the root of launch set `vseq` after its verdict words
  u64 rsv[31];
};
static_assert(sizeof(XHeader) == XCH_HDR_BYTES, "window header");

// per launch set, copied to the device right before the graph launch (the graph itself is static)
struct XDyn {
  u64 seq;         // launch-set counter of this channel: the same on every rank, strictly increasing from 1
  u32 root;        // rank whose window receives the partials and which runs the pairing checks
  u32 rsv;
  u64 timeout_ns;  // bound of every device-side wait
};

struct XLayout {
  u32 rank, world, max_groups, rsv;
  H2V_HD size_t arrive_off() const { return XCH_HDR_BYTES; }
  H2V_HD size_t verdict_off() const { return XCH_HDR_BYTES + 8 * (size_t)XCH_MAX_RANKS; }
  H2V_HD size_t partials_off() const { return (verdict_off() + 4 * ((size_t)max_groups + 4) + 255) & ~(size_t)255; }
  H2V_HD size_t bytes() const { return partials_off() + (size_t)world * max_groups * XCH_PARTIAL_BYTES; }
};

#if defined(__CUDACC__)
__device__ __forceinline__ void st_release_sys(u64* p, u64 v) { asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory"); }
__device__ __forceinline__ u64 ld_acquire_sys(const u64* p) {
  u64 v;
  asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ u32 ld_relaxed_sys(const u32* p) {
  u32 v;
  asm volatile("ld.relaxed.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ u64 global_ns() {
  u64 t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
// waits until *p >= want; false on timeout
__device__ __forceinline__ bool spin_until_ge(const u64* p, u64 want, u64 timeout_ns) {
  if (ld_acquire_sys(p) >= want) return true;
  const u64 t0 = global_ns();
  for (;;) {
    __nanosleep(100);
    if (ld_acquire_sys(p) >= want) return true;
    if (global_ns() - t0 > timeout_ns) return false;
  }
}

// (The header of a partial carries its window bits and window count, not whether the windows came from a GLV split: the
// window sums of a split scalar keep their meaning, sum_w 2^(c w) S_w = sum k P, and every rank derives the same geometry
// from the same batch shape, so partials of equal (c, W) add up either way.)
// Packs the window sums of fold group blockIdx.x into a partial (32-byte header + 128 Jacobian slots) and stores it
// into slot [rank][group] of the ROOT's window (peer memory over NVLink; the root's own window when rank == root);
// the last block to finish publishes this rank's sequence number there.  16-byte stores.
__global__ void __launch_bounds__(256) k_pack_partial_x(u32 cbits, u32 windows, u32 npts, const G1Jac* __restrict__ wsums, const XDyn* __restrict__ dyn,
                                                        u8* const* __restrict__ peers, XLayout lay, u32* done) {
  asm volatile("griddepcontrol.wait;" ::: "memory");
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  const u32 g = blockIdx.x, t = threadIdx.x;
  const u64 seq = dyn->seq;
  u8* root = peers[dyn->root];
  uint4* o = (uint4*)(root + lay.partials_off() + ((size_t)lay.rank * lay.max_groups + g) * XCH_PARTIAL_BYTES);
  const uint4* src = (const uint4*)(wsums + (size_t)g * npts);
  if (t == 0) {
    o[0] = make_uint4(0x50563248u, cbits, windows, npts);  // H2V_PARTIAL_MAGIC
    o[1] = make_uint4(0, 0, 0, 0);
  }
  const u32 live = npts * (u32)(sizeof(G1Jac) / 16);
  for (u32 i = t; i < (XCH_PARTIAL_BYTES - 32) / 16; i += 256) o[2 + i] = i < live ? src[i] : make_uint4(0, 0, 0, 0);
  __threadfence_system();
  __syncthreads();
  if (t == 0) {
    const u32 prev = atomicAdd(done, 1u);
    if (prev == gridDim.x - 1) {  // every block's stores are ordered before this point (fence + atomic)
      *done = 0;
      __threadfence_system();
      st_release_sys((u64*)(root + lay.arrive_off()) + lay.rank, seq);
    }
  }
}

// Root: verdict words of this launch set -> every rank's window, then the sequence number (warp per rank).
// *status = the root's error bits (k_sum_partials: 1 = a partial never arrived, 2 = window geometries differ); they
// travel with the verdicts so that every rank fails alike, and a failed exchange never reads as "accepted".
__global__ void __launch_bounds__(256) k_bcast_verdict(const XDyn* __restrict__ dyn, u8* const* __restrict__ peers, XLayout lay, u32 groups,
                                                       const u32* __restrict__ verdict, const u32* __restrict__ status) {
  const u32 lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = blockDim.x >> 5;
  const u64 seq = dyn->seq;
  const u32 st = *status;
  for (u32 r = wid; r < lay.world; r += nw) {
    u8* w = peers[r];
    u32* vd = (u32*)(w + lay.verdict_off());
    for (u32 g = lane; g < groups; g += 32) vd[g] = st ? 0u : verdict[g];
    if (lane == 0) vd[lay.max_groups] = st;
    __threadfence_system();
    __syncwarp();
    if (lane == 0) st_release_sys(&((XHeader*)w)->vseq, seq);
  }
}

// Every rank: waits for the verdicts of this launch set in its own window and copies them next to the batch
// (out[0..groups) verdicts, out[groups] |= 4 when the wait timed out, out[groups + 1] = root's status word).
__global__ void __launch_bounds__(64) k_wait_verdict(const XDyn* __restrict__ dyn, const u8* __restrict__ window, XLayout lay, u32 groups, u32* out) {
  __shared__ u32 ok;
  if (threadIdx.x == 0) ok = spin_until_ge(&((const XHeader*)window)->vseq, dyn->seq, dyn->timeout_ns) ? 1u : 0u;
  __syncthreads();
  const u32* vd = (const u32*)(window + lay.verdict_off());
  for (u32 g = threadIdx.x; g < groups; g += 64) out[g] = ok ? ld_relaxed_sys(vd + g) : 0u;
  if (threadIdx.x == 0) {
    if (!ok) atomicOr(out + groups, 4u);  // bit 2: the verdicts never arrived (bit 0: a partial never arrived, k_sum_partials)
    out[groups + 1] = ok ? ld_relaxed_sys(vd + lay.max_groups) : 0u;
  }
}
#endif

}  // namespace h2v
