// allreduce.cu — the data-parallel hot path: per-step DDP gradient-bucket allreduce across the
// job's replicas, fused with the bucket cast/scale, hand-written for sm_100a.
//
// Replaces (reference side, third-party): DDP default comm hook `tensor.div_(N)` + `all_reduce`
// (torch/distributed/algorithms/ddp_comm_hooks/default_hooks.py:18-33), the compress hooks' cast +
// scale (:57-92) and ProcessGroupGloo/NCCL::allreduce, which the reference operator only configures
// (controllers/train/torchjob_controller.go:394-446).
//
// Semantics (all algorithms, every replica bit-identical):
//     wire_r[i] = cast_wire( f32(in_r[i]) * pre )                pre  = scale (PRE) or 1 (POST)
//     acc[i]    = f32(wire_0[i]) + f32(wire_1[i]) + ... (rank order, fp32)
//     out[i]    = cast_out( f32( cast_wire( acc[i] * post ) ) )  post = 1 (PRE) or scale (POST)
// (NVLS: the switch performs the fp32-accumulated sum; its order is unspecified.)
//
// Kernels (one launch per bucket, 512 threads/CTA, CTA b of every replica owns the same slab of
// 16-byte packs so that all cross-replica dependencies are between same-index CTAs and a per-CTA
// flag barrier in peer HBM is sufficient — no grid-wide sync):
//   local      (world 1)  out = cast(in*scale): HBM-bound, one even wave of CTAs (LDG.128 x 8 in
//              flight per thread), or — same dtype — cp.async.bulk (TMA) through a shared-memory ring
//   one-shot   push wire packs into slot[rank] of every peer's staging buffer; barrier; reduce the
//              `world` local slots                                              1 barrier, (N-1)S out
//   two-shot   stage locally; barrier; replica r reduces sub-slab r from all peers (LDG.128 over
//              NVLink, all peers in flight), writes it back in place; barrier; pull the other
//              sub-slabs                                                  2 barriers, 2(N-1)/N S
//   nvls       stage locally; barrier; multimem.ld_reduce sub-slab r through the NVSwitch multicast
//              mapping and multimem.st the result to every replica; barrier; local copy-out
//   arrive     1 warp: "my bucket is ready" to every peer + wait for theirs (and the zero-copy
//              symmetry check) — the wait for the slowest replica's backward costs one warp, not a grid
//   nvls-inplace / two-shot-inplace (after arrive): reduce sub-slab r straight from the peers'
//              buckets and write the result into EVERY replica's bucket (multimem.st / P2P stores);
//              one trailing barrier                                    0 extra HBM passes
//   broadcast  root's buffer to every replica (multimem.st, or peers pull over NVLink)
// Tensor cores are deliberately unused: this is a bandwidth-bound reduction, not a contraction.
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>

#include <string.h>

#include <type_traits>

#include "tok_internal.h"

namespace tok {
namespace {

// ------------------------------------------------------------------------------------------------
// PTX helpers
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ unsigned long long globaltimer_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
__device__ __forceinline__ void st_release_sys(uint32_t* p, uint32_t v) {
  asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t ld_relaxed_sys(const uint32_t* p) {
  uint32_t v;
  asm volatile("ld.relaxed.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ unsigned long long ld_relaxed_sys(const unsigned long long* p) {
  unsigned long long v;
  asm volatile("ld.relaxed.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_relaxed_sys(uint32_t* p, uint32_t v) {
  asm volatile("st.relaxed.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ void st_relaxed_sys(unsigned long long* p, unsigned long long v) {
  asm volatile("st.relaxed.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ void fence_sys() { asm volatile("fence.acq_rel.sys;" ::: "memory"); }
// One arrive for the whole group: the NVSwitch applies the add to the counter of EVERY replica bound
// to the multicast object (release: ordered after this CTA's data writes, cumulative over bar.sync).
__device__ __forceinline__ void multimem_red_release_add(uint32_t* mc_ptr, uint32_t v) {
  asm volatile("multimem.red.release.sys.global.add.u32 [%0], %1;" ::"l"(mc_ptr), "r"(v) : "memory");
}
__device__ __forceinline__ void multimem_red_relaxed_add(uint32_t* mc_ptr, uint32_t v) {
  asm volatile("multimem.red.relaxed.sys.global.add.u32 [%0], %1;" ::"l"(mc_ptr), "r"(v) : "memory");
}
// Data written by other GPUs during this kernel is always read at system scope (served by the
// home L2, never by a stale local L1 line).
__device__ __forceinline__ uint4 ld_sys(const uint4* p) {
  uint4 v;
  asm volatile("ld.relaxed.sys.global.v4.u32 {%0,%1,%2,%3}, [%4];"
               : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w)
               : "l"(p)
               : "memory");
  return v;
}
__device__ __forceinline__ uint2 ld_sys(const uint2* p) {
  uint2 v;
  asm volatile("ld.relaxed.sys.global.v2.u32 {%0,%1}, [%2];"
               : "=r"(v.x), "=r"(v.y)
               : "l"(p)
               : "memory");
  return v;
}

template <int BYTES>
struct RawT;
template <>
struct RawT<16> {
  using type = uint4;
};
template <>
struct RawT<8> {
  using type = uint2;
};

// ------------------------------------------------------------------------------------------------
// pack <-> fp32 conversion.  A pack is P elements; P = 4 when any dtype of the launch is f32
// (16 B of f32, 8 B of a 16-bit type), else 8 (16 B of a 16-bit type).
// ------------------------------------------------------------------------------------------------
template <class T, int P>
struct Cvt;

template <>
struct Cvt<float, 4> {
  using raw_t = uint4;
  static __device__ __forceinline__ void to_f32(const raw_t& r, float (&v)[4]) {
    v[0] = __uint_as_float(r.x);
    v[1] = __uint_as_float(r.y);
    v[2] = __uint_as_float(r.z);
    v[3] = __uint_as_float(r.w);
  }
  static __device__ __forceinline__ raw_t from_f32(const float (&v)[4]) {
    return make_uint4(__float_as_uint(v[0]), __float_as_uint(v[1]), __float_as_uint(v[2]),
                      __float_as_uint(v[3]));
  }
  static __device__ __forceinline__ float scalar(float x) { return x; }
  static __device__ __forceinline__ float from_scalar(float x) { return x; }
};

template <int P>
struct Cvt<__nv_bfloat16, P> {
  using raw_t = typename RawT<2 * P>::type;
  static __device__ __forceinline__ void to_f32(const raw_t& r, float (&v)[P]) {
    const uint32_t* w = reinterpret_cast<const uint32_t*>(&r);
#pragma unroll
    for (int k = 0; k < P / 2; ++k) {
      v[2 * k] = __uint_as_float(w[k] << 16);
      v[2 * k + 1] = __uint_as_float(w[k] & 0xffff0000u);
    }
  }
  static __device__ __forceinline__ raw_t from_f32(const float (&v)[P]) {
    raw_t r;
    uint32_t* w = reinterpret_cast<uint32_t*>(&r);
#pragma unroll
    for (int k = 0; k < P / 2; ++k) {
      __nv_bfloat162 h = __floats2bfloat162_rn(v[2 * k], v[2 * k + 1]);
      w[k] = *reinterpret_cast<uint32_t*>(&h);
    }
    return r;
  }
  static __device__ __forceinline__ float scalar(__nv_bfloat16 x) { return __bfloat162float(x); }
  static __device__ __forceinline__ __nv_bfloat16 from_scalar(float x) {
    return __float2bfloat16_rn(x);
  }
};

template <int P>
struct Cvt<__half, P> {
  using raw_t = typename RawT<2 * P>::type;
  static __device__ __forceinline__ void to_f32(const raw_t& r, float (&v)[P]) {
    const uint32_t* w = reinterpret_cast<const uint32_t*>(&r);
#pragma unroll
    for (int k = 0; k < P / 2; ++k) {
      float2 f = __half22float2(*reinterpret_cast<const __half2*>(&w[k]));
      v[2 * k] = f.x;
      v[2 * k + 1] = f.y;
    }
  }
  static __device__ __forceinline__ raw_t from_f32(const float (&v)[P]) {
    raw_t r;
    uint32_t* w = reinterpret_cast<uint32_t*>(&r);
#pragma unroll
    for (int k = 0; k < P / 2; ++k) {
      __half2 h = __floats2half2_rn(v[2 * k], v[2 * k + 1]);
      w[k] = *reinterpret_cast<uint32_t*>(&h);
    }
    return r;
  }
  static __device__ __forceinline__ float scalar(__half x) { return __half2float(x); }
  static __device__ __forceinline__ __half from_scalar(float x) { return __float2half_rn(x); }
};

// ------------------------------------------------------------------------------------------------
// NVSwitch multicast (NVLS) load-reduce / store, fp32 accumulation inside the switch.
// ------------------------------------------------------------------------------------------------
template <class T, int BYTES>
struct MM;
template <>
struct MM<float, 16> {
  static __device__ __forceinline__ uint4 ld_reduce(const void* p) {
    uint4 v;
    asm volatile("multimem.ld_reduce.relaxed.sys.global.add.v4.f32 {%0,%1,%2,%3}, [%4];"
                 : "=f"(*reinterpret_cast<float*>(&v.x)), "=f"(*reinterpret_cast<float*>(&v.y)),
                   "=f"(*reinterpret_cast<float*>(&v.z)), "=f"(*reinterpret_cast<float*>(&v.w))
                 : "l"(p)
                 : "memory");
    return v;
  }
  static __device__ __forceinline__ void st(void* p, const uint4& v) {
    asm volatile("multimem.st.relaxed.sys.global.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(p),
                 "f"(__uint_as_float(v.x)), "f"(__uint_as_float(v.y)), "f"(__uint_as_float(v.z)),
                 "f"(__uint_as_float(v.w))
                 : "memory");
  }
};
#define TOK_MM_16BIT(T, SFX)                                                                      \
  template <>                                                                                     \
  struct MM<T, 16> {                                                                              \
    static __device__ __forceinline__ uint4 ld_reduce(const void* p) {                            \
      uint4 v;                                                                                    \
      asm volatile("multimem.ld_reduce.relaxed.sys.global.add.acc::f32.v4." SFX                   \
                   " {%0,%1,%2,%3}, [%4];"                                                        \
                   : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w)                                   \
                   : "l"(p)                                                                       \
                   : "memory");                                                                   \
      return v;                                                                                   \
    }                                                                                             \
    static __device__ __forceinline__ void st(void* p, const uint4& v) {                          \
      asm volatile("multimem.st.relaxed.sys.global.v4." SFX " [%0], {%1,%2,%3,%4};" ::"l"(p),     \
                   "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w)                                         \
                   : "memory");                                                                   \
    }                                                                                             \
  };                                                                                              \
  template <>                                                                                     \
  struct MM<T, 8> {                                                                               \
    static __device__ __forceinline__ uint2 ld_reduce(const void* p) {                            \
      uint2 v;                                                                                    \
      asm volatile("multimem.ld_reduce.relaxed.sys.global.add.acc::f32.v2." SFX                   \
                   " {%0,%1}, [%2];"                                                              \
                   : "=r"(v.x), "=r"(v.y)                                                         \
                   : "l"(p)                                                                       \
                   : "memory");                                                                   \
      return v;                                                                                   \
    }                                                                                             \
    static __device__ __forceinline__ void st(void* p, const uint2& v) {                          \
      asm volatile("multimem.st.relaxed.sys.global.v2." SFX " [%0], {%1,%2};" ::"l"(p), "r"(v.x), \
                   "r"(v.y)                                                                       \
                   : "memory");                                                                   \
    }                                                                                             \
  };
TOK_MM_16BIT(__nv_bfloat16, "bf16x2")
TOK_MM_16BIT(__half, "f16x2")
#undef TOK_MM_16BIT

// ------------------------------------------------------------------------------------------------
// Per-CTA cross-replica barrier, run by warp 0 of the CTA (the other warps park in bar.sync).
//
// With an NVSwitch multicast mapping (a.mc): ONE `multimem.red.release.sys.add` bumps counter mcnt[b]
// on every replica at once; lane 0 spins (relaxed, system scope) on its own copy until it reached
// world * target.  Without multicast: lanes 0..world-1 publish `target` into flag[b][rank] of one peer
// each (a single warp-wide st.release.sys) and poll flag[b][lane] of their own heap.
// Either way the polling lanes fold their "how far behind" words with a warp-shuffle butterfly so
// that the warp leaves the spin loop as one, then fence (acquire, system scope) before the CTA's
// bar.sync releases the workers.  Values only grow; a replica can be at most one barrier ahead.
// Gives up on host abort or after timeout_ns (a dead peer must not hang the GPU): checked by lane 0
// every 4096 spins — the abort word lives in pinned HOST memory, a PCIe round trip per look.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ int warp_min8(int d) {
  d = min(d, __shfl_xor_sync(0xffffffffu, d, 4));
  d = min(d, __shfl_xor_sync(0xffffffffu, d, 2));
  d = min(d, __shfl_xor_sync(0xffffffffu, d, 1));
  return __shfl_sync(0xffffffffu, d, 0);  // lanes 0..7 cover every possible source rank
}

// Spin until `*word - want >= 0` on every polling lane.  Returns 0, or the status code to report.
// `where`: 1 = bucket arrival, 2 = in-kernel CTA barrier (recorded with the lanes that were still
// behind when the wait was given up, so that tok_comm_status can say WHICH replica is missing).
__device__ __forceinline__ int warp_spin(const KArgs& a, const uint32_t* word, uint32_t want,
                                         bool polls, uint32_t where) {
  const int lane = threadIdx.x & 31;
  unsigned long long t0 = 0;
  uint32_t spins = 0;
  for (;;) {
    int mine = 0;
    if (polls) mine = static_cast<int32_t>(ld_relaxed_sys(word) - want);
    const int d = warp_min8(mine);
    if (d >= 0) return 0;
    if ((++spins & 0xfffu) == 0) {
      int code = 0;
      if (lane == 0) {
        if (a.hostctl[kCtlAbort] != 0) {
          code = 2;
        } else {
          const unsigned long long now = globaltimer_ns();
          if (t0 == 0)
            t0 = now;
          else if (now - t0 > a.timeout_ns)
            code = 1;
        }
      }
      code = __shfl_sync(0xffffffffu, code, 0);
      if (code) {
        const unsigned behind = __ballot_sync(0xffffffffu, polls && mine < 0);
        if (lane == 0 && a.hostctl[kCtlWhere] == 0) {
          a.hostctl[kCtlBehind] = behind;
          a.hostctl[kCtlWant] = want;
          a.hostctl[kCtlWhere] = where | (blockIdx.x << 8);
        }
        return code;
      }
    }
  }
}

// Warp 0's part of the barrier on flag slot `slot`: signal `target` through the multicast counter
// (mc) or the P2P flags, as a release or a relaxed store, wait for every replica, record a failure
// in *s_fail, and fence if `acquire`.  The exchange kernels signal with release; relaxed signalling
// only exists so that tools/barrier_bench.py can time the flags without the ordering.
__device__ __forceinline__ void warp_barrier(const KArgs& a, uint32_t slot, uint32_t target, bool mc,
                                             bool release, bool acquire, int* s_fail) {
  const int lane = threadIdx.x;
  const uint32_t* word;
  uint32_t want;
  bool polls;
  if (mc) {
    uint32_t* cnt = reinterpret_cast<uint32_t*>(a.mc + kMcntOff) + slot;
    if (lane == 0) {
      if (release)
        multimem_red_release_add(cnt, 1u);
      else
        multimem_red_relaxed_add(cnt, 1u);
    }
    word = reinterpret_cast<const uint32_t*>(a.peer[a.rank] + kMcntOff) + slot;
    want = target * static_cast<uint32_t>(a.world);
    polls = lane == 0;
  } else {
    polls = lane < a.world;
    if (polls) {
      uint32_t* flag = reinterpret_cast<uint32_t*>(a.peer[lane]) + (slot * kMaxWorld + a.rank);
      if (release)
        st_release_sys(flag, target);
      else
        st_relaxed_sys(flag, target);
    }
    word = reinterpret_cast<const uint32_t*>(a.peer[a.rank]) + (slot * kMaxWorld + (polls ? lane : 0));
    want = target;
  }
  const int code = warp_spin(a, word, want, polls, 2u);
  if (code != 0 && lane == 0) {
    a.hostctl[kCtlStatus] = code;
    *s_fail = 1;
  }
  if (acquire) fence_sys();  // acquire side of the flag hand-off; bar.sync extends it to the CTA
}

// Optional phase timestamps for tools/phase_breakdown.py (never enabled on the product path).
__device__ __forceinline__ void dbg_stamp(const KArgs& a, int slot) {
  if (a.dbg != nullptr && threadIdx.x == 0) a.dbg[blockIdx.x * 8 + slot] = globaltimer_ns();
}

struct CtaState {
  uint32_t seq;      // launches completed before this one (buffer parity)
  uint32_t bar;      // barriers this CTA index has passed
  uint32_t arrived;  // verdict of the last arrive_kernel (0 = every replica's bucket is ready)
  int* fail;         // CtaShared::fail
};

// Declared __shared__ by each kernel, not here: a kernel's own variable lets the compiler drop the
// words that kernel never reads.
struct CtaShared {
  uint32_t words[3];  // CtaState's first three fields, read once by thread 0
  int fail;           // set by a barrier that was given up
};

__device__ __forceinline__ CtaState cta_begin(const KArgs& a, CtaShared& sh) {
  if (threadIdx.x == 0) {
    sh.words[0] = a.ctr[kCtrCallSeq];
    sh.words[1] = a.ctr[blockIdx.x];
    sh.words[2] = a.ctr[kCtrArriveCode];
    sh.fail = 0;
  }
  __syncthreads();
  CtaState st;
  st.seq = sh.words[0];
  st.bar = sh.words[1];
  st.arrived = sh.words[2];
  st.fail = &sh.fail;
  return st;
}

// ACQUIRE: fence (system scope) after the wait.  Needed when the CTA goes on to read what the peers
// wrote; the trailing barrier of the zero-copy kernels is followed by nothing but the kernel's end
// (the next kernel starts with a clean L1 and reads local memory through the coherent L2), so it
// skips the fence — measured (tools/barrier_bench.py, 8 GPUs, 64 CTAs): signalling alone 2.0 us,
// with release + acquire fences 10.5 us; the fences, not the flags, are what a barrier costs.
template <bool ACQUIRE = true>
__device__ __forceinline__ bool cta_barrier(const KArgs& a, CtaState& st) {
  st.bar += 1;
  __syncthreads();
  if (threadIdx.x < 32) warp_barrier(a, blockIdx.x, st.bar, a.mc != nullptr, true, ACQUIRE, st.fail);
  __syncthreads();
  return *st.fail == 0;
}

// Last CTA out bumps the launch sequence (selects the other staging buffer next time); works under
// CUDA-graph replay because nothing about the sequence lives on the host.
__device__ __forceinline__ void cta_end(const KArgs& a, const CtaState& st) {
  __syncthreads();
  if (threadIdx.x == 0) {
    a.ctr[blockIdx.x] = st.bar;
    __threadfence();
    const unsigned ticket = atomicAdd(&a.ctr[kCtrDone], 1u);
    if (ticket == gridDim.x - 1) {
      a.ctr[kCtrDone] = 0;
      a.ctr[kCtrCallSeq] = st.seq + 1;
    }
  }
}

template <class T>
__device__ __forceinline__ T min_sz(T a, T b) {
  return a < b ? a : b;
}

struct Range {
  size_t lo, hi;
};

// The PRE/POST scale pair and a CTA's slab: CTA b owns packs [b * packs_per_cta, +packs_per_cta),
// clipped to `end`.
struct Slab {
  float pre;   // each contribution's scale: scale (PRE) or 1 (POST)
  float post;  // the sum's scale: 1 (PRE) or scale (POST)
  size_t lo, hi;
  size_t M;  // sub-slab length
  // The sub-slab replica `rank` reduces (two-shot, NVLS): M packs from lo + rank * M, clipped to
  // the slab.  Call it where it is used; computed up front, it is scheduled ahead of the barrier.
  __device__ __forceinline__ Range sub(int rank) const {
    const size_t slo = min_sz(lo + static_cast<size_t>(rank) * M, hi);
    return Range{slo, min_sz(slo + M, hi)};
  }
};

__device__ __forceinline__ Slab cta_slab(const KArgs& a, size_t end) {
  Slab s;
  s.pre = (a.flags & TOK_FLAG_SCALE_POST) ? 1.f : a.scale;
  s.post = (a.flags & TOK_FLAG_SCALE_POST) ? a.scale : 1.f;
  s.lo = static_cast<size_t>(blockIdx.x) * a.packs_per_cta;
  s.hi = min_sz(s.lo + a.packs_per_cta, end);
  s.M = a.packs_per_cta / a.world;
  return s;
}

// The streaming loop over packs [lo, hi): each thread issues U independent loads, kThreads packs
// apart, before the first of their U stores, then finishes one pack at a time.  Each caller's U was
// tuned for its load.
template <int U, class Load, class Store>
__device__ __forceinline__ void stream(size_t lo, size_t hi, Load load, Store store) {
  size_t i = lo + threadIdx.x;
  for (; i + (U - 1) * kThreads < hi; i += U * kThreads) {
    decltype(load(i)) r[U];
#pragma unroll
    for (int u = 0; u < U; ++u) r[u] = load(i + u * kThreads);
#pragma unroll
    for (int u = 0; u < U; ++u) store(i + u * kThreads, r[u]);
  }
  for (; i < hi; i += kThreads) store(i, load(i));
}

// ------------------------------------------------------------------------------------------------
// The kernels.
// ------------------------------------------------------------------------------------------------
template <class IN, class WIRE, class OUT>
struct AR {
  static constexpr int kMaxSz =
      sizeof(IN) > sizeof(WIRE) ? (sizeof(IN) > sizeof(OUT) ? sizeof(IN) : sizeof(OUT))
                                : (sizeof(WIRE) > sizeof(OUT) ? sizeof(WIRE) : sizeof(OUT));
  static constexpr int P = 16 / kMaxSz;
  using CI = Cvt<IN, P>;
  using CW = Cvt<WIRE, P>;
  using CO = Cvt<OUT, P>;
  using RI = typename CI::raw_t;
  using RW = typename CW::raw_t;
  using RO = typename CO::raw_t;

  // in pack -> wire pack (fused cast + pre-scale)
  static __device__ __forceinline__ RW in_to_wire(const RI& r, float pre) {
    float v[P];
    CI::to_f32(r, v);
#pragma unroll
    for (int k = 0; k < P; ++k) v[k] *= pre;
    return CW::from_f32(v);
  }
  // partial last pack of `in` (count % P != 0), zero padded
  static __device__ __forceinline__ RW in_tail_to_wire(const KArgs& a, size_t pack, float pre) {
    const IN* in = static_cast<const IN*>(a.in);
    float v[P];
#pragma unroll
    for (int k = 0; k < P; ++k) {
      const size_t e = pack * P + k;
      v[k] = e < a.count ? CI::scalar(in[e]) * pre : 0.f;
    }
    return CW::from_f32(v);
  }
  // wire pack * post (the sum's scale), through fp32
  static __device__ __forceinline__ RW scale_wire(RW w, float post) {
    if (post != 1.f) {
      float v[P];
      CW::to_f32(w, v);
#pragma unroll
      for (int k = 0; k < P; ++k) v[k] *= post;
      w = CW::from_f32(v);
    }
    return w;
  }
  // wire pack -> out (vector store, or guarded scalar stores for the partial last pack)
  static __device__ __forceinline__ void wire_to_out(const KArgs& a, size_t pack, const RW& w) {
    OUT* out = static_cast<OUT*>(a.out);
    const size_t full = a.count / P;
    if (pack < full) {
      if constexpr (std::is_same<WIRE, OUT>::value) {
        reinterpret_cast<RW*>(out)[pack] = w;
      } else {
        float v[P];
        CW::to_f32(w, v);
        reinterpret_cast<RO*>(out)[pack] = CO::from_f32(v);
      }
    } else {
      float v[P];
      CW::to_f32(w, v);
#pragma unroll
      for (int k = 0; k < P; ++k) {
        const size_t e = pack * P + k;
        if (e < a.count) out[e] = CO::from_scalar(v[k]);
      }
    }
  }

  // ---- phase 0 (two-shot / NVLS): in -> own staging buffer, packs [lo, hi) -----------------------
  static __device__ __forceinline__ void stage_local(const KArgs& a, RW* dst, size_t lo, size_t hi,
                                                     float pre) {
    const RI* in = static_cast<const RI*>(a.in);
    const size_t full = a.count / P;
    const size_t hv = hi < full ? hi : full;
    stream<4>(lo, hv, [&](size_t i) { return __ldcs(in + i); },
              [&](size_t i, const RI& r) { dst[i] = in_to_wire(r, pre); });
    if (threadIdx.x == 0 && full < a.total_packs && full >= lo && full < hi)
      dst[full] = in_tail_to_wire(a, full, pre);
  }

  // ---- phase 0 (one-shot): in -> slot[rank] of every replica's staging buffer ---------------------
  static __device__ __forceinline__ void stage_push(const KArgs& a, int q, size_t lo, size_t hi,
                                                    float pre) {
    const RI* in = static_cast<const RI*>(a.in);
    RW* dst[kMaxWorld];
#pragma unroll
    for (int p = 0; p < kMaxWorld; ++p)
      dst[p] = reinterpret_cast<RW*>(a.peer[p < a.world ? p : 0] + a.stage_off[q] +
                                     static_cast<size_t>(a.rank) * a.slot_bytes);
    auto put = [&](size_t i, const RW& w) {
#pragma unroll
      for (int p = 0; p < kMaxWorld; ++p)
        if (p < a.world) dst[p][i] = w;
    };
    const size_t full = a.count / P;
    const size_t hv = hi < full ? hi : full;
    stream<2>(lo, hv, [&](size_t i) { return __ldcs(in + i); },
              [&](size_t i, const RI& r) { put(i, in_to_wire(r, pre)); });
    if (threadIdx.x == 0 && full < a.total_packs && full >= lo && full < hi)
      put(full, in_tail_to_wire(a, full, pre));
  }

  // The streaming loop over rows: pack i of src[0..world).  All U x world loads of a batch are issued
  // before the first row is reduced; world x U 16-byte requests in flight per thread hide the ~2 us
  // NVLink round trip.
  template <int MAXW, int U, class Row>
  static __device__ __forceinline__ void stream_rows(const KArgs& a, const RW* const* src, size_t lo,
                                                     size_t hi, Row row) {
    size_t i = lo + threadIdx.x;
    for (; i + (U - 1) * kThreads < hi; i += U * kThreads) {
      RW r[U][MAXW];
#pragma unroll
      for (int u = 0; u < U; ++u)
#pragma unroll
        for (int p = 0; p < MAXW; ++p)
          if (p < a.world) r[u][p] = ld_sys(src[p] + i + u * kThreads);
#pragma unroll
      for (int u = 0; u < U; ++u) row(r[u], i + u * kThreads);
    }
    for (; i < hi; i += kThreads) {
      RW r[MAXW];
#pragma unroll
      for (int p = 0; p < MAXW; ++p)
        if (p < a.world) r[p] = ld_sys(src[p] + i);
      row(r, i);
    }
  }

  // ---- rank-ordered fp32 reduction of packs [lo, hi) from src[0..world) --------------------------
  // `mine` (two-shot) receives the reduced wire pack in place so that peers can pull it in phase 2.
  template <int MAXW, int U>
  static __device__ __forceinline__ void reduce_packs(const KArgs& a, const RW* const (&src)[kMaxWorld],
                                                      RW* mine, size_t lo, size_t hi, float post) {
    auto one = [&](const RW (&r)[MAXW], size_t idx) {
      float acc[P];
      CW::to_f32(r[0], acc);
#pragma unroll
      for (int p = 1; p < MAXW; ++p)
        if (p < a.world) {
          float v[P];
          CW::to_f32(r[p], v);
#pragma unroll
          for (int k = 0; k < P; ++k) acc[k] += v[k];
        }
#pragma unroll
      for (int k = 0; k < P; ++k) acc[k] *= post;
      const RW w = CW::from_f32(acc);
      if (mine) mine[idx] = w;
      wire_to_out(a, idx, w);
    };
    stream_rows<MAXW, U>(a, src, lo, hi, one);
  }

  static __device__ __forceinline__ void reduce_dispatch(const KArgs& a,
                                                         const RW* const (&src)[kMaxWorld], RW* mine,
                                                         size_t lo, size_t hi, float post) {
    if (a.world <= 4)
      reduce_packs<4, 4>(a, src, mine, lo, hi, post);
    else
      reduce_packs<kMaxWorld, 2>(a, src, mine, lo, hi, post);
  }

  // ---- phase 2 (two-shot): pull the other replicas' reduced sub-slabs -----------------------------
  // (peer, offset) is flattened so that every thread keeps 8 independent remote loads in flight
  // whatever the world size.
  static __device__ __forceinline__ void gather_packs(const KArgs& a, size_t base_off,
                                                      size_t slab_lo, size_t M) {
    const size_t J = static_cast<size_t>(a.world - 1) * M;
    constexpr int U = 8;
    auto locate = [&](size_t j, const RW*& p_src, size_t& idx) -> bool {
      int pp = 0;
#pragma unroll
      for (int k = 1; k < kMaxWorld - 1; ++k) pp += (j >= k * M) ? 1 : 0;
      const size_t off = j - pp * M;
      int p = a.rank + 1 + pp;
      if (p >= a.world) p -= a.world;
      idx = slab_lo + static_cast<size_t>(p) * M + off;
      p_src = reinterpret_cast<const RW*>(a.peer[p] + base_off);
      return idx < a.total_packs;
    };
    size_t j = threadIdx.x;
    for (; j + (U - 1) * kThreads < J; j += U * kThreads) {
      RW r[U];
      size_t idx[U];
      bool ok[U];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const RW* s;
        ok[u] = locate(j + u * kThreads, s, idx[u]);
        if (ok[u]) r[u] = ld_sys(s + idx[u]);
      }
#pragma unroll
      for (int u = 0; u < U; ++u)
        if (ok[u]) wire_to_out(a, idx[u], r[u]);
    }
    for (; j < J; j += kThreads) {
      const RW* s;
      size_t idx;
      if (locate(j, s, idx)) wire_to_out(a, idx, ld_sys(s + idx));
    }
  }

  // ---- phase 2 (NVLS): local staging -> out over packs [lo, hi) -----------------------------------
  static __device__ __forceinline__ void copy_out(const KArgs& a, const RW* src, size_t lo,
                                                  size_t hi) {
    stream<8>(lo, hi, [&](size_t i) { return ld_sys(src + i); },
              [&](size_t i, const RW& w) { wire_to_out(a, i, w); });
  }

  // ---- NVLS phase 1: in-switch reduce of my sub-slab, broadcast of the result ----------------------
  template <int U = 8>
  static __device__ __forceinline__ void nvls_reduce(const KArgs& a, char* mc_stage, size_t lo,
                                                     size_t hi, float post) {
    using M = MM<WIRE, sizeof(RW)>;
    RW* mc = reinterpret_cast<RW*>(mc_stage);
    stream<U>(lo, hi, [&](size_t i) { return M::ld_reduce(mc + i); },
              [&](size_t i, const RW& r) { M::st(mc + i, scale_wire(r, post)); });
  }

  // ---- zero-copy two-shot: reduce packs [lo, hi) straight from every replica's bucket (rank order,
  // fp32; PRE scale applied to each contribution exactly as the staged path's wire cast does) and
  // push the result into every replica's bucket -------------------------------------------------------
  template <int MAXW, int U>
  static __device__ __forceinline__ void reduce_push(const KArgs& a, size_t lo, size_t hi, float pre,
                                                     float post) {
    RW* buf[MAXW];
#pragma unroll
    for (int p = 0; p < MAXW; ++p)
      buf[p] = reinterpret_cast<RW*>(a.peer[p < a.world ? p : 0] + a.buf_off);
    auto one = [&](const RW (&r)[MAXW], size_t idx) {
      float acc[P];
#pragma unroll
      for (int p = 0; p < MAXW; ++p)
        if (p < a.world) {
          float v[P];
          CW::to_f32(r[p], v);
          if (pre != 1.f) {  // wire_p = cast_wire(f32(in_p) * pre); __fmul_rn: a separately rounded
                             // product, never contracted with the sum below into an FMA
#pragma unroll
            for (int k = 0; k < P; ++k) v[k] = __fmul_rn(v[k], pre);
            const RW w = CW::from_f32(v);
            CW::to_f32(w, v);
          }
#pragma unroll
          for (int k = 0; k < P; ++k) acc[k] = (p == 0) ? v[k] : acc[k] + v[k];
        }
#pragma unroll
      for (int k = 0; k < P; ++k) acc[k] *= post;
      const RW w = CW::from_f32(acc);
#pragma unroll
      for (int p = 0; p < MAXW; ++p)
        if (p < a.world) buf[p][idx] = w;
    };
    stream_rows<MAXW, U>(a, buf, lo, hi, one);
  }

  // A failed barrier leaves the bucket half exchanged: overwrite this CTA's slab of `out` with NaN so
  // that the optimizer cannot silently consume it (the error itself surfaces through tok_comm_status).
  static __device__ __forceinline__ void poison(const KArgs& a, size_t lo, size_t hi) {
    OUT* out = static_cast<OUT*>(a.out);
    const size_t e_lo = lo * P;
    const size_t e_hi = hi * P < a.count ? hi * P : a.count;
    const OUT nan = CO::from_scalar(__int_as_float(0x7fc00000));
    for (size_t e = e_lo + threadIdx.x; e < e_hi; e += kThreads) out[e] = nan;
  }

  // The end of an exchange CTA: poison on failure, last phase stamp, hand over the launch state.
  static __device__ __forceinline__ void finish(const KArgs& a, const CtaState& st, const Slab& s,
                                                bool ok) {
    if (!ok) poison(a, s.lo, s.hi);
    dbg_stamp(a, 5);
    cta_end(a, st);
  }
};

// world == 1: fused scale/cast only (HBM bound: S_in + S_out).  ONE even wave: CTA b owns the
// contiguous packs [b*L, (b+1)*L) with L = packs_per_cta chosen by the host so that the grid is at
// most 2 CTAs per SM and every CTA has the same amount of work — no second, partially filled wave.
// Each thread keeps 8 x 16-byte streaming loads in flight.
template <class IN, class WIRE, class OUT>
__global__ void __launch_bounds__(kThreads, 2) local_kernel(const __grid_constant__ KArgs a) {
  using A = AR<IN, WIRE, OUT>;
  const typename A::RI* in = static_cast<const typename A::RI*>(a.in);
  const size_t full = a.count / A::P;
  const Slab sl = cta_slab(a, full);
  auto finish = [&](size_t i, const typename A::RW& w) {
    A::wire_to_out(a, i, A::scale_wire(w, sl.post));
  };
  stream<8>(sl.lo, sl.hi, [&](size_t i) { return __ldcs(in + i); },
            [&](size_t i, const typename A::RI& r) { finish(i, A::in_to_wire(r, sl.pre)); });
  if (blockIdx.x == 0 && threadIdx.x == 0 && full < a.total_packs)
    finish(full, A::in_tail_to_wire(a, full, sl.pre));
}

// ------------------------------------------------------------------------------------------------
// world == 1, one dtype: the same pass with the copies done by the TMA engine.  A CTA streams its
// tiles through a ring of kTmaStages shared-memory buffers: one elected thread issues
// cp.async.bulk global->shared (completion counted in bytes on an mbarrier), all threads scale the
// tile in shared memory, the elected thread issues cp.async.bulk shared->global and refills the
// stage whose store has finished reading.  SASS: UBLKCP + SYNCS.  Whether this beats the LDG.128
// wave above is a measurement (tools/local_bench.py -> profiles/); the host picks by TOK_LOCAL_TMA.
// ------------------------------------------------------------------------------------------------
constexpr int kTmaStages = 4;
constexpr int kTmaTileBytes = 16384;
constexpr int kTmaThreads = 256;

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)),
               "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "WAIT_%=:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra DONE_%=;\n"
      "bra WAIT_%=;\n"
      "DONE_%=:\n"
      "}\n" ::"r"(smem_u32(bar)),
      "r"(parity)
      : "memory");
}
__device__ __forceinline__ void bulk_g2s(void* smem_dst, const void* gmem_src, uint32_t bytes,
                                         uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
          smem_u32(smem_dst)),
      "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar))
      : "memory");
}
__device__ __forceinline__ void bulk_s2g(void* gmem_dst, const void* smem_src, uint32_t bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gmem_dst),
               "r"(smem_u32(smem_src)), "r"(bytes)
               : "memory");
  asm volatile("cp.async.bulk.commit_group;" ::: "memory");
}
template <int N>
__device__ __forceinline__ void bulk_wait_read() {
  asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}

template <class T>
__global__ void __launch_bounds__(kTmaThreads) local_tma_kernel(const __grid_constant__ KArgs a) {
  using A = AR<T, T, T>;
  extern __shared__ __align__(128) unsigned char tma_smem[];
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(tma_smem + kTmaStages * kTmaTileBytes);
  const char* in = static_cast<const char*>(a.in);
  char* out = static_cast<char*>(a.out);
  const size_t full = a.count / A::P;
  const Slab sl = cta_slab(a, full);  // only the scales: the tiles are strided over the grid
  const size_t nbytes = full * 16;
  const size_t ntiles = (nbytes + kTmaTileBytes - 1) / kTmaTileBytes;
  const size_t nk = ntiles > blockIdx.x ? (ntiles - blockIdx.x - 1) / gridDim.x + 1 : 0;
  const int tid = threadIdx.x;
  auto tile_off = [&](size_t k) { return (blockIdx.x + k * gridDim.x) * static_cast<size_t>(kTmaTileBytes); };
  auto tile_len = [&](size_t k) {
    return static_cast<uint32_t>(min_sz<size_t>(kTmaTileBytes, nbytes - tile_off(k)));
  };
  auto load = [&](size_t k) {
    const int s = static_cast<int>(k % kTmaStages);
    mbar_expect_tx(&full_bar[s], tile_len(k));
    bulk_g2s(tma_smem + s * kTmaTileBytes, in + tile_off(k), tile_len(k), &full_bar[s]);
  };
  if (tid == 0) {
#pragma unroll
    for (int s = 0; s < kTmaStages; ++s) mbar_init(&full_bar[s], 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  if (tid == 0)
    for (size_t k = 0; k < nk && k < kTmaStages; ++k) load(k);
  for (size_t k = 0; k < nk; ++k) {
    const int s = static_cast<int>(k % kTmaStages);
    mbar_wait(&full_bar[s], static_cast<uint32_t>((k / kTmaStages) & 1));
    typename A::RW* tile = reinterpret_cast<typename A::RW*>(tma_smem + s * kTmaTileBytes);
    const uint32_t packs = tile_len(k) / 16;
    for (uint32_t i = tid; i < packs; i += kTmaThreads)
      tile[i] = A::scale_wire(A::in_to_wire(tile[i], sl.pre), sl.post);
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // generic writes -> async proxy
    __syncthreads();
    if (tid == 0) {
      bulk_s2g(out + tile_off(k), tile, tile_len(k));
      // the stage processed one iteration ago is free once its store has finished READING it
      if (k >= 1 && k - 1 + kTmaStages < nk) {
        bulk_wait_read<1>();
        load(k - 1 + kTmaStages);
      }
    }
  }
  if (tid == 0) bulk_wait_read<0>();  // shared memory must outlive the stores that read it
  if (blockIdx.x == 0 && tid == 0 && full < a.total_packs)
    A::wire_to_out(a, full, A::scale_wire(A::in_tail_to_wire(a, full, sl.pre), sl.post));
}

template <class IN, class WIRE, class OUT>
__global__ void __launch_bounds__(kThreads, 1) one_shot_kernel(const __grid_constant__ KArgs a) {
  using A = AR<IN, WIRE, OUT>;
  __shared__ CtaShared sh;
  CtaState st = cta_begin(a, sh);
  const Slab sl = cta_slab(a, a.total_packs);
  const int q = st.seq & 1;

  dbg_stamp(a, 0);
  A::stage_push(a, q, sl.lo, sl.hi, sl.pre);
  dbg_stamp(a, 1);
  if (cta_barrier(a, st)) {
    dbg_stamp(a, 2);
    const typename A::RW* src[kMaxWorld];
#pragma unroll
    for (int p = 0; p < kMaxWorld; ++p)
      src[p] = reinterpret_cast<const typename A::RW*>(a.peer[a.rank] + a.stage_off[q] +
                                                       static_cast<size_t>(p) * a.slot_bytes);
    A::reduce_dispatch(a, src, nullptr, sl.lo, sl.hi, sl.post);
    dbg_stamp(a, 3);
  } else {
    A::poison(a, sl.lo, sl.hi);
  }
  cta_end(a, st);
}

template <class IN, class WIRE, class OUT>
__global__ void __launch_bounds__(kThreads, 1) two_shot_kernel(const __grid_constant__ KArgs a) {
  using A = AR<IN, WIRE, OUT>;
  __shared__ CtaShared sh;
  CtaState st = cta_begin(a, sh);
  const Slab sl = cta_slab(a, a.total_packs);
  const int q = st.seq & 1;
  typename A::RW* mine = reinterpret_cast<typename A::RW*>(a.peer[a.rank] + a.stage_off[q]);

  dbg_stamp(a, 0);
  A::stage_local(a, mine, sl.lo, sl.hi, sl.pre);
  dbg_stamp(a, 1);
  bool ok = cta_barrier(a, st);
  dbg_stamp(a, 2);
  if (ok) {
    const typename A::RW* src[kMaxWorld];
#pragma unroll
    for (int p = 0; p < kMaxWorld; ++p)
      src[p] = reinterpret_cast<const typename A::RW*>(a.peer[p < a.world ? p : 0] + a.stage_off[q]);
    const Range sub = sl.sub(a.rank);
    A::reduce_dispatch(a, src, mine, sub.lo, sub.hi, sl.post);
    dbg_stamp(a, 3);
    ok = cta_barrier(a, st);
    dbg_stamp(a, 4);
  }
  if (ok) A::gather_packs(a, a.stage_off[q], sl.lo, sl.M);
  A::finish(a, st, sl, ok);
}

template <class IN, class WIRE, class OUT>
__global__ void __launch_bounds__(kThreads, 1) nvls_kernel(const __grid_constant__ KArgs a) {
  using A = AR<IN, WIRE, OUT>;
  __shared__ CtaShared sh;
  CtaState st = cta_begin(a, sh);
  const Slab sl = cta_slab(a, a.total_packs);
  const int q = st.seq & 1;
  typename A::RW* mine = reinterpret_cast<typename A::RW*>(a.peer[a.rank] + a.stage_off[q]);

  dbg_stamp(a, 0);
  A::stage_local(a, mine, sl.lo, sl.hi, sl.pre);
  dbg_stamp(a, 1);
  bool ok = cta_barrier(a, st);
  dbg_stamp(a, 2);
  if (ok) {
    const Range sub = sl.sub(a.rank);
    A::nvls_reduce(a, a.mc + a.stage_off[q], sub.lo, sub.hi, sl.post);
    dbg_stamp(a, 3);
    ok = cta_barrier(a, st);
    dbg_stamp(a, 4);
  }
  if (ok) A::copy_out(a, mine, sl.lo, sl.hi);
  A::finish(a, st, sl, ok);
}

// ------------------------------------------------------------------------------------------------
// Bucket arrival (1 warp).  "My bucket is ready" to every peer, then wait until every peer said the
// same.  Stream-ordered after the kernels that produced the bucket, so when it completes every
// replica's copy may be read AND overwritten by the exchange kernel that follows on the stream —
// which therefore needs no leading barrier.  While a replica waits for the slowest peer's backward
// it occupies one warp instead of a whole exchange grid.  Zero-copy symmetry check rides along: each
// replica announces the heap offset of its bucket (buf_off != 0) and compares.
// Constraint (measured, tools/thread_arrival_diag.py): replicas must not share a CUDA context.  With
// replicas as THREADS of one process, the exchange kernel queued behind a waiting arrival blocks the
// context's work queue, a peer's arrival enqueued later is never dispatched, and both sides time out.
// One process per replica — the product shape — has one context each.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(32) arrive_kernel(const __grid_constant__ KArgs a) {
  const int lane = threadIdx.x;
  const uint32_t target = a.ctr[kCtrArrive] + 1;
  const bool polls = lane < a.world;
  if (polls) {
    st_relaxed_sys(reinterpret_cast<unsigned long long*>(a.peer[lane] + kArrSymOff) + a.rank,
                   static_cast<unsigned long long>(a.buf_off));
    st_release_sys(reinterpret_cast<uint32_t*>(a.peer[lane] + kArrOff) + a.rank, target);
  }
  const uint32_t* word =
      reinterpret_cast<const uint32_t*>(a.peer[a.rank] + kArrOff) + (polls ? lane : 0);
  int code = warp_spin(a, word, target, polls, 1u);
  // no fence: the offset word below is read with a system-scope load issued after (control-dependent
  // on) the flag value, and its writer released the flag after writing it
  if (code == 0 && polls && a.buf_off != 0) {
    const unsigned long long theirs = ld_relaxed_sys(
        reinterpret_cast<const unsigned long long*>(a.peer[a.rank] + kArrSymOff) + lane);
    if (theirs != static_cast<unsigned long long>(a.buf_off)) code = 3;
  }
  code = max(code, __shfl_xor_sync(0xffffffffu, code, 4));
  code = max(code, __shfl_xor_sync(0xffffffffu, code, 2));
  code = max(code, __shfl_xor_sync(0xffffffffu, code, 1));
  if (lane == 0) {
    if (code != 0) a.hostctl[kCtlStatus] = code;  // 3: replicas did not allocate symmetrically
    a.ctr[kCtrArriveCode] = code;                 // device copy for the exchange kernel that follows
    a.ctr[kCtrArrive] = target;
  }
}

// ------------------------------------------------------------------------------------------------
// Zero-copy variants (always preceded by arrive_kernel): the bucket itself lives in the symmetric
// pool of every replica's heap at the same offset (a.buf_off), so peers read / multicast-write it
// directly — no staging pass, no copy-out.  in == out, one dtype, whole 16-byte packs.  Replica r
// reduces sub-slab r of every CTA slab and writes the result into EVERY replica's bucket; the only
// barrier is the trailing one ("all writes into my bucket have landed, all reads of it are done").
// A status left by a failed arrival (timeout / abort / asymmetric bucket) poisons instead.
// ------------------------------------------------------------------------------------------------
template <class WIRE>
__global__ void __launch_bounds__(kThreads, 1) nvls_inplace_kernel(const __grid_constant__ KArgs a) {
  using A = AR<WIRE, WIRE, WIRE>;
  __shared__ CtaShared sh;
  CtaState st = cta_begin(a, sh);
  const Slab sl = cta_slab(a, a.total_packs);
  dbg_stamp(a, 0);
  bool ok = st.arrived == 0;
  dbg_stamp(a, 2);
  if (ok) {
    const Range sub = sl.sub(a.rank);
    if (a.unroll == 16)  // the switch sums; scale the sum
      A::template nvls_reduce<16>(a, a.mc + a.buf_off, sub.lo, sub.hi, a.scale);
    else
      A::template nvls_reduce<8>(a, a.mc + a.buf_off, sub.lo, sub.hi, a.scale);
    dbg_stamp(a, 3);
    ok = cta_barrier<false>(a, st);
    dbg_stamp(a, 4);
  }
  A::finish(a, st, sl, ok);
}

template <class WIRE>
__global__ void __launch_bounds__(kThreads, 1)
    two_shot_inplace_kernel(const __grid_constant__ KArgs a) {
  using A = AR<WIRE, WIRE, WIRE>;
  __shared__ CtaShared sh;
  CtaState st = cta_begin(a, sh);
  const Slab sl = cta_slab(a, a.total_packs);
  dbg_stamp(a, 0);
  bool ok = st.arrived == 0;
  dbg_stamp(a, 2);
  if (ok) {
    const Range sub = sl.sub(a.rank);
    // reduce-scatter (reads over NVLink) fused with a push all-gather (posted writes over NVLink)
    if (a.world <= 2)
      A::template reduce_push<2, 8>(a, sub.lo, sub.hi, sl.pre, sl.post);
    else if (a.world <= 4)
      A::template reduce_push<4, 4>(a, sub.lo, sub.hi, sl.pre, sl.post);
    else
      A::template reduce_push<kMaxWorld, 2>(a, sub.lo, sub.hi, sl.pre, sl.post);
    dbg_stamp(a, 3);
    ok = cta_barrier<false>(a, st);
    dbg_stamp(a, 4);
  }
  A::finish(a, st, sl, ok);
}

// ------------------------------------------------------------------------------------------------
// Broadcast (parameter / optimizer-state replication at start-up and after an elastic re-form;
// replaces dist._broadcast_coalesced, torch/nn/parallel/distributed.py:1032).  count = BYTES.
//   kBcastMcPush  buffer in the pool, multicast bound: after arrive, the root multimem.st's its
//                 slab into every replica (one NVLink egress of S feeds all N-1 receivers), everybody
//                 meets at the trailing barrier
//   kBcastPull    buffer in the pool, no multicast: after arrive, receivers read the root's copy
//   kBcastStaged  buffer anywhere: root copies into its staging buffer; barrier; receivers pull it
//                 into their own buffer (double-buffered staging: no trailing barrier)
// ------------------------------------------------------------------------------------------------
template <int MODE>
__global__ void __launch_bounds__(kThreads, 1) bcast_kernel(const __grid_constant__ KArgs a) {
  __shared__ CtaShared sh;
  CtaState st = cta_begin(a, sh);
  const int q = st.seq & 1;
  const size_t packs = a.count / 16;  // whole 16-byte packs; the byte tail is handled below
  const size_t lo = min_sz(static_cast<size_t>(blockIdx.x) * a.packs_per_cta, packs);
  const size_t hi = min_sz(lo + a.packs_per_cta, packs);
  const bool root = a.rank == a.root;
  bool ok = true;
  if (MODE == kBcastStaged) {
    uint4* stage = reinterpret_cast<uint4*>(a.peer[a.root] + a.stage_off[q]);
    if (root) {
      const uint4* src = static_cast<const uint4*>(a.in);
      for (size_t i = lo + threadIdx.x; i < hi; i += kThreads) stage[i] = __ldcs(src + i);
      if (blockIdx.x == 0 && threadIdx.x < (a.count & 15))
        reinterpret_cast<char*>(stage)[packs * 16 + threadIdx.x] =
            static_cast<const char*>(a.in)[packs * 16 + threadIdx.x];
    }
    ok = cta_barrier(a, st);
    if (ok && !root) {
      uint4* dst = static_cast<uint4*>(a.out);
      stream<8>(lo, hi, [&](size_t i) { return ld_sys(stage + i); },
                [&](size_t i, const uint4& v) { dst[i] = v; });
      if (blockIdx.x == 0 && threadIdx.x < (a.count & 15)) {
        const volatile char* sb = reinterpret_cast<const volatile char*>(stage);
        static_cast<char*>(a.out)[packs * 16 + threadIdx.x] = sb[packs * 16 + threadIdx.x];
      }
    }
  } else {
    ok = st.arrived == 0;  // arrival verdict (the kernel runs after arrive_kernel)
    if (ok) {
      if (MODE == kBcastMcPush) {
        if (root) {
          const uint4* src = reinterpret_cast<const uint4*>(a.peer[a.rank] + a.buf_off);
          uint4* mc = reinterpret_cast<uint4*>(a.mc + a.buf_off);
          // written out: on stream() this loop compiles to differently scheduled machine code
          constexpr int U = 8;
          size_t i = lo + threadIdx.x;
          for (; i + (U - 1) * kThreads < hi; i += U * kThreads) {
            uint4 r[U];
#pragma unroll
            for (int u = 0; u < U; ++u) r[u] = __ldcs(src + i + u * kThreads);
#pragma unroll
            for (int u = 0; u < U; ++u) MM<float, 16>::st(mc + i + u * kThreads, r[u]);
          }
          for (; i < hi; i += kThreads) MM<float, 16>::st(mc + i, __ldcs(src + i));
        }
      } else if (!root) {
        const uint4* src = reinterpret_cast<const uint4*>(a.peer[a.root] + a.buf_off);
        uint4* dst = reinterpret_cast<uint4*>(a.peer[a.rank] + a.buf_off);
        stream<8>(lo, hi, [&](size_t i) { return ld_sys(src + i); },
                  [&](size_t i, const uint4& v) { dst[i] = v; });
      }
      ok = cta_barrier(a, st);
    }
  }
  cta_end(a, st);
}

// ------------------------------------------------------------------------------------------------
// Profiling aid (tools/barrier_bench.py): `count` cross-replica barriers back to back, nothing else —
// what one barrier costs, and which part of it.  Every variant runs warp_barrier, the routine of the
// exchange kernels' cta_barrier:
//   0 production barrier (multimem.red.release when a multicast mapping exists, else P2P flags)
//   1 production P2P-flag barrier even when a multicast mapping exists
//   2 signalling only: relaxed multimem.red + relaxed poll, no release, no acquire fence
//   3 signalling only over P2P flags: relaxed stores + relaxed polls
//   4 as 0, with 64 KiB of posted P2P / multicast stores in front of every barrier (a data tail)
// Uses the flag words of CTA slots [128, 128 + grid) so that it never disturbs the exchange state.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kThreads, 1) barrier_bench_kernel(const __grid_constant__ KArgs a) {
  __shared__ int s_fail;
  const int variant = static_cast<int>(a.flags);
  // the multicast counters (slots 192..255) and the P2P flags (slots 128..191) count separately
  const bool mc_variant = a.mc != nullptr && (variant == 0 || variant == 2 || variant == 4);
  const bool ordered = variant == 0 || variant == 1 || variant == 4;
  const uint32_t slot = (mc_variant ? 192 : 128) + blockIdx.x;
  if (threadIdx.x == 0) s_fail = 0;
  uint32_t bar = a.ctr[slot];
  __syncthreads();
  for (size_t it = 0; it < a.count; ++it) {
    bar += 1;
    if (variant == 4) {
      uint4* dst = reinterpret_cast<uint4*>(a.peer[(a.rank + 1) % a.world] + a.stage_off[0]) +
                   static_cast<size_t>(blockIdx.x) * 4096;
      const uint4 v = make_uint4(bar, bar, bar, bar);
#pragma unroll
      for (int k = 0; k < 8; ++k) dst[threadIdx.x + k * kThreads] = v;
    }
    __syncthreads();
    if (threadIdx.x < 32) warp_barrier(a, slot, bar, mc_variant, ordered, ordered, &s_fail);
    __syncthreads();
    if (s_fail) break;
  }
  if (threadIdx.x == 0) a.ctr[slot] = bar;
}

// ------------------------------------------------------------------------------------------------
// dispatch
// ------------------------------------------------------------------------------------------------
template <class IN, class WIRE, class OUT>
int launch_typed(int algo, int ctas, const KArgs& a, cudaStream_t s) {
  switch (algo) {
    case TOK_ALGO_LOCAL:
      local_kernel<IN, WIRE, OUT><<<ctas, kThreads, 0, s>>>(a);
      break;
    case kAlgoLocalTma:
      if constexpr (std::is_same<IN, WIRE>::value && std::is_same<WIRE, OUT>::value) {
        static bool attr_set = false;  // per instantiation; benign if two threads race
        if (!attr_set) {
          cudaFuncSetAttribute(local_tma_kernel<WIRE>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                               static_cast<int>(local_tma_smem_bytes()));
          attr_set = true;
        }
        local_tma_kernel<WIRE><<<ctas, kTmaThreads, local_tma_smem_bytes(), s>>>(a);
        break;
      }
      return static_cast<int>(cudaErrorInvalidValue);
    case TOK_ALGO_ONE_SHOT:
      one_shot_kernel<IN, WIRE, OUT><<<ctas, kThreads, 0, s>>>(a);
      break;
    case TOK_ALGO_TWO_SHOT:
      two_shot_kernel<IN, WIRE, OUT><<<ctas, kThreads, 0, s>>>(a);
      break;
    case TOK_ALGO_NVLS:
      nvls_kernel<IN, WIRE, OUT><<<ctas, kThreads, 0, s>>>(a);
      break;
    case kAlgoTwoShotInplace:
    case kAlgoNvlsInplace:
      if constexpr (std::is_same<IN, WIRE>::value && std::is_same<WIRE, OUT>::value) {
        if (algo == kAlgoNvlsInplace)
          nvls_inplace_kernel<WIRE><<<ctas, kThreads, 0, s>>>(a);
        else
          two_shot_inplace_kernel<WIRE><<<ctas, kThreads, 0, s>>>(a);
        break;
      }
      return static_cast<int>(cudaErrorInvalidValue);
    default:
      return static_cast<int>(cudaErrorInvalidValue);
  }
  return static_cast<int>(cudaGetLastError());
}

template <class IN, class WIRE>
int launch_out(int out_dtype, int algo, int ctas, const KArgs& a, cudaStream_t s) {
  switch (out_dtype) {
    case TOK_F32:
      return launch_typed<IN, WIRE, float>(algo, ctas, a, s);
    case TOK_BF16:
      return launch_typed<IN, WIRE, __nv_bfloat16>(algo, ctas, a, s);
    case TOK_F16:
      return launch_typed<IN, WIRE, __half>(algo, ctas, a, s);
  }
  return static_cast<int>(cudaErrorInvalidValue);
}

template <class IN>
int launch_wire(int wire_dtype, int out_dtype, int algo, int ctas, const KArgs& a, cudaStream_t s) {
  switch (wire_dtype) {
    case TOK_F32:
      return launch_out<IN, float>(out_dtype, algo, ctas, a, s);
    case TOK_BF16:
      return launch_out<IN, __nv_bfloat16>(out_dtype, algo, ctas, a, s);
    case TOK_F16:
      return launch_out<IN, __half>(out_dtype, algo, ctas, a, s);
  }
  return static_cast<int>(cudaErrorInvalidValue);
}

}  // namespace

size_t local_tma_smem_bytes() { return kTmaStages * kTmaTileBytes + 64; }

int launch_arrive(const KArgs& args, void* stream) {
  arrive_kernel<<<1, 32, 0, static_cast<cudaStream_t>(stream)>>>(args);
  return static_cast<int>(cudaGetLastError());
}

int launch_barrier_bench(int ctas, const KArgs& args, void* stream) {
  barrier_bench_kernel<<<ctas, kThreads, 0, static_cast<cudaStream_t>(stream)>>>(args);
  return static_cast<int>(cudaGetLastError());
}

int launch_broadcast(int mode, int ctas, const KArgs& args, void* stream) {
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  switch (mode) {
    case kBcastMcPush:
      bcast_kernel<kBcastMcPush><<<ctas, kThreads, 0, s>>>(args);
      break;
    case kBcastPull:
      bcast_kernel<kBcastPull><<<ctas, kThreads, 0, s>>>(args);
      break;
    case kBcastStaged:
      bcast_kernel<kBcastStaged><<<ctas, kThreads, 0, s>>>(args);
      break;
    default:
      return static_cast<int>(cudaErrorInvalidValue);
  }
  return static_cast<int>(cudaGetLastError());
}

size_t dtype_size(int dtype) { return dtype == TOK_F32 ? 4 : 2; }

int pack_elems(int in_dtype, int wire_dtype, int out_dtype) {
  return (in_dtype == TOK_F32 || wire_dtype == TOK_F32 || out_dtype == TOK_F32) ? 4 : 8;
}

int launch_allreduce(int algo, int in_dtype, int wire_dtype, int out_dtype, int ctas,
                     const KArgs& args, void* stream) {
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  switch (in_dtype) {
    case TOK_F32:
      return launch_wire<float>(wire_dtype, out_dtype, algo, ctas, args, s);
    case TOK_BF16:
      return launch_wire<__nv_bfloat16>(wire_dtype, out_dtype, algo, ctas, args, s);
    case TOK_F16:
      return launch_wire<__half>(wire_dtype, out_dtype, algo, ctas, args, s);
  }
  return static_cast<int>(cudaErrorInvalidValue);
}

}  // namespace tok
