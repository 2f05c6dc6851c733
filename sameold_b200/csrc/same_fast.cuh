// same_fast.cuh — sample-rate building blocks of the 22050 Hz class (42 taps, DC length 16, s16 samples), shared by the
// fast receiver kernels and the front-end kernel (same_kernels.cu) and by the long-stream path (same_long.cu):
// integer unpacking, the exact integer DC blocker (DcInt / dc_chunk / dc_store), the raw-sample feed with prefetch
// (RawFeedT) and the AGC step.  One copy of each: an arithmetic fix lands in one place.
#pragma once

#include <cuda_runtime.h>

#include "same_lane.cuh"

namespace same_dev {

#define FAST_NTAPS 42
#define FAST_DCL 16
#define FAST_CHUNK 32     // samples produced per refill step (2 x DC length: the S1 history recycles in place twice)
#define FAST_RING 64

// Explicit shared-memory accesses on 32-bit shared addresses (keeps ptxas from re-deriving the shared window base
// around every predicated store).
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ float lds_f32(uint32_t addr) {
  float v;
  asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(addr));
  return v;
}
__device__ __forceinline__ void sts_f32(uint32_t addr, float v) {
  asm volatile("st.shared.f32 [%0], %1;" ::"r"(addr), "f"(v) : "memory");
}
__device__ __forceinline__ void sts_f32_mirrored(uint32_t addr, float v) {  // y ring slot j and its mirror j + 64
  asm volatile("st.shared.f32 [%0], %1;\n\tst.shared.f32 [%0+8192], %1;" ::"r"(addr), "f"(v) : "memory");
}

__device__ __forceinline__ int s16_lo(uint32_t w) {   // sign-extended low half in one PRMT
  int r;
  asm("prmt.b32 %0, %1, 0, 0x9910;" : "=r"(r) : "r"(w));
  return r;
}
__device__ __forceinline__ int s16_hi(uint32_t w) { return ((int)w) >> 16; }
__device__ __forceinline__ int s16_at(const uint32_t* w, int i) { return (i & 1) ? s16_hi(w[i >> 1]) : s16_lo(w[i >> 1]); }

// ----------------------------------------------------------------------------------------------------------------
// Exact integer DC blocker (A0 + A1 for the 22050 Hz geometry), shared by every fast kernel and the front-end kernel.
//
// With s16 input and length 16 every intermediate of dcblock.rs:45-49,104-108 is an integer / 16 / 256 below 2^24, so
// the f32 running sums have no rounding error and equal these integer recursions (SURVEY.md §8a row A1):
//     S1 += x - x[-16]            ff: moving_sum += input - aged      dcblock.rs:106     (S1 = 16 * ma0)
//     S2 += S1 - S1[-16]          fb: moving_sum += ma0 - aged        dcblock.rs:106     (S2 = 256 * ma1)
//     d   = (256 * x[-15] - S2) / 256                                  dcblock.rs:48
// State: the last 16 raw samples (packed pairs, oldest first) and the last 16 values of S1.  One chunk = 32 samples,
// everything statically indexed (registers).
// ----------------------------------------------------------------------------------------------------------------
struct DcInt {
  uint32_t rawh[FAST_DCL / 2];   // last 16 raw samples, packed pairs, oldest first   (ff window, dcblock.rs:63)
  int s1h[FAST_DCL];             // S1 of the last 16 samples                         (fb window)
  int S1, S2;
};

// word index of the DC state inside a 34-word block: ff window 0..15, fb window 16..31, ff sum 32, fb sum 33
#define DCW_FF 0
#define DCW_FB 16
#define DCW_FFSUM 32
#define DCW_FBSUM 33
#define DCW_WORDS 34

__device__ __forceinline__ void dc_load(DcInt& q, const uint32_t* st, const SameLayout& L) {
  q.S1 = __float2int_rn(__uint_as_float(LANE_ST(st, L, F_DC_FFSUM)));              // ff moving_sum
  q.S2 = __float2int_rn(__uint_as_float(LANE_ST(st, L, F_DC_FBSUM)) * 16.0f);      // 16 * fb moving_sum
#pragma unroll
  for (int i = 0; i < FAST_DCL / 2; ++i) {
    const int lo = __float2int_rn(__uint_as_float(LANE_ST(st, L, L.dc_ff + 2 * i)));
    const int hi = __float2int_rn(__uint_as_float(LANE_ST(st, L, L.dc_ff + 2 * i + 1)));
    q.rawh[i] = ((uint32_t)lo & 0xffffu) | ((uint32_t)hi << 16);
  }
#pragma unroll
  for (int i = 0; i < FAST_DCL; ++i) q.s1h[i] = __float2int_rn(__uint_as_float(LANE_ST(st, L, L.dc_fb + i)) * 16.0f);
}

__device__ __forceinline__ void dc_zero(DcInt& q) {
  q.S1 = 0; q.S2 = 0;
#pragma unroll
  for (int i = 0; i < FAST_DCL / 2; ++i) q.rawh[i] = 0u;
#pragma unroll
  for (int i = 0; i < FAST_DCL; ++i) q.s1h[i] = 0;
}

// One full chunk of CHUNK (16 or 32) samples (packed pairs in cur); emit(i, d) receives the DC-blocked sample i as exact f32.
template <int CHUNK, class Emit>
__device__ __forceinline__ void dc_chunk(DcInt& q, const uint32_t (&cur)[CHUNK / 2], Emit&& emit) {
  static_assert(CHUNK == 16 || CHUNK == 32, "the S1 history recycles in place: chunk = 1 or 2 DC lengths");
#pragma unroll
  for (int i = 0; i < CHUNK; ++i) {
    const int x = s16_at(cur, i);
    const int x16 = (i < FAST_DCL) ? s16_at(q.rawh, i) : s16_at(cur, i - FAST_DCL);
    const int x15 = (i < FAST_DCL - 1) ? s16_at(q.rawh, i + 1) : s16_at(cur, i - (FAST_DCL - 1));
    q.S1 += x - x16;
    q.S2 += q.S1 - q.s1h[i & 15];
    q.s1h[i & 15] = q.S1;
    const int D = (x15 << 8) - q.S2;
    emit(i, (float)D * 0.00390625f);
  }
#pragma unroll
  for (int i = 0; i < FAST_DCL / 2; ++i) q.rawh[i] = cur[CHUNK / 2 - FAST_DCL / 2 + i];
}

// The final, partial chunk of a submit (nnew < CHUNK samples; cur zero-filled beyond nnew).  The histories are NOT
// rotated afterwards: dc_store_after_partial writes them out in canonical order.
template <int CHUNK, class Emit>
__device__ __forceinline__ void dc_chunk_partial(DcInt& q, const uint32_t (&cur)[CHUNK / 2], const int nnew, Emit&& emit) {
#pragma unroll
  for (int i = 0; i < CHUNK; ++i) {
    if (i < nnew) {
      const int x = s16_at(cur, i);
      const int x16 = (i < FAST_DCL) ? s16_at(q.rawh, i) : s16_at(cur, i - FAST_DCL);
      const int x15 = (i < FAST_DCL - 1) ? s16_at(q.rawh, i + 1) : s16_at(cur, i - (FAST_DCL - 1));
      q.S1 += x - x16;
      q.S2 += q.S1 - q.s1h[i & 15];
      q.s1h[i & 15] = q.S1;
      const int D = (x15 << 8) - q.S2;
      emit(i, (float)D * 0.00390625f);
    }
  }
}

// DC state out, canonical f32 form (the generic kernel's layout), through store(word, bits) with word in 0..33.
// After whole chunks only: the histories are in order.
template <class Store>
__device__ __forceinline__ void dc_store(const DcInt& q, Store&& store) {
  store(DCW_FFSUM, __float_as_uint((float)q.S1));
  store(DCW_FBSUM, __float_as_uint((float)q.S2 * 0.0625f));
#pragma unroll
  for (int i = 0; i < FAST_DCL; ++i) {
    store(DCW_FF + i, __float_as_uint((float)s16_at(q.rawh, i)));
    store(DCW_FB + i, __float_as_uint((float)q.s1h[i] * 0.0625f));
  }
}
// After a partial chunk of nnew samples: rotate so that index 0 is the oldest sample again (static register indices,
// run-time word numbers -- no dynamically indexed register arrays).  The last 16 samples are old-history entries
// i >= nnew and chunk samples nnew-16 <= i < nnew; the S1 of chunk sample j lives in s1h[j & 15].
template <int CHUNK, class Store>
__device__ __forceinline__ void dc_store_after_partial(const DcInt& q, const uint32_t (&cur)[CHUNK / 2], const uint32_t nnew,
                                                       Store&& store) {
  store(DCW_FFSUM, __float_as_uint((float)q.S1));
  store(DCW_FBSUM, __float_as_uint((float)q.S2 * 0.0625f));
#pragma unroll
  for (int i = 0; i < FAST_DCL; ++i) {
    if (i >= (int)nnew) store(DCW_FF + ((uint32_t)i - nnew), __float_as_uint((float)s16_at(q.rawh, i)));
    store(DCW_FB + (((uint32_t)i - nnew) & 15u), __float_as_uint((float)q.s1h[i] * 0.0625f));
  }
#pragma unroll
  for (int i = 0; i < CHUNK; ++i) {
    if (i < (int)nnew && i + FAST_DCL >= (int)nnew)
      store(DCW_FF + ((uint32_t)(i + FAST_DCL) - nnew), __float_as_uint((float)s16_at(cur, i)));
  }
}
// store target: the resident state words of this lane
struct DcToState {
  uint32_t* st; const SameLayout& L;
  __device__ __forceinline__ void operator()(uint32_t w, uint32_t bits) const {
    const uint32_t word = w < DCW_FB ? L.dc_ff + w : w < DCW_FFSUM ? L.dc_fb + (w - DCW_FB) : (w == DCW_FFSUM ? (uint32_t)F_DC_FFSUM : (uint32_t)F_DC_FBSUM);
    LANE_ST(st, L, word) = bits;
  }
};

// Raw-sample feed of one lane: CHUNK-sample chunks as packed pairs, 16-byte loads issued one chunk ahead (a refill
// happens at most once or twice per round, so the global-load latency overlaps a round of sequential work).
template <int CHUNK>
struct RawFeedT {
  static constexpr int NV = CHUNK / 8;   // int4 loads per chunk
  const int16_t* src;
  int4 nx[NV];
  bool aligned, pf_ok;
  __device__ __forceinline__ void init(const int16_t* s, uint32_t first, uint32_t len) {
    src = s;
    aligned = (reinterpret_cast<uintptr_t>(s) & 15u) == 0;
#pragma unroll
    for (int i = 0; i < NV; ++i) nx[i] = make_int4(0, 0, 0, 0);
    pf_ok = src != nullptr && aligned && first + (uint32_t)CHUNK <= len;
    if (pf_ok) {
      const int4* q = reinterpret_cast<const int4*>(src + first);
#pragma unroll
      for (int i = 0; i < NV; ++i) nx[i] = __ldg(q + i);
    }
  }
  // the full chunk at rp (rp % 8 == 0 relative to an aligned src); prefetches the chunk after it
  __device__ __forceinline__ void take_full(uint32_t (&cur)[CHUNK / 2], uint32_t rp, uint32_t len) {
    if (pf_ok) {
#pragma unroll
      for (int i = 0; i < NV; ++i) { cur[4 * i] = nx[i].x; cur[4 * i + 1] = nx[i].y; cur[4 * i + 2] = nx[i].z; cur[4 * i + 3] = nx[i].w; }
    } else {
#pragma unroll
      for (int i = 0; i < CHUNK / 2; ++i) {
        const uint32_t lo = src ? (uint32_t)(uint16_t)src[rp + 2 * i] : 0u;
        const uint32_t hi = src ? (uint32_t)(uint16_t)src[rp + 2 * i + 1] : 0u;
        cur[i] = lo | (hi << 16);
      }
    }
    pf_ok = src != nullptr && aligned && (len - rp) >= 2u * CHUNK;
    if (pf_ok) {
      const int4* q = reinterpret_cast<const int4*>(src + rp + CHUNK);
#pragma unroll
      for (int i = 0; i < NV; ++i) nx[i] = __ldg(q + i);
    }
  }
  // a partial chunk of nnew < CHUNK samples at rp: scalar loads, zero-filled
  __device__ __forceinline__ void take_partial(uint32_t (&cur)[CHUNK / 2], uint32_t rp, uint32_t nnew) const {
#pragma unroll
    for (int i = 0; i < CHUNK / 2; ++i) cur[i] = 0u;
#pragma unroll
    for (int i = 0; i < CHUNK; ++i) {
      const uint32_t v = (src && i < (int)nnew) ? (uint32_t)(uint16_t)src[rp + i] : 0u;
      cur[i >> 1] |= (i & 1) ? (v << 16) : v;
    }
  }
};
using RawFeed = RawFeedT<FAST_CHUNK>;

// One AGC step (agc.rs:72-77): y = x*g; g += (!locked as f32)*(1-|y|)*bw; g = clamp(g, min, max).  `bw_eff` is bw or 0.
__device__ __forceinline__ float agc_step(float& g, const float d, const float bw_eff, const float gmin, const float gmax) {
  const float y = FMUL(d, g);                                                       // agc.rs:73
  g = fminf(fmaxf(FADD(g, FMUL(FSUB(1.0f, fabsf(y)), bw_eff)), gmin), gmax);        // agc.rs:74-75
  return y;
}

// Ring counters between warps of one block (same_long_seq_kernel, same_rx_pipe_kernel).  LS_RELEASE_ACQUIRE=1:
// st.release.cta / ld.acquire.cta, the hand-off the PTX memory model defines (the acquire load is a plain LDS in SASS,
// the release store a MEMBAR.ALL.CTA + STS).  0: volatile accesses, relying on one
// thread's shared-memory stores being performed in program order.  Both are bit-exact over 24 h
// (tests/test_zz_config5_24h.py); profiles/README.md has the A/B.
#ifndef LS_RELEASE_ACQUIRE
#define LS_RELEASE_ACQUIRE 1
#endif
__device__ __forceinline__ void ls_publish(volatile uint32_t* w, uint32_t v) {
#if LS_RELEASE_ACQUIRE
  asm volatile("st.release.cta.shared.u32 [%0], %1;" ::"r"((uint32_t)__cvta_generic_to_shared(const_cast<uint32_t*>(w))), "r"(v)
               : "memory");
#else
  *w = v;
#endif
}
__device__ __forceinline__ uint32_t ls_observe(const volatile uint32_t* w) {
#if LS_RELEASE_ACQUIRE
  uint32_t v;
  asm volatile("ld.acquire.cta.shared.u32 %0, [%1];" : "=r"(v) : "r"((uint32_t)__cvta_generic_to_shared(const_cast<uint32_t*>(w)))
               : "memory");
  return v;
#else
  return *w;
#endif
}

}  // namespace same_dev
