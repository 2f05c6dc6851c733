// same_long.cu — the long-stream path: ONE stream (BASELINE config 5: a single 24 h stream with sparse bursts), where
// there is no second stream to fill a warp and the receiver's dependent chain per TED round (~1500 cycles) is all there
// is.  What the north star asks for here — "time-parallel FIR/correlator tiles, per-stream loop kernels" — is possible
// bit-exactly as long as the AGC is unlocked, i.e. everywhere except inside bursts (0.5 % of such a stream):
//
//   A  same_long_dc_kernel    s16 -> exact DC-blocked f32, time-parallel (the integer recursion has 31 samples of memory)
//   B  same_long_agc_kernel   the AGC recurrence (agc.rs:72-77) in blocks of 2048 samples, one thread per block.  Block 0
//                             starts from the stream's true gain; every other block warms up on the 1024 samples before
//                             it from a guessed gain.  The unlocked AGC map contracts (|1 - |d| bw| per sample), so the
//                             trajectories coalesce BITWISE within ~300 samples on noise (worst seen 481) — and whether a
//                             block's start gain really equals its predecessor's end gain is CHECKED, bit for bit:
//      same_long_verify_kernel   first block whose hand-over fails -> end of the range that may be consumed.
//   C  same_long_mf_kernel    the mark/space matched filters (demod.rs:156-164) at EVERY sample position of that AGC
//                             output, time-parallel: 21x the arithmetic of the sequential receiver, in parallel.
//   D  same_long_seq_kernel   the timing loop (A5) strictly sequential on one lane, picking its soft symbols out of C's
//                             output (staged through shared memory), and the squelch, equalizer, framer and transport
//                             (A6-A9) on a second warp, one ring of symbol records behind: ~250 cycles per TED round
//                             instead of ~1500.  It stops when the symbol stages lock the AGC (sync found: a burst
//                             begins) or reset the timing loop, at the end of the verified range, or at the end.
//   burst / unverified spans  the ordinary tile-fed single-warp kernel (same_rx_fast_kernel<true>) on A's output, until
//                             the AGC is unlocked again; then B-D restart from the true state.
// The speculation in B never decides anything: a block is used only after its hand-over gain was verified, and D's
// arithmetic is the sequential receiver's (same_lane.cuh), so the events are those of the reference, bit for bit
// (tests: the full 24 h stream, the 16-minute stream in chunks, every single-stream test above the length threshold).
// All state stays in the ordinary resident layout between kernels; the DC-blocker state is committed at the end.
#include <cuda_runtime.h>

#include "same_fast.cuh"
#include "same_internal.h"
#include "same_lane.cuh"

namespace same_dev {

#define LS_RUN 256        // samples per thread in A
#define LS_BLOCK 2048     // samples per thread in B
#define LS_WARM 1024      // warm-up samples of a speculative block
#define LS_TILE 4096      // soft symbols staged per shared-memory tile in D

// ---------------------------------------------------------------------------------------------------------------- A
__global__ void same_long_dc_kernel(const __grid_constant__ SameParams p, const int16_t* __restrict__ src, const uint32_t len,
                                    float* __restrict__ d, uint32_t* __restrict__ dc_next) {
  const SameLayout& L = p.layout;
  const uint32_t run = blockIdx.x * blockDim.x + threadIdx.x;
  const uint32_t r0 = run * LS_RUN;
  if (r0 >= len) return;
  const uint32_t r1 = min(r0 + (uint32_t)LS_RUN, len);
  const uint32_t* st = p.state32;   // stream 0
  DcInt dc;
  RawFeed feed;
  uint32_t cur[FAST_CHUNK / 2];
  if (run == 0) {
    dc_load(dc, st, L);
    feed.init(src, 0u, len);
  } else {
    dc_zero(dc);
    feed.init(src, r0 - FAST_CHUNK, len);
    feed.take_full(cur, r0 - FAST_CHUNK, len);
    dc_chunk<FAST_CHUNK>(dc, cur, [](int, float) {});      // warm-up: exact from the 32nd sample on
  }
  uint32_t c = r0;
  for (; c + FAST_CHUNK <= r1; c += FAST_CHUNK) {
    feed.take_full(cur, c, len);
    float* dst = d + c;
    dc_chunk<FAST_CHUNK>(dc, cur, [&](int i, float v) { dst[i] = v; });
  }
  const auto to_next = [&](uint32_t w, uint32_t bits) { dc_next[(size_t)w * L.n_pad] = bits; };
  if (c < r1) {
    const uint32_t nnew = r1 - c;
    feed.take_partial(cur, c, nnew);
    float* dst = d + c;
    dc_chunk_partial<FAST_CHUNK>(dc, cur, (int)nnew, [&](int i, float v) { dst[i] = v; });
    dc_store_after_partial<FAST_CHUNK>(dc, cur, nnew, to_next);
  } else if (r1 == len) {
    dc_store(dc, to_next);
  }
}

// commit A's DC-blocker state (end of the submit)
__global__ void same_long_commit_dc_kernel(const __grid_constant__ SameParams p, const uint32_t* __restrict__ dc_next) {
  const SameLayout& L = p.layout;
  if (threadIdx.x < DCW_WORDS) DcToState{p.state32, L}(threadIdx.x, dc_next[(size_t)threadIdx.x * L.n_pad]);
}

// ---------------------------------------------------------------------------------------------------------------- B
// d: DC-blocked samples of the submit; the range is [pos0, end).  yfull[42 + (n - pos0)] = AGC output of sample n,
// yfull[0..42) = the demod window before pos0 (copied from the state); gspec[n - pos0] = gain AFTER sample n;
// g_in[k] = the gain block k > 0 started with after its warm-up.
__global__ void same_long_agc_kernel(const __grid_constant__ SameParams p, const float* __restrict__ d, const uint32_t pos0,
                                     const uint32_t end, float* __restrict__ yfull, float* __restrict__ gspec,
                                     float* __restrict__ g_in) {
  const SameLayout& L = p.layout;
  const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
  const unsigned long long sk64 = (unsigned long long)pos0 + (unsigned long long)k * LS_BLOCK;
  if (sk64 >= end) return;
  const uint32_t sk = (uint32_t)sk64;
  const float bw = p.agc_bw, gmin = p.agc_min, gmax = p.agc_max;
  const float g_true = __uint_as_float(LANE_ST(p.state32, L, F_AGC_GAIN));   // gain at pos0
  float g = g_true;
  if (k == 0) {
    for (int i = 0; i < FAST_NTAPS; ++i) yfull[i] = __uint_as_float(LANE_ST(p.state32, L, L.win + i));
  } else {
    for (uint32_t n = sk - LS_WARM; n < sk; ++n) (void)agc_step(g, d[n], bw, gmin, gmax);   // LS_BLOCK >= LS_WARM: n >= pos0
    g_in[k] = g;
  }
  const uint32_t e = min(sk + (uint32_t)LS_BLOCK, end);
  float* yo = yfull + FAST_NTAPS - pos0;
  float* go = gspec - pos0;
  for (uint32_t n = sk; n < e; ++n) {
    yo[n] = agc_step(g, d[n], bw, gmin, gmax);
    go[n] = g;
  }
}

// ctrl[0] = end of the verified range: the start of the first block whose warm-started gain differs (bitwise) from its
// predecessor's end gain, or `end`.  (ctrl[0] is preset to `end` by the host.)
__global__ void same_long_verify_kernel(const float* __restrict__ gspec, const float* __restrict__ g_in, const uint32_t pos0,
                                        const uint32_t end, uint32_t* __restrict__ ctrl) {
  const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x + 1u;
  const unsigned long long sk64 = (unsigned long long)pos0 + (unsigned long long)k * LS_BLOCK;
  if (sk64 >= end) return;
  const uint32_t sk = (uint32_t)sk64;
  if (__float_as_uint(g_in[k]) != __float_as_uint(gspec[sk - 1u - pos0])) atomicMin(&ctrl[0], sk);
}

// ---------------------------------------------------------------------------------------------------------------- C
// soft[i] = demodulated sample at the position pos0 + i (window = samples pos0 + i - 42 .. pos0 + i - 1 = yfull[i .. i+41]),
// i = 1 .. n_out: one rounded multiply and one rounded add per component and tap, newest sample first
// (filter.rs:363-377), |mark| - |space| clamped (demod.rs:163).
__global__ void __launch_bounds__(256) same_long_mf_kernel(const __grid_constant__ SameTaps2 taps, const float* __restrict__ yfull,
                                                           const uint32_t n_out, float* __restrict__ soft) {
  __shared__ float tile[256 + FAST_NTAPS];
  const uint32_t i0 = blockIdx.x * 256u + 1u;
  for (uint32_t j = threadIdx.x; j < 256u + FAST_NTAPS - 1u; j += 256u) {
    const uint32_t idx = i0 + j;                       // yfull index; valid up to n_out + 41
    tile[j] = (idx <= n_out + FAST_NTAPS - 1u) ? yfull[idx] : 0.0f;
  }
  __syncthreads();
  const uint32_t i = i0 + threadIdx.x;
  if (i > n_out) return;
  float mr = 0.0f, mi = 0.0f, sr = 0.0f, si = 0.0f;
#pragma unroll
  for (int j = 0; j < FAST_NTAPS; ++j) {
    const float v = tile[threadIdx.x + (FAST_NTAPS - 1) - j];
    mr = FADD(mr, FMUL(v, taps.mark[j].x));
    mi = FADD(mi, FMUL(v, taps.mark[j].y));
    sr = FADD(sr, FMUL(v, taps.space[j].x));
    si = FADD(si, FMUL(v, taps.space[j].y));
  }
  soft[i] = rclamp(FSUB(hypot_fixed(mr, mi), hypot_fixed(sr, si)), -1.0f, 1.0f);
}

// ---------------------------------------------------------------------------------------------------------------- D
// Two warps, one lane each doing sequential work, pipelined:
//   warp T  the timing loop (A5): picks its soft symbol out of the staged tile (the warp's other lanes stage tiles one
//           ahead with 16-byte asynchronous copies), TED, PI loop, next fire clock; every emitted symbol goes into a ring
//           of records together with the loop state it left behind.
//   warp S  the symbol stages (A6-A9) on those records: squelch, equalizer, framer, events, transport.
// Until the squelch finds sync nothing the symbol stages do feeds back into the timing loop (receiver.rs:423-438,
// 479-490 all hang off sync / carrier-drop / burst-end), so T may run ahead of S by the ring.  When S's symbol locks the
// AGC (sync found: a burst begins) or resets the timing loop (end()), the record's state IS the receiver's state at that
// symbol: S stops the kernel there and whatever T did beyond it is dropped (T touches no global state).
// ctrl[0] in: end of the verified range (absolute position in the submit).  Out: ctrl[1] = position reached,
// ctrl[2] = why it stopped (0 range end, 1 AGC locked by the symbol stages, 2 timing loop reset by them).
#define LS_RING 64
struct LsRec { uint32_t pos; float zero, sym, until, pavg, pinst, ted0; uint32_t pad; };

// Ring counters.  LS_RELEASE_ACQUIRE=1: st.release.cta / ld.acquire.cta, the hand-off the PTX memory model defines (the
// acquire load is a plain LDS in SASS, the release store a MEMBAR.ALL.CTA + STS).  0: volatile accesses, relying on one
// thread's shared-memory stores being performed in program order.  Both are bit-exact over 24 h
// (tests/test_zz_config5_24h.py); profiles/README.md has the A/B.
#ifndef LS_RELEASE_ACQUIRE
#define LS_RELEASE_ACQUIRE 1
#endif
// The counters are published in batches (the release store's MEMBAR is what costs): T every LS_HEAD_BATCH records and
// when it finishes, S every LS_TAIL_BATCH records and whenever it has drained the ring.
#ifndef LS_HEAD_BATCH
#define LS_HEAD_BATCH 4u
#endif
#define LS_TAIL_BATCH 8u
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

__global__ void __launch_bounds__(64) same_long_seq_kernel(const __grid_constant__ SameParams p, const float* __restrict__ soft,
                                                           const float* __restrict__ yfull, const float* __restrict__ gspec,
                                                           const uint32_t pos0, uint32_t* __restrict__ ctrl) {
  __shared__ __align__(16) float tile[2][LS_TILE];
  __shared__ LsRec ring[LS_RING];
  __shared__ volatile uint32_t sh_head, sh_tail, sh_stop, sh_tdone;
  __shared__ float t_final[8];          // T's loop state at the end of the range: until, pavg, pinst, ted0, ted1, ted2, tedcnt, clock
  __shared__ uint32_t t_pos;
  const SameLayout& L = p.layout;
  const int lane = threadIdx.x & 31;
  const int role = threadIdx.x >> 5;   // 0 = T, 1 = S
  uint32_t* st = p.state32;            // stream 0
  StreamBlob* blob = p.blobs;
  const uint32_t range = ctrl[0] - pos0;   // samples that may be consumed
  if (threadIdx.x == 0) { sh_head = 0u; sh_tail = 0u; sh_stop = 0u; sh_tdone = 0u; }
  __syncthreads();

  Lane a;
  lane_load(a, p, st, 0u);
  uint32_t why = 0, stop_pos = 0;

  if (role == 0) {
    // ================================================ T: timing loop ================================================
    uint32_t pos = 0;                    // relative to pos0
    int cfire = fire_clock(a.until, a.clock);
    uint32_t done = 0, head = 0, tail_seen = 0;
    const auto stage = [&](uint32_t tbase, int buf) {   // `soft` is padded by two tiles: reading past `range` is harmless
      const uint32_t dst = (uint32_t)__cvta_generic_to_shared(&tile[buf][0]);
#pragma unroll 4
      for (uint32_t j = (uint32_t)lane * 4u; j < LS_TILE; j += 128u)
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst + j * 4u), "l"(soft + tbase + j) : "memory");
      asm volatile("cp.async.commit_group;" ::: "memory");
    };
    stage(0u, 0);
    int buf = 0;
    for (uint32_t tbase = 0; !done; tbase += LS_TILE, buf ^= 1) {
      stage(tbase + LS_TILE, buf ^ 1);
      asm volatile("cp.async.wait_group 1;" ::: "memory");
      __syncwarp();
      if (lane == 0) {
        const float* tl = &tile[buf][0];
        if (sh_stop) done = 1;                                           // checked per tile and while the ring is full
        while (!done) {
          const uint32_t next = pos + (uint32_t)(cfire - a.clock);      // position of the next TED instant
          if (next > range) {                                            // not inside the range: consume what is left
            a.clock += (int)(range - pos);
            pos = range;
            done = 1;
            break;
          }
          if (next >= tbase + LS_TILE) break;                            // in the next tile
          a.clock = cfire;
          pos = next;
          const float s_in = tl[pos - tbase];
          const float rem = FSUB(a.until, (float)a.clock);               // receiver.rs:352
          a.clock = 0;
          const bool have_sym = ted_step(a, p, s_in, rem);
          cfire = fire_clock(a.until, 0);
          if (have_sym) {
            if (head - tail_seen >= (uint32_t)LS_RING) {                   // ring full as far as T knows: look again, wait for S
              while (head - (tail_seen = ls_observe(&sh_tail)) >= (uint32_t)LS_RING) { if (sh_stop) { done = 1; break; } }
              if (done) break;
            }
            // the record, then the head counter that publishes it (ls_publish)
            volatile float* q = reinterpret_cast<volatile float*>(&ring[head & (LS_RING - 1)]);
            q[1] = a.ted1; q[2] = a.ted2; q[3] = a.until; q[4] = a.pavg; q[5] = a.pinst; q[6] = a.ted0;
            reinterpret_cast<volatile uint32_t*>(q)[0] = pos;
            head += 1u;
            if ((head & (LS_HEAD_BATCH - 1u)) == 0u) ls_publish(&sh_head, head);   // S may lag: it feeds back only by stopping
          }
        }
        if (done) {
          t_final[0] = a.until; t_final[1] = a.pavg; t_final[2] = a.pinst; t_final[3] = a.ted0; t_final[4] = a.ted1;
          t_final[5] = a.ted2; t_final[6] = __uint_as_float(a.tedcnt); t_final[7] = __int_as_float(a.clock);
          t_pos = pos;
          ls_publish(&sh_head, head);          // whatever the batching held back
          ls_publish(&sh_tdone, 1u);
        }
      }
      done = __shfl_sync(0xffffffffu, done, 0);
      __syncwarp();
    }
    asm volatile("cp.async.wait_group 0;" ::: "memory");
  } else if (lane == 0) {
    // ================================================ S: symbol stages ================================================
    uint32_t tail = 0, tail_pub = 0;
    while (true) {
      uint32_t head = ls_observe(&sh_head);
      if (tail == head) {
        if (tail_pub != tail) { ls_publish(&sh_tail, tail); tail_pub = tail; }   // ring drained: T may be waiting for room
        if (ls_observe(&sh_tdone)) { head = ls_observe(&sh_head); if (tail == head) break; }
        else continue;
      }
      LsRec r;
      {
        const volatile float* q = reinterpret_cast<const volatile float*>(&ring[tail & (LS_RING - 1)]);
        r.pos = reinterpret_cast<const volatile uint32_t*>(q)[0];
        r.zero = q[1]; r.sym = q[2]; r.until = q[3]; r.pavg = q[4]; r.pinst = q[5]; r.ted0 = q[6];
      }
      // The quiet symbol (nearly all of a long stream): no carrier, framer idle, nothing pending in the transport layer
      // and this symbol does not complete the sync word.  Then symbol_squelch + symbol_finish reduce to the squelch's
      // own bookkeeping (same expressions as same_lane.cuh:symbol_squelch, codesquelch.rs:228-304,421-428,483-488) --
      // written out here because a single lane pays for every instruction of the select-based general form.
      bool quiet = false;
      if (p.trace == nullptr && a.byteclk < 0 && a.fr.st == 0u && a.link_last == 0u) {
        const uint32_t nd = (a.sq_data >> 1) | ((r.sym >= 0.0f) ? 0x80000000u : 0u);
        const uint32_t cerr = __popc(nd ^ p.sq_sync_word);
        const float pw = fmaxf(FADD(a.sq_power, FMUL(FSUB(FMUL(r.sym, r.sym), a.sq_power), p.sq_bw)), 0.0f);
        const unsigned long long sc = a.symcount + 1ull;
        const unsigned long long n = a.n0 + r.pos;
        const bool acquire = sc >= 32ull && !(a.flags & FLAG_SQ_LOCK) && cerr <= p.sq_max_err && pw >= p.sq_open;
        const bool transport_due = (a.tr.have_eom && n > a.tr.eom_at) || sc >= a.tr.next_deadline ||
                                   ((a.tr.hist_n ? 1u : 0u) != a.tr.tr_state);
        if (!acquire && !transport_due) {
          LANE_ST(st, L, L.sqh + (a.sq_head & 63u)) = __float_as_uint(r.zero);
          LANE_ST(st, L, L.sqh + ((a.sq_head + 1u) & 63u)) = __float_as_uint(r.sym);
          a.sq_head = (a.sq_head + 2u) & 63u;
          a.sq_data = nd;
          a.sq_power = pw;
          a.sq_pflags = (a.sq_pflags >> 1) | ((pw >= p.sq_close) ? 0x80000000u : 0u);
          a.symcount = sc;
          quiet = true;
        }
      }
      if (quiet) {
        tail += 1u;
        if ((tail & (LS_TAIL_BATCH - 1u)) == 0u) { ls_publish(&sh_tail, tail); tail_pub = tail; }
        continue;
      }
      a.until = r.until; a.pavg = r.pavg; a.pinst = r.pinst;
      a.ted0 = r.ted0; a.ted1 = r.zero; a.ted2 = r.sym; a.tedcnt = 1u; a.clock = 0;
      symbol_step(a, p, 0u, st, blob, r.zero, r.sym, a.n0 + r.pos);
      tail += 1u;
      ls_publish(&sh_tail, tail);
      tail_pub = tail;
      if ((a.flags & FLAG_AGC_LOCKED) || a.tedcnt != 1u) {       // sync found (AGC locked) or end() reset the timing loop
        why = (a.flags & FLAG_AGC_LOCKED) ? 1u : 2u;
        stop_pos = r.pos;
        __threadfence_block();
        sh_stop = 1u;
        break;
      }
    }
  }
  __syncthreads();
  if (threadIdx.x != 32) return;
  // ---- state out (S's lane): the symbol stages' state + the timing loop's state at the stop symbol / at the range end ----
  uint32_t pos = stop_pos;
  if (why == 0u) {
    a.until = t_final[0]; a.pavg = t_final[1]; a.pinst = t_final[2]; a.ted0 = t_final[3]; a.ted1 = t_final[4];
    a.ted2 = t_final[5]; a.tedcnt = __float_as_uint(t_final[6]); a.clock = __float_as_int(t_final[7]);
    pos = t_pos;
  }
  if (pos > 0u) a.g = gspec[pos - 1u];
  lane_store(a, p, st, a.n0 + pos);
  for (int i = 0; i < FAST_NTAPS; ++i) LANE_ST(st, L, L.win + i) = __float_as_uint(yfull[pos + i]);
  ctrl[1] = pos0 + pos;
  ctrl[2] = why;
}

}  // namespace same_dev

// ----------------------------------------------------------------------------------------------------------------
// Launchers (called from same_engine.cu)
// ----------------------------------------------------------------------------------------------------------------
extern "C" cudaError_t same_long_launch_dc(const SameParams* p, const int16_t* d_src, uint32_t len, float* d, uint32_t* dc_next,
                                           cudaStream_t stream) {
  const uint32_t runs = (len + LS_RUN - 1u) / LS_RUN;
  same_dev::same_long_dc_kernel<<<(runs + 127u) / 128u, 128, 0, stream>>>(*p, d_src, len, d, dc_next);
  return cudaGetLastError();
}

extern "C" cudaError_t same_long_launch_commit_dc(const SameParams* p, const uint32_t* dc_next, cudaStream_t stream) {
  same_dev::same_long_commit_dc_kernel<<<1, 64, 0, stream>>>(*p, dc_next);
  return cudaGetLastError();
}

// B + verify + C + D for the range [pos0, end) of the submit; ctrl (device, 4 words) receives {verified end, position
// reached, reason}.  The caller presets nothing: ctrl[0] is set here.
extern "C" cudaError_t same_long_launch_speculative(const SameParams* p, const SameTaps2* taps2, const float* d, uint32_t pos0,
                                                    uint32_t end, float* yfull, float* gspec, float* g_in, float* soft,
                                                    uint32_t* ctrl, cudaStream_t stream) {
  const uint32_t n = end - pos0;
  const uint32_t blocks = (n + LS_BLOCK - 1u) / LS_BLOCK;
  cudaError_t err = cudaMemcpyAsync(ctrl, &end, sizeof(uint32_t), cudaMemcpyHostToDevice, stream);   // pageable source: staged
  if (err != cudaSuccess) return err;
  same_dev::same_long_agc_kernel<<<(blocks + 63u) / 64u, 64, 0, stream>>>(*p, d, pos0, end, yfull, gspec, g_in);
  if (blocks > 1u)
    same_dev::same_long_verify_kernel<<<(blocks - 1u + 127u) / 128u, 128, 0, stream>>>(gspec, g_in, pos0, end, ctrl);
  same_dev::same_long_mf_kernel<<<(n + 255u) / 256u, 256, 0, stream>>>(*taps2, yfull, n, soft);
  same_dev::same_long_seq_kernel<<<1, 64, 0, stream>>>(*p, soft, yfull, gspec, pos0, ctrl);
  return cudaGetLastError();
}
