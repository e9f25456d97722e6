// smooth_chain3.cuh -- sweep kernel of the chained strip smoother (smooth_chain.cuh explains the mapping and the
// {value, launch tag} protocol), third generation: WARP-SPECIALISED.
// Included by solver_kernels.cu after smooth_chain.cuh, inside namespace rlfc::{anonymous}.
//
// Measured on B200 (tools/ubench/shfl_lat.cu, profiles/r02_chain_sweeps.md): the loop-carried chain of one step
// (SHFL.UP of the previous result, select, 6 dependent FP ops without FMA) is 51.5 cycles; the first generation of the
// kernel (since removed) spent 156 cycles per step (cp.async bookkeeping, tag votes and operand addressing in the same
// warp), a batched single-warp variant 166 (two mbarrier waits at ~90 cycles and five bulk-copy issues per 8 steps).
// So everything that is not the chain moves to a second warp:
//   * CTA = one COMPUTE warp + one LOADER warp + one EDGE-FORWARDER warp per (sweep, strip);
//   * the loader streams the strip's operands in batches of kC3B steps with bulk copies (coefficients, r, previous
//     sweep's entries: contiguous along t in the strip-skewed layout), VALIDATES the tags of the previous sweep's entries
//     once they have landed (a stale batch is simply fetched again until its producer has passed) and only then hands
//     the batch to the compute warp through an mbarrier -- the compute warp never sees a tag;
//   * the two neighbour-strip operands (lane 0's S, lane 31's N) are the latency-critical ones: every strip-to-strip
//     hand-off is on the critical path of a sweep.  Producers write their lane-0 / lane-31 results to compact EDGE arrays
//     indexed by the consumer's step; the loader polls them 32 entries at a time with plain loads, forwards the run of
//     entries whose tag is current into a shared-memory ring of plain floats and publishes a counter;
//   * the compute warp: one mbarrier wait per batch, one counter check per 8 steps, and per step three shared-memory
//     loads, two shuffles, the arithmetic and two stores.
// Arithmetic per update, unchanged (MG.pde:85-86):  d = (dW*lxW + dE*lxE + dS*lyS + dN*lyN - r) * (-inv).
#pragma once

#ifndef RLFC_C3B
#define RLFC_C3B 16
#endif
#ifndef RLFC_C3SLOTS
#define RLFC_C3SLOTS 4
#endif
constexpr int kC3B = RLFC_C3B;           // steps per batch (multiple of 8)
constexpr int kC3Slots = RLFC_C3SLOTS;   // batches in flight
#ifndef RLFC_C3_LSLEEP
#define RLFC_C3_LSLEEP 0
#endif
#ifndef RLFC_C3_FSLEEP
#define RLFC_C3_FSLEEP 0
#endif
constexpr int kC3EdgeRing = 128;         // entries of the edge ring (power of two, >= 64)

struct __align__(128) Chain3Smem {
  float4 coef[kC3Slots][kC3B][32];       // {lx[i+1][j], ly[i][j], ly[i][j+1], -inv[i][j]}
  float r[kC3Slots][kC3B][32];
  uint2 e[kC3Slots][kC3B][32];           // previous sweep, entries t+1
  float edge[2][kC3EdgeRing];            // [0] S of lane 0, [1] N of lane 31, validated, by step & (ring - 1)
  unsigned long long full[kC3Slots];     // bulk copies of the slot have landed        (waited for by the loader)
  unsigned long long ready[kC3Slots];    // loader -> compute: batch validated
  unsigned long long empty[kC3Slots];    // compute -> loader: batch consumed
  int edge_ready;                        // loader -> compute: edge operands of steps < edge_ready are in the ring
  int compute_pos;                       // compute -> loader: steps < compute_pos are done
#ifdef RLFC_CHAIN_STATS
  unsigned long long dbg_forward;
  int dbg_run;
#endif
};

__device__ __forceinline__ int c3_lds_volatile(const int* p) {
  int v;
  asm volatile("ld.volatile.shared.s32 %0, [%1];" : "=r"(v) : "r"((unsigned)__cvta_generic_to_shared(p)) : "memory");
  return v;
}
__device__ __forceinline__ void c3_sts_volatile(int* p, int v) {
  asm volatile("st.volatile.shared.s32 [%0], %1;" ::"r"((unsigned)__cvta_generic_to_shared(p)), "r"(v) : "memory");
}
__device__ __forceinline__ float4 c3_lds128v(unsigned a) {
  float4 v;
  asm volatile("ld.volatile.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(a) : "memory");
  return v;
}
// {value, tag} hand-offs: device scope on one GPU; system scope when strips of one sweep run on several devices (slab mode)
template <bool SYS>
__device__ __forceinline__ void c3_st64(uint2* p, unsigned v, unsigned tag) {
  if (SYS) asm volatile("st.relaxed.sys.global.v2.u32 [%0], {%1,%2};" ::"l"(p), "r"(v), "r"(tag) : "memory");
  else asm volatile("st.relaxed.gpu.global.v2.u32 [%0], {%1,%2};" ::"l"(p), "r"(v), "r"(tag) : "memory");
}
template <bool SYS>
__device__ __forceinline__ uint2 c3_ld64(const uint2* p) {
  uint2 v;
  if (SYS) asm volatile("ld.relaxed.sys.global.v2.u32 {%0,%1}, [%2];" : "=r"(v.x), "=r"(v.y) : "l"(p) : "memory");
  else asm volatile("ld.relaxed.gpu.global.v2.u32 {%0,%1}, [%2];" : "=r"(v.x), "=r"(v.y) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void c3_mbar_arrive(unsigned long long* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"((unsigned)__cvta_generic_to_shared(bar)) : "memory");
}
__device__ __forceinline__ bool c3_mbar_test(unsigned long long* bar, unsigned parity) {
  unsigned ok;
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n"
      "selp.u32 %0, 1, 0, p;\n"
      "}\n" : "=r"(ok) : "r"((unsigned)__cvta_generic_to_shared(bar)), "r"(parity) : "memory");
  return ok != 0;
}

template <bool SYS>
__global__ void __launch_bounds__(96)
k_chain_sweeps3(const __grid_constant__ SolverParams q, int level) {
  using namespace rows_detail;           // mbarrier / bulk-copy wrappers (smooth_rows.cuh)
  extern __shared__ __align__(16) unsigned char ch_smem[];
  __shared__ unsigned long long s_ticket;
  const DevLevel& Lv = q.lev[level];
  const ChainLevel& ch = Lv.ch;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const unsigned long long G = (unsigned long long)q.B * 4ull * (unsigned)ch.ns_loc;
  Chain3Smem& R = *reinterpret_cast<Chain3Smem*>(ch_smem);
  if (threadIdx.x == 0) {
    s_ticket = atomicAdd(ch.ticket, 1ull);
    for (int k = 0; k < kC3Slots; k++) { mbar_init(&R.full[k], 1); mbar_init(&R.ready[k], 1); mbar_init(&R.empty[k], 1); }
    R.edge_ready = 0;
    R.compute_pos = 0;
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    fence_proxy_async();
  }
  __syncthreads();
  const unsigned long long ticket = s_ticket;
  const unsigned tag = ch.tag_hi | (unsigned)((ticket / G) & 0x3ffffffull);      // same for every CTA of this launch
  const unsigned role = (unsigned)(ticket % G);
  const int e = (int)(role / (4u * ch.ns_loc)), rem = (int)(role % (4u * ch.ns_loc));
  const int g = rem / ch.ns_loc + 1;
  const int s = ch.s0 + rem % ch.ns_loc;
  if (!q.sc.active[e]) return;
  const int ni = Lv.n - 2, T = ch.T, NS = ch.NS;
  const int Tend = ni + 32;                                   // entries 0 .. Tend carry rows 0 .. ni+1 of every lane
  const int nbat = (Tend + kC3B) / kC3B;                      // batches; steps up to kC3B nbat - 1 < T stay inside the strip
  const int nsteps = nbat * kC3B;
  const size_t eo = (size_t)e * ch.sk_stride;
  const unsigned tagp = (g == 1) ? 0u : tag;                  // sweep 0 (= r*inv) was written by the kernel before this one
  const bool hasS = s > 0, hasN = s + 1 < NS;

  if (warp == 2) {
    // ====================================== EDGE FORWARDER ======================================
    // Polls the two edge arrays 32 steps at a time and forwards the leading run of entries whose tag is current.  This
    // loop's period (one L2 round trip) is part of every strip-to-strip hand-off, hence a warp of its own.
    const uint2* g_es = c2_edge(ch, g, 0, e, hasS ? s - 1 : s) + kC2EdgePad;       // by consumer step
    const uint2* g_en = c2_edge(ch, g - 1, 1, e, hasN ? s + 1 : s) + kC2EdgePad;
    int efill = 0;                                            // edge operands of steps < efill are in the ring
    int cpos = 0;
    unsigned idle = 0;
#ifdef RLFC_CHAIN_STATS
    unsigned n_polls = 0, n_full = 0;
    unsigned long long fw_t0, fw_t1;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(fw_t0));
#endif
    while (efill < nsteps) {
#ifdef RLFC_CHAIN_STATS
      if (efill + 32 > cpos + kC3EdgeRing) n_full++; else n_polls++;
#endif
      if (efill + 32 > cpos + kC3EdgeRing) {                  // ring full: wait for the compute warp (without hammering
        __nanosleep(200);                                     // the shared-memory port it loads its operands through)
        cpos = c3_lds_volatile(&R.compute_pos);
        if (++idle > kChSpinMax) __trap();
        continue;
      }
      const int te = efill + lane;
      uint2 vs = make_uint2(0u, tag), vn = make_uint2(0u, tagp);
      if (hasS && te >= 1 && te <= ni) vs = c3_ld64<SYS>(g_es + te);
      if (hasN && te >= 32 && te <= ni + 31) vn = c3_ld64<SYS>(g_en + te);
      const unsigned okm = __ballot_sync(0xffffffffu, vs.y == tag && vn.y == tagp);
      const int cnt = (okm == 0xffffffffu) ? 32 : (__ffs(~okm) - 1);            // leading run of current entries
      const int lim = min(cnt, nsteps - efill);
      if (lane < lim) {
        R.edge[0][te & (kC3EdgeRing - 1)] = __uint_as_float(vs.x);
        R.edge[1][te & (kC3EdgeRing - 1)] = __uint_as_float(vn.x);
      }
      __syncwarp();
      if (lim > 0) {
#ifdef RLFC_CHAIN_STATS
        if (lane == 0 && g == 1 && level == 0 && (ticket / G) == RLFC_CHAIN_STATS && efill <= 969 && efill + lim > 969) {
          unsigned long long tt; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(tt));
          R.dbg_forward = tt; R.dbg_run = lim;
        }
#endif
        efill += lim;
        if (lane == 0) c3_sts_volatile(&R.edge_ready, efill);
        idle = 0;
      } else {
        if (++idle > kChSpinMax) __trap();                    // a tag that never comes is a bug, and a trap beats a hung GPU
#if RLFC_C3_FSLEEP > 0
        __nanosleep(RLFC_C3_FSLEEP);
#endif
      }
    }
#ifdef RLFC_CHAIN_STATS
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(fw_t1));
    if (lane == 0 && g == 1 && level == 0 && (ticket / G) == RLFC_CHAIN_STATS)
      printf("fwd s%d polls %u full %u time %llu ns\n", s, n_polls, n_full, fw_t1 - fw_t0);
#endif
    return;
  }
  if (warp == 1) {
    // =========================================== LOADER ===========================================
    const char* g_coef = reinterpret_cast<const char*>(ch.ct + (size_t)s * T * 32);
    const char* g_r = reinterpret_cast<const char*>(ch.rsk + eo + (size_t)s * T * 32);
    const char* g_e = reinterpret_cast<const char*>(ch.dsk[g - 1] + eo + ((size_t)s * T + 1) * 32);
    int b_issue = 0, b_valid = 0;                             // next batch to fetch / to validate
    unsigned ph_full = 0, ph_empty = 0;                       // phase parity per slot (bit = slot)
    bool settling = false;                                    // a stale batch was seen: wait for the producer to pass the
    unsigned idle = 0;                                        // furthest batch in flight, then fetch all of them again
    while (b_valid < nbat) {
      bool progress = false;
      if (settling) {
        const int tl = min(b_issue * kC3B - 1, Tend - 1);     // last step in flight whose E operand is checked
        const bool ok = c3_ld64<SYS>(reinterpret_cast<const uint2*>(g_e + (size_t)tl * 256) + lane).y == tagp;
        if (__all_sync(0xffffffffu, ok)) {
          for (int bb = b_valid + 1; bb < b_issue; bb++) {    // drain the copies in flight (stale), ...
            const int sl = bb % kC3Slots;
            mbar_wait(&R.full[sl], (ph_full >> sl) & 1u);
            ph_full ^= 1u << sl;
          }
          __syncwarp();
          if (lane == 0)
            for (int bb = b_valid; bb < b_issue; bb++) {      // ... fetch the entries of all of them again
              const int sl = bb % kC3Slots;
              mbar_expect_tx(&R.full[sl], (unsigned)(kC3B * 256));
              bulk_g2s(&R.e[sl][0][0], g_e + (size_t)bb * (kC3B * 256), kC3B * 256u, &R.full[sl]);
            }
          settling = false;
          progress = true;
        }
      } else {
        // ---- fetch ahead ----
        if (b_issue < nbat) {
          const int slot = b_issue % kC3Slots;
          bool free_slot = b_issue < kC3Slots;
          if (!free_slot && c3_mbar_test(&R.empty[slot], (ph_empty >> slot) & 1u)) { free_slot = true; ph_empty ^= 1u << slot; }
          if (free_slot) {
            if (lane == 0) {
              mbar_expect_tx(&R.full[slot], (unsigned)(kC3B * (512 + 128 + 256)));
              bulk_g2s(&R.coef[slot][0][0], g_coef + (size_t)b_issue * (kC3B * 512), kC3B * 512u, &R.full[slot]);
              bulk_g2s(&R.r[slot][0][0], g_r + (size_t)b_issue * (kC3B * 128), kC3B * 128u, &R.full[slot]);
              bulk_g2s(&R.e[slot][0][0], g_e + (size_t)b_issue * (kC3B * 256), kC3B * 256u, &R.full[slot]);
            }
            b_issue++;
            progress = true;
          }
        }
        // ---- validate the oldest batch in flight, hand it over ----
        if (b_valid < b_issue) {
          const int slot = b_valid % kC3Slots;
          if (c3_mbar_test(&R.full[slot], (ph_full >> slot) & 1u)) {
            ph_full ^= 1u << slot;
            bool bad = false;
            if (g > 1) {
              const int t0 = b_valid * kC3B;
#pragma unroll 4
              for (int k = 0; k < kC3B; k++) bad |= (t0 + k < Tend) && R.e[slot][k][lane].y != tagp;
            }
            if (__any_sync(0xffffffffu, bad)) {
              settling = true;                                // the producer is less than the prefetch distance ahead
            } else {
              __syncwarp();
              if (lane == 0) c3_mbar_arrive(&R.ready[slot]);
              b_valid++;
            }
            progress = true;
          }
        }
      }
      if (progress) idle = 0;
      else {
        if (++idle > kChSpinMax) __trap();
#if RLFC_C3_LSLEEP > 0
        __nanosleep(RLFC_C3_LSLEEP);                          // (do not hammer the shared-memory port the compute warp loads through)
#endif
      }
    }
    return;
  }

  // ============================================= COMPUTE =============================================
  const unsigned a_ring = sm_addr(&R);
  const unsigned a_edge = a_ring + (unsigned)offsetof(Chain3Smem, edge) + (lane == 0 ? 0u : 4u * kC3EdgeRing);
  const bool l0 = lane == 0, l31 = lane == 31;
  // results: every lane its element of the strip-skewed array; lanes 0 / 31 also the edge arrays, by consumer step
  uint2* out = ch.dsk[g] + eo + (size_t)s * T * 32 + lane;
  uint2* eout = (l0 ? c2_edge(ch, g, 1, e, s) + 31 : c2_edge(ch, g, 0, e, s) - 31) + kC2EdgePad;
  const bool edge_lane = l0 || l31;
  float W = 0.f, cxW = 0.f;
  unsigned ph_ready = 0;
  int slot = 0;
#ifdef RLFC_CHAIN_STATS
  unsigned long long st_t0, st_t1, st_consume = 0, st_produce = 0;
  unsigned st_spins = 0;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(st_t0));
#endif
  for (int b = 0; b < nbat; b++) {
    mbar_wait(&R.ready[slot], (ph_ready >> slot) & 1u);
    ph_ready ^= 1u << slot;
    const unsigned a_c = a_ring + (unsigned)offsetof(Chain3Smem, coef) + (unsigned)slot * (kC3B * 512u) + 16u * lane;
    const unsigned a_r = a_ring + (unsigned)offsetof(Chain3Smem, r) + (unsigned)slot * (kC3B * 128u) + 4u * lane;
    const unsigned a_e = a_ring + (unsigned)offsetof(Chain3Smem, e) + (unsigned)slot * (kC3B * 256u) + 8u * lane;
#pragma unroll 1
    for (int h = 0; h < kC3B / 8; h++) {
      const int t0 = b * kC3B + h * 8;
      while (c3_lds_volatile(&R.edge_ready) < t0 + 8) {
#ifdef RLFC_CHAIN_STATS
        st_spins++;
#endif
      }
#ifdef RLFC_CHAIN_STATS
      if (lane == 0 && g == 1 && level == 0 && (ticket / G) == RLFC_CHAIN_STATS && (t0 == 968 || t0 == 1000)) {
        unsigned long long tt; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(tt));
        if (t0 == 968) st_consume = tt; else st_produce = tt;
      }
#endif
      const unsigned a_x = a_edge + 4u * ((unsigned)t0 & (kC3EdgeRing - 1));
      float4 cn = c3_lds128v(a_c + 512u * (8 * h));
#pragma unroll
      for (int k = 0; k < 8; k++) {
        // (volatile loads and stores keep their program order in the SASS: the coefficient load of step k+1 sits between
        // the stores of steps k-1 and k, which pins every store to its own step instead of the end of the block)
        const float4 c = cn;
        if (k + 1 < 8) cn = c3_lds128v(a_c + 512u * (8 * h + k + 1));
        const float rv = ch_lds32(a_r + 128u * (8 * h + k));
        const float E = ch_lds32(a_e + 256u * (8 * h + k));
        const float axv = ch_lds32(a_x + 4u * k);
        float S = __shfl_up_sync(0xffffffffu, W, 1);          // the loop-carried chain
        float N = __shfl_down_sync(0xffffffffu, E, 1);
        if (l31) N = axv;
        if (l0) S = axv;
        const float res = (W * cxW + E * c.x + S * c.y + N * c.z - rv) * c.w;      // MG.pde:85-86
        if (edge_lane) c3_st64<SYS>(eout + t0 + k, __float_as_uint(res), tag);
        c3_st64<SYS>(out + (size_t)k * 32, __float_as_uint(res), tag);
        W = res;
        cxW = c.x;
      }
      out += 8 * 32;
    }
    __syncwarp();
    if (lane == 0) {
      c3_mbar_arrive(&R.empty[slot]);
      c3_sts_volatile(&R.compute_pos, (b + 1) * kC3B);
    }
    slot = (slot + 1 == kC3Slots) ? 0 : slot + 1;
  }
#ifdef RLFC_CHAIN_STATS
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(st_t1));
  if (lane == 0 && (ticket / G) == RLFC_CHAIN_STATS)
    printf("chain L%d g%d s%d start %llu end %llu miss %u spins %u steps %d\n", level, g, s, st_t0, st_t1, 0u, st_spins, Tend + 1);
  if (lane == 0 && g == 1 && level == 0 && (ticket / G) == RLFC_CHAIN_STATS)
    printf("hop s%d forward969 %llu run %d consume968 %llu produce1000 %llu\n", s, R.dbg_forward - st_t0, R.dbg_run, st_consume - st_t0, st_produce - st_t0);
#endif
}
