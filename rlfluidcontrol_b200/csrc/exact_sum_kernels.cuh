// exact_sum_kernels.cuh -- Field.sum (Field.pde:311-318) as two kernels around exact_sum.cuh:
//   k_xsum_tables  one thread per segment of 32 additions: predicted accumulator before the segment (chunk totals
//                  handed from CTA to CTA + block scan), then the segment summary (exact_sum.cuh); each warp condenses
//                  its 32 summaries into a batch record of a few "table + float additions" entries
//   k_xsum_chain   one warp per environment walks the batch records with the true accumulator; a batch whose record
//                  does not provably apply is redone as genuine float additions
// The result is bit-identical to the serial loop for any input (tests/test_exact_sum.py, tests/test_gpu_parity.py).
// Included by solver_kernels.cu inside namespace rlfc::{anonymous}.
#pragma once
// (exact_sum.cuh is included at file scope by solver_kernels.cu)

constexpr int kXsThreads = 256;
constexpr int kXsChunk = kXsThreads * xsum::kSeg;       // additions per CTA
constexpr int kXsPad = xsum::kSeg + 1;                  // shared-memory stride of a segment (bank-conflict free)
constexpr int kXsEntWords = 12;                         // record entry: table (7), three float additions, 2 unused
constexpr int kXsRecEntries = 15;
constexpr int kXsRecWords = 8 + kXsRecEntries * kXsEntWords + 4;   // batch record: 8 header words + entries (192 words)

// Chunk loader: serial index K (i-major over the interior) -> pitched array.  The pointer update is branch-free when
// a row is at least half a CTA wide (WIDE: at most two row ends per stride of kXsThreads elements), so that the loads
// of the unrolled loop are not separated by control flow.
template <bool WIDE>
__device__ __forceinline__ void xs_fill(const SolverParams& q, const float* p, long long base, long long N, int t, float* buf) {
  // 32-bit incremental addressing (rlfc_env_create rejects grids beyond 2^31 cells): element K = base + t + 256 u
  // sits at row 1 + K / len, column 1 + K % len; a stride of 256 elements passes at most two row ends when WIDE.
  const int len = q.m - 2, P = q.P, skip = P - len;
  const unsigned k0 = (unsigned)base + (unsigned)t;
  int j = 1 + (int)(k0 % (unsigned)len);
  int off = (1 + (int)(k0 / (unsigned)len)) * P + j;
  const int left = (int)((N - base) < (long long)kXsChunk ? (N - base) : (long long)kXsChunk) - t;   // u*256 < left <=> in range
  float* dst = buf + (t >> 5) * kXsPad + (t & 31);                // local index t + 256 u: segment (t >> 5) + 8 u
  const float* ptr = p + off;                                     // running pointer: one 64-bit add per element
  const unsigned uskip = (unsigned)skip;
  asm volatile("" : "+l"(ptr), "+r"(j));                          // keep them in registers (no rematerialisation per load)
#pragma unroll 8
  for (int u = 0; u < xsum::kSeg; u++) {
    dst[u * (kXsThreads / 32) * kXsPad] = (u * kXsThreads < left) ? *ptr : 0.f;
    j += kXsThreads;
    unsigned inc = kXsThreads;
    if (WIDE) {
      const bool a = j > len; j -= a ? len : 0; inc += a ? uskip : 0u;
      const bool b = j > len; j -= b ? len : 0; inc += b ? uskip : 0u;
    } else {
      while (j > len) { j -= len; inc += uskip; }
    }
    ptr += inc;
  }
}

// PASS (large domains only; 0 otherwise): 1 = first of two passes -- also records, per batch, the predicted accumulator at
// its start and what the batch really does to a float accumulator (its table's increment: the rounding BIAS of a long run
// of small addends against a large accumulator is systematic, thousands of ulps per million additions, and the exact
// prefix sums the prediction is made of know nothing about it); k_xsum_refine turns these into a per-batch correction;
// 2 = second pass: the prediction includes that correction, so the records are built for the binade the accumulator is
// really in.  A prediction is only a prediction: exactness rests on the validity checks of the serial pass alone.
template <int PASS>
__global__ void __launch_bounds__(kXsThreads)
k_xsum_tables(const __grid_constant__ SolverParams q) {
  __shared__ float buf[kXsThreads * kXsPad];
  __shared__ double wsum[kXsThreads / 32];
  __shared__ double base_pred;
  __shared__ double wpart[kXsThreads / 32];
  const int e = blockIdx.x, c = blockIdx.y, t = threadIdx.x, lane = t & 31, warp = t >> 5;
  if (q.sc.frozen[e]) return;
  const int len = q.m - 2;
  const long long N = (long long)(q.n - 2) * len, base = (long long)c * kXsChunk;
  const float* p = q.lev[0].x + (size_t)e * q.stride;
  if (2 * len >= kXsThreads) xs_fill<true>(q, p, base, N, t, buf);
  else xs_fill<false>(q, p, base, N, t, buf);
  __syncthreads();
  const long long g = (long long)c * kXsThreads + t;              // this thread's segment
  const long long left = N - g * xsum::kSeg;
  const int cnt = left >= xsum::kSeg ? xsum::kSeg : (left > 0 ? (int)left : 0);
  const float* seg = buf + t * kXsPad;
  float fsum = 0.f;                                               // a prediction only: float precision is plenty
#pragma unroll 8
  for (int k = 0; k < xsum::kSeg; k++) fsum += seg[k];            // (tail elements are stored as +0)
  const double ssum = (double)fsum;
  // exclusive scan of the segment sums over the CTA
  double incl = ssum;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const double v = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += v;
  }
  if (lane == 31) wsum[warp] = incl;
  __syncthreads();
  {
    // Chunk totals travel between the CTAs of one environment through global memory (single pass, "look-back"):
    // publish this chunk's total, then wait for the totals of the chunks before it.  CTAs are dispatched in
    // blockIdx order and the chunk index is the SLOW grid dimension, so the CTAs waited for started a whole row of
    // environments earlier and have normally published already; the wait is bounded
    // all the same -- the total only feeds the PREDICTION, a wrong one merely sends segments to the serial path.
    const unsigned ep = q.xs_epoch[e] + 1u;                       // k_xsum_chain bumps the epoch after every pass
    volatile double* ct = q.xs_ctot + (size_t)e * q.xs_nchunks;
    volatile unsigned* cf = q.xs_cflag + (size_t)e * q.xs_nchunks;
    if (t == 0) {
      double tot = 0.0;
      for (int w = 0; w < kXsThreads / 32; w++) tot += wsum[w];
      ct[c] = tot;
      __threadfence();
      cf[c] = ep;
    }
    double part = 0.0;
    for (int k = t; k < c; k += kXsThreads) {
      int spins = 0;
      while (cf[k] != ep && ++spins < (1 << 20)) {}
      __threadfence();
      part += ct[k];
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) part += __shfl_down_sync(0xffffffffu, part, o);
    if (lane == 0) wpart[warp] = part;
    __syncthreads();
    if (t == 0) {
      double bsum = 0.0;
      for (int w = 0; w < kXsThreads / 32; w++) bsum += wpart[w];
      base_pred = bsum;
    }
  }
  __syncthreads();
  double pred = base_pred;
  for (int w = 0; w < warp; w++) pred += wsum[w];
  const long long batch_ = (long long)c * (kXsThreads / 32) + warp;
  if (PASS == 1 && lane == 0 && batch_ < q.xs_nbatches) q.xs_pred[(size_t)e * q.xs_nbatches + batch_] = pred;
  if (PASS >= 2 && batch_ < q.xs_nbatches) pred += q.xs_corr[(size_t)e * q.xs_nbatches + batch_];
  pred += incl - ssum;
  uint32_t slot[xsum::kSlotWords];
  if (cnt > 0) {
    xsum::build_segment([&](int k) { return seg[k]; }, cnt, pred, slot);
  } else {                                                        // past the end: an empty table
#pragma unroll
    for (int w = 0; w < xsum::kSlotWords; w++) slot[w] = 0u;
    slot[0] = xsum::kOne; slot[1] = xsum::kAnyKey;
  }
  // Batch record: the 32 summaries of this warp (= one batch of the serial pass) condensed into a few entries
  // "table, then one float addition".  A split or serial summary (a "head") closes the running group of tables:
  //   C_k = table of the group that is open after slot k  (head: what it restarts with -- the second table of
  //         a split summary, nothing for a serial one; otherwise C_{k-1} followed by the slot's table),
  //   E_k = C_{k-1} followed by the head's first table = the entry that ends at head k, with the head's float
  //         addition (split) or the 32 genuine additions of the segment (serial) right behind it;
  // the last entry is C_31.  C is a Kogge-Stone scan of table compositions, segmented at the heads.
  {
    const uint32_t type = slot[0];
    const bool head = type != xsum::kOne;
    uint32_t X[7], acc[7];
    const uint32_t ident[7] = {xsum::kAnyKey, 0u, 0u, (uint32_t)INT32_MIN, (uint32_t)INT32_MAX, (uint32_t)INT32_MIN, (uint32_t)INT32_MAX};
    xsum::normalise_table(slot + 1);
    if (type == xsum::kSplit) xsum::normalise_table(slot + xsum::kSlotB);
#pragma unroll
    for (int w = 0; w < 7; w++) {
      X[w] = (type == xsum::kSerial) ? ident[w] : slot[1 + w];
      acc[w] = (type == xsum::kOne) ? slot[1 + w] : (type == xsum::kSplit ? slot[xsum::kSlotB + w] : ident[w]);
    }
    const uint32_t headmask = __ballot_sync(0xffffffffu, head);
    const uint32_t upto = headmask & ((2u << lane) - 1u);         // heads at or below this lane
    const int dist = lane - (upto ? 31 - __clz(upto) : 0);
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      uint32_t prev[7];
#pragma unroll
      for (int w = 0; w < 7; w++) prev[w] = __shfl_up_sync(0xffffffffu, acc[w], o);
      if (dist >= o) xsum::compose_tables(prev, acc);
    }
    uint32_t cprev[7];
#pragma unroll
    for (int w = 0; w < 7; w++) {
      cprev[w] = __shfl_up_sync(0xffffffffu, acc[w], 1);
      if (lane == 0) cprev[w] = ident[w];
    }
    xsum::compose_tables(cprev, X);                               // X = E_k on head lanes
    // a run of consecutive serial summaries is ONE entry: the table before it, then `run` whole segments
    const uint32_t sermask = __ballot_sync(0xffffffffu, type == xsum::kSerial);
    const bool absorbed = type == xsum::kSerial && lane > 0 && ((sermask >> (lane - 1)) & 1u);
    const uint32_t emitmask = __ballot_sync(0xffffffffu, head && !absorbed);
    const int idx = __popc(emitmask & ((1u << lane) - 1u));       // entry index of an emitting head lane
    const int count = __popc(emitmask) + 1;
    // serial summaries from this lane on (all the way to lane 31: the shifted mask has no zero bit left when lane == 0)
    const uint32_t nser = ~(sermask >> lane);
    const int run = type == xsum::kSerial ? (nser ? __ffs(nser) - 1 : 32 - lane) : 0;
    const long long batch = (long long)c * (kXsThreads / 32) + warp;
    if (batch < q.xs_nbatches) {
      uint32_t* rec = q.xs_recs + ((size_t)e * q.xs_nbatches + batch) * kXsRecWords;
      if (lane == 0)
        *reinterpret_cast<uint4*>(rec) = make_uint4(count <= kXsRecEntries ? (uint32_t)count : 0xffffffffu, sermask, 0u, 0u);
      if ((PASS == 1 || PASS == 3) && lane == 31 && count > kXsRecEntries) q.xs_inc[(size_t)e * q.xs_nbatches + batch] = incl;
      if (count <= kXsRecEntries) {
        const uint32_t nz = xsum::kNegZero;                        // serial heads and the last entry add nothing
        if (head && !absorbed) {
          const bool sp = type == xsum::kSplit;
          uint4* ent = reinterpret_cast<uint4*>(rec + 8 + kXsEntWords * idx);
          ent[0] = make_uint4(X[0], X[1], X[2], X[3]);
          ent[1] = make_uint4(X[4], X[5], X[6], sp ? slot[xsum::kSlotRaw] : nz);
          ent[2] = make_uint4(sp ? slot[xsum::kSlotRaw + 1] : nz, sp ? slot[xsum::kSlotRaw + 2] : nz, (uint32_t)run, (uint32_t)lane);
        }
        if ((PASS == 1 || PASS == 3) && lane == 31) {
          // the batch's effect on a float accumulator: the table's increment where the batch is one valid table,
          // otherwise its exact sum
          double inc = incl;
          if (count == 1 && acc[0] != xsum::kAnyKey && (int32_t)acc[3] != xsum::kNever) {
            const int ex = (int)(acc[0] & 255u);
            inc = ldexp((double)(int32_t)acc[1], ex - 150);
            if (acc[0] >> 8) inc = -inc;
          }
          q.xs_inc[(size_t)e * q.xs_nbatches + batch] = inc;
        }
        if (lane == 31) {
          uint4* ent = reinterpret_cast<uint4*>(rec + 8 + kXsEntWords * (count - 1));
          ent[0] = make_uint4(acc[0], acc[1], acc[2], acc[3]);
          ent[1] = make_uint4(acc[4], acc[5], acc[6], nz);
          ent[2] = make_uint4(nz, nz, 0u, 0u);
        }
      }
    }
  }
}

// Between the two table passes of a large domain: prefix sums of the batches' float increments = the refined prediction
// of the accumulator at every batch start; its difference from the first pass's prediction is the correction.
__global__ void __launch_bounds__(1024)
k_xsum_refine(const __grid_constant__ SolverParams q) {
  __shared__ double wtot[32];
  const int e = blockIdx.x, t = threadIdx.x, lane = t & 31, warp = t >> 5;
  if (q.sc.frozen[e]) return;
  const int nb = q.xs_nbatches, per = (nb + 1023) / 1024;
  const double* inc = q.xs_inc + (size_t)e * nb;
  const double* pred = q.xs_pred + (size_t)e * nb;
  double* corr = q.xs_corr + (size_t)e * nb;
  const int b0 = t * per, b1 = min(b0 + per, nb);
  double mine = 0.0;
  for (int b = b0; b < b1; b++) mine += inc[b];
  double incl = mine;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const double v = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += v;
  }
  if (lane == 31) wtot[warp] = incl;
  __syncthreads();
  double run = incl - mine;
  for (int w = 0; w < warp; w++) run += wtot[w];
  for (int b = b0; b < b1; b++) {
    corr[b] = run - pred[b];
    run += inc[b];
  }
}

// Serial pass.  One warp per environment walks the batch records: per entry one table application (checked),
// three float additions, and the genuine additions of a run of serial segments where the entry says so.  If any
// entry of a batch does not provably apply (or the batch has too many heads for a record), the whole batch is
// redone from its start as 1024 genuine float additions.
constexpr int kXsGroup = kXsThreads / 32;   // batch records per cp.async group = one chunk of k_xsum_tables; the ring holds two
constexpr int kXsRawPf = 4;       // serial segments per batch whose elements are prefetched

__device__ __forceinline__ void xs_cp16(void* smem, const void* gmem) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((unsigned)__cvta_generic_to_shared(smem)), "l"(gmem) : "memory");
}

__device__ __forceinline__ void xs_cp4(void* smem, const void* gmem) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"((unsigned)__cvta_generic_to_shared(smem)), "l"(gmem) : "memory");
}

__global__ void __launch_bounds__(32)
k_xsum_chain(const __grid_constant__ SolverParams q) {
  __shared__ __align__(16) uint32_t ring[2 * kXsGroup][kXsRecWords];
  __shared__ float stage[32][32];
  const int e = blockIdx.x, lane = threadIdx.x;
  if (q.sc.frozen[e]) return;
  const unsigned len = (unsigned)(q.m - 2), P = (unsigned)q.P;
  const unsigned N = (unsigned)(q.n - 2) * len;                   // rlfc_env_create rejects grids beyond 2^31 cells
  const int nseg = q.xs_nseg, nb = q.xs_nbatches;
  const float* p = q.lev[0].x + (size_t)e * q.stride;
  const uint32_t* recs = q.xs_recs + (size_t)e * nb * kXsRecWords;
  auto element = [&](unsigned g) {                                 // this lane's element of segment g (-0 past the end:
    const unsigned K = g * xsum::kSeg + lane;                      //  s + -0.f == s for every s)
    return K < N ? p[(size_t)(1u + K / len) * P + 1u + K % len] : -0.f;
  };
  auto fetch = [&](int grp) {                                     // records of batches grp*kXsGroup ..; one commit group
    const int b0 = grp * kXsGroup, n16 = min(kXsGroup, nb - b0) * (kXsRecWords / 4);   // 16-byte pieces (contiguous records)
    uint32_t* dst = ring[b0 % (2 * kXsGroup)];
    const uint32_t* src = recs + (size_t)b0 * kXsRecWords;
    for (int k = lane; k < n16; k += 32) xs_cp16(dst + 4 * k, src + 4 * k);
    asm volatile("cp.async.commit_group;" ::: "memory");
  };
  // xs_stats[e][0..3]: batches crossed by their record / walked summary by summary, record entries applied,
  // segments redone as float additions
  int st_rec = 0, st_walk = 0, st_ent = 0, st_redo = 0;
#ifdef RLFC_XS_TIMING           // cycles: [4] batch set-up + prefetch, [5] record entries, [6] serial segments, [7] walks
  long long tk = clock64(), tacc[4] = {0, 0, 0, 0};
#define XS_TICK(i) do { const long long n_ = clock64(); tacc[i] += n_ - tk; tk = n_; } while (0)
#else
#define XS_TICK(i)
#endif
  uint32_t bits = 0u;                                             // s = +0.f
  // 32 genuine additions of segment g; lane u holds element u in v
  auto redo = [&](float v) {
    st_redo++;
    float el[xsum::kSeg];
#pragma unroll
    for (int u = 0; u < xsum::kSeg; u++) el[u] = __shfl_sync(0xffffffffu, v, u);
    float s = xsum::u2f(bits);
#pragma unroll
    for (int u = 0; u < xsum::kSeg; u++) s += el[u];
    bits = xsum::f2u(s);
  };
  // batch b as genuine additions, from the accumulator in `bits`: all 1024 elements land in shared memory by
  // cp.async (one memory round trip for the batch); rolled loops and one call site of redo keep the code small
  auto redo_batch = [&](int b) {
    st_walk++;
    __syncwarp();
#pragma unroll 1
    for (int k = 0; k < 32; k++) {
      const unsigned K = (unsigned)(b * 32 + k) * xsum::kSeg + lane;
      if (K < N) xs_cp4(&stage[k][lane], p + (size_t)(1u + K / len) * P + 1u + K % len);
      else stage[k][lane] = -0.f;
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
    asm volatile("cp.async.wait_group 0;" ::: "memory");          // (also waits for the record group in flight: rare path)
    __syncwarp();
#pragma unroll 1
    for (int k = 0; k < 32; k++) redo(stage[k][lane]);
  };
  const int ngrp = (nb + kXsGroup - 1) / kXsGroup;
  float rawn[kXsRawPf];                                           // elements of the next batch's first serial segments
#pragma unroll
  for (int i = 0; i < kXsRawPf; i++) rawn[i] = 0.f;
  bool have_raw = false, prefetched = false;
  for (int b = 0; b < nb; b++) {
    if (b % kXsGroup == 0) {                                      // chunk boundary
      const int grp = b / kXsGroup;
      __syncwarp();
      if (!prefetched) fetch(grp);
      prefetched = false;
      if (grp + 1 < ngrp) {                                       // next chunk's records: in flight now
        fetch(grp + 1);
        prefetched = true;
        asm volatile("cp.async.wait_group 1;" ::: "memory");
      } else {
        asm volatile("cp.async.wait_group 0;" ::: "memory");
      }
      __syncwarp();
    }
    const uint32_t* rec = ring[b % (2 * kXsGroup)];
    const uint4 hdr = *reinterpret_cast<const uint4*>(rec);       // count, serial entries, head summaries
    float raw[kXsRawPf];
#pragma unroll
    for (int i = 0; i < kXsRawPf; i++) raw[i] = rawn[i];
    const bool raw_ok = have_raw;
    have_raw = false;
    if ((b + 1) % kXsGroup != 0 && b + 1 < nb) {                  // elements of the next batch's serial segments (same group)
      const uint4 nh = *reinterpret_cast<const uint4*>(ring[(b + 1) % (2 * kXsGroup)]);
      uint32_t m = nh.x == 0xffffffffu ? 0u : nh.y;
      if (m) {
        have_raw = true;
#pragma unroll
        for (int i = 0; i < kXsRawPf; i++) {
          rawn[i] = 0.f;
          if (m) {
            const int k = __ffs(m) - 1;
            m &= m - 1u;
            rawn[i] = element((unsigned)((b + 1) * 32 + k));
          }
        }
      }
    }
    XS_TICK(0);
    if (hdr.x == 0xffffffffu) { redo_batch(b); XS_TICK(3); continue; }
    const uint32_t start = bits;
    const int st_redo0 = st_redo;
    bool ok = true;
    const int count = (int)hdr.x;
    for (int i = 0; i < count; i++) {
      const uint4 t0 = *reinterpret_cast<const uint4*>(rec + 8 + kXsEntWords * i);
      const uint4 t1 = *reinterpret_cast<const uint4*>(rec + 12 + kXsEntWords * i);
      const uint2 t2 = *reinterpret_cast<const uint2*>(rec + 16 + kXsEntWords * i);
      bits = xsum::apply_table(bits, t0.x, (int32_t)t0.y, (int32_t)t0.z, (int32_t)t0.w, (int32_t)t1.x, (int32_t)t1.y,
                               (int32_t)t1.z, ok);
      bits = xsum::f2u(((xsum::u2f(bits) + xsum::u2f(t1.w)) + xsum::u2f(t2.x)) + xsum::u2f(t2.y));
      XS_TICK(1);
      const uint2 sr = *reinterpret_cast<const uint2*>(rec + 18 + kXsEntWords * i);   // serial run: length, first slot
      for (int j = 0; j < (int)sr.x; j++) {
        const int k = (int)sr.y + j;
        const unsigned g = (unsigned)(b * 32 + k);
        const int si = __popc(hdr.y & ((1u << k) - 1u));
        float v;
        if (raw_ok && si < kXsRawPf) {
          v = raw[0];
#pragma unroll
          for (int r = 1; r < kXsRawPf; r++) v = (si == r) ? raw[r] : v;
        } else {
          v = element(g);                                         // (no prefetch across group boundaries / beyond kXsRawPf)
        }
        redo(v);
      }
      XS_TICK(2);
    }
    if (ok) { st_rec++; st_ent += count; }
    else { bits = start; st_redo = st_redo0; redo_batch(b); XS_TICK(3); }
  }
  if (lane == 0) {
    q.sc.psum[e] = xsum::u2f(bits);
    q.xs_epoch[e] += 1u;                                          // next pass: fresh chunk-total flags
    int* st = q.xs_stats + 8 * e;
    st[0] = st_rec; st[1] = st_walk; st[2] = st_ent; st[3] = st_redo;
#ifdef RLFC_XS_TIMING
    for (int k = 0; k < 4; k++) st[4 + k] = (int)tacc[k];
#endif
  }
#undef XS_TICK
}

// Large domains: blocks of 32 consecutive batch records condensed IN PARALLEL (one warp per block), ahead of the serial
// pass: a segmented scan of table compositions over the lanes, runs broken at the records that are more than one table.
// Lane l of block k ends up with the composition of the tables of records (start of its run) .. l; the serial pass
// (k_xsum_chain_blocks) crosses a whole run with one checked application of the run's last lane.  Output layout
// xs_blk[e][block][8][32]: words 0..6 the composed table, word 7 the block's mask of one-table records.
__global__ void __launch_bounds__(32)
k_xsum_condense(const __grid_constant__ SolverParams q) {
  const int e = blockIdx.y, bk = blockIdx.x, lane = threadIdx.x;
  if (q.sc.frozen[e]) return;
  const int nb = q.xs_nbatches, b0 = bk * 32;
  const int kend = min(32, nb - b0);
  const uint32_t* mine = q.xs_recs + ((size_t)e * nb + b0 + lane) * kXsRecWords;
  const uint32_t ident[7] = {xsum::kAnyKey, 0u, 0u, (uint32_t)INT32_MIN, (uint32_t)INT32_MAX, (uint32_t)INT32_MIN, (uint32_t)INT32_MAX};
  uint32_t cnt = 0xffffffffu;
  uint4 w0 = make_uint4(0u, 0u, 0u, 0u), w1 = w0;
  if (lane < kend) {
    cnt = mine[0];
    w0 = *reinterpret_cast<const uint4*>(mine + 8);
    w1 = *reinterpret_cast<const uint4*>(mine + 12);
  }
  const bool pure = cnt == 1u;                                    // the whole batch is one table (no float additions, no serial run)
  uint32_t acc[7] = {w0.x, w0.y, w0.z, w0.w, w1.x, w1.y, w1.z};
  if (!pure)
#pragma unroll
    for (int w = 0; w < 7; w++) acc[w] = ident[w];
  const uint32_t puremask = __ballot_sync(0xffffffffu, pure);
  const uint32_t headmask = ~puremask;
  const uint32_t upto = headmask & ((2u << lane) - 1u);
  const int dist = upto ? lane - (31 - __clz(upto)) : lane + 1;    // lanes since the last non-table record (itself: 0)
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    uint32_t prev[7];
#pragma unroll
    for (int w = 0; w < 7; w++) prev[w] = __shfl_up_sync(0xffffffffu, acc[w], o);
    if (dist > o && lane >= o) xsum::compose_tables(prev, acc);    // (the partner is inside this lane's run)
  }
  uint32_t* out = q.xs_blk + (((size_t)e * gridDim.x + bk) * 8) * 32 + lane;
#pragma unroll
  for (int w = 0; w < 7; w++) out[w * 32] = acc[w];
  out[7 * 32] = puremask;
}

// Serial pass for LARGE domains (thousands of batches per environment, e.g. 2048 for a 2048 x 1024 grid): there almost
// every batch record is ONE table (no binade change inside 1024 additions), and tables compose, so every block of 32
// consecutive batch records is condensed first (k_xsum_condense, in parallel: a segmented scan of table compositions
// over the lanes, runs broken at the records that are more than one table) and this warp crosses a whole run with one
// checked table application.  Records with float additions or serial segments are walked entry by entry as in k_xsum_chain; a run whose
// composed table does not provably apply is walked record by record.  Exactness is unchanged: a table is only applied
// when its validity condition holds for the true accumulator.
// Batches whose record does not apply are rebuilt for the TRUE accumulator.  On very large domains such batches come in long
// stretches (the running sum of a zero-mean field sits next to a power of two for millions of additions and the records
// were built for the neighbouring binade: profiles/r02_field_sum_large.md), and rebuilding is 5 200 cycles of one warp per
// batch.  So the CTA carries kXsBulkWarps - 1 HELPER warps that sleep at a named barrier: when warp 0 meets such a batch b,
// every warp rebuilds one of the batches b .. b + kXsBulkWarps - 1 for the accumulator's current key (the whole-batch
// table only), and warp 0 then crosses them one checked application after the other for as long as they apply.  A batch
// whose whole-batch table does not apply falls back to the single-warp path (prefix tables, element-wise additions).
constexpr int kXsBulkWarps = 16;
struct XsBulk {
  float stage[kXsBulkWarps][32][33];     // a batch's 1024 elements per warp, one segment per row (pitch 33: conflict-free)
  uint32_t table[kXsBulkWarps][8];       // the whole-batch table each warp built
  int cmd_batch;                         // first batch of the round, -1 = exit
  uint32_t cmd_key;
};

__device__ __forceinline__ void xs_bulk_barrier() { asm volatile("bar.sync 1, %0;" ::"n"(32 * kXsBulkWarps) : "memory"); }

// one warp: the table of batch `b` for an accumulator of key `key` (lane 31's result is the whole batch), into out[0..6]
__device__ __forceinline__ void xs_bulk_build(const float* __restrict__ p, unsigned N, unsigned len, unsigned P, int nb, int b,
                                              uint32_t key, float (*st)[33], uint32_t* out, int lane) {
  uint32_t w[7] = {key, 0u, 0u, (uint32_t)xsum::kNever, (uint32_t)(-xsum::kNever), (uint32_t)xsum::kNever, (uint32_t)(-xsum::kNever)};
  if (b < nb) {                                                    // (warp-uniform)
    const unsigned K0 = (unsigned)b * 1024u + lane;
    unsigned row = K0 / len, col = K0 - row * len, K = K0;
    const float* src = p + (size_t)(1u + row) * P + 1u + col;
#pragma unroll 4
    for (int k = 0; k < 32; k++) {
      if (K < N) xs_cp4(&st[k][lane], src);
      else st[k][lane] = -0.f;
      K += 32u; col += 32u; src += 32;
      while (col >= len) { col -= len; src += P - len; }
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
    asm volatile("cp.async.wait_group 0;" ::: "memory");
    __syncwarp();
    xsum::Run run;
    run.start(key);
#pragma unroll 8
    for (int j = 0; j < 32; j++) run.add(st[lane][j]);
    if (run.good) { run.store(w); xsum::normalise_table(w); }
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      uint32_t prev[7];
#pragma unroll
      for (int k = 0; k < 7; k++) prev[k] = __shfl_up_sync(0xffffffffu, w[k], o);
      if (lane >= o) xsum::compose_tables(prev, w);
    }
  }
  if (lane == 31) {
#pragma unroll
    for (int k = 0; k < 7; k++) out[k] = w[k];
  }
  __syncwarp();
}

template <bool BULK>               // BULK: launched with kXsBulkWarps warps (helpers); otherwise one warp and none of the bulk code
__global__ void __launch_bounds__(BULK ? 32 * kXsBulkWarps : 32)
k_xsum_chain_blocks(const __grid_constant__ SolverParams q) {
  extern __shared__ __align__(16) uint32_t xs_dyn[];               // [32][32] float stage | [32][33] float stage (redo) | XsBulk
  float (*stage)[32] = reinterpret_cast<float (*)[32]>(xs_dyn);
  float (*stageP)[33] = reinterpret_cast<float (*)[33]>(xs_dyn + 32 * 32);
  XsBulk& bulk = *reinterpret_cast<XsBulk*>(xs_dyn + 32 * 32 + 32 * 33);
  const int e = blockIdx.x, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (q.sc.frozen[e]) return;
  const unsigned len = (unsigned)(q.m - 2), P = (unsigned)q.P;
  const unsigned N = (unsigned)(q.n - 2) * len;
  const int nb = q.xs_nbatches;
  const float* p = q.lev[0].x + (size_t)e * q.stride;
  const uint32_t* recs = q.xs_recs + (size_t)e * nb * kXsRecWords;
  if (BULK && warp != 0) {
    // ---- helper warps: one batch per round ----
    for (;;) {
      xs_bulk_barrier();                                           // a command has been posted
      const int b0 = *(volatile int*)&bulk.cmd_batch;
      if (b0 < 0) return;
      xs_bulk_build(p, N, len, P, nb, b0 + warp, *(volatile uint32_t*)&bulk.cmd_key, bulk.stage[warp], bulk.table[warp], lane);
      xs_bulk_barrier();                                           // the tables are in shared memory
    }
  }
  constexpr bool bulk_on = BULK;
  int done_upto = 0;                                               // batches below this index have been crossed (bulk rounds run ahead)
  int st_rec = 0, st_walk = 0, st_ent = 0, st_redo = 0, st_km = 0;
  long long tk = clock64(), tacc[4] = {0, 0, 0, 0};                // cycles: [0] block set-up + scan, [1] table runs, [2] record walks, [3] batches redone
#define XSB_TICK(i) do { const long long n_ = clock64(); tacc[i] += n_ - tk; tk = n_; } while (0)
  uint32_t bits = 0u;                                             // s = +0.f
  auto element = [&](unsigned g) {
    const unsigned K = g * xsum::kSeg + lane;
    return K < N ? p[(size_t)(1u + K / len) * P + 1u + K % len] : -0.f;
  };
  // 32 genuine additions of the values in seg[0..31] (shared memory; every lane runs the same chain on broadcast loads)
  auto add_segment = [&](const float* seg) {
    st_redo++;
    float s = xsum::u2f(bits);
    const float4* v4 = reinterpret_cast<const float4*>(seg);
#pragma unroll
    for (int k = 0; k < 8; k++) {
      const float4 v = v4[k];
      s += v.x; s += v.y; s += v.z; s += v.w;
    }
    bits = xsum::f2u(s);
  };
  // A batch whose record does not apply -- in practice: the accumulator sits in the other binade than predicted, or
  // comes closer to a binade boundary than the prediction did -- is redone with tables built for the TRUE accumulator:
  // lane L summarises segment L for the accumulator's actual key, a scan composes the prefixes, every lane checks its
  // prefix against the accumulator, the longest valid prefix is applied in one step, the segment behind it (the real
  // binade change) is added element by element, and the rest is rebuilt for the new key.  Exact for the same reason as
  // everywhere else: a table is applied only where its validity condition holds for the true accumulator.
  auto redo_batch = [&](int b) {
    st_walk++;
    XSB_TICK(2);
    __syncwarp();
    if (bulk_on && !(q.xs_flags & 1) && xsum::key_ok(bits >> 23)) {
      // ---- bulk round: batches b .. b + kXsBulkWarps - 1 rebuilt by all warps for the accumulator's current key ----
      if (lane == 0) { bulk.cmd_batch = b; bulk.cmd_key = bits >> 23; }
      xs_bulk_barrier();
      xs_bulk_build(p, N, len, P, nb, b, bits >> 23, bulk.stage[0], bulk.table[0], lane);
      xs_bulk_barrier();
      int crossed = 0;
      for (int w = 0; w < kXsBulkWarps && b + w < nb; w++) {
        const uint32_t* T = bulk.table[w];
        bool ok = true;
        const uint32_t nbits = xsum::apply_table(bits, T[0], (int32_t)T[1], (int32_t)T[2], (int32_t)T[3], (int32_t)T[4], (int32_t)T[5],
                                                 (int32_t)T[6], ok);
        if (!ok) break;
        bits = nbits;
        crossed++;
      }
      if (crossed > 0) {
        st_walk += crossed - 1;
        done_upto = b + crossed;
        XSB_TICK(3);
        return;
      }
    }
    {
      // element (b*32 + k)*32 + lane for k = 0..31: one division, then 32 elements further per k
      const unsigned K0 = (unsigned)b * 1024u + lane;
      unsigned row = K0 / len, col = K0 - row * len, K = K0;
      const float* src = p + (size_t)(1u + row) * P + 1u + col;
#pragma unroll 4
      for (int k = 0; k < 32; k++) {
        if (K < N) xs_cp4(&stageP[k][lane], src);
        else stageP[k][lane] = -0.f;
        K += 32u; col += 32u; src += 32;
        while (col >= len) { col -= len; src += P - len; }
      }
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
    asm volatile("cp.async.wait_group 0;" ::: "memory");
    __syncwarp();
    auto add_row = [&](int k) {                                   // 32 genuine additions (every lane the same chain, broadcast loads)
      float s = xsum::u2f(bits);
#pragma unroll 8
      for (int j = 0; j < 32; j++) s += stageP[k][j];
      bits = xsum::f2u(s);
      st_redo++;
    };
    int done = 0;
    if (q.xs_flags & 1) {                                         // RLFC_XS_REDO=serial: plain genuine additions (cross-check)
      for (int k = 0; k < 32; k++) add_row(k);
      done = 32;
    }
    while (done < 32) {
      const uint32_t key = bits >> 23;
      if (!xsum::key_ok(key)) { add_row(done); done++; continue; }
      uint32_t w[7] = {xsum::kAnyKey, 0u, 0u, (uint32_t)INT32_MIN, (uint32_t)INT32_MAX, (uint32_t)INT32_MIN, (uint32_t)INT32_MAX};
      if (lane >= done) {
        xsum::Run run;
        run.start(key);
#pragma unroll 8
        for (int j = 0; j < 32; j++) run.add(stageP[lane][j]);    // (row pitch 33: conflict-free)
        if (run.good) { run.store(w); xsum::normalise_table(w); }
        else { w[0] = key; w[1] = w[2] = 0u; w[3] = w[5] = (uint32_t)xsum::kNever; w[4] = w[6] = (uint32_t)(-xsum::kNever); }
      }
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        uint32_t prev[7];
#pragma unroll
        for (int k = 0; k < 7; k++) prev[k] = __shfl_up_sync(0xffffffffu, w[k], o);
        if (lane >= o) xsum::compose_tables(prev, w);
      }
      bool ok = true;
      const uint32_t nbits = xsum::apply_table(bits, w[0], (int32_t)w[1], (int32_t)w[2], (int32_t)w[3], (int32_t)w[4], (int32_t)w[5],
                                               (int32_t)w[6], ok);
      const uint32_t okm = __ballot_sync(0xffffffffu, ok || lane < done);
      const int f = (okm == 0xffffffffu) ? 32 : (__ffs(~okm) - 1);               // first segment whose prefix does not apply
      if (f > done) bits = __shfl_sync(0xffffffffu, nbits, f - 1);
      if (f < 32) { add_row(f); done = f + 1; } else done = 32;
    }
    __syncwarp();
    XSB_TICK(3);
  };
  auto walk_batch = [&](int b, const uint32_t* rec) {              // one record, entry by entry (as k_xsum_chain)
    if (BULK && b < done_upto) return;                             // (crossed by a bulk round already)
    const uint4 hdr = *reinterpret_cast<const uint4*>(rec);
#ifdef RLFC_XS_DIAG
    if (lane == 0 && b >= 503 && b <= 505) printf("xswalk %d hdr %08x %08x bits %08x\n", b, hdr.x, hdr.y, bits);
#endif
    if (hdr.x == 0xffffffffu) { st_walk += 1 << 16; redo_batch(b); return; }
    const uint32_t start = bits;
    const int st_redo0 = st_redo;
    bool ok = true;
    const int count = (int)hdr.x;
    if (count > 0 && rec[8] != xsum::kAnyKey && rec[8] != (bits >> 23)) st_km++;   // (diagnostic: the record was built for another binade)
#ifdef RLFC_XS_DIAG
    if (lane == 0 && count > 0 && rec[8] != xsum::kAnyKey && rec[8] != (bits >> 23) && (st_km % 16) == 1)
      printf("xs miss batch %d of %d: accumulator %.9g (key %u), record key %u\n", b, nb, xsum::u2f(bits), bits >> 23, rec[8]);
#endif
    for (int i = 0; i < count; i++) {
      const uint4 t0 = *reinterpret_cast<const uint4*>(rec + 8 + kXsEntWords * i);
      const uint4 t1 = *reinterpret_cast<const uint4*>(rec + 12 + kXsEntWords * i);
      const uint4 t2 = *reinterpret_cast<const uint4*>(rec + 16 + kXsEntWords * i);
      bits = xsum::apply_table(bits, t0.x, (int32_t)t0.y, (int32_t)t0.z, (int32_t)t0.w, (int32_t)t1.x, (int32_t)t1.y,
                               (int32_t)t1.z, ok);
      bits = xsum::f2u(((xsum::u2f(bits) + xsum::u2f(t1.w)) + xsum::u2f(t2.x)) + xsum::u2f(t2.y));
      for (int j = 0; j < (int)t2.z; j++) {                        // a run of serial segments
        __syncwarp();
        stage[0][lane] = element((unsigned)(b * 32 + (int)t2.w + j));
        __syncwarp();
        add_segment(stage[0]);
      }
    }
    if (ok) { st_rec++; st_ent += count; }
    else { bits = start; st_redo = st_redo0; redo_batch(b); }
  };
  const uint32_t* cblk = q.xs_blk + (size_t)e * ((nb + 31) / 32) * 8 * 32;
  uint32_t nxt[8];
#pragma unroll
  for (int w = 0; w < 8; w++) nxt[w] = cblk[w * 32 + lane];
  // (the records themselves are only read where a run does not apply or a record is more than one table: straight from
  // global memory, a few dozen per pass)
  bool midrun = false;
  for (int b0 = 0; b0 < nb; b0 += 32) {
    const int kend = min(32, nb - b0);
    midrun = false;                                                // (runs do not extend across blocks)
    // this block's condensed tables (k_xsum_condense), fetched one block ahead
    uint32_t acc[7];
#pragma unroll
    for (int w = 0; w < 7; w++) acc[w] = nxt[w];
    const uint32_t puremask = nxt[7];
    if (b0 + 32 < nb) {
      const uint32_t* src = cblk + ((size_t)(b0 / 32 + 1) * 8) * 32 + lane;
#pragma unroll
      for (int w = 0; w < 8; w++) nxt[w] = src[w * 32];
    }
    int k = 0;
    XSB_TICK(0);
#ifdef RLFC_XS_DIAG
    if (lane == 0) printf("xsblk %d bits %08x puremask %08x\n", b0, bits, puremask);
#endif
    while (k < kend) {
#ifdef RLFC_XS_DIAG
      if (lane == 0) printf("xsbat %d bits %08x\n", b0 + k, bits);
#endif
      if (BULK && b0 + k < done_upto) { k++; midrun = true; continue; }    // crossed by a bulk round
      if (BULK && !((puremask >> k) & 1u)) midrun = false;         // a record that is more than one table starts the runs afresh
      if (BULK && midrun) {
        // inside a run of one-table records whose beginning a bulk round consumed: the condensed tables start at the run's
        // first record, so the rest of the run is crossed record by record
        walk_batch(b0 + k, recs + (size_t)(b0 + k) * kXsRecWords);
        k++;
        XSB_TICK(2);
        continue;
      }
      if ((puremask >> k) & 1u) {
        const uint32_t rest = ~(puremask >> k);                    // first non-table record at or after k
        int run = rest ? __ffs(rest) - 1 : 32 - k;
        run = min(run, kend - k);
        uint32_t tbl[7];
#pragma unroll
        for (int w = 0; w < 7; w++) tbl[w] = __shfl_sync(0xffffffffu, acc[w], k + run - 1);
        bool ok = true;
        const uint32_t nb_bits = xsum::apply_table(bits, tbl[0], (int32_t)tbl[1], (int32_t)tbl[2], (int32_t)tbl[3], (int32_t)tbl[4],
                                                   (int32_t)tbl[5], (int32_t)tbl[6], ok);
#ifdef RLFC_XS_DIAG
        if (lane == 0 && b0 + k <= 505 && b0 + k + run > 503) printf("xsrun %d..%d key %08x D0 %d ok %d\n", b0 + k, b0 + k + run - 1, tbl[0], (int)tbl[1], (int)ok);
#endif
        if (ok) { bits = nb_bits; st_rec += run; st_ent++; }
        else for (int j = 0; j < run; j++) walk_batch(b0 + k + j, recs + (size_t)(b0 + k + j) * kXsRecWords);
        k += run;
        XSB_TICK(1);
      } else {
        walk_batch(b0 + k, recs + (size_t)(b0 + k) * kXsRecWords);
        k++;
        XSB_TICK(2);
      }
    }
  }
  asm volatile("cp.async.wait_group 0;" ::: "memory");
  if (bulk_on) {
    if (lane == 0) bulk.cmd_batch = -1;                            // release the helper warps
    xs_bulk_barrier();
  }
  if (lane == 0) {
    q.sc.psum[e] = xsum::u2f(bits);
    q.xs_epoch[e] += 1u;
    int* st = q.xs_stats + 8 * e;
    st[0] = st_rec; st[1] = st_walk; st[2] = st_ent | (st_km << 16); st[3] = st_redo;
    for (int k = 0; k < 4; k++) st[4 + k] = (int)tacc[k];
  }
#undef XSB_TICK
}
constexpr size_t kXsBlocksSmem = (size_t)(32 * 32 + 32 * 33) * 4 + sizeof(XsBulk);
