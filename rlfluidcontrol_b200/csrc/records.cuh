// records.cuh -- one environment's complete state as a portable byte record (rlfc_env_export / rlfc_env_import and their
// _device variants; the format is rlfc.h "State records").  Included at the end of solver_kernels.cu, after snapshot.cuh,
// whose snap_word (the scalar record) and pair_applies (the last in-range pair wins) it shares.
//
// A record holds what a snapshot slot holds, with the three fields in the reference layout n x m (ghosts included) instead
// of the pitched one.  A record is a multiple of 16 bytes and so is each field, so every field starts 16-byte aligned in a
// 16-byte aligned buffer, but a field row (m floats, m even) starts only 8-byte aligned.  The copy therefore walks each
// field as flat float4 of the reference layout (16-byte accesses on the record side) and moves each float4 as two float2
// of the pitched layout, which sit in one row or, at an odd row's end, in two (8-byte accesses on the device side).
//
//   k_export        grid (3 fields x chunks, pairs): copies its chunk, CTA 0 of a pair also writes the header, the scalar
//                   record and the sensors; every CTA writes its partial checksum, the pair's last CTA (ticket) adds them
//                   in chunk order and stores the checksum.
//   k_import_check  grid (chunks of the whole record, pairs): the winning pair of each destination recomputes the
//                   checksum the same way, CTA 0 checks the header against the destination; verdict[k] only.
//   k_import        grid (3 fields x chunks, pairs): pairs with verdict "apply" copy back, CTA 0 writes the scalar record
//                   (honouring keep), the sensors when the tables match, the refusal flag and skip[e] = 0.
#pragma once
#include "snapshot.cuh"

namespace rlfc {
namespace {

constexpr int kRecThreads = 256;
constexpr int kRecVec = 4;                            // float4 per thread: 16 KB of one field per CTA
constexpr int kRecChunk = kRecThreads * kRecVec;      // float4 per chunk
constexpr int kRecHdrWords = RLFC_RECORD_HEADER_BYTES / 4;
constexpr unsigned kRecMagic0 = 0x43464c52u, kRecMagic1 = 0x54415453u;   // "RLFC", "STAT" little-endian

struct RecArgs {
  EnvScalars sc;
  int B, nprobe;
  float *ux, *uy, *p;                         // the environments' fields (batch base)
  size_t stride;                              // level-0 per-environment stride (floats)
  int n, m, P;                                // level-0 dims incl. ghosts, pitch
  SensorSet sens;                             // the environments' sensors (sens.n = 0: none)
  const rlfc_sensor* table;                   // [sens.n] the handle's sensor table as given at create
  const unsigned* env_par;                    // [5][B] each environment's parameter tuple (bits)
  unsigned grid[3];                           // resolution, x_lengths, y_lengths
  int adaptive;
  unsigned char* rec;                         // n records of `bytes` each
  size_t bytes;
  int K;                                      // sensors of a record of `bytes` bytes on this grid
  const int* ids;
  int npairs, keep;
  unsigned long long* partial;                // [npairs][chunks]
  unsigned* ticket;                           // [npairs], zero between launches
  int* hcode;                                 // [npairs] header verdict of k_import_check
  int* verdict;                               // [npairs] kRecSkip, 0 = apply, else the failed check (RecordCheck)
  int* refused;                               // [B] flags bit 3
  int* skip;                                  // [B] mask of the following launch_poisson_rebuild* (nullptr: none)
};

__device__ __forceinline__ unsigned f2u(float x) { return __float_as_uint(x); }

// sum over the CTA, then the pair's ticket: the CTA that takes the last one adds all partials in chunk order and returns
// the pair's total in *sum (thread 0 only); true in every thread of that CTA
__device__ __forceinline__ bool rec_combine(unsigned long long part, unsigned long long* partial, unsigned* ticket, int nch,
                                           unsigned long long* sum) {
  __shared__ unsigned long long s_part[kRecThreads / 32];
  __shared__ int s_last;
  for (int o = 16; o > 0; o >>= 1) part += __shfl_xor_sync(0xffffffffu, part, o);
  if ((threadIdx.x & 31) == 0) s_part[threadIdx.x >> 5] = part;
  __syncthreads();
  if (threadIdx.x == 0) {
    unsigned long long t = 0;
    for (int w = 0; w < kRecThreads / 32; w++) t += s_part[w];
    partial[blockIdx.x] = t;
    __threadfence();
    s_last = atomicAdd(ticket, 1u) == (unsigned)nch - 1;
  }
  __syncthreads();
  const bool last = s_last;
  if (last && threadIdx.x == 0) {
    __threadfence();
    unsigned long long t = 0;
    for (int c = 0; c < nch; c++) t += __ldcg(partial + c);
    *sum = t;
    *ticket = 0;                              // ready for the next launch
  }
  __syncthreads();                            // (s_part, s_last are reused by the next pair)
  return last;
}

// float4 q of a reference-layout field (n x m, m even) as two float2 offsets into the pitched layout
__device__ __forceinline__ void rec_offsets(int q, int m, int P, size_t& o0, size_t& o1) {
  const int j0 = 4 * q, i = j0 / m, j = j0 - i * m;
  o0 = (size_t)i * P + j;
  o1 = j + 2 < m ? o0 + 2 : (size_t)(i + 1) * P;
}

__device__ __forceinline__ unsigned long long mix4(unsigned long long w, uint4 v) {
  return record_mix(w, v.x) + record_mix(w + 1, v.y) + record_mix(w + 2, v.z) + record_mix(w + 3, v.w);
}

// word w (>= 4) of the head of environment e's record (header, scalar record, sensor table, sensor values)
__device__ __forceinline__ unsigned head_word(const RecArgs& a, int e, int w) {
  const int K = a.sens.n;
  if (w < kRecHdrWords) switch (w) {
    case 4: return RLFC_RECORD_VERSION;
    case 5: return (unsigned)a.adaptive;
    case 6: return (unsigned)a.bytes;
    case 7: return (unsigned)((unsigned long long)a.bytes >> 32);
    case 8: case 9: case 10: return a.grid[w - 8];
    case 11: return (unsigned)a.n;
    case 12: return (unsigned)a.m;
    case 18: return (unsigned)a.nprobe;
    case 19: return (unsigned)K;
    default: return a.env_par[(size_t)(w - 13) * a.B + e];   // 13 .. 17
  }
  w -= kRecHdrWords;
  if (w < kSnapWords) {
    const unsigned* x = snap_word(a.sc, a.nprobe, e, w);
    return x ? *x : 0u;
  }
  w -= kSnapWords;
  if (w < 3 * K) return reinterpret_cast<const unsigned*>(a.table)[w];
  return f2u(a.sens.out[(size_t)e * K + (w - 3 * K)]);
}

__global__ void __launch_bounds__(kRecThreads) k_export(const __grid_constant__ RecArgs a) {
  const int nv = a.n * a.m / 4, cpf = (nv + kRecChunk - 1) / kRecChunk, nch = 3 * cpf;
  const int f = blockIdx.x / cpf, c = blockIdx.x - f * cpf;
  const size_t head = RLFC_RECORD_HEADER_BYTES + 4 * kSnapWords + 16 * (size_t)a.sens.n;
  for (int k = blockIdx.y; k < a.npairs; k += gridDim.y) {
    unsigned* rw = reinterpret_cast<unsigned*>(a.rec + (size_t)k * a.bytes);
    const int e = a.ids[k];
    if (e < 0 || e >= a.B) {                  // a record every import refuses: zero magic and header
      if (blockIdx.x == 0 && threadIdx.x < kRecHdrWords) rw[threadIdx.x] = 0u;
      continue;
    }
    const float* src = (f == 0 ? a.ux : f == 1 ? a.uy : a.p) + (size_t)e * a.stride;
    const size_t off = head + (size_t)f * nv * 16;   // byte offset of field f
    float4* dst = reinterpret_cast<float4*>(a.rec + (size_t)k * a.bytes + off);
    unsigned long long part = 0;
#pragma unroll
    for (int u = 0; u < kRecVec; u++) {
      const int q = c * kRecChunk + u * kRecThreads + (int)threadIdx.x;
      if (q < nv) {
        size_t o0, o1;
        rec_offsets(q, a.m, a.P, o0, o1);
        const float2 v0 = *reinterpret_cast<const float2*>(src + o0), v1 = *reinterpret_cast<const float2*>(src + o1);
        const float4 v = make_float4(v0.x, v0.y, v1.x, v1.y);
        __stcs(dst + q, v);
        part += mix4(off / 4 + 4 * (size_t)q, make_uint4(f2u(v.x), f2u(v.y), f2u(v.z), f2u(v.w)));
      }
    }
    if (blockIdx.x == 0) {
      if (threadIdx.x == 0) { rw[0] = kRecMagic0; rw[1] = kRecMagic1; }
      for (int w = 4 + (int)threadIdx.x; w < (int)(head / 4); w += kRecThreads) {
        const unsigned x = head_word(a, e, w);
        rw[w] = x;
        part += record_mix(w, x);
      }
    }
    unsigned long long sum;
    if (rec_combine(part, a.partial + (size_t)k * nch, a.ticket + k, nch, &sum) && threadIdx.x == 0)
      *reinterpret_cast<unsigned long long*>(rw + 2) = sum;
  }
}

// the checks of record rw against the handle and environment e, in the order of RecordCheck (0: all pass)
__device__ int rec_header_check(const RecArgs& a, const unsigned* rw) {
  if (rw[0] != kRecMagic0 || rw[1] != kRecMagic1) return kRecMagic;
  if (rw[4] != RLFC_RECORD_VERSION) return kRecVersion;
  const unsigned long long len = rw[6] | (unsigned long long)rw[7] << 32, n = rw[11], m = rw[12];
  if (len != a.bytes || n > 0xffffu || m > 0xffffu ||
      len != RLFC_RECORD_HEADER_BYTES + 4 * kSnapWords + 16ull * rw[19] + 12 * n * m) return kRecLength;
  if (rw[8] != a.grid[0] || rw[9] != a.grid[1] || rw[10] != a.grid[2] || n != (unsigned)a.n || m != (unsigned)a.m ||
      rw[18] != (unsigned)a.nprobe) return kRecGrid;
  return 0;
}
__device__ int rec_state_check(const RecArgs& a, const unsigned* rw, int e) {
  for (int w = 0; w < 5; w++)
    if (rw[13 + w] != a.env_par[(size_t)w * a.B + e]) return kRecTuple;
  const unsigned dt = rw[kRecHdrWords + 4];   // scalar word 4
  if (a.adaptive) {
    const float x = __uint_as_float(dt);
    if (!(x > 0.f) || !isfinite(x)) return kRecDt;
  } else if (dt != f2u(a.sc.dt[e])) return kRecDt;
  return 0;
}

__global__ void __launch_bounds__(kRecThreads) k_import_check(const __grid_constant__ RecArgs a) {
  const int nq = (int)(a.bytes / 16), nch = (nq + kRecChunk - 1) / kRecChunk, c = blockIdx.x;
  for (int k = blockIdx.y; k < a.npairs; k += gridDim.y) {
    if (!pair_applies(a.ids, a.ids, k, a.npairs, a.B, a.B, true)) {
      if (c == 0 && threadIdx.x == 0) a.verdict[k] = kRecSkip;
      continue;
    }
    const int e = a.ids[k];
    const unsigned char* r = a.rec + (size_t)k * a.bytes;
    unsigned long long part = 0;
#pragma unroll
    for (int u = 0; u < kRecVec; u++) {
      const int q = c * kRecChunk + u * kRecThreads + (int)threadIdx.x;
      if (q < nq) {
        // words 0 .. 3 (magic, checksum) are not covered
        if (q > 0) part += mix4(4 * (unsigned long long)q, __ldcs(reinterpret_cast<const uint4*>(r) + q));
      }
    }
    if (c == 0 && threadIdx.x == 0) {
      const unsigned* rw = reinterpret_cast<const unsigned*>(r);
      const int h = rec_header_check(a, rw);
      a.hcode[k] = h ? h : rec_state_check(a, rw, e);
    }
    unsigned long long sum;
    if (rec_combine(part, a.partial + (size_t)k * nch, a.ticket + k, nch, &sum) && threadIdx.x == 0) {
      const int h = __ldcg(a.hcode + k);
      const unsigned long long stored = *reinterpret_cast<const unsigned long long*>(r + 8);
      a.verdict[k] = h && h < kRecChecksum ? h : sum != stored ? (int)kRecChecksum : h;
    }
  }
}

__global__ void __launch_bounds__(kRecThreads) k_import(const __grid_constant__ RecArgs a) {
  const int nv = a.n * a.m / 4, cpf = (nv + kRecChunk - 1) / kRecChunk;
  const int f = blockIdx.x / cpf, c = blockIdx.x - f * cpf;
  const size_t head = RLFC_RECORD_HEADER_BYTES + 4 * kSnapWords + 16 * (size_t)a.K;
  for (int k = blockIdx.y; k < a.npairs; k += gridDim.y) {
    const int v = a.verdict[k];
    if (v == kRecSkip) continue;
    const int e = a.ids[k];
    if (blockIdx.x == 0 && threadIdx.x == 0) {
      a.refused[e] = v != 0;
      if (v == 0 && a.skip) a.skip[e] = 0;
    }
    if (v != 0) continue;
    const unsigned char* r = a.rec + (size_t)k * a.bytes;
    const size_t off = head + (size_t)f * nv * 16;
    const float4* src = reinterpret_cast<const float4*>(r + off);
    float* dst = (f == 0 ? a.ux : f == 1 ? a.uy : a.p) + (size_t)e * a.stride;
#pragma unroll
    for (int u = 0; u < kRecVec; u++) {
      const int q = c * kRecChunk + u * kRecThreads + (int)threadIdx.x;
      if (q < nv) {
        size_t o0, o1;
        rec_offsets(q, a.m, a.P, o0, o1);
        const float4 x = __ldcs(src + q);
        *reinterpret_cast<float2*>(dst + o0) = make_float2(x.x, x.y);
        *reinterpret_cast<float2*>(dst + o1) = make_float2(x.z, x.w);
      }
    }
    if (blockIdx.x == 0) {
      const unsigned* rw = reinterpret_cast<const unsigned*>(r);
      if (threadIdx.x < kSnapWords) {
        const int w = threadIdx.x;
        unsigned* x = snap_word(a.sc, a.nprobe, e, w);
        if (x && !(a.keep && w >= kSnapAcc0 && w < kSnapAcc1)) *x = rw[kRecHdrWords + w];
      }
      // sensor values only under a byte-equal sensor table (else the next step overwrites the destination's)
      const int K = a.sens.n;
      const unsigned* tab = rw + kRecHdrWords + kSnapWords;
      int differ = a.K != K;
      for (int w = threadIdx.x; !differ && w < 3 * K; w += kRecThreads)
        differ = tab[w] != reinterpret_cast<const unsigned*>(a.table)[w];
      if (!__syncthreads_or(differ))
        for (int s = threadIdx.x; s < K; s += kRecThreads) a.sens.out[(size_t)e * K + s] = __uint_as_float(tab[3 * K + s]);
    }
  }
}

RecArgs record_args(const SolverParams& q, const SensorSet& sens, const RecordBufs& rb, float* ux, float* uy, const int* d_ids,
                    int n, void* rec, size_t bytes) {
  RecArgs a{};
  a.sc = q.sc;
  a.B = q.B;
  a.nprobe = q.nprobe;
  a.ux = ux;
  a.uy = uy;
  a.p = q.lev[0].x;
  a.stride = q.stride;
  a.n = q.n; a.m = q.m; a.P = q.P;
  a.sens = sens;
  a.table = rb.sensors;
  a.env_par = rb.env_par;
  for (int i = 0; i < 3; i++) a.grid[i] = (unsigned)rb.grid[i];
  a.adaptive = q.adaptive;
  a.rec = static_cast<unsigned char*>(rec);
  a.bytes = bytes;
  a.K = (int)((bytes - RLFC_RECORD_HEADER_BYTES - 4 * kSnapWords - 12 * (size_t)q.n * q.m) / 16);
  a.ids = d_ids;
  a.npairs = n;
  a.partial = rb.partial;
  a.ticket = rb.ticket;
  a.hcode = rb.hcode;
  a.verdict = rb.verdict;
  a.refused = rb.refused;
  return a;
}

}  // namespace

int record_chunks(int n, int m, size_t bytes) {
  const int nv = n * m / 4, cpf = (nv + kRecChunk - 1) / kRecChunk;
  const int nch = (int)((bytes / 16 + kRecChunk - 1) / kRecChunk);
  return 3 * cpf > nch ? 3 * cpf : nch;
}

int launch_record_export(const SolverParams& q, const SensorSet& sens, const RecordBufs& rb, float* ux, float* uy,
                         const int* d_ids, int n, void* rec, cudaStream_t st) {
  if (n <= 0) return 0;
  const size_t bytes = record_bytes(q.n, q.m, sens.n);
  const RecArgs a = record_args(q, sens, rb, ux, uy, d_ids, n, rec, bytes);
  const int cpf = (q.n * q.m / 4 + kRecChunk - 1) / kRecChunk;
  k_export<<<dim3(3 * cpf, n < 65535 ? n : 65535), kRecThreads, 0, st>>>(a);
  return 1;
}

int launch_record_import(const SolverParams& q, const SensorSet& sens, const RecordBufs& rb, float* ux, float* uy,
                         const int* d_ids, int n, const void* rec, size_t bytes, int check, int keep_accumulators, int* skip,
                         cudaStream_t st) {
  if (n <= 0) return 0;
  RecArgs a = record_args(q, sens, rb, ux, uy, d_ids, n, const_cast<void*>(rec), bytes);
  a.keep = keep_accumulators;
  a.skip = skip;
  const dim3 pairs(1, n < 65535 ? n : 65535);
  if (check) {
    const int nch = (int)((bytes / 16 + kRecChunk - 1) / kRecChunk);
    k_import_check<<<dim3(nch, pairs.y), kRecThreads, 0, st>>>(a);
  } else {
    const int cpf = (q.n * q.m / 4 + kRecChunk - 1) / kRecChunk;
    k_import<<<dim3(3 * cpf, pairs.y), kRecThreads, 0, st>>>(a);
  }
  return 1;
}

}  // namespace rlfc
