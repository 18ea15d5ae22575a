// Device helpers: mbarrier + TMA bulk copy (sm_100a), Philox4x32-10.
#pragma once
#include <cstdint>

namespace cmb {

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  do {
    asm volatile(
        "{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n selp.u32 %0, 1, 0, p;\n}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
  } while (!ok);
}
// Producer-side wait: back off with nanosleep between polls.  try_wait returns at once when
// the phase is not complete, so a bare poll loop issues an instruction every few cycles and
// starves the consumer warps that share the SM sub-partition (ncu r1e: 60 % of all issued
// instructions were producer spin iterations).
__device__ __forceinline__ void mbar_wait_sleep(uint64_t* bar, uint32_t parity, uint32_t ns) {
  uint32_t ok;
  for (;;) {
    asm volatile(
        "{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n selp.u32 %0, 1, 0, p;\n}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    if (ok) break;
    __nanosleep(ns);
  }
}
// TMA 1-D bulk copy global -> shared, completion signalled on an mbarrier.
__device__ __forceinline__ void tma_bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_u32(dst)),
               "l"(src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void fence_proxy_async() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}

// Double-buffered stream of op chunks through shared memory.  All threads of the CTA
// call wait()/release() in lock step; thread 0 issues the TMA copies.
struct ChunkStream {
  const unsigned char* src;
  const uint32_t* off;
  const uint32_t* bytes;
  uint32_t n_chunks, cap;
  unsigned char* buf;
  uint64_t* bar;
  __device__ __forceinline__ void issue(uint32_t k) {
    uint32_t nb = __ldg(bytes + k);
    mbar_expect_tx(&bar[k & 1], nb);
    tma_bulk_g2s(buf + (size_t)(k & 1) * cap, src + __ldg(off + k), nb, &bar[k & 1]);
  }
  __device__ __forceinline__ void start(unsigned char* smem, uint64_t* bars) {
    buf = smem;
    bar = bars;
    if (threadIdx.x == 0) {
      mbar_init(&bar[0], 1);
      mbar_init(&bar[1], 1);
      mbar_fence_init();
    }
    __syncthreads();
    if (threadIdx.x == 0) {
      issue(0);
      if (n_chunks > 1) issue(1);
    }
  }
  __device__ __forceinline__ const unsigned char* wait(uint32_t k) {
    mbar_wait(&bar[k & 1], (k >> 1) & 1);
    return buf + (size_t)(k & 1) * cap;
  }
  __device__ __forceinline__ void release(uint32_t k) {
    __syncthreads();
    if (threadIdx.x == 0 && k + 2 < n_chunks) {
      fence_proxy_async();
      issue(k + 2);
    }
  }
};

// Philox4x32-10 (Salmon et al., SC'11); counter (site lo, site hi, node, tag), key = seed.
__host__ __device__ __forceinline__ void philox4x32_10(uint32_t c[4], uint32_t k0, uint32_t k1) {
#pragma unroll
  for (int r = 0; r < 10; r++) {
    uint64_t p0 = (uint64_t)0xD2511F53u * c[0];
    uint64_t p1 = (uint64_t)0xCD9E8D57u * c[2];
    uint32_t n0 = (uint32_t)(p1 >> 32) ^ c[1] ^ k0;
    uint32_t n1 = (uint32_t)p1;
    uint32_t n2 = (uint32_t)(p0 >> 32) ^ c[3] ^ k1;
    uint32_t n3 = (uint32_t)p0;
    c[0] = n0; c[1] = n1; c[2] = n2; c[3] = n3;
    k0 += 0x9E3779B9u;
    k1 += 0xBB67AE85u;
  }
}
__host__ __device__ __forceinline__ double philox_u01(uint64_t seed, uint64_t site, uint32_t node, uint32_t tag) {
  uint32_t c[4] = {(uint32_t)site, (uint32_t)(site >> 32), node, tag};
  philox4x32_10(c, (uint32_t)seed, (uint32_t)(seed >> 32));
  uint64_t u = (((uint64_t)c[0] << 32) | c[1]) >> 11;
  return (double)u * (1.0 / 9007199254740992.0);
}

// Two uniforms from one Philox block: (c0, c1) and (c2, c3).  The simulator draws the states of
// the (2 k)-th and (2 k + 1)-th child of a node from ONE block keyed by the parent.
__host__ __device__ __forceinline__ void philox_u01x2(uint64_t seed, uint64_t site, uint32_t node, uint32_t tag,
                                                      double& u0, double& u1) {
  uint32_t c[4] = {(uint32_t)site, (uint32_t)(site >> 32), node, tag};
  philox4x32_10(c, (uint32_t)seed, (uint32_t)(seed >> 32));
  u0 = (double)((((uint64_t)c[0] << 32) | c[1]) >> 11) * (1.0 / 9007199254740992.0);
  u1 = (double)((((uint64_t)c[2] << 32) | c[3]) >> 11) * (1.0 / 9007199254740992.0);
}

// Key of a nucleotide column for the null's pattern compression (k2_pairs.cu launch_compress_patterns): the tips
// at 2 bits each, 16 to a 32-bit word in the order the simulation walk reaches the leaves, and a 64-bit hash of
// those words folded in the same order.  k3_simulate and k2_column_keys must produce the same key.
constexpr uint64_t kColumnHashInit = 0x243F6A8885A308D3ull;
__device__ __forceinline__ uint64_t column_hash_step(uint64_t h, uint32_t w) {
  h = (h ^ w) * 0xFF51AFD7ED558CCDull;
  return h ^ (h >> 32);
}
__device__ __forceinline__ uint64_t column_hash_final(uint64_t h) { // MurmurHash3's fmix64
  h ^= h >> 33; h *= 0xFF51AFD7ED558CCDull;
  h ^= h >> 33; h *= 0xC4CEB9FE1A85EC53ull;
  return h ^ (h >> 33);
}

// Continuous site rate (simulations.continuous = yes; NonHomogeneousSequenceSimulator::enableContinuousRates,
// CoMap.cpp:209-219 -> rDist->randC()): Gamma(alpha, beta = alpha) by Marsaglia & Tsang's squeeze method with
// Box-Muller normals, every uniform from the site's Philox stream (node = root, tags 98.. ), so a site's rate
// depends only on (seed, site).  kind: 1 constant rate 1, 2 gamma, 3 invariant (rate 0 with probability p_inv)
// + gamma / (1 - p_inv).
__host__ __device__ __forceinline__ double continuous_rate(int kind, double alpha, double p_inv, uint64_t seed,
                                                           uint64_t site, uint32_t node) {
  if (kind == 1) return 1.;
  double scale = 1.;
  if (kind == 3) {
    if (philox_u01(seed, site, node, 98) < p_inv) return 0.;
    scale = 1. / (1. - p_inv);
  }
  double a = alpha, boost = 1.;
  if (a < 1.) { // G(a) = G(a + 1) U^(1/a)
    boost = pow(1. - philox_u01(seed, site, node, 99), 1. / a);
    a += 1.;
  }
  const double d = a - 1. / 3., c = 1. / sqrt(9. * d);
  double g = d;
  for (uint32_t k = 0; k < 64; k++) {
    double u1, u2;
    philox_u01x2(seed, site, node, 100 + 2 * k, u1, u2);
    const double x = sqrt(-2. * log(1. - u1)) * cos(6.283185307179586 * u2);
    double v = 1. + c * x;
    if (v <= 0.) continue;
    v = v * v * v;
    const double u = 1. - philox_u01(seed, site, node, 101 + 2 * k);
    if (u < 1. - 0.0331 * (x * x) * (x * x) || log(u) < 0.5 * x * x + d * (1. - v + log(v))) { g = d * v; break; }
  }
  return g * boost / alpha * scale;
}

} // namespace cmb
