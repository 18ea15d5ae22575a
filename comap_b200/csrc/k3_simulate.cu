// K3: on-device sequence simulation for the parametric-bootstrap null.
//
// Replaces NonHomogeneousSequenceSimulator::simulate(n) in discrete-rate mode (call sites
// CoMap.cpp:209-219, AnalysisTools.cpp:591,614, ClusterTools.cpp:224; SURVEY.md s8 a11):
// root state ~ pi (first i with r <= cumulative pi), rate class uniform over classes
// (upstream behaviour) or ~ probs, child state by linear inverse-CDF over the cumulative
// row of P_c(b).  Randomness is counter based -- Philox4x32-10 keyed (seed; site, node,
// tag) -- so a site's column does not depend on batching, GPU count or launch geometry.
// The k-th child of node p (children in id order) uses half k % 2 of the block keyed
// (p, tag 2 + k / 2): one Philox block serves both children of a binary node (the RNG was
// 3/4 of this kernel's instructions with one block per child).
// One thread per site walks the precompiled pre-order stream (schedule.cpp); tips are
// written [row][site] (site contiguous) in the layout K1 reads.
#include "device_utils.cuh"
#include "kernels.h"

namespace cmb {
namespace {

constexpr int NT = 256;

struct SimParams {
  const unsigned char* src;
  const uint32_t *off, *bytes, *nrec;
  uint32_t n_chunks, cap;
  int A, C, root_node, weighted;
  uint64_t seed;
  uint32_t rk[20];             // Philox round keys of `seed` (k0, k1 per round): constant-bank operands of the XORs
  int64_t base, group, stride; // site id = base + (idx / group) * stride + idx % group
  int64_t n, n_pad;
  int64_t half_n, half_col, half_shift; // two batches in one launch: threads >= half_n simulate site ids shifted by
                                        // half_shift and write columns from half_col (half_n = 0: one batch)
  const double *pi, *probs;
  uint8_t* tips;
  int32_t* classes;
  // pattern compression of the null (k2_pairs.cu launch_compress_patterns), fused: the column's key, built in
  // registers while the column is produced instead of re-read from the tip matrix (nullable; A = 4)
  uint64_t* key_hash;
  int32_t* key_col;
  uint32_t* key_packed;
};

// Philox4x32-10 with the key schedule taken from the launch parameters: the round keys depend on the seed only,
// so they sit in the constant bank and fold into the XORs (LOP3 with a uniform operand); high and low product
// words through __umulhi / mul.lo (the 64-bit product form left one add of a zero carry per multiply).  42
// instructions per block instead of 91 (cuobjdump); the same function of (seed, counter) as philox4x32_10.
// Measured and left out: 53-bit integer uniforms against integer thresholds ceil(cum 2^53) instead of the
// conversion to double + DSETP (the same draws, 5.8 vs 5.6 ms per config-4 step: no gain).
__device__ __forceinline__ void philox_rk(const SimParams& p, uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3,
                                          double& u0, double& u1) {
#pragma unroll
  for (int r = 0; r < 10; r++) {
    const uint32_t h0 = __umulhi(0xD2511F53u, c0), l0 = 0xD2511F53u * c0;
    const uint32_t h1 = __umulhi(0xCD9E8D57u, c2), l1 = 0xCD9E8D57u * c2;
    c0 = h1 ^ c1 ^ p.rk[2 * r];
    c2 = h0 ^ c3 ^ p.rk[2 * r + 1];
    c1 = l1; c3 = l0;
  }
  u0 = (double)((((uint64_t)c0 << 32) | c1) >> 11) * (1.0 / 9007199254740992.0);
  u1 = (double)((((uint64_t)c2 << 32) | c3) >> 11) * (1.0 / 9007199254740992.0);
}

__device__ __forceinline__ int draw_state(const double* __restrict__ row, int A, double u) {
  if (A == 4) { // nucleotides: the cumulative row is two 128-bit shared loads
    const double2 lo = *reinterpret_cast<const double2*>(row), hi = *reinterpret_cast<const double2*>(row + 2);
    return u < lo.x ? 0 : u < lo.y ? 1 : u < hi.x ? 2 : 3;
  }
  int y = A - 1;
  for (int k = A - 1; k >= 0; k--)
    if (u < row[k]) y = k;
  return y;
}

// AT = 4 / 20: the alphabet size at compile time (table strides become shifts / immediates); 0 = read it from p
template <int AT>
__global__ void __launch_bounds__(NT) k3_simulate(const __grid_constant__ SimParams p) {
  extern __shared__ __align__(128) unsigned char smem[];
  const int64_t tid = (int64_t)blockIdx.x * NT + threadIdx.x;
  const bool live = tid < p.n;
  const int64_t tt = live ? tid : p.n - 1;
  const bool second = p.half_n > 0 && tt >= p.half_n;
  const int64_t ii = second ? tt - p.half_n : tt;                   // index inside its batch
  const int64_t idx = second ? p.half_col + ii : ii;                // column of the tip matrix
  const uint64_t site = (uint64_t)(p.base + (second ? p.half_shift : 0) + (ii / p.group) * p.stride + ii % p.group);
  ChunkStream cs{p.src, p.off, p.bytes, p.n_chunks, p.cap, nullptr, nullptr};
  cs.start(smem + 128, reinterpret_cast<uint64_t*>(smem));
  const int A = AT > 0 ? AT : p.A, C = p.C, AA = A * A;
  const uint32_t site_lo = (uint32_t)site, site_hi = (uint32_t)(site >> 32);

  int st;
  {
    double r, r_unused;
    philox_rk(p, site_lo, site_hi, (uint32_t)p.root_node, 0u, r, r_unused);
    st = A - 1;
    double cp = 0.;
    bool done = false;
    for (int i = 0; i < A; i++) {
      cp += __ldg(p.pi + i);
      if (!done && r <= cp) { st = i; done = true; }
    }
  }
  int c;
  {
    double r, r_unused;
    philox_rk(p, site_lo, site_hi, (uint32_t)p.root_node, 1u, r, r_unused);
    if (p.weighted) {
      c = C - 1;
      double cq = 0.;
      bool done = false;
      for (int i = 0; i < C; i++) {
        cq += __ldg(p.probs + i);
        if (!done && r <= cq) { c = i; done = true; }
      }
    } else {
      c = (int)(r * (double)C);
      if (c >= C) c = C - 1;
    }
  }
  if (live && p.classes) p.classes[idx] = c;

  uint8_t stk[kMaxStack];
  int sp = 0;
  uint8_t* const tip_col = p.tips + idx;
  const uint32_t npad32 = (uint32_t)p.n_pad;
  // column key: 16 tips per word in walk order (every thread counts the same tips: the branches are uniform)
  const bool keyed = AT == 4 && p.key_hash != nullptr;
  uint64_t hash = kColumnHashInit;
  uint32_t word = 0, n_tips = 0;
  uint32_t* const packed_col = keyed ? p.key_packed + idx : nullptr;
  auto key_tip = [&](int s) {
    word |= (uint32_t)s << (2 * (n_tips & 15));
    if ((++n_tips & 15) == 0) {
      if (live) packed_col[(uint64_t)(n_tips / 16 - 1) * npad32] = word;
      hash = column_hash_step(hash, word);
      word = 0;
    }
  };
  const size_t tab = (size_t)C * AA;
  for (uint32_t k = 0; k < p.n_chunks; k++) {
    const unsigned char* rp = cs.wait(k);
    const uint32_t nrec = __ldg(p.nrec + k);
    for (uint32_t r = 0; r < nrec; r++) {
      const int4 h0 = *reinterpret_cast<const int4*>(rp);
      const int4 h1 = *reinterpret_cast<const int4*>(rp + 16);
      const uint32_t flags = (uint32_t)h0.x;
      const double* cumA = reinterpret_cast<const double*>(rp + 32);
      const double* cumB = cumA + tab;
      rp += (32 + 2 * tab * sizeof(double) + 15) & ~size_t(15);
      int sa = st, sb = st;
      // h1.y / h1.z = (block index << 1 | half) of child a / b among the children of node h1.w
      double u0 = 0., u1 = 0.;
      if (h0.w >= 0) {
        philox_rk(p, site_lo, site_hi, (uint32_t)h1.w, 2u + ((uint32_t)h1.y >> 1), u0, u1);
        sa = draw_state(cumA + ((size_t)c * A + st) * A, A, (h1.y & 1) ? u1 : u0);
      }
      if (h1.x >= 0) {
        if (h0.w < 0 || (h1.y >> 1) != (h1.z >> 1))
          philox_rk(p, site_lo, site_hi, (uint32_t)h1.w, 2u + ((uint32_t)h1.z >> 1), u0, u1);
        sb = draw_state(cumB + ((size_t)c * A + st) * A, A, (h1.z & 1) ? u1 : u0);
      }
      // row * n_pad as one 32 x 32 -> 64 bit multiply (rows and padded site counts are below 2^32)
      if (flags & kUpTipA) {
        if (live) tip_col[(uint64_t)(uint32_t)h0.y * npad32] = (uint8_t)sa;
        if (keyed) key_tip(sa);
      }
      if (flags & kUpTipB) {
        if (live) tip_col[(uint64_t)(uint32_t)h0.z * npad32] = (uint8_t)sb;
        if (keyed) key_tip(sb);
      }
      if (flags & kUpTakeA) {
        if (flags & kUpPush) stk[sp++] = (uint8_t)sb;
        st = sa;
      } else if (flags & kUpTakeB) st = sb;
      else if (flags & kUpPop) st = stk[--sp];
    }
    cs.release(k);
  }
  if (keyed && live) {
    if (n_tips & 15) {
      packed_col[(uint64_t)(n_tips / 16) * npad32] = word;
      hash = column_hash_step(hash, word);
    }
    p.key_hash[tid] = column_hash_final(hash);
    p.key_col[tid] = (int32_t)idx;
  }
}

// Continuous rates: the site's rate r is drawn once (continuous_rate), the transition probabilities of a branch
// are P(d_b r) = R exp(ev d_b r) L evaluated for the parent's state only (A exponentials + A^2 multiply-adds per
// branch), the child state is drawn by the same linear inverse-CDF and the same Philox blocks as the discrete walk.
struct ContParams { int kind; double alpha, p_inv; const double* spec; int n_nodes; };

template <int AMAX>
__global__ void __launch_bounds__(NT) k3_simulate_cont(SimParams p, ContParams cp) {
  extern __shared__ __align__(128) unsigned char smem[];
  const int A = p.A, AA = A * A;
  double* sp = reinterpret_cast<double*>(smem);          // ev | R | L
  for (int i = threadIdx.x; i < A + 2 * AA; i += NT) sp[i] = __ldg(cp.spec + i);
  const double* ev = sp;
  const double* R = sp + A;
  const double* L = sp + A + AA;
  const double* brlen = cp.spec + A + 2 * AA;
  unsigned char* ring = smem + ((sizeof(double) * (A + 2 * AA) + 127) & ~size_t(127));
  const int64_t tid = (int64_t)blockIdx.x * NT + threadIdx.x;
  const bool live = tid < p.n;
  const int64_t tt = live ? tid : p.n - 1;
  const bool second = p.half_n > 0 && tt >= p.half_n;
  const int64_t ii = second ? tt - p.half_n : tt;
  const int64_t idx = second ? p.half_col + ii : ii;
  const uint64_t site = (uint64_t)(p.base + (second ? p.half_shift : 0) + (ii / p.group) * p.stride + ii % p.group);
  ChunkStream cs{p.src, p.off, p.bytes, p.n_chunks, p.cap, nullptr, nullptr};
  cs.start(ring + 128, reinterpret_cast<uint64_t*>(ring));   // includes the __syncthreads that publishes sp
  int st;
  {
    double r = philox_u01(p.seed, site, (uint32_t)p.root_node, 0);
    st = A - 1;
    double cpi = 0.;
    bool done = false;
    for (int i = 0; i < A; i++) {
      cpi += __ldg(p.pi + i);
      if (!done && r <= cpi) { st = i; done = true; }
    }
  }
  const double rate = continuous_rate(cp.kind, cp.alpha, cp.p_inv, p.seed, site, (uint32_t)p.root_node);
  if (live && p.classes) p.classes[idx] = -1;
  auto draw = [&](int x, int node, double u) {
    if (rate == 0.) return x;                       // invariant site: P = I
    const double t = __ldg(brlen + node) * rate;
    double ek[AMAX];
#pragma unroll
    for (int k = 0; k < AMAX; k++) ek[k] = k < A ? R[x * A + k] * exp(ev[k] * t) : 0.;
    double cum = 0.;
    int y = A - 1;
    bool done = false;
    for (int j = 0; j < A; j++) {
      double pj = 0.;
#pragma unroll
      for (int k = 0; k < AMAX; k++) if (k < A) pj += ek[k] * L[k * A + j];
      cum += pj;
      if (!done && u < cum) { y = j; done = true; }
    }
    return y;
  };
  uint8_t stk[kMaxStack];
  int spt = 0;
  const size_t tab = (size_t)p.C * AA;
  for (uint32_t k = 0; k < p.n_chunks; k++) {
    const unsigned char* rp = cs.wait(k);
    const uint32_t nrec = __ldg(p.nrec + k);
    for (uint32_t r = 0; r < nrec; r++) {
      const int4 h0 = *reinterpret_cast<const int4*>(rp);
      const int4 h1 = *reinterpret_cast<const int4*>(rp + 16);
      const uint32_t flags = (uint32_t)h0.x;
      rp += (32 + 2 * tab * sizeof(double) + 15) & ~size_t(15);
      int sa = st, sb = st;
      double u0 = 0., u1 = 0.;
      if (h0.w >= 0) {
        philox_u01x2(p.seed, site, (uint32_t)h1.w, 2u + ((uint32_t)h1.y >> 1), u0, u1);
        sa = draw(st, h0.w, (h1.y & 1) ? u1 : u0);
      }
      if (h1.x >= 0) {
        if (h0.w < 0 || (h1.y >> 1) != (h1.z >> 1))
          philox_u01x2(p.seed, site, (uint32_t)h1.w, 2u + ((uint32_t)h1.z >> 1), u0, u1);
        sb = draw(st, h1.x, (h1.z & 1) ? u1 : u0);
      }
      if ((flags & kUpTipA) && live) p.tips[(size_t)h0.y * p.n_pad + idx] = (uint8_t)sa;
      if ((flags & kUpTipB) && live) p.tips[(size_t)h0.z * p.n_pad + idx] = (uint8_t)sb;
      if (flags & kUpTakeA) {
        if (flags & kUpPush) stk[spt++] = (uint8_t)sb;
        st = sa;
      } else if (flags & kUpTakeB) st = sb;
      else if (flags & kUpPop) st = stk[--spt];
    }
    cs.release(k);
  }
}

} // namespace

void launch_simulate(const MapModel& m, const DevStream& s, uint64_t seed, int64_t base, int64_t group,
                     int64_t stride, int64_t n, int64_t n_pad, int weighted, int root_node, uint8_t* tips,
                     int32_t* classes, cudaStream_t st, int64_t half_n, int64_t half_col, int64_t half_shift,
                     const ColumnKeys* keys) {
  if (n_pad >= ((int64_t)1 << 32)) fail("internal: simulated batch of %lld padded sites", (long long)n_pad);
  SimParams p;
  p.half_n = half_n; p.half_col = half_col; p.half_shift = half_shift;
  p.src = s.bytes.as<unsigned char>(); p.off = s.off.as<uint32_t>(); p.bytes = s.nbytes.as<uint32_t>();
  p.nrec = s.nrec.as<uint32_t>(); p.n_chunks = s.n_chunks; p.cap = s.cap;
  p.A = m.A; p.C = m.C; p.root_node = root_node; p.weighted = weighted; p.seed = seed;
  for (int r = 0; r < 10; r++) { // Philox4x32 key schedule: both halves bumped by their Weyl constants every round
    p.rk[2 * r] = (uint32_t)seed + (uint32_t)r * 0x9E3779B9u;
    p.rk[2 * r + 1] = (uint32_t)(seed >> 32) + (uint32_t)r * 0xBB67AE85u;
  }
  p.base = base; p.group = group; p.stride = stride; p.n = n; p.n_pad = n_pad;
  p.pi = m.pi; p.probs = m.probs; p.tips = tips; p.classes = classes;
  p.key_hash = keys ? keys->hash : nullptr;
  p.key_col = keys ? keys->col : nullptr;
  p.key_packed = keys ? keys->packed : nullptr;
  if (keys && (m.cont_kind != 0 || m.A != 4)) fail("internal: fused column keys need the discrete nucleotide simulator");
  size_t smem = 128 + 2 * (size_t)s.cap;
  if (m.cont_kind != 0) {
    if (!m.spec) fail("internal: continuous simulation without the generator's spectrum");
    ContParams cp{m.cont_kind, m.cont_alpha, m.cont_pinv, m.spec, 0};
    smem += (sizeof(double) * (m.A + 2 * (size_t)m.A * m.A) + 127) & ~size_t(127);
    if (m.A <= 4) {
      CMB_CUDA(cudaFuncSetAttribute(k3_simulate_cont<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      k3_simulate_cont<4><<<(unsigned)((n + NT - 1) / NT), NT, smem, st>>>(p, cp);
    } else if (m.A <= 20) {
      CMB_CUDA(cudaFuncSetAttribute(k3_simulate_cont<20>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      k3_simulate_cont<20><<<(unsigned)((n + NT - 1) / NT), NT, smem, st>>>(p, cp);
    } else fail("continuous simulation supports up to 20 states");
    CMB_CUDA(cudaGetLastError());
    return;
  }
  const unsigned grid = (unsigned)((n + NT - 1) / NT);
  if (m.A == 4) {
    CMB_CUDA(cudaFuncSetAttribute(k3_simulate<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    k3_simulate<4><<<grid, NT, smem, st>>>(p);
  } else if (m.A == 20) {
    CMB_CUDA(cudaFuncSetAttribute(k3_simulate<20>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    k3_simulate<20><<<grid, NT, smem, st>>>(p);
  } else {
    CMB_CUDA(cudaFuncSetAttribute(k3_simulate<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    k3_simulate<0><<<grid, NT, smem, st>>>(p);
  }
  CMB_CUDA(cudaGetLastError());
}

} // namespace cmb
