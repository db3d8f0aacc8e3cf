// Weight gradient of the sparse convolutions on 5th-generation tensor cores (sm_100a only):
//     dW[k] (+)= sum over pairs (i, o) of rules[k]   x[i, :]^T . dout[o, :]          (bf16 or TF32 operands, fp32 accumulate)
//
// The contraction index is the PAIR, so -- unlike the forward, where missing neighbours are masked output rows -- the
// live pairs of an offset can be compacted freely: a stage is 64 compacted pairs, its A operand the 64 gathered x rows
// and its B operand the 64 gathered dout rows, both stored exactly like the forward's A tiles (one 128-byte row per
// pair and 64-channel block, SWIZZLE_128B).  Read through MN-MAJOR shared-memory descriptors the same bytes are
// x^T (M = input channels, K = pairs) and dout (K = pairs, N = output channels), so one tcgen05.mma (M=128, N=Cout,
// K=16) contracts 16 pairs and the Cin x Cout accumulator of the offset stays in TMEM for the whole CTA.
//
// Work split: every CTA owns ONE offset k and a contiguous range of output rows (the centre offset of a submanifold
// table holds every row and gets proportionally more CTAs).  A CTA writes its Cin x Cout partial sum to a slab of its
// own; k_wgrad_reduce adds the slabs of an offset into dW in a fixed order.
// Roles: producer warps (each walks its share of 128-row blocks, ballots the neighbour indices, appends the live pairs
// to a ring and emits a stage whenever 64 are pending; LDGSTS copies that signal their own landing), one issuing warp
// that consumes the producers' stages in a fixed round-robin order (so dW is bitwise reproducible), 4 epilogue warps
// (tcgen05.ld -> slab stores).
//
// TF32 instantiation (precision SCN_PREC_TF32, fp32 x and dout): a stage row is 128 bytes = 32 fp32 channels, so blocks
// are 32 channels wide (nca, ncb up to 8: runtime counts, one instantiation per pairs-per-stage) and one
// tcgen05.mma (kind::tf32) contracts K = 8 pairs.  MN-major TF32 operands must use the 128-byte swizzle with 32-byte
// atomicity (SWIZZLE_128B_BASE32B, descriptor layout type 1; CUTLASS cute/arch/mma_sm100_desc.hpp and
// Layout_MN_SW128_32B_Atom = Swizzle<2,5,2>): the 32-byte granule g of row r sits at g ^ (r & 3), 4-row atoms of
// 512 bytes (SBO), instead of the 16-byte chunk c at c ^ (r & 7) in 8-row atoms of 1024 bytes.
//
// Replaces SCN's dConvolution_KMxKN_backward_dW_A/B (SURVEY.md 2.2); reference call sites
// src/networks/sparse_building_blocks.py:29-34,110-117 (backward).
#include <cstdlib>
#include <map>
#include <mutex>

#include "common.cuh"
#include "tc_ptx.cuh"

namespace wg {

using namespace tcptx;

constexpr int EPI_WARPS = 4;              // warps 0..3 (TMEM lane quarter = warp index)
constexpr int PROD_WARPS = 6;             // warps 4..9; the first NPW are active, two slots each
constexpr int WARP_MMA = EPI_WARPS + PROD_WARPS;
constexpr int THREADS = 32 * (WARP_MMA + 1);
constexpr int MAX_SLOTS = 2 * PROD_WARPS;
constexpr int RING = 256;                 // pending-pair ring per producer warp (entries), a power of two

struct Params {
  const void* x;                // [n_in_rows, Cin] bf16 (fp32 for the TF32 instantiation)
  const void* dout;             // [n_rows, Cout], the element type of x
  const int32_t* nbr;           // [K][n_pad]: input row of output row o at offset k, or -1
  float* part;                  // [gridDim.x][Cin][Cout] partial sums, one slab per CTA
  int64_t n_rows, n_pad;
  int K, Cin, Cout;
  int nca, ncb;                 // channel blocks (128-byte rows: 64 bf16 / 32 fp32 channels) per stage: A, B
  int nmb;                      // M blocks of 128 input channels
  int slots, npw;               // stage slots, active producer warps (slots == 2 * npw)
  int s_other, s_centre, centre;   // CTAs per ordinary offset / for the centre offset (or -1)
};

// MN-major 128-byte-swizzled descriptor: rows of 128 bytes along M/N, `lbo` bytes between consecutive 128-byte blocks
// along M/N.  bf16: SWIZZLE_128B, 8 K-rows per 1024-byte atom (SBO); TF32: SWIZZLE_128B_BASE32B, 4 K-rows per 512-byte
// atom.
template <bool TF32>
__device__ __forceinline__ uint64_t make_desc_mn_sw128(uint32_t saddr, uint32_t lbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr & 0x3FFFFu) >> 4);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFFu) << 16;
  d |= (uint64_t)((TF32 ? 512 : 1024) >> 4) << 32;
  d |= (uint64_t)1 << 46;       // descriptor version 1 (sm_100)
  d |= (uint64_t)(TF32 ? 1 : 2) << 61;   // LayoutType::SWIZZLE_128B_BASE32B / SWIZZLE_128B
  return d;
}
// fp32 accumulate, A and B MN-major, M = 128, N = n; bf16 (kind::f16) or TF32 (kind::tf32) operands
template <bool TF32>
__device__ __forceinline__ uint32_t make_idesc_mn(int n) {
  constexpr uint32_t fmt = TF32 ? 2u : 1u;
  return (1u << 4) | (fmt << 7) | (fmt << 10) | (1u << 15) | (1u << 16) | ((uint32_t)(n >> 3) << 17) | (8u << 24);
}
template <bool TF32>
__device__ __forceinline__ void umma(uint32_t tmem_d, uint64_t da, uint64_t db, uint32_t idesc, uint32_t accumulate) {
  if constexpr (TF32)
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(da), "l"(db), "r"(idesc), "r"(accumulate)
        : "memory");
  else
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(da), "l"(db), "r"(idesc), "r"(accumulate)
        : "memory");
}

// NA / NB: 64-channel blocks of a stage's A (x rows) / B (dout rows) operand = ceil(Cin / 64), ceil(Cout / 64)
// HALF: Cin == Cout == 32, rows are 64 bytes: 4 lanes per row and 8 rows per pass instead of 8 lanes / 4 rows
// PAIRS: pairs (MMA K rows) per stage: 64, or 32 for the wide layers (NA + NB >= 5: a 64-pair stage is 40-48 KB, only 4
// slots = 2 producer warps fit; measured 78 us for 258 k pairs at 160 channels against 73 us for 805 k pairs at 128).
// (Two-warp producer teams per stage were measured too and are slower: 117 -> 168 us at 96 channels.)
// TF32: NA == NB == 0, the block counts (1..8 each) are p.nca / p.ncb; PAIRS 64, 32 or 16 (see scn_wgrad_tc).
template <int NA, int NB, bool HALF, int PAIRS, bool TF32 = false>
__global__ void __launch_bounds__(THREADS, 1) k_wgrad_tc(const Params p) {
  static_assert(TF32 == (NA == 0 && NB == 0), "TF32 takes its block counts at run time");
  static_assert(!(TF32 && HALF), "fp32 rows of 32 channels are whole 128-byte rows");
  constexpr int NAM = TF32 ? 8 : NA, NBM = TF32 ? 8 : NB;   // bounds of the (unrolled) block loops
  const int na = TF32 ? p.nca : NA, nb = TF32 ? p.ncb : NB;
  constexpr int BLK_BYTES = PAIRS * 128;                 // one channel block of a stage: PAIRS rows x 128 B
  extern __shared__ unsigned char smem_raw[];
  pdl_launch_dependents();                               // see common.cuh: programmatic dependent launch
  const uint32_t raw = smem_u32(smem_raw);
  const uint32_t base = (raw + 1023u) & ~1023u;
  unsigned char* gbase = smem_raw + (base - raw);
  const int slots = p.slots, NPW = p.npw;
  const uint32_t slot_bytes = (uint32_t)(na + nb) * BLK_BYTES;
  const uint32_t bar0 = base + (uint32_t)slots * slot_bytes;
  auto afull = [&](int s) { return bar0 + 8u * (uint32_t)s; };
  auto aempty = [&](int s) { return bar0 + 8u * (uint32_t)(MAX_SLOTS + s); };
  const uint32_t accf = bar0 + 8u * (uint32_t)(2 * MAX_SLOTS);
  unsigned char* tail = gbase + (size_t)slots * slot_bytes + 8 * (2 * MAX_SLOTS + 2);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tail);
  const uint32_t seq = smem_u32(tail + 16);                          // [MAX_SLOTS] u32: per-warp stage number + 1 (| parity << 31)
  const uint32_t done = smem_u32(tail + 16 + 4 * MAX_SLOTS);         // [PROD_WARPS] u32: stages emitted + 1 once the warp is finished
  int2* rings = reinterpret_cast<int2*>(tail + 16 + 4 * MAX_SLOTS + 4 * PROD_WARPS + 8);   // [PROD_WARPS][RING]

  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;

  // ---- this CTA's offset and row range ------------------------------------------------------------------
  int k, piece, pieces;
  {
    const int b = (int)blockIdx.x;
    const int before = p.centre >= 0 ? p.centre * p.s_other : 0x7fffffff;
    if (b < before) { k = b / p.s_other; piece = b % p.s_other; pieces = p.s_other; }
    else if (b < before + p.s_centre) { k = p.centre; piece = b - before; pieces = p.s_centre; }
    else { const int b2 = b - p.s_centre + p.s_other; k = b2 / p.s_other; piece = b2 % p.s_other; pieces = p.s_other; }
  }
  const int64_t nblocks = (p.n_rows + 127) / 128;                    // 128-row blocks of the table
  const int64_t blk_lo = nblocks * piece / pieces, blk_hi = nblocks * (piece + 1) / pieces;

  if (warp == WARP_MMA) {
    if (lane == 0) {
      for (int s = 0; s < slots; ++s) {
        st_release_u32(seq + 4u * (uint32_t)s, 0u);
        mbar_init(afull(s), 32);                 // the 32 lanes of the owning producer warp, each when its copies landed
        mbar_init(aempty(s), 1);                 // one tcgen05.commit
      }
      for (int w = 0; w < PROD_WARPS; ++w) st_release_u32(done + 4u * (uint32_t)w, 0u);
      mbar_init(accf, 1);
      asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncwarp();
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  pdl_wait();                                            // everything above overlapped the previous kernel's tail

  if (warp >= EPI_WARPS && warp < EPI_WARPS + PROD_WARPS) {
    // ================================ producers =============================================
    const int pw = warp - EPI_WARPS;
    if (pw < NPW) {
      int2* ring = rings + pw * RING;                       // .x: x row offset / 16 B, .y: dout row offset / 16 B
      const uint32_t xvec = (uint32_t)p.Cin >> (TF32 ? 2 : 3), dvec = (uint32_t)p.Cout >> (TF32 ? 2 : 3);
      const uint32_t lt = (1u << lane) - 1u;
      constexpr int LPR = HALF ? 4 : 8;                     // lanes per row
      constexpr int RPP = 32 / LPR;                         // rows per pass
      const int chunk = lane % LPR, sub = lane / LPR;
      const uint32_t csw = (uint32_t)chunk << 4;
      const unsigned char* xb = reinterpret_cast<const unsigned char*>(p.x);
      const unsigned char* db = reinterpret_cast<const unsigned char*>(p.dout);
      int head = 0, pending = 0, emitted = 0;

      // per-lane invariants of the copies: this lane moves 16-byte chunk `chunk` of every channel block (TF32: the
      // channel counts are multiples of 32, every block is a whole row)
      bool a_ok[NAM], b_ok[NBM];
#pragma unroll
      for (int b = 0; b < NAM; ++b) a_ok[b] = TF32 || b * 64 + chunk * 8 < p.Cin;
#pragma unroll
      for (int b = 0; b < NBM; ++b) b_ok[b] = TF32 || b * 64 + chunk * 8 < p.Cout;
      const unsigned char* xsrc = xb + ((uint32_t)chunk << 4);
      const unsigned char* dsrc = db + ((uint32_t)chunk << 4);

      // emits one stage from the first `take` (<= 64) pending pairs; rows beyond `take` are zero-filled.
      // ~6 instructions per 16-byte copy: LDS.64 (shared by the row's copies), IMAD.WIDE, LOP3, LDGSTS.
      auto emit = [&](int take) {
        const int slot = pw + (emitted & 1) * NPW;
        const uint32_t sbase = base + (uint32_t)slot * slot_bytes;
        mbar_wait(aempty(slot), (((uint32_t)emitted >> 1) & 1u) ^ 1u);   // MMAs of this slot's previous stage retired
#pragma unroll 4
        for (int pass = 0; pass < PAIRS / RPP; ++pass) {
          const int row = pass * RPP + sub;                  // stage row (pair), LPR lanes per row
          const bool live = row < take;
          const int2 e = live ? ring[(head + row) & (RING - 1)] : make_int2(0, 0);
          // SWIZZLE_128B: 16-byte chunk c at c ^ (row & 7); TF32 (SWIZZLE_128B_BASE32B): 32-byte granule c / 2 at
          // (c / 2) ^ (row & 3)
          const uint32_t rsw = TF32 ? ((uint32_t)(row & 3) << 5) : ((uint32_t)(row & 7) << 4);
          const uint32_t dst = (sbase + (uint32_t)row * 128u + rsw) ^ csw;
          const unsigned char* xs = xsrc + ((uint64_t)(uint32_t)e.x << 4);
          const unsigned char* ds = dsrc + ((uint64_t)(uint32_t)e.y << 4);
#pragma unroll
          for (int b = 0; b < NAM; ++b) {                    // x row -> A blocks
            if (TF32 && b >= na) break;
            const bool ok = live && a_ok[b];
            cp_async16(dst + (uint32_t)b * BLK_BYTES, ok ? xs + b * 128 : xs, ok ? 16u : 0u);
          }
#pragma unroll
          for (int b = 0; b < NBM; ++b) {                    // dout row -> B blocks
            if (TF32 && b >= nb) break;
            const bool ok = live && b_ok[b];
            cp_async16(dst + (uint32_t)(na + b) * BLK_BYTES, ok ? ds + b * 128 : ds, ok ? 16u : 0u);
          }
        }
        cp_async_arrive_noinc(afull(slot));
        __syncwarp();
        if (lane == 0)
          st_release_u32(seq + 4u * (uint32_t)slot, ((uint32_t)emitted + 1u) | ((((uint32_t)emitted >> 1) & 1u) << 31));
        head = (head + take) & (RING - 1);
        pending -= take;
        ++emitted;
      };

      const int32_t* tab = p.nbr + (int64_t)k * p.n_pad;
      int jn[4] = {-1, -1, -1, -1};                       // indices of the NEXT block, loaded one block ahead
      if (blk_lo + pw < blk_hi) {
#pragma unroll
        for (int i = 0; i < 4; ++i) jn[i] = ldg_nc32(tab + (blk_lo + pw) * 128 + 32 * i + lane);
      }
      for (int64_t blk = blk_lo + pw; blk < blk_hi; blk += NPW) {
        const int64_t o0 = blk * 128;
        int j[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) j[i] = jn[i];          // (table rows beyond n_rows are -1 padding)
        if (blk + NPW < blk_hi) {
#pragma unroll
          for (int i = 0; i < 4; ++i) jn[i] = ldg_nc32(tab + (blk + NPW) * 128 + 32 * i + lane);
        }
        int at = pending;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const uint32_t m = __ballot_sync(0xffffffffu, j[i] >= 0);
          if (j[i] >= 0)
            ring[(head + at + __popc(m & lt)) & (RING - 1)] =
                make_int2((int)((uint32_t)j[i] * xvec), (int)((uint32_t)(o0 + 32 * i + lane) * dvec));
          at += __popc(m);
        }
        pending = at;
        __syncwarp();
        while (pending >= PAIRS) emit(PAIRS);
      }
      if (pending > 0) emit(pending);
      if (lane == 0) st_release_u32(done + 4u * (uint32_t)pw, (uint32_t)emitted + 1u);
    }
  } else if (warp == WARP_MMA) {
    // ================================ MMA issuer ============================================
    const uint32_t idesc = make_idesc_mn<TF32>(p.Cout);
    const uint32_t a_lbo = BLK_BYTES, b_lbo = BLK_BYTES;
    int consumed[PROD_WARPS];
#pragma unroll
    for (int w = 0; w < PROD_WARPS; ++w) consumed[w] = 0;
    bool first = true;
    for (;;) {
      bool all_done = true;
#pragma unroll
      for (int w = 0; w < PROD_WARPS; ++w) {
        if (w >= NPW) continue;
        // Stages are consumed in a FIXED order (round robin over the producers, each in its own order), so the fp32
        // accumulation order in TMEM, and with it every bit of dW, does not depend on timing: wait for producer w's
        // next stage, or for w to be finished and drained.  (Taking whichever producer was ready first made repeated
        // launches differ in the last bits.)  One lane's view of the flags, broadcast: the branches must be warp-uniform.
        const int slot = w + (consumed[w] & 1) * NPW;
        bool drained = false;
        uint32_t f = 0, idle = 0;
        for (;;) {
          const uint32_t dn = __shfl_sync(0xffffffffu, ld_acquire_u32(done + 4u * (uint32_t)w), 0);
          if (dn != 0u && (uint32_t)consumed[w] + 1u == dn) { drained = true; break; }
          f = __shfl_sync(0xffffffffu, ld_acquire_u32(seq + 4u * (uint32_t)slot), 0);
          if ((f & 0x7fffffffu) == (uint32_t)consumed[w] + 1u) break;         // its next stage is issued
          if (++idle > 8u * SPIN_LIMIT) __trap();                             // polls of ONE producer (not all NPW)
        }
        if (drained) continue;
        all_done = false;
        __syncwarp();
        mbar_wait(afull(slot), f >> 31);                                       // ... and landed
        tc_fence_after();
        const uint32_t sbase = base + (uint32_t)slot * slot_bytes;
        if (elect_one()) {
          // M = 128 reads BPM blocks (two of 64 bf16 / four of 32 fp32 channels); a single last block is read BPM times
          // (LBO = 0), a last M block of 2 or 3 TF32 blocks reads on into the following blocks: accumulator rows beyond
          // Cin are never looked at by the epilogue
          constexpr int BPM = TF32 ? 4 : 2;
          constexpr int KPM = TF32 ? 8 : 16;                 // pairs (K rows) per MMA: 32 bytes of K
#pragma unroll
          for (int mb = 0; mb < (NAM + BPM - 1) / BPM; ++mb) {
            if (TF32 && mb * BPM >= na) break;
            const uint32_t tmem_d = tmem_base + (uint32_t)(mb * p.Cout);
            const uint32_t lbo = (BPM * mb + 1 < na) ? a_lbo : 0u;
#pragma unroll
            for (int kk = 0; kk < PAIRS / KPM; ++kk) {
              const uint32_t koff = (uint32_t)kk * (uint32_t)(KPM * 128);
              const uint64_t da = make_desc_mn_sw128<TF32>(sbase + (uint32_t)(BPM * mb) * BLK_BYTES + koff, lbo);
              const uint64_t db = make_desc_mn_sw128<TF32>(sbase + (uint32_t)na * BLK_BYTES + koff, b_lbo);
              umma<TF32>(tmem_d, da, db, idesc, (first && kk == 0) ? 0u : 1u);
            }
          }
          umma_commit(aempty(slot));
        }
        __syncwarp();
        first = false;
        ++consumed[w];
      }
      if (all_done) break;
    }
    // `first` still true <=> no pair at all in this CTA's range: the epilogue must not add the (uninitialised) accumulator.
    // Written before the commit: the epilogue reads it after the commit's barrier has completed.
    if (lane == 0) st_release_u32(done + 4u * (uint32_t)PROD_WARPS, first ? 1u : 2u);
    __syncwarp();
    if (elect_one()) umma_commit(accf);
    __syncwarp();
  } else if (warp < EPI_WARPS) {
    // ================================ epilogue: TMEM -> slab ==================================
    mbar_wait_long(accf, 0u);
    tc_fence_after();
    const uint32_t any = ld_acquire_u32(done + 4u * (uint32_t)PROD_WARPS);
    // The CTA's Cin x Cout partial sum goes to its own slab with plain 16-byte stores; k_wgrad_reduce then adds the slabs of
    // an offset in a fixed order (deterministic).  Atomics straight into dW were ~44% of the kernel's time on the
    // deep levels (148-296 CTAs x 25-37 k red.global.add each; ncu: the other warps idle at the exit barrier meanwhile).
    for (int mb = 0; mb < (TF32 ? p.nmb : (NA + 1) / 2); ++mb) {
      const int cin = mb * 128 + warp * 32 + lane;                            // accumulator row == input channel
      const uint32_t taddr = tmem_base + ((uint32_t)(warp * 32) << 16) + (uint32_t)(mb * p.Cout);
      // one 32-column chunk at a time: unrolled, this loop takes 76-78 registers instead of 43-56
#pragma unroll 1
      for (int c0 = 0; c0 < p.Cout; c0 += 32) {
        uint32_t v[32];
        if (any == 2u) {
          tmem_ld32(taddr + (uint32_t)c0, v);
        } else {
#pragma unroll
          for (int e = 0; e < 32; ++e) v[e] = 0u;                             // no pair in this CTA's range: a slab of zeros
        }
        if (cin < p.Cin) {
          uint4* dst = reinterpret_cast<uint4*>(p.part + ((size_t)blockIdx.x * p.Cin + cin) * p.Cout + c0);
#pragma unroll
          for (int e = 0; e < 8; ++e) dst[e] = make_uint4(v[4 * e], v[4 * e + 1], v[4 * e + 2], v[4 * e + 3]);
        }
      }
    }
    tc_fence_before();
  }

  tc_fence_before();
  __syncthreads();
  if (warp == WARP_MMA) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512) : "memory");
  }
}

// dW[k] += sum over the CTAs of offset k of their slabs (4 floats per thread, slabs added in CTA order: deterministic)
// Block 0 also finishes the convolution's bias gradient when the column sums of dout are already known (they come out
// of the BatchNorm backward that produced dout): dbias (+)= colsum, folded in here instead of one more launch.
__global__ void k_wgrad_reduce(const float* __restrict__ part, float* __restrict__ dW, int K, int CC, int s_other, int s_centre,
                               int centre, const float* __restrict__ colsum, float* dbias, int nbias, int accumulate_bias) {
  pdl_launch_dependents();
  pdl_wait();
  if (blockIdx.x == 0 && colsum != nullptr)
    for (int c = threadIdx.x; c < nbias; c += blockDim.x) dbias[c] = (accumulate_bias ? dbias[c] : 0.f) + colsum[c];
  const int64_t i = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) * 4;
  if (i >= (int64_t)K * CC) return;
  const int k = (int)(i / CC);
  const int e = (int)(i - (int64_t)k * CC);
  int first, count;
  if (centre < 0 || k < centre) { first = k * s_other; count = s_other; }
  else if (k == centre) { first = centre * s_other; count = s_centre; }
  else { first = centre * s_other + s_centre + (k - centre - 1) * s_other; count = s_other; }
  // dW may be a view into a flat gradient arena: only 4-byte aligned, so it is read and written as scalars
  float4 acc = make_float4(dW[i], dW[i + 1], dW[i + 2], dW[i + 3]);
  for (int c = 0; c < count; ++c) {
    const float4 v = *reinterpret_cast<const float4*>(part + (size_t)(first + c) * CC + e);
    acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
  }
  dW[i] = acc.x; dW[i + 1] = acc.y; dW[i + 2] = acc.z; dW[i + 3] = acc.w;
}

// library-owned slab buffer per (device, stream), grown on demand (a growth is a cudaFree + cudaMalloc, i.e. a device
// synchronisation; it happens a handful of times in the first step)
int wgrad_slabs(size_t bytes, cudaStream_t s, float** out) {
  static std::mutex mu;
  static std::map<std::pair<int, cudaStream_t>, std::pair<float*, size_t>> table;
  int dev = 0;
  SCN_CUDA(cudaGetDevice(&dev));
  std::lock_guard<std::mutex> lock(mu);
  auto& e = table[{dev, s}];
  if (e.second < bytes) {
    if (e.first != nullptr) {
      SCN_CUDA(cudaStreamSynchronize(s));
      cudaFree(e.first);
      e = {nullptr, 0};
    }
    const size_t want = bytes + bytes / 4;
    float* p = nullptr;
    const cudaError_t err = cudaMalloc(&p, want);
    if (err != cudaSuccess) { (void)cudaGetLastError(); return (int)err; }
    e = {p, want};
  }
  *out = e.first;
  return SCN_OK;
}

struct BiasFold { const float* colsum; float* dbias; int C; int accumulate; };
static thread_local BiasFold g_fold = {nullptr, nullptr, 0, 0};

}  // namespace wg

// module_api.cu: "dbias (+)= colsum" is pending for the next weight-gradient launch of this thread; scn_wgrad_tc folds
// it into its reduction kernel when it runs one (and clears it), otherwise the caller does it itself.
void scn_wgrad_set_bias_fold(const float* colsum, float* dbias, int C, int accumulate) {
  wg::g_fold = {colsum, dbias, C, accumulate};
}
bool scn_wgrad_bias_fold_pending() { return wg::g_fold.colsum != nullptr; }

// the configuration of the last k_wgrad_tc launch (developer entry like scn_tc_debug_knobs, for the tests' coverage
// check): grid, s_other, s_centre, pairs per stage, slots, nca, ncb; written on the host just before the launch
static int32_t g_wg_last_launch[7] = {0, 0, 0, 0, 0, 0, 0};
extern "C" void scn_wgrad_debug_last_launch(int32_t* out) {
  for (int i = 0; i < 7; ++i) out[i] = g_wg_last_launch[i];
}

// dW[K][Cin][Cout] += ...; x, dout bf16, or fp32 with tf32 != 0 (TF32 MMAs).  Returns SCN_ERR_UNSUPPORTED for shapes
// outside the kernel (caller falls back).  Gathered rows are addressed through 32-bit offsets in 16-byte units: x and
// dout up to 64 GB each.
int scn_wgrad_tc(const void* x, const void* dout, const int32_t* nbr, int K, int64_t n_rows, int64_t n_pad, int Cin, int Cout,
                 int tf32, float* dW, cudaStream_t s) {
  if ((Cin % 32) || (Cout % 32) || Cin < 32 || Cout < 32 || Cin > 256 || Cout > 256 || K < 1) return SCN_ERR_UNSUPPORTED;
  if ((uint64_t)n_rows * (uint64_t)(Cout * (tf32 ? 4 : 2) / 16) >= 0xffffffffull) return SCN_ERR_UNSUPPORTED;
  if (n_pad < ((n_rows + 127) / 128) * 128) return SCN_ERR_ARG;      // whole 128-row blocks are read
  wg::Params p;
  p.x = x; p.dout = dout; p.nbr = nbr; p.n_rows = n_rows; p.n_pad = n_pad; p.K = K; p.Cin = Cin; p.Cout = Cout;
  p.nmb = (Cin + 127) / 128;
  const int blk = tf32 ? 32 : 64;                            // channels per 128-byte block
  p.nca = (Cin + blk - 1) / blk;
  p.ncb = (Cout + blk - 1) / blk;
  if (p.nmb * Cout > 512) return SCN_ERR_UNSUPPORTED;
  // pairs per stage (see the kernel).  TF32 blocks hold half the channels of bf16 ones: the same thresholds in bytes per
  // pair, and one more halving for the widest layers (a 32-pair stage of 256 x 256 fp32 is 64 KB: 2 slots only)
  const int nbl = p.nca + p.ncb;
  const int pairs = tf32 ? (nbl >= 10 ? 16 : (nbl >= 5 ? 32 : 64)) : (nbl >= 5 ? 32 : 64);
  const uint32_t slot_bytes = (uint32_t)(p.nca + p.ncb) * (uint32_t)pairs * 128u;
  const uint32_t fixed = 1024u + 8u * (2 * wg::MAX_SLOTS + 2) + 16u + 4u * wg::MAX_SLOTS + 4u * wg::PROD_WARPS + 8u +
                         (uint32_t)wg::PROD_WARPS * wg::RING * 8u;
  int slots = (int)((226u * 1024u - fixed) / slot_bytes);
  if (slots > wg::MAX_SLOTS) slots = wg::MAX_SLOTS;
  slots &= ~1;
  if (slots < 2) return SCN_ERR_UNSUPPORTED;
  p.slots = slots;
  p.npw = slots / 2;
  // CTAs (one per SM at a time: the kernel uses all of shared memory): ONE full wave, or two for big tables -- never
  // a few CTAs more than a wave (150 CTAs on 148 SMs run for two waves: measured 86 us instead of ~45 at 20 k rows x
  // 160 channels).  The centre offset of an odd-sized (submanifold) table holds every row -> 3.5x the share of the
  // others.  Small tables get fewer CTAs: every CTA pays a fixed price (TMEM allocation, a Cin*Cout slab), so it
  // should own ~500 pairs or more (about 30% of the K*n table entries are pairs in the reference's networks).
  static const int pairs_per_cta = [] {                      // developer knob for sweeps: SCN_B200_WG_PAIRS=<pairs per CTA>
    const char* e = std::getenv("SCN_B200_WG_PAIRS");
    const int v = e ? std::atoi(e) : 0;
    return v > 0 ? v : 512;
  }();
  const int64_t by_work = (int64_t)((double)n_rows * K * 0.3 / (double)pairs_per_cta);
  int target = by_work >= (int64_t)(2 * kNumSMs * 0.85) ? 2 * kNumSMs : (by_work >= kNumSMs ? kNumSMs : (int)by_work);
  if (target < K) target = K;
  const int64_t nblocks = (n_rows + 127) / 128;
  if ((K & 1) && K > 1) {
    p.centre = K / 2;
    const double unit = (double)target / ((double)(K - 1) + 3.5);
    p.s_other = (int)unit;
    if (p.s_other < 1) p.s_other = 1;
    p.s_centre = target - (K - 1) * p.s_other;
    if (p.s_centre > (int)(3.5 * unit + 1.5)) p.s_centre = (int)(3.5 * unit + 1.5);
  } else {
    p.centre = -1;
    p.s_other = target / K;
    p.s_centre = 0;
  }
  if (p.s_other < 1) p.s_other = 1;
  if (p.s_other > nblocks) p.s_other = (int)(nblocks > 0 ? nblocks : 1);
  if (p.centre >= 0) {
    if (p.s_centre < 1) p.s_centre = 1;
    if (p.s_centre > nblocks) p.s_centre = (int)(nblocks > 0 ? nblocks : 1);
  }
  const int grid = (p.centre >= 0 ? (K - 1) * p.s_other + p.s_centre : K * p.s_other);
  const size_t smem = (size_t)fixed + (size_t)slots * slot_bytes;
  const int CC = Cin * Cout;
  const int rc = wg::wgrad_slabs((size_t)grid * CC * sizeof(float), s, &p.part);
  if (rc != SCN_OK) return rc;
  {
    const int32_t rec[7] = {grid, p.s_other, p.s_centre, pairs, slots, p.nca, p.ncb};
    for (int i = 0; i < 7; ++i) g_wg_last_launch[i] = rec[i];
  }
  auto launch = [&](auto kern) -> int {
    SCN_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    SCN_CUDA(scn_launch_pdl(kern, dim3((unsigned)grid), dim3(wg::THREADS), smem, s, p));
    SCN_LAUNCH_CHECK();
    const wg::BiasFold bf = wg::g_fold;
    wg::g_fold = {nullptr, nullptr, 0, 0};
    SCN_CUDA(scn_launch_pdl(wg::k_wgrad_reduce, dim3(grid_for((int64_t)K * CC / 4, 256)), dim3(256), 0, s, (const float*)p.part, dW,
                            K, CC, p.s_other, p.s_centre, p.centre, bf.colsum, bf.dbias, bf.C, bf.accumulate));
    SCN_LAUNCH_CHECK();
    return SCN_OK;
  };
  if (tf32) {
    if (pairs == 64) return launch(wg::k_wgrad_tc<0, 0, false, 64, true>);
    if (pairs == 32) return launch(wg::k_wgrad_tc<0, 0, false, 32, true>);
    return launch(wg::k_wgrad_tc<0, 0, false, 16, true>);
  }
  if (Cin == 32 && Cout == 32) return launch(wg::k_wgrad_tc<1, 1, true, 64>);
#define WG_CASE(a, b) if (p.nca == a && p.ncb == b) return launch(wg::k_wgrad_tc<a, b, false, ((a) + (b) >= 5 ? 32 : 64)>)
  WG_CASE(1, 1); WG_CASE(1, 2); WG_CASE(1, 3); WG_CASE(1, 4);
  WG_CASE(2, 1); WG_CASE(2, 2); WG_CASE(2, 3); WG_CASE(2, 4);
  WG_CASE(3, 1); WG_CASE(3, 2); WG_CASE(3, 3); WG_CASE(3, 4);
  WG_CASE(4, 1); WG_CASE(4, 2); WG_CASE(4, 3); WG_CASE(4, 4);
#undef WG_CASE
  return SCN_ERR_UNSUPPORTED;
}
