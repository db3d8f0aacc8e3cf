// Output-stationary gather-GEMM convolution on 5th-generation tensor cores (sm_100a only):
//     out[o, :] = bias + sum_k  in[nbr[k][o], :] . B_k            (bf16 or TF32 operands, fp32 accumulate)
//
// One persistent CTA per SM owns a contiguous range of 128-row output tiles (an even split of the tiles over the
// grid) and walks it in GROUPS of T tiles whose accumulators live in TMEM together (T * n_out <= 256 columns with two
// groups double-buffered, or <= 512 columns single-buffered when a CTA has one group anyway).  The contraction
// (K offsets x n_in channels) is cut into stages of 64 channels (one 128-byte shared-memory row).  Per stage:
//   * the weight tile B(q) (n_out x 128 B, pre-swizzled image) is streamed ONCE per group by a 1-D bulk async copy
//     (TMA engine, mbarrier complete_tx) and reused by the T tiles of the group,
//   * for each tile ONE producer warp gathers the A tile: it reads the tile's 128 neighbour indices (prefetched one
//     stage ahead), ballots them, compacts the LIVE rows into a warp-private list of (source offset, swizzled
//     destination) pairs and copies only those rows with 16-byte LDGSTS (8 lanes per 128-byte row).  The ballots are
//     published as the stage's disable-output-lane mask.  The copies signal their landing themselves
//     (cp.async.mbarrier.arrive.noinc), the warp never waits for them and alternates between its two A slots,
//   * up to 4 issuing warps (tile t -> warp t mod NM) issue tcgen05.mma (M=128, N=n_out, K=16) with that mask:
//     accumulator rows without a neighbour at this offset are not updated, so their stale A rows never reach a
//     result.  Only the first stage of a tile, which initialises the accumulator, is written in full,
//   * 4 epilogue warps drain finished accumulators (tcgen05.ld), add bias, convert and store.
// Every output row is written exactly once: no atomics, deterministic.
//
// TF32 instantiation (precision SCN_PREC_TF32, fp32 features): the same machinery at byte level -- a stage is still one
// 128-byte row per output row, now 32 fp32 channels, and one tcgen05.mma (kind::tf32, K = 8) still consumes 32 bytes of
// it, so only the channels per stage (32), the instruction descriptor, the weight image and the fp32 epilogue differ.
// The MMA reads the fp32 bits of the gathered rows as they are (the tensor core uses their upper 19 bits); the weight
// image holds values rounded to TF32 (cvt.rna).  No offset pairing: a 32-channel fp32 row already fills a stage.
//
// Synchronisation notes.  A slot's mbarriers must see consecutive phases from each waiter (a parity wait cannot tell
// phase r from r-2), hence one producer warp per pair of slots; the issuing warps run up to SA stages apart, so the
// "which stage is in this slot" handshake is a monotonically increasing sequence flag (release store / acquire poll)
// and only then the landing barrier, whose parity the flag carries.
//
// What bounds it (timeline marks, -DSCN_TC_TIMELINE + tools/tc_timeline.py; DESIGN.md 4.1): neither L2 latency
// nor the tensor pipe but the dependent-issue rate of the single warps that build a stage (~5 cycles per
// instruction), so every role's per-stage instruction count was cut (6 instructions per gathered row segment,
// ~70 per issued stage) and the roles were multiplied (5-6 producer warps, 4 issuing warps).
// History (profiles/): dense zero-filled A tiles via cp.async, TMA tile::gather4 and lock-step LDG/STS batches
// were measured first; they moved all 128 rows per stage although ~30% are live.
//
// Replaces SCN's dConvolution_KMxKN_forwardA/B (SURVEY.md 2.2); reference call sites
// src/networks/sparse_building_blocks.py:29-34,110-117.
#include <cstring>

#include "common.cuh"
#include "tc_ptx.cuh"

namespace tc {

constexpr int BM = 128;                 // output rows per tile == TMEM lanes
constexpr int KC = 64;                  // bf16 channels per pipeline stage (one 128-byte swizzle row)
constexpr int KC_TF32 = 32;             // fp32 channels per pipeline stage
constexpr int A_BYTES = BM * 128;       // 16 KB
constexpr int EPI_WARPS = 4;            // warps 0..3  (TMEM lane quarter = warp index)
constexpr int NGRP = 4;                 // producer groups: stage n is gathered by group n mod NGRP ...
constexpr int PROD_WARPS = 4 * NGRP;    // ... whose 4 warps own one 32-row quarter of the tile each (warps 4..19)
constexpr int WARP_MMA = EPI_WARPS + PROD_WARPS;   // first of MMA_WARPS issuing warps (tile t -> warp t mod NM)
constexpr int MMA_WARPS = 4;
constexpr int WARP_BLOAD = WARP_MMA + MMA_WARPS;   // weight tiles
constexpr int THREADS = 32 * (WARP_BLOAD + 1);     // 800
constexpr int MAX_A = 12, MAX_B = 8;    // ring depths: A tiles (a multiple of NGRP), B tiles
constexpr int MASK_BYTES = 32;          // per A slot: 2 x 128-bit disable-output-lane masks (second: PAIR upper half)
constexpr int LIST_BYTES = 64 * 8;      // per producer warp: live items of its quarter stage, (source row, smem address)
using namespace tcptx;

// K-major, SWIZZLE_128B shared-memory matrix descriptor (cute::UMMA::SmemDescriptor layout):
// rows are 128 bytes, groups of 8 rows are 1024 bytes apart (SBO); LBO unused for swizzled K-major.
__device__ __forceinline__ uint64_t make_desc_sw128(uint32_t saddr) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr & 0x3FFFFu) >> 4);
  d |= (uint64_t)1 << 16;
  d |= (uint64_t)(1024 >> 4) << 32;
  d |= (uint64_t)1 << 46;       // descriptor version 1 (sm_100)
  d |= (uint64_t)2 << 61;       // LayoutType::SWIZZLE_128B
  return d;
}
// base + 16 * units as ONE instruction (IMAD.WIDE.U32 with a 64-bit addend)
__device__ __forceinline__ const unsigned char* mad_wide16(uint32_t units, const unsigned char* base) {
  uint64_t r;
  asm("mad.wide.u32 %0, %1, 16, %2;" : "=l"(r) : "r"(units), "l"((uint64_t)(uintptr_t)base));
  return reinterpret_cast<const unsigned char*>((uintptr_t)r);
}
// instruction descriptor: fp32 accumulate, A and B K-major, M=128, N=n; a/b format bf16 (kind::f16) or TF32 (kind::tf32)
template <bool TF32>
__device__ __forceinline__ uint32_t make_idesc(int n) {
  constexpr uint32_t fmt = TF32 ? 2u : 1u;
  return (1u << 4) | (fmt << 7) | (fmt << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);
}
// 8 consecutive output values of a row, out + idx .. out + idx + 7: one 16-byte store (bf16) or two (fp32)
template <bool TF32>
__device__ __forceinline__ void store8(void* out, int64_t idx, const float* f) {
  if constexpr (TF32) {
    float4* d = reinterpret_cast<float4*>(reinterpret_cast<float*>(out) + idx);
    d[0] = make_float4(f[0], f[1], f[2], f[3]);
    d[1] = make_float4(f[4], f[5], f[6], f[7]);
  } else {
    uint4 u;
    u.x = pack_bf16x2(f[0], f[1]); u.y = pack_bf16x2(f[2], f[3]);
    u.z = pack_bf16x2(f[4], f[5]); u.w = pack_bf16x2(f[6], f[7]);
    *reinterpret_cast<uint4*>(reinterpret_cast<__nv_bfloat16*>(out) + idx) = u;
  }
}
struct Params {
  const void* in;               // [n_in_rows, n_in] bf16 (fp32 for the TF32 instantiation)
  const int32_t* nbr;           // [K][n_pad]
  const unsigned char* bimg;    // [K*nch][n_out][128 B] pre-swizzled weight tiles, one per stage
  const float* bias;            // [n_out] or null
  void* out;                    // [n_rows, n_out], the element type of `in`
  int64_t n_rows, n_pad;
  int K, n_in, n_out;
  int nch;                      // channel chunks (stages) per offset
  int last_kc;                  // channels in the last chunk of an offset (bf16: 64 or 32; TF32: 32)
  int T;                        // tiles per group
  int SA, SB;                   // A / B ring depth
  int num_tiles;
  int NM;                       // active MMA-issuing warps = min(T, MMA_WARPS)
  int nbuf;                     // 2: groups alternate between the TMEM halves (T*n_out <= 256); 1: one group uses all 512 columns
  int ksplit;                   // NM == 2 only: a CTA that owns a single tile splits its stages over the two classes (see kernel)
  unsigned long long* dbg;      // optional timeline buffer (scn_tc_debug_timeline): CTA 0 records clock64() marks
  int exp;                      // -DSCN_TC_TIMELINE builds only: timing experiments with WRONG results (SCN_B200_TC_EXP):
                                // 1 no gather copies, 2 no MMAs, 4 no output stores
};

// NCH: 64-channel chunks per offset = ceil(n_in / 64).  PAIR (n_in == 32, NCH == 1): one stage holds TWO offsets,
// 32 channels each (chunks 0-3 from offset 2q, chunks 4-7 from offset 2q+1), halving the stage count.
// TF32: fp32 features and TF32 MMAs, 32-channel chunks; NCH == 0 takes the chunk count (1..8) from p.nch, so that one
// instantiation serves every width.
template <int NCH, bool PAIR, bool TF32 = false>
__global__ void __launch_bounds__(THREADS, 1) k_conv_tc(const Params p) {
  static_assert(!(TF32 && PAIR), "a 32-channel fp32 row fills a stage");
  constexpr int ESZ = TF32 ? 4 : 2;                        // bytes per element
  constexpr int KCE = 128 / ESZ;                           // channels per full stage
  const int nch = NCH > 0 ? NCH : p.nch;
  extern __shared__ unsigned char smem_raw[];
  pdl_launch_dependents();                                 // the next kernel's CTAs may be scheduled as ours retire (common.cuh)
  const uint32_t raw = smem_u32(smem_raw);
  const uint32_t base = (raw + 1023u) & ~1023u;            // SWIZZLE_128B tiles need 1024-byte alignment
  unsigned char* gbase = smem_raw + (base - raw);
  const int SA = p.SA, SB = p.SB;
  const uint32_t b_bytes = (uint32_t)p.n_out * 128u;
  const uint32_t a_base = base;
  const uint32_t b_base = base + (uint32_t)SA * A_BYTES;
  const uint32_t bar0 = b_base + (uint32_t)SB * b_bytes;   // 8-byte aligned
  auto afull = [&](int s) { return bar0 + 8u * (uint32_t)s; };
  auto aempty = [&](int s) { return bar0 + 8u * (uint32_t)(MAX_A + s); };
  auto bfull = [&](int s) { return bar0 + 8u * (uint32_t)(2 * MAX_A + s); };
  auto bempty = [&](int s) { return bar0 + 8u * (uint32_t)(2 * MAX_A + MAX_B + s); };
  auto accf = [&](int b) { return bar0 + 8u * (uint32_t)(2 * MAX_A + 2 * MAX_B + b); };
  auto acce = [&](int b) { return bar0 + 8u * (uint32_t)(2 * MAX_A + 2 * MAX_B + 2 + b); };
  constexpr int NBAR = 2 * MAX_A + 2 * MAX_B + 4;          // 44 -> 352 bytes (a multiple of 16: amask stays 16-byte aligned)
  unsigned char* tail = gbase + (size_t)SA * A_BYTES + (size_t)SB * b_bytes + 8 * NBAR;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tail);
  uint32_t* amask = reinterpret_cast<uint32_t*>(tail + 16);                    // [MAX_A][8], 16-byte aligned
  unsigned char* lists = tail + 16 + MAX_A * MASK_BYTES;                       // [PROD_WARPS][2][LIST_BYTES]

  // warp index through a broadcast shuffle: the compiler then knows it is warp-uniform (role branches, barrier
  // addresses and slot numbers stay in uniform registers instead of per-lane copies with R2UR waterfalls)
  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;
  // timeline marks: dbg[((role * 256 + stage) * 8 + event)] = clock64(), CTA 0 only, first 256 stages of each role
  // (compiled in only with -DSCN_TC_TIMELINE: the marks cost the single-warp issue loops real time).  Roles: 0-3
  // producer groups, 4-7 issuing warps (per stage), 8 weight loader, 9 epilogue warp 0, 10-13 issuing warps (per q)
  auto mark = [&](int role, int stage, int ev) {
#ifdef SCN_TC_TIMELINE
    if (p.dbg != nullptr && blockIdx.x == 0 && lane == 0 && stage < 256)
      p.dbg[((size_t)role * 256 + stage) * 8 + ev] = (unsigned long long)clock64();
#else
    (void)role; (void)stage; (void)ev;
#endif
  };
#ifdef SCN_TC_TIMELINE
  const int exp_flags = p.exp;
#else
  constexpr int exp_flags = 0;
#endif

  // This CTA's contiguous range of tiles [tile_lo, tile_hi): an even split of the tiles over the grid, cut into groups
  // of T tiles (only the last group of a CTA can be partial; its missing tiles are not processed by anybody).
  const int T = p.T;
  const int tile_lo = (int)(((int64_t)p.num_tiles * blockIdx.x) / gridDim.x);
  const int tile_hi = (int)(((int64_t)p.num_tiles * (blockIdx.x + 1)) / gridDim.x);
  const int my_tiles = tile_hi - tile_lo;
  const int my_groups = (my_tiles + T - 1) / T;
  auto tiles_in_group = [&](int g) { return my_tiles - g * T < T ? my_tiles - g * T : T; };
  const int NSTEP = PAIR ? (p.K + 1) / 2 : p.K;            // offsets (offset pairs) per tile
  const int Q = NSTEP * nch;                                // stages per tile
  // K-split: a CTA with ONE tile (the deep levels: fewer tiles than SMs) would run all its stages through one issuing
  // warp, a serial chain of ~800 cycles per stage.  With two classes the stages are dealt q = 0, 2, 4, ... / 1, 3, 5, ...
  // to two issuing warps with separate TMEM accumulators (columns 0 and n_out), which the epilogue adds.
  const bool ksplit = p.ksplit != 0 && p.NM == 2 && my_tiles == 1;

  if (warp == WARP_MMA) {
    if (lane == 0) {
      for (int s = 0; s < SA; ++s) {
        mbar_init(afull(s), 132);                 // the 4 x 32 lanes of the stage's producer group, each when its copies landed, + 4 mask publications
        mbar_init(aempty(s), 1);                  // one tcgen05.commit
      }
      for (int s = 0; s < SB; ++s) {
        mbar_init(bfull(s), 1);                   // the loader's expect_tx arrival (+ complete_tx bytes)
        mbar_init(bempty(s), ksplit ? 1 : p.NM);  // one tcgen05.commit per issuing warp that consumes the tile
      }
      for (int b = 0; b < 2; ++b) {
        mbar_init(accf(b), p.NM);
        mbar_init(acce(b), EPI_WARPS);
      }
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
  pdl_wait();                                              // barrier init and TMEM allocation above overlapped the previous kernel's tail

  // Classes: tile t of a group belongs to class t mod NM (NM = 1, 2 or 4).  A class is an independent pipeline: ONE issuing
  // warp, NGRP / NM producer groups and a private ring of SA / NM A slots.  Every slot therefore has a single consumer
  // and its producers see consecutive phases, so plain parity mbarriers are safe (no sequence flags, no fences).
  const int NM = p.NM;
  const int spc = SA / NM;                                  // A slots per class (a multiple of NGRP / NM)

  if (warp >= EPI_WARPS && warp < EPI_WARPS + PROD_WARPS) {
    // ================================ A producers ============================================
    // Group grp serves class grp mod NM as sub-worker grp / NM: it gathers every (NGRP / NM)-th stage of the class, in
    // the class's MMA order (group, stage, tile).  Warp wq of the group owns rows 32 wq .. 32 wq + 31 of the tile: ONE
    // neighbour index per lane, one ballot, one 32-bit word of the stage's disable-output-lane mask.  A single warp
    // issues roughly one dependent instruction per 5 cycles, so the per-stage instruction count of a warp IS its
    // gather rate: a quarter stage costs ~100 instructions (the 128-row stages of the first version of this kernel:
    // ~470), and 16 warps work at once.  Live rows are compacted into a warp-private list of (source row, swizzled
    // destination) items so that every 16-byte LDGSTS pass moves 4 whole rows (8 lanes per 128-byte row; PAIR: 8 half
    // rows).  The copies signal their landing themselves (cp.async.mbarrier.arrive.noinc); the warp never waits for
    // them, and nothing in the loop is a memory fence (a MEMBAR would wait for the copies in flight).
    const int pw = warp - EPI_WARPS;
    const int grp = pw >> 2, wq = pw & 3;
    const int cls = grp % NM, sub = grp / NM, gpc = NGRP / NM;
    constexpr int LPI = PAIR ? 4 : 8;                    // lanes per item (a 128-byte row, or a 64-byte half row)
    constexpr int IPP = 32 / LPI;                        // items per pass
    const int chunk = lane % LPI, isub = lane / LPI;
    // list items: .x source row offset / 16 B (-1: zeros), .y smem address
    const uint32_t row_vec = (uint32_t)p.n_in >> (TF32 ? 2 : 3);   // 16-byte units per feature row (list offsets are in these units)
    const int last_chunks = p.last_kc * ESZ / 16;
    const uint32_t lt = (1u << lane) - 1u;
    const uint32_t csw = (uint32_t)chunk << 4;
    // swizzled address of (row 32 wq + lane, 16-byte chunk 0) in slot 0 (upper half, PAIR: ^ 0x40)
    const uint32_t myrow = 32u * (uint32_t)wq + (uint32_t)lane;
    const uint32_t drow = a_base + (myrow << 7) + ((myrow & 7u) << 4);

    // cursor over the class's stages: tile t (= cls, cls + NM, ...) of stage q (chunk cc of its offset) of group g;
    // qptr -> this lane's entry of the stage's (first) offset in tile 0 of the group: the address of a fetch is one
    // IMAD.WIDE (the 64-bit index arithmetic written out per stage was 41 of a quarter stage's 187 instructions)
    int t = cls, q = 0, cc = 0, g = 0, tv = my_groups > 0 ? tiles_in_group(0) : 0;
    const int32_t* gptr = p.nbr + (int64_t)tile_lo * BM + myrow;
    const int32_t* qptr = gptr;
    const int64_t qstride = (int64_t)p.n_pad * (PAIR ? 2 : 1);
    auto next_q = [&]() {
      ++q;
      if (++cc == nch) { cc = 0; qptr += qstride; }
    };
    auto step = [&]() {
      if (ksplit) {                                      // this class's stages: q = cls, cls + 2, ... of the only tile
        next_q(); next_q();
        if (q >= Q) { g = my_groups; tv = 0; }
        return;
      }
      t += NM;
      if (t >= tv) {
        t = cls;
        next_q();
        if (q == Q) {
          q = 0; ++g;
          gptr += (int64_t)T * BM;
          qptr = gptr;
          tv = g < my_groups ? tiles_in_group(g) : 0;
        }
      }
    };
    // only the last group of a CTA can be partial: once the class has no tile in a group it has no stage left
    auto valid = [&]() { return g < my_groups && (ksplit ? q < Q : cls < tv); };
    if (ksplit) {
      t = 0;
      if (cls == 1) next_q();
    }
    for (int i = 0; i < sub; ++i)
      if (valid()) step();
    // Neighbour indices are fetched TWO stages ahead (the cursor runs ahead of the stage being gathered): one stage of
    // lead (~500 cycles of this warp's own work) does not cover an L2 round trip under load.  A fetch returns the
    // stage's (q << 3 | cc), or -1 when no stage is left, so the cursor never has to be rewound.
    auto fetch = [&](int& jl_, int& jh_, int& q_) {
      q_ = -1; jl_ = -1; jh_ = -1;
      if (valid()) {
        const int32_t* src = qptr + t * BM;
        jl_ = ldg_nc32(src);
        if (PAIR && (2 * q + 1 < p.K)) jh_ = ldg_nc32(src + p.n_pad);
        q_ = (q << 3) | cc;
        for (int i = 0; i < gpc; ++i) step();
      }
    };

    int ls = sub;                                        // slot within the class ring (sub < gpc <= spc)
    uint32_t round = 0;
    int it = 0;
    auto do_stage = [&](const int jl, const int jh, const int qc) {
      if (wq == 0) mark(grp, it, 0);
      int2* list = reinterpret_cast<int2*>(lists + (pw * 2 + (it & 1)) * LIST_BYTES);   // two list buffers per warp, alternating
      const int slot = cls * spc + ls;
      const int ccur = qc & 7;                           // channel chunk of the offset
      const bool full = qc < (ksplit ? 16 : 8);          // first stage of an accumulator (q == 0; K-split: q < 2): unmasked MMA, every row written
      const uint32_t dst = drow + (uint32_t)slot * A_BYTES;
      // ---- live rows -> list (full stage: every row, missing ones as zeros) ----------------------------------
      const uint32_t bl = __ballot_sync(0xffffffffu, jl >= 0);
      const uint32_t bh = PAIR ? __ballot_sync(0xffffffffu, jh >= 0) : 0u;
      int nlive;
      if (full) {
        list[lane] = make_int2(jl >= 0 ? (int)((uint32_t)jl * row_vec) : -1, (int)dst);
        if (PAIR) list[32 + lane] = make_int2(jh >= 0 ? (int)((uint32_t)jh * row_vec) : -1, (int)(dst ^ 0x40u));
        nlive = PAIR ? 64 : 32;
      } else {
        const int2 el = make_int2((int)((uint32_t)jl * row_vec), (int)dst);
        const int2 eh = make_int2((int)((uint32_t)jh * row_vec), (int)(dst ^ 0x40u));
        if (jl >= 0) list[__popc(bl & lt)] = el;
        nlive = __popc(bl);
        if (PAIR) {
          if (jh >= 0) list[nlive + __popc(bh & lt)] = eh;
          nlive += __popc(bh);
        }
        // pad the list to whole passes with copies of its last item (copying a row twice is harmless): the gather
        // loop below then needs no per-item predicates (they were a third of its instructions)
        if (nlive & (IPP - 1)) {
          const bool from_hi = PAIR && bh != 0u;
          const int top = 31 - __clz(from_hi ? bh : bl);
          const int lx = __shfl_sync(0xffffffffu, from_hi ? eh.x : el.x, top);
          const int ly = __shfl_sync(0xffffffffu, from_hi ? eh.y : el.y, top);
          const int padded = (nlive + IPP - 1) & ~(IPP - 1);
          if (nlive + lane < padded) list[nlive + lane] = make_int2(lx, ly);
        }
      }
      __syncwarp();                                      // the list is complete (its buffer is rewritten two stages later)
      if (wq == 0) mark(grp, it, 1);

      // the MMAs that read this slot's previous stage have retired
      mbar_wait(aempty(slot), (round & 1u) ^ 1u);
      if (wq == 0) mark(grp, it, 2);
      if (lane == 0) {
        amask[slot * 8 + wq] = ~bl;
        if (PAIR) amask[slot * 8 + 4 + wq] = ~bh;
      }
      const int npass = (nlive + IPP - 1) / IPP;         // <= 8
      const bool lane_on = PAIR ? true : chunk < (ccur == nch - 1 ? last_chunks : 8);
      const unsigned char* src0 = reinterpret_cast<const unsigned char*>(p.in) + ((uint32_t)ccur * 128u + csw);
      if (lane_on && !(exp_flags & 1)) {
        if (!full) {
          // hot path per pass: LDS.64, one 32x32+64 multiply-add (source address), LOP3 (destination), LDGSTS
          for (int p0 = 0; p0 < npass; p0 += 4) {        // up to 4 list entries are read before their copies are issued
            int2 e[4];
#pragma unroll
            for (int u = 0; u < 4; ++u)
              if (p0 + u < npass) e[u] = list[(p0 + u) * IPP + isub];
#pragma unroll
            for (int u = 0; u < 4; ++u)
              if (p0 + u < npass) cp_async16((uint32_t)e[u].y ^ csw, mad_wide16((uint32_t)e[u].x, src0), 16u);
          }
        } else {
          // first stage of a tile: every row is written, missing neighbours as zeros (src-size 0 reads nothing)
#pragma unroll
          for (int pass = 0; pass < 8; ++pass) {
            const int2 e = list[pass * IPP + isub];
            const bool live = e.x != -1;
            cp_async16((uint32_t)e.y ^ csw, mad_wide16(live ? (uint32_t)e.x : 0u, src0), live ? 16u : 0u);
          }
        }
      }
      // Landing is signalled by the copies themselves: every lane's arrival on afull(slot) fires when its cp.async
      // have completed.  Lane 0's ordinary arrival (release) publishes the mask words it stored above.
      cp_async_arrive_noinc(afull(slot));
      if (lane == 0) mbar_arrive(afull(slot));
      if (wq == 0) mark(grp, it, 3);
      ++it;
      ls += gpc;
      if (ls >= spc) { ls -= spc; ++round; }
    };

    // Indices are fetched two stages ahead.  (Two stages per loop iteration, so that the register hand-over below never
    // waits for a load in flight, was measured and is slower: 76 -> 89 us at 495 k rows x 32 channels.)
    int jlA, jhA, qA, jlB, jhB, qB;
    fetch(jlA, jhA, qA);
    fetch(jlB, jhB, qB);
    while (qA >= 0) {
      int jlC, jhC, qC;
      fetch(jlC, jhC, qC);
      do_stage(jlA, jhA, qA);
      jlA = jlB; jhA = jhB; qA = qB;
      jlB = jlC; jhB = jhC; qB = qC;
    }
  } else if (warp == WARP_BLOAD) {
    // ================================ weight-tile loader (1 elected lane, bulk async copies) ==
    // The tiles (n_out x 128 B each, already in the swizzled shared-memory image) stream from L2 in stage order; the
    // copy engine signals bfull itself (complete_tx), so landing needs no warp and no proxy fence.
    const int total_b = my_groups * Q;
    int bslot = 0;
    uint32_t bround = 0;
    for (int i = 0; i < total_b; ++i) {
      mark(8, i, 0);
      if (ksplit) mbar_wait_sleep(bempty(bslot), (bround & 1u) ^ 1u, 100u);
      else mbar_wait(bempty(bslot), (bround & 1u) ^ 1u);
      mark(8, i, 1);
      if (elect_one()) {
        mbar_expect_tx(bfull(bslot), b_bytes);
        bulk_g2s(b_base + (uint32_t)bslot * b_bytes, p.bimg + (size_t)(i % Q) * b_bytes, b_bytes, bfull(bslot));
      }
      __syncwarp();
      if (++bslot == SB) { bslot = 0; ++bround; }
    }
  } else if (warp >= WARP_MMA && warp < WARP_MMA + MMA_WARPS) {
    // ================================ MMA issuers (warp-uniform loops, 1 elected lane issues) =
    // The per-stage issue path (two mbarrier waits, mask fetch, 4 UTCHMMA, commit) costs one warp several hundred
    // cycles, more than the tensor pipe needs for the stage, so the T tiles of a group (independent accumulators)
    // are dealt to NM = 1, 2 or 4 issuing warps (classes): warp m issues tiles m, m + NM, ...
    const int m = warp - WARP_MMA;                                    // == class
    if (m < NM) {
      const uint32_t idesc = make_idesc<TF32>(p.n_out);
      const uint64_t da0 = make_desc_sw128(a_base), db0 = make_desc_sw128(b_base);
      const int nbuf = p.nbuf;
      int bslot = 0;
      uint32_t bround = 0;
      int ls = 0;                                                     // this class's next stage: slot m * spc + ls ...
      uint32_t around = 0;                                            // ... in round `around` of that slot
      int it = 0;
      // one stage: wait for its four quarters (and their masks), issue its MMAs into columns `col`, free the A slot
      auto issue_stage = [&](int q, uint32_t col, uint64_t db, bool first) {
        const int cc = PAIR ? 0 : q % nch;
        const int step = PAIR ? q : q / nch;
        // MMAs of 32 bytes of K each.  PAIR with an odd K: the last stage holds one offset only, its upper 32 channels
        // are never written
        const int nk = PAIR ? ((2 * step + 1 < p.K) ? 4 : 2) : ((cc == nch - 1 ? p.last_kc : KCE) * ESZ / 32);
        const int aslot = m * spc + ls;
        mark(4 + m, it, 0);
        mbar_wait(afull(aslot), around & 1u);                // all four quarters of the stage have landed (and their masks)
        mark(4 + m, it, 1);
        tc_fence_after();
        // disable-output-lane masks published by the stage's producers: bit r set <=> output row r has no
        // neighbour at this offset (its A row is stale).  Every lane loads the same words; the ballots make
        // them provably warp-uniform so they are moved to uniform registers once.
        uint32_t m0 = 0, m1 = 0, m2 = 0, m3 = 0, h0 = 0, h1 = 0, h2 = 0, h3 = 0;
        if (!first) {
          const uint4 mw = *reinterpret_cast<const uint4*>(amask + aslot * 8);
          m0 = __ballot_sync(0xffffffffu, (mw.x >> lane) & 1u);
          m1 = __ballot_sync(0xffffffffu, (mw.y >> lane) & 1u);
          m2 = __ballot_sync(0xffffffffu, (mw.z >> lane) & 1u);
          m3 = __ballot_sync(0xffffffffu, (mw.w >> lane) & 1u);
          if (PAIR) {
            const uint4 hw = *reinterpret_cast<const uint4*>(amask + aslot * 8 + 4);
            h0 = __ballot_sync(0xffffffffu, (hw.x >> lane) & 1u);
            h1 = __ballot_sync(0xffffffffu, (hw.y >> lane) & 1u);
            h2 = __ballot_sync(0xffffffffu, (hw.z >> lane) & 1u);
            h3 = __ballot_sync(0xffffffffu, (hw.w >> lane) & 1u);
          }
        }
        const uint64_t da = da0 + (uint64_t)((uint32_t)aslot * (A_BYTES >> 4));
        const uint32_t tmem_d = tmem_base + col;
        if (elect_one()) {
#pragma unroll
          for (int kk = 0; kk < 4; ++kk) {
            if (kk < nk && !(exp_flags & 2)) {
              const bool hi = PAIR && kk >= 2;
              umma_masked<TF32>(tmem_d, da + (uint64_t)(kk * 2), db + (uint64_t)(kk * 2), idesc, (!first || kk > 0) ? 1u : 0u,
                                hi ? h0 : m0, hi ? h1 : m1, hi ? h2 : m2, hi ? h3 : m3);
            }
          }
          umma_commit(aempty(aslot));                                  // frees the A slot when these MMAs retire
        }
        __syncwarp();
        mark(4 + m, it, 2);
        ++it;
        if (++ls == spc) { ls = 0; ++around; }
      };
      if (ksplit) {
        // one tile, one group: this warp issues the stages q = m, m + 2, ... into its own accumulator (columns m * n_out);
        // a weight tile is consumed by one class only (SB is even: a B slot always belongs to the same class)
        mbar_wait(acce(0), 1u);
        tc_fence_after();
        bslot = m;
        for (int q = m; q < Q; q += 2) {
          mbar_wait(bfull(bslot), bround & 1u);
          issue_stage(q, (uint32_t)(m * p.n_out), db0 + (uint64_t)(((uint32_t)bslot * b_bytes) >> 4), q < 2);
          if (elect_one()) umma_commit(bempty(bslot));
          __syncwarp();
          bslot += 2;
          if (bslot >= SB) { bslot -= SB; ++bround; }
        }
        if (elect_one()) umma_commit(accf(0));
        __syncwarp();
      } else
      for (int g = 0; g < my_groups; ++g) {
        const int buf = nbuf == 2 ? (g & 1) : 0;
        const uint32_t use = (uint32_t)(nbuf == 2 ? (g >> 1) : g);    // how many times this buffer has been used before
        const int tv = tiles_in_group(g);
        mbar_wait(acce(buf), (use & 1u) ^ 1u);                        // epilogue has drained this accumulator buffer
        tc_fence_after();
        for (int q = 0; q < Q; ++q) {
          mark(10 + m, g * Q + q, 0);
          mbar_wait(bfull(bslot), bround & 1u);
          mark(10 + m, g * Q + q, 1);
          const uint64_t db = db0 + (uint64_t)(((uint32_t)bslot * b_bytes) >> 4);
          for (int t = m; t < tv; t += NM) issue_stage(q, (uint32_t)buf * 256u + (uint32_t)(t * p.n_out), db, q == 0);
          if (elect_one()) umma_commit(bempty(bslot));
          __syncwarp();
          if (++bslot == SB) { bslot = 0; ++bround; }
        }
        if (elect_one()) umma_commit(accf(buf));                       // this warp's accumulators of the group are complete
        __syncwarp();
      }
    }
  } else if (warp < EPI_WARPS) {
    // ================================ epilogue (warps 0..3) ==================================
    if (ksplit) {
      // one tile whose two partial accumulators (columns 0.. and n_out..) are added on the way out
      mbar_wait_sleep(accf(0), 0u, 100u);                  // one tile per CTA: the epilogue is on the critical path
      tc_fence_after();
      const int64_t row = (int64_t)tile_lo * BM + warp * 32 + lane;
      const uint32_t taddr = tmem_base + ((uint32_t)(warp * 32) << 16);
      for (int c0 = 0; c0 < p.n_out; c0 += 16) {
        uint32_t a[16], b[16];
        tmem_ld16x2(taddr + (uint32_t)c0, taddr + (uint32_t)(p.n_out + c0), a, b);
        if (row < p.n_rows && !(exp_flags & 4)) {
#pragma unroll
          for (int gq = 0; gq < 2; ++gq) {
            float f[8];
#pragma unroll
            for (int e = 0; e < 8; ++e)
              f[e] = __uint_as_float(a[gq * 8 + e]) + __uint_as_float(b[gq * 8 + e]) +
                     (p.bias ? __ldg(p.bias + c0 + gq * 8 + e) : 0.f);
            store8<TF32>(p.out, row * p.n_out + c0 + gq * 8, f);
          }
        }
      }
      tc_fence_before();
    } else
    for (int g = 0; g < my_groups; ++g) {
      const int buf = p.nbuf == 2 ? (g & 1) : 0;
      if (warp == 0) mark(9, g, 0);
      mbar_wait_long(accf(buf), (uint32_t)(p.nbuf == 2 ? (g >> 1) : g) & 1u);
      if (warp == 0) mark(9, g, 1);
      tc_fence_after();
      const int tv = tiles_in_group(g);
      for (int t = 0; t < tv; ++t) {
        const int64_t tile = (int64_t)tile_lo + (int64_t)g * T + t;
        const int64_t row = tile * BM + warp * 32 + lane;
        const uint32_t taddr = tmem_base + ((uint32_t)(warp * 32) << 16) + (uint32_t)buf * 256u + (uint32_t)(t * p.n_out);
        for (int c0 = 0; c0 < p.n_out; c0 += 32) {
          uint32_t v[32];
          tmem_ld32(taddr + (uint32_t)c0, v);
          if (row < p.n_rows && !(exp_flags & 4)) {
#pragma unroll
            for (int gq = 0; gq < 4; ++gq) {
              float f[8];
#pragma unroll
              for (int e = 0; e < 8; ++e)
                f[e] = __uint_as_float(v[gq * 8 + e]) + (p.bias ? __ldg(p.bias + c0 + gq * 8 + e) : 0.f);
              store8<TF32>(p.out, row * p.n_out + c0 + gq * 8, f);
            }
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (warp == 0) mark(9, g, 2);
      if (lane == 0) mbar_arrive(acce(buf));
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == WARP_MMA) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512) : "memory");
  }
}

// Weight image: one tile per stage q = k*nch + c/64: n_out rows of 128 bytes; the 16-byte chunk (c%64)/8 of row n
// is stored at chunk position chunk ^ (n & 7) (the SWIZZLE_128B pattern); unused half rows stay zero.
// tf32: q = k*nch + c/32, chunk (c%32)/4, values rounded to TF32 (cvt.rna) and stored as fp32 bits.
__global__ void k_prep_weights_tc(const float* __restrict__ W, int K, int Cin, int Cout, int transpose, int mirror,
                                  int nch, int pair, int tf32, void* __restrict__ img) {
  const int n_in = transpose ? Cout : Cin, n_out = transpose ? Cin : Cout;
  int64_t total = (int64_t)K * n_in * n_out;
  int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= total) return;
  int k = (int)(i / ((int64_t)n_in * n_out));
  int rem = (int)(i - (int64_t)k * n_in * n_out);
  int n = rem / n_in, c = rem % n_in;
  int src_k = (transpose && mirror) ? K - 1 - k : k;
  int ci = transpose ? n : c, co = transpose ? c : n;
  float v = W[((int64_t)src_k * Cin + ci) * Cout + co];
  if (tf32) {
    const int q = k * nch + c / KC_TF32, chunk = (c % KC_TF32) >> 2;
    reinterpret_cast<float*>(img)[((size_t)q * n_out + n) * 32 + (size_t)((chunk ^ (n & 7)) << 2) + (c & 3)] = to_tf32_rna(v);
    return;
  }
  // pair (n_in == 32): stage q = k/2, chunks 0-3 <- offset 2q, chunks 4-7 <- offset 2q+1
  const int q = pair ? (k >> 1) : k * nch + c / KC;
  const int chunk = pair ? (k & 1) * 4 + (c >> 3) : (c % KC) >> 3;
  size_t off = ((size_t)q * n_out + n) * 64 + (size_t)((chunk ^ (n & 7)) << 3) + (c & 7);
  reinterpret_cast<__nv_bfloat16*>(img)[off] = __float2bfloat16_rn(v);
}

// All weight images of a network in ONE launch (the trainer calls it once per step instead of 112 per-module launches):
// descs = n x 8 int64 {W, img, K, Cin, Cout, transpose | mirror << 1, first element index, precision}; element i of the
// concatenated index space belongs to the descriptor d with first[d] <= i < first[d + 1].  A thread builds ONE 16-byte
// chunk of an image (8 consecutive input channels of one output channel): units of a descriptor are numbered
// (offset, 8-channel block, output channel) with the output channel fastest, so that the forward image's strided reads
// of W[k][c][n] are coalesced over n and the transposed image reads 32 contiguous bytes per thread.  (One thread per
// ELEMENT with 2-byte scattered stores took 360 us per step for the 41 M elements of the default network.)
__global__ void __launch_bounds__(256) k_prep_weights_tc_batched(const long long* __restrict__ descs, int n, long long units) {
  pdl_launch_dependents();
  pdl_wait();
  const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i >= units) return;
  const long long e = i * 8;
  int lo = 0, hi = n - 1;
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (__ldg(descs + mid * 8 + 6) <= e) lo = mid; else hi = mid - 1;
  }
  const long long* d = descs + lo * 8;
  const float* W = reinterpret_cast<const float*>(d[0]);
  unsigned char* img = reinterpret_cast<unsigned char*>(d[1]);
  const int K = (int)d[2], Cin = (int)d[3], Cout = (int)d[4], transpose = (int)(d[5] & 1), mirror = (int)((d[5] >> 1) & 1);
  const int n_in = transpose ? Cout : Cin, n_out = transpose ? Cin : Cout;
  const bool tf32 = d[7] == SCN_PREC_TF32;
  const int kc = tf32 ? KC_TF32 : KC;
  const int nch = (n_in + kc - 1) / kc, pair = !tf32 && n_in == 32;
  const int u = (int)((e - d[6]) >> 3);               // unit within the descriptor
  const int per_k = (n_in >> 3) * n_out;
  const int k = u / per_k;
  const int r = u - k * per_k;
  const int cb = r / n_out, nn = r - cb * n_out;      // 8-channel block, output channel
  const int c0 = cb * 8;
  const int src_k = (transpose && mirror) ? K - 1 - k : k;
  float v[8];
  if (transpose) {                                    // W[src_k][ci = nn][co = c0 .. c0 + 7]: contiguous
    const float4* src = reinterpret_cast<const float4*>(W + ((long long)src_k * Cin + nn) * Cout + c0);
    const float4 a = __ldg(src), b = __ldg(src + 1);
    v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
  } else {                                            // W[k][ci = c0 .. c0 + 7][co = nn]: stride Cout, coalesced over nn
    const float* src = W + ((long long)src_k * Cin + c0) * Cout + nn;
#pragma unroll
    for (int j = 0; j < 8; ++j) v[j] = __ldg(src + (long long)j * Cout);
  }
  if (tf32) {                                         // the 8 channels are 16-byte chunks c, c + 1 (4 fp32 each)
    const int q = k * nch + c0 / KC_TF32, chunk = (c0 % KC_TF32) >> 2;
    unsigned char* row = img + ((size_t)q * n_out + nn) * 128;
    *reinterpret_cast<float4*>(row + ((chunk ^ (nn & 7)) << 4)) =
        make_float4(to_tf32_rna(v[0]), to_tf32_rna(v[1]), to_tf32_rna(v[2]), to_tf32_rna(v[3]));
    *reinterpret_cast<float4*>(row + (((chunk + 1) ^ (nn & 7)) << 4)) =
        make_float4(to_tf32_rna(v[4]), to_tf32_rna(v[5]), to_tf32_rna(v[6]), to_tf32_rna(v[7]));
    return;
  }
  // pair (n_in == 32): stage q = k/2, chunks 0-3 <- offset 2q, chunks 4-7 <- offset 2q+1
  const int q = pair ? (k >> 1) : k * nch + c0 / KC;
  const int chunk = pair ? (k & 1) * 4 + cb : (c0 % KC) >> 3;
  uint4 o;
  o.x = pack_bf16x2(v[0], v[1]); o.y = pack_bf16x2(v[2], v[3]);
  o.z = pack_bf16x2(v[4], v[5]); o.w = pack_bf16x2(v[6], v[7]);
  *reinterpret_cast<uint4*>(img + ((size_t)q * n_out + nn) * 128 + (size_t)((chunk ^ (nn & 7)) << 4)) = o;
}

}  // namespace tc

// descs: device array of n x 8 int64 (see k_prep_weights_tc_batched); images whose n_in is not a multiple of 64 must
// have been zero-filled once by the caller (their unused half rows are never written).  tcgen05-path images only.
extern "C" int scn_conv_prep_weights_batched(const void* descs, int n, int64_t total, void* stream) {
  if (n <= 0 || total <= 0) return SCN_OK;
  if (!descs) return SCN_ERR_ARG;
  SCN_CUDA(scn_launch_pdl(tc::k_prep_weights_tc_batched, dim3(grid_for(total / 8, 256)), dim3(256), 0, (cudaStream_t)stream,
                          (const long long*)descs, n, (long long)(total / 8)));
  SCN_LAUNCH_CHECK();
  return SCN_OK;
}

// Debug: device buffer of 4 roles x 256 stages x 8 marks (uint64) filled by CTA 0 of the following launches; NULL disables.
static unsigned long long* g_tc_dbg = nullptr;
extern "C" void scn_tc_debug_timeline(void* device_buffer) { g_tc_dbg = (unsigned long long*)device_buffer; }
// timing experiments (WRONG results; honoured only by -DSCN_TC_TIMELINE builds): 1 no gather copies, 2 no MMAs, 4 no stores
#ifdef SCN_TC_TIMELINE
static int g_tc_exp = 0;
extern "C" void scn_tc_debug_exp(int flags) { g_tc_exp = flags; }
#else
extern "C" void scn_tc_debug_exp(int) {}
#endif

bool scn_tc_shape_ok(int K, int n_in, int n_out) {
  return K >= 1 && (n_in % 32) == 0 && (n_out % 32) == 0 && n_in >= 32 && n_in <= 256 && n_out >= 32 && n_out <= 256;
}

// bf16, n_in == 32: two offsets share a 64-channel stage
static bool tc_pair(int n_in, int tf32) { return !tf32 && n_in == 32; }
// channel chunks (stages) per offset: 64 bf16 or 32 fp32 channels each
static int tc_nch(int n_in, int tf32) {
  const int kc = tf32 ? tc::KC_TF32 : tc::KC;
  return (n_in + kc - 1) / kc;
}

size_t scn_tc_image_bytes(int K, int n_in, int n_out, int tf32) {
  const size_t stages = tc_pair(n_in, tf32) ? (size_t)(K + 1) / 2 : (size_t)K * tc_nch(n_in, tf32);
  return stages * n_out * 128;
}

int scn_tc_prep(const float* W, int K, int Cin, int Cout, int transpose, int mirror, int tf32, void* out, cudaStream_t s) {
  const int n_in = transpose ? Cout : Cin, n_out = transpose ? Cin : Cout;
  const int nch = tc_nch(n_in, tf32);
  if (!tf32 && (n_in % tc::KC) != 0) SCN_CUDA(cudaMemsetAsync(out, 0, scn_tc_image_bytes(K, n_in, n_out, tf32), s));
  int64_t total = (int64_t)K * Cin * Cout;
  tc::k_prep_weights_tc<<<grid_for(total, 256), 256, 0, s>>>(W, K, Cin, Cout, transpose, mirror, nch,
                                                             tc_pair(n_in, tf32) ? 1 : 0, tf32, out);
  SCN_LAUNCH_CHECK();
  return SCN_OK;
}

// developer knobs for sweeps: a cap on the CTAs, forced tiles per group, forced A / B ring depths; 0 = automatic
static int g_knob[4] = {0, 0, 0, 0};          // grid, T, SA, SB
// developer entry for the sweep tools (like scn_tc_debug_timeline: not part of the product ABI)
extern "C" void scn_tc_debug_knobs(int grid, int t, int sa, int sb) {
  g_knob[0] = grid; g_knob[1] = t; g_knob[2] = sa; g_knob[3] = sb;
}
// the configuration of the last k_conv_tc launch (developer entry like the knobs, for the tests' coverage check):
// grid, T, NM, nbuf, ksplit, SA, SB, min and max tiles per CTA; written on the host just before the launch
static int32_t g_last_launch[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
extern "C" void scn_tc_debug_last_launch(int32_t* out) {
  for (int i = 0; i < 9; ++i) out[i] = g_last_launch[i];
}

// in / out: bf16, or fp32 with tf32 != 0 (TF32 MMAs)
int scn_tc_forward(const void* in, int64_t n_in_rows, const int32_t* nbr, int K, int64_t n_rows, int64_t n_pad, int n_in,
                   int n_out, const void* bimg, const float* bias, void* out, int tf32, cudaStream_t s) {
  const uint64_t row_units = (uint64_t)n_in * (tf32 ? 4u : 2u) / 16u;                // 16-byte units per input row
  if ((uint64_t)n_in_rows * row_units >= 0xffffffffull) return SCN_ERR_UNSUPPORTED;   // 32-bit offsets in 16-byte units (64 GB)
  const int force_grid = g_knob[0], force_t = g_knob[1], force_sa = g_knob[2], force_sb = g_knob[3];
  tc::Params p;
  p.dbg = g_tc_dbg;
#ifdef SCN_TC_TIMELINE
  p.exp = g_tc_exp;
#else
  p.exp = 0;
#endif
  p.in = in; p.nbr = nbr; p.bimg = (const unsigned char*)bimg; p.bias = bias; p.out = out;
  p.n_rows = n_rows; p.n_pad = n_pad; p.K = K; p.n_in = n_in; p.n_out = n_out;
  const bool pair = tc_pair(n_in, tf32);
  const int nch = tc_nch(n_in, tf32);
  p.nch = nch;
  p.last_kc = n_in - (nch - 1) * (tf32 ? tc::KC_TF32 : tc::KC);
  p.num_tiles = (int)((n_rows + tc::BM - 1) / tc::BM);
  // Tiles per group.  A group's T tiles are dealt to NM = 1, 2 or 4 classes (one issuing warp + producer group each) and
  // every class walks its tiles' stages as ONE serial chain (~1400 cycles per stage), so a CTA's time is, in units of
  // one tile's chain,   sum over its groups of ceil(tiles of the group / NM)   -- T = 5 on 4 classes costs 2 units per
  // group, like T = 8 -- plus the epilogue of every group where it is not overlapped (one group in all 512 TMEM columns
  // instead of two alternating halves).  T is the candidate that minimises that estimate for the CTA with the most
  // tiles; ties go to the larger T (fewer passes over the weight image).  Measured, 96 channels: 138 k rows (8 tiles per
  // CTA) T = 5 -> 4: 108 -> 84 us; 155 k rows (9 tiles per CTA): T = 5 stays, 111 us.
  int max_ctas = kNumSMs;
  if (force_grid > 0 && force_grid < max_ctas) max_ctas = force_grid;
  const int per_cta = (p.num_tiles + max_ctas - 1) / max_ctas;
  const int q_per_tile = (pair ? (K + 1) / 2 : K) * nch;
  int T = 1;
  p.nbuf = 2;
  {
    double best = 1e30;
    for (int t = 1; t <= 8 && t * n_out <= 512 && t <= (per_cta > 0 ? per_cta : 1); ++t) {
      const int nm = t >= 4 ? 4 : (t >= 2 ? 2 : 1);
      const int full = per_cta / t, rem = per_cta % t;
      const int groups = full + (rem ? 1 : 0);
      const double units = (double)full * ((t + nm - 1) / nm) + (rem ? (rem + nm - 1) / nm : 0);
      const int nbuf = t * n_out <= 256 ? 2 : 1;
      // epilogue of a group (~600 cycles per tile and 32 output columns) relative to a tile's chain; hidden behind the
      // next group's main loop when double-buffered, except for the last group
      const double ep = (double)t * (n_out / 32.0) * 600.0 / ((double)q_per_tile * 1400.0);
      const double cost = units + (nbuf == 1 ? groups * ep : ep + 0.15 * (groups - 1) * ep);
      if (cost <= best + 1e-9) { best = cost; T = t; p.nbuf = nbuf; }
    }
  }
  if (force_t > 0) {
    T = force_t;
    if (T > 8) T = 8;
    if (T * n_out > 512) T = 512 / n_out;
    if (T > per_cta) T = per_cta;
    if (T < 1) T = 1;
    p.nbuf = T * n_out <= 256 ? 2 : 1;
  }
  p.T = T;
  p.NM = T >= 4 ? 4 : (T >= 2 ? 2 : 1);         // classes (issuing warps): a power of two that divides NGRP
  // K-split (see the kernel): CTAs that own a single tile deal its stages to two classes.  Possible when a launch has two
  // classes anyway (T == 2 or 3: the deep levels with one or two tiles per CTA) or one tile per CTA and room for a second
  // accumulator.
  p.ksplit = 0;
  const int stages_per_tile = (pair ? (K + 1) / 2 : K) * nch;
  if (stages_per_tile >= 2) {          // both accumulators must receive a first stage
    if (p.NM == 1 && per_cta == 1 && 2 * n_out <= 512) { p.NM = 2; p.nbuf = 1; p.ksplit = 1; }
    else if (p.NM == 2) p.ksplit = 1;
  }
  const uint32_t b_bytes = (uint32_t)n_out * 128u;
  constexpr int NBAR = 2 * tc::MAX_A + 2 * tc::MAX_B + 4;
  const uint32_t fixed = 1024u + 8u * NBAR + 16u + (uint32_t)tc::MAX_A * tc::MASK_BYTES +
                         2u * (uint32_t)tc::PROD_WARPS * tc::LIST_BYTES + 16u;
  const uint32_t budget = 226u * 1024u - fixed;
  // A ring: a multiple of NGRP slots (every class ring then is a multiple of its producer groups: parity-safe), 8 by
  // default (measured: depth beyond 6 buys nothing); the weight ring gets the rest, up to MAX_B tiles
  int SA = 8;
  // K-split launches (one or two tiles per CTA, wide layers): the weight tiles (n_out x 128 B per stage, consumed by one
  // class each) need the depth, the A ring does not (measured: 4 slots == 8 slots at these shapes)
  if (p.ksplit && per_cta <= 2) SA = 4;
  if (force_sa > 0) SA = force_sa;
  SA = SA / tc::NGRP * tc::NGRP;
  if (SA > tc::MAX_A) SA = tc::MAX_A;
  if (SA < tc::NGRP) SA = tc::NGRP;
  while (SA > tc::NGRP && (uint32_t)SA * tc::A_BYTES + 2u * b_bytes > budget) SA -= tc::NGRP;
  if ((uint32_t)SA * tc::A_BYTES + 2u * b_bytes > budget) return SCN_ERR_UNSUPPORTED;
  int SB = (int)((budget - (uint32_t)SA * tc::A_BYTES) / b_bytes);
  if (SB > tc::MAX_B) SB = tc::MAX_B;
  if (force_sb >= 2 && force_sb < SB) SB = force_sb;
  if (p.ksplit && (SB & 1)) --SB;                // K-split: a B slot must always belong to the same class
  p.SA = SA;
  p.SB = SB;
  const size_t smem = (size_t)fixed + (size_t)SA * tc::A_BYTES + (size_t)SB * b_bytes;
  int grid = p.num_tiles < max_ctas ? p.num_tiles : max_ctas;
  {
    static bool attr_set = false;          // opt in to > 48 KB of dynamic shared memory, once per kernel
    if (!attr_set) {
      SCN_CUDA(cudaFuncSetAttribute(tc::k_conv_tc<1, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
      SCN_CUDA(cudaFuncSetAttribute(tc::k_conv_tc<1, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
      SCN_CUDA(cudaFuncSetAttribute(tc::k_conv_tc<2, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
      SCN_CUDA(cudaFuncSetAttribute(tc::k_conv_tc<3, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
      SCN_CUDA(cudaFuncSetAttribute(tc::k_conv_tc<4, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
      SCN_CUDA(cudaFuncSetAttribute(tc::k_conv_tc<0, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
      attr_set = true;
    }
  }
  if (grid < 1) return SCN_OK;                   // no output row
  {
    const int32_t rec[9] = {grid, p.T, p.NM, p.nbuf, p.ksplit, p.SA, p.SB, p.num_tiles / grid,
                            (p.num_tiles + grid - 1) / grid};
    for (int i = 0; i < 9; ++i) g_last_launch[i] = rec[i];
  }
  auto launch = [&](auto kern) -> int {
    SCN_CUDA(scn_launch_pdl(kern, dim3((unsigned)grid), dim3(tc::THREADS), smem, s, p));
    SCN_LAUNCH_CHECK();
    return SCN_OK;
  };
  if (tf32) return nch <= 8 ? launch(tc::k_conv_tc<0, false, true>) : SCN_ERR_UNSUPPORTED;
  if (pair) return launch(tc::k_conv_tc<1, true>);
  switch (nch) {
    case 1: return launch(tc::k_conv_tc<1, false>);
    case 2: return launch(tc::k_conv_tc<2, false>);
    case 3: return launch(tc::k_conv_tc<3, false>);
    case 4: return launch(tc::k_conv_tc<4, false>);
    default: return SCN_ERR_UNSUPPORTED;
  }
}
