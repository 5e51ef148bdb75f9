// dp_kernels.cuh -- device code of the PEX verification path for sm_100a.
//
// One engine computes every alignment::align mode (src/lib/alignment.cpp:83-181 of the reference):
// a banded, bit-parallel (Myers/Hyyroe) semi-global edit-distance pass in which a RING of G lanes
// of one warp sweeps the DP matrix as a skewed wavefront.  Rows are cut into blocks of 32*W rows
// (W 32-bit words held in registers per lane); lane r of the ring owns blocks r, r+G, r+2G, ...;
// block b processes column j at step t = j + b, so the only cross-lane traffic is the two
// horizontal-delta bits (and the running score) of the block above, handed down with warp shuffles.
// A lane takes its next block as soon as its own has ended; the block below a block that has ended
// substitutes the "+1 per column" bound for the neighbour's deltas itself (run_steps: Upper), so a
// ring needs G >= 2 + (B - 3) / (32 W + 1) lanes for a band of B diagonals and no more.
// Only the cells inside the diagonal band [dlo, dhi] that can lie on an alignment with <= k errors
// are computed (a block is active for columns cs(b)..ce(b)); outside values are replaced by upper
// bounds (+1 steps), which keeps every value <= k exact.
//
// Not a dense contraction: no tensor cores.  The hot loop is LOP3 / IADD3(.X) / SHF on the integer
// pipes, Eq words and window characters come from shared memory, the carries from SHFL.
//
// Around the engine: walk2_kernel (traceback + CIGAR from the checkpoint records a root pass leaves),
// range_min_kernel (a window's result read off a pass over the union of several windows), the
// level_*_kernel family (the PEX tree walk's inner levels: windows, per-node election, engine tasks,
// survivors -- all on the device), build_peq_kernel / pack_nibbles_kernel (input encoding).
#pragma once

#include <cstdint>
#include <cuda_runtime.h>

namespace fxg {

constexpr int kNumSymbols = 6;          // ranks 0..5, include/input.hpp:63-66 of the reference
constexpr int kPeqFrontPadWords = 64;   // table words in front of position 0 (wildcard rows read there)
constexpr int kPeqBackPadWords = 66;
constexpr uint32_t kFlagReverse = 1u;   // run on reversed views (alignment.cpp:118-125)
constexpr uint32_t kFlagInlineRef = 2u; // window comes from the per-batch inline pool
constexpr int32_t kNoScore = 0x3fffffff;
constexpr int32_t kPoisonScore = 0x7ffffff0;   // the engine found its own bookkeeping inconsistent (host turns it into an error)
constexpr uint32_t kWinChunks = 8;      // 32-base chunks of the window a ring keeps in shared memory at a time
constexpr uint32_t kWinBytes = 2 * kWinChunks * 32;   // every chunk is stored twice (slot and slot + kWinChunks): reads never wrap

// One bit-vector DP pass.  All coordinates are in bases.
struct DpTask {
    uint64_t ref_base;     // position of window[0] in the packed reference store (or inline pool)
    uint64_t query_base;   // position of query[0] in the pool the Peq table was built from
    uint64_t trace_base;   // first 32-bit word of this task's trace planes (trace passes only)
    uint32_t n;            // window length
    uint32_t m;            // query length (>= 1)
    int32_t dlo, dhi;      // band of diagonals j - i (1-based DP coordinates) that is computed
    uint32_t flags;
    uint32_t out;          // result slot
};

struct DpResult {
    int32_t score;         // minimum of the last row inside the band (kNoScore if the last row was never reached)
    uint32_t end_col;      // rightmost column (1-based, == exclusive end) attaining it
};

// ---------------------------------------------------------------------------------------------
// Peq table: bit p of plane s is (pool[p] == s).  kPeqFrontPadWords zero words in front.
// ---------------------------------------------------------------------------------------------
__global__ void build_peq_kernel(const uint8_t* __restrict__ pool, uint64_t len, uint32_t* __restrict__ table,
                                 uint64_t plane_words, uint32_t* __restrict__ bad_rank_flag) {
    uint64_t const n_words = (len + 31) / 32;
    uint32_t const lane = threadIdx.x & 31;
    uint64_t const warp = (uint64_t(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
    uint64_t const n_warps = (uint64_t(gridDim.x) * blockDim.x) >> 5;
    bool bad = false;
    for (uint64_t w = warp; w < n_words; w += n_warps) {
        uint64_t const p = w * 32 + lane;
        uint32_t const c = p < len ? pool[p] : 0xffu;
        bad |= p < len && c >= uint32_t(kNumSymbols);       // such a byte matches no plane (harmless here); the host reports it
        uint32_t mine = 0;
#pragma unroll
        for (int s = 0; s < kNumSymbols; ++s) {
            uint32_t const bal = __ballot_sync(0xffffffffu, c == uint32_t(s));
            if (lane == uint32_t(s)) mine = bal;
        }
        if (lane < kNumSymbols) table[uint64_t(lane) * plane_words + kPeqFrontPadWords + w] = mine;
    }
    if (bad_rank_flag && __any_sync(0xffffffffu, bad) && lane == 0) atomicOr(bad_rank_flag, 1u);
}

// 32 bits of plane starting at (signed) bit position x
__device__ __forceinline__ uint32_t peq_window(const uint32_t* __restrict__ plane, int64_t x) {
    int64_t const X = x + int64_t(kPeqFrontPadWords) * 32;
    uint32_t const lo = plane[X >> 5], hi = plane[(X >> 5) + 1];
    return __funnelshift_r(lo, hi, uint32_t(X) & 31u);
}

// ---------------------------------------------------------------------------------------------
// reference store: 4 bits per base (ranks 0..15 exact), 32 bases per 16-byte chunk
// ---------------------------------------------------------------------------------------------
__global__ void pack_nibbles_kernel(const uint8_t* __restrict__ ranks, uint64_t len, uint32_t* __restrict__ packed) {
    uint64_t const n_words = (len + 7) / 8;
    for (uint64_t w = uint64_t(blockIdx.x) * blockDim.x + threadIdx.x; w < n_words; w += uint64_t(gridDim.x) * blockDim.x) {
        uint32_t x = 0;
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            uint64_t const p = w * 8 + i;
            uint32_t const c = p < len ? ranks[p] : 0u;
            x |= (c & 15u) << (4 * i);
        }
        packed[w] = x;
    }
}

__device__ __forceinline__ uint32_t packed_base(const uint32_t* __restrict__ packed, uint64_t p) {
    return (packed[p >> 3] >> (4 * (uint32_t(p) & 7u))) & 15u;
}

// 8 packed bases -> 8 bytes (two words, base order preserved)
__device__ __forceinline__ void unpack8(uint32_t x, uint32_t& lo, uint32_t& hi) {
    uint32_t const e = x & 0x0f0f0f0fu, o = (x >> 4) & 0x0f0f0f0fu;
    lo = __byte_perm(e, o, 0x5140);
    hi = __byte_perm(e, o, 0x7362);
}

// ---------------------------------------------------------------------------------------------
// the DP engine
// ---------------------------------------------------------------------------------------------
struct DpLaunch {
    const DpTask* tasks;        // sorted so that the tasks of one warp have similar step counts
    uint32_t n_tasks;
    uint32_t group;             // G: lanes per task (1..32); floor(32 / G) tasks per warp
    uint32_t win_stride;        // bytes of shared memory per task window buffer (kWinBytes)
    uint32_t peq_stride;        // words per symbol row of the per-task Eq table
    const uint32_t* ref_packed; // resident references
    const uint32_t* inline_packed;
    uint64_t ref_chunks, inline_chunks;   // 16-byte chunks that may be read from each store
    uint32_t two;               // the constant 2, kept opaque to the compiler (see run_steps)
    const uint32_t* peq_table;  // kNumSymbols planes
    uint64_t peq_plane_words;
    DpResult* results;
    uint32_t* trace;            // trace planes [step][ring lane][word][hp, vp]
    const uint32_t* n_tasks_dev;// if set: the number of tasks is read from here (tasks built on the device; the grid is
                                // sized for an upper bound and surplus CTAs leave at once)
    const uint32_t* class_active; // if set: the tasks of class `cls` begin at tasks + class_active[0] + .. + class_active[cls - 1]
    uint32_t cls;
};

// S = T + P + carry over CH consecutive words with the hardware carry chain (IADD3.X); one asm
// statement per chunk so that nothing can clobber CC in between.  cin: zero or anything else (= a carry); the return value is 0 or 1.
template <int CH, bool COUT> struct Chain;
template <bool COUT> struct Chain<1, COUT> {
    static __device__ __forceinline__ uint32_t run(uint32_t* S, const uint32_t* T, const uint32_t* P, uint32_t cin) {
        uint32_t d, co = 0;
        if (COUT) asm("add.cc.u32 %0, %3, 0xffffffff; addc.cc.u32 %1, %4, %5; addc.u32 %2, 0, 0;"
                      : "=&r"(d), "=&r"(S[0]), "=&r"(co) : "r"(cin), "r"(T[0]), "r"(P[0]));
        else asm("add.cc.u32 %0, %2, 0xffffffff; addc.u32 %1, %3, %4;" : "=&r"(d), "=&r"(S[0]) : "r"(cin), "r"(T[0]), "r"(P[0]));
        return co;
    }
};
template <bool COUT> struct Chain<2, COUT> {
    static __device__ __forceinline__ uint32_t run(uint32_t* S, const uint32_t* T, const uint32_t* P, uint32_t cin) {
        uint32_t d, co = 0;
        if (COUT) asm("add.cc.u32 %0, %4, 0xffffffff; addc.cc.u32 %1, %5, %7; addc.cc.u32 %2, %6, %8; addc.u32 %3, 0, 0;"
                      : "=&r"(d), "=&r"(S[0]), "=&r"(S[1]), "=&r"(co) : "r"(cin), "r"(T[0]), "r"(T[1]), "r"(P[0]), "r"(P[1]));
        else asm("add.cc.u32 %0, %3, 0xffffffff; addc.cc.u32 %1, %4, %6; addc.u32 %2, %5, %7;"
                 : "=&r"(d), "=&r"(S[0]), "=&r"(S[1]) : "r"(cin), "r"(T[0]), "r"(T[1]), "r"(P[0]), "r"(P[1]));
        return co;
    }
};
template <bool COUT> struct Chain<4, COUT> {
    static __device__ __forceinline__ uint32_t run(uint32_t* S, const uint32_t* T, const uint32_t* P, uint32_t cin) {
        uint32_t d, co = 0;
        if (COUT) asm("add.cc.u32 %0, %6, 0xffffffff; addc.cc.u32 %1, %7, %11; addc.cc.u32 %2, %8, %12; addc.cc.u32 %3, %9, %13; "
                      "addc.cc.u32 %4, %10, %14; addc.u32 %5, 0, 0;"
                      : "=&r"(d), "=&r"(S[0]), "=&r"(S[1]), "=&r"(S[2]), "=&r"(S[3]), "=&r"(co)
                      : "r"(cin), "r"(T[0]), "r"(T[1]), "r"(T[2]), "r"(T[3]), "r"(P[0]), "r"(P[1]), "r"(P[2]), "r"(P[3]));
        else asm("add.cc.u32 %0, %5, 0xffffffff; addc.cc.u32 %1, %6, %10; addc.cc.u32 %2, %7, %11; addc.cc.u32 %3, %8, %12; "
                 "addc.u32 %4, %9, %13;"
                 : "=&r"(d), "=&r"(S[0]), "=&r"(S[1]), "=&r"(S[2]), "=&r"(S[3])
                 : "r"(cin), "r"(T[0]), "r"(T[1]), "r"(T[2]), "r"(T[3]), "r"(P[0]), "r"(P[1]), "r"(P[2]), "r"(P[3]));
        return co;
    }
};
template <bool COUT> struct Chain<8, COUT> {
    static __device__ __forceinline__ uint32_t run(uint32_t* S, const uint32_t* T, const uint32_t* P, uint32_t cin) {
        uint32_t d, co = 0;
        if (COUT) asm("add.cc.u32 %0, %10, 0xffffffff; addc.cc.u32 %1, %11, %19; addc.cc.u32 %2, %12, %20; addc.cc.u32 %3, %13, %21; "
                      "addc.cc.u32 %4, %14, %22; addc.cc.u32 %5, %15, %23; addc.cc.u32 %6, %16, %24; addc.cc.u32 %7, %17, %25; "
                      "addc.cc.u32 %8, %18, %26; addc.u32 %9, 0, 0;"
                      : "=&r"(d), "=&r"(S[0]), "=&r"(S[1]), "=&r"(S[2]), "=&r"(S[3]), "=&r"(S[4]), "=&r"(S[5]), "=&r"(S[6]), "=&r"(S[7]), "=&r"(co)
                      : "r"(cin), "r"(T[0]), "r"(T[1]), "r"(T[2]), "r"(T[3]), "r"(T[4]), "r"(T[5]), "r"(T[6]), "r"(T[7]),
                        "r"(P[0]), "r"(P[1]), "r"(P[2]), "r"(P[3]), "r"(P[4]), "r"(P[5]), "r"(P[6]), "r"(P[7]));
        else asm("add.cc.u32 %0, %9, 0xffffffff; addc.cc.u32 %1, %10, %18; addc.cc.u32 %2, %11, %19; addc.cc.u32 %3, %12, %20; "
                 "addc.cc.u32 %4, %13, %21; addc.cc.u32 %5, %14, %22; addc.cc.u32 %6, %15, %23; addc.cc.u32 %7, %16, %24; "
                 "addc.u32 %8, %17, %25;"
                 : "=&r"(d), "=&r"(S[0]), "=&r"(S[1]), "=&r"(S[2]), "=&r"(S[3]), "=&r"(S[4]), "=&r"(S[5]), "=&r"(S[6]), "=&r"(S[7])
                 : "r"(cin), "r"(T[0]), "r"(T[1]), "r"(T[2]), "r"(T[3]), "r"(T[4]), "r"(T[5]), "r"(T[6]), "r"(T[7]),
                   "r"(P[0]), "r"(P[1]), "r"(P[2]), "r"(P[3]), "r"(P[4]), "r"(P[5]), "r"(P[6]), "r"(P[7]));
        return co;
    }
};

// Per-lane state of the ring.  Everything lives in registers (all loops over W are unrolled).
template <int W>
struct LaneState {
    uint32_t Pv[W], Mv[W];      // vertical +1 / -1 deltas of the W words of the current block
    uint32_t b;                 // current block
    int32_t cs, ce;             // its active column range (cs > ce: none)
    uint32_t o_hp, o_hn;        // HP / HN of the block's last word after the latest step (bit 31 = bottom row)
    int32_t score;              // value of the block's bottom row after the latest step
    int32_t best;               // last block only: minimum of the last row so far ...
    uint32_t best_col;          // ... and the rightmost column attaining it
    const uint32_t* eqb;        // Eq rows of the current block: symbol s at eqb + s * W
    // checkpoint passes only: the horizontal deltas of the block's bottom row, one bit per step (latest step in bit 0),
    // and where the block's next checkpoint record goes
    uint32_t acc_hp, acc_hn;
    uint32_t* ckp;
};

// ---- checkpoints (root alignments whose CIGAR is wanted) ----
// Instead of trace planes for every cell, the score pass leaves just enough behind for the traceback to recompute any
// (block x 32 steps) tile of the matrix exactly: every 32 steps each working block writes one record
//   [ Pv[W] | Mv[W] | HP bits | HN bits | 0 | 0 ]   (ck_record_words(W) words)
// -- its vertical deltas after step t = 32 q (block b is at column t - b then), and the horizontal deltas of its bottom
// row for the steps 32 (q - 1) + 1 .. 32 q (bit p = step 32 (q - 1) + 1 + p), which are the upper boundary of the block
// below.  A block's records follow each other, the first one being q_first = ceil(first step / 32); a block that ends
// between two multiples of 32 adds a last record with the remaining boundary bits.
constexpr uint32_t kCkExtra = 4;
__host__ __device__ constexpr uint32_t ck_record_words(uint32_t W) { return W == 1 ? 8u : 2 * W + kCkExtra; }   // a multiple of 16 bytes
// records reserved per block: a block works for at most (band width + rows) steps
__host__ __device__ inline uint32_t ck_records_per_block(int64_t band_width, uint32_t rows) { return uint32_t((band_width + rows) / 32 + 3); }

// shared-memory loads by 32-bit shared-space address (keeps the address arithmetic in one register and off the ALU pipe)
__device__ __forceinline__ uint32_t lds_u8(uint32_t addr) {
    uint32_t v;
    asm volatile("ld.shared.u8 %0, [%1];" : "=r"(v) : "r"(addr));
    return v;
}
template <int W>
__device__ __forceinline__ void load_eq(uint32_t (&Eq)[W], uint32_t addr) {
    if constexpr (W % 4 == 0) {
#pragma unroll
        for (int i = 0; i < W; i += 4)
            asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(Eq[i]), "=r"(Eq[i + 1]), "=r"(Eq[i + 2]), "=r"(Eq[i + 3]) : "r"(addr + 4 * i));
    } else if constexpr (W == 2) {
        asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(Eq[0]), "=r"(Eq[1]) : "r"(addr));
    } else {
#pragma unroll
        for (int i = 0; i < W; ++i) asm volatile("ld.shared.u32 %0, [%1];" : "=r"(Eq[i]) : "r"(addr + 4 * i));
    }
}
template <int LUT>
__device__ __forceinline__ uint32_t lop3(uint32_t a, uint32_t b, uint32_t c) {
    uint32_t d;
    asm("lop3.b32 %0, %1, %2, %3, %4;" : "=r"(d) : "r"(a), "r"(b), "r"(c), "n"(LUT));
    return d;
}
// integer multiply-add pipe (IMAD / IMAD.HI), which the recurrence itself leaves idle
__device__ __forceinline__ uint32_t mad_lo(uint32_t a, uint32_t b, uint32_t c) {
    uint32_t d;
    asm("mad.lo.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
    return d;
}
__device__ __forceinline__ uint32_t mad_hi(uint32_t a, uint32_t b, uint32_t c) {
    uint32_t d;
    asm("mad.hi.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
    return d;
}
// acc += hi(a * b), in place (no copy of the accumulator)
__device__ __forceinline__ void mad_hi_acc(uint32_t& acc, uint32_t a, uint32_t b) {
    asm("mad.hi.u32 %0, %1, %2, %0;" : "+r"(acc) : "r"(a), "r"(b));
}

// One column of one block: the Myers/Hyyroe word-step over W words with the horizontal deltas (in_hp, in_hn: bit 31 =
// the row above the block) of the block above.  Returns HP / HN of the last word (bit 31 = the block's bottom row).
//
// Per word, on the ALU pipe: T = Eq & Pv;  S = T + Pv + carry (one carry chain through the block);
//   HN<<1 = S ^ T ^ Pv      -- the carries INTO every bit of that sum are exactly the shifted HN vector
//                              (carry out of bit i = Pv_i & (Eq_i | carry_i) = Pv_i & D0_i = HN_i), word boundaries included;
//   D0' = (S ^ Pv) | Eq  (D0 = D0' | Mv);  HP = Mv | ~(Pv | D0');  Mv' = HP<<1 & D0;  Pv' = HN<<1 | ~(HP<<1 | D0).
// (Measured on B200: IMAD / IMAD.HI share their issue slots with the ALU pipe, so shifting HP with multiply-adds
// instead of one funnel shift gains nothing.)
// KEEP_HP: also hand back HP of every word (the traceback wants HP and the new Pv of each cell).
// RAW_CARRY (the engine): in_hn is either zero or 0x80000000 and goes into the adder's carry chain as it is (any non-zero
// value is a carry), and out_hn is handed back in the same form -- bit 31 alone -- so that the lane below can use it
// without a shift or a mask on the ALU pipe.
template <int W, bool KEEP_HP, bool RAW_CARRY = false>
__device__ __forceinline__ void block_column(uint32_t (&Pv)[W], uint32_t (&Mv)[W], const uint32_t (&Eq)[W], uint32_t in_hp, uint32_t in_hn,
                                             uint32_t& out_hp, uint32_t& out_hn, uint32_t (&hp_all)[KEEP_HP ? W : 1]) {
    constexpr int CH = W < 8 ? W : 8;
    uint32_t hp_prev = in_hp;
    uint32_t hp_last = in_hp, hn_last = in_hn;
    uint32_t carry = RAW_CARRY ? in_hn : in_hn >> 31;     // the adder's carry across a word boundary equals the HN bit there
#pragma unroll
    for (int c0 = 0; c0 < W; c0 += CH) {
        uint32_t Tt[CH], Sm[CH];
#pragma unroll
        for (int i = 0; i < CH; ++i) Tt[i] = Eq[c0 + i] & Pv[c0 + i];
        if (c0 + CH < W) carry = Chain<CH, true>::run(Sm, Tt, &Pv[c0], carry);
        else Chain<CH, false>::run(Sm, Tt, &Pv[c0], carry);
#pragma unroll
        for (int i = 0; i < CH; ++i) {
            uint32_t const pv = Pv[c0 + i], mv = Mv[c0 + i];
            // (LOP3 by hand: left to itself the compiler expands D0p again and spends an extra instruction per word)
            uint32_t const HNs = lop3<0x96>(Sm[i], Tt[i], pv);                // S ^ T ^ Pv
            uint32_t const D0p = lop3<0xBE>(Sm[i], pv, Eq[c0 + i]);           // (S ^ Pv) | Eq;  D0 = D0p | Mv
            uint32_t const HP = lop3<0xF1>(mv, pv, D0p);                      // Mv | ~(Pv | D0p)
            uint32_t const HPs = __funnelshift_l(hp_prev, HP, 1);
            hp_prev = HP;
            if (c0 + i == W - 1) { hp_last = HP; hn_last = RAW_CARRY ? lop3<0x80>(pv, D0p, 0x80000000u) : (pv & D0p); }   // Pv & Mv == 0
            Mv[c0 + i] = lop3<0xE0>(HPs, D0p, mv);                            // HPs & (D0p | Mv)
            uint32_t const u = lop3<0xFE>(HPs, D0p, mv);                      // HPs | D0
            Pv[c0 + i] = lop3<0xF3>(HNs, u, 0u);                              // HNs | ~(HPs | D0)
            if (KEEP_HP) hp_all[c0 + i] = HP;
        }
    }
    out_hp = hp_last; out_hn = hn_last;
}

template <int W>
__device__ __forceinline__ void write_checkpoint(uint32_t* rec, const uint32_t (&Pv)[W], const uint32_t (&Mv)[W], uint32_t hp_bits, uint32_t hn_bits) {
    if constexpr (W == 1) {
        *reinterpret_cast<uint4*>(rec) = make_uint4(Pv[0], Mv[0], hp_bits, hn_bits);
    } else if constexpr (W == 2) {
        *reinterpret_cast<uint4*>(rec) = make_uint4(Pv[0], Pv[1], Mv[0], Mv[1]);
        *reinterpret_cast<uint4*>(rec + 4) = make_uint4(hp_bits, hn_bits, 0u, 0u);
    } else {
#pragma unroll
        for (int i = 0; i < W; i += 4) {
            *reinterpret_cast<uint4*>(rec + i) = make_uint4(Pv[i], Pv[i + 1], Pv[i + 2], Pv[i + 3]);
            *reinterpret_cast<uint4*>(rec + W + i) = make_uint4(Mv[i], Mv[i + 1], Mv[i + 2], Mv[i + 3]);
        }
        *reinterpret_cast<uint4*>(rec + 2 * W) = make_uint4(hp_bits, hn_bits, 0u, 0u);
    }
}

// Steps t .. evt-1 of every lane of the warp: no block starts or ends in this range, so the loop is the recurrence
// and nothing else -- no divergent branch (inactive lanes run the same instructions on dead state and keep publishing
// the "+1 per column" boundary), window characters two steps and Eq rows one step ahead of their use.
// What a lane takes from the lane of the block above goes through three masks (Upper): the neighbour's deltas as they
// are, or zeros (block 0: row 0 of a semi-global matrix is all zeros), or "+1 per column" (the block above has ended:
// its lane may already be at work on its next block, and what lies beyond a block's last column is bounded by +1 steps).
// The block above ends with the step before an event, and the step of the event still reads its last column: `peel`
// (warp-uniform) runs that one step with the masks `first` and the others with `rest`.
// LAST:  some lane is on the last block (tracks the minimum of the last row);
// CKPT:  working blocks leave a checkpoint record after every step that is a multiple of 32 (the loop is cut there, so
//        that the stores stay out of the recurrence).
struct Upper { uint32_t keep, hp_add; };      // x * keep + hp_add (multiply-add pipe): keep = 1 takes the neighbour's deltas, keep = 0 replaces them; hp_add = 0x80000000: "+1 per column"
template <int W, bool CKPT, bool LAST>
__device__ __forceinline__ void run_steps(LaneState<W>& S, uint32_t t, uint32_t const evt, bool const active, uint32_t const src_lane,
                                          uint32_t const last_block, const uint8_t* const win0, const uint8_t* const idle_chars, uint32_t const two,
                                          Upper const first, Upper const rest, bool peel) {
    uint32_t const inc = active ? 1u : 0u;
    Upper up = peel ? first : rest;
    bool const track = LAST && active && S.b == last_block;
    // character of column j is win0[j - 1] (inside the ring buffer); idle lanes keep reading one valid character
    uint32_t wp = uint32_t(__cvta_generic_to_shared(active ? win0 + (int32_t(t) - int32_t(S.b) - 1) : idle_chars));
    uint32_t const eqb = uint32_t(__cvta_generic_to_shared(S.eqb));
    // published deltas: a * x + b with (a, b) = (1, 0) for a working lane and (0, boundary) for an idle one
    uint32_t const pub_a = inc, pub_hp_b = active ? 0u : 0x80000000u;
    // bottom-row value = base + (#steps with HP) - (#steps with HN), the two counts kept by multiply-adds
    // (`two` = 2 comes in as a kernel parameter: as a literal, mad.hi(x, 2, c) is turned back into an ALU-pipe LEA.HI)
    int32_t const score_base = S.score;
    uint32_t n_hp = 0, n_hn = 0;
    uint32_t EqA[W], EqB[W];
    uint32_t no_hp[1];
    load_eq<W>(EqA, mad_lo(lds_u8(wp), 4 * W, eqb));
    wp += inc;
    uint32_t cn = lds_u8(wp);                             // character of step t + 1
#define FXG_STEP(EQ_USE, EQ_LOAD)                                                                          \
    {                                                                                                      \
        load_eq<W>(EQ_LOAD, mad_lo(cn, 4 * W, eqb));      /* Eq of the next step */                        \
        wp += inc; cn = lds_u8(wp);                       /* character of the step after it */             \
        uint32_t r_hp = __shfl_sync(0xffffffffu, S.o_hp, src_lane);                                        \
        uint32_t r_hn = __shfl_sync(0xffffffffu, S.o_hn, src_lane);                                        \
        r_hp = mad_lo(r_hp, up.keep, up.hp_add);          /* only bit 31 is looked at */                   \
        r_hn = mad_lo(r_hn, up.keep, 0u);                 /* 0 or 0x80000000 */                            \
        uint32_t hp, hn;                                                                                   \
        block_column<W, false, true>(S.Pv, S.Mv, EQ_USE, r_hp, r_hn, hp, hn, no_hp);                       \
        S.o_hp = mad_lo(hp, pub_a, pub_hp_b); S.o_hn = mad_lo(hn, pub_a, 0u);                              \
        mad_hi_acc(n_hp, hp, two); mad_hi_acc(n_hn, hn, two);                                        \
        if (LAST) {                                                                                        \
            int32_t const sc = score_base + int32_t(n_hp) - int32_t(n_hn);                                 \
            if (track && sc <= S.best) { S.best = sc; S.best_col = t - S.b; }                              \
        }                                                                                                  \
        if (CKPT) { S.acc_hp = __funnelshift_l(hp, S.acc_hp, 1); S.acc_hn = __funnelshift_l(hn, S.acc_hn, 1); } \
        ++t;                                                                                               \
    }
    while (t < evt) {
        // up to and including the next multiple of 32 (checkpoint passes), or all the way
        uint32_t const seg = peel ? t + 1u : (CKPT ? min(evt, ((t + 31u) & ~31u) + 1u) : evt);
        while (t + 1 < seg) { FXG_STEP(EqA, EqB) FXG_STEP(EqB, EqA) }
        if (t < seg) {
            FXG_STEP(EqA, EqB)
#pragma unroll
            for (int i = 0; i < W; ++i) EqA[i] = EqB[i];
        }
        if (CKPT) {
            if (((t - 1) & 31u) == 0 && active) { write_checkpoint<W>(S.ckp, S.Pv, S.Mv, __brev(S.acc_hp), __brev(S.acc_hn)); S.ckp += ck_record_words(W); }
        }
        if (peel) { peel = false; up = rest; }
    }
#undef FXG_STEP
    // (a lane that did not work keeps the value its last block ended with: a band of one diagonal starts the block below from it)
    S.score = active ? score_base + int32_t(n_hp) - int32_t(n_hn) : score_base;
}

// 32 consecutive window characters (one 16-byte chunk of the packed store) as bytes.  `logical` counts chunks in sweep
// order: forward passes read the store upwards from the chunk of window[0]; reverse passes (alignment.cpp:118-125)
// read it downwards from the chunk of window[n-1], each chunk back to front, so that the sweep is always forward.
__device__ __forceinline__ void load_window_chunk(const uint4* __restrict__ packed, int64_t n_chunks, int64_t first_chunk, bool reverse,
                                                  uint32_t logical, uint8_t* buf) {
    int64_t g = reverse ? first_chunk - int64_t(logical) : first_chunk + int64_t(logical);
    if (g < 0) g = 0;                                     // only characters past the window's end can come from here
    if (g >= n_chunks) g = n_chunks - 1;
    uint4 const v = __ldg(packed + g);
    uint4 a, b2;
    unpack8(v.x, a.x, a.y); unpack8(v.y, a.z, a.w); unpack8(v.z, b2.x, b2.y); unpack8(v.w, b2.z, b2.w);
    if (reverse) {
        uint4 const ra = make_uint4(__byte_perm(b2.w, 0, 0x0123), __byte_perm(b2.z, 0, 0x0123), __byte_perm(b2.y, 0, 0x0123), __byte_perm(b2.x, 0, 0x0123));
        uint4 const rb = make_uint4(__byte_perm(a.w, 0, 0x0123), __byte_perm(a.z, 0, 0x0123), __byte_perm(a.y, 0, 0x0123), __byte_perm(a.x, 0, 0x0123));
        a = ra; b2 = rb;
    }
    uint32_t const slot = logical % kWinChunks;
    uint4* d0 = reinterpret_cast<uint4*>(buf + slot * 32);
    uint4* d1 = reinterpret_cast<uint4*>(buf + (slot + kWinChunks) * 32);
    d0[0] = a; d0[1] = b2; d1[0] = a; d1[1] = b2;
}

// the tasks_per_warp tasks number `group_index` of a launch, on one warp
template <int W, bool CKPT>
__device__ __forceinline__ void dp_task_group(DpLaunch const& L, const DpTask* const tasks, uint32_t const group_index, uint32_t const n_tasks, uint8_t* const smem) {
    uint32_t const lane = threadIdx.x;
    uint32_t const G = L.group;
    uint32_t const tasks_per_warp = 32u / G;
    uint32_t const slot = lane / G;                 // which task of this warp
    uint32_t const r = lane % G;                    // ring position
    uint32_t const task_id = group_index * tasks_per_warp + slot;
    bool const in_ring = slot < tasks_per_warp;     // G need not divide 32: spare lanes idle
    bool const have_task = in_ring && task_id < n_tasks;

    // lanes without a task idle on the (always present) first task's buffers: whatever they read there is valid
    uint8_t* const win = smem + size_t(have_task ? slot : 0) * kWinBytes;
    uint32_t* const peq = reinterpret_cast<uint32_t*>(smem + size_t(tasks_per_warp) * kWinBytes) +
                          size_t(have_task ? slot : 0) * kNumSymbols * L.peq_stride;

    DpTask T;
    if (have_task) T = tasks[task_id];
    else { T.n = 0; T.m = 1; T.dlo = 0; T.dhi = 0; T.flags = 0; T.ref_base = 0; T.query_base = 0; T.trace_base = 0; T.out = 0; }

    constexpr int ROWS = 32 * W;
    uint32_t const nb = (T.m + ROWS - 1) / ROWS;               // blocks of this task
    uint32_t const pad = nb * ROWS - T.m;                      // wildcard rows in front, so that row m is the last bit
    int32_t const dlo = T.dlo - int32_t(pad), dhi = T.dhi - int32_t(pad);
    bool const reverse = (T.flags & kFlagReverse) != 0;

    // ---- the window streams through a small ring buffer: character i (0-based, sweep order) sits in logical chunk
    //      (phase + i) / 32; the buffer holds chunks [c_base, c_base + kWinChunks)
    const uint4* const packed = reinterpret_cast<const uint4*>((T.flags & kFlagInlineRef) ? L.inline_packed : L.ref_packed);
    int64_t const store_chunks = int64_t((T.flags & kFlagInlineRef) ? L.inline_chunks : L.ref_chunks);
    uint64_t const w_last = T.ref_base + (T.n ? T.n - 1 : 0);  // store position of window[n-1]
    int64_t const first_chunk = reverse ? int64_t(w_last >> 5) : int64_t(T.ref_base >> 5);
    uint32_t const phase = reverse ? 31u - uint32_t(w_last & 31u) : uint32_t(T.ref_base & 31u);
    uint32_t c_base = 0;
    bool dead = false;                                         // internal inconsistency: the task reports kPoisonScore
    if (have_task) {
        // (a short window does not fill the buffer: the sweep reads up to two characters past the window's end and no further)
        uint32_t const fill = min(kWinChunks, (phase + T.n + 2u + 31u) / 32u);
        for (uint32_t c = r; c < fill; c += G) load_window_chunk(packed, store_chunks, first_chunk, reverse, c, win);
        // ---- stage the Eq table of the query piece from the pool-level Peq planes: block-major, then symbol, then word ----
        uint32_t const n_words = nb * W;
        for (uint32_t w = r; w < n_words; w += G) {
            int32_t const virt = int32_t(pad) - int32_t(32 * w);            // wildcard bits in this word
            uint32_t const wild = virt >= 32 ? 0xffffffffu : (virt > 0 ? ((1u << virt) - 1u) : 0u);
            uint32_t* const dst = peq + (w / W) * (kNumSymbols * W) + (w % W);
#pragma unroll
            for (int s = 0; s < kNumSymbols; ++s) {
                const uint32_t* plane = L.peq_table + uint64_t(s) * L.peq_plane_words;
                uint32_t x;
                if (!reverse) {
                    x = peq_window(plane, int64_t(T.query_base) - int64_t(pad) + int64_t(32 * w));
                } else {
                    int64_t const y = int64_t(T.query_base) + int64_t(T.m) - 1 + int64_t(pad) - int64_t(32 * w);
                    x = __brev(peq_window(plane, y - 31));
                }
                dst[s * W] = x | wild;
            }
        }
    }
    __syncwarp();

    uint32_t const last_block = nb - 1;
    uint32_t const ck_per_block = ck_records_per_block(int64_t(T.dhi) - int64_t(T.dlo) + 1, ROWS);
    LaneState<W> S;
    S.acc_hp = 0; S.acc_hn = 0; S.ckp = nullptr;
#pragma unroll
    for (int i = 0; i < W; ++i) { S.Pv[i] = 0; S.Mv[i] = 0; }
    S.b = r; S.o_hp = 0x80000000u; S.o_hn = 0;      // an idle lane publishes "the boundary grows by +1 per column"
    S.score = 0; S.best = kNoScore; S.best_col = 0;
    S.eqb = peq;
    int32_t ce_up = 0;                              // last column of the block above the lane's current block
    auto set_block = [&](uint32_t blk) {
        S.cs = 0x7fffffff; S.ce = -1;
        if (!have_task || blk >= nb) return;
        {
            int32_t const hi_up = int32_t(ROWS) * int32_t(blk) + dhi;
            ce_up = hi_up > int32_t(T.n) ? int32_t(T.n) : hi_up;
        }
        // (all quantities are far below 2^31: queries are at most FXG_MAX_QUERY_LENGTH long)
        int32_t const lo = int32_t(ROWS) * int32_t(blk) + 1 + dlo;
        int32_t const hi = int32_t(ROWS) * int32_t(blk + 1) + dhi;
        int32_t const cs = lo < 1 ? 1 : lo;
        int32_t const ce = hi > int32_t(T.n) ? int32_t(T.n) : hi;
        if (cs <= ce) { S.cs = cs; S.ce = ce; }
    };
    set_block(S.b);
    uint32_t const src_lane = in_ring ? slot * G + (r + G - 1) % G : lane;

    // number of steps of this warp: last block of the longest task
    uint32_t const my_end = __reduce_max_sync(0xffffffffu, have_task ? (T.n + nb - 1) : 0u);
    constexpr uint32_t kNever = 0x7fffffffu;

    // (checkpoint passes) the block of this lane ended with step t - 1: the boundary bits since the last multiple of 32 go
    // into one more record
    auto flush_boundary_bits = [&](uint32_t t) {
        uint32_t const left_over = (t - 1) & 31u;
        if (left_over) {
            uint32_t const hb = __brev(S.acc_hp) >> (32 - left_over), nbits = __brev(S.acc_hn) >> (32 - left_over);
            if constexpr (W == 1) *reinterpret_cast<uint2*>(S.ckp + 2) = make_uint2(hb, nbits);
            else *reinterpret_cast<uint4*>(S.ckp + 2 * W) = make_uint4(hb, nbits, 0u, 0u);
        }
    };

    uint32_t my_refill = 0;                                    // first step that would read past this ring's window buffer (0: not planned yet)
    uint32_t t = 1;
    while (t <= my_end) {
        // ---------------- between steps t-1 and t: blocks that ended move on, blocks that begin are set up ----------------
        uint32_t const r_hp = __shfl_sync(0xffffffffu, S.o_hp, src_lane);
        uint32_t const r_hn = __shfl_sync(0xffffffffu, S.o_hn, src_lane);
        int32_t const r_sc = __shfl_sync(0xffffffffu, S.score, src_lane);
        if (S.ce >= 0 && int32_t(t) - int32_t(S.b) > S.ce) {
            if (CKPT) flush_boundary_bits(t);
            S.b += G; set_block(S.b);
        }
        int32_t const j = int32_t(t) - int32_t(S.b);
        if (j == S.cs) {
            // (re)start: column cs-1 of this block is (bottom of the block above at cs-1) + 1, 2, ...
#pragma unroll
            for (int i = 0; i < W; ++i) { S.Pv[i] = 0xffffffffu; S.Mv[i] = 0; }
            if (S.b == 0) {
                // wildcard rows carry value 0: no vertical step there
#pragma unroll
                for (int i = 0; i < W; ++i) {
                    int32_t const virt = int32_t(pad) - 32 * i;
                    S.Pv[i] = virt >= 32 ? 0u : (virt > 0 ? (0xffffffffu << virt) : 0xffffffffu);
                }
                S.score = int32_t(ROWS) - int32_t(pad);
            } else if (S.cs - 1 == ce_up) {
                // a band of a single diagonal (k = 0, window as long as the query): the block above ended at column cs - 1 and
                // its lane, idle since, still holds that column's value
                S.score = r_sc + ROWS;
            } else {
                // the block above has just done column cs: its deltas there lead back to column cs - 1
                S.score = r_sc - int32_t(r_hp >> 31) + int32_t(r_hn >> 31) + ROWS;
            }
            S.eqb = peq + S.b * (kNumSymbols * W);
            if (CKPT) {
                // steps before the block's first one read as "boundary grows by +1 per column", like an idle lane's output
                S.acc_hp = 0xffffffffu; S.acc_hn = 0;
                S.ckp = L.trace + T.trace_base + uint64_t(S.b) * ck_per_block * ck_record_words(W);
            }
        }
        bool const active = j >= S.cs && j <= S.ce && !dead;
        // ---------------- window ring buffer: the blocks of a ring read characters t-1-b .. t+1-b (two ahead) ----------------
        // Computed from the band geometry alone, identically by every lane of the ring (no voting):
        //   b_top = first block that has not ended yet (it reads furthest ahead: ce(b) + b grows with b),
        //   b_low = last block that has begun (blocks that begin later start at or beyond its position).
        // (looked at only when some ring's buffer runs out with this step: until then the step computed at the last
        //  look stays valid -- the first unfinished block only moves down, so reads never reach further ahead than planned)
        if (__any_sync(0xffffffffu, t >= my_refill)) {
            my_refill = kNever;
            uint32_t new_base = c_base;
            uint32_t i_hi = 0;
            bool reading = false;
            if (have_task && !dead) {
                // (all quantities are far below 2^31: n, m <= a few 100 000)
                int32_t const ti = int32_t(t);
                int32_t const e1 = ti - int32_t(T.n);                                               // n + b >= t
                int32_t const e2n = ti - dhi - ROWS;                                                // ROWS (b+1) + dhi + b >= t
                int32_t const e2 = e2n > 0 ? (e2n + ROWS) / (ROWS + 1) : 0;
                int32_t const b_top = e1 > e2 ? e1 : e2;
                int32_t const s1 = ti - 1 - dlo;                                                    // ROWS b + 1 + dlo + b <= t
                int32_t b_low = s1 > 0 ? s1 / (ROWS + 1) : 0;
                if (b_low > ti - 1) b_low = ti - 1;                                                 // blocks clipped to column 1 begin at step 1 + b
                if (b_low > int32_t(last_block)) b_low = int32_t(last_block);
                reading = b_top <= int32_t(last_block);
                if (reading) {
                    i_hi = uint32_t(int32_t(phase) + ti + 1 - b_top);                               // buffer position of the furthest read of step t
                    if (i_hi >= 32 * (c_base + kWinChunks)) {
                        int32_t const lo = ti - 3 - b_low;                                          // everything before it is done with
                        new_base = uint32_t(int32_t(phase) + (lo > 0 ? lo : 0)) >> 5;
                        if (new_base <= c_base || i_hi >= 32 * (new_base + kWinChunks)) { dead = true; new_base = c_base; }   // cannot happen: a ring spans < 40 characters
                    }
                }
            }
            // the refill itself in warp-uniform control flow (the hot loops below rely on a converged warp)
            uint32_t const rounds = __reduce_max_sync(0xffffffffu, (new_base - c_base + G - 1) / G);
            for (uint32_t k = 0; k < rounds; ++k) {
                uint32_t const c = c_base + kWinChunks + r + k * G;
                if (c < new_base + kWinChunks) load_window_chunk(packed, store_chunks, first_chunk, reverse, c, win);
            }
            c_base = new_base;
            if (reading && !dead) my_refill = t + (32 * (c_base + kWinChunks) - i_hi);              // first step that would read past the buffer
        }
        __syncwarp();
        // character of column j is win0[j - 1]: chunk c lives at slot c % kWinChunks (and kWinChunks above it)
        uint8_t const* const win0 = win + phase - 32 * kWinChunks * (c_base / kWinChunks);
        // next step at which some lane's block ends (it moves on before the step after) or begins, or a buffer runs out
        uint32_t my_evt = active ? uint32_t(S.ce) + S.b + 1u : (S.cs == 0x7fffffff ? kNever : uint32_t(S.cs) + S.b);
        my_evt = min(my_evt, my_refill);
        // What the lane takes from the lane of the block above (run_steps): nothing for block 0, "+1 per column" once the
        // block above has ended.  Its last step is ce_up + b - 1; the step after it is an event (the block's end) and still
        // reads that last column, the steps after that read the bound.
        auto upper_at = [&](uint32_t step) {
            if (S.b == 0) return Upper{0u, 0u};
            return int32_t(step) - int32_t(S.b) > ce_up ? Upper{0u, 0x80000000u} : Upper{1u, 0u};
        };
        Upper const up_first = upper_at(t), up_rest = upper_at(t + 1);
        bool const peel = __any_sync(0xffffffffu, up_first.keep != up_rest.keep);
        if (active && S.b > 0 && int32_t(t) - int32_t(S.b) < ce_up) my_evt = min(my_evt, uint32_t(ce_up) + S.b);   // (coincides with the end of the block above)
        uint32_t const evt = min(__reduce_min_sync(0xffffffffu, my_evt), my_end + 1);
        bool const any_last = __any_sync(0xffffffffu, active && S.b == last_block);
        if (any_last) run_steps<W, CKPT, true>(S, t, evt, active, src_lane, last_block, win0, win, L.two, up_first, up_rest, peel);
        else run_steps<W, CKPT, false>(S, t, evt, active, src_lane, last_block, win0, win, L.two, up_first, up_rest, peel);
        t = evt;
    }
    // the blocks that worked up to the warp's very last step never came back to the bookkeeping above: the last block of
    // the longest task still owes its final boundary bits (the last row's deltas, which range_min_kernel reads)
    if (CKPT && S.ce >= 0 && int32_t(t) - int32_t(S.b) > S.ce) flush_boundary_bits(t);
    // the lane that owned the last block reports
    uint32_t const owner = last_block % G;
    if (have_task && r == owner) {
        DpResult res; res.score = dead ? kPoisonScore : S.best; res.end_col = S.best_col;
        L.results[T.out] = res;
    }
}

// One warp per CTA.  Launches whose task count is known on the host have one CTA per group of tasks; launches whose tasks
// were built on the device (n_tasks_dev) get a grid that is only an upper bound, capped by the host at what the machine
// can hold at once: CTAs take the groups in turn and leave when none is left.
// (the second launch bound keeps the register count where it was before the loop around the task groups: 25 warps per SM
//  for W = 4 with checkpoints instead of 23)
__host__ __device__ constexpr int dp_min_ctas(int W) { return W <= 2 ? 28 : (W == 4 ? 25 : (W == 8 ? 19 : (W == 16 ? 14 : 8))); }
template <int W, bool CKPT>
__global__ void __launch_bounds__(32, dp_min_ctas(W)) dp_kernel(DpLaunch const L) {
    extern __shared__ __align__(16) uint8_t smem[];
    uint32_t const tasks_per_warp = 32u / L.group;
    uint32_t const n_tasks = L.n_tasks_dev ? __ldg(L.n_tasks_dev) : L.n_tasks;
    const DpTask* tasks = L.tasks;
    if (L.class_active) { for (uint32_t c = 0; c < L.cls; ++c) tasks += __ldg(L.class_active + c); }
    for (uint32_t g = blockIdx.x; g * tasks_per_warp < n_tasks; g += gridDim.x) {
        dp_task_group<W, CKPT>(L, tasks, g, n_tasks, smem);
        __syncwarp();                               // the next group reuses the window and Eq buffers
    }
}

// ---------------------------------------------------------------------------------------------
// The engine for bands that no ring of one warp can hold (more than ~29 700 diagonals: reads near the 100 kbp limit of
// input.hpp:42 at 10-15 % errors).  One CTA of kWideThreads threads per task, W = 32: thread l owns block l (1 024 rows)
// and nothing else -- 128 blocks cover every legal query -- and the hand-over of the horizontal deltas between neighbours
// goes through shared memory with one barrier per step instead of a shuffle.  Same band rule, same boundary conventions
// (a block outside its working range publishes "+1 per column"; a fresh block starts from the block above + 1, 2, ...),
// same checkpoint records as dp_kernel<32, CKPT>, so walk2_kernel<32> and range_min_kernel read its output unchanged.
// These tasks are rare and long (a 100 kbp root is 1.4e10 cells); the kernel is written for exactness, not for the roofline.
// ---------------------------------------------------------------------------------------------
constexpr uint32_t kWideThreads = 128;
constexpr uint32_t kWideG = 64;                     // marks the wide configuration in the host's (W, G) tables
__host__ __device__ constexpr size_t wide_smem_bytes() { return size_t(kNumSymbols) * 32 * kWideThreads * 4 + 2 * kWideThreads * 16; }

template <bool CKPT>
__global__ void __launch_bounds__(kWideThreads, 1) dp_wide_kernel(DpLaunch const L) {
    extern __shared__ __align__(16) uint8_t smem[];
    constexpr int W = 32;
    constexpr int ROWS = 32 * W;
    uint32_t* const eq_all = reinterpret_cast<uint32_t*>(smem);                     // Eq[sym][word][thread]
    uint4* const pub = reinterpret_cast<uint4*>(smem + size_t(kNumSymbols) * 32 * kWideThreads * 4);   // [2][thread]: hp, hn, score
    uint32_t const l = threadIdx.x;
    uint32_t const n_tasks = L.n_tasks_dev ? __ldg(L.n_tasks_dev) : L.n_tasks;
    const DpTask* tasks = L.tasks;
    if (L.class_active) { for (uint32_t c = 0; c < L.cls; ++c) tasks += __ldg(L.class_active + c); }
    for (uint32_t task_id = blockIdx.x; task_id < n_tasks; task_id += gridDim.x) {
        DpTask const T = tasks[task_id];
        uint32_t const nb = (T.m + ROWS - 1) / ROWS;               // <= kWideThreads (checked by the host)
        uint32_t const pad = nb * ROWS - T.m;
        int32_t const dlo = T.dlo - int32_t(pad), dhi = T.dhi - int32_t(pad);
        bool const reverse = (T.flags & kFlagReverse) != 0;
        const uint32_t* const packed = (T.flags & kFlagInlineRef) ? L.inline_packed : L.ref_packed;
        bool const have = l < nb;
        int32_t cs = 0x7fffffff, ce = -1;
        if (have) {
            int32_t const lo = int32_t(ROWS) * int32_t(l) + 1 + dlo, hi = int32_t(ROWS) * int32_t(l + 1) + dhi;
            int32_t const a = lo < 1 ? 1 : lo, b = hi > int32_t(T.n) ? int32_t(T.n) : hi;
            if (a <= b) { cs = a; ce = b; }
        }
        // ---- Eq rows of this thread's block ----
        if (have) {
            for (int w = 0; w < W; ++w) {
                uint32_t const gw = l * W + uint32_t(w);
                int32_t const virt = int32_t(pad) - int32_t(32 * gw);
                uint32_t const wild = virt >= 32 ? 0xffffffffu : (virt > 0 ? ((1u << virt) - 1u) : 0u);
                for (int sym = 0; sym < kNumSymbols; ++sym) {
                    const uint32_t* plane = L.peq_table + uint64_t(sym) * L.peq_plane_words;
                    uint32_t x;
                    if (!reverse) x = peq_window(plane, int64_t(T.query_base) - int64_t(pad) + int64_t(32 * gw));
                    else x = __brev(peq_window(plane, int64_t(T.query_base) + int64_t(T.m) - 1 + int64_t(pad) - int64_t(32 * gw) - 31));
                    eq_all[(uint32_t(sym) * 32 + uint32_t(w)) * kWideThreads + l] = x | wild;
                }
            }
        }
        uint32_t Pv[W], Mv[W];
#pragma unroll
        for (int i = 0; i < W; ++i) { Pv[i] = 0; Mv[i] = 0; }
        int32_t score = 0, best = kNoScore;
        uint32_t best_col = 0;
        uint32_t acc_hp = 0xffffffffu, acc_hn = 0;
        uint32_t const ck_per_block = ck_records_per_block(int64_t(T.dhi) - int64_t(T.dlo) + 1, ROWS);
        uint32_t* ckp = CKPT ? L.trace + T.trace_base + uint64_t(l) * ck_per_block * ck_record_words(W) : nullptr;
        pub[l] = make_uint4(0x80000000u, 0u, 0u, 0u);
        pub[kWideThreads + l] = make_uint4(0x80000000u, 0u, 0u, 0u);
        __syncthreads();
        uint32_t const t_end = T.n + nb - 1;
        bool const is_last = have && l == nb - 1;
        for (uint32_t t = 1; t <= t_end; ++t) {
            int32_t const j = int32_t(t) - int32_t(l);
            uint4 const up = l > 0 ? pub[((t - 1) & 1u) * kWideThreads + l - 1] : make_uint4(0u, 0u, 0u, 0u);   // the block above after step t - 1
            bool const active = have && j >= cs && j <= ce;
            uint4 mine = make_uint4(0x80000000u, 0u, uint32_t(score), 0u);         // outside its range a block publishes "+1 per column"
            if (active) {
                if (j == cs) {
                    // column cs - 1 of this block is (bottom of the block above at cs - 1) + 1, 2, ...
#pragma unroll
                    for (int i = 0; i < W; ++i) { Pv[i] = 0xffffffffu; Mv[i] = 0; }
                    if (l == 0) {
#pragma unroll
                        for (int i = 0; i < W; ++i) {
                            int32_t const virt = int32_t(pad) - 32 * i;            // wildcard rows carry value 0: no vertical step there
                            Pv[i] = virt >= 32 ? 0u : (virt > 0 ? (0xffffffffu << virt) : 0xffffffffu);
                        }
                        score = int32_t(ROWS) - int32_t(pad);
                    } else if (cs - 1 == (int32_t(ROWS) * int32_t(l) + dhi > int32_t(T.n) ? int32_t(T.n) : int32_t(ROWS) * int32_t(l) + dhi)) {
                        score = int32_t(up.z) + ROWS;                              // band of a single diagonal: the block above ended at column cs - 1
                    } else {
                        score = int32_t(up.z) - int32_t(up.x >> 31) + int32_t(up.y >> 31) + ROWS;
                    }
                    acc_hp = 0xffffffffu; acc_hn = 0;
                }
                // character of column j: window[j - 1] in sweep order
                uint64_t const pos = reverse ? T.ref_base + uint64_t(T.n) - uint64_t(j) : T.ref_base + uint64_t(j) - 1;
                uint32_t c = packed_base(packed, pos);
                if (c >= uint32_t(kNumSymbols)) c = 0;                               // (cannot happen: ranks are checked on upload)
                uint32_t Eq[W];
#pragma unroll
                for (int w = 0; w < W; ++w) Eq[w] = eq_all[(c * 32 + uint32_t(w)) * kWideThreads + l];
                uint32_t hp, hn, no_hp[1];
                block_column<W, false>(Pv, Mv, Eq, l == 0 ? 0u : up.x, l == 0 ? 0u : up.y, hp, hn, no_hp);
                score += int32_t(hp >> 31) - int32_t(hn >> 31);
                if (is_last && score <= best) { best = score; best_col = uint32_t(j); }
                mine = make_uint4(hp, hn, uint32_t(score), 0u);
                if (CKPT) {
                    acc_hp = __funnelshift_l(hp, acc_hp, 1); acc_hn = __funnelshift_l(hn, acc_hn, 1);
                    if ((t & 31u) == 0) { write_checkpoint<W>(ckp, Pv, Mv, __brev(acc_hp), __brev(acc_hn)); ckp += ck_record_words(W); }
                    else if (j == ce) {
                        // the block ends between two multiples of 32: the boundary bits since the last one go into one more record
                        uint32_t const left_over = t & 31u;
                        *reinterpret_cast<uint4*>(ckp + 2 * W) = make_uint4(__brev(acc_hp) >> (32 - left_over), __brev(acc_hn) >> (32 - left_over), 0u, 0u);
                    }
                }
            }
            pub[(t & 1u) * kWideThreads + l] = mine;
            __syncthreads();
        }
        if (is_last) { DpResult res; res.score = best; res.end_col = best_col; L.results[T.out] = res; }
        __syncthreads();                                   // the next task reuses the Eq rows
    }
}

struct WalkResult {
    uint32_t begin_col;     // column where the traceback reached row 0 (sequence1_begin_position)
    uint32_t cigar_len;     // 0xffffffff on overflow / inconsistency; the ops are the LAST cigar_len entries of the slot
};

// ---------------------------------------------------------------------------------------------
// traceback from checkpoints (alignment.cpp:156-178 of the reference): one LANE per alignment.
//
// The score pass of a root alignment left one record per block and 32 steps (see ck_record_words).  The cell the
// traceback stands on belongs to exactly one tile = (block b) x (steps 32 (q-1)+1 .. 32 q, i.e. columns t - b); the lane
// recomputes that tile with the engine's own word-step -- from the block's record at step 32 (q-1) and the boundary bits
// of the block above, exactly as the score pass computed it -- keeps its HP / VP' bits in local memory, follows the path
// until it leaves the tile, and repeats.  No trace planes ever reach HBM.
// ---------------------------------------------------------------------------------------------
struct Walk2Task {
    uint64_t ck_base;       // first word of the task's checkpoint records
    uint64_t ref_base;      // packed-store position of the score pass' window[0]
    uint64_t query_base;    // position of query[0] in the pool (bytes and Peq planes)
    uint64_t cigar_base;    // first op of the task's slot; the cigar ends at cigar_base + cigar_cap
    uint32_t n, m;          // window and query length of the score pass
    int32_t dlo, dhi;       // its band
    uint32_t end_col;       // column of the alignment's last cell (row m)
    uint32_t score;         // its number of errors
    uint32_t flags;
    uint32_t cigar_cap;
    uint32_t out;
    uint32_t reserved;
};

struct Walk2Launch {
    const Walk2Task* tasks; uint32_t n_tasks;
    const uint32_t* ck;
    const uint32_t* ref_packed; const uint32_t* inline_packed;
    const uint32_t* peq_table; uint64_t peq_plane_words;
    uint32_t* cigars;
    WalkResult* results;
    uint32_t two;
};

// One GROUP of W lanes per alignment (W = the block width of its score pass: lane w owns word w of the block), 64 / W
// alignments per CTA.  The tile the traceback stands on is recomputed as a skewed wavefront -- lane w does column step s
// at time s + w, the carries of word w - 1 arrive by shuffle -- so a tile of 32 steps costs 32 + W single-word steps
// instead of 32 W-word steps on one lane; only the words at or above the path's row are computed (carries run downwards).
// What the path does in a cell -- left, up, match, mismatch, two bits -- goes to shared memory as two bit planes, and every
// lane of the group follows the path through them in lockstep (same addresses: broadcasts), one 8-byte load per cell, so
// that all of them know where the next tile is; lane 0 writes the cigar.
__host__ __device__ constexpr uint32_t walk2_threads() { return 64u; }
__host__ __device__ constexpr uint32_t walk2_per_cta(uint32_t W) { return walk2_threads() / W; }
// shared memory per alignment: the two operation planes of 32 steps x W words (+ 2 words, so that the groups of a warp
// start in different banks and every pair of plane words stays 8-byte aligned), the Eq rows of its current block
// (6 symbols x W words) and the tile's 32 window characters as bytes
__host__ __device__ constexpr uint32_t walk2_words_per_group(uint32_t W) { return 64 * W + 2 + kNumSymbols * W + 8; }
__host__ __device__ constexpr size_t walk2_smem_bytes(uint32_t W) { return size_t(walk2_words_per_group(W)) * walk2_per_cta(W) * 4; }

template <int W>
__global__ void __launch_bounds__(walk2_threads()) walk2_kernel(Walk2Launch const L) {
    extern __shared__ __align__(16) uint32_t w2_smem[];
    constexpr int ROWS = 32 * W;
    constexpr uint32_t RECW = ck_record_words(W);
    constexpr uint32_t PER_CTA = walk2_per_cta(W);
    uint32_t const w = threadIdx.x % W;                                    // this lane's word of the block
    uint32_t const grp = threadIdx.x / W;                                  // alignment within the CTA
    // operation code of the cell in row bit r of word x at step p: bit r of bits[(p * W + x) * 2] (low) and of the word
    // after it (high); 0 match, 1 mismatch, 2 up (I), 3 left (D) -- trace priority left > up > diagonal, decided in the
    // one place that writes the planes (oracle: FXO_TRACE_PRIORITY)
    uint32_t* const bits = w2_smem + grp * walk2_words_per_group(W);
    uint32_t* const eq_g = bits + 64 * W + 2;                              // Eq[sym][x] at eq_g[sym * W + x]
    uint8_t* const tile_chars = reinterpret_cast<uint8_t*>(eq_g + kNumSymbols * W);   // window character of step p of the tile
    uint32_t const id = blockIdx.x * PER_CTA + grp;
    bool const mine = id < L.n_tasks;
    bool done = !mine;
    Walk2Task T;
    if (!done) T = L.tasks[id];
    else { T = Walk2Task{}; T.m = 1; }
    const uint32_t* const ref = (T.flags & kFlagInlineRef) ? L.inline_packed : L.ref_packed;
    uint32_t const nb = (T.m + ROWS - 1) / ROWS;
    uint32_t const pad = nb * ROWS - T.m;
    int32_t const dlo = T.dlo - int32_t(pad), dhi = T.dhi - int32_t(pad);
    uint32_t const ck_per_block = ck_records_per_block(int64_t(T.dhi) - int64_t(T.dlo) + 1, ROWS);
    const uint32_t* const ck = L.ck + T.ck_base;
    uint32_t* const slot_end = L.cigars + T.cigar_base + T.cigar_cap;
    bool const writer = w == 0;

    // first / last step of block b in the score pass (block b is at column t - b at step t)
    auto block_steps = [&](uint32_t b, int32_t& ts, int32_t& te) {
        int32_t const lo = int32_t(ROWS) * int32_t(b) + 1 + dlo, hi = int32_t(ROWS) * int32_t(b + 1) + dhi;
        ts = (lo < 1 ? 1 : lo) + int32_t(b);
        te = (hi > int32_t(T.n) ? int32_t(T.n) : hi) + int32_t(b);
    };

    uint32_t i = T.m, j = T.end_col;                             // the cell the traceback stands on (row, column; 1-based)
    uint32_t n_runs = 0, cur_code = 0, cur_len = 0, errors = 0;  // the run being collected, by operation code
    bool bad = false;
    uint32_t eq_block = 0xffffffffu;                             // block whose Eq rows are in shared memory
    // the cigar operation of a code: =, X, I, D as 7, 8, 1, 2 (output.cpp of the reference writes them as "=XID")
    auto flush_run = [&]() {
        if (cur_len) {
            if (n_runs < T.cigar_cap) { if (writer) slot_end[-1 - int64_t(n_runs)] = (cur_len << 4) | ((0x2187u >> (4 * cur_code)) & 15u); }
            else bad = true;
            ++n_runs;
        }
    };
    auto emit = [&](uint32_t code, uint32_t len) {
        if (code == cur_code) { cur_len += len; return; }
        flush_run();
        cur_code = code; cur_len = len;
    };

    // inputs of a tile, as loaded: window characters, this lane's word of the block's record at the step before the tile,
    // boundary bits of the block above for the tile's steps (A) and the 32 steps before (B)
    struct TileIn { uint32_t raw[5]; uint32_t sh; uint32_t pv, mv; uint32_t hpA, hnA, hpB, hnB; };
    TileIn X;
    bool pf_valid = false; uint32_t pf_b = 0, pf_q = 0;
    auto fetch_tile = [&](uint32_t b, uint32_t q, TileIn& Y) {
        int32_t ts, te; block_steps(b, ts, te);
        int32_t const t0 = 32 * int32_t(q - 1);
        int64_t const pos0 = int64_t(T.ref_base) + int64_t(t0) - int64_t(b);      // store position of step t0 + 1 (column - 1)
        int64_t const w0 = pos0 >= 0 ? (pos0 >> 3) : -((7 - pos0) >> 3);          // floor(pos0 / 8); positions before the window are never used
        Y.sh = uint32_t(pos0 - w0 * 8) * 4;
#pragma unroll
        for (int k = 0; k < 5; ++k) Y.raw[k] = w0 + k >= 0 ? __ldg(ref + (w0 + k)) : 0u;
        Y.pv = 0; Y.mv = 0;
        if (t0 >= ts) {
            const uint32_t* rec = ck + (uint64_t(b) * ck_per_block + uint32_t(int32_t(q - 1) - ((ts + 31) >> 5))) * RECW;
            Y.pv = rec[w]; Y.mv = rec[W + w];
        }
        Y.hpA = 0xffffffffu; Y.hnA = 0; Y.hpB = 0xffffffffu; Y.hnB = 0;
        if (b > 0) {
            int32_t us, ue; block_steps(b - 1, us, ue);
            int32_t const uq_first = (us + 31) >> 5, uq_last = (ue + 31) >> 5;
            const uint32_t* const urec = ck + uint64_t(b - 1) * ck_per_block * RECW;
            constexpr int BO = W == 1 ? 2 : 2 * W;                           // where a record keeps its boundary bits
            if (int32_t(q) >= uq_first && int32_t(q) <= uq_last) { uint2 const v = *reinterpret_cast<const uint2*>(urec + uint64_t(int32_t(q) - uq_first) * RECW + BO); Y.hpA = v.x; Y.hnA = v.y; }
            if (int32_t(q) - 1 >= uq_first && int32_t(q) - 1 <= uq_last) { uint2 const v = *reinterpret_cast<const uint2*>(urec + uint64_t(int32_t(q) - 1 - uq_first) * RECW + BO); Y.hpB = v.x; Y.hnB = v.y; }
        }
    };

    while (!__all_sync(0xffffffffu, done)) {
        uint32_t b = 0, q = 0;
        if (!done) {
            if (i == 0) done = true;
            else if (j == 0) { emit(2, i); errors += i; i = 0; done = true; }     // column 0: only "up" remains
        }
        // ---------------- recompute the tile of (i, j): what this group needs, then the wavefront with the whole warp ----------------
        uint32_t Pv1[1] = {0}, Mv1[1] = {0};
        uint32_t top_hp = 0, top_hn = 0;
        int32_t p_first = 0, n_steps = 0;                                  // the tile's steps p_first .. p_first + n_steps - 1 are computed
        uint32_t wi0 = 0;                                                  // word of the path's row: words above it are all that is needed
        if (!done) {
            uint32_t const u = i + pad;                                          // row in the padded numbering (1-based)
            b = (u - 1) / ROWS;
            wi0 = ((u - 1) % ROWS) >> 5;
            uint32_t const t_cell = j + b;
            q = (t_cell + 31) >> 5;
            int32_t ts, te; block_steps(b, ts, te);
            int32_t const t0 = 32 * int32_t(q - 1);                              // the tile covers steps t0 + 1 .. t0 + 32
            // the path only moves up and left: nothing after the step of (i, j) is needed
            int32_t const t_lo = t0 + 1 > ts ? t0 + 1 : ts, t_hi = int32_t(t_cell) < te ? int32_t(t_cell) : te;
            p_first = t_lo - t0 - 1; n_steps = t_hi - t_lo + 1;
            if (n_steps < 0) n_steps = 0;
            // what the tile is computed from: fetched while the previous tile was being walked, if the guess was right
            if (!(pf_valid && pf_b == b && pf_q == q)) fetch_tile(b, q, X);
            pf_valid = false;
            // the tile's window characters, one byte per step: the lanes of the group share the four words of eight
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                if (uint32_t(k) % uint32_t(W) == w % 4u) {
                    uint32_t lo8, hi8;
                    unpack8(__funnelshift_r(X.raw[k], X.raw[k + 1], X.sh), lo8, hi8);
                    *reinterpret_cast<uint2*>(tile_chars + 8 * k) = make_uint2(lo8, hi8);
                }
            }
            if (t0 >= ts) { Pv1[0] = X.pv; Mv1[0] = X.mv; }
            else {
                // the block begins inside the tile: "block above + 1, 2, ..." (wildcard rows of block 0 carry value 0)
                int32_t const virt = b == 0 ? int32_t(pad) - 32 * int32_t(w) : 0;
                Pv1[0] = virt >= 32 ? 0u : (virt > 0 ? (0xffffffffu << virt) : 0xffffffffu);
                Mv1[0] = 0;
            }
            // upper boundary: bit p = horizontal delta of the row above the block at step t0 + 1 + p
            if (b > 0) {
                int32_t us, ue; block_steps(b - 1, us, ue);                      // the block above is one step ahead: its step t - 1
                top_hp = (X.hpA << 1) | (X.hpB >> 31);
                top_hn = (X.hnA << 1) | (X.hnB >> 31);
                // steps of the block above outside its working range publish the "+1" boundary
                int32_t const p_lo = us - t0, p_hi = ue - t0;                    // bit p <-> upper step t0 + p
                uint32_t valid = 0;
                if (p_hi >= 0 && p_lo <= 31) {
                    uint32_t const lo = p_lo > 0 ? uint32_t(p_lo) : 0u, hi = p_hi < 31 ? uint32_t(p_hi) : 31u;
                    valid = (hi == 31 ? 0xffffffffu : ((1u << (hi + 1)) - 1u)) & ~((1u << lo) - 1u);
                }
                top_hp = (top_hp & valid) | ~valid;
                top_hn &= valid;
            }
            // Eq rows of this block: every lane its own word
            if (eq_block != b) {
                eq_block = b;
                uint32_t const gw = b * W + w;
                int32_t const virt = int32_t(pad) - int32_t(32 * gw);
                uint32_t const wild = virt >= 32 ? 0xffffffffu : (virt > 0 ? ((1u << virt) - 1u) : 0u);
#pragma unroll
                for (int sym = 0; sym < kNumSymbols; ++sym) {
                    const uint32_t* plane = L.peq_table + uint64_t(sym) * L.peq_plane_words;
                    eq_g[sym * W + w] = peq_window(plane, int64_t(T.query_base) - int64_t(pad) + int64_t(32 * gw)) | wild;
                }
            }
        }
        __syncwarp();
        {
            // lane w computes step s of the tile at time s + w
            int32_t const my_last = (!done && w <= wi0) ? n_steps - 1 + int32_t(wi0) : -1;
            int32_t const t_max = __reduce_max_sync(0xffffffffu, my_last);
            uint32_t out_hp = 0, out_hn = 0;
            bool const works = !done && w <= wi0;
            // Eq word of this lane's next step, fetched one step ahead (clamped: the word of a step that is never done is not used)
            auto eq_of = [&](int32_t sidx) -> uint32_t {
                int32_t const p = p_first + (sidx < 0 ? 0 : sidx);
                return eq_g[uint32_t(tile_chars[p > 31 ? 31 : p]) * W + w];
            };
            uint32_t eq_next = works ? eq_of(-int32_t(w)) : 0u;
            for (int32_t tau = 0; tau <= t_max; ++tau) {
                uint32_t in_hp = __shfl_up_sync(0xffffffffu, out_hp, 1, W);
                uint32_t in_hn = __shfl_up_sync(0xffffffffu, out_hn, 1, W);
                int32_t const sidx = tau - int32_t(w);
                if (works && sidx >= 0 && sidx < n_steps) {
                    uint32_t const p = uint32_t(p_first + sidx);
                    if (w == 0) { in_hp = ((top_hp >> p) & 1u) << 31; in_hn = ((top_hn >> p) & 1u) << 31; }
                    uint32_t Eq1[1], hp_all[1];
                    Eq1[0] = eq_next;
                    eq_next = eq_of(sidx + 1);
                    block_column<1, true>(Pv1, Mv1, Eq1, in_hp, in_hn, out_hp, out_hn, hp_all);
                    // left where HP (D[i][j] = D[i][j-1] + 1), else up where the new Pv (D[i][j] = D[i-1][j] + 1), else the
                    // diagonal: a match where Eq (query[i-1] == window[j-1]), a mismatch otherwise
                    uint32_t const hp = hp_all[0], vp = Pv1[0];
                    uint32_t const low = hp | ~(vp | Eq1[0]);                          // codes 1 and 3
                    uint32_t const high = hp | vp;                                    // codes 2 and 3
                    *reinterpret_cast<uint2*>(bits + (p * W + w) * 2) = make_uint2(low, high);
                }
            }
        }
        __syncwarp();
        // the path most likely continues into the same block's previous 32 steps: get that tile's inputs on their
        // way now, they arrive while this tile is being walked
        if (!done) {
            int32_t ts, te; block_steps(b, ts, te);
            if (q >= 2 && 32 * int32_t(q - 1) >= ts) { fetch_tile(b, q - 1, X); pf_valid = true; pf_b = b; pf_q = q - 1; }
        }
        // ---------------- follow the path while it stays inside the tile (every lane of the group, in lockstep) ----------------
        if (!done) {
            // position inside the tile: step p (column), row r of the block (0-based); the tile is left when p < 0 (column
            // before the tile), r < 0 (row of the block above), or the matrix' row 0 / column 0 is reached
            uint32_t const u0 = i + pad;
            int32_t p = int32_t(j + b) - 32 * int32_t(q - 1) - 1;
            int32_t r = int32_t((u0 - 1) % ROWS);
            int32_t const r_min = b == 0 ? int32_t(pad) : 0;                       // first real row of the block
            int32_t const p_min = (int32_t(b) + 1 - 32 * int32_t(q - 1) - 1) > 0 ? (int32_t(b) + 1 - 32 * int32_t(q - 1) - 1) : 0;   // step of column 1
            uint32_t ops_err = 0;
            while (p >= p_min && r >= r_min) {
                uint2 const v = *reinterpret_cast<const uint2*>(bits + (uint32_t(p) * W + (uint32_t(r) >> 5)) * 2);
                uint32_t const bit = uint32_t(r) & 31u;
                uint32_t const lo1 = (v.x >> bit) & 1u, hi1 = (v.y >> bit) & 1u;
                uint32_t const code = lo1 | (hi1 << 1);
                p -= int32_t(code != 2u);                                          // every move but "up" (code 2) goes one column back
                r -= int32_t(code != 3u);                                          // every move but "left" (code 3) goes one row up
                ops_err += code != 0u;
                if (code == cur_code) ++cur_len;
                else { flush_run(); cur_code = code; cur_len = 1; }
            }
            // back to matrix coordinates
            int32_t const p0 = int32_t(j + b) - 32 * int32_t(q - 1) - 1, r0 = int32_t((u0 - 1) % ROWS);
            j -= uint32_t(p0 - p); i -= uint32_t(r0 - r);
            errors += ops_err;
        }
        __syncwarp();                                                      // the next tile overwrites the bits
    }
    if (mine && writer) {
        flush_run();
        if (errors != T.score) bad = true;                                       // the path must cost exactly what the score pass found
        WalkResult R; R.begin_col = j; R.cigar_len = bad ? 0xffffffffu : n_runs;
        L.results[T.out] = R;
    }
}

// ---------------------------------------------------------------------------------------------
// The tree walk on the device (query_verifier::verify, verification.cpp:8-136).
//
// A batch arrives as compact records made once per job (host: prepare_job): one NodeRec per inner node, one LeafRec per
// leaf, one ReadRec per read, one AnchorRec16 per anchor (= walk).  The walks climb their trees level by level without the
// host: per level one kernel computes every waiting walk's window (compute_reference_span_start_and_length,
// verification.cpp:157-184, extra length 0) and elects per (node, strand) the walk with the rightmost window start; the
// elected ones become engine tasks (per configuration class, in one array: class c starts where the active walks of the
// classes before it would end); after the engine ran, the others take the elected walk's answer where it carries over,
// or become tasks of a second / third engine launch; a last kernel moves the survivors to their parent node.  Then
// decide_kernel settles, per read and strand in anchor order, which walks count and which verify their root -- the
// interval optimisation's sequential rule (verification.cpp:119-136) included -- and sums the statistics per member
// job; the walks that verify their root are handed to the host as a list.  The host only enqueues kernels (the engine
// reads its task counts from device memory) and synchronises once, before the root level.
// ---------------------------------------------------------------------------------------------
struct NodeRec {                       // an inner node of a read's tree
    uint32_t from, m, k;               // query_index_from, piece length, num_errors
    uint16_t parent;                   // inner index of the parent within the read's tree (unused for the root)
    uint8_t depth;                     // hops to the root
    uint8_t cls;                       // configuration class of its score passes
};
struct LeafRec { uint32_t from; uint32_t parent; };          // query_index_from, inner index of the parent (kNoParent: none)
struct AnchorRec16 { uint64_t reference_position; uint32_t pex_leaf_index; uint32_t reference_id; };   // search::anchor_t without num_errors
struct ReadRec {                       // 64 bytes; bases are relative to the job until gather_reads_kernel shifts them
    uint32_t walk_begin;               // first walk (= anchor) of the read
    uint32_t n_forward;                // its forward anchors come first
    uint32_t node_base, leaf_base;     // where the read's NodeRecs / LeafRecs begin
    uint64_t qoff_forward, qoff_reverse;   // pool position of query[0] per orientation
    uint32_t root_from, root_m, root_k;    // the root node
    uint32_t root_extra;               // ceil_eps((m + 2k + 1) * extra_verification_ratio), verification.cpp:165-166
    uint32_t member;                   // member job the read belongs to (statistics are kept per member)
    uint32_t n_walks;                  // forward + reverse anchors
    uint32_t reserved0, reserved1;
};
struct WalkRec {
    int64_t diag;                      // anchor position - first query index of its leaf (reference coordinates)
    uint64_t qoff;                     // pool position of query[0] in the walk's orientation
    uint32_t node;                     // first node to align (index into the batch's NodeRec array), or kDeadNode / kAtRootNode
    uint32_t node_base;                // where the read's NodeRecs begin
    uint32_t ref_id;
    uint32_t orient;
};
constexpr uint32_t kDeadNode = 0xffffffffu;        // the walk failed at an inner level
constexpr uint32_t kAtRootNode = 0xfffffffeu;      // the walk starts at its root: nothing to do below it
constexpr uint32_t kNoParent = 0xffffffffu;
constexpr int kWalkBits = 28;                       // a walk's index shares a 64-bit word with its window start (a store position below 2^36)
constexpr uint32_t kMaxDeviceWalks = 1u << kWalkBits;
constexpr unsigned long long kWalkMask = (1ull << kWalkBits) - 1;
constexpr int kMaxLevelClasses = 32;             // configuration classes of a context (a bit each in the per-depth masks)

// a member job's ReadRecs copied into the batch, bases shifted to the member's place in it
__global__ void gather_reads_kernel(const ReadRec* __restrict__ src, ReadRec* __restrict__ dst, uint32_t n, uint32_t walk0, uint32_t node0,
                                    uint32_t leaf0, uint64_t pool_shift, uint32_t member) {
    uint32_t const i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    ReadRec r = src[i];
    r.walk_begin += walk0; r.node_base += node0; r.leaf_base += leaf0;
    r.qoff_forward += pool_shift; r.qoff_reverse += pool_shift; r.member = member;
    dst[i] = r;
}

// last read with walk_begin <= i
__device__ __forceinline__ uint32_t read_of_walk(const ReadRec* __restrict__ reads, uint32_t n_reads, uint32_t i) {
    uint32_t lo = 0, hi = n_reads;
    while (hi - lo > 1) { uint32_t const mid = (lo + hi) >> 1; if (reads[mid].walk_begin <= i) lo = mid; else hi = mid; }
    return lo;
}

// The walk records from the anchors: the first node of a walk is its leaf's parent (verification.cpp:66-70), or the root
// itself for direct_full_verification (verification.cpp:23-42) and for leaves that hang off the root.
__global__ void walk_init_kernel(const AnchorRec16* __restrict__ anchors, const ReadRec* __restrict__ reads, uint32_t n_reads,
                                 const LeafRec* __restrict__ leaves, WalkRec* __restrict__ walks, uint32_t* __restrict__ node, uint32_t n_walks,
                                 uint32_t direct) {
    uint32_t const i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_walks) return;
    ReadRec const R = reads[read_of_walk(reads, n_reads, i)];
    AnchorRec16 const A = anchors[i];
    LeafRec const L = leaves[R.leaf_base + A.pex_leaf_index];
    uint32_t const orient = i - R.walk_begin >= R.n_forward ? 1u : 0u;
    WalkRec w;
    w.diag = int64_t(A.reference_position) - int64_t(L.from);
    w.qoff = orient ? R.qoff_reverse : R.qoff_forward;
    w.node_base = R.node_base; w.ref_id = A.reference_id; w.orient = orient;
    w.node = (!direct && L.parent != kNoParent && L.parent != 0) ? R.node_base + L.parent : kAtRootNode;      // inner[0] is the root
    walks[i] = w;
    node[i] = w.node;
}

struct LevelCtx {
    const WalkRec* walks; const NodeRec* nodes; uint32_t n_walks;
    const uint64_t* ref_base; const uint64_t* ref_len;
    uint32_t* node;                    // per walk: node to align next
    uint64_t* ask_ws; uint32_t* ask_len; uint8_t* flag;
    unsigned long long* rep;           // per (node, strand): (window start << kWalkBits | walk) of the elected walk, 0 = none
    unsigned long long* rep_min;       // the same for the walk with the leftmost window start (all ones = none)
    uint32_t* n_inner; uint64_t* sum_inner; uint64_t* cells_inner;     // statistics per walk, verification.cpp:238-242
    DpTask* tasks;                     // one array for all classes: class c begins at class_active[0] + .. + class_active[c-1]
    uint32_t* counts;                  // tasks appended per class by the phase at hand
    uint32_t* class_active;            // walks per class that wait at this level (set by level_begin_kernel)
    const DpResult* results;           // per walk
    unsigned long long* totals;        // [0] engine tasks, [1] their word-steps, [2] answers inferred
    uint32_t level, infer;
    uint8_t cls_W[kMaxLevelClasses];   // block width of every class (for the word-step count)
};
enum : uint8_t { kWalkActive = 1, kWalkComputed = 2, kWalkYes = 4, kWalkAsksLeftmost = 8 };

__device__ __forceinline__ uint32_t class_offset(const uint32_t* __restrict__ class_active, uint32_t cls) {
    uint32_t o = 0;
    for (uint32_t c = 0; c < cls; ++c) o += class_active[c];
    return o;
}

// Counters that every thread of a kernel bumps are bumped once per warp: tens of millions of atomics on one address
// (one per false-positive anchor of a config-4 batch) would otherwise take longer than the alignments themselves.
// Both may be called from divergent code: the lanes that arrive together share one atomic.
__device__ __forceinline__ void warp_add(unsigned long long* addr, unsigned long long v) {          // v < 2^50
    unsigned const active = __activemask();
    unsigned const lo = __reduce_add_sync(active, unsigned(v & 0xffffffu)), hi = __reduce_add_sync(active, unsigned(v >> 24));
    if ((threadIdx.x & 31u) == unsigned(__ffs(int(active)) - 1)) atomicAdd(addr, (unsigned long long)lo + ((unsigned long long)hi << 24));
}
__device__ __forceinline__ void warp_add_keyed(unsigned long long* base, uint32_t stride, uint32_t key, unsigned long long v) {   // base[key * stride] += v
    unsigned const active = __activemask();
    unsigned const peers = __match_any_sync(active, key);
    unsigned const lo = __reduce_add_sync(peers, unsigned(v & 0xffffffu)), hi = __reduce_add_sync(peers, unsigned(v >> 24));
    if ((threadIdx.x & 31u) == unsigned(__ffs(int(peers)) - 1)) atomicAdd(base + size_t(key) * stride, (unsigned long long)lo + ((unsigned long long)hi << 24));
}
__device__ __forceinline__ uint32_t warp_slot(uint32_t* counters, uint32_t key) {                  // atomicAdd(counters + key, 1), one atomic per key and warp
    unsigned const active = __activemask();
    unsigned const peers = __match_any_sync(active, key);
    unsigned const lane = threadIdx.x & 31u;
    int const leader = __ffs(int(peers)) - 1;
    uint32_t base = 0;
    if (int(lane) == leader) base = atomicAdd(counters + key, uint32_t(__popc(peers)));
    base = __shfl_sync(peers, base, leader);
    return base + uint32_t(__popc(peers & ((1u << lane) - 1u)));
}

__device__ __forceinline__ void emit_level_task(LevelCtx const& C, uint32_t i, NodeRec const& N, uint64_t qoff) {
    uint32_t const slot = class_offset(C.class_active, N.cls) + warp_slot(C.counts, N.cls);
    DpTask t;
    t.ref_base = C.ask_ws[i]; t.query_base = qoff + N.from; t.trace_base = 0;
    t.n = C.ask_len[i]; t.m = N.m; t.dlo = -int32_t(N.k); t.dhi = int32_t(t.n) - int32_t(N.m) + int32_t(N.k);
    t.flags = 0; t.out = i;
    C.tasks[slot] = t;
    // word-steps the engine issues for it (host: word_steps_of): block b works on columns cs(b)..ce(b)
    uint32_t const W = C.cls_W[N.cls], rows = 32 * W, nb = W ? (N.m + rows - 1) / rows : 0;
    int64_t const pad = int64_t(nb) * rows - N.m;
    unsigned long long ws = 0;
    for (uint32_t b = 0; b < nb; ++b) {
        int64_t lo = int64_t(rows) * b + 1 + t.dlo - pad, hi = int64_t(rows) * (b + 1) + t.dhi - pad;
        if (lo < 1) lo = 1;
        if (hi > int64_t(t.n)) hi = t.n;
        if (hi >= lo) ws += (unsigned long long)(hi - lo + 1) * W;
    }
    warp_add(C.totals, 1ull);
    warp_add(C.totals + 1, ws);
}

__global__ void level_begin_kernel(LevelCtx const C) {
    uint32_t const i = blockIdx.x * blockDim.x + threadIdx.x;
    uint8_t f = 0;
    uint32_t cls = 0xffu;
    if (i < C.n_walks) {
        uint32_t const nd = C.node[i];
        if (nd < kAtRootNode) {
            NodeRec const N = C.nodes[nd];
            if (N.depth == C.level) {
                WalkRec const Wk = C.walks[i];
                int64_t const s = Wk.diag + int64_t(N.from) - int64_t(N.k);
                uint64_t const offset = s >= 0 ? uint64_t(s) : 0;
                uint64_t const base = uint64_t(N.m) + 2ull * N.k + 1;
                uint64_t const room = C.ref_len[Wk.ref_id] - offset;
                uint64_t const len = base < room ? base : room;
                C.n_inner[i] += 1; C.sum_inner[i] += len; C.cells_inner[i] += uint64_t(N.m) * len;
                if (int64_t(N.m) - int64_t(len) > int64_t(N.k)) {
                    C.node[i] = kDeadNode;                   // more insertions needed than errors allowed: no alignment
                } else {
                    uint64_t const ws = C.ref_base[Wk.ref_id] + offset;
                    C.ask_ws[i] = ws; C.ask_len[i] = uint32_t(len);
                    f = kWalkActive;
                    cls = N.cls;
                    if (C.infer) {
                        atomicMax(C.rep + (size_t(nd) * 2 + Wk.orient), (unsigned long long)((ws << kWalkBits) | i));
                        atomicMin(C.rep_min + (size_t(nd) * 2 + Wk.orient), (unsigned long long)((ws << kWalkBits) | i));
                    }
                }
            }
        }
        C.flag[i] = f;
    }
    // walks per class (the classes share one task array), one atomic per class and warp
    uint32_t const peers = __match_any_sync(0xffffffffu, cls);
    if (cls != 0xffu && (threadIdx.x & 31u) == uint32_t(__ffs(int(peers)) - 1)) atomicAdd(C.class_active + cls, uint32_t(__popc(peers)));
}

__global__ void level_first_kernel(LevelCtx const C) {
    uint32_t const i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= C.n_walks || !(C.flag[i] & kWalkActive)) return;
    uint32_t const nd = C.node[i];
    WalkRec const Wk = C.walks[i];
    if (C.infer && uint32_t(C.rep[size_t(nd) * 2 + Wk.orient] & kWalkMask) != i) return;
    emit_level_task(C, i, C.nodes[nd], Wk.qoff);
    C.flag[i] |= kWalkComputed;
}

// After the elected walks (rightmost window start per node and strand) have their answers.  A = the elected walk's
// window, B = this walk's (B starts at or before A, both on the same reference or nothing is inferred):
//  * A holds an alignment: B holds it too if it is A's window or ends at or after the alignment's end; else B is computed;
//  * A holds none: neither does the same window.  Otherwise let C be the node's leftmost window.  If A and C start at most
//    k + 1 apart, every alignment inside B (at most m + k columns, starting at or after C's start) lies inside A (when it
//    starts at or after A's start: B ends at or before A) or inside C (when it starts before A's start: it ends before
//    A.start + m + k <= C.start + m + 2k + 1 = C's end, or C is clipped by the reference's end and B with it) -- so C is
//    computed, and the others wait for its answer (level_third_kernel); if the windows spread further, B is computed.
__global__ void level_second_kernel(LevelCtx const C) {
    uint32_t const i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= C.n_walks) return;
    uint8_t const f = C.flag[i];
    if (!(f & kWalkActive) || (f & kWalkComputed)) return;
    uint32_t const nd = C.node[i];
    NodeRec const N = C.nodes[nd];
    WalkRec const Wk = C.walks[i];
    size_t const key = size_t(nd) * 2 + Wk.orient;
    uint32_t const a = uint32_t(C.rep[key] & kWalkMask);
    DpResult const R = C.results[a];
    bool const a_yes = R.score <= int32_t(N.k);
    uint64_t const ws = C.ask_ws[i]; uint32_t const len = C.ask_len[i];
    if (ws == C.ask_ws[a] && len == C.ask_len[a]) { if (a_yes) C.flag[i] = f | kWalkYes; return; }                           // the same window
    bool const same_ref = C.walks[a].ref_id == Wk.ref_id;
    if (a_yes) {
        if (same_ref && ws + len >= C.ask_ws[a] + R.end_col) { C.flag[i] = f | kWalkYes; warp_add(C.totals + 2, 1ull); return; }
    } else if (same_ref) {
        uint32_t const c = uint32_t(C.rep_min[key] & kWalkMask);
        if (C.walks[c].ref_id == Wk.ref_id && C.ask_ws[a] - C.ask_ws[c] <= uint64_t(N.k) + 1) {
            if (i != c) { C.flag[i] = f | kWalkAsksLeftmost; return; }
        }
    }
    emit_level_task(C, i, N, Wk.qoff);
    C.flag[i] = f | kWalkComputed;
}

// After the leftmost windows have their answers: none there either means none in between (see above); an alignment there
// carries over to B if it is the same window or the alignment provably lies inside B; what is left is computed.
__global__ void level_third_kernel(LevelCtx const C) {
    uint32_t const i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= C.n_walks) return;
    uint8_t const f = C.flag[i];
    if (!(f & kWalkAsksLeftmost)) return;
    uint32_t const nd = C.node[i];
    NodeRec const N = C.nodes[nd];
    WalkRec const Wk = C.walks[i];
    uint32_t const c = uint32_t(C.rep_min[size_t(nd) * 2 + Wk.orient] & kWalkMask);
    DpResult const R = C.results[c];
    if (R.score > int32_t(N.k)) { warp_add(C.totals + 2, 1ull); return; }                    // no alignment in A, none in C: none in B
    uint64_t const ws = C.ask_ws[i]; uint32_t const len = C.ask_len[i];
    uint64_t const end = C.ask_ws[c] + R.end_col;                                             // exclusive end of C's alignment
    if ((ws == C.ask_ws[c] && len == C.ask_len[c]) ||
        (end <= ws + len && int64_t(end) - int64_t(N.m) - int64_t(R.score) >= int64_t(ws))) {
        C.flag[i] = f | kWalkYes; warp_add(C.totals + 2, 1ull); return;
    }
    emit_level_task(C, i, N, Wk.qoff);
    C.flag[i] = f | kWalkComputed;
}

__global__ void level_advance_kernel(LevelCtx const C) {
    uint32_t const i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= C.n_walks) return;
    uint8_t const f = C.flag[i];
    if (!(f & kWalkActive)) return;
    uint32_t const nd = C.node[i];
    NodeRec const N = C.nodes[nd];
    bool const yes = (f & kWalkComputed) ? C.results[i].score <= int32_t(N.k) : (f & kWalkYes) != 0;
    C.node[i] = yes ? C.walks[i].node_base + N.parent : kDeadNode;      // pex_tree::get_parent_of_child, pex.cpp:70-76
}

// ---------------------------------------------------------------------------------------------
// Which walks count, and which of them verify their root (verification.cpp:45-71, 106-109, 119-136).
//
// One warp per (read, strand), walks in anchor order -- the order of the reference's anchor loop
// (parallelization.cpp:230-249).  Without the interval optimisation every walk counts and every walk that stands at its
// root verifies it.  With it, a walk whose root window, trimmed by the extra length on both sides
// (half_open_interval::trim_from_both_sides, intervals.cpp:48-58), lies inside the root window of an EARLIER walk of the
// same reference that reached its root (and was not avoided itself) is avoided: its inner alignments, computed
// speculatively, do not count, and it verifies nothing (root_was_already_verified, verification.cpp:119-136; the
// window is inserted whenever the root is reached, even if the root alignment then fails, :106-109).  Whether a walk
// reaches its root depends on its inner alignments alone, so this one pass decides everything.
// The windows inserted so far sit in registers (one per lane); beyond 32 they spill to `inserted` (walk indices).
// ---------------------------------------------------------------------------------------------
struct DecideCtx {
    const WalkRec* walks; const uint32_t* node; const ReadRec* reads; uint32_t n_reads;
    const uint64_t* ref_len;
    const uint32_t* n_inner; const uint64_t* sum_inner; const uint64_t* cells_inner;
    uint8_t* root_flag;                // out, per walk: 1 = verifies its root
    uint32_t* root_count;              // out, per (read, strand): how many do
    uint32_t* inserted;                // scratch, one entry per walk
    unsigned long long* member_totals; // per member: n_aligned_inner, sum_aligned_inner, cells_inner, n_avoided_root, sum_avoided_root, 3 spare
    uint32_t ivopt;
};
constexpr int kMemberTotals = 8;

// root window of a walk: [start, start + len) in its reference's coordinates (compute_reference_span_start_and_length)
__device__ __forceinline__ void root_window(ReadRec const& R, int64_t diag, uint64_t ref_len, uint64_t& start, uint64_t& len) {
    uint64_t const base = uint64_t(R.root_m) + 2ull * R.root_k + 1;
    int64_t const s = diag + int64_t(R.root_from) - int64_t(R.root_k) - int64_t(R.root_extra);
    start = s >= 0 ? uint64_t(s) : 0;
    uint64_t const full = base + 2ull * R.root_extra, room = ref_len - start;
    len = full < room ? full : room;
}

__global__ void decide_kernel(DecideCtx const C) {
    uint32_t const lane = threadIdx.x & 31u;
    uint32_t const pair = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;          // (read, strand)
    if (pair >= 2 * C.n_reads) return;
    ReadRec const R = C.reads[pair >> 1];
    uint32_t const orient = pair & 1u;
    uint32_t const w0 = R.walk_begin + (orient ? R.n_forward : 0u);
    uint32_t const w1 = orient ? R.walk_begin + R.n_walks : R.walk_begin + R.n_forward;
    uint32_t n_ins = 0, n_root = 0;
    uint32_t ins_ref = 0; uint64_t ins_start = 0, ins_end = 0;                    // entry `lane` of the inserted windows
    unsigned long long s_n = 0, s_sum = 0, s_cells = 0, s_av = 0, s_avsum = 0;
    for (uint32_t base = w0; base < w1; base += 32) {
        uint32_t const i = base + lane;
        bool const have = i < w1;
        uint32_t ref = 0; uint64_t rs = 0, len = 0; bool reached = false;
        if (have) {
            WalkRec const Wk = C.walks[i];
            ref = Wk.ref_id;
            root_window(R, Wk.diag, C.ref_len[ref], rs, len);
            reached = C.node[i] != kDeadNode;
        }
        uint64_t const re = rs + len;
        // trimmed by the extra length on both sides (intervals.cpp:48-58)
        uint64_t const e0 = R.root_extra > re ? 0 : re - R.root_extra;
        uint64_t const te = e0 > rs + 1 ? e0 : rs + 1;
        uint64_t const ts = te - 1 < rs + R.root_extra ? te - 1 : rs + R.root_extra;
        bool my_avoided = false, my_root = false;
        uint32_t const n_here = min(32u, w1 - base);
        for (uint32_t q = 0; q < n_here; ++q) {
            uint32_t const q_ref = __shfl_sync(0xffffffffu, ref, q);
            uint64_t const q_rs = __shfl_sync(0xffffffffu, rs, q), q_re = __shfl_sync(0xffffffffu, re, q);
            uint64_t const q_ts = __shfl_sync(0xffffffffu, ts, q), q_te = __shfl_sync(0xffffffffu, te, q);
            bool const q_reached = __shfl_sync(0xffffffffu, int(reached), q) != 0;
            bool avoided = false;
            if (C.ivopt) {
                bool hit = lane < min(n_ins, 32u) && ins_ref == q_ref && ins_start <= q_ts && ins_end >= q_te;
                for (uint32_t e = 32 + lane; e < n_ins; e += 32) {
                    WalkRec const Wi = C.walks[C.inserted[w0 + e]];
                    uint64_t is, il;
                    root_window(R, Wi.diag, C.ref_len[Wi.ref_id], is, il);
                    hit |= Wi.ref_id == q_ref && is <= q_ts && is + il >= q_te;
                }
                avoided = __any_sync(0xffffffffu, hit);
            }
            if (avoided) {
                if (lane == q) my_avoided = true;
            } else if (q_reached) {
                if (lane == q) my_root = true;
                if (C.ivopt) {
                    if (n_ins < 32) { if (lane == n_ins) { ins_ref = q_ref; ins_start = q_rs; ins_end = q_re; } }
                    else { if (lane == 0) C.inserted[w0 + n_ins] = base + q; __syncwarp(); }
                    ++n_ins;
                }
                ++n_root;
            }
        }
        if (have) {
            C.root_flag[i] = my_root ? 1 : 0;
            if (my_avoided) { s_av += 1; s_avsum += len; }
            else { s_n += C.n_inner[i]; s_sum += C.sum_inner[i]; s_cells += C.cells_inner[i]; }
        }
    }
    for (int off = 16; off > 0; off >>= 1) {
        s_n += __shfl_down_sync(0xffffffffu, s_n, off); s_sum += __shfl_down_sync(0xffffffffu, s_sum, off);
        s_cells += __shfl_down_sync(0xffffffffu, s_cells, off); s_av += __shfl_down_sync(0xffffffffu, s_av, off);
        s_avsum += __shfl_down_sync(0xffffffffu, s_avsum, off);
    }
    if (lane == 0) {
        C.root_count[pair] = n_root;
        unsigned long long* const T = C.member_totals + size_t(R.member) * kMemberTotals;
        if (s_n | s_sum | s_cells) { atomicAdd(T + 0, s_n); atomicAdd(T + 1, s_sum); atomicAdd(T + 2, s_cells); }
        if (s_av) { atomicAdd(T + 3, s_av); atomicAdd(T + 4, s_avsum); }
    }
}

// exclusive prefix sums of `counts` (one CTA; n is the number of (read, strand) pairs of a batch); total -> *total
__global__ void scan_counts_kernel(const uint32_t* __restrict__ counts, uint32_t* __restrict__ offsets, uint32_t n, uint32_t* __restrict__ total) {
    __shared__ uint32_t warp_sums[32];
    __shared__ uint32_t carry;
    uint32_t const lane = threadIdx.x & 31u, wid = threadIdx.x >> 5;
    if (threadIdx.x == 0) carry = 0;
    __syncthreads();
    for (uint32_t base = 0; base < n; base += blockDim.x) {
        uint32_t const i = base + threadIdx.x;
        uint32_t const v = i < n ? counts[i] : 0u;
        uint32_t x = v;
        for (int off = 1; off < 32; off <<= 1) { uint32_t const y = __shfl_up_sync(0xffffffffu, x, off); if (lane >= uint32_t(off)) x += y; }
        if (lane == 31) warp_sums[wid] = x;
        __syncthreads();
        if (wid == 0) {
            uint32_t s = lane < (blockDim.x >> 5) ? warp_sums[lane] : 0u;
            for (int off = 1; off < 32; off <<= 1) { uint32_t const y = __shfl_up_sync(0xffffffffu, s, off); if (lane >= uint32_t(off)) s += y; }
            warp_sums[lane] = s;                                       // inclusive sums of the warps
        }
        __syncthreads();
        uint32_t const before = carry + (wid ? warp_sums[wid - 1] : 0u);
        if (i < n) offsets[i] = before + x - v;
        __syncthreads();
        if (threadIdx.x == blockDim.x - 1) carry = before + x;
        __syncthreads();
    }
    if (threadIdx.x == 0) *total = carry;
}

// the walks that verify their root, in walk order
struct RootEntry { int64_t diag; uint32_t walk; uint32_t ref_id; };
__global__ void root_emit_kernel(DecideCtx const C, const uint32_t* __restrict__ offsets, RootEntry* __restrict__ out) {
    uint32_t const lane = threadIdx.x & 31u;
    uint32_t const pair = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (pair >= 2 * C.n_reads) return;
    if (C.root_count[pair] == 0) return;
    ReadRec const R = C.reads[pair >> 1];
    uint32_t const orient = pair & 1u;
    uint32_t const w0 = R.walk_begin + (orient ? R.n_forward : 0u);
    uint32_t const w1 = orient ? R.walk_begin + R.n_walks : R.walk_begin + R.n_forward;
    uint32_t at = offsets[pair];
    for (uint32_t base = w0; base < w1; base += 32) {
        uint32_t const i = base + lane;
        bool const is_root = i < w1 && C.root_flag[i] != 0;
        uint32_t const bal = __ballot_sync(0xffffffffu, is_root);
        if (is_root) {
            WalkRec const Wk = C.walks[i];
            RootEntry e; e.diag = Wk.diag; e.walk = i; e.ref_id = Wk.ref_id;
            out[at + __popc(bal & ((1u << lane) - 1u))] = e;
        }
        at += __popc(bal);
    }
}

// ---------------------------------------------------------------------------------------------
// Last-row minimum over a range of columns, from the checkpoint records of a score pass.
//
// Several root windows of one query piece that nearly coincide are scored by ONE pass over their union (host side:
// run_root_passes).  The records of the pass' last block hold the horizontal deltas of row m for every column the block
// worked on, and the pass reported one (value, column) of that row; so the values of row m at all those columns follow by
// summing deltas, and each member window gets the minimum over its own columns and the rightmost column attaining it
// (alignment.cpp:128-139 / the engine's `sc <= best`).  One thread per member window.
// ---------------------------------------------------------------------------------------------
struct RangeMinTask {
    uint64_t ck_base;                  // first word of the pass' checkpoint records
    uint32_t n, m; int32_t dlo, dhi;   // the pass
    uint32_t W;                        // its block width (words per lane)
    uint32_t col_from, col_to;         // the member's columns in the pass' numbering (1-based, inclusive)
    uint32_t unit;                     // the pass' slot in the engine's result array: the (value, column) it reported
    uint32_t out;
    uint32_t reserved;
};

__global__ void range_min_kernel(const RangeMinTask* __restrict__ tasks, uint32_t n_tasks, const uint32_t* __restrict__ ck_all,
                                 const DpResult* __restrict__ unit_results, DpResult* __restrict__ results) {
    uint32_t const id = blockIdx.x * blockDim.x + threadIdx.x;
    if (id >= n_tasks) return;
    RangeMinTask const T = tasks[id];
    DpResult const known = unit_results[T.unit];
    uint32_t const W = T.W, ROWS = 32 * W, RECW = ck_record_words(W), BO = W == 1 ? 2 : 2 * W;
    uint32_t const nb = (T.m + ROWS - 1) / ROWS, lb = nb - 1;
    uint32_t const pad = nb * ROWS - T.m;
    int32_t const dlo = T.dlo - int32_t(pad), dhi = T.dhi - int32_t(pad);
    int32_t const lo = int32_t(ROWS) * int32_t(lb) + 1 + dlo, hi = int32_t(ROWS) * int32_t(nb) + dhi;
    int32_t const cs = lo < 1 ? 1 : lo, ce = hi > int32_t(T.n) ? int32_t(T.n) : hi;       // columns the last block worked on
    uint32_t const ck_per_block = ck_records_per_block(int64_t(T.dhi) - int64_t(T.dlo) + 1, ROWS);
    uint32_t const q_first = uint32_t(cs + int32_t(lb) + 31) >> 5;
    const uint32_t* const recs = ck_all + T.ck_base + uint64_t(lb) * ck_per_block * RECW + BO;
    // deltas of step t (column t - lb): bit (t - 1) % 32 of record (t + 31) / 32
    auto rec_of = [&](uint32_t t) { return reinterpret_cast<const uint2*>(recs + uint64_t(((t + 31) >> 5) - q_first) * RECW); };
    // sum of the deltas of columns cs .. x (0 for x < cs)
    auto prefix = [&](int32_t x) -> int32_t {
        if (x < cs) return 0;
        uint32_t const t0 = uint32_t(cs) + lb, t1 = uint32_t(x) + lb;
        int32_t sum = 0;
        for (uint32_t q = (t0 + 31) >> 5; q <= (t1 + 31) >> 5; ++q) {
            uint2 const v = *rec_of(32 * (q - 1) + 1);
            uint32_t const first = 32 * (q - 1) + 1;                  // step of bit 0
            uint32_t mask = 0xffffffffu;
            if (t0 > first) mask &= 0xffffffffu << (t0 - first);
            if (t1 < first + 31) mask &= 0xffffffffu >> (first + 31 - t1);
            sum += __popc(v.x & mask) - __popc(v.y & mask);
        }
        return sum;
    };
    DpResult R; R.score = kNoScore; R.end_col = 0;
    int32_t const a = int32_t(T.col_from) > cs ? int32_t(T.col_from) : cs, b = int32_t(T.col_to) < ce ? int32_t(T.col_to) : ce;
    if (a <= b && known.score < kNoScore && int32_t(known.end_col) >= cs && int32_t(known.end_col) <= ce) {
        int32_t sc = known.score - prefix(int32_t(known.end_col)) + prefix(a - 1);        // row m at column a - 1
        uint2 v = make_uint2(0u, 0u);
        for (int32_t col = a; col <= b; ++col) {
            uint32_t const t = uint32_t(col) + lb, bit = (t - 1) & 31u;
            if (col == a || bit == 0) v = *rec_of(t);
            sc += int32_t((v.x >> bit) & 1u) - int32_t((v.y >> bit) & 1u);
            if (sc <= R.score) { R.score = sc; R.end_col = uint32_t(col); }
        }
    }
    results[T.out] = R;
}

// ---------------------------------------------------------------------------------------------
// int32 issue-rate microbenchmark: the 8 LOP3 : 1 IADD3 : 2 SHF mix of one Myers word-step,
// 8 independent chains per thread so that the pipes, not dependencies, limit the rate.
// ---------------------------------------------------------------------------------------------
__global__ void int32_peak_kernel(uint32_t* out, uint32_t iters, uint32_t seed) {
    uint32_t a[8], b2[8], c[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) { a[i] = seed + threadIdx.x * 7 + i; b2[i] = seed * 3 + i * 11 + blockIdx.x; c[i] = ~seed + i; }
    for (uint32_t it = 0; it < iters; ++it) {
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            uint32_t x = a[i], y = b2[i], z = c[i];
            uint32_t t0 = (x & y) | z;            // LOP3
            uint32_t t1 = (x ^ z) & ~y;           // LOP3
            uint32_t t2 = t0 + t1 + y;            // IADD3
            uint32_t t3 = (t2 ^ x) | t0;          // LOP3
            uint32_t t4 = y & t3;                 // LOP3
            uint32_t t5 = z | ~(y | t3);          // LOP3
            uint32_t t6 = __funnelshift_l(t4, t5, 1);   // SHF
            uint32_t t7 = __funnelshift_l(t5, t4, 1);   // SHF
            uint32_t t8 = t6 & t3;                // LOP3
            uint32_t t9 = t7 | ~(t6 | t3);        // LOP3
            uint32_t t10 = (t8 ^ t9) | t1;        // LOP3
            a[i] = t8; b2[i] = t9; c[i] = t10;
        }
    }
    uint32_t acc = 0;
#pragma unroll
    for (int i = 0; i < 8; ++i) acc ^= a[i] ^ b2[i] ^ c[i];
    if (acc == 0x12345678u) out[0] = acc;       // keep the result alive without a store in the common case
}

}  // namespace fxg
