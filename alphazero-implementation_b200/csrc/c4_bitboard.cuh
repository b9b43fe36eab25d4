// Connect4 (6x7, 4-in-line) rules on two 64-bit bitboards.
//
// Replaces the third-party `simulator.game.connect` State/Action calls the reference makes
// (SURVEY.md Appendix B): Action.sample_next_state() search.py:89 / node.py:38, State.actions
// models/games/connect4/model.py:29, State.has_ended node.py:63, State.reward node.py:68.
//
// Layout: bit index = column*7 + row, row 0 = bottom; each column owns 7 bits, the 7th (row 6)
// is a guard that stays zero so that shifted-AND line tests never wrap between columns.
#pragma once
#include <stdint.h>

#if defined(__CUDACC__)
#define C4_HD __host__ __device__ __forceinline__
#else
#define C4_HD static inline
#endif

namespace c4 {

constexpr int H = 6;
constexpr int W = 7;
constexpr int STRIDE = 7;  // bits per column
constexpr uint64_t TOP_ROW = 0x810204081020ull;     // bit (7c+5) for c = 0..6
constexpr uint64_t BOARD = 0xFDFBF7EFDFBFull;       // 6 playable cells of every column
constexpr uint64_t LEGAL_MAGIC = 0x1041041041ull;   // sum 2^(36-6c): gathers bits 7c -> bits 36+c

C4_HD uint64_t col_cells(int c) { return 0x3Full << (STRIDE * c); }

// 4-in-line anywhere in one player's stones: vertical (1), horizontal (7), diagonals (6, 8)
C4_HD bool has4(uint64_t b) {
    uint64_t m;
    m = b & (b >> 1);
    if (m & (m >> 2)) return true;
    m = b & (b >> 7);
    if (m & (m >> 14)) return true;
    m = b & (b >> 6);
    if (m & (m >> 12)) return true;
    m = b & (b >> 8);
    return (m & (m >> 16)) != 0;
}

// branch-free variant for divergent warp code
C4_HD bool has4_nb(uint64_t b) {
    uint64_t v = b & (b >> 1), h = b & (b >> 7), d1 = b & (b >> 6), d2 = b & (b >> 8);
    return ((v & (v >> 2)) | (h & (h >> 14)) | (d1 & (d1 >> 12)) | (d2 & (d2 >> 16))) != 0;
}

C4_HD bool is_full(uint64_t occ) { return (occ & TOP_ROW) == TOP_ROW; }

// State.actions as a 7-bit column mask of a NON-ended position: column legal iff its top cell is empty
C4_HD uint32_t legal_mask(uint64_t occ) {
    uint64_t t = (~occ & TOP_ROW) >> 5;  // bit 7c set iff column c has room
    return (uint32_t)((t * LEGAL_MAGIC) >> 36) & 0x7Fu;
}

// the cell a stone dropped in column c lands on (column must have room): carry of occ + bottom(c)
C4_HD uint64_t drop_bit(uint64_t occ, int c) { return (occ + (1ull << (STRIDE * c))) & col_cells(c); }

// c-th legal column in ascending order -> column index (idx < popcount(legal))
C4_HD int nth_legal_column(uint32_t legal, int idx) {
    int col = 0;
#pragma unroll
    for (int c = 0; c < W; ++c) {
        uint32_t below = legal & ((1u << c) - 1u);
        int rank = 0;
#if defined(__CUDA_ARCH__)
        rank = __popc(below);
#else
        rank = __builtin_popcount(below);
#endif
        if (((legal >> c) & 1u) && rank == idx) col = c;
    }
    return col;
}

// Left-right mirror of one player's stones: column c's 7 bits (bit 7c + r) move to column 6 - c.  A position and its mirror
// have the same value, and their policies are the same with the columns reversed; the side to move does not change.
C4_HD uint64_t mirror(uint64_t b) {
    constexpr uint64_t C0 = 0x7Full, C1 = C0 << 7, C2 = C0 << 14, C3 = C0 << 21;
    return (b & C3) | ((b & C0) << 42) | ((b >> 42) & C0) | ((b & C1) << 28) | ((b >> 28) & C1) | ((b & C2) << 14) |
           ((b >> 14) & C2);
}

// Canonical form of a position: the smaller of (b0, b1) and (mirror(b0), mirror(b1)) as unsigned 64-bit values, b0 first.
// `mirrored` is set only when the mirror was taken; a palindrome (its own mirror) is its own canonical form.
struct Canonical {
    uint64_t b0, b1;
    bool mirrored;
};
C4_HD Canonical canonical(uint64_t b0, uint64_t b1) {
    const uint64_t m0 = mirror(b0), m1 = mirror(b1);
    Canonical r;
    r.mirrored = m0 < b0 || (m0 == b0 && m1 < b1);
    r.b0 = r.mirrored ? m0 : b0;
    r.b1 = r.mirrored ? m1 : b1;
    return r;
}

// has_ended / reward of an arbitrary position (root states handed in by the caller):
// winner = whoever owns a 4-in-line (player 0 tested first), else draw iff board full.
struct Terminal {
    bool ended;
    int8_t reward0;  // reward of player 0; player 1 gets the negation (+1 win / -1 loss / 0 draw)
};
C4_HD Terminal terminal_of(uint64_t b0, uint64_t b1) {
    Terminal t;
    bool w0 = has4(b0), w1 = has4(b1);
    t.ended = w0 || w1 || is_full(b0 | b1);
    t.reward0 = w0 ? 1 : (w1 ? -1 : 0);
    return t;
}


// ---- the same rules on the two 32-bit halves of a board, for the streaming rules kernels (k_env_step_h / k_state_info_h).
// On sm_100 the integer work of a kernel is split over two issue pipes of 64 lanes / clk / SM each: shifts and logic ops (SHF,
// LOP3, IADD3, SEL) on the ALU pipe, integer multiply-adds (IMAD, IMAD.HI) on the FMA pipe.  The 64-bit formulation above
// compiles to ALU-pipe instructions only and that pipe, not HBM, bounds the kernels (DESIGN.md 3a).  Here the 4-in-line test
// shifts LEFT, the low word by a multiplication with a power of two (FMA pipe), the high word by one funnel shift (ALU pipe) or
// by a multiply-add on a mulhi (FMA pipe), and the byte packing / unpacking around it uses multiply-adds and byte permutes.
namespace h32 {

constexpr uint32_t TOP_LO = 0x04081020u, TOP_HI = 0x8102u;          // TOP_ROW
constexpr uint32_t BOARD_LO = 0xF7EFDFBFu, BOARD_HI = 0xFDFBu;      // BOARD

C4_HD uint32_t mulhi_u32(uint32_t a, uint32_t b) {
#if defined(__CUDA_ARCH__)
    uint32_t r;
    asm("mul.hi.u32 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(b));
    return r;
#else
    return (uint32_t)(((uint64_t)a * (uint64_t)b) >> 32);
#endif
}
C4_HD uint32_t mad_u32(uint32_t a, uint32_t b, uint32_t c) {
#if defined(__CUDA_ARCH__)
    uint32_t r;
    asm("mad.lo.u32 %0, %1, %2, %3;" : "=r"(r) : "r"(a), "r"(b), "r"(c));
    return r;
#else
    return a * b + c;
#endif
}
// PTX shl.b32: amounts above 31 give 0 (C++ leaves them undefined)
C4_HD uint32_t shl_clamp(uint32_t a, uint32_t s) {
#if defined(__CUDA_ARCH__)
    uint32_t r;
    asm("shl.b32 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(s));
    return r;
#else
    return s > 31u ? 0u : a << s;
#endif
}

// (hi:lo) >> S for a constant 1 <= S <= 31 (two ALU-pipe shifts)
template <int S>
C4_HD void shr64(uint32_t lo, uint32_t hi, uint32_t &olo, uint32_t &ohi) {
    olo = (lo >> S) | (hi << (32 - S));
    ohi = hi >> S;
}

// (hi:lo) << S for a constant 1 <= S <= 31: the low word as a multiplication (FMA pipe); the high word as one funnel shift (ALU
// pipe) or, HM, as hi * 2^S + mulhi(lo, 2^S) (FMA pipe, the mulhi at about a third of a multiply-add's rate)
template <int S, bool HM>
C4_HD void shl64(uint32_t lo, uint32_t hi, uint32_t &olo, uint32_t &ohi) {
    olo = mad_u32(lo, 1u << S, 0u);
    if (HM) {
        ohi = mad_u32(hi, 1u << S, mulhi_u32(lo, 1u << S));
    } else {
#if defined(__CUDA_ARCH__)
        ohi = __funnelshift_l(lo, hi, S);
#else
        ohi = (hi << S) | (lo >> (32 - S));
#endif
    }
}
// the same test with left shifts: stones at p, p - S, p - 2 S, p - 3 S (bits shifted out of the 64 belong to no cell)
template <int S, bool HM>
C4_HD void line4_l(uint32_t lo, uint32_t hi, uint32_t &rlo, uint32_t &rhi) {
    uint32_t al, ah, bl, bh;
    shl64<S, HM>(lo, hi, al, ah);
    const uint32_t ml = lo & al, mh = hi & ah;
    shl64<2 * S, HM>(ml, mh, bl, bh);
    rlo |= ml & bl;
    rhi |= mh & bh;
}
// (hi:lo) + (bhi:blo)
C4_HD void add64(uint32_t lo, uint32_t hi, uint32_t blo, uint32_t bhi, uint32_t &olo, uint32_t &ohi) {
#if defined(__CUDA_ARCH__)
    asm("add.cc.u32 %0, %2, %3;\n\taddc.u32 %1, %4, %5;" : "=&r"(olo), "=r"(ohi) : "r"(lo), "r"(blo), "r"(hi), "r"(bhi));  // & : written before hi / bhi are read
#else
    olo = lo + blo;
    ohi = hi + bhi + (olo < lo ? 1u : 0u);
#endif
}

// one direction of the 4-in-line test: stones at p, p + S, p + 2 S, p + 3 S
template <int S>
C4_HD void line4(uint32_t lo, uint32_t hi, uint32_t &rlo, uint32_t &rhi) {
    uint32_t al, ah, bl, bh;
    shr64<S>(lo, hi, al, ah);
    const uint32_t ml = lo & al, mh = hi & ah;
    shr64<2 * S>(ml, mh, bl, bh);
    rlo |= ml & bl;
    rhi |= mh & bh;
}

// has4 of a board given as halves.  MODE >= 1: left shifts - low words on the FMA pipe, high words on the ALU pipe (MODE 1: 24 ALU
// + 8 FMA instructions) or, for MODE - 1 of the four directions, on the FMA pipe too (MODE 4, what the kernels run: 18 ALU + 20
// FMA); MODE 0: right shifts, everything on the ALU pipe (32), kept for the A/B.  (Right shifts as mulhi everywhere were
// measured too: IMAD.HI issues at about a third of IMAD's rate and the kernels got no faster.)
template <int MODE>
C4_HD bool has4(uint32_t lo, uint32_t hi) {
    uint32_t rlo = 0u, rhi = 0u;
    if (MODE >= 1) {  // MODE - 1 = directions whose high-word shifts run on the FMA pipe as well
        line4_l<1, (MODE >= 2)>(lo, hi, rlo, rhi);
        line4_l<7, (MODE >= 3)>(lo, hi, rlo, rhi);
        line4_l<6, (MODE >= 4)>(lo, hi, rlo, rhi);
        line4_l<8, (MODE >= 5)>(lo, hi, rlo, rhi);
    } else {
        line4<1>(lo, hi, rlo, rhi);
        line4<7>(lo, hi, rlo, rhi);
        line4<6>(lo, hi, rlo, rhi);
        line4<8>(lo, hi, rlo, rhi);
    }
    return (rlo | rhi) != 0u;
}

// State.actions of a non-ended position from t = ~occ & TOP_ROW (halves): two multiplications gather the top-row bits - bits
// 5 + 7 i of t_lo to bits 32 + i of the 64-bit product (all other partial products fall on bits 7.. of the high word or into
// the low word), bits 1 + 7 i of t_hi to bits 13 + i (the others on bits 1, 7, 8, 20, 21, 27)
C4_HD uint32_t legal_from_top(uint32_t t_lo, uint32_t t_hi) {
    return (mulhi_u32(t_lo, 0x08208200u) | (mad_u32(t_hi, 0x1041u, 0u) >> 9)) & 0x7Fu;
}

struct Info {
    uint32_t legal, ended, pair;  // 7-bit column mask (0 when ended), 0 / 1, reward bytes {player 0, player 1} as a 16-bit pair
};
// has_ended / reward / actions of an arbitrary position (terminal_of + legal_mask above)
template <int MODE>
C4_HD Info state_info(uint32_t lo0, uint32_t hi0, uint32_t lo1, uint32_t hi1) {
    const bool w0 = has4<MODE>(lo0, hi0), w1 = has4<MODE>(lo1, hi1);
    const uint32_t t_lo = ~(lo0 | lo1) & TOP_LO, t_hi = ~(hi0 | hi1) & TOP_HI;
    const bool ended = w0 || w1 || (t_lo | t_hi) == 0u;
    Info r;
    r.legal = ended ? 0u : legal_from_top(t_lo, t_hi);
    r.ended = ended ? 1u : 0u;
    r.pair = w0 ? 0xFF01u : (w1 ? 0x01FFu : 0u);  // {+1, -1} / {-1, +1} / {0, 0}
    return r;
}

struct Step {
    uint32_t lo0, hi0, lo1, hi1, status;  // the successor (the input when the move is refused), 0 = moved / 1 = refused
    Info info;
};
// Action.sample_next_state() with the checks of k_env_step: an ended position, a column >= 7 or a full column leave the state
// as it is (status 1).  `z` = all ones when player 1 is to move, 0 when player 0 is.  The stone lands on
// (occ + bottom(col)) & ~occ - the carry of the addition runs up the column's stones - and the move is legal iff that cell is
// one of the 42 (a full column carries into its guard bit, a column >= 7 into bits the board never uses or out of the word).
template <int MODE>
C4_HD Step env_step(uint32_t lo0, uint32_t hi0, uint32_t lo1, uint32_t hi1, uint32_t z, uint32_t col) {
    const bool w0 = has4<MODE>(lo0, hi0), w1 = has4<MODE>(lo1, hi1);
    const uint32_t olo = lo0 | lo1, ohi = hi0 | hi1;
    const uint32_t t_lo = ~olo & TOP_LO, t_hi = ~ohi & TOP_HI;
    const bool ended0 = w0 || w1 || (t_lo | t_hi) == 0u;
    const uint32_t blo = shl_clamp(1u, mad_u32(col, 7u, 0u)), bhi = shl_clamp(1u, mad_u32(col, 7u, 0xFFFFFFE0u));  // 1 << 7 col
    uint32_t slo, shi;
    add64(olo, ohi, blo, bhi, slo, shi);
    uint32_t nlo = slo & ~olo, nhi = shi & ~ohi;
    const bool valid = !ended0 && ((nlo & BOARD_LO) | (nhi & BOARD_HI)) != 0u;
    nlo = valid ? nlo : 0u;
    nhi = valid ? nhi : 0u;
    Step r;
    r.lo0 = lo0 | (nlo & ~z);
    r.hi0 = hi0 | (nhi & ~z);
    r.lo1 = lo1 | (nlo & z);
    r.hi1 = hi1 | (nhi & z);
    const bool win = has4<MODE>((r.lo0 & ~z) | (r.lo1 & z), (r.hi0 & ~z) | (r.hi1 & z)) && valid;  // the mover's stones
    const uint32_t u_lo = t_lo & ~nlo, u_hi = t_hi & ~nhi;  // empty top cells after the move
    const bool ended = valid ? (win || (u_lo | u_hi) == 0u) : ended0;
    r.status = valid ? 0u : 1u;
    r.info.legal = ended ? 0u : legal_from_top(u_lo, u_hi);
    r.info.ended = ended ? 1u : 0u;
    const uint32_t pair0 = w0 ? 0xFF01u : (w1 ? 0x01FFu : 0u);
    r.info.pair = valid ? (win ? (0xFF01u ^ (z & 0xFEFEu)) : 0u) : pair0;  // {+1, -1} when player 0 made the line, {-1, +1} when player 1 did
    return r;
}

// four player bytes (bit 0 = the player) -> per position a word of all ones (player 1) or zero: one multiplication puts the bit
// on the byte's sign, one byte permute per position replicates it
C4_HD uint32_t player_mask(uint32_t players_x80, int k) {
#if defined(__CUDA_ARCH__)
    uint32_t r;  // prmt: bit 3 of a selector nibble replicates the selected byte's sign (__byte_perm drops that bit)
    asm("prmt.b32 %0, %1, %2, %3;" : "=r"(r) : "r"(players_x80), "r"(0u), "r"(0x8888u + 0x1111u * (uint32_t)k));
    return r;
#else
    return ((players_x80 >> (8 * k + 7)) & 1u) ? 0xFFFFFFFFu : 0u;
#endif
}
C4_HD uint32_t byte_of(uint32_t w, int k) {
#if defined(__CUDA_ARCH__)
    return __byte_perm(w, 0u, 0x4440u + (uint32_t)k);
#else
    return (w >> (8 * k)) & 0xFFu;
#endif
}

}  // namespace h32

}  // namespace c4
