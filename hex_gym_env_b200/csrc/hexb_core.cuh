// hexb_core.cuh - per-game and per-word logic of the batched Hex simulator (sm_100a).
//
// Everything here is written against the REFERENCE SEMANTICS (MBPrdctns/hex_gym_env), cited as
// file:line relative to the reference root, but in a representation chosen for the B200:
//
//   * one TAGGED LABEL BYTE per cell, C bytes per game, in the AGENT'S PERSPECTIVE ("stored") coordinates:
//       0 = empty, else (region label & 0x7f) | (player << 7), player 0 = "R" (connects stored row 0
//       to row N-1; the agent), player 1 = "C" (connects stored col 0 to col N-1; the opponent).
//     It replaces the reference's board f64[N,N] plus regions f64[2,N+2,N+2] (HexGame.py:23,38-45,
//     HexSingleGame.py:27,42-49): the padded borders are implicit (near edge = label 1, far edge =
//     label 2 until that player connects, then 1) and a cell belongs to at most one player, so one
//     plane with a tag bit carries both region planes. Labels stay < 128 for N <= 19 (3 + the size
//     of an independent set of the hex adjacency graph on the interior rows).
//   * "stored" = true coordinates when the agent is BLACK, the transpose when the agent is WHITE
//     (the hex neighbourhood is symmetric under transposition), so the agent's observation, mask and
//     action index are the stored row-major order and never need a transpose on the hot path.
//   * a small per-game record (u32 words): the occupancy bitboard in stored row-major order,
//     counters, flags, RNG draw index. (The random opponent picks the k-th empty cell of ITS
//     perspective = stored column-major order, SelfplayWrapper.py:17-22, minihex/__init__.py:8-12:
//     select_kth_zero_colmajor finds it from the same bitboard.)
//   * games are stored chunk-major, 32 games (one warp) per contiguous block: their label bytes
//     [32][C], then their record words [word][lane] (see chunk_state_bytes below).
//
// The same source compiles for the device (hexb_kernels.cu) and, with HEXB_HOST_EMU defined, for the
// host-side emulator under tests/emu/ that replays the kernel phases serially. The emulator is test
// infrastructure; the product has no CPU path.
#pragma once
#include <stdint.h>

#if defined(__CUDACC__) && !defined(HEXB_HOST_EMU)
#define HEXB_HD __host__ __device__ __forceinline__
#else
#define HEXB_HD static inline
#endif

namespace hexb {

// ----------------------------------------------------------------------------------------------
// constants
// ----------------------------------------------------------------------------------------------
constexpr int kTile = 128;  // a shard's game count is padded to a multiple of this (4 chunks of 32 games), so 1, 2 or 4 warps per CTA all divide it

enum : int { VARIANT_A = 0, VARIANT_B = 1 };
enum : int { MODE_STEP = 0, MODE_RESET = 1, MODE_PLY = 2, MODE_HALF = 3 };

// meta word
constexpr uint32_t M_CTR_R_SHIFT = 0;   // bits 0-7   region_counter of R
constexpr uint32_t M_CTR_C_SHIFT = 8;   // bits 8-15  region_counter of C
constexpr uint32_t M_TOMOVE = 1u << 16;  // 1 = C to move (simulator.current_player_num in stored terms)
constexpr uint32_t M_DONE = 1u << 17;
constexpr uint32_t M_TRANSPOSED = 1u << 18;  // agent is true WHITE: stored = true^T, R = WHITE, C = BLACK
constexpr uint32_t M_FAR_R1 = 1u << 19;      // R's far border label has become 1 (R connected)
constexpr uint32_t M_FAR_C1 = 1u << 20;
constexpr uint32_t M_WIN_SHIFT = 21;         // bits 21-22: simulator.winner 0 none, 1 R, 2 C
constexpr uint32_t M_WIN_MASK = 3u << 21;
constexpr uint32_t M_INVALID = 1u << 23;      // the episode ended on an illegal agent move (winner == 3)
constexpr uint32_t M_COLOUR_SET = 1u << 24;   // SelfplayWrapper.py:72-73 ran (agent colour fixed for the env's lifetime)
constexpr uint32_t M_LIVE = 1u << 25;         // reset() has been called at least once
constexpr uint32_t M_AGENT_ENDED = 1u << 26;  // the agent's own ply ended the episode (terminal obs is the opponent's view)

// per-game scratch words handed from the thread-per-game phases to the cooperative byte passes
//   prm: bits 0-7 o1 (tagged), 8-15 o2 (tagged), 16-23 m (tagged), 24 need-relabel
constexpr uint32_t P_NEED = 1u << 24;
//   flg: bit 0 resetting, bit 1 output view is the opponent's (transposed+swapped), bit 2 has opening stone,
//        bit 3 emit terminal obs, bit 4 terminal view is the opponent's, bit 5 row needs the relabel sweep;
//        bits 8-15 opening byte, 16-31 opening cell
constexpr uint32_t F_RESET = 1u << 0;
constexpr uint32_t F_VIEW_OPP = 1u << 1;
constexpr uint32_t F_OPEN = 1u << 2;
constexpr uint32_t F_TERM = 1u << 3;
constexpr uint32_t F_TERM_OPP = 1u << 4;
constexpr uint32_t F_RELABEL = 1u << 5;
constexpr uint32_t F_ROWJOB = F_RESET | F_TERM | F_RELABEL;  // anything the warp has to sweep the row for

constexpr int ceil_log2(int n) { return n <= 1 ? 0 : 1 + ceil_log2((n + 1) / 2); }

template <int N>
struct Geo {
    static constexpr int C = N * N;
    static constexpr int W = (C + 31) / 32;      // bitboard words
    static constexpr int R = W + 2;              // record words: occ_rm[W], meta, draws
    static constexpr int CHUNK_LAB = 32 * C;               // label bytes of a chunk (multiple of 16)
    static constexpr int CHUNK_STATE = 32 * (C + 4 * R);   // whole chunk: labels + records (multiple of 16)
    static constexpr int COL_STEPS = ceil_log2(N);         // bisection steps over the columns (select_kth_zero_colmajor)
    static constexpr uint32_t LAST_MASK = (C % 32) ? ((1u << (C % 32)) - 1u) : 0xffffffffu;
};

template <int N>
struct Rec {
    uint32_t occ_rm[Geo<N>::W];   // occupancy bitboard, stored row-major order (bit y*N + x)
    uint32_t meta, draws;  // (plies of the running episode = stones on the board = popcount of the occupancy)
};

// Packed state, chunk-major: games are grouped in chunks of 32 (one warp); chunk k occupies CHUNK_STATE contiguous,
// 16-byte aligned bytes = the 32 games' label bytes [32][C] followed by their record words [R][32] (word-major so that lane
// i reads word w at [w*32 + i] without bank conflicts). One bulk copy moves a whole chunk.
HEXB_HD long long chunk_state_bytes(int C) { return 32ll * (C + 4 * ((C + 31) / 32 + 2)); }
HEXB_HD long long labels_offset(long long g, int C) { return (g >> 5) * chunk_state_bytes(C) + (g & 31) * C; }
HEXB_HD long long rec_offset(long long g, int C) { return (g >> 5) * chunk_state_bytes(C) + 32ll * C + 4 * (g & 31); }  // word w: + 128*w
constexpr int kRecStride = 32;  // words between consecutive record words of one game

struct Params {
    // packed state (owned by the handle)
    uint8_t *state;       // [Gpad/32] chunks of { labels u8[32][C], records u32[R][32] }
    long long *stats;     // [kStatStripes][8]
    long long G, Gpad, game_offset;
    unsigned long long seed;
    int variant, auto_reset, eval_state, opponent_first, agent_mode, mode;
    int raw;  // 1: bare HexGame batch (hexb_ply): reset draws nothing and nobody opens
    int steps;            // MODE_STEP: env steps per launch (hexb_rollout: T > 1 keeps the state on chip between steps; outputs [T,G,..])
    int manual_opponent;  // 1: the opponent's moves come from the caller (hexb_half_step); resets never play the opening move
    int half_side;        // MODE_HALF: 0 = the agent's ply, 1 = the opponent's ply
    int pool_size;        // setup_opponents: size of the opponent pool the index is drawn from
    int32_t *opp_index;   // [G] nullable: opponent chosen at reset, -1 = best model, k = pool entry (SelfplayWrapper.py:97-103)
    int32_t *eval_episode;  // [G] nullable: episodes started since SelfPlayEnv.set_eval (hexb_set_eval; SelfplayWrapper.py:93-95)
    double opp_eps;       // MODE_HALF, variant A, side 1 with caller actions: HexEnv.eps of opponent_predict (HexGame.py:354-359): one draw
                          // rv per opponent ply, rv < eps -> random_policy moves instead of the caller's action; < 0 = off
    uint8_t *to_move;     // [G] MODE_HALF / MODE_RESET out: 0 agent to move, 1 opponent to move, 2 finished
    int32_t *info_opp;    // [G] nullable, MODE_STEP out: the opponent's move of this step (info["last_move_opponent"]), -1 = none
    int8_t *info_winner;  // [G] nullable, MODE_STEP out: env.winner after the step: -1 None, 0 BLACK, 1 WHITE, 3 illegal move
    uint32_t enc_ka, enc_kb, enc_kc;   // observation bytes of a label word: obs = mask * ka + C-stones * kb + kc (enc_consts; per variant)
    long long keep_chunks;  // chunks [0, keep_chunks) are kept in L2 between steps (evict_last), the others streamed (evict_first)
    int early;     // 1: the record-only half of the env step (game_step_pre) runs on record words fetched with plain loads while
                   // the chunk's bulk copy is still in flight (set per launch: pays for launches of at most one wave)
    uint32_t one;  // always 1, but opaque to the compiler: a * one + b is issued as IMAD on the FMA pipe (see fma_add)
    int obs_f32;   // 1: obs / term_obs point to float32 buffers (hexb_config.obs_dtype = HEXB_OBS_F32: the reference's observation
                   // is a float array, HexSingleGame.py:175, and SB3's policies take float32), 0: int8
    // borrowed I/O (device pointers, any may be null unless noted)
    const int32_t *actions;    // [G]   null => sample the agent's move on device (one draw)
    const double *opp_u;       // [G,2] null => Philox stream
    const uint8_t *reset_mask;  // [G]   MODE_RESET: null => all
    const double *open_u;      // [G]   MODE_RESET: injected opening draw
    int8_t *obs;               // [G,N,N]
    uint8_t *mask;             // [G,C]
    float *reward;             // [G]
    uint8_t *done;             // [G]
    int8_t *term_obs;          // [G,N,N] written only for games that finished in this step
    int32_t *actions_out;      // [G]   the agent action actually played
    int8_t *ret;               // [G]   MODE_PLY: -1 none, 0 BLACK, 1 WHITE, 3 illegal
};

// ----------------------------------------------------------------------------------------------
// small helpers
// ----------------------------------------------------------------------------------------------
HEXB_HD int popc32(uint32_t v) {
#if defined(__CUDA_ARCH__)
    return __popc(v);
#else
    return __builtin_popcount(v);
#endif
}
HEXB_HD uint32_t mulhi32(uint32_t a, uint32_t b) {
#if defined(__CUDA_ARCH__)
    return __umulhi(a, b);
#else
    return (uint32_t)(((uint64_t)a * b) >> 32);
#endif
}
HEXB_HD uint32_t splat(uint32_t b) { return b * 0x01010101u; }
HEXB_HD uint32_t umin32(uint32_t a, uint32_t b) { return a < b ? a : b; }
// a + b issued as a multiply-add (IMAD, FMA pipe) instead of an add (IADD3 / VIADD, ALU pipe). `one` is Params::one: the
// step kernel is bound by the ALU pipe (LOP3 / SHF / PRMT / ISETP, rt 2 cycles per warp instruction and SMSP) while the FMA
// pipe idles, so the adds and shifts of the byte-SIMD loops are steered there.
HEXB_HD uint32_t fma_add(uint32_t a, uint32_t b, uint32_t one) { return a * one + b; }

// Philox4x32-10 (Random123); pinned by the Random123 known-answer vectors in tests/test_philox.py.
HEXB_HD void philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1, uint32_t &o0, uint32_t &o1) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint32_t hi0 = mulhi32(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
        const uint32_t hi1 = mulhi32(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
        c0 = hi1 ^ c1 ^ k0;
        c1 = lo1;
        c2 = hi0 ^ c3 ^ k1;
        c3 = lo0;
        k0 += 0x9E3779B9u;
        k1 += 0xBB67AE85u;
    }
    o0 = c0;
    o1 = c1;
}

// Draw idx of global game `game`: the double CPython's random.random() would build from two 32-bit outputs.
HEXB_HD double draw01(unsigned long long seed, unsigned long long game, uint32_t idx) {
    uint32_t a, b;
    philox4x32_10(idx, (uint32_t)game, (uint32_t)(game >> 32), 0u, (uint32_t)seed, (uint32_t)(seed >> 32), a, b);
    return ((double)(a >> 5) * 67108864.0 + (double)(b >> 6)) * (1.0 / 9007199254740992.0);
}

// The same draw as a real function call, for the restart path (reset_game: up to four draws, taken by one or two lanes of a
// warp in a step): inlined there, every draw is another copy of the ten Philox rounds in the step kernel, whose
// instruction-cache footprint is worth more than the call (ncu: 18 % of the stall samples at 1 Mi games were 'no_instructions').
#if defined(__CUDACC__) && !defined(HEXB_HOST_EMU)
static __host__ __device__ __noinline__ double draw01_cold(unsigned long long seed, unsigned long long game, uint32_t idx) {
    return draw01(seed, game, idx);
}
#else
static inline double draw01_cold(unsigned long long seed, unsigned long long game, uint32_t idx) { return draw01(seed, game, idx); }
#endif

// choice = int(random.random() * n)   (SelfplayWrapper.py:20, minihex/__init__.py:11): one fp64 multiply, truncation.
HEXB_HD int choice_of(double u, int n) {
#if defined(__CUDA_ARCH__)
    int k = __double2int_rz(__dmul_rn(u, (double)n));
#else
    int k = (int)(u * (double)n);
#endif
    return k < 0 ? 0 : (k >= n ? n - 1 : k);
}

// index of the k-th (0-based) SET bit of a W-word bit set (k < number of set bits)
template <int N>
HEXB_HD int select_kth_set(const uint32_t (&bits)[Geo<N>::W], int k) {
    constexpr int W = Geo<N>::W;
    // the word holding it is the last word w whose preceding words hold at most k set bits (the counts below only grow)
    uint32_t z = bits[0];
    int base = 0, below = 0, before = popc32(bits[0]);   // set bits in the words before w
#pragma unroll
    for (int w = 1; w < W; ++w) {
        if (k >= before) { z = bits[w]; base = 32 * w; below = before; }
        before += popc32(bits[w]);
    }
    k -= below;
    // k-th set bit of z by halving
    int pos = 0, c;
    c = popc32(z & 0xffffu); if (k >= c) { k -= c; pos += 16; z >>= 16; }
    c = popc32(z & 0xffu);   if (k >= c) { k -= c; pos += 8;  z >>= 8; }
    c = popc32(z & 0xfu);    if (k >= c) { k -= c; pos += 4;  z >>= 4; }
    c = popc32(z & 0x3u);    if (k >= c) { k -= c; pos += 2;  z >>= 2; }
    c = (int)(z & 1u);       if (k >= c) { pos += 1; }
    return base + pos;
}

// the empty cells of a bitboard as a bit set (bits >= C cleared)
template <int N>
HEXB_HD void empty_bits(const uint32_t (&occ)[Geo<N>::W], uint32_t (&e)[Geo<N>::W]) {
#pragma unroll
    for (int w = 0; w < Geo<N>::W; ++w) e[w] = ~occ[w];
    e[Geo<N>::W - 1] &= Geo<N>::LAST_MASK;
}

// index of the k-th (0-based) ZERO bit among the first C bits of a W-word bitboard: the k-th empty cell in row-major order
template <int N>
HEXB_HD int select_kth_zero(const uint32_t (&occ)[Geo<N>::W], int k) {
    uint32_t e[Geo<N>::W];
    empty_bits<N>(occ, e);
    return select_kth_set<N>(e, k);
}

// ---- the k-th empty cell in COLUMN-major order, from the row-major bitboard.
// The random opponent picks the k-th empty cell of ITS view (SelfplayWrapper.py:17-22, minihex/__init__.py:8-12), which is the
// stored board transposed, i.e. stored column-major order. Instead of carrying a second, transposed bitboard in the state
// (W words read and written per game and step), the column is found by bisection on "empty cells in columns < X" and the row
// by a k-th-set-bit selection inside that column. The masks are periodic with period N bits, so they are made by ONE multiply
// per word: an N-bit field times the constant with a one at every multiple of N (the copies cannot overlap, so no carries).
template <int N>
HEXB_HD constexpr uint32_t rep_word(int w) {   // word w of the C-bit constant with bits 0, N, 2N, ..., (N-1)N set
    uint32_t v = 0;
    for (int y = 0; y < N; ++y) {
        const int b = y * N;
        if ((b >> 5) == w) v |= 1u << (b & 31);
    }
    return v;
}
template <int N>
HEXB_HD void spread_field(uint32_t field, uint32_t (&out)[Geo<N>::W]) {   // field (< 2^N) copied to bit offsets 0, N, 2N, ...
    uint32_t carry = 0;
#pragma unroll
    for (int w = 0; w < Geo<N>::W; ++w) {
        constexpr uint32_t REP[] = {rep_word<N>(0), rep_word<N>(1), rep_word<N>(2), rep_word<N>(3), rep_word<N>(4), rep_word<N>(5),
                                    rep_word<N>(6), rep_word<N>(7), rep_word<N>(8), rep_word<N>(9), rep_word<N>(10), rep_word<N>(11)};
        const unsigned long long p = (unsigned long long)field * REP[w];
        out[w] = (uint32_t)p | carry;
        carry = (uint32_t)(p >> 32);
    }
}
// returns the stored (row-major) cell of the k-th empty cell in column-major order and its column in `col`
template <int N>
HEXB_HD int select_kth_zero_colmajor(const uint32_t (&occ)[Geo<N>::W], int k, int &col) {
    constexpr int W = Geo<N>::W;
    uint32_t e[W], m[W];
    empty_bits<N>(occ, e);
    // invariant: empties in columns < lo  <=  k  <  empties in columns < hi
    int lo = 0, hi = N, below = 0;
#pragma unroll
    for (int it = 0; it < Geo<N>::COL_STEPS; ++it) {
        const int mid = (lo + hi + 1) >> 1;   // lo < mid <= hi while hi - lo > 1; mid == hi when hi - lo == 1 (then c > k: no change)
        spread_field<N>((1u << mid) - 1u, m);
        int c = 0;
#pragma unroll
        for (int w = 0; w < W; ++w) c += popc32(e[w] & m[w]);
        if (c <= k) { lo = mid; below = c; }
        else hi = mid;
    }
    col = lo;
    spread_field<N>(1u << lo, m);
#pragma unroll
    for (int w = 0; w < W; ++w) m[w] &= e[w];
    return select_kth_set<N>(m, k - below);
}

template <int N>
HEXB_HD int count_empty(const uint32_t (&occ)[Geo<N>::W]) {
    int n = 0;
#pragma unroll
    for (int w = 0; w < Geo<N>::W; ++w) n += popc32(occ[w]);
    return Geo<N>::C - n;
}

template <int N>
HEXB_HD bool test_bit(const uint32_t (&bb)[Geo<N>::W], int i) {
    // (written as mask-and-or: a select chain `v = (w == i >> 5) ? bb[w] : v` is turned into an indexed load by the compiler,
    // which moves the whole record from registers to local memory: 43 LDL/STL in the step kernel, +2 us per 1 Mi-game step at
    // 11x11 and +12 us at 19x19)
    uint32_t v = 0;
#pragma unroll
    for (int w = 0; w < Geo<N>::W; ++w) v |= bb[w] & (0u - (uint32_t)(w == (i >> 5)));
    return (v >> (i & 31)) & 1u;
}
// the bit of cell i in word w of a bitboard, 0 when i lies in another word: one shift by i - 32w, which the device clamps (shl.b32
// with a count >= 32, negative counts included, gives 0), instead of a compare and a select per word (ALU pipe; the subtraction
// is a multiply-add, see fma_add)
HEXB_HD uint32_t word_bit(int i, int w, uint32_t one) {
    const uint32_t s = fma_add((uint32_t)i, (uint32_t)(-32 * w), one);
#if defined(__CUDA_ARCH__)
    uint32_t d;
    asm("shl.b32 %0, %1, %2;" : "=r"(d) : "r"(1u), "r"(s));
    return d;
#else
    return s < 32u ? 1u << s : 0u;
#endif
}
template <int N>
HEXB_HD void set_bit(uint32_t (&bb)[Geo<N>::W], int i, uint32_t one = 1u) {
#pragma unroll
    for (int w = 0; w < Geo<N>::W; ++w) bb[w] |= word_bit(i, w, one);
}

template <int N>
HEXB_HD int transpose_cell(int a) {
    const int y = a / N;
    return (a - y * N) * N + y;
}

// ----------------------------------------------------------------------------------------------
// one stone: HexGame.fast_move (HexGame.py:85-111, HexSingleGame.py:88-122) + flood_fill
// (HexGame.py:124-142, HexSingleGame.py:135-153) on the tagged label plane of ONE game.
//   L      this game's C label bytes (shared memory on the device)
//   p      0 = R, 1 = C      cell  stored row-major index, known to be empty
//   one    Params::one (see fma_add)
// Writes the new cell's byte, updates occupancy/counters/far flags in `rec`, and returns the relabel
// request for the cooperative byte pass (regions[regions == label] = new_region_label, :141-142 / :152-153):
// at most two labels besides the minimum can be adjacent (the six neighbours form a cycle; own stones
// that are adjacent on the cycle already share a label), so `prm` carries o1, o2 and m.
// Returns true iff the mover's far border now carries label 1 (regions[-1,-1] == 1, :102 / :111).
// ----------------------------------------------------------------------------------------------
// A neighbour's byte as the mover's label biased by tag = p << 7: an own stone gives label + tag (tag + 1 .. tag + 127), an empty
// cell or a stone of the other colour a value <= tag as a signed int (for R the byte is sign-extended, so C stones are negative
// and an empty cell is 0; for C the plain byte of an R stone or an empty cell is below 128).
HEXB_HD int32_t own_biased(uint32_t b, int p) { return p ? (int32_t)b : (int32_t)(int8_t)b; }
// The smallest biased label above kb among s[], as d = label - (kb + 1) >= 0, or a negative d (as a signed int) if there is none:
// every s <= kb gives s - (kb + 1) in [-384, -1], i.e. >= 2^31 unsigned, so one unsigned min filters and selects at once. The
// subtractions are multiply-adds (FMA pipe), the mins VIMNMX3 (ALU pipe).
HEXB_HD uint32_t next_above(const int32_t (&s)[6], uint32_t kb, uint32_t one) {
    uint32_t d[6];
#pragma unroll
    for (int i = 0; i < 6; ++i) d[i] = fma_add((uint32_t)s[i], ~kb, one);   // s - kb - 1
    return umin32(umin32(umin32(d[0], d[1]), d[2]), umin32(umin32(d[3], d[4]), d[5]));
}
template <int N>
HEXB_HD bool place_stone(uint8_t *L, Rec<N> &rec, int p, int cell, uint32_t &prm, uint32_t one = 1u) {
    const int y = cell / N, x = cell - y * N;
    const uint32_t tag = (uint32_t)p << 7;
    const bool up = y > 0, dn = y < N - 1, lf = x > 0, rt = x < N - 1;
    // implicit borders of the mover's padded plane: near border label 1, far border 1 once connected, else 2. Each takes the place
    // of the one off-board neighbour that lies on it (R: up = row -1 / down = row N; C: left = column -1 / right = column N), which
    // is off the board exactly when the cell touches that border; the other off-board neighbours count as nothing (0).
    const uint32_t far1 = p ? (rec.meta & M_FAR_C1) : (rec.meta & M_FAR_R1);
    const int32_t nb = (int32_t)tag + 1, fb = (int32_t)tag + (far1 ? 1 : 2);
    // the hex neighbourhood: 3x3 window minus [0,0] and [2,2] (neighborhood[0,0] = neighborhood[2,2] = 0)
    int32_t s[6];
    s[0] = up ? own_biased(L[cell - N], p) : (p ? 0 : nb);
    s[1] = (up && rt) ? own_biased(L[cell - N + 1], p) : 0;
    s[2] = lf ? own_biased(L[cell - 1], p) : (p ? nb : 0);
    s[3] = rt ? own_biased(L[cell + 1], p) : (p ? fb : 0);
    s[4] = (dn && lf) ? own_biased(L[cell + N - 1], p) : 0;
    s[5] = dn ? own_biased(L[cell + N], p) : (p ? 0 : fb);
    // m = the smallest adjacent own label, o1 < o2 the next larger ones (biased by tag, i.e. the tagged bytes)
    const uint32_t dm = next_above(s, tag, one);
    const uint32_t cshift = p ? M_CTR_C_SHIFT : M_CTR_R_SHIFT;
    uint32_t lab;
    prm = 0;
    if ((int32_t)dm < 0) {  // no adjacent region: new label = region_counter, counter += 1
        lab = ((rec.meta >> cshift) & 0xffu) | tag;
        rec.meta += 1u << cshift;
    } else {
        lab = dm + tag + 1u;
        const uint32_t d1 = next_above(s, lab, one);
        if ((int32_t)d1 >= 0) {
            const uint32_t o1 = d1 + lab + 1u;
            const uint32_t d2 = next_above(s, o1, one);
            const uint32_t o2e = (int32_t)d2 >= 0 ? d2 + o1 + 1u : o1;
            prm = o1 | (o2e << 8) | (lab << 16) | P_NEED;
            // the relabel runs over the whole padded plane, borders included: 2 -> 1 moves the far border (m = 1 < o1 < o2, so
            // label 2 can only be o1)
            if (lab == tag + 1u && o1 == tag + 2u && !far1) rec.meta |= p ? M_FAR_C1 : M_FAR_R1;
        }
    }
    L[cell] = (uint8_t)lab;
    set_bit<N>(rec.occ_rm, cell, one);
    return (rec.meta & (p ? M_FAR_C1 : M_FAR_R1)) != 0u;
}

// ----------------------------------------------------------------------------------------------
// byte-SIMD helpers for the cooperative passes (4 cells per 32-bit word)
// ----------------------------------------------------------------------------------------------
HEXB_HD uint32_t relabel_byte(uint32_t b, uint32_t prm) {
    return ((prm & P_NEED) && (b == (prm & 0xffu) || b == ((prm >> 8) & 0xffu))) ? ((prm >> 16) & 0xffu) : b;
}
// observation / mask bytes in the STORED orientation (the agent's view)
//   variant B (HexSingleGame.py:15-19, 265-271): own -1, opponent +1, empty 0; own = R
//   variant A (HexGame.py:10-13): BLACK 0 (= R, the agent), WHITE 1, EMPTY 2
// 0xff in every byte of f whose top bit is set (PRMT with the sign-replicate selector bit on the device)
HEXB_HD uint32_t sign_fill(uint32_t f) {
#if defined(__CUDA_ARCH__)
    uint32_t d;
    asm("prmt.b32 %0, %1, %2, %3;" : "=r"(d) : "r"(f), "r"(0u), "r"(0xba98u));  // selector bit 3 = replicate the byte's msb
    return d;
#else
    return ((f >> 7) & 0x01010101u) * 0xffu;
#endif
}
// byte p (0..3, run-time) of v replicated into all four bytes: one PRMT with a register selector on the device
HEXB_HD uint32_t splat_byte_dyn(uint32_t v, int p) {
#if defined(__CUDA_ARCH__)
    uint32_t d;
    asm("prmt.b32 %0, %1, %2, %3;" : "=r"(d) : "r"(v), "r"(0u), "r"(0x1111u * (uint32_t)p));
    return d;
#else
    return ((v >> (8 * p)) & 0xffu) * 0x01010101u;
#endif
}

// x >> 7 for a word of 0x80 byte flags, issued as a multiply-high so that it runs on the (idle) FMA pipe instead of the ALU
// pipe, which is the busy one in the step kernel (ncu: sm__pipe_alu_cycles_active is the top pipe)
HEXB_HD uint32_t flags_to_ones(uint32_t f) { return mulhi32(f, 1u << 25); }

// One label word (4 cells) -> observation bytes + mask bytes, the same code for both variants: with msk = 0x01 per empty cell and
// c1 = 0x01 per C stone (at most one of them per byte),
//   variant B   R -> 0xff, C -> 0x01, empty -> 0x00:  obs = 0xffffffff - 0xff * msk - 0xfe * c1   (no byte ever borrows)
//   variant A   BLACK (= R) 0, WHITE (= C) 1, EMPTY 2: obs = 2 * msk + c1
// i.e. obs = msk * ka + (c1 * kb + kc) with per-variant constants (Params::enc_k*, filled by enc_consts): two multiply-adds on the
// FMA pipe and no logic op for the observation itself. Per word: 3 ALU-pipe ops (LOP3: t's operand, z, c1's operand) + 5
// FMA-pipe ops (one add issued as IMAD, two multiply-highs, two IMAD) - the ALU pipe is the busy one in the step kernel.
HEXB_HD void enc_consts(int variant, uint32_t &ka, uint32_t &kb, uint32_t &kc) {
    if (variant == VARIANT_B) { ka = 0u - 0xffu; kb = 0u - 0xfeu; kc = 0xffffffffu; }
    else { ka = 2u; kb = 1u; kc = 0u; }
}
HEXB_HD void encode_word_k(uint32_t x, uint32_t one, uint32_t ka, uint32_t kb, uint32_t kc, uint32_t &obs, uint32_t &msk) {
    const uint32_t t = fma_add(x & 0x7f7f7f7fu, 0x7f7f7f7fu, one);
    const uint32_t z = ~(t | x) & 0x80808080u;           // 0x80 per EMPTY cell
    const uint32_t c1 = flags_to_ones(x & 0x80808080u);  // 0x01 per C stone
    msk = flags_to_ones(z);                              // legal == empty
    obs = msk * ka + (c1 * kb + kc);
}
// one byte, optionally seen from the opponent's side (sign swap; the caller transposes the cell index)
HEXB_HD uint32_t encode_byte(uint32_t b, int variant, bool opp_view, uint32_t &msk) {
    msk = (b == 0u);
    if (variant == VARIANT_A) return b == 0u ? 2u : ((b >> 7) ^ (opp_view ? 1u : 0u));  // invert_board swaps 0 <-> 1 (HexGame.py:297-303)
    if (b == 0u) return 0u;
    const bool own = ((b >> 7) != 0u) == opp_view;  // R is "own" in the agent's view, C in the opponent's
    return own ? 0xffu : 0x01u;
}

// one observation cell into the caller's buffer in its dtype (the per-cell paths: terminal observations, opponent views, K5)
HEXB_HD void store_obs(int8_t *obs, int obs_f32, long long i, uint32_t byte) {
    if (obs_f32) reinterpret_cast<float *>(obs)[i] = (float)(int8_t)byte;
    else obs[i] = (int8_t)byte;
}

// ----------------------------------------------------------------------------------------------
// reset: HexGame.__init__ on an empty board (HexGame.py:21-68 / HexSingleGame.py:26-71) + HexEnv.reset
// (HexGame.py:206-242 / HexSingleGame.py:208-231) + SelfPlayEnv.reset / setup_opponents / continue_game
// (SelfplayWrapper.py:69-104,146-172). The label bytes themselves are cleared by the caller; this fills
// `rec` and returns the opening stone (if the opponent moves first) through `flg`.
// ----------------------------------------------------------------------------------------------
template <int N>
HEXB_HD void reset_game(Rec<N> &rec, const Params &P, unsigned long long gid, const double *inj_u, uint32_t &flg) {
    constexpr int C = Geo<N>::C;
    uint32_t meta = rec.meta & (M_TRANSPOSED | M_COLOUR_SET);
    meta |= M_LIVE | (3u << M_CTR_R_SHIFT) | (3u << M_CTR_C_SHIFT);
#pragma unroll
    for (int w = 0; w < Geo<N>::W; ++w) rec.occ_rm[w] = 0u;
    bool opp_opens;
    if (P.raw) {
        opp_opens = false;
    } else if (P.variant == VARIANT_B) {
        if (!(meta & M_COLOUR_SET)) {  // random.randint(0,1) once per env (SelfplayWrapper.py:72-73)
            int colour = P.agent_mode;
            if (P.agent_mode == 2) colour = (int)(draw01_cold(P.seed, gid, rec.draws++) * 2.0);
            meta |= M_COLOUR_SET | (colour ? M_TRANSPOSED : 0u);
        }
        if (P.eval_state) {  // setup_opponents while evaluating (:92-96): episode k since set_eval meets pool entry k, nothing is drawn
            if (P.opp_index && P.eval_episode) {
                const unsigned long long i = gid - (unsigned long long)P.game_offset;
                const int ep = P.eval_episode[i];
                if (ep <= P.pool_size - 1) {   // past the end of the pool the game keeps the opponent it has
                    P.opp_index[i] = ep;
                    P.eval_episode[i] = ep + 1;
                }
            }
        } else if (!inj_u) {  // setup_opponents (:97-103): 80 % the best model, else a uniformly drawn pool entry
            const double rv = draw01_cold(P.seed, gid, rec.draws++);
            int pick = -1;
            if (!(rv < 0.8)) {   // random.random() for the pool index: the draw is always consumed, its value only matters to a caller-driven opponent
                const uint32_t at = rec.draws++;
                if (P.opp_index && P.pool_size > 0) pick = choice_of(draw01_cold(P.seed, gid, at), P.pool_size);
            }
            if (P.opp_index) P.opp_index[gid - (unsigned long long)P.game_offset] = pick;
        }
        opp_opens = (meta & M_TRANSPOSED) != 0u;  // agent WHITE: BLACK (the opponent) opens (:79-80)
    } else {
        opp_opens = P.opponent_first != 0;  // HexGame.py:224-230
    }
    if (opp_opens && P.manual_opponent) {
        meta |= M_TOMOVE;  // the caller's opponent policy opens: nothing is placed here
    } else if (opp_opens) {
        double u;
        if (inj_u) u = *inj_u;
        else {
            if (P.variant == VARIANT_B) rec.draws++;  // rv = random.uniform(0,1), unused (:159)
            u = draw01_cold(P.seed, gid, rec.draws++);
        }
        const int k = choice_of(u, C);         // k-th empty cell of the opponent's view of an empty board
        const int x = k / N, y = k - x * N;    // stored column-major index -> stored (y, x)
        uint32_t lab;
        if (x == 0) lab = 1u;
        else if (x == N - 1) lab = 2u;
        else { lab = 3u; meta += 1u << M_CTR_C_SHIFT; }
        set_bit<N>(rec.occ_rm, y * N + x);
        flg |= F_OPEN | ((lab | 0x80u) << 8) | ((uint32_t)(y * N + x) << 16);
    }
    rec.meta = meta;  // R (the agent) to move unless a caller-driven opponent opens
    flg |= F_RESET;
}

}  // namespace hexb
