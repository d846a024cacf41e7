// tetris_dev.cuh — device-side Tetris board step for sm_100a (bitboard form of /SPEC_PYTETRIS.md).
//
// Replaces the pyTetris C++ env at the reference call sites agents/agent.py:103,114,143-144 (copy_from/play/
// getState), agents/cppmodule/agent.cpp:205,233,243 and play.py:150.  The whole game lives in registers:
// the 20x10 board is ten 32-bit words (two 16-bit rows per word), the falling piece is (piece, rot, px, py) and
// a 16-bit 4x4 shape mask.  One thread owns one game for the duration of a step; nothing here touches memory
// except rec_load / rec_store.
#pragma once
#include <stdint.h>

namespace b200 {

constexpr int REC_WORDS = 20;   // SPEC §6 packed record (80 B)
constexpr int KEY_WORDS = 12;   // SPEC §6 observation key (48 B)
constexpr int N_ACTIONS = 7;    // reference core.h:17

// SPEC §2 shapes: bit (4*r + c) of SHAPES[piece][rot] = cell (r, c) of the 4x4 box.
__device__ __constant__ uint16_t SHAPES[7][4] = {
    /* I */ {0x00F0, 0x4444, 0x0F00, 0x2222},
    /* O */ {0x0066, 0x0066, 0x0066, 0x0066},
    /* T */ {0x0072, 0x0262, 0x0270, 0x0232},
    /* S */ {0x0036, 0x0462, 0x0360, 0x0231},
    /* Z */ {0x0063, 0x0264, 0x0630, 0x0132},
    /* J */ {0x0071, 0x0226, 0x0470, 0x0322},
    /* L */ {0x0074, 0x0622, 0x0170, 0x0223},
};

struct Game {
    uint32_t w[10];   // board, word i = row 2i | row 2i+1 << 16
    int piece, rot, px, py;
    uint32_t bag;
    int dropcnt, end, app, scoring, randomizer, combo;
    uint32_t rng;
    int score, lines, ls[4];
};

__device__ __forceinline__ uint32_t shape_of(int piece, int rot) { return SHAPES[piece][rot]; }

// Row r (0..19) of the board; r is dynamic, so pick the word with a predicated chain instead of local memory.
__device__ __forceinline__ uint32_t get_row(const uint32_t (&w)[10], int r) {
    int i = r >> 1;
    uint32_t x = w[0];
#pragma unroll
    for (int k = 1; k < 10; ++k) x = (i == k) ? w[k] : x;
    return (r & 1) ? (x >> 16) : (x & 0xffffu);
}

__device__ __forceinline__ void or_row(uint32_t (&w)[10], int r, uint32_t m) {
    int i = r >> 1;
    uint32_t v = (r & 1) ? (m << 16) : m;
#pragma unroll
    for (int k = 0; k < 10; ++k) w[k] |= (i == k) ? v : 0u;
}

// Remove row r: rows above it move down one, row 0 becomes empty (SPEC §3.3).
__device__ __forceinline__ void remove_row(uint32_t (&w)[10], int r) {
#pragma unroll
    for (int i = 9; i >= 0; --i) {
        uint32_t below = (i > 0) ? (w[i - 1] >> 16) : 0u;   // row 2i-1
        if (2 * i + 1 <= r) w[i] = (w[i] << 16) | below;                 // both rows of the word shift down
        else if (2 * i == r) w[i] = (w[i] & 0xffff0000u) | below;        // only the low row is replaced
    }
}

// SPEC §3: true if the piece would leave the board or overlap a locked cell.
__device__ __forceinline__ bool collides(const uint32_t (&w)[10], uint32_t shape, int px, int py) {
    bool hit = false;
#pragma unroll
    for (int r = 0; r < 4; ++r) {
        uint32_t m = (shape >> (4 * r)) & 0xfu;
        if (m) {
            int br = py + r;
            if (br < 0 || br > 19) { hit = true; }
            else {
                uint32_t mm;
                if (px < 0) { if (m & ((1u << (-px)) - 1u)) hit = true; mm = m >> (-px); }
                else mm = m << px;
                if (mm >> 10) hit = true;
                if (get_row(w, br) & mm) hit = true;
            }
        }
    }
    return hit;
}

// SPEC §3.2 hard drop: how many rows the piece at the LEGAL position (px, py) falls.  Closed form of the reference-style loop
// `while (!collides(px, py + 1)) ++py` (one dependent collision test of ~80 instructions per row fallen; the hard-drop lane made
// every expansion wait): for each of the four shape rows r, bit y of hit[r] says that board row y has a locked cell under that
// shape row's cells; the first set bit below row py + r (or the floor) bounds the fall of that row, the piece falls the minimum.
// The board rows are walked with static indices only (no dynamic row select), four independent chains.
__device__ __forceinline__ int drop_distance(const uint32_t (&w)[10], uint32_t shape, int px, int py) {
    uint32_t mm[4], hit[4];
#pragma unroll
    for (int r = 0; r < 4; ++r) {
        const uint32_t m = (shape >> (4 * r)) & 0xfu;
        mm[r] = px < 0 ? (m >> (-px)) : (m << px);     // legal position: no cell is shifted off the board
        hit[r] = 0u;
    }
#pragma unroll
    for (int y = 0; y < 20; ++y) {
        const uint32_t row = (y & 1) ? (w[y >> 1] >> 16) : (w[y >> 1] & 0xffffu);
#pragma unroll
        for (int r = 0; r < 4; ++r) hit[r] |= (row & mm[r]) ? (1u << y) : 0u;
    }
    int d = 32;
#pragma unroll
    for (int r = 0; r < 4; ++r) {
        if (mm[r]) {
            const int br = py + r;                                   // >= 0 for a non-empty shape row at a legal position
            const uint32_t below = hit[r] >> (br + 1);               // rows br+1 .. 19
            const int free_rows = below ? (__ffs((int)below) - 1) : (19 - br);
            d = free_rows < d ? free_rows : d;
        }
    }
    return d;
}

__device__ __forceinline__ uint32_t rng_next(uint32_t &s) {   // SPEC §4 xorshift32
    s ^= s << 13; s ^= s >> 17; s ^= s << 5;
    return s;
}

__device__ __forceinline__ void spawn(Game &g) {   // SPEC §3.4 + §4
    int piece;
    if (g.randomizer == 0) {
        if (g.bag == 0) g.bag = 0x7fu;
        uint32_t k = rng_next(g.rng) % (uint32_t)__popc(g.bag);
        piece = (int)__fns(g.bag, 0, (int)k + 1);
        g.bag &= ~(1u << piece);
    } else {
        piece = (int)(rng_next(g.rng) % 7u);
    }
    g.piece = piece; g.rot = 0; g.px = 3; g.py = (piece == 0) ? -1 : 0;
    if (collides(g.w, shape_of(piece, 0), g.px, g.py)) g.end = 1;
}

__device__ __forceinline__ void lock_piece(Game &g) {   // SPEC §3.3
    uint32_t shape = shape_of(g.piece, g.rot);
#pragma unroll
    for (int r = 0; r < 4; ++r) {
        uint32_t m = (shape >> (4 * r)) & 0xfu;
        if (m) or_row(g.w, g.py + r, (g.px < 0) ? (m >> (-g.px)) : (m << g.px));
    }
    int n = 0;
#pragma unroll
    for (int r = 0; r < 4; ++r) {   // top to bottom: removing a row never moves the rows below it
        int br = g.py + r;
        if (br >= 0 && br <= 19 && get_row(g.w, br) == 0x3ffu) { remove_row(g.w, br); ++n; }
    }
    if (n > 0) {
        g.combo += 1;
        g.lines += n;
#pragma unroll
        for (int i = 0; i < 4; ++i) g.ls[i] += (i == n - 1) ? 1 : 0;
        if (g.scoring == 0) g.score += (n == 1 ? 100 : n == 2 ? 300 : n == 3 ? 500 : 800) + 50 * (g.combo - 1);
        else g.score += n;
    } else {
        g.combo = 0;
    }
    spawn(g);
}

// One environment step (SPEC §3).  The reference entry point is Tetris.play(action).
// In an expansion the seven lanes of a group play the seven different actions, so every action-specific branch is executed
// serially by the warp.  The step is therefore written with ONE collision test for all shifting / rotating / soft-drop actions
// (a candidate position per action, accepted if it does not collide; action 0 proposes the current position) and ONE lock_piece
// site shared by the hard drop and by gravity; only the hard drop's distance computation is a branch of its own.
__device__ __forceinline__ void play(Game &g, int action) {
    if (g.end) return;
    uint32_t shape = shape_of(g.piece, g.rot);
    bool lock = false;
    if (action == 5) {   // hard drop
        const int d = drop_distance(g.w, shape, g.px, g.py);
        g.py += d;
        if (g.scoring == 0) g.score += 2 * d;
        g.dropcnt = 0;
        lock = true;
    } else {
        const bool rotate = action == 3 || action == 4;
        const int nr = rotate ? ((g.rot + (action == 3 ? 1 : 3)) & 3) : g.rot;
        const uint32_t ns = rotate ? shape_of(g.piece, nr) : shape;
        const int nx = g.px + (action == 2 ? 1 : 0) - (action == 1 ? 1 : 0);
        const int ny = g.py + (action == 6 ? 1 : 0);
        if (!collides(g.w, ns, nx, ny)) {          // action 0 (and any action code outside 1..6) proposes the current, legal position
            g.rot = nr; shape = ns; g.px = nx;
            if (ny != g.py) { g.py = ny; if (g.scoring == 0) g.score += 1; }
        }
        g.dropcnt += 1;
        if (g.dropcnt >= g.app) {
            g.dropcnt = 0;
            if (!collides(g.w, shape, g.px, g.py + 1)) g.py += 1;
            else lock = true;
        }
    }
    if (lock) lock_piece(g);
}

// ---- SPEC §6 packed record <-> registers
__device__ __forceinline__ void unpack(Game &g, const uint32_t (&r)[REC_WORDS]) {
#pragma unroll
    for (int i = 0; i < 10; ++i) g.w[i] = r[i];
    uint32_t a = r[10], b = r[11];
    g.piece = a & 7; g.rot = (a >> 3) & 3; g.px = (int)((a >> 5) & 15) - 2; g.py = (int)((a >> 9) & 31) - 2;
    g.bag = (a >> 14) & 0x7f; g.end = (a >> 21) & 1; g.scoring = (a >> 22) & 1; g.randomizer = (a >> 23) & 1;
    g.dropcnt = (a >> 24) & 0xff; g.app = b & 0xff; g.combo = (int)(b >> 8);
    g.rng = r[12]; g.score = (int)r[13]; g.lines = (int)r[14];
#pragma unroll
    for (int i = 0; i < 4; ++i) g.ls[i] = (int)r[15 + i];
}

__device__ __forceinline__ void pack(const Game &g, uint32_t (&r)[REC_WORDS]) {
#pragma unroll
    for (int i = 0; i < 10; ++i) r[i] = g.w[i];
    r[10] = (uint32_t)g.piece | ((uint32_t)g.rot << 3) | ((uint32_t)(g.px + 2) << 5) | ((uint32_t)(g.py + 2) << 9) |
            ((g.bag & 0x7fu) << 14) | ((uint32_t)(g.end & 1) << 21) | ((uint32_t)g.scoring << 22) |
            ((uint32_t)g.randomizer << 23) | ((uint32_t)(g.dropcnt & 0xff) << 24);
    r[11] = (uint32_t)(g.app & 0xff) | ((uint32_t)(g.combo & 0xffffff) << 8);
    r[12] = g.rng; r[13] = (uint32_t)g.score; r[14] = (uint32_t)g.lines;
#pragma unroll
    for (int i = 0; i < 4; ++i) r[15 + i] = (uint32_t)g.ls[i];
    r[19] = 0;
}

// SPEC §6 observation key: board words with the piece's own cells cleared + the four piece cells (ascending).
__device__ __forceinline__ void obskey(const Game &g, uint32_t (&k)[KEY_WORDS]) {
#pragma unroll
    for (int i = 0; i < 10; ++i) k[i] = g.w[i];
    uint32_t shape = shape_of(g.piece, g.rot);
    uint32_t cells = 0;
    int n = 0;
#pragma unroll
    for (int r = 0; r < 4; ++r) {       // row-major scan of the box yields ascending row*10+col
        uint32_t m = (shape >> (4 * r)) & 0xfu;
        int br = g.py + r;
        if (m) {                        // clear the whole shape row at once (one pass over the board words per row, not per cell)
            const uint32_t mm = (g.px < 0) ? (m >> (-g.px)) : (m << g.px);
            const uint32_t bits = (br & 1) ? (mm << 16) : mm;
            const int wi = br >> 1;
#pragma unroll
            for (int q = 0; q < 10; ++q) k[q] &= (wi == q) ? ~bits : 0xffffffffu;
        }
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            if ((m >> c) & 1u) {
                cells |= (uint32_t)(br * 10 + g.px + c) << (8 * n);
                ++n;
            }
        }
    }
    k[10] = cells;
    k[11] = 0;
}

__device__ __forceinline__ uint64_t hash_words(const uint32_t *w, int n) {
    uint64_t h = 0x9E3779B97F4A7C15ull;
#pragma unroll
    for (int i = 0; i < n; ++i) {
        h ^= w[i];
        h *= 0xff51afd7ed558ccdull;
        h ^= h >> 32;
    }
    return h;
}

}  // namespace b200
