// twr_common.cuh -- device-side primitives shared by every kernel of the rollout engine:
// Philox4x32-10, the packed env state and the Env-trait methods on it.
//
// Env state layout in HBM (structure of arrays over envs, one coalesced vector load each):
//   cells : uint4 per env, in one of two encodings, chosen by the board size alone (cells_wide):
//           bytes  -- Puzzle of up to 16 cells: byte i = tile at cell i.  GridWorld: byte 0/1/2 = agent/goal/trap cell.
//           5-bit  -- Puzzle of 17..25 cells: bits [5i, 5i+5) = tile at cell i (25 x 5 = 125 bits).
//           Unused fields (cells >= N) hold their own index in either form, so "solved" is one 128-bit compare
//           against TWR_IDENT_* / TWR_IDENT5_*.  Only the accessors below know either layout.
//   meta  : uint32 per env = blank cell (bits 0..7) | depth or steps_left (bits 8..31).
// Reference semantics: rust/src/envs/puzzle.rs, examples/grid_world/src/lib.rs (cited per function).
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

#define TWR_MAX_ACTIONS 4
#define TWR_MAX_CELLS_PUZZLE 25   // 5-bit cells in the 128-bit state
#define TWR_MAX_CELLS_BYTES 16    // the byte encoding
#define TWR_MAX_CELLS 32          // boards whose N*N-row table the forwards stage whole (and the observation length a policy's fit assumes)
#define TWR_MAX_OBS 64            // observation indices per env: GridWorld of up to 64 cells (4 * 64 compact rows, 256)

enum : uint32_t { TWR_RNG_RESET = 0, TWR_RNG_PERM = 1, TWR_RNG_SAMPLE = 2, TWR_RNG_SOLVE = 3, TWR_RNG_MCTS = 4, TWR_RNG_AZ_ACT = 5 };

struct EnvParams {
    int kind;  // 0 puzzle, 1 grid_world
    int W, H, N;
    int difficulty, depth_slope, max_depth;
};

// Global (Philox) env id of local env e: base + (e + off) mod `mod` (mod == 0: base + e).  The rotation lets
// a collect lay episodes out directly in the reference's merge order [last, 0, 1, ..., n-2]
// (collector/collector.rs:40-46): local 0 is the LAST episode id, local i is episode i-1.
struct EnvIds {
    uint32_t base, off, mod;
    uint32_t div;   // > 1: `div` consecutive local envs share one id (the searches of one evaluate() episode)
    __host__ __device__ __forceinline__ uint32_t gid(uint32_t e) const {
        if (div > 1) e /= div;
        return base + (mod ? (e + off) % mod : e);
    }
};

// ------------------------------------------------------------------ Philox ---
__host__ __device__ __forceinline__ void philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3,
                                                       uint32_t k0, uint32_t k1, uint32_t out[4]) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
#ifdef __CUDA_ARCH__
        const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
        const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
#else
        const uint64_t p0 = (uint64_t)0xD2511F53u * c0, p1 = (uint64_t)0xCD9E8D57u * c2;
        const uint32_t hi0 = (uint32_t)(p0 >> 32), lo0 = (uint32_t)p0;
        const uint32_t hi1 = (uint32_t)(p1 >> 32), lo1 = (uint32_t)p1;
#endif
        const uint32_t n0 = hi1 ^ c1 ^ k0, n2 = hi0 ^ c3 ^ k1;
        c0 = n0; c1 = lo1; c2 = n2; c3 = lo0;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

// 24 high bits * 2^-24, in [0,1): rand 0.8.5 `gen::<f32>()` (call site nn/policy.rs:171)
__host__ __device__ __forceinline__ float u32_to_unit_f32(uint32_t w) {
    return (float)(w >> 8) * (1.0f / 16777216.0f);
}

__device__ __forceinline__ uint32_t mulhi_u32(uint32_t a, uint32_t n) { return __umulhi(a, n); }

// --------------------------------------------------------------- env state ---
struct EnvState {
    uint64_t lo, hi;  // the 128-bit board (bytes or 5-bit fields)
    uint32_t blank;   // puzzle: blank cell index
    uint32_t depth;   // puzzle: depth budget; grid_world: steps_left
};

// Which encodings a kernel is compiled for.  TWR_CELLS_ANY picks one from the board size at run time (one uniform branch);
// TWR_CELLS_BYTES fixes the byte form at compile time.  The pair kernel (k_forward_tc2) is built with the latter: every
// instruction of its per-item path costs about 1 % of the collect, and it never meets a wide board (an N >= 17 board
// has an N*N >= 289-row table, which that kernel takes only as a compact GridWorld image).
enum : int { TWR_CELLS_ANY = 0, TWR_CELLS_BYTES = 1 };
template <int F = TWR_CELLS_ANY>
__host__ __device__ __forceinline__ bool cells_wide(const EnvParams& p) {
    return F == TWR_CELLS_ANY && p.kind == 0 && p.N > TWR_MAX_CELLS_BYTES;
}

__host__ __device__ __forceinline__ uint32_t cell_get(const EnvState& s, int i, bool wide) {
    if (wide) {
        const unsigned __int128 w = ((unsigned __int128)s.hi << 64) | s.lo;
        return (uint32_t)(w >> (5 * i)) & 0x1Fu;
    }
    const uint64_t w = (i < 8) ? s.lo : s.hi;
    return (uint32_t)(w >> (8 * (i & 7))) & 0xFFu;
}
__host__ __device__ __forceinline__ void cell_set(EnvState& s, int i, uint32_t v, bool wide) {
    if (wide) {
        const int sh = 5 * i;
        unsigned __int128 w = ((unsigned __int128)s.hi << 64) | s.lo;
        w = (w & ~((unsigned __int128)0x1Fu << sh)) | ((unsigned __int128)(v & 0x1Fu) << sh);
        s.lo = (uint64_t)w; s.hi = (uint64_t)(w >> 64);
        return;
    }
    const int sh = 8 * (i & 7);
    const uint64_t m = ~(0xFFull << sh), b = (uint64_t)(v & 0xFFu) << sh;
    if (i < 8) s.lo = (s.lo & m) | b; else s.hi = (s.hi & m) | b;
}

#define TWR_IDENT_LO 0x0706050403020100ull    // byte i = i
#define TWR_IDENT_HI 0x0F0E0D0C0B0A0908ull
#define TWR_IDENT5_LO 0xC5A928398A418820ull   // 5-bit field i = i, i < 25
#define TWR_IDENT5_HI 0x18BDAB49CA307B9Aull

// the cell words of one env (blank and depth zero): what the forwards, the compaction and the search read from a
// trajectory record or a leaf message
__host__ __device__ __forceinline__ EnvState env_from_cells(const uint4& c) {
    EnvState s;
    s.lo = (uint64_t)c.x | ((uint64_t)c.y << 32);
    s.hi = (uint64_t)c.z | ((uint64_t)c.w << 32);
    s.blank = 0; s.depth = 0;
    return s;
}
__device__ __forceinline__ EnvState env_load(const uint4* __restrict__ cells, const uint32_t* __restrict__ meta, int64_t e) {
    EnvState s = env_from_cells(cells[e]);
    const uint32_t m = meta[e];
    s.blank = m & 0xFFu; s.depth = m >> 8;
    return s;
}
__host__ __device__ __forceinline__ uint4 env_pack_cells(const EnvState& s) {
    return make_uint4((uint32_t)s.lo, (uint32_t)(s.lo >> 32), (uint32_t)s.hi, (uint32_t)(s.hi >> 32));
}
__device__ __forceinline__ void env_store(uint4* __restrict__ cells, uint32_t* __restrict__ meta, int64_t e, const EnvState& s) {
    cells[e] = env_pack_cells(s);
    meta[e] = (s.blank & 0xFFu) | (s.depth << 8);
}

// the solved board of a Puzzle (every field i holds i), in the env's encoding
__host__ __device__ __forceinline__ void env_set_identity(const EnvParams& p, EnvState& s) {
    const bool wide = cells_wide(p);
    s.lo = wide ? TWR_IDENT5_LO : TWR_IDENT_LO;
    s.hi = wide ? TWR_IDENT5_HI : TWR_IDENT_HI;
}

// Puzzle::new (envs/puzzle.rs:34-42) / GridWorld::new (lib.rs:23-41)
__device__ __forceinline__ EnvState env_fresh(const EnvParams& p) {
    EnvState s;
    s.blank = 0;
    if (p.kind == 0) { env_set_identity(p, s); s.depth = 1; } else { s.lo = 0; s.hi = 0; s.depth = (uint32_t)p.max_depth; }
    return s;
}

// GridWorld's agent / goal / trap cells are bytes 0..2 of the state in either build
template <int F = TWR_CELLS_ANY>
__device__ __forceinline__ bool env_success(const EnvParams& p, const EnvState& s) {
    if (p.kind == 0) {                                                      // puzzle.rs:44-50
        const bool wide = cells_wide<F>(p);
        return s.lo == (wide ? TWR_IDENT5_LO : TWR_IDENT_LO) && s.hi == (wide ? TWR_IDENT5_HI : TWR_IDENT_HI);
    }
    return cell_get(s, 0, false) == cell_get(s, 1, false);                  // lib.rs:67 at_goal
}

template <int F = TWR_CELLS_ANY>
__device__ __forceinline__ bool env_is_final(const EnvParams& p, const EnvState& s) {
    if (p.kind == 0) return s.depth == 0 || env_success<F>(p, s);          // puzzle.rs:167-169
    const uint32_t a = cell_get(s, 0, false);
    return s.depth == 0 || a == cell_get(s, 1, false) || a == cell_get(s, 2, false);   // lib.rs:147-149
}

template <int F = TWR_CELLS_ANY>
__device__ __forceinline__ float env_reward(const EnvParams& p, const EnvState& s) {
    if (p.kind == 0) {                                                      // puzzle.rs:171-177
        if (env_success<F>(p, s)) return 1.0f;
        if (s.depth == 0) return -0.5f;
        return __fdiv_rn(-0.5f, (float)p.max_depth);
    }
    const uint32_t a = cell_get(s, 0, false);                               // lib.rs:151-155
    if (a == cell_get(s, 1, false)) return 1.0f;
    if (a == cell_get(s, 2, false)) return -0.5f;
    if (s.depth == 0) return -0.5f;
    return __fdiv_rn(-0.5f, (float)s.depth);
}

// bit a set <=> action a legal.  puzzle.rs:162-165 / lib.rs:138-145
__device__ __forceinline__ uint32_t env_masks(const EnvParams& p, const EnvState& s) {
    if (p.kind == 0) {
        const int zx = (int)s.blank % p.W, zy = (int)s.blank / p.W;
        return (zx > 0 ? 1u : 0u) | (zy > 0 ? 2u : 0u) | (zx < p.W - 1 ? 4u : 0u) | (zy < p.H - 1 ? 8u : 0u);
    }
    const int a = (int)cell_get(s, 0, false), ax = a % p.W, ay = a / p.W;
    return (ay > 0 ? 1u : 0u) | (ay + 1 < p.H ? 2u : 0u) | (ax > 0 ? 4u : 0u) | (ax + 1 < p.W ? 8u : 0u);
}

// Env::step.  puzzle.rs:135-160 (blank moves 0 left,1 up,2 right,3 down; illegal = no-op; depth
// always saturating -1) / lib.rs:127-136 (0 up,1 down,2 left,3 right; steps_left saturating -1)
template <int F = TWR_CELLS_ANY>
__device__ __forceinline__ void env_step(const EnvParams& p, EnvState& s, int action) {
    if (p.kind == 0) {
        const int z = (int)s.blank, zx = z % p.W, zy = z / p.W;
        int t = -1;
        if (action == 0 && zx > 0) t = z - 1;
        else if (action == 1 && zy > 0) t = z - p.W;
        else if (action == 2 && zx < p.W - 1) t = z + 1;
        else if (action == 3 && zy < p.H - 1) t = z + p.W;
        if (t >= 0) {
            const bool wide = cells_wide<F>(p);
            cell_set(s, z, cell_get(s, t, wide), wide);
            cell_set(s, t, 0, wide);
            s.blank = (uint32_t)t;
        }
    } else {
        int a = (int)cell_get(s, 0, false);
        const int ax = a % p.W, ay = a / p.W;
        if (action == 0 && ay > 0) a -= p.W;
        else if (action == 1 && ay + 1 < p.H) a += p.W;
        else if (action == 2 && ax > 0) a -= 1;
        else if (action == 3 && ax + 1 < p.W) a += 1;
        cell_set(s, 0, (uint32_t)a, false);
    }
    if (s.depth > 0) s.depth -= 1;
}

// board value at cell i as Env::observe / get_state see it.  puzzle.rs:183-185 ; lib.rs:74-81
// (goal 2, trap 3, agent 1 written last so the agent overwrites).
template <int F = TWR_CELLS_ANY>
__device__ __forceinline__ uint32_t env_board(const EnvParams& p, const EnvState& s, int i) {
    if (p.kind == 0) return cell_get(s, i, cells_wide<F>(p));
    const uint32_t a = cell_get(s, 0, false), g = cell_get(s, 1, false), t = cell_get(s, 2, false);
    uint32_t v = 0;
    if ((uint32_t)i == g) v = 2;
    if ((uint32_t)i == t) v = 3;
    if ((uint32_t)i == a) v = 1;
    return v;
}

// Sequential u32 draws of one Philox stream: word k = philox(env_id, k/4, kind, collect_id)[k%4]
struct RngStream {
    uint32_t k0, k1, env_id, kind, cid, next, buf[4];
    __device__ __forceinline__ RngStream(uint64_t seed, uint32_t env, uint32_t kind_, uint32_t cid_)
        : k0((uint32_t)seed), k1((uint32_t)(seed >> 32)), env_id(env), kind(kind_), cid(cid_), next(0) {}
    __device__ __forceinline__ uint32_t draw() {
        if ((next & 3u) == 0) philox4x32_10(env_id, next >> 2, kind, cid, k0, k1, buf);
        const uint32_t i = next++ & 3u;
        return i == 0 ? buf[0] : i == 1 ? buf[1] : i == 2 ? buf[2] : buf[3];
    }
};

// Env::reset with the shared stream.  puzzle.rs:119-133: `difficulty` draws from {0,1,2,3}
// applied through step() (illegal = no-op), then depth = depth_slope*difficulty; draw j is the
// 2-bit field j%16 of stream word j/16.  lib.rs:114-125: agent uniform; goal uniform among cells
// within Manhattan distance `difficulty` (candidates x-outer / y-inner, lib.rs:50-65) rejecting
// the agent cell; trap uniform rejecting agent and goal; steps_left = max_steps.
__device__ __forceinline__ EnvState env_reset(const EnvParams& p, uint64_t seed, uint32_t env_id, uint32_t cid) {
    EnvState s = env_fresh(p);
    RngStream rng(seed, env_id, TWR_RNG_RESET, cid);
    if (p.kind == 0) {
        uint32_t w = 0;
        for (int j = 0; j < p.difficulty; ++j) {
            if ((j & 15) == 0) w = rng.draw();
            env_step(p, s, (int)((w >> (2 * (j & 15))) & 3u));
        }
        s.depth = (uint32_t)(p.depth_slope * p.difficulty);
    } else {
        const uint32_t n = (uint32_t)p.N;
        const int a = (int)mulhi_u32(rng.draw(), n), ax = a % p.W, ay = a / p.W;
        int nc = 0;
        for (int x = 0; x < p.W; ++x)
            for (int y = 0; y < p.H; ++y)
                nc += (abs(x - ax) + abs(y - ay) <= p.difficulty) ? 1 : 0;
        int g = a;
        while (g == a) {
            int k = (int)mulhi_u32(rng.draw(), (uint32_t)nc);
            for (int x = 0; x < p.W && k >= 0; ++x)
                for (int y = 0; y < p.H && k >= 0; ++y)
                    if (abs(x - ax) + abs(y - ay) <= p.difficulty) {
                        if (k == 0) g = y * p.W + x;
                        --k;
                    }
        }
        int t = a;
        while (t == a || t == g) t = (int)mulhi_u32(rng.draw(), n);
        cell_set(s, 0, (uint32_t)a, false); cell_set(s, 1, (uint32_t)g, false); cell_set(s, 2, (uint32_t)t, false);
        s.depth = (uint32_t)p.max_depth;
    }
    return s;
}

// ------------------------------------------------------------ sampling ---
// nn/policy.rs:169-172 + argmax :130-151: argmax_i(l_i - ln|ln u_i|), strict '>', first max wins.
// logf (not __logf) so the oracle's libm and the device agree to <= 1 ulp.
__device__ __forceinline__ int sample_from_logits4(const float l[4], const float u[4], int n) {
    int best = 0;
    float bv = l[0] - logf(fabsf(logf(u[0])));
#pragma unroll
    for (int i = 1; i < TWR_MAX_ACTIONS; ++i) {
        if (i < n) {
            const float g = l[i] - logf(fabsf(logf(u[i])));
            if (g > bv) { bv = g; best = i; }
        }
    }
    return best;
}
