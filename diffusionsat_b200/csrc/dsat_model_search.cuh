// Every model of a formula over n <= 1024 variables by ordered search (dsat_enumerate_models_search): the same list, in the
// same ascending order, as the brute force of dsat_models.cuh, for formulas too large to go through 2^n assignments.
//
// Fixed branching order: a node branches on its highest unassigned variable, 0 before 1.  Inside a subtree every higher
// variable is already fixed, so a depth-first walk meets the models in ascending order of the integer they encode (x1 =
// bit 0).  Unit propagation only fixes what every model of the node fixes, so it leaves that order alone.  A leaf is a node
// where every clause holds: its f unassigned variables are free, and it stands for 2^f models, written as a binary counter
// deposited into the free variables in ascending variable order.
//
// A node is its assignment: two bitsets of `words` 64-bit words, `set` (assigned) and `val` (value; 0 where unassigned).
// The bits of `set` at and above n_vars are always 1, so they never count as unassigned.
//
// Host flow (dsat_api.cu):
//   1. Frontier.  Starting from the root, expand_kernel<false> counts the surviving children of every node (0 for a
//      conflict, 1 for a leaf, which is kept as it is, up to 2 for a branch), scan_kernel turns the counts into offsets
//      and expand_kernel<true> writes the children there: a stable compaction, so the frontier stays in depth-first order.
//      Levels repeat until the frontier holds FRONTIER_TARGET nodes, every node is a leaf, or MAX_LEVELS levels ran.
//   2. Search, CHUNK_NODES frontier nodes per launch: search_kernel<false> writes each node's model count (saturated at
//      2^63, which the host reports as an overflow), scan_kernel makes offsets, search_kernel<true> searches again and
//      writes each node's models at its offset.  Warps take nodes from an atomic cursor in any order: the offsets fix
//      where each node's models go.
//      The count pass needs no order, so it branches on the highest variable of an open clause instead: variables that no
//      open clause holds stay free down to the leaves.  Its work then does not double with each such variable (a formula
//      over 66 variables with the one clause [1, 2] is one branch, 3 * 2^64 models: an overflow found at once).  The emit
//      pass runs only on counts that fit the caller's capacity, so its work is bounded by what it writes.
//
// Propagation in a warp: the 32 lanes evaluate 32 clauses at a time against the warp's bitsets in shared memory.  A clause
// with no true and no unassigned literal is a conflict; one with a single unassigned literal ORs that literal into the
// warp's `pos` / `neg` masks.  After a pass over all clauses the masks are applied at once (a variable in both is a
// conflict) and their variables appended to the trail, which backtracking walks to clear them again.
#pragma once
#include "dsat_common.cuh"

namespace dsat {
namespace msearch {

constexpr int MAX_VARS = 1024;
constexpr int MAX_WORDS = MAX_VARS / 64;
constexpr int WARPS = 8;                                        // warps per block, one node each
constexpr int THREADS = WARPS * 32;
constexpr int FRONTIER_TARGET = 1 << 15;                        // nodes that fill a B200 several times over
constexpr int MAX_LEVELS = 64;                                  // breadth-first levels at most
constexpr int CHUNK_NODES = 1 << 14;                            // frontier nodes per search launch
constexpr int SCAN_THREADS = 1024, SCAN_ITEMS = 4;
constexpr int CLAUSE_SMEM_MAX = 32 * 1024;                      // clause arrays staged in shared memory up to this size
constexpr unsigned long long SAT = 1ull << 63;                  // a saturated count: 2^63 or more models
enum { CONFLICT = 0, LEAF = 1, OPEN = 2 };

// a + b for counts <= SAT, saturated at SAT
__host__ __device__ __forceinline__ unsigned long long sat_add(unsigned long long a, unsigned long long b) {
    const unsigned long long r = a + b;
    return r < a || r > SAT ? SAT : r;
}

// Clauses after the host's normalisation (no empty clause, no tautology, no repeated literal): clause j is the literals
// lit[off[j] .. off[j+1]), each coded var << 1 | negated with var 0-based.
struct Formula {
    const int* off;
    const unsigned short* lit;
    int m, n_vars, words;
};

struct WarpState { unsigned long long set[MAX_WORDS], val[MAX_WORDS], pos[MAX_WORDS], neg[MAX_WORDS]; };

// shared memory of one warp: its state, the output index at each decision (n_vars u64, emit pass), the decision levels
// (n_vars u32) and the trail (n_vars u16)
__host__ __device__ inline int warp_smem_bytes(int n_vars) {
    return (int)sizeof(WarpState) + ((n_vars * 14 + 15) & ~15);
}
__host__ __device__ inline long long clause_smem_bytes(int m, long long nnz) {
    return ((long long)(m + 1) * 4 + nnz * 2 + 15) & ~15ll;
}

// Stage the clause arrays in shared memory when the host reserved room for them (stage != 0) and point F at them; then
// carve this warp's state, levels and trail out of the rest.
__device__ __forceinline__ void setup_block(Formula& F, int stage, long long nnz, WarpState*& s,
                                           unsigned long long*& level_at, unsigned*& levels, unsigned short*& trail) {
    extern __shared__ __align__(16) unsigned char smem[];
    int clause_bytes = 0;
    if (stage) {
        int* s_off = reinterpret_cast<int*>(smem);
        unsigned short* s_lit = reinterpret_cast<unsigned short*>(smem + (size_t)(F.m + 1) * 4);
        for (int j = threadIdx.x; j <= F.m; j += blockDim.x) s_off[j] = F.off[j];
        for (long long q = threadIdx.x; q < nnz; q += blockDim.x) s_lit[q] = F.lit[q];
        __syncthreads();
        F.off = s_off;
        F.lit = s_lit;
        clause_bytes = (int)clause_smem_bytes(F.m, nnz);
    }
    unsigned char* mine = smem + clause_bytes + (size_t)(threadIdx.x >> 5) * warp_smem_bytes(F.n_vars);
    s = reinterpret_cast<WarpState*>(mine);
    level_at = reinterpret_cast<unsigned long long*>(mine + sizeof(WarpState));
    levels = reinterpret_cast<unsigned*>(mine + sizeof(WarpState) + (size_t)F.n_vars * 8);
    trail = reinterpret_cast<unsigned short*>(mine + sizeof(WarpState) + (size_t)F.n_vars * 12);
}

__device__ __forceinline__ void load_node(WarpState* s, const unsigned long long* __restrict__ node, int words, int lane) {
    __syncwarp();                                               // the previous node's state has been read by every lane
    if (lane < words) {
        s->set[lane] = node[lane];
        s->val[lane] = node[words + lane];
        s->pos[lane] = s->neg[lane] = 0ull;
    }
    __syncwarp();
}

__device__ __forceinline__ void store_node(const WarpState* s, unsigned long long* __restrict__ node, int words, int lane) {
    if (lane < words) {
        node[lane] = s->set[lane];
        node[words + lane] = s->val[lane];
    }
}

// Unit propagation to a fixpoint.  Returns CONFLICT, LEAF (every clause holds) or OPEN (no unit left, a clause is open);
// the variables it assigns are appended to trail[tlen...].  On OPEN, open_top = the highest unassigned variable of an
// open clause.  Warp-uniform.
__device__ int propagate(const Formula& F, WarpState* s, unsigned short* trail, int& tlen, unsigned& open_top, int lane) {
    for (;;) {
        bool open = false, unit = false;
        unsigned top = 0;                                       // 1 + highest free variable of this lane's open clauses
        for (int base = 0; base < F.m; base += 32) {
            const int j = base + lane;
            bool conflict = false;
            if (j < F.m) {
                bool sat = false;
                int free_lits = 0;
                unsigned last = 0, clause_top = 0;
                for (int q = F.off[j], e = F.off[j + 1]; q < e; ++q) {
                    const unsigned l = F.lit[q], v = l >> 1;
                    const unsigned long long bit = 1ull << (v & 63);
                    if (s->set[v >> 6] & bit) {
                        if (((s->val[v >> 6] & bit) != 0) != (bool)(l & 1)) { sat = true; break; }
                    } else {
                        ++free_lits;
                        last = l;
                        clause_top = max(clause_top, v + 1);
                    }
                }
                if (!sat) {
                    open = true;
                    top = max(top, clause_top);
                    if (free_lits == 0) conflict = true;
                    else if (free_lits == 1) {
                        unit = true;
                        const unsigned v = last >> 1;
                        atomicOr((last & 1) ? &s->neg[v >> 6] : &s->pos[v >> 6], 1ull << (v & 63));
                    }
                }
            }
            if (__any_sync(0xffffffffu, conflict)) {
                __syncwarp();
                if (lane < F.words) s->pos[lane] = s->neg[lane] = 0ull;
                __syncwarp();
                return CONFLICT;
            }
        }
        if (!__any_sync(0xffffffffu, open)) return LEAF;
        if (!__any_sync(0xffffffffu, unit)) {
            open_top = __reduce_max_sync(0xffffffffu, top) - 1;  // an open clause has two free literals here
            return OPEN;
        }
        __syncwarp();
        unsigned long long p = 0, n = 0;
        if (lane < F.words) {
            p = s->pos[lane];
            n = s->neg[lane];
            s->pos[lane] = s->neg[lane] = 0ull;
        }
        if (__any_sync(0xffffffffu, (p & n) != 0)) { __syncwarp(); return CONFLICT; }    // x and not x both forced
        const unsigned long long fresh = p | n;                 // units are on unassigned variables only
        if (lane < F.words) {
            s->set[lane] |= fresh;
            s->val[lane] |= p;
        }
        const int cnt = __popcll(fresh);
        int incl = cnt;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += t; }
        int at = tlen + incl - cnt;
        for (unsigned long long x = fresh; x; x &= x - 1) {
            DSAT_CHECK(at < F.n_vars);
            trail[at++] = (unsigned short)(lane * 64 + __ffsll((long long)x) - 1);
        }
        tlen += __shfl_sync(0xffffffffu, incl, 31);
        __syncwarp();
    }
}

// unassign trail[keep .. tlen)
__device__ __forceinline__ void undo(WarpState* s, const unsigned short* trail, int keep, int tlen, int lane) {
    __syncwarp();                                               // every lane has finished reading the state
    for (int i = keep + lane; i < tlen; i += 32) {
        const unsigned v = trail[i];
        const unsigned long long clear = ~(1ull << (v & 63));
        atomicAnd(&s->set[v >> 6], clear);
        atomicAnd(&s->val[v >> 6], clear);
    }
    __syncwarp();
}

// assign variable v = b and push it on the trail
__device__ __forceinline__ void decide(const Formula& F, WarpState* s, unsigned short* trail, int& tlen, unsigned v, int b,
                                       int lane) {
    DSAT_CHECK(tlen < F.n_vars);
    if (lane == 0) {
        s->set[v >> 6] |= 1ull << (v & 63);
        if (b) s->val[v >> 6] |= 1ull << (v & 63);
        trail[tlen] = (unsigned short)v;
    }
    ++tlen;
    __syncwarp();
}

// highest unassigned variable (the node is OPEN, so there is one)
__device__ __forceinline__ unsigned highest_unassigned(const Formula& F, const WarpState* s, int lane) {
    const unsigned long long un = lane < F.words ? ~s->set[lane] : 0ull;
    const unsigned ball = __ballot_sync(0xffffffffu, un != 0);
    const int w = 31 - __clz((int)ball);
    const unsigned long long top = __shfl_sync(0xffffffffu, un, w);
    return (unsigned)(w * 64 + 63 - __clzll((long long)top));
}

__device__ __forceinline__ int free_vars(const Formula& F, const WarpState* s, int lane) {
    int f = lane < F.words ? __popcll(~s->set[lane]) : 0;
#pragma unroll
    for (int o = 16; o; o >>= 1) f += __shfl_xor_sync(0xffffffffu, f, o);
    return f;
}

// One breadth-first level.  COUNT (EMIT = false): kids[i] = surviving children of frontier node i, *open_nodes += nodes
// that branch.  EMIT: the children, in order, at next[offsets[i]...].  One warp per node, grid-stride.
// ordered (a frontier the emit pass will walk): branch on the highest unassigned variable, and keep a node whole when that
// variable is in no open clause (branching on it would only copy the node; the node's own search branches on it first, so
// the order holds).  Otherwise (count only) branch on the highest variable of an open clause.
template <bool EMIT>
__global__ void __launch_bounds__(THREADS) expand_kernel(Formula F, int stage, long long nnz, int ordered,
                                                         const unsigned long long* __restrict__ cur, int n_nodes,
                                                         unsigned long long* __restrict__ kids,
                                                         unsigned* __restrict__ open_nodes,
                                                         const unsigned long long* __restrict__ offsets,
                                                         unsigned long long* __restrict__ next, int next_cap) {
    WarpState* s; unsigned long long* level_at; unsigned* levels; unsigned short* trail;
    setup_block(F, stage, nnz, s, level_at, levels, trail);
    const int lane = threadIdx.x & 31;
    const int stride = gridDim.x * WARPS, node_words = 2 * F.words;
    for (int i = blockIdx.x * WARPS + (threadIdx.x >> 5); i < n_nodes; i += stride) {
        load_node(s, cur + (size_t)i * node_words, F.words, lane);
        int tlen = 0;
        unsigned open_top;
        const int st = propagate(F, s, trail, tlen, open_top, lane);
        unsigned long long out = 0;
        if (EMIT) out = offsets[i];
        int alive = 0;
        const unsigned top = st == OPEN ? highest_unassigned(F, s, lane) : 0u;
        if (st == LEAF || (st == OPEN && ordered && top != open_top)) {
            alive = 1;
            if (EMIT) { DSAT_CHECK(out < (unsigned long long)next_cap); store_node(s, next + out * node_words, F.words, lane); }
        } else if (st == OPEN) {
            const unsigned v = ordered ? top : open_top;
            const int base = tlen;
            for (int b = 0; b < 2; ++b) {
                decide(F, s, trail, tlen, v, b, lane);
                if (propagate(F, s, trail, tlen, open_top, lane) != CONFLICT) {
                    if (EMIT) {
                        DSAT_CHECK(out + alive < (unsigned long long)next_cap);
                        store_node(s, next + (out + alive) * node_words, F.words, lane);
                    }
                    ++alive;
                }
                undo(s, trail, base, tlen, lane);
                tlen = base;
            }
            if (!EMIT && lane == 0) atomicAdd(open_nodes, 1u);
        }
        if (!EMIT && lane == 0) kids[i] = alive;
        __syncwarp();
    }
}

// The models of a leaf: model c (c < 2^f) has the node's values and the bits of c deposited into the free variables in
// ascending order.  Models at out index base + c for c < count, `words` words each.
__device__ __forceinline__ void emit_leaf(const Formula& F, const WarpState* s, unsigned long long base,
                                          unsigned long long count, unsigned long long limit,
                                          unsigned long long* __restrict__ out, int lane) {
    for (unsigned long long c = lane; c < count; c += 32) {
        DSAT_CHECK(base + c < limit);
        unsigned long long rest = c;                            // the bits of c not yet deposited
        for (int w = 0; w < F.words; ++w) {
            unsigned long long key = s->val[w];
            for (unsigned long long fm = ~s->set[w]; fm && rest; fm &= fm - 1, rest >>= 1)
                if (rest & 1) key |= fm & (0ull - fm);
            out[(base + c) * F.words + w] = key;
        }
    }
}

// Branch 1 of a variable v in no open clause: the models of branch 0, out[a0, at), with bit v set, at out[at...]
__device__ __forceinline__ void copy_with_bit(const Formula& F, unsigned long long a0, unsigned long long at,
                                              unsigned long long count, unsigned long long limit, unsigned v,
                                              unsigned long long* __restrict__ out, int lane) {
    __syncwarp();                                               // branch 0's keys, written by every lane, are visible
    for (unsigned long long c = lane; c < count; c += 32) {
        DSAT_CHECK(at + c < limit);
        for (int w = 0; w < F.words; ++w)
            out[(at + c) * F.words + w] = out[(a0 + c) * F.words + w] | (w == (int)(v >> 6) ? 1ull << (v & 63) : 0ull);
    }
}

// Depth-first search of frontier nodes taken from *cursor.  COUNT: counts[i] = models below node i (saturated at SAT).
// EMIT: node i's models at out[offsets[i]...], only indices below `limit`; nodes with counts[i] == 0 are skipped.
template <bool EMIT>
__global__ void __launch_bounds__(THREADS) search_kernel(Formula F, int stage, long long nnz,
                                                         const unsigned long long* __restrict__ frontier, int n_nodes,
                                                         unsigned* __restrict__ cursor,
                                                         unsigned long long* __restrict__ counts,
                                                         const unsigned long long* __restrict__ offsets,
                                                         unsigned long long limit, unsigned long long* __restrict__ out) {
    WarpState* s; unsigned long long* level_at; unsigned* levels; unsigned short* trail;
    setup_block(F, stage, nnz, s, level_at, levels, trail);
    const int lane = threadIdx.x & 31, node_words = 2 * F.words;
    constexpr unsigned BRANCH1 = 1u << 31, COPY = 1u << 30;   // a level: trail length | variable << 16 | flags
    for (;;) {
        unsigned i = 0;
        if (lane == 0) i = atomicAdd(cursor, 1u);
        i = __shfl_sync(0xffffffffu, i, 0);
        if (i >= (unsigned)n_nodes) break;
        unsigned long long at = 0, total = 0;
        if (EMIT) {
            at = offsets[i];
            if (at >= limit || counts[i] == 0) continue;
        }
        load_node(s, frontier + (size_t)i * node_words, F.words, lane);
        int tlen = 0, depth = 0;
        for (;;) {
            unsigned open_top;
            const int st = propagate(F, s, trail, tlen, open_top, lane);
            if (st == OPEN) {
                // COUNT branches on the highest variable of an open clause: a higher unassigned variable is in no open
                // clause here nor below, stays unassigned and so counts as free at every leaf, which makes the count the
                // same without the 2^k subtrees of k such variables.  EMIT keeps the ordered branching; when its
                // variable is in no open clause, branch 1 is branch 0's models with that bit set (COPY), not a search.
                const unsigned v = EMIT ? highest_unassigned(F, s, lane) : open_top;
                DSAT_CHECK(depth < F.n_vars);
                if (lane == 0) {
                    levels[depth] = (unsigned)tlen | v << 16 | (EMIT && v != open_top ? COPY : 0u);
                    level_at[depth] = at;
                }
                ++depth;
                decide(F, s, trail, tlen, v, 0, lane);
                continue;
            }
            if (st == LEAF) {
                const int f = free_vars(F, s, lane);
                if (!EMIT) {
                    total = sat_add(total, f >= 63 ? SAT : 1ull << f);
                    if (total == SAT) break;                     // the count overflows: no need to go on
                } else {
                    const unsigned long long n_leaf = 1ull << f, room = limit - at;
                    emit_leaf(F, s, at, n_leaf < room ? n_leaf : room, limit, out, lane);
                    at += n_leaf;
                    if (at >= limit) break;
                }
            }
            bool resumed = false;                                // backtrack to the deepest level still on branch 0
            while (depth > 0) {
                const unsigned L = levels[depth - 1];
                const int keep = (int)(L & 0xffffu);
                undo(s, trail, keep, tlen, lane);
                tlen = keep;
                if (EMIT && (L & COPY) && !(L & BRANCH1)) {
                    const unsigned long long a0 = level_at[depth - 1], n0 = at - a0, room = limit - at;
                    copy_with_bit(F, a0, at, n0 < room ? n0 : room, limit, (L >> 16) & 0x3ffu, out, lane);
                    at += n0;
                    if (at >= limit) break;                      // resumed stays false: the node is done
                    --depth;
                    continue;
                }
                if (!(L & BRANCH1)) {
                    if (lane == 0) levels[depth - 1] = L | BRANCH1;
                    decide(F, s, trail, tlen, (L >> 16) & 0x3ffu, 1, lane);
                    resumed = true;
                    break;
                }
                --depth;
            }
            if (!resumed) break;
        }
        if (!EMIT && lane == 0) counts[i] = total;
        __syncwarp();
    }
}

// offsets[i] = sum of counts[0, i), *total = sum of all n, saturated at SAT (one CTA, SCAN_ITEMS consecutive items per
// thread)
__global__ void __launch_bounds__(SCAN_THREADS) scan_kernel(const unsigned long long* __restrict__ counts, int n,
                                                            unsigned long long* __restrict__ offsets,
                                                            unsigned long long* __restrict__ total) {
    __shared__ unsigned long long warp_tot[SCAN_THREADS / 32];
    __shared__ unsigned long long carry;
    if (threadIdx.x == 0) carry = 0;
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int base = 0; base < n; base += SCAN_THREADS * SCAN_ITEMS) {
        const int i0 = base + threadIdx.x * SCAN_ITEMS;
        unsigned long long v[SCAN_ITEMS], mine = 0;
#pragma unroll
        for (int q = 0; q < SCAN_ITEMS; ++q) { v[q] = i0 + q < n ? counts[i0 + q] : 0ull; mine = sat_add(mine, v[q]); }
        unsigned long long x = mine;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const unsigned long long t = __shfl_up_sync(0xffffffffu, x, o); if (lane >= o) x = sat_add(x, t); }
        if (lane == 31) warp_tot[warp] = x;
        __syncthreads();
        if (warp == 0) {
            unsigned long long w = warp_tot[lane];
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) { const unsigned long long t = __shfl_up_sync(0xffffffffu, w, o); if (lane >= o) w = sat_add(w, t); }
            warp_tot[lane] = w;
        }
        __syncthreads();
        unsigned long long at = sat_add(carry, warp ? warp_tot[warp - 1] : 0ull);
        // x - mine is the warp-exclusive prefix unless saturation hid it; then every later offset is unused anyway
        at = sat_add(at, x == SAT ? SAT : x - mine);
#pragma unroll
        for (int q = 0; q < SCAN_ITEMS; ++q) {
            if (i0 + q < n) offsets[i0 + q] = at;
            at = sat_add(at, v[q]);
        }
        __syncthreads();
        if (threadIdx.x == 0) carry = sat_add(carry, warp_tot[31]);
        __syncthreads();
    }
    if (threadIdx.x == 0) *total = carry;
}

}  // namespace msearch
}  // namespace dsat
