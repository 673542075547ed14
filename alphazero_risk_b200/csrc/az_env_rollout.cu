// az_env_rollout.cu — the translation unit of the environment: az_env.cu itself (included byte for byte: the ncu capture of
// k_env_rollout in profiles/traffic.json is keyed by that file's hash) with az_env_rollout launching k_env_rollout_slots, the pooled
// rollout whose games keep their land bytes in their pool slot.  The previous kernel stays reachable as az_env_rollout_lane_columns
// (profiles/rollout_slots.py times the two side by side); the public API has one rollout.
#include "az_b200.h"

extern "C" AZ_API int az_env_rollout_lane_columns(az_env* e, int n_steps, void* stream);
#define az_env_rollout az_env_rollout_lane_columns
#include "az_env.cu"
#undef az_env_rollout

// ---------------------------------------------------------------- the pooled rollout, land bytes in the slot
// Same pool, categories, sequence-numbered rings and service order rules as k_env_rollout (comment above it in az_env.cu); what
// moves is the game's storage.  There a warp that takes a game copied its 11 land words from the 28-word context into the lane's
// private column (7 x LDS.128 + 11 STS) and back after the move (11 LDS + 7 x STS.128): about 36 warp instructions and a third of
// a warp-step's shared-memory wavefronts, with a store -> load round trip at the head of every move's dependency chain — while the
// rules touch the land bytes about ten times per move.  Here the land words live in a SLOT-indexed column (word w of slot s at
// col[w * ENV_POOL_SLOTS + s]: the first 11 words of EnvSmemWide's column, so the HBM load / store helpers of az_env.cu fill and
// drain it unchanged while thread t owns slot t) and a lane that takes slot s points its AzLandColumn at that slot: the rules read
// and write the game in place.  The context shrinks to the non-land words (4 x uint4, structure of arrays so that the eight lanes
// of a quarter-warp, which hold eight different slot residues, hit eight different 16-byte bank groups); the lane column's other
// 11 words stay the per-lane fortify-DFS parents.
#define ENV_SLOT_CTX_Q 4                         // uint4 per game context: scalars, (ply, done, parked fortify land), own0/own1, gt1/full
static_assert(ENV_POOL_SLOTS == ENV_BLOCK, "the slot land column is the first 11 words of the lane column");

// The queues stay eight rings per category keyed by slot % 8.  Every land word of slot s sits in bank s % 32, so the four lanes of a
// warp that share a ring residue can conflict on land bytes; rings keyed by slot % 32 (one game per lane and ring, conflict-free land
// accesses) were measured and lose 10 %: 22.8 instead of 25.2 games per warp-step (profiles/README.md).

struct EnvSmemSlots {                            // starts like EnvSmemWide / EnvSmem: the per-thread helpers of az_env.cu work on it
    uint64_t tab[AZ_TABLE_U64];
    uint32_t col[ENV_COL_WORDS * ENV_BLOCK];     // words 0..10 per SLOT: the land bytes; words 11..21 per LANE: fortify-DFS parents
    uint64_t lut11[AZ_LUT11_U64];
    uint4 ctx[ENV_SLOT_CTX_Q * ENV_POOL_SLOTS];  // context word q of slot s at ctx[q * ENV_POOL_SLOTS + s]
    uint32_t q[ENV_POOL_NCAT][ENV_POOL_NSUB][ENV_POOL_QSUB];  // cells as in EnvSmemPool: (sequence << 16) | slot
    uint32_t head[ENV_POOL_NCAT][ENV_POOL_NSUB], tail[ENV_POOL_NCAT][ENV_POOL_NSUB];
    int cnt[ENV_POOL_NCAT][ENV_POOL_NSUB];
    uint32_t remaining;
};

__device__ __forceinline__ void slot_load(EnvCtx& c, EnvSmemSlots& sp, int slot, int& done, int& park_li)
{
    const uint4 a = sp.ctx[0 * ENV_POOL_SLOTS + slot], b = sp.ctx[1 * ENV_POOL_SLOTS + slot];
    const uint4 d = sp.ctx[2 * ENV_POOL_SLOTS + slot], f = sp.ctx[3 * ENV_POOL_SLOTS + slot];
    c.land.base = (uint8_t*)sp.col + 4 * slot;
    az_unpack_scalars(c.g, a.x, a.y, a.z, a.w);
    c.ply = b.x; done = (int)b.y; park_li = (int)b.z;
    c.g.own0 = (uint64_t)d.x | ((uint64_t)d.y << 32); c.g.own1 = (uint64_t)d.z | ((uint64_t)d.w << 32);
    c.g.gt1 = (uint64_t)f.x | ((uint64_t)f.y << 32); c.g.full = (uint64_t)f.z | ((uint64_t)f.w << 32);
}

__device__ __forceinline__ void slot_store(const EnvCtx& c, EnvSmemSlots& sp, int slot, int done, int park_li)
{
    sp.ctx[0 * ENV_POOL_SLOTS + slot] = make_uint4((c.g.cards0 << 16) | (c.g.cards1 << 24), az_pack_w11(c.g), az_pack_w12(c.g), az_pack_w13(c.g));
    sp.ctx[1 * ENV_POOL_SLOTS + slot] = make_uint4(c.ply, (uint32_t)done, (uint32_t)park_li, 0u);
    sp.ctx[2 * ENV_POOL_SLOTS + slot] = make_uint4((uint32_t)c.g.own0, (uint32_t)(c.g.own0 >> 32), (uint32_t)c.g.own1, (uint32_t)(c.g.own1 >> 32));
    sp.ctx[3 * ENV_POOL_SLOTS + slot] = make_uint4((uint32_t)c.g.gt1, (uint32_t)(c.g.gt1 >> 32), (uint32_t)c.g.full, (uint32_t)(c.g.full >> 32));
}

__device__ __forceinline__ void slot_push(EnvSmemSlots& sp, int newcat, int slot)
{
    if (newcat >= 0 && newcat < ENV_POOL_NCAT) {
        const int r = slot & (ENV_POOL_NSUB - 1);
        const uint32_t pos = atomicAdd(&sp.tail[newcat][r], 1u);
        volatile uint32_t* e = &sp.q[newcat][r][pos & (ENV_POOL_QSUB - 1)];
        while ((*e >> 16) != (pos & 0xffffu)) { }                        // the cell's previous lap has been taken
        *e = (((pos + 1u) & 0xffffu) << 16) | (uint32_t)slot;
        atomicAdd(&sp.cnt[newcat][r], 1);
    }
}

// as pool_choose: returns (priority << 2) | rotated category, 0 = every queue is empty
__device__ __forceinline__ uint32_t slot_choose(const EnvSmemSlots& sp, int lane, unsigned rot)
{
    const int grp = lane >> 3, sub = lane & 7;
    int a = *reinterpret_cast<const volatile int*>(&sp.cnt[grp][sub]);
    a = a < 0 ? 0 : (a > 4 ? 4 : a);
#pragma unroll
    for (int o = 1; o < 8; o <<= 1) a += __shfl_xor_sync(0xffffffffu, a, o);
    const uint32_t pr = grp >= ENV_CAT_REDEAL ? (a >= ENV_POOL_MIN_BATCH ? 64u + (uint32_t)a : (a ? 1u : 0u)) : (a ? 8u + (uint32_t)a : 0u);
    const uint32_t score = sub == 0 ? (pr << 2) | (((uint32_t)grp + rot) & 3u) : 0u;
    return __reduce_max_sync(0xffffffffu, score);
}

__global__ void __launch_bounds__(ENV_BLOCK, 1) k_env_rollout_slots(uint32_t* __restrict__ st, int n, const uint64_t* __restrict__ g_tab,
                                                                     int n_steps, uint64_t seed, uint32_t first_game, AzRulesDev rules,
                                                                     unsigned long long* __restrict__ counters)
{
    extern __shared__ __align__(16) unsigned char env_dyn_smem[];
    EnvSmemSlots& sp = *reinterpret_cast<EnvSmemSlots*>(env_dyn_smem);
    EnvSmemWide& smw = *reinterpret_cast<EnvSmemWide*>(env_dyn_smem);
    EnvSmem& sm = *reinterpret_cast<EnvSmem*>(env_dyn_smem);
    for (int i = threadIdx.x; i < ENV_POOL_NCAT * ENV_POOL_NSUB * ENV_POOL_QSUB; i += ENV_BLOCK) (&sp.q[0][0][0])[i] = (uint32_t)(i & (ENV_POOL_QSUB - 1)) << 16;
    if (threadIdx.x < ENV_POOL_NCAT * ENV_POOL_NSUB) { (&sp.head[0][0])[threadIdx.x] = 0; (&sp.tail[0][0])[threadIdx.x] = 0; (&sp.cnt[0][0])[threadIdx.x] = 0; }
    if (threadIdx.x == 0) sp.remaining = 0;
    const AzTablesWide T = env_stage_tables_wide(smw, g_tab);              // __syncthreads inside
    const int lane = threadIdx.x & 31;
    const int gi0 = blockIdx.x * ENV_POOL_SLOTS, gi = gi0 + (int)threadIdx.x;
    const bool live = gi < n;
    unsigned games = 0, w0 = 0, w1 = 0, dr = 0;
    EnvCtx c;
    {
        // every thread brings its own game into slot threadIdx.x (env_load writes the land words straight into the slot's column)
        // and queues it
        int cat = -1;
        if (live) {
            env_load(c, sm, st, n, gi);
            cat = pool_classify(c.g, 0, n_steps, rules, games, w0, w1, dr);
            slot_store(c, sp, (int)threadIdx.x, 0, 0);
        } else env_bind(c, sm);
        const int nq = __popc(__ballot_sync(0xffffffffu, cat >= 0 && cat < ENV_POOL_NCAT));
        if (lane == 0 && nq) atomicAdd(&sp.remaining, (uint32_t)nq);
        __threadfence_block();
        slot_push(sp, cat, (int)threadIdx.x);
    }
    __syncthreads();
    unsigned rot = threadIdx.x >> 5;
    const int sub = lane & (ENV_POOL_NSUB - 1), grp = lane >> 3;           // ring this lane is served from; its place in the ring's batch of 4
    uint32_t best = slot_choose(sp, lane, rot);
    for (;;) {
        if ((best >> 2) == 0) {
            if (*reinterpret_cast<volatile uint32_t*>(&sp.remaining) == 0) break;
            __nanosleep(64);
            best = slot_choose(sp, lane, rot);
            continue;
        }
        const int cat = (int)(((best & 3u) - rot) & 3u);
        // lanes 0..7 each take up to 4 games from one ring: reserve 4 at once and give back what was not there
        int kq = 0; uint32_t hq = 0;
        if (lane < ENV_POOL_NSUB) {
            const int old = atomicSub(&sp.cnt[cat][lane], 4);
            kq = old >= 4 ? 4 : (old > 0 ? old : 0);
            if (kq < 4) atomicAdd(&sp.cnt[cat][lane], 4 - kq);
            if (kq) hq = atomicAdd(&sp.head[cat][lane], (uint32_t)kq);
        }
        kq = __shfl_sync(0xffffffffu, kq, sub); hq = __shfl_sync(0xffffffffu, hq, sub);
        const bool has = grp < kq;
        if (!__any_sync(0xffffffffu, has)) { best = slot_choose(sp, lane, rot); continue; }
        ++rot;
        int slot = -1;
        if (has) {
            const uint32_t pos = hq + (uint32_t)grp;
            volatile uint32_t* e = &sp.q[cat][sub][pos & (ENV_POOL_QSUB - 1)];
            uint32_t v;
            while (((v = *e) >> 16) != ((pos + 1u) & 0xffffu)) { }
            *e = ((pos + ENV_POOL_QSUB) & 0xffffu) << 16;
            slot = (int)(v & 0xffffu);
        }
        __threadfence_block();
        int newcat = -1, done = 0, park_li = 0;
        if (slot >= 0) {
            slot_load(c, sp, slot, done, park_li);
            const uint32_t game = first_game + (uint32_t)(gi0 + slot);
            if (cat == ENV_CAT_REDEAL) {
                az_new_game(c.g, c.land, seed, game, c.ply);
                newcat = pool_phase_cat(c.g.phase);
            } else if (cat == ENV_CAT_FORTIFY) {
                az_fortify_finish(c.g, c.land, c.scratch, T, park_li);
                c.ply++; done++;
                newcat = pool_classify(c.g, done, n_steps, rules, games, w0, w1, dr);
            } else if (cat == ENV_CAT_ATTACK) {
                __builtin_assume(c.g.phase == AZ_PH_ATTACK);
                const uint64_t valid = az_valid_moves_flat(c.g, T, rules);
                const az_u32x4 blk = az_rng_block(seed, game, c.ply, AZ_STREAM_REAL, 0);
                const int action = az_nth_set_bit(valid, az_mulhi32(blk.y, (uint32_t)__popcll(valid)));
                az_move_flat(c.g, c.land, T, rules, action, blk.x);
                c.ply++; done++;
                newcat = pool_classify(c.g, done, n_steps, rules, games, w0, w1, dr);
            } else {
                __builtin_assume(c.g.phase != AZ_PH_ATTACK);
                const uint64_t valid = az_valid_moves_flat(c.g, T, rules);
                const az_u32x4 blk = az_rng_block(seed, game, c.ply, AZ_STREAM_REAL, 0);
                const int action = az_nth_set_bit(valid, az_mulhi32(blk.y, (uint32_t)__popcll(valid)));
                if (az_move_flat(c.g, c.land, T, rules, action, blk.x)) { newcat = ENV_CAT_FORTIFY; park_li = action; }
                else { c.ply++; done++; newcat = pool_classify(c.g, done, n_steps, rules, games, w0, w1, dr); }
            }
        }
        best = slot_choose(sp, lane, rot);                                    // before the stores, as in k_env_rollout
        if (slot >= 0) slot_store(c, sp, slot, done, park_li);
        __threadfence_block();
        slot_push(sp, newcat, slot);
        const int nfin = __popc(__ballot_sync(0xffffffffu, newcat == ENV_CAT_NONE));
        if (lane == 0 && nfin) atomicSub(&sp.remaining, (uint32_t)nfin);
    }
    __syncthreads();
    unsigned steps = 0;
    if (live) {
        int done, park_li;
        slot_load(c, sp, (int)threadIdx.x, done, park_li);
        env_store(c, sm, st, n, gi);                                          // reads slot threadIdx.x's land column
        steps = (unsigned)done;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        steps += __shfl_xor_sync(0xffffffffu, steps, o); games += __shfl_xor_sync(0xffffffffu, games, o);
        w0 += __shfl_xor_sync(0xffffffffu, w0, o); w1 += __shfl_xor_sync(0xffffffffu, w1, o); dr += __shfl_xor_sync(0xffffffffu, dr, o);
    }
    if (lane == 0) {
        atomicAdd(&counters[0], (unsigned long long)steps);
        if (games) atomicAdd(&counters[1], (unsigned long long)games);
        if (w0) atomicAdd(&counters[2], (unsigned long long)w0);
        if (w1) atomicAdd(&counters[3], (unsigned long long)w1);
        if (dr) atomicAdd(&counters[4], (unsigned long long)dr);
    }
}

extern "C" int az_env_rollout(az_env* e, int n_steps, void* stream)
{
    AZ_REQUIRE(e != nullptr, "env is NULL");
    AZ_REQUIRE(n_steps >= 0, "n_steps must be >= 0");
    AzDeviceGuard guard(e->device);
    cudaStream_t s = (cudaStream_t)stream;
    AZ_CUDA(cudaEventRecord(e->ev0, s));
    static bool smem_set[64] = { false };                      // wide tables + columns + game contexts: above the 48 KB default
    if (!smem_set[e->device & 63]) {
        AZ_CUDA(cudaFuncSetAttribute(k_env_rollout_slots, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(EnvSmemSlots)));
        smem_set[e->device & 63] = true;
    }
    k_env_rollout_slots<<<env_grid(e->n), ENV_BLOCK, sizeof(EnvSmemSlots), s>>>(e->d_state, e->n, az_device_tables(), n_steps, e->seed,
                                                                                e->first_game, dev_rules(e->rules), e->d_counters);
    AZ_CUDA(cudaGetLastError());
    AZ_CUDA(cudaEventRecord(e->ev1, s));
    e->timed = true;
    return AZ_OK;
}
