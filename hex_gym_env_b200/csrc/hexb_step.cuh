// hexb_step.cuh - the fused env-step kernels (K1/K2/K3) of the batched Hex simulator and their launcher, for ONE board size per
// translation unit (hexb_step_inst.cu instantiates launch_tile<N> for N = HEXB_INST_N).
//
//   hexb_step_kernel<N, KIND, BATCHED>   one warp per chunk of 32 games; BATCHED picks the relabel sweep (several rows per pass
//                                        for launches of at most one wave, one row per pass for deep, issue-bound launches)
//   hexb_coop_kernel<N, KIND>            one CTA of 4 warps per chunk, for sub-wave launches (latency-bound)
#pragma once
#include "hexb_host.h"

using namespace hexb;

// ------------------------------------------------------------------------------------------------ PTX helpers
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
    uint32_t ok = 0;
    for (uint32_t spin = 0; !ok; ++spin) {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(ok)
            : "r"(smem_u32(bar)), "r"(parity)
            : "memory");
        if (spin > (1u << 26)) __trap();  // never hang the GPU: a lost copy becomes a CUDA error
    }
}
// global -> shared bulk copy (TMA 1-D), completes `bytes` on the mbarrier
__device__ __forceinline__ void bulk_g2s(void *dst_smem, const void *src, uint32_t bytes, uint64_t *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst_smem)),
                 "l"(src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
// shared -> global bulk copy
__device__ __forceinline__ void bulk_s2g(void *dst, const void *src_smem, uint32_t bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst), "r"(smem_u32(src_smem)), "r"(bytes) : "memory");
    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
}
// L2 eviction policies for the chunk copies: a fixed part of the state (the first keep_chunks chunks) is marked evict_last and
// stays in the 126 MB L2 from one step to the next, the rest is marked evict_first so that it does not push that part out.
// (Marking ALL of a state larger than L2 evict_last just recreates LRU thrashing: every line is evicted before its reuse.)
__device__ __forceinline__ uint64_t l2_policy(bool keep) {
    uint64_t p;
    if (keep) asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p));
    else asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
    return p;
}
__device__ __forceinline__ void bulk_g2s_hint(void *dst_smem, const void *src, uint32_t bytes, uint64_t *bar, uint64_t policy) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;" ::"r"(
                     smem_u32(dst_smem)),
                 "l"(src), "r"(bytes), "r"(smem_u32(bar)), "l"(policy)
                 : "memory");
}
__device__ __forceinline__ void bulk_s2g_hint(void *dst, const void *src_smem, uint32_t bytes, uint64_t policy) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group.L2::cache_hint [%0], [%1], %2, %3;" ::"l"(dst), "r"(smem_u32(src_smem)),
                 "r"(bytes), "l"(policy)
                 : "memory");
    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
}
__device__ __forceinline__ void bulk_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// ------------------------------------------------------------------------------------------------ step kernel
// One warp = one chunk of 32 games; a CTA is kWarpsPerCta independent warps (no __syncthreads anywhere). Per warp:
//   lane 0 starts ONE bulk asynchronous copy (cp.async.bulk = the 1-D TMA path, completion on the warp's own mbarrier)
//   of the chunk (32 games' label bytes + record words, one contiguous block) into shared memory; meanwhile every lane
//   fetches its game's meta / stream-position words and runs the Philox rounds of the step's two draws; then the
//   thread-per-game plies, the rare finished-game rows, the elementwise obs/mask encode with 16-byte coalesced stores, the
//   warp-per-game relabel sweeps, and one bulk copy of the chunk back to global memory.
constexpr int kWarpsPerCta = 1;   // measured (r1h): 1 warp per CTA 90.0 us, 2: 94.0 us, 4: 94.7 us per 1 Mi-game step (finer-grained tail)
constexpr int kCtaThreads = kWarpsPerCta * kWarp;
// resident CTAs per SM the register allocation should allow (the hardware holds at most 32 CTAs per SM, i.e. 32 warps with one
// warp per CTA; the step kernel uses 56 registers, so registers are not the limit), for large boards whatever the shared-memory
// footprint of the chunk permits
constexpr int min_ctas(int n) {
    const int smem = kWarpsPerCta * 32 * (n * n + 4 * ((n * n + 31) / 32 + 2)) + 64;
    const int by_smem = 220 * 1024 / smem;
    const int want = 10 * 4 / kWarpsPerCta;   // 40 warps per SM (48 registers): measured equal to 48 warps, and no spills
    const int cap = 8 * 4 / kWarpsPerCta;
    return n <= 12 ? (want > 32 ? 32 : want) : (by_smem < 1 ? 1 : (by_smem > cap ? cap : by_smem));
}

template <int N>
struct SmemLayout {
    static constexpr int CHUNK = Geo<N>::CHUNK_STATE;    // labels + records of 32 games
    static constexpr int BAR = kWarpsPerCta * CHUNK;   // multiple of 16
    static constexpr int BYTES = BAR + kWarpsPerCta * 8;
};

template <int N>
__device__ __forceinline__ void encode_loop(const uint4 *src, uint4 *po, uint4 *pm, int lane, int nthr, const Params &P) {
#pragma unroll 4
    for (int i = lane; i < Chunk<N>::VECS; i += nthr) {
        const uint4 x = src[i];
        Vec4 in = {x.x, x.y, x.z, x.w}, o, m;
        encode_vec_k(in, P.one, P.enc_ka, P.enc_kb, P.enc_kc, o, m);
        __stcs(po + i, make_uint4(o.x, o.y, o.z, o.w));
        __stcs(pm + i, make_uint4(m.x, m.y, m.z, m.w));
    }
}
// Everything a slow encode needs, by value: a noinline function must not take the kernel's Params by reference (that would copy the
// whole struct from the constant bank to the stack of every thread).
struct EncArgs {
    void *obs;           // int8 or float32 [.., C]
    uint8_t *mask;
    int obs_f32;
    uint32_t one, ka, kb, kc;
    long long out0, limit;   // element offset of the chunk in the outputs, elements that exist
};
// float32 observations (hexb_config.obs_dtype = HEXB_OBS_F32): one label word = four cells = one 16-byte store per lane, so
// that consecutive lanes write consecutive 16-byte pieces of the [G,N,N] float array
template <int N>
__device__ __forceinline__ void encode_obs_f32(const uint8_t *chunk, const EncArgs &A, int lane, int nthr) {
    const uint32_t *src = reinterpret_cast<const uint32_t *>(chunk);
    float *obs = reinterpret_cast<float *>(A.obs);
    const bool vec_ok = ((((uintptr_t)obs) | (uintptr_t)(4 * A.out0)) & 15) == 0;
    for (int i = lane; i < Chunk<N>::WORDS; i += nthr) {
        uint32_t o, m;
        encode_word_k(src[i], A.one, A.ka, A.kb, A.kc, o, m);
        const float4 f = make_float4((float)(int8_t)(o & 0xffu), (float)(int8_t)((o >> 8) & 0xffu), (float)(int8_t)((o >> 16) & 0xffu),
                                     (float)(int8_t)(o >> 24));
        const long long off = A.out0 + 4ll * i;   // element index
        if (vec_ok && off + 4 <= A.limit) {
            __stcs(reinterpret_cast<float4 *>(obs + off), f);
        } else {
            const float a[4] = {f.x, f.y, f.z, f.w};
            for (int k = 0; k < 4; ++k)
                if (off + k < A.limit) obs[off + k] = a[k];
        }
    }
}
// Every case but the common one (see encode_chunk): float32 observations, one of the two outputs missing, a ragged last chunk,
// unaligned buffers. Out of line: it is a quarter of the step kernel's code and almost never runs.
template <int N>
__device__ __noinline__ void encode_chunk_slow(const uint8_t *chunk, EncArgs A, int lane, int nthr) {
    const uint4 *src = reinterpret_cast<const uint4 *>(chunk);
    uint8_t *obs = reinterpret_cast<uint8_t *>(A.obs);
    uint8_t *msk = A.mask;
    if (A.obs_f32) {
        if (obs) encode_obs_f32<N>(chunk, A, lane, nthr);
        obs = nullptr;   // the byte loop below then writes the mask only
    }
    if (!obs && !msk) return;
    const bool vec_ok = ((((uintptr_t)obs) | ((uintptr_t)msk) | (uintptr_t)A.out0) & 15) == 0;
    for (int i = lane; i < Chunk<N>::VECS; i += nthr) {
        const uint4 x = src[i];
        Vec4 in = {x.x, x.y, x.z, x.w}, o, m;
        encode_vec_k(in, A.one, A.ka, A.kb, A.kc, o, m);
        const long long off = A.out0 + 16ll * i;
        if (vec_ok && off + 16 <= A.limit) {
            if (obs) __stcs(reinterpret_cast<uint4 *>(obs + off), make_uint4(o.x, o.y, o.z, o.w));
            if (msk) __stcs(reinterpret_cast<uint4 *>(msk + off), make_uint4(m.x, m.y, m.z, m.w));
        } else {
            if (obs) store_tail(obs, off, A.limit, o);
            if (msk) store_tail(msk, off, A.limit, m);
        }
    }
}
// (lane, nthr): the calling thread's index among the nthr threads that share the chunk (one warp, or the whole CTA in the
// cooperative form)
template <int N>
__device__ __forceinline__ void encode_chunk(const uint8_t *chunk, const Params &P, long long g0, int t, int lane, int nthr = kWarp) {
    constexpr int C = Geo<N>::C;
    const long long out0 = (g0 + (long long)t * P.G) * C;   // byte offset of the chunk in obs / mask (row t of [T,G,C])
    const long long limit = ((long long)t + 1) * P.G * C;   // bytes of that row that exist in the caller's buffers
    uint8_t *obs = reinterpret_cast<uint8_t *>(P.obs);
    uint8_t *msk = P.mask;
    const bool vec_ok = ((((uintptr_t)obs) | ((uintptr_t)msk) | (uintptr_t)out0) & 15) == 0;
    if (!P.obs_f32 && vec_ok && obs && msk && out0 + Chunk<N>::BYTES <= limit) {
        // the common case (warp-uniform): int8 observations, whole chunk inside the buffers, both outputs wanted, 16-byte aligned.
        // (An explicit L2 evict_first policy on these streaming stores was measured both ways in round 1 - 95.5 -> 92.4 us per
        // 1 Mi-game step in one process layout, 92.3 -> 96.3 us in bench.py on another box - and its code path removed in r2p: every
        // instantiation of this loop that is compiled in but not run costs instruction-cache space in the step kernel.)
        encode_loop<N>(reinterpret_cast<const uint4 *>(chunk), reinterpret_cast<uint4 *>(obs + out0), reinterpret_cast<uint4 *>(msk + out0),
                       lane, nthr, P);
        return;
    }
    const EncArgs A = {P.obs, P.mask, P.obs_f32, P.one, P.enc_ka, P.enc_kb, P.enc_kc, out0, limit};
    encode_chunk_slow<N>(chunk, A, lane, nthr);
}

// The rare per-row views, out of line for the same reason: info["terminal_observation"] of a game that finished in this step
// (term_row_lane) and the opponent's-side observation of a finished, not restarted game (view_row_lane). variant / dtype by value.
template <int N>
__device__ __noinline__ void rare_row_view(const uint8_t *chunk, int r, int8_t *obs, uint8_t *mask, int obs_f32, int variant, bool opp,
                                           long long g, int lane) {
    constexpr int C = Geo<N>::C;
    const uint8_t *Lg = chunk + r * C;
    for (int c = lane; c < C; c += kWarp) {
        uint32_t mk;
        const uint32_t ob = encode_byte(Lg[opp ? transpose_cell<N>(c) : c], variant, opp, mk);
        if (obs) store_obs(obs, obs_f32, g * C + c, ob);
        if (mask) mask[g * C + c] = (uint8_t)mk;
    }
}

// K7: lane 0 adds the warp's packed, reduced statistics (see the packing at the call sites) to the warp's stripe
__device__ __forceinline__ void add_stats(const Params &P, long long wglobal, int lane, uint32_t sa, uint32_t sb) {
    if (lane != 0) return;
    unsigned long long *stripe = reinterpret_cast<unsigned long long *>(P.stats) + 8 * (wglobal & (kStatStripes - 1));
    if (sa) {
        if (sa & 63u) atomicAdd(stripe + 0, (unsigned long long)(sa & 63u));
        if ((sa >> 6) & 63u) atomicAdd(stripe + 1, (unsigned long long)((sa >> 6) & 63u));
        if ((sa >> 12) & 63u) atomicAdd(stripe + 2, (unsigned long long)((sa >> 12) & 63u));
        if ((sa >> 18) & 63u) atomicAdd(stripe + 3, (unsigned long long)((sa >> 18) & 63u));
        if ((sa >> 24) & 63u) atomicAdd(stripe + 5, (unsigned long long)((sa >> 24) & 63u));
        atomicAdd(stripe + 4, (unsigned long long)(sb & 0x3fffu));
    }
    if ((sb >> 14) & 63u) atomicAdd(stripe + 6, (unsigned long long)((sb >> 14) & 63u));
    if (sb >> 20) atomicAdd(stripe + 7, (unsigned long long)(sb >> 20));
}

// KIND_STEP: the instantiation the timed path launches (one env step, nothing else compiled in, step index folded to 0);
// KIND_ROLLOUT: P.steps env steps per launch on the resident chunk (hexb_rollout);
// KIND_OTHER: reset / raw ply / half step, selected at run time by P.mode.
enum : int { KIND_OTHER = 0, KIND_STEP = 1, KIND_ROLLOUT = 2 };
template <int N, int KIND, bool BATCHED>
__global__ void __launch_bounds__(kCtaThreads, min_ctas(N)) hexb_step_kernel(const Params P) {
    constexpr bool STEP_ONLY = KIND != KIND_OTHER;
    extern __shared__ __align__(128) uint8_t smem[];
    using SL = SmemLayout<N>;
    constexpr int C = Geo<N>::C;
    constexpr uint32_t FULL = 0xffffffffu;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    uint8_t *chunk = smem + wid * SL::CHUNK;
    uint64_t *bar = reinterpret_cast<uint64_t *>(smem + SL::BAR) + wid;
    const long long wglobal = (long long)blockIdx.x * kWarpsPerCta + wid;
    const long long g0 = wglobal * kWarp;   // first game of the chunk
    const long long g = g0 + lane;          // this lane's game
    uint8_t *gl = P.state + wglobal * SL::CHUNK;

    // ---- programmatic dependent launch: the step kernels are launched with the programmatic-stream-serialization attribute, so
    //      a launch that follows another kernel on the stream may be set up while that kernel drains; it waits HERE, before its
    //      first global access, until the previous grid has completed and its writes are visible (a no-op without the attribute).
    //      This hides ~2 us of launch gap per step for steps issued one by one (1 Mi games 11x11: 93.6 -> 91.4 us; a CUDA graph
    //      has no such gap). Letting the next grid in EARLY (griddepcontrol.launch_dependents at the top) was measured and
    //      rejected: its waiting CTAs take slots from this grid (65,536 games of 7x7: 9.1 -> 12.7 us per step).
    asm volatile("griddepcontrol.wait;" ::: "memory");

    // ---- chunk in (asynchronous: labels and records in ONE bulk copy); meanwhile the two draws of the (first) step, which
    //      only need the game's meta and stream-position words (two plain loads of lines the bulk copy is fetching anyway)
    const bool use_hint = P.keep_chunks > 0;               // warp-uniform (kernel-uniform)
    const bool keep = wglobal < P.keep_chunks;
    if (lane == 0) {
        mbar_init(bar, 1);
        mbar_expect_tx(bar, SL::CHUNK);
        if (use_hint) bulk_g2s_hint(chunk, gl, SL::CHUNK, bar, l2_policy(keep));
        else bulk_g2s(chunk, gl, SL::CHUNK, bar);
    }
    uint32_t *recw = reinterpret_cast<uint32_t *>(chunk + Geo<N>::CHUNK_LAB) + lane;   // this lane's record word 0 (shared memory)
    uint32_t *lab32 = reinterpret_cast<uint32_t *>(chunk);
    double u_agent = 0.0, u_opp = 0.0;
    Rec<N> rec = {};
    // Params::early (kernel-uniform, set per launch): the record-only half of the step (game_step_pre) runs BEFORE the chunk has
    // landed, on record words fetched with plain coalesced loads - for launches of at most one wave, where every warp waits for
    // its bulk copy at the same moment and the Philox rounds alone do not cover it. Deep launches fetch only meta / draws here.
    const bool early = STEP_ONLY && P.early;
    if (STEP_ONLY && g < P.G) {
        const uint32_t *grec = reinterpret_cast<const uint32_t *>(gl + Geo<N>::CHUNK_LAB) + lane;
        rec.meta = grec[Geo<N>::W * kRecStride];
        rec.draws = grec[(Geo<N>::W + 1) * kRecStride];
        if (early) {
#pragma unroll
            for (int w = 0; w < Geo<N>::W; ++w) rec.occ_rm[w] = grec[w * kRecStride];
        }
        pre_draws(P, rec.meta, rec.draws, (unsigned long long)(P.game_offset + g), u_agent, u_opp);
    }
    __syncwarp();  // the barrier's initialisation is visible to the other lanes
    uint8_t *L = chunk + lane * C;

    // One env step per iteration. hexb_step launches with steps == 1; hexb_rollout runs T steps with the chunk staying in
    // shared memory and the records in registers: the state crosses HBM once per launch instead of once per step.
    const int steps = KIND == KIND_ROLLOUT ? P.steps : 1;
    for (int tt = 0; tt < steps; ++tt) {
        const int t = KIND == KIND_ROLLOUT ? tt : 0;   // a compile-time 0 on the single-step path
        // ---- thread-per-game phase
        uint32_t prmA = 0, prmB = 0, flg = 0;
        if (!STEP_ONLY) {
            mbar_wait(bar, 0);
            load_rec<N>(recw, rec);
        }
        if (STEP_ONLY) {
            if (tt > 0 && g < P.G) pre_draws(P, rec.meta, rec.draws, (unsigned long long)(P.game_offset + g), u_agent, u_opp);
            if (tt == 0 && !early) {
                mbar_wait(bar, 0);
                load_rec<N>(recw, rec);
            }
            Pre pre;
            game_step_pre<N>(P, g, rec, u_agent, u_opp, pre);   // one copy of this code whichever side of the wait it runs on
            if (tt == 0 && early) mbar_wait(bar, 0);
            Loc loc;
            game_step_post<N>(L, P, g, t, rec, pre, loc, prmA, prmB, flg);
            // K7: episode statistics - the eight per-game increments are packed into two words (fields wide enough for the
            // sum over 32 lanes), reduced with two redux.sync, and lane 0 adds the non-zero counters to this warp's stripe
            const uint32_t pa = (uint32_t)loc.st[0] | ((uint32_t)loc.st[1] << 6) | ((uint32_t)loc.st[2] << 12) |
                                ((uint32_t)loc.st[3] << 18) | ((uint32_t)loc.st[5] << 24);
            const uint32_t pb = (uint32_t)loc.st[4] | ((uint32_t)loc.st[6] << 14) | ((uint32_t)loc.st[7] << 20);
            add_stats(P, wglobal, lane, __reduce_add_sync(FULL, pa), __reduce_add_sync(FULL, pb));
        } else if (P.mode == MODE_RESET) {
            game_reset<N>(P, g, rec, flg);
        } else if (P.mode == MODE_HALF) {
            Loc loc;
            game_half<N>(L, P, g, rec, loc, prmA, prmB, flg);
            const uint32_t pa = (uint32_t)loc.st[0] | ((uint32_t)loc.st[1] << 6) | ((uint32_t)loc.st[2] << 12) |
                                ((uint32_t)loc.st[3] << 18) | ((uint32_t)loc.st[5] << 24);
            const uint32_t pb = (uint32_t)loc.st[4] | ((uint32_t)loc.st[6] << 14) | ((uint32_t)loc.st[7] << 20);
            add_stats(P, wglobal, lane, __reduce_add_sync(FULL, pa), __reduce_add_sync(FULL, pb));
        } else {
            game_ply<N>(L, P, g, rec, prmA, flg);
        }
        if ((KIND != KIND_ROLLOUT || tt == steps - 1) && g < P.G) store_rec<N>(recw, rec);
        __syncwarp();  // every game's new stones (and record) are in shared memory

        // ---- warp-per-game row jobs, part 1 (rare): games that finished - terminal observation, clear, opening stone
        uint32_t pending = __ballot_sync(FULL, (flg & (F_RESET | F_TERM)) != 0u);
        while (pending) {
            const int r = __ffs(pending) - 1;
            pending &= pending - 1;
            const uint32_t rf = __shfl_sync(FULL, flg, r);
            if (rf & F_TERM) {   // terminal observation (reads the finished board), then the clear: different lanes touch the same words
                rare_row_view<N>(chunk, r, P.term_obs, nullptr, P.obs_f32, P.variant, (rf & F_TERM_OPP) != 0u, g0 + r + (long long)t * P.G, lane);
                __syncwarp();
            }
            if (rf & F_RESET) clear_row_lane<N>(lab32, r, rf, lane);
            __syncwarp();
        }

        // ---- observation + mask. They depend on emptiness and owner bits only, not on the labels, so they are issued
        //      BEFORE the relabel sweeps: the output stores drain to HBM while the warp works through its relabel rows.
        if ((STEP_ONLY || (P.mode != MODE_PLY && P.mode != MODE_HALF)) && (P.obs || P.mask)) {
            encode_chunk<N>(chunk, P, g0, t, lane);
            uint32_t views = __ballot_sync(FULL, (flg & F_VIEW_OPP) != 0u);  // only without auto-reset: finished by the agent's own ply
            if (views) __syncwarp();
            while (views) {
                const int r = __ffs(views) - 1;
                views &= views - 1;
                rare_row_view<N>(chunk, r, P.obs, P.mask, P.obs_f32, P.variant, true, g0 + r + (long long)t * P.G, lane);
            }
        }

        // ---- row jobs, part 2: relabel sweeps (regions[regions == label] = new label, both plies of the step at once)
        if (!BATCHED) {
            // one row per pass, one word per lane: the faster form when the launch is several waves deep (issue-bound regime)
            const bool need = (flg & (F_RELABEL | F_RESET)) == F_RELABEL;
            RelabelReq q = {0u, 0u, 0u, 0u, 0u};
            if (need) prep_request(prmA, prmB, q);   // each game's own lane decodes its requests once
            const uint32_t all_rows = __ballot_sync(FULL, need);
            const uint32_t extra = __ballot_sync(FULL, need && q.nx != 0u);   // rows with more than one (old -> new) pair
            uint32_t pending = all_rows & ~extra;                             // the common case first: one pair, no inner loop
            while (pending) {
                const int r = __ffs(pending) - 1;
                pending &= pending - 1;
                const uint32_t so = __shfl_sync(FULL, q.so0, r), sn = __shfl_sync(FULL, q.sn0, r);
                relabel_row_lane2<N, false>(lab32, row_desc<N>(r), lane, so, sn, 0u, 0u, 0, P.one);
                __syncwarp();
            }
            pending = extra;
            while (pending) {
                const int r = __ffs(pending) - 1;
                pending &= pending - 1;
                const uint32_t so = __shfl_sync(FULL, q.so0, r), sn = __shfl_sync(FULL, q.sn0, r);
                const uint32_t xo = __shfl_sync(FULL, q.xo, r), xn = __shfl_sync(FULL, q.xn, r), nx = __shfl_sync(FULL, q.nx, r);
                relabel_row_lane2<N, true>(lab32, row_desc<N>(r), lane, so, sn, xo, xn, (int)nx, P.one);
                __syncwarp();
            }
        } else {
            // RPS rows per pass (Sweep<N>): fewer, wider passes shorten a warp's dependent chain - the faster form when the
            // launch is at most about one wave of warps and the step time is a single warp's latency (small batches, rollouts)
            using SW = Sweep<N>;
            const bool need = (flg & (F_RELABEL | F_RESET)) == F_RELABEL;
            uint32_t olds_l = 0, news_l = 0, n_l = 0;
            if (need) canon_request(prmA, prmB, olds_l, news_l, n_l);
            const uint32_t pend_all = __ballot_sync(FULL, need);
            const int sg = lane / SW::LPR, sl = lane % SW::LPR;
            constexpr int CLASSES = (Chunk<N>::ALIGNED_ROWS || SW::RPS == 1) ? 1 : 2;
#pragma unroll
            for (int cls = 0; cls < CLASSES; ++cls) {
                uint32_t pp = CLASSES == 1 ? pend_all : (pend_all & (cls ? 0xaaaaaaaau : 0x55555555u));
                while (pp) {
                    const int row = pick_row<N>(pp, sg);
                    const int srcl = row & 31;
                    const uint32_t o = __shfl_sync(FULL, olds_l, srcl), nw = __shfl_sync(FULL, news_l, srcl);
                    const uint32_t n = __shfl_sync(FULL, n_l, srcl);
                    relabel_rows_lane<N>(lab32, row, sl, o, nw, (int)n, P.one);
                    __syncwarp();
                }
            }
        }
        // the next step's thread-per-game phase writes label bytes other lanes' encode loops have just read
        if (KIND == KIND_ROLLOUT) __syncwarp();
    }

    // ---- chunk out. The next grid on the stream (the next env step) may start launching now: it still waits at its
    //      griddepcontrol.wait for this whole grid to complete and flush, but its CTAs are dispatched and set up while this grid's
    //      chunks drain to global memory: about 1 % on every batch size measured (profiles/r2n_pdl_ab.jsonl). Triggering at the
    //      TOP of the kernel was measured and rejected in round 1.
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    fence_async_smem();  // generic-proxy writes to shared memory -> visible to the async proxy
    __syncwarp();
    if (lane == 0) {
        if (use_hint) bulk_s2g_hint(gl, chunk, SL::CHUNK, l2_policy(keep));
        else bulk_s2g(gl, chunk, SL::CHUNK);
        bulk_wait_read();
    }
}

// ------------------------------------------------------------------------------------------------ cooperative form (sub-wave launches)
// When a launch holds at most about one wave of warps, a step costs one warp's dependent instruction chain (about 2,300
// instructions at 11x11), not bandwidth. This form gives a 32-game chunk to a CTA of WPC = 4 warps instead of one warp (2 and 8
// warps per chunk were measured too and never won, profiles/r2b_forms.jsonl):
//   thread-per-game phase   warp w plays games [w*32/WPC, (w+1)*32/WPC) on its first 32/WPC lanes (the chain of ONE game is what
//                           it is, but a warp now runs the union of the branches of 32/WPC games instead of 32: the restart path
//                           with its extra Philox draws is taken by far fewer warps per step)
//   row jobs + encode       split over all WPC*32 threads: lane group k of the CTA takes the k-th pending row (several rows per
//                           pass like Sweep<N>, WPC times as many), the encode loop strides by the CTA size
// with one __syncthreads between phases (requests and flags go through shared memory instead of shuffles). Rows that share an
// edge word (odd N) are never swept in the same pass: passes are split by row parity, as in the batched warp form.
// Results are bit-identical to the warp form (rows are independent, the encode is elementwise).
constexpr int WPC = 4;   // warps per chunk of the cooperative form
template <int N>
struct CoopSmem {
    static constexpr int CHUNK = Geo<N>::CHUNK_STATE;        // multiple of 16
    static constexpr int BAR = CHUNK;                         // one mbarrier (8 bytes), padded to 16
    static constexpr int FLG = BAR + 16;                      // u32 flg[32]
    static constexpr int OLDS = FLG + 128, NEWS = OLDS + 128, CNT = NEWS + 128;   // canonical relabel requests per game
    static constexpr int MASKS = CNT + 128;                   // u32 [3][8]: per-warp ballots (finished rows, opponent views, relabel rows)
    static constexpr int STATS = MASKS + 96;                  // u32 [2][8]: per-warp packed statistics
    static constexpr int BYTES = STATS + 64;
};

template <int N, int KIND>
__global__ void __launch_bounds__(WPC * 32) hexb_coop_kernel(const Params P) {
    static_assert(KIND == KIND_STEP || KIND == KIND_ROLLOUT, "the cooperative form exists for the env step only");
    extern __shared__ __align__(128) uint8_t smem[];
    using SL = CoopSmem<N>;
    using SW = Sweep<N>;
    constexpr int C = Geo<N>::C;
    constexpr int GPW = kWarp / WPC;          // games per warp
    constexpr int NT = WPC * kWarp;
    constexpr uint32_t FULL = 0xffffffffu;
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    uint8_t *chunk = smem;
    uint64_t *bar = reinterpret_cast<uint64_t *>(smem + SL::BAR);
    uint32_t *s_flg = reinterpret_cast<uint32_t *>(smem + SL::FLG);
    uint32_t *s_olds = reinterpret_cast<uint32_t *>(smem + SL::OLDS);
    uint32_t *s_news = reinterpret_cast<uint32_t *>(smem + SL::NEWS);
    uint32_t *s_cnt = reinterpret_cast<uint32_t *>(smem + SL::CNT);
    uint32_t *s_masks = reinterpret_cast<uint32_t *>(smem + SL::MASKS);
    uint32_t *s_stats = reinterpret_cast<uint32_t *>(smem + SL::STATS);
    const long long wglobal = blockIdx.x;     // chunk index
    const long long g0 = wglobal * kWarp;
    const bool owner = lane < GPW;            // this thread plays a game
    const int gi = wid * GPW + lane;          // its index inside the chunk (owners only)
    const long long g = g0 + gi;
    uint8_t *gl = P.state + wglobal * SL::CHUNK;

    asm volatile("griddepcontrol.wait;" ::: "memory");   // programmatic dependent launch (see hexb_step_kernel)

    const bool use_hint = P.keep_chunks > 0;
    const bool keep = wglobal < P.keep_chunks;
    if (tid == 0) {
        mbar_init(bar, 1);
        mbar_expect_tx(bar, SL::CHUNK);
        if (use_hint) bulk_g2s_hint(chunk, gl, SL::CHUNK, bar, l2_policy(keep));
        else bulk_g2s(chunk, gl, SL::CHUNK, bar);
    }
    uint32_t *recw = reinterpret_cast<uint32_t *>(chunk + Geo<N>::CHUNK_LAB) + gi;
    uint32_t *lab32 = reinterpret_cast<uint32_t *>(chunk);
    double u_agent = 0.0, u_opp = 0.0;
    if (owner && g < P.G) {   // the step's two draws while the chunk is in flight
        const uint32_t *grec = reinterpret_cast<const uint32_t *>(gl + Geo<N>::CHUNK_LAB) + gi;
        pre_draws(P, grec[Geo<N>::W * kRecStride], grec[(Geo<N>::W + 1) * kRecStride], (unsigned long long)(P.game_offset + g), u_agent, u_opp);
    }
    __syncthreads();   // the barrier's initialisation is visible to every thread
    mbar_wait(bar, 0);
    Rec<N> rec;
    if (owner) load_rec<N>(recw, rec);
    uint8_t *L = chunk + gi * C;

    const int steps = KIND == KIND_ROLLOUT ? P.steps : 1;
    for (int tt = 0; tt < steps; ++tt) {
        const int t = KIND == KIND_ROLLOUT ? tt : 0;
        // ---- thread-per-game phase (owners), statistics, requests and flags into shared memory
        uint32_t prmA = 0, prmB = 0, flg = 0, pa = 0, pb = 0;
        if (owner) {
            if (t > 0 && g < P.G) pre_draws(P, rec.meta, rec.draws, (unsigned long long)(P.game_offset + g), u_agent, u_opp);
            Loc loc;
            game_step<N>(L, P, g, t, rec, u_agent, u_opp, loc, prmA, prmB, flg);
            pa = (uint32_t)loc.st[0] | ((uint32_t)loc.st[1] << 6) | ((uint32_t)loc.st[2] << 12) | ((uint32_t)loc.st[3] << 18) |
                 ((uint32_t)loc.st[5] << 24);
            pb = (uint32_t)loc.st[4] | ((uint32_t)loc.st[6] << 14) | ((uint32_t)loc.st[7] << 20);
            if ((KIND != KIND_ROLLOUT || tt == steps - 1) && g < P.G) store_rec<N>(recw, rec);
            const bool need = (flg & (F_RELABEL | F_RESET)) == F_RELABEL;
            uint32_t o = 0, nw = 0, n = 0;
            if (need) canon_request(prmA, prmB, o, nw, n);
            s_flg[gi] = flg;
            s_olds[gi] = o;
            s_news[gi] = nw;
            s_cnt[gi] = n;
        }
        {
            const uint32_t sa = __reduce_add_sync(FULL, pa), sb = __reduce_add_sync(FULL, pb);
            const uint32_t bt = __ballot_sync(FULL, (flg & (F_RESET | F_TERM)) != 0u);
            const uint32_t bv = __ballot_sync(FULL, (flg & F_VIEW_OPP) != 0u);
            const uint32_t br = __ballot_sync(FULL, (flg & (F_RELABEL | F_RESET)) == F_RELABEL);
            if (lane == 0) {
                s_masks[wid] = bt; s_masks[8 + wid] = bv; s_masks[16 + wid] = br;
                s_stats[wid] = sa; s_stats[8 + wid] = sb;
            }
        }
        __syncthreads();   // every game's new stones, record, flags and requests are in shared memory
        uint32_t m_fin = 0, m_view = 0, m_rel = 0;
#pragma unroll
        for (int w = 0; w < WPC; ++w) {
            m_fin |= s_masks[w] << (w * GPW);
            m_view |= s_masks[8 + w] << (w * GPW);
            m_rel |= s_masks[16 + w] << (w * GPW);
        }
        if (tid == 0) {   // K7: one set of atomics per chunk
            uint32_t sa = 0, sb = 0;
#pragma unroll
            for (int w = 0; w < WPC; ++w) { sa += s_stats[w]; sb += s_stats[8 + w]; }
            add_stats(P, wglobal, 0, sa, sb);
        }

        // ---- finished games (CTA-uniform, rare): terminal observation, clear, opening stone; warp k % WPC takes the k-th of them.
        //      Terminal observations only read; the clears of rows that share an edge word (odd N) go in two parity passes.
        if (m_fin) {
            int k = 0;
            for (uint32_t pend = m_fin; pend; pend &= pend - 1, ++k) {
                const int r = __ffs(pend) - 1;
                const uint32_t rf = s_flg[r];
                if ((k % WPC) == wid && (rf & F_TERM)) term_row_lane<N>(chunk, r, rf, P, g0 + r + (long long)t * P.G, lane);
            }
            __syncthreads();
            constexpr int CLASSES = Chunk<N>::ALIGNED_ROWS ? 1 : 2;
#pragma unroll
            for (int cls = 0; cls < CLASSES; ++cls) {
                k = 0;
                for (uint32_t pend = CLASSES == 1 ? m_fin : (m_fin & (cls ? 0xaaaaaaaau : 0x55555555u)); pend; pend &= pend - 1, ++k) {
                    const int r = __ffs(pend) - 1;
                    const uint32_t rf = s_flg[r];
                    if ((k % WPC) == wid && (rf & F_RESET)) clear_row_lane<N>(lab32, r, rf, lane);
                }
                __syncthreads();
            }
        }

        // ---- observation + mask, all threads
        if (P.obs || P.mask) {
            encode_chunk<N>(chunk, P, g0, t, tid, NT);
            if (m_view) {   // only without auto-reset: games the agent's own ply finished are shown from the opponent's side
                __syncthreads();   // these rows' outputs were first written by the whole-chunk encode, possibly by other warps
                int k = 0;
                for (uint32_t pend = m_view; pend; pend &= pend - 1, ++k) {
                    const int r = __ffs(pend) - 1;
                    if ((k % WPC) == wid) view_row_lane<N>(chunk, r, P, g0 + r + (long long)t * P.G, lane);
                }
            }
        }

        // ---- relabel sweeps: lane group q of the CTA (LPR lanes) takes the q-th pending row of the pass's parity class
        if (m_rel) {
            if (P.obs || P.mask) __syncthreads();   // the encode loops have read the label words the sweeps rewrite
            constexpr int CLASSES = Chunk<N>::ALIGNED_ROWS ? 1 : 2;
            const int grp = tid / SW::LPR, sl = tid % SW::LPR;
            constexpr int GROUPS = NT / SW::LPR;
#pragma unroll
            for (int cls = 0; cls < CLASSES; ++cls) {
                const uint32_t pp = CLASSES == 1 ? m_rel : (m_rel & (cls ? 0xaaaaaaaau : 0x55555555u));
                const int cnt = __popc(pp);
                for (int q = grp; q < cnt; q += GROUPS) {
                    const int row = kth_set_bit32(pp, q);
                    relabel_rows_lane<N>(lab32, row, sl, s_olds[row], s_news[row], (int)s_cnt[row], P.one);
                }
                if (CLASSES == 2 && cls == 0) __syncthreads();
            }
        }
        if (KIND == KIND_ROLLOUT && tt + 1 < steps) __syncthreads();   // the next step reads what this one wrote
    }

    // ---- chunk out (no early launch trigger here: with at most one chunk per SM it measured 2 % slower, profiles/r2n_pdl_ab.jsonl)
    fence_async_smem();
    __syncthreads();
    if (tid == 0) {
        if (use_hint) bulk_s2g_hint(gl, chunk, SL::CHUNK, l2_policy(keep));
        else bulk_s2g(gl, chunk, SL::CHUNK);
        bulk_wait_read();
    }
}

// ------------------------------------------------------------------------------------------------ launcher
// number of chunk-warps one wave of the step kernel holds on this device (SMs x resident warps per SM)
static long long wave_warps(int device) {
    static long long cached[64] = {0};
    if (device < 0 || device >= 64) return 148ll * 32;
    long long v = __atomic_load_n(&cached[device], __ATOMIC_RELAXED);
    if (!v) {
        int sms = 0;
        if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device) != cudaSuccess || sms <= 0) sms = 148;
        v = (long long)sms * 32;
        __atomic_store_n(&cached[device], v, __ATOMIC_RELAXED);   // idempotent: racing threads store the same value
    }
    return v;
}

// Warps per chunk (1 or WPC) for a launch of `chunks` chunks (hexb_set_launch_form overrides). Measured on B200 (profiles/r2b_forms.jsonl,
// CUDA-graph step time, 1 / 2 / 4 / 8 warps per chunk): 4,096 games of 6x6 6.16 / 6.16 / 5.88 / 5.93 us; 16,384 games of 7x7
// 6.20 / 6.46 / 6.84 / 9.61; 65,536 games of 7x7 8.12 / 11.2 / 16.1 / 26.0; 131,072 games of 11x11 15.8 / 23.8 / 34.7 / 55.5.
// The cooperative form only shortens the row sweeps and the encode (about a fifth of one warp's chain, profiles/r2b_*): the
// thread-per-game phase is one game's dependent chain whatever the number of warps, and its sparsely populated warps cost issue
// slots as soon as an SM holds more than a few chunks. So it is chosen only while there is at most one chunk per SM.
static int auto_form(long long chunks, int device) {
    const long long sms = wave_warps(device) / 32;
    return chunks <= sms ? WPC : 1;
}

template <int N>
static int set_attrs_once(int dev) {
    // function attributes are per device; std::call_once-style guard per (N, device) (two host threads may create handles at once)
    static int done[64] = {0};
    if (dev >= 0 && dev < 64 && __atomic_load_n(&done[dev], __ATOMIC_ACQUIRE)) return HEXB_OK;
    constexpr int smem = SmemLayout<N>::BYTES;
#define HEXB_ATTR(F, B)                                                                       \
    CK(cudaFuncSetAttribute(F, cudaFuncAttributeMaxDynamicSharedMemorySize, B));             \
    CK(cudaFuncSetAttribute(F, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    HEXB_ATTR((hexb_step_kernel<N, KIND_STEP, false>), smem)
    HEXB_ATTR((hexb_step_kernel<N, KIND_STEP, true>), smem)
    HEXB_ATTR((hexb_step_kernel<N, KIND_ROLLOUT, false>), smem)
    HEXB_ATTR((hexb_step_kernel<N, KIND_ROLLOUT, true>), smem)
    HEXB_ATTR((hexb_step_kernel<N, KIND_OTHER, false>), smem)
    HEXB_ATTR((hexb_coop_kernel<N, KIND_STEP>), CoopSmem<N>::BYTES)
    HEXB_ATTR((hexb_coop_kernel<N, KIND_ROLLOUT>), CoopSmem<N>::BYTES)
#undef HEXB_ATTR
    if (dev >= 0 && dev < 64) __atomic_store_n(&done[dev], 1, __ATOMIC_RELEASE);   // setting the attributes twice is harmless
    return HEXB_OK;
}

template <int N>
static int launch_tile(const hexb_env *e, const Params &P, cudaStream_t s) {
    const int rc = set_attrs_once<N>(e->cfg.device);
    if (rc != HEXB_OK) return rc;
    cudaLaunchConfig_t lc = {};
    lc.stream = s;
    cudaLaunchAttribute la[1];
    la[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    la[0].val.programmaticStreamSerializationAllowed = 1;
    lc.attrs = la;
    lc.numAttrs = 1;
    const long long chunks = P.Gpad / kWarp;
    // The record-only half of the step before the chunk has landed (Params::early): while a launch is at most one wave of warps
    // every warp waits for its bulk copy at the same time, and the copy of a whole wave's chunks takes longer than the Philox
    // rounds that used to cover it. Measured on one box (profiles/r2p_early_ab.jsonl, us per step off / on): 11x11 32,768 games
    // 8.01 / 7.88, 65,536 10.29 / 10.14, 131,072 15.43 / 15.14; 7x7 65,536 8.23 / 8.11, 131,072 12.49 / 12.35; 19x19 65,536
    // 17.1 / 16.9; no change at 4,096 games; 1 Mi games of 11x11 99.7 / 101.3 (deep launches hide the wait behind other warps and
    // pay for the second fetch of the record words), hence by launch depth.
    Params Q = P;
    Q.early = chunks <= wave_warps(e->cfg.device) ? 1 : 0;
    int form = 1;
    if (P.mode == MODE_STEP) form = e->launch_form ? e->launch_form : auto_form(chunks, e->cfg.device);
    if (form == WPC) {   // cooperative form: one CTA of WPC warps per chunk
        lc.gridDim = dim3((unsigned)chunks);
        lc.blockDim = dim3(WPC * kWarp);
        lc.dynamicSmemBytes = CoopSmem<N>::BYTES;
        if (P.steps == 1) CK(cudaLaunchKernelEx(&lc, hexb_coop_kernel<N, KIND_STEP>, Q));
        else CK(cudaLaunchKernelEx(&lc, hexb_coop_kernel<N, KIND_ROLLOUT>, Q));
        CK(cudaGetLastError());
        return HEXB_OK;
    }
    lc.gridDim = dim3((unsigned)(P.Gpad / kCtaThreads));
    lc.blockDim = dim3(kCtaThreads);
    lc.dynamicSmemBytes = SmemLayout<N>::BYTES;
    // Which relabel sweep: several rows per pass shortens a warp's dependent chain and pays while the SMs are sparsely filled;
    // one row per pass executes fewer instructions and wins once a launch is issue- or bandwidth-bound. Measured on the same box
    // (profiles/r2i_sweep_ab.jsonl, us per step batched / one-row): 11x11 32,768 games 7.79 / 8.12, 65,536 10.25 / 10.11, 131,072
    // 15.69 / 15.11, 1 Mi 106.4 / 94.9; 7x7 65,536 8.04 / 8.34, 131,072 12.13 / 12.14; 19x19 65,536 17.47 / 17.14. Short rows
    // (small boards) leave most lanes of a one-row pass idle, so the cross-over comes later there.
    const long long sms = wave_warps(e->cfg.device) / 32;
    const bool small = chunks <= sms * (N <= 8 ? 28 : 12);
    if (P.mode == MODE_STEP && P.steps == 1) {
        if (small) CK(cudaLaunchKernelEx(&lc, hexb_step_kernel<N, KIND_STEP, true>, Q));
        else CK(cudaLaunchKernelEx(&lc, hexb_step_kernel<N, KIND_STEP, false>, Q));
    } else if (P.mode == MODE_STEP) {
        if (small) CK(cudaLaunchKernelEx(&lc, hexb_step_kernel<N, KIND_ROLLOUT, true>, Q));
        else CK(cudaLaunchKernelEx(&lc, hexb_step_kernel<N, KIND_ROLLOUT, false>, Q));
    } else {
        CK(cudaLaunchKernelEx(&lc, hexb_step_kernel<N, KIND_OTHER, false>, Q));
    }
    CK(cudaGetLastError());
    return HEXB_OK;
}
