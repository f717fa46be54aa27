// render_pool.cuh -- the pooled render kernel: paths live in a per-warp POOL in shared memory, not in lanes.
// (included by kernels.cu inside its anonymous namespace, after shade_event / geodesic_step / geodesic_scan;
// the work counters of bt_render_stats come from render_kernel_stats: they are properties of the paths,
// which are the same in both kernels)
//
// render_body (kernels.cu) binds a lane to one pixel and one path at a time; whenever a lane's path
// waits for a phase that the warp is not running (a pending chord, a resolved segment, a finished
// path) the lane idles: 18..21 of 32 lanes were active per instruction on the shipped scenes.
// Here a warp owns P = 32 W path SLOTS in shared memory (flight state F: position, direction,
// travelled length, free distance, pending chord, hit; path state Q: RNG, throughput, counters, AOV
// latches) and runs one PHASE at a time on the 32 slots that need it:
//
//   REGEN  retire finished paths into their pixel's sum IN PATH ORDER, hand finished pixels back,
//          start new camera paths in idle slots (ray generation, mod.rs:244-320)
//   STEP   (lens field) RK4 steps; a lane keeps its flight in registers while it can fly, and the lanes
//          whose flight left the FLY state are refilled from the stack of parked flights: lane compaction
//   SCAN   pending chords / straight segments against the scene (try_hit, mod.rs:389-427)
//   SHADE  resolved segments: shade_event (sample_surface / sample_volume / sample_root)
//
// The next phase is the one with the most slots waiting (a ballot-compacted list in shared memory: the
// "warp-shuffle ballot queues" of the north star), so every pass runs with a full or nearly full warp.
// A lane is a PIXEL STREAM: it owns one pixel at a time (its sum lives in registers) -- pixel `lane` of the
// warp's k-th 8 x 4 tile -- and issues its pixel's paths in the reference's order (pass-major, sub-pixel
// minor, mod.rs:277-278).  The warps of the persistent grid draw their tiles from ONE global counter
// (dynamic: a tile under the lens costs several times a tile of sky, and a static split left the slowest
// warp 10 % behind the average); the lanes of a warp advance through the warp's tiles at their own pace,
// at most POOL_TILES tiles apart.  Paths finish out of
// order; a finished path keeps its slot (state DONE, contribution in place of the throughput) until the
// pixel's earlier paths have been added, so the pixel sum is formed in exactly the order render_body
// forms it: the two kernels give bit-identical images, whatever the scheduling.
#pragma once

enum {
    ST_IDLE = 0, ST_DONE = 1,
    ST_FLY = FL_FLY + 2, ST_PEND = FL_PEND + 2, ST_PEND_FAR = FL_PEND_FAR + 2, ST_PEND_STRAIGHT = 5,
    ST_HIT = FL_HIT + 2, ST_HIT_FAR = FL_HIT_FAR + 2, ST_ESCAPED = FL_ESCAPED + 2, ST_CAPTURED = FL_CAPTURED + 2,
    ST_HIT_STRAIGHT = 10,
    ST_NODE = 11, ST_LEAF = 12  // BVH scenes: a traversal waiting at an inner node / holding a leaf
};
#ifndef BT_POOL_BVH_K
#define BT_POOL_BVH_K 8
#endif
enum { POOL_BVH_K = BT_POOL_BVH_K };  // traversal stack levels of a slot kept in shared memory (the rest: the arena)
enum { POOL_RING = 16 };  // paths of one pixel in flight at most (in-order retirement window)
enum { POOL_TILES = 8 };  // window of tiles a warp's lanes may be spread over

struct Pool {
    // F, a flight:  fa = (x, travelled)  fb = (v, free)  fc = (rest, near, steps, h.t)  fd = (xp, h.prim | face)
    //    a straight ray (flat field): fa = (o, h.t)  fb = (d, h.prim | face) only
    float4 *fa, *fb, *fc, *fd;
    uint4 *qa, *qb;             // Q: xoshiro256++ state
    float4* qc;                 //    (T, misc)   misc = ring index | latched << 4 | (vol_obj + 1) << 5 | bounce << 12 | volume bounce << 20
    float4 *qe, *qf;            //    AOV latches (albedo, depth) (normal, -)   [CT_AOV kernels]
    uint2* tv;                  // BVH: (node reference, stack height)
    uint32_t* bstack;           // BVH: traversal stacks (BvhStack: stride P, POOL_BVH_K levels)
    uint2* bover;               // BVH: the stack levels beyond, BVH_STACK - POOL_BVH_K per slot (arena)
    uint8_t *st, *list, *stack, *ring;
    unsigned long long* tiles;  // the warp's window of tile indices: tile k of its stream is tiles[k % POOL_TILES]
};
// misc packs the counters of a path into 8 bits each: the pooled kernel serves the calls within POOL_MAX_BOUNCES and
// POOL_MAX_OBJECTS (variants.h: render_family; the lane kernel renders the others)
BT_DEV uint32_t pack_misc(uint32_t ring, bool latched, int vol_obj, uint32_t bounce, uint32_t vb) {
    return ring | (latched ? 16u : 0u) | ((uint32_t)(vol_obj + 1) << 5) | (bounce << 12) | (vb << 20);
}
// Bytes of one warp's pool.  Shared memory holds what the STEP and SCAN phases touch: the flights F, the slot states
// and the queues.  The path state Q (48 B per slot, + 32 B of AOV latches) is read and written once per EVENT (1.5 .. 5
// per path) by SHADE / REGEN only and lives in global memory (an L2-resident scratch arena of the engine,
// pool_q_bytes per warp of the persistent grid): the shared memory it would take is worth two more CTAs per SM.
__host__ __device__ inline size_t pool_warp_bytes(uint32_t w, bool lens, bool bvh = false) {
    const size_t P = 32u * w;
    return P * (lens ? 64 : 32) + (bvh ? P * (8 + POOL_BVH_K * 8) : 0) + POOL_TILES * 8 + 3 * P + POOL_RING * 32;
}
__host__ __device__ inline size_t pool_q_bytes(uint32_t w, bool bvh = false) {
    return (size_t)32u * w * (80 + (bvh ? (BVH_STACK - POOL_BVH_K) * 8 : 0));
}
template <bool LENS, bool AOV, bool BVH>
BT_DEV Pool pool_carve(char* base, char* qbase, uint32_t P) {
    Pool pl;
    float4* f = reinterpret_cast<float4*>(base);
    pl.fa = f; f += P;
    pl.fb = f; f += P;
    pl.fc = pl.fd = f;
    if (LENS) { pl.fc = f; f += P; pl.fd = f; f += P; }
    pl.tv = reinterpret_cast<uint2*>(f);
    pl.bstack = reinterpret_cast<uint32_t*>(pl.tv + P);
    if (BVH) f = reinterpret_cast<float4*>(pl.bstack + 2 * POOL_BVH_K * P);
    pl.tiles = reinterpret_cast<unsigned long long*>(f);
    uint8_t* b = reinterpret_cast<uint8_t*>(pl.tiles + POOL_TILES);
    pl.st = b; b += P;
    pl.list = b; b += P;
    pl.stack = b; b += P;
    pl.ring = b;
    float4* q = reinterpret_cast<float4*>(qbase);
    pl.qa = reinterpret_cast<uint4*>(q);
    pl.qb = reinterpret_cast<uint4*>(q + P);
    pl.qc = q + 2 * P;
    pl.qe = q + 3 * P;
    pl.qf = q + 4 * P;
    pl.bover = reinterpret_cast<uint2*>(q + 5 * P);
    return pl;
}
// The slots whose state lies in [lo, hi], compacted into pl.list (ballot + popc); stops once 32 are found.
// Home slots are visited starting at row w0 so that no row of the pool is served last every time.
BT_DEV uint32_t pool_collect(const Pool& pl, uint32_t W, uint32_t w0, int lo, int hi, int lane) {
    const unsigned lt = (1u << lane) - 1u;
    uint32_t n = 0;
    for (uint32_t i = 0; i < W && n < 32; ++i) {
        uint32_t w = w0 + i;
        if (w >= W) w -= W;
        const uint32_t s = w * 32 + lane;
        const int v = pl.st[s];
        const bool m = v >= lo && v <= hi;
        const unsigned b = __ballot_sync(0xffffffffu, m);
        if (m) pl.list[n + __popc(b & lt)] = (uint8_t)s;
        n += __popc(b);
    }
    __syncwarp();
    return n;
}
BT_DEV uint32_t pack_hit(const Hit& h) { return ((uint32_t)(h.prim + 1) << 4) | (uint32_t)(h.face & 15); }
BT_DEV void unpack_hit(uint32_t w, Hit& h) {
    h.prim = (int)(w >> 4) - 1;
    h.face = (int)(w & 15);
}

// PSTATS: scheduling counters (bt_render_pool_stats; never timed): p.stats[0..11] = STEP iterations, flying lanes summed
// over them, refill rounds, STEP entries, SCAN passes, slots scanned, SHADE passes, slots shaded, REGEN passes,
// paths issued, paths retired, turns; [12..16] = SM clocks the warps spent in STEP, SCAN, SHADE, REGEN and in the kernel;
// [17..20] = free-distance grid refreshes: STEP iterations in which any lane refreshed, those in which lanes inside and
// outside the grid's box both did, lanes refreshed from a cell of the grid, lanes refreshed outside its box
template <bool LENS, bool EXACT, int NL, int C, bool PSTATS = false, bool BVH = false>
BT_DEV void render_pool_body(const RenderParams& p) {
    static_assert(!(BVH && LENS), "the pooled traversal serves flat fields (a lensed BVH scene renders through render_body)");
    extern __shared__ float4 smem[];
    const SceneView sc = stage_scene<BVH>(p, smem);
    const typename LensSel<NL>::type lens = LensSel<NL>::make(sc.lens, (int)p.scene.n_lens);
    Consts k;
    k.tau_scale = p.tau_scale;
    k.one_scale = p.one_scale;
    constexpr bool AOV = (C & CT_AOV) != 0;
    constexpr bool VOL = (C & CT_VOLUMES) != 0;

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const unsigned lt = (1u << lane) - 1u;
    const uint32_t W = p.pool_w, P = 32u * W;
    const Pool pl = pool_carve<LENS, AOV, BVH>(reinterpret_cast<char*>(smem + p.scene.stage_f4) + warp * pool_warp_bytes(W, LENS, BVH),
                                               p.pool_q + ((size_t)blockIdx.x * (blockDim.x >> 5) + warp) * pool_q_bytes(W, BVH), P);
    for (uint32_t w = 0; w < W; ++w) pl.st[w * 32 + lane] = ST_IDLE;
    __syncwarp();

    // ---- this lane's pixel stream: pixel (lane & 7, lane >> 3) of the warp's tile number `seq` ---------------------
    // Up to TWO pixels are open per lane: A, the older one, whose paths are being retired (they retire in issue order, so every
    // finished path belongs to A until A is complete), and B, which the lane starts issuing as soon as A's last path is out --
    // a lane never waits for the slowest path of a pixel before it starts the next one (calls of a few paths per pixel: the
    // reference's progressive loop renders ONE pass per call, and a frame split over 8 GPUs leaves 8 spp per call).
    // (everything that is only needed when a pixel starts or ends is recomputed there: the STEP loop is short of registers)
    uint32_t seq = 0;       // the next tile of the warp's stream this lane will take a pixel from
    uint32_t fetched = 0;   // tiles the warp has drawn from the global counter so far (warp-uniform)
    bool exhausted = false;
    uint32_t n_pix = 0;     // open pixels: 0, 1 (A) or 2 (A and B)
    uint32_t ax = 0, ay = 0, a_issued = 0, a_retired = 0, bx = 0, by = 0, b_issued = 0;
    uint32_t tot_issued = 0, tot_retired = 0;   // running path counters of this lane (the ring of in-flight paths is indexed by them)
    V3 acc = v3(0.0f, 0.0f, 0.0f);              // the sum of A's retired paths
    uint32_t sub_i = 0, sub_j = 0;              // sub-pixel of the next path of the pixel being issued

    // warp-uniform queue sizes
    uint32_t n_fly = 0 /* parked on pl.stack */, n_pend = 0, n_res = 0, n_done = 0, n_free = P;
    uint32_t n_node = 0, n_leaf = 0;  // BVH: traversals at an inner node / holding a leaf (n_pend stays 0)
    bool regen_futile = false;
    uint32_t turn = 0, w0 = 0;  // w0: the pool row the slot lists start at (rotates)
    uint32_t ps[16] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0};  // PSTATS only (warp-uniform)
    long long pc[5] = {0, 0, 0, 0, 0}, pc_t0 = 0;            // PSTATS only: SM clocks in STEP / SCAN / SHADE / REGEN, and in all
    if (PSTATS) pc_t0 = clock64();

#pragma unroll 1
    for (;;) {
        ++turn;
        // ---- the phase with the most slots waiting ----------------------------------------------
        const uint32_t c_step = LENS ? min(n_fly, 32u) : 0u, c_scan = min(n_pend, 32u), c_shade = min(n_res, 32u);
        const uint32_t c_regen = regen_futile ? 0u : min(n_free + n_done, 32u);
        const uint32_t c_node = BVH ? min(n_node, 32u) : 0u, c_leaf = BVH ? min(n_leaf, 32u) : 0u;
        const uint32_t best = max(max(max(c_step, c_scan), max(c_shade, c_regen)), max(c_node, c_leaf));
        if (best == 0) break;
        if (++w0 >= W) w0 = 0;

        long long pc_in = 0;
        if (PSTATS) pc_in = clock64();
        int pc_phase = 3;
        if (LENS && c_step == best) {
            if (PSTATS) pc_phase = 0;
            // ================================ STEP ================================
            // A lane keeps its flight in registers while it flies.  Lanes whose flight left the FLY state
            // (a chord to intersect, an escape, a capture) write it back and take another one from the
            // stack of parked flights -- once `pool_refill` more lanes are waiting, so that the bookkeeping
            // is paid every other step, not every step.  The phase ends when the stack is empty and fewer
            // lanes fly than another phase has slots waiting.
            int slot = -1, fs = FL_FLY;
            P3 x = p3(make_float2(0.0f, 0.0f), 0.0f), v = x;  // the stepper's paired layout: no conversion per step
            Flight f;
            flight_reset(f);
            uint32_t round_at = 0;  // a refill round runs once this many lanes wait (0: at once)
            if (PSTATS) ++ps[3];
#pragma unroll 1
            for (;;) {
                const bool waiting = slot < 0 || fs != FL_FLY;
                const unsigned m_wait = __ballot_sync(0xffffffffu, waiting);
                if ((uint32_t)__popc(m_wait) >= round_at) {
                    if (PSTATS) ++ps[2];
                    // write back the flights that left the FLY state
                    const bool left = slot >= 0 && waiting;
                    const bool pend = fs == FL_PEND || fs == FL_PEND_FAR;
                    if (left) {
                        pl.fa[slot] = make_float4(x.xy.x, x.xy.y, x.z, f.travelled);
                        pl.fb[slot] = make_float4(v.xy.x, v.xy.y, v.z, f.free);
                        pl.fc[slot] = make_float4(f.rest, __int_as_float(f.near), __uint_as_float(f.steps), 0.0f);
                        pl.fd[slot] = make_float4(f.xp.xy.x, f.xp.xy.y, f.xp.z, 0.0f);
                        pl.st[slot] = (uint8_t)(fs + 2);
                    }
                    const uint32_t n_left = __popc(__ballot_sync(0xffffffffu, left)), n_lp = __popc(__ballot_sync(0xffffffffu, left && pend));
                    n_pend += n_lp;
                    n_res += n_left - n_lp;
                    // refill from the stack of parked flights: every waiting lane is empty now
                    const uint32_t n_wait = __popc(m_wait), take = min(n_wait, n_fly);
                    slot = waiting ? -1 : slot;
                    if (waiting && (uint32_t)__popc(m_wait & lt) < take) {
                        slot = pl.stack[n_fly - 1 - __popc(m_wait & lt)];
                        const float4 a = pl.fa[slot], b = pl.fb[slot], c = pl.fc[slot];
                        x = p3(a);
                        v = p3(b);
                        f.travelled = a.w;
                        f.free = b.w;
                        f.rest = c.x;
                        f.near = __float_as_int(c.y);
                        f.steps = __float_as_uint(c.z);
                        fs = FL_FLY;
                    }
                    n_fly -= take;
                    const uint32_t unfilled = n_wait - take;
                    round_at = min(unfilled + p.pool_refill, 32u);
                    if (n_fly == 0) {
                        // leave when another phase would run with more lanes than keep flying here
                        const uint32_t flying = 32u - unfilled;
                        const uint32_t other = max(max(min(n_pend, 32u), min(n_res, 32u)), regen_futile ? 0u : min(n_free + n_done, 32u));
                        if (flying == 0 || (flying < other && flying < p.pool_step_min)) break;
                    }
                }
                if (PSTATS) {
                    ++ps[0];
                    ps[1] += __popc(__ballot_sync(0xffffffffu, slot >= 0 && fs == FL_FLY));
                }
                if (PSTATS) {
                    int rf = 0;
                    if (slot >= 0 && fs == FL_FLY) fs = geodesic_step<EXACT, C>(p, lens, sc.prims, x, v, f, p.clip_max, &rf);
                    const uint32_t n_in = __popc(__ballot_sync(0xffffffffu, rf == 1)), n_out = __popc(__ballot_sync(0xffffffffu, rf == 2));
                    ps[12] += (n_in + n_out) != 0;
                    ps[13] += n_in != 0 && n_out != 0;
                    ps[14] += n_in;
                    ps[15] += n_out;
                } else if (slot >= 0 && fs == FL_FLY) {
                    fs = geodesic_step<EXACT, C>(p, lens, sc.prims, x, v, f, p.clip_max);
                }
            }
            // park the flights still flying
            {
                const bool fly = slot >= 0;
                const unsigned m = __ballot_sync(0xffffffffu, fly);
                if (fly) {
                    pl.fa[slot] = make_float4(x.xy.x, x.xy.y, x.z, f.travelled);
                    pl.fb[slot] = make_float4(v.xy.x, v.xy.y, v.z, f.free);
                    pl.fc[slot] = make_float4(f.rest, __int_as_float(f.near), __uint_as_float(f.steps), 0.0f);
                    pl.stack[n_fly + __popc(m & lt)] = (uint8_t)slot;
                }
                n_fly += __popc(m);
            }
            __syncwarp();
        } else if (BVH && c_node == best) {
            if (PSTATS) pc_phase = 1;
            // ================================ NODE ================================
            // BVH scenes: the SCAN phase is a traversal, run as two kinds of unit on the slots that want them -- here
            // visits of 4-wide inner nodes (up to steps_per_turn in a row while a slot stays at an inner node), below
            // leaf tests.  Each runs with a full warp of rays that need exactly that, whatever their origin.
            const uint32_t n = min(pool_collect(pl, W, w0, ST_NODE, ST_NODE, lane), 32u);
            bool to_leaf = false, resolved = false;
            if ((uint32_t)lane < n) {
                const int slot = pl.list[lane];
                const float4 a = pl.fa[slot], b = pl.fb[slot];
                const uint2 tv = pl.tv[slot];
                const V3 o = v3(a), d = v3(b);
                BvhTrav t;
                t.cur = tv.x;
                t.sp = tv.y;
                t.h.t = a.w;
                BvhStack bs;
                bs.base = pl.bstack;
                bs.stride = P;
                bs.idx = (uint32_t)slot;
                bs.k = min(p.bvh_stack_k, (uint32_t)POOL_BVH_K);
                bs.over = pl.bover + (size_t)slot * (BVH_STACK - POOL_BVH_K);
                const V3 inv = v3(m_rcp(d.x), m_rcp(d.y), m_rcp(d.z));
                const uint32_t sgn = bvh_signs(inv);
#pragma unroll 1
                for (uint32_t r = 0; r < p.steps_per_turn && !(t.cur & BVH_LEAF); ++r) bvh_node(t, sc.nodes, bs, o, inv, sgn, p.clip_min);
                pl.tv[slot] = make_uint2(t.cur, t.sp);
                if (t.cur == BVH_DONE) {
                    pl.st[slot] = ST_HIT_STRAIGHT;
                    resolved = true;
                } else if (t.cur & BVH_LEAF) {
                    pl.st[slot] = ST_LEAF;
                    to_leaf = true;
                }
            }
            const uint32_t n_tl = __popc(__ballot_sync(0xffffffffu, to_leaf)), n_rs = __popc(__ballot_sync(0xffffffffu, resolved));
            n_node -= n_tl + n_rs;
            n_leaf += n_tl;
            n_res += n_rs;
            if (PSTATS) {
                ++ps[4];
                ps[5] += n;
            }
            __syncwarp();
        } else if (BVH && c_leaf == best) {
            if (PSTATS) pc_phase = 1;
            // ================================ LEAF ================================
            const uint32_t n = min(pool_collect(pl, W, w0, ST_LEAF, ST_LEAF, lane), 32u);
            bool to_node = false, resolved = false;
            if ((uint32_t)lane < n) {
                const int slot = pl.list[lane];
                const float4 a = pl.fa[slot], b = pl.fb[slot];
                const uint2 tv = pl.tv[slot];
                const V3 o = v3(a), d = v3(b);
                BvhTrav t;
                t.cur = tv.x;
                t.sp = tv.y;
                t.h.t = a.w;
                unpack_hit(__float_as_uint(b.w), t.h);
                BvhStack bs;
                bs.base = pl.bstack;
                bs.stride = P;
                bs.idx = (uint32_t)slot;
                bs.k = min(p.bvh_stack_k, (uint32_t)POOL_BVH_K);
                bs.over = pl.bover + (size_t)slot * (BVH_STACK - POOL_BVH_K);
                bvh_leaf(t, sc.prims, bs, o, d, p.clip_min);
                pl.fa[slot].w = t.h.t;
                pl.fb[slot].w = __uint_as_float(pack_hit(t.h));
                pl.tv[slot] = make_uint2(t.cur, t.sp);
                if (t.cur == BVH_DONE) {
                    pl.st[slot] = ST_HIT_STRAIGHT;
                    resolved = true;
                } else if (!(t.cur & BVH_LEAF)) {
                    pl.st[slot] = ST_NODE;
                    to_node = true;
                }
            }
            const uint32_t n_tn = __popc(__ballot_sync(0xffffffffu, to_node)), n_rs = __popc(__ballot_sync(0xffffffffu, resolved));
            n_leaf -= n_tn + n_rs;
            n_node += n_tn;
            n_res += n_rs;
            if (PSTATS) {
                ++ps[4];
                ps[5] += n;
            }
            __syncwarp();
        } else if (c_scan == best) {
            if (PSTATS) pc_phase = 1;
            // ================================ SCAN ================================
            const uint32_t n = min(pool_collect(pl, W, w0, ST_PEND, ST_PEND_STRAIGHT, lane), 32u);
            bool to_fly = false, resolved = false;
            int slot = -1;
            if ((uint32_t)lane < n) {
                slot = pl.list[lane];
                const int s = pl.st[slot];
                const float4 a = pl.fa[slot], b = pl.fb[slot];
                const V3 x = v3(a), v = v3(b);
                if (!LENS || s == ST_PEND_STRAIGHT) {
                    const int vol_obj = VOL ? (int)((__float_as_uint(pl.qc[slot].w) >> 5) & 127u) - 1 : -1;
                    const bool in_volume = VOL && vol_obj >= 0;
                    const Hit h = scan_prims<C>(sc.prims, sc.boxes, (int)p.scene.n_prims, x, v, in_volume ? 0.0f : p.clip_min,
                                                in_volume ? p.volume_step : p.clip_max, vol_obj);
                    if (LENS) {
                        pl.fc[slot].w = h.t;
                        pl.fd[slot].w = __uint_as_float(pack_hit(h));
                    } else {
                        pl.fa[slot].w = h.t;
                        pl.fb[slot].w = __uint_as_float(pack_hit(h));
                    }
                    pl.st[slot] = ST_HIT_STRAIGHT;
                    resolved = true;
                } else if (LENS) {
                    const float4 c = pl.fc[slot], e = pl.fd[slot];
                    Flight f;
                    f.travelled = a.w;
                    f.free = b.w;
                    f.rest = c.x;
                    f.near = -1;
                    f.steps = __float_as_uint(c.z);
                    f.scans = 0;
                    f.xp = p3(e);
                    const int fs = geodesic_scan<EXACT, false, C>(p, sc, p3(x), p3(v), f, s - 2, p.clip_min, p.clip_max);
                    pl.fa[slot].w = f.travelled;
                    if (fs == FL_FLY) {
                        pl.fb[slot].w = f.free;
                        pl.fc[slot] = make_float4(f.rest, __int_as_float(f.near), __uint_as_float(f.steps), 0.0f);
                        pl.st[slot] = ST_FLY;
                        to_fly = true;
                    } else {
                        pl.fc[slot] = make_float4(0.0f, __int_as_float(-1), __uint_as_float(f.steps), f.h.t);
                        pl.fd[slot].w = __uint_as_float(pack_hit(f.h));
                        pl.st[slot] = (uint8_t)(fs + 2);
                        resolved = true;
                    }
                }
            }
            const unsigned m_fly = __ballot_sync(0xffffffffu, to_fly);
            if (LENS && to_fly) pl.stack[n_fly + __popc(m_fly & lt)] = (uint8_t)slot;
            n_fly += __popc(m_fly);
            n_res += __popc(__ballot_sync(0xffffffffu, resolved));
            n_pend -= n;
            if (PSTATS) {
                ++ps[4];
                ps[5] += n;
            }
            __syncwarp();
        } else if (c_shade == best) {
            if (PSTATS) pc_phase = 2;
            // ================================ SHADE ===============================
            const uint32_t n = min(pool_collect(pl, W, w0, ST_HIT, ST_HIT_STRAIGHT, lane), 32u);
            bool to_fly = false, to_pend = false, to_node = false, finished = false;
            int slot = -1;
            if ((uint32_t)lane < n) {
                slot = pl.list[lane];
                const int s = pl.st[slot];
                const float4 a = pl.fa[slot], b = pl.fb[slot];
                V3 o = v3(a), d = v3(b);
                Traced tr;
                if (!LENS || s == ST_HIT_STRAIGHT) {
                    const float ht = LENS ? pl.fc[slot].w : a.w;
                    const uint32_t hw = __float_as_uint(LENS ? pl.fd[slot].w : b.w);
                    tr.h.t = ht;
                    unpack_hit(hw, tr.h);
                    tr.o = o;
                    tr.d = d;
                    tr.t_total = ht;
                    tr.steps = 0;
                    tr.scans = 1;
                    tr.captured = false;
                } else if (LENS) {
                    const float4 c = pl.fc[slot], e = pl.fd[slot];
                    Flight f;
                    f.travelled = a.w;
                    f.steps = __float_as_uint(c.z);
                    f.scans = 0;
                    f.h.t = c.w;
                    unpack_hit(__float_as_uint(e.w), f.h);
                    f.xp = p3(e);
                    tr = flight_result<EXACT>(s - 2, p3(o), p3(d), f);
                }
                PathQ q;
                {
                    const uint4 r0 = pl.qa[slot], r1 = pl.qb[slot];
                    q.rng.s0 = ((uint64_t)r0.y << 32) | r0.x;
                    q.rng.s1 = ((uint64_t)r0.w << 32) | r0.z;
                    q.rng.s2 = ((uint64_t)r1.y << 32) | r1.x;
                    q.rng.s3 = ((uint64_t)r1.w << 32) | r1.z;
                }
                const float4 tc = pl.qc[slot];
                const uint32_t misc = __float_as_uint(tc.w);
                q.T = v3(tc);
                q.bounce = (misc >> 12) & 255u;
                q.vb = (misc >> 20) & 255u;
                q.vol_obj = VOL ? (int)((misc >> 5) & 127u) - 1 : -1;
                q.latched = AOV && ((misc >> 4) & 1u);
                q.aov_albedo = q.aov_normal = v3(0.0f, 0.0f, 0.0f);
                q.aov_depth = __int_as_float(0x7f800000);
                if (AOV) {
                    const float4 e0 = pl.qe[slot], e1 = pl.qf[slot];
                    q.aov_albedo = v3(e0);
                    q.aov_depth = e0.w;
                    q.aov_normal = v3(e1);
                }
                V3 contrib;
                if (shade_event<C>(p, sc, k, tr, q, o, d, contrib)) {
                    pl.qc[slot] = make_float4(contrib.x, contrib.y, contrib.z, tc.w);
                    pl.st[slot] = ST_DONE;
                    finished = true;
                } else {
                    pl.qa[slot] = make_uint4((uint32_t)q.rng.s0, (uint32_t)(q.rng.s0 >> 32), (uint32_t)q.rng.s1, (uint32_t)(q.rng.s1 >> 32));
                    pl.qb[slot] = make_uint4((uint32_t)q.rng.s2, (uint32_t)(q.rng.s2 >> 32), (uint32_t)q.rng.s3, (uint32_t)(q.rng.s3 >> 32));
                    pl.qc[slot] = make_float4(q.T.x, q.T.y, q.T.z,
                                              __uint_as_float(pack_misc(misc & 15u, AOV && q.latched, VOL ? q.vol_obj : -1, q.bounce, q.vb)));
                    if (AOV) {
                        pl.qe[slot] = make_float4(q.aov_albedo.x, q.aov_albedo.y, q.aov_albedo.z, q.aov_depth);
                        pl.qf[slot] = make_float4(q.aov_normal.x, q.aov_normal.y, q.aov_normal.z, 0.0f);
                    }
                    // the scattered ray: a new flight, or a straight segment (flat field / volume march)
                    pl.fa[slot] = make_float4(o.x, o.y, o.z, BVH ? p.clip_max : 0.0f);
                    pl.fb[slot] = make_float4(d.x, d.y, d.z, 0.0f);
                    if (BVH) {  // a new traversal: at the root, no hit (pack_hit of prim -1 = 0)
                        pl.tv[slot] = make_uint2(0u, 0u);
                        pl.st[slot] = ST_NODE;
                        to_node = true;
                    } else if (LENS && !(VOL && q.vol_obj >= 0)) {
                        pl.fc[slot] = make_float4(0.0f, __int_as_float(-1), __uint_as_float(0u), 0.0f);
                        pl.st[slot] = ST_FLY;
                        to_fly = true;
                    } else {
                        pl.st[slot] = ST_PEND_STRAIGHT;
                        to_pend = true;
                    }
                }
            }
            const unsigned m_fly = __ballot_sync(0xffffffffu, to_fly);
            if (LENS && to_fly) pl.stack[n_fly + __popc(m_fly & lt)] = (uint8_t)slot;
            n_fly += __popc(m_fly);
            n_pend += __popc(__ballot_sync(0xffffffffu, to_pend));
            if (BVH) n_node += __popc(__ballot_sync(0xffffffffu, to_node));
            const uint32_t fin = __popc(__ballot_sync(0xffffffffu, finished));
            n_done += fin;
            n_res -= n;
            if (fin) regen_futile = false;
            if (PSTATS) {
                ++ps[6];
                ps[7] += n;
            }
            __syncwarp();
        } else {
            // ================================ REGEN ===============================
            // 1. retire finished paths in issue order (Chunk::write_*: rgb += value); a completed pixel goes back to the frame
            uint32_t r_cnt = 0;
            while (tot_retired != tot_issued) {
                const uint32_t s = pl.ring[(tot_retired & (POOL_RING - 1)) * 32 + lane];
                if (pl.st[s] != ST_DONE) break;
                const float4 c = pl.qc[s];
                acc = v3(__fadd_rn(acc.x, c.x), __fadd_rn(acc.y, c.y), __fadd_rn(acc.z, c.z));
                pl.st[s] = ST_IDLE;
                ++tot_retired;
                ++r_cnt;
                if (++a_retired == p.paths_per_pixel) {  // Buffer::write_color: rgb += value, alpha untouched (buffer.rs:159-178)
                    float4* dst = p.fb + ((uint64_t)ay * p.width + ax);
                    float4 fbv = *dst;
                    fbv.x += acc.x;
                    fbv.y += acc.y;
                    fbv.z += acc.z;
                    *dst = fbv;
                    acc = v3(0.0f, 0.0f, 0.0f);
                    ax = bx;  // B (if open) becomes A
                    ay = by;
                    a_issued = b_issued;
                    a_retired = 0;
                    --n_pix;
                }
            }
            const uint32_t n_ret = __reduce_add_sync(0xffffffffu, r_cnt);
            n_done -= n_ret;
            n_free += n_ret;
            // 2. open the next pixel of this lane's stream -- pixel `lane` of the warp's tile number seq -- once every path of the
            //    newest open pixel is issued.  The warp draws tiles from the grid-wide counter as its lanes reach them; a lane may
            //    run at most POOL_TILES tiles ahead of the slowest one (the window the tile indices are kept in).
            {
                const uint32_t tiles_x = (p.width + 7) / 8, tiles_y = (p.row_end - p.row0 + 3) / 4;
                const unsigned long long n_tiles = (unsigned long long)tiles_x * tiles_y;
#pragma unroll 1
                for (;;) {
                    const uint32_t lo = __reduce_min_sync(0xffffffffu, exhausted ? 0xffffffffu : seq);
                    const bool room = n_pix == 0 || (n_pix == 1 && a_issued == p.paths_per_pixel);
                    const bool want = room && !exhausted && seq - lo < POOL_TILES;
                    const uint32_t upto = __reduce_max_sync(0xffffffffu, want ? seq + 1 : 0u);
                    if (upto == 0) break;  // nobody can take a pixel now
                    while (fetched < upto) {
                        if (lane == 0) pl.tiles[fetched % POOL_TILES] = atomicAdd(p.pool_counter, 1ULL);
                        ++fetched;
                    }
                    __syncwarp();
                    bool skipped = false;
                    if (want) {
                        const unsigned long long t = pl.tiles[seq % POOL_TILES];
                        ++seq;
                        if (t >= n_tiles) {
                            exhausted = true;
                        } else {
                            const uint32_t ty = (uint32_t)(t / tiles_x), tx = (uint32_t)(t - (unsigned long long)ty * tiles_x);
                            const uint32_t px = tx * 8 + (lane & 7), py = p.row0 + ty * 4 + (lane >> 3);
                            if (px < p.width && py < p.row_end) {
                                if (n_pix == 0) {
                                    ax = px;
                                    ay = py;
                                    a_issued = a_retired = 0;
                                } else {
                                    bx = px;
                                    by = py;
                                    b_issued = 0;
                                }
                                ++n_pix;
                                sub_i = sub_j = 0;  // path_base is a multiple of sub_count: a call starts at sub-pixel (0, 0)
                            } else {
                                skipped = true;  // a tile that hangs over the frame's edge: on to the next one
                            }
                        }
                    }
                    __syncwarp();
                    if (!__any_sync(0xffffffffu, skipped)) break;
                }
            }
            // 3. start new camera paths in idle slots: the next path of the newest open pixel
            const bool on_b = n_pix == 2;
            const uint32_t issued = on_b ? b_issued : a_issued, px = on_b ? bx : ax, py = on_b ? by : ay;
            const bool can_issue = n_pix != 0 && issued < p.paths_per_pixel && tot_issued - tot_retired < POOL_RING;
            const uint32_t rot = turn & 31u;
            const unsigned m_issue = __ballot_sync(0xffffffffu, can_issue);
            uint32_t take = 0;
            if (m_issue != 0 && n_free != 0) {
                const uint32_t n_idle = min(pool_collect(pl, W, w0, ST_IDLE, ST_IDLE, lane), 32u);
                take = min((uint32_t)__popc(m_issue), n_idle);
                // rank among the issuing lanes, counted from lane `rot` so that no lane is served last every time
                const unsigned m_rot = __funnelshift_r(m_issue, m_issue, rot);
                const uint32_t rank = __popc(m_rot & ((1u << ((lane - rot) & 31u)) - 1u));
                if (can_issue && rank < take) {
                    const int slot = pl.list[rank];
                    Rng rng;
                    rng.seed_from_u64(path_seed(p.seed, (uint64_t)py * p.width + px, p.path_base + issued));
                    V3 o, d;
                    camera_ray(p.cam, k, rng, px, py, sub_i, sub_j, o, d);
                    if (++sub_i == p.cam.sub_n) {  // the next path's sub-pixel, counted instead of divided out
                        sub_i = 0;
                        if (++sub_j == p.cam.sub_n) sub_j = 0;
                    }
                    pl.qa[slot] = make_uint4((uint32_t)rng.s0, (uint32_t)(rng.s0 >> 32), (uint32_t)rng.s1, (uint32_t)(rng.s1 >> 32));
                    pl.qb[slot] = make_uint4((uint32_t)rng.s2, (uint32_t)(rng.s2 >> 32), (uint32_t)rng.s3, (uint32_t)(rng.s3 >> 32));
                    const uint32_t ri = tot_issued & (POOL_RING - 1);
                    pl.qc[slot] = make_float4(1.0f, 1.0f, 1.0f, __uint_as_float(pack_misc(ri, false, -1, 0u, 0u)));
                    if (AOV) {
                        pl.qe[slot] = make_float4(0.0f, 0.0f, 0.0f, __int_as_float(0x7f800000));
                        pl.qf[slot] = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
                    }
                    pl.fa[slot] = make_float4(o.x, o.y, o.z, BVH ? p.clip_max : 0.0f);
                    pl.fb[slot] = make_float4(d.x, d.y, d.z, 0.0f);
                    if (LENS) {
                        pl.fc[slot] = make_float4(0.0f, __int_as_float(-1), __uint_as_float(0u), 0.0f);
                        pl.stack[n_fly + rank] = (uint8_t)slot;
                    }
                    if (BVH) pl.tv[slot] = make_uint2(0u, 0u);
                    pl.st[slot] = LENS ? ST_FLY : (BVH ? ST_NODE : ST_PEND_STRAIGHT);
                    pl.ring[ri * 32 + lane] = (uint8_t)slot;
                    ++tot_issued;
                    if (on_b) ++b_issued; else ++a_issued;
                }
                if (LENS) n_fly += take; else if (BVH) n_node += take; else n_pend += take;
                n_free -= take;
            }
            if (PSTATS) {
                ++ps[8];
                ps[9] += take;
                ps[10] += n_ret;
            }
            regen_futile = n_ret == 0 && take == 0;  // nothing to do here until a path finishes (SHADE clears it)
            __syncwarp();
        }
        if (PSTATS) pc[pc_phase] += clock64() - pc_in;
    }
    if (PSTATS) {
        ps[11] = turn;
        pc[4] = clock64() - pc_t0;
        if (lane == 0) {
            for (int i = 0; i < 12; ++i) atomicAdd(p.stats + i, (unsigned long long)ps[i]);
            for (int i = 0; i < 5; ++i) atomicAdd(p.stats + 12 + i, (unsigned long long)pc[i]);
            for (int i = 0; i < 4; ++i) atomicAdd(p.stats + 17 + i, (unsigned long long)ps[12 + i]);
        }
    }
}
