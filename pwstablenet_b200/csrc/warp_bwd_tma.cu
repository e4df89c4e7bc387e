// warp_bwd_tma.cu -- TMA-pipelined persistent backward warp (sm_100a).
//
// Autograd of R/main_new.py:106,116 (grad -> map) and :197 (grad -> frame), triggered at :214.
//
// One persistent CTA per SM walks 64x16 tiles of OUTPUT pixels, handed out dynamically.  Its 20 warps:
//   2 scouts     one per consumer group, alternate tiles: TMA-load the map of the next tile, reduce this tile's map
//                to the bounding box of its source taps, TMA-load its grad_output and that box of the frame (only when
//                grad_grid is wanted, it is its one use), and hold the tile back until the bands of grad_input its taps
//                can reach are zero-filled by every CTA;
//   16 consumers two groups of 8 warps, each group owning every other tile; inside a tile a warp owns a 32-pixel-wide
//                strip of 4 rows and marches down it;
//   2 zero-fill  zero-fill grad_input band by band, kZeroAhead bands ahead of the scouts.
// The scatter into grad_input is the marching scheme of warp_bwd_lean.cu: a lane whose right neighbour
// samples the next source pixel hands its east taps over by shuffle, the south taps ride down the strip
// in registers, and what is left is ~1 RED.ADD.F32 per source pixel and channel on consecutive addresses.
// The stragglers (east taps nobody takes over, parked sums whose chain broke) are compacted through a
// per-warp queue in shared memory and leave as dense 32-lane REDs (the L2 accepts ~25 G RED
// instructions/s whether 1 or 32 lanes are active: tools/exp/exp_red.cu).
// grad_grid is accumulated in ATen's exact statement order from taps read out of the shared-memory box:
// bit-identical to the other backward kernels; grad_input differs only by atomic order.
#include "pws_pipe.cuh"
#include "pws_launch.cuh"
#include "pws_f32x2.cuh"

#include <atomic>
#include <cstdio>
#include <cstdlib>

namespace pws {

using namespace pipe;

namespace {

// Tunables (measured on a B200; DESIGN 3.3 has the record of the alternatives).
constexpr int kGroups = 2, kGroupWarps = 8;     // consumer groups of 8 warps
constexpr int kScouts = kGroups;                // scout w feeds consumer group w (and tells it when the tiles have run out)
constexpr int kConsumers = kGroups * kGroupWarps;
// The zero-fill of grad_input paces the whole kernel when ONE warp does it: a band costs that warp its stores plus a
// gpu-scope fence (~2 us while the REDs keep the memory system busy), 128 bands of a 16-frame launch = the kernel's 0.46 ms
// (ncu: the zero-fill warp never sleeps, half of its samples sit on the fence).  kZeroWarps warps take the bands round-robin.
constexpr int kZeroWarps = 2;
// how far the zero-fill runs ahead of the scatter, in bands: the best look-ahead is 3-4 bands (0.593 / 0.482 / 0.469 /
// 0.468 ms at 1 / 2 / 3 / 4)
constexpr int kZeroAhead = 4;
// pause of a zero-fill warp between two looks at the scouts' progress (a band lasts ~5 us; at 256 ns the polls were 7 % of
// the kernel's instructions)
constexpr int kZeroPollNs = 1000;
// grad_input bytes per band (see below)
constexpr int64_t kBandBytes = (int64_t)4 << 20;
// main-ring depth of the fp32 kernel with frame boxes (without boxes, or with 16-bit boxes, the ring is 6 deep: Smem)
constexpr int kBoxStages = 4;

constexpr int kThreads = (kScouts + kConsumers + kZeroWarps) * 32;  // scouts, consumers, the warps that zero-fill grad_input
constexpr int kZeroWarp = kScouts + kConsumers;                      // first of them
constexpr int kInfoStop = 1 << 11;  // info.z: no more tiles for this consumer group

// grad_input is zero-filled INSIDE the kernel, kZeroAhead bands ahead of the scatter: the zeroed lines are still in L2
// when the REDs land and no separate memset pass runs ahead of the kernel.  Band b of a frame split into B bands is rows
// [ceil(b*H/B), ceil((b+1)*H/B)) of every channel plane; a tile only waits for the bands its taps can reach.  Every band
// costs its CTA's zero-fill warp a fence, an atomic and a poll (~1 us): a launch of many SMALL frames must not pay many of
// them per frame, so B follows the frame size (about kBandBytes of grad_input per band, 1..kMaxBands).
// A launch owns one slot of per-band completion counters; the last CTA to leave resets the slot.
constexpr int kSyncSlots = kLaunchSlots, kSyncFrames = 256;
constexpr int kMaxBands = 32;   // (a 4K fp32 grad_input frame is 25 bands of 4 MB)
__device__ unsigned int g_zero_done[kSyncSlots][kSyncFrames * kMaxBands];
__device__ unsigned int g_exit_count[kSyncSlots];
// Tiles are handed out dynamically: the SMs of a B200 do not run this kernel at the same pace (the spread is several
// per cent: distance to the L2 slices, neighbours on the same TPC), and with a static round-robin every frame ended
// with the fast CTAs waiting at the zero-fill counter of the next frame for the slow ones.
__device__ unsigned int g_tile_next[kSyncSlots];
// (slots are leased per device and reused only after their previous launch has finished: pws_launch.cuh)

// the scouts' progress words: a flag polled by the zero-fill warp, not data
#ifdef PWS_BWD_ATOMIC_PROGRESS   // shared-memory atomics: silences compute-sanitizer's racecheck (used for the sanitizer runs)
__device__ __forceinline__ void progress_store(int *p, int v) { atomicExch(p, v); }
__device__ __forceinline__ int progress_load(int *p) { return atomicOr(p, 0); }
#else
__device__ __forceinline__ void progress_store(int *p, int v) { *reinterpret_cast<volatile int *>(p) = v; }
__device__ __forceinline__ int progress_load(int *p) { return *reinterpret_cast<volatile int *>(p); }
#endif
__device__ __forceinline__ unsigned int ld_acquire(const unsigned int *p)
{
    unsigned int v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
constexpr int kStripRows = 2 * kTH / kGroupWarps;  // a warp owns a 32-column strip of this many rows
constexpr int kQueueCap = 64;  // entries per consumer warp: 31 left over + one class of stragglers from 32 lanes

// Two rings.  A stage of the main ring holds a tile's grad_output, its frame box (room for the largest box shape) and its
// info words behind one `full` and one `empty` mbarrier.  The map tiles live in a ring of their own that is two slots
// deeper: a scout loads the map of its NEXT tile while it dispatches the current one, so that the bounding box of a tile
// is known before the tile's stage frees up and the grad_output and box loads leave the moment it does.
// kElem: bytes per frame / grad_output element (4, or 2 for f16 / bf16 frames: the smaller stages buy a deeper ring)
template <int CS, bool kGgrid, int kElem = 4> struct Smem {
    static constexpr int kStages = kGgrid ? (kElem == 2 ? 6 : kBoxStages) : 6;
    static constexpr int kMapStages = kStages + kScouts;
    static constexpr int kGoutBytes = CS * kTW * kTH * kElem;
    static constexpr int kBoxBytes = kGgrid ? (box_w(kNumShapes - 1) * box_h(kNumShapes - 1) * CS * kElem + 127) / 128 * 128 : 0;
    static constexpr int kMapOff = 0;
    static constexpr int kGoutOff = kMapStages * kMapTileBytes;
    static constexpr int kBoxOff = kGoutOff + kStages * kGoutBytes;
    static constexpr int kQueueOff = kBoxOff + kStages * kBoxBytes;
    static constexpr int kQueueEntry = CS == 3 ? 16 : 8;
    static constexpr int kInfoOff = kQueueOff + kConsumers * kQueueCap * kQueueEntry;
    static constexpr int kBarOff = kInfoOff + kStages * 48;   // per stage: info, where, two base pointers
    static constexpr int kProgressOff = kBarOff + 2 * (kStages + kMapStages) * 8;
    static constexpr int kTotal = kProgressOff + 16;
    static_assert(kGoutBytes % 128 == 0 && kBoxBytes % 128 == 0, "TMA destinations must stay 128-byte aligned");
    static_assert(kTotal <= 227 * 1024, "shared memory budget");
};

struct TmaParams {
    CUtensorMap map;              // as in warp_fwd_tma.cu
    CUtensorMap gout;             // (Wo, Ho, C, N), box (64,16,CS,1)
    CUtensorMap box[kNumShapes];  // frame (W, H, C, N), box (BW, BH, CS, 1)
};

template <int CS>
struct Carry {
    int x, y;  // target of the parked south-west sums
    bool live;
    float v[CS];
};

// Straggler queue of a consumer warp: one entry = a source pixel offset plus its CS channel values.
template <int CS> struct QEntry;
template <> struct QEntry<1> { int off; float v[1]; };
template <> struct QEntry<3> { int off; float v[3]; };
template <int CS>
struct Queue {
    QEntry<CS> *buf;  // shared memory, kQueueCap entries
    int count;        // warp-uniform
};

template <int CS>
__device__ __forceinline__ void queue_put(Queue<CS> &q, int pos, int off, const float (&v)[CS])
{
    if (CS == 3) *reinterpret_cast<int4 *>(q.buf + pos) = make_int4(off, __float_as_int(v[0]), __float_as_int(v[CS > 1 ? 1 : 0]), __float_as_int(v[CS > 2 ? 2 : 0]));
    else *reinterpret_cast<int2 *>(q.buf + pos) = make_int2(off, __float_as_int(v[0]));
}
// element `off` of a plane: one IMAD.WIDE (the compiler otherwise widens the offset once and adds it to every plane base
// with carry chains)
__device__ __forceinline__ float *at(float *base, int off)
{
    float *p;
    asm("mad.wide.s32 %0, %1, 4, %2;" : "=l"(p) : "r"(off), "l"(base));
    return p;
}

// gp[k]: this frame's grad_input plane of channel k (one 64-bit base per plane; an entry's offset is 32-bit).
// grad_input's adds are tma::red_add_f32, an explicit fire-and-forget reduction: with a fence elsewhere in the kernel nvcc
// turns atomicAdd into the returning ATOMG form, whose round trip to L2 the scatter would then wait for.
template <int CS>
__device__ __forceinline__ void queue_pop_red(const Queue<CS> &q, int pos, float *const (&gp)[CS])
{
    if (CS == 3) {
        const int4 e = *reinterpret_cast<const int4 *>(q.buf + pos);
        tma::red_add_f32(at(gp[0], e.x), __int_as_float(e.y));
        tma::red_add_f32(at(gp[CS > 1 ? 1 : 0], e.x), __int_as_float(e.z));
        tma::red_add_f32(at(gp[CS > 2 ? 2 : 0], e.x), __int_as_float(e.w));
    } else {
        const int2 e = *reinterpret_cast<const int2 *>(q.buf + pos);
        tma::red_add_f32(at(gp[0], e.x), __int_as_float(e.y));
    }
}
// one dense 32-lane RED per channel once a warp's worth of entries is queued (a push adds at most 32 entries to fewer
// than 32, so one round always brings the count back below 32)
template <int CS>
__device__ __forceinline__ void queue_drain(Queue<CS> &q, float *const (&gp)[CS], int lane)
{
    __syncwarp();
    if (q.count >= 32) {
        queue_pop_red<CS>(q, q.count - 32 + lane, gp);
        q.count -= 32;
    }
    __syncwarp();
}
template <int CS>
__device__ __forceinline__ void queue_flush(Queue<CS> &q, float *const (&gp)[CS], int lane)
{
    queue_drain<CS>(q, gp, lane);
    if (lane < q.count) queue_pop_red<CS>(q, lane, gp);
    q.count = 0;
    __syncwarp();
}

// One output row (32 pixels) of a warp in a tile that is NOT interior (frame border, partial tile, no box): every tap and
// every lane is checked.  kBoxTaps: the taps of grad_grid come from the shared-memory box
// (tap = box[(y - by) * pitch + (x - bx)] per plane), else from global memory.
template <typename T, int CS, bool kGin, bool kGgrid, bool kBoxTaps>
__device__ __forceinline__ void masked_row(
    const int lane, const bool px_ok, const unsigned live,
    const float ix, const float iy, const float x0f, const float y0f, const int x0, const int y0,
    const float gxm, const float gym, const float (&go)[CS],
    const T *__restrict__ box, const int pitch, const int plane,
    const T *__restrict__ ip, const int sH, const int i_ch, const int H, const int W,
    float *const (&gp)[CS], float *__restrict__ ggq, const int gg_s3, Carry<CS> &cy, Queue<CS> &q, const uint64_t pol_first)
{
    const float dw = fsub(x0f + 1.0f, ix), de = fsub(ix, x0f), dn = fsub(y0f + 1.0f, iy), ds = fsub(iy, y0f);
    const bool xw = (unsigned)x0 < (unsigned)W, xe = (unsigned)(x0 + 1) < (unsigned)W;
    const bool yn = (unsigned)y0 < (unsigned)H, ys = (unsigned)(y0 + 1) < (unsigned)H;
    unsigned mask = ((xw && yn) ? 1u : 0u) | ((xe && yn) ? 2u : 0u) | ((xw && ys) ? 4u : 0u) | ((xe && ys) ? 8u : 0u);
    if (!px_ok) mask = 0u;

    if (kGgrid && px_ok) {
        float gix = 0.f, giy = 0.f;
        const T *__restrict__ p0 = kBoxTaps ? box + (y0 * pitch + x0) : ip + (y0 * sH + x0);
        const int row = kBoxTaps ? pitch : sH, ch = kBoxTaps ? plane : i_ch;
#pragma unroll
        for (int k = 0; k < CS; ++k) {
            const T *__restrict__ pc = p0 + k * ch;
            float v0 = 0.f, v1 = 0.f, v2 = 0.f, v3 = 0.f;
            if (kBoxTaps) {
                if (mask & 1u) v0 = to_acc(pc[0]);
                if (mask & 2u) v1 = to_acc(pc[1]);
                if (mask & 4u) v2 = to_acc(pc[row]);
                if (mask & 8u) v3 = to_acc(pc[row + 1]);
            } else {
                if (mask & 1u) v0 = to_acc(__ldg(pc));
                if (mask & 2u) v1 = to_acc(__ldg(pc + 1));
                if (mask & 4u) v2 = to_acc(__ldg(pc + row));
                if (mask & 8u) v3 = to_acc(__ldg(pc + row + 1));
            }
            // ATen's statement order: t = v*d rounded, then one fma with gOut
            if (mask & 1u) { gix = ffma(-fmul(v0, dn), go[k], gix); giy = ffma(-fmul(v0, dw), go[k], giy); }
            if (mask & 2u) { gix = ffma(fmul(v1, dn), go[k], gix);  giy = ffma(-fmul(v1, de), go[k], giy); }
            if (mask & 4u) { gix = ffma(-fmul(v2, ds), go[k], gix); giy = ffma(fmul(v2, dw), go[k], giy); }
            if (mask & 8u) { gix = ffma(fmul(v3, ds), go[k], gix);  giy = ffma(fmul(v3, de), go[k], giy); }
        }
        gix = fmul(gxm, gix); giy = fmul(gym, giy);
        tma::st_f32_hint(ggq, gix, pol_first); tma::st_f32_hint(ggq + gg_s3, giy, pol_first);
    }

    if (kGin) {
        const float nw = fmul(dw, dn), ne = fmul(de, dn), sw = fmul(dw, ds), se = fmul(de, ds);
        const int o_nw = y0 * W + x0;  // grad_input is dense NCHW
        const int px0 = __shfl_up_sync(0xffffffffu, x0, 1), py0 = __shfl_up_sync(0xffffffffu, y0, 1);
        const int nx0 = __shfl_down_sync(0xffffffffu, x0, 1), ny0 = __shfl_down_sync(0xffffffffu, y0, 1);
        const bool take = lane > 0 && px0 + 1 == x0 && py0 == y0 && px_ok && ((live >> (lane - 1)) & 1u);
        const bool given = lane < 31 && nx0 == x0 + 1 && ny0 == y0 && px_ok && ((live >> (lane + 1)) & 1u);
        const bool chain = cy.live && cy.x == x0 && cy.y == y0;
        const int o_cy = cy.y * W + cy.x;
        // stragglers of this row -> queue: east taps nobody takes over (top and bottom), parked sums whose chain broke
        const bool p_e1 = !given && (mask & 2u), p_e2 = !given && (mask & 8u), p_f = cy.live && !chain;
        const unsigned lt = (1u << lane) - 1u;
        float etop[CS], ebot[CS], brk[CS];
#pragma unroll
        for (int k = 0; k < CS; ++k) {
            float top = fmul(nw, go[k]), bot = fmul(sw, go[k]);
            etop[k] = fmul(ne, go[k]); ebot[k] = fmul(se, go[k]);
            const float ptop = __shfl_up_sync(0xffffffffu, etop[k], 1), pbot = __shfl_up_sync(0xffffffffu, ebot[k], 1);
            if (take) { top += ptop; bot += pbot; }
            brk[k] = cy.v[k];
            if (chain) top += cy.v[k];
            if (mask & 1u) tma::red_add_f32(at(gp[k], o_nw), top);
            cy.v[k] = bot;
        }
        const unsigned b1 = __ballot_sync(0xffffffffu, p_e1), b2 = __ballot_sync(0xffffffffu, p_e2), b3 = __ballot_sync(0xffffffffu, p_f);
        if (b1) {
            if (p_e1) queue_put<CS>(q, q.count + __popc(b1 & lt), o_nw + 1, etop);
            q.count += __popc(b1);
            if (q.count >= 32) queue_drain<CS>(q, gp, lane);
        }
        if (b2) {
            if (p_e2) queue_put<CS>(q, q.count + __popc(b2 & lt), o_nw + W + 1, ebot);
            q.count += __popc(b2);
            if (q.count >= 32) queue_drain<CS>(q, gp, lane);
        }
        if (b3) {
            if (p_f) queue_put<CS>(q, q.count + __popc(b3 & lt), o_cy, brk);
            q.count += __popc(b3);
            if (q.count >= 32) queue_drain<CS>(q, gp, lane);
        }
        cy.x = x0; cy.y = y0 + 1;
        cy.live = (mask & 4u) != 0u;
    }
}

// A strip of a tile that is not "interior": the masked rows, then the parked south-west sums.
template <typename T, int CS, bool kBorder, bool kAlign, bool kInter, bool kGin, bool kGgrid>
__device__ __forceinline__ void masked_strip(
    const int lane, const int4 info, const int h0, const int w0, const int row0, const int col0,
    const float *__restrict__ mp, const T *__restrict__ gop, const T *__restrict__ bp, const int pitch, const int plane,
    const T *__restrict__ ip, const int sH, const int i_ch, const Geometry g,
    float *const (&gp)[CS], float *__restrict__ ggq, const int gg_s1, const int gg_s3, Queue<CS> &q, const uint64_t pol_first)
{
    const float Wf = (float)g.W, Hf = (float)g.H, Wm1 = (float)(g.W - 1), Hm1 = (float)(g.H - 1);
    const bool col_ok = w0 + lane < g.Wo;
    const unsigned live = __ballot_sync(0xffffffffu, col_ok);
    const bool box_taps = kGgrid && !(info.z & (kInfoFallback | kInfoEmpty));
    const int rows = min(kStripRows, g.Ho - h0);  // may be <= 0 for the strips below the last row
    Carry<CS> cy;
    cy.x = 0; cy.y = 0; cy.live = false;
#pragma unroll
    for (int k = 0; k < CS; ++k) cy.v[k] = 0.f;
    for (int r = 0; r < rows; ++r) {
        float gx, gy, go[CS];
        if (kInter) { const float2 v = *reinterpret_cast<const float2 *>(mp + (row0 + r) * (2 * kTW) + 2 * (col0 + lane)); gx = v.x; gy = v.y; }
        else { gx = mp[(row0 + r) * kTW + col0 + lane]; gy = mp[kTW * kTH + (row0 + r) * kTW + col0 + lane]; }
#pragma unroll
        for (int k = 0; k < CS; ++k) go[k] = to_acc(gop[k * (kTW * kTH) + r * kTW]);
        float gxm, gym;
        const float ix = src_index_grad<kBorder, kAlign>(gx, Wf, Wm1, &gxm);
        const float iy = src_index_grad<kBorder, kAlign>(gy, Hf, Hm1, &gym);
        const float x0f = floorf(ix), y0f = floorf(iy);
        const int x0 = (int)x0f, y0 = (int)y0f;
        if (box_taps)
            masked_row<T, CS, kGin, kGgrid, true>(lane, col_ok, live, ix, iy, x0f, y0f, x0, y0, gxm, gym, go,
                                               bp, pitch, plane, ip, sH, i_ch, g.H, g.W, gp, ggq, gg_s3, cy, q, pol_first);
        else
            masked_row<T, CS, kGin, kGgrid, false>(lane, col_ok, live, ix, iy, x0f, y0f, x0, y0, gxm, gym, go,
                                                bp, pitch, plane, ip, sH, i_ch, g.H, g.W, gp, ggq, gg_s3, cy, q, pol_first);
        if (kGgrid) ggq += gg_s1;
    }
    if (kGin && cy.live) {
        const int o_cy = cy.y * g.W + cy.x;
#pragma unroll
        for (int k = 0; k < CS; ++k) tma::red_add_f32(at(gp[k], o_cy), cy.v[k]);
    }
}

// insert one class of stragglers (predicate p, entry (off, v)) into the warp's queue; all 32 lanes call this
template <int CS>
__device__ __forceinline__ void queue_push(Queue<CS> &q, const bool p, const int off, const float (&v)[CS], const unsigned lt,
                                           float *const (&gp)[CS], const int lane)
{
    const unsigned b = __ballot_sync(0xffffffffu, p);
    if (b) {
        if (p) queue_put<CS>(q, q.count + __popc(b & lt), off, v);
        q.count += __popc(b);
        if (q.count >= 32) queue_drain<CS>(q, gp, lane);
    }
}

// A strip (32 pixels x kStripRows rows) of an INTERIOR tile: the tile is full and every tap of every pixel lies inside
// the frame, so there are no masks, the floor is one round-down add, and a source pixel is identified by its linear
// offset alone.  grad_grid and the scatter of a row run in one body: one pass over the map and grad_output in shared memory.
// Coordinates run on fp32 PAIRS (pws_f32x2.cuh); grad_grid accumulates (giy, gix) as one pair: per tap and channel one
// FMUL2 (tap value x the pair of fraction weights, ATen's sign folded into the weights: -(v*d) == v*(-d) exactly) and one
// FFMA2 with grad_output -- ATen's statements, operation for operation, so the result is bit-identical.
// dw = 1 - de instead of (x0 + 1) - ix: de = ix - x0 is exact, so both are the rounding of the same real number.
// Two refinements of the scatter trade ~16 issue slots per row for a quarter fewer queue entries (0.383 -> 0.367 ms / 16
// 1080p frames with grad_input only, 0.426 -> 0.409 with grad_grid too):
//   east carry    an east-bottom tap nobody takes over is parked like the south-west sum and merges into the lane's own
//                 east tap of the next row (one queue entry per broken horizontal chain instead of two);
//   vertical dup  a row that samples the SAME source row as the one above adds the parked sum to its own bottom sum
//                 instead of flushing it.
template <typename T, int CS, bool kAlign, bool kInter, bool kGin, bool kGgrid>
__device__ __forceinline__ void interior_strip(
    const int lane, const float *__restrict__ mq /* this lane's map element(s) in the strip's first row */,
    const T *__restrict__ gop, const T *__restrict__ bp, const int pitch, const int plane,
    const float2 size2 /* (W, H) as floats; (W-1, H-1) when kAlign */, const int W, const float2 gmul2 /* (gym, gxm) */,
    float *const (&gp)[CS], float *__restrict__ ggq, const int gg_s1, const int gg_s3, Queue<CS> &q, const uint64_t pol_first)
{
    // the two grad_grid stores of a pixel: running byte pointers, one 64-bit add each per row
    char *gq_x = reinterpret_cast<char *>(ggq), *gq_y = reinterpret_cast<char *>(ggq + gg_s3);
    const int64_t gq_step = (int64_t)gg_s1 * 4;
    const unsigned lt = (1u << lane) - 1u;
    int co = -1, eo = -1;        // linear offsets of the parked south-west / south-east sums' targets; -1: nothing parked
    float cv[CS], ev[CS];
#pragma unroll
    for (int k = 0; k < CS; ++k) { cv[k] = 0.f; ev[k] = 0.f; }

#pragma unroll
    for (int r = 0; r < kStripRows; ++r) {
        float2 gxy;
        if (kInter) gxy = *reinterpret_cast<const float2 *>(mq + r * (2 * kTW));
        else { gxy.x = mq[r * kTW]; gxy.y = mq[kTW * kTH + r * kTW]; }
        float go[CS];
#pragma unroll
        for (int k = 0; k < CS; ++k) go[k] = to_acc(gop[k * (kTW * kTH) + r * kTW]);
        // unnormalise (ATen's operation order), floor, fractions
        const float2 t = x2::add(gxy, x2::bc(1.0f));
        const float2 ixy = kAlign ? x2::mul(x2::mul(t, x2::bc(0.5f)), size2) : x2::mul(x2::fma(t, size2, x2::bc(-1.0f)), x2::bc(0.5f));
        const float2 fl = x2::add_rm(ixy, x2::bc(12582912.0f));              // 1.5 * 2^23: the integer part lands in the mantissa
        const int x0 = __float_as_int(fl.x) - 0x4B400000, y0 = __float_as_int(fl.y) - 0x4B400000;
        const float2 es = x2::sub(ixy, x2::add(fl, x2::bc(-12582912.0f)));   // (de, ds) = (ix - x0, iy - y0)
        const float2 wn = x2::sub(x2::bc(1.0f), es);                         // (dw, dn)
        const float de = es.x, ds = es.y, dw = wn.x, dn = wn.y;

        if (kGgrid) {
            const T *__restrict__ p0 = bp + (y0 * pitch + x0);
            // per tap the weights of (giy, gix) with ATen's signs: nw (-dw, -dn), ne (-de, +dn), sw (+dw, -ds), se (+de, +ds)
            const float2 c_nw = make_float2(-dw, -dn), c_ne = make_float2(-de, dn), c_sw = make_float2(dw, -ds), c_se = es;
            float2 acc = make_float2(0.f, 0.f);
#pragma unroll
            for (int k = 0; k < CS; ++k) {
                const float v0 = to_acc(p0[k * plane]), v1 = to_acc(p0[k * plane + 1]), v2 = to_acc(p0[k * plane + pitch]), v3 = to_acc(p0[k * plane + pitch + 1]);
                const float2 g2 = x2::bc(go[k]);
                acc = x2::fma(x2::mul(x2::bc(v0), c_nw), g2, acc);
                acc = x2::fma(x2::mul(x2::bc(v1), c_ne), g2, acc);
                acc = x2::fma(x2::mul(x2::bc(v2), c_sw), g2, acc);
                acc = x2::fma(x2::mul(x2::bc(v3), c_se), g2, acc);
            }
            acc = x2::mul(gmul2, acc);
            tma::st_f32_hint(reinterpret_cast<float *>(gq_x), acc.y, pol_first); tma::st_f32_hint(reinterpret_cast<float *>(gq_y), acc.x, pol_first);
            // (volatile: the unrolled rows otherwise recompute base + r * step with twice the 64-bit adds)
            asm volatile("add.s64 %0, %0, %1;" : "+l"(gq_x) : "l"(gq_step));
            asm volatile("add.s64 %0, %0, %1;" : "+l"(gq_y) : "l"(gq_step));
        }

        if (kGin) {
            const int o = y0 * W + x0;                      // north-west tap; the others are o + 1, o + W, o + W + 1
            const int o_left = __shfl_up_sync(0xffffffffu, o, 1);
            // lane l hands its east taps to lane l + 1 when that lane's north-west tap is this lane's north-east one
            // (x0 <= W - 2 in an interior tile: "offset + 1" never wraps into the next row)
            const bool take = lane > 0 && o_left + 1 == o;
            const bool given = ((__ballot_sync(0xffffffffu, take) >> 1) >> lane) & 1u;
            // (r > 0: nothing is parked in the strip's first row; the loop is unrolled, the test is free)
            const bool chain = r > 0 && co == o;                    // the parked south-west sum lands on this row's north-west tap
            const bool vdup = r > 0 && co == o + W;                 // ... on its south-west tap: same source row again
            const bool broke = r > 0 && !chain && !vdup;
            const bool e_chain = r > 0 && eo == o + 1, e_vdup = r > 0 && eo == o + W + 1;
            const bool e_broke = r > 0 && eo >= 0 && !e_chain && !e_vdup;
            // (scalar: pairs would need as many register moves here as they save multiplies)
            const float nw = fmul(dw, dn), ne = fmul(de, dn), sw = fmul(dw, ds), se = fmul(de, ds);
            float et[CS], eb[CS], old_c[CS], old_e[CS];
#pragma unroll
            for (int k = 0; k < CS; ++k) {
                float top = fmul(nw, go[k]), bot = fmul(sw, go[k]);   // west column
                et[k] = fmul(ne, go[k]); eb[k] = fmul(se, go[k]);     // east column
                old_e[k] = ev[k];
                if (e_chain) et[k] += ev[k];                // parked south-east sum: this row's north-east tap
                if (e_vdup) eb[k] += ev[k];
                const float pt = __shfl_up_sync(0xffffffffu, et[k], 1), pb = __shfl_up_sync(0xffffffffu, eb[k], 1);
                if (take) { top += pt; bot += pb; }
                old_c[k] = cv[k];
                if (chain) top += cv[k];
                if (vdup) bot += cv[k];
                tma::red_add_f32(at(gp[k], o), top);
                cv[k] = bot;
                ev[k] = eb[k];
            }
            // stragglers -> queue: the north-east tap nobody took, parked sums whose chain broke
            queue_push<CS>(q, !given, o + 1, et, lt, gp, lane);
            queue_push<CS>(q, broke, co, old_c, lt, gp, lane);
            queue_push<CS>(q, e_broke, eo, old_e, lt, gp, lane);
            co = o + W;
            eo = !given ? o + W + 1 : -1;
        }
    }
    if (kGin) {
#pragma unroll
        for (int k = 0; k < CS; ++k) tma::red_add_f32(at(gp[k], co), cv[k]);   // every lane parked a south-west sum in the last row
        queue_push<CS>(q, eo >= 0, eo, ev, lt, gp, lane);
    }
}

template <typename T, int CS, bool kBorder, bool kAlign, bool kInter, bool kGin, bool kGgrid>
__global__ void __launch_bounds__(kThreads, 1)
bwd_tma_kernel(const __grid_constant__ TmaParams tp, const View in, const View grid, const View gin, const View ggrid, const Geometry g,
               const int tiles_x, const int tiles_y, const int total_tiles, const int n_begin, const int n_frames, const int slot, const int kBands)
{
    using S = Smem<CS, kGgrid, (int)sizeof(T)>;
    constexpr int kStages = S::kStages, kMapStages = S::kMapStages;
    extern __shared__ __align__(1024) unsigned char smem[];
    float *const s_map = reinterpret_cast<float *>(smem + S::kMapOff);
    unsigned char *const s_gout = smem + S::kGoutOff;
    unsigned char *const s_box = smem + S::kBoxOff;
    QEntry<CS> *const s_queue = reinterpret_cast<QEntry<CS> *>(smem + S::kQueueOff);
    int4 *const s_info = reinterpret_cast<int4 *>(smem + S::kInfoOff);
    uint64_t *const full = reinterpret_cast<uint64_t *>(smem + S::kBarOff);
    uint64_t *const empty = full + kStages;
    uint64_t *const map_full = empty + kStages;
    uint64_t *const map_empty = map_full + kMapStages;
    // [0], [1]: how far scout 0 / 1 has dispatched, in bands (kBands * frame + band).  Written by the scouts and polled by
    // the zero-fill warps (volatile; compute-sanitizer's racecheck flags exactly this pair and nothing else -- build with
    // -DPWS_BWD_ATOMIC_PROGRESS to run it clean).  The other two words of the 16 bytes are unused.
    int *const s_progress = reinterpret_cast<int *>(smem + S::kProgressOff);

    // Roles are numbered from the TOP warp of the CTA down (the scheduler favours the higher warp ids when several
    // warps are ready; the scouts are a handful of instructions per tile, but every consumer waits on them).
    const int warp = (kThreads / 32 - 1) - (threadIdx.x >> 5), lane = threadIdx.x & 31;
    const int tiles_xy = tiles_x * tiles_y;
    const float Wf = (float)g.W, Hf = (float)g.H, Wm1 = (float)(g.W - 1), Hm1 = (float)(g.H - 1);
    // L2 priorities: everything that streams through once (map, grad_output, frame boxes, grad_grid) is evict_first,
    // so the replacement order favours grad_input, which is revisited between its zero-fill and its last RED.
    // (evict_last for grad_input was tried: its lines then outlive the kernel and crowd the next one out of L2.)
    const uint64_t pol_first = tma::policy_evict_first();
    const uint64_t pol_box = pol_first, pol_gg = pol_first, pol_zero = tma::policy_evict_normal();

    if (threadIdx.x == 0) {
        s_progress[0] = 0; s_progress[1] = 0;
        // full: the scout arrives twice -- once with the byte count of the TMA loads, once when the tile's frame is known
        // to be zero-filled by every CTA; empty: one arrival per consumer warp of the group
        for (int s = 0; s < kStages; ++s) { tma::mbar_init(full + s, 2); tma::mbar_init(empty + s, kGroupWarps); }
        for (int s = 0; s < kMapStages; ++s) { tma::mbar_init(map_full + s, 1); tma::mbar_init(map_empty + s, kGroupWarps); }
        tma::fence_barrier_init();
    }
    __syncthreads();

    if (warp < kScouts) {
        // ===== scouts: scout w serves the iterations it = w, w + 2, ... = consumer group w =====
        // Per tile: fetch the tile index, start the map load of the NEXT tile, reduce this tile's map (already in the map
        // ring) to the bounding box of its taps, wait for the ring stage, issue the grad_output and frame box loads on the
        // stage's barrier, and make sure the tile's frame has been zero-filled by every CTA before giving the stage its
        // second arrival.  The consumers do none of this: between two tiles they wait on
        // one mbarrier.
        if (lane == 0) {
            tma::prefetch_desc(&tp.map); tma::prefetch_desc(&tp.gout);
            if (kGgrid) { tma::prefetch_desc(&tp.box[0]); tma::prefetch_desc(&tp.box[1]); tma::prefetch_desc(&tp.box[2]); }
        }
        // The first 2 * kScouts tiles of a CTA are static, the rest comes from the launch's counter.  The scout works
        // on tile `t` while the map of its next tile `t1` is being loaded into the map ring and the index of the one
        // after is being fetched.
        const int stride = kScouts * (int)gridDim.x;
        int t = blockIdx.x + warp * gridDim.x, t1 = t + stride;
        // map load of iteration `i` (tile coordinates c) into its slot of the map ring; lane 0 only
        auto load_map = [&](int i, const TileCoord &c) {
            const int ms = i % kMapStages;
            tma::mbar_arrive_expect_tx(map_full + ms, kMapTileBytes);
            if (kInter) tma::load_3d_hint(s_map + ms * kMapTileFloats, &tp.map, map_full + ms, 2 * c.w0, c.h0, n_begin + c.n, pol_first);
            else tma::load_4d_hint(s_map + ms * kMapTileFloats, &tp.map, map_full + ms, c.w0, c.h0, 0, n_begin + c.n, pol_first);
        };
        TileCoord tc = tile_coord(min(t, total_tiles - 1), tiles_x, tiles_xy);
        if (lane == 0 && t < total_tiles) load_map(warp, tc);  // the ring starts out empty
        int zero_seen = -1;  // bands [0, zero_seen] (index = bands * frame + band) are known to be zero-filled by every CTA
        for (int it = warp;; it += kScouts) {
            const int st = it % kStages, ph = (it / kStages) & 1;
            const int ms = it % kMapStages, mph = (it / kMapStages) & 1;
            const int ms1 = (it + kScouts) % kMapStages, mph1 = ((it + kScouts) / kMapStages) & 1;
            if (t >= total_tiles) {
                tma::mbar_wait_relaxed(empty + st, ph ^ 1);
                if (lane == 0) {
                    s_info[3 * st] = make_int4(0, 0, kInfoStop, 0);
                    tma::mbar_arrive(full + st); tma::mbar_arrive(full + st);
                    progress_store(&s_progress[warp], INT_MAX - kZeroAhead);  // out of tiles: let the zero-fill warp run to the end
                }
                break;
            }
            int t2 = 0;
            if (lane == 0) t2 = (int)atomicAdd(&g_tile_next[slot], 1u) + 2 * stride;  // the tile after the next
            const TileCoord tc1 = tile_coord(min(t1, total_tiles - 1), tiles_x, tiles_xy);
            // next tile's map: its slot was last used kMapStages iterations ago and is normally free by now
            bool next_loaded = t1 >= total_tiles;
            if (!next_loaded && __shfl_sync(0xffffffffu, (int)tma::mbar_test(map_empty + ms1, mph1 ^ 1), 0)) {
                if (lane == 0) load_map(it + kScouts, tc1);
                next_loaded = true;
            }
            // this tile: bounding box of its taps from the map tile in shared memory
            const int cols = min(kTW, g.Wo - tc.w0), rows = min(kTH, g.Ho - tc.h0);
            tma::mbar_wait_relaxed(map_full + ms, mph);
            float xlo, xhi, ylo, yhi;
            map_tile_range<kInter>(s_map + ms * kMapTileFloats, rows, cols, lane, xlo, xhi, ylo, yhi);
            int4 info = box_of_range<kBorder, kAlign, false, 16 / (int)sizeof(T)>(xlo, xhi, ylo, yhi, g.W, g.H, cols == kTW && rows == kTH);
            info.w = tc.n;
            const int progress = kBands * tc.n + (kBands * (t - tc.n * tiles_xy)) / tiles_xy;  // in bands
            const bool want_box = kGgrid && !(info.z & (kInfoFallback | kInfoEmpty));
            const int shape = info.z & 0xff;
            tma::mbar_wait_relaxed(empty + st, ph ^ 1);
            if (lane == 0) {
                s_info[3 * st] = info;
                s_info[3 * st + 1] = make_int4(tc.h0, tc.w0, 0, 0);
                // the tile's base pointers, computed once here instead of by each of the group's eight warps: this frame's
                // grad_input plane 0 and the tile's first grad_grid element
                {
                    const uint64_t p_gin = kGin ? reinterpret_cast<uint64_t>((float *)gin.p + (int64_t)(n_begin + tc.n) * gin.sN) : 0;
                    const uint64_t p_gg = kGgrid ? reinterpret_cast<uint64_t>((float *)ggrid.p + ((int64_t)(n_begin + tc.n) * ggrid.sN +
                                                                                               (int64_t)tc.h0 * ggrid.s1 + (int64_t)tc.w0 * ggrid.s2)) : 0;
                    reinterpret_cast<ulonglong2 *>(s_info)[3 * st + 2] = make_ulonglong2(p_gin, p_gg);
                }
                tma::mbar_arrive_expect_tx(full + st, S::kGoutBytes + (want_box ? box_w(shape) * box_h(shape) * CS * (int)sizeof(T) : 0));
                tma::load_4d_hint(s_gout + (size_t)st * S::kGoutBytes, &tp.gout, full + st, tc.w0, tc.h0, 0, n_begin + tc.n, pol_first);
                if (want_box) tma::load_4d_hint(s_box + (size_t)st * S::kBoxBytes, &tp.box[shape], full + st, info.x, info.y, 0, n_begin + tc.n, pol_box);
                if (kGin && !(info.z & kInfoEmpty)) {
                    // the last band this tile's REDs can land in: the box rows when the taps were bounded, else the whole frame
                    const int y_hi = (info.z & kInfoFallback) ? g.H - 1 : min(info.y + box_h(shape), g.H) - 1;
                    const int need = kBands * tc.n + (kBands * y_hi) / g.H;
                    // the zero-fill warp keeps `zero_ahead` bands ahead of what the scouts publish: the output position of
                    // the tile, or the band it needs if that is further on (a map that samples far away must not starve)
                    progress_store(&s_progress[warp], max(progress, need));
                    // (the zero-fill warps of a CTA take the bands round-robin: completion is not in order, check every band)
                    for (int b = zero_seen + 1; b <= need; ++b)
                        while (ld_acquire(&g_zero_done[slot][b]) < gridDim.x) __nanosleep(64);
                    zero_seen = max(zero_seen, need);
                } else if (kGin) {
                    progress_store(&s_progress[warp], progress);
                }
                // second arrival: passes on (cta scope) the acquire above and this scout's view of the map tile
                tma::mbar_arrive(full + st);
            }
            if (!next_loaded) {
                tma::mbar_wait_relaxed(map_empty + ms1, mph1 ^ 1);
                if (lane == 0) load_map(it + kScouts, tc1);
            }
            t = t1; tc = tc1;
            t1 = __shfl_sync(0xffffffffu, t2, 0);
        }
    } else if (warp >= kZeroWarp) {
        // ===== zero-fill of grad_input: this CTA's 1/gridDim share of every band, kZeroAhead bands ahead of the scouts; the
        // zero-fill warps take the bands round-robin =====
        if (kGin) {
            const int64_t plane = (int64_t)g.H * g.W;  // dense NCHW frame (host-checked), W % 4 == 0, base 16-byte aligned
            const int last = n_frames * kBands - 1;
            for (int idx = warp - kZeroWarp; idx <= last; idx += kZeroWarps) {
                const int f = idx / kBands, b = idx % kBands;
                while (max(progress_load(&s_progress[0]), progress_load(&s_progress[1])) + kZeroAhead < idx) __nanosleep(kZeroPollNs);
                const int r0 = (b * g.H + kBands - 1) / kBands, r1 = ((b + 1) * g.H + kBands - 1) / kBands;
                const int band_vec = (r1 - r0) * (g.W / 4);  // float4 per channel plane
                const int share = (band_vec + gridDim.x - 1) / gridDim.x;
                const int v0 = blockIdx.x * share, v1 = min(band_vec, v0 + share);
                float *const fp = (float *)gin.p + (int64_t)(n_begin + f) * gin.sN + (int64_t)r0 * g.W;
                for (int c = 0; c < CS; ++c) {
                    float4 *__restrict__ dst = reinterpret_cast<float4 *>(fp + c * plane);
                    for (int v = v0 + lane; v < v1; v += 32) tma::st_zero_v4_hint(dst + v, pol_zero);
                }
                __threadfence();
                __syncwarp();
                if (lane == 0) atomicAdd(&g_zero_done[slot][idx], 1u);
            }
        }
    } else {
        // ===== consumers: group `grp` owns the iterations it = grp, grp + 2, ...; a warp owns a 32 x 4 strip of the tile =====
        const int cw = warp - kScouts, grp = cw / kGroupWarps, wg = cw % kGroupWarps;
        const int col0 = (wg & 1) * 32, row0 = (wg >> 1) * kStripRows;
        Queue<CS> q;
        q.buf = s_queue + cw * kQueueCap;
        q.count = 0;
        const float2 size2 = kAlign ? make_float2(Wm1, Hm1) : make_float2(Wf, Hf);
        const float2 gmul2 = make_float2((kAlign ? Hm1 : Hf) * 0.5f, (kAlign ? Wm1 : Wf) * 0.5f);   // (gym, gxm)
        // this lane's first map element, grad_output element and grad_grid element of a tile, relative to the tile
        const int map_lane = kInter ? row0 * (2 * kTW) + 2 * (col0 + lane) : row0 * kTW + col0 + lane;
        const int gout_lane = row0 * kTW + col0 + lane;
        const int64_t gg_lane = kGgrid ? (int64_t)row0 * ggrid.s1 + (int64_t)(col0 + lane) * ggrid.s2 : 0;
        const int plane_elems = g.H * g.W;   // grad_input is dense NCHW (host-checked)
        for (int it = grp;; it += kGroups) {
            const int is = it % kStages, ph = (it / kStages) & 1;
            // one warp of the group waits on the stage's mbarrier, the others park on a hardware barrier and spin on nothing
            if (wg == 0) tma::mbar_wait(full + is, ph);
            tma::named_bar_sync(1 + grp, kGroupWarps * 32);
            const int4 info = s_info[3 * is], where = s_info[3 * is + 1];
            if (info.z & kInfoStop) break;
            const int n = n_begin + info.w;
            const int shape = info.z & 0xff;
            const int ms = it % kMapStages;
            const float *mp = s_map + ms * kMapTileFloats;
            const T *gop = reinterpret_cast<const T *>(s_gout + (size_t)is * S::kGoutBytes) + gout_lane;
            const T *box0 = reinterpret_cast<const T *>(s_box + (size_t)is * S::kBoxBytes);
            // this frame's grad_input planes: one 64-bit base per channel, source pixels are 32-bit offsets from them
            const ulonglong2 base = reinterpret_cast<const ulonglong2 *>(s_info)[3 * is + 2];   // published by the scout
            float *gp[CS];
            gp[0] = reinterpret_cast<float *>(base.x);
#pragma unroll
            for (int k = 1; k < CS; ++k) gp[k] = gp[k - 1] + plane_elems;
            float *__restrict__ ggq = kGgrid ? reinterpret_cast<float *>(base.y) + gg_lane : nullptr;

            if (info.z & kInfoInterior) {
                // the box address of source pixel (x, y) is bp + y * pitch + x: fold the box origin into the base
                const int pitch = box_w(shape), plane = box_w(shape) * box_h(shape);
                interior_strip<T, CS, kAlign, kInter, kGin, kGgrid>(lane, mp + map_lane, gop, box0 - (info.y * pitch + info.x), pitch, plane,
                                                                    size2, g.W, gmul2, gp, ggq, ggrid.s1, ggrid.s3, q, pol_gg);
            } else {
                const int pitch = box_w(shape), plane = box_w(shape) * box_h(shape);
                const T *__restrict__ ip = (const T *)in.p + (int64_t)n * in.sN;
                masked_strip<T, CS, kBorder, kAlign, kInter, kGin, kGgrid>(lane, info, where.x + row0, where.y + col0, row0, col0, mp, gop,
                                                                        box0 - (info.y * pitch + info.x), pitch, plane, ip, in.s2, in.s1,
                                                                        g, gp, ggq, ggrid.s1, ggrid.s3, q, pol_gg);
            }
            if (kGin) queue_flush<CS>(q, gp, lane);
            __syncwarp();
            if (lane == 0) { tma::mbar_arrive(empty + is); tma::mbar_arrive(map_empty + ms); }
        }
    }
    __syncthreads();
    // the last CTA to leave hands the counter slot back clean
    if (threadIdx.x == 0) {
        __threadfence();
        if (atomicAdd(&g_exit_count[slot], 1u) == gridDim.x - 1) {
            if (kGin) for (int i = 0; i < n_frames * kBands; ++i) g_zero_done[slot][i] = 0u;
            g_tile_next[slot] = 0u;
            g_exit_count[slot] = 0u;
            __threadfence();
        }
    }
}

template <typename T, int CS, bool kBorder, bool kAlign, bool kInter, bool kGin, bool kGgrid>
bool launch_k(const TmaParams &tp, const Problem &pb, int tiles_x, int tiles_y, int total, int n0, cudaStream_t st)
{
    auto kern = bwd_tma_kernel<T, CS, kBorder, kAlign, kInter, kGin, kGgrid>;
    using S = Smem<CS, kGgrid, (int)sizeof(T)>;
    static std::atomic<uint64_t> attr_done{0};  // per instantiation, one bit per device
    if (!ensure_dynamic_smem(reinterpret_cast<const void *>(kern), S::kTotal, attr_done)) return false;
    const int grid = total < sm_count() ? total : sm_count();
    int n_frames = total / (tiles_x * tiles_y);
    SlotLease lease(kRingBackward, st);
    if (!lease.ok()) return false;  // stream capture: the caller takes the memset + non-persistent kernel path
    int slot = lease.slot();
    const int64_t frame_bytes = (int64_t)CS * pb.g.H * pb.g.W * 4;
    int bands = (int)((frame_bytes + kBandBytes - 1) / kBandBytes);
    bands = bands < 1 ? 1 : bands > kMaxBands ? kMaxBands : bands;
    // The scouts wait for EVERY CTA of the launch to have zero-filled a band of grad_input: all CTAs must be resident at
    // the same time.  A cooperative launch makes the driver guarantee that (or refuse the launch: SM-limited contexts
    // such as MPS partitions or green contexts, where the caller then falls back to the non-persistent kernels).
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)grid); cfg.blockDim = dim3(kThreads); cfg.dynamicSmemBytes = S::kTotal; cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeCooperative; attr[0].val.cooperative = 1;
    cfg.attrs = attr; cfg.numAttrs = 1;
    if (cudaLaunchKernelEx(&cfg, kern, tp, pb.in, pb.grid, pb.gin, pb.ggrid, pb.g, tiles_x, tiles_y, total, n0, n_frames, slot, bands) != cudaSuccess) {
        cudaGetLastError();
        lease.cancel();
        return false;
    }
    note_launch();
    note_kernel(sizeof(T) == 2 ? "bwd_tma_16" : "bwd_tma");
    return true;
}

template <typename T, int CS, bool kBorder, bool kAlign, bool kInter>
bool launch_mask(const TmaParams &tp, const Problem &pb, int tx, int ty, int total, int n0, cudaStream_t st)
{
    if (pb.want_gin && pb.want_ggrid) return launch_k<T, CS, kBorder, kAlign, kInter, true, true>(tp, pb, tx, ty, total, n0, st);
    if (pb.want_gin) return launch_k<T, CS, kBorder, kAlign, kInter, true, false>(tp, pb, tx, ty, total, n0, st);
    return launch_k<T, CS, kBorder, kAlign, kInter, false, true>(tp, pb, tx, ty, total, n0, st);
}

template <typename T, int CS, bool kInter>
bool launch_ba(const TmaParams &tp, const Problem &pb, int tx, int ty, int total, int n0, cudaStream_t st)
{
    const bool border = pb.g.padding == PWS_PAD_BORDER, align = pb.g.align != 0;
    if (border && align) return launch_mask<T, CS, true, true, kInter>(tp, pb, tx, ty, total, n0, st);
    if (border) return launch_mask<T, CS, true, false, kInter>(tp, pb, tx, ty, total, n0, st);
    if (align) return launch_mask<T, CS, false, true, kInter>(tp, pb, tx, ty, total, n0, st);
    return launch_mask<T, CS, false, false, kInter>(tp, pb, tx, ty, total, n0, st);
}

}  // namespace

// Prepared launch state of an eligible problem (tensor maps are encoded once per call, not per chunk).
struct BwdTmaPlan {
    TmaParams tp;
    bool inter;
    int tiles_x, tiles_y;
};

// Returns a heap plan when the TMA backward can take the problem, nullptr otherwise.
BwdTmaPlan *backward_tma_plan(const Problem &pb)
{
    const Geometry &g = pb.g;
    if (tma_disabled()) return nullptr;
    if (pb.grid_dtype != PWS_F32) return nullptr;
    const bool half_frames = pb.in_dtype == PWS_F16 || pb.in_dtype == PWS_BF16;   // grad_output has the frames' type, grad_input is fp32
    if (pb.in_dtype != PWS_F32 && !half_frames) return nullptr;
    if (half_frames ? g.C != 3 : (g.C != 1 && g.C != 3)) return nullptr;   // (16-bit: the RGB instantiations only)
    if (g.W > (1 << 22) || g.H > (1 << 22)) return nullptr;
    if (pb.want_gin && !(pb.gin.s3 == 1 && pb.gin.s2 == g.W && pb.gin.s1 == g.W * g.H)) return nullptr;
    // in-kernel zero-fill writes float4: frame base and frame stride 16-byte aligned
    if (pb.want_gin && ((reinterpret_cast<uintptr_t>(pb.gin.p) & 15) || (pb.gin.sN % 4) || (g.W % 4))) return nullptr;
    if (pb.want_ggrid) {
        // written with plain stores: planar (two scalars) or interleaved (one float2)
        if (pb.ggrid.s3 == 1 && ((reinterpret_cast<uintptr_t>(pb.ggrid.p) & 7) || (pb.ggrid.sN & 1) || (pb.ggrid.s1 & 1) || (pb.ggrid.s2 & 1)))
            return nullptr;
    }
    BwdTmaPlan *pl = new BwdTmaPlan;
    pl->tiles_x = (g.Wo + kTW - 1) / kTW;
    pl->tiles_y = (g.Ho + kTH - 1) / kTH;
    bool ok = encode_map_tma(pb.grid, g, &pl->tp.map, &pl->inter);
    ok = ok && encode_frame_tma(pb.gout, g.Wo, g.Ho, g.C, g.N, kTW, kTH, g.C, &pl->tp.gout, pb.in_dtype);
    for (int s = 0; ok && s < kNumShapes; ++s) ok = encode_frame_tma(pb.in, g.W, g.H, g.C, g.N, box_w(s), box_h(s), g.C, &pl->tp.box[s], pb.in_dtype);
    if ((int64_t)pl->tiles_x * pl->tiles_y * g.N > INT_MAX) ok = false;
    if (!ok) { delete pl; return nullptr; }
    return pl;
}

void backward_tma_free(BwdTmaPlan *pl) { delete pl; }

int backward_tma_max_frames() { return kSyncFrames; }

// Launch frames [n0, n0+nn), nn <= backward_tma_max_frames().  Zero-fills grad_input of those frames itself.
bool launch_backward_tma(const BwdTmaPlan *pl, const Problem &pb, int n0, int nn, cudaStream_t st)
{
    const int total = pl->tiles_x * pl->tiles_y * nn;
    if (total <= 0) return true;
    if (pb.in_dtype == PWS_F16)
        return pl->inter ? launch_ba<__half, 3, true>(pl->tp, pb, pl->tiles_x, pl->tiles_y, total, n0, st)
                         : launch_ba<__half, 3, false>(pl->tp, pb, pl->tiles_x, pl->tiles_y, total, n0, st);
    if (pb.in_dtype == PWS_BF16)
        return pl->inter ? launch_ba<__nv_bfloat16, 3, true>(pl->tp, pb, pl->tiles_x, pl->tiles_y, total, n0, st)
                         : launch_ba<__nv_bfloat16, 3, false>(pl->tp, pb, pl->tiles_x, pl->tiles_y, total, n0, st);
    if (pb.g.C == 3)
        return pl->inter ? launch_ba<float, 3, true>(pl->tp, pb, pl->tiles_x, pl->tiles_y, total, n0, st)
                         : launch_ba<float, 3, false>(pl->tp, pb, pl->tiles_x, pl->tiles_y, total, n0, st);
    return pl->inter ? launch_ba<float, 1, true>(pl->tp, pb, pl->tiles_x, pl->tiles_y, total, n0, st)
                     : launch_ba<float, 1, false>(pl->tp, pb, pl->tiles_x, pl->tiles_y, total, n0, st);
}

}  // namespace pws
