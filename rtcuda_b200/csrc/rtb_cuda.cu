// rtb_cuda.cu — the shipped backend: sm_100a kernels, device memory, CUB
// radix sort / select, CUDA events, and the C ABI of include/rtb.h.
//
// Kernels (all plain SIMT; nothing on this path is a dense contraction, so
// no tensor cores):
//   k_trace<which, pool>  persistent traversal kernel for the extend (closest
//                         hit) and shadow (any hit) rays of one iteration:
//                         grid = SMs x resident blocks, a warp claims 128 queue
//                         entries with one atomicAdd (lane 0) and a shuffle
//                         broadcast and refills idle lanes while the others
//                         keep traversing; triangle tests pooled per warp in
//                         shared memory on large scenes (replaces kernels ch /
//                         ah, render.cuh:278-328, which launch one thread per
//                         ray in 64-thread blocks)
//   k_shade<type>         grid-stride over one material queue, writes the next
//                         rays in place (replaces mat + init, render.cuh:84-248)
//   k_generate            new camera paths behind the shaded ones (gen, :250-275)
//   k_control             single-thread queue bookkeeping; raises `done` in
//                         mapped host memory (replaces the four blocking
//                         4-byte device->host copies per iteration,
//                         render.cuh:433-445)
//   k_for<Functor>        one thread per element for builder / utility bodies
#include <cuda_runtime.h>
#include <dlfcn.h>
#include <nccl.h>  // types and prototypes only: the library is opened with dlopen on first use (no link-time dependency)

#include <cctype>
#include <cstdlib>
#include <mutex>

#include <cub/block/block_scan.cuh>
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>
#include <cub/device/device_select.cuh>

#include "rtb_engine.h"

#define RTB_CUDA_CHECK(expr)                                                                              \
    do {                                                                                                  \
        cudaError_t e_ = (expr);                                                                          \
        if (e_ != cudaSuccess)                                                                            \
            throw rtb::Error(e_ == cudaErrorMemoryAllocation ? RTB_ERR_OOM : RTB_ERR_CUDA,                \
                             std::string(#expr) + ": " + cudaGetErrorName(e_) + " (" + cudaGetErrorString(e_) + ")"); \
    } while (0)

namespace rtb {

constexpr int kBlock = 256;
// Threads per block of the persistent trace kernels (warps are independent there).  At 64 registers 32 warps fill the
// register file of an SM: a trace kernel launched at full occupancy leaves no room for any block of the OTHER
// wavefront, whose kernels then only start in its tail.  With W wavefronts each trace launch therefore takes 1 / W of
// the SM (8 / W blocks of 128 threads, trace_grid()), so that the wavefronts really run side by side — one's
// issue-bound traversal next to another's DRAM-bound shading (128-thread shade blocks fit the registers left):
// two wavefronts C2 37.4 -> 35.4 ms, C4 37.6 -> 29.2 ms, C1 3.34 -> 2.97 ms; four 34.9 / 27.5 / 2.92 ms
// (profiles/r1/README.md, sessions 74-77).
#ifndef RTB_TRACE_BLOCK
#define RTB_TRACE_BLOCK 128
#endif
constexpr int kTraceBlock = RTB_TRACE_BLOCK;
#ifndef RTB_TRACE_MIN_BLOCKS
#define RTB_TRACE_MIN_BLOCKS (1024 / RTB_TRACE_BLOCK)  // 32 warps per SM at 64 registers (40 warps at 51 registers: A/B in profiles/r2)
#endif
constexpr int kTraceBlocksPerSm = RTB_TRACE_MIN_BLOCKS;

template <class F>
__global__ void __launch_bounds__(kBlock) k_for(int n, F f) {
    const int i = blockIdx.x * kBlock + threadIdx.x;
    if (i < n) f(i);
}

__global__ void __launch_bounds__(kBlock) k_generate(WaveState W, RenderConsts rc) {
    const int n = generate_count(W);
    for (int i = blockIdx.x * kBlock + threadIdx.x; i < n; i += gridDim.x * kBlock) generate_body(W, rc, i);
}

__device__ __forceinline__ void prefetch_l2(const void *p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }

// The hit records are a pure stream (read once, in order): each thread copies the record of its NEXT loop iteration
// into its own shared-memory slot with cp.async (LDGSTS: no registers, nothing waits) while it shades the current
// one.  ncu before: 35 % of the kernel's stall samples sat on the first use of the record (DRAM latency).
__device__ __forceinline__ void cp_async16(void *smem, const void *gmem) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((unsigned)__cvta_generic_to_shared(smem)), "l"(gmem));
}
// Up to 128 registers (no spills; the matte / glossy kernels take 94, 80 would spill): shade is bound by DRAM and
// latency, not by its occupancy.  The specular kernels need 64 registers and get half as many more blocks.
#ifndef RTB_SHADE_BLOCK
#define RTB_SHADE_BLOCK 128
#endif
constexpr int kShadeBlock = RTB_SHADE_BLOCK;  // small blocks: they fit the registers a half-occupancy trace kernel leaves free
#ifndef RTB_SHADE_MATTE_BLOCKS
#define RTB_SHADE_MATTE_BLOCKS 2  // per 256 threads: 2 -> up to 128 registers; 3 -> 85 (spills), 4 -> 64 (A/B: profiles/r2)
#endif
constexpr int shade_blocks_per_sm(int type) { return ((type == RTB_MIRROR || type == RTB_GLASS) ? 3 : RTB_SHADE_MATTE_BLOCKS) * (256 / kShadeBlock); }
template <int TYPE, bool EXT = false>
__global__ void __launch_bounds__(kShadeBlock, shade_blocks_per_sm(TYPE)) k_shade(WaveState W, SceneView S, RenderConsts rc, bool shadows) {
    __shared__ float4 stage[2][3][kShadeBlock];
    const int n = W.c->n_mat[TYPE];
    const int stride = gridDim.x * kShadeBlock, t = threadIdx.x;
    ShadeTally tally; tally.extend = 0u; tally.shadow = 0u;
    int i = blockIdx.x * kShadeBlock + t;
    if (i < n) {
        const size_t q = (size_t)W.qbase[TYPE] + (size_t)i;
        cp_async16(&stage[0][0][t], W.ma + q); cp_async16(&stage[0][1][t], W.mb + q); cp_async16(&stage[0][2][t], W.mc + q);
    }
    asm volatile("cp.async.commit_group;");
    for (int buf = 0; i < n; i += stride, buf ^= 1) {
        if (i + stride < n) {
            const size_t q = (size_t)W.qbase[TYPE] + (size_t)(i + stride);
            cp_async16(&stage[buf ^ 1][0][t], W.ma + q); cp_async16(&stage[buf ^ 1][1][t], W.mb + q); cp_async16(&stage[buf ^ 1][2][t], W.mc + q);
        }
        asm volatile("cp.async.commit_group;");
        asm volatile("cp.async.wait_group 1;" ::: "memory");  // everything but the group just committed has landed
        const float4 a4 = stage[buf][0][t], b4 = stage[buf][1][t], h4 = stage[buf][2][t];
        F4 a, b, hr;
        a.x = a4.x; a.y = a4.y; a.z = a4.z; a.w = a4.w; b.x = b4.x; b.y = b4.y; b.z = b4.z; b.w = b4.w;
        hr.x = h4.x; hr.y = h4.y; hr.z = h4.z; hr.w = h4.w;
        shade_item<TYPE, EXT>(W, S, rc, shadows, i, a, b, hr, tally);
    }
    asm volatile("cp.async.wait_all;" ::: "memory");
    tally_flush(W.c, tally);
}

__global__ void k_control(WaveState W, bool shadows) { control_body(W, shadows); }

// Persistent traversal with dynamic ray fetch (after Aila & Laine 2009): the
// grid is SMs x resident blocks whatever the queue size; a warp claims `chunk`
// queue entries with one atomicAdd (elected lane) + shuffle broadcast, and
// whenever fewer than `refill` of its lanes still hold a live ray the idle
// lanes take new entries while the others keep their traversal state, so short
// rays (a wall) do not wait for long ones (the bunny) in the same warp.  ncu r1
// before this: 6.9-11 of 32 lanes active per instruction in k_extend.
struct FetchTuning {
    int refill;    // refill idle lanes when fewer than this many lanes hold a live ray
    int chunk;     // queue entries a warp claims with one atomicAdd
    int prefetch;  // prefetch a claimed chunk's rays into L2
    int tri_step;  // own-lane triangle tests: 0 = all of a node's triangles at once, k = at most k per step (the rest carries over)
};

// Pooled triangle tests (POOL).  ncu r1 (profiles/r1/r1_ncu_full_big_launches_session6.txt and the
// source page of the same capture): the node step ran with 24 of 32 lanes but the per-ray triangle
// loop with 5-8, and took 31 % of the issue slots of k_extend for ~1 triangle per ray and step.
// With POOL the hit triangles of all the rays of a warp are gathered in shared memory after every
// node step and tested 32 at a time, one candidate per lane whatever ray it belongs to; the
// order-dependent accept rule (0 < t <= tmax, tmax shrinking, last tie wins: triangle.cuh:49,
// bvh.cuh:231) stays with the ray's own lane, which walks its candidates in the same order as the
// per-ray loop, so results are bit-identical.
struct alignas(16) WarpScratch {
    float4 ro[32];   // per lane: ray origin | pixel (extend)
    float4 rd[32];   // per lane: ray direction | sample<<8|bounces (extend)
    float4 fin[32];  // per lane: the queue word only the finish needs (extend: beta | pdf, shadow: radiance | pixel), by cp.async
    float4 res[32];  // per candidate: t (or -1), u, v, leaf-order triangle index
    uint2 item[32];  // per candidate: leaf-order triangle index, owner lane
};
template <bool ANY>
__device__ __forceinline__ void pooled_triangles(WarpScratch &ws, const Bvh8View &B, Traversal<ANY, false> &T, uint32_t tx,
                                                 uint32_t ty, bool &has, bool &pending, const unsigned lane,
                                                 const unsigned lanes_below) {
    // A lane submits at most 3 candidates per round (one leaf child holds <= 3 triangles), so the
    // positions come from two ballots instead of a 5-step shuffle scan and the per-lane loops are
    // three predicated steps; a lane's surplus, and whatever does not fit in 32 slots, waits for the
    // next round.
    while (__any_sync(0xffffffffu, ty != 0u)) {
        const int cnt = min(__popc(ty), 3);
        const unsigned b0 = __ballot_sync(0xffffffffu, cnt & 1), b1 = __ballot_sync(0xffffffffu, cnt & 2);
        const int first = __popc(b0 & lanes_below) + 2 * __popc(b1 & lanes_below);
        const int total = __popc(b0) + 2 * __popc(b1);
        const int take = max(0, min(cnt, 32 - first));
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            if (k < take) {
                const int bit = 31 - __clz(ty);
                ty &= ~(1u << bit);
                ws.item[first + k] = make_uint2(tx + (uint32_t)bit, lane);
            }
        }
        __syncwarp();
        if ((int)lane < min(total, 32)) {
            const uint2 it = ws.item[lane];
            const float4 o = ws.ro[it.y], d = ws.rd[it.y];
            const Tri48 tr = load_tri(B.tris, (int)it.x);
            float u, v;
            const float t = tri_candidate(tr, v3(o.x, o.y, o.z), v3(d.x, d.y, d.z), u, v);
            ws.res[lane] = make_float4(t, u, v, __int_as_float((int)it.x));
        }
        __syncwarp();
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            if (k < take && has) {
                const float4 c = ws.res[first + k];
                if (T.accept(B, __float_as_int(c.w), c.x, c.y, c.z)) {  // any-hit ray occluded: finished
                    ty = 0u; has = false; pending = true;
                }
            }
        }
        __syncwarp();
    }
}
// the same triangles, each ray's lane on its own (A/B, and the better choice when rays meet ~1 triangle per step)
template <bool ANY>
__device__ __forceinline__ void own_triangles(const Bvh8View &B, Traversal<ANY, false> &T, uint32_t tx, uint32_t ty, bool &has,
                                              bool &pending) {
    while (ty) {
        const int bit = 31 - __clz(ty);
        ty &= ~(1u << bit);
        const int idx = (int)(tx + (uint32_t)bit);
        const Tri48 tr = load_tri(B.tris, idx);
        float u, v;
        const float t = tri_candidate(tr, T.r.o, T.r.d, u, v);
        if (T.accept(B, idx, t, u, v)) { has = false; pending = true; break; }
    }
}

// Stack variants of the persistent kernel.  Default: LocalStack (rtb_bvh8.h).  HybridStack<N> keeps the first N
// entries of every thread in shared memory ([N][kBlock] uint2: the bank is the thread, so lanes at different depths
// never conflict) and the rest in local memory; RTB_SMEM_STACK=N selects it (N = 8) for an A/B.  The shared memory it
// takes (N x 2 KB per block, four blocks per SM) comes out of the L1 that caches the nodes.
struct LocalStackK : LocalStack {
    __device__ explicit LocalStackK(uint2 *) {}
};
template <int N>
struct HybridStack {
    uint2 *s;
    uint32_t x[kStackSize - N], y[kStackSize - N];
    __device__ explicit HybridStack(uint2 *column) : s(column) {}
    __device__ __forceinline__ void put(int i, uint32_t a, uint32_t b) {
        if (i < N) s[i * kTraceBlock] = make_uint2(a, b);
        else { x[i - N] = a; y[i - N] = b; }
    }
    __device__ __forceinline__ void get(int i, uint32_t &a, uint32_t &b) const {
        if (i < N) { const uint2 v = s[i * kTraceBlock]; a = v.x; b = v.y; }
        else { a = x[i - N]; b = y[i - N]; }
    }
};
// INST: two-level scenes (rtb_bvh8.h, Traversal<.., INST>): stepped schedule only; the world ray a lane needs when it
// enters or leaves an instance is the one in its shared-memory slot (ws.ro / ws.rd).
template <bool ANY, bool POOL, bool INST = false, class STACK = LocalStackK>
__device__ __forceinline__ void persistent_trace(WarpScratch &ws, const WaveState &W, const SceneView &S, FetchTuning tune, uint2 *ws_stack = nullptr) {
    const int n = ANY ? W.c->n_shadow : W.c->n_extend;
    int32_t *head = ANY ? &W.c->shadow_head : &W.c->extend_head;
    const unsigned lane = threadIdx.x & 31u;
    const unsigned lanes_below = (1u << lane) - 1u;
    Traversal<ANY, false, INST> T;
    STACK st(ws_stack);
    bool has = false, exhausted = false, pending = false;
    int qi = 0;
    int chunk_next = 0, chunk_end = 0;  // warp-uniform: the part of the queue this warp has claimed
    uint32_t tx = 0u, ty = 0u;          // triangles of the current node still to test: base | bits
    while (true) {
        // results of the rays that finished since the last refill are written here, together, so
        // that the hit-record / atomic code runs with many lanes instead of one at a time
        if (pending) {
            asm volatile("cp.async.wait_all;" ::: "memory");  // this lane's finish word (copied when the ray was fetched)
            const float4 fw = ws.fin[lane];
            if (ANY) {
                if (!T.found) {  // ah, render.cuh:278-294: unoccluded -> splat
                    const V3 L = v3(fw.x, fw.y, fw.z);
                    if (finite3(L)) accum_add(W, __float_as_uint(fw.w), L);
                }
            } else if (T.hit.tri < 0) {
                if (W.has_env) extend_miss(W, __float_as_uint(ws.ro[lane].w), v3(fw.x, fw.y, fw.z));
            } else {
                const int mat = INST ? hit_material(S, T.hit.tri, T.hit_inst) : S.tri_meta[T.hit.tri].material;
                const int type = mat >> 24;
                const int j = hit_queue_push(W, type);
                if (INST) W.hit_inst[j] = T.hit_inst;
                F4 beta; beta.x = fw.x; beta.y = fw.y; beta.z = fw.z; beta.w = fw.w;
                const float4 o = ws.ro[lane], d = ws.rd[lane];
                F4 ma; ma.x = d.x; ma.y = d.y; ma.z = d.z; ma.w = o.w;
                F4 mb; mb.x = beta.x; mb.y = beta.y; mb.z = beta.z; mb.w = d.w;
                F4 mc; mc.x = i2f(mat); mc.y = T.hit.u; mc.z = T.hit.v; mc.w = i2f(T.hit.tri);
                W.ma[j] = ma; W.mb[j] = mb; W.mc[j] = mc;
                if (W.mis) { W.mis[2 * (size_t)j] = beta.w; W.mis[2 * (size_t)j + 1] = T.hit.t; }
            }
            pending = false;
        }
        // hand queue entries to the idle lanes; a new chunk is claimed (one atomic per warp) when the
        // current one runs out, so most refills cost no global round trip at all.  Holes (slots whose
        // path cast no ray) leave their lane idle for this round.
        unsigned need = __ballot_sync(0xffffffffu, !has);
        for (int round = 0; round < 2 && need != 0u && !exhausted; ++round) {
            if (chunk_next >= chunk_end) {
                int base = 0;
                if (lane == 0u) base = atomicAdd(head, tune.chunk);
                base = __shfl_sync(0xffffffffu, base, 0);
                chunk_next = base;
                chunk_end = min(base + tune.chunk, n);
                if (base >= n) { exhausted = true; break; }
                if (tune.prefetch) {  // pull the chunk's rays towards L2 while the warp still traverses
                    for (int i = base + (int)lane; i < chunk_end; i += 32) {
                        if (ANY) { prefetch_l2(W.sh_o + i); prefetch_l2(W.sh_d + i); }
                        else { prefetch_l2(W.ea + i); prefetch_l2(W.eb + i); prefetch_l2(W.ec + i); }
                    }
                }
            }
            const int idx = chunk_next + __popc(need & lanes_below);
            if (!has && idx < chunk_end) {
                if (ANY) {
                    const F4 o = ldg(W.sh_o + idx), d = ldg(W.sh_d + idx);  // both at once: holes are rare, latency is not
                    if (o.w > 0.f) {
                        cp_async16(&ws.fin[lane], W.sh_L + idx);
                        ws.ro[lane] = make_float4(o.x, o.y, o.z, 0.f);
                        ws.rd[lane] = make_float4(d.x, d.y, d.z, 0.f);
                        T.init(xyz(o), xyz(d), o.w, f2i(d.w));
                        qi = idx; has = true; ty = 0u;
                    }
                } else {
                    const F4 a = ldg(W.ea + idx), b = ldg(W.eb + idx);
                    if (f2u(a.w) != kHolePixel) {
                        cp_async16(&ws.fin[lane], W.ec + idx);
                        ws.ro[lane] = make_float4(a.x, a.y, a.z, a.w);
                        ws.rd[lane] = make_float4(b.x, b.y, b.z, b.w);
                        T.init(xyz(a), xyz(b), FLT_MAX, -1);
                        qi = idx; has = true; ty = 0u;
                    }
                }
            }
            chunk_next = min(chunk_next + __popc(need), chunk_end);
            need = __ballot_sync(0xffffffffu, !has);
        }
        unsigned act = __ballot_sync(0xffffffffu, has);
        if (act == 0u) {
            if (exhausted) return;
            continue;  // chunk boundary (or a run of holes): claim more
        }
        const int keep_going = exhausted ? 1 : tune.refill;
        do {
            if constexpr (INST) {
                if (has && ty == 0u) T.node_part(S.bvh, st, tx, ty);
                if (has && T.cur < 0) {  // (tx, ty) is a leaf list of the top tree: enter its nearest instance
                    if (ty != 0u) {
                        const float4 o = ws.ro[lane], d = ws.rd[lane];
                        T.enter_instance(S.bvh, st, tx, ty, v3(o.x, o.y, o.z), v3(d.x, d.y, d.z));
                    }
                } else if (ty != 0u) {  // two triangles of the list together, as in the flat kernel below
                    const int bit1 = 31 - __clz(ty);
                    ty &= ~(1u << bit1);
                    const bool two = ty != 0u;
                    const int bit2 = two ? 31 - __clz(ty) : bit1;
                    ty &= ~(1u << bit2);
                    const int idx1 = (int)(tx + (uint32_t)bit1), idx2 = (int)(tx + (uint32_t)bit2);
                    const Tri48 tr1 = load_tri(S.bvh.tris, idx1), tr2 = load_tri(S.bvh.tris, idx2);
                    float u1, v1, u2, v2;
                    const float t1 = tri_candidate(tr1, T.r.o, T.r.d, u1, v1);
                    const float t2 = tri_candidate(tr2, T.r.o, T.r.d, u2, v2);
                    if (T.accept(S.bvh, idx1, t1, u1, v1)) { has = false; pending = true; ty = 0u; }
                    else if (two && T.accept(S.bvh, idx2, t2, u2, v2)) { has = false; pending = true; ty = 0u; }
                }
                if (has && ty == 0u) {
                    const float4 o = ws.ro[lane], d = ws.rd[lane];
                    if (!T.advance_inst(st, tx, ty, v3(o.x, o.y, o.z), v3(d.x, d.y, d.z))) { has = false; pending = true; }
                }
            } else if constexpr (POOL) {
                tx = 0u; ty = 0u;
                if (has) T.node_part(S.bvh, st, tx, ty);
                pooled_triangles<ANY>(ws, S.bvh, T, tx, ty, has, pending, lane, lanes_below);
                ty = 0u;
                if (has && !T.advance(st)) { has = false; pending = true; }
            } else if (tune.tri_step > 0) {
                // stepped: at most tri_step triangle tests per lane and step; a lane with more keeps them for
                // the next steps and sits out the node phase meanwhile (its own order of events is unchanged:
                // the next node is fetched only once all triangles of the current one are tested), so one
                // lane's long triangle list no longer idles the rest of the warp
                if (has && ty == 0u) T.node_part(S.bvh, st, tx, ty);
                // tri_step 2 (default): both triangles are fetched and tested together — the loads of the second overlap the
                // arithmetic of the first (C3 105.0 -> 100.0 ms, C2 / C4 unchanged: profiles/r1/README.md, session 64) — and the
                // accept rule then runs on them in list order, so the ray's own order of events is what it was
                if (tune.tri_step == 2) {
                  if (ty != 0u) {
                    const int bit1 = 31 - __clz(ty);
                    ty &= ~(1u << bit1);
                    const bool two = ty != 0u;
                    const int bit2 = two ? 31 - __clz(ty) : bit1;
                    ty &= ~(1u << bit2);
                    const int idx1 = (int)(tx + (uint32_t)bit1), idx2 = (int)(tx + (uint32_t)bit2);
                    const Tri48 tr1 = load_tri(S.bvh.tris, idx1), tr2 = load_tri(S.bvh.tris, idx2);
                    float u1, v1, u2, v2;
                    const float t1 = tri_candidate(tr1, T.r.o, T.r.d, u1, v1);
                    const float t2 = tri_candidate(tr2, T.r.o, T.r.d, u2, v2);
                    if (T.accept(S.bvh, idx1, t1, u1, v1)) { has = false; pending = true; ty = 0u; }
                    else if (two && T.accept(S.bvh, idx2, t2, u2, v2)) { has = false; pending = true; ty = 0u; }
                  }
                } else {
#pragma unroll 1
                for (int k = 0; k < tune.tri_step && ty != 0u; ++k) {
                    const int bit = 31 - __clz(ty);
                    ty &= ~(1u << bit);
                    const int idx = (int)(tx + (uint32_t)bit);
                    const Tri48 tr = load_tri(S.bvh.tris, idx);
                    float u, v;
                    const float t = tri_candidate(tr, T.r.o, T.r.d, u, v);
                    if (T.accept(S.bvh, idx, t, u, v)) { has = false; pending = true; ty = 0u; }
                }
                }
                if (has && ty == 0u && !T.advance(st)) { has = false; pending = true; }
            } else {
                tx = 0u; ty = 0u;
                if (has) T.node_part(S.bvh, st, tx, ty);
                own_triangles<ANY>(S.bvh, T, tx, ty, has, pending);
                ty = 0u;
                if (has && !T.advance(st)) { has = false; pending = true; }
            }
            act = __ballot_sync(0xffffffffu, has);
        } while (__popc(act) >= keep_going);
    }
}
// extend and shadow rays of one iteration in ONE launch (WHICH = 3): a warp that runs out of extend
// rays goes on with shadow rays, so the tail of the first queue overlaps the start of the second.
// WHICH = 1 / 2: extend / shadow only (A/B, and per-stage timing).
// Triangle tests, three schedules (profiles/r1/README.md): each lane walks all the triangles of its node at once
// (tri_step 0); at most tri_step per step, the rest carried over (default, 2: C2 39.5 -> 39.1 ms, C3 116.5 ->
// 108.9 ms); pooled per warp in shared memory (POOL, RTB_POOLED=1: C3 113.5 ms, C2 47.9 ms).
// Tried and dropped: prefetching the next node into L2 during the triangle tests (C3 116 -> 140 ms, C2 40 -> 49 ms).
template <int WHICH, bool POOL, bool INST = false>
__global__ void __launch_bounds__(kTraceBlock, kTraceBlocksPerSm) k_trace(WaveState W, SceneView S, FetchTuning tune) {
    __shared__ WarpScratch scratch[kTraceBlock / 32];
    WarpScratch &ws = scratch[threadIdx.x >> 5];
    if (WHICH & 1) persistent_trace<false, POOL, INST>(ws, W, S, tune);
    if (WHICH == 3) __syncwarp();
    if (WHICH & 2) persistent_trace<true, POOL, INST>(ws, W, S, tune);
}
constexpr int kSmemStack = 8;
__global__ void __launch_bounds__(kTraceBlock, kTraceBlocksPerSm) k_trace_smem_stack(WaveState W, SceneView S, FetchTuning tune) {  // k_trace<3, false> with HybridStack
    __shared__ WarpScratch scratch[kTraceBlock / 32];
    __shared__ uint2 sstack[kSmemStack][kTraceBlock];
    WarpScratch &ws = scratch[threadIdx.x >> 5];
    persistent_trace<false, false, false, HybridStack<kSmemStack>>(ws, W, S, tune, &sstack[0][threadIdx.x]);
    __syncwarp();
    persistent_trace<true, false, false, HybridStack<kSmemStack>>(ws, W, S, tune, &sstack[0][threadIdx.x]);
}
template <int WHICH>
static void launch_trace_kernel(int grid, cudaStream_t st, bool pooled, bool smem_stack, const WaveState &W, const SceneView &S, const FetchTuning &tune) {
    if (WHICH == 3 && smem_stack && !S.bvh.inst && !pooled) { k_trace_smem_stack<<<grid, kTraceBlock, 0, st>>>(W, S, tune); return; }
    if (S.bvh.inst) {  // two-level scene: stepped schedule, two triangles per step
        k_trace<WHICH, false, true><<<grid, kTraceBlock, 0, st>>>(W, S, tune);
    } else if (pooled) k_trace<WHICH, true><<<grid, kTraceBlock, 0, st>>>(W, S, tune);
    else k_trace<WHICH, false><<<grid, kTraceBlock, 0, st>>>(W, S, tune);
}
// one thread per queue entry (A/B against the persistent kernels; COUNT = work counters)
template <bool COUNT>
__global__ void __launch_bounds__(kBlock) k_extend_flat(WaveState W, SceneView S) {
    const int i = blockIdx.x * kBlock + threadIdx.x;
    if (i < W.c->n_extend) extend_body<COUNT>(W, S, i);
}
template <bool COUNT>
__global__ void __launch_bounds__(kBlock) k_shadow_flat(WaveState W, SceneView S) {
    const int i = blockIdx.x * kBlock + threadIdx.x;
    if (i < W.c->n_shadow) shadow_body<COUNT>(W, S, i);
}

// prim_setup_body with the block's vertices (36 bytes per triangle) and records (48 bytes) passing through shared memory,
// so that global memory sees whole 128-bit words at consecutive addresses: one thread per triangle reading nine floats at a
// 36-byte stride and storing twelve at a 48-byte stride took 1.48 ms for the 1.2 GB of a 10 M-triangle scene.
constexpr int kSetupBlock = 256;
__global__ void __launch_bounds__(kSetupBlock) k_prim_setup_tiled(PrimSetupArgs a) {
    __shared__ __align__(16) float vin[kSetupBlock * 9];
    __shared__ float4 rec[kSetupBlock * 3];
    const int b0 = blockIdx.x * kSetupBlock;
    const int cnt = min(kSetupBlock, a.n - b0);
    const float *src = a.vertices + 9 * (size_t)b0;  // (36 * 256 bytes per block: 16-byte aligned like the array)
    if (cnt == kSetupBlock && (reinterpret_cast<uintptr_t>(src) & 15u) == 0) {
        const float4 *s4 = reinterpret_cast<const float4 *>(src);
        float4 *d4 = reinterpret_cast<float4 *>(vin);
        for (int t = threadIdx.x; t < kSetupBlock * 9 / 4; t += kSetupBlock) d4[t] = s4[t];
    } else {
        for (int t = threadIdx.x; t < cnt * 9; t += kSetupBlock) vin[t] = src[t];
    }
    __syncthreads();
    const int i = b0 + threadIdx.x;
    Tri48 tr;
    if (i < a.n) {
        const float *v = vin + 9 * threadIdx.x;
        tr = tri_from_vertices(v3(v[0], v[1], v[2]), v3(v[3], v[4], v[5]), v3(v[6], v[7], v[8]));
        float4 *r = rec + 3 * threadIdx.x;
        r[0] = make_float4(tr.p0x, tr.p0y, tr.p0z, tr.e1x);
        r[1] = make_float4(tr.e1y, tr.e1z, tr.e2x, tr.e2y);
        r[2] = make_float4(tr.e2z, tr.nx, tr.ny, tr.nz);
    }
    __syncthreads();
    float4 *dst = reinterpret_cast<float4 *>(a.tri_in + b0);
    for (int t = threadIdx.x; t < cnt * 3; t += kSetupBlock) dst[t] = rec[t];
    // scene bounds: one reduction per warp, one per block, SIX atomics per block (one per warp was still 1.9 M atomics
    // to six addresses for 10 M triangles — the kernel's whole 1.5 ms)
    __shared__ int32_t part[kSetupBlock / 32][6];
    int32_t o[6] = {0x7fffffff, 0x7fffffff, 0x7fffffff, (int32_t)0x80000000, (int32_t)0x80000000, (int32_t)0x80000000};
    if (i < a.n) {
        V3 lo, hi;
        prim_setup_box(a, i, tr, lo, hi);
        o[0] = float_to_ordered(lo.x); o[1] = float_to_ordered(lo.y); o[2] = float_to_ordered(lo.z);
        o[3] = float_to_ordered(hi.x); o[4] = float_to_ordered(hi.y); o[5] = float_to_ordered(hi.z);
    }
#pragma unroll
    for (int k = 0; k < 3; ++k) { o[k] = __reduce_min_sync(0xffffffffu, o[k]); o[3 + k] = __reduce_max_sync(0xffffffffu, o[3 + k]); }
    if ((threadIdx.x & 31) == 0) for (int k = 0; k < 6; ++k) part[threadIdx.x >> 5][k] = o[k];
    __syncthreads();
    if (threadIdx.x < 6) {
        const int k = threadIdx.x;
        int32_t v = part[0][k];
        for (int w = 1; w < kSetupBlock / 32; ++w) v = k < 3 ? min(v, part[w][k]) : max(v, part[w][k]);
        if (k < 3) atomicMin(a.scene_bounds + k, v); else atomicMax(a.scene_bounds + k, v);
    }
}

// Nearest-neighbour search of one PLOC round (ploc_nn_body) with the cluster boxes of a block's window staged in
// shared memory: every cluster compares itself with 2 x radius neighbours, so the one-thread-per-cluster form reads
// 32 boxes of 32 bytes through the cluster index for every thread — 8.1 of the 17.7 ms of kernel time of a
// 10 M-triangle build (profiles/r2/r2_launches_c3s_session5.csv).  Same arithmetic, same tie rule, same result.
constexpr int kNnBlock = 256, kNnMaxRadius = 64;
__global__ void __launch_bounds__(kNnBlock) k_ploc_nn_tiled(PlocArgs a) {
    __shared__ float lox[kNnBlock + 2 * kNnMaxRadius], loy[kNnBlock + 2 * kNnMaxRadius], loz[kNnBlock + 2 * kNnMaxRadius];
    __shared__ float hix[kNnBlock + 2 * kNnMaxRadius], hiy[kNnBlock + 2 * kNnMaxRadius], hiz[kNnBlock + 2 * kNnMaxRadius];
    const int ncl = ploc_ncl(a);
    const int b0 = blockIdx.x * kNnBlock, first = b0 - a.radius;
    if (blockIdx.x == 0 && threadIdx.x == 0 && a.log) a.log[a.round] = ncl;
    if (b0 >= ncl) return;  // (the grid covers the host's bound of the count)
    const int span = kNnBlock + 2 * a.radius;
    for (int t = threadIdx.x; t < span; t += kNnBlock) {
        const int j = first + t;
        if (j >= 0 && j < ncl) {
            const B2Node b = a.nodes[a.cin[j]];
            lox[t] = b.lox; loy[t] = b.loy; loz[t] = b.loz; hix[t] = b.hix; hiy[t] = b.hiy; hiz[t] = b.hiz;
        }
    }
    __syncthreads();
    const int i = b0 + threadIdx.x;
    if (i >= ncl) return;
    const int ti = threadIdx.x + a.radius;
    B2Node me;
    me.lox = lox[ti]; me.loy = loy[ti]; me.loz = loz[ti]; me.hix = hix[ti]; me.hiy = hiy[ti]; me.hiz = hiz[ti];
    float best = FLT_MAX;
    int bj = -1;
    const int j0 = i - a.radius < 0 ? 0 : i - a.radius;
    const int j1 = i + a.radius > ncl - 1 ? ncl - 1 : i + a.radius;
    for (int j = j0; j <= j1; ++j) {
        if (j == i) continue;
        const int t = j - first;
        B2Node o;
        o.lox = lox[t]; o.loy = loy[t]; o.loz = loz[t]; o.hix = hix[t]; o.hiy = hiy[t]; o.hiz = hiz[t];
        const float ar = union_half_area(me, o);
        if (bj < 0 || ar < best) { best = ar; bj = j; }
    }
    a.nn[i] = bj;
}

// All remaining PLOC rounds in ONE launch once the clusters fit a thread block: cluster list, nearest neighbours and
// merge results live in shared memory, the same round bodies (rtb_build.h) run between block barriers, the
// order-preserving compaction is a block scan.  out[0] = rounds run, out[1] = root node, counts[r] = nodes made by round r.
constexpr int kPlocTail = 1024;
__global__ void __launch_bounds__(kPlocTail) k_ploc_tail(PlocArgs a, int n_leaves, int32_t *out, int32_t *counts) {
    __shared__ int32_t cin[kPlocTail], cout[kPlocTail], nn[kPlocTail];
    // boxes of the clusters by position: the neighbour search of a round reads 2 x radius of them per thread
    __shared__ float lox[kPlocTail], loy[kPlocTail], loz[kPlocTail], hix[kPlocTail], hiy[kPlocTail], hiz[kPlocTail];
    typedef cub::BlockScan<int, kPlocTail> Scan;
    __shared__ typename Scan::TempStorage scan_tmp;
    const int t = threadIdx.x;
    int n = ploc_ncl(a);
    if (n > kPlocTail) { if (t == 0) { out[0] = -1; out[1] = -1; } return; }  // (the host launches it on a bound <= kPlocTail)
    if (t < n) {
        const int c = a.cin[t];
        cin[t] = c;
        const B2Node b = a.nodes[c];
        lox[t] = b.lox; loy[t] = b.loy; loz[t] = b.loz; hix[t] = b.hix; hiy[t] = b.hiy; hiz[t] = b.hiz;
    }
    __syncthreads();
    PlocArgs b = a;
    b.cin = cin; b.cout = cout; b.nn = nn; b.ncl_dev = nullptr; b.log = nullptr;
    int rounds = 0;
    while (n > 1) {
        b.ncl = n;
        B2Node me;
        if (t < n) {  // ploc_nn_body on the shared-memory boxes: same arithmetic, same tie rule
            me.lox = lox[t]; me.loy = loy[t]; me.loz = loz[t]; me.hix = hix[t]; me.hiy = hiy[t]; me.hiz = hiz[t];
            float best = FLT_MAX;
            int bj = -1;
            const int j0 = t - a.radius < 0 ? 0 : t - a.radius;
            const int j1 = t + a.radius > n - 1 ? n - 1 : t + a.radius;
            for (int j = j0; j <= j1; ++j) {
                if (j == t) continue;
                B2Node o;
                o.lox = lox[j]; o.loy = loy[j]; o.loz = loz[j]; o.hix = hix[j]; o.hiy = hiy[j]; o.hiz = hiz[j];
                const float ar = union_half_area(me, o);
                if (bj < 0 || ar < best) { best = ar; bj = j; }
            }
            nn[t] = bj;
        }
        __syncthreads();
        ploc_merge_body(b, n_leaves, t);  // (new nodes go to global memory: visible to the block after the barrier)
        // box of what this position holds after the merge (the union is the one ploc_merge_body stores: same min / max)
        if (t < n) {
            const int j = nn[t];
            if (j >= 0 && nn[j] == t && t < j) {
                me.lox = fminf(me.lox, lox[j]); me.loy = fminf(me.loy, loy[j]); me.loz = fminf(me.loz, loz[j]);
                me.hix = fmaxf(me.hix, hix[j]); me.hiy = fmaxf(me.hiy, hiy[j]); me.hiz = fmaxf(me.hiz, hiz[j]);
            }
        }
        __syncthreads();
        const int v = t < n ? cout[t] : -1;
        const int flag = v >= 0 ? 1 : 0;
        int pos, total;
        Scan(scan_tmp).ExclusiveSum(flag, pos, total);
        __syncthreads();
        if (flag) {
            cin[pos] = v;
            lox[pos] = me.lox; loy[pos] = me.loy; loz[pos] = me.loz; hix[pos] = me.hix; hiy[pos] = me.hiy; hiz[pos] = me.hiz;
        }
        if (t == 0) counts[rounds] = n - total;
        const bool stuck = total >= n;  // a round that merged nothing would spin here for ever (cannot happen with finite boxes)
        n = total;
        ++rounds;
        __syncthreads();
        if (stuck) break;
    }
    if (t == 0) { out[0] = n > 1 ? -1 : rounds; out[1] = cin[0]; }
}

__global__ void __launch_bounds__(kBlock) k_collapse_level(CollapseArgs a, int32_t *zero, int32_t *levels) {
    const int n = *a.n_in_dev;
    if (blockIdx.x == 0 && threadIdx.x == 0) { *zero = 0; if (n > 0) *levels += 1; }
    for (int i = blockIdx.x * kBlock + threadIdx.x; i < n; i += gridDim.x * kBlock) collapse_body(a, i);
}

// ---- binned SAH builder (RTB_BUILDER_BINNED_SAH, rtb_build.h 3') ----
// A level of large ranges: every range has ceil(size / kSahChunk) blocks (blk_in: block -> range).  k_sah_bounds reduces
// box and centroid bounds per block (12 atomics per block and range), k_sah_bin bins in shared memory and flushes once
// per block and range, k_sah_split chooses with one warp per range and makes the children, k_sah_flag / a scan /
// k_sah_scatter / k_sah_copy partition every range stably in place.
constexpr int kSahBlock = 256;
__device__ __forceinline__ bool sah_block_range(const SahArgs &a, int &t, int &p0, int &p1) {
    if ((int)blockIdx.x >= *a.n_blk_in) return false;
    t = a.blk_in[blockIdx.x];
    const SahRange r = a.tin_c[t].r;
    p0 = r.begin + ((int)blockIdx.x - a.tin_c[t].blk0) * kSahChunk;
    p1 = min(p0 + kSahChunk, r.end);
    return true;
}
__device__ __forceinline__ void sah_load_bnd(const SahTask &T, int32_t *bnd, float *scale) {
#pragma unroll
    for (int k = 0; k < 12; ++k) bnd[k] = T.bnd[k];
#pragma unroll
    for (int k = 0; k < 3; ++k) scale[k] = sah_scale(bnd, k);
}
// warp-wide sah_choose: lane k holds bin k of an axis; prefix / suffix merges by shuffles (integer sums and min / max:
// exact in any order), the same costs and the same tie rule (lowest cost, then lowest axis, then lowest plane)
__device__ __forceinline__ SahSplit sah_choose_warp(const int32_t *bins, const float *scale, int size, int lane) {
    SahSplit s; s.axis = -1; s.plane = 0; s.nl = size / 2;
    float best = sah_inf();
    for (int a = 0; a < 3; ++a) {
        if (scale[a] <= 0.f) continue;  // (warp-uniform)
        int32_t L[kSahBinWords], R[kSahBinWords];
        const int32_t *w = bins + (a * kSahBins + lane) * kSahBinWords;
#pragma unroll
        for (int j = 0; j < kSahBinWords; ++j) L[j] = R[j] = w[j];
#pragma unroll
        for (int off = 1; off < 32; off <<= 1) {
            int32_t u[kSahBinWords], d[kSahBinWords];
#pragma unroll
            for (int j = 0; j < kSahBinWords; ++j) { u[j] = __shfl_up_sync(0xffffffffu, L[j], off); d[j] = __shfl_down_sync(0xffffffffu, R[j], off); }
            if (lane >= off) sah_bin_merge(L, u);
            if (lane + off < 32) sah_bin_merge(R, d);
        }
        int32_t R1[kSahBinWords];
#pragma unroll
        for (int j = 0; j < kSahBinWords; ++j) R1[j] = __shfl_down_sync(0xffffffffu, R[j], 1);
        const float c = lane + 1 < kSahBins ? sah_plane_cost(L, R1) : sah_inf();
        const unsigned cb = __float_as_uint(c);  // (c >= 0: the bits order as the values)
        const unsigned m = __reduce_min_sync(0xffffffffu, cb);
        const int k = __ffs(__ballot_sync(0xffffffffu, cb == m)) - 1;
        const int nl = __shfl_sync(0xffffffffu, L[0], k);
        if (__uint_as_float(m) < best) { best = __uint_as_float(m); s.axis = a; s.plane = k; s.nl = nl; }
    }
    return s;
}
__global__ void __launch_bounds__(kSahBlock) k_sah_bounds(SahArgs a) {
    __shared__ int32_t part[kSahBlock / 32][12];
    int t, p0, p1;
    if (!sah_block_range(a, t, p0, p1)) return;
    int32_t b[12];
    sah_bnd_init(b);
    for (int p = p0 + threadIdx.x; p < p1; p += kSahBlock) { const int g = a.idx[p]; sah_bnd_add(b, a.prim_lo[g], a.prim_hi[g]); }
    __syncwarp();
#pragma unroll
    for (int k = 0; k < 12; ++k) b[k] = (k % 6) < 3 ? __reduce_min_sync(0xffffffffu, b[k]) : __reduce_max_sync(0xffffffffu, b[k]);
    if ((threadIdx.x & 31) == 0)
        for (int k = 0; k < 12; ++k) part[threadIdx.x >> 5][k] = b[k];
    __syncthreads();
    if (threadIdx.x < 12) {
        const int k = threadIdx.x;
        int32_t v = part[0][k];
        for (int w = 1; w < kSahBlock / 32; ++w) v = (k % 6) < 3 ? min(v, part[w][k]) : max(v, part[w][k]);
        if ((k % 6) < 3) atomicMin(&a.tin[t].bnd[k], v); else atomicMax(&a.tin[t].bnd[k], v);
    }
}
__global__ void __launch_bounds__(kSahBlock) k_sah_bin(SahArgs a) {
    __shared__ int32_t bins[kSahBinsWords];
    int t, p0, p1;
    if (!sah_block_range(a, t, p0, p1)) return;
    int32_t bnd[12]; float scale[3];
    sah_load_bnd(a.tin_c[t], bnd, scale);
    if (!(scale[0] > 0.f || scale[1] > 0.f || scale[2] > 0.f)) return;  // split by position: no bins
    for (int k = threadIdx.x; k < 3 * kSahBins; k += kSahBlock) sah_bin_init(bins + k * kSahBinWords);
    __syncthreads();
    for (int p = p0 + threadIdx.x; p < p1; p += kSahBlock) { const int g = a.idx[p]; sah_bin_add(bins, a.prim_lo[g], a.prim_hi[g], bnd, scale); }
    __syncthreads();
    int32_t *dst = a.bins + (size_t)t * kSahBinsWords;
    for (int k = threadIdx.x; k < 3 * kSahBins; k += kSahBlock) {
        const int32_t *w = bins + k * kSahBinWords;
        if (w[0] == 0) continue;
        int32_t *d = dst + k * kSahBinWords;
        atomicAdd(d, w[0]);
        for (int j = 0; j < 3; ++j) { atomicMin(d + 1 + j, w[1 + j]); atomicMax(d + 4 + j, w[4 + j]); }
    }
}
__global__ void __launch_bounds__(kSahBlock) k_sah_split(SahArgs a) {
    if (blockIdx.x == 0 && threadIdx.x == 0) { *a.n_clear = 0; *a.n_blk_clear = 0; }
    const int t = (blockIdx.x * kSahBlock + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (t >= *a.n_tin) return;  // (warp-uniform)
    SahTask &T = a.tin[t];
    int32_t bnd[12]; float scale[3];
    sah_load_bnd(T, bnd, scale);
    int32_t *bins = a.bins + (size_t)t * kSahBinsWords;
    const SahSplit s = sah_choose_warp(bins, scale, T.r.end - T.r.begin, lane);
    __syncwarp();
    for (int k = lane; k < 3 * kSahBins; k += 32) sah_bin_init(bins + k * kSahBinWords);  // neutral for the next level
    if (lane == 0) {
        T.axis = s.axis; T.plane = s.plane; T.nl = s.nl;
        SahRange ch[2];
        sah_make_node(a, T.r, bnd, s.nl, a.node_counter, ch);
        sah_push_child(a, ch[0]); sah_push_child(a, ch[1]);
    }
}
__global__ void __launch_bounds__(kSahBlock) k_sah_flag(SahArgs a) {
    int t, p0, p1;
    if (!sah_block_range(a, t, p0, p1)) return;
    const SahTask &T = a.tin_c[t];
    int32_t bnd[12]; float scale[3];
    sah_load_bnd(T, bnd, scale);
    SahSplit s; s.axis = T.axis; s.plane = T.plane; s.nl = T.nl;
    for (int p = p0 + threadIdx.x; p < p1; p += kSahBlock) {
        const int g = a.idx[p];
        a.flags[p] = sah_goes_left(s, p - T.r.begin, a.prim_lo[g], a.prim_hi[g], bnd) ? 1 : 0;
    }
}
__global__ void __launch_bounds__(kSahBlock) k_sah_scatter(SahArgs a) {
    int t, p0, p1;
    if (!sah_block_range(a, t, p0, p1)) return;
    const SahTask &T = a.tin_c[t];
    const int b = T.r.begin, nl = T.nl, base = a.scan[b];
    for (int p = p0 + threadIdx.x; p < p1; p += kSahBlock) {
        const int before = a.scan[p] - base;  // left-goers in [b, p)
        a.idx2[a.flags[p] ? b + before : b + nl + (p - b - before)] = a.idx[p];
    }
}
__global__ void __launch_bounds__(kSahBlock) k_sah_copy(SahArgs a) {
    int t, p0, p1;
    if (!sah_block_range(a, t, p0, p1)) return;
    for (int p = p0 + threadIdx.x; p < p1; p += kSahBlock) a.idx[p] = a.idx2[p];
}
// The ranges of <= kSahSmall primitives, one block each: boxes and positions in shared memory, the subtree level by
// level inside the block, one warp per range of a level (the rule of the large levels: same bounds, bins, choice and
// stable partition).  Inner ids: one atomic per block for the whole subtree.
constexpr int kSahSmallWarps = 8;
struct SahSmallSmem {
    float box[6][kSahSmall];  // lo xyz, hi xyz of local primitive slot
    int32_t gidx[kSahSmall], slot[kSahSmall], scratch[kSahSmall];  // slot at each position of the range, partition buffer
    SahRange list[2][kSahSmall / 2];
    int32_t bins[kSahSmallWarps][kSahBinsWords];
    int32_t n_cur, n_next, ids;
};
__device__ __forceinline__ void sah_small_box(const SahSmallSmem &S, int sl, F4 &lo, F4 &hi) {
    lo.x = S.box[0][sl]; lo.y = S.box[1][sl]; lo.z = S.box[2][sl]; lo.w = 0.f;
    hi.x = S.box[3][sl]; hi.y = S.box[4][sl]; hi.z = S.box[5][sl]; hi.w = 0.f;
}
__device__ void sah_small_range(const SahArgs &a, SahSmallSmem &S, const SahRange r, int B, int lane, int warp, int nxt) {
    const int b = r.begin - B, e = r.end - B;
    int32_t bnd[12];
    sah_bnd_init(bnd);
    for (int j = b + lane; j < e; j += 32) { F4 lo, hi; sah_small_box(S, S.slot[j], lo, hi); sah_bnd_add(bnd, lo, hi); }
    __syncwarp();
#pragma unroll
    for (int k = 0; k < 12; ++k) bnd[k] = (k % 6) < 3 ? __reduce_min_sync(0xffffffffu, bnd[k]) : __reduce_max_sync(0xffffffffu, bnd[k]);
    float scale[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) scale[k] = sah_scale(bnd, k);
    int32_t *bins = S.bins[warp];
    for (int k = lane; k < 3 * kSahBins; k += 32) sah_bin_init(bins + k * kSahBinWords);
    __syncwarp();
    if (scale[0] > 0.f || scale[1] > 0.f || scale[2] > 0.f)
        for (int j = b + lane; j < e; j += 32) { F4 lo, hi; sah_small_box(S, S.slot[j], lo, hi); sah_bin_add(bins, lo, hi, bnd, scale); }
    __syncwarp();
    const SahSplit s = sah_choose_warp(bins, scale, e - b, lane);
    int nl_seen = 0, nr_seen = 0;
    const unsigned below = (1u << lane) - 1u;
    for (int base = b; base < e; base += 32) {  // (warp-uniform)
        const int j = base + lane;
        const bool in = j < e;
        const int sl = in ? S.slot[j] : 0;
        F4 lo, hi;
        sah_small_box(S, sl, lo, hi);
        const bool f = in && sah_goes_left(s, j - b, lo, hi, bnd);
        const unsigned lm = __ballot_sync(0xffffffffu, f), rm = __ballot_sync(0xffffffffu, in && !f);
        if (f) S.scratch[b + nl_seen + __popc(lm & below)] = sl;
        else if (in) S.scratch[b + s.nl + nr_seen + __popc(rm & below)] = sl;
        nl_seen += __popc(lm); nr_seen += __popc(rm);
    }
    __syncwarp();
    for (int j = b + lane; j < e; j += 32) S.slot[j] = S.scratch[j];
    __syncwarp();
    if (lane == 0) {
        SahRange ch[2];
        sah_make_node(a, r, bnd, s.nl, &S.ids, ch);
        for (int k = 0; k < 2; ++k)
            if (ch[k].end - ch[k].begin > 1) S.list[nxt][atomicAdd(&S.n_next, 1)] = ch[k];
    }
    __syncwarp();
}
__global__ void __launch_bounds__(kSahSmallWarps * 32) k_sah_small(SahArgs a) {
    extern __shared__ __align__(16) unsigned char sah_smem[];
    SahSmallSmem &S = *reinterpret_cast<SahSmallSmem *>(sah_smem);
    const SahRange R = a.small[blockIdx.x];
    const int B = R.begin, size = R.end - R.begin, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    for (int i = tid; i < size; i += kSahSmallWarps * 32) {
        const int g = a.idx[B + i];
        const F4 lo = a.prim_lo[g], hi = a.prim_hi[g];
        S.gidx[i] = g; S.slot[i] = i;
        S.box[0][i] = lo.x; S.box[1][i] = lo.y; S.box[2][i] = lo.z; S.box[3][i] = hi.x; S.box[4][i] = hi.y; S.box[5][i] = hi.z;
    }
    if (tid == 0) {
        S.list[0][0] = R; S.n_cur = 1;
        S.ids = atomicAdd(a.node_counter, size - 2);  // ids of the subtree's size - 1 inner nodes but its root (R.id)
    }
    __syncthreads();
    int cur = 0;
    while (true) {  // one level of the subtree per pass; each pass splits every range in two, so sizes fall
        const int m = S.n_cur;
        if (m == 0) break;
        if (tid == 0) S.n_next = 0;
        __syncthreads();
        for (int i = warp; i < m; i += kSahSmallWarps) sah_small_range(a, S, S.list[cur][i], B, lane, warp, cur ^ 1);
        __syncthreads();
        if (tid == 0) S.n_cur = S.n_next;
        cur ^= 1;
        __syncthreads();
    }
    for (int i = tid; i < size; i += kSahSmallWarps * 32) a.idx[B + i] = S.gidx[S.slot[i]];
}

// ---- treelet restructuring (RTB_BUILDER_TREELET_PASSES, rtb_build.h 3.5) ----
// One warp per treelet root of one depth: lane 0 forms the treelet and rewires it, the 32 lanes share the (<= 127)
// subsets of the dynamic programme; the treelet's tables live in shared memory.
constexpr int kTloWarps = 4;
__global__ void __launch_bounds__(kTloWarps * 32) k_tlo_treelet(TloArgs a) {
    __shared__ TloWork W[kTloWarps];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int i = blockIdx.x * kTloWarps + warp;
    if (i >= a.num) return;  // (a whole warp)
    tlo_treelet(a, W[warp], i, lane, 32);
}

// ---- refit (rtb_scene_refit, rtb_build.h 6) ----
// The nodes of one depth, one thread each.  Every lane of a block exists (the grid is rounded up, out-of-range lanes
// contribute 0), so the SAH terms are summed over the full warp mask and one lane per warp adds them to the total.
__global__ void __launch_bounds__(kBlock) k_refit_level(RefitArgs a) {
    const int i = blockIdx.x * kBlock + threadIdx.x;
    float v = i < a.num ? refit_body(a, i) : 0.f;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if ((threadIdx.x & 31) == 0 && v != 0.f) atomicAdd(a.sah, v);
}

// NCCL, loaded on first use.  A process that already holds a libnccl.so.2 (torch brings its own) gets that one.
struct Nccl {
    void *lib = nullptr;
    decltype(&ncclGetUniqueId) GetUniqueId = nullptr;
    decltype(&ncclCommInitRank) CommInitRank = nullptr;
    decltype(&ncclCommInitAll) CommInitAll = nullptr;
    decltype(&ncclCommDestroy) CommDestroy = nullptr;
    decltype(&ncclAllReduce) AllReduce = nullptr;
    decltype(&ncclReduce) Reduce = nullptr;
    decltype(&ncclGroupStart) GroupStart = nullptr;
    decltype(&ncclGroupEnd) GroupEnd = nullptr;
    decltype(&ncclGetErrorString) GetErrorString = nullptr;
    static Nccl &get() {
        static Nccl n;
        static std::once_flag once;
        std::call_once(once, [] {
            for (const char *name : {"libnccl.so.2", "libnccl.so"}) {
                n.lib = dlopen(name, RTLD_NOW | RTLD_GLOBAL);
                if (n.lib) break;
            }
            if (!n.lib) return;
#define RTB_NCCL_SYM(f) n.f = (decltype(n.f))dlsym(n.lib, "nccl" #f)
            RTB_NCCL_SYM(GetUniqueId); RTB_NCCL_SYM(CommInitRank); RTB_NCCL_SYM(CommInitAll); RTB_NCCL_SYM(CommDestroy);
            RTB_NCCL_SYM(AllReduce); RTB_NCCL_SYM(Reduce); RTB_NCCL_SYM(GroupStart); RTB_NCCL_SYM(GroupEnd); RTB_NCCL_SYM(GetErrorString);
#undef RTB_NCCL_SYM
        });
        if (!n.lib || !n.GetUniqueId || !n.CommInitRank || !n.CommInitAll || !n.CommDestroy || !n.AllReduce || !n.Reduce || !n.GroupStart ||
            !n.GroupEnd || !n.GetErrorString)
            throw Error(RTB_ERR_NO_DEVICE, "NCCL (libnccl.so.2) could not be loaded: multi-GPU entry points need it");
        return n;
    }
};
#define RTB_NCCL_CHECK(expr)                                                                                               \
    do {                                                                                                                   \
        ncclResult_t r_ = (expr);                                                                                          \
        if (r_ != ncclSuccess) throw rtb::Error(RTB_ERR_CUDA, std::string(#expr) + ": " + rtb::Nccl::get().GetErrorString(r_)); \
    } while (0)
static_assert(sizeof(ncclUniqueId) == RTB_COMM_ID_BYTES, "rtb.h: RTB_COMM_ID_BYTES must be sizeof(ncclUniqueId)");

struct NonNegative {
    __host__ __device__ bool operator()(const int32_t &v) const { return v >= 0; }
};

struct CudaBackend {
    int dev_ = -1;
    int num_sms_ = 0;
    cudaStream_t stream_ = nullptr;  // the stream launches go to: streams_[0] unless use_stream(k) says otherwise
    cudaStream_t streams_[kMaxPipelines] = {nullptr, nullptr};
    cudaEvent_t sync_ev_ = nullptr;
    cudaMemPool_t pool_mem_ = nullptr;
    int pipelines_ = 0;  // RTB_PIPELINES: concurrent wavefronts per render (1..4); 0 = by scene size, see pipelines()
    int blocks_trace_ = 0, blocks_generate_ = 0;
    int trace_blocks_per_sm_ = 1, trace_cap_ = 0, active_pipelines_ = 1;
    void *cub_temp_ = nullptr;
    size_t cub_temp_bytes_ = 0;
    int32_t *h_done_ = nullptr, *d_done_ = nullptr;  // mapped pinned word raised by k_control
    FetchTuning tune_{24, 128, 1, 2};  // RTB_REFILL / RTB_CHUNK / RTB_PREFETCH override (tuning runs)
    int pooled_ = 0;  // RTB_POOLED: pooled triangle tests (1), each ray's lane on its own (0, default), by scene size (-1)
    int fused_ = 1;   // "fused": extend + shadow rays of one iteration in one launch
    int smem_stack_ = 0;  // "smem_stack": first stack entries in shared memory (A/B, k_trace_smem_stack)
    WaveCache wave_cache_;  // queues of the last destroyed scene (rtb_engine.h)
    WaveCache &wave_cache() { return wave_cache_; }
    int pool_ = 0;          // "pool": path slots of a render; 0 = automatic (default_pool)
    size_t pool_budget_ = 0;  // an eighth of the device memory that was free when the context was created
    int ploc_tail_off_ = 0; // RTB_PLOC_TAIL=0: every PLOC round its own launches (A/B)
    int nn_tiled_off_ = 0;  // "nn_tiled" = 0: nearest-neighbour search of a PLOC round one thread per cluster from global memory (A/B)

    explicit CudaBackend(int device) {
        int count = 0;
        cudaError_t e = cudaGetDeviceCount(&count);
        if (e != cudaSuccess || count == 0)
            throw Error(RTB_ERR_NO_DEVICE, std::string("no CUDA device available (") + cudaGetErrorString(e) +
                                               "); rtcuda_b200 has no CPU fallback");
        if (device < 0 || device >= count) throw Error(RTB_ERR_INVALID, "device ordinal out of range");
        cudaDeviceProp prop;
        RTB_CUDA_CHECK(cudaGetDeviceProperties(&prop, device));
        if (prop.major != 10)
            throw Error(RTB_ERR_NO_DEVICE, std::string("device '") + prop.name + "' is sm_" + std::to_string(prop.major) +
                                               std::to_string(prop.minor) + "; this library is built for sm_100a (B200) only");
        dev_ = device;
        num_sms_ = prop.multiProcessorCount;
        RTB_CUDA_CHECK(cudaSetDevice(dev_));
        for (int k = 0; k < kMaxPipelines; ++k) RTB_CUDA_CHECK(cudaStreamCreateWithFlags(&streams_[k], cudaStreamDefault));
        stream_ = streams_[0];
        RTB_CUDA_CHECK(cudaEventCreateWithFlags(&sync_ev_, cudaEventDisableTiming));
        // stream-ordered allocator that keeps freed blocks: scene builds and renders reuse memory instead of paying
        // cudaMalloc / cudaFree (each an implicit device synchronisation) every call.  The pool is this context's own
        // (the device's default pool is process-wide state that a host framework may also use); it is destroyed with
        // the context, which returns every byte to the driver.
        cudaMemPoolProps props = {};
        props.allocType = cudaMemAllocationTypePinned;
        props.handleTypes = cudaMemHandleTypeNone;
        props.location.type = cudaMemLocationTypeDevice;
        props.location.id = dev_;
        RTB_CUDA_CHECK(cudaMemPoolCreate(&pool_mem_, &props));
        unsigned long long keep = ~0ull;
        RTB_CUDA_CHECK(cudaMemPoolSetAttribute(pool_mem_, cudaMemPoolAttrReleaseThreshold, &keep));
        {
            size_t free_b = 0, total_b = 0;
            RTB_CUDA_CHECK(cudaMemGetInfo(&free_b, &total_b));
            pool_budget_ = free_b / 8;
        }
        RTB_CUDA_CHECK(cudaHostAlloc((void **)&h_done_, kMaxPipelines * sizeof(int32_t), cudaHostAllocMapped));
        RTB_CUDA_CHECK(cudaHostGetDevicePointer((void **)&d_done_, h_done_, 0));
        for (int k = 0; k < kMaxPipelines; ++k) h_done_[k] = 0;
        int per_sm = 0;
        RTB_CUDA_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_trace<3, true>, kTraceBlock, 0));
        trace_blocks_per_sm_ = per_sm > 0 ? per_sm : 1;
        // tuning runs (tools/sweep.py) may preset the options of rtb_context_set_option through the environment:
        // RTB_<NAME IN CAPITALS>=value, read once here; the ABI call is the documented way
        static const char *const names[] = {"refill", "chunk", "prefetch", "tri_step", "pooled", "fused", "smem_stack", "pipelines", "pool",
                                            "ploc_tail", "trace_blocks", "nn_tiled"};
        for (const char *nm : names) {
            std::string env = "RTB_";
            for (const char *c = nm; *c; ++c) env += (char)toupper((unsigned char)*c);
            if (const char *e = getenv(env.c_str())) set_option(nm, atoll(e));
        }
        blocks_trace_ = num_sms_ * trace_blocks_per_sm_;
        RTB_CUDA_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_generate, kBlock, 0));
        blocks_generate_ = num_sms_ * (per_sm > 0 ? per_sm : 1);
    }
    ~CudaBackend() {
        if (dev_ < 0) return;
        cudaSetDevice(dev_);
        stream_ = streams_[0];
        for (int k = 0; k < kMaxPipelines; ++k) if (streams_[k]) cudaStreamSynchronize(streams_[k]);
        wave_cache_release(*this, wave_cache_);
        if (cub_temp_) cudaFreeAsync(cub_temp_, stream_);
        if (tail_counts_) cudaFreeAsync(tail_counts_, stream_);
        if (h_done_) cudaFreeHost(h_done_);
        if (sync_ev_) cudaEventDestroy(sync_ev_);
        for (int k = 0; k < kMaxPipelines; ++k) if (streams_[k]) { cudaStreamSynchronize(streams_[k]); cudaStreamDestroy(streams_[k]); }
        if (pool_mem_) cudaMemPoolDestroy(pool_mem_);
    }
    CudaBackend(const CudaBackend &) = delete;
    CudaBackend &operator=(const CudaBackend &) = delete;

    // rtb_context_set_option / rtb_context_get_option (include/rtb.h lists the names)
    bool set_option(const std::string &name, long long v) {
        auto in = [&](long long lo, long long hi) { return v >= lo && v <= hi; };
        if (name == "refill") { if (!in(1, 32)) return false; tune_.refill = (int)v; }
        else if (name == "chunk") { if (!in(32, 1 << 20)) return false; tune_.chunk = (int)v; }
        else if (name == "prefetch") { if (!in(0, 1)) return false; tune_.prefetch = (int)v; }
        else if (name == "tri_step") { if (!in(0, 4)) return false; tune_.tri_step = (int)v; }
        else if (name == "pooled") { if (!in(-1, 1)) return false; pooled_ = (int)v; }
        else if (name == "fused") { if (!in(0, 1)) return false; fused_ = (int)v; }
        else if (name == "smem_stack") { if (!in(0, 1)) return false; smem_stack_ = (int)v; }
        else if (name == "pipelines") { if (!in(0, kMaxPipelines)) return false; pipelines_ = (int)v; }
        else if (name == "pool") { if (v != 0 && !in(1024, 1ll << 30)) return false; pool_ = (int)v; }
        else if (name == "ploc_tail") { if (!in(0, 1)) return false; ploc_tail_off_ = v == 0; }
        else if (name == "trace_blocks") { if (!in(0, trace_blocks_per_sm_)) return false; trace_cap_ = (int)v; }
        else if (name == "nn_tiled") { if (!in(0, 1)) return false; nn_tiled_off_ = v == 0; }
        else return false;
        return true;
    }
    bool get_option(const std::string &name, long long &v) const {
        if (name == "refill") v = tune_.refill;
        else if (name == "chunk") v = tune_.chunk;
        else if (name == "prefetch") v = tune_.prefetch;
        else if (name == "tri_step") v = tune_.tri_step;
        else if (name == "pooled") v = pooled_;
        else if (name == "fused") v = fused_;
        else if (name == "smem_stack") v = smem_stack_;
        else if (name == "pipelines") v = pipelines_;
        else if (name == "pool") v = pool_;
        else if (name == "ploc_tail") v = ploc_tail_off_ ? 0 : 1;
        else if (name == "trace_blocks") v = trace_cap_;
        else if (name == "nn_tiled") v = nn_tiled_off_ ? 0 : 1;
        else return false;
        return true;
    }
    int device() const { return dev_; }
    void make_current() { RTB_CUDA_CHECK(cudaSetDevice(dev_)); }
    void sync() { RTB_CUDA_CHECK(cudaStreamSynchronize(stream_)); }
    // Path slots of a render that does not name a pool.  Fewer, larger iterations win (C2, four wavefronts: 34.5 ms at
    // 32 Mi slots, 34.3 at 64 Mi, 33.7 with all 132.7 M paths in flight; C4 27.6 / 27.2 / 26.4 ms: profiles/README.md,
    // session 45), and a B200 has 180 GB: as many slots as fit an eighth of what was free when the context was created,
    // at least 4 Mi; render_accumulate caps it at the paths of the render.
    long long default_pool(size_t slot_bytes) const {
        if (pool_ > 0) return pool_;
        long long n = (long long)(pool_budget_ / (slot_bytes ? slot_bytes : 144));
        if (n < (1ll << 22)) n = 1ll << 22;
        if (n > (1ll << 28)) n = 1ll << 28;
        return n;
    }

    template <class T> T *alloc(size_t n) {
        void *p = nullptr;
        RTB_CUDA_CHECK(cudaMallocFromPoolAsync(&p, sizeof(T) * (n ? n : 1), pool_mem_, stream_));
        return (T *)p;
    }
    void free(void *p) { if (p) cudaFreeAsync(p, stream_); }
    template <class T> void upload(T *dst, const T *src, size_t n) {
        RTB_CUDA_CHECK(cudaMemcpyAsync(dst, src, sizeof(T) * n, cudaMemcpyHostToDevice, stream_));
        RTB_CUDA_CHECK(cudaStreamSynchronize(stream_));  // src may be a temporary
    }
    template <class T> void download(T *dst, const T *src, size_t n) {
        RTB_CUDA_CHECK(cudaMemcpyAsync(dst, src, sizeof(T) * n, cudaMemcpyDeviceToHost, stream_));
        RTB_CUDA_CHECK(cudaStreamSynchronize(stream_));
    }
    template <class T> void copy(T *dst, const T *src, size_t n) {
        RTB_CUDA_CHECK(cudaMemcpyAsync(dst, src, sizeof(T) * n, cudaMemcpyDeviceToDevice, stream_));
    }
    template <class T> void zero(T *p, size_t n) { RTB_CUDA_CHECK(cudaMemsetAsync(p, 0, sizeof(T) * n, stream_)); }
    // device memory of another context's GPU -> this one's (NVLink peer copy when the driver can, staged otherwise)
    template <class T> void copy_from(CudaBackend &src_be, T *dst, const T *src, size_t n) {
        if (!n) return;
        if (src_be.dev_ == dev_) { copy(dst, src, n); return; }
        RTB_CUDA_CHECK(cudaMemcpyPeerAsync(dst, dev_, src, src_be.dev_, sizeof(T) * n, stream_));
    }
    // ---- collectives over the GPUs of one process (rtb_multi) and over processes (rtb_comm) ----
    struct Group { std::vector<ncclComm_t> comms; };
    static Group *group_create(const std::vector<CudaBackend *> &members) {
        Nccl &nc = Nccl::get();
        std::vector<int> devs;
        for (CudaBackend *b : members) devs.push_back(b->dev_);
        Group *g = new Group();
        g->comms.resize(members.size());
        ncclResult_t r = nc.CommInitAll(g->comms.data(), (int)devs.size(), devs.data());
        if (r != ncclSuccess) { delete g; throw Error(RTB_ERR_CUDA, std::string("ncclCommInitAll: ") + nc.GetErrorString(r)); }
        return g;
    }
    static void group_destroy(Group *g) {
        if (!g) return;
        for (ncclComm_t c : g->comms) if (c) Nccl::get().CommDestroy(c);
        delete g;
    }
    // sum of every member's buffer into the root's, in place; enqueued on each member's stream, one NCCL group
    template <class T>
    static void group_reduce(Group *g, const std::vector<CudaBackend *> &members, const std::vector<T *> &bufs, size_t n, int root) {
        Nccl &nc = Nccl::get();
        const ncclDataType_t dt = sizeof(T) == 8 ? ncclInt64 : ncclFloat32;
        RTB_NCCL_CHECK(nc.GroupStart());
        for (size_t r = 0; r < members.size(); ++r) {
            ncclResult_t e = nc.Reduce(bufs[r], bufs[r], n, dt, ncclSum, root, g->comms[r], members[r]->streams_[0]);
            if (e != ncclSuccess) { nc.GroupEnd(); throw Error(RTB_ERR_CUDA, std::string("ncclReduce: ") + nc.GetErrorString(e)); }
        }
        RTB_NCCL_CHECK(nc.GroupEnd());
    }
    struct Comm { ncclComm_t comm = nullptr; int rank = 0, world = 1; };
    static void comm_unique_id(uint8_t *out) {
        ncclUniqueId id;
        RTB_NCCL_CHECK(Nccl::get().GetUniqueId(&id));
        memcpy(out, &id, sizeof id);
    }
    Comm *comm_create(const uint8_t *id_bytes, int rank, int world) {
        ncclUniqueId id;
        memcpy(&id, id_bytes, sizeof id);
        make_current();
        Comm *c = new Comm();
        c->rank = rank; c->world = world;
        ncclResult_t r = Nccl::get().CommInitRank(&c->comm, world, id, rank);
        if (r != ncclSuccess) { delete c; throw Error(RTB_ERR_CUDA, std::string("ncclCommInitRank: ") + Nccl::get().GetErrorString(r)); }
        return c;
    }
    static void comm_destroy(Comm *c) {
        if (!c) return;
        if (c->comm) Nccl::get().CommDestroy(c->comm);
        delete c;
    }
    template <class T> void comm_allreduce(Comm *c, T *buf, size_t n) {
        const ncclDataType_t dt = sizeof(T) == 8 ? ncclInt64 : ncclFloat32;
        RTB_NCCL_CHECK(Nccl::get().AllReduce(buf, buf, n, dt, ncclSum, c->comm, streams_[0]));
        RTB_CUDA_CHECK(cudaStreamSynchronize(streams_[0]));
    }

    template <class F> void launch(int n, F f) {
        if (n <= 0) return;
        k_for<F><<<(n + kBlock - 1) / kBlock, kBlock, 0, stream_>>>(n, f);
        RTB_CUDA_CHECK(cudaGetLastError());
    }
    template <class F> void launch_trace(int n, F f) { launch(n, f); }
    void generate(const GenerateK &k) {
        k_generate<<<blocks_generate_, kBlock, 0, stream_>>>(k.W, k.rc);
        RTB_CUDA_CHECK(cudaGetLastError());
    }
    void shade(const ShadeK &k) {
        const int grid = num_sms_ * shade_blocks_per_sm(k.type);  // one resident wave: the kernels are grid-stride loops
        if ((k.rc.flags & (RTB_RENDER_TRUE_MIS | RTB_RENDER_RR_TERMINATE)) || k.S.bvh.inst) {  // beyond-the-reference estimator, instanced scenes
            if (k.type == 0) k_shade<0, true><<<grid, kShadeBlock, 0, stream_>>>(k.W, k.S, k.rc, k.shadows);
            else if (k.type == 1) k_shade<1, true><<<grid, kShadeBlock, 0, stream_>>>(k.W, k.S, k.rc, k.shadows);
            else if (k.type == 2) k_shade<2, true><<<grid, kShadeBlock, 0, stream_>>>(k.W, k.S, k.rc, k.shadows);
            else k_shade<3, true><<<grid, kShadeBlock, 0, stream_>>>(k.W, k.S, k.rc, k.shadows);
        } else {
            if (k.type == 0) k_shade<0><<<grid, kShadeBlock, 0, stream_>>>(k.W, k.S, k.rc, k.shadows);
            else if (k.type == 1) k_shade<1><<<grid, kShadeBlock, 0, stream_>>>(k.W, k.S, k.rc, k.shadows);
            else if (k.type == 2) k_shade<2><<<grid, kShadeBlock, 0, stream_>>>(k.W, k.S, k.rc, k.shadows);
            else k_shade<3><<<grid, kShadeBlock, 0, stream_>>>(k.W, k.S, k.rc, k.shadows);
        }
        RTB_CUDA_CHECK(cudaGetLastError());
    }
    void control(const WaveState &W, bool shadows) {
        k_control<<<1, 1, 0, stream_>>>(W, shadows);
        RTB_CUDA_CHECK(cudaGetLastError());
    }
    // Grid of a persistent trace launch.  Two wavefronts: half the resident blocks each (see kTraceBlock) — unless the
    // scene is far beyond L2: there the kernel waits on DRAM latency, wants every warp it can get, and the half-size
    // launches were measured 1 % slower (C3 99.4 -> 100.3 ms).
    void begin_render(int pipelines) { active_pipelines_ = pipelines; }
    int trace_grid(const SceneView &S) const {
        int per = trace_blocks_per_sm_;
        if (trace_cap_ > 0) per = trace_cap_;
        else if (active_pipelines_ > 1 && !big_scene(S)) per = per / active_pipelines_ > 0 ? per / active_pipelines_ : 1;
        return num_sms_ * per;
    }
    // mode 0: persistent, 1: one thread per ray, 2: one thread per ray + work counters
    bool big_scene(const SceneView &S) const {  // nodes + triangles beyond what stays resident in the 126 MB L2
        return (size_t)S.bvh.num_nodes * 80 + (size_t)S.bvh.num_tris * 48 > ((size_t)48 << 20);
    }
    bool use_pooled(const SceneView &S) const { return pooled_ < 0 ? big_scene(S) : pooled_ != 0; }
    void extend(const WaveState &W, const SceneView &S, int mode) {
        const int flat_grid = (W.pool + kBlock - 1) / kBlock;
        if (mode == 2) k_extend_flat<true><<<flat_grid, kBlock, 0, stream_>>>(W, S);
        else if (mode == 1) k_extend_flat<false><<<flat_grid, kBlock, 0, stream_>>>(W, S);
        else launch_trace_kernel<1>(trace_grid(S), stream_, use_pooled(S), smem_stack_ != 0, W, S, tune_);
        RTB_CUDA_CHECK(cudaGetLastError());
    }
    void shadow(const WaveState &W, const SceneView &S, int mode) {
        const int flat_grid = (W.pool + kBlock - 1) / kBlock;
        if (mode == 2) k_shadow_flat<true><<<flat_grid, kBlock, 0, stream_>>>(W, S);
        else if (mode == 1) k_shadow_flat<false><<<flat_grid, kBlock, 0, stream_>>>(W, S);
        else launch_trace_kernel<2>(trace_grid(S), stream_, use_pooled(S), smem_stack_ != 0, W, S, tune_);
        RTB_CUDA_CHECK(cudaGetLastError());
    }
    // both ray types in one launch; false = not available in this mode
    bool trace_fused(const WaveState &W, const SceneView &S, int mode) {
        if (mode != 0 || !fused_) return false;
        launch_trace_kernel<3>(trace_grid(S), stream_, use_pooled(S), smem_stack_ != 0, W, S, tune_);
        RTB_CUDA_CHECK(cudaGetLastError());
        return true;
    }
    // ---- concurrent wavefronts (rtb_engine.h, render_accumulate) ----
    // Four wavefronts, each trace kernel a quarter of the SM, while nodes + triangles stay in L2 (C4 29.0 -> 27.5 ms,
    // C2 35.2 -> 34.9 ms against two); two full-size ones on a scene far beyond it (C3 98.7 ms against 101.6 with four).
    int pipelines(const SceneView &S) const { return pipelines_ > 0 ? pipelines_ : (big_scene(S) ? 2 : 4); }
    void use_stream(int k) { stream_ = streams_[k]; }
    void fork(int k) {  // stream k continues after what is queued on the main stream
        RTB_CUDA_CHECK(cudaEventRecord(sync_ev_, streams_[0]));
        RTB_CUDA_CHECK(cudaStreamWaitEvent(streams_[k], sync_ev_, 0));
    }
    void join(int k) {  // the main stream continues after what is queued on stream k
        RTB_CUDA_CHECK(cudaEventRecord(sync_ev_, streams_[k]));
        RTB_CUDA_CHECK(cudaStreamWaitEvent(streams_[0], sync_ev_, 0));
    }
    int32_t *done_flag_device(int k) { return d_done_ + k; }
    void reset_done(int k) { ((volatile int32_t *)h_done_)[k] = 0; }
    bool done(int k) const { return ((volatile int32_t *)h_done_)[k] != 0; }
    void wait(cudaEvent_t e) { RTB_CUDA_CHECK(cudaEventSynchronize(e)); }

    void ensure_temp(size_t bytes) {
        if (bytes <= cub_temp_bytes_) return;
        if (cub_temp_) cudaFreeAsync(cub_temp_, stream_);
        cub_temp_ = nullptr; cub_temp_bytes_ = 0;
        RTB_CUDA_CHECK(cudaMallocFromPoolAsync(&cub_temp_, bytes, pool_mem_, stream_));
        cub_temp_bytes_ = bytes;
    }
    void sort_pairs(uint64_t *keys, int32_t *vals, int n) {
        uint64_t *k2 = alloc<uint64_t>(n);
        int32_t *v2 = alloc<int32_t>(n);
        cub::DoubleBuffer<uint64_t> dk(keys, k2);
        cub::DoubleBuffer<int32_t> dv(vals, v2);
        size_t bytes = 0;
        RTB_CUDA_CHECK(cub::DeviceRadixSort::SortPairs(nullptr, bytes, dk, dv, n, 0, 63, stream_));
        ensure_temp(bytes);
        RTB_CUDA_CHECK(cub::DeviceRadixSort::SortPairs(cub_temp_, bytes, dk, dv, n, 0, 63, stream_));
        if (dk.Current() != keys) copy(keys, dk.Current(), n);
        if (dv.Current() != vals) copy(vals, dv.Current(), n);
        free(k2); free(v2);  // (stream-ordered: released when the copies above have run)
    }
    void prim_setup(const PrimSetupArgs &a) {
        if (a.n <= 0) return;
        if (!a.vertices) { PrimSetupK k; k.a = a; launch(a.n, k); return; }  // records already filled (reference-pointer ingest)
        k_prim_setup_tiled<<<(a.n + kSetupBlock - 1) / kSetupBlock, kSetupBlock, 0, stream_>>>(a);
        RTB_CUDA_CHECK(cudaGetLastError());
    }
    void ploc_nn(const PlocArgs &a) {
        if (a.ncl <= 0) return;
        if (a.radius > kNnMaxRadius || nn_tiled_off_) { PlocNnK k; k.a = a; launch(a.ncl, k); return; }
        k_ploc_nn_tiled<<<(a.ncl + kNnBlock - 1) / kNnBlock, kNnBlock, 0, stream_>>>(a);
        RTB_CUDA_CHECK(cudaGetLastError());
    }
    // all remaining rounds in one launch once the host's bound of the cluster count fits a thread block; out[0] = rounds
    // (-1: a round merged nothing), out[1] = root, ploc_tail_counts()[r] = nodes made by round r — all left on the device
    int32_t *tail_counts_ = nullptr;
    int32_t *ploc_tail_counts() {
        if (!tail_counts_) tail_counts_ = alloc<int32_t>(kPlocTail);
        return tail_counts_;
    }
    bool ploc_tail(const PlocArgs &a, int n_leaves, int32_t *d_out) {
        if (a.ncl > kPlocTail || ploc_tail_off_) return false;
        k_ploc_tail<<<1, kPlocTail, 0, stream_>>>(a, n_leaves, d_out, ploc_tail_counts());
        RTB_CUDA_CHECK(cudaGetLastError());
        return true;
    }
    // order-preserving compaction of the entries >= 0 of in[0, n) into out; their number goes to *d_count (device memory)
    void compact_nonneg(const int32_t *in, int32_t *out, int n, int32_t *d_count) {
        size_t bytes = 0;
        RTB_CUDA_CHECK(cub::DeviceSelect::If(nullptr, bytes, in, out, d_count, n, NonNegative(), stream_));
        ensure_temp(bytes);
        RTB_CUDA_CHECK(cub::DeviceSelect::If(cub_temp_, bytes, in, out, d_count, n, NonNegative(), stream_));
    }
    // binned SAH: one level of large ranges (counts in device memory; grids cover the bounds) / all small ranges
    void sah_level(const SahArgs &a, int block_bound, int task_bound) {
        k_sah_bounds<<<block_bound, kSahBlock, 0, stream_>>>(a);
        k_sah_bin<<<block_bound, kSahBlock, 0, stream_>>>(a);
        k_sah_split<<<(task_bound * 32 + kSahBlock - 1) / kSahBlock, kSahBlock, 0, stream_>>>(a);
        k_sah_flag<<<block_bound, kSahBlock, 0, stream_>>>(a);
        RTB_CUDA_CHECK(cudaGetLastError());
        size_t bytes = 0;
        RTB_CUDA_CHECK(cub::DeviceScan::ExclusiveSum(nullptr, bytes, a.flags, a.scan, a.n, stream_));
        ensure_temp(bytes);
        RTB_CUDA_CHECK(cub::DeviceScan::ExclusiveSum(cub_temp_, bytes, a.flags, a.scan, a.n, stream_));
        k_sah_scatter<<<block_bound, kSahBlock, 0, stream_>>>(a);
        k_sah_copy<<<block_bound, kSahBlock, 0, stream_>>>(a);
        RTB_CUDA_CHECK(cudaGetLastError());
    }
    void sah_small(const SahArgs &a, int count) {
        if (count <= 0) return;
        RTB_CUDA_CHECK(cudaFuncSetAttribute(k_sah_small, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(SahSmallSmem)));
        k_sah_small<<<count, kSahSmallWarps * 32, sizeof(SahSmallSmem), stream_>>>(a);
        RTB_CUDA_CHECK(cudaGetLastError());
    }
    // treelet restructuring: the treelets of one depth (a.num roots)
    void tlo_treelets(const TloArgs &a) {
        if (a.num <= 0) return;
        k_tlo_treelet<<<(a.num + kTloWarps - 1) / kTloWarps, kTloWarps * 32, 0, stream_>>>(a);
        RTB_CUDA_CHECK(cudaGetLastError());
    }
    // one level of the collapse over the work items counted in device memory (k.a.n_in_dev): a resident grid strides
    // over them; *zero is cleared for the level after the next, *levels counts the levels that had work
    void collapse_level(const CollapseK &k, int bound, int32_t *zero, int32_t *levels) {
        int grid = (bound + kBlock - 1) / kBlock;
        if (grid > num_sms_ * 8) grid = num_sms_ * 8;
        k_collapse_level<<<grid, kBlock, 0, stream_>>>(k.a, zero, levels);
        RTB_CUDA_CHECK(cudaGetLastError());
    }

    // refit: the nodes of one depth (a.num of them)
    void refit_level(const RefitArgs &a) {
        if (a.num <= 0) return;
        k_refit_level<<<(a.num + kBlock - 1) / kBlock, kBlock, 0, stream_>>>(a);
        RTB_CUDA_CHECK(cudaGetLastError());
    }

    using Time = cudaEvent_t;
    Time now() {
        cudaEvent_t e;
        RTB_CUDA_CHECK(cudaEventCreate(&e));
        RTB_CUDA_CHECK(cudaEventRecord(e, stream_));
        return e;
    }
    float elapsed_keep(Time a, Time b) {  // both events already completed or on the same stream
        float ms = 0.f;
        RTB_CUDA_CHECK(cudaEventSynchronize(b));
        RTB_CUDA_CHECK(cudaEventElapsedTime(&ms, a, b));
        return ms;
    }
    void release(Time e) { cudaEventDestroy(e); }
    float elapsed_ms(Time a, Time b) {
        float ms = 0.f;
        RTB_CUDA_CHECK(cudaEventSynchronize(b));
        RTB_CUDA_CHECK(cudaEventElapsedTime(&ms, a, b));
        cudaEventDestroy(a);
        cudaEventDestroy(b);
        return ms;
    }
};

static_assert(HasSahKernels<CudaBackend>::value, "the binned-SAH builder runs as k_sah_* kernels on the GPU");
static_assert(HasTreeletKernels<CudaBackend>::value, "treelet restructuring runs as k_tlo_treelet on the GPU");
static_assert(HasRefitKernels<CudaBackend>::value, "the refit runs as k_refit_level on the GPU");

}  // namespace rtb

#define RTB_BACKEND rtb::CudaBackend
#include "rtb_api_impl.h"
