// spf_quad.cuh — the fast path of the batched SPF engine (sm_100a): one CTA per job,
// three CTAs per SM, the whole per-job state in shared memory, the link-state graph
// read as 16-byte QUADS from L2 (quad_layout.h).
//
// Same results as spf_batch_kernel (spf_kernel.cuh) and as the reference Dijkstra
//   holo-ospf/src/spf.rs:587-729 (run_area) / holo-isis/src/spf.rs:525-707 (compute_spt)
// under the static-order conditions of SURVEY.md §8a #1; what differs is the data
// layout and the shape of the parallel work:
//
//   1. SSSP    label-correcting relaxation in QUAD SPACE: the frontier is a bitmap over
//              forward quads, a work item is one quad (one 128-bit load, four branch-free
//              relaxations, atomicMin on the slot-indexed distance array).  Buckets are a
//              ring of four frontier bitmaps indexed by (distance >> shift) & 3, so moving
//              to the next bucket is a bitmap switch, not a scan of the distance array.
//              A round is: compact the current bucket's bitmap into a bounded queue
//              (chains of a multi-quad vertex are spread with bit operations), barrier,
//              expand, barrier.
//   2. parents one thread per IN-quad (edge-uniform, no per-vertex degree loop): ECMP-DAG
//              predicate dist[u] + c == dist[v] on four records, chain partials combined
//              with warp shuffles; writes dist / first_parent / n_parents planes.
//   3. hops and next hops: pointer jumping over the first-parent tree, ECMP vertices as
//              jump terminals (the scheme of spf_kernel.cuh phase 3J), 16 first-hop atoms
//              per pass, up to four passes (64 atoms).
//
// Eligibility (decided by the host at graph upload, hspf_capi.cu): packed ids and costs (V,
// quads < 65535, costs <= 65534, degrees <= 128), no LEAF vertex flags, no hop-count mode,
// per-job state within shared memory; and one next-hop word.  Everything else runs
// spf_batch_kernel.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

#include "spf_kernel.cuh"

namespace hspf {

constexpr uint32_t kJsInvalid = 8u;   // HSPF_JS_INVALID
constexpr uint32_t kJsInternal = 16u; // HSPF_JS_INTERNAL: a loop bound that cannot be reached was reached
constexpr uint32_t kJsNarrow = 32u;   // HSPF_JS_NARROW: the job's result does not fit 16-bit planes
constexpr int kQMaxRoot = 64;         // non-HOP root neighbours tracked (>= 64 atoms is refused anyway)
constexpr int kQuadThreads = 512;     // CTA size, the fastest of the sweep in profiles/r2_kernel_history.md

struct QuadDev {
    uint32_t NQ, NIQ, shift, isteps;
    const uint4 *fq;            // [NQ]
    const uint32_t *fcont;      // [NQ/32]
    const uint16_t *slot_of;    // [V]
    const uint16_t *vert_of;    // [NQ]
    const uint4 *iq;            // [NIQ]
    const uint2 *imeta;         // [NIQ]
    const uint32_t *fpos;       // [E]
    const uint32_t *ipos;       // [E]
};

struct QuadLayout {   // byte offsets into dynamic shared memory
    uint32_t dist, ring, cont, h0, ecmp, elist, total;
};

struct QuadArgs {
    DevGraph g;
    QuadDev q;
    QuadLayout lay;
    uint32_t n_jobs;
    const uint32_t *roots;
    const uint32_t *ov_off;
    const uint32_t *ov_edge;
    const uint32_t *ov_cost;
    uint32_t *out_dist;
    uint16_t *out_hops;
    uint32_t *out_fp;
    uint16_t *out_npar;
    uint64_t *out_nh;
    uint32_t *out_status;
    uint32_t *job_counter;
    uint32_t narrow;            // 1: 16-bit result planes (hspf_result16): out_dist / out_fp / out_nh point at u16 arrays
    // Fused exchange (multi-GPU, 16-bit planes): the result writer also stores the planes the
    // consumers need (dist, hops, nh_mask, job status) into this rank's slot on every peer GPU,
    // over NVLink, job by job while the batch computes: peer address = local address + peer_delta[k].
    uint32_t n_peers;
    long long peer_delta[7];
    uint32_t *done;             // optional: done[job / done_chunk] counts finished jobs (release: planes first), so
    uint32_t done_chunk;        // that the host call can copy a chunk's planes back while the launch still runs
    unsigned long long *prof;   // optional [gridDim][16] cycle counters
};

// The jump words are padded to a multiple of 4 * kQuadThreads (unrolled rounds without bounds checks).
inline QuadLayout make_quad_layout(uint32_t V, uint32_t NQ) {
    QuadLayout L{};
    auto al = [](size_t x) { return (uint32_t)((x + 15) / 16 * 16); };
    const uint32_t nbv = (V + 31) / 32, nbw = (NQ / 32 + 1u) & ~1u;   // bitmap rows: an even number of words
    const uint32_t Vp = (V + 4 * kQuadThreads - 1) / (4 * kQuadThreads) * (4 * kQuadThreads);
    uint32_t o = 0;
    L.dist = o; o += al((size_t)NQ * 4);
    // phase 3: jump words u32[Vp] over dist, ECMP vertex list u16[V] behind them
    L.elist = al((size_t)Vp * 4);
    if (L.elist + al((size_t)V * 2) > o) o = L.elist + al((size_t)V * 2);
    L.ring = o; o += al((size_t)4 * nbw * 4);      // [word][bucket & 3]
    L.cont = o; o += al((size_t)nbw * 4);
    L.h0 = o; o += al((size_t)nbv * 4);
    L.ecmp = o; o += al((size_t)nbv * 4);
    L.total = o;
    return L;
}

struct QSmall {
    long long t_mark;     // phase profile clock of thread 0 (here, not in a register held through the kernel)
    uint32_t cnt[2];
    uint32_t wake;        // epoch: bumped by a working warp that sees plenty of work while others sleep
    uint32_t status;
    uint32_t job;
    uint32_t n_ov, sh;
    uint32_t ov_edge[kMaxOv], ov_cost[kMaxOv];          // forward edge, new cost (kInf = disabled)
    uint32_t ov_fq[kMaxOv], ov_iq[kMaxOv];              // quad * 4 + record in fq / iq
    uint32_t n_roottab, root_rb, n_atoms;
    uint32_t rt_target[kQMaxRoot], rt_base[kQMaxRoot], rt_cost[kQMaxRoot];
};

#define HSPF_QMARK(k)                                                            \
    do {                                                                         \
        if (a.prof && tid == 0) {                                                \
            const long long now_ = clock64();                                    \
            a.prof[(size_t)blockIdx.x * 16 + (k)] += (unsigned long long)(now_ - S.t_mark); \
            S.t_mark = now_;                                                     \
        }                                                                        \
    } while (0)

template <bool kOv>
__global__ void __launch_bounds__(kQuadThreads, 3) spf_quad_kernel(const QuadArgs a) {
    constexpr int T = kQuadThreads;
    extern __shared__ __align__(16) uint8_t qsm[];
    __shared__ QSmall S;

    const DevGraph &g = a.g;
    const QuadDev &Q = a.q;
    const QuadLayout &L = a.lay;
    const uint32_t V = g.V, NQ = Q.NQ, NBW = NQ >> 5, nbv = (V + 31) >> 5;
    const uint32_t NBWp = (NBW + 1u) & ~1u;     // bitmap row stride: an even number of words
    const uint32_t tid = threadIdx.x, lane = tid & 31;

    uint32_t *dist = reinterpret_cast<uint32_t *>(qsm + L.dist);
    uint32_t *ring = reinterpret_cast<uint32_t *>(qsm + L.ring);     // frontier bitmaps, word w of bucket b at [w * 4 + (b & 3)]
    uint32_t *cont_s = reinterpret_cast<uint32_t *>(qsm + L.cont);
    uint32_t *h0bm = reinterpret_cast<uint32_t *>(qsm + L.h0);
    uint32_t *ecmpbm = reinterpret_cast<uint32_t *>(qsm + L.ecmp);
    uint32_t *word = dist;                                   // phase 3
    uint16_t *elist = reinterpret_cast<uint16_t *>(qsm + L.elist);

    if (tid == 0) S.t_mark = clock64();

    // once per CTA: chain-continuation bits
    for (uint32_t w = tid; w < NBWp; w += T) cont_s[w] = (w < NBW) ? Q.fcont[w] : 0u;
    auto is_hop = [&](uint32_t v) -> bool { return (__ldg(&g.vflags[v]) & kVfHop) != 0; };
    const uint32_t Vp = (V + 4 * T - 1) / (4 * T) * (4 * T);
    // Unreached sentinel: a relaxed distance above reject_above must be rejected (IS-IS
    // MAX_PATH_METRIC, holo-isis/src/spf.rs:636-645).  With every distance initialised to
    // reject_above + 1 the improvement test nd < dist[head] does that by itself.
    const uint32_t U = g.reject_above + 1u ? g.reject_above + 1u : kInf;

    for (;;) {
        // ---- fetch next job -------------------------------------------------------
        __syncthreads();
        if (tid == 0) S.job = atomicAdd(a.job_counter, 1u);
        __syncthreads();
        const uint32_t job = S.job;
        if (job >= a.n_jobs) break;
        const uint32_t root = a.roots[job];
        uint32_t n_ov_raw = 0;
        if (kOv && a.ov_off) n_ov_raw = a.ov_off[job + 1] - a.ov_off[job];
        if (root >= V || n_ov_raw > (uint32_t)kMaxOv) {      // device-pointer callers are not validated on the host
            if (tid == 0) {
                a.out_status[job] = kJsInvalid;
                for (uint32_t k = 0; k < (a.narrow ? a.n_peers : 0u); ++k)
                    *reinterpret_cast<uint32_t *>(reinterpret_cast<char *>(&a.out_status[job]) + a.peer_delta[k]) = kJsInvalid;
                if (a.done) { __threadfence(); atomicAdd(&a.done[job / a.done_chunk], 1u); }
            }
            continue;
        }
        const size_t jo = (size_t)job * V;
        const bool narrow = a.narrow != 0;
        uint32_t *o_dist = a.out_dist + jo;
        uint16_t *o_hops = a.out_hops + jo;
        uint32_t *o_fp = a.out_fp + jo;
        uint16_t *o_npar = a.out_npar + jo;
        uint64_t *o_nh = a.out_nh + jo;
        uint16_t *o_dist16 = reinterpret_cast<uint16_t *>(a.out_dist) + jo;     // narrow planes (hspf_result16)
        uint16_t *o_fp16 = reinterpret_cast<uint16_t *>(a.out_fp) + jo;
        uint16_t *o_nh16 = reinterpret_cast<uint16_t *>(a.out_nh) + jo;
        // the planes just written are read back in phase 3 (first parents, distances of ECMP parents)
        const uint32_t n_peers = narrow ? a.n_peers : 0u;
        // Fused exchange: a finished job's row of a travelling plane goes to the same position of
        // every peer's copy of this rank's slot, as 16-byte stores (full NVLink write packets; the
        // row was just written, so the loads hit L2), unaligned ends as 2-byte stores.
        auto peer_push_row = [&](uint16_t *row) {
            char *src = reinterpret_cast<char *>(row);
            const size_t bytes = (size_t)V * 2;
            const size_t head = (16 - (reinterpret_cast<uintptr_t>(src) & 15)) & 15;       // (deltas are multiples of 256)
            const size_t h = head < bytes ? head : bytes;
            const size_t n16 = (bytes - h) / 16, tail0 = h + n16 * 16;
            for (size_t i = tid; i < n16; i += T) {
                const uint4 val = __ldcg(reinterpret_cast<const uint4 *>(src + h) + i);
                for (uint32_t k = 0; k < n_peers; ++k)
                    reinterpret_cast<uint4 *>(src + h + a.peer_delta[k])[i] = val;
            }
            auto push16 = [&](size_t o) {
                const uint16_t val = __ldcg(reinterpret_cast<const uint16_t *>(src + o));
                for (uint32_t k = 0; k < n_peers; ++k) *reinterpret_cast<uint16_t *>(src + o + a.peer_delta[k]) = val;
            };
            for (size_t o = (size_t)tid * 2; o < h; o += (size_t)T * 2) push16(o);
            for (size_t o = tail0 + (size_t)tid * 2; o < bytes; o += (size_t)T * 2) push16(o);
        };
        auto ld_fp = [&](uint32_t v) -> uint32_t {
            if (narrow) { const uint32_t f = __ldcg(&o_fp16[v]); return f == 0xFFFFu ? kInf : f; }
            return __ldcg(&o_fp[v]);
        };
        auto ld_dist = [&](uint32_t v) -> uint32_t {
            if (narrow) { const uint32_t d = __ldcg(&o_dist16[v]); return d == 0xFFFFu ? kInf : d; }
            return __ldcg(&o_dist[v]);
        };

        // ---- per-job init -----------------------------------------------------------
        {
            uint4 *d4 = reinterpret_cast<uint4 *>(dist);
            const uint4 inf4 = make_uint4(U, U, U, U);
            for (uint32_t i = tid; i < NQ / 4; i += T) d4[i] = inf4;
            for (uint32_t i = tid; i < 4 * NBWp; i += T) ring[i] = 0;
            for (uint32_t w = tid; w < nbv; w += T) { h0bm[w] = 0; ecmpbm[w] = 0; }
        }
        if (tid == 0) {
            S.status = 0;
            S.cnt[0] = 0;
            S.cnt[1] = 0;
            S.wake = 0;
            S.n_ov = n_ov_raw;
            S.sh = Q.shift;
        }
        __syncthreads();
        if (kOv && tid < n_ov_raw) {
            const uint32_t e = a.ov_edge[a.ov_off[job] + tid];
            const uint32_t c = a.ov_cost[a.ov_off[job] + tid];
            if (e >= g.E) {
                atomicOr(&S.status, kJsInvalid);
                S.ov_edge[tid] = kInf; S.ov_cost[tid] = kInf; S.ov_fq[tid] = kInf; S.ov_iq[tid] = kInf;
            } else {
                S.ov_edge[tid] = e;
                S.ov_cost[tid] = c;
                S.ov_fq[tid] = Q.fpos[e];
                S.ov_iq[tid] = Q.ipos[e];
                const uint32_t tail = Q.vert_of[Q.fpos[e] >> 2];
                if (c == 0 && (g.vflags[tail] & kVfHop)) atomicOr(&S.status, kJsOrder);
                if (c != kInf) {
                    // a relaxation out of bucket b must land in b .. b+3 (ring of four bitmaps)
                    uint32_t sh = Q.shift;
                    while (sh < 31 && (3ull << sh) < (unsigned long long)c) ++sh;
                    atomicMax(&S.sh, sh);
                }
            }
        }
        const uint32_t rs = Q.slot_of[root];
        if (tid == 0) {
            dist[rs] = 0;
            ring[(rs >> 5) << 2] = 1u << (rs & 31);     // bucket 0
        }
        __syncthreads();
        const uint32_t n_ov = kOv ? S.n_ov : 0u;
        auto ov_cost_of = [&](uint32_t e, uint32_t c) -> uint32_t {   // cost of forward edge e under this job's overrides
            for (uint32_t k = 0; k < n_ov; ++k)
                if (S.ov_edge[k] == e) c = S.ov_cost[k];
            return c;
        };
        // root edge table: first-hop atom bases behind the root's non-HOP neighbours
        if (tid == 32 % T) {
            const uint32_t rb = g.row[root], re = g.row[root + 1];
            uint32_t nt = 0, nextbase = re - rb;
            for (uint32_t e = rb; e < re; ++e) {
                const uint2 ec = g.edge[e];
                const uint32_t h = ec.x;
                if (!(g.vflags[h] & kVfHop)) {
                    if (nt < (uint32_t)kQMaxRoot) {
                        S.rt_target[nt] = h;
                        S.rt_base[nt] = nextbase;
                        S.rt_cost[nt] = ov_cost_of(e, ec.y);
                        ++nt;
                    } else {
                        atomicOr(&S.status, kJsTooManyAtoms);
                    }
                    nextbase += g.row[h + 1] - g.row[h];
                }
            }
            S.n_roottab = nt;
            S.root_rb = rb;
            if (nextbase > 64u) { atomicOr(&S.status, kJsTooManyAtoms); nextbase = 64u; }
            S.n_atoms = nextbase;
        }
        __syncthreads();
        HSPF_QMARK(0);   // job fetch + init

        // ======================= phase 1: SSSP in quad space ===========================
        const uint32_t sh = kOv ? S.sh : Q.shift;
        {
            // one quad: four relaxations (pad records never improve anything)
            auto relax = [&](uint32_t q, uint32_t first, uint32_t du, const uint4 &r4) {
                uint32_t hs[4] = {r4.x & 0xFFFFu, r4.y & 0xFFFFu, r4.z & 0xFFFFu, r4.w & 0xFFFFu};
                uint32_t cs[4] = {r4.x >> 16, r4.y >> 16, r4.z >> 16, r4.w >> 16};
                if (kOv) {
                    for (uint32_t k = 0; k < n_ov; ++k) {
                        const uint32_t fp_ = S.ov_fq[k];
                        if ((fp_ >> 2) != q) continue;
                        const uint32_t c = S.ov_cost[k];
#pragma unroll
                        for (int j = 0; j < 4; ++j)
                            if ((fp_ & 3u) == (uint32_t)j) {
                                if (c == kInf) { hs[j] = first; cs[j] = 0xFFFFu; } else cs[j] = c;
                            }
                    }
                }
                uint32_t dh[4];
#pragma unroll
                for (int j = 0; j < 4; ++j) dh[j] = dist[hs[j]];
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const uint32_t nd = kOv ? sat_add(du, cs[j]) : du + cs[j];
                    if (nd < dh[j]) {      // also rejects nd > reject_above (see U)
                        // The mark must not become visible before the distance (another warp may claim
                        // it at once): it takes the atomic's result as an operand.  A mark is only needed
                        // when this relaxation was the improvement.
                        const uint32_t old = atomicMin(&dist[hs[j]], nd);
                        if (old > nd) atomicOr(&ring[((hs[j] >> 5) << 2) + ((nd >> sh) & 3u)], 1u << (hs[j] & 31));
                    }
                }
            };
            // Buckets are processed in order; a bucket takes rounds.  In a round every warp claims
            // its own chunk of the bucket's bitmap (one word per lane; atomicExch: a mark made
            // meanwhile by another warp is either taken now or stays for the next claim).  A warp
            // scan of the popcounts gives every quad of the chunk an output index, and output lane t
            // finds its quad by itself — owner word by binary search over the scanned counts
            // (shuffles), then the k-th set bit of that word — so all lanes work in every pass,
            // whatever the distribution of bits over the words, and the quad goes straight from the
            // lane's registers into the relaxation: no queue, no CTA-wide scan.  One CTA barrier per
            // round; the bucket is finished by a round that claimed nothing.
            constexpr uint32_t kWarps_ = T / 32;
            const uint32_t warp = tid >> 5;
            // chunk = the bitmap words of one claim (one per lane): sized so that every warp owns one
            const uint32_t cw = min(32u, (NBWp + kWarps_ - 1) / kWarps_);
            const uint32_t nchunks = (NBWp + cw - 1) / cw;
            // output index t of a claimed chunk -> queue-less entry (quad | first quad of its chain << 16)
            auto pick = [&](uint32_t t, uint32_t incl, uint32_t bits, uint32_t meta, uint32_t C) -> uint32_t {
                uint32_t lo = 0;      // owner = number of lanes whose inclusive count is <= t
#pragma unroll
                for (uint32_t step = 16; step >= 1; step >>= 1) {
                    const uint32_t v = __shfl_sync(0xffffffffu, incl, lo + step - 1);
                    if (v <= t) lo += step;
                }
                lo &= 31u;
                const uint32_t ob = __shfl_sync(0xffffffffu, bits, lo);
                const uint32_t om = __shfl_sync(0xffffffffu, meta, lo);
                const uint32_t oc = __shfl_sync(0xffffffffu, C, lo);
                // k-th set bit of the owner's word
                uint32_t k = t - (om & 0xFFFFu), pos = 0, cc;
                cc = __popc(ob & 0xFFFFu); if (k >= cc) { k -= cc; pos = 16; }
                cc = __popc((ob >> pos) & 0xFFu); if (k >= cc) { k -= cc; pos += 8; }
                cc = __popc((ob >> pos) & 0xFu); if (k >= cc) { k -= cc; pos += 4; }
                cc = __popc((ob >> pos) & 0x3u); if (k >= cc) { k -= cc; pos += 2; }
                cc = (ob >> pos) & 1u; if (k >= cc) pos += 1;
                pos &= 31u;
                // first quad of the chain: the nearest bit at or below pos that continues nothing
                const uint32_t fb = 31u - __clz((~oc & ((2u << pos) - 1u)) | 1u);
                const uint32_t qb = (om >> 16) * 32;
                return (qb + pos) | ((qb + fb) << 16);
            };
            uint32_t cur = 0, empties = 0;
            bool bucket_work = false;
            for (uint32_t guard = 0;; ++guard) {
                if (guard > (1u << 24)) { if (tid == 0) atomicOr(&S.status, kJsInternal); break; }   // defensive
                uint32_t *bm = ring + (cur & 3u);
                int claimed = 0;
                for (uint32_t c = warp; c < nchunks; c += kWarps_) {
                    const uint32_t w = c * cw + lane;
                    const bool mine = lane < cw && w < NBWp;
                    uint32_t bits = mine ? *reinterpret_cast<volatile uint32_t *>(&bm[w << 2]) : 0u;
                    if (!__any_sync(0xffffffffu, bits != 0)) continue;
                    claimed = 1;
                    uint32_t C = 0;
                    if (bits) {
                        bits = atomicExch(&bm[w << 2], 0u);
                        C = cont_s[w];
                        uint32_t m = bits;
                        while ((m = (m << 1) & C) != 0) bits |= m;      // the other quads of a multi-quad vertex
                    }
                    const uint32_t cnt = __popc(bits);
                    uint32_t incl = cnt;
#pragma unroll
                    for (int o = 1; o < 32; o <<= 1) {
                        const uint32_t t = __shfl_up_sync(0xffffffffu, incl, o);
                        if ((int)lane >= o) incl += t;
                    }
                    const uint32_t n = __shfl_sync(0xffffffffu, incl, 31);
                    const uint32_t meta = (incl - cnt) | (w << 16);
                    if (a.prof && lane == 0) atomicAdd(&a.prof[(size_t)blockIdx.x * 16 + 12], (unsigned long long)n);
                    // two quads of a lane in flight
                    for (uint32_t t0 = 0; t0 < n; t0 += 64) {
                        const uint32_t ta = t0 + lane, tb = ta + 32;
                        const bool hb = t0 + 32 < n;                       // warp-uniform
                        const uint32_t e0 = pick(ta, incl, bits, meta, C);
                        const uint32_t e1 = hb ? pick(tb, incl, bits, meta, C) : 0u;
                        const uint32_t du0 = (ta < n) ? dist[e0 >> 16] : kInf;     // the chain owner's distance
                        const uint32_t du1 = (hb && tb < n) ? dist[e1 >> 16] : kInf;
                        // a mark is stale when the vertex was settled in an earlier bucket
                        const bool l0 = (du0 >> sh) == cur, l1 = (du1 >> sh) == cur;
                        uint4 r0 = make_uint4(0u, 0u, 0u, 0u), r1 = r0;
                        if (l0) r0 = __ldg(&Q.fq[e0 & 0xFFFFu]);
                        if (l1) r1 = __ldg(&Q.fq[e1 & 0xFFFFu]);
                        if (l0) relax(e0 & 0xFFFFu, e0 >> 16, du0, r0);
                        if (l1) relax(e1 & 0xFFFFu, e1 >> 16, du1, r1);
                    }
                }
                if (a.prof && tid == 0) a.prof[(size_t)blockIdx.x * 16 + 7] += 1;
                if (__syncthreads_or(claimed)) { bucket_work = true; continue; }      // another round of this bucket
                if (bucket_work) empties = 0;
                else if (++empties == 4) break;      // bucket width >= a third of the largest cost: gaps span < 4 buckets
                bucket_work = false;
                ++cur;
            }
        }
        HSPF_QMARK(1);   // SSSP

        // hops-0 non-HOP heads of root edges (their out-edges carry first-hop atoms)
        if (tid < S.n_roottab) {
            const uint32_t h = S.rt_target[tid], c = S.rt_cost[tid];
            if (c < U && dist[Q.slot_of[h]] == c) atomicOr(&h0bm[h >> 5], 1u << (h & 31));
        }
        __syncthreads();
        auto hops0 = [&](uint32_t u) -> bool { return u == root || ((h0bm[u >> 5] >> (u & 31)) & 1u); };

        // first-hop atom seeds: one thread per atom, is its edge in the DAG?
        const uint32_t n_atoms = S.n_atoms;
        uint32_t seed_v = kInf;
        if (tid < n_atoms) {
            const uint32_t atom = tid, rdeg = g.row[root + 1] - S.root_rb;
            uint32_t e = kInf, u = root;
            if (atom < rdeg) {
                e = S.root_rb + atom;
            } else {
                for (uint32_t k = 0; k < S.n_roottab; ++k) {
                    const uint32_t N = S.rt_target[k], nb = S.rt_base[k];
                    if (atom < nb || atom >= nb + (g.row[N + 1] - g.row[N])) continue;
                    uint32_t q = 0;      // parallel root edges: only the first one's range is used
                    while (q < k && S.rt_target[q] != N) ++q;
                    if (q == k && hops0(N)) { u = N; e = g.row[N] + (atom - nb); }
                    break;
                }
            }
            if (e != kInf) {
                const uint2 ec = g.edge[e];
                const uint32_t c = kOv ? ov_cost_of(e, ec.y) : ec.y;
                const uint32_t du = dist[Q.slot_of[u]], dh = dist[Q.slot_of[ec.x]];
                if (du < U && dh < U && c != kInf && sat_add(du, c) == dh &&
                    !((g.flags & kGfNoHopTargetNoNh) && !is_hop(ec.x)))
                    seed_v = ec.x;
            }
        }

        // ======================= phase 2: ECMP parents, one thread per in-quad =============
        {
            uint32_t sat_flag = 0, narrow_flag = 0;
            const uint32_t NIQ = Q.NIQ, isteps = Q.isteps;
            // DAG predicate on the four records of one in-quad -> (count, best (dist, slot) parent)
            auto pull = [&](uint32_t i, const uint2 &m, const uint4 &r4, uint32_t &dv, uint32_t &cnt, uint32_t &bd, uint32_t &bs) {
                const uint32_t sv = (m.x != 0xFFFFFFFFu) ? (m.x & 0xFFFFu) : 0u;
                dv = dist[sv];
                uint32_t su[4] = {r4.x & 0xFFFFu, r4.y & 0xFFFFu, r4.z & 0xFFFFu, r4.w & 0xFFFFu};
                uint32_t cs[4] = {r4.x >> 16, r4.y >> 16, r4.z >> 16, r4.w >> 16};
                if (kOv) {
                    for (uint32_t k = 0; k < n_ov; ++k) {
                        const uint32_t ip_ = S.ov_iq[k];
                        if ((ip_ >> 2) != i) continue;
                        const uint32_t c = S.ov_cost[k];
#pragma unroll
                        for (int j = 0; j < 4; ++j)
                            if ((ip_ & 3u) == (uint32_t)j) {
                                if (c == kInf) { su[j] = sv; cs[j] = 0xFFFFu; } else cs[j] = c;
                            }
                    }
                }
                uint32_t du[4];
#pragma unroll
                for (int j = 0; j < 4; ++j) du[j] = dist[su[j]];
                cnt = 0; bd = kInf; bs = kInf;
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const uint32_t nd = kOv ? sat_add(du[j], cs[j]) : du[j] + cs[j];
                    const bool ok = du[j] < U && nd == dv;
                    const bool better = ok && (du[j] < bd || (du[j] == bd && su[j] < bs));
                    cnt += ok ? 1u : 0u;
                    bd = better ? du[j] : bd;
                    bs = better ? su[j] : bs;
                }
            };
            // combine the partial results of a chain (the quads of one vertex are adjacent lanes)
            auto combine = [&](uint32_t rem, uint32_t &cnt, uint32_t &bd, uint32_t &bs) {
                for (uint32_t s = 0, d = 1; s < isteps; ++s, d <<= 1) {
                    const uint32_t ocnt = __shfl_down_sync(0xffffffffu, cnt, d);
                    const uint32_t obd = __shfl_down_sync(0xffffffffu, bd, d);
                    const uint32_t obs = __shfl_down_sync(0xffffffffu, bs, d);
                    if (d <= rem) {
                        cnt += ocnt;
                        if (obd < bd || (obd == bd && obs < bs)) { bd = obd; bs = obs; }
                    }
                }
            };
            auto emit_v = [&](const uint2 &m, uint32_t dv, uint32_t cnt, uint32_t bs) {
                if (m.x != 0xFFFFFFFFu && ((m.y >> 8) & 0xFFu) == 0) {      // first quad of a real vertex
                    const uint32_t v = m.x >> 16;
                    if (dv >= U) dv = kInf;                                   // unreached
                    if (v == root || dv == kInf) { cnt = 0; bs = kInf; }
                    if (dv != kInf && g.saturate_at && dv >= g.saturate_at) sat_flag = 1;
                    const uint32_t fpv = cnt ? (uint32_t)__ldg(&Q.vert_of[bs]) : kInf;
                    if (narrow) {
                        if (dv != kInf && dv >= 0xFFFFu) narrow_flag = 1;      // does not fit; 0xFFFF means "not on the SPT"
                        o_dist16[v] = (uint16_t)min(dv, 0xFFFFu);
                        o_fp16[v] = (uint16_t)min(fpv, 0xFFFFu);

                    } else {
                        o_dist[v] = dv;
                        o_fp[v] = fpv;
                    }
                    o_npar[v] = (uint16_t)min(cnt, 0xFFFFu);
                    if (cnt >= 2) atomicOr(&ecmpbm[v >> 5], 1u << (v & 31));
                }
            };
            // two in-quads of a thread in flight (NIQ % 32 == 0: a warp is in range as a whole)
            const uint32_t wbase = tid & ~31u;
            for (uint32_t i0 = 0; i0 + wbase < NIQ; i0 += 2 * T) {
                const uint32_t ia = i0 + tid, ib = ia + T;
                const bool hb = i0 + T + wbase < NIQ;                          // warp-uniform
                const uint2 ma = __ldg(&Q.imeta[ia]);
                const uint4 ra = __ldg(&Q.iq[ia]);
                uint2 mb = make_uint2(0xFFFFFFFFu, 0u);
                uint4 rb = make_uint4(0u, 0u, 0u, 0u);
                if (hb) { mb = __ldg(&Q.imeta[ib]); rb = __ldg(&Q.iq[ib]); }
                uint32_t dva, ca, bda, bsa, dvb = kInf, cb = 0, bdb = kInf, bsb = kInf;
                pull(ia, ma, ra, dva, ca, bda, bsa);
                if (hb) pull(ib, mb, rb, dvb, cb, bdb, bsb);
                combine(ma.y & 0xFFu, ca, bda, bsa);
                if (hb) combine(mb.y & 0xFFu, cb, bdb, bsb);
                emit_v(ma, dva, ca, bsa);
                if (hb) emit_v(mb, dvb, cb, bsb);
            }
            if (sat_flag) atomicOr(&S.status, kJsSaturated);
            if (narrow_flag) atomicOr(&S.status, kJsNarrow);
        }
        __syncthreads();
        HSPF_QMARK(2);   // parents

        // ======================= phase 3: pointer jumping ===============================
        // Hops and next hops are path aggregates over the first-parent tree (sum of the HOP
        // flags, OR of the first-hop atoms): pointer doubling, one 32-bit word per vertex
        // (ancestor:16 | aggregate:16) that only its owner thread stores, so the rounds update
        // in place (a reader sees the old or the new pair, both consistent).  Terminals point
        // at themselves with an aggregate that is neutral under the update, so the update is
        // unconditional: word[v] = (anc(word[A]), agg(v) (+) agg(word[A])).
        // See spf_kernel.cuh phase 3J for the derivation; the first parents are read back
        // from the plane just written.
        // -- hops: sum of HOP flags over (root, v]; the root and unreached vertices are terminals
        for (uint32_t v = tid; v < Vp; v += T) {      // (padding words are terminals: no bounds checks in the rounds)
            const uint32_t f = (v < V) ? ld_fp(v) : kInf;
            word[v] = (f == kInf) ? (v << 16) : ((f << 16) | (is_hop(v) ? 1u : 0u));
        }
        __syncthreads();
        uint32_t jump_rounds = 0;     // rounds in which some vertex still moved
        for (;;) {
            uint32_t moved = 0;
            for (uint32_t v0 = tid; v0 < Vp; v0 += 4 * T) {      // Vp % (4 * T) == 0
                // two jumps per round (v -> A -> A'): fewer barrier-separated rounds
                uint32_t w[4], w2[4], w3[4];
#pragma unroll
                for (int k = 0; k < 4; ++k) w[k] = word[v0 + k * T];
#pragma unroll
                for (int k = 0; k < 4; ++k) w2[k] = word[w[k] >> 16];
#pragma unroll
                for (int k = 0; k < 4; ++k) w3[k] = word[w2[k] >> 16];
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    // w2 / w3 are terminals (point at themselves, sum 0: read twice they add nothing)
                    // or ordinary vertices
                    word[v0 + k * T] = (w3[k] & 0xFFFF0000u) | ((w[k] + w2[k] + w3[k]) & 0xFFFFu);
                    moved |= w3[k] ^ w[k];
                }
            }
            if (a.prof && tid == 0) a.prof[(size_t)blockIdx.x * 16 + 13] += 1;
            if (!__syncthreads_or((moved >> 16) != 0)) break;
            if (++jump_rounds > 32u) { if (tid == 0) atomicOr(&S.status, kJsInternal); break; }   // depth < 2^32: cannot happen
        }
        for (uint32_t v = tid; v < V; v += T) {
            const uint32_t w = word[v];
            const uint32_t h = (w >> 16) == v ? 0u : (w & 0xFFFFu);
            o_hops[v] = (uint16_t)h;
            // a hops-0 vertex that is not a head of a root edge cannot own atoms
            if (h == 0 && v != root && (w >> 16) != v && !hops0(v) && g.row[v + 1] != g.row[v])
                atomicOr(&S.status, kJsTooManyAtoms);
        }
        __syncthreads();
        HSPF_QMARK(5);   // hops

        // -- next hops.  nh[v] = atoms entering v | U nh[p] over DAG parents p that are not at
        // hops 0.  The tree is cut below hops-0 vertices and AT ECMP vertices (jump terminals):
        //   word[v] = (top[v], atoms on the segment (top[v], v])
        // then the ECMP vertices are resolved among themselves (monotone sweeps to the fixpoint)
        // and every vertex adds the final set of its top.  16 atoms per pass.
        auto is_ecmp = [&](uint32_t v) -> bool { return (ecmpbm[v >> 5] >> (v & 31)) & 1u; };
        // ECMP vertex list (ascending ids), built once
        if (tid == 0) S.cnt[0] = 0;
        __syncthreads();
        for (uint32_t w0 = 0; w0 < nbv; w0 += T) {
            const uint32_t w = w0 + tid;
            const uint32_t bits = (w < nbv) ? ecmpbm[w] : 0u;
            if (!__any_sync(0xffffffffu, bits != 0)) continue;
            const uint32_t n = __popc(bits);
            uint32_t incl = n;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const uint32_t t = __shfl_up_sync(0xffffffffu, incl, o);
                if ((int)lane >= o) incl += t;
            }
            const uint32_t tot = __shfl_sync(0xffffffffu, incl, 31);
            uint32_t base = 0;
            if (lane == 31) base = atomicAdd(&S.cnt[0], tot);
            base = __shfl_sync(0xffffffffu, base, 31);
            uint32_t pos = base + incl - n;
            for (uint32_t b = bits; b; b &= b - 1) elist[pos++] = (uint16_t)(w * 32 + (__ffs(b) - 1));
        }
        __syncthreads();
        const uint32_t n_e = S.cnt[0];
        // DAG parents of an ECMP vertex are re-derived from the distance plane just written
        auto parents = [&](uint32_t x, auto &&f) {
            const uint32_t dx = ld_dist(x);
            for (uint32_t j = g.irow[x]; j < g.irow[x + 1]; ++j) {
                uint32_t u, c;
                if constexpr (kOv) {
                    const uint4 r = g.iedge[j];
                    u = r.x; c = ov_cost_of(r.z, r.y);
                    if (c == kInf) continue;
                } else {
                    const uint32_t r = g.iedge16[j];
                    u = r & 0xFFFFu; c = r >> 16;
                }
                const uint32_t du = ld_dist(u);
                if (du != kInf && sat_add(du, c) == dx && !hops0(u)) f(u);
            }
        };
        uint32_t pc[4] = {kInf, kInf, kInf, kInf};
        bool cached = false;
        if (n_e <= (uint32_t)T && tid < n_e) {
            uint32_t n = 0;
            parents(elist[tid], [&](uint32_t u) {
#pragma unroll
                for (int k = 0; k < 4; ++k) if (n == (uint32_t)k) pc[k] = u;
                ++n;
            });
            cached = n <= 4;
        }
        for (uint32_t pass = 0; pass * 16u < n_atoms || pass == 0; ++pass) {
            // terminals (the root, unreached vertices, ECMP vertices) point at themselves
            for (uint32_t v = tid; v < Vp; v += T) {
                uint32_t A = v;
                if (v < V) {
                    const uint32_t f = ld_fp(v);
                    if (f != kInf && !is_ecmp(v)) A = hops0(f) ? root : f;
                }
                word[v] = A << 16;
            }
            __syncthreads();
            if (seed_v != kInf && (tid >> 4) == pass) atomicOr(&word[seed_v], 1u << (tid & 15));
            __syncthreads();
            // the cut tree is no deeper than the first-parent tree: the hop pass's round count suffices
            for (uint32_t r = 0; r < jump_rounds; ++r) {
                for (uint32_t v0 = tid; v0 < Vp; v0 += 4 * T) {
                    uint32_t w[4], w2[4], w3[4];
#pragma unroll
                    for (int k = 0; k < 4; ++k) w[k] = word[v0 + k * T];
#pragma unroll
                    for (int k = 0; k < 4; ++k) w2[k] = word[w[k] >> 16];
#pragma unroll
                    for (int k = 0; k < 4; ++k) w3[k] = word[w2[k] >> 16];
#pragma unroll
                    for (int k = 0; k < 4; ++k)   // OR-ing a terminal's own seeds again is harmless (every vertex ORs in its top's set below)
                        word[v0 + k * T] = (w3[k] & 0xFFFF0000u) | ((w[k] | w2[k] | w3[k]) & 0xFFFFu);
                }
                if (a.prof && tid == 0) a.prof[(size_t)blockIdx.x * 16 + 14] += 1;
                __syncthreads();
            }
            // ECMP vertices: from the self-pointing terminal form to (top, own segment) through the first parent
            if (n_e) {
                for (uint32_t i = tid; i < n_e; i += T) {
                    const uint32_t x = elist[i];
                    const uint32_t seeds = word[x] & 0xFFFFu;
                    const uint32_t f = ld_fp(x);      // an ECMP vertex has parents
                    uint32_t nw;
                    if (hops0(f)) nw = (root << 16) | seeds;
                    else if (is_ecmp(f)) nw = (f << 16) | seeds;
                    else { const uint32_t wf = word[f]; nw = (wf & 0xFFFF0000u) | ((wf | seeds) & 0xFFFFu); }
                    // (word[f] of a non-ECMP f is final and is not rewritten here)
                    word[x] = nw;
                }
                __syncthreads();
                // own segment | final set of own top | the same of every other parent
                for (uint32_t sweeps = 0;;) {
                    int ch = 0;
                    for (uint32_t i = tid; i < n_e; i += T) {
                        const uint32_t x = elist[i];
                        const uint32_t w = word[x], Tx = w >> 16;
                        uint32_t need = (Tx != root) ? word[Tx] : 0u;
                        auto pull_parent = [&](uint32_t u) {
                            const uint32_t wp = word[u], Tp = wp >> 16;
                            need |= wp;
                            if (Tp != root && Tp != u) need |= word[Tp];
                        };
                        if (cached) {
#pragma unroll
                            for (int k = 0; k < 4; ++k) if (pc[k] != kInf) pull_parent(pc[k]);
                        } else {
                            parents(x, pull_parent);
                        }
                        need &= 0xFFFFu & ~w;
                        if (need) { word[x] = w | need; ch = 1; }
                    }
                    if (a.prof && tid == 0) a.prof[(size_t)blockIdx.x * 16 + 15] += 1;
                    if (!__syncthreads_or(ch)) break;
                    if (++sweeps > 16u * n_e + 16u) { if (tid == 0) atomicOr(&S.status, kJsInternal); break; }   // <= 16 bits per vertex
                }
            }
            for (uint32_t v = tid; v < V; v += T) {
                const uint32_t w = word[v], Tv = w >> 16;
                uint32_t m = w;
                if (Tv != root && Tv != v) m |= word[Tv];
                if (narrow) {
                    if (pass == 0) {      // (more than 16 atoms: HSPF_JS_NARROW, set below)
                        o_nh16[v] = (uint16_t)(m & 0xFFFFu);
                    }
                } else {
                    const uint64_t bits = (uint64_t)(m & 0xFFFFu) << (16 * pass);
                    if (pass == 0) o_nh[v] = bits; else o_nh[v] |= bits;
                }
            }
            __syncthreads();
        }
        if (n_peers) {
            __syncthreads();                      // every plane of this job is written (this CTA wrote them all)
            peer_push_row(o_dist16);
            peer_push_row(o_hops);
            peer_push_row(o_nh16);
        }
        if (tid == 0) {
            const uint32_t st = S.status | ((narrow && n_atoms > 16u) ? kJsNarrow : 0u);
            a.out_status[job] = st;
            for (uint32_t k = 0; k < n_peers; ++k)
                *reinterpret_cast<uint32_t *>(reinterpret_cast<char *>(&a.out_status[job]) + a.peer_delta[k]) = st;
        }
        if (a.done) {
            // every plane of this job is written: publish (barrier: the other threads' stores happen
            // before thread 0's fence; fence: before the count becomes visible to the copy engine's wait)
            __syncthreads();
            if (tid == 0) { __threadfence(); atomicAdd(&a.done[job / a.done_chunk], 1u); }
        }
        HSPF_QMARK(4);   // next hops
    }
}

// Permanent cost change of listed forward edges (hspf_graph_update_costs): every copy of an edge's cost in
// the device image — CSR edge, transposed edge (found by its forward index among the head's in-edges),
// their packed twins, the quad-padded in-edge rows of spf_batch_kernel and the two quad-space records
// (QuadHost::fpos / ipos) — is rewritten by one thread per edge.  Runs alone on the ctx stream.
__global__ void patch_costs_kernel(DevGraph g, QuadDev q, bool has_quads, uint32_t n, const uint32_t *edges,
                                   const uint32_t *costs) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint32_t e = edges[i], c = costs[i];
    uint2 *edge = const_cast<uint2 *>(g.edge);
    const uint32_t v = edge[e].x;
    edge[e].y = c;
    if (g.edge16) const_cast<uint32_t *>(g.edge16)[e] = v | (c << 16);
    uint4 *iedge = const_cast<uint4 *>(g.iedge);
    for (uint32_t k = g.irow[v]; k < g.irow[v + 1]; ++k) {
        if (iedge[k].z != e) continue;
        iedge[k].y = c;
        if (g.iedge16) {
            const uint32_t rec = iedge[k].x | (c << 16);
            const_cast<uint32_t *>(g.iedge16)[k] = rec;
            if (g.iquad) reinterpret_cast<uint32_t *>(const_cast<uint4 *>(g.iquad))[(size_t)g.iquad_row[v] * 4 + (k - g.irow[v])] = rec;
        }
        break;
    }
    if (has_quads) {
        uint32_t *fq = reinterpret_cast<uint32_t *>(const_cast<uint4 *>(q.fq));
        uint32_t *iq = reinterpret_cast<uint32_t *>(const_cast<uint4 *>(q.iq));
        const uint32_t fp = q.fpos[e], ip = q.ipos[e];
        fq[fp] = (fq[fp] & 0xFFFFu) | (c << 16);
        iq[ip] = (iq[ip] & 0xFFFFu) | (c << 16);
    }
}

}  // namespace hspf
