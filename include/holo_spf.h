/*
 * holo_spf.h — C ABI of the B200 batched shortest-path-first engine.
 *
 * This is the drop-in boundary for the one hot path this repo replaces in
 * holo-routing/holo: the Dijkstra bodies of
 *
 *   holo-ospf/src/spf.rs:587-729   run_area<V>()      (OSPFv2 / OSPFv3, per area)
 *   holo-isis/src/spf.rs:525-707   compute_spt()      (IS-IS, per level / MT)
 *
 * The reference has no FFI for this path (workspace forbids unsafe,
 * Cargo.toml:92-94), so the seam is defined here: the Rust caller flattens
 * its LSDB into the CSR described below (walking V::vertex_lsa_find /
 * V::vertex_lsa_links once, holo-ospf/src/ospfv2/spf.rs:356-461, or
 * vertex_edges, holo-isis/src/spf.rs:1005-1138), calls hspf_run_batch() and
 * rebuilds `Vertex{distance,hops,nexthops}` / `Spt` from the SoA result.
 * INTEGRATION.md shows the `extern "C"` block a maintainer would add.
 *
 * Conventions
 *  - plain pointers and sizes only; inputs are borrowed for the call, outputs
 *    are written into caller-allocated buffers, nothing is returned by
 *    library-owned pointer; no callbacks.
 *  - every entry point returns HSPF_OK (0) or a negative HSPF_E_*; C++
 *    exceptions never cross the boundary.  A non-zero status tells the caller
 *    to fall back to its in-tree CPU path, matching the reference's
 *    "log and continue" convention (holo-ospf/src/spf.rs:608,718).
 *  - one hspf_ctx per protocol instance (one caller thread each,
 *    holo-protocol/src/lib.rs:258-287,405-408); no process-global mutable
 *    state; a ctx owns its CUDA stream and device buffers.
 *  - there is NO CPU fallback inside this library: without a usable CUDA
 *    device every call fails with HSPF_E_CUDA.
 */
#ifndef HOLO_SPF_H
#define HOLO_SPF_H

#include <stdint.h>
#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define HSPF_OK                  0
#define HSPF_E_INVAL            (-1) /* malformed argument / CSR                      */
#define HSPF_E_CUDA             (-2) /* CUDA runtime error (see hspf_last_error)       */
#define HSPF_E_NOMEM            (-3)
#define HSPF_E_NEEDS_ORACLE     (-4) /* order-dependent semantics: zero-cost link out
                                        of a hop-counting vertex (see SURVEY §8a #1);
                                        caller must use its CPU path                  */
#define HSPF_E_UNSUPPORTED      (-5)
#define HSPF_E_JOB_STATUS       (-6) /* call completed, but >=1 job_status != 0       */

/* ---- vertex flags (hspf_csr.vflags) -------------------------------------- */
/* Vertex counts a hop when entered: OSPF Router vertex (spf.rs:675-678) /
 * IS-IS non-pseudonode (holo-isis spf.rs:648-651).                           */
#define HSPF_VF_HOP              0x01u
/* Vertex is never expanded (its out-edges are ignored): IS-IS vertex without
 * zeroth LSP (spf.rs:556-559) or failing the protocols-supported check
 * (spf.rs:580-602).                                                           */
#define HSPF_VF_LEAF             0x02u
/* Vertex is not expanded unless it is the root: IS-IS overload bit
 * (spf.rs:566-572; `hops != 0` is equivalent to "not the root" for a
 * non-pseudonode).                                                            */
#define HSPF_VF_LEAF_UNLESS_ROOT 0x04u

/* ---- graph flags (hspf_csr.flags) ----------------------------------------- */
/* IS-IS first-hop rule (spf.rs:678-702): an edge out of a hops==0 vertex into a
 * NON-hop vertex (pseudonode) contributes no next hop.  OSPF leaves this clear
 * (root -> transit network yields (iface, None), ospfv2/spf.rs:297-303).      */
#define HSPF_GF_NOHOP_TARGET_NO_NEXTHOP 0x01u

/* Hop-count topology (holo-isis MetricMode::HopCount, flooding/manet.rs:59,
 * spf.rs:1122-1138): every HOP -> non-HOP edge costs 0 and every other edge costs
 * 1 (checked at upload).  Zero-cost links out of HOP vertices make the reference's
 * result depend on pop order, but here in one simple way the device reproduces
 * exactly: a pseudonode enters the candidate list when the lowest-numbered
 * attached router of its distance level is expanded and is popped before the
 * next router ((d, false, ..) < (d, true, ..)), so that router is its only ECMP
 * parent.  Without this flag such graphs are refused (HSPF_E_NEEDS_ORACLE). */
#define HSPF_GF_HOPCOUNT 0x02u

#define HSPF_COST_DISABLED 0xFFFFFFFFu /* edge override: remove the edge       */
#define HSPF_DIST_INF      0xFFFFFFFFu /* result: vertex is not on the SPT     */
#define HSPF_NO_PARENT     0xFFFFFFFFu

/* ---- per-job status bits (hspf_result.job_status) --------------------------- */
#define HSPF_JS_SATURATED      0x1u /* some distance reached csr.saturate_at:
                                       OSPF u16 saturating_add (spf.rs:672) makes the
                                       ECMP DAG pop-order dependent; use the CPU path */
#define HSPF_JS_TOO_MANY_ATOMS 0x2u /* first-hop atoms > 64*nh_words              */
#define HSPF_JS_ORDER          0x4u /* an override put a zero cost on a link out of a
                                       hop-counting vertex: pop-order dependent, use the
                                       CPU path (same reason as HSPF_E_NEEDS_ORACLE)    */
#define HSPF_JS_INVALID        0x8u /* malformed job (root >= n_vertices, more than
                                       HSPF_MAX_OVERRIDES overrides, override edge >= n_edges):
                                       the job was skipped, its planes are not written.  Only
                                       reachable with HSPF_RUN_DEVICE_PTRS / hspf_run_batch_async,
                                       whose job arrays the host cannot see; host-pointer calls
                                       fail with HSPF_E_INVAL before anything runs            */

#define HSPF_JS_NARROW         0x20u /* hspf_run_batch16 only: the result does not fit 16-bit planes */
#define HSPF_JS_INTERNAL       0x10u /* a device loop hit a bound that cannot be reached on a
                                        valid graph (defensive; please report): planes undefined */

/*
 * Flattened link-state graph of one area / level / topology.
 *
 * Vertices MUST be numbered in the reference's VertexId order, because that
 * order is the tie-break of the candidate list `(distance, VertexId)`:
 *   OSPFv2: every Network{dr_addr} before every Router{router_id}, each by
 *           IPv4 value (derived Ord, holo-ospf/src/ospfv2/spf.rs:40-44);
 *   OSPFv3: Network{router_id, iface_id} before Router (ospfv3/spf.rs:37-41);
 *   IS-IS : pseudonodes (non_pseudonode=false) before routers, then LanId
 *           (holo-isis/src/spf.rs:94-98).
 *
 * Edges of a vertex MUST appear in the reference's link iteration order
 * (vertex_lsa_links / vertex_edges) and only contain links that survive the
 * structural filters there: target LSA exists and is not MaxAge, and the
 * mutual-link check ("target has any link back", spf.rs:654-664) passes.
 * Self loops are not allowed.  No edge may join two non-HOP vertices.
 */
typedef struct hspf_csr {
    uint32_t n_vertices;
    uint32_t n_edges;
    const uint32_t *row_ptr;   /* [n_vertices + 1]                              */
    const uint32_t *col;       /* [n_edges] head vertex                          */
    const uint32_t *cost;      /* [n_edges] link cost (OSPF u16 / IS-IS u32)     */
    const uint8_t  *vflags;    /* [n_vertices] HSPF_VF_*                         */
    /* A relaxed distance strictly greater than this is rejected (IS-IS
     * MAX_PATH_METRIC 1023 / 0xFE000000, spf.rs:45-47,636-645).  OSPF passes
     * 0xFFFFFFFE (no rejection).                                               */
    uint32_t reject_above;
    /* If non-zero: a final distance >= this value marks the job
     * HSPF_JS_SATURATED (OSPF passes 0xFFFF).                                  */
    uint32_t saturate_at;
    uint32_t flags;            /* HSPF_GF_*                                      */
    /* Near/far bucket width of the device SSSP; 0 = let the library choose.    */
    uint32_t delta;
} hspf_csr;

/*
 * One batch of independent SPF jobs over one uploaded graph: job j computes the
 * SPT rooted at roots[j] over the graph with edge overrides
 * ov_edge/ov_cost[ov_off[j] .. ov_off[j+1]) applied (what-if perturbations:
 * new cost, or HSPF_COST_DISABLED).  ov_off may be NULL (no overrides).
 * The caller is responsible for keeping the mutual-link property under
 * overrides (disable both directions of an adjacency).  At most
 * HSPF_MAX_OVERRIDES per job.
 */
#define HSPF_MAX_OVERRIDES 8
typedef struct hspf_jobs {
    uint32_t n_jobs;
    const uint32_t *roots;     /* [n_jobs]                                       */
    const uint32_t *ov_off;    /* [n_jobs + 1] or NULL                           */
    const uint32_t *ov_edge;   /* CSR edge index                                 */
    const uint32_t *ov_cost;   /* new cost or HSPF_COST_DISABLED                 */
} hspf_jobs;

/*
 * SoA results, caller-allocated, [n_jobs][n_vertices] row-major.  Any pointer
 * may be NULL to skip that plane.  With HSPF_RUN_DEVICE_PTRS the pointers (and
 * the hspf_jobs arrays) are device pointers on the ctx's device and no
 * host<->device copy is made.
 *
 *  dist         : distance from the root, HSPF_DIST_INF if not on the SPT
 *                 (Vertex.distance, holo-ospf spf.rs:42 / holo-isis spf.rs:79)
 *  hops         : Vertex.hops (number of HOP vertices on the first-found
 *                 shortest path, root excluded)
 *  first_parent : DAG parent with the smallest (distance, VertexId): the vertex
 *                 whose relaxation created the final candidate entry
 *                 (spf.rs:700-703); HSPF_NO_PARENT for the root / unreached
 *  n_parents    : number of ECMP DAG in-edges (IS-IS Vertex.parents.len(),
 *                 parallel edges counted, spf.rs:675)
 *  nh_mask      : [n_jobs][n_vertices][nh_words] bitset of first-hop atoms
 *                 (see hspf_atom_decode): the union the reference builds in
 *                 calc_nexthops / spf.rs:678-702 before the host maps atoms to
 *                 interface/address next hops
 *  job_status   : [n_jobs] HSPF_JS_* bits
 */
typedef struct hspf_result {
    uint32_t *dist;
    uint16_t *hops;
    uint32_t *first_parent;
    uint16_t *n_parents;
    uint64_t *nh_mask;
    uint32_t  nh_words;        /* 1..4                                           */
    uint32_t *job_status;
} hspf_result;

#define HSPF_RUN_DEVICE_PTRS 0x1u

/*
 * The same results in 16-bit planes: 10 bytes per vertex instead of 20, or 6 when the
 * caller skips first_parent / n_parents (holo-ospf keeps neither in its Vertex,
 * holo-ospf/src/spf.rs:38-46; holo-isis does, spf.rs:76-86).  Half the bytes over PCIe in the
 * host-pointer call and over NVLink in the multi-GPU exchange.  OSPF always fits: its
 * distances are u16 (spf.rs:672) and a job whose distances reach 0xFFFF is HSPF_JS_SATURATED
 * anyway.  Encoding: dist 0xFFFF = not on the SPT, first_parent 0xFFFF = none, nh_mask = atoms
 * 0..15.  A job whose result does not fit (a distance >= 0xFFFF on a graph without
 * saturate_at, or more than 16 first-hop atoms) gets HSPF_JS_NARROW and must be re-run through
 * hspf_run_batch.  Graph requirements: fewer than 65535 vertices, link costs <= 65534, no
 * HSPF_VF_LEAF* flags, no HSPF_GF_HOPCOUNT (hspf_graph_info tells); otherwise
 * HSPF_E_UNSUPPORTED.  Any plane pointer may be NULL.
 */
typedef struct hspf_result16 {
    uint16_t *dist;
    uint16_t *hops;
    uint16_t *first_parent;
    uint16_t *n_parents;
    uint16_t *nh_mask;
    uint32_t *job_status;
} hspf_result16;

typedef struct hspf_ctx hspf_ctx;
typedef struct hspf_graph hspf_graph;

/* Create / destroy a context bound to CUDA device `device`. */
int hspf_ctx_create(int device, hspf_ctx **out);
void hspf_ctx_destroy(hspf_ctx *ctx);
/* Last error text of this ctx (never NULL; valid until the next call on ctx). */
const char *hspf_last_error(const hspf_ctx *ctx);

/* Validate `g`, build the transposed CSR and upload both to the device.
 * Returns HSPF_E_NEEDS_ORACLE if a zero-cost edge leaves a HOP vertex. */
int hspf_graph_upload(hspf_ctx *ctx, const hspf_csr *g, hspf_graph **out);
void hspf_graph_free(hspf_ctx *ctx, hspf_graph *g);

/* Run a batch; blocks until results are visible in `out`.  Returns
 * HSPF_E_JOB_STATUS if the batch ran but some job_status is non-zero. */
int hspf_run_batch(hspf_ctx *ctx, const hspf_graph *g, const hspf_jobs *jobs,
                   const hspf_result *out, uint32_t flags);

/* Permanent cost change of existing edges of an uploaded graph (an interface cost change: the structure
 * stands).  Every cost-bearing array of the device image is patched in place on the ctx stream, behind
 * batches already enqueued; the call returns when the patch is done.  edges[]: forward CSR edge indices,
 * costs[]: their new costs.  HSPF_E_UNSUPPORTED when a cost does not fit the image as uploaded (16-bit
 * packing, bucket ring of the fast path, hop-count graphs): free the graph and upload the new CSR.
 * HSPF_E_NEEDS_ORACLE: zero cost out of a HOP vertex.  Nothing is changed on an error. */
int hspf_graph_update_costs(hspf_ctx *ctx, hspf_graph *g, uint32_t n, const uint32_t *edges, const uint32_t *costs);

/* Asynchronous variant used by the benchmark: enqueue on the ctx stream and
 * return; requires HSPF_RUN_DEVICE_PTRS.  hspf_sync() waits for completion. */
int hspf_run_batch_async(hspf_ctx *ctx, const hspf_graph *g,
                         const hspf_jobs *jobs, const hspf_result *out);
int hspf_sync(hspf_ctx *ctx);
/* 16-bit planes (hspf_result16), same contracts as the two calls above. */
int hspf_run_batch16(hspf_ctx *ctx, const hspf_graph *g, const hspf_jobs *jobs,
                     const hspf_result16 *out, uint32_t flags);
int hspf_run_batch16_async(hspf_ctx *ctx, const hspf_graph *g,
                           const hspf_jobs *jobs, const hspf_result16 *out);
/* info = {1 if the packed fast path (and so hspf_run_batch16) serves this graph: packed quad image,
 * no LEAF flags, no hop-count mode, per-job state within the device's shared memory; forward quads,
 * in-quads, log2 of the bucket width, n_vertices, n_edges, largest in-degree, 0}. */
int hspf_graph_info(const hspf_graph *g, uint32_t info[8]);
/* The ctx's cudaStream_t (as void*) so callers can record CUDA events on it. */
void *hspf_stream(hspf_ctx *ctx);
/* Number of kernels this ctx has launched so far (bench `gpu_launches`). */
uint64_t hspf_launch_count(const hspf_ctx *ctx);

/*
 * First-hop atoms.  For a job rooted at `root`, atom a < deg(root) is the a-th
 * CSR out-edge of the root.  Further atoms cover the out-edges of the non-HOP
 * vertices (transit networks / pseudonodes) directly attached to the root: for
 * the j-th root edge whose head N is a non-HOP vertex,
 *   base_j = deg(root) + sum_{i<j, head_i non-HOP} deg(head_i)
 * and atom base_j + k is the k-th out-edge of N (the first such j is used when
 * parallel root->N edges exist).  hspf_atom_decode maps an atom back to
 * (tail vertex, CSR edge index); it only reads the host CSR.
 */
int hspf_atom_decode(const hspf_csr *g, uint32_t root, uint32_t atom,
                     uint32_t *tail, uint32_t *edge);
int hspf_atom_count(const hspf_csr *g, uint32_t root, uint32_t *n_atoms);

/* Leave `n_sms` SMs free in every batch launch of this ctx so that a concurrent kernel on
 * another stream (the NCCL all-gather of the previous batch's results) can run beside
 * the persistent batch kernel.  Default 0. */
int hspf_ctx_reserve_sms(hspf_ctx *ctx, int n_sms);

/* Debug aid: enable/disable per-phase cycle counters of the batch kernel and read
 * the sums of the last launch (SM cycles summed over CTAs).  Slots: 0 init, 1 SSSP,
 * 2 parents, 3 dist write-back, 4 next hops (jump phase) or Kahn push, 5 hops (jump phase) or
 * hops write-back, 6 Kahn rounds, 7 SSSP rounds, 8-11 SSSP round internals (expand, barrier,
 * compaction, barrier), 12 frontier entries, 13-15 jump phase: hop rounds, next-hop rounds,
 * ECMP sweeps (Kahn path: round internals).  `out` may be NULL. */
int hspf_debug_phase_profile(hspf_ctx *ctx, int enable, uint64_t out[16]);

/* Test aid: which kernel the batches of this ctx run.  HSPF_PATH_AUTO (the default) takes the packed
 * fast path wherever it serves the graph (hspf_graph_info) and one next-hop word is asked for;
 * HSPF_PATH_GENERAL always runs the general kernel, HSPF_PATH_GENERAL_KAHN the general kernel
 * without its pointer-jumping next-hop phase.  Every path gives the same planes; 16-bit planes
 * need HSPF_PATH_AUTO. */
#define HSPF_PATH_AUTO 0
#define HSPF_PATH_GENERAL 1
#define HSPF_PATH_GENERAL_KAHN 2
int hspf_debug_set_path(hspf_ctx *ctx, int path);

/* Debug / test aid (host only, no CUDA call): build the quad-space image the fast-path kernel
 * reads (holo_b200/csrc/quad_layout.h) and copy it out.  hdr = {eligible, n_fwd_quads, n_in_quads,
 * bucket shift, longest in-quad chain, largest atom count, 0, 0}.  Call once with NULL arrays to
 * get the sizes: fq/iq [4*quads], fcont [quads/32], slot_of [V], vert_of [fwd quads],
 * imeta [2*in quads], fpos/ipos [E]. */
int hspf_debug_quad_image(const hspf_csr *g, uint32_t hdr[8], uint32_t *fq, uint32_t *fcont, uint16_t *slot_of,
                          uint16_t *vert_of, uint32_t *iq, uint32_t *imeta, uint32_t *fpos, uint32_t *ipos);

/* ---- Multi-GPU result exchange over NVLink peer memory (one process per GPU) --------
 * SURVEY.md §8e / BASELINE north_star: batches larger than one GPU are sharded by root and
 * the per-partition SPT results are all-gathered over NVLink.  The reference has no
 * counterpart (holo-ospf / holo-isis are single-process).
 *
 * Every rank owns `n_buffers` x `world` slots of `slot_bytes`; the batch kernel of rank r
 * writes its result planes into slot r of its own buffer (hspf_xchg_slot), hspf_xchg_push
 * copies that slot to slot r of the same buffer on every peer with the copy engines, and
 * sequence flags travel behind the data.  Waiting and acknowledging use stream memory
 * operations, so no step of the exchange needs an SM and the next batch kernel overlaps it.
 *
 * Per step on buffer k (all ranks, in lockstep):
 *     hspf_xchg_acquire(x, k);            engine stream waits until the previous push(k) has left the
 *                                         device and the local consumer has released buffer k
 *     hspf_run_batch_async(... planes inside hspf_xchg_slot(x, k, rank) ...);
 *     hspf_xchg_push(x, k);
 *     hspf_xchg_wait(x, k);               consumer stream: all `world` slots of buffer k are in
 *     ... consumer work on hspf_xchg_consumer_stream(x) ...
 *     hspf_xchg_release(x, k);            peers may overwrite buffer k again
 * Setup: create (returns this rank's IPC handle), exchange the 64-byte handles between the
 * ranks by any means, attach every peer's handle.  Tear-down: make sure every rank has
 * synced before any rank destroys its exchange (the allocations are mapped by the peers). */
#define HSPF_IPC_HANDLE_BYTES 64
typedef struct hspf_xchg hspf_xchg;
int hspf_xchg_create(hspf_ctx *ctx, int device, uint32_t rank, uint32_t world, size_t slot_bytes,
                     uint32_t n_buffers, hspf_xchg **out, uint8_t handle[HSPF_IPC_HANDLE_BYTES]);
int hspf_xchg_attach(hspf_xchg *x, uint32_t peer_rank, const uint8_t handle[HSPF_IPC_HANDLE_BYTES]);
/* Same-process peers (two contexts on one device, or devices with peer access): attach by the
 * base pointer hspf_xchg_base() of the peer's exchange instead of an IPC handle. */
int hspf_xchg_attach_ptr(hspf_xchg *x, uint32_t peer_rank, void *peer_base);
void *hspf_xchg_base(hspf_xchg *x);
/* Only the first nbytes of the own slot travel in hspf_xchg_push (0 = the whole slot): lay the
 * planes the consumers need first.  Sequence numbers are 32 bits: no limit on the number of pushes. */
int hspf_xchg_set_push_bytes(hspf_xchg *x, size_t nbytes);
/* Fused exchange: the batch kernel stores the planes the consumers need (16-bit dist, hops,
 * nh_mask; job status) into this rank's slot on every peer while it computes, over NVLink, and
 * only the sequence flags travel afterwards.  Per step on buffer k:
 *     hspf_xchg_acquire_direct(x, k);     as acquire, and every peer has released this rank's slot
 *     hspf_xchg_peer_deltas(x, k, d, &n); hspf_ctx_set_peer_slots(ctx, n, d);
 *     hspf_run_batch16_async(... planes inside hspf_xchg_slot(x, k, rank) ...);
 *     hspf_ctx_set_peer_slots(ctx, 0, NULL);
 *     hspf_xchg_publish(x, k);            flags behind the kernel
 *     hspf_xchg_wait / consumer work / hspf_xchg_release as before.
 * deltas[]: room for world - 1 entries; at most 7 peers.  first_parent / n_parents stay local. */
int hspf_xchg_acquire_direct(hspf_xchg *x, uint32_t buffer);
int hspf_xchg_peer_deltas(hspf_xchg *x, uint32_t buffer, int64_t *deltas, uint32_t *n_peers);
int hspf_xchg_publish(hspf_xchg *x, uint32_t buffer);
int hspf_ctx_set_peer_slots(hspf_ctx *ctx, uint32_t n_peers, const int64_t *deltas);
void *hspf_xchg_slot(hspf_xchg *x, uint32_t buffer, uint32_t slot);   /* device pointer, local copy */
size_t hspf_xchg_slot_bytes(const hspf_xchg *x);                      /* slot_bytes rounded up to 256 */
int hspf_xchg_acquire(hspf_xchg *x, uint32_t buffer);
int hspf_xchg_push(hspf_xchg *x, uint32_t buffer);
int hspf_xchg_wait(hspf_xchg *x, uint32_t buffer);
int hspf_xchg_release(hspf_xchg *x, uint32_t buffer);
void *hspf_xchg_consumer_stream(hspf_xchg *x);                        /* cudaStream_t */
int hspf_xchg_sync(hspf_xchg *x);                                     /* host blocks: pushes + consumer done */
const char *hspf_xchg_last_error(const hspf_xchg *x);
int hspf_xchg_destroy(hspf_xchg *x);

/* Library build info, e.g. "holo_spf 0.1 sm_100a". */
const char *hspf_version(void);

#ifdef __cplusplus
}
#endif
#endif /* HOLO_SPF_H */
