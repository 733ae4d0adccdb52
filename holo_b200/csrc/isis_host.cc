// isis_host.cc — IS-IS host side of the engine: level LSDB image -> CSR, and device
// result planes -> the reference's Spt (vertices with ordered ECMP parents, next-hop
// Vecs, first/second hops).
//
// The LSDB walk the reference repeats for every visited edge (vertex_edges over up
// to 256 fragments x 4 TLV kinds, plus the mutual-link re-iteration,
// holo-isis/src/spf.rs:605-625,1005-1120) happens here once; the per-vertex transit
// gates (missing zeroth LSP, overload bit, protocols-supported, spf.rs:556-602)
// become vertex flags.  Distances / hops / first-hop sets come from the CUDA kernel
// (hspf_run_batch); this file only orders what the kernel found the way the
// reference's pop order would have (parents: spf.rs:675, nexthops: spf.rs:678-702).
#include <algorithm>
#include <cstring>
#include <new>
#include <unordered_map>
#include <unordered_set>
#include <vector>

#include "holo_spf_lsdb.h"
#include "spf_one_root.h"

namespace {
constexpr uint32_t kNone = 0xFFFFFFFFu;
constexpr uint32_t kMaxWide = 0xFE000000u;
inline bool is_pn(hl_lan_id id) { return (id & 0xFF) != 0; }
}  // namespace

struct hspf_isis_flat {
    const hl_isis_level *lvl = nullptr;
    std::vector<hl_lan_id> ids;                 // [V] in VertexId order
    std::vector<uint32_t> row, col, cost;
    std::vector<uint8_t> vflags;
    std::vector<uint32_t> irow, isrc, ieid;     // transposed (host copy)
    std::unordered_map<uint64_t, uint32_t> index;
    uint32_t reject_above = 0, gflags = 0;
};

namespace {

int flatten(const hl_isis_level *l, hspf_isis_flat &f) {
    f.lvl = l;
    const bool mt_none = l->mt_id == HL_ISIS_MT_NONE, mt_std = l->mt_id == HL_ISIS_MT_STANDARD;
    const bool std_en = l->metric_type == HL_ISIS_METRIC_STANDARD || l->metric_type == HL_ISIS_METRIC_BOTH;
    const bool wide_en = l->metric_type == HL_ISIS_METRIC_WIDE || l->metric_type == HL_ISIS_METRIC_BOTH;
    const bool hopcount = l->metric_mode == HL_ISIS_MODE_HOPCOUNT;
    auto valid = [&](const hl_isis_lsp &p) { return p.seqno != 0 && p.rem_lifetime != 0; };

    // fragments in LspId order
    std::vector<uint32_t> order(l->n_lsps);
    for (uint32_t i = 0; i < l->n_lsps; ++i) order[i] = i;
    std::stable_sort(order.begin(), order.end(), [&](uint32_t a, uint32_t b) {
        const auto &x = l->lsps[a], &y = l->lsps[b];
        return x.lan_id != y.lan_id ? x.lan_id < y.lan_id : x.fragment < y.fragment;
    });
    // vertices: every LAN id owning at least one valid fragment
    std::vector<hl_lan_id> pn, rt;
    for (uint32_t i : order) {
        const auto &p = l->lsps[i];
        if (!valid(p)) continue;
        auto &dst = is_pn(p.lan_id) ? pn : rt;
        if (dst.empty() || dst.back() != p.lan_id) dst.push_back(p.lan_id);
    }
    f.ids = pn;
    f.ids.insert(f.ids.end(), rt.begin(), rt.end());
    const uint32_t V = (uint32_t)f.ids.size();
    for (uint32_t v = 0; v < V; ++v) f.index.emplace(f.ids[v], v);
    f.vflags.assign(V, 0);
    std::vector<uint8_t> has_zeroth(V, 0);
    for (uint32_t v = 0; v < V; ++v) if (!is_pn(f.ids[v])) f.vflags[v] |= HSPF_VF_HOP;

    struct Raw { uint32_t u, v, cost; };
    std::vector<Raw> raw;
    raw.reserve(l->n_reaches);
    auto ecost = [&](hl_lan_id nbr, uint32_t metric) { return hopcount ? (is_pn(nbr) ? 0u : 1u) : metric; };
    for (uint32_t i : order) {
        const auto &p = l->lsps[i];
        if (!valid(p)) continue;
        const uint32_t u = f.index[p.lan_id];
        if (p.fragment == 0) {
            has_zeroth[u] = 1;
            if (!is_pn(p.lan_id)) {
                // overload bit: skipped unless root (spf.rs:566-572), only with an MT id
                if (!mt_none) {
                    const bool ol = mt_std ? (p.flags & HL_LSPF_OL) : (p.flags & HL_LSPF_MT_IPV6_OL);
                    if (ol) f.vflags[u] |= HSPF_VF_LEAF_UNLESS_ROOT;
                }
                // protocols-supported gate (spf.rs:580-602), standard topology only
                if (mt_std) {
                    bool ok = p.flags & HL_LSPF_HAS_PROTOCOLS;
                    if (ok && l->ipv4_enabled && !(p.flags & HL_LSPF_NLPID_IPV4)) ok = false;
                    if (ok && l->ipv6_enabled && !(p.flags & HL_LSPF_NLPID_IPV6)) ok = false;
                    if (!ok) f.vflags[u] |= HSPF_VF_LEAF;
                }
            }
        }
        const hl_isis_reach *re = l->reaches + p.reach_off;
        auto emit = [&](const hl_isis_reach &r) {
            auto it = f.index.find(r.neighbor);
            if (it == f.index.end()) return;       // no LSP: the mutual check can never pass
            raw.push_back({u, it->second, ecost(r.neighbor, r.metric)});
        };
        if ((mt_none || mt_std) && std_en)
            for (uint32_t k = 0; k < p.n_reach; ++k) if (re[k].kind == HL_ISIS_REACH_LEGACY) emit(re[k]);
        if (((mt_none || mt_std) || is_pn(p.lan_id)) && wide_en)
            for (uint32_t k = 0; k < p.n_reach; ++k)
                if (re[k].kind == HL_ISIS_REACH_EXT && re[k].metric < kMaxWide) emit(re[k]);
        if (!mt_none && !mt_std)
            for (uint32_t k = 0; k < p.n_reach; ++k)
                if (re[k].kind == HL_ISIS_REACH_MT && re[k].mt_id == l->mt_id && re[k].metric < kMaxWide) emit(re[k]);
        if (mt_none)
            for (uint32_t k = 0; k < p.n_reach; ++k)
                if (re[k].kind == HL_ISIS_REACH_MT && re[k].metric < kMaxWide) emit(re[k]);
    }
    for (uint32_t v = 0; v < V; ++v) if (!has_zeroth[v]) f.vflags[v] |= HSPF_VF_LEAF;

    // mutual-link filter; raw is grouped by u in iteration order (fragments of one
    // LAN id are contiguous in LspId order)
    std::unordered_set<uint64_t> have;
    have.reserve(raw.size() * 2);
    for (auto &e : raw) have.insert(((uint64_t)e.u << 32) | e.v);
    auto keep = [&](const Raw &e) {
        if (e.u == e.v) return false;
        // a link between two pseudonodes can never be mutual-checked into the SPT in
        // a sane LSDB; the engine's CSR forbids it, so drop it
        if (!(f.vflags[e.u] & HSPF_VF_HOP) && !(f.vflags[e.v] & HSPF_VF_HOP)) return false;
        return have.count(((uint64_t)e.v << 32) | e.u) != 0;
    };
    f.row.assign(V + 1, 0);
    for (auto &e : raw) if (keep(e)) f.row[e.u + 1]++;
    for (uint32_t v = 0; v < V; ++v) f.row[v + 1] += f.row[v];
    const uint32_t E = f.row[V];
    f.col.resize(E); f.cost.resize(E);
    std::vector<uint32_t> fill(f.row.begin(), f.row.end() - 1);
    for (auto &e : raw) if (keep(e)) { const uint32_t k = fill[e.u]++; f.col[k] = e.v; f.cost[k] = e.cost; }
    // transposed copy for the host-side ordering passes
    f.irow.assign(V + 1, 0);
    for (uint32_t e = 0; e < E; ++e) f.irow[f.col[e] + 1]++;
    for (uint32_t v = 0; v < V; ++v) f.irow[v + 1] += f.irow[v];
    f.isrc.resize(E); f.ieid.resize(E);
    std::vector<uint32_t> ifill(f.irow.begin(), f.irow.end() - 1);
    for (uint32_t u = 0; u < V; ++u)
        for (uint32_t e = f.row[u]; e < f.row[u + 1]; ++e) { const uint32_t k = ifill[f.col[e]]++; f.isrc[k] = u; f.ieid[k] = e; }
    f.reject_above = l->metric_type == HL_ISIS_METRIC_STANDARD ? 1023u : kMaxWide;
    f.gflags = HSPF_GF_NOHOP_TARGET_NO_NEXTHOP | (hopcount ? HSPF_GF_HOPCOUNT : 0u);
    return HSPF_OK;
}

void fill_csr(const hspf_isis_flat &f, hspf_csr *c) {
    std::memset(c, 0, sizeof(*c));
    c->n_vertices = (uint32_t)f.ids.size();
    c->n_edges = (uint32_t)f.col.size();
    c->row_ptr = f.row.data(); c->col = f.col.data(); c->cost = f.cost.data(); c->vflags = f.vflags.data();
    c->reject_above = f.reject_above;
    c->saturate_at = 0;
    c->flags = f.gflags;
    c->delta = 0;
}

inline bool expands(uint8_t fl, uint32_t u, uint32_t root) {
    return !((fl & HSPF_VF_LEAF) || ((fl & HSPF_VF_LEAF_UNLESS_ROOT) && u != root));
}

int spt_from_planes(const hspf_isis_flat &f, uint32_t root, const uint32_t *dist, const uint16_t *hops,
                    uint32_t n_ov, const uint32_t *ov_edge, const uint32_t *ov_cost, hl_isis_spt *out) {
    const uint32_t V = (uint32_t)f.ids.size();
    const bool hopcount = f.gflags & HSPF_GF_HOPCOUNT;
    auto ecost = [&](uint32_t e) {
        uint32_t c = f.cost[e];
        for (uint32_t k = 0; k < n_ov; ++k) if (ov_edge[k] == e) c = ov_cost[k];
        return c;
    };
    auto is_dag = [&](uint32_t u, uint32_t e, uint32_t v) {
        if (v == root || dist[u] == HSPF_DIST_INF || dist[v] == HSPF_DIST_INF) return false;
        if (!expands(f.vflags[u], u, root)) return false;
        const uint32_t c = ecost(e);
        if (c == HSPF_COST_DISABLED) return false;
        const uint64_t s = (uint64_t)dist[u] + c;
        return s == dist[v];
    };
    // hop-count mode: a pseudonode's only parent is its lowest-numbered router of the same level
    std::vector<uint32_t> owner;
    if (hopcount) {
        owner.assign(V, kNone);
        for (uint32_t v = 0; v < V; ++v) {
            if ((f.vflags[v] & HSPF_VF_HOP) || dist[v] == HSPF_DIST_INF) continue;
            for (uint32_t i = f.irow[v]; i < f.irow[v + 1]; ++i)
                if (is_dag(f.isrc[i], f.ieid[i], v)) owner[v] = std::min(owner[v], f.isrc[i]);
        }
    }
    // pop order
    std::vector<uint32_t> spt;
    for (uint32_t v = 0; v < V; ++v) if (dist[v] != HSPF_DIST_INF) spt.push_back(v);
    std::vector<uint32_t> pop = spt;
    auto key = [&](uint32_t v) {
        // (distance, tie): plain VertexId order, or the interleaved hop-count order
        uint64_t tie = v;
        if (hopcount) tie = (f.vflags[v] & HSPF_VF_HOP) ? ((uint64_t)v << 33) : (((uint64_t)owner[v] << 33) | (1ull << 32) | v);
        return std::make_pair(dist[v], tie);
    };
    std::sort(pop.begin(), pop.end(), [&](uint32_t a, uint32_t b) { return key(a) < key(b); });
    std::vector<uint32_t> pos(V, kNone), rank(V, kNone);
    for (uint32_t i = 0; i < pop.size(); ++i) pos[pop[i]] = i;
    for (uint32_t i = 0; i < spt.size(); ++i) rank[spt[i]] = i;

    // parents in push order: by (pop position of the tail, edge order of the tail)
    std::vector<std::vector<uint32_t>> parents(V);
    size_t n_par = 0;
    std::vector<std::pair<uint64_t, uint32_t>> tmp;
    for (uint32_t v : spt) {
        tmp.clear();
        for (uint32_t i = f.irow[v]; i < f.irow[v + 1]; ++i) {
            const uint32_t u = f.isrc[i], e = f.ieid[i];
            if (!is_dag(u, e, v)) continue;
            if (hopcount && !(f.vflags[v] & HSPF_VF_HOP) && u != owner[v]) continue;
            tmp.emplace_back(((uint64_t)pos[u] << 32) | e, u);
        }
        std::sort(tmp.begin(), tmp.end());
        for (auto &t : tmp) parents[v].push_back(t.second);
        n_par += tmp.size();
    }
    // next-hop Vecs in pop order
    std::vector<std::vector<uint64_t>> nh(V);
    size_t n_nh = 0;
    const size_t cap = (size_t)1 << 22;
    for (uint32_t v : pop) {
        auto &dst = nh[v];
        for (uint32_t p : parents[v]) {
            if (hops[p] == 0) {
                if (f.vflags[v] & HSPF_VF_HOP) dst.push_back(f.ids[v] >> 8);
            } else {
                if (n_nh + dst.size() + nh[p].size() > cap) return HSPF_E_UNSUPPORTED;
                dst.insert(dst.end(), nh[p].begin(), nh[p].end());
            }
        }
        n_nh += dst.size();
    }
    std::vector<uint32_t> fh, sh;
    for (uint32_t v : pop) {
        if (!(f.vflags[v] & HSPF_VF_HOP)) continue;
        if (hops[v] == 1) fh.push_back(rank[v]);
        if (hops[v] == 2) sh.push_back(rank[v]);
    }
    out->n_vertices = (uint32_t)spt.size();
    out->n_parents = (uint32_t)n_par;
    out->n_nexthops = (uint32_t)n_nh;
    out->n_first_hops = (uint32_t)fh.size();
    out->n_second_hops = (uint32_t)sh.size();
    if (out->n_vertices > out->vertices_cap || out->n_parents > out->parents_cap ||
        out->n_nexthops > out->nexthops_cap || out->n_first_hops > out->first_hops_cap ||
        out->n_second_hops > out->second_hops_cap)
        return HSPF_E_NOMEM;
    uint32_t i = 0, p = 0, n = 0;
    for (uint32_t v : spt) {
        hl_isis_vertex o{};
        o.lan_id = f.ids[v]; o.distance = dist[v]; o.hops = hops[v];
        o.par_off = p; o.n_par = (uint32_t)parents[v].size();
        o.nh_off = n; o.n_nh = (uint32_t)nh[v].size();
        for (uint32_t u : parents[v]) out->parents[p++] = rank[u];
        for (uint64_t x : nh[v]) out->nexthops[n++] = x;
        out->vertices[i++] = o;
    }
    std::copy(fh.begin(), fh.end(), out->first_hops);
    std::copy(sh.begin(), sh.end(), out->second_hops);
    return HSPF_OK;
}

}  // namespace

extern "C" {

int hspf_isis_flatten(const hl_isis_level *lvl, hspf_isis_flat **out) {
    if (!lvl || !out) return HSPF_E_INVAL;
    *out = nullptr;
    try {
        auto *f = new hspf_isis_flat();
        int rc = flatten(lvl, *f);
        if (rc) { delete f; return rc; }
        *out = f;
        return HSPF_OK;
    } catch (const std::bad_alloc &) { return HSPF_E_NOMEM; } catch (...) { return HSPF_E_INVAL; }
}

void hspf_isis_flat_free(hspf_isis_flat *flat) { delete flat; }

int hspf_isis_flat_csr(const hspf_isis_flat *flat, hspf_csr *out) {
    if (!flat || !out) return HSPF_E_INVAL;
    fill_csr(*flat, out);
    return HSPF_OK;
}

int hspf_isis_spf_type(const hl_isis_level *ol, const hl_isis_level *nl, const hl_isis_lsp_trigger *tr, uint32_t n,
                       uint32_t *spf_type) {
    if (!ol || !nl || !spf_type || (n && !tr)) return HSPF_E_INVAL;
    auto find = [](const hl_isis_level *l, hl_lan_id id, uint8_t frag) -> const hl_isis_lsp * {
        for (uint32_t i = 0; i < l->n_lsps; ++i)
            if (l->lsps[i].lan_id == id && l->lsps[i].fragment == frag) return &l->lsps[i];
        return nullptr;
    };
    // the IS-reachability entries of one TLV kind, in TLV order
    auto same_kind = [](const hl_isis_level *a, const hl_isis_lsp *x, const hl_isis_level *b, const hl_isis_lsp *y, uint8_t kind) {
        uint32_t i = 0, j = 0;
        for (;;) {
            while (i < x->n_reach && a->reaches[x->reach_off + i].kind != kind) ++i;
            while (j < y->n_reach && b->reaches[y->reach_off + j].kind != kind) ++j;
            if (i == x->n_reach || j == y->n_reach) return i == x->n_reach && j == y->n_reach;
            const hl_isis_reach &p = a->reaches[x->reach_off + i], &q = b->reaches[y->reach_off + j];
            if (p.neighbor != q.neighbor || p.metric != q.metric) return false;
            ++i; ++j;
        }
    };
    *spf_type = HL_ISIS_SPF_ROUTE_ONLY;
    for (uint32_t k = 0; k < n; ++k) {
        const hl_isis_lsp *x = find(ol, tr[k].lan_id, tr[k].fragment), *y = find(nl, tr[k].lan_id, tr[k].fragment);
        if (!y) return HSPF_E_INVAL;                         // a trigger is an LSP that was just installed
        bool topology_change = true;
        // lsp.flags (LspFlags: the image carries its OL and ATT bits; the other image flags come from TLVs, which the
        // reference does not compare here)
        const uint8_t hdr_bits = HL_LSPF_OL | HL_LSPF_ATT;
        if (x && (x->rem_lifetime == 0) == (y->rem_lifetime == 0) && (x->flags & hdr_bits) == (y->flags & hdr_bits) &&
            same_kind(ol, x, nl, y, HL_ISIS_REACH_LEGACY) && same_kind(ol, x, nl, y, HL_ISIS_REACH_EXT))
            topology_change = false;
        if (topology_change) { *spf_type = HL_ISIS_SPF_FULL; break; }
    }
    return HSPF_OK;
}

int hspf_isis_flat_update(hspf_isis_flat *flat, const hl_isis_level *nl, uint32_t *kind, uint32_t *edges, uint32_t *costs,
                          uint32_t cap, uint32_t *n_changed) {
    if (!flat || !nl || !kind || !n_changed) return HSPF_E_INVAL;
    try {
        *n_changed = 0;
        hspf_isis_flat fresh;
        const int rc = flatten(nl, fresh);
        if (rc) return rc;
        hspf_isis_flat &f = *flat;
        const bool same_graph = f.ids == fresh.ids && f.row == fresh.row && f.col == fresh.col && f.vflags == fresh.vflags &&
                                f.reject_above == fresh.reject_above && f.gflags == fresh.gflags;
        if (!same_graph) {
            f = std::move(fresh);
            *kind = HSPF_FLAT_REBUILT;
            return HSPF_OK;
        }
        uint32_t changed = 0;
        for (uint32_t e = 0; e < (uint32_t)f.cost.size(); ++e) {
            if (f.cost[e] == fresh.cost[e]) continue;
            if (changed < cap && edges && costs) { edges[changed] = e; costs[changed] = fresh.cost[e]; }
            ++changed;
        }
        f.cost = std::move(fresh.cost);
        f.lvl = nl;
        *n_changed = changed;
        *kind = changed ? HSPF_FLAT_COSTS : HSPF_FLAT_UNCHANGED;
        return changed > cap ? HSPF_E_NOMEM : HSPF_OK;
    } catch (const std::bad_alloc &) { return HSPF_E_NOMEM; } catch (...) { return HSPF_E_INVAL; }
}

int hspf_isis_flat_vertices(const hspf_isis_flat *flat, const uint64_t **lan_ids, uint32_t *n_vertices) {
    if (!flat) return HSPF_E_INVAL;
    if (lan_ids) *lan_ids = flat->ids.data();
    if (n_vertices) *n_vertices = (uint32_t)flat->ids.size();
    return HSPF_OK;
}

uint32_t hspf_isis_flat_vertex(const hspf_isis_flat *flat, uint64_t lan_id) {
    if (!flat) return kNone;
    auto it = flat->index.find(lan_id);
    return it == flat->index.end() ? kNone : it->second;
}

int hspf_isis_spt_from_planes(const hspf_isis_flat *flat, uint32_t root_vertex, const uint32_t *dist,
                              const uint16_t *hops, uint32_t n_ov, const uint32_t *ov_edge,
                              const uint32_t *ov_cost, hl_isis_spt *out) {
    if (!flat || !dist || !hops || !out || root_vertex >= flat->ids.size()) return HSPF_E_INVAL;
    try {
        return spt_from_planes(*flat, root_vertex, dist, hops, n_ov, ov_edge, ov_cost, out);
    } catch (const std::bad_alloc &) { return HSPF_E_NOMEM; } catch (...) { return HSPF_E_INVAL; }
}

int hspf_isis_compute_spt(hspf_ctx *ctx, const hl_isis_level *lvl, uint64_t root_system_id, hl_isis_spt *out) {
    if (!ctx || !lvl || !out) return HSPF_E_INVAL;
    try {
        hspf_isis_flat f;
        int rc = flatten(lvl, f);
        if (rc) return rc;
        const hl_lan_id root_id = (hl_lan_id)(root_system_id << 8);
        auto it = f.index.find(root_id);
        if (it == f.index.end()) {
            // the root owns no LSP: the SPT is the root alone (popped, zeroth LSP missing)
            out->n_vertices = 1; out->n_parents = out->n_nexthops = out->n_first_hops = out->n_second_hops = 0;
            if (out->vertices_cap < 1) return HSPF_E_NOMEM;
            hl_isis_vertex o{};
            o.lan_id = root_id;
            out->vertices[0] = o;
            return HSPF_OK;
        }
        const uint32_t root = it->second;
        hspf_csr csr;
        fill_csr(f, &csr);
        hspf::OneRootPlanes p;
        rc = hspf::run_one_root(ctx, csr, root, 4, false, p);
        // first-hop atom overflow is irrelevant here: the Vec is rebuilt from parents
        if (rc == HSPF_E_JOB_STATUS && !(p.status & ~HSPF_JS_TOO_MANY_ATOMS)) rc = HSPF_OK;
        if (rc) return rc;
        return spt_from_planes(f, root, p.dist.data(), p.hops.data(), 0, nullptr, nullptr, out);
    } catch (const std::bad_alloc &) { return HSPF_E_NOMEM; } catch (...) { return HSPF_E_INVAL; }
}

}  // extern "C"

// =====================================================================================
// Route path of compute_spf (holo-isis/src/spf.rs:742-799): per enabled topology one
// SPT with `local = true` next-hop resolution (resolve_nexthop, spf.rs:948-1002), then
// compute_routes (spf.rs:838-941).  Distances/hops come from the device; the host
// replays only the first-hop bookkeeping of the hops==0 vertices (root and the
// pseudonodes attached to it) in pop order, because resolve_nexthop is stateful
// ("the same adjacency shouldn't be used more than once", used_adjs).
// =====================================================================================
#include <array>
#include <map>
#include <set>

namespace {

struct LNh { uint64_t sysid; bool has_iface; uint32_t iface; bool has4; uint32_t ipv4; bool has6; hl_ip_addr ipv6; };

struct IpLess {
    bool operator()(const hl_ip_addr &a, const hl_ip_addr &b) const {
        if (a.is_v6 != b.is_v6) return a.is_v6 < b.is_v6;
        return std::memcmp(a.bytes, b.bytes, 16) < 0;
    }
};
struct NetKey {
    hl_ip_addr a; uint8_t len;
    bool operator<(const NetKey &o) const {
        if (a.is_v6 != o.a.is_v6) return a.is_v6 < o.a.is_v6;
        int c = std::memcmp(a.bytes, o.a.bytes, 16);
        return c ? c < 0 : len < o.len;
    }
};
struct RNh { uint64_t sysid; uint32_t iface; hl_ip_addr addr; bool has_label = false; uint32_t label = 0; };
struct PrefixSid { bool present = false; uint8_t flags = 0; bool is_label = false; uint32_t value = 0; };
struct RouteE {
    uint8_t type, flags; uint32_t metric; std::map<hl_ip_addr, RNh, IpLess> nh;
    PrefixSid psid;                               // Route.prefix_sid (route.rs:100)
    bool has_label = false; uint32_t label = 0;   // Route.sr_label
};

// SR view of one level's LSDB (holo-isis/src/sr.rs): per system the label blocks and address
// family flags of its first valid SR-Capabilities sub-TLV, per LAN id whether a valid fragment
// lists SPF in an SR-Algorithm sub-TLV.  Built once per route computation.
struct SrView {
    struct Cap { const hl_srgb *blocks; uint32_t n; uint8_t flags; };
    std::unordered_map<uint64_t, Cap> cap;          // system id -> capabilities
    std::unordered_map<uint64_t, bool> algo_spf;    // LAN id -> SR-Algorithm contains SPF
    explicit SrView(const hl_isis_level &l) {
        // LspId order: (lan_id, fragment); the first valid LSP with the sub-TLV wins
        std::vector<uint32_t> order(l.n_lsps);
        for (uint32_t i = 0; i < l.n_lsps; ++i) order[i] = i;
        std::stable_sort(order.begin(), order.end(), [&](uint32_t a, uint32_t b) {
            const auto &x = l.lsps[a], &y = l.lsps[b];
            return x.lan_id != y.lan_id ? x.lan_id < y.lan_id : x.fragment < y.fragment;
        });
        for (uint32_t i : order) {
            const auto &p = l.lsps[i];
            if (!p.seqno || !p.rem_lifetime) continue;
            if (p.sr_flags & HL_LSP_SR_ALGO_SPF) algo_spf[p.lan_id] = true;
            if ((p.sr_flags & HL_LSP_SR_HAS_CAP) && !cap.count(p.lan_id >> 8))
                cap.emplace(p.lan_id >> 8, Cap{l.srgbs + p.srgb_off, p.n_srgb, p.sr_flags});
        }
    }
    // index_to_label (sr.rs:268-300)
    static bool label_of(const Cap &c, uint32_t index, uint32_t &label) {
        for (uint32_t i = 0; i < c.n; ++i) {
            if (c.blocks[i].first_is_index) continue;
            if (index >= c.blocks[i].range) { index -= c.blocks[i].range; continue; }
            label = c.blocks[i].first + index;
            return true;
        }
        return false;
    }
    // prefix_sid_update (sr.rs:33-99) with prefix_sid_input_label / prefix_sid_output_label
    void update(RouteE &r, uint64_t own_system, uint64_t adv_lan_id, bool v6, bool local, bool last_hop) const {
        const PrefixSid &ps = r.psid;
        auto al = algo_spf.find(adv_lan_id);
        if (al == algo_spf.end()) return;                 // remote node does not run SPF for SR
        const bool p_flag = ps.flags & HL_ISIS_PSID_P, e_flag = ps.flags & HL_ISIS_PSID_E;
        if (local && (!p_flag || e_flag)) {
            r.has_label = false;
        } else if (ps.is_label) {
            r.has_label = true; r.label = ps.value;
        } else {
            auto own = cap.find(own_system);
            uint32_t lab;
            if (own != cap.end() && label_of(own->second, ps.value, lab)) { r.has_label = true; r.label = lab; }
        }
        for (auto &kv : r.nh) {
            RNh &nh = kv.second;
            if (last_hop && !p_flag) { nh.has_label = true; nh.label = 3; continue; }                 // implicit null
            auto c = cap.find(nh.sysid);
            if (c == cap.end()) continue;
            if (!(c->second.flags & (v6 ? HL_LSP_SR_CAP_V : HL_LSP_SR_CAP_I))) continue;
            if (last_hop && e_flag) { nh.has_label = true; nh.label = v6 ? 2u : 0u; continue; }      // explicit null
            uint32_t lab;
            if (ps.is_label) { nh.has_label = true; nh.label = last_hop ? ps.value : 3u; }
            else if (label_of(c->second, ps.value, lab)) { nh.has_label = true; nh.label = lab; }
        }
    }
};

// Next-hop Vecs of a `local = true` SPT for every SPT vertex (indexed by vertex).
int local_nexthops(const hspf_isis_flat &f, const hl_isis_instance *in, uint8_t mt_id, uint32_t root,
                   const uint32_t *dist, const uint16_t *hops, std::vector<std::vector<LNh>> &out) {
    const uint32_t V = (uint32_t)f.ids.size();
    const uint8_t level_bit = in->level == 1 ? 1 : 2;
    // pop order
    std::vector<uint32_t> pop;
    for (uint32_t v = 0; v < V; ++v) if (dist[v] != HSPF_DIST_INF) pop.push_back(v);
    std::sort(pop.begin(), pop.end(), [&](uint32_t a, uint32_t b) { return dist[a] != dist[b] ? dist[a] < dist[b] : a < b; });
    std::vector<uint32_t> pos(V, kNone);
    for (uint32_t i = 0; i < pop.size(); ++i) pos[pop[i]] = i;
    auto relax_ok = [&](uint32_t u, uint32_t e) {     // would the reference relax this edge at all?
        if (dist[u] == HSPF_DIST_INF || !expands(f.vflags[u], u, root)) return false;
        return (uint64_t)dist[u] + f.cost[e] <= f.reject_above;
    };
    std::set<std::array<uint8_t, 6>> used;
    auto resolve = [&](uint32_t P, uint32_t e, uint32_t R) {
        LNh nh{f.ids[R] >> 8, false, 0, false, 0, false, hl_ip_addr{}};
        const bool want_bcast = is_pn(f.ids[P]);
        for (uint32_t i = 0; i < in->n_ifaces; ++i) {
            const auto &iface = in->ifaces[i];
            if ((bool)iface.is_broadcast != want_bcast) continue;
            const hl_isis_adj *adj = nullptr;
            if (iface.is_broadcast) {
                for (uint32_t k = 0; k < iface.n_adj && !adj; ++k)
                    if (in->adjs[iface.adj_off + k].system_id == nh.sysid) adj = &in->adjs[iface.adj_off + k];
                if (adj && (!(mt_id == HL_ISIS_MT_STANDARD ? adj->topo_std : adj->topo_ipv6) || !adj->up)) adj = nullptr;
            } else {
                if (iface.metric != f.cost[e] || !iface.n_adj) continue;
                const auto &a = in->adjs[iface.adj_off];
                if ((mt_id == HL_ISIS_MT_STANDARD ? a.topo_std : a.topo_ipv6) && (a.level_usage & level_bit) &&
                    a.system_id == nh.sysid && a.up)
                    adj = &a;
            }
            if (!adj) continue;
            std::array<uint8_t, 6> snpa;
            std::memcpy(snpa.data(), adj->snpa, 6);
            if (!used.insert(snpa).second) continue;
            nh.has_iface = true; nh.iface = i;
            nh.has4 = adj->has_ipv4; nh.ipv4 = adj->ipv4;
            nh.has6 = adj->has_ipv6; nh.ipv6 = adj->ipv6;
            break;
        }
        return nh;
    };
    // replay the relaxations out of the hops==0 vertices, in pop order
    std::map<uint32_t, LNh> first_hop;    // forward edge id -> resolved next hop (final DAG edges only)
    for (uint32_t P : pop) {
        if (hops[P] != 0 || !expands(f.vflags[P], P, root)) continue;
        for (uint32_t e = f.row[P]; e < f.row[P + 1]; ++e) {
            const uint32_t R = f.col[e];
            if (pos[R] != kNone && pos[R] < pos[P]) continue;            // already on the SPT
            const uint64_t d = (uint64_t)dist[P] + f.cost[e];
            if (d > f.reject_above) continue;
            // candidate distance of R at this moment
            uint64_t cb = ~0ull;
            for (uint32_t i = f.irow[R]; i < f.irow[R + 1]; ++i) {
                const uint32_t u = f.isrc[i], e2 = f.ieid[i];
                if (!relax_ok(u, e2)) continue;
                const bool earlier = (u == P) ? (e2 < e) : (pos[u] < pos[P]);
                if (earlier) cb = std::min<uint64_t>(cb, (uint64_t)dist[u] + f.cost[e2]);
            }
            if (d > cb) continue;
            if (!(f.vflags[R] & HSPF_VF_HOP)) continue;                  // pseudonode: nothing is pushed
            LNh nh = resolve(P, e, R);
            if (d == dist[R]) first_hop[e] = nh;
        }
    }
    // final Vecs in pop order: parents in (pop position, edge order)
    out.assign(V, {});
    std::vector<std::pair<uint64_t, uint32_t>> tmp;
    for (uint32_t v : pop) {
        if (v == root) continue;
        tmp.clear();
        for (uint32_t i = f.irow[v]; i < f.irow[v + 1]; ++i) {
            const uint32_t u = f.isrc[i], e = f.ieid[i];
            if (!relax_ok(u, e) || (uint64_t)dist[u] + f.cost[e] != dist[v]) continue;
            tmp.emplace_back(((uint64_t)pos[u] << 32) | e, u);
        }
        std::sort(tmp.begin(), tmp.end());
        for (auto &t : tmp) {
            const uint32_t u = t.second, e = (uint32_t)(t.first & 0xFFFFFFFFu);
            if (hops[u] == 0) {
                if (f.vflags[v] & HSPF_VF_HOP) {
                    auto it = first_hop.find(e);
                    if (it != first_hop.end()) out[v].push_back(it->second);
                }
            } else {
                if (out[v].size() + out[u].size() > ((size_t)1 << 22)) return HSPF_E_UNSUPPORTED;
                out[v].insert(out[v].end(), out[u].begin(), out[u].end());
            }
        }
    }
    return HSPF_OK;
}

}  // namespace

namespace {

// One topology of compute_spf's route path: flatten with the topology's edge rules and find
// the root.  Returns HSPF_OK and `have_root`.
int topology_flat(const hl_isis_instance *in, uint8_t mt_id, hspf_isis_flat &f, uint32_t &root, bool &have_root) {
    hl_isis_level l = in->lvl;
    l.mt_id = mt_id;
    l.metric_mode = HL_ISIS_MODE_NORMAL;
    int rc = flatten(&l, f);
    if (rc) return rc;
    const hl_lan_id root_id = (hl_lan_id)(in->system_id << 8);
    auto it = f.index.find(root_id);
    have_root = it != f.index.end();      // root owns no LSP: nothing reachable, no routes
    root = have_root ? it->second : 0;
    return HSPF_OK;
}

// compute_routes (spf.rs:838-941) for one topology, over that topology's SPT planes
// (vertex order of `f`).
int topology_routes(const hl_isis_instance *in, const hspf_isis_flat &f, uint8_t mt_id, uint32_t root,
                    const uint32_t *dist_p, const uint16_t *hops_p, std::map<NetKey, RouteE> &rib) {
    const hl_isis_level &l0 = in->lvl;
    const bool std_en = l0.metric_type == HL_ISIS_METRIC_STANDARD || l0.metric_type == HL_ISIS_METRIC_BOTH;
    const bool wide_en = l0.metric_type == HL_ISIS_METRIC_WIDE || l0.metric_type == HL_ISIS_METRIC_BOTH;
    const uint32_t V = (uint32_t)f.ids.size();
    const uint32_t *dist = dist_p;
    const uint16_t *hops = hops_p;
    int rc = HSPF_OK;
    const SrView sr(l0);
        std::vector<std::vector<LNh>> vnh;
        rc = local_nexthops(f, in, mt_id, root, dist, hops, vnh);
        if (rc) return rc;

        // ---- compute_routes over the SPT in id_tree (= vertex index) order -------------
        bool attached = false;
        for (uint32_t i = 0; i < in->n_adjs; ++i) {
            const auto &a = in->adjs[i];
            if ((mt_id == HL_ISIS_MT_STANDARD ? a.topo_std : a.topo_ipv6) && a.up && (a.level_usage & 2) && a.area_disjoint) attached = true;
        }
        const bool ipv4_enabled = l0.ipv4_enabled && mt_id == HL_ISIS_MT_STANDARD;
        const bool ipv6_enabled = l0.ipv6_enabled && (mt_id == HL_ISIS_MT_STANDARD ? !in->mt_ipv6_enabled : true);
        // fragments per LAN id in LspId order
        std::vector<uint32_t> order(l0.n_lsps);
        for (uint32_t i = 0; i < l0.n_lsps; ++i) order[i] = i;
        std::stable_sort(order.begin(), order.end(), [&](uint32_t a, uint32_t b) {
            const auto &x = l0.lsps[a], &y = l0.lsps[b];
            return x.lan_id != y.lan_id ? x.lan_id < y.lan_id : x.fragment < y.fragment;
        });
        std::unordered_map<uint64_t, std::vector<uint32_t>> frags;
        for (uint32_t i : order) frags[l0.lsps[i].lan_id].push_back(i);
        for (uint32_t v = 0; v < V; ++v) {
            if (dist[v] == HSPF_DIST_INF) continue;
            const auto &fr = frags[f.ids[v]];
            const hl_isis_lsp *z = nullptr;
            for (uint32_t i : fr)
                if (l0.lsps[i].fragment == 0) { if (l0.lsps[i].seqno && l0.lsps[i].rem_lifetime) z = &l0.lsps[i]; break; }
            if (!z) continue;
            const bool att_bit = !in->att_ignore &&
                                 (mt_id == HL_ISIS_MT_STANDARD ? (z->flags & HL_LSPF_ATT) : (z->flags & HL_LSPF_MT_IPV6_ATT));
            auto add = [&](const hl_ip_addr &prefix, uint8_t len, uint32_t nmetric, bool external, const hl_isis_ipreach *src = nullptr) {
                auto build = [&](std::map<hl_ip_addr, RNh, IpLess> &m) {
                    for (const LNh &nh : vnh[v]) {
                        hl_ip_addr addr{};
                        if (!prefix.is_v6) {
                            if (!nh.has4) continue;
                            addr.bytes[0] = (uint8_t)(nh.ipv4 >> 24); addr.bytes[1] = (uint8_t)(nh.ipv4 >> 16);
                            addr.bytes[2] = (uint8_t)(nh.ipv4 >> 8); addr.bytes[3] = (uint8_t)nh.ipv4;
                        } else {
                            if (!nh.has6) continue;
                            addr = nh.ipv6; addr.is_v6 = 1;
                        }
                        m[addr] = RNh{nh.sysid, nh.iface, addr};
                    }
                };
                const uint32_t metric = dist[v] + nmetric;
                NetKey key{prefix, len};
                auto rit = rib.find(key);
                RouteE *route;
                if (rit == rib.end() || metric < rit->second.metric) {
                    RouteE r{};
                    r.flags = hops[v] == 0 ? HL_ROUTE_CONNECTED : 0;
                    r.type = in->level == 1 ? (external ? HL_ISIS_RT_L1_EXT : HL_ISIS_RT_L1_INTRA)
                                            : (external ? HL_ISIS_RT_L2_EXT : HL_ISIS_RT_L2_INTRA);
                    r.metric = metric;
                    build(r.nh);
                    if (src && src->has_psid) r.psid = PrefixSid{true, src->psid_flags, src->psid_is_label != 0, src->psid_value};
                    if (rit == rib.end()) route = &rib.emplace(key, std::move(r)).first->second;
                    else { rit->second = std::move(r); route = &rit->second; }
                } else if (metric == rit->second.metric) {
                    build(rit->second.nh);
                    route = &rit->second;
                } else {
                    return;
                }
                while (route->nh.size() > in->max_paths) route->nh.erase(std::prev(route->nh.end()));
                if (in->sr_enabled && route->psid.present)      // spf.rs:923-939
                    sr.update(*route, in->system_id, f.ids[v], prefix.is_v6 != 0, hops[v] == 0, hops[v] == 1);
            };
            for (uint32_t i : fr) {
                const auto &lsp = l0.lsps[i];
                if (!lsp.seqno || !lsp.rem_lifetime) continue;
                if (att_bit && in->level == 1 && (in->level_type == 1 || !attached)) {
                    if (ipv4_enabled) add(hl_ip_addr{}, 0, 0, false);
                    if (ipv6_enabled) { hl_ip_addr z6{}; z6.is_v6 = 1; add(z6, 0, 0, false); }
                }
                const hl_isis_ipreach *ip = l0.ipreaches + lsp.ipreach_off;
                if (mt_id == HL_ISIS_MT_STANDARD && ipv4_enabled) {
                    if (std_en) {
                        for (uint32_t k = 0; k < lsp.n_ipreach; ++k)
                            if (ip[k].kind == HL_ISIS_IP_V4_INTERNAL) add(ip[k].prefix, ip[k].len, ip[k].metric, false);
                        for (uint32_t k = 0; k < lsp.n_ipreach; ++k)
                            if (ip[k].kind == HL_ISIS_IP_V4_EXTERNAL) add(ip[k].prefix, ip[k].len, ip[k].metric, true);
                    }
                    if (wide_en)
                        for (uint32_t k = 0; k < lsp.n_ipreach; ++k)
                            if (ip[k].kind == HL_ISIS_IP_V4_EXT && ip[k].metric <= kMaxWide)
                                add(ip[k].prefix, ip[k].len, ip[k].metric, ip[k].external, &ip[k]);
                }
                if (ipv6_enabled)
                    for (uint32_t k = 0; k < lsp.n_ipreach; ++k) {
                        const bool take = mt_id == HL_ISIS_MT_IPV6 ? (ip[k].kind == HL_ISIS_IP_MT_V6 && ip[k].mt_id == HL_ISIS_MT_IPV6)
                                                                   : (ip[k].kind == HL_ISIS_IP_V6);
                        if (take) add(ip[k].prefix, ip[k].len, ip[k].metric, ip[k].external, &ip[k]);
                    }
            }
        }
    return HSPF_OK;
}

int emit_rib(std::map<NetKey, RouteE> &rib, hl_isis_rib *out) {
    uint32_t need_h = 0;
    for (auto &kv : rib) need_h += (uint32_t)kv.second.nh.size();
    out->n_routes = (uint32_t)rib.size(); out->n_nexthops = need_h;
    if (out->n_routes > out->routes_cap || need_h > out->nexthops_cap) return HSPF_E_NOMEM;
    uint32_t i = 0, h = 0;
    for (auto &kv : rib) {
        hl_isis_route o{};
        o.prefix = kv.first.a; o.len = kv.first.len; o.metric = kv.second.metric; o.route_type = kv.second.type;
        o.flags = kv.second.flags; o.nh_off = h; o.n_nh = (uint32_t)kv.second.nh.size();
        o.has_sr_label = kv.second.has_label ? 1 : 0; o.sr_label = kv.second.has_label ? kv.second.label : 0;
        for (auto &nk : kv.second.nh) {
            hl_isis_nexthop x{};
            x.system_id = nk.second.sysid; x.iface = nk.second.iface; x.addr = nk.second.addr;
            x.has_label = nk.second.has_label ? 1 : 0; x.sr_label = nk.second.has_label ? nk.second.label : 0;
            out->nexthops[h++] = x;
        }
        out->routes[i++] = o;
    }
    return HSPF_OK;
}

}  // namespace

extern "C" int hspf_isis_compute_routes(hspf_ctx *ctx, const hl_isis_instance *in, hl_isis_rib *out) {
    if (!ctx || !in || !out) return HSPF_E_INVAL;
    try {
        std::map<NetKey, RouteE> rib;
        const uint8_t mts[2] = {HL_ISIS_MT_STANDARD, HL_ISIS_MT_IPV6};
        for (uint8_t mt_id : mts) {
            if (mt_id == HL_ISIS_MT_IPV6 && !in->mt_ipv6_enabled) continue;
            hspf_isis_flat f;
            uint32_t root = 0;
            bool have_root = false;
            int rc = topology_flat(in, mt_id, f, root, have_root);
            if (rc) return rc;
            if (!have_root) continue;
            hspf_csr csr;
            fill_csr(f, &csr);
            hspf::OneRootPlanes p;
            rc = hspf::run_one_root(ctx, csr, root, 4, false, p);
            if (rc == HSPF_E_JOB_STATUS && !(p.status & ~HSPF_JS_TOO_MANY_ATOMS)) rc = HSPF_OK;
            if (rc) return rc;
            rc = topology_routes(in, f, mt_id, root, p.dist.data(), p.hops.data(), rib);
            if (rc) return rc;
        }
        return emit_rib(rib, out);
    } catch (const std::bad_alloc &) { return HSPF_E_NOMEM; } catch (...) { return HSPF_E_INVAL; }
}

/* The same route stage over SPT planes the caller already has (e.g. one job of a what-if batch
 * run through hspf_isis_flatten + hspf_run_batch): `dist_*` / `hops_*` are indexed by the vertex
 * order of hspf_isis_flatten for that topology (lvl.mt_id = HL_ISIS_MT_STANDARD / HL_ISIS_MT_IPV6,
 * lvl.metric_mode = HL_ISIS_MODE_NORMAL); the IPv6-topology planes are ignored unless
 * inst->mt_ipv6_enabled.  Host only. */
extern "C" int hspf_isis_routes_from_planes(const hl_isis_instance *in, const uint32_t *dist_std, const uint16_t *hops_std,
                                            const uint32_t *dist_mt6, const uint16_t *hops_mt6, hl_isis_rib *out) {
    if (!in || !out) return HSPF_E_INVAL;
    try {
        std::map<NetKey, RouteE> rib;
        const uint8_t mts[2] = {HL_ISIS_MT_STANDARD, HL_ISIS_MT_IPV6};
        for (uint8_t mt_id : mts) {
            if (mt_id == HL_ISIS_MT_IPV6 && !in->mt_ipv6_enabled) continue;
            const uint32_t *dist = mt_id == HL_ISIS_MT_STANDARD ? dist_std : dist_mt6;
            const uint16_t *hops = mt_id == HL_ISIS_MT_STANDARD ? hops_std : hops_mt6;
            hspf_isis_flat f;
            uint32_t root = 0;
            bool have_root = false;
            int rc = topology_flat(in, mt_id, f, root, have_root);
            if (rc) return rc;
            if (!have_root) continue;
            if (!dist || !hops) return HSPF_E_INVAL;
            rc = topology_routes(in, f, mt_id, root, dist, hops, rib);
            if (rc) return rc;
        }
        return emit_rib(rib, out);
    } catch (const std::bad_alloc &) { return HSPF_E_NOMEM; } catch (...) { return HSPF_E_INVAL; }
}
