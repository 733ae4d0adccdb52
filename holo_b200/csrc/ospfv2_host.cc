// ospfv2_host.cc — OSPFv2 host side of the engine: LSDB image -> CSR, and device
// results -> Vertex.nexthops / area router table / intra-area routes.
//
// What the reference does inside its Dijkstra loop per visited link
// (vertex_lsa_find + vertex_lsa_links + mutual-link re-iteration,
// holo-ospf/src/ospfv2/spf.rs:356-461, spf.rs:654-664) is done here ONCE per
// LSDB with sorted tables, so the device sees a clean CSR; the SPT itself comes
// from spf_batch_kernel through hspf_run_batch.  After the kernel the first-hop
// atoms are mapped to interface/address next hops following
// Ospfv2::calc_nexthops (ospfv2/spf.rs:173-354), then the intra-area route table
// is assembled per update_rib_intra_area / route_update (route.rs:343-446,
// 895-942) with SR labels per sr.rs:29-77,127-255.
#include <algorithm>
#include <cstring>
#include <memory>
#include <new>
#include <stdexcept>
#include <unordered_map>
#include <unordered_set>
#include <vector>

#include "holo_spf_lsdb.h"
#include "route_cells.h"
#include "spf_one_root.h"

namespace {

constexpr uint32_t kNone = 0xFFFFFFFFu;

struct Nh {   // one next hop; ordering key = (iface sort_key, has_addr, addr)
    uint32_t sort, iface, addr, nbr, label;
    uint8_t has_addr, has_nbr, has_label;
};
inline bool nh_less(const Nh &a, const Nh &b) {
    if (a.sort != b.sort) return a.sort < b.sort;
    if (a.has_addr != b.has_addr) return a.has_addr < b.has_addr;
    return a.addr < b.addr;
}
inline bool nh_same_key(const Nh &a, const Nh &b) { return a.sort == b.sort && a.has_addr == b.has_addr && a.addr == b.addr; }

// sorted-unique insert; an existing key is overwritten (BTreeMap::insert/extend)
void nh_insert(std::vector<Nh> &set, const Nh &x) {
    auto it = std::lower_bound(set.begin(), set.end(), x, nh_less);
    if (it != set.end() && nh_same_key(*it, x)) *it = x; else set.insert(it, x);
}

}  // namespace

struct hspf_ospfv2_flat {
    const hl_ospfv2_area *area = nullptr;
    uint32_t n_net = 0, n_rtr = 0;
    std::vector<uint32_t> ids;          // [V] dr_addr / router_id
    std::vector<uint8_t> is_router;     // [V]
    std::vector<uint32_t> lsa_of;       // [V] index into network_lsas / router_lsas
    std::vector<uint32_t> row, col, cost, link_index, link_pos;
    std::vector<uint8_t> vflags;
    std::unordered_map<uint32_t, uint32_t> net_vertex, rtr_vertex;   // id -> vertex
};

namespace {

int flatten(const hl_ospfv2_area *a, hspf_ospfv2_flat &f) {
    f.area = a;
    // ---- vertices ---------------------------------------------------------------
    // Router vertex: LSA key (adv_rtr == lsa_id == router_id), not MaxAge.
    std::vector<std::pair<uint32_t, uint32_t>> rtrs;   // (router_id, lsa index)
    for (uint32_t i = 0; i < a->n_router_lsas; ++i) {
        const auto &l = a->router_lsas[i];
        if (l.adv_rtr == l.lsa_id && l.age != HL_LSA_MAX_AGE) rtrs.emplace_back(l.adv_rtr, i);
    }
    std::sort(rtrs.begin(), rtrs.end());
    rtrs.erase(std::unique(rtrs.begin(), rtrs.end(), [](auto &x, auto &y) { return x.first == y.first; }), rtrs.end());
    // Network vertex: the FIRST Network-LSA in LsaKey order with that LS-ID; if that
    // one is MaxAge the vertex does not exist (find() before filter()).
    std::vector<uint32_t> order(a->n_network_lsas);
    for (uint32_t i = 0; i < a->n_network_lsas; ++i) order[i] = i;
    std::stable_sort(order.begin(), order.end(), [&](uint32_t x, uint32_t y) {
        const auto &p = a->network_lsas[x], &q = a->network_lsas[y];
        return p.adv_rtr != q.adv_rtr ? p.adv_rtr < q.adv_rtr : p.lsa_id < q.lsa_id;
    });
    std::unordered_map<uint32_t, uint32_t> first_net;   // lsa_id -> lsa index
    for (uint32_t i : order) first_net.emplace(a->network_lsas[i].lsa_id, i);
    std::vector<std::pair<uint32_t, uint32_t>> nets;
    for (auto &kv : first_net)
        if (a->network_lsas[kv.second].age != HL_LSA_MAX_AGE) nets.emplace_back(kv.first, kv.second);
    std::sort(nets.begin(), nets.end());

    f.n_net = (uint32_t)nets.size();
    f.n_rtr = (uint32_t)rtrs.size();
    const uint32_t V = f.n_net + f.n_rtr;
    f.ids.resize(V); f.is_router.resize(V); f.lsa_of.resize(V); f.vflags.resize(V);
    for (uint32_t i = 0; i < f.n_net; ++i) {
        f.ids[i] = nets[i].first; f.is_router[i] = 0; f.lsa_of[i] = nets[i].second; f.vflags[i] = 0;
        f.net_vertex.emplace(nets[i].first, i);
    }
    for (uint32_t i = 0; i < f.n_rtr; ++i) {
        const uint32_t v = f.n_net + i;
        f.ids[v] = rtrs[i].first; f.is_router[v] = 1; f.lsa_of[v] = rtrs[i].second; f.vflags[v] = HSPF_VF_HOP;
        f.rtr_vertex.emplace(rtrs[i].first, v);
    }

    // ---- raw links (before the mutual-link filter) ---------------------------------
    struct Raw { uint32_t u, v, cost, link, pos; };
    std::vector<Raw> raw;
    raw.reserve(a->n_links + a->n_attached);
    std::vector<uint32_t> att;
    for (uint32_t v = 0; v < V; ++v) {
        if (!f.is_router[v]) {
            const auto &n = a->network_lsas[f.lsa_of[v]];
            att.assign(a->attached + n.att_off, a->attached + n.att_off + n.n_att);
            std::sort(att.begin(), att.end());
            att.erase(std::unique(att.begin(), att.end()), att.end());
            for (uint32_t rid : att) {
                auto it = f.rtr_vertex.find(rid);
                if (it == f.rtr_vertex.end()) continue;
                raw.push_back({v, it->second, 0, kNone, 0});
            }
        } else {
            const auto &r = a->router_lsas[f.lsa_of[v]];
            uint32_t pos = 0;
            for (uint32_t k = 0; k < r.n_links; ++k) {
                const auto &l = a->links[r.link_off + k];
                uint32_t tgt = kNone;
                if (l.link_type == HL_LINK_P2P || l.link_type == HL_LINK_VLINK) {
                    auto it = f.rtr_vertex.find(l.link_id);
                    if (it != f.rtr_vertex.end()) tgt = it->second;
                } else if (l.link_type == HL_LINK_TRANSIT) {
                    auto it = f.net_vertex.find(l.link_id);
                    if (it != f.net_vertex.end()) tgt = it->second;
                } else {
                    continue;   // stub links are dropped before enumerate()
                }
                const uint32_t p = pos++;
                if (tgt == kNone) continue;
                raw.push_back({v, tgt, l.metric, r.link_off + k, p});
            }
        }
    }
    // ---- mutual-link filter: keep u->v iff v has any raw link to u -----------------
    // raw is grouped by u (vertices were walked in order): "v links back to u" is a scan of v's few raw links
    std::vector<uint32_t> rrow(V + 1, 0);
    for (auto &e : raw) rrow[e.u + 1]++;
    for (uint32_t v = 0; v < V; ++v) rrow[v + 1] += rrow[v];
    std::vector<uint8_t> keep(raw.size(), 0);
    for (size_t i = 0; i < raw.size(); ++i) {
        const Raw &e = raw[i];
        if (e.u == e.v) continue;   // a link to oneself is skipped by `spt.contains_key`
        for (uint32_t k = rrow[e.v]; k < rrow[e.v + 1]; ++k)
            if (raw[k].v == e.u) { keep[i] = 1; break; }
    }
    f.row.assign(V + 1, 0);
    for (size_t i = 0; i < raw.size(); ++i) if (keep[i]) f.row[raw[i].u + 1]++;
    for (uint32_t v = 0; v < V; ++v) f.row[v + 1] += f.row[v];
    const uint32_t E = f.row[V];
    f.col.resize(E); f.cost.resize(E); f.link_index.resize(E); f.link_pos.resize(E);
    uint32_t k = 0;
    for (size_t i = 0; i < raw.size(); ++i) {   // grouped by u in link order: edges come out in CSR order
        if (!keep[i]) continue;
        const Raw &e = raw[i];
        f.col[k] = e.v; f.cost[k] = e.cost; f.link_index[k] = e.link; f.link_pos[k] = e.pos;
        ++k;
    }
    return HSPF_OK;
}

void fill_csr(const hspf_ospfv2_flat &f, hspf_csr *c) {
    std::memset(c, 0, sizeof(*c));
    c->n_vertices = (uint32_t)f.ids.size();
    c->n_edges = (uint32_t)f.col.size();
    c->row_ptr = f.row.data();
    c->col = f.col.data();
    c->cost = f.cost.data();
    c->vflags = f.vflags.data();
    c->reject_above = 0xFFFFFFFEu;
    c->saturate_at = 0xFFFFu;
    c->flags = 0;
    c->delta = 0;
}

// ---- first hops (Ospfv2::calc_nexthops) ------------------------------------------------
struct Resolver {
    const hspf_ospfv2_flat &f;
    const hl_ospfv2_area *a;
    uint32_t root;
    const uint64_t *nh_mask;   // [V][nhw]
    uint32_t nhw;
    std::vector<std::vector<Nh>> atom_nh;   // per atom
    std::vector<uint8_t> atom_done;
    std::vector<int> ifaces_with_nbrs;      // nth(link_pos) table

    // parent is the root (ospfv2/spf.rs:188-305)
    void root_atom(uint32_t e, std::vector<Nh> &out) const {
        const uint32_t pos = f.link_pos[e];
        if (pos >= ifaces_with_nbrs.size()) return;                  // Err(SpfNexthopCalcError)
        const uint32_t ii = (uint32_t)ifaces_with_nbrs[pos];
        const hl_ospf_iface &iface = a->ifaces[ii];
        if (iface.if_type == HL_IF_VLINK) return;                    // resolved later (RFC 2328 16.3)
        const uint32_t dest = f.col[e];
        if (f.is_router[dest]) {
            const auto &dl = a->router_lsas[f.lsa_of[dest]];
            if (iface.if_type == HL_IF_P2P || iface.if_type == HL_IF_VLINK) {
                for (uint32_t k = 0; k < iface.n_nbrs; ++k) {
                    const auto &nbr = a->nbrs[iface.nbr_off + k];
                    if (nbr.router_id != dl.adv_rtr) continue;
                    out.push_back(Nh{iface.sort_key, ii, nbr.src, dl.adv_rtr, 0, 1, 1, 0});
                    break;
                }
            } else if (iface.if_type == HL_IF_P2MP) {
                for (uint32_t k = 0; k < dl.n_links; ++k) {
                    const auto &l = a->links[dl.link_off + k];
                    bool in = false;
                    for (uint32_t q = 0; q < iface.n_addrs && !in; ++q) {
                        const auto &net = a->iface_addrs[iface.addr_off + q];
                        in = (l.link_data & net.mask) == (net.addr & net.mask);
                    }
                    if (in) nh_insert(out, Nh{iface.sort_key, ii, l.link_data, dl.adv_rtr, 0, 1, 1, 0});
                }
            }
        } else {
            out.push_back(Nh{iface.sort_key, ii, 0, 0, 0, 0, 0, 0});
        }
    }

    std::vector<Nh> vertex_nexthops(uint32_t v) {
        std::vector<Nh> set;
        for (uint32_t w = 0; w < nhw; ++w) {
            uint64_t m = nh_mask[(size_t)v * nhw + w];
            while (m) {
                const uint32_t atom = w * 64 + (uint32_t)__builtin_ctzll(m);
                m &= m - 1;
                for (const Nh &x : resolve(atom)) nh_insert(set, x);
            }
        }
        return set;
    }

    const std::vector<Nh> &resolve(uint32_t atom) {
        if (atom_done[atom]) return atom_nh[atom];
        atom_done[atom] = 1;   // (the DAG has no cycles; set first to be safe)
        hspf_csr c;
        fill_csr(f, &c);
        uint32_t tail = 0, e = 0;
        std::vector<Nh> out;
        if (hspf_atom_decode(&c, root, atom, &tail, &e) == HSPF_OK) {
            if (tail == root) {
                root_atom(e, out);
            } else {
                // parent is a transit network attached to the root (ospfv2/spf.rs:306-350)
                const auto &pl = a->network_lsas[f.lsa_of[tail]];
                const uint32_t dest = f.col[e];
                const auto &dl = a->router_lsas[f.lsa_of[dest]];
                const hl_ospfv2_link *dest_link = nullptr;
                for (uint32_t k = 0; k < dl.n_links; ++k) {
                    const auto &l = a->links[dl.link_off + k];
                    if ((l.link_data & pl.mask) == (pl.lsa_id & pl.mask)) { dest_link = &l; break; }
                }
                if (dest_link) {
                    std::vector<Nh> pn = vertex_nexthops(tail);     // parent.nexthops, final when it is expanded
                    if (!pn.empty()) {
                        const Nh &p0 = pn.front();
                        out.push_back(Nh{p0.sort, p0.iface, dest_link->link_data, dl.adv_rtr, 0, 1, 1, 0});
                    }
                }
            }
        }
        atom_nh[atom] = std::move(out);
        return atom_nh[atom];
    }
};

struct RouterInfo { bool has_sr_algo = false; std::vector<const hl_srgb *> srgb; };

bool index_to_label(uint32_t index, const std::vector<const hl_srgb *> &srgbs, uint32_t *label) {
    for (auto *s : srgbs) {
        if (s->first_is_index) continue;
        if (index >= s->range) { index -= s->range; continue; }
        *label = s->first + index;
        return true;
    }
    return false;
}

// open-addressing u64 -> u32 table sized once (the tables below know their bound): a find is a multiply and a probe
struct FlatMap64 {
    static constexpr uint64_t kEmpty = ~0ull;
    std::vector<uint64_t> keys;
    std::vector<uint32_t> vals;
    uint64_t mask = 0;
    void init(size_t n) {
        size_t cap = 16;
        while (cap < 2 * n + 2) cap <<= 1;
        keys.assign(cap, kEmpty);
        vals.assign(cap, 0);
        mask = cap - 1;
    }
    static uint64_t mix(uint64_t k) { k ^= k >> 29; k *= 0x9E3779B97F4A7C15ull; return k ^ (k >> 32); }
    uint32_t *find(uint64_t k) {
        for (uint64_t i = mix(k) & mask;; i = (i + 1) & mask) {
            if (keys[i] == k) return &vals[i];
            if (keys[i] == kEmpty) return nullptr;
        }
    }
    // inserts when absent; returns the slot's value either way
    uint32_t &at(uint64_t k, uint32_t v_if_new, bool *inserted) {
        for (uint64_t i = mix(k) & mask;; i = (i + 1) & mask) {
            if (keys[i] == k) { *inserted = false; return vals[i]; }
            if (keys[i] == kEmpty) { keys[i] = k; vals[i] = v_if_new; *inserted = true; return vals[i]; }
        }
    }
};

struct Route {
    uint32_t prefix, plen, metric;
    uint8_t flags, origin_type;
    uint32_t origin_adv, origin_id;
    bool has_sid = false; uint32_t sid_value = 0; uint8_t sid_flags = 0; bool sid_is_label = false;
    bool has_label = false; uint32_t label = 0;
    std::vector<Nh> nh;                          // owned next hops (labelled, merged or truncated) ...
    const std::vector<Nh> *shared = nullptr;     // ... or the vertex's own set, untouched (most routes)
    const std::vector<Nh> &hops() const { return shared ? *shared : nh; }
    void own() { if (shared) { nh = *shared; shared = nullptr; } }
};

inline uint64_t pkey(uint32_t prefix, uint32_t plen) { return ((uint64_t)prefix << 8) | plen; }

}  // namespace

extern "C" {

int hspf_ospfv2_flatten(const hl_ospfv2_area *area, hspf_ospfv2_flat **out) {
    if (!area || !out) return HSPF_E_INVAL;
    *out = nullptr;
    try {
        auto *f = new hspf_ospfv2_flat();
        int rc = flatten(area, *f);
        if (rc) { delete f; return rc; }
        *out = f;
        return HSPF_OK;
    } catch (const std::bad_alloc &) {
        return HSPF_E_NOMEM;
    } catch (...) {
        return HSPF_E_INVAL;
    }
}

void hspf_ospfv2_flat_free(hspf_ospfv2_flat *flat) { delete flat; }

int hspf_ospfv2_flat_csr(const hspf_ospfv2_flat *flat, hspf_csr *out) {
    if (!flat || !out) return HSPF_E_INVAL;
    fill_csr(*flat, out);
    return HSPF_OK;
}

int hspf_ospfv2_flat_vertices(const hspf_ospfv2_flat *flat, const uint32_t **ids, const uint8_t **is_router,
                              uint32_t *n_vertices) {
    if (!flat) return HSPF_E_INVAL;
    if (ids) *ids = flat->ids.data();
    if (is_router) *is_router = flat->is_router.data();
    if (n_vertices) *n_vertices = (uint32_t)flat->ids.size();
    return HSPF_OK;
}

int hspf_ospfv2_flat_edge_tags(const hspf_ospfv2_flat *flat, const uint32_t **link_index, const uint32_t **link_pos) {
    if (!flat) return HSPF_E_INVAL;
    if (link_index) *link_index = flat->link_index.data();
    if (link_pos) *link_pos = flat->link_pos.data();
    return HSPF_OK;
}

uint32_t hspf_ospfv2_flat_router_vertex(const hspf_ospfv2_flat *flat, uint32_t router_id) {
    if (!flat) return kNone;
    auto it = flat->rtr_vertex.find(router_id);
    return it == flat->rtr_vertex.end() ? kNone : it->second;
}

uint32_t hspf_ospfv2_flat_network_vertex(const hspf_ospfv2_flat *flat, uint32_t dr_addr) {
    if (!flat) return kNone;
    auto it = flat->net_vertex.find(dr_addr);
    return it == flat->net_vertex.end() ? kNone : it->second;
}

/* sizeof() of every struct that crosses the ABI, for binding self-checks. */
int hspf_abi_sizes(uint32_t *out, uint32_t cap) {
    const uint32_t v[] = {
        (uint32_t)sizeof(hspf_csr), (uint32_t)sizeof(hspf_jobs), (uint32_t)sizeof(hspf_result),
        (uint32_t)sizeof(hl_ospfv2_link), (uint32_t)sizeof(hl_ospfv2_router_lsa), (uint32_t)sizeof(hl_ospfv2_network_lsa),
        (uint32_t)sizeof(hl_ospf_iface), (uint32_t)sizeof(hl_ipv4_net), (uint32_t)sizeof(hl_ospf_nbr),
        (uint32_t)sizeof(hl_srgb), (uint32_t)sizeof(hl_ospfv2_ri_lsa), (uint32_t)sizeof(hl_ospfv2_ext_prefix),
        (uint32_t)sizeof(hl_ospfv2_area), (uint32_t)sizeof(hl_nexthop), (uint32_t)sizeof(hl_spt_vertex),
        (uint32_t)sizeof(hl_route_rtr), (uint32_t)sizeof(hl_route_net), (uint32_t)sizeof(hl_ospfv2_result),
        (uint32_t)sizeof(hl_isis_reach), (uint32_t)sizeof(hl_isis_lsp), (uint32_t)sizeof(hl_isis_level),
        (uint32_t)sizeof(hl_isis_vertex), (uint32_t)sizeof(hl_isis_spt),
        (uint32_t)sizeof(hl_isis_ipreach), (uint32_t)sizeof(hl_isis_adj), (uint32_t)sizeof(hl_isis_iface),
        (uint32_t)sizeof(hl_isis_instance), (uint32_t)sizeof(hl_isis_nexthop), (uint32_t)sizeof(hl_isis_route),
        (uint32_t)sizeof(hl_isis_rib),
        (uint32_t)sizeof(hl_ospfv3_link), (uint32_t)sizeof(hl_ospfv3_router_lsa), (uint32_t)sizeof(hl_ospfv3_network_lsa),
        (uint32_t)sizeof(hl_ip_addr), (uint32_t)sizeof(hl_ospfv3_prefix), (uint32_t)sizeof(hl_ospfv3_iap_lsa),
        (uint32_t)sizeof(hl_ospfv3_link_lsa), (uint32_t)sizeof(hl_ospfv3_iface), (uint32_t)sizeof(hl_ospfv3_area),
        (uint32_t)sizeof(hl_nexthop6), (uint32_t)sizeof(hl_spt_vertex6), (uint32_t)sizeof(hl_route_net6),
        (uint32_t)sizeof(hl_ospfv3_result),
        (uint32_t)sizeof(hl_ospfv2_summary_lsa), (uint32_t)sizeof(hl_ospfv2_external_lsa),
        (uint32_t)sizeof(hl_ospfv2_rib_area), (uint32_t)sizeof(hl_rib_route), (uint32_t)sizeof(hl_ospfv2_rib),
        (uint32_t)sizeof(hl_ospfv3_inter_area_lsa), (uint32_t)sizeof(hl_ospfv3_external_lsa),
        (uint32_t)sizeof(hl_ospfv3_rib_area), (uint32_t)sizeof(hl_rib_route6), (uint32_t)sizeof(hl_ospfv3_rib),
        (uint32_t)sizeof(hl_rib_action),
        (uint32_t)sizeof(hl_isis_rnl_entry),
        (uint32_t)sizeof(hl_route_cell),
        (uint32_t)sizeof(hl_lsa_trigger), (uint32_t)sizeof(hl_spf_computation), (uint32_t)sizeof(hl_rib_rtr),
        (uint32_t)sizeof(hl_ospfv2_rtr_tables),
        (uint32_t)sizeof(hl_isis_lsp_trigger), (uint32_t)sizeof(hl_ip_prefix), (uint32_t)sizeof(hl_lsa_trigger6),
        (uint32_t)sizeof(hl_spf_computation6),
    };
    static_assert(sizeof(hl_rib_action) == 12, "hl_rib_action layout");
    const uint32_t n = sizeof(v) / sizeof(v[0]);
    if (!out || cap < n) return (int)n;
    for (uint32_t i = 0; i < n; ++i) out[i] = v[i];
    return (int)n;
}

}  // extern "C" (reopened below)

namespace {

// Everything run_area + update_rib_intra_area do after the SPT (holo-ospf/src/spf.rs:627-724,
// route.rs:343-446, sr.rs): Vertex.nexthops from the atom sets, the area's router table,
// transit_capability, intra-area routes with SR labels.  `dist` / `hops` / `nh` are the planes
// of the root's job in the vertex order of `f`.
int area_from_planes(const hspf_ospfv2_flat &f, const hl_ospfv2_area *a, uint32_t root, const uint32_t *dist,
                     const uint16_t *hops, const uint64_t *nh, uint32_t nhw, hl_ospfv2_result *out) {
    const uint32_t V = (uint32_t)f.ids.size();
    // ---- Vertex.nexthops --------------------------------------------------------------
    Resolver rs{f, a, root, nh, nhw, {}, {}, {}};
    rs.atom_nh.resize((size_t)64 * nhw);
    rs.atom_done.assign((size_t)64 * nhw, 0);
    for (uint32_t i = 0; i < a->n_ifaces; ++i)
        if (a->ifaces[i].n_nbrs > 0) rs.ifaces_with_nbrs.push_back((int)i);
    std::vector<uint32_t> spt;            // vertices on the SPT, VertexId order
    for (uint32_t v = 0; v < V; ++v) if (dist[v] != HSPF_DIST_INF) spt.push_back(v);
    std::vector<std::vector<Nh>> vnh(V);
    for (uint32_t v : spt) vnh[v] = rs.vertex_nexthops(v);

    // ---- intra-area routes (update_rib_intra_area) ------------------------------------
    FlatMap64 extp;                      // (adv_rtr, prefix/len) -> index of the first live entry
    auto ekey = [](uint32_t adv, uint32_t prefix, uint32_t plen) {
        return (((uint64_t)adv << 38) ^ ((uint64_t)prefix << 6) ^ plen) & 0x7FFFFFFFFFFFFFFFull;
    };
    if (a->sr_enabled) {
        extp.init(a->n_ext_prefixes);
        for (uint32_t i = 0; i < a->n_ext_prefixes; ++i) {
            const auto &e = a->ext_prefixes[i];
            if (e.age == HL_LSA_MAX_AGE) continue;
            bool fresh;
            extp.at(ekey(e.adv_rtr, e.prefix, (uint32_t)__builtin_popcount(e.mask)), i, &fresh);
        }
    }
    auto ext_find = [&](uint32_t adv, uint32_t prefix, uint32_t plen) -> const hl_ospfv2_ext_prefix * {
        const uint32_t *slot = extp.find(ekey(adv, prefix, plen));
        if (!slot) return nullptr;
        const auto *e = &a->ext_prefixes[*slot];
        if (e->adv_rtr == adv && e->prefix == prefix && (uint32_t)__builtin_popcount(e->mask) == plen) return e;
        // hash-key collision: fall back to a scan (first match in LSDB order)
        for (uint32_t i = 0; i < a->n_ext_prefixes; ++i) {
            const auto &x = a->ext_prefixes[i];
            if (x.age != HL_LSA_MAX_AGE && x.adv_rtr == adv && x.prefix == prefix &&
                (uint32_t)__builtin_popcount(x.mask) == plen) return &x;
        }
        return nullptr;
    };
    FlatMap64 rib_idx;
    std::vector<Route> rib;
    std::vector<uint8_t> rib_live;
    {   // at most one entry per stub link / network vertex: no rehash, no vector regrowth
        const size_t cap = (size_t)a->n_links + a->n_network_lsas + 1;
        rib_idx.init(cap);
        rib.reserve(cap);
        rib_live.reserve(cap);
    }
    RouterInfo local_ri; bool local_ri_loaded = false;
    // per-router aggregate of the Router-Information LSAs (area_router_information,
    // ospfv2/spf.rs:617-654), built in one pass over the LSDB-ordered array
    std::unordered_map<uint32_t, RouterInfo> ri_cache;
    const RouterInfo no_ri;
    if (a->sr_enabled) {
        ri_cache.reserve(a->n_ri_lsas);
        for (uint32_t i = 0; i < a->n_ri_lsas; ++i) {
            const auto &l = a->ri_lsas[i];
            if (l.age == HL_LSA_MAX_AGE) continue;
            RouterInfo &ri = ri_cache[l.adv_rtr];
            if (l.has_sr_algo) ri.has_sr_algo = true;
            for (uint32_t k = 0; k < l.n_srgb; ++k) ri.srgb.push_back(&a->srgbs[l.srgb_off + k]);
        }
    }
    auto cached_ri = [&](uint32_t rid) -> const RouterInfo & {
        auto it = ri_cache.find(rid);
        if (it == ri_cache.end()) return no_ri;
        return it->second;
    };

    // the neighbours that next hops name are the root's few: remember their entries
    std::vector<std::pair<uint32_t, const RouterInfo *>> nbr_memo;
    auto nbr_ri = [&](uint32_t rid) -> const RouterInfo & {
        for (auto &kv : nbr_memo) if (kv.first == rid) return *kv.second;
        const RouterInfo &ri = cached_ri(rid);
        if (nbr_memo.size() < 64) nbr_memo.emplace_back(rid, &ri);
        return ri;
    };
    auto add_stub = [&](uint32_t v, uint32_t prefix, uint32_t plen, uint32_t stub_metric, uint32_t adv_rtr) {
        uint32_t m = dist[v] + stub_metric;
        if (m > 0xFFFF) m = 0xFFFF;
        const uint64_t key = pkey(prefix, plen);
        const uint32_t *slot = rib_idx.find(key);
        Route *cur = (slot && rib_live[*slot]) ? &rib[*slot] : nullptr;
        if (cur && m > cur->metric) return;
        uint8_t otype; uint32_t oadv, oid;
        if (f.is_router[v]) { const auto &l = a->router_lsas[f.lsa_of[v]]; otype = 1; oadv = l.adv_rtr; oid = l.lsa_id; }
        else { const auto &l = a->network_lsas[f.lsa_of[v]]; otype = 2; oadv = l.adv_rtr; oid = l.lsa_id; }
        if (!f.is_router[v] && cur) {
            if (m > cur->metric || oid < cur->origin_id) return;
            rib_live[*slot] = 0;        // o.remove()
            cur = nullptr;
        }
        Route nr;
        nr.prefix = prefix; nr.plen = plen; nr.metric = m;
        nr.flags = hops[v] == 0 ? HL_ROUTE_CONNECTED : 0;
        nr.origin_type = otype; nr.origin_adv = oadv; nr.origin_id = oid;
        nr.shared = &vnh[v];
        if (a->sr_enabled) {
            const hl_ospfv2_ext_prefix *ep = ext_find(adv_rtr, prefix, plen);
            if (ep && ep->route_type == 1 && ep->has_sid && cached_ri(oadv).has_sr_algo) {
                nr.own();                        // per-route labels on the next hops
                const bool local = hops[v] == 0, last_hop = hops[v] == 1;
                nr.has_sid = true; nr.sid_value = ep->sid_value; nr.sid_flags = ep->sid_flags;
                nr.sid_is_label = ep->sid_is_label;
                if (!(local && (!(ep->sid_flags & HL_PSID_NP) || (ep->sid_flags & HL_PSID_E)))) {
                    if (!ep->sid_is_label) {
                        if (!local_ri_loaded) { local_ri = cached_ri(a->router_id); local_ri_loaded = true; }
                        uint32_t lab;
                        if (!local_ri.srgb.empty() && index_to_label(ep->sid_value, local_ri.srgb, &lab)) {
                            nr.has_label = true; nr.label = lab;
                        }
                    } else {
                        nr.has_label = true; nr.label = ep->sid_value;
                    }
                }
                for (Nh &x : nr.nh) {
                    if (!x.has_nbr) continue;
                    uint32_t lab = 0; bool ok = false, decided = false;
                    if (last_hop) {
                        if (!(ep->sid_flags & HL_PSID_NP)) { lab = 3; ok = decided = true; }
                        else if (ep->sid_flags & HL_PSID_E) { lab = 0; ok = decided = true; }
                    }
                    if (!decided) {
                        if (!ep->sid_is_label) {
                            const RouterInfo &nri = nbr_ri(x.nbr);
                            if (!nri.srgb.empty()) ok = index_to_label(ep->sid_value, nri.srgb, &lab);
                        } else {
                            lab = last_hop ? ep->sid_value : 3u; ok = true;
                        }
                    }
                    if (ok) { x.has_label = 1; x.label = lab; }
                }
            }
        }
        // route_update
        Route *route;
        if (cur) {
            if (nr.metric < cur->metric) *cur = std::move(nr);
            else if (nr.metric == cur->metric) { cur->own(); for (const Nh &x : nr.hops()) nh_insert(cur->nh, x); }
            route = cur;
        } else {
            if (slot) { rib[*slot] = std::move(nr); rib_live[*slot] = 1; route = &rib[*slot]; }
            else {
                bool fresh;
                rib_idx.at(key, (uint32_t)rib.size(), &fresh);
                rib.push_back(std::move(nr)); rib_live.push_back(1); route = &rib.back();
            }
        }
        if (route->hops().size() > a->max_paths) { route->own(); route->nh.resize(a->max_paths); }
    };
    for (uint32_t v : spt) {
        if (!f.is_router[v]) {
            const auto &nl = a->network_lsas[f.lsa_of[v]];
            add_stub(v, nl.lsa_id & nl.mask, (uint32_t)__builtin_popcount(nl.mask), 0, nl.adv_rtr);
        } else {
            const auto &rl = a->router_lsas[f.lsa_of[v]];
            for (uint32_t k = 0; k < rl.n_links; ++k) {
                const auto &l = a->links[rl.link_off + k];
                if (l.link_type != HL_LINK_STUB) continue;
                add_stub(v, l.link_id & l.link_data, (uint32_t)__builtin_popcount(l.link_data), l.metric, rl.adv_rtr);
            }
        }
    }

    // ---- export ---------------------------------------------------------------------------
    std::vector<std::pair<uint64_t, uint32_t>> order;      // (prefix, length) key next to the index: a flat sort
    order.reserve(rib.size());
    for (uint32_t i = 0; i < rib.size(); ++i) if (rib_live[i]) order.emplace_back(pkey(rib[i].prefix, rib[i].plen), i);
    std::sort(order.begin(), order.end());
    std::vector<uint32_t> live;
    live.reserve(order.size());
    for (auto &kv : order) live.push_back(kv.second);
    uint32_t n_rtr_in_spt = 0, need_h = 0;
    for (uint32_t v : spt) { need_h += (uint32_t)vnh[v].size(); if (f.is_router[v]) { ++n_rtr_in_spt; need_h += (uint32_t)vnh[v].size(); } }
    for (uint32_t i : live) need_h += (uint32_t)rib[i].hops().size();
    out->n_vertices = (uint32_t)spt.size();
    out->n_routers = n_rtr_in_spt;
    out->n_routes = (uint32_t)live.size();
    out->n_nexthops = need_h;
    bool tc = false;
    for (uint32_t v : spt)
        if (f.is_router[v] && (a->router_lsas[f.lsa_of[v]].flags & HL_RTR_FLAG_V)) tc = true;
    out->transit_capability = tc;
    if (out->n_vertices > out->vertices_cap || out->n_routers > out->routers_cap ||
        out->n_routes > out->routes_cap || out->n_nexthops > out->nexthops_cap)
        return HSPF_E_NOMEM;
    uint32_t h = 0;
    auto put = [&](const std::vector<Nh> &s) {
        for (const Nh &x : s) {
            hl_nexthop o{};
            o.iface = x.iface; o.addr = x.has_addr ? x.addr : 0; o.nbr_router_id = x.has_nbr ? x.nbr : 0;
            o.sr_label = x.has_label ? x.label : 0;
            o.has_addr = x.has_addr; o.has_nbr = x.has_nbr; o.has_label = x.has_label;
            out->nexthops[h++] = o;
        }
    };
    uint32_t i = 0;
    for (uint32_t v : spt) {
        hl_spt_vertex o{};
        o.id = f.ids[v]; o.distance = dist[v]; o.hops = hops[v]; o.is_router = f.is_router[v];
        o.nh_off = h; o.n_nh = (uint32_t)vnh[v].size();
        put(vnh[v]);
        out->vertices[i++] = o;
    }
    i = 0;
    for (uint32_t v : spt) {   // router vertices are already in router-id order
        if (!f.is_router[v]) continue;
        const auto &rl = a->router_lsas[f.lsa_of[v]];
        hl_route_rtr o{};
        o.router_id = rl.adv_rtr; o.metric = dist[v]; o.flags = rl.flags; o.options = rl.options;
        o.nh_off = h; o.n_nh = (uint32_t)vnh[v].size();
        put(vnh[v]);
        out->routers[i++] = o;
    }
    i = 0;
    for (uint32_t k : live) {
        const Route &r = rib[k];
        hl_route_net o{};
        o.prefix = r.prefix; o.mask = r.plen == 0 ? 0 : 0xFFFFFFFFu << (32 - r.plen);
        o.metric = r.metric; o.flags = r.flags; o.origin_type = r.origin_type;
        o.origin_adv_rtr = r.origin_adv; o.origin_lsa_id = r.origin_id;
        o.has_prefix_sid = r.has_sid; o.prefix_sid_value = r.sid_value; o.prefix_sid_flags = r.sid_flags;
        o.prefix_sid_is_label = r.sid_is_label;
        o.has_sr_label = r.has_label; o.sr_label = r.has_label ? r.label : 0;
        o.nh_off = h; o.n_nh = (uint32_t)r.hops().size();
        put(r.hops());
        out->routes[i++] = o;
    }
    return HSPF_OK;
}

}  // namespace

extern "C" {

int hspf_ospfv2_run_area(hspf_ctx *ctx, const hl_ospfv2_area *a, hl_ospfv2_result *out) {
    if (!ctx || !a || !out) return HSPF_E_INVAL;
    try {
        out->n_vertices = out->n_routers = out->n_routes = out->n_nexthops = 0;
        out->transit_capability = 0;
        out->root_found = 0;
        hspf_ospfv2_flat f;
        int rc = flatten(a, f);
        if (rc) return rc;
        auto rit = f.rtr_vertex.find(a->router_id);
        if (rit == f.rtr_vertex.end()) return HSPF_OK;   // SpfRootNotFound: logged, nothing computed
        out->root_found = 1;
        const uint32_t root = rit->second;

        // ---- SPT on the device ---------------------------------------------------------
        hspf_csr csr;
        fill_csr(f, &csr);
        uint32_t n_atoms = 0;
        hspf_atom_count(&csr, root, &n_atoms);
        const uint32_t nhw = std::max(1u, (n_atoms + 63) / 64);
        if (nhw > 4) return HSPF_E_UNSUPPORTED;   // > 256 first-hop atoms: caller's CPU path
        hspf::OneRootPlanes p;
        rc = hspf::run_one_root(ctx, csr, root, nhw, true, p);
        if (rc) return rc;   // includes HSPF_E_JOB_STATUS (saturation): caller's CPU path
        return area_from_planes(f, a, root, p.dist.data(), p.hops.data(), p.nh.data(), nhw, out);
    } catch (const std::bad_alloc &) {
        return HSPF_E_NOMEM;
    } catch (...) {
        return HSPF_E_INVAL;
    }
}

/* The post-SPT half of hspf_ospfv2_run_area over planes the caller already has (one job of a
 * batch run through hspf_ospfv2_flatten + hspf_run_batch with the local router as root): planes
 * are indexed by the vertex order of hspf_ospfv2_flatten; nh_words as passed to the engine.
 * Host only. */
int hspf_ospfv2_area_from_planes(const hl_ospfv2_area *a, const uint32_t *dist, const uint16_t *hops,
                                 const uint64_t *nh_mask, uint32_t nh_words, hl_ospfv2_result *out) {
    if (!a || !out || !dist || !hops || !nh_mask || nh_words < 1 || nh_words > 4) return HSPF_E_INVAL;
    try {
        out->n_vertices = out->n_routers = out->n_routes = out->n_nexthops = 0;
        out->transit_capability = 0;
        out->root_found = 0;
        hspf_ospfv2_flat f;
        int rc = flatten(a, f);
        if (rc) return rc;
        auto rit = f.rtr_vertex.find(a->router_id);
        if (rit == f.rtr_vertex.end()) return HSPF_OK;
        out->root_found = 1;
        return area_from_planes(f, a, rit->second, dist, hops, nh_mask, nh_words, out);
    } catch (const std::bad_alloc &) {
        return HSPF_E_NOMEM;
    } catch (...) {
        return HSPF_E_INVAL;
    }
}


/* ---- batched route stage: the table and the per-job decode (route_cells.h) ------------------- */

void hspf_ospfv2_rtable_free(hspf_ospfv2_rtable *rt) {
    if (!rt) return;
    hspf_rtable_release_device(rt);
    delete rt;
}

int hspf_ospfv2_rtable_create(const hspf_ospfv2_flat *flat, hspf_ospfv2_rtable **out) {
    if (!flat || !flat->area || !out) return HSPF_E_INVAL;
    try {
        const hspf_ospfv2_flat &f = *flat;
        const hl_ospfv2_area *a = f.area;
        const uint32_t V = (uint32_t)f.ids.size();
        // Extended-Prefix entries by (advertising router, prefix): the first live one in LSDB order
        // (lsdb iteration + find, sr.rs:29-49), and which routers announce the SPF algorithm
        // (advertising router, prefix) -> first live Extended-Prefix entry in LSDB order (lsdb iteration + find,
        // sr.rs:29-49): a flat table on a folded key, verified on the entry, with a scan behind a false hit
        FlatMap64 extp;
        auto ekey = [](uint32_t adv, uint32_t prefix, uint32_t plen) {
            return (((uint64_t)adv << 38) ^ ((uint64_t)prefix << 6) ^ plen) & 0x7FFFFFFFFFFFFFFFull;
        };
        auto ext_lookup = [&](uint32_t adv, uint32_t prefix, uint32_t plen) -> int32_t {
            const uint32_t *slot = extp.find(ekey(adv, prefix, plen));
            if (!slot) return -1;
            const auto &e = a->ext_prefixes[*slot];
            if (e.adv_rtr == adv && e.prefix == prefix && (uint32_t)__builtin_popcount(e.mask) == plen) return (int32_t)*slot;
            for (uint32_t i = 0; i < a->n_ext_prefixes; ++i) {
                const auto &x = a->ext_prefixes[i];
                if (x.age != HL_LSA_MAX_AGE && x.adv_rtr == adv && x.prefix == prefix && (uint32_t)__builtin_popcount(x.mask) == plen)
                    return (int32_t)i;
            }
            return -1;
        };
        std::unordered_set<uint32_t> sr_algo;
        if (a->sr_enabled) {
            extp.init(a->n_ext_prefixes);
            for (uint32_t i = 0; i < a->n_ext_prefixes; ++i) {
                const auto &e = a->ext_prefixes[i];
                if (e.age == HL_LSA_MAX_AGE) continue;
                bool fresh;
                extp.at(ekey(e.adv_rtr, e.prefix, (uint32_t)__builtin_popcount(e.mask)), i, &fresh);
            }
            for (uint32_t i = 0; i < a->n_ri_lsas; ++i)
                if (a->ri_lsas[i].age != HL_LSA_MAX_AGE && a->ri_lsas[i].has_sr_algo) sr_algo.insert(a->ri_lsas[i].adv_rtr);
        }
        struct Raw { uint32_t prefix, plen, seq; hspf::RouteContrib c; uint8_t otype; uint32_t oadv; int32_t ext; };
        std::vector<Raw> raw;
        raw.reserve((size_t)a->n_links + a->n_network_lsas);
        auto rt = new hspf_ospfv2_rtable();
        std::unique_ptr<hspf_ospfv2_rtable> guard(rt);
        rt->t.sids.push_back(hspf::SidDesc{0, 0, 0});
        std::unordered_map<uint64_t, uint16_t> sid_class;
        auto add = [&](uint32_t v, uint32_t prefix, uint32_t plen, uint32_t metric, uint8_t otype, uint32_t oadv, uint32_t oid) {
            Raw r{};
            r.prefix = prefix; r.plen = plen; r.seq = (uint32_t)raw.size();
            r.c.vertex = v; r.c.origin_id = oid; r.c.metric = (uint16_t)metric; r.c.is_network = otype == 2;
            r.otype = otype; r.oadv = oadv; r.ext = -1;
            if (a->sr_enabled && sr_algo.count(oadv)) {
                const int32_t ei = ext_lookup(oadv, prefix, plen);
                if (ei >= 0) {
                    const auto &e = a->ext_prefixes[ei];
                    if (e.route_type == 1 && e.has_sid) {
                        r.ext = ei;
                        const uint64_t key = ((uint64_t)e.sid_value << 16) | ((uint64_t)e.sid_flags << 8) | (e.sid_is_label ? 1u : 0u);
                        auto ins = sid_class.emplace(key, (uint16_t)rt->t.sids.size());
                        if (ins.second) {
                            if (rt->t.sids.size() >= 0xFFFFu) throw std::length_error("sid classes");
                            rt->t.sids.push_back(hspf::SidDesc{e.sid_value, e.sid_flags, (uint8_t)(e.sid_is_label ? 1 : 0)});
                        }
                        r.c.sid_class = ins.first->second;
                    }
                }
            }
            raw.push_back(r);
        };
        for (uint32_t v = 0; v < V; ++v) {
            if (!f.is_router[v]) {
                const auto &nl = a->network_lsas[f.lsa_of[v]];
                add(v, nl.lsa_id & nl.mask, (uint32_t)__builtin_popcount(nl.mask), 0, 2, nl.adv_rtr, nl.lsa_id);
            } else {
                const auto &rl = a->router_lsas[f.lsa_of[v]];
                for (uint32_t k = 0; k < rl.n_links; ++k) {
                    const auto &l = a->links[rl.link_off + k];
                    if (l.link_type != HL_LINK_STUB) continue;
                    add(v, l.link_id & l.link_data, (uint32_t)__builtin_popcount(l.link_data), l.metric, 1, rl.adv_rtr, rl.lsa_id);
                }
            }
        }
        {   // (prefix, length, order of appearance): sort flat keys, then gather the records
            std::vector<std::pair<uint64_t, uint32_t>> order(raw.size());
            for (size_t i = 0; i < raw.size(); ++i) order[i] = {pkey(raw[i].prefix, raw[i].plen), raw[i].seq};
            std::sort(order.begin(), order.end());
            std::vector<Raw> sorted;
            sorted.reserve(raw.size());
            for (auto &kv : order) sorted.push_back(raw[kv.second]);
            raw.swap(sorted);
        }
        auto &t = rt->t;
        t.n_vertices = V;
        for (size_t i = 0; i < raw.size(); ++i) {
            if (i == 0 || raw[i].prefix != raw[i - 1].prefix || raw[i].plen != raw[i - 1].plen) {
                t.prefix.push_back(raw[i].prefix); t.plen.push_back(raw[i].plen); t.off.push_back((uint32_t)i);
            }
            t.contribs.push_back(raw[i].c);
            t.origin_type.push_back(raw[i].otype);
            t.origin_adv.push_back(raw[i].oadv);
            rt->ext_of.push_back(raw[i].ext);
        }
        t.off.push_back((uint32_t)raw.size());
        *out = guard.release();
        return HSPF_OK;
    } catch (const std::bad_alloc &) {
        return HSPF_E_NOMEM;
    } catch (...) {
        return HSPF_E_UNSUPPORTED;
    }
}

uint32_t hspf_ospfv2_rtable_prefixes(const hspf_ospfv2_rtable *rt) { return rt ? (uint32_t)rt->t.prefix.size() : 0; }
uint32_t hspf_ospfv2_rtable_contributors(const hspf_ospfv2_rtable *rt) { return rt ? (uint32_t)rt->t.contribs.size() : 0; }

int hspf_ospfv2_rtable_arrays(const hspf_ospfv2_rtable *rt, const uint32_t **prefix, const uint32_t **plen,
                              const uint32_t **off, const void **contribs) {
    if (!rt) return HSPF_E_INVAL;
    if (prefix) *prefix = rt->t.prefix.data();
    if (plen) *plen = rt->t.plen.data();
    if (off) *off = rt->t.off.data();
    if (contribs) *contribs = rt->t.contribs.data();
    return HSPF_OK;
}

int hspf_ospfv2_routes_from_cells(const hl_ospfv2_area *a, const hspf_ospfv2_rtable *rt, const hl_route_cell *cells,
                                  const uint32_t *gather_v, const uint64_t *gather_nh, uint32_t n_gather,
                                  hl_ospfv2_result *out) {
    if (!a || !rt || !cells || !out || (n_gather && (!gather_v || !gather_nh))) return HSPF_E_INVAL;
    try {
        out->n_vertices = out->n_routers = out->n_routes = out->n_nexthops = 0;
        out->transit_capability = 0;
        out->root_found = 0;
        hspf_ospfv2_flat f;
        int rc = flatten(a, f);
        if (rc) return rc;
        const uint32_t V = (uint32_t)f.ids.size();
        if (V != rt->t.n_vertices) return HSPF_E_INVAL;          // not the LSDB the table was built from
        auto rit = f.rtr_vertex.find(a->router_id);
        if (rit == f.rtr_vertex.end()) return HSPF_OK;
        out->root_found = 1;
        const uint32_t root = rit->second;
        // atoms -> next hops: only the transit networks next to the root are ever looked up (Resolver::resolve)
        std::vector<uint64_t> sparse_nh(V, 0);
        for (uint32_t i = 0; i < n_gather; ++i) {
            if (gather_v[i] >= V) return HSPF_E_INVAL;
            sparse_nh[gather_v[i]] = gather_nh[i];
        }
        Resolver rs{f, a, root, sparse_nh.data(), 1, {}, {}, {}};
        rs.atom_nh.resize(64);
        rs.atom_done.assign(64, 0);
        for (uint32_t i = 0; i < a->n_ifaces; ++i)
            if (a->ifaces[i].n_nbrs > 0) rs.ifaces_with_nbrs.push_back((int)i);
        // SRGBs per router (area_router_information, ospfv2/spf.rs:617-654)
        std::unordered_map<uint32_t, RouterInfo> ri_cache;
        const RouterInfo no_ri;
        if (a->sr_enabled) {
            for (uint32_t i = 0; i < a->n_ri_lsas; ++i) {
                const auto &l = a->ri_lsas[i];
                if (l.age == HL_LSA_MAX_AGE) continue;
                RouterInfo &ri = ri_cache[l.adv_rtr];
                if (l.has_sr_algo) ri.has_sr_algo = true;
                for (uint32_t k = 0; k < l.n_srgb; ++k) ri.srgb.push_back(&a->srgbs[l.srgb_off + k]);
            }
        }
        auto cached_ri = [&](uint32_t rid) -> const RouterInfo & {
            auto it = ri_cache.find(rid);
            return it == ri_cache.end() ? no_ri : it->second;
        };
        const RouterInfo &local_ri = cached_ri(a->router_id);

        const auto &t = rt->t;
        const uint32_t P = (uint32_t)t.prefix.size();
        uint32_t n_routes = 0, n_nh = 0;
        std::vector<Nh> set;
        for (uint32_t p = 0; p < P; ++p) {
            const hl_route_cell &c = cells[p];
            if (!(c.flags & HL_CELL_PRESENT)) continue;
            if (c.flags & HL_CELL_MIXED_SID) return HSPF_E_UNSUPPORTED;
            if (c.winner < t.off[p] || c.winner >= t.off[p + 1]) return HSPF_E_INVAL;
            const hspf::RouteContrib &w = t.contribs[c.winner];
            const hl_ospfv2_ext_prefix *ep = nullptr;
            if (w.sid_class) {
                const int32_t e = rt->ext_of[c.winner];
                if (e < 0 || (uint32_t)e >= a->n_ext_prefixes) return HSPF_E_INVAL;
                ep = &a->ext_prefixes[e];
            }
            const bool local = (c.flags & HL_CELL_CONNECTED) != 0;
            hl_route_net o{};
            o.prefix = t.prefix[p]; o.mask = t.plen[p] == 0 ? 0 : 0xFFFFFFFFu << (32 - t.plen[p]);
            o.metric = c.metric; o.flags = local ? HL_ROUTE_CONNECTED : 0; o.origin_type = t.origin_type[c.winner];
            o.origin_adv_rtr = t.origin_adv[c.winner]; o.origin_lsa_id = w.origin_id;
            if (ep) {
                o.has_prefix_sid = 1; o.prefix_sid_value = ep->sid_value; o.prefix_sid_flags = ep->sid_flags;
                o.prefix_sid_is_label = ep->sid_is_label;
                if (!(local && (!(ep->sid_flags & HL_PSID_NP) || (ep->sid_flags & HL_PSID_E)))) {
                    if (!ep->sid_is_label) {
                        uint32_t lab;
                        if (!local_ri.srgb.empty() && index_to_label(ep->sid_value, local_ri.srgb, &lab)) { o.has_sr_label = 1; o.sr_label = lab; }
                    } else {
                        o.has_sr_label = 1; o.sr_label = ep->sid_value;
                    }
                }
            }
            set.clear();
            uint64_t m = c.nh_mask;
            while (m) {
                const uint32_t atom = (uint32_t)__builtin_ctzll(m);
                m &= m - 1;
                const bool last_hop = (c.lasthop_mask >> atom) & 1u;
                for (Nh x : rs.resolve(atom)) {
                    if (ep && x.has_nbr) {
                        uint32_t lab = 0; bool ok = false, decided = false;
                        if (last_hop) {
                            if (!(ep->sid_flags & HL_PSID_NP)) { lab = 3; ok = decided = true; }
                            else if (ep->sid_flags & HL_PSID_E) { lab = 0; ok = decided = true; }
                        }
                        if (!decided) {
                            if (!ep->sid_is_label) {
                                const RouterInfo &nri = cached_ri(x.nbr);
                                if (!nri.srgb.empty()) ok = index_to_label(ep->sid_value, nri.srgb, &lab);
                            } else {
                                lab = last_hop ? ep->sid_value : 3u; ok = true;
                            }
                        }
                        if (ok) { x.has_label = 1; x.label = lab; }
                    }
                    auto it = std::lower_bound(set.begin(), set.end(), x, nh_less);
                    if (it != set.end() && nh_same_key(*it, x)) {
                        // two atoms, one next hop: the reference keeps whichever advertiser came last; the
                        // cell cannot tell unless both agree
                        if (it->iface != x.iface || it->nbr != x.nbr || it->has_nbr != x.has_nbr ||
                            it->has_label != x.has_label || it->label != x.label) return HSPF_E_UNSUPPORTED;
                    } else {
                        set.insert(it, x);
                    }
                }
            }
            if (set.size() > a->max_paths) set.resize(a->max_paths);
            o.nh_off = n_nh; o.n_nh = (uint32_t)set.size();
            if (n_routes < out->routes_cap && n_nh + set.size() <= out->nexthops_cap) {
                out->routes[n_routes] = o;
                for (const Nh &x : set) {
                    hl_nexthop h{};
                    h.iface = x.iface; h.addr = x.has_addr ? x.addr : 0; h.nbr_router_id = x.has_nbr ? x.nbr : 0;
                    h.sr_label = x.has_label ? x.label : 0;
                    h.has_addr = x.has_addr; h.has_nbr = x.has_nbr; h.has_label = x.has_label;
                    out->nexthops[n_nh + (&x - set.data())] = h;
                }
            }
            ++n_routes; n_nh += (uint32_t)set.size();
        }
        out->n_routes = n_routes; out->n_nexthops = n_nh;
        if (n_routes > out->routes_cap || n_nh > out->nexthops_cap) return HSPF_E_NOMEM;
        return HSPF_OK;
    } catch (const std::bad_alloc &) {
        return HSPF_E_NOMEM;
    } catch (...) {
        return HSPF_E_INVAL;
    }
}


/* ---- trigger-keyed recomputation (holo_spf_lsdb.h) ---------------------------------------------- */

int hspf_ospfv2_spf_computation_type(const hl_lsa_trigger *tr, uint32_t n, hl_spf_computation *out) {
    if (!out || (n && !tr)) return HSPF_E_INVAL;
    out->kind = HL_SPF_PARTIAL;
    out->n_inter_network = out->n_inter_router = out->n_external = 0;
    // Router- and Network-LSAs are topology; the SR opaque LSAs are treated the same way (ospfv2/spf.rs:101-121)
    for (uint32_t i = 0; i < n; ++i) {
        const auto &t = tr[i];
        const bool sr_opaque_area = t.lsa_type == 10 && (t.opaque_type == 4 || t.opaque_type == 7 || t.opaque_type == 8);
        const bool sr_opaque_as = t.lsa_type == 11 && t.opaque_type == 7;
        if (t.lsa_type == 1 || t.lsa_type == 2 || sr_opaque_area || sr_opaque_as) {
            out->kind = HL_SPF_FULL;
            return HSPF_OK;
        }
    }
    try {
        std::vector<std::pair<uint32_t, uint32_t>> net, ext;      // (address, prefix length): Ipv4Network order
        std::vector<uint32_t> rtr;
        for (uint32_t i = 0; i < n; ++i) {
            const auto &t = tr[i];
            if (t.lsa_type == 3) net.emplace_back(t.lsa_id, (uint32_t)__builtin_popcount(t.mask));
            else if (t.lsa_type == 4) rtr.push_back(t.lsa_id);
            else if (t.lsa_type == 5) ext.emplace_back(t.lsa_id, (uint32_t)__builtin_popcount(t.mask));
        }
        auto uniq = [](auto &v) { std::sort(v.begin(), v.end()); v.erase(std::unique(v.begin(), v.end()), v.end()); };
        uniq(net); uniq(rtr); uniq(ext);
        out->n_inter_network = (uint32_t)net.size();
        out->n_inter_router = (uint32_t)rtr.size();
        out->n_external = (uint32_t)ext.size();
        if (net.size() > out->cap || rtr.size() > out->cap || ext.size() > out->cap) return HSPF_E_NOMEM;
        if ((!net.empty() && !out->inter_network) || (!rtr.empty() && !out->inter_router) || (!ext.empty() && !out->external))
            return HSPF_E_INVAL;
        auto mask_of = [](uint32_t len) { return len == 0 ? 0u : 0xFFFFFFFFu << (32 - len); };
        for (size_t i = 0; i < net.size(); ++i) out->inter_network[i] = hl_ipv4_net{net[i].first, mask_of(net[i].second)};
        for (size_t i = 0; i < rtr.size(); ++i) out->inter_router[i] = rtr[i];
        for (size_t i = 0; i < ext.size(); ++i) out->external[i] = hl_ipv4_net{ext[i].first, mask_of(ext[i].second)};
        return HSPF_OK;
    } catch (const std::bad_alloc &) {
        return HSPF_E_NOMEM;
    }
}

int hspf_ospfv2_flat_update(hspf_ospfv2_flat *flat, const hl_ospfv2_area *na, const hl_lsa_trigger *tr, uint32_t n,
                            uint32_t *kind, uint32_t *edges, uint32_t *costs, uint32_t cap, uint32_t *n_changed) {
    if (!flat || !flat->area || !na || !kind || !n_changed || (n && !tr)) return HSPF_E_INVAL;
    try {
        *n_changed = 0;
        hspf_ospfv2_flat &f = *flat;
        const hl_ospfv2_area *oa = f.area;
        auto rebuild = [&]() -> int {
            hspf_ospfv2_flat fresh;
            const int rc = flatten(na, fresh);
            if (rc) return rc;
            f = std::move(fresh);
            *kind = HSPF_FLAT_REBUILT;
            return HSPF_OK;
        };
        // the shortcuts below index the new image with the old image's LSA and link positions
        const bool same_layout = oa->n_router_lsas == na->n_router_lsas && oa->n_network_lsas == na->n_network_lsas &&
                                 oa->n_links == na->n_links && oa->n_attached == na->n_attached;
        std::vector<uint32_t> cost_rows;       // router vertices whose link metrics may have changed
        bool graph_trigger = false;
        for (uint32_t i = 0; i < n; ++i) {
            const auto &t = tr[i];
            if (t.lsa_type != 1 && t.lsa_type != 2) continue;   // nothing else bears on the graph
            graph_trigger = true;
            if (!same_layout) return rebuild();
            if (t.lsa_type == 1) {
                // the LSA at the same index must be this LSA, before and after, with the same links
                const hl_ospfv2_router_lsa *ol = nullptr, *nl = nullptr;
                uint32_t idx = 0;
                for (; idx < oa->n_router_lsas; ++idx)
                    if (oa->router_lsas[idx].adv_rtr == t.adv_rtr && oa->router_lsas[idx].lsa_id == t.lsa_id) { ol = &oa->router_lsas[idx]; break; }
                if (!ol) return rebuild();                                      // a new LSA: a vertex may appear
                nl = &na->router_lsas[idx];
                if (nl->adv_rtr != t.adv_rtr || nl->lsa_id != t.lsa_id) return rebuild();
                if ((ol->age == HL_LSA_MAX_AGE) != (nl->age == HL_LSA_MAX_AGE)) return rebuild();
                if (ol->n_links != nl->n_links || ol->link_off != nl->link_off) return rebuild();
                for (uint32_t k = 0; k < ol->n_links; ++k) {
                    const auto &x = oa->links[ol->link_off + k], &y = na->links[nl->link_off + k];
                    if (x.link_type != y.link_type || x.link_id != y.link_id || x.link_data != y.link_data) return rebuild();
                }
                if (t.adv_rtr == t.lsa_id && nl->age != HL_LSA_MAX_AGE) {
                    auto it = f.rtr_vertex.find(t.adv_rtr);
                    if (it == f.rtr_vertex.end() || f.lsa_of[it->second] != idx) return rebuild();
                    cost_rows.push_back(it->second);
                }
            } else {
                const hl_ospfv2_network_lsa *ol = nullptr;
                uint32_t idx = 0;
                for (; idx < oa->n_network_lsas; ++idx)
                    if (oa->network_lsas[idx].adv_rtr == t.adv_rtr && oa->network_lsas[idx].lsa_id == t.lsa_id) { ol = &oa->network_lsas[idx]; break; }
                if (!ol) return rebuild();
                const hl_ospfv2_network_lsa *nl = &na->network_lsas[idx];
                if (nl->adv_rtr != t.adv_rtr || nl->lsa_id != t.lsa_id) return rebuild();
                if ((ol->age == HL_LSA_MAX_AGE) != (nl->age == HL_LSA_MAX_AGE)) return rebuild();
                if (ol->n_att != nl->n_att || ol->att_off != nl->att_off) return rebuild();
                for (uint32_t k = 0; k < ol->n_att; ++k)
                    if (oa->attached[ol->att_off + k] != na->attached[nl->att_off + k]) return rebuild();
            }
        }
        f.area = na;
        if (!graph_trigger) { *kind = HSPF_FLAT_UNCHANGED; return HSPF_OK; }
        uint32_t changed = 0;
        for (uint32_t v : cost_rows)
            for (uint32_t e = f.row[v]; e < f.row[v + 1]; ++e) {
                const uint32_t c = na->links[f.link_index[e]].metric;
                if (c == f.cost[e]) continue;
                f.cost[e] = c;
                if (changed < cap && edges && costs) { edges[changed] = e; costs[changed] = c; }
                ++changed;
            }
        *n_changed = changed;
        *kind = changed ? HSPF_FLAT_COSTS : HSPF_FLAT_UNCHANGED;
        return changed > cap ? HSPF_E_NOMEM : HSPF_OK;
    } catch (const std::bad_alloc &) {
        return HSPF_E_NOMEM;
    } catch (...) {
        return HSPF_E_INVAL;
    }
}

}  // extern "C"
