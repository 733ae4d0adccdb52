// ospfv3_host.cc — OSPFv3 host side of the engine: LSDB image -> CSR and device
// results -> Vertex.nexthops / area router table / intra-area routes.
//
// OSPFv3 differences from the OSPFv2 flattener (holo-ospf/src/ospfv3/spf.rs):
//  * VertexId::Network is (router_id, iface_id) (:37-41);
//  * a Router vertex aggregates ALL Router-LSA fragments of its advertising router that
//    carry the R-bit (and the V6-bit for the IPv6 address family) (:316-342); its links
//    are the concatenation of the fragments in LsaKey order (:381-398);
//  * first hops use the interface named by the root's link (`iface_id` == system
//    ifindex, :187-190) and the neighbour's Link-LSA link-local address (:592-611);
//  * stub prefixes come from Intra-Area-Prefix-LSAs in LSDB order (:420-477).
// The SPT (distance, hops, first-hop atom sets) is computed by spf_batch_kernel.
#include <algorithm>
#include <cstring>
#include <map>
#include <new>
#include <unordered_map>
#include <unordered_set>
#include <array>
#include <set>
#include <tuple>
#include <memory>
#include <vector>

#include "holo_spf_lsdb.h"
#include "route_cells.h"
#include "spf_one_root.h"

namespace {

constexpr uint32_t kNone = 0xFFFFFFFFu;

struct Nh6 { uint32_t sort, iface, nbr; hl_ip_addr addr; uint8_t has_addr, has_nbr; };
inline int addr_cmp(const hl_ip_addr &a, const hl_ip_addr &b) {
    if (a.is_v6 != b.is_v6) return a.is_v6 < b.is_v6 ? -1 : 1;
    return std::memcmp(a.bytes, b.bytes, 16);
}
inline bool nh_less(const Nh6 &a, const Nh6 &b) {
    if (a.sort != b.sort) return a.sort < b.sort;
    if (a.has_addr != b.has_addr) return a.has_addr < b.has_addr;
    return a.has_addr && addr_cmp(a.addr, b.addr) < 0;
}
inline bool nh_same(const Nh6 &a, const Nh6 &b) {
    return a.sort == b.sort && a.has_addr == b.has_addr && (!a.has_addr || addr_cmp(a.addr, b.addr) == 0);
}
void nh_insert(std::vector<Nh6> &set, const Nh6 &x) {
    auto it = std::lower_bound(set.begin(), set.end(), x, nh_less);
    if (it != set.end() && nh_same(*it, x)) *it = x; else set.insert(it, x);
}

}  // namespace

struct hspf_ospfv3_flat {
    const hl_ospfv3_area *area = nullptr;
    uint32_t n_net = 0;
    std::vector<uint32_t> rid, ifid;            // [V] vertex identity
    std::vector<uint8_t> is_router;
    std::vector<uint32_t> first_lsa;            // [V] network LSA index / first router fragment index
    std::vector<std::vector<uint32_t>> frags;   // [V] router fragments in LsaKey order
    std::vector<uint32_t> row, col, cost, link_index;
    std::vector<uint8_t> vflags;
    std::unordered_map<uint64_t, uint32_t> net_vertex;   // (router_id<<32 | iface_id) -> vertex
    std::unordered_map<uint32_t, uint32_t> rtr_vertex;
};

namespace {

int flatten(const hl_ospfv3_area *a, hspf_ospfv3_flat &f) {
    f.area = a;
    // fragments in LsaKey order
    std::vector<uint32_t> ord(a->n_router_lsas);
    for (uint32_t i = 0; i < a->n_router_lsas; ++i) ord[i] = i;
    std::stable_sort(ord.begin(), ord.end(), [&](uint32_t x, uint32_t y) {
        const auto &p = a->router_lsas[x], &q = a->router_lsas[y];
        return p.adv_rtr != q.adv_rtr ? p.adv_rtr < q.adv_rtr : p.lsa_id < q.lsa_id;
    });
    std::map<uint32_t, std::vector<uint32_t>> by_rtr;
    for (uint32_t i : ord) {
        const auto &r = a->router_lsas[i];
        if (r.age == HL_LSA_MAX_AGE || !(r.options & HL_V3_OPT_R)) continue;
        if (a->af_ipv6 && !(r.options & HL_V3_OPT_V6)) continue;
        by_rtr[r.adv_rtr].push_back(i);
    }
    std::map<std::pair<uint32_t, uint32_t>, uint32_t> nets;
    for (uint32_t i = 0; i < a->n_network_lsas; ++i) {
        const auto &n = a->network_lsas[i];
        auto key = std::make_pair(n.adv_rtr, n.lsa_id);
        if (nets.count(key)) continue;             // LSDB keys are unique; keep the first
        nets.emplace(key, i);
    }
    for (auto it = nets.begin(); it != nets.end();) {
        if (a->network_lsas[it->second].age == HL_LSA_MAX_AGE) it = nets.erase(it); else ++it;
    }
    f.n_net = (uint32_t)nets.size();
    const uint32_t V = f.n_net + (uint32_t)by_rtr.size();
    f.rid.resize(V); f.ifid.assign(V, 0); f.is_router.resize(V); f.first_lsa.resize(V); f.frags.resize(V); f.vflags.resize(V);
    uint32_t v = 0;
    for (auto &kv : nets) {
        f.rid[v] = kv.first.first; f.ifid[v] = kv.first.second; f.is_router[v] = 0; f.first_lsa[v] = kv.second; f.vflags[v] = 0;
        f.net_vertex.emplace(((uint64_t)kv.first.first << 32) | kv.first.second, v);
        ++v;
    }
    for (auto &kv : by_rtr) {
        f.rid[v] = kv.first; f.is_router[v] = 1; f.first_lsa[v] = kv.second[0]; f.frags[v] = kv.second; f.vflags[v] = HSPF_VF_HOP;
        f.rtr_vertex.emplace(kv.first, v);
        ++v;
    }
    struct Raw { uint32_t u, v, cost, link; };
    std::vector<Raw> raw;
    std::vector<uint32_t> att;
    for (uint32_t u = 0; u < V; ++u) {
        if (!f.is_router[u]) {
            const auto &n = a->network_lsas[f.first_lsa[u]];
            att.assign(a->attached + n.att_off, a->attached + n.att_off + n.n_att);
            std::sort(att.begin(), att.end());
            att.erase(std::unique(att.begin(), att.end()), att.end());
            for (uint32_t r : att) {
                auto it = f.rtr_vertex.find(r);
                if (it != f.rtr_vertex.end()) raw.push_back({u, it->second, 0, kNone});
            }
        } else {
            for (uint32_t li : f.frags[u]) {
                const auto &r = a->router_lsas[li];
                for (uint32_t k = 0; k < r.n_links; ++k) {
                    const auto &l = a->links[r.link_off + k];
                    uint32_t tgt = kNone;
                    if (l.link_type == HL_LINK_TRANSIT) {
                        auto it = f.net_vertex.find(((uint64_t)l.nbr_router_id << 32) | l.nbr_iface_id);
                        if (it != f.net_vertex.end()) tgt = it->second;
                    } else {
                        auto it = f.rtr_vertex.find(l.nbr_router_id);
                        if (it != f.rtr_vertex.end()) tgt = it->second;
                    }
                    if (tgt != kNone) raw.push_back({u, tgt, l.metric, r.link_off + k});
                }
            }
        }
    }
    std::unordered_set<uint64_t> have;
    have.reserve(raw.size() * 2);
    for (auto &e : raw) have.insert(((uint64_t)e.u << 32) | e.v);
    auto keep = [&](const Raw &e) { return e.u != e.v && have.count(((uint64_t)e.v << 32) | e.u); };
    f.row.assign(V + 1, 0);
    for (auto &e : raw) if (keep(e)) f.row[e.u + 1]++;
    for (uint32_t i = 0; i < V; ++i) f.row[i + 1] += f.row[i];
    const uint32_t E = f.row[V];
    f.col.resize(E); f.cost.resize(E); f.link_index.resize(E);
    std::vector<uint32_t> fill(f.row.begin(), f.row.end() - 1);
    for (auto &e : raw) if (keep(e)) { const uint32_t k = fill[e.u]++; f.col[k] = e.v; f.cost[k] = e.cost; f.link_index[k] = e.link; }
    return HSPF_OK;
}

void fill_csr(const hspf_ospfv3_flat &f, hspf_csr *c) {
    std::memset(c, 0, sizeof(*c));
    c->n_vertices = (uint32_t)f.rid.size();
    c->n_edges = (uint32_t)f.col.size();
    c->row_ptr = f.row.data(); c->col = f.col.data(); c->cost = f.cost.data(); c->vflags = f.vflags.data();
    c->reject_above = 0xFFFFFFFEu;
    c->saturate_at = 0xFFFFu;
}

struct Resolver {
    const hspf_ospfv3_flat &f;
    const hl_ospfv3_area *a;
    uint32_t root;
    const uint64_t *nh_mask;
    uint32_t nhw;
    std::vector<std::vector<Nh6>> atom_nh;
    std::vector<uint8_t> atom_done;

    int iface_by_ifindex(uint32_t ifindex) const {
        for (uint32_t i = 0; i < a->n_ifaces; ++i) if (a->ifaces[i].ifindex == ifindex) return (int)i;
        return -1;
    }
    bool lladdr(uint32_t iface, uint32_t nbr_rid, uint32_t nbr_ifid, hl_ip_addr *out) const {
        for (uint32_t i = 0; i < a->n_link_lsas; ++i) {
            const auto &l = a->link_lsas[i];
            if (l.iface == iface && l.adv_rtr == nbr_rid && l.lsa_id == nbr_ifid) {
                if (l.age == HL_LSA_MAX_AGE) return false;
                *out = l.linklocal;
                return true;
            }
        }
        return false;
    }
    std::vector<Nh6> vertex_nexthops(uint32_t v) {
        std::vector<Nh6> set;
        for (uint32_t w = 0; w < nhw; ++w) {
            uint64_t m = nh_mask[(size_t)v * nhw + w];
            while (m) {
                const uint32_t atom = w * 64 + (uint32_t)__builtin_ctzll(m);
                m &= m - 1;
                for (const Nh6 &x : resolve(atom)) nh_insert(set, x);
            }
        }
        return set;
    }
    const std::vector<Nh6> &resolve(uint32_t atom) {
        if (atom_done[atom]) return atom_nh[atom];
        atom_done[atom] = 1;
        hspf_csr c;
        fill_csr(f, &c);
        uint32_t tail = 0, e = 0;
        std::vector<Nh6> out;
        if (hspf_atom_decode(&c, root, atom, &tail, &e) == HSPF_OK) {
            const uint32_t dest = f.col[e];
            if (tail == root) {
                const auto &pl = a->links[f.link_index[e]];
                const int ii = iface_by_ifindex(pl.iface_id);
                if (ii >= 0 && a->ifaces[ii].if_type != HL_IF_VLINK) {
                    const auto &iface = a->ifaces[ii];
                    if (f.is_router[dest]) {
                        hl_ip_addr addr;
                        if (lladdr((uint32_t)ii, pl.nbr_router_id, pl.nbr_iface_id, &addr))
                            out.push_back(Nh6{iface.sort_key, (uint32_t)ii, f.rid[dest], addr, 1, 1});
                    } else {
                        out.push_back(Nh6{iface.sort_key, (uint32_t)ii, 0, hl_ip_addr{}, 0, 0});
                    }
                }
            } else {
                // parent is a transit network attached to the root (ospfv3/spf.rs:229-279)
                const auto &pn = a->network_lsas[f.first_lsa[tail]];
                const hl_ospfv3_link *dest_link = nullptr;
                for (uint32_t li : f.frags[dest]) {
                    const auto &r = a->router_lsas[li];
                    for (uint32_t k = 0; k < r.n_links && !dest_link; ++k) {
                        const auto &l = a->links[r.link_off + k];
                        if (l.nbr_router_id == pn.adv_rtr && l.nbr_iface_id == pn.lsa_id) dest_link = &l;
                    }
                    if (dest_link) break;
                }
                if (dest_link) {
                    std::vector<Nh6> pnh = vertex_nexthops(tail);
                    if (!pnh.empty()) {
                        const Nh6 &p0 = pnh.front();
                        hl_ip_addr addr;
                        if (lladdr(p0.iface, f.rid[dest], dest_link->iface_id, &addr))
                            out.push_back(Nh6{p0.sort, p0.iface, f.rid[dest], addr, 1, 1});
                    }
                }
            }
        }
        atom_nh[atom] = std::move(out);
        return atom_nh[atom];
    }
};

struct Route6 { hl_ip_addr prefix; uint8_t len, flags, otype, options; uint32_t metric, oadv, oid; std::vector<Nh6> nh; bool live; };

struct PKey {
    hl_ip_addr a; uint8_t len;
    bool operator<(const PKey &o) const {
        int c = addr_cmp(a, o.a);
        if (c) return c < 0;
        return len < o.len;
    }
};

}  // namespace

extern "C" {

int hspf_ospfv3_flatten(const hl_ospfv3_area *area, hspf_ospfv3_flat **out) {
    if (!area || !out) return HSPF_E_INVAL;
    *out = nullptr;
    try {
        auto *f = new hspf_ospfv3_flat();
        int rc = flatten(area, *f);
        if (rc) { delete f; return rc; }
        *out = f;
        return HSPF_OK;
    } catch (const std::bad_alloc &) { return HSPF_E_NOMEM; } catch (...) { return HSPF_E_INVAL; }
}

void hspf_ospfv3_flat_free(hspf_ospfv3_flat *flat) { delete flat; }

int hspf_ospfv3_spf_computation_type(const hl_lsa_trigger6 *tr, uint32_t n, const hl_ip_prefix *prefixes, uint32_t n_prefixes,
                                     hl_spf_computation6 *out) {
    if (!out || (n && !tr) || (n_prefixes && !prefixes)) return HSPF_E_INVAL;
    out->kind = HL_SPF_PARTIAL;
    out->n_intra = out->n_inter_network = out->n_inter_router = out->n_external = 0;
    auto normalized = [](uint16_t c) -> uint16_t { return (c >= 33 && c <= 41) ? (uint16_t)(c - 32) : c; };   // Ext* -> legacy code
    for (uint32_t i = 0; i < n; ++i) {
        const uint16_t c = normalized(tr[i].function_code);
        if (c == 1 || c == 2 || c == 8 || c == 12) { out->kind = HL_SPF_FULL; return HSPF_OK; }
        if ((uint64_t)tr[i].prefix_off + tr[i].n_prefixes > n_prefixes) return HSPF_E_INVAL;
    }
    try {
        using Key = std::tuple<uint8_t, std::array<uint8_t, 16>, uint8_t>;      // IpNetwork Ord: family, address, length
        auto key = [](const hl_ip_prefix &p) { std::array<uint8_t, 16> b; std::memcpy(b.data(), p.addr.bytes, 16); return Key{p.addr.is_v6, b, p.len}; };
        std::map<Key, hl_ip_prefix> intra, inter, ext;
        std::set<uint32_t> rtr;
        for (uint32_t i = 0; i < n; ++i) {
            const uint16_t c = normalized(tr[i].function_code);
            const hl_ip_prefix *p = prefixes + tr[i].prefix_off;
            if (c == 9) for (uint32_t k = 0; k < tr[i].n_prefixes; ++k) intra.emplace(key(p[k]), p[k]);
            else if (c == 3) { if (tr[i].n_prefixes) inter.emplace(key(p[0]), p[0]); }
            else if (c == 4) rtr.insert(tr[i].router_id);
            else if (c == 5) { if (tr[i].n_prefixes) ext.emplace(key(p[0]), p[0]); }
        }
        out->n_intra = (uint32_t)intra.size(); out->n_inter_network = (uint32_t)inter.size();
        out->n_inter_router = (uint32_t)rtr.size(); out->n_external = (uint32_t)ext.size();
        if (intra.size() > out->cap || inter.size() > out->cap || rtr.size() > out->cap || ext.size() > out->cap) return HSPF_E_NOMEM;
        if ((!intra.empty() && !out->intra) || (!inter.empty() && !out->inter_network) || (!rtr.empty() && !out->inter_router) ||
            (!ext.empty() && !out->external)) return HSPF_E_INVAL;
        uint32_t k = 0;
        for (auto &kv : intra) out->intra[k++] = kv.second;
        k = 0;
        for (auto &kv : inter) out->inter_network[k++] = kv.second;
        k = 0;
        for (uint32_t r : rtr) out->inter_router[k++] = r;
        k = 0;
        for (auto &kv : ext) out->external[k++] = kv.second;
        return HSPF_OK;
    } catch (const std::bad_alloc &) { return HSPF_E_NOMEM; }
}

int hspf_ospfv3_flat_update(hspf_ospfv3_flat *flat, const hl_ospfv3_area *na, uint32_t *kind, uint32_t *edges,
                            uint32_t *costs, uint32_t cap, uint32_t *n_changed) {
    if (!flat || !na || !kind || !n_changed) return HSPF_E_INVAL;
    try {
        *n_changed = 0;
        hspf_ospfv3_flat fresh;
        const int rc = flatten(na, fresh);
        if (rc) return rc;
        hspf_ospfv3_flat &f = *flat;
        // same vertices, same edges between them, same per-edge link records: only metrics can differ
        const bool same_graph = f.rid == fresh.rid && f.ifid == fresh.ifid && f.is_router == fresh.is_router && f.row == fresh.row &&
                                f.col == fresh.col && f.vflags == fresh.vflags;
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
        f = std::move(fresh);                    // LSA / link indices of the new image
        *n_changed = changed;
        *kind = changed ? HSPF_FLAT_COSTS : HSPF_FLAT_UNCHANGED;
        return changed > cap ? HSPF_E_NOMEM : HSPF_OK;
    } catch (const std::bad_alloc &) { return HSPF_E_NOMEM; } catch (...) { return HSPF_E_INVAL; }
}

int hspf_ospfv3_flat_csr(const hspf_ospfv3_flat *flat, hspf_csr *out) {
    if (!flat || !out) return HSPF_E_INVAL;
    fill_csr(*flat, out);
    return HSPF_OK;
}

int hspf_ospfv3_flat_vertices(const hspf_ospfv3_flat *flat, const uint32_t **router_ids, const uint32_t **iface_ids,
                              const uint8_t **is_router, uint32_t *n_vertices) {
    if (!flat) return HSPF_E_INVAL;
    if (router_ids) *router_ids = flat->rid.data();
    if (iface_ids) *iface_ids = flat->ifid.data();
    if (is_router) *is_router = flat->is_router.data();
    if (n_vertices) *n_vertices = (uint32_t)flat->rid.size();
    return HSPF_OK;
}

uint32_t hspf_ospfv3_flat_router_vertex(const hspf_ospfv3_flat *flat, uint32_t router_id) {
    if (!flat) return kNone;
    auto it = flat->rtr_vertex.find(router_id);
    return it == flat->rtr_vertex.end() ? kNone : it->second;
}

}  // extern "C" (reopened below)

namespace {

// Everything run_area + update_rib_intra_area do after the SPT for OSPFv3 (spf.rs:627-724 with
// the hooks of ospfv3/spf.rs:164-283, 420-477, 592-611; route.rs:343-446), over the planes of
// the root's job in the vertex order of `f`.
int area_from_planes(const hspf_ospfv3_flat &f, const hl_ospfv3_area *a, uint32_t root, const uint32_t *dist,
                     const uint16_t *hops, const uint64_t *nh, uint32_t nhw, hl_ospfv3_result *out) {
    const uint32_t V = (uint32_t)f.rid.size();
    Resolver rs{f, a, root, nh, nhw, {}, {}};
    rs.atom_nh.resize((size_t)64 * nhw);
    rs.atom_done.assign((size_t)64 * nhw, 0);
    std::vector<uint32_t> spt;
    for (uint32_t v = 0; v < V; ++v) if (dist[v] != HSPF_DIST_INF) spt.push_back(v);
    std::vector<std::vector<Nh6>> vnh(V);
    for (uint32_t v : spt) vnh[v] = rs.vertex_nexthops(v);

    // ---- intra-area routes from Intra-Area-Prefix-LSAs in LsaKey order ----------
    std::vector<uint32_t> iord(a->n_iap_lsas);
    for (uint32_t i = 0; i < a->n_iap_lsas; ++i) iord[i] = i;
    std::stable_sort(iord.begin(), iord.end(), [&](uint32_t x, uint32_t y) {
        const auto &p = a->iap_lsas[x], &q = a->iap_lsas[y];
        return p.adv_rtr != q.adv_rtr ? p.adv_rtr < q.adv_rtr : p.lsa_id < q.lsa_id;
    });
    std::map<PKey, uint32_t> rib_idx;
    std::vector<Route6> rib;
    for (uint32_t i : iord) {
        const auto &l = a->iap_lsas[i];
        if (l.age == HL_LSA_MAX_AGE) continue;
        uint32_t v = kNone;
        if (l.ref_type == HL_V3_REF_ROUTER) {
            if (l.ref_lsa_id != 0) continue;
            auto it = f.rtr_vertex.find(l.ref_adv_rtr);
            if (it != f.rtr_vertex.end()) v = it->second;
        } else if (l.ref_type == HL_V3_REF_NETWORK) {
            auto it = f.net_vertex.find(((uint64_t)l.ref_adv_rtr << 32) | l.ref_lsa_id);
            if (it != f.net_vertex.end()) v = it->second;
        }
        if (v == kNone || dist[v] == HSPF_DIST_INF) continue;
        for (uint32_t k = 0; k < l.n_prefixes; ++k) {
            const auto &px = a->prefixes[l.prefix_off + k];
            if (px.options & HL_PFX_OPT_NU) continue;
            uint32_t m = dist[v] + px.metric;
            if (m > 0xFFFF) m = 0xFFFF;
            PKey key{px.addr, px.len};
            auto it = rib_idx.find(key);
            Route6 *cur = (it != rib_idx.end() && rib[it->second].live) ? &rib[it->second] : nullptr;
            if (cur && m > cur->metric) continue;
            uint8_t otype; uint32_t oadv, oid;
            if (f.is_router[v]) { const auto &r = a->router_lsas[f.first_lsa[v]]; otype = 1; oadv = r.adv_rtr; oid = r.lsa_id; }
            else { const auto &n = a->network_lsas[f.first_lsa[v]]; otype = 2; oadv = n.adv_rtr; oid = n.lsa_id; }
            if (!f.is_router[v] && cur) {
                if (m > cur->metric || oid < cur->oid) continue;
                cur->live = false;
                cur = nullptr;
            }
            Route6 nr{px.addr, px.len, (uint8_t)(hops[v] == 0 ? HL_ROUTE_CONNECTED : 0), otype, px.options, m, oadv, oid, vnh[v], true};
            Route6 *route;
            if (cur) {
                if (nr.metric < cur->metric) *cur = nr;
                else if (nr.metric == cur->metric) for (const Nh6 &x : nr.nh) nh_insert(cur->nh, x);
                route = cur;
            } else if (it != rib_idx.end()) {
                rib[it->second] = nr; route = &rib[it->second];
            } else {
                rib_idx.emplace(key, (uint32_t)rib.size()); rib.push_back(nr); route = &rib.back();
            }
            if (route->nh.size() > a->max_paths) route->nh.resize(a->max_paths);
        }
    }

    // ---- export --------------------------------------------------------------------
    uint32_t n_rtr = 0, need_h = 0, n_routes = 0;
    for (uint32_t v : spt) { need_h += (uint32_t)vnh[v].size(); if (f.is_router[v]) { ++n_rtr; need_h += (uint32_t)vnh[v].size(); } }
    for (auto &kv : rib_idx) if (rib[kv.second].live) { ++n_routes; need_h += (uint32_t)rib[kv.second].nh.size(); }
    out->n_vertices = (uint32_t)spt.size(); out->n_routers = n_rtr; out->n_routes = n_routes; out->n_nexthops = need_h;
    bool tc = false;
    for (uint32_t v : spt) if (f.is_router[v] && (a->router_lsas[f.first_lsa[v]].flags & HL_RTR_FLAG_V)) tc = true;
    out->transit_capability = tc;
    if (out->n_vertices > out->vertices_cap || n_rtr > out->routers_cap || n_routes > out->routes_cap ||
        need_h > out->nexthops_cap)
        return HSPF_E_NOMEM;
    uint32_t h = 0;
    auto put = [&](const std::vector<Nh6> &s) {
        for (const Nh6 &x : s) {
            hl_nexthop6 o{};
            o.iface = x.iface; o.nbr_router_id = x.has_nbr ? x.nbr : 0;
            if (x.has_addr) o.addr = x.addr;
            o.has_addr = x.has_addr; o.has_nbr = x.has_nbr;
            out->nexthops[h++] = o;
        }
    };
    uint32_t i = 0;
    for (uint32_t v : spt) {
        hl_spt_vertex6 o{};
        o.router_id = f.rid[v]; o.iface_id = f.ifid[v]; o.distance = dist[v]; o.hops = hops[v]; o.is_router = f.is_router[v];
        o.nh_off = h; o.n_nh = (uint32_t)vnh[v].size();
        put(vnh[v]);
        out->vertices[i++] = o;
    }
    i = 0;
    for (uint32_t v : spt) {
        if (!f.is_router[v]) continue;
        const auto &r = a->router_lsas[f.first_lsa[v]];
        hl_route_rtr o{};
        o.router_id = r.adv_rtr; o.metric = dist[v]; o.flags = r.flags; o.options = r.options;
        o.nh_off = h; o.n_nh = (uint32_t)vnh[v].size();
        put(vnh[v]);
        out->routers[i++] = o;
    }
    i = 0;
    for (auto &kv : rib_idx) {
        const Route6 &r = rib[kv.second];
        if (!r.live) continue;
        hl_route_net6 o{};
        o.prefix = r.prefix; o.len = r.len; o.flags = r.flags; o.origin_type = r.otype; o.prefix_options = r.options;
        o.metric = r.metric; o.origin_adv_rtr = r.oadv; o.origin_lsa_id = r.oid; o.nh_off = h; o.n_nh = (uint32_t)r.nh.size();
        put(r.nh);
        out->routes[i++] = o;
    }
    return HSPF_OK;
}

}  // namespace

extern "C" {

int hspf_ospfv3_run_area(hspf_ctx *ctx, const hl_ospfv3_area *a, hl_ospfv3_result *out) {
    if (!ctx || !a || !out) return HSPF_E_INVAL;
    try {
        out->n_vertices = out->n_routers = out->n_routes = out->n_nexthops = 0;
        out->transit_capability = 0;
        out->root_found = 0;
        hspf_ospfv3_flat f;
        int rc = flatten(a, f);
        if (rc) return rc;
        auto rit = f.rtr_vertex.find(a->router_id);
        if (rit == f.rtr_vertex.end()) return HSPF_OK;
        out->root_found = 1;
        const uint32_t root = rit->second;
        hspf_csr csr;
        fill_csr(f, &csr);
        uint32_t n_atoms = 0;
        hspf_atom_count(&csr, root, &n_atoms);
        const uint32_t nhw = std::max(1u, (n_atoms + 63) / 64);
        if (nhw > 4) return HSPF_E_UNSUPPORTED;
        hspf::OneRootPlanes p;
        rc = hspf::run_one_root(ctx, csr, root, nhw, true, p);
        if (rc) return rc;
        return area_from_planes(f, a, root, p.dist.data(), p.hops.data(), p.nh.data(), nhw, out);
    } catch (const std::bad_alloc &) {
        return HSPF_E_NOMEM;
    } catch (...) {
        return HSPF_E_INVAL;
    }
}

/* The post-SPT half of hspf_ospfv3_run_area over planes the caller already has (vertex order of
 * hspf_ospfv3_flatten, area->router_id as root).  Host only. */
int hspf_ospfv3_area_from_planes(const hl_ospfv3_area *a, const uint32_t *dist, const uint16_t *hops,
                                 const uint64_t *nh_mask, uint32_t nh_words, hl_ospfv3_result *out) {
    if (!a || !out || !dist || !hops || !nh_mask || nh_words < 1 || nh_words > 4) return HSPF_E_INVAL;
    try {
        out->n_vertices = out->n_routers = out->n_routes = out->n_nexthops = 0;
        out->transit_capability = 0;
        out->root_found = 0;
        hspf_ospfv3_flat f;
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


/* ---- batched route stage: table and per-job decode for OSPFv3 areas (route_cells.h) ---------------------- */

int hspf_ospfv3_rtable_create(const hspf_ospfv3_flat *flat, hspf_ospfv2_rtable **out) {
    if (!flat || !flat->area || !out) return HSPF_E_INVAL;
    try {
        const hspf_ospfv3_flat &f = *flat;
        const hl_ospfv3_area *a = f.area;
        // update_rib_intra_area meets the advertisements LSA by LSA in LsaKey order (ospfv3/spf.rs:420-477)
        std::vector<uint32_t> iord(a->n_iap_lsas);
        for (uint32_t i = 0; i < a->n_iap_lsas; ++i) iord[i] = i;
        std::stable_sort(iord.begin(), iord.end(), [&](uint32_t x, uint32_t y) {
            const auto &p = a->iap_lsas[x], &q = a->iap_lsas[y];
            return p.adv_rtr != q.adv_rtr ? p.adv_rtr < q.adv_rtr : p.lsa_id < q.lsa_id;
        });
        struct Raw { PKey key; uint32_t seq; hspf::RouteContrib c; uint8_t otype, options; uint32_t oadv; };
        std::vector<Raw> raw;
        for (uint32_t i : iord) {
            const auto &l = a->iap_lsas[i];
            if (l.age == HL_LSA_MAX_AGE) continue;
            uint32_t v = kNone;
            if (l.ref_type == HL_V3_REF_ROUTER) {
                if (l.ref_lsa_id != 0) continue;
                auto it = f.rtr_vertex.find(l.ref_adv_rtr);
                if (it != f.rtr_vertex.end()) v = it->second;
            } else if (l.ref_type == HL_V3_REF_NETWORK) {
                auto it = f.net_vertex.find(((uint64_t)l.ref_adv_rtr << 32) | l.ref_lsa_id);
                if (it != f.net_vertex.end()) v = it->second;
            }
            if (v == kNone) continue;
            uint8_t otype; uint32_t oadv, oid;
            if (f.is_router[v]) { const auto &r = a->router_lsas[f.first_lsa[v]]; otype = 1; oadv = r.adv_rtr; oid = r.lsa_id; }
            else { const auto &n = a->network_lsas[f.first_lsa[v]]; otype = 2; oadv = n.adv_rtr; oid = n.lsa_id; }
            for (uint32_t k = 0; k < l.n_prefixes; ++k) {
                const auto &px = a->prefixes[l.prefix_off + k];
                if (px.options & HL_PFX_OPT_NU) continue;
                Raw r{};
                r.key = PKey{px.addr, px.len}; r.seq = (uint32_t)raw.size();
                r.c.vertex = v; r.c.origin_id = oid; r.c.metric = px.metric; r.c.sid_class = 0; r.c.is_network = otype == 2;
                r.otype = otype; r.options = px.options; r.oadv = oadv;
                raw.push_back(r);
            }
        }
        std::sort(raw.begin(), raw.end(), [](const Raw &x, const Raw &y) {
            if (x.key < y.key) return true;
            if (y.key < x.key) return false;
            return x.seq < y.seq;
        });
        auto rt = std::make_unique<hspf_ospfv2_rtable>();
        auto &t = rt->t;
        t.v3 = true;
        t.n_vertices = (uint32_t)f.rid.size();
        t.sids.push_back(hspf::SidDesc{0, 0, 0});
        for (size_t i = 0; i < raw.size(); ++i) {
            if (i == 0 || raw[i - 1].key < raw[i].key) {
                t.prefix6.push_back(raw[i].key.a); t.prefix.push_back(0); t.plen.push_back(raw[i].key.len); t.off.push_back((uint32_t)i);
            }
            t.contribs.push_back(raw[i].c);
            t.origin_type.push_back(raw[i].otype);
            t.origin_adv.push_back(raw[i].oadv);
            t.options6.push_back(raw[i].options);
            rt->ext_of.push_back(-1);
        }
        t.off.push_back((uint32_t)raw.size());
        *out = rt.release();
        return HSPF_OK;
    } catch (const std::bad_alloc &) { return HSPF_E_NOMEM; } catch (...) { return HSPF_E_INVAL; }
}

int hspf_ospfv3_rtable_prefixes6(const hspf_ospfv2_rtable *rt, const hl_ip_addr **prefixes, const uint32_t **lens) {
    if (!rt || !rt->t.v3) return HSPF_E_INVAL;
    if (prefixes) *prefixes = rt->t.prefix6.data();
    if (lens) *lens = rt->t.plen.data();
    return HSPF_OK;
}

int hspf_ospfv3_routes_from_cells(const hl_ospfv3_area *a, const hspf_ospfv2_rtable *rt, const hl_route_cell *cells,
                                  const uint32_t *gather_v, const uint64_t *gather_nh, uint32_t n_gather, hl_ospfv3_result *out) {
    if (!a || !rt || !rt->t.v3 || !cells || !out || (n_gather && (!gather_v || !gather_nh))) return HSPF_E_INVAL;
    try {
        out->n_vertices = out->n_routers = out->n_routes = out->n_nexthops = 0;
        out->transit_capability = 0;
        out->root_found = 0;
        hspf_ospfv3_flat f;
        int rc = flatten(a, f);
        if (rc) return rc;
        const uint32_t V = (uint32_t)f.rid.size();
        if (V != rt->t.n_vertices) return HSPF_E_INVAL;                   // not the LSDB the table was built from
        auto rit = f.rtr_vertex.find(a->router_id);
        if (rit == f.rtr_vertex.end()) return HSPF_OK;
        out->root_found = 1;
        std::vector<uint64_t> sparse_nh(V, 0);                             // only the transit networks next to the root are read
        for (uint32_t i = 0; i < n_gather; ++i) {
            if (gather_v[i] >= V) return HSPF_E_INVAL;
            sparse_nh[gather_v[i]] = gather_nh[i];
        }
        Resolver rs{f, a, rit->second, sparse_nh.data(), 1, {}, {}};
        rs.atom_nh.resize(64);
        rs.atom_done.assign(64, 0);
        const auto &t = rt->t;
        const uint32_t P = (uint32_t)t.prefix6.size();
        uint32_t n_routes = 0, n_nh = 0;
        std::vector<Nh6> set;
        for (uint32_t p = 0; p < P; ++p) {
            const hl_route_cell &c = cells[p];
            if (!(c.flags & HL_CELL_PRESENT)) continue;
            if (c.flags & HL_CELL_MIXED_SID) return HSPF_E_UNSUPPORTED;
            if (c.winner < t.off[p] || c.winner >= t.off[p + 1]) return HSPF_E_INVAL;
            hl_route_net6 o{};
            o.prefix = t.prefix6[p]; o.len = (uint8_t)t.plen[p];
            o.flags = (c.flags & HL_CELL_CONNECTED) ? HL_ROUTE_CONNECTED : 0;
            o.origin_type = t.origin_type[c.winner]; o.prefix_options = t.options6[c.winner]; o.metric = c.metric;
            o.origin_adv_rtr = t.origin_adv[c.winner]; o.origin_lsa_id = t.contribs[c.winner].origin_id;
            set.clear();
            uint64_t m = c.nh_mask;
            while (m) {
                const uint32_t atom = (uint32_t)__builtin_ctzll(m);
                m &= m - 1;
                for (const Nh6 &x : rs.resolve(atom)) {
                    auto it = std::lower_bound(set.begin(), set.end(), x, nh_less);
                    if (it != set.end() && nh_same(*it, x)) {
                        // same NexthopKey from another atom: the reference keeps the later advertiser's; both must agree
                        if (it->iface != x.iface || it->has_nbr != x.has_nbr || (x.has_nbr && it->nbr != x.nbr)) return HSPF_E_UNSUPPORTED;
                    } else {
                        set.insert(it, x);
                    }
                }
            }
            if (set.size() > a->max_paths) set.resize(a->max_paths);
            o.nh_off = n_nh; o.n_nh = (uint32_t)set.size();
            if (n_routes < out->routes_cap && n_nh + set.size() <= out->nexthops_cap) {
                out->routes[n_routes] = o;
                uint32_t h = n_nh;
                for (const Nh6 &x : set) {
                    hl_nexthop6 q{};
                    q.iface = x.iface; q.nbr_router_id = x.has_nbr ? x.nbr : 0;
                    if (x.has_addr) q.addr = x.addr;
                    q.has_addr = x.has_addr; q.has_nbr = x.has_nbr;
                    out->nexthops[h++] = q;
                }
            }
            ++n_routes; n_nh += (uint32_t)set.size();
        }
        out->n_routes = n_routes; out->n_nexthops = n_nh;
        if (n_routes > out->routes_cap || n_nh > out->nexthops_cap) return HSPF_E_NOMEM;
        return HSPF_OK;
    } catch (const std::bad_alloc &) { return HSPF_E_NOMEM; } catch (...) { return HSPF_E_INVAL; }
}

}  // extern "C"
