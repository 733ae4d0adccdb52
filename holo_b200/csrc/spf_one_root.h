// spf_one_root.h — one SPF job on a graph uploaded for it alone: the device half of the
// single-root calls (hspf_ospfv2_run_area, hspf_ospfv3_run_area, hspf_isis_compute_spt,
// hspf_isis_compute_routes).
#pragma once
#include <cstdint>
#include <vector>

#include "holo_spf.h"

namespace hspf {

struct OneRootPlanes {
    std::vector<uint32_t> dist;
    std::vector<uint16_t> hops;
    std::vector<uint64_t> nh;    // [V][nh_words]; empty unless asked for
    uint32_t status = 0;         // job_status of the job
};

// Upload `csr`, run the job rooted at `root` and free the graph.  Returns the error of the upload or
// what hspf_run_batch returned (HSPF_E_JOB_STATUS included: `out.status` says why).
inline int run_one_root(hspf_ctx *ctx, const hspf_csr &csr, uint32_t root, uint32_t nh_words, bool want_nh,
                        OneRootPlanes &out) {
    hspf_graph *g = nullptr;
    int rc = hspf_graph_upload(ctx, &csr, &g);
    if (rc) return rc;
    const uint32_t V = csr.n_vertices;
    out.dist.resize(V);
    out.hops.resize(V);
    out.nh.resize(want_nh ? (size_t)V * nh_words : 0);
    hspf_jobs jobs{};
    jobs.n_jobs = 1;
    jobs.roots = &root;
    hspf_result res{};
    res.dist = out.dist.data();
    res.hops = out.hops.data();
    res.nh_mask = want_nh ? out.nh.data() : nullptr;
    res.nh_words = nh_words;
    res.job_status = &out.status;
    rc = hspf_run_batch(ctx, g, &jobs, &res, 0);
    hspf_graph_free(ctx, g);
    return rc;
}

}  // namespace hspf
