// options.cc — storage and name table of the plan-time options (options.h).
#include "options.h"

#include <string.h>

namespace fd {

Options& options() {
    static Options o;
    return o;
}

int* option_slot(const char* name) {
    if (!name) return nullptr;
    Options& o = options();
    struct Entry { const char* name; int* slot; };
    const Entry table[] = {
        {"strip", &o.strip}, {"strip_min_w", &o.strip_min_w}, {"swap", &o.swap}, {"two_cta", &o.two_cta},
        {"split_k", &o.split_k}, {"split_k_min_kb", &o.split_k_min_kb}, {"split_k_max", &o.split_k_max},
        {"b_resident", &o.b_resident}, {"latency_bn", &o.latency_bn}, {"stem", &o.stem}, {"block", &o.block}, {"halo", &o.halo}, {"halo_skew", &o.halo_skew}, {"halo_slots", &o.halo_slots}, {"fuse_pool", &o.fuse_pool}, {"pdl", &o.pdl}, {"graph", &o.graph},
        {"exact_batch", &o.exact_batch}, {"nms_general", &o.nms_general}, {"jpeg_threads", &o.jpeg_threads},
        {"detect_overlap", &o.detect_overlap}, {"server_inflight", &o.server_inflight},
    };
    for (const Entry& e : table)
        if (!strcmp(e.name, name)) return e.slot;
    return nullptr;
}

}  // namespace fd
