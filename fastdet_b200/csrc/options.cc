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
        {"strip", &o.strip}, {"stem", &o.stem}, {"block", &o.block}, {"fuse_pool", &o.fuse_pool},
        {"nms_general", &o.nms_general}, {"jpeg_threads", &o.jpeg_threads}, {"server_inflight", &o.server_inflight},
    };
    for (const Entry& e : table)
        if (!strcmp(e.name, name)) return e.slot;
    return nullptr;
}

}  // namespace fd
