// Library tunables.  Every switch the planners consult lives in ONE table that is filled from the environment exactly
// once (first use) and can be changed programmatically with gd_set_option(); nothing on the launch path calls getenv().
#pragma once
#include <stdint.h>

namespace gd {

enum Opt {
    OPT_NO_CTAB,          // GD_NO_CTAB        decoder_v2_4 check-phase MLP evaluated directly
    OPT_NO_VTAB,          // GD_NO_VTAB        decoder_v2_4 variable-phase MLP evaluated directly
    OPT_FORCE_STREAMED,   // GD_FORCE_STREAMED take the streamed global-memory kernel even when the state fits on chip
    OPT_NO_VSKIP,         // GD_NO_VSKIP       re-evaluate degree-1 variables every iteration
    OPT_FORCE_LIGHT,      // GD_FORCE_LIGHT    node-owner kernel even where the planner declines
    OPT_NO_LEAN,          // GD_NO_LEAN        decoder_v2_4 on surface/toric codes: skip the table-only check-owner kernel
    OPT_LEAN_R,           // GD_LEAN_R         its owners (warps) per group of 32 syndromes
    OPT_LEAN_G,           // GD_LEAN_G         its groups per CTA
    OPT_LEAN_PARTS,       // GD_LEAN_PARTS     1: decode the graph's connected components in separate launches, 0: never (unset: when that seats more groups)
    OPT_COUNT
};

constexpr long long kOptUnset = INT64_MIN;

// value of an option, kOptUnset when neither the environment (at first use) nor gd_set_option() gave one
long long opt_get(Opt o);
// bumped by every gd_set_option(): planners cache their searches per epoch
long long opt_epoch();
inline bool opt_on(Opt o) { return opt_get(o) != kOptUnset; }                       // flag-style switches: set at all
inline long long opt_int(Opt o, long long dflt) { const long long v = opt_get(o); return v == kOptUnset ? dflt : v; }

}  // namespace gd
