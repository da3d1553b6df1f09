// Option table of the library (gd_options.cuh): environment read ONCE, then plain loads on the launch path.
#include "gd_common.cuh"
#include "gd_options.cuh"
#include <stdlib.h>
#include <string.h>
#include <atomic>
#include <mutex>

namespace gd {

static const char* const kOptNames[OPT_COUNT] = {
    "GD_NO_CTAB", "GD_NO_VTAB", "GD_FORCE_STREAMED", "GD_NO_VSKIP", "GD_FORCE_LIGHT", "GD_NO_LEAN", "GD_LEAN_R", "GD_LEAN_G",
    "GD_LEAN_PARTS"};

static std::atomic<long long> g_opt[OPT_COUNT];
static std::once_flag g_opt_once;
static std::atomic<long long> g_opt_epoch{0};

long long opt_epoch() { return g_opt_epoch.load(std::memory_order_relaxed); }

static void load_env() {
    for (int i = 0; i < OPT_COUNT; ++i) {
        const char* e = getenv(kOptNames[i]);
        g_opt[i].store(e ? atoll(e) : kOptUnset, std::memory_order_relaxed);
    }
}

long long opt_get(Opt o) {
    std::call_once(g_opt_once, load_env);
    return g_opt[o].load(std::memory_order_relaxed);
}

}  // namespace gd

extern "C" int gd_set_option(const char* name, int64_t value, int32_t unset) {
    GD_CHECK_ARG(name != nullptr, "gd_set_option: name is NULL");
    std::call_once(gd::g_opt_once, gd::load_env);
    for (int i = 0; i < gd::OPT_COUNT; ++i)
        if (strcmp(name, gd::kOptNames[i]) == 0) {
            gd::g_opt[i].store(unset ? gd::kOptUnset : (long long)value, std::memory_order_relaxed);
            gd::g_opt_epoch.fetch_add(1, std::memory_order_relaxed);
            return GD_OK;
        }
    gd::set_error("gd_set_option: unknown option '%s'", name);
    return GD_ERR_INVALID;
}
