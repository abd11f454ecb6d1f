// tunables.cu -- run-time knobs of the library (GENPC_*), read from the environment ONCE when the library is loaded.
//
// r01 called getenv() on every forward (five times in the Chamfer host path alone).  The knobs now live in a small table
// that a static initialiser fills from the environment at load time; the hot host paths only do a handful of short
// strcmp()s against it.  Tests and the tools/ experiments flip a knob at run time through genpc_set_tunable() (the
// environment is NOT re-read).  Not meant to be changed while launches are being issued from other threads.
#include <cstdlib>
#include <cstring>

#include "common.cuh"

namespace genpc {

struct Knob {
    const char *name;
    char value[32];
    bool set;
};

static Knob g_knobs[] = {
    {"GENPC_CHAMFER_MODE", "", false},   // "sym" | "scan"
    {"GENPC_SYM_BALANCED", "", false},   {"GENPC_CHAMFER_PRUNE", "", false}, {"GENPC_HOST_PRUNE", "", false},
    {"GENPC_PRUNE_COOP", "", false},     {"GENPC_SORT_CLUSTER", "", false},  {"GENPC_EMD_GETMAX", "", false},
    {"GENPC_EMD_PRUNE", "", false},      {"GENPC_EMD_SORT", "", false},      {"GENPC_FPS_MODE", "", false},
    {"GENPC_FPS_CLUSTER16", "", false},  {"GENPC_FPS_SMEM", "", false},      {"GENPC_REGISTER_MODE", "", false},
    {"GENPC_REGISTER_PERSIST", "", false}, {"GENPC_REGISTER_PRUNE", "", false},
};
constexpr int N_KNOBS = sizeof(g_knobs) / sizeof(g_knobs[0]);

static void knob_assign(Knob &k, const char *v) {
    k.set = (v != nullptr);
    k.value[0] = 0;
    if (v != nullptr) {
        strncpy(k.value, v, sizeof(k.value) - 1);
        k.value[sizeof(k.value) - 1] = 0;
    }
}

static struct KnobInit {
    KnobInit() {
        for (int i = 0; i < N_KNOBS; ++i) knob_assign(g_knobs[i], getenv(g_knobs[i].name));
    }
} g_knob_init;

const char *tunable(const char *name) {
    for (int i = 0; i < N_KNOBS; ++i)
        if (strcmp(g_knobs[i].name, name) == 0) return g_knobs[i].set ? g_knobs[i].value : nullptr;
    return nullptr;
}

int num_sms() {
    static int cache[64] = {0};   // 0 = not asked yet; racing first calls write the same value
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return GENPC_NUM_SMS_B200;
    int n = cache[dev];
    if (n <= 0) {
        if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = GENPC_NUM_SMS_B200;
        cache[dev] = n;
    }
    return n;
}

}  // namespace genpc

extern "C" int genpc_set_tunable(const char *name, const char *value) {
    if (name == nullptr) return GENPC_ERR_SHAPE;
    for (int i = 0; i < genpc::N_KNOBS; ++i)
        if (strcmp(genpc::g_knobs[i].name, name) == 0) {
            genpc::knob_assign(genpc::g_knobs[i], value);
            return GENPC_OK;
        }
    return GENPC_ERR_SHAPE;  // unknown knob
}

extern "C" const char *genpc_get_tunable(const char *name) { return name ? genpc::tunable(name) : nullptr; }
