// b200dp_cli.cpp -- a compiled-language host over the C ABI (include/b200dp.h), the way the
// reference's Go binaries sit over internal/pkg/*: no Python, no ctypes.  Used for
// measurements without interpreter overhead and as a worked example of the ABI contracts
// (caller-owned arrays, E_NOSPC growth, error strings).
//
//   g++ -O2 -std=c++17 -I include tools/b200dp_cli.cpp -L k8s-device-plugin_b200 -lb200dp \
//       -Wl,-rpath,'$ORIGIN/../k8s-device-plugin_b200' -o tools/b200dp_cli
//
//   b200dp_cli <backend-uri> enumerate | health | cycle [steps [idle_ms]] | probe [steps] | resources <single|mixed>
//                            | labels <csv> | alloc <size> | p2p | compute [tiles [n]]
#include <algorithm>
#include <chrono>
#include <ctime>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "b200dp.h"

static double now_ms() {
    using namespace std::chrono;
    return duration<double, std::milli>(steady_clock::now().time_since_epoch()).count();
}
static int die(b2dp_ctx* c, const char* what, int rc) {
    fprintf(stderr, "%s: %s [%d] %s\n", what, b2dp_strerror(rc), rc, c ? b2dp_last_error(c) : "");
    return 1;
}
static double median(std::vector<double> v) { std::sort(v.begin(), v.end()); return v.empty() ? 0 : v[v.size() / 2]; }
static double pct(std::vector<double> v, double q) {
    std::sort(v.begin(), v.end());
    return v.empty() ? 0 : v[(size_t)(q * (double)(v.size() - 1) + 0.5)];
}

int main(int argc, char** argv) {
    if (argc < 3) { fprintf(stderr, "usage: %s <backend-uri> <command> [args]\n", argv[0]); return 2; }
    if (b2dp_abi_version() != B2DP_ABI_VERSION) {
        fprintf(stderr, "libb200dp.so has ABI %d, this host was built against %d\n", b2dp_abi_version(), B2DP_ABI_VERSION);
        return 3;
    }
    b2dp_ctx* ctx = nullptr;
    int rc = b2dp_open(argv[1], &ctx);
    if (rc != B2DP_OK) return die(nullptr, "b2dp_open", rc);
    const std::string cmd = argv[2];

    std::vector<b2dp_device> devs(64);
    int n = 0;
    while ((rc = b2dp_enumerate(ctx, devs.data(), (int)devs.size(), &n)) == B2DP_E_NOSPC) devs.resize(n);
    if (rc != B2DP_OK) return die(ctx, "b2dp_enumerate", rc);
    devs.resize(n);

    if (cmd == "enumerate") {
        for (auto& d : devs)
            printf("%s devID=%s card=%d renderD=%d node=%d numa=%d partition=%s_%s\n", d.id, d.dev_id, d.card, d.render_d,
                   d.node_id, d.numa_node, d.compute_partition, d.memory_partition);
    } else if (cmd == "health") {
        int32_t h = 0;
        b2dp_node_health(ctx, &h);
        printf("node %s\n", h ? "Healthy" : "Unhealthy");
    } else if (cmd == "compute") {  // tensor-core check: n event-timed checks, per GPU the median ms, TFLOP/s and SMs
        b2dp_compute_opts o{};
        o.tiles = argc > 3 ? (uint32_t)atoi(argv[3]) : 0;
        o.flags = B2DP_COMPUTE_EVENT_TIMING;
        const int steps = argc > 4 ? atoi(argv[4]) : 1;
        std::vector<b2dp_compute_result> res(devs.size());
        std::vector<std::vector<double>> ms(devs.size());
        bool all_ok = true;
        for (int s = 0; s < steps; ++s) {
            int m = 0;
            if ((rc = b2dp_compute_check(ctx, &o, res.data(), (int)res.size(), &m)) != B2DP_OK) return die(ctx, "b2dp_compute_check", rc);
            for (int i = 0; i < m; ++i) { ms[i].push_back(res[i].ms_event); all_ok = all_ok && res[i].healthy; }
        }
        for (size_t i = 0; i < res.size(); ++i) {
            const b2dp_compute_result& r = res[i];
            const double t = median(ms[i]);
            printf("%s %s ms=%.4f tflops=%.1f tiles=%llu sms=%d covered=%d failed=%d bad_rows=%llu first_bad_sm=%d\n", devs[i].id,
                   r.healthy ? "Healthy" : "Unhealthy", t, t > 0 ? 2.0 * 128 * 128 * 128 * (double)r.tiles / (t * 1e-3) * 1e-12 : 0.0,
                   (unsigned long long)r.tiles, r.sms, r.sms_covered, r.sms_failed, (unsigned long long)r.bad_rows, r.first_bad_sm);
        }
        if (!all_ok) { b2dp_close(ctx); return 1; }  // a failed check is a failing exit status
    } else if (cmd == "probe" || cmd == "cycle") {
        const int steps = argc > 3 ? atoi(argv[3]) : 200;
        const int idle_ms = argc > 4 ? atoi(argv[4]) : 0;  // sleep between cycles: the production shape is a heartbeat every few seconds
        std::vector<b2dp_probe_result> res(n ? n : 1);
        std::vector<uint8_t> buf(1 << 16);
        b2dp_cycle_opts co{};
        co.flags = B2DP_LW_HEARTBEAT;
        size_t len = 0;
        b2dp_cycle_stats st{};
        if ((rc = b2dp_list_and_watch(ctx, "gpu", nullptr, buf.data(), buf.size(), &len, &st)) != B2DP_OK)
            return die(ctx, "b2dp_list_and_watch(initial)", rc);
        std::vector<double> wall, kern, kmax, host;
        double bytes = 0, frac_min = 1e30;
        for (int i = -5; i < steps; ++i) {
            if (idle_ms > 0) { struct timespec ts{idle_ms / 1000, (long)(idle_ms % 1000) * 1000000L}; nanosleep(&ts, nullptr); }
            const double t0 = now_ms();
            if (cmd == "probe") {
                int m = 0;
                b2dp_probe_opts po{};
                po.flags = B2DP_PROBE_EVENT_TIMING;   // kernel_ms_median below is the CUDA-event time
                if ((rc = b2dp_probe_health(ctx, &po, res.data(), (int)res.size(), &m)) != B2DP_OK) return die(ctx, "b2dp_probe_health", rc);
                if (i >= 0) { bytes = 0; for (int k = 0; k < m; ++k) { bytes += (double)res[k].bytes; kern.push_back(res[k].ms_event); if (!res[k].healthy) return die(ctx, "unhealthy device", res[k].err); } }
            } else {
                if ((rc = b2dp_list_and_watch(ctx, "gpu", &co, buf.data(), buf.size(), &len, &st)) != B2DP_OK) return die(ctx, "b2dp_list_and_watch", rc);
                if (i >= 0) { bytes = (double)st.probe_bytes; if (st.n_unhealthy) return die(ctx, "unhealthy device", 0); }
            }
            if (i >= 0) {
                wall.push_back(now_ms() - t0);
                if (cmd == "cycle") {  // tail attribution: the slowest GPU's in-kernel span vs everything the host adds
                    kmax.push_back(st.probe_ms_device_max);
                    host.push_back(wall.back() - st.probe_ms_device_max);
                    if (st.probe_frac_min > 0 && st.probe_frac_min < frac_min) frac_min = st.probe_frac_min;
                }
            }
        }
        const double w = median(wall);
        printf("{\"command\": \"%s\", \"idle_ms_between_cycles\": %d, \"n_devices\": %d, \"steps\": %d, \"wall_ms_median\": %.4f, \"wall_ms_p99\": %.4f, "
               "\"wall_ms_max\": %.4f, \"aggregate_gbs\": %.1f, \"kernel_ms_median\": %.4f, \"response_bytes\": %zu, "
               "\"slowest_kernel_ms_p50\": %.4f, \"slowest_kernel_ms_p99\": %.4f, \"host_overhead_ms_p50\": %.4f, "
               "\"host_overhead_ms_p99\": %.4f, \"probe_frac_min\": %.4f}\n",
               cmd.c_str(), idle_ms, n, steps, w, pct(wall, 0.99), *std::max_element(wall.begin(), wall.end()), bytes / w / 1e6,
               median(kern), len, pct(kmax, 0.5), pct(kmax, 0.99), pct(host, 0.5), pct(host, 0.99), frac_min > 1e29 ? 0.0 : frac_min);
    } else if (cmd == "resources") {
        char names[16][64];
        int m = 0;
        if ((rc = b2dp_resource_list(ctx, argc > 3 ? argv[3] : "single", names, 16, &m)) != B2DP_OK) return die(ctx, "b2dp_resource_list", rc);
        for (int i = 0; i < m; ++i) printf("amd.com/%s\n", names[i]);
    } else if (cmd == "labels") {
        std::vector<b2dp_label> labels(256);
        int m = 0;
        if ((rc = b2dp_generate_labels(ctx, argc > 3 ? argv[3] : "vram,cu-count,product-name", labels.data(), 256, &m)) != B2DP_OK)
            return die(ctx, "b2dp_generate_labels", rc);
        for (int i = 0; i < m; ++i) printf("%s=%s\n", labels[i].key, labels[i].value);
    } else if (cmd == "alloc") {
        const int size = argc > 3 ? atoi(argv[3]) : 1;
        if ((rc = b2dp_start(ctx)) != B2DP_OK) return die(ctx, "b2dp_start", rc);
        std::vector<const char*> ids;
        for (auto& d : devs) ids.push_back(d.id);
        std::vector<char[64]> out(devs.size() + 1);
        int m = 0;
        const double t0 = now_ms();
        rc = b2dp_preferred_allocation(ctx, ids.data(), (int)ids.size(), nullptr, 0, size, out.data(), (int)out.size(), &m);
        const double dt = now_ms() - t0;
        if (rc != B2DP_OK) return die(ctx, "b2dp_preferred_allocation", rc);
        for (int i = 0; i < m; ++i) printf("%s\n", out[i]);
        fprintf(stderr, "allocated %d of %zu in %.4f ms\n", m, ids.size(), dt);
    } else if (cmd == "p2p") {
        std::vector<float> gbs((size_t)n * n);
        std::vector<int32_t> lt((size_t)n * n);
        std::vector<uint64_t> mm((size_t)n * n);
        if ((rc = b2dp_p2p_matrix(ctx, nullptr, gbs.data(), lt.data(), mm.data(), n)) != B2DP_OK) return die(ctx, "b2dp_p2p_matrix", rc);
        for (int i = 0; i < n; ++i) {
            for (int j = 0; j < n; ++j) printf("%7.1f/%-2d ", gbs[(size_t)i * n + j], lt[(size_t)i * n + j]);
            printf("\n");
        }
    } else {
        fprintf(stderr, "unknown command %s\n", cmd.c_str());
        b2dp_close(ctx);
        return 2;
    }
    b2dp_close(ctx);
    return 0;
}
