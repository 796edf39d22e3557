// Prints what hmc.jl_b200/csrc/plan_policy.cuh decides, for tests/test_plan_policy.py (compiled there with g++; no GPU).
//
//   plan_policy_driver plan key=value ...   one problem (keys below); the HMCGPU_* tuning variables are read from the
//                                           environment.  Prints the sweep choice, the layout counts, the draw chunks and
//                                           the launch schedule, or "error <code> <message>".
//   plan_policy_driver schedule             reads lines "burnin nrun chunk n_bufs n_groups sweeps_per_launch" from stdin and
//                                           prints each one's launch schedule, followed by "end"
//   plan_policy_driver limits precision K lanes   prints scan_max_T and seg_max_T
//
// Schedule lines: "L group sweep0 n_sweeps chunk wait closes_chunk last" for a launch, "P chunk" for a post.
#include "plan_policy.cuh"

#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

using namespace hmc;

static void print_schedule(const std::vector<RunOp>& ops) {
    for (const RunOp& op : ops) {
        if (op.post) printf("P %lld\n", op.chunk);
        else printf("L %d %lld %lld %lld %lld %d %d\n", op.group, op.sweep0, op.n_sweeps, op.chunk, op.wait, (int)op.closes_chunk, (int)op.last);
    }
}

static int plan(int argc, char** argv) {
    int sm = 148, K = 3, precision = 32, nc = 1, nser = 1, sig = 0, n_h = 1;
    unsigned flags = HMCGPU_FLAG_REF_Q1;
    long long burnin = 0, nrun = 1;
    std::vector<int> T;
    for (int i = 2; i < argc; ++i) {
        const char* eq = strchr(argv[i], '=');
        if (!eq) { fprintf(stderr, "bad argument %s\n", argv[i]); return 2; }
        const std::string k(argv[i], eq - argv[i]);
        const char* v = eq + 1;
        if (k == "sm") sm = atoi(v);
        else if (k == "K") K = atoi(v);
        else if (k == "precision") precision = atoi(v);
        else if (k == "nc") nc = atoi(v);
        else if (k == "nser") nser = atoi(v);
        else if (k == "sig") sig = atoi(v);
        else if (k == "n_h") n_h = atoi(v);
        else if (k == "flags") flags = (unsigned)atol(v);
        else if (k == "burnin") burnin = atoll(v);
        else if (k == "nrun") nrun = atoll(v);
        else if (k == "T") {                                  // the window lengths, comma-separated
            char* s = const_cast<char*>(v);
            do T.push_back((int)strtol(s, &s, 10)); while (*s++ == ',');
        }
        else { fprintf(stderr, "unknown key %s\n", k.c_str()); return 2; }
    }
    // windows [1, T_w] of series w % nser; sig: every observation a signal
    const int nw = (int)T.size();
    std::vector<int32_t> start(nw, 1), end(T.begin(), T.end()), series(nw);
    for (int w = 0; w < nw; ++w) series[w] = w % nser;
    const uint8_t mask = 1;
    hmcgpu_problem p{};
    p.n_series = nser; p.n_windows = nw; p.win_series = nser > 1 ? series.data() : nullptr;
    p.win_start = start.data(); p.win_end = end.data(); p.K = K; p.n_chains = nc; p.burnin = burnin; p.nrun = nrun;
    p.is_signal = sig ? &mask : nullptr; p.n_h = n_h; p.precision = precision; p.flags = flags;

    // as plan_build: the windows by decreasing length
    std::vector<int> order(nw);
    std::iota(order.begin(), order.end(), 0);
    std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return T[a] > T[b]; });
    const Tuning t = read_tuning();
    SweepChoice c;
    const char* err = nullptr;
    if (const int rc = choose_sweep(sm, &p, T, order, t, c, &err)) { printf("error %d %s\n", rc, err); return 0; }
    const SlotLayout lay = layout_slots(&p, T, order, c, t);
    const int F = 3 * K + K * K + 2 * n_h + 1;              // summary_fields (hmcgpu.cu)
    const DrawChunks dc = draw_chunks((int)lay.groups.size(), flags, F, lay.n_slots, precision / 8, nrun);
    printf("kernel %d\nseg_lanes %d\nn_long %d\nseg_threads %d\nsweeps_per_launch %d\n", (int)c.kernel, c.seg_lanes, c.n_long,
           c.seg_threads, c.sweeps_per_launch);
    printf("n_slots %d\nn_warps %d\nn_tasks %d\nn_groups %d\nchunk %d\nn_bufs %d\n", lay.n_slots, lay.n_warps, lay.n_tasks,
           (int)lay.groups.size(), dc.chunk, dc.n_bufs);
    print_schedule(launch_schedule(burnin, nrun, dc.chunk, dc.n_bufs, (int)lay.groups.size(), c.sweeps_per_launch));
    return 0;
}

int main(int argc, char** argv) {
    const std::string mode = argc > 1 ? argv[1] : "";
    if (mode == "plan") return plan(argc, argv);
    if (mode == "schedule") {
        long long burnin, nrun, chunk;
        int n_bufs, G, L;
        while (scanf("%lld %lld %lld %d %d %d", &burnin, &nrun, &chunk, &n_bufs, &G, &L) == 6) {
            print_schedule(launch_schedule(burnin, nrun, chunk, n_bufs, G, L));
            printf("end\n");
        }
        return 0;
    }
    if (mode == "limits" && argc == 5) {
        printf("scan_max_T %d\nseg_max_T %lld\n", scan_max_T(atoi(argv[2]), atoi(argv[3])), seg_max_T(atoi(argv[3]), atoi(argv[4])));
        return 0;
    }
    fprintf(stderr, "usage: %s plan key=value ... | schedule | limits precision K lanes\n", argv[0]);
    return 2;
}
