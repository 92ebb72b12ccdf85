// Per-problem MPC ticks through hkd-mpc_b200/host/MultiPhaseDDP.hpp: robots of one batch tick at their own times
// (HKDMPCSolver::update of the robots whose mpc_data message arrived, HKDMPC/HKDMPC.cpp:169-200).
//   g++ -std=c++17 examples/subset_tick.cpp -Lhkd-mpc_b200 -lhsddp_b200 -Wl,-rpath,hkd-mpc_b200 -o subset_tick
//   ./subset_tick <input.bin> <commands.bin>
// input.bin: one gait table and the initial states of 6 problems -- int32 rows, float dt, then body_state, qJ, foot placements,
// grf ([rows][12] doubles each), contact ([rows][4] int32), x0 ([6][24] doubles).  Problems 0, 1, 4 use window 0 of the gait,
// problems 2, 3, 5 window 20.  After a cold solve, tick t = 1 .. 4 ticks problems {0, 2, 5} every tick and {1, 3} on even
// ticks (update, initial states, 2 x 1 solve, commands), once on MultiPhaseDDP and once on MultiGpuDDP with one part; the
// command records of every tick of the first are written to commands.bin, and the second must give the same bytes.
#include <cstdio>
#include <cstring>
#include <vector>
#include "../hkd-mpc_b200/host/MultiPhaseDDP.hpp"

namespace {
template <class T>
bool read(std::FILE* f, std::vector<T>& v, size_t n) { v.resize(n); return std::fread(v.data(), sizeof(T), n, f) == n; }

// the states a tick sets: x0 with the body x position moved by 0.5 mm per tick
std::vector<double> tick_states(const std::vector<double>& x0, const std::vector<int32_t>& problem, int tick) {
    std::vector<double> x;
    for (int32_t p : problem) {
        x.insert(x.end(), x0.begin() + 24 * p, x0.begin() + 24 * (p + 1));
        x[x.size() - 24 + 3] += 0.0005 * tick;
    }
    return x;
}

template <class Solver>
std::vector<hsddp_mpc_command> run(Solver& s, const std::vector<double>& x0) {
    hsddp_b200::HSDDP_OPTION cold, tick;
    tick.max_AL_iter = 2; tick.max_DDP_iter = 1;
    s.set_initial_condition(x0);
    s.solve(cold);
    std::vector<hsddp_mpc_command> all;
    for (int t = 1; t <= 4; ++t) {
        const std::vector<int32_t> list = (t % 2 == 0) ? std::vector<int32_t>{0, 2, 5, 1, 3} : std::vector<int32_t>{0, 2, 5};
        s.update_problems(list);
        s.set_initial_condition_problems(list, tick_states(x0, list, t));
        s.solve_problems(list, tick);
        const std::vector<hsddp_mpc_command> c = s.get_mpc_command_problems(list, 8);
        all.insert(all.end(), c.begin(), c.end());
    }
    return all;
}
}  // namespace

int main(int argc, char** argv) {
    if (argc < 3) { std::fprintf(stderr, "usage: %s input.bin commands.bin\n", argv[0]); return 2; }
    try {
        std::FILE* f = std::fopen(argv[1], "rb");
        if (!f) { std::fprintf(stderr, "error: cannot open %s\n", argv[1]); return 2; }
        int32_t rows = 0;
        float dt = 0.f;
        std::vector<double> body, qJ, foot, grf, x0;
        std::vector<int32_t> contact;
        const bool ok = std::fread(&rows, 4, 1, f) == 1 && std::fread(&dt, 4, 1, f) == 1 && read(f, body, 12 * (size_t)rows) && read(f, qJ, 12 * (size_t)rows) &&
                        read(f, foot, 12 * (size_t)rows) && read(f, grf, 12 * (size_t)rows) && read(f, contact, 4 * (size_t)rows) && read(f, x0, 6 * 24);
        std::fclose(f);
        if (!ok) { std::fprintf(stderr, "error: %s is truncated\n", argv[1]); return 2; }
        const std::vector<int32_t> sched_gait{0, 0}, sched_window{0, 20}, schedule_id{0, 0, 1, 1, 0, 1};
        hsddp_b200::MultiPhaseDDP<double> solver(0);
        solver.set_multiPhaseProblem_from_gaits({rows}, {dt}, body, qJ, foot, grf, contact, sched_gait, sched_window, 0.6f, schedule_id);
        const std::vector<hsddp_mpc_command> a = run(solver, x0);
        hsddp_b200::MultiGpuDDP multi({0});
        multi.set_multiPhaseProblem_from_gaits({rows}, {dt}, body, qJ, foot, grf, contact, sched_gait, sched_window, 0.6f, schedule_id);
        const std::vector<hsddp_mpc_command> b = run(multi, x0);
        if (a.size() != b.size() || std::memcmp(a.data(), b.data(), a.size() * sizeof(hsddp_mpc_command)) != 0) {
            std::fprintf(stderr, "error: MultiGpuDDP commands differ from MultiPhaseDDP's\n");
            return 4;
        }
        std::FILE* o = std::fopen(argv[2], "wb");
        if (!o || std::fwrite(a.data(), sizeof(hsddp_mpc_command), a.size(), o) != a.size()) { std::fprintf(stderr, "error: cannot write %s\n", argv[2]); return 2; }
        std::fclose(o);
        std::printf("%zu command records, first GRF z of leg 0 = %.4f N\n", a.size(), a[0].hkd_controls[0][2]);
    } catch (const std::exception& e) {
        std::fprintf(stderr, "error: %s\n", e.what());
        return 1;
    }
    return 0;
}
