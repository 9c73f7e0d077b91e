// Drives include/pqp_base_solver.hpp exactly the way PathOptimizer::optimizePath drives the
// reference's BaseSolver (path_optimizer.cpp:128-157): construct on the stack, solve(), then
// updateProblemFormulationAndSolve(*final_path, final_path) with input and output aliased.
// Input: a text file written by tests/test_dropin.py; output: one line per knot.
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <fstream>
#include <iostream>

// Two builds of this file (tests/test_dropin.py):
//   dropin_test       against tests/cpp/ref_stub.hpp (stand-ins; builds anywhere);
//   dropin_test_real  with -DPQP_TEST_REAL_TYPES -I oracle/_ref/include, i.e. against the reference's
//                     OWN State / SlState / VehicleStateBound (include/data_struct/data_struct.hpp) and
//                     VehicleState (vehicle_state_frenet.hpp and an object of its .cpp), as staged from
//                     a checkout of the original project by `make -C oracle ref`. Only
//                     the reference's ReferencePath cannot be compiled standalone (it needs grid_map / glog), so
//                     a holder with the three accessors the solver reads carries the real element types.
#include "../../include/pqp_base_solver.hpp"
#ifdef PQP_TEST_REAL_TYPES
#include "data_struct/data_struct.hpp"
#include "data_struct/vehicle_state_frenet.hpp"
namespace stub {
using State = PathOptimizationNS::State;
using SlState = PathOptimizationNS::SlState;
using VehicleStateBound = PathOptimizationNS::VehicleStateBound;
using VehicleState = PathOptimizationNS::VehicleState;
class ReferencePath {  // accessors of reference_path.hpp:21-46 that base_solver.cpp reads
 public:
    const std::vector<State> &getReferenceStates() const { return states_; }
    const std::vector<VehicleStateBound> &getBounds() const { return bounds_; }
    std::shared_ptr<VehicleStateBound> isBlocked() const { return blocked_; }
    double getLength() const { return states_.empty() ? 0.0 : states_.back().s; }
    std::vector<State> states_;
    std::vector<VehicleStateBound> bounds_;
    std::shared_ptr<VehicleStateBound> blocked_;
};
}  // namespace stub
#else
#include "ref_stub.hpp"
#endif

using Solver = pqp::dropin::BaseSolverT<stub::ReferencePath, stub::VehicleState, stub::SlState>;

int main(int argc, char **argv) {
    if (argc < 2) return 2;
    std::ifstream f(argv[1]);
    size_t n;
    f >> n;
    stub::ReferencePath ref;
    ref.states_.resize(n);
    ref.bounds_.resize(n);
    for (size_t i = 0; i < n; ++i) {
        auto &s = ref.states_[i];
        auto &b = ref.bounds_[i];
        f >> s.s >> s.k >> s.x >> s.y >> s.heading >> b.front.lb >> b.front.ub >> b.rear.lb >> b.rear.ub;
        b.center.lb = b.front.lb;
        b.center.ub = b.front.ub;
    }
    double offset, heading_error;
    stub::State start, target;
    f >> offset >> heading_error >> start.k >> target.heading;
    stub::VehicleState veh(start, target, offset, heading_error);
    int constraint_end_heading;
    f >> constraint_end_heading;
    std::vector<stub::SlState> input_path;
    for (const auto &rs : ref.states_) {  // path_optimizer.cpp:128-137
        stub::SlState st;
        st.x = rs.x; st.y = rs.y; st.heading = rs.heading; st.s = rs.s; st.k = rs.k;
        input_path.push_back(st);
    }
    pqp::dropin::SolverFlags flags;
    flags.constraint_end_heading = constraint_end_heading != 0;
    // argv[2] = number of extra plans: the reference constructs a BaseSolver per plan at 30 Hz
    // (path_optimizer.cpp:138); report wall time per plan (construct + solve + re-solve + destruct) and
    // what the handle pool did
    const int extra = argc > 2 ? std::atoi(argv[2]) : 0;
    if (extra > 0) {
        double first_ms = 0.0, rest_ms = 0.0;
        float stage_last[PQP_NSTAGES] = {0, 0, 0, 0, 0};
        for (int rep = 0; rep <= extra; ++rep) {
            const auto t0 = std::chrono::steady_clock::now();
            {
                Solver sv(ref, veh, input_path, flags);
                std::vector<stub::SlState> out;
                if (!sv.solve(&out) || !sv.updateProblemFormulationAndSolve(out, &out)) {
                    std::printf("plan %d failed: status %d err '%s'\n", rep, sv.lastStatus(), sv.lastError().c_str());
                    return 0;
                }
                for (int k = 0; k < PQP_NSTAGES; ++k) stage_last[k] = sv.lastStageMs()[k];
            }
            const double ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
            if (rep == 0) first_ms = ms;
            else rest_ms += ms;
        }
        auto &pool = pqp::dropin::HandlePool::instance();
        std::printf("plans %d first_ms %.4f later_ms %.4f creates %zu hits %zu stage_ms h2d %.4f kernel %.4f d2h %.4f total %.4f\n",
                    extra + 1, first_ms, rest_ms / extra, pool.creates(), pool.hits(), stage_last[PQP_STAGE_H2D],
                    stage_last[PQP_STAGE_KERNEL], stage_last[PQP_STAGE_D2H], stage_last[PQP_STAGE_TOTAL]);
    }
    Solver solver(ref, veh, input_path, flags);
    std::vector<stub::SlState> final_path;
    const bool ok1 = solver.solve(&final_path);
    std::printf("solve %d status %d iters %d cost %.17g err '%s'\n", ok1 ? 1 : 0, solver.lastStatus(),
                solver.lastIterations(), solver.lastCost(), solver.lastError().c_str());
    if (!ok1) return 0;
    const bool ok2 = solver.updateProblemFormulationAndSolve(final_path, &final_path);
    std::printf("resolve %d status %d iters %d cost %.17g\n", ok2 ? 1 : 0, solver.lastStatus(),
                solver.lastIterations(), solver.lastCost());
    if (!ok2) return 0;
    for (const auto &p : final_path)
        std::printf("%.17g %.17g %.17g %.17g %.17g %.17g %.17g\n", p.x, p.y, p.heading, p.k, p.d_k, p.l, p.d_heading);
    return 0;
}
