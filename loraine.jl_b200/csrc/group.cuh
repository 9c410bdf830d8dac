// In-process multi-GPU: ONE host thread (the Julia task) drives N devices through a single handle.
// lrn_create_multi builds one ordinary single-device solver per GPU ("members", rank r on device r) that share an NCCL
// communicator made with ncclCommInitAll, and returns a facade handle.  Every ABI call on the facade is fanned out: member r
// runs the same entry point on its own device from its own short-lived host thread (rank 0 on the caller's thread), exactly
// as the ranks of a one-process-per-GPU launch would, so the sharded Schur assembly / row-block-cyclic Cholesky code is the
// same in both modes.  Host-visible outputs are taken from member 0; the other members write into thread-local scratch.
// The facade is generic over the handle type: lrn_create_multi (Float64, lrn_solver) and lrn_dd_create_multi (double-double
// LP path, lrn_dd_solver) share it.  A handle type needs `void* group` and `std::string err`.
#pragma once
#include "solver.cuh"
#include <thread>

namespace lrn {

template <typename Hd>
struct GroupOf {
    std::vector<Hd*> members;
};
using Group = GroupOf<lrn_solver>;

template <typename Hd, typename F>
int32_t group_call(Hd* facade, F&& f) {
    GroupOf<Hd>* g = static_cast<GroupOf<Hd>*>(facade->group);
    const int N = (int)g->members.size();
    facade->err.clear();
    std::vector<int32_t> rc(N, 0);
    std::vector<std::thread> th;
    th.reserve(N > 0 ? N - 1 : 0);
    for (int r = 1; r < N; r++) th.emplace_back([&, r] { rc[r] = f(g->members[r], r); });
    rc[0] = f(g->members[0], 0);
    for (auto& t : th) t.join();
    for (int r = 0; r < N; r++)
        if (rc[r] < 0) {
            facade->err = "[rank " + std::to_string(r) + "] " + g->members[r]->err;
            return rc[r];
        }
    return rc[0];
}

// scratch outputs of the members with rank > 0
struct GroupScratch {
    double d[16];
    int32_t i32[4];
    int64_t i64[4];
    std::vector<double> a, b;
};
inline GroupScratch& group_scratch() {
    thread_local GroupScratch s;
    return s;
}

}  // namespace lrn

// first statement of an entry point: fan the call out when `h` is a facade.  CALL uses m_ (member handle) and r_ (rank).
#define LRN_GROUP(h, CALL)                                                                          \
    do {                                                                                            \
        if ((h) && (h)->group)                                                                      \
            return lrn::group_call((h), [&](auto* m_, int r_) -> int32_t { (void)r_; return CALL; }); \
    } while (0)
