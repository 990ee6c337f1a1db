// fork_join.hpp -- run n jobs at once and wait for all of them; an exception of a job reaches the caller.
#pragma once
#include <exception>
#include <thread>
#include <vector>

// job(0 .. n-2) on threads of their own, job(n-1) on the calling thread.  Every thread that was started is joined, also when
// starting one fails; then the exception of the lowest-index job that threw is rethrown here (a throw on a thread of its own
// would end the process).  n <= 0: nothing runs.
template <class F>
void fork_join(int n, F &&job)
{
    if (n <= 0) return;
    std::vector<std::exception_ptr> err(n);
    auto run = [&](int i) {
        try { job(i); }
        catch (...) { err[i] = std::current_exception(); }
    };
    std::vector<std::thread> th;
    try {
        th.reserve(n - 1);
        for (int i = 0; i + 1 < n; ++i) th.emplace_back(run, i);
    } catch (...) {
        for (std::thread &t : th) t.join();
        throw;
    }
    run(n - 1);
    for (std::thread &t : th) t.join();
    for (const std::exception_ptr &e : err)
        if (e) std::rethrow_exception(e);
}
