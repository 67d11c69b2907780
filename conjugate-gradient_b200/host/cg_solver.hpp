// cg_solver.hpp -- host-side mirror of the reference's `CGSolver` class: the union of the MPI
// interface (/root/reference/code/MPI/cg.hh:11-57) and the CUDA one (code/CUDA/cg.hh:13-45),
// same method names and argument meaning, so that a driver written against the reference
// compiles against this header.  Underneath, every method is a thin call into the C ABI
// (include/cgb200.h) -- one rank context per GPU, one host thread per rank for the collective
// steps.  Nothing is computed on the host; without a B200 the methods throw.
#pragma once

#include <cstdint>
#include <stdexcept>
#include <string>
#include <vector>

struct cgb_ctx;

class CGSolver {
public:
    CGSolver();
    ~CGSolver();
    CGSolver(const CGSolver &) = delete;
    CGSolver &operator=(const CGSolver &) = delete;

    /// read matrix from .mtx file (cg.cu:307-321: also sets m and n; max_iter = n)
    void read_matrix(const std::string &filename);

    /// initialize source term b_i = -2 i pi^2 sin(10 pi i h)^2 on the host (cg.cc:218-234)
    void init_source_term(double h);

    /// the reference's row partition (cg.cc:236-268)
    void partition_matrix(int N, int psize, int start_rows[], int num_rows[]);

    /// generate the synthetic Laplacian-like matrix directly in device memory (cg.cc:159-188)
    void generate_lap2d_matrix(int size);

    /// MPI-form solve (cg.cc:38-156): x holds x0 on entry and the solution on return; prints
    /// the DEBUG line
    void solve(std::vector<double> &x);

    /// CUDA-form solve (cg.cu:166-305): x is zero-filled first (cg.cu:217), the loop bound is
    /// n; NUM_THREADS / BLOCK_WIDTH / T select the mat-vec launch shape
    void solve(double *x, int NUM_THREADS, int BLOCK_WIDTH, bool T);

    /// fix maximum number of iterations for weak scaling experiments (cg.cc:204-216)
    void set_max_iter(int maxIter);

    inline int m() const { return m_m; }
    inline int n() const { return m_n; }

    /// prescribe residual tolerance for ending of the algorithm (cg.hh:39)
    void tolerance(double tolerance) { m_tolerance = tolerance; }

    // ---- additions of the B200 build ----------------------------------------------------
    /// CUDA devices to shard the rows over (the "psize" of the results row); default {0}
    void set_devices(const std::vector<int> &devices);
    int psize() const { return static_cast<int>(m_devices.size()); }

    struct Stats {
        int64_t k = 0;            // the k of "[STEP k]"
        int64_t iterations = 0;   // loop bodies executed
        bool converged = false;
        double rsold = 0, norm_x = 0, rel_resid = 0;
        double loop_seconds = 0;  // device-timed iteration loop (max over ranks)
        std::string gemv_variant;
    };
    const Stats &last_stats() const { return m_stats; }
    /// direct choice of the mat-vec variant (index or -1 = default)
    void set_gemv_variant(int v) { m_variant = v; }
    void set_quiet(bool q) { m_quiet = q; }
    /// the shards are held in CSR storage (environment CGB_STORAGE=csr at context creation)
    bool csr_storage() const { return m_csr; }

private:
    void ensure_contexts(int64_t n);
    void destroy_contexts();
    void run_solve(double *x, int64_t max_iter);
    void autotune();
    template <class F> void on_all_ranks(F &&f);

    int m_m{0};
    int m_n{0};
    int m_maxIter{0};
    std::vector<double> m_b;
    double m_tolerance{1e-10};

    std::vector<int> m_devices{0};
    std::vector<cgb_ctx *> m_ctx;
    int64_t m_ctx_n{0};
    bool m_rhs_uploaded{false};
    int m_variant{-1};
    bool m_quiet{false};
    bool m_csr{false};
    Stats m_stats;
};

/// map the reference's NUM_THREADS / BLOCK_WIDTH knobs (code/CUDA/cg_main.cc:21-25) onto the
/// nearest mat-vec variant: NUM_THREADS -> consumer warps per CTA, BLOCK_WIDTH -> column tile
int gemv_variant_for(int NUM_THREADS, int BLOCK_WIDTH);
