// cgsolver_main.cpp -- the `cgsolver` program with BOTH command lines of the reference:
//
//   cgsolver N outfile [max_iter]
//       (/root/reference/code/MPI/cg_main.cc:13-69)  synthetic generate_lap2d_matrix(N) system,
//       appends "n,psize,seconds" to outfile; psize = number of GPUs.
//   cgsolver file.mtx NUM_THREADS BLOCK_WIDTH true/false outfile
//       (/root/reference/code/CUDA/cg_main.cc:16-63)  Matrix Market system, appends
//       "NUM_THREADS,BLOCK_WIDTH,seconds", also prints "Time for CG (dense solver)  = ... [s]".
//
// The reference ships these as two binaries; here argv[1] decides: an integer selects the
// first form.  The MPI launcher's rank count (`srun -n P`) becomes the environment variable
// CGB_GPUS (number of GPUs, default 1) or CGB_DEVICES (comma-separated device list).
// CGB_STORAGE=csr holds the matrix in CSR storage instead of dense shards (same output).
#include "cg_solver.hpp"

#include <chrono>
#include <cstdlib>
#include <fstream>
#include <iostream>
#include <sstream>
#include <string>
#include <vector>

using clk = std::chrono::high_resolution_clock;
using second = std::chrono::duration<double>;

static bool is_integer(const std::string &s)
{
    if (s.empty()) return false;
    size_t i = (s[0] == '+' || s[0] == '-') ? 1 : 0;
    if (i == s.size()) return false;
    for (; i < s.size(); ++i)
        if (s[i] < '0' || s[i] > '9') return false;
    return true;
}

static std::vector<int> devices_from_env()
{
    std::vector<int> dev;
    if (const char *list = std::getenv("CGB_DEVICES")) {
        std::stringstream ss(list);
        std::string tok;
        while (std::getline(ss, tok, ','))
            if (!tok.empty()) dev.push_back(std::stoi(tok));
    } else if (const char *g = std::getenv("CGB_GPUS")) {
        for (int d = 0; d < std::stoi(g); ++d) dev.push_back(d);
    }
    if (dev.empty()) dev.push_back(0);
    return dev;
}

static void write_json(const CGSolver &solver, double elapsed)
{
    // optional side channel (never read by the reference tooling): CGB_JSON=<path>
    const char *path = std::getenv("CGB_JSON");
    if (!path) return;
    const CGSolver::Stats &s = solver.last_stats();
    std::ofstream js(path, std::ios_base::app);
    js.precision(17);
    js << "{\"n\": " << solver.n() << ", \"gpus\": " << solver.psize() << ", \"k\": " << s.k
       << ", \"iterations\": " << s.iterations << ", \"converged\": " << (s.converged ? "true" : "false")
       << ", \"solve_seconds\": " << elapsed << ", \"loop_seconds\": " << s.loop_seconds
       << ", \"it_per_s\": " << (s.loop_seconds > 0 ? s.iterations / s.loop_seconds : 0.0)
       << ", \"gemv_variant\": \"" << s.gemv_variant << "\", \"norm_x\": " << s.norm_x
       << ", \"rel_resid\": " << s.rel_resid << ", \"rsold\": " << s.rsold
       << (solver.csr_storage() ? ", \"storage\": \"csr\"" : "") << "}" << std::endl;
}

// cgsolver N outfile [max_iter]
static int main_generated(int argc, char **argv)
{
    CGSolver solver;
    solver.set_devices(devices_from_env());
    solver.generate_lap2d_matrix(std::stoi(argv[1]));
    int n = solver.n();

    if (argc >= 4) { // weak-scaling runs cap the iteration count
        int maxIter;
        std::stringstream arg(argv[3]);
        arg >> maxIter;
        solver.set_max_iter(maxIter);
    }

    double h = 1. / n;
    solver.init_source_term(h);
    std::vector<double> x_d(n, 0.);

    auto t1 = clk::now();
    solver.solve(x_d);
    second elapsed = clk::now() - t1;

    if (argc >= 3) {
        std::ofstream outfile(argv[2], std::ios_base::app);
        outfile << n << "," << solver.psize() << "," << elapsed.count() << std::endl;
    }
    write_json(solver, elapsed.count());
    return 0;
}

// cgsolver file.mtx NUM_THREADS BLOCK_WIDTH true/false outfile
static int main_matrix_market(int argc, char **argv)
{
    if (argc < 6) {
        // the reference's CUDA program prints its usage on stderr and exits 0 (code/CUDA/cg_main.cc:11-18;
        // its MPI program returns 1, cg_main.cc:22-26 -- kept in main() below)
        std::cerr << "Usage: " << argv[0] << " file.mtx NUM_THREADS BLOCK_WIDTH true/false outfile" << std::endl;
        return 0;
    }
    int NUM_THREADS = std::stoi(argv[2]); // stoi on purpose: cg.run passes "64," style tokens
    int BLOCK_WIDTH = std::stoi(argv[3]);
    bool T = std::string(argv[4]) == "true";
    std::string OUTPUT_FILE(argv[5]);

    CGSolver solver;
    solver.set_devices(devices_from_env());
    solver.read_matrix(argv[1]);
    int n = solver.n();
    double h = 1. / n;
    solver.init_source_term(h);
    std::vector<double> x_d(n);

    auto t1 = clk::now();
    solver.solve(x_d.data(), NUM_THREADS, BLOCK_WIDTH, T);
    second elapsed = clk::now() - t1;
    // std::scientific set by the DEBUG line is sticky on cout, exactly as in the reference
    std::cout << "Time for CG (dense solver)  = " << elapsed.count() << " [s]\n";

    std::ofstream outfile(OUTPUT_FILE.c_str(), std::ios_base::app);
    outfile << NUM_THREADS << "," << BLOCK_WIDTH << "," << elapsed.count() << std::endl;
    write_json(solver, elapsed.count());
    return 0;
}

int main(int argc, char **argv)
{
    if (argc < 2) {
        std::cerr << "Usage: " << argv[0] << " N outfile [max_iter]" << std::endl
                  << "       " << argv[0] << " file.mtx NUM_THREADS BLOCK_WIDTH true/false outfile" << std::endl;
        return 1; // code/MPI/cg_main.cc:22-26
    }
    try {
        return is_integer(argv[1]) ? main_generated(argc, argv) : main_matrix_market(argc, argv);
    } catch (const std::exception &e) {
        std::cerr << "cgsolver: " << e.what() << std::endl;
        return 2;
    }
}
