// final.cc — driver mirroring the reference's parallel-final/main.cu:34-161 on the B200-native library.
//
//   ./final -k 30 -f NAME                  reads ../data/NAME/NAME.mtx (main.cu:54), or --path FILE for an explicit file
//   ./final -k 50 --graph rmat --scale 20 [--ef 8] [--seed 1]     seeded generators (BASELINE.json configs)
//   ./final -k 20 --graph er -n 10000 -e 50000 [--seed S]
//   ./final -k 100 --graph band -n 1048576 [--seed S]
//   ./final -k 30 --graph ba -n 100000 -b 20                      Barabasi-Albert, as main.cu:67-71
//   options: --reorth (full reorthogonalisation)  --gpus N (row-sharded, one host thread per GPU, NCCL)
//            --check FILE (raw float64 e^A x to compare with, e.g. written by oracle/_ref/ref_final --out)
//            --write FILE (one value per line, write_ans)   --top M (print the M most central vertices, device-side ranking)
//            --t T (e^{TA} x, inverse temperature T)   --scaled (e^{T(A - sI)} x, s = largest Ritz value: never overflows; the log
//            scale T*s is printed)   --katz ALPHA ((I - ALPHA A)^{-1} x, Katz centrality)
//            --ritz M (the top M Ritz pairs with their certified eigenvalue intervals)   --eigcent (eigenvector centrality: the result
//            and --top are y_0; prints the spectral-radius bracket)   --katz-frac F (Katz with alpha = F / hi, hi the certified upper
//            bound on lambda_max, so F < 1 guarantees alpha < 1 / lambda_max; prints alpha and the bracket)
//
// Same object sequence as the reference: adjMatrix -> lanczosDecomp<double>(A,k,x,cuda=true) -> eigenDecomp<double> ->
// multOut(L,E,A,true), same TIMING / ERROR CHECKING tables. The reference's serial arm (main.cu:83-99) is not here: this
// library has no CPU path; the serial code is the test oracle (oracle/), whose answer can be passed with --check.
#include <cstdio>
#include <cstring>
#include <fstream>
#include <iomanip>
#include <iostream>
#include <string>
#include <thread>
#include <vector>
#include <sys/time.h>

#include "adjMatrix.h"
#include "check_ans.h"
#include "cu_lanczos.h"
#include "eigen.h"
#include "helpers.h"
#include "multiplyOut.h"
#include "ritz.h"
#include "write_ans.h"

#define WIDTH 81

static double seconds_between(timeval s, timeval e) { return e.tv_sec - s.tv_sec + (e.tv_usec - s.tv_usec) / 1000000.0; }

struct ritz_out {
  std::vector<double> theta, rho, res;
  double lo = 0.0, hi = 0.0;
};

static void print_ritz(const ritz_out& R, bool pairs) {
  std::cout << std::setprecision(17);
  if (pairs) {
    std::cout << "Ritz pairs (j theta rayleigh residual; [rayleigh - residual, rayleigh + residual] holds an eigenvalue of A)\n";
    for (size_t j = 0; j < R.theta.size(); j++)
      std::cout << "ritz " << j << ' ' << R.theta[j] << ' ' << R.rho[j] << ' ' << R.res[j] << " [" << R.rho[j] - R.res[j] << ", "
                << R.rho[j] + R.res[j] << "]\n";
  }
  std::cout << "spectral radius bracket: " << R.lo << ' ' << R.hi << '\n' << std::setprecision(6);
}

// Row-sharded run over `gpus` devices: one host thread per GPU, each driving its own lz_ctx (C ABI directly). ritz_m > 0: lz_ritz
// after the run; katz_frac > 0: then Katz with alpha = katz_frac / hi; eigcent: the result is y_0 (no coefficient solve).
static int run_multi(adjMatrix& A, unsigned k, int reorth, int gpus, int fkind, double fparam, std::vector<double>& ans, double& log_scale,
                     double& t_lanczos, double& t_mult, unsigned ritz_m, double katz_frac, bool eigcent, ritz_out& R) {
  unsigned char uid[LZ_NCCL_UID_BYTES];
  if (lz_nccl_unique_id(uid) != LZ_OK) { std::cerr << lz_last_error() << '\n'; return 1; }
  std::vector<int> rc(gpus, 0);
  std::vector<std::string> err(gpus);
  std::vector<double> tl(gpus, 0.0), tm(gpus, 0.0);
  std::vector<std::thread> th;
  for (int r = 0; r < gpus; r++) {
    th.emplace_back([&, r]() {
      lz_ctx* c = nullptr;
      auto bad = [&](int code) { rc[r] = code; err[r] = lz_last_error(); if (c) lz_destroy(c); };
      int e;
      if ((e = lz_create_dist(r, r, gpus, uid, &c)) != LZ_OK) return bad(e);
      if ((e = lz_set_matfun(c, fkind, fparam)) != LZ_OK) return bad(e);
      if ((e = lz_csr_upload(c, A.get_n(), A.get_row_offset(), A.get_col_idx())) != LZ_OK) return bad(e);
      if ((e = lz_set_start_vector(c, nullptr)) != LZ_OK) return bad(e);
      if ((e = lz_sync(c)) != LZ_OK) return bad(e);
      timeval s, e1, e2;
      gettimeofday(&s, NULL);
      if ((e = lz_lanczos_run(c, k, reorth)) != LZ_OK) return bad(e);
      if ((e = lz_sync(c)) != LZ_OK) return bad(e);
      gettimeofday(&e1, NULL);
      if (ritz_m) {
        ritz_out mine;
        mine.theta.resize(ritz_m); mine.rho.resize(ritz_m); mine.res.resize(ritz_m);
        if ((e = lz_ritz(c, ritz_m)) != LZ_OK) return bad(e);
        if ((e = lz_get_ritz(c, mine.theta.data(), mine.rho.data(), mine.res.data())) != LZ_OK) return bad(e);
        if ((e = lz_spectral_radius_bounds(c, &mine.lo, &mine.hi)) != LZ_OK) return bad(e);
        if (katz_frac > 0.0 && (e = lz_set_matfun(c, LZ_MATFUN_RESOLVENT, katz_frac / mine.hi)) != LZ_OK) return bad(e);
        if (r == 0) R = mine;
      }
      if (!eigcent) {
        if ((e = lz_tridiag_expv(c)) != LZ_OK) return bad(e);
        if ((e = lz_multout(c)) != LZ_OK) return bad(e);
      }
      std::vector<double> y(A.get_n());
      if ((e = lz_get_ans(c, y.data())) != LZ_OK) return bad(e);
      gettimeofday(&e2, NULL);
      tl[r] = seconds_between(s, e1); tm[r] = seconds_between(e1, e2);
      if (r == 0) {
        if (!eigcent && (e = lz_get_matfun_scale(c, &log_scale)) != LZ_OK) return bad(e);
        ans.swap(y);
      }
      lz_destroy(c);
    });
  }
  for (auto& t : th) t.join();
  for (int r = 0; r < gpus; r++)
    if (rc[r]) { std::cerr << "rank " << r << ": " << err[r] << '\n'; return 1; }
  t_lanczos = *std::max_element(tl.begin(), tl.end());
  t_mult = *std::max_element(tm.begin(), tm.end());
  return 0;
}

int main(int argc, char** argv) {
  unsigned n{10'000}, deg{5}, edges{n * 10}, krylov_dim{100}, width{17};
  bool verbose{true};
  std::string filename{"bn1000000e9999944"}, graph{"file"}, path, check_file, write_file;
  unsigned scale = 16, ef = 8;
  uint64_t seed = 1;
  int reorth = LZ_REORTH_NONE, gpus = 1;
  unsigned top = 0;
  double t = 1.0, katz = 0.0, katz_frac = 0.0;
  bool scaled = false, have_t = false, have_katz = false, have_katz_frac = false, eigcent = false;
  unsigned ritz_req = 0;

  // long options first; what is left goes to the reference's getopt string
  std::vector<char*> rest{argv[0]};
  for (int i = 1; i < argc; i++) {
    std::string a = argv[i];
    auto val = [&]() -> const char* { if (i + 1 >= argc) { std::cerr << "missing value for " << a << '\n'; exit(2); } return argv[++i]; };
    auto num = [&]() -> double {
      const char* v = val();
      char* end = nullptr;
      const double d = strtod(v, &end);
      if (end == v || *end) { std::cerr << "not a number for " << a << ": " << v << '\n'; exit(2); }
      return d;
    };
    if (a == "--graph") graph = val();
    else if (a == "--scale") scale = (unsigned)atoi(val());
    else if (a == "--ef") ef = (unsigned)atoi(val());
    else if (a == "--seed") seed = strtoull(val(), nullptr, 10);
    else if (a == "--path") path = val();
    else if (a == "--check") check_file = val();
    else if (a == "--write") write_file = val();
    else if (a == "--gpus") gpus = atoi(val());
    else if (a == "--reorth") reorth = LZ_REORTH_FULL;
    else if (a == "--top") top = (unsigned)atoi(val());
    else if (a == "--t") { t = num(); have_t = true; }
    else if (a == "--scaled") scaled = true;
    else if (a == "--katz") { katz = num(); have_katz = true; }
    else if (a == "--katz-frac") { katz_frac = num(); have_katz_frac = true; }
    else if (a == "--eigcent") eigcent = true;
    else if (a == "--ritz") { const double v = num(); ritz_req = (unsigned)v; if (v < 1 || v > LZ_RITZ_MAX || v != ritz_req) { std::cerr << "--ritz takes 1.." << LZ_RITZ_MAX << '\n'; return 2; } }
    else rest.push_back(argv[i]);
  }
  if (parseArguments((int)rest.size(), rest.data(), filename, krylov_dim, verbose, n, deg, edges) != 0) return 2;
  if (have_katz && (have_t || scaled)) { std::cerr << "--katz excludes --t and --scaled\n"; return 2; }
  if (have_katz_frac && (have_katz || have_t || scaled)) { std::cerr << "--katz-frac excludes --katz, --t and --scaled\n"; return 2; }
  if (have_katz_frac && !(katz_frac > 0.0 && katz_frac < 1.0)) { std::cerr << "--katz-frac takes a fraction in (0, 1)\n"; return 2; }
  if (eigcent && (have_katz || have_katz_frac || have_t || scaled)) { std::cerr << "--eigcent excludes --katz, --katz-frac, --t and --scaled\n"; return 2; }
  const unsigned ritz_m = ritz_req ? ritz_req : (eigcent || have_katz_frac) ? 1u : 0u;
  const int fkind = (have_katz || have_katz_frac) ? LZ_MATFUN_RESOLVENT : scaled ? LZ_MATFUN_EXP_SCALED : LZ_MATFUN_EXP;
  double fparam = have_katz ? katz : t;
  const bool default_fun = fkind == LZ_MATFUN_EXP && fparam == 1.0 && !eigcent;

  timeval start, end;
  gettimeofday(&start, NULL);
  adjMatrix A;
  adjMatrix::generator_seed = seed;
  if (graph == "file") {
    std::string filepath = path.empty() ? "../data/" + filename + "/" + filename + ".mtx" : path;
    std::cout << "Going to open file: " << filepath << std::endl;
    std::ifstream fs;
    fs.open(filepath);
    if (fs.fail()) { std::cerr << "File opening failed\n"; return 1; }
    fs >> n >> n >> edges;
    adjMatrix B(n, edges, fs);
    A = std::move(B);
  } else if (graph == "rmat") {
    A = adjMatrix::rmat(scale, ef, seed);
  } else if (graph == "er") {
    adjMatrix B(n, edges);
    A = std::move(B);
  } else if (graph == "band") {
    A = adjMatrix::banded(n, seed);
  } else if (graph == "ba") {
    adjMatrix B(n, deg, 'b');
    A = std::move(B);
  } else {
    std::cerr << "unknown --graph " << graph << '\n';
    return 2;
  }
  n = A.get_n();
  edges = A.get_edges();
  gettimeofday(&end, NULL);
  std::cout << "\nTime elapsed to build adjacency matrix with n = " << n << " edges = " << edges << ":\n\t" << seconds_between(start, end)
            << " seconds\n\n";
  std::cout << "Running Lanczos algorithm for krylov_dim " << krylov_dim << (reorth ? " with full reorthogonalisation" : "") << " on "
            << gpus << " GPU(s)\n\n";

  std::vector<double> x_double(n, 1);   // main.cu:79
  std::vector<double> result;
  double gpu_time_lanczos = 0, gpu_time_mult = 0, gpu_time_whole = 0, log_scale = 0;
  lz_timings tm{};
  ritz_out rz;
  auto label = [&]() {
    if (eigcent) return std::string("eigenvector centrality");
    if (fkind == LZ_MATFUN_RESOLVENT) return "Katz centrality (I - alpha A)^-1 x, alpha = " + std::to_string(fparam);
    if (!default_fun) return "total communicability e^{tA} x, t = " + std::to_string(fparam) + (scaled ? ", scaled by e^-log_scale" : "");
    return std::string("total communicability");
  };
  std::string fun_label;
  if (gpus > 1) {
    if (run_multi(A, krylov_dim, reorth, gpus, fkind, fparam, result, log_scale, gpu_time_lanczos, gpu_time_mult, ritz_m, katz_frac, eigcent, rz))
      return 1;
    if (have_katz_frac) fparam = katz_frac / rz.hi;
    fun_label = label();
    gpu_time_whole = gpu_time_lanczos + gpu_time_mult;
  } else {
    timeval s, e1, e2, e3;
    gettimeofday(&s, NULL);
    lanczosDecomp<double> cu_L(A, krylov_dim, &x_double[0], /*cuda=*/true, reorth);   // main.cu:115
    gettimeofday(&e1, NULL);
    if (ritz_m) {
      ritzPairs<double> R(cu_L, ritz_m);
      rz.theta = R.values(); rz.rho = R.rayleigh(); rz.res = R.residuals();
      R.spectral_radius_bounds(rz.lo, rz.hi);
      if (have_katz_frac) fparam = katz_frac / rz.hi;                                 // certified: alpha < 1 / lambda_max
      if (eigcent) {
        result.resize(n);
        R.vector(0, result.data());
      }
    }
    fun_label = label();
    if (eigcent) {                                                                    // the answer (and top_k) is y_0 until a multOut
      e2 = e3 = e1;
    } else {
      eigenDecomp<double> cu_E(cu_L, fkind, fparam);                                  // main.cu:124
      gettimeofday(&e2, NULL);
      multOut(cu_L, cu_E, A, true);                                                   // main.cu:127
      gettimeofday(&e3, NULL);
      result.assign(cu_L.get_ans_ptr(), cu_L.get_ans_ptr() + n);
      log_scale = cu_E.log_scale();
    }
    gpu_time_lanczos = seconds_between(s, e1);
    gpu_time_mult = seconds_between(e2, e3);
    gpu_time_whole = seconds_between(s, e3);
    tm = cu_L.timings();
    if (!write_file.empty() && !eigcent) write_ans(write_file, cu_L);                             // main.cu:159
    if (top) {
      std::vector<unsigned> ti(top);
      std::vector<double> tv(top);
      const unsigned cnt = cu_L.top_k(top, ti.data(), tv.data());
      std::cout << "TOP " << cnt << " vertices by " << fun_label << " (rank vertex value)\n" << std::setprecision(17);
      for (unsigned i = 0; i < cnt; i++) std::cout << "rank " << i + 1 << ' ' << ti[i] << ' ' << tv[i] << '\n';
      std::cout << std::setprecision(6);
    }
  }

  if (ritz_m) print_ritz(rz, ritz_req > 0);
  if (have_katz_frac) std::cout << "katz alpha: " << std::setprecision(17) << fparam << std::setprecision(6) << " (= " << katz_frac << " / hi)\n";
  if (eigcent) std::cout << "result: eigenvector centrality y_0 (unit 2-norm)\n";
  else if (!default_fun)
    std::cout << "matrix function: " << fun_label << "\nlog scale: " << std::setprecision(17) << log_scale << std::setprecision(6)
              << " (f(A) x = result * e^log_scale)\n";
  std::cout << std::setfill('~') << std::setw(WIDTH) << '\n' << std::setfill(' ');
  std::cout << "TIMING (host wall clock, seconds; Lanczos includes CSR upload and relabelling as the reference's includes its cudaMalloc + H2D)\n";
  std::cout << std::setfill('~') << std::setw(WIDTH) << '\n' << std::setfill(' ');
  std::cout << std::setw(width) << std::left << "Lanczos" << std::right << std::setw(width) << gpu_time_lanczos << "\n\n";
  std::cout << std::setw(width) << std::left << "Multiply Out" << std::right << std::setw(width) << gpu_time_mult << "\n\n";
  std::cout << std::setw(width) << std::left << "Entire algorithm" << std::right << std::setw(width) << gpu_time_whole << "\n\n";
  if (gpus == 1)
    std::cout << "device time: Lanczos loop " << tm.lanczos_ms << " ms (" << krylov_dim / (tm.lanczos_ms * 1e-3) << " iterations/s), tridiagonal "
              << tm.tridiag_ms << " ms, multOut " << tm.multout_ms << " ms, kernels launched " << tm.kernel_launches << "\n\n";

  std::cout << std::setfill('~') << std::setw(WIDTH) << '\n' << std::setfill(' ');
  std::cout << "ERROR CHECKING\n";
  std::cout << std::setfill('~') << std::setw(WIDTH) << '\n' << std::setfill(' ');
  bool finite = true;
  for (double v : result) finite &= std::isfinite(v);
  std::cout << "result finite: " << (finite ? "yes" : "NO") << ", ||ans||_2 = " << std::setprecision(17) << norm(result.data(), n) << '\n';
  int status = finite ? 0 : 3;
  if (!check_file.empty()) {
    std::vector<double> ref(n);
    FILE* f = fopen(check_file.c_str(), "rb");
    if (!f || fread(ref.data(), 8, n, f) != n) { std::cerr << "cannot read " << check_file << '\n'; return 1; }
    fclose(f);
    check_result r = compare_ans(ref.data(), result.data(), n);
    std::cout << "Max difference of " << std::setprecision(10) << r.max_abs << " found at index " << r.max_idx << '\n';
    std::cout << std::setw(30) << std::left << "Total norm of differences" << "=" << std::right << std::setprecision(20) << std::setw(30)
              << r.total_norm << '\n';
    std::cout << std::setw(30) << std::left << "Relative norm of differences" << "=" << std::right << std::setprecision(20)
              << std::setw(30) << r.relative_norm << std::endl;
    if (!(r.relative_norm < 1e-9)) status = 4;
  }
  if ((gpus > 1 || eigcent) && !write_file.empty()) {
    std::ofstream fs(write_file);
    fs << std::setprecision(17);
    for (double v : result) fs << v << '\n';
  }
  std::cout << std::setfill('~') << std::setw(WIDTH) << '\n' << std::setfill(' ');
  return status;
}
