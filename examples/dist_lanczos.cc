// examples/dist_lanczos.cc -- E0 of the square-lattice Fermi-Hubbard model on SEVERAL GPUs from a plain C++ host: no Python, no
// MPI, no NCCL -- only the C ABI of libqbgpu (include/qbgpu.h, "multi-GPU drivers").
//
// The reference's driver is one C++ process (model<T>::locate_E0_lanczos, src/model.cc:1124-1316, as called by
// examples/trans_absent/latt_square/square_Fermi_Hubbard.cc).  Here the same call is spread over N processes, one per GPU
// (fork), each holding a row shard of H in the species order; the Krylov vector travels through peer memory (CUDA IPC over
// NVLink) and the Lanczos scalars through the library's push all-reduce kernel.  The only thing the host has to provide is
// a way to hand 64-byte handles around -- here: small files in /tmp.
//
//   g++ -std=c++17 -O2 -I include examples/dist_lanczos.cc -L quantum_basis_b200 -lqbgpu -Wl,-rpath,$PWD/quantum_basis_b200 -o dist_lanczos
//   ./dist_lanczos NGPUS [Lx Ly NUP NDN] [NEV]    (default 4 3 6 6: E0 = -16.879382788684, the reference's own value)
//
// NEV = 2 runs all of locate_E0_lanczos(nev = 2, ncv = 2) in one call (qbgpu_dist_locate_e0_lanczos): E0, phi0, E1 by the
// Lanczos run re-orthogonalised against phi0, phi1; it prints E0, E1, the gap and the four step counts.
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>
#include <sys/wait.h>
#include <unistd.h>
#include "qbgpu.h"

#define CHECK(call) do { int rc_ = (call); if (rc_ != 0) { fprintf(stderr, "rank %d: %s failed: %s\n", rank, #call, qbgpu_last_error()); _exit(3); } } while (0)

static long long binom(int n, int k) { long long r = 1; for (int i = 1; i <= k; i++) r = r * (n - k + i) / i; return r; }

static int run_rank(int rank, int world, int Lx, int Ly, int nup, int ndn, int nev, const std::string &tag)
{
    CHECK(qbgpu_init(rank));
    const int ns = Lx * Ly;
    std::vector<int32_t> bonds;                                   // the example's bond list: +x and +y bond of every site, PBC
    auto site = [&](int x, int y) { return ((x % Lx + Lx) % Lx) + ((y % Ly + Ly) % Ly) * Lx; };
    for (int x = 0; x < Lx; x++) for (int y = 0; y < Ly; y++) {
        bonds.push_back(site(x, y)); bonds.push_back(site(x + 1, y));
        bonds.push_back(site(x, y)); bonds.push_back(site(x, y + 1));
    }
    const long long Du = binom(ns, nup), Dd = binom(ns, ndn), n = Du * Dd;
    std::vector<int64_t> bounds(world + 1);                       // whole up configurations per rank (species-order shards)
    for (int r = 0; r <= world; r++) bounds[r] = (Du * r / world) * Dd;
    qbgpu_matrix_t A = nullptr, Ar = nullptr, local = nullptr, cross = nullptr;
    CHECK(qbgpu_build_hubbard(&A, ns, nup, ndn, (int)bonds.size() / 2, bonds.data(), 1.0, 1.1, /*api_complex=*/1,
                              QBGPU_SPECIES_ORDER, bounds[rank], bounds[rank + 1]));
    CHECK(qbgpu_real_view(A, &Ar));                               // H and the start vector are real: fp64 vectors
    CHECK(qbgpu_species_parts(Ar, &local, &cross));
    qbgpu_dist_t D = nullptr;
    CHECK(qbgpu_dist_create(&D, rank, world, n, bounds.data(), /*vec_complex=*/0));
    // hand the 64-byte handles around: every rank writes a file, then reads everybody's
    unsigned char mine[64];
    CHECK(qbgpu_dist_export(D, mine));
    { std::string p = tag + "." + std::to_string(rank) + ".tmp"; FILE *f = fopen(p.c_str(), "wb"); fwrite(mine, 1, 64, f); fclose(f);
      rename(p.c_str(), (tag + "." + std::to_string(rank)).c_str()); }
    std::vector<unsigned char> all(64 * world);
    for (int r = 0; r < world; r++) {
        const std::string p = tag + "." + std::to_string(r);
        FILE *f = nullptr;
        for (int tries = 0; tries < 6000 && !(f = fopen(p.c_str(), "rb")); tries++) usleep(10000);
        if (!f || fread(all.data() + 64 * r, 1, 64, f) != 64) { fprintf(stderr, "rank %d: no handle from rank %d\n", rank, r); _exit(4); }
        fclose(f);
    }
    CHECK(qbgpu_dist_connect(D, all.data()));
    // the reference's start vector vec_randomize(seed 1) (src/model.cc:1165), this rank's rows in the internal order
    int32_t *ref_rows = nullptr;
    CHECK(qbgpu_malloc((void **)&ref_rows, sizeof(int32_t) * (size_t)(bounds[rank + 1] - bounds[rank] + 1)));
    CHECK(qbgpu_species_ref_rows(ns, nup, ndn, bounds[rank], bounds[rank + 1], ref_rows));
    const int64_t maxit = 1000;
    if (nev == 2) {
        // E0, phi0, E1, phi1: the four stages of locate_E0_lanczos(nev = 2, ncv = 2) (src/model.cc:1124-1316); the start
        // vectors are drawn inside, so only the reference rows of the shard are passed
        double *phi = nullptr;                                    // this rank's rows of phi0 and phi1, one after the other
        CHECK(qbgpu_malloc((void **)&phi, sizeof(double) * 2 * (size_t)(bounds[rank + 1] - bounds[rank] + 1)));
        double E[2] = {0.0, 0.0}, accu[4];
        int64_t steps[4];
        CHECK(qbgpu_dist_locate_e0_lanczos(D, local, cross, ref_rows, 2, 2, maxit, E, phi, steps, accu));
        if (rank == 0) printf("E0 = %.12f   E1 = %.12f   gap = %.12f   steps: Lanczos E0 %lld, CG phi0 %lld, Lanczos E1 %lld, CG phi1 %lld   dim = %lld   GPUs = %d\n",
                              E[0], E[1], E[1] - E[0], (long long)steps[0], (long long)steps[1], (long long)steps[2], (long long)steps[3], n, world);
        qbgpu_free(phi);
    } else {
        CHECK(qbgpu_dist_randomize(D, 0, 1, ref_rows));
        std::vector<double> hess(2 * maxit), ritz(maxit);
        int64_t m = 0;
        CHECK(qbgpu_dist_lanczos(D, local, cross, maxit - 1, maxit, &m, hess.data(), "sr_val0", 1));     // stop rule of src/lanczos.cc:228-248
        CHECK(qbgpu_hess_eigen(hess.data(), maxit, m, ritz.data(), nullptr));
        if (rank == 0) printf("E0 = %.12f   Lanczos steps = %lld   dim = %lld   GPUs = %d\n", ritz[0], (long long)m, n, world);
    }
    fflush(stdout);                                               // the rank leaves through _exit, which does not flush
    qbgpu_free(ref_rows);
    qbgpu_dist_destroy(D);
    qbgpu_destroy(local); qbgpu_destroy(cross); qbgpu_destroy(Ar); qbgpu_destroy(A);
    unlink((tag + "." + std::to_string(rank)).c_str());
    return 0;
}

int main(int argc, char **argv)
{
    const int world = argc > 1 ? atoi(argv[1]) : 2;
    int Lx = 4, Ly = 3, nup = 6, ndn = 6;
    if (argc >= 6) { Lx = atoi(argv[2]); Ly = atoi(argv[3]); nup = atoi(argv[4]); ndn = atoi(argv[5]); }
    const int nev = argc == 3 ? atoi(argv[2]) : (argc >= 7 ? atoi(argv[6]) : 1);
    if (nev != 1 && nev != 2) { fprintf(stderr, "NEV must be 1 or 2\n"); return 2; }
    const std::string tag = "/tmp/qbgpu_dist_handles_" + std::to_string((long long)getpid());
    std::vector<pid_t> kids;
    for (int r = 0; r < world; r++) {                              // one process per GPU
        pid_t pid = fork();
        if (pid == 0) _exit(run_rank(r, world, Lx, Ly, nup, ndn, nev, tag));
        kids.push_back(pid);
    }
    int bad = 0;
    for (pid_t k : kids) { int st = 0; waitpid(k, &st, 0); bad += !(WIFEXITED(st) && WEXITSTATUS(st) == 0); }
    return bad ? 1 : 0;
}
