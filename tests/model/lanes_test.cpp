// CPU check that the state step's result does not depend on how many lanes run it
// (nka_b200/csrc/nka_state.h, DESIGN.md section 4).  On the device the step runs on the 32 lanes of
// a warp and par.sync() is __syncwarp(); here the lanes are std::threads and par.sync() is a
// barrier, so a missing sync shows up as a data race (under -fsanitize=thread) and, mostly, as
// different bits.  Every op sequence given on the command line is run with the one-lane model
// from a zeroed and from a 0xFF-filled state, and on 2, 3, 32 and 33 threads; the outputs and the
// h, c, s arrays after every op must be bit-identical to the one-lane run.  Driven by
// tests/test_model.py.
//
//   lanes_test FILE...     FILE: int32 n, mvec, nops; float64 vtol; then per op int32 kind
//                          (0 update, 1 relax, 2 restart), followed by n float64 for an update
#include <atomic>
#include <chrono>
#include <thread>

#include <stdio.h>

#include "nka_model.cpp"

// A reusable barrier whose wait gives up after a while: a sync that not every lane reaches
// fails the run with a message instead of hanging it.  The lanes outnumber the cores, so a waiting
// lane yields its core rather than spinning on it or sleeping (a wake-up per lane per sync made the
// 33-lane runs ten times slower).
struct Barrier {
  int n = 1;
  std::atomic<int> count{0};
  std::atomic<unsigned> gen{0};
  void wait() {
    const unsigned g = gen.load(std::memory_order_acquire);
    if (count.fetch_add(1, std::memory_order_acq_rel) == n - 1) {
      count.store(0, std::memory_order_relaxed);
      gen.store(g + 1, std::memory_order_release);
      return;
    }
    const auto t0 = std::chrono::steady_clock::now();
    for (unsigned spins = 1; gen.load(std::memory_order_acquire) == g; ++spins) {
      std::this_thread::yield();
      if (spins % 4096 == 0 && std::chrono::steady_clock::now() - t0 > std::chrono::seconds(60)) {
        fprintf(stderr, "lanes_test: barrier timeout: a par.sync() was not reached by every lane\n");
        fflush(stderr);
        abort();
      }
    }
  }
};

struct ThreadPar {
  int l, n;
  Barrier* bar;
  int lane() const { return l; }
  int nlanes() const { return n; }
  void sync() const { bar->wait(); }
};

// The calling thread is lane 0; lanes 1..n-1 wait for a step, run their share and wait again.
struct Lanes {
  int n;
  Barrier bar;
  std::vector<std::thread> th;
  bool quit = false;
  NkaDevState* S = nullptr;
  NkaStepScratch* X = nullptr;
  const double* dots = nullptr;
  int have_last = 0;

  explicit Lanes(int nl) : n(nl) {
    bar.n = nl;
    for (int l = 1; l < nl; ++l) th.emplace_back([this, l] { loop(l); });
  }
  ~Lanes() {
    quit = true;
    bar.wait();
    for (std::thread& t : th) t.join();
  }
  void loop(int l) {
    for (;;) {
      bar.wait();
      if (quit) return;
      run(l);
      bar.wait();
    }
  }
  int run(int l) { return nka_state_step(*S, *X, dots, NKA_MAXSLOT, have_last, ThreadPar{l, n, &bar}); }
  int step(NkaDevState& s, NkaStepScratch& x, const double* d, int hl) {
    S = &s; X = &x; dots = d; have_last = hl;
    bar.wait();
    const int r = run(0);
    bar.wait();
    return r;
  }
};

static Lanes* g_lanes = nullptr;
static int lanes_step(NkaDevState& S, NkaStepScratch& X, const double* dots, int have_last)
{
  return g_lanes->step(S, X, dots, have_last);
}

struct Op { int kind; std::vector<double> f; };
struct Seq { int n = 0, mvec = 0; double vtol = 0.0; std::vector<Op> ops; };

static bool read_seq(const char* path, Seq& q)
{
  FILE* fp = fopen(path, "rb");
  if (!fp) return false;
  int hdr[3];
  bool ok = fread(hdr, sizeof hdr, 1, fp) == 1 && fread(&q.vtol, sizeof q.vtol, 1, fp) == 1;
  q.n = hdr[0]; q.mvec = hdr[1];
  for (int k = 0; ok && k < hdr[2]; ++k) {
    Op op;
    ok = fread(&op.kind, sizeof op.kind, 1, fp) == 1;
    if (ok && op.kind == 0) {
      op.f.resize(q.n);
      ok = q.n == 0 || fread(op.f.data(), sizeof(double), q.n, fp) == (size_t)q.n;
    }
    q.ops.push_back(std::move(op));
  }
  fclose(fp);
  return ok;
}

// What is compared after every op: the output of an update, then h, c, s of the state.
static std::vector<double> run_seq(const Seq& q, bool lazy, int poison, ModelStepFn step, int* ndrops)
{
  Model* m = model_init_ex(q.n, q.mvec, q.vtol, poison);
  if (!lazy) model_set_lazy(m, 0);
  m->step = step;
  std::vector<double> rec, f;
  for (const Op& op : q.ops) {
    if (op.kind == 0) {
      f = op.f;
      model_accel_update(m, f.data());
      rec.insert(rec.end(), f.begin(), f.end());
      *ndrops += m->S.ndrop_last;
    } else if (op.kind == 1) {
      model_relax(m);
    } else {
      model_restart(m);
    }
    rec.insert(rec.end(), m->S.h, m->S.h + NKA_MAXSLOT * NKA_MAXSLOT);
    rec.insert(rec.end(), m->S.c, m->S.c + NKA_MAXSLOT);
    rec.insert(rec.end(), m->S.s, m->S.s + NKA_MAXSLOT);
    if (m->S.error || model_bound_violations(m)) { fprintf(stderr, "model error\n"); exit(1); }
  }
  model_delete(m);
  return rec;
}

int main(int argc, char** argv)
{
  const int lane_counts[] = {2, 3, 32, 33};
  long runs = 0, calls = 0;
  int drops = 0;
  for (int a = 1; a < argc; ++a) {
    Seq q;
    if (!read_seq(argv[a], q)) { printf("FAIL cannot read %s\n", argv[a]); return 1; }
    for (int lazy = 1; lazy >= 0; --lazy) {
      int nd = 0;
      const std::vector<double> want = run_seq(q, lazy, 0, serial_step, &nd);
      drops += nd;
      auto check = [&](const std::vector<double>& got, const char* what, int lanes) {
        ++runs;
        if (got.size() == want.size() && memcmp(got.data(), want.data(), want.size() * sizeof(double)) == 0) return;
        size_t i = 0;
        while (i < got.size() && i < want.size() && memcmp(&got[i], &want[i], sizeof(double)) == 0) ++i;
        printf("FAIL %s lazy=%d %s lanes=%d: first difference at record word %zu (%.17g vs %.17g)\n", argv[a], lazy,
               what, lanes, i, i < got.size() ? got[i] : 0.0, i < want.size() ? want[i] : 0.0);
        exit(1);
      };
      check(run_seq(q, lazy, 1, serial_step, &nd), "0xFF-filled state", 1);
      for (int nl : lane_counts) {
        Lanes lanes(nl);
        g_lanes = &lanes;
        check(run_seq(q, lazy, 0, lanes_step, &nd), "zeroed state", nl);
        g_lanes = nullptr;
      }
    }
    for (const Op& op : q.ops) calls += op.kind == 0;
  }
  printf("lanes ok: %d sequences, %ld updates, %d vtol drops (lazy on and off), %ld runs bit-identical\n",
         argc - 1, calls, drops, runs);
  return 0;
}
