// Error plumbing, version and launch accounting for libb200rl.
#include <atomic>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>

#include "common.cuh"

namespace b200rl {

static thread_local char g_err[512] = "";
static std::atomic<int64_t> g_launches{0};

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

void count_launch(int n) { g_launches.fetch_add(n, std::memory_order_relaxed); }

static int g_pdl = -1;
int pdl_enabled() {
  if (g_pdl < 0) {
    const char* e = getenv("B200RL_PDL");
    g_pdl = e ? (atoi(e) != 0) : 1;   // on by default (B200RL_PDL=0 switches it off)
  }
  return g_pdl;
}

}  // namespace b200rl

extern "C" {

const char* b200rl_last_error(void) { return b200rl::g_err; }
int b200rl_version(void) { return 101; }
int64_t b200rl_launch_count(void) { return b200rl::g_launches.load(); }

int b200rl_set_pdl(int enabled) {
  b200rl::g_pdl = enabled ? 1 : 0;
  return B200RL_OK;
}
int b200rl_get_pdl(void) { return b200rl::pdl_enabled(); }

// Emission order of a `tf.data` style shuffle(buffer) over a stream of n elements
// (train/ppo_learner.py:236-238).  Host-side like the reference's input pipeline; the
// minibatch rows are then gathered on the device with b200rl_rb_read_rows.
int b200rl_shuffle_order(int64_t n, int64_t buffer, uint64_t seed, uint64_t call,
                         int64_t* out_host) {
  if (n < 0 || buffer < 1 || (n > 0 && out_host == nullptr)) {
    b200rl::set_error("shuffle_order: need n >= 0, buffer >= 1 and an output array");
    return B200RL_ERR_INVALID;
  }
  const int64_t cap = buffer < n ? buffer : n;
  int64_t* slots = cap > 0 ? new int64_t[cap] : nullptr;
  for (int64_t i = 0; i < cap; ++i) slots[i] = i;       // reservoir = first `cap` elements
  int64_t next_in = cap, fill = cap;
  for (int64_t i = 0; i < n; ++i) {
    const b200rl::Philox4 r = b200rl::philox4x32_10((uint64_t)i, call, seed);
    const int64_t j = b200rl::uniform_i64(r.x, r.y, 0, fill);
    out_host[i] = slots[j];
    if (next_in < n) {
      slots[j] = next_in++;                              // refill from the stream
    } else {
      slots[j] = slots[--fill];                          // stream exhausted: shrink
    }
  }
  delete[] slots;
  return B200RL_OK;
}

}  // extern "C"
