// hostemu_tiers.cpp — TEST INFRASTRUCTURE ONLY: the host emulation (hostemu_backend.cpp) with the tick
// kernel's fast gossip tier in front of the generic row step, so that the emulation takes a member
// through the same three tiers as gs_tick_kernel: the probe fast path for an empty mailbox whose ticker
// fires, gs_fast_gossip for a member with mail, gs_row_step for whatever either declines.  The
// emulation's single-tick loop calls gs_row_step after its probe fast path; that call is routed through
// gs_row_step_tiered below.  Its quiet-window loop calls the generic step with an empty mailbox only,
// which the tier declines, as the window kernel never runs it.
// GSIM_HOSTEMU_NO_FAST (generic step only) turns the tier off as well; GSIM_FLAG_NO_FAST_GOSSIP is
// honoured inside gs_fast_gossip itself.
#include "../../consul_b200/csrc/gs_aux.h"
#include "../../consul_b200/csrc/gs_backend.h"

#include <stdlib.h>

namespace {

// rows of single-tick launches each tier after the probe fast path took (gsim_hostemu_row_counts)
uint64_t g_fast_gossip_rows = 0, g_generic_rows = 0;

template <class Sink>
void gs_row_step_tiered(const GsDev& d, const GsGlobals& g, uint32_t i, uint32_t t, uint32_t gslot, uint32_t inb,
                        Sink& sink) {
  static const bool no_fast = getenv("GSIM_HOSTEMU_NO_FAST") != nullptr;
  // the kernel's drain reads `due` without the tile gate, as here
  if (inb != 0u && !no_fast && gs_fast_gossip(d, g, sink, i, t, gslot, inb, d.due[i] == t)) {
    __atomic_fetch_add(&g_fast_gossip_rows, 1ull, __ATOMIC_RELAXED);
    return;
  }
  if (inb != 0u) __atomic_fetch_add(&g_generic_rows, 1ull, __ATOMIC_RELAXED);
  gs_row_step(d, g, i, t, gslot, inb, sink);
}

}  // namespace

#define gs_row_step gs_row_step_tiered
#include "hostemu_backend.cpp"
#undef gs_row_step

// Test-only counters (not part of libgsim): rows with mail that the fast gossip tier took, and rows with
// mail that took the generic step, in single-tick launches since the library was loaded.
extern "C" void gsim_hostemu_row_counts(uint64_t out[2]) {
  out[0] = __atomic_load_n(&g_fast_gossip_rows, __ATOMIC_RELAXED);
  out[1] = __atomic_load_n(&g_generic_rows, __ATOMIC_RELAXED);
}
