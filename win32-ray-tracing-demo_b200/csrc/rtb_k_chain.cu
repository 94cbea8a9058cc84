// rtb_k_chain.cu -- k_whitted_chain: the per-ray Whitted reflection chain, throughput kernel of the k-d trees, the flat
// grid, the linear scan and the convex accelerators (reference MainWindow.cpp:69-143 over Tunnel.cpp:786-1309).
#include "rtb_launch.h"

namespace rtb {

template <class Probe, int FOLD> static void go(const Launch &L)
{
    if (L.mesh) k_whitted_chain<Probe, FOLD, true><<<L.grid, RTB_CTA_THREADS, 0, L.stream>>>(*L.S, *L.F, L.out, L.counters);
    else k_whitted_chain<Probe, FOLD><<<L.grid, RTB_CTA_THREADS, 0, L.stream>>>(*L.S, *L.F, L.out, L.counters);
}

void launchChain(const Launch &L)
{
    const bool s = shortFold(*L.F);
    if (L.count) { if (s) go<CountProbe, RTB_FOLD_SHORT>(L); else go<CountProbe, RTB_FOLD_LONG>(L); }
    else { if (s) go<NoProbe, RTB_FOLD_SHORT>(L); else go<NoProbe, RTB_FOLD_LONG>(L); }
}

} // namespace rtb
