// rtb_k_mc.cu -- k_montecarlo (reference MainWindow.cpp:145-249 `radiance`) and k_whitted_tree (`trace` on scenes with
// refractive materials, MainWindow.cpp:69-143).
#include "rtb_launch.h"

namespace rtb {

template <bool MESH> static void tree(const Launch &L)
{
    if (L.count) k_whitted_tree<CountProbe, MESH><<<L.grid, RTB_CTA_THREADS, 0, L.stream>>>(*L.S, *L.F, L.out, L.counters);
    else k_whitted_tree<NoProbe, MESH><<<L.grid, RTB_CTA_THREADS, 0, L.stream>>>(*L.S, *L.F, L.out, L.counters);
}
void launchTree(const Launch &L) { if (L.mesh) tree<true>(L); else tree<false>(L); }

template <bool MESH> static void monteCarlo(const Launch &L)
{
    if (L.count) k_montecarlo<CountProbe, MESH><<<L.grid, RTB_CTA_THREADS, 0, L.stream>>>(*L.S, *L.F, L.out, L.counters);
    else k_montecarlo<NoProbe, MESH><<<L.grid, RTB_CTA_THREADS, 0, L.stream>>>(*L.S, *L.F, L.out, L.counters);
}
void launchMonteCarlo(const Launch &L) { if (L.mesh) monteCarlo<true>(L); else monteCarlo<false>(L); }

} // namespace rtb
