// rtb_launch.h -- host-side launchers of the render kernels.  Every kernel family lives in its own translation unit
// (rtb_k_*.cu: the kernels are templates over the observation probe, the accelerator family and the fold-stack size,
// and one file with all of them took a minute to compile); rtb_abi.cu decides WHICH kernels share a frame
// (launchRender) and calls these.
#pragma once
#include "rtb_kernels.cuh"

namespace rtb {

struct Launch
{
    const DScene *S;
    const FrameParams *F;
    float *out;
    Counters *counters;
    dim3 grid;           // CTAs of RTB_CTA_THREADS threads
    cudaStream_t stream;
    bool count;          // CountProbe (frame.counters) instead of NoProbe
    bool mesh;           // the scene has RTB_PRIM_MESH records: the MESH instantiations (chain, tree, Monte Carlo only)
};

void launchChain(const Launch &L);                // k_whitted_chain        (rtb_k_chain.cu)
void launchChainSm(const Launch &L, bool grid);   // k_whitted_chain_sm     (rtb_k_sm.cu)
void launchChainOct(const Launch &L, bool grid);  // k_whitted_chain_oct    (rtb_k_oct.cu)
int octWarpsPerTile(int accel, int n_tiles);                   // warps the 8-lane / 16-lane kernel gives a tile (its grid is sized with this)
void launchChainWide(const Launch &L);            // k_whitted_chain_wide   (rtb_k_wide.cu)
void launchTree(const Launch &L);                 // k_whitted_tree         (rtb_k_mc.cu)
void launchMonteCarlo(const Launch &L);           // k_montecarlo           (rtb_k_mc.cu)

// the fold stack a frame needs (rtb_kernels.cuh: RTB_FOLD_SHORT / RTB_FOLD_LONG)
inline bool shortFold(const FrameParams &F) { return foldShortEnough(F.setting.max_depth); }

} // namespace rtb
