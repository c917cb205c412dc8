// TEST INFRASTRUCTURE ONLY — CPU oracle (restatement) of DM-VIO's pixel selection for new keyframes:
// PixelSelector::makeHists / select / makeMaps (FullSystem/PixelSelector2.cpp:L94-454), the gamma-weighted absSquaredGrad it reads
// (FrameHessian::makeImages, HessianBlocks.cpp:L168-188; CalibHessian::getBGradOnly, HessianBlocks.h:L394-400) and the loop of
// FullSystem::makeNewTraces (FullSystem.cpp:L1640-1665).  Pinned bit-exact against the reference's own PixelSelector2.cpp compiled into
// oracle/_ref (tests/test_ref_pin_select.py).  Plain float arithmetic in the reference's operation order, no FMA contraction.
#pragma once
#include <cstdint>

namespace orc {

struct SelectSettings {  // util/settings.cpp:L167-170
  float minGradHistCut = 0.5f, minGradHistAdd = 7.f, gradDownweightPerLevel = 0.75f;
  int selectDirectionDistribution = 1;
};

// the bytes of PixelSelector::randomPattern (PixelSelector2.cpp:L45-47): glibc srand(3141592), then rand() & 0xFF, n times
void randomPattern(int n, uint8_t* out);

// PixelSelector::makeMaps on the frame whose levels 0..2 are dIp[l] (w_l*h_l*3 floats, [I,dx,dy]); B256 = CalibHessian::B or nullptr.
// currentPotential is the selector's state (in/out).  map_out: w*h floats of 0/1/2/4.  Returns numHaveSub.
int makeMaps(int w, int h, const float* const dIp[3], const float* B256, const SelectSettings& s, float density, int recursionsLeft, float thFactor,
             int& currentPotential, float* map_out);

}  // namespace orc

extern "C" {
void orc_random_pattern(int n, uint8_t* out);
/* settings4 = minGradHistCut, minGradHistAdd, gradDownweightPerLevel, selectDirectionDistribution (NULL = defaults) */
int orc_make_maps(int w, int h, const float* dIp0, const float* dIp1, const float* dIp2, const float* B256, const float* settings4, float density,
                  int recursionsLeft, float thFactor, int32_t* currentPotential, float* map_out);
/* FullSystem::makeNewTraces: makeMaps with (density, recursionsLeft, thFactor), then an ImmaturePoint per selected pixel in
 * [patternPadding+1, dim-patternPadding-2) in raster order, dropping those whose energyTH is not finite.  Writes at most cap points;
 * returns the number kept (larger than cap: nothing but *numHaveSub / *currentPotential written). */
int orc_make_new_traces(int w, int h, const float* dIp0, const float* dIp1, const float* dIp2, const float* B256, const float* settings4, float density,
                        int recursionsLeft, float thFactor, int32_t* currentPotential, int32_t* numHaveSub, int cap, int32_t* u, int32_t* v, float* type,
                        float* color8, float* weights8, float* gradH4, float* energyTH);
}
