// TEST INFRASTRUCTURE ONLY — C harness around the REFERENCE's own pixel selector: PixelSelector::makeMaps (FullSystem/PixelSelector2.cpp:
// L94-454) on a FrameHessian built by the reference's own FrameHessian::makeImages (HessianBlocks.cpp:L128-191).  Compiled by
// oracle/ref_select_build.sh into oracle/_ref/libdso_ref_select.so, linked against oracle/_ref/libdso_ref.so, which holds the reference's
// compiled translation units (PixelSelector2.cpp, HessianBlocks.cpp, settings.cpp, globalCalib.cpp among them; oracle/ref_build.sh).
// Nothing of the reference is copied into this repo.  tests/golden/make_select_golden.py records its results into
// tests/golden/ref_select.npz, against which tests/test_ref_pin_select.py pins the oracle (oracle/orc_select.cpp).
#include <cstdint>
#include <cstdlib>
#include <vector>

#define private public
#define protected public
#include "FullSystem/FullSystem.h"
#include "FullSystem/HessianBlocks.h"
#include "FullSystem/PixelSelector2.h"
#include "util/globalCalib.h"
#include "util/settings.h"
#undef private
#undef protected

using namespace dso;

extern "C" {

// settings4 = setting_minGradHistCut, setting_minGradHistAdd, setting_gradDownweightPerLevel, setting_selectDirectionDistribution (NULL = the
// defaults of util/settings.cpp:L167-170).  B256 = CalibHessian::B (NULL = the identity the CalibHessian constructor sets).
// currentPotential: the selector's state before (in) and after (out) the call.  map_out: w*h.  dIp_out (may be NULL): levels 0..2 of
// [I,dx,dy] concatenated, as the selector read them.  Returns makeMaps' numHaveSub.
int ref_make_maps(int w, int h, const double K[4], const float* image, const float* B256, const float* settings4, float density, int recursionsLeft,
                  float thFactor, int32_t* currentPotential, float* map_out, float* dIp_out) {
  Eigen::Matrix3f Km;
  Km.setZero();
  Km(0, 0) = (float)K[0]; Km(1, 1) = (float)K[1]; Km(0, 2) = (float)K[2]; Km(1, 2) = (float)K[3]; Km(2, 2) = 1.f;
  setGlobalCalib(w, h, Km);
  const float saved[4] = {setting_minGradHistCut, setting_minGradHistAdd, setting_gradDownweightPerLevel, (float)setting_selectDirectionDistribution};
  if (settings4) {
    setting_minGradHistCut = settings4[0]; setting_minGradHistAdd = settings4[1]; setting_gradDownweightPerLevel = settings4[2];
    setting_selectDirectionDistribution = settings4[3] != 0;
  }
  CalibHessian Hc;
  if (B256) for (int i = 0; i < 256; i++) Hc.B[i] = B256[i];
  FrameHessian* fh = new FrameHessian();
  for (int l = 0; l < PYR_LEVELS; l++) { fh->dIp[l] = 0; fh->absSquaredGrad[l] = 0; }
  std::vector<float> img(image, image + (size_t)w * h);
  fh->makeImages(img.data(), &Hc);
  // the first and last rows' gradients are left uninitialised by makeImages (L169-179): zero them, as the oracle and the product do
  for (int l = 0; l < 3; l++)
    for (int r : {0, hG[l] - 1})
      for (int x = 0; x < wG[l]; x++) {
        fh->dIp[l][r * wG[l] + x][1] = 0; fh->dIp[l][r * wG[l] + x][2] = 0; fh->absSquaredGrad[l][r * wG[l] + x] = 0;
      }
  // The fields PixelSelector::PixelSelector (L43-72) sets, set here without running it: its std::cout line faults when the reference's
  // objects are loaded into a Python process.  Same values, same sizes; randomPattern through the C library's own srand / rand.
  alignas(PixelSelector) unsigned char storage[sizeof(PixelSelector)];
  PixelSelector& sel = *reinterpret_cast<PixelSelector*>(storage);
  sel.randomPattern = new unsigned char[w * h];
  std::srand(3141592);
  for (int i = 0; i < w * h; i++) sel.randomPattern[i] = rand() & 0xFF;
  sel.bW = 16; sel.bH = 16; sel.nbW = w / 16; sel.nbH = h / 16;
  sel.gradHist = new int[100 * (1 + sel.nbW) * (1 + sel.nbH)];
  sel.ths = new float[sel.nbW * sel.nbH + 100];
  sel.thsSmoothed = new float[sel.nbW * sel.nbH + 100];
  sel.allowFast = false;
  sel.gradHistFrame = 0;
  sel.currentPotential = *currentPotential;
  const int numHaveSub = sel.makeMaps(fh, map_out, density, recursionsLeft, false, thFactor);
  *currentPotential = sel.currentPotential;
  sel.~PixelSelector();
  if (dIp_out)
    for (int l = 0, n = 0; l < 3; l++)
      for (int i = 0; i < wG[l] * hG[l]; i++)
        for (int k = 0; k < 3; k++) dIp_out[n++] = fh->dIp[l][i][k];
  delete fh;
  setting_minGradHistCut = saved[0]; setting_minGradHistAdd = saved[1]; setting_gradDownweightPerLevel = saved[2]; setting_selectDirectionDistribution = saved[3] != 0;
  return numHaveSub;
}

}  // extern "C"
