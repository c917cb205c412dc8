// TEST INFRASTRUCTURE ONLY — see orc_select.h.
#include "orc_select.h"
#include "orc_trace.h"
#include <algorithm>
#include <cmath>
#include <cstring>
#include <vector>

namespace orc {

void randomPattern(int n, uint8_t* out) {
  // glibc's TYPE_3 additive generator (random_r.c): 31 words seeded by the Park-Miller step, 310 outputs discarded, then
  // r[i] = r[i-31] + r[i-3] (mod 2^32) and rand() = r[i] >> 1
  std::vector<uint32_t> r((size_t)n + 344);
  int32_t word = 3141592;
  r[0] = (uint32_t)word;
  for (int i = 1; i < 31; i++) {
    const int32_t hi = word / 127773, lo = word % 127773;
    word = 16807 * lo - 2836 * hi;
    if (word < 0) word += 2147483647;
    r[i] = (uint32_t)word;
  }
  for (int i = 31; i < 34; i++) r[i] = r[i - 31];
  for (size_t i = 34; i < r.size(); i++) r[i] = r[i - 31] + r[i - 3];
  for (int i = 0; i < n; i++) out[i] = (uint8_t)((r[(size_t)i + 344] >> 1) & 0xFF);
}

namespace {

const float kDirections[16][2] = {  // PixelSelector2.cpp:L328-344
    {0, 1.0000f},       {0.3827f, 0.9239f}, {0.1951f, 0.9808f}, {0.9239f, 0.3827f},  {0.7071f, 0.7071f}, {0.3827f, -0.9239f},
    {0.8315f, 0.5556f}, {0.8315f, -0.5556f}, {0.5556f, -0.8315f}, {0.9808f, 0.1951f}, {0.9239f, -0.3827f}, {0.7071f, -0.7071f},
    {0.5556f, 0.8315f}, {0.9808f, -0.1951f}, {1.0000f, 0.0000f}, {0.1951f, -0.9808f}};

int histQuantil(const int* hist, float below) {  // computeHistQuantil, L82-91
  int th = hist[0] * below + 0.5f;
  for (int i = 0; i < 90; i++) {
    th -= hist[i + 1];
    if (th < 0) return i;
  }
  return 90;
}

struct Selector {
  int w, h, nbW, nbH;
  const float* dI;           // level 0, [I,dx,dy]
  std::vector<float> ag[3];  // absSquaredGrad[0..2]
  std::vector<float> ths, thsSmoothed;
  std::vector<uint8_t> rp;
  SelectSettings s;
};

// absSquaredGrad of one level (HessianBlocks.cpp:L168-188): dx*dx+dy*dy, times gw*gw (getBGradOnly) when B is given; first / last row 0
void absSquaredGrad(const float* dI, int wl, int hl, const float* B, std::vector<float>& out) {
  out.assign((size_t)wl * hl, 0.f);
  for (int idx = wl; idx < wl * (hl - 1); idx++) {
    const float dx = dI[3 * idx + 1], dy = dI[3 * idx + 2];
    out[idx] = dx * dx + dy * dy;
    if (B) {
      int c = dI[3 * idx] + 0.5f;
      if (c < 5) c = 5;
      if (c > 250) c = 250;
      const float gw = B[c + 1] - B[c];
      out[idx] *= gw * gw;
    }
  }
}

void makeHists(Selector& S) {  // L94-157
  const int w = S.w, h = S.h, w32 = S.nbW, h32 = S.nbH;
  S.ths.assign((size_t)w32 * h32, 0.f);
  S.thsSmoothed.assign((size_t)w32 * h32, 0.f);
  int hist[91];  // computeHistQuantil reads bins up to 90; the reference clears 50 of its (larger) buffer, bins past 49 are taken as 0
  for (int y = 0; y < h32; y++)
    for (int x = 0; x < w32; x++) {
      const float* map0 = S.ag[0].data() + 16 * x + 16 * y * w;
      std::memset(hist, 0, sizeof(hist));
      for (int j = 0; j < 16; j++)
        for (int i = 0; i < 16; i++) {
          const int it = i + 16 * x, jt = j + 16 * y;
          if (it > w - 2 || jt > h - 2 || it < 1 || jt < 1) continue;
          int g = sqrtf(map0[i + j * w]);
          if (g > 48) g = 48;
          hist[g + 1]++;
          hist[0]++;
        }
      S.ths[x + y * w32] = histQuantil(hist, S.s.minGradHistCut) + S.s.minGradHistAdd;
    }
  const float* ths = S.ths.data();
  for (int y = 0; y < h32; y++)
    for (int x = 0; x < w32; x++) {
      float sum = 0, num = 0;
      if (x > 0) {
        if (y > 0) { num++; sum += ths[x - 1 + (y - 1) * w32]; }
        if (y < h32 - 1) { num++; sum += ths[x - 1 + (y + 1) * w32]; }
        num++; sum += ths[x - 1 + y * w32];
      }
      if (x < w32 - 1) {
        if (y > 0) { num++; sum += ths[x + 1 + (y - 1) * w32]; }
        if (y < h32 - 1) { num++; sum += ths[x + 1 + (y + 1) * w32]; }
        num++; sum += ths[x + 1 + y * w32];
      }
      if (y > 0) { num++; sum += ths[x + (y - 1) * w32]; }
      if (y < h32 - 1) { num++; sum += ths[x + (y + 1) * w32]; }
      num++; sum += ths[x + y * w32];
      S.thsSmoothed[x + y * w32] = (sum / num) * (sum / num);
    }
}

// PixelSelector::select (L311-454): one raster walk over 4pot / 2pot / pot blocks; returns n2 + n3 + n4 through n[3]
void select(const Selector& S, float* map_out, int pot, float thFactor, int n[3]) {
  const int w = S.w, h = S.h, w1 = w / 2, w2 = w / 4;
  const float *mapmax0 = S.ag[0].data(), *mapmax1 = S.ag[1].data(), *mapmax2 = S.ag[2].data();
  std::memset(map_out, 0, sizeof(float) * w * h);
  const float dw1 = S.s.gradDownweightPerLevel, dw2 = dw1 * dw1;
  const bool useDir = S.s.selectDirectionDistribution != 0;
  auto dirNormOf = [&](int idx, const float* d) { return fabsf(S.dI[3 * idx + 1] * d[0] + S.dI[3 * idx + 2] * d[1]); };
  int n3 = 0, n2 = 0, n4 = 0;
  for (int y4 = 0; y4 < h; y4 += 4 * pot)
    for (int x4 = 0; x4 < w; x4 += 4 * pot) {
      const int my3 = std::min(4 * pot, h - y4), mx3 = std::min(4 * pot, w - x4);
      int bestIdx4 = -1;
      float bestVal4 = 0;
      const float* dir4 = kDirections[S.rp[n2] & 0xF];
      for (int y3 = 0; y3 < my3; y3 += 2 * pot)
        for (int x3 = 0; x3 < mx3; x3 += 2 * pot) {
          const int x34 = x3 + x4, y34 = y3 + y4;
          const int my2 = std::min(2 * pot, h - y34), mx2 = std::min(2 * pot, w - x34);
          int bestIdx3 = -1;
          float bestVal3 = 0;
          const float* dir3 = kDirections[S.rp[n2] & 0xF];
          for (int y2 = 0; y2 < my2; y2 += pot)
            for (int x2 = 0; x2 < mx2; x2 += pot) {
              const int x234 = x2 + x34, y234 = y2 + y34;
              const int my1 = std::min(pot, h - y234), mx1 = std::min(pot, w - x234);
              int bestIdx2 = -1;
              float bestVal2 = 0;
              const float* dir2 = kDirections[S.rp[n2] & 0xF];
              for (int y1 = 0; y1 < my1; y1++)
                for (int x1 = 0; x1 < mx1; x1++) {
                  const int xf = x1 + x234, yf = y1 + y234, idx = xf + w * yf;
                  if (xf < 4 || xf >= w - 5 || yf < 4 || yf > h - 4) continue;
                  const float pixelTH0 = S.thsSmoothed[xf / 16 + (yf / 16) * S.nbW];
                  const float pixelTH1 = pixelTH0 * dw1;
                  const float pixelTH2 = pixelTH1 * dw2;
                  const float ag0 = mapmax0[idx];
                  if (ag0 > pixelTH0 * thFactor) {
                    const float dn = useDir ? dirNormOf(idx, dir2) : ag0;
                    if (dn > bestVal2) { bestVal2 = dn; bestIdx2 = idx; bestIdx3 = -2; bestIdx4 = -2; }
                  }
                  if (bestIdx3 == -2) continue;
                  // (int)(xf*0.5f+0.25f) == xf/2 and (int)(xf*0.25f+0.125) == xf/4 exactly for the non-negative integers here
                  const float ag1 = mapmax1[(int)(xf * 0.5f + 0.25f) + (int)(yf * 0.5f + 0.25f) * w1];
                  if (ag1 > pixelTH1 * thFactor) {
                    const float dn = useDir ? dirNormOf(idx, dir3) : ag1;
                    if (dn > bestVal3) { bestVal3 = dn; bestIdx3 = idx; bestIdx4 = -2; }
                  }
                  if (bestIdx4 == -2) continue;
                  const float ag2 = mapmax2[(int)(xf * 0.25f + 0.125) + (int)(yf * 0.25f + 0.125) * w2];
                  if (ag2 > pixelTH2 * thFactor) {
                    const float dn = useDir ? dirNormOf(idx, dir4) : ag2;
                    if (dn > bestVal4) { bestVal4 = dn; bestIdx4 = idx; }
                  }
                }
              if (bestIdx2 > 0) { map_out[bestIdx2] = 1; bestVal3 = 1e10; n2++; }
            }
          if (bestIdx3 > 0) { map_out[bestIdx3] = 2; bestVal4 = 1e10; n3++; }
        }
      if (bestIdx4 > 0) { map_out[bestIdx4] = 4; n4++; }
    }
  n[0] = n2; n[1] = n3; n[2] = n4;
}

int makeMapsRec(const Selector& S, float* map_out, float density, int recursionsLeft, float thFactor, int& currentPotential) {  // L158-307
  float numHave = 0, numWant = density, quotia;
  int idealPotential = currentPotential;
  {
    int n[3];
    select(S, map_out, currentPotential, thFactor, n);
    numHave = n[0] + n[1] + n[2];
    quotia = numWant / numHave;
    float K = numHave * (currentPotential + 1) * (currentPotential + 1);
    idealPotential = sqrtf(K / numWant) - 1;
    if (idealPotential < 1) idealPotential = 1;
    if (recursionsLeft > 0 && quotia > 1.25 && currentPotential > 1) {
      if (idealPotential >= currentPotential) idealPotential = currentPotential - 1;
      currentPotential = idealPotential;
      return makeMapsRec(S, map_out, density, recursionsLeft - 1, thFactor, currentPotential);
    } else if (recursionsLeft > 0 && quotia < 0.25) {
      if (idealPotential <= currentPotential) idealPotential = currentPotential + 1;
      currentPotential = idealPotential;
      return makeMapsRec(S, map_out, density, recursionsLeft - 1, thFactor, currentPotential);
    }
  }
  int numHaveSub = numHave;
  if (quotia < 0.95) {
    int rn = 0;
    unsigned char charTH = 255 * quotia;
    for (int i = 0; i < S.w * S.h; i++)
      if (map_out[i] != 0) {
        if (S.rp[rn] > charTH) { map_out[i] = 0; numHaveSub--; }
        rn++;
      }
  }
  currentPotential = idealPotential;
  return numHaveSub;
}

}  // namespace

int makeMaps(int w, int h, const float* const dIp[3], const float* B256, const SelectSettings& s, float density, int recursionsLeft, float thFactor,
             int& currentPotential, float* map_out) {
  Selector S;
  S.w = w; S.h = h; S.nbW = w / 16; S.nbH = h / 16; S.dI = dIp[0]; S.s = s;
  for (int l = 0; l < 3; l++) absSquaredGrad(dIp[l], w >> l, h >> l, B256, S.ag[l]);
  S.rp.resize((size_t)w * h);
  randomPattern(w * h, S.rp.data());
  makeHists(S);
  return makeMapsRec(S, map_out, density, recursionsLeft, thFactor, currentPotential);
}

}  // namespace orc

namespace {
orc::SelectSettings settings_of(const float* s4) {
  orc::SelectSettings s;
  if (s4) { s.minGradHistCut = s4[0]; s.minGradHistAdd = s4[1]; s.gradDownweightPerLevel = s4[2]; s.selectDirectionDistribution = (int)s4[3]; }
  return s;
}
}  // namespace

extern "C" {
void orc_random_pattern(int n, uint8_t* out) { orc::randomPattern(n, out); }

int orc_make_maps(int w, int h, const float* dIp0, const float* dIp1, const float* dIp2, const float* B256, const float* settings4, float density,
                  int recursionsLeft, float thFactor, int32_t* currentPotential, float* map_out) {
  const float* lv[3] = {dIp0, dIp1, dIp2};
  int pot = *currentPotential;
  const int r = orc::makeMaps(w, h, lv, B256, settings_of(settings4), density, recursionsLeft, thFactor, pot, map_out);
  *currentPotential = pot;
  return r;
}

int orc_make_new_traces(int w, int h, const float* dIp0, const float* dIp1, const float* dIp2, const float* B256, const float* settings4, float density,
                        int recursionsLeft, float thFactor, int32_t* currentPotential, int32_t* numHaveSub, int cap, int32_t* u, int32_t* v, float* type,
                        float* color8, float* weights8, float* gradH4, float* energyTH) {
  std::vector<float> map((size_t)w * h);
  *numHaveSub = orc_make_maps(w, h, dIp0, dIp1, dIp2, B256, settings4, density, recursionsLeft, thFactor, currentPotential, map.data());
  const int patternPadding = 2;  // FullSystem.cpp:L1652-1664
  std::vector<orc::ImmaturePt> kept;
  std::vector<float> types;
  const orc::TraceSettings ts;
  for (int y = patternPadding + 1; y < h - patternPadding - 2; y++)
    for (int x = patternPadding + 1; x < w - patternPadding - 2; x++) {
      const int i = x + y * w;
      if (map[i] == 0) continue;
      orc::ImmaturePt p;
      orc::initImmature(p, dIp0, w, x, y, ts);
      if (!std::isfinite(p.energyTH)) continue;
      kept.push_back(p);
      types.push_back(map[i]);
    }
  const int n = (int)kept.size();
  if (n > cap) return n;
  for (int k = 0; k < n; k++) {
    const orc::ImmaturePt& p = kept[k];
    u[k] = (int32_t)p.u; v[k] = (int32_t)p.v; type[k] = types[k];
    std::memcpy(color8 + 8 * k, p.color, 32); std::memcpy(weights8 + 8 * k, p.weights, 32); std::memcpy(gradH4 + 4 * k, p.gradH, 16);
    energyTH[k] = p.energyTH;
  }
  return n;
}
}
