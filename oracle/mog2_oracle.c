/* mog2_oracle.c -- TEST INFRASTRUCTURE ONLY: a scalar C restatement of OpenCV's BackgroundSubtractorMOG2
 * (cv2.createBackgroundSubtractorMOG2(detectShadows=False), one uint8 channel, five modes), which tests/test_mog2_oracle.py
 * holds equal to live cv2 (4.13) on every foreground mask and on getBackgroundImage, and tests/test_mog2_gpu.py holds the
 * device kernels (csrc/mog2_kernels.cu) to.  Layout per pixel: gmm[npx][5] = {weight, variance}, mean[npx][5], used[npx].
 * Built with -ffp-contract=off: every a*b+c is two rounded operations, as in cv2's build (a fused multiply-add changes
 * background pixels).  The per-frame learning-rate rule is host logic (oracle/mog2_oracle.py).
 *
 * stats (may be NULL) counts, over all pixels of the call, which branches ran:
 *   [0] a mode pruned (weight < -prune: the nmodes-- quirk)      [1] variance clamped at var_min
 *   [2] variance clamped at var_max                             [3] the weakest of five modes replaced
 *   [4] a fitting mode swapped with an equal weight above it     [5] pixels with five modes after the call
 *   [6] a new mode created (not fitting, alphaT > 0)             [7] pixels marked background */
#include <math.h>
#include <stdint.h>

#define NM 5
typedef struct { float weight, variance; } GMM;
static void swapg(GMM *a, GMM *b) { GMM t = *a; *a = *b; *b = t; }
static void swapf(float *a, float *b) { float t = *a; *a = *b; *b = t; }

void mog2_apply(const uint8_t *img, int npx, GMM *gmm0, float *mean0, uint8_t *used, uint8_t *mask, float alphaT, float prune,
                float Tb, float TB, float Tg, float varInit, float varMin, float varMax, int64_t *stats) {
    int64_t s[8] = {0};
    float alpha1 = 1.f - alphaT;
    for (int x = 0; x < npx; x++) {
        GMM *gmm = gmm0 + x * NM; float *mean = mean0 + x * NM; float data = (float)img[x];
        int background = 0, fits = 0, nmodes = used[x]; float totalWeight = 0.f;
        for (int mode = 0; mode < nmodes; mode++) {
            float weight = alpha1 * gmm[mode].weight + prune; int swap_count = 0;
            if (!fits) {
                float var = gmm[mode].variance;
                float d = mean[mode] - data; float dist2 = d * d;
                if (totalWeight < TB && dist2 < Tb * var) background = 1;
                if (dist2 < Tg * var) {
                    fits = 1; weight += alphaT; float k = alphaT / weight;
                    mean[mode] -= k * d;
                    float varnew = var + k * (dist2 - var);
                    if (!(varnew > varMin)) s[1]++;
                    varnew = varnew > varMin ? varnew : varMin;
                    if (!(varnew < varMax)) s[2]++;
                    varnew = varnew < varMax ? varnew : varMax;
                    gmm[mode].variance = varnew;
                    for (int i = mode; i > 0; i--) {
                        if (weight < gmm[i - 1].weight) break;
                        if (weight == gmm[i - 1].weight) s[4]++;
                        swap_count++; swapg(&gmm[i], &gmm[i - 1]); swapf(&mean[i], &mean[i - 1]);
                    }
                }
            }
            if (weight < -prune) { weight = 0.f; nmodes--; s[0]++; }
            gmm[mode - swap_count].weight = weight;
            totalWeight += weight;
        }
        /* cv2 4.x: no 1/0 when every visited mode was pruned (the scalar form 1.f / totalWeight turns the weights to NaN) */
        float invWeight = 0.f;
        if (fabsf(totalWeight) > 1.1920928955078125e-07f) invWeight = 1.f / totalWeight;
        for (int mode = 0; mode < nmodes; mode++) gmm[mode].weight *= invWeight;
        if (!fits && alphaT > 0.f) {
            s[6]++;
            if (nmodes == NM) s[3]++;
            int mode = nmodes == NM ? NM - 1 : nmodes++;
            if (nmodes == 1) gmm[mode].weight = 1.f;
            else { gmm[mode].weight = alphaT; for (int i = 0; i < nmodes - 1; i++) gmm[i].weight *= alpha1; }
            mean[mode] = data; gmm[mode].variance = varInit;
            for (int i = nmodes - 1; i > 0; i--) {
                if (alphaT < gmm[i - 1].weight) break;
                swapg(&gmm[i], &gmm[i - 1]); swapf(&mean[i], &mean[i - 1]);
            }
        }
        used[x] = (uint8_t)nmodes;
        if (nmodes == NM) s[5]++;
        if (background) s[7]++;
        mask[x] = background ? 0 : 255;
    }
    if (stats)
        for (int i = 0; i < 8; i++) stats[i] += s[i];
}

void mog2_background(int npx, const GMM *gmm0, const float *mean0, const uint8_t *used, float TB, uint8_t *out) {
    for (int x = 0; x < npx; x++) {
        const GMM *gmm = gmm0 + x * NM; const float *mean = mean0 + x * NM;
        float meanVal = 0.f, totalWeight = 0.f;
        for (int g = 0; g < used[x]; g++) {
            meanVal += gmm[g].weight * mean[g]; totalWeight += gmm[g].weight;
            if (totalWeight > TB) break;
        }
        float inv = 0.f;
        if (fabsf(totalWeight) > 1.1920928955078125e-07f) inv = 1.f / totalWeight;
        float v = meanVal * inv; int r = (int)lrintf(v);
        out[x] = (uint8_t)(r < 0 ? 0 : r > 255 ? 255 : r);
    }
}
