/* Per-site rescaling shared by every kernel family: exponents are counted in units of 2^256. */
#pragma once
#define PLF_SCALE_BITS 256
#define PLF_TWO_P256 1.157920892373162e+77      /* 2^256  */
#define PLF_TWO_M256 8.636168555094445e-78      /* 2^-256 */

/* number of 2^256 up-scalings applied so that max(v) >= 2^-256 (v >= 0) */
__device__ __forceinline__ int f4_rescale_up(double v[4])
{
    /* non-negative doubles order like their high words */
    int h = max(max(__double2hiint(v[0]), __double2hiint(v[1])), max(__double2hiint(v[2]), __double2hiint(v[3])));
    int s = 0;
    if (h < 0x2FF00000) {          /* high word of 2^-256 */
        double m = fmax(fmax(v[0], v[1]), fmax(v[2], v[3]));
        while (m > 0.0 && m < PLF_TWO_M256 && s < 3) {
#pragma unroll
            for (int i = 0; i < 4; i++) v[i] *= PLF_TWO_P256;
            m *= PLF_TWO_P256;
            s++;
        }
    }
    return s;
}
