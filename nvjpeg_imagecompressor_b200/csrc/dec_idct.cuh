// dec_idct.cuh -- the islow 1-D inverse DCT (jidctint.c jpeg_idct_islow), shared by k_idct and k_idct_scaled
#pragma once

namespace b2j {

#define FIX_0_298631336 2446
#define FIX_0_390180644 3196
#define FIX_0_541196100 4433
#define FIX_0_765366865 6270
#define FIX_0_899976223 7373
#define FIX_1_175875602 9633
#define FIX_1_501321110 12299
#define FIX_1_847759065 15137
#define FIX_1_961570560 16069
#define FIX_2_053119869 16819
#define FIX_2_562915447 20995
#define FIX_3_072711026 25172

template <int SH>
__device__ __forceinline__ void idct8(int &i0, int &i1, int &i2, int &i3, int &i4, int &i5, int &i6, int &i7) {
    constexpr int RND = 1 << (SH - 1);
    int z1 = (i2 + i6) * FIX_0_541196100;
    const int t2 = z1 - i6 * FIX_1_847759065, t3 = z1 + i2 * FIX_0_765366865;
    const int t0 = (i0 + i4) << 13, t1 = (i0 - i4) << 13;
    const int t10 = t0 + t3, t13 = t0 - t3, t11 = t1 + t2, t12 = t1 - t2;
    int a0 = i7, a1 = i5, a2 = i3, a3 = i1;
    z1 = a0 + a3;
    int z2 = a1 + a2, z3 = a0 + a2, z4 = a1 + a3;
    const int z5 = (z3 + z4) * FIX_1_175875602;
    a0 *= FIX_0_298631336; a1 *= FIX_2_053119869; a2 *= FIX_3_072711026; a3 *= FIX_1_501321110;
    z1 *= -FIX_0_899976223; z2 *= -FIX_2_562915447;
    z3 = z3 * (-FIX_1_961570560) + z5;
    z4 = z4 * (-FIX_0_390180644) + z5;
    a0 += z1 + z3; a1 += z2 + z4; a2 += z2 + z3; a3 += z1 + z4;
    i0 = (t10 + a3 + RND) >> SH; i7 = (t10 - a3 + RND) >> SH;
    i1 = (t11 + a2 + RND) >> SH; i6 = (t11 - a2 + RND) >> SH;
    i2 = (t12 + a1 + RND) >> SH; i5 = (t12 - a1 + RND) >> SH;
    i3 = (t13 + a0 + RND) >> SH; i4 = (t13 - a0 + RND) >> SH;
}

}  // namespace b2j
