// Internal pieces shared by the FFT translation units (fft.cu: power-of-two sizes, fft_mixed.cu: 2^a 3^b 5^c 7^d):
// complex arithmetic, the radix-4 / radix-8 butterflies, the Hermitian split / merge of the packed real <-> complex
// z pass, and the per-device twiddle cache.  Not part of the C ABI.
#pragma once
#include "common.cuh"

template <typename T> struct C2;
template <> struct C2<float> { typedef float2 type; };
template <> struct C2<double> { typedef double2 type; };

template <typename C> __device__ __forceinline__ C cadd(C a, C b) { return C{a.x + b.x, a.y + b.y}; }
template <typename C> __device__ __forceinline__ C csub(C a, C b) { return C{a.x - b.x, a.y - b.y}; }
template <typename C> __device__ __forceinline__ C cmul(C a, C b) {
    return C{a.x * b.x - a.y * b.y, a.x * b.y + a.y * b.x};
}
template <typename C> __device__ __forceinline__ C cconj(C a) { return C{a.x, -a.y}; }
template <typename C> __device__ __forceinline__ C cmuli_neg(C a) { return C{a.y, -a.x}; }  // a * (-i)

template <typename C> struct Sqrt1_2;
template <> struct Sqrt1_2<float2> { static __device__ __forceinline__ float v() { return 0.70710678118654752440f; } };
template <> struct Sqrt1_2<double2> { static __device__ __forceinline__ double v() { return 0.70710678118654752440; } };

// 4-point DFT (forward): X0 = c0+c1, X1 = c2+c3, X2 = c0-c1, X3 = c2-c3
template <typename C>
__device__ __forceinline__ void dft4(C &a0, C &a1, C &a2, C &a3) {
    C c0 = cadd(a0, a2), c1 = cadd(a1, a3), c2 = csub(a0, a2), c3 = cmuli_neg(csub(a1, a3));
    a0 = cadd(c0, c1);
    a1 = cadd(c2, c3);
    a2 = csub(c0, c1);
    a3 = csub(c2, c3);
}

template <typename C>
__device__ __forceinline__ void radix8(C (&a)[8]) {   // in: a[j] = x_j ; out: a[m] = X_m (8-point forward DFT)
    C b0 = cadd(a[0], a[4]), b1 = cadd(a[1], a[5]), b2 = cadd(a[2], a[6]), b3 = cadd(a[3], a[7]);
    C b4 = csub(a[0], a[4]), d5 = csub(a[1], a[5]), d6 = csub(a[2], a[6]), d7 = csub(a[3], a[7]);
    const auto h = Sqrt1_2<C>::v();
    C b5 = C{(d5.x + d5.y) * h, (d5.y - d5.x) * h};
    C b6 = cmuli_neg(d6);
    C b7 = C{(d7.y - d7.x) * h, -(d7.x + d7.y) * h};
    dft4(b0, b1, b2, b3);      // -> X0, X2, X4, X6
    dft4(b4, b5, b6, b7);      // -> X1, X3, X5, X7
    a[0] = b0; a[1] = b4; a[2] = b1; a[3] = b5; a[4] = b2; a[5] = b6; a[6] = b3; a[7] = b7;
}

// Forward z pass, Hermitian split of the packed transform Z = FFT_M(x[2n] + i x[2n+1]), M = Nz/2:
//   X[k] = h [ (Z[k] + conj Z[M-k]) - i W_Nz^k (Z[k] - conj Z[M-k]) ],  zm = conj Z[M-k], w = W_Nz^k, h = scale / 2
template <typename C, typename T>
__device__ __forceinline__ C hermitian_split(C zk, C zm, C w, T h) {
    C e = cadd(zk, zm), o = csub(zk, zm);
    C wo = cmul(w, o);
    return C{(e.x + wo.y) * h, (e.y - wo.x) * h};
}

// Backward z pass, the inverse merge: with xm = conj X[M-k] and w = W_Nz^k, returns conj Z[k] where
//   Z[k] = E + i O,  E = X[k] + conj X[M-k],  O = conj(w) (X[k] - conj X[M-k])
// (the factor 2 of the unnormalised inverse cancels the 1/2 of the split); x[2n] + i x[2n+1] = conj(FFT_M(conj Z))[n]
template <typename C>
__device__ __forceinline__ C hermitian_merge(C xk, C xm, C w) {
    C e = cadd(xk, xm), d = csub(xk, xm);
    C o = cmul(cconj(w), d);
    C z = C{e.x - o.y, e.y + o.x};
    return cconj(z);
}

// tw[k] = exp(-2 pi i k / N), k < N, f8-accurate (sincospi), built once per (device, N, dtype) and kept for the life
// of the process.  dtype NBK_F4 -> float2 table, NBK_F8 -> double2.
int get_twiddle(int N, int dtype, cudaStream_t s, void **out);

// the size rule of the mixed-radix whole-mesh transforms: every side even and 7-smooth, Nx, Ny <= 8192, Nz <= 16384
int nbk_check_mixed_dims(const char *who, int dtype, int64_t Nx, int64_t Ny, int64_t Nz);
