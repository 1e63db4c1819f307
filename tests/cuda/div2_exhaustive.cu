// Exhaustive check of exact_math.cuh's div_const2 against IEEE division (__fdiv_rn): for every divisor on the command
// line and ALL 2^32 f32 dividends, whenever the acceptance rule (min|a| >= 2^-96, max|a| <= 2^96) holds its result must be
// bit-identical (NaNs compared as NaNs).  zh = RN(1/b), zl = RN(1/b - zh) in double, as the engine forms them.
// Prints "divisor mismatches flagged".
#include <cstdio>
#include <cstdlib>

#include "../../dsp_stuff_b200/csrc/exact_math.cuh"

__global__ void check(float b, float zh, float zl, unsigned long long* mism, unsigned long long* flagged) {
    unsigned long long base = ((unsigned long long)blockIdx.x * blockDim.x + threadIdx.x) * 256ull;
    unsigned long long m = 0, f = 0;
    for (int k = 0; k < 256; k++) {
        const float a = __uint_as_float((unsigned)(base + k));
        float mn = dspb::kDiv2Hi, mx = 0.0f;
        const float q = dspb::div_const2(a, dspb::ConstDiv2{zh, zl}, mn, mx);
        const float ref = __fdiv_rn(a, b);
        if (!dspb::div_const2_accept(mn, mx)) f++;
        else if (__float_as_uint(q) != __float_as_uint(ref) && !(q != q && ref != ref)) m++;
    }
    if (m) atomicAdd(mism, m);
    if (f) atomicAdd(flagged, f);
}

int main(int argc, char** argv) {
    unsigned long long *d, h[2];
    if (cudaMalloc(&d, 16) != cudaSuccess) { printf("cuda error\n"); return 2; }
    int rc = 0;
    for (int i = 1; i < argc; i++) {
        const float b = strtof(argv[i], nullptr);
        const float zh = 1.0f / b;
        const float zl = (float)(1.0 / (double)b - (double)zh);
        cudaMemset(d, 0, 16);
        check<<<65536, 256>>>(b, zh, zl, d, d + 1);
        if (cudaDeviceSynchronize() != cudaSuccess) { printf("cuda error\n"); return 2; }
        cudaMemcpy(h, d, 16, cudaMemcpyDeviceToHost);
        printf("%.9g %llu %llu\n", b, h[0], h[1]);
        if (h[0]) rc = 1;
    }
    return rc;
}
