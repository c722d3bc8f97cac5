// Micro-benchmark (tooling, not product): FP32 issue rates on sm_100a that decide the
// channelizer's inner-loop shape: scalar FMUL+FADD vs FFMA vs packed f32x2 (FMUL2/FADD2/FFMA2),
// with register, shared-broadcast and __constant__ second operands.
//
// Modes 0-23 are one row per thread.  Mode x2 is NOT exact: ptxas 12.9 contracts its FMUL2 feeding
// FADD2 into FFMA2 even under -fmad=false (SASS: FMUL2 + FFMA2 + FADD2), which skips a product rounding.
// Modes 30-33 (kx) are the exact candidates for k_channelize<IN_U8IQ> with its operand pattern: a
// warp-uniform shared-memory table, 2 output rows per thread, 8 channels, tap after tap.
#include <cstdio>
#include <cuda_runtime.h>
#define CK(x) do{cudaError_t e=(x); if(e!=cudaSuccess){printf("ERR %s line %d\n",cudaGetErrorString(e),__LINE__);return 1;}}while(0)

__constant__ float4 cw[256];

template<int MODE> __global__ void __launch_bounds__(256) k(float *out, const float4 *gw, int iters)
{
    __shared__ float4 sw[256];
    sw[threadIdx.x] = gw[threadIdx.x];
    __syncthreads();
    float x = threadIdx.x * 0.001f + 1.0f, y = 0.5f + blockIdx.x * 1e-3f;
    float2 acc[8];
    #pragma unroll
    for (int c = 0; c < 8; c++) acc[c] = make_float2(0.f, 0.f);
    for (int it = 0; it < iters; it++) {
        #pragma unroll 8
        for (int j = 0; j < 32; j++) {
            float a = x + j, b = y - j;   // stand-in for the converted sample
            #pragma unroll
            for (int c = 0; c < 8; c++) {
                float4 w;
                if (MODE >= 10 && MODE < 20) w = sw[(j * 8 + c) & 255];
                else if (MODE >= 20) w = cw[(j * 8 + c) & 255];
                else w = make_float4(x + c, y + c, -(y + c), x + c);
                int m = MODE % 10;
                if (m == 0) {        // exact scalar: 4 FMUL + 4 FADD
                    float pr = __fadd_rn(__fmul_rn(a, w.x), __fmul_rn(b, w.z));
                    float pi = __fadd_rn(__fmul_rn(a, w.y), __fmul_rn(b, w.w));
                    acc[c].x = __fadd_rn(acc[c].x, pr);
                    acc[c].y = __fadd_rn(acc[c].y, pi);
                } else if (m == 1) { // scalar FFMA: 4 FFMA
                    acc[c].x = fmaf(a, w.x, acc[c].x); acc[c].x = fmaf(b, w.z, acc[c].x);
                    acc[c].y = fmaf(a, w.y, acc[c].y); acc[c].y = fmaf(b, w.w, acc[c].y);
                } else if (m == 2) { // packed 2 FMUL2 + 2 FADD2, contracted by ptxas (not exact)
                    float2 p1 = __fmul2_rn(make_float2(a, a), make_float2(w.x, w.y));
                    float2 p2 = __fmul2_rn(make_float2(b, b), make_float2(w.z, w.w));
                    acc[c] = __fadd2_rn(acc[c], __fadd2_rn(p1, p2));
                } else if (m == 3) { // packed FFMA2: 2
                    acc[c] = __ffma2_rn(make_float2(a, a), make_float2(w.x, w.y), acc[c]);
                    acc[c] = __ffma2_rn(make_float2(b, b), make_float2(w.z, w.w), acc[c]);
                } else if (m == 4) { // exact, FMUL2 for products, scalar adds
                    float2 p1 = __fmul2_rn(make_float2(a, a), make_float2(w.x, w.y));
                    float2 p2 = __fmul2_rn(make_float2(b, b), make_float2(w.z, w.w));
                    acc[c].x = __fadd_rn(acc[c].x, __fadd_rn(p1.x, p2.x));
                    acc[c].y = __fadd_rn(acc[c].y, __fadd_rn(p1.y, p2.y));
                }
            }
        }
        x += 1e-7f;
    }
    float s = 0;
    #pragma unroll
    for (int c = 0; c < 8; c++) s += acc[c].x + acc[c].y;
    out[blockIdx.x * blockDim.x + threadIdx.x] = s;
}

// Exact shapes, 2 rows per thread (A, B) x 8 channels per tap; the table is 32 taps x 8 channels.
//   30: 2 FMUL2 + 2 FADD + 1 FADD2 per complex MAC, float4 (c, d, -d, c) entries (k_channelize before r3)
//   31: scalar 4 FMUL + 4 FADD, float4 entries
//   32: (c, d)-paired 2 FFMA2(x, w, -0) + 2 FADD2, float4 entries
//   33: row-packed 4 FFMA2(x, w, -0) + 4 FADD2 per two complex MACs, float2 (c, d) entries, two channels per LDS.128
// nz is -0.0f passed at run time: with a literal -0 ptxas rewrites FFMA2(x, w, -0) into FMUL2 and contracts again.
template<int MODE> __global__ void __launch_bounds__(128) kx(float *out, const float4 *gw, int iters, float nz)
{
    __shared__ float4 sw[256];
    for (int i = threadIdx.x; i < 256; i += blockDim.x) sw[i] = gw[i];
    __syncthreads();
    const float xa = threadIdx.x * 0.001f + 1.0f, xb = threadIdx.x * 0.002f + 2.0f;
    const float ya = 0.5f + blockIdx.x * 1e-3f, yb = 0.25f + blockIdx.x * 1e-3f;
    float2 p[8], q[8];                       // 30-32: p = row A (re, im), q = row B; 33: p = re (A, B), q = im (A, B)
    #pragma unroll
    for (int c = 0; c < 8; c++) p[c] = q[c] = make_float2(0.f, 0.f);
    const float2 z = make_float2(nz, nz);
    for (int it = 0; it < iters; it++) {
        #pragma unroll 4
        for (int j = 0; j < 32; j++) {
            const float fj = (float)j;
            const float aA = __fadd_rn(xa, fj), bA = __fadd_rn(ya, -fj), aB = __fadd_rn(xb, fj), bB = __fadd_rn(yb, -fj);
            if (MODE == 33) {
                const float2 re = make_float2(aA, aB), im = make_float2(bA, bB);
                const float4 *wj = reinterpret_cast<const float4 *>(sw) + j * 4;
                #pragma unroll
                for (int c = 0; c < 8; c++) {
                    const float4 w4 = wj[c / 2];
                    const float wc = c & 1 ? w4.z : w4.x, wd = c & 1 ? w4.w : w4.y;
                    const float2 cc = make_float2(wc, wc), dd = make_float2(wd, wd);
                    const float2 ac = __ffma2_rn(re, cc, z), bd = __ffma2_rn(im, dd, z);
                    const float2 ad = __ffma2_rn(re, dd, z), bc = __ffma2_rn(im, cc, z);
                    p[c] = __fadd2_rn(p[c], __fadd2_rn(ac, make_float2(-bd.x, -bd.y)));
                    q[c] = __fadd2_rn(q[c], __fadd2_rn(ad, bc));
                }
            } else {
                #pragma unroll
                for (int c = 0; c < 8; c++) {
                    const float4 w = sw[j * 8 + c];
                    #pragma unroll
                    for (int r = 0; r < 2; r++) {
                        float2 &acc = r ? q[c] : p[c];
                        const float a = r ? aB : aA, b = r ? bB : bA;
                        if (MODE == 30) {
                            const float2 p1 = __fmul2_rn(make_float2(a, a), make_float2(w.x, w.y));
                            const float2 p2 = __fmul2_rn(make_float2(b, b), make_float2(w.z, w.w));
                            acc = __fadd2_rn(acc, make_float2(__fadd_rn(p1.x, p2.x), __fadd_rn(p1.y, p2.y)));
                        } else if (MODE == 31) {
                            acc.x = __fadd_rn(acc.x, __fadd_rn(__fmul_rn(a, w.x), __fmul_rn(b, w.z)));
                            acc.y = __fadd_rn(acc.y, __fadd_rn(__fmul_rn(a, w.y), __fmul_rn(b, w.w)));
                        } else {
                            const float2 p1 = __ffma2_rn(make_float2(a, a), make_float2(w.x, w.y), z);
                            const float2 p2 = __ffma2_rn(make_float2(b, b), make_float2(w.z, w.w), z);
                            acc = __fadd2_rn(acc, __fadd2_rn(p1, p2));
                        }
                    }
                }
            }
        }
    }
    float s = 0;
    #pragma unroll
    for (int c = 0; c < 8; c++) s += p[c].x + p[c].y + q[c].x + q[c].y;
    out[blockIdx.x * blockDim.x + threadIdx.x] = s;
}

template<int MODE> int runx(const char *name, float *out, float4 *gw, int blocks)
{
    int iters = 200;
    cudaEvent_t e0, e1; cudaEventCreate(&e0); cudaEventCreate(&e1);
    kx<MODE><<<blocks, 128>>>(out, gw, 10, -0.0f);
    CK(cudaDeviceSynchronize());
    float best = 1e9;
    for (int r = 0; r < 5; r++) {
        cudaEventRecord(e0);
        kx<MODE><<<blocks, 128>>>(out, gw, iters, -0.0f);
        cudaEventRecord(e1);
        CK(cudaEventSynchronize(e1));
        float ms; cudaEventElapsedTime(&ms, e0, e1);
        if (ms < best) best = ms;
    }
    double macs = (double)blocks * 128 * iters * 32 * 8 * 2;   // complex MACs: 2 rows x 8 channels per tap
    printf("%-34s %8.3f ms  %8.1f G complex-MAC/s  (%.1f per clk per SM @1.9GHz)\n", name, best, macs / best * 1e-6,
           macs / best * 1e-6 / 148 / 1.9);
    return 0;
}

template<int MODE> int run(const char *name, float *out, float4 *gw, int blocks)
{
    int iters = 200;
    cudaEvent_t e0, e1; cudaEventCreate(&e0); cudaEventCreate(&e1);
    k<MODE><<<blocks, 256>>>(out, gw, 10);
    CK(cudaDeviceSynchronize());
    float best = 1e9;
    for (int r = 0; r < 5; r++) {
        cudaEventRecord(e0);
        k<MODE><<<blocks, 256>>>(out, gw, iters);
        cudaEventRecord(e1);
        CK(cudaEventSynchronize(e1));
        float ms; cudaEventElapsedTime(&ms, e0, e1);
        if (ms < best) best = ms;
    }
    double macs = (double)blocks * 256 * iters * 32 * 8;   // complex MACs
    printf("%-34s %8.3f ms  %8.1f G complex-MAC/s  (%.1f per clk per SM @1.9GHz)\n", name, best, macs / best * 1e-6,
           macs / best * 1e-6 / 148 / 1.9);
    return 0;
}

int main()
{
    float *out; float4 *gw; float4 h[256];
    for (int i = 0; i < 256; i++) h[i] = make_float4(1.f + i * 1e-3f, 0.5f, -0.5f, 1.f + i * 1e-3f);
    CK(cudaMalloc(&out, 148 * 16 * 256 * 4)); CK(cudaMalloc(&gw, sizeof(h)));
    CK(cudaMemcpy(gw, h, sizeof(h), cudaMemcpyHostToDevice));
    CK(cudaMemcpyToSymbol(cw, h, sizeof(h)));
    int blocks = 148 * 8;
    run<0>("reg  exact scalar 4FMUL+4FADD", out, gw, blocks);
    run<1>("reg  scalar 4FFMA", out, gw, blocks);
    run<2>("reg  contracted 2FMUL2+2FADD2", out, gw, blocks);
    run<3>("reg  packed 2FFMA2", out, gw, blocks);
    run<4>("reg  exact 2FMUL2+4FADD", out, gw, blocks);
    run<10>("smem exact scalar", out, gw, blocks);
    run<11>("smem scalar FFMA", out, gw, blocks);
    run<12>("smem contracted packed", out, gw, blocks);
    run<13>("smem packed FFMA2", out, gw, blocks);
    run<20>("cmem exact scalar", out, gw, blocks);
    run<21>("cmem scalar FFMA", out, gw, blocks);
    run<22>("cmem contracted packed", out, gw, blocks);
    run<23>("cmem packed FFMA2", out, gw, blocks);
    // 16 CTAs of 128 threads per SM
    const int xblocks = 148 * 16;
    runx<30>("2row exact 2FMUL2+2FADD+FADD2", out, gw, xblocks);
    runx<31>("2row exact scalar 4FMUL+4FADD", out, gw, xblocks);
    runx<32>("2row exact (c,d) 2FFMA2+2FADD2", out, gw, xblocks);
    runx<33>("2row exact row-packed 4FFMA2+4FADD2", out, gw, xblocks);
    return 0;
}
