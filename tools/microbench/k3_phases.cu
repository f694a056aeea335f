// Where the time of K3 (huffman_kernel) goes for ONE table: cycle stamps of thread 0 around the phases of
// build_one_table on a typical AC-luma histogram (h2j_k_huffman.cuh, H2J_K3_CLOCKS).  Prints microseconds per phase
// and the whole kernel's CUDA-event time for 1 frame (4 CTAs) -- the single-frame call shape.
#define H2J_K3_CLOCKS 1
#include <cstdio>
#include <cstdlib>
#include <vector>

#include "../../h264-h265-to-jpeg_b200/csrc/h2j_kernels.cuh"

using namespace h2j;

int main(int argc, char **argv)
{
    const int nsym = argc > 1 ? atoi(argv[1]) : 60;
    FrameState *st;
    FrameTab *tab;
    uint8_t *out;
    char *comment;
    cudaMalloc(&st, sizeof(FrameState));
    cudaMalloc(&tab, sizeof(FrameTab));
    cudaMalloc(&out, 1 << 20);
    cudaMalloc(&comment, 32);
    FrameState h{};
    // AC tables: geometric counts with ties at the tail (the tie order is what makes the sorts sequential)
    for (int t = 2; t < 4; t++) {
        srand(7 + t);
        for (int i = 0; i < nsym; i++) {
            const int sym = ((i % 11) + 1) | (((i / 11) & 15) << 4);  // (run, size) symbols, up to 176 distinct
            h.hist[t][sym] = 1 + (unsigned)(200000.0 / ((i + 1) * (i + 1))) + (i > 30 ? rand() % 3 : 0);
        }
        h.hist[t][0] = 40000;
        h.hist[t][0xf0] = 3;
    }
    for (int t = 0; t < 2; t++)
        for (int i = 0; i < 9; i++) h.hist[t][i] = 1000 >> i | 1;
    FrameLayout L{};
    L.w = 322; L.h = 242;
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0);
    cudaEventCreate(&e1);
    float best = 1e9f;
    for (int rep = 0; rep < 5; rep++) {
        cudaMemcpy(st, &h, sizeof h, cudaMemcpyHostToDevice);
        cudaEventRecord(e0);
        huffman_kernel<<<4, kHuffGroup>>>(L, tab, st, 1, out, 1 << 20, 1 << 20, comment, 14);
        cudaEventRecord(e1);
        cudaDeviceSynchronize();
        float ms;
        cudaEventElapsedTime(&ms, e0, e1);
        best = ms < best ? ms : best;
    }
    long long c[16];
    cudaMemcpyFromSymbol(c, g_k3_clocks, sizeof c);
    int clk_khz = 0;
    cudaDeviceGetAttribute(&clk_khz, cudaDevAttrClockRate, 0);
    const double us = 1e3 / clk_khz;
    const char *names[] = {"gather used symbols", "sort by count (AV_QSORT replay)", "package-merge, 16 levels", "back-trace + lengths + gather",
                           "sort by length (AV_QSORT replay)", "BITS/HUFFVAL + code table"};
    printf("{\"symbols\": %d, \"kernel_us_1_frame\": %.2f, \"sm_clock_mhz\": %.0f", nsym, best * 1e3, clk_khz / 1e3);
    for (int i = 0; i < 6; i++) printf(", \"%s_us\": %.2f", names[i], (c[i + 1] - c[i]) * us);
    printf(", \"table_total_us\": %.2f, \"rounds_of_the_second_sort\": %lld}\n", (c[6] - c[0]) * us, c[15]);
    cudaError_t err = cudaGetLastError();
    if (err != cudaSuccess) { fprintf(stderr, "%s\n", cudaGetErrorString(err)); return 1; }
    return 0;
}
