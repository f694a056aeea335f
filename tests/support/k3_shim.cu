// K3 (huffman_kernel, csrc/h2j_k_huffman.cuh) on histograms the caller gives, for tests/test_gpu_huffman_k3.py.
// Built at test time as a shared library for sm_100a; the product library is not involved.  TEST INFRASTRUCTURE ONLY.
#include <cstring>
#include <vector>

#include "../../h264-h265-to-jpeg_b200/csrc/h2j_k_huffman.cuh"

using namespace h2j;

// hist: n x 4 x 256 counts (tables DC luma, DC chroma, AC luma, AC chroma; the DC ones may only use symbols 0..15).
// Out, per frame: bits n x 4 x 17, vals n x 4 x 256, nvals n x 4, hcode n x 4 x 256 (FrameTab::hcode as K3 leaves it, the DC
// tables inside hcode[1]), hdr n x hdr_cap header bytes, hdr_bytes n, status n.  Returns 0, or the CUDA error code.
extern "C" int k3_run(int n, const uint32_t *hist, uint8_t *bits, uint8_t *vals, int *nvals, uint32_t *hcode, uint8_t *hdr,
                      int hdr_cap, int *hdr_bytes, int *status)
{
    static const char kComment[] = "k3 shim";
    FrameState *d_state = nullptr;
    FrameTab *d_tabs = nullptr;
    uint8_t *d_out = nullptr;
    char *d_comment = nullptr;
    cudaError_t err = cudaSuccess;
    std::vector<FrameState> st(n);
    std::vector<FrameTab> tabs(n);
    FrameLayout L{};
    L.w = 64;
    L.h = 48;
    L.fmt = kFmt420;
    memset(st.data(), 0, sizeof(FrameState) * n);
    memset(tabs.data(), 0, sizeof(FrameTab) * n);
    for (int f = 0; f < n; f++) {
        memcpy(st[f].hist, hist + (size_t)f * 4 * 256, sizeof st[f].hist);
        for (int i = 0; i < 64; i++) tabs[f].dqt_zz[i] = (uint8_t)(i + 1);
    }
#define K3_TRY(call) do { err = (call); if (err != cudaSuccess) goto done; } while (0)
    K3_TRY(cudaMalloc(&d_state, sizeof(FrameState) * n));
    K3_TRY(cudaMalloc(&d_tabs, sizeof(FrameTab) * n));
    K3_TRY(cudaMalloc(&d_out, (size_t)hdr_cap * n));
    K3_TRY(cudaMalloc(&d_comment, sizeof kComment));
    K3_TRY(cudaMemcpy(d_state, st.data(), sizeof(FrameState) * n, cudaMemcpyHostToDevice));
    K3_TRY(cudaMemcpy(d_tabs, tabs.data(), sizeof(FrameTab) * n, cudaMemcpyHostToDevice));
    K3_TRY(cudaMemset(d_out, 0, (size_t)hdr_cap * n));
    K3_TRY(cudaMemcpy(d_comment, kComment, sizeof kComment, cudaMemcpyHostToDevice));
    huffman_kernel<<<4 * n, kHuffGroup>>>(L, d_tabs, d_state, n, d_out, hdr_cap, hdr_cap, d_comment, (int)strlen(kComment));
    K3_TRY(cudaGetLastError());
    K3_TRY(cudaDeviceSynchronize());
    K3_TRY(cudaMemcpy(tabs.data(), d_tabs, sizeof(FrameTab) * n, cudaMemcpyDeviceToHost));
    K3_TRY(cudaMemcpy(hdr, d_out, (size_t)hdr_cap * n, cudaMemcpyDeviceToHost));
    for (int f = 0; f < n; f++) {
        const FrameTab &T = tabs[f];
        memcpy(bits + (size_t)f * 4 * 17, T.bits, sizeof T.bits);
        memcpy(vals + (size_t)f * 4 * 256, T.vals, sizeof T.vals);
        memcpy(nvals + (size_t)f * 4, T.nvals, sizeof T.nvals);
        memcpy(hcode + (size_t)f * 4 * 256, T.hcode, sizeof T.hcode);
        hdr_bytes[f] = T.header_bytes;
        status[f] = T.status;
    }
done:
#undef K3_TRY
    cudaFree(d_state);
    cudaFree(d_tabs);
    cudaFree(d_out);
    cudaFree(d_comment);
    return (int)err;
}
