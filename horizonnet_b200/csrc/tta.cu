// Device-side test-time augmentation around the forward (reference inference.py:32-62 augment /
// augment_undo and inference.py:77-93): the flip / horizontal-roll views are built on the device from ONE
// uploaded panorama, and un-flip / un-roll + mean over views + sigmoid(cor) + the boundary -> pixel-row
// conversion with clipping are one kernel, so a TTA inference is 3 launches around hn_model_forward instead
// of numpy work and two device->host round trips per image.  Both kernels take B panoramas at once.  ("next" row f2 of SURVEY.md section 8f.)
#include "hn_common.cuh"

namespace hn {

namespace {

// views[v*B + b][c][h][w] = x[b][c][h][src(w)] (the view-major order of the reference's np.concatenate);
// mode 0: identity, 1: flip (np.flip axis -1), 2: roll by shift (np.roll)
__global__ void tta_views_kernel(const float* __restrict__ x, float* __restrict__ views, int B, int V,
                                 const int* __restrict__ modes, const int* __restrict__ shifts, int H, int W) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const size_t per = (size_t)3 * H * W;
    if (i >= per * V * B) return;
    const int vb = (int)(i / per);
    const int v = vb / B, b = vb - v * B;
    const size_t r = i - (size_t)vb * per;
    const int w = (int)(r % W);
    const size_t row = r / W;                       // c*H + h
    int src = w;
    if (modes[v] == 1) src = W - 1 - w;
    else if (modes[v] == 2) { src = (w - shifts[v]) % W; if (src < 0) src += W; }      // np.roll(x, shift): out[w] = in[w - shift]
    views[i] = __ldg(x + (size_t)b * per + row * W + src);
}

// y_bon_pix[b][s][w] = clip(((mean_v undo(bon[v*B + b][s]))[w] / pi + 0.5) * H - 0.5),
// y_cor[b][w] = mean_v undo(sigmoid(cor[v*B + b]))[w]
__global__ void tta_merge_kernel(const float* __restrict__ bon, const float* __restrict__ cor, int B, int V,
                                 const int* __restrict__ modes, const int* __restrict__ shifts, float* __restrict__ y_bon,
                                 float* __restrict__ y_cor, int H, int W) {
    const int w = blockIdx.x * blockDim.x + threadIdx.x;
    const int b = blockIdx.y;
    if (w >= W) return;
    float sb0 = 0.f, sb1 = 0.f, sc = 0.f;
    for (int v = 0; v < V; ++v) {
        int src = w;
        if (modes[v] == 1) src = W - 1 - w;                                   // undo flip
        else if (modes[v] == 2) { src = (w + shifts[v]) % W; if (src < 0) src += W; }   // np.roll(x, -shift)
        const size_t vb = (size_t)v * B + b;
        sb0 += bon[(vb * 2 + 0) * W + src];
        sb1 += bon[(vb * 2 + 1) * W + src];
        sc += 1.f / (1.f + expf(-cor[vb * W + src]));                  // torch.sigmoid before the undo (inference.py:80)
    }
    const float inv = (float)V;
    const float pi = 3.14159265358979323846f;
    float b0 = (sb0 / inv / pi + 0.5f) * (float)H - 0.5f;                     // inference.py:90
    float b1 = (sb1 / inv / pi + 0.5f) * (float)H - 0.5f;
    b0 = fminf(fmaxf(b0, 1.f), (float)H / 2 - 1);                             // inference.py:91
    b1 = fminf(fmaxf(b1, (float)H / 2 + 1), (float)H - 2);                    // inference.py:92
    y_bon[(size_t)b * 2 * W + w] = b0;
    y_bon[(size_t)b * 2 * W + W + w] = b1;
    y_cor[(size_t)b * W + w] = sc / inv;
}

}  // namespace

int tta_views(const float* x, float* views, int B, int V, const int* modes_dev, const int* shifts_dev, cudaStream_t st) {
    const size_t total = (size_t)B * V * 3 * 512 * 1024;
    tta_views_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(x, views, B, V, modes_dev, shifts_dev, 512, 1024);
    HN_LAUNCH_OK();
    return 0;
}

int tta_merge(const float* bon, const float* cor, int B, int V, const int* modes_dev, const int* shifts_dev, float* y_bon,
              float* y_cor, cudaStream_t st) {
    tta_merge_kernel<<<dim3(4, B), 256, 0, st>>>(bon, cor, B, V, modes_dev, shifts_dev, y_bon, y_cor, 512, 1024);
    HN_LAUNCH_OK();
    return 0;
}

}  // namespace hn
