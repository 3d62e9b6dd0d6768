/* libhorizonnet_b200 -- C ABI of the B200-native HorizonNet hot path.
 *
 * The reference (sunset1995/HorizonNet @ c9a7df9) is pure Python and has no FFI of its own, so this
 * ABI sits *beneath* the two Python entry points it keeps drop-in compatible (see INTEGRATION.md):
 *
 *   model.HorizonNet('resnet50', use_rnn=True).forward(x)        reference model.py:254-281
 *   misc.panostretch.pano_stretch(img, corners, kx, ky, order)   reference misc/panostretch.py:81-117
 *
 * Conventions: plain pointers and sizes only (no torch types); the caller owns every buffer;
 * device entry points are asynchronous on the CUstream/cudaStream_t passed as `void* stream`
 * (NULL = legacy default stream); every function returns 0 on success and a negative value on
 * failure, with the message available from hn_last_error() (thread-local).  A handle is bound to
 * one device and is not thread-safe; use one handle per replica (reference train.py:190-192
 * replicates the module per device).  There is no CPU path: without a CUDA device every compute
 * entry point fails.
 */
#ifndef HORIZONNET_B200_H
#define HORIZONNET_B200_H

#ifdef __cplusplus
extern "C" {
#endif

typedef struct hn_model hn_model;

/* Last error message of the calling thread ("" if none). */
const char* hn_last_error(void);
/* ABI version (bumped on any signature change). */
int hn_abi_version(void);
/* Digest of the sources this binary was built from (horizonnet_b200/build.py embeds it; the Python binding
 * refuses to run a binary whose digest differs from the checked-out sources). */
const char* hn_build_digest(void);
/* Number of kernels this library has launched in this process (bench.py "gpu_launches"). */
long long hn_kernel_launches(void);

/* ---- model.HorizonNet (reference model.py:185-281), resnet50 + bi-LSTM head only ------------- */

/* Creates the model on CUDA device `device`, with activation workspace for up to `max_batch`
 * panoramas per forward.  Replaces HorizonNet.__init__ (model.py:189-246) minus the ImageNet
 * download. */
int hn_model_create(int device, int max_batch, hn_model** out);

/* Number of tensors of the reference checkpoint layout (448, misc/utils.py:49-58) and the i-th key
 * with its element count; lets a binding iterate the state_dict without knowing the topology. */
int hn_model_num_tensors(const hn_model* m);
int hn_model_tensor_info(const hn_model* m, int index, const char** key, long long* numel);

/* Uploads one fp32 tensor of the reference state_dict (same key names and PyTorch layouts:
 * conv OIHW, LSTM [4H, in], linear [out, in]).  `data` may be a host (on_device=0) or a device
 * pointer (on_device=1).  `*.num_batches_tracked` keys are accepted and ignored.
 * Replaces nn.Module.load_state_dict for this module (misc/utils.py:64). */
int hn_model_set_tensor(hn_model* m, const char* key, const float* data, long long numel, int on_device);

/* Folds eval-mode BN / conv bias and re-packs all weights into the kernels' layouts.  Fails if a
 * tensor was never set.  Must be called after the last hn_model_set_tensor and before forward. */
int hn_model_finalize(hn_model* m);

/* HorizonNet.forward (model.py:254-281), eval mode.  x: [batch][in_channels >= 3][512][1024] fp32
 * NCHW in [0,1] on the device (only the first 3 channels are read, model.py:252);
 * bon: [batch][2][1024], cor: [batch][1][1024] fp32 on the device (raw: cor is a logit). */
int hn_model_forward(hn_model* m, const float* x_nchw_dev, int batch, int in_channels,
                     float* bon_dev, float* cor_dev, void* stream);

/* Throughput form of hn_model_forward for streams of batches.  The forward is split over two internal streams:
 * the encoder + height reduction of call i+1 (all 148 SMs, tensor-core bound) run while the bi-LSTM recurrence + head
 * of call i (16-CTA clusters on 64 SMs, latency-bound: 512 dependent steps) are still in flight.  Ordering contract
 * on `stream`: x must be ready in stream order at the call; x may be reused by work enqueued on `stream` after the
 * call returns; bon/cor of call i are complete for work enqueued on `stream` after call i+1 returns, or after
 * hn_model_flush(m, stream).  Results are bit-identical to hn_model_forward.  Keep bon/cor of consecutive calls in
 * distinct buffers. */
int hn_model_forward_async(hn_model* m, const float* x_nchw_dev, int batch, int in_channels,
                           float* bon_dev, float* cor_dev, void* stream);
/* Makes `stream` wait for every forward enqueued so far by hn_model_forward_async. */
int hn_model_flush(hn_model* m, void* stream);

/* TRAIN-mode forward: what `net(x)` computes under `net.train()` (reference train.py:52 inside feed_forward,
 * model.py:254-281 with every nn.BatchNorm2d in training mode and both dropouts active) -- the first step of the
 * "next" row f1; the backward pass is NOT built.
 *   - BatchNorm2d i (i < hn_model_num_bn(m), state_dict prefix hn_model_bn_name(m, i)): bn_train[i] = 1 normalises
 *     with the batch mean / biased variance of the raw conv output and moves running_mean / running_var (the device
 *     copies inside the model, read them back with hn_model_get_tensor) by bn_factor[i] (= the module's momentum, or
 *     1/num_batches_tracked for momentum=None; < 0: track_running_stats off) using the unbiased variance;
 *     bn_train[i] = 0 keeps that module in eval mode (train.py:251-256, --freeze_earlier_blocks).
 *   - rnn_dropout: nn.LSTM(dropout=0.5) between the recurrent layers (model.py:226); head_dropout: self.drop_out
 *     (model.py:228, :265); 0 disables.  Masks are Philox4x32-10 functions of (seed, which, element index):
 *     hn_dropout_mask writes the factors (0 or 1/(1-p)) the forward multiplies with, which = 0 inter-layer
 *     [256][batch][1024], 1 head [256][batch][1024].  torch's own generator stream is not reproduced; for parity
 *     against a torch run, rnn_mask_dev / head_mask_dev (same shapes, or NULL) replace the Philox masks.
 * Each convolution runs twice (statistics pass + real pass); eval-mode entry points called afterwards fold the moved
 * running statistics again on their own. */
int hn_model_num_bn(const hn_model* m);
const char* hn_model_bn_name(const hn_model* m, int i);
int hn_model_forward_train(hn_model* m, const float* x_nchw_dev, int batch, int in_channels, float* bon_dev,
                           float* cor_dev, const unsigned char* bn_train, const double* bn_factor, int n_bn,
                           unsigned long long seed, double rnn_dropout, double head_dropout,
                           const float* rnn_mask_dev, const float* head_mask_dev, void* stream);
int hn_dropout_mask(unsigned long long seed, int which, double p, float* out_dev, long long n, void* stream);
/* Current device copy of a state_dict tensor (e.g. "...bn1.running_mean" after train forwards) -> out
 * (device pointer if on_device, else host; the host form synchronises). */
int hn_model_get_tensor(hn_model* m, const char* key, float* out, long long numel, int on_device, void* stream);

/* Training step (row f1; reference train.py:44-58 feed_forward + :272-281 backward).  hn_train_forward = the train-mode
 * forward above (same arguments) but on exact-fp32 kernels and with a tape: every conv output and activation is kept.
 * hn_train_backward takes d(loss)/d(bon) [batch][2][1024] and d(loss)/d(cor) [batch][1][1024] (device) -- the losses
 * themselves (train.py:53-56: L1 + BCE-with-logits) and the optimizer (train.py:216-223) stay with the caller -- and
 * leaves d(loss)/d(parameter) for every state_dict parameter in the reference's layout (nn.Conv2d OIHW, nn.LSTM
 * [4H][in], ...), read back with hn_model_get_grad (device pointer).  One backward per forward.  First correct path:
 * fp32 CUDA-core kernels; no tensor-core dgrad/wgrad, loss scaling or gradient all-reduce yet. */
int hn_train_forward(hn_model* m, const float* x_nchw_dev, int batch, int in_channels, float* bon_dev, float* cor_dev,
                     const unsigned char* bn_train, const double* bn_factor, int n_bn, unsigned long long seed,
                     double rnn_dropout, double head_dropout, const float* rnn_mask_dev, const float* head_mask_dev,
                     void* stream);
int hn_train_backward(hn_model* m, const float* dbon_dev, const float* dcor_dev, void* stream);
int hn_model_get_grad(hn_model* m, const char* key, float* out_dev, long long numel, void* stream);
/* Device time (ms) of the phases of the last hn_train_backward: head, bi-LSTM BPTT, sequence adjoint, the 69 conv units. */
int hn_train_profile(hn_model* m, double ms[4]);
/* HN_TRAIN_PROF=1 during the last hn_train_backward: the conv-unit phase split into ms[0] BatchNorm backward, ms[1] weight
 * gradients, ms[2] data gradients (device ms, summed over the units); -1 when that backward was not profiled. */
int hn_train_profile_units(hn_model* m, double ms[3]);
/* Tape inspection for tests: conv unit i of the last hn_train_forward (graph order: stem, blocks, height reduction);
 * what = 0 activation, 1 raw conv output, 2 gradient of the activation; halo-1 NHWC copy, dims = {B, H, W, C}. */
int hn_train_debug_unit(hn_model* m, int i, int what, float* out_dev, long long capacity, int dims[4], char* name,
                        int name_cap, void* stream);

/* Same call with HOST buffers: H2D of x, forward, D2H of bon/cor, synchronous.  This is what
 * inference.py:78-79 (`net(x.to(device))` + `.cpu()`) amounts to. */
int hn_model_forward_host(hn_model* m, const float* x_nchw_host, int batch, int in_channels,
                          float* bon_host, float* cor_host);

/* Pipelined form of the host call for streams of batches: hn_model_submit_host enqueues the H2D
 * copy of a batch (pinned memory recommended) on an internal copy stream into one of two input
 * slots, enqueues its forward behind it (two-stream schedule of hn_model_forward_async) and returns;
 * hn_model_collect_host waits for the OLDEST submitted batch, copies bon/cor back and synchronises
 * (a device-side failure of that batch is reported here).  Calling submit(i+1) before collect(i)
 * overlaps the upload and the encoder of the next batch with the forward / recurrence of the current
 * one (at most 2 batches in flight).  Results are identical to hn_model_forward_host. */
int hn_model_submit_host(hn_model* m, const float* x_nchw_host, int batch, int in_channels);
int hn_model_collect_host(hn_model* m, float* bon_host, float* cor_host);

/* Test-time-augmented inference on the device ("next" row f2; reference inference.py:32-62 augment /
 * augment_undo and inference.py:77-93).  x: ONE panorama [3][512][1024] fp32 on the device; views =
 * identity (+ horizontal flip if `flip`) + one np.roll per entry of shifts_host (pixels, as computed by
 * inference.py:40 `int(round(shift_p * W))`).  Outputs on the device: y_bon_pix [2][1024] = boundary rows in
 * pixels, mean over un-augmented views, clipped like inference.py:90-92; y_cor [1024] = mean of the
 * un-augmented sigmoid(cor).  Needs max_batch >= number of views. */
int hn_model_infer_tta(hn_model* m, const float* x_dev, int in_channels, int flip, const int* shifts_host,
                       int n_rotate, float* y_bon_pix_dev, float* y_cor_dev, void* stream);

/* Room-layout post-processing on the device (reference inference.py:21-29 find_N_peaks and :95-139 with the
 * misc/post_proc.py functions they call: floor/ceiling plane, wall-wall peaks, wall fitting, the Polygon validity
 * check with its cuboid fallback, corner assembly).  One CTA per panorama; every input and output is on the device.
 *   y_bon_pix [B][2][1024]  boundary rows in pixels and y_cor [B][1024] corner probabilities, exactly what
 *                           hn_model_infer_tta / hn_model_infer_layout write (inference.py:90-93);
 *   mode                    HN_LAYOUT_GENERAL, HN_LAYOUT_CUBOID (force_cuboid) or HN_LAYOUT_RAW (force_raw);
 *   min_v                   peak threshold (the caller applies the reference's default: 0 cuboid, 0.05 general);
 *   r_px                    peak window int(round(W * r / 2)) (inference.py:108; 26 for the default r = 0.05);
 *   workspace               hn_layout_workspace_bytes(B) bytes of device memory (no allocation inside);
 *   cor_id [B][HN_LAYOUT_MAX_COR][2]  normalised (u, v) corners, n_cor[B] rows valid per panorama;
 *   z1 [B]                  the floor plane (np_refine_by_fix_z, float32);
 *   status [B][4]           {HN_LAYOUT_OK / HN_LAYOUT_ASSERT / HN_LAYOUT_RING, fell back to the cuboid (1/0),
 *                            number of peaks, number of walls}; ASSERT = the reference raises AssertionError
 *                            (gen_ww_cuboid / gen_ww_general / vote asserts), RING = the reference raises ValueError
 *                            (a wall ring shapely cannot build); cor_id is empty for both;
 *   peaks [B][1024], types [B][HN_LAYOUT_MAX_WALLS]  (optional, NULL to skip) the peak columns and wall types
 *                            (0: x = const, 1: y = const) of the final result. */
#define HN_LAYOUT_GENERAL 0
#define HN_LAYOUT_CUBOID 1
#define HN_LAYOUT_RAW 2
#define HN_LAYOUT_OK 0
#define HN_LAYOUT_ASSERT 1
#define HN_LAYOUT_RING 2
#define HN_LAYOUT_MAX_WALLS 2048
#define HN_LAYOUT_MAX_COR 4096
long long hn_layout_workspace_bytes(int batch);
int hn_layout(const float* y_bon_pix_dev, const float* y_cor_dev, int batch, int mode, float min_v, int r_px,
              void* workspace_dev, float* cor_id_dev, int* n_cor_dev, float* z1_dev, int* status_dev, int* peaks_dev,
              int* types_dev, void* stream);

/* Batched test-time augmentation + forward + layout in one call: x [batch][3][512][1024] on the device, views as in
 * hn_model_infer_tta (view-major order v * batch + b, chunked so that chunk * views <= max_batch), the merged
 * signals go to y_bon_pix_dev [batch][2][1024] / y_cor_dev [batch][1024], then hn_layout with the remaining
 * arguments.  With batch 1 the signals are the bits hn_model_infer_tta writes. */
int hn_model_infer_layout(hn_model* m, const float* x_dev, int batch, int flip, const int* shifts_host, int n_rotate,
                          int mode, float min_v, int r_px, void* workspace_dev, float* y_bon_pix_dev, float* y_cor_dev,
                          float* cor_id_dev, int* n_cor_dev, float* z1_dev, int* status_dev, int* peaks_dev,
                          int* types_dev, void* stream);

/* Test hook: copies an intermediate result of the LAST forward, converted to the reference's
 * layout, into `out_dev` (fp32).  Stages: "stem" (conv1+bn1+relu, NCHW [B,64,256,512], model.py:73-75),
 * "layer1".."layer4" (NCHW [B,C,H,W], model.py:78-81),
 * "feature" ([B,1024,256], model.py:175-178), "rnn_out" ([256,B,1024], model.py:264).
 * dims receives the 4 (or 3, last = 0) extents. */
int hn_model_stage(hn_model* m, const char* stage, float* out_dev, long long capacity, int dims[4],
                   void* stream);

/* Options: "tensor_cores" = 1 routes every conv / projection GEMM the tcgen05 kernel supports
 * through the split-fp16 tensor-core path (default), 0 = exact fp32 CUDA-core kernels everywhere;
 * "stem_tc" = 1 (default; env HN_TC_STEM) runs the 7x7 stem on tcgen05 when "tensor_cores" is on, 0 = fp32 CUDA-core stem;
 * "fuse_bottleneck" = 1 (default; env HN_TC_FUSE) runs conv2 + conv3 of the layer1 bottlenecks as one kernel (bit-identical results);
 * "profile" = 1 turns on per-launch CUDA-event timing (see hn_model_profile_read). */
int hn_model_set_option(hn_model* m, const char* name, int value);

/* With option "profile" = 1 every forward records CUDA-event pairs (on the forward's stream)
 * around each launch; this call waits for them and returns, per op class
 * {0 stem, 1 maxpool, 2 encoder convs, 3 height-reduction convs, 4 upsample/concat tail,
 *  5 LSTM input-projection GEMMs, 6 LSTM recurrence, 7 linear head},
 * the accumulated device milliseconds, algorithmic FLOPs and launch counts (arrays of 8). */
int hn_model_profile_read(hn_model* m, double* ms, double* flops, long long* launches, int reset);

/* Synchronises the device and reports device-side failures recorded by earlier asynchronous
 * forwards (e.g. the persistent LSTM kernel's peer-wait timeout). */
int hn_model_check(hn_model* m);

void hn_model_destroy(hn_model* m);

/* ---- misc.panostretch.pano_stretch, image part (reference misc/panostretch.py:81-102) -------- */

/* n images [h][w][c] fp32 (HWC, c in 1..4) on the device, one (kx[i], ky[i]) pair per image
 * (host arrays of n doubles); order 0 (nearest) or 1 (bilinear); scipy legacy 'wrap' semantics. */
int hn_pano_stretch(const float* img_dev, float* out_dev, int n, int h, int w, int c,
                    const double* kx_host, const double* ky_host, int order, void* stream);
/* Same with host images (H2D + kernel + D2H inside), i.e. the numpy-in / numpy-out call of
 * dataset.py:82. */
int hn_pano_stretch_host(const float* img_host, float* out_host, int n, int h, int w, int c,
                         const double* kx_host, const double* ky_host, int order);

/* float64 images (the reference's own CLI feeds float64 0-255, misc/panostretch.py:171): taps, blend and result in double,
 * like scipy returns for a float64 input. */
int hn_pano_stretch_f64(const double* img_dev, double* out_dev, int n, int h, int w, int c,
                        const double* kx_host, const double* ky_host, int order, void* stream);
int hn_pano_stretch_host_f64(const double* img_host, double* out_host, int n, int h, int w, int c,
                             const double* kx_host, const double* ky_host, int order);

/* ---- dataset.PanoCorBonDataset.__getitem__, image path (reference dataset.py:53, 69-105, 124) ------
 *
 * One fused gather pass per image:  uint8 HWC / 255 -> pano_stretch(kx, ky) -> flip -> roll(dx) -> ** gamma -> CHW:
 * n uint8 images [h][w][3] on the device -> n float32 images [3][h][w] on the device (the network input layout,
 * dataset.py:124).  Host arrays of n entries: kx/ky (dataset.py:71-82; NULL or <= 0: no stretch for that image),
 * flip (dataset.py:88-91; NULL: none), dx (np.roll shift, dataset.py:95-98, 0 <= dx < w; NULL: 0),
 * gamma (exponent p of dataset.py:102-105; NULL or <= 0: none).  The random draws and the corner / boundary label
 * bookkeeping stay with the caller (horizonnet_b200/dataset.py mirrors them). */
int hn_augment(const unsigned char* img_u8_dev, float* out_chw_dev, int n, int h, int w,
               const double* kx_host, const double* ky_host, const int* flip_host, const int* dx_host,
               const float* gamma_host, void* stream);

/* ---- misc.pano_lsd_align.rotatePanorama (reference misc/pano_lsd_align.py:125-171, warpImageFast :101-122) ----
 *
 * n images [h][w][c] on the device, float32 (in_is_f64 = 0) or float64 (1) -> n float64 images [h][w][c] rotated by
 * R; rinv_host = 9 doubles, row-major inverse of the reference's R (= vp.T when called with a vanishing-point
 * matrix, pano_lsd_align.py:143).  w must be even (the reference's padding rule, :160-163). */
int hn_rotate_panorama(const void* img_dev, int in_is_f64, double* out_dev, int n, int h, int w, int c,
                       const double* rinv_host, void* stream);

/* ---- kernel-level entry points (unit tests; halo-NHWC activations, see DESIGN.md) ------------ */

/* One convolution + folded BN/bias + optional residual + optional ReLU.
 * in:  [B][H][W + 2*in_halo][Cin]   out: [B][Ho][Wo + 2*out_halo][Cout]   (fp32, device)
 * w_packed: [kh*kw*Cin][Cout], k = (dy*kw + dx)*Cin + c;  scale/shift: [Cout];
 * ph = zero padding along H, pw = circular padding along W (<= in_halo).
 * impl: 0 = exact fp32 CUDA-core kernel, 1 = split-fp16 tcgen05 tensor-core kernel. */
int hn_conv2d(const float* in_dev, int B, int H, int W, int Cin, int in_halo,
              const float* w_packed_dev, const float* scale_dev, const float* shift_dev,
              const float* residual_dev, int Cout, int kh, int kw, int sh, int sw, int ph, int pw,
              int relu, float* out_dev, int out_halo, int impl, void* stream);
/* Backward building blocks of the training step, for unit tests against torch.autograd (train_step.cu):
 * weight + data gradient of one convolution (dz: halo-1 NHWC with circular halo columns; din may be NULL),
 * BatchNorm2d (+identity, ReLU) forward+backward (bn_scratch: 4*C floats, sums: 3*C doubles, C a multiple of 4), and one
 * bidirectional LSTM layer's gate gradients. */
int hn_conv2d_backward(const float* in, int B, int H, int W, int Cin, int in_halo, const float* w_oihw, const float* dz,
                       int Cout, int kh, int kw, int sh, int sw, int ph, int pw, float* din, float* dw_oihw, void* stream);
/* The weight gradient alone on the tcgen05 kernel (wgrad_tc.cu; in / dz: halo-1 NHWC fp32, Cin and Cout multiples of 64,
 * strides 1 or 2): the planes are made inside.  Returns -1 for a shape that kernel does not take. */
int hn_conv2d_wgrad_tc(const float* in, int B, int H, int W, int Cin, const float* dz, int Cout, int kh, int kw, int sh,
                       int sw, int ph, int pw, float* dw_oihw, void* stream);
/* Host-side plan of that kernel for one shape (no GPU work; sms = SM count to plan for): plan[10] = tile columns, rows per
 * tile, tiles per row, box rows, images per tile, pixel tiles (64 pixels each), tiles per slice, slices, work items per slice,
 * CTAs.  -1 for a shape the kernel does not take. */
int hn_wgrad_tc_plan(int B, int H, int W, int Cin, int Cout, int kh, int kw, int sh, int sw, int ph, int pw, int sms, int plan[10]);
int hn_wgrad_tc_enabled(void);   /* 1: the training step uses that kernel where it applies (env HN_WGRAD_TC=0/1 overrides the default) */
int hn_bn_forward_backward(const float* z, int B, int H, int W, int C, const float* gamma, const float* beta,
                           float* running_mean, float* running_var, double factor, int train, int relu, const float* res,
                           float* y, const float* dy, float* dz, float* dres, float* dgamma, float* dbeta, float* bn_scratch,
                           double* sums, void* stream);
int hn_lstm_layer_backward(const float* xp, const float* hout, const float* whf, const float* whb, const float* dout, int T,
                           int B, float* dgates, float* scratch, void* stream);

/* One bidirectional LSTM layer recurrence: xproj [T][B][4096] (input projection + both biases,
 * column = dir*2048 + gate*512 + unit), w_hh_* [2048][512] (PyTorch layout), out [T][B][1024]. */
int hn_lstm_layer(const float* xproj_dev, const float* w_hh_fwd_dev, const float* w_hh_bwd_dev,
                  float* out_dev, int T, int B, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* HORIZONNET_B200_H */
