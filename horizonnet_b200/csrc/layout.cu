// Room-layout post-processing on the device (reference inference.py:21-29 find_N_peaks and :95-139, with the
// misc/post_proc.py functions they call).  One CTA of 1024 threads per panorama, one thread per column:
//   plane     np_refine_by_fix_z / mean_percentile in float32 (bitonic sort of the 1024 per-column heights)
//   peaks     maximum_filter(size=r, mode='wrap') == signal, signal > float32(min_v), optional top 4
//   walls     per segment between peaks and per axis, `vote` as "widest window of the sorted segment whose spread
//             is within tol, leftmost first" (each sorted position binary-searches its window end), then the
//             sequential gen_ww_cuboid / gen_ww_general logic on one thread
//   validity  Polygon(xy2d).is_valid as an exact simple-ring test; an invalid ring falls back to the cuboid
//   corners   np_xy2coor, roll by -2*argmin, infer_coory, normalised cor_id
// Exceptions the reference raises become a per-panorama status (HN_LAYOUT_ASSERT / HN_LAYOUT_RING), never a silent
// result.
#include "hn_common.cuh"

namespace hn {

namespace {

constexpr int W = 1024;
constexpr int MAXW = 2 * W;            // walls: every peak adds at most one forced wall (gen_ww_general)
constexpr double PI = 3.14159265358979323846;

enum { ST_OK = 0, ST_ASSERT = 1, ST_RING = 2 };

struct LayoutWs {                      // per-panorama scratch in the caller's workspace
    double val[MAXW], score[MAXW], u0[MAXW], u1[MAXW];
    int type[MAXW], gpid[MAXW], tbd[MAXW];
    double seg_val[2][W], seg_score[2][W], seg_l1[2][W], seg_mean[2][W];
    double corx[MAXW], cory[MAXW];
    float ringx[MAXW], ringy[MAXW];
};

struct Smem {
    float yb0[W], ycor[W], zs[W];
    double xy[2][W];
    double sv[W];
    int sseg[W];
    int wv[W];
    int peaks[W];
    double redd[32];
    int redi[32];
    int K, nw, status, invalid, nring;
};

__device__ __forceinline__ double coorx2u(double x) { return ((x + 0.5) / W - 0.5) * 2 * PI; }      // post_proc.py:22-23
__device__ __forceinline__ double coory2v(double y) { return -((y + 0.5) / 512 - 0.5) * PI; }        // :26-27

__device__ double x_u_solve_y(double x, double u) {                                                  // :43-45
    const double c = (x - 512.0 + 0.5) / sin(u);
    return -c * cos(u) + 256.0 - 0.5;
}
__device__ double y_u_solve_x(double y, double u) {                                                  // :48-50
    const double c = -(y - 256.0 + 0.5) / cos(u);
    return c * sin(u) + 512.0 - 0.5;
}

__device__ double block_sum(double v, Smem& s) {
    for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    __syncthreads();
    if ((threadIdx.x & 31) == 0) s.redd[threadIdx.x >> 5] = v;
    __syncthreads();
    double t = 0.0;
    for (int i = 0; i < 32; ++i) t += s.redd[i];
    __syncthreads();
    return t;
}

__device__ int block_count(int pred, Smem& s) {
    const int c = __popc(__ballot_sync(0xffffffffu, pred));
    __syncthreads();
    if ((threadIdx.x & 31) == 0) s.redi[threadIdx.x >> 5] = c;
    __syncthreads();
    int t = 0;
    for (int i = 0; i < 32; ++i) t += s.redi[i];
    __syncthreads();
    return t;
}

// sign of a*b - c*d, exact in sign (Kahan's fma form has a relative error below 2 ulp)
__device__ __forceinline__ int sign_ab_cd(double a, double b, double c, double d) {
    const double w = c * d;
    const double e = fma(-c, d, w);
    const double f = fma(a, b, -w);
    const double r = f + e;
    return (r > 0) - (r < 0);
}
__device__ __forceinline__ int orient(float ax, float ay, float bx, float by, float cx, float cy) {
    return sign_ab_cd((double)bx - ax, (double)cy - ay, (double)by - ay, (double)cx - ax);
}
__device__ __forceinline__ bool on_box(float ax, float ay, float bx, float by, float px, float py) {
    return fminf(ax, bx) <= px && px <= fmaxf(ax, bx) && fminf(ay, by) <= py && py <= fmaxf(ay, by);
}

// Peaks, per-segment votes and the wall list for one peak setting; returns with s.status / s.K / s.nw set.
__device__ void walls_pass(Smem& s, LayoutWs* ws, int r, float min_v, bool top4, bool cuboid, float tol) {
    const int t = threadIdx.x;
    // ---- find_N_peaks (inference.py:21-29): window [t - r/2, t - r/2 + r - 1], wrap
    float m = -INFINITY;
    const int lo = t - r / 2;
    for (int k = 0; k < r; ++k) {
        int c = (lo + k) % W;
        if (c < 0) c += W;
        m = fmaxf(m, s.ycor[c]);
    }
    const int is_pk = (s.ycor[t] == m) && (s.ycor[t] > min_v);
    {
        const unsigned bal = __ballot_sync(0xffffffffu, is_pk);
        if ((t & 31) == 0) s.redi[t >> 5] = __popc(bal);
        __syncthreads();
        int off = 0;
        for (int i = 0; i < (t >> 5); ++i) off += s.redi[i];
        if (is_pk) s.peaks[off + __popc(bal & ((1u << (t & 31)) - 1u))] = t;
        if (t == 31) {
            int tot = 0;
            for (int i = 0; i < 32; ++i) tot += s.redi[i];
            s.K = tot;
        }
        __syncthreads();
    }
    if (top4 && t == 0 && s.K > 4) {      // top 4 by value (ties: lower column), re-sorted by column
        int sel[4];
        for (int q = 0; q < 4; ++q) {
            int best = -1;
            for (int i = 0; i < s.K; ++i) {
                const int c = s.peaks[i];
                bool used = false;
                for (int u = 0; u < q; ++u) used |= sel[u] == c;
                if (!used && (best < 0 || s.ycor[c] > s.ycor[best])) best = c;
            }
            sel[q] = best;
        }
        for (int a = 0; a < 4; ++a)
            for (int b = a + 1; b < 4; ++b)
                if (sel[b] < sel[a]) { const int x = sel[a]; sel[a] = sel[b]; sel[b] = x; }
        for (int q = 0; q < 4; ++q) s.peaks[q] = sel[q];
        s.K = 4;
    }
    __syncthreads();
    const int K = s.K;
    if ((cuboid && K != 4) || K == 0) {   // gen_ww_cuboid :207 / gen_ww_general :243 asserts
        if (t == 0) { s.status = ST_ASSERT; s.nw = 0; }
        __syncthreads();
        return;
    }
    // ---- get_gpid (post_proc.py:134-139): segment j >= 1 = [p[j-1], p[j]), segment 0 = the rest (wrapping)
    int g;
    {
        int lo2 = 0, hi2 = K;                         // number of peaks <= t
        while (lo2 < hi2) { const int mid = (lo2 + hi2) >> 1; if (s.peaks[mid] <= t) lo2 = mid + 1; else hi2 = mid; }
        g = lo2 == K ? 0 : lo2;
    }
    const int size0 = W - s.peaks[K - 1] + s.peaks[0];
    // ---- vote (post_proc.py:75-98) on both axes of every segment
    for (int a = 0; a < 2; ++a) {
        s.sv[t] = s.xy[a][t];
        s.sseg[t] = g;
        __syncthreads();
        for (int k = 2; k <= W; k <<= 1)
            for (int j = k >> 1; j > 0; j >>= 1) {
                const int ixj = t ^ j;
                if (ixj > t) {
                    const bool up = (t & k) == 0;
                    const int ga = s.sseg[t], gb = s.sseg[ixj];
                    const double va = s.sv[t], vb = s.sv[ixj];
                    const bool gt = ga > gb || (ga == gb && va > vb);
                    if (gt == up) { s.sseg[t] = gb; s.sseg[ixj] = ga; s.sv[t] = vb; s.sv[ixj] = va; }
                }
                __syncthreads();
            }
        {   // widest window starting at this sorted position: last j with (v[j] - v[t]) + 1e-9 <= tol
            const int seg = s.sseg[t];
            const int st = seg == 0 ? 0 : size0 + s.peaks[seg - 1] - s.peaks[0];
            const int L = seg == 0 ? size0 : s.peaks[seg] - s.peaks[seg - 1];
            const int en = st + L;
            int lo3 = t, hi3 = en - 1;
            while (lo3 < hi3) {
                const int mid = (lo3 + hi3 + 1) >> 1;
                if ((s.sv[mid] - s.sv[t]) + 1e-9 <= (double)tol) lo3 = mid; else hi3 = mid - 1;
            }
            const int w = lo3 - t + 1;
            s.wv[t] = ((double)w < L * 0.4) ? -1 : w;          // n < len * 0.4 is invalid
        }
        __syncthreads();
        const int lane = t & 31;
        for (int seg = t >> 5; seg < K; seg += 32) {           // one warp per segment
            const int st = seg == 0 ? 0 : size0 + s.peaks[seg - 1] - s.peaks[0];
            const int L = seg == 0 ? size0 : s.peaks[seg] - s.peaks[seg - 1];
            int bw = -1, bi = 0x7fffffff;
            double sum = 0.0;
            for (int i = st + lane; i < st + L; i += 32) {
                const int w = s.wv[i];
                if (w > bw || (w == bw && i < bi)) { bw = w; bi = i; }
                sum += s.sv[i];
            }
            for (int o = 16; o; o >>= 1) {
                const int w2 = __shfl_xor_sync(0xffffffffu, bw, o), i2 = __shfl_xor_sync(0xffffffffu, bi, o);
                if (w2 > bw || (w2 == bw && i2 < bi)) { bw = w2; bi = i2; }
                sum += __shfl_xor_sync(0xffffffffu, sum, o);
            }
            double best, score;
            bool bad = false;
            if (bw < 0 || (double)L < (double)tol) {           // no valid entry, or len(vec) < tol: median
                best = (L & 1) ? s.sv[st + L / 2] : (s.sv[st + L / 2 - 1] + s.sv[st + L / 2]) / 2;
                score = 0.0;
            } else {
                bad = bw < 2;                                  // assert max_col > max_row
                double bs = 0.0;
                for (int i = bi + lane; i < bi + bw; i += 32) bs += s.sv[i];
                for (int o = 16; o; o >>= 1) bs += __shfl_xor_sync(0xffffffffu, bs, o);
                best = bs / bw;
                score = (double)bw / L;
            }
            double l1 = 0.0;
            for (int i = st + lane; i < st + L; i += 32) l1 += fabs(s.sv[i] - best);
            for (int o = 16; o; o >>= 1) l1 += __shfl_xor_sync(0xffffffffu, l1, o);
            if (lane == 0) {
                ws->seg_val[a][seg] = best;
                ws->seg_score[a][seg] = score;
                ws->seg_l1[a][seg] = l1 / L;
                ws->seg_mean[a][seg] = sum / L;
                if (bad) s.status = ST_ASSERT;
            }
        }
        __syncthreads();
    }
    if (s.status != ST_OK) {
        if (t == 0) s.nw = 0;
        __syncthreads();
        return;
    }
    if (t == 0) {
        for (int j = 0; j < K; ++j) {                          // :210-218 / :246-256
            const double xs = ws->seg_score[0][j], ys = ws->seg_score[1][j];
            const bool tx = xs > ys || (xs == ys && -ws->seg_l1[0][j] > -ws->seg_l1[1][j]);
            ws->type[j] = tx ? 0 : 1;
            ws->val[j] = tx ? ws->seg_val[0][j] : ws->seg_val[1][j];
            ws->score[j] = tx ? xs : ys;
            ws->gpid[j] = j;
            ws->u0[j] = coorx2u((double)s.peaks[(j - 1 + K) % K]);
            ws->u1[j] = coorx2u((double)s.peaks[j]);
            ws->tbd[j] = 1;
        }
        int n = K;
        if (cuboid) {                                          // sanity fallback :220-236 (types only)
            double sc[2] = {0.0, 0.0};
            for (int j = 0; j < 4; ++j) sc[j % 2] += ws->type[j] == 0 ? ws->score[j] : -ws->score[j];
            for (int j = 0; j < 4; ++j) ws->type[j] = (sc[0] > sc[1]) ? (j & 1) : 1 - (j & 1);
        } else {                                               // gen_ww_general :258-332
            while (true) {
                int tb = -1;
                for (int i = 0; i < n; ++i)
                    if (ws->tbd[i] && (tb == -1 || ws->score[i] > ws->score[tb])) tb = i;
                if (tb == -1) break;
                ws->tbd[tb] = 0;
                const int p = (tb - 1 + n) % n, q = (tb + 1) % n;
                const int ntbd = ws->tbd[p] + ws->tbd[q];
                if (ntbd == 2) continue;
                if (ntbd == 1) {
                    if ((!ws->tbd[p] && ws->type[p] == ws->type[tb]) || (!ws->tbd[q] && ws->type[q] == ws->type[tb])) {
                        if (ws->score[tb] >= -1) {             // re-queue
                            ws->tbd[tb] = 1;
                            ws->score[tb] -= 100;
                        } else {                               // forced infer: insert one wall
                            int at, nt;
                            double nv;
                            if (!ws->tbd[p]) {
                                at = tb;
                                if (ws->type[p] == 0) { nv = x_u_solve_y(ws->val[p], ws->u1[p]); nt = 1; }
                                else { nv = y_u_solve_x(ws->val[p], ws->u1[p]); nt = 0; }
                            } else {
                                at = q;
                                if (ws->type[q] == 0) { nv = x_u_solve_y(ws->val[q], ws->u0[q]); nt = 1; }
                                else { nv = y_u_solve_x(ws->val[q], ws->u0[q]); nt = 0; }
                            }
                            if (n >= MAXW) { s.status = ST_ASSERT; break; }
                            for (int i = n; i > at; --i) {
                                ws->val[i] = ws->val[i - 1]; ws->score[i] = ws->score[i - 1];
                                ws->u0[i] = ws->u0[i - 1]; ws->u1[i] = ws->u1[i - 1];
                                ws->type[i] = ws->type[i - 1]; ws->gpid[i] = ws->gpid[i - 1]; ws->tbd[i] = ws->tbd[i - 1];
                            }
                            ws->val[at] = nv; ws->score[at] = 0; ws->u0[at] = -1; ws->u1[at] = -1;
                            ws->type[at] = nt; ws->gpid[at] = -1; ws->tbd[at] = 0;
                            ++n;
                        }
                    }
                    continue;
                }
                if (ws->type[p] == ws->type[q]) {
                    if (ws->type[tb] == ws->type[p]) {         // forced change
                        ws->type[tb] = (ws->type[tb] + 1) % 2;
                        ws->val[tb] = ws->seg_mean[ws->type[tb]][ws->gpid[tb]];
                    }
                } else {                                       // two inferred walls replace this one
                    const int tp0 = ws->type[q], tp1 = ws->type[p];
                    double v0, v1;
                    if (ws->type[p] == 0) {
                        v0 = x_u_solve_y(ws->val[p], ws->u1[p]);
                        v1 = y_u_solve_x(ws->val[q], ws->u0[q]);
                    } else {
                        v0 = y_u_solve_x(ws->val[p], ws->u1[p]);
                        v1 = x_u_solve_y(ws->val[q], ws->u0[q]);
                    }
                    if (n >= MAXW) { s.status = ST_ASSERT; break; }
                    for (int i = n; i > tb + 1; --i) {
                        ws->val[i] = ws->val[i - 1]; ws->score[i] = ws->score[i - 1];
                        ws->u0[i] = ws->u0[i - 1]; ws->u1[i] = ws->u1[i - 1];
                        ws->type[i] = ws->type[i - 1]; ws->gpid[i] = ws->gpid[i - 1]; ws->tbd[i] = ws->tbd[i - 1];
                    }
                    ws->val[tb] = v0; ws->score[tb] = 0; ws->u0[tb] = -1; ws->u1[tb] = -1;
                    ws->type[tb] = tp0; ws->gpid[tb] = -1; ws->tbd[tb] = 0;
                    ws->val[tb + 1] = v1; ws->score[tb + 1] = 0; ws->u0[tb + 1] = -1; ws->u1[tb + 1] = -1;
                    ws->type[tb + 1] = tp1; ws->gpid[tb + 1] = -1; ws->tbd[tb + 1] = 0;
                    ++n;
                }
            }
        }
        s.nw = n;
    }
    __syncthreads();
}

// Polygon(xy2d).is_valid (inference.py:114-120) as an exact simple-ring test; sets s.invalid / s.status.
__device__ void check_ring(Smem& s, LayoutWs* ws) {
    const int t = threadIdx.x;
    const int n0 = s.nw;
    if (t == 0) {
        s.invalid = 0;
        if (n0 < 3) {
            s.status = ST_RING;                                // shapely: a ring needs at least 4 coordinates
        } else {
            int n = 0;
            for (int i = 0; i < n0; ++i) {                     // xy2d row i, then drop repeated consecutive vertices
                const int pi = (i - 1 + n0) % n0;
                float v[2] = {0.f, 0.f};
                v[ws->type[i]] = (float)ws->val[i];
                v[ws->type[pi]] = (float)ws->val[pi];
                if (n == 0 || v[0] != ws->ringx[n - 1] || v[1] != ws->ringy[n - 1]) {
                    ws->ringx[n] = v[0]; ws->ringy[n] = v[1]; ++n;
                }
            }
            while (n > 1 && ws->ringx[n - 1] == ws->ringx[0] && ws->ringy[n - 1] == ws->ringy[0]) --n;
            if (n < 3) s.invalid = 1;
            s.nring = n;
        }
    }
    __syncthreads();
    if (s.status != ST_OK || s.invalid) return;
    const int n = s.nring;
    const float* X = ws->ringx;
    const float* Y = ws->ringy;
    bool bad = false;
    for (int i = t; i < n && !bad; i += blockDim.x) {
        const int i1 = (i + 1) % n;
        for (int j = i + 1; j < n; ++j) {
            const int j1 = (j + 1) % n;
            if (j == i + 1 || (i == 0 && j == n - 1)) {        // adjacent: a spike folds back over the shared vertex
                float px, py, qx, qy, rx, ry;
                if (j == i + 1) { px = X[i]; py = Y[i]; qx = X[i1]; qy = Y[i1]; rx = X[j1]; ry = Y[j1]; }
                else { px = X[i1]; py = Y[i1]; qx = X[i]; qy = Y[i]; rx = X[j]; ry = Y[j]; }
                if (orient(px, py, qx, qy, rx, ry) == 0 &&
                    sign_ab_cd((double)qx - px, (double)rx - qx, -((double)qy - py), (double)ry - qy) < 0) {
                    bad = true; break;
                }
                continue;
            }
            const float ax = X[i], ay = Y[i], bx = X[i1], by = Y[i1], cx = X[j], cy = Y[j], dx = X[j1], dy = Y[j1];
            const int o1 = orient(ax, ay, bx, by, cx, cy), o2 = orient(ax, ay, bx, by, dx, dy);
            const int o3 = orient(cx, cy, dx, dy, ax, ay), o4 = orient(cx, cy, dx, dy, bx, by);
            if (o1 * o2 <= 0 && o3 * o4 <= 0 && !(o1 == 0 && o2 == 0)) { bad = true; break; }
            if ((o1 == 0 && on_box(ax, ay, bx, by, cx, cy)) || (o2 == 0 && on_box(ax, ay, bx, by, dx, dy)) ||
                (o3 == 0 && on_box(cx, cy, dx, dy, ax, ay)) || (o4 == 0 && on_box(cx, cy, dx, dy, bx, by))) {
                bad = true; break;
            }
        }
    }
    if (bad) s.invalid = 1;                                    // benign race: every writer stores 1
    __syncthreads();
}

__global__ void __launch_bounds__(1024, 1)
layout_kernel(const float* __restrict__ y_bon_pix, const float* __restrict__ y_cor, int mode, float min_v, int r,
              unsigned char* __restrict__ workspace, float* __restrict__ cor_id, int* __restrict__ n_cor,
              float* __restrict__ z1_out, int* __restrict__ status_out, int* __restrict__ peaks_out,
              int* __restrict__ types_out) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    Smem& s = *reinterpret_cast<Smem*>(smem_raw);
    const int b = blockIdx.x, t = threadIdx.x;
    LayoutWs* ws = reinterpret_cast<LayoutWs*>(workspace) + b;
    float* out = cor_id + (size_t)b * 2 * MAXW * 2;
    const float yb0 = y_bon_pix[(size_t)b * 2 * W + t], yb1 = y_bon_pix[(size_t)b * 2 * W + W + t];
    s.yb0[t] = yb0;
    s.ycor[t] = y_cor[(size_t)b * W + t];
    if (t == 0) { s.status = ST_OK; s.invalid = 0; s.K = 0; s.nw = 0; }

    // ---- np_refine_by_fix_z (post_proc.py:109-123) in float32, as the reference runs it on float32 rows
    const float pif = 3.14159265358979323846f;
    const float v0 = -(((yb0 + 0.5f) / 512.f) - 0.5f) * pif, v1 = -(((yb1 + 0.5f) / 512.f) - 0.5f) * pif;
    s.zs[t] = (50.f / tanf(v0)) * tanf(v1);
    __syncthreads();
    for (int k = 2; k <= W; k <<= 1)
        for (int j = k >> 1; j > 0; j >>= 1) {
            const int ixj = t ^ j;
            if (ixj > t) {
                const float a = s.zs[t], c = s.zs[ixj];
                if ((a > c) == ((t & k) == 0)) { s.zs[t] = c; s.zs[ixj] = a; }
            }
            __syncthreads();
        }
    // np.percentile (linear) at 25 / 75: positions 255.75 and 767.25 of 1024, numpy's _lerp
    const float lo_a = s.zs[255], lo_b = s.zs[256], hi_a = s.zs[767], hi_b = s.zs[768];
    const float vmin = lo_b - (lo_b - lo_a) * 0.25f, vmax = hi_a + (hi_b - hi_a) * 0.25f;
    const float zt = s.zs[t];
    const bool inr = vmin <= zt && zt <= vmax;
    const double zsum = block_sum(inr ? (double)zt : 0.0, s);
    const int zcnt = block_count(inr, s);
    const float z1 = (float)(zsum / zcnt);
    const float tol = fabsf(0.16f * z1 / 1.6f);                // inference.py:113, float32

    // ---- np_coor2xy of every column (post_proc.py:30-40), float64
    {
        const double u = coorx2u((double)t), v = coory2v((double)yb0);
        const double c = 50.0 / tan(v);
        s.xy[0][t] = c * sin(u) + 1024 / 2 - 0.5;
        s.xy[1][t] = -c * cos(u) + 512 / 2 - 0.5;
    }
    __syncthreads();

    int fallback = 0;
    int nrow;                                                  // rows of `cor` before infer_coory
    if (mode == 2) {                                           // force_raw: (column, ceiling row) for every column
        ws->corx[t] = (double)t;
        ws->cory[t] = (double)yb0;
        nrow = W;
    } else {
        const bool cuboid = mode == 1;
        walls_pass(s, ws, r, min_v, cuboid, cuboid, tol);
        if (!cuboid && s.status == ST_OK) {
            check_ring(s, ws);
            if (s.status == ST_OK && s.invalid) {              // inference.py:120-126
                fallback = 1;
                walls_pass(s, ws, r, 0.f, true, true, tol);
            }
        }
        nrow = s.nw;
        if (s.status == ST_OK) {
            for (int j = t; j < nrow; j += blockDim.x) {       // gen_ww :349-356 -> np_xy2coor
                const int nj = (j + 1) % nrow;
                const double px = ws->type[j] == 1 ? ws->val[nj] : ws->val[j];
                const double py = ws->type[j] == 1 ? ws->val[j] : ws->val[nj];
                const double x = px - 1024 / 2 + 0.5, y = py - 512 / 2 + 0.5;
                const double u = atan2(x, -y);
                const double v = atan(50 / sqrt(x * x + y * y));
                ws->corx[j] = (u / (2 * PI) + 0.5) * 1024 - 0.5;
                ws->cory[j] = (-v / PI + 0.5) * 512 - 0.5;
            }
        }
    }
    __syncthreads();
    const int status = s.status;
    int shift = 0;
    if (status == ST_OK && mode != 2) {                        // np.roll(cor, -2 * cor[::2, 0].argmin())
        double bv = INFINITY;
        int bi = 0x7fffffff;
        for (int j = 2 * t; j < nrow; j += 2 * blockDim.x)
            if (ws->corx[j] < bv) { bv = ws->corx[j]; bi = j; }
        for (int o = 16; o; o >>= 1) {
            const double v2 = __shfl_xor_sync(0xffffffffu, bv, o);
            const int i2 = __shfl_xor_sync(0xffffffffu, bi, o);
            if (v2 < bv || (v2 == bv && i2 < bi)) { bv = v2; bi = i2; }
        }
        if ((t & 31) == 0) { s.redd[t >> 5] = bv; s.redi[t >> 5] = bi; }
        __syncthreads();
        if (t == 0) {
            for (int i = 1; i < 32; ++i)
                if (s.redd[i] < s.redd[0] || (s.redd[i] == s.redd[0] && s.redi[i] < s.redi[0])) {
                    s.redd[0] = s.redd[i]; s.redi[0] = s.redi[i];
                }
        }
        __syncthreads();
        shift = s.redi[0];
    }
    if (status == ST_OK) {                                     // infer_coory + cor_id (inference.py:128-139)
        const float zz = 50.f + (z1 - 50.f);                   // z1 - z0 and z0 + h, both float32
        for (int rr = t; rr < nrow; rr += blockDim.x) {
            const int j = (rr + shift) % nrow;
            const double cx = ws->corx[j], cy = ws->cory[j];
            const double c0 = 50.0 / tan(coory2v(cy));
            const double y2 = (-atan2((double)zz, c0) / PI + 0.5) * 512 - 0.5;
            const float fx = (float)cx / 1024.f;
            out[(size_t)(2 * rr) * 2 + 0] = fx;
            out[(size_t)(2 * rr) * 2 + 1] = (float)cy / 512.f;
            out[(size_t)(2 * rr + 1) * 2 + 0] = fx;
            out[(size_t)(2 * rr + 1) * 2 + 1] = (float)y2 / 512.f;
        }
    }
    if (peaks_out && mode != 2)
        for (int i = t; i < s.K; i += blockDim.x) peaks_out[(size_t)b * W + i] = s.peaks[i];
    if (types_out && mode != 2 && status == ST_OK)
        for (int i = t; i < nrow; i += blockDim.x) types_out[(size_t)b * MAXW + i] = ws->type[i];
    if (t == 0) {
        n_cor[b] = status == ST_OK ? 2 * nrow : 0;
        z1_out[b] = z1;
        status_out[4 * b + 0] = status;
        status_out[4 * b + 1] = fallback;
        status_out[4 * b + 2] = mode == 2 ? 0 : s.K;
        status_out[4 * b + 3] = (mode == 2 || status != ST_OK) ? 0 : nrow;
    }
}

}  // namespace

size_t layout_workspace_bytes(int B) { return (size_t)B * sizeof(LayoutWs); }

int layout(const float* y_bon_pix, const float* y_cor, int B, int mode, float min_v, int r_px, void* workspace,
           float* cor_id, int* n_cor, float* z1, int* status, int* peaks, int* types, cudaStream_t st) {
    HN_CUDA_OK(cudaFuncSetAttribute(layout_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(Smem)));
    layout_kernel<<<B, W, sizeof(Smem), st>>>(y_bon_pix, y_cor, mode, min_v, r_px, (unsigned char*)workspace, cor_id,
                                               n_cor, z1, status, peaks, types);
    HN_LAUNCH_OK();
    return 0;
}

}  // namespace hn
