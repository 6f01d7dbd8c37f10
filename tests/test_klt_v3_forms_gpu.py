"""The staged tracker's conversions (csrc/klt_v3_forms.cuh) beside the shared forms of klt.cu, on the device and bit for
bit: the magic-constant floor over every fraction class near integers, near 0 and near the limits of [-2^22, 2^22)
(and beyond them, where the range test must still reject), the FADD cvRound of the packed weights over ties and weight sums of 2^14 + 1,
and the host bound that replaces the minEig division.  Then whole-tracker runs against the oracle at image borders,
far outside the image and over a sweep of minEig thresholds."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from monocular_visual_odometry_va4mr_b200 import _lib, synth

pytestmark = pytest.mark.gpu

CSRC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "monocular_visual_odometry_va4mr_b200", "csrc")
NVCC = os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin", "nvcc")

# floor_to_int and bilinear_weights as klt.cu has them (the generic tracker still runs these), next to the v3 forms
SRC = r"""
#define W_BITS 14
#include "klt_v3_forms.cuh"
__device__ __forceinline__ int floor_to_int(float v)
{
    if (!(fabsf(v) < 1.0e9f)) return INT_MIN;
    return __float2int_rd(v);
}
__device__ __forceinline__ void bilinear_weights(float a, float b, int& w00, int& w01, int& w10, int& w11)
{
    const float s = (float)(1 << W_BITS);
    w00 = __float2int_rn(__fmul_rn(__fmul_rn(__fsub_rn(1.f, a), __fsub_rn(1.f, b)), s));
    w01 = __float2int_rn(__fmul_rn(__fmul_rn(a, __fsub_rn(1.f, b)), s));
    w10 = __float2int_rn(__fmul_rn(__fmul_rn(__fsub_rn(1.f, a), b), s));
    w11 = (1 << W_BITS) - w00 - w01 - w10;
}
__global__ void floor_k(const float* x, int n, int* o)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint32_t bits;
    const float f = floor_v3(x[i], bits);
    const int old = floor_to_int(x[i]);
    o[5 * i] = old;
    o[5 * i + 1] = __float_as_int(__fsub_rn(x[i], (float)old));
    o[5 * i + 2] = floor_bits_to_int(bits);
    o[5 * i + 3] = __float_as_int(__fsub_rn(x[i], f));
    o[5 * i + 4] = __float2int_rd(x[i]);
}
__global__ void weights_k(const float* a, const float* b, int n, uint32_t* o)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    int w00, w01, w10, w11;
    bilinear_weights(a[i], b[i], w00, w01, w10, w11);
    uint32_t wt, wb;
    bilinear_weights_v3(a[i], b[i], wt, wb);
    o[5 * i] = (uint32_t)(w01 * 65536 + w00);
    o[5 * i + 1] = (uint32_t)w11 * 65536u + (uint32_t)w10;
    o[5 * i + 2] = wt;
    o[5 * i + 3] = wb;
    o[5 * i + 4] = (uint32_t)w11;
}
__global__ void min_eig_k(const float* num, int n, float d, float thr, float bound, uint8_t* o)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    o[2 * i] = __fdiv_rn(num[i], d) < thr;
    o[2 * i + 1] = num[i] < bound;
}
extern "C" float t_bound(float thr, float d) { return min_eig_num_bound(thr, d); }
extern "C" int t_floor(const float* x, int n, int* o) { floor_k<<<(n + 255) / 256, 256>>>(x, n, o); return (int)cudaDeviceSynchronize(); }
extern "C" int t_weights(const float* a, const float* b, int n, uint32_t* o) { weights_k<<<(n + 255) / 256, 256>>>(a, b, n, o); return (int)cudaDeviceSynchronize(); }
extern "C" int t_min_eig(const float* num, int n, float d, float thr, float bound, uint8_t* o)
{
    min_eig_k<<<(n + 255) / 256, 256>>>(num, n, d, thr, bound, o);
    return (int)cudaDeviceSynchronize();
}
"""


@pytest.fixture(scope="module")
def forms(tmp_path_factory):
    import torch
    torch.cuda.init()
    d = tmp_path_factory.mktemp("klt_v3_forms")
    src, so = d / "forms.cu", d / "forms.so"
    src.write_text(SRC)
    subprocess.check_call([NVCC, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "--fmad=false",
                           "-Xcompiler", "-fPIC", "-shared", "-I", CSRC, str(src), "-o", str(so)])
    lib = C.CDLL(str(so))
    lib.t_bound.restype = C.c_float
    lib.t_bound.argtypes = [C.c_float, C.c_float]
    for f in (lib.t_floor, lib.t_weights, lib.t_min_eig):
        f.restype = C.c_int
    return lib, torch


def _dev(torch, a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _around(v, k):
    """k floats on each side of every value of v, v included"""
    v = np.float32(v).ravel()
    out = [v]
    lo, hi = v.copy(), v.copy()
    for _ in range(k):
        lo, hi = np.nextafter(lo, np.float32(-np.inf)), np.nextafter(hi, np.float32(np.inf))
        out += [lo, hi]
    return np.concatenate(out)


def test_floor_matches_shared_form(forms):
    lib, torch = forms
    rng = np.random.default_rng(0)
    ints = np.float32(np.arange(-300, 301))
    big = np.float32([2.0 ** 22, 2.0 ** 23, 1.5 * 2.0 ** 23, 2.0 ** 24, 2.0 ** 30, 1e9, 3e38])
    x = np.concatenate([
        _around(ints, 300),                                         # every fraction class next to integers, both sides
        _around(np.float32([0.0, -0.0, 0.5, -0.5]), 2000),          # +-0, subnormals, near 1/2
        np.float32(rng.uniform(-5000, 5000, 1 << 20)),
        _around(np.concatenate([big, -big]), 600),                  # the +-2^22 limit and far beyond
        np.float32([np.inf, -np.inf, np.nan, 1.5 * 2.0 ** 23 - 0.5, -1.5 * 2.0 ** 23]),
    ]).astype(np.float32)
    o = torch.zeros((len(x), 5), dtype=torch.int32, device="cuda")
    assert lib.t_floor(C.c_void_p(_dev(torch, x).data_ptr()), len(x), C.c_void_p(o.data_ptr())) == 0
    o = o.cpu().numpy()
    exact = (x >= -2.0 ** 22) & (x < 2.0 ** 22)
    assert exact.sum() > 1_000_000
    # in [-2^22, 2^22): the same integer and the same fraction bits as floor_to_int / __float2int_rd
    assert np.array_equal(o[exact, 2], o[exact, 0]) and np.array_equal(o[exact, 2], o[exact, 4])
    assert np.array_equal(o[exact, 3], o[exact, 1])
    # beyond (and non-finite): outside [-2^22, 2^22], so every range test of a level below 2^22 px rejects it
    far = o[~exact, 2]
    assert len(far) > 1000 and np.all((far >= 1 << 22) | (far < -(1 << 22)))


def test_weights_match_shared_form(forms):
    lib, torch = forms
    rng = np.random.default_rng(1)
    one = np.float32(1)
    k = np.arange(0, 1 << 14, dtype=np.float64)
    ties = np.float32((k + 0.5) / 16384.0)                          # a * 1 * 2^14 exactly k + 1/2: ties to even
    edge = _around(np.float32([0.0, 1.0, 0.5, 0.25, 0.75]), 3000)
    edge = edge[(edge >= 0) & (edge <= 1)]
    a = np.concatenate([ties, ties, np.zeros_like(ties), np.float32(rng.random(1 << 21)), edge, np.repeat(edge, 7)])
    b = np.concatenate([np.zeros_like(ties), one - ties, ties, np.float32(rng.random(1 << 21)), edge[::-1],
                        np.tile(np.float32([0, 1e-5, 3e-5, 0.5, 1 - 3e-5, 1 - 1e-5, 1]), len(edge))])
    # fractions of ~0 in both axes: the three rounded weights add up to 2^14 + 1 (iw11 = -1)
    t = np.float32(rng.uniform(0, 6e-5, 1 << 18))
    a = np.concatenate([a, t, one - t]).astype(np.float32)
    b = np.concatenate([b, t[::-1], t]).astype(np.float32)
    o = torch.zeros((len(a), 5), dtype=torch.int32, device="cuda")
    assert lib.t_weights(C.c_void_p(_dev(torch, a).data_ptr()), C.c_void_p(_dev(torch, b).data_ptr()), len(a),
                         C.c_void_p(o.data_ptr())) == 0
    o = o.cpu().numpy()
    assert np.array_equal(o[:, 2], o[:, 0]) and np.array_equal(o[:, 3], o[:, 1])
    assert (o[:, 4] == -1).sum() > 100


@pytest.mark.parametrize("thr", [1e-4, 1e-3, 0.01, 0.37, 5e-8, 0.0, -1.0, float("inf"), float("nan")])
@pytest.mark.parametrize("win", [15, 21])
def test_min_eig_bound_matches_division(forms, thr, win):
    lib, torch = forms
    d = np.float32(2 * win * win)
    thr = np.float32(thr)
    bound = np.float32(lib.t_bound(float(thr), float(d)))
    rng = np.random.default_rng(2)
    cands = [bound, thr * d] if np.isfinite(bound) else [thr * d]
    cands = [c for c in cands if np.isfinite(c)]
    num = np.concatenate([_around(np.float32(cands), 4000) if cands else np.float32([]),
                          np.float32(rng.uniform(-1, 60, 1 << 18)), _around(np.float32([0.0, -0.0]), 100),
                          np.float32([np.inf, -np.inf, 3e38, -3e38])]).astype(np.float32)
    o = torch.zeros((len(num), 2), dtype=torch.uint8, device="cuda")
    assert lib.t_min_eig(C.c_void_p(_dev(torch, num).data_ptr()), len(num), C.c_float(d), C.c_float(thr),
                         C.c_float(bound), C.c_void_p(o.data_ptr())) == 0
    o = o.cpu().numpy()
    assert np.array_equal(o[:, 0], o[:, 1])
    with np.errstate(invalid="ignore"):
        assert np.array_equal(o[:, 0], (num / d < thr).astype(np.uint8))   # numpy's float32 division is IEEE too


CRIT = (3, 30, 0.01)


@pytest.fixture(scope="module")
def env():
    import torch
    return _lib.default_context(0), torch


def _track(env, f0, f1, pts, win, ml, min_eig):
    ctx, torch = env
    dev = torch.device("cuda", 0)
    h, w = f0.shape
    n = len(pts)
    d0, d1 = torch.from_numpy(f0).to(dev), torch.from_numpy(f1).to(dev)
    dp = torch.from_numpy(np.ascontiguousarray(pts, np.float32)).to(dev)
    o_p = torch.zeros((n, 2), dtype=torch.float32, device=dev)
    o_s = torch.zeros((n,), dtype=torch.uint8, device=dev)
    o_e = torch.zeros((n,), dtype=torch.float32, device=dev)
    rc = ctx.lib.b200vo_calc_optical_flow_pyr_lk_dev(ctx.h, d0.data_ptr(), d1.data_ptr(), h, w, w, w, dp.data_ptr(), n,
                                                     win, win, ml, CRIT[0], CRIT[1], CRIT[2], 0, min_eig,
                                                     o_p.data_ptr(), o_s.data_ptr(), o_e.data_ptr())
    assert rc == 0, ctx.last_error()
    ctx.sync()
    torch.cuda.synchronize()
    return o_p.cpu().numpy(), o_s.cpu().numpy(), o_e.cpu().numpy()


@pytest.mark.parametrize("win,ml", [(15, 4), (21, 3)])
def test_tracker_borders_and_min_eig_sweep_vs_oracle(env, win, ml):
    """Points straddling every edge at every level and points far outside, over minEig thresholds from accept-all to
    reject-most: status, positions and errors equal the oracle's bit for bit."""
    import oracle
    s = synth.render_sequence("kitti", 2, seed=23, width=520, height=180)
    f0, f1 = s["frames"]
    h, w = f0.shape
    rng = np.random.default_rng(9)
    pts = []
    for lvl in range(ml + 1):
        sc = 1 << lvl
        for dd in range(-3, win + 3):
            f = rng.uniform(0, 1, 2)
            pts += [((dd + f[0]) * sc, rng.uniform(0.2, 0.8) * h), (w - 1 - (dd + f[0]) * sc, rng.uniform(0.2, 0.8) * h),
                    (rng.uniform(0.2, 0.8) * w, (dd + f[1]) * sc), (rng.uniform(0.2, 0.8) * w, h - 1 - (dd + f[1]) * sc)]
    pts += [(-1e7, 50.0), (50.0, 5e6), (4194304.0, 10.0), (-4194305.0, -3.0), (3e30, 1.0)]
    pts += list(zip(rng.uniform(0, w, 300), rng.uniform(0, h, 300)))
    pts = np.float32(pts)
    counts = []
    for thr in (0.0, 1e-4, 1e-3, 4e-3, 0.01, 0.03):
        rp, rst, rerr = oracle.calc_optical_flow_pyr_lk(f0, f1, pts, (win, win), ml, CRIT, min_eig=thr)
        rst, rerr = rst.ravel(), rerr.ravel()
        p, st, err = _track(env, f0, f1, pts, win, ml, thr)
        ok = rst == 1
        assert np.array_equal(st, rst), thr
        assert np.array_equal(p[ok], rp[ok]) and np.array_equal(err[ok], rerr[ok]), thr
        counts.append(int(ok.sum()))
    assert counts[0] > counts[-1] > 0   # the thresholds do reject windows
