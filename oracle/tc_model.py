"""oracle/tc_model.py -- float64 model of the tensor-core path's own arithmetic (TEST INFRASTRUCTURE ONLY).

The tensor-core kernels (fused_tc.cu / fused_mg.cuh: LNB_PATH_TC train and render steps of MLPs of up to 4 layers of
width <= 63; wide_tc.cu: the layerwise path of everything wider or deeper) multiply bf16 operands and accumulate in
fp32.  ``nerf_f64`` / ``mlp_fit_f64`` restate the mathematics exactly, so a comparison with them has to absorb the
whole bf16 error (~5e-3 on the gradients of the C2 network) and cannot see a kernel that is wrong by less.  This model
rounds to bf16 exactly where the kernels do and keeps float64 everywhere else (sums of bf16 products are then exact up
to the fp32 roundings it states), so a kernel differs from it only by its fp32 summation order and its fast
transcendentals: 1e-5 and below.

Rounding points (variant "fused": fused_tc.cu / fused_mg.cuh; variant "wide": wide_tc.cu):
  * A_0 = bf16(X); the ones column that carries the bias is exact (pack_features in fused_tc.cu; f32_to_bf16_rows_kernel
    in wide_tc.cu, which has no ones column: its biases are added in the epilogue).
  * W_l = bf16(w_l), zero-padded (ImgMap::put_w via tc_prep_kernel; wide_prep_all_kernel).
  * hidden pre-activations: "fused" adds bf16(b_l) inside the MMA (ImgMap::put_b writes the bias into the weight
    operand's row in_l), Z_l = fp32(A_l W_l + bf16(b_l)); "wide" adds the fp32 bias in the epilogue (EPI_RELU_BF16),
    Z_l = fp32(fp32(A_l W_l) + b_l).
  * A_{l+1} = bf16(relu(Z_l)) (cvt.rn.relu.bf16x2 in the fused epilogue; fmaxf + pack_bf16 in EPI_RELU_BF16).
  * the head's pre-activations hz = fp32(fp32(A_{L-1} W_{L-1}) + b_head), b_head fp32 in both variants (the fp32 bias
    tail of the weight image; EPI_HEAD_F32).  Head, compositing, loss and head adjoint: the float64 formulas of the
    restatement (oracle.head_f64, composite_f64, fit_loss_f64, head_adjoint_f64).
  * dZ_{L-1} = bf16(dz), dz the unit-seed adjoint of hz (the dZ_{L-1} pack in fused_mg.cuh / fused_v1_kernel;
    f32_to_bf16_rows_kernel of the head adjoint in lnb_wide_tc_step).
  * dZ_{l-1} = bf16(fp32(dZ_l W_l^T)) . [A_l > 0], the mask from the STORED bf16 activation (relu_adjoint in
    fused_tc.cu; the ReLU bit pattern of EPI_RELU_BF16 read back by EPI_MASK_BF16).
  * dW_l = A_l^T dZ_l and db_l = sum_rows dZ_l from the bf16 operands (the weight-gradient MMAs; the bias gradient is
    the ones column in the fused kernels, a column sum in wide_tc.cu), then scaled by the seed after the reduction
    (tc_reduce_kernel, wide_reduce_all_kernel): with g = 'loss' that is the loss times the unit-seed gradient.

Rays input (``rays=(rays_o, rays_d, t, E)``): x = fp32(o + d t) as sample_inputs in fused_tc.cu forms it, then the
positional encoding of that x in float64, rounded to fp32 and bf16.  The kernels' sin / cos are faster and less
accurate (MUFU with angle doubling in the fused kernel, fp32 sincosf of fp32(2^i x) in the wide one), so a bf16
rounding of a high band can flip: compare rays mode with this model at E <= 2 only.

``_exact=True`` switches every rounding off; the model then is the float64 restatement (tests/test_tc_model.py checks
that the two agree to 1e-12, so they cannot drift apart).
"""
import numpy as np

from oracle import oracle as O


def bf16(x):
    """Round-to-nearest-even to bf16 of float32 values; float64 input is rounded to float32 first (the kernels round an
    fp32 accumulator).  Returns the bf16 values as float64.  NaN stays NaN."""
    with np.errstate(invalid="ignore", over="ignore"):
        x32 = np.ascontiguousarray(np.asarray(x, np.float64).astype(np.float32))
    b = x32.view(np.uint32).astype(np.uint64)
    r = ((b + (((b >> np.uint64(16)) & np.uint64(1)) + np.uint64(0x7FFF))) & np.uint64(0xFFFF0000)).astype(np.uint32)
    out = r.view(np.float32).astype(np.float64)
    return np.where(np.isnan(x32), np.nan, out)


def f32(x):
    """Round float64 values to float32 (returned as float64)."""
    return np.asarray(x, np.float64).astype(np.float32).astype(np.float64)


def _ident(x):
    return np.asarray(x, np.float64)


def rays_features(rays_o, rays_d, t, E):
    """A_0 before its bf16 rounding in rays mode: the positional encoding of x = fp32(o + d t) (float64 math, float32
    result), [R*S][3 + 6E]."""
    pts, _ = O.sample_points(rays_o, rays_d, t)
    return O.positional_encoding(f32(pts), E).reshape(-1, 3 + 6 * E)


def _forward(A0, ws, bs, dims, variant, rb, rf, head):
    L = len(dims) - 1
    W = [rb(ws[l, :dims[l], :dims[l + 1]]) for l in range(L)]
    A = [rb(A0)]
    for l in range(L - 1):
        b = np.asarray(bs[l, :dims[l + 1]], np.float64)
        if variant == "fused":
            Z = rf(A[l] @ W[l] + rb(b))
        elif variant == "wide":
            Z = rf(rf(A[l] @ W[l]) + b)
        else:
            raise ValueError(variant)
        A.append(rb(np.maximum(Z, 0.0)))
    hz = rf(rf(A[-1] @ W[-1]) + np.asarray(bs[L - 1, :dims[L]], np.float64))
    return W, A, hz, O.head_f64(hz, head)


def _backward(res, W, A, dz, ws, bs, dims, g, rb, rf):
    """Unit-seed adjoint chain from dz, weight / bias gradients scaled by the seed after the reduction."""
    L = len(dims) - 1
    dZ = [None] * L
    dZ[L - 1] = rb(dz)
    for l in range(L - 1, 0, -1):
        dZ[l - 1] = rb(rf(dZ[l] @ W[l].T)) * (A[l] > 0)
    scale = float(res["loss"]) if isinstance(g, str) else float(g)
    d_ws = np.zeros(ws.shape, np.float64)
    d_bs = np.zeros(bs.shape, np.float64)
    for l in range(L):
        d_ws[l, :dims[l], :dims[l + 1]] = scale * (A[l].T @ dZ[l])
        d_bs[l, :dims[l + 1]] = scale * dZ[l].sum(0)
    res.update(d_ws=d_ws, d_bs=d_bs, dz=dZ, scale=scale)
    return res


def nerf_tc_model(X, ws, bs, dims, target, dists, R, S, g=None, variant="fused", rays=None, _exact=False):
    """The tensor-core nerf step as the kernels compute it (see the module docstring).  Same arguments and keys as
    oracle.nerf_f64 (loss, color, d_ws, d_bs) plus the intermediates: A_l (the bf16 layer inputs, A_l[0] = A_0), hz (the
    head's pre-activations), dz (the bf16 adjoints dZ_l), scale (the seed the gradients were multiplied by).  rays =
    (rays_o, rays_d, t, E) builds A_0 from rays (X is then ignored)."""
    rb, rf = (_ident, _ident) if _exact else (bf16, f32)
    dims = [int(v) for v in dims]
    A0 = rays_features(*rays) if rays is not None else X
    W, A, hz, Y = _forward(A0, ws, bs, dims, variant, rb, rf, "nerf")
    res = O.composite_f64(Y, dists, target, R, S, None if g is None else 1.0)
    res.update(A_l=A, hz=hz)
    if g is None:
        return res
    return _backward(res, W, A, O.head_adjoint_f64(Y, res.pop("dY"), "nerf"), ws, bs, dims, g, rb, rf)


def fit_tc_model(X, ws, bs, dims, target, g=None, variant="fused", _exact=False):
    """The tensor-core mlp_fit step (sigmoid head, SSE), as nerf_tc_model; same keys as oracle.mlp_fit_f64."""
    rb, rf = (_ident, _ident) if _exact else (bf16, f32)
    dims = [int(v) for v in dims]
    W, A, hz, Y = _forward(X, ws, bs, dims, variant, rb, rf, "sigmoid")
    res = O.fit_loss_f64(Y, target, None if g is None else 1.0)
    res.update(A_l=A, hz=hz)
    if g is None:
        return res
    return _backward(res, W, A, O.head_adjoint_f64(Y, res.pop("dY"), "sigmoid"), ws, bs, dims, g, rb, rf)


def without_rows(res, rows):
    """d_ws / d_bs of a model result with the contributions of the sample rows `rows` left out of the reduction (what a
    kernel that lost those rows' tile would return)."""
    d_ws, d_bs = res["d_ws"].copy(), res["d_bs"].copy()
    for l, (A, dZ) in enumerate(zip(res["A_l"], res["dz"])):
        i, o = A.shape[1], dZ.shape[1]
        d_ws[l, :i, :o] -= res["scale"] * (A[rows].T @ dZ[rows])
        d_bs[l, :o] -= res["scale"] * dZ[rows].sum(0)
    return dict(res, d_ws=d_ws, d_bs=d_bs)
