"""TEST INFRASTRUCTURE ONLY: a numpy / torch-CPU emulation of the C-ABI in include/cgan_b200.h.

It lets the `-m "not gpu"` suite execute the REAL host code of the package — `kernels.py` (every taped op and its
vector-Jacobian product), `tape.py`, `variables.py` (flat packing), `gans/modular_gan.py` (the unrolled cycle, Adam, EMA,
step counters, checkpoints) — on the CPU and compare it with the oracle, so host-side logic errors show up without a
GPU.  Each entry point follows the header's contract literally (raw addresses and sizes; nothing knows about tensors).

This is NOT a fallback: nothing under `compare_gan_b200/` imports it, and the package still refuses to run without the
CUDA library.  Tests opt in explicitly with `with emulated_library(): ...`.
"""
import contextlib
import ctypes

import numpy as np
import torch
import torch.nn.functional as F


def f32(ptr, n):
  return np.ctypeslib.as_array((ctypes.c_float * int(n)).from_address(int(ptr)))


def i32(ptr, n):
  return np.ctypeslib.as_array((ctypes.c_int32 * int(n)).from_address(int(ptr)))


def f64(ptr, n):
  return np.ctypeslib.as_array((ctypes.c_double * int(n)).from_address(int(ptr)))


def rna_tf32(a):
  """cvt.rna.tf32.f32 on a float32 array: round the 13 low mantissa bits to nearest, ties away from zero."""
  a = np.ascontiguousarray(a, np.float32)
  return ((a.view(np.uint32) + np.uint32(0x1000)) & np.uint32(0xFFFFE000)).view(np.float32)


def _desc(ref):
  d = ref._obj            # ctypes.byref(ConvDesc)
  return d


def _conv_forward(x, w, d):
  """x: torch [n,h,w,cin] (real input), w: torch HWIO.  Returns [n,oh,ow,cout] per cgan_conv_desc."""
  xt = x.permute(0, 3, 1, 2)
  if d.upsample:
    up = torch.zeros(xt.shape[0], xt.shape[1], 2 * d.h, 2 * d.w, dtype=xt.dtype)
    up[:, :, ::2, ::2] = xt
    xt = up
  vh, vw = xt.shape[2], xt.shape[3]
  pad_b = max((d.oh - 1) * d.stride + d.kh - vh - d.pad_t, 0)
  pad_r = max((d.ow - 1) * d.stride + d.kw - vw - d.pad_l, 0)
  xt = F.pad(xt, (d.pad_l, pad_r, d.pad_t, pad_b))
  y = F.conv2d(xt, w.permute(3, 2, 0, 1), stride=d.stride)
  y = y[:, :, :d.oh, :d.ow]
  assert y.shape[2] == d.oh and y.shape[3] == d.ow, (tuple(y.shape), d.oh, d.ow)
  return y.permute(0, 2, 3, 1)


class EmulatedLib(object):
  """Same surface as compare_gan_b200._lib.Lib: call(name, *args), launch_count(), set_stream()."""

  emulated = True

  def __init__(self):
    self.launches = 0
    self.math_mode = 0
    self.last_path = 0

  def set_stream(self, stream):
    pass

  def launch_count(self):
    return self.launches

  def get_option(self, key):
    return {1: 2, 2: self.last_path, 3: 1, 6: 1}[key]

  def set_option(self, key, value):
    assert (key == 1 and value in (1, 2)) or (key == 3 and value in (0, 1, 2)) or (key == 6 and value in (0, 1))

  def call(self, name, *args):
    self.launches += 1
    getattr(self, "cgan_" + name)(*args)

  # ---- context / utilities ------------------------------------------------------------------
  def cgan_ctx_set_math_mode(self, mode):
    assert mode in (0, 1)
    self.math_mode = mode

  def cgan_ctx_set_option(self, key, value):
    self.set_option(key, value)

  def cgan_ctx_get_option(self, key, out):
    out._obj.value = self.get_option(key)

  def _tc(self, d=None):
    """math_mode 1 is emulated as the tensor-core ARITHMETIC (operands rounded to the nearest TF32 value, fp32
    accumulation) for every contraction with more than 4 input and output channels, and for the image-side layers whose
    taps fit one 32-wide patch row (the library runs those as 32-wide GEMMs, csrc/thin_tc.cu); other thin layers stay exact.  Sets the path CGAN_OPT_LAST_PATH reports."""
    thin = d is not None and min(d.cin, d.cout) <= 4
    if thin:      # image-side layers: a 32-wide GEMM over patch tensors (csrc/thin_tc.cu) when kh*kw*channels fits one row
      thin_tc = (not d.upsample and d.kh * d.kw > 1 and d.kh * d.kw * min(d.cin, d.cout) <= 32 and
                 max(d.cin, d.cout) >= 32 and max(d.cin, d.cout) % 4 == 0 and (d.cin <= 4 or d.stride == 1))
    tc = self.math_mode == 1 and (d is None or not thin or thin_tc)
    self.last_path = 1 if tc else 0
    return tc

  def cgan_fill(self, dst, value, n):
    f32(dst, n)[:] = np.float32(value)

  def cgan_copy(self, dst, src, n):
    f32(dst, n)[:] = f32(src, n).copy()

  def cgan_copy2d(self, dst, dst_ld, dst_off, src, src_ld, src_off, rows, cols):
    d = f32(dst, rows * dst_ld).reshape(rows, dst_ld)
    s = f32(src, rows * src_ld).reshape(rows, src_ld)
    d[:, dst_off:dst_off + cols] = s[:, src_off:src_off + cols].copy()

  def cgan_axpby(self, y, a, x, b, y0, c, n):
    out = np.float32(a) * f32(x, n)
    if y0 is not None:
      out = out + np.float32(b) * f32(y0, n)
    f32(y, n)[:] = out + np.float32(c)

  def cgan_scale_by_dev(self, y, x, scalar_dev, mul, inverse, n):
    s = f32(scalar_dev, 1)[0]
    s = np.float32(1.0) / s if inverse else s
    f32(y, n)[:] = f32(x, n) * (s * np.float32(mul))

  def cgan_dot(self, out_dev, a, b, n):
    f32(out_dev, 1)[0] = np.float32(np.dot(f32(a, n).astype(np.float64), f32(b, n).astype(np.float64)))

  def cgan_random_uniform(self, out, n, seed, offset):
    m = np.uint64(0xFFFFFFFFFFFFFFFF)
    with np.errstate(over="ignore"):
      z = np.uint64(seed) + np.uint64(0x9E3779B97F4A7C15) * (np.uint64(offset) + np.arange(1, n + 1, dtype=np.uint64))
      z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
      z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
      z = z ^ (z >> np.uint64(31))
    f32(out, n)[:] = (z >> np.uint64(40)).astype(np.float32) * np.float32(1.0 / 16777216.0)

  def cgan_interpolate(self, y, x, xf, alpha, n, per):
    xa, xb = f32(x, n * per).reshape(n, per), f32(xf, n * per).reshape(n, per)
    f32(y, n * per).reshape(n, per)[:] = xa + f32(alpha, n).reshape(n, 1) * (xb - xa)

  def cgan_one_hot(self, out, labels, n, classes):
    o = f32(out, n * classes).reshape(n, classes)
    o[:] = 0
    lab = i32(labels, n)
    ok = (lab >= 0) & (lab < classes)          # tf.one_hot: an out-of-range index (S3GAN's -1 = "no label") is a zero row
    o[np.arange(n)[ok], lab[ok]] = 1

  # ---- contractions -------------------------------------------------------------------------
  def _conv_tensors(self, d, x_ptr, w_ptr):
    x = torch.from_numpy(f32(x_ptr, d.n * d.h * d.w * d.cin).reshape(d.n, d.h, d.w, d.cin).copy())
    w = torch.from_numpy(f32(w_ptr, d.kh * d.kw * d.cin * d.cout).reshape(d.kh, d.kw, d.cin, d.cout).copy())
    return x, w

  def cgan_conv2d_fwd(self, dref, x, w, bias, y):
    self.cgan_conv2d_fwd_act_ld(dref, x, w, bias, 0, y, _desc(dref).cout)

  def cgan_conv2d_fwd_act(self, dref, x, w, bias, act, y):
    self.cgan_conv2d_fwd_act_ld(dref, x, w, bias, act, y, _desc(dref).cout)

  def cgan_conv2d_fwd_act_ld(self, dref, x, w, bias, act, y, ldy):
    d = _desc(dref)
    xt, wt = self._conv_tensors(d, x, w)
    if self._tc(d):
      xt, wt = torch.from_numpy(rna_tf32(xt.numpy())), torch.from_numpy(rna_tf32(wt.numpy()))
    out = _conv_forward(xt, wt, d).numpy()
    if bias is not None:
      out = out + f32(bias, d.cout)
    if act == 1:
      out = np.maximum(out, 0)
    pixels = d.n * d.oh * d.ow
    out = out.reshape(pixels, d.cout).astype(np.float32)
    if ldy == d.cout:
      f32(y, pixels * d.cout).reshape(pixels, d.cout)[:] = out
    else:                                # channel slice of a wider NHWC tensor: the last row owns only cout floats
      for p in range(pixels):
        f32(y + 4 * p * ldy, d.cout)[:] = out[p]

  def _post(self, out_ptr, n, ep, relu_done=False):
    """Epilogue of the *_ex convolution entry points on a dense output of n floats."""
    o = f32(out_ptr, n)
    if ep.residual:
      o += f32(ep.residual, n)
    if (ep.flags & 1) and not relu_done:
      np.maximum(o, 0, out=o)
    if ep.mask:
      m = f32(ep.mask, n)
      o[:] = np.where(m > 0, o, np.float32(ep.mask_leak) * o)
    if ep.flags & 2:
      o[:] = rna_tf32(o)

  def cgan_conv2d_fwd_ex(self, dref, x, w, epref, y):
    d, ep = _desc(dref), epref._obj
    ldy = ep.ldy or d.cout
    assert ldy == d.cout or not (ep.residual or ep.mask or (ep.flags & 2)), "strided fused outputs are not emulated"
    plain_relu = (ep.flags & 1) and not (ep.residual or ep.mask)
    self.cgan_conv2d_fwd_act_ld(dref, x, w, ep.bias, 1 if plain_relu else 0, y, ldy)
    if ldy == d.cout:
      self._post(y, d.n * d.oh * d.ow * d.cout, ep, relu_done=plain_relu)

  def cgan_conv2d_dgrad_ex(self, dref, dy, w, epref, dx):
    d = _desc(dref)
    self.cgan_conv2d_dgrad(dref, dy, w, dx)
    if epref is not None:
      ep = epref._obj
      n = d.n * d.h * d.w * d.cin
      if ep.bias:
        f32(dx, n).reshape(-1, d.cin)[:] += f32(ep.bias, d.cin)
      self._post(dx, n, ep)

  def cgan_conv2d_wgrad_ex(self, dref, x, dy, flags, dw):
    self.cgan_conv2d_wgrad(dref, x, dy, dw)

  def cgan_conv2d_dgrad(self, dref, dy, w, dx):
    d = _desc(dref)
    x = torch.zeros(d.n, d.h, d.w, d.cin, requires_grad=True)
    wt = torch.from_numpy(f32(w, d.kh * d.kw * d.cin * d.cout).reshape(d.kh, d.kw, d.cin, d.cout).copy())
    g = torch.from_numpy(f32(dy, d.n * d.oh * d.ow * d.cout).reshape(d.n, d.oh, d.ow, d.cout).copy())
    if self._tc(d):
      wt, g = torch.from_numpy(rna_tf32(wt.numpy())), torch.from_numpy(rna_tf32(g.numpy()))
    _conv_forward(x, wt, d).backward(g)
    f32(dx, x.numel())[:] = x.grad.numpy().ravel()

  def cgan_conv2d_wgrad(self, dref, x, dy, dw):
    d = _desc(dref)
    xt = torch.from_numpy(f32(x, d.n * d.h * d.w * d.cin).reshape(d.n, d.h, d.w, d.cin).copy())
    wt = torch.zeros(d.kh, d.kw, d.cin, d.cout, requires_grad=True)
    g = torch.from_numpy(f32(dy, d.n * d.oh * d.ow * d.cout).reshape(d.n, d.oh, d.ow, d.cout).copy())
    if self._tc(d):
      xt, g = torch.from_numpy(rna_tf32(xt.numpy())), torch.from_numpy(rna_tf32(g.numpy()))
    _conv_forward(xt, wt, d).backward(g)
    f32(dw, wt.numel())[:] = wt.grad.numpy().ravel()

  def cgan_gemm(self, ta, tb, m, n, k, alpha, a, lda, b, ldb, beta, c, ldc):
    self.cgan_gemm_batched(ta, tb, m, n, k, alpha, a, lda, 0, b, ldb, 0, beta, c, ldc, 0, 1)

  def cgan_gemm_batched(self, ta, tb, m, n, k, alpha, a, lda, sa, b, ldb, sb, beta, c, ldc, sc, batch):
    tc = self._tc() and batch > 1
    self.last_path = 1 if tc else 0
    for i in range(batch):
      ar, ac = (k, m) if ta else (m, k)
      br, bc = (n, k) if tb else (k, n)
      am = f32(a + 4 * i * sa, (ar - 1) * lda + ac).copy()
      bm = f32(b + 4 * i * sb, (br - 1) * ldb + bc).copy()
      A = np.lib.stride_tricks.as_strided(am, (ar, ac), (4 * lda, 4))
      B = np.lib.stride_tricks.as_strided(bm, (br, bc), (4 * ldb, 4))
      A = A.T if ta else A
      B = B.T if tb else B
      if tc:
        A, B = rna_tf32(A), rna_tf32(B)
      cm = f32(c + 4 * i * sc, (m - 1) * ldc + n)
      C = np.lib.stride_tricks.as_strided(cm, (m, n), (4 * ldc, 4))
      res = np.float32(alpha) * (A.astype(np.float32) @ B.astype(np.float32))
      C[:] = res + (np.float32(beta) * C if beta != 0 else 0)

  # ---- rows x channels ----------------------------------------------------------------------
  def cgan_bias_add(self, y, x, bias, rows, c):
    f32(y, rows * c).reshape(rows, c)[:] = f32(x, rows * c).reshape(rows, c) + f32(bias, c)

  def cgan_colsum(self, out, x, groups, rows_per_group, c):
    v = f32(x, groups * rows_per_group * c).reshape(groups, rows_per_group, c)
    f32(out, groups * c).reshape(groups, c)[:] = v.sum(axis=1, dtype=np.float64).astype(np.float32)

  # ---- batch norm ---------------------------------------------------------------------------
  def cgan_bn_moments(self, stats, x, rows, c):
    v = f32(x, rows * c).reshape(rows, c).astype(np.float64)
    s = f32(stats, 2 * c)
    s[:c] = v.mean(0)
    s[c:] = (v * v).mean(0)

  def cgan_bn_finalize(self, mean_var, stats, c, moving_mean, moving_var, decay):
    s, out = f32(stats, 2 * c), f32(mean_var, 2 * c)
    mean = s[:c].copy()
    var = s[c:] - mean * mean
    out[:c], out[c:] = mean, var
    if moving_mean is not None:
      mm = f32(moving_mean, c)
      mm -= (mm - mean) * np.float32(1.0 - decay)
    if moving_var is not None:
      mv = f32(moving_var, c)
      mv -= (mv - var) * np.float32(1.0 - decay)

  def cgan_bn_accumulate(self, mean_var, batch, c, accu_mean, accu_var, accu_counter, update_accus):
    am, av, ac = f32(accu_mean, c), f32(accu_var, c), f32(accu_counter, 1)
    if f32(update_accus, 1)[0] == 1.0:
      b = f32(batch, 2 * c)
      am += b[:c]
      av += b[c:]
      ac += 1
    out = f32(mean_var, 2 * c)
    out[:c] = am / ac[0]
    out[c:] = av / ac[0]

  @staticmethod
  def _per_row(ptr, rows, c, rows_per_sample, cond):
    if ptr is None:
      return None
    if not cond:
      return f32(ptr, c).reshape(1, c)
    samples = rows // rows_per_sample
    return np.repeat(f32(ptr, samples * c).reshape(samples, c), rows_per_sample, axis=0)

  def cgan_bn_apply(self, y, x, rows, c, rows_per_sample, mean_var, eps, gamma, beta, cond, act):
    rnd, act = act & 0x100, act & 0xFF
    mv = f32(mean_var, 2 * c)
    xv = f32(x, rows * c).reshape(rows, c)
    out = (xv - mv[:c]) * (np.float32(1.0) / np.sqrt(mv[c:] + np.float32(eps)))
    g, b = self._per_row(gamma, rows, c, rows_per_sample, cond), self._per_row(beta, rows, c, rows_per_sample, cond)
    if g is not None:
      out = out * g
    if b is not None:
      out = out + b
    if act == 1:
      out = np.maximum(out, 0)
    f32(y, rows * c).reshape(rows, c)[:] = rna_tf32(out) if rnd else out

  def cgan_bn_bwd_reduce(self, sums, dgamma, dbeta, dy, x, rows, c, rows_per_sample, mean_var, eps, gamma, cond):
    mv = f32(mean_var, 2 * c)
    inv = 1.0 / np.sqrt(mv[c:].astype(np.float64) + eps)
    xhat = (f32(x, rows * c).reshape(rows, c).astype(np.float64) - mv[:c]) * inv
    g = f32(dy, rows * c).reshape(rows, c).astype(np.float64)
    gam = self._per_row(gamma, rows, c, rows_per_sample, cond)
    dxhat = g * gam if gam is not None else g
    s = f32(sums, 2 * c)
    s[:c] = dxhat.sum(0)
    s[c:] = (dxhat * xhat).sum(0)
    groups = rows // rows_per_sample if cond else 1
    if dgamma is not None:
      f32(dgamma, groups * c).reshape(groups, c)[:] = (g * xhat).reshape(groups, -1, c).sum(1)
    if dbeta is not None:
      f32(dbeta, groups * c).reshape(groups, c)[:] = g.reshape(groups, -1, c).sum(1)

  def cgan_bn_bwd_apply(self, dx, dy, x, rows, c, rows_per_sample, mean_var, eps, gamma, cond, sums, inv_count,
                        round_tf32=0):
    mv = f32(mean_var, 2 * c)
    inv = 1.0 / np.sqrt(mv[c:].astype(np.float64) + eps)
    xhat = (f32(x, rows * c).reshape(rows, c).astype(np.float64) - mv[:c]) * inv
    g = f32(dy, rows * c).reshape(rows, c).astype(np.float64)
    gam = self._per_row(gamma, rows, c, rows_per_sample, cond)
    dxhat = g * gam if gam is not None else g
    s = f32(sums, 2 * c).astype(np.float64)
    out = (inv * (dxhat - s[:c] * inv_count - xhat * s[c:] * inv_count)).astype(np.float32)
    f32(dx, rows * c).reshape(rows, c)[:] = rna_tf32(out) if round_tf32 else out

  # ---- spectral norm --------------------------------------------------------------------------
  @staticmethod
  def _l2n(v, eps):
    return v / np.sqrt(max(float((v.astype(np.float64) ** 2).sum()), eps))

  def cgan_spectral_norm(self, w, rows, cols, left, eps, u_inout, v_out, sigma_out, wbar_out):
    W = f32(w, rows * cols).reshape(rows, cols).astype(np.float64)
    if left:
      u = f32(u_inout, rows).astype(np.float64)
      v = self._l2n(W.T @ u, eps)
      un = self._l2n(W @ v, eps)
      sigma = float(un @ W @ v)
      f32(u_inout, rows)[:] = un
      f32(v_out, cols)[:] = v
    else:
      u = f32(u_inout, cols).astype(np.float64)
      v = self._l2n(W @ u, eps)          # (u W^T)^T
      un = self._l2n(W.T @ v, eps)       # (v W)^T
      sigma = float(v @ W @ un)
      f32(u_inout, cols)[:] = un
      f32(v_out, rows)[:] = v
    f32(sigma_out, 1)[0] = sigma
    if wbar_out is not None:
      f32(wbar_out, rows * cols)[:] = (W / sigma).ravel()

  def cgan_spectral_norm_batched(self, items, n, max_dims, eps, wbar_base, v_base, sigma_base, u_used_base):
    raw = np.ctypeslib.as_array((ctypes.c_uint8 * (56 * n)).from_address(int(items)))
    rec = raw.view(np.dtype([("w", "<u8"), ("u", "<u8"), ("rows", "<i4"), ("cols", "<i4"), ("left", "<i4"), ("reserved", "<i4"),
                             ("wbar_off", "<i8"), ("v_off", "<i8"), ("u_off", "<i8")]))
    for i in range(n):
      r = rec[i]
      rows, cols, left = int(r["rows"]), int(r["cols"]), int(r["left"])
      assert rows + cols <= max_dims
      nu = rows if left else cols
      self.cgan_spectral_norm(int(r["w"]), rows, cols, left, eps, int(r["u"]), v_base + 4 * int(r["v_off"]),
                              sigma_base + 4 * i, wbar_base + 4 * int(r["wbar_off"]))
      f32(u_used_base + 4 * int(r["u_off"]), nu)[:] = f32(int(r["u"]), nu)

  def cgan_spectral_norm_bwd(self, dw, dwbar, wbar, rows, cols, left, u, v, sigma):
    g = f32(dwbar, rows * cols).reshape(rows, cols).astype(np.float64)
    wb = f32(wbar, rows * cols).reshape(rows, cols).astype(np.float64)
    s = float(f32(sigma, 1)[0])
    if left:
      outer = np.outer(f32(u, rows), f32(v, cols)).astype(np.float64)
    else:
      outer = np.outer(f32(v, rows), f32(u, cols)).astype(np.float64)
    f32(dw, rows * cols)[:] = ((g - (g * wb).sum() * outer) / s).ravel()

  # ---- pointwise / pooling --------------------------------------------------------------------
  def cgan_act_fwd(self, y, x, kind, leak, n):
    rnd, kind = kind & 0x100, kind & 0xFF
    v = f32(x, n)
    out = {1: lambda: np.maximum(v, 0), 2: lambda: np.maximum(v, np.float32(leak) * v),
           3: lambda: (1.0 / (1.0 + np.exp(-v.astype(np.float64)))).astype(np.float32),
           4: lambda: ((np.tanh(v.astype(np.float64)) + 1.0) / 2.0).astype(np.float32)}[kind]()
    f32(y, n)[:] = rna_tf32(out) if rnd else out

  def cgan_act_bwd(self, dx, dy, ref, kind, leak, n):
    rnd, kind = kind & 0x100, kind & 0xFF
    g, r = f32(dy, n), f32(ref, n)
    if kind == 1:
      out = g * (r > 0)
    elif kind == 2:
      out = g * np.where(r > 0, np.float32(1.0), np.float32(leak))
    elif kind == 3:
      out = g * r * (1 - r)
    else:                                  # y = (tanh+1)/2  =>  dy/dx = (1 - tanh^2)/2 = 2 y (1 - y)
      out = g * 2 * r * (1 - r)
    f32(dx, n)[:] = rna_tf32(out) if rnd else out

  def cgan_rot90(self, y, x, n, hw, c, k):
    v = f32(x, n * hw * hw * c).reshape(n, hw, hw, c)
    tr = lambda a: a.transpose(0, 2, 1, 3)
    out = {1: lambda: tr(v)[:, ::-1], 2: lambda: v[:, ::-1, ::-1], 3: lambda: tr(v[:, ::-1])}[k]()
    f32(y, n * hw * hw * c)[:] = np.ascontiguousarray(out).ravel()

  def cgan_rotation_loss(self, loss_out, dlogits, logits, rows, nrot):
    z = torch.from_numpy(f32(logits, rows * nrot).reshape(rows, nrot).copy()).double().requires_grad_(True)
    labels = torch.arange(nrot).repeat_interleave(rows // nrot)
    p = torch.softmax(z, -1)[torch.arange(rows), labels]
    loss = -(torch.log(p + 1e-10)).mean()
    loss.backward()
    f32(loss_out, 1)[0] = float(loss.detach())
    if dlogits is not None:
      f32(dlogits, rows * nrot)[:] = z.grad.numpy().astype(np.float32).ravel()

  def cgan_row_has_label(self, out, y, rows, cols):
    f32(out, rows)[:] = (f32(y, rows * cols).reshape(rows, cols).sum(1) > 0.5).astype(np.float32)

  def cgan_argmax_one_hot(self, out, logits, rows, cols):
    z = f32(logits, rows * cols).reshape(rows, cols)
    o = f32(out, rows * cols).reshape(rows, cols)
    o[:] = 0
    o[np.arange(rows), z.argmax(1)] = 1

  def cgan_softmax_xent(self, loss_out, dlogits, logits, labels, weights, rows, cols):
    z = torch.from_numpy(f32(logits, rows * cols).reshape(rows, cols).copy()).double().requires_grad_(True)
    lab = torch.from_numpy(f32(labels, rows * cols).reshape(rows, cols).copy()).double()
    w = torch.ones(rows, dtype=torch.float64) if weights is None else torch.from_numpy(f32(weights, rows).copy()).double()
    ce = -(lab * torch.log_softmax(z, -1)).sum(1)
    present = float((w != 0).sum())
    loss = (w * ce).sum() / present if present > 0 else (w * ce).sum() * 0.0
    loss.backward()
    f32(loss_out, 1)[0] = float(loss.detach())
    if dlogits is not None:
      f32(dlogits, rows * cols)[:] = z.grad.numpy().astype(np.float32).ravel()

  def cgan_add(self, y, a, b, n):
    f32(y, n)[:] = f32(a, n) + f32(b, n)

  def cgan_add_tf32(self, y, a, b, n, round_tf32):
    out = f32(a, n) + f32(b, n)
    f32(y, n)[:] = rna_tf32(out) if round_tf32 else out

  def cgan_avgpool2_fwd(self, y, x, n, h, w, c):
    v = f32(x, n * h * w * c).reshape(n, h // 2, 2, w // 2, 2, c)
    f32(y, n * (h // 2) * (w // 2) * c)[:] = v.mean(axis=(2, 4)).ravel()

  def cgan_avgpool2_bwd(self, dx, dy, n, h, w, c):
    g = f32(dy, n * (h // 2) * (w // 2) * c).reshape(n, h // 2, 1, w // 2, 1, c)
    f32(dx, n * h * w * c)[:] = np.broadcast_to(g * np.float32(0.25), (n, h // 2, 2, w // 2, 2, c)).ravel()

  def cgan_maxpool2_fwd(self, y, x, n, h, w, c):
    v = f32(x, n * h * w * c).reshape(n, h // 2, 2, w // 2, 2, c)
    f32(y, n * (h // 2) * (w // 2) * c)[:] = v.max(axis=(2, 4)).ravel()

  def cgan_maxpool2_bwd(self, dx, dy, x, n, h, w, c):
    v = f32(x, n * h * w * c).reshape(n, h // 2, 2, w // 2, 2, c).transpose(0, 1, 3, 5, 2, 4).reshape(-1, 4)
    g = f32(dy, n * (h // 2) * (w // 2) * c).reshape(-1)
    out = np.zeros_like(v)
    out[np.arange(v.shape[0]), v.argmax(axis=1)] = g        # first maximum wins, as TF's MaxPoolGrad
    out = out.reshape(n, h // 2, w // 2, c, 2, 2).transpose(0, 1, 4, 2, 5, 3)
    f32(dx, n * h * w * c)[:] = out.ravel()

  def cgan_globalpool_fwd(self, y, x, n, hw, c, scale):
    f32(y, n * c).reshape(n, c)[:] = f32(x, n * hw * c).reshape(n, hw, c).sum(1, dtype=np.float64) * scale

  def cgan_globalpool_bwd(self, dx, dy, n, hw, c, scale):
    g = f32(dy, n * c).reshape(n, 1, c) * np.float32(scale)
    f32(dx, n * hw * c)[:] = np.broadcast_to(g, (n, hw, c)).ravel()

  def cgan_softmax_fwd(self, y, x, rows, cols):
    v = f32(x, rows * cols).reshape(rows, cols).astype(np.float64)
    e = np.exp(v - v.max(1, keepdims=True))
    f32(y, rows * cols).reshape(rows, cols)[:] = e / e.sum(1, keepdims=True)

  def cgan_softmax_bwd(self, dx, dy, y, rows, cols):
    g = f32(dy, rows * cols).reshape(rows, cols).astype(np.float64)
    p = f32(y, rows * cols).reshape(rows, cols).astype(np.float64)
    f32(dx, rows * cols).reshape(rows, cols)[:] = p * (g - (g * p).sum(1, keepdims=True))

  # ---- fused attention (csrc/attn_tc.cu): same contract, same shape rule, TF32 probabilities ----
  def attention_supported(self, batch, lq, lk, dk, dv):
    return (self.math_mode == 1 and 1 <= batch <= 65535 and lq >= 128 and lq % 128 == 0 and lk >= 128 and lk % 128 == 0 and
            4 <= dk <= 32 and dk % 4 == 0 and 16 <= dv <= 128 and dv % 16 == 0)

  def cgan_round_tf32(self, y, x, n):
    f32(y, n)[:] = rna_tf32(f32(x, n))

  def cgan_attention_fwd(self, q, k, v, out, lse, batch, lq, lk, dk, dv):
    assert self.attention_supported(batch, lq, lk, dk, dv)
    self.last_path = 1
    Q = f32(q, batch * lq * dk).reshape(batch, lq, dk)
    Kk = f32(k, batch * lk * dk).reshape(batch, lk, dk)
    Vv = f32(v, batch * lk * dv).reshape(batch, lk, dv)
    s = np.einsum("bqd,bkd->bqk", Q, Kk).astype(np.float32)
    m = s.max(2, keepdims=True)
    pe = rna_tf32(np.exp(s - m).astype(np.float32))
    l = pe.sum(2, keepdims=True, dtype=np.float32)
    f32(out, batch * lq * dv).reshape(batch, lq, dv)[:] = np.einsum("bqk,bkd->bqd", pe, Vv) / l
    f32(lse, batch * lq).reshape(batch, lq)[:] = (m + np.log(l))[:, :, 0]

  def cgan_attention_bwd(self, q, k, v, out, lse, dout, dq, dk_out, dv_out, batch, lq, lk, dk, dv):
    assert self.attention_supported(batch, lq, lk, dk, dv)
    self.last_path = 1
    Q = f32(q, batch * lq * dk).reshape(batch, lq, dk)
    Kk = f32(k, batch * lk * dk).reshape(batch, lk, dk)
    Vv = f32(v, batch * lk * dv).reshape(batch, lk, dv)
    O = f32(out, batch * lq * dv).reshape(batch, lq, dv)
    dO = f32(dout, batch * lq * dv).reshape(batch, lq, dv)
    L = f32(lse, batch * lq).reshape(batch, lq, 1)
    p = np.exp(np.einsum("bqd,bkd->bqk", Q, Kk).astype(np.float32) - L).astype(np.float32)
    dsum = (dO * O).sum(2, keepdims=True, dtype=np.float32)
    ds = rna_tf32(p * (np.einsum("bqd,bkd->bqk", dO, Vv).astype(np.float32) - dsum))
    p = rna_tf32(p)
    f32(dq, batch * lq * dk).reshape(batch, lq, dk)[:] = np.einsum("bqk,bkd->bqd", ds, Kk)
    f32(dk_out, batch * lk * dk).reshape(batch, lk, dk)[:] = np.einsum("bqk,bqd->bkd", ds, Q)
    f32(dv_out, batch * lk * dv).reshape(batch, lk, dv)[:] = np.einsum("bqk,bqd->bkd", p, dO)

  def cgan_rowdot(self, out, a, b, rows, cols):
    f32(out, rows)[:] = (f32(a, rows * cols).reshape(rows, cols).astype(np.float64) *
                         f32(b, rows * cols).reshape(rows, cols)).sum(1)

  def cgan_rowscale(self, y, a, s, rows, cols):
    f32(y, rows * cols).reshape(rows, cols)[:] = f32(a, rows * cols).reshape(rows, cols) * f32(s, rows).reshape(rows, 1)

  # ---- losses / penalties / optimizer -----------------------------------------------------------
  def cgan_gan_loss(self, kind, logits_real, logits_fake, b, out4, dlogits, which):
    from oracle import gan as ogan
    name = {0: "non_saturating", 1: "hinge", 2: "wasserstein", 3: "least_squares"}[kind]
    r = torch.from_numpy(f32(logits_real, b).reshape(b, 1).copy()).requires_grad_(True)
    f = torch.from_numpy(f32(logits_fake, b).reshape(b, 1).copy()).requires_grad_(True)
    losses = ogan.get_losses(name, torch.sigmoid(r), torch.sigmoid(f), r, f)
    f32(out4, 4)[:] = [float(v.detach()) for v in losses]
    if dlogits is not None:
      target = losses[0] if which == 0 else losses[3]
      gr, gf = torch.autograd.grad(target, [r, f], allow_unused=True)
      zero = torch.zeros(b, 1)
      f32(dlogits, 2 * b)[:] = torch.cat([zero if gr is None else gr, zero if gf is None else gf]).numpy().ravel()

  def cgan_gp_penalty(self, penalty_out, dg, g, n, per, weight):
    gt = torch.from_numpy(f32(g, n * per).reshape(n, per).copy()).requires_grad_(True)
    slopes = torch.sqrt(1e-4 + (gt * gt).sum(1))
    pen = ((slopes - 1.0) ** 2).mean()
    f32(penalty_out, 1)[0] = float(pen.detach())
    if dg is not None:
      (weight * pen).backward()
      f32(dg, n * per)[:] = gt.grad.numpy().ravel()

  def cgan_adam_step(self, p, g, m, v, n, lr, beta1, beta2, eps, grad_scale, step_dev, ema, ema_decay, ema_start_step):
    step = i32(step_dev, 1)
    step[0] += 1
    t = int(step[0])
    lr_t = np.float32(lr * np.sqrt(1.0 - beta2 ** t) / (1.0 - beta1 ** t))
    pv, gv, mv, vv = f32(p, n), f32(g, n) * np.float32(grad_scale), f32(m, n), f32(v, n)
    mv[:] = np.float32(beta1) * mv + np.float32(1.0 - beta1) * gv
    vv[:] = np.float32(beta2) * vv + np.float32(1.0 - beta2) * gv * gv
    pv -= lr_t * mv / (np.sqrt(vv) + np.float32(eps))
    if ema is not None:
      d = np.float32(ema_decay if (t - 1) >= ema_start_step else 0.0)
      ev = f32(ema, n)
      ev -= (ev - pv) * (np.float32(1.0) - d)

  # ---- evaluation ---------------------------------------------------------------------------------
  def cgan_pool2d_fwd(self, y, x, n, h, w, c, k, stride, pad_t, pad_l, oh, ow, mode):
    xt = torch.from_numpy(f32(x, n * h * w * c).reshape(n, h, w, c).copy()).permute(0, 3, 1, 2)
    pad_b = max((oh - 1) * stride + k - h - pad_t, 0)
    pad_r = max((ow - 1) * stride + k - w - pad_l, 0)
    if mode == 0:
      out = F.max_pool2d(F.pad(xt, (pad_l, pad_r, pad_t, pad_b), value=float("-inf")), k, stride)
    else:             # tf.nn.avg_pool "SAME": padded cells are excluded from the divisor
      total = F.avg_pool2d(F.pad(xt, (pad_l, pad_r, pad_t, pad_b)), k, stride, divisor_override=1)
      count = F.avg_pool2d(F.pad(torch.ones(1, 1, h, w), (pad_l, pad_r, pad_t, pad_b)), k, stride, divisor_override=1)
      out = total / count
    out = out[:, :, :oh, :ow]
    f32(y, n * oh * ow * c)[:] = out.permute(0, 2, 3, 1).contiguous().numpy().ravel()

  def cgan_resize_bilinear(self, y, x, n, h, w, c, oh, ow, inception_scale):
    from oracle import inception as oinc
    out = oinc.resize_bilinear_tf(torch.from_numpy(f32(x, n * h * w * c).reshape(n, h, w, c).copy()), oh, ow)
    if inception_scale:
      out = (out * 255.0 - 128.0) / 128.0
    f32(y, n * oh * ow * c)[:] = out.contiguous().numpy().ravel()

  def cgan_cov_accumulate(self, act, n, d, s, sxx):
    a = f32(act, n * d).reshape(n, d).astype(np.float64)
    f64(s, d)[:] += a.sum(0)
    f64(sxx, d * d).reshape(d, d)[:] += a.T @ a


@contextlib.contextmanager
def emulated_library():
  """Runs the package's host code against the emulator: kernels._RT points at an EmulatedLib on the CPU and the few
  torch.cuda calls of the host code (synchronize / current_stream / empty_cache) become no-ops."""
  from compare_gan_b200 import kernels as K
  saved_rt = dict(K._RT)
  saved_cuda = {name: getattr(torch.cuda, name) for name in ("synchronize", "current_stream", "empty_cache", "Event")}

  class _Stream(object):
    cuda_stream = 0
  lib = EmulatedLib()
  K._RT["lib"], K._RT["device"] = lib, torch.device("cpu")
  saved_from_numpy = K.from_numpy

  def from_numpy(a, req=False):
    # on the GPU `.to(device)` copies; on the CPU it would alias the caller's array (e.g. VariableStore.init_values)
    return K.DT(torch.from_numpy(np.array(a, copy=True)).contiguous(), req)
  K.from_numpy = from_numpy
  torch.cuda.synchronize = lambda *a, **k: None
  torch.cuda.current_stream = lambda *a, **k: _Stream()
  torch.cuda.empty_cache = lambda: None

  class _Event(object):            # runner_lib.PipelineFeeder: copies are synchronous on the CPU
    def __init__(self, *a, **k):
      pass

    def record(self, *a, **k):
      pass

    def synchronize(self):
      pass
  torch.cuda.Event = _Event
  try:
    yield lib
  finally:
    K._RT.update(saved_rt)
    K.from_numpy = saved_from_numpy
    for name, fn in saved_cuda.items():
      setattr(torch.cuda, name, fn)
