"""LayerNorm epilogue of the tensor-core layer and chain kernels against an fp64 reference,
on rows that are hard for the row statistics (one outlier column, a large offset on every
column, constant and near-constant rows), at every cluster size, at both output widths with
and without padding columns, and for every LayerNorm output kind.

A row family lives in the bias vector or in the weight scale, which every row of a launch
shares, so each family is a launch of its own.  The products stay ordinary, and the fp64
reference of the same op, built from the fp32 inputs, is exact.  The error is
max |got - want| / max |want|.  Its bound adds twice the error of torch's fp32 LayerNorm
applied to the fp64 pre-LayerNorm values rounded to fp32: on the offset families fp32
itself loses digits, everywhere else that term is ~0."""
import ctypes as C

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import _cases
from _cases import cluster  # noqa: F401  (fixture)
from graphcast_b200 import _native, engine
from oracle import gnn as oracle_gnn

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
TOL = {"bf16x3": 3e-5, "bf16": 2e-2, "fp32_simt": 5e-6}
CONST = 0.3      # the value of every pre-LayerNorm column in the (near-)constant families

# Outliers at the first column of each 256-column unit (0, 256), at the last ones (255, 511)
# and at an interior column (37).
OUTLIERS = [f"col{c}+{a}" for a in (30, 100, 1000) for c in (0, 256, 255, 511, 37)]
FAMILIES = ["ordinary", "offset+1e2", "offset+1e3", "constant", "near_constant"] + OUTLIERS


def _stream():
  return torch.cuda.current_stream().cuda_stream


def _rel(got, want):
  return float((got - want).abs().max() / want.abs().max())


def _ln64(pre, scale, offset):
  return F.layer_norm(pre, (pre.shape[1],), scale.double(), offset.double(), 1e-5)


def _e32(pre, scale, offset, want, add=0):
  """Error of torch's fp32 LayerNorm of the fp64 pre-LayerNorm values rounded to fp32."""
  y32 = F.layer_norm(pre.float(), (pre.shape[1],), scale.float(), offset.float(), 1e-5).double()
  return _rel(y32 + add, want + add)


def _family(name, rows, k, n_valid, n, g):
  """(x [rows, k], w [k, n_valid], bias [n]) fp32: N(0, 1) pre-activations plus the family."""
  x = torch.randn(rows, k, generator=g)
  w = torch.randn(k, n_valid, generator=g) / np.sqrt(k)
  bias = 0.1 * torch.randn(n, generator=g)
  if name == "constant":
    x.zero_()
    bias.fill_(CONST)
  elif name == "near_constant":          # variance ~1e-8: eps dominates
    w *= 1e-4
    bias.fill_(CONST)
  elif name.startswith("offset+"):
    bias += float(name[7:])
  elif name.startswith("col"):
    col, a = name[3:].split("+")
    bias[int(col)] += float(a)
  else:
    assert name == "ordinary", name
  return x, w, bias


def _ln_params(n, g):
  return 1 + 0.1 * torch.randn(n, generator=g), 0.1 * torch.randn(n, generator=g)


def _packed(x):
  """Weight [k, n] fp32 -> (packed bf16 hi/lo image, fp32 copy) on the device."""
  lib = _native.lib()
  k, n = x.shape
  wp = np.ascontiguousarray(x.numpy(), dtype=np.float32)
  img = np.empty(lib.gcb_packed_weight_bytes(k, n), np.uint8)
  assert lib.gcb_pack_weight_host(wp.ctypes.data, k, n, k, n, img.ctypes.data) == 0
  return torch.as_tensor(img).to(DEV), torch.as_tensor(wp).to(DEV)


def _canary_ld(n_valid):
  return n_valid + (4 - n_valid % 4) % 4 + 4      # NaN-filled columns past n_valid


def _decode_image(img, rows):
  """Operand image of a 512-wide result -> fp32 [rows, 512] (hi + lo), on the host."""
  raw = img.cpu().numpy().view(np.uint16).reshape(-1, 32, 2, 2112)      # [tile, kstep, hi|lo, 2112 u16]
  pieces = np.stack([raw[..., :1024], raw[..., 1056:2080]], axis=3)      # chunks c = 0, 1 (64 B skew)
  pieces = pieces.reshape(-1, 32, 2, 2, 128, 8)                           # [tile, ks, part, c, row, 8]
  f = (pieces.astype(np.uint32) << 16).view(np.float32)
  x = f[:, :, 0] + f[:, :, 1]
  return torch.as_tensor(x.transpose(0, 3, 1, 2, 4).reshape(-1, 512)[:rows])


def _layer(prec, x, w, bias, n, *, ln=None, act=False, residual=None, out=False, out_y=True,
           out_img=False):
  """One gcb_layer_forward on table input x.  Returns (status, {output name: host tensor})."""
  lib = _native.lib()
  rows, k = x.shape
  n_valid = w.shape[1]
  wpad = torch.zeros(k, n)
  wpad[:, :n_valid] = w
  wimg, wf = _packed(wpad)
  alive = [x.to(DEV), wimg, wf, bias.to(DEV)]
  d = _native.LayerDesc()
  d.rows, d.n, d.n_valid, d.nseg = rows, n, n_valid, 1
  d.seg[0].table, d.seg[0].ld, d.seg[0].k, d.seg[0].k_valid, d.seg[0].fan = alive[0].data_ptr(), k, k, k, 1
  d.w_packed, d.w_f32, d.bias = wimg.data_ptr(), wf.data_ptr(), alive[3].data_ptr()
  if ln is not None:
    alive += [ln[0].to(DEV), ln[1].to(DEV)]
    d.ln_scale, d.ln_offset = alive[-2].data_ptr(), alive[-1].data_ptr()
  d.act = _native.ACT_SWISH if act else _native.ACT_NONE
  ld = _canary_ld(n_valid)
  bufs = {}
  if residual is not None:
    alive.append(residual.to(DEV))
    d.residual, d.ld_res = alive[-1].data_ptr(), residual.shape[1]
  if out:
    bufs["out"] = torch.full((rows, ld), float("nan"), device=DEV)
    d.out, d.ld_out = bufs["out"].data_ptr(), ld
  if out_y:
    bufs["out_y"] = torch.full((rows, ld), float("nan"), device=DEV)
    d.out_y, d.ld_out_y = bufs["out_y"].data_ptr(), ld
  if out_img:
    bufs["img"] = torch.zeros(lib.gcb_a_image_bytes(rows, n), dtype=torch.uint8, device=DEV)
    d.out_img = bufs["img"].data_ptr()
  d.precision = _native.PRECISIONS[prec]
  rc = lib.gcb_layer_forward(C.byref(d), _stream())
  torch.cuda.synchronize()
  return rc, {name: t.cpu() for name, t in bufs.items()}


def _check_canary(got, n_valid):
  assert torch.isnan(got[:, n_valid:]).all(), "kernel wrote beyond n_valid"


def test_cluster_size_is_validated():
  lib = _native.lib()
  for bad in (0, 3, 8):
    assert lib.gcb_set_cluster_size(bad) == -1
    assert b"cluster size" in lib.gcb_last_error()


@pytest.mark.parametrize("prec,cluster", [("bf16x3", 1), ("bf16x3", 2), ("bf16x3", 4),
                                          ("fp32_simt", 2)], indirect=["cluster"])
@pytest.mark.parametrize("family", FAMILIES)
def test_layernorm_row_families(family, prec, cluster):
  """fp32_simt (two-pass statistics, no cluster) is the control that the bound is fair."""
  g = torch.Generator().manual_seed(FAMILIES.index(family))
  rows, k, n = 3 * 128 + 45, 256, 512
  x, w, bias = _family(family, rows, k, n, n, g)
  scale, offset = _ln_params(n, g)
  rc, o = _layer(prec, x, w, bias, n, ln=(scale, offset))
  _native.check(rc, "layer")
  got = o["out_y"]
  _check_canary(got, n)
  pre = x.double() @ w.double() + bias.double()
  want = _ln64(pre, scale, offset)
  err, e32 = _rel(got[:, :n].double(), want), _e32(pre, scale, offset, want)
  print(f"\n{family:>14} {prec:>9} cluster {cluster}: err {err:.2e}  fp32 LayerNorm {e32:.2e}")
  if family == "constant":
    assert float((got[:, :n] - offset).abs().max()) <= 1e-6
  assert err <= TOL[prec] + 2 * e32, (err, e32)


@pytest.mark.parametrize("cluster", [1, 2, 4], indirect=True)
@pytest.mark.parametrize("prec", ["bf16x3", "bf16"])
@pytest.mark.parametrize("n,n_valid", [(512, 512), (512, 500), (256, 256), (256, 227)])
def test_layernorm_outputs_at_every_cluster_size(n, n_valid, prec, cluster):
  """All three outputs of one launch: out_y, out = residual + y, and (n_valid = 512 only) the
  operand image of out.  At cluster 4 the 6 tiles are one full cluster and one with two idle CTAs."""
  g = torch.Generator().manual_seed(n + n_valid)
  rows, k = 5 * 128 + 1, 256
  x, w, bias = _family("ordinary", rows, k, n_valid, n, g)
  scale, offset = _ln_params(n, g)
  res = torch.randn(rows, _canary_ld(n_valid), generator=g)
  rc, o = _layer(prec, x, w, bias, n, ln=(scale, offset), residual=res, out=True,
                 out_img=n_valid == 512)
  _native.check(rc, "layer")
  for name in ("out_y", "out"):
    _check_canary(o[name], n_valid)
  pre = x.double() @ w.double() + bias[:n_valid].double()
  sc, of = scale[:n_valid], offset[:n_valid]
  want = _ln64(pre, sc, of)
  r = res[:, :n_valid].double()
  e32 = _e32(pre, sc, of, want)
  err_y = _rel(o["out_y"][:, :n_valid].double(), want)
  err_o = _rel(o["out"][:, :n_valid].double(), want + r)
  print(f"\n({n}, {n_valid}) {prec} cluster {cluster}: out_y {err_y:.2e}  out {err_o:.2e}")
  assert err_y <= TOL[prec] + 2 * e32, err_y
  assert err_o <= TOL[prec] + 2 * _e32(pre, sc, of, want, r), err_o
  if n_valid == 512:
    # the image holds residual + y as bf16 hi + lo (2^-17 relative)
    assert _rel(_decode_image(o["img"], rows), o["out"][:, :512]) < 2 ** -16


@pytest.mark.parametrize("prec", ["bf16x3", "bf16", "fp32_simt"])
def test_swish_with_layernorm_is_refused(prec):
  """LN(swish(.)) in one layer is not a supported layer (no model layer needs it)."""
  g = torch.Generator().manual_seed(1)
  x, w, bias = _family("ordinary", 130, 64, 512, 512, g)
  rc, _ = _layer(prec, x, w, bias, 512, ln=_ln_params(512, g), act=True)
  assert rc == -1
  assert b"swish" in _native.lib().gcb_last_error()


def _chain_layer(cl, layer_w, bias, ln=None, act=False, keep=False):
  cl.w_packed, cl.bias = layer_w.data_ptr(), bias.data_ptr()
  if ln is not None:
    cl.ln_scale, cl.ln_offset = ln[0].data_ptr(), ln[1].data_ptr()
  cl.act, cl.keep = (_native.ACT_SWISH if act else _native.ACT_NONE), int(keep)
  for i in range(3):
    cl.seg_from[i] = -1


@pytest.mark.parametrize("kind", ["out_y", "residual", "residual_img"])
@pytest.mark.parametrize("family", ["ordinary"] + OUTLIERS)
def test_chain_layernorm_row_families(family, kind):
  """[swish layer (kept on chip) -> LayerNorm layer with the family in its bias] as one chain
  launch: bit-identical to the two layers launched one by one, and within the bound of fp64."""
  lib = _native.lib()
  prec = "bf16x3"
  g = torch.Generator().manual_seed(100 + OUTLIERS.index(family) if family in OUTLIERS else 99)
  rows = 128 * 9 + 7
  x = torch.randn(rows, 512, generator=g)
  w0 = torch.randn(512, 512, generator=g) / np.sqrt(512)
  b0 = 0.1 * torch.randn(512, generator=g)
  _, w1, b1 = _family(family, 1, 512, 512, 512, g)
  scale, offset = _ln_params(512, g)
  res = torch.randn(rows, 512, generator=g)
  (w0i, _), (w1i, _) = _packed(w0), _packed(w1)
  xd, b0d, b1d, sd, od, rd = (t.to(DEV) for t in (x, b0, b1, scale, offset, res))
  nbytes = lib.gcb_a_image_bytes(rows, 512)
  nan = lambda: torch.full((rows, 512), float("nan"), device=DEV)
  res_img = torch.zeros(nbytes, dtype=torch.uint8, device=DEV)
  _native.check(lib.gcb_rows_to_image(rd.data_ptr(), 512, 1, rows, 512, res_img.data_ptr(), _stream()),
                "rows_to_image")

  # layer by layer: hidden activation through an HBM operand image
  hidden = torch.zeros(nbytes, dtype=torch.uint8, device=DEV)
  y1, o1 = nan(), nan()
  d0 = _native.LayerDesc()
  d0.rows, d0.n, d0.n_valid, d0.nseg = rows, 512, 512, 1
  d0.seg[0].table, d0.seg[0].ld, d0.seg[0].k, d0.seg[0].k_valid, d0.seg[0].fan = xd.data_ptr(), 512, 512, 512, 1
  d0.w_packed, d0.bias, d0.act, d0.out_img = w0i.data_ptr(), b0d.data_ptr(), _native.ACT_SWISH, hidden.data_ptr()
  d0.precision = _native.PRECISIONS[prec]
  _native.check(lib.gcb_layer_forward(C.byref(d0), _stream()), "layer 0")
  d1 = _native.LayerDesc()
  d1.rows, d1.n, d1.n_valid, d1.nseg = rows, 512, 512, 1
  d1.seg[0].img, d1.seg[0].k = hidden.data_ptr(), 512
  d1.w_packed, d1.bias = w1i.data_ptr(), b1d.data_ptr()
  d1.ln_scale, d1.ln_offset = sd.data_ptr(), od.data_ptr()
  d1.out_y, d1.ld_out_y = y1.data_ptr(), 512
  if kind == "residual":
    d1.residual, d1.ld_res, d1.out, d1.ld_out = rd.data_ptr(), 512, o1.data_ptr(), 512
  d1.precision = _native.PRECISIONS[prec]
  _native.check(lib.gcb_layer_forward(C.byref(d1), _stream()), "layer 1")

  # one chain launch
  y2, o2 = nan(), nan()
  out_img = torch.zeros(nbytes, dtype=torch.uint8, device=DEV)
  scratch = torch.zeros(lib.gcb_chain_scratch_bytes(0, 1, 1, 1), dtype=torch.uint8, device=DEV)
  ch = _native.ChainDesc()
  ch.rows, ch.nlayers, ch.precision, ch.lag = rows, 2, _native.PRECISIONS[prec], 1
  ch.scratch, ch.scratch_bytes = scratch.data_ptr(), scratch.numel()
  l0, l1 = ch.layer[0], ch.layer[1]
  _chain_layer(l0, w0i, b0d, act=True, keep=True)
  l0.nseg = 1
  l0.seg[0].table, l0.seg[0].ld, l0.seg[0].k, l0.seg[0].k_valid, l0.seg[0].fan = xd.data_ptr(), 512, 512, 512, 1
  _chain_layer(l1, w1i, b1d, ln=(sd, od))
  l1.nseg, l1.seg_from[0], l1.seg[0].k = 1, 0, 512
  l1.out_y, l1.ld_out_y = y2.data_ptr(), 512
  if kind == "residual":
    l1.residual, l1.ld_res, l1.out, l1.ld_out = rd.data_ptr(), 512, o2.data_ptr(), 512
  elif kind == "residual_img":
    l1.residual_img, l1.out_img = res_img.data_ptr(), out_img.data_ptr()
  _native.check(lib.gcb_chain_forward(C.byref(ch), _stream()), "chain")
  torch.cuda.synchronize()

  assert torch.equal(y1, y2)
  h = x.double() @ w0.double() + b0.double()
  pre = (h * torch.sigmoid(h)) @ w1.double() + b1.double()
  want = _ln64(pre, scale, offset)
  e32 = _e32(pre, scale, offset, want)
  err = _rel(y2.cpu().double(), want)
  print(f"\n{family:>10} {kind:>12}: err {err:.2e}  fp32 LayerNorm {e32:.2e}")
  assert err <= TOL[prec] + 2 * e32, (err, e32)
  if kind == "residual":
    assert torch.equal(o1, o2)
    r = res.double()
    err_o = _rel(o2.cpu().double(), want + r)
    assert err_o <= TOL[prec] + 2 * _e32(pre, scale, offset, want, r), err_o
  elif kind == "residual_img":
    # the image holds residual (as the image held it) + y, as bf16 hi + lo (2^-17 relative)
    want_img = _decode_image(res_img, rows).double() + y2.cpu().double()
    assert _rel(_decode_image(out_img, rows).double(), want_img) < 2 ** -16


@pytest.mark.parametrize("cluster", [1, 4], indirect=True)
def test_unfused_step_at_cluster_size(cluster):
  """Every layer its own launch (fuse=False), so every layer runs at this cluster size."""
  g, params, x = _cases.small_case(c_in=31, n_out=23, msg_steps=2)
  ref = oracle_gnn.Oracle(params, torch.float64).forward(g.as_dict(), x).numpy()
  eng = engine.Engine(g, params, c_in=31, n_out=23, msg_steps=2, precision="bf16x3", fuse=False)
  xt = torch.as_tensor(x)
  y1 = eng.forward_features(xt).clone()
  y2 = eng.forward_features(xt).clone()
  assert torch.equal(y1, y2)
  y = y1.cpu().numpy()
  err = float(np.abs(y - ref).max() / np.abs(ref).max())
  print(f"\ncluster {cluster}: {err:.3e} vs fp64 oracle")
  assert err <= 1e-4
