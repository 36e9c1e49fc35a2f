"""Parity of the fused layer kernel (through the C ABI) against a plain PyTorch
fp32/fp64 reference of the same op: gathers, fan-in sums, zero padding, bias,
swish, LayerNorm, residual, both outputs, ragged row counts, both output widths."""
import ctypes as C

import numpy as np
import pytest
import torch

from _cases import cluster  # noqa: F401  (fixture)
from graphcast_b200 import _native

pytestmark = pytest.mark.gpu

TOL = {"bf16x3": 3e-5, "bf16": 2e-2, "fp32_simt": 5e-6}


def _pack(lib, w, k_pad, n_pad, dev):
  img = np.empty(lib.gcb_packed_weight_bytes(k_pad, n_pad), np.uint8)
  wp = np.zeros((k_pad, n_pad), np.float32)
  wp[:w.shape[0], :w.shape[1]] = w
  assert lib.gcb_pack_weight_host(wp.ctypes.data, k_pad, n_pad, k_pad, n_pad, img.ctypes.data) == 0
  return torch.as_tensor(img).to(dev), torch.as_tensor(wp).to(dev)


def _run_case(prec, rows, segs, n, n_valid, act, ln, residual, out_y, seed=0):
  """segs: list of (table_rows, k_valid, k_pad, use_idx, fan)."""
  lib = _native.lib()
  dev = torch.device("cuda:0")
  g = torch.Generator().manual_seed(seed)
  d = _native.LayerDesc()
  d.rows, d.n, d.n_valid, d.nseg = rows, n, n_valid, len(segs)
  keep, cols, w_rows = [], [], []
  for i, (trows, kv, kp, use_idx, fan) in enumerate(segs):
    ld = kv + 4                                   # row stride wider than the data
    table = torch.randn(trows * fan, ld, generator=g)
    idx = torch.randint(0, trows, (rows,), generator=g, dtype=torch.int32) if use_idx else None
    tdev = table.to(dev); keep.append(tdev)
    d.seg[i].table, d.seg[i].ld, d.seg[i].k, d.seg[i].k_valid, d.seg[i].fan = tdev.data_ptr(), ld, kp, kv, fan
    if idx is not None:
      idev = idx.to(dev); keep.append(idev); d.seg[i].idx = idev.data_ptr()
    src = idx.long() if idx is not None else torch.arange(rows)
    assert trows >= rows or use_idx
    gathered = table.view(trows, fan, ld)[src][:, :, :kv].double().sum(1)
    cols.append(gathered)
    w_rows.append((kv, kp))
  k_real = sum(kv for kv, _ in w_rows)
  w = torch.randn(k_real, n_valid, generator=g) / np.sqrt(k_real)
  # lay weight rows out with per-segment padding
  k_pad = sum(kp for _, kp in w_rows)
  wp = np.zeros((k_pad, n_valid), np.float32)
  s = dst = 0
  for kv, kp in w_rows:
    wp[dst:dst + kv] = w[s:s + kv].numpy(); s += kv; dst += kp
  img, wf = _pack(lib, wp, k_pad, n, dev)
  bias = torch.randn(n, generator=g) * 0.1
  scale = 1 + 0.1 * torch.randn(n, generator=g)
  offset = 0.1 * torch.randn(n, generator=g)
  bdev, sdev, odev = bias.to(dev), scale.to(dev), offset.to(dev)
  d.w_packed, d.w_f32, d.bias = img.data_ptr(), wf.data_ptr(), bdev.data_ptr()
  if ln:
    d.ln_scale, d.ln_offset = sdev.data_ptr(), odev.data_ptr()
  d.act = 1 if act else 0
  ld_out = n_valid + (4 - n_valid % 4) % 4 + 4
  res = torch.randn(rows, ld_out, generator=g)
  rdev = res.to(dev)
  out = torch.full((rows, ld_out), float("nan"), device=dev)
  outy = torch.full((rows, 512), float("nan"), device=dev)
  if residual:
    d.residual, d.ld_res = rdev.data_ptr(), ld_out
  d.out, d.ld_out = out.data_ptr(), ld_out
  if out_y:
    d.out_y, d.ld_out_y = outy.data_ptr(), 512
  d.precision = _native.PRECISIONS[prec]
  _native.check(lib.gcb_layer_forward(C.byref(d), torch.cuda.current_stream().cuda_stream), "layer")
  torch.cuda.synchronize()
  # reference in float64
  z = torch.cat(cols, 1)
  y = z @ w.double() + bias[:n_valid].double()
  if act:
    y = y * torch.sigmoid(y)
  if ln:
    y = torch.nn.functional.layer_norm(y, (n_valid,), scale[:n_valid].double(), offset[:n_valid].double(), 1e-5)
  want = y + (res[:, :n_valid].double() if residual else 0)
  got = out[:, :n_valid].cpu().double()
  denom = want.abs().max()
  err = float((got - want).abs().max() / denom)
  assert torch.isnan(out[:, n_valid:]).all(), "kernel wrote beyond n_valid"
  if out_y:
    erry = float((outy[:, :n_valid].cpu().double() - y).abs().max() / y.abs().max())
    err = max(err, erry)
  return err


@pytest.mark.parametrize("prec", ["fp32_simt", "bf16x3", "bf16"])
def test_edge_block_three_gathered_segments(prec):
  err = _run_case(prec, rows=1000, segs=[(1000, 512, 512, False, 1), (300, 512, 512, True, 1),
                                         (77, 512, 512, True, 1)],
                  n=512, n_valid=512, act=True, ln=False, residual=False, out_y=False)
  assert err < TOL[prec], err


@pytest.mark.parametrize("prec", ["fp32_simt", "bf16x3", "bf16"])
def test_layernorm_residual_and_message_output(prec):
  err = _run_case(prec, rows=333, segs=[(333, 512, 512, False, 1)], n=512, n_valid=512,
                  act=False, ln=True, residual=True, out_y=True)
  assert err < TOL[prec], err


@pytest.mark.parametrize("prec", ["fp32_simt", "bf16x3"])
def test_padded_inputs_and_narrow_output(prec):
  # K=474 real columns padded to 480 (first encoder layer), K=4 padded to 16 (edge embed)
  err = _run_case(prec, rows=257, segs=[(257, 476, 480, False, 1)], n=512, n_valid=512,
                  act=True, ln=False, residual=False, out_y=False)
  assert err < TOL[prec], err
  err = _run_case(prec, rows=129, segs=[(129, 4, 16, False, 1)], n=512, n_valid=512,
                  act=True, ln=False, residual=False, out_y=False)
  assert err < TOL[prec], err
  # decoder output layer: 227 of 256 columns, no LayerNorm
  err = _run_case(prec, rows=500, segs=[(500, 512, 512, False, 1)], n=256, n_valid=227,
                  act=False, ln=False, residual=False, out_y=False)
  assert err < TOL[prec], err


@pytest.mark.parametrize("prec", ["fp32_simt", "bf16x3"])
def test_fan_in_three_segment(prec):
  err = _run_case(prec, rows=700, segs=[(700, 512, 512, False, 1), (700, 512, 512, False, 3)],
                  n=512, n_valid=512, act=True, ln=False, residual=False, out_y=False)
  assert err < TOL[prec], err


# 5 * 128 + 1 rows at a cluster of 4: one full cluster, then one with two idle CTAs
RAGGED_ROWS = [1, 127, 128, 129, 5 * 128 + 1, 148 * 128 + 5]


@pytest.mark.parametrize("rows", RAGGED_ROWS)
def test_ragged_row_counts(rows):
  err = _run_case("bf16x3", rows=rows, segs=[(max(rows, 1), 512, 512, False, 1)], n=512,
                  n_valid=512, act=False, ln=True, residual=True, out_y=False)
  assert err < TOL["bf16x3"], err


@pytest.mark.parametrize("prec", ["fp32_simt", "bf16x3", "bf16"])
@pytest.mark.parametrize("rows", [700, 128 * 148 + 77])
def test_gathered_pre_activation_addends(prec, rows):
  """Split first edge-MLP layer: swish(e @ W_e + b + P_s[snd] + P_r[rcv])."""
  lib = _native.lib()
  dev = torch.device("cuda:0")
  g = torch.Generator().manual_seed(3)
  e = torch.randn(rows, 512, generator=g)
  ps, pr = torch.randn(301, 512, generator=g), torch.randn(97, 516, generator=g)
  snd = torch.randint(0, 301, (rows,), generator=g, dtype=torch.int32)
  rcv = torch.randint(0, 97, (rows,), generator=g, dtype=torch.int32)
  w = torch.randn(512, 512, generator=g) / np.sqrt(512)
  bias = 0.1 * torch.randn(512, generator=g)
  img, wf = _pack(lib, w.numpy(), 512, 512, dev)
  ed, psd, prd, sd, rd, bd = (t.to(dev) for t in (e, ps, pr, snd, rcv, bias))
  out = torch.empty(rows, 512, device=dev)
  d = _native.LayerDesc()
  d.rows, d.n, d.n_valid, d.nseg = rows, 512, 512, 1
  d.seg[0].table, d.seg[0].ld, d.seg[0].k, d.seg[0].k_valid, d.seg[0].fan = ed.data_ptr(), 512, 512, 512, 1
  d.w_packed, d.w_f32, d.bias, d.act = img.data_ptr(), wf.data_ptr(), bd.data_ptr(), 1
  d.out, d.ld_out = out.data_ptr(), 512
  d.precision = _native.PRECISIONS[prec]
  d.n_pre_add = 2
  d.pre_add[0].table, d.pre_add[0].idx, d.pre_add[0].ld = psd.data_ptr(), sd.data_ptr(), 512
  d.pre_add[1].table, d.pre_add[1].idx, d.pre_add[1].ld = prd.data_ptr(), rd.data_ptr(), 516
  _native.check(lib.gcb_layer_forward(C.byref(d), torch.cuda.current_stream().cuda_stream), "layer")
  torch.cuda.synchronize()
  y = e.double() @ w.double() + bias.double() + ps.double()[snd.long()] + pr.double()[rcv.long(), :512]
  want = y * torch.sigmoid(y)
  err = float((out.cpu().double() - want).abs().max() / want.abs().max())
  assert err < TOL[prec], err
  # LayerNorm + pre_add is rejected
  d.ln_scale, d.ln_offset = bd.data_ptr(), bd.data_ptr()
  assert lib.gcb_layer_forward(C.byref(d), None) == -1


@pytest.mark.parametrize("prec", ["fp32_simt", "bf16x3", "bf16"])
@pytest.mark.parametrize("rows", [1, 333, 128 * 148 * 2 + 5])
def test_operand_image_chain(prec, rows):
  """Two-layer MLP with the hidden activations handed over as an operand image:
  layer 0 writes out_img, layer 1 reads a_img (TMA-fed A operand, no gather warps)."""
  lib = _native.lib()
  dev = torch.device("cuda:0")
  g = torch.Generator().manual_seed(5)
  x = torch.randn(rows, 512, generator=g)
  w0 = torch.randn(512, 512, generator=g) / np.sqrt(512)
  w1 = torch.randn(512, 512, generator=g) / np.sqrt(512)
  b0, b1 = 0.1 * torch.randn(512, generator=g), 0.1 * torch.randn(512, generator=g)
  sc, of = 1 + 0.1 * torch.randn(512, generator=g), 0.1 * torch.randn(512, generator=g)
  img0, wf0 = _pack(lib, w0.numpy(), 512, 512, dev)
  img1, wf1 = _pack(lib, w1.numpy(), 512, 512, dev)
  xd, b0d, b1d, scd, ofd = (t.to(dev) for t in (x, b0, b1, sc, of))
  nbytes = lib.gcb_a_image_bytes(rows, 512)
  assert nbytes == ((rows + 127) // 128) * 32 * 8448
  himg = torch.zeros(nbytes, dtype=torch.uint8, device=dev)
  out = torch.empty(rows, 512, device=dev)
  st = torch.cuda.current_stream().cuda_stream
  d = _native.LayerDesc()
  d.rows, d.n, d.n_valid, d.nseg = rows, 512, 512, 1
  d.seg[0].table, d.seg[0].ld, d.seg[0].k, d.seg[0].k_valid, d.seg[0].fan = xd.data_ptr(), 512, 512, 512, 1
  d.w_packed, d.w_f32, d.bias, d.act = img0.data_ptr(), wf0.data_ptr(), b0d.data_ptr(), 1
  d.out_img = himg.data_ptr()
  d.precision = _native.PRECISIONS[prec]
  _native.check(lib.gcb_layer_forward(C.byref(d), st), "layer0")
  d1 = _native.LayerDesc()
  d1.rows, d1.n, d1.n_valid, d1.nseg = rows, 512, 512, 1
  d1.seg[0].img, d1.seg[0].k = himg.data_ptr(), 512
  d1.w_packed, d1.w_f32, d1.bias = img1.data_ptr(), wf1.data_ptr(), b1d.data_ptr()
  d1.ln_scale, d1.ln_offset = scd.data_ptr(), ofd.data_ptr()
  d1.out, d1.ld_out = out.data_ptr(), 512
  d1.precision = _native.PRECISIONS[prec]
  _native.check(lib.gcb_layer_forward(C.byref(d1), st), "layer1")
  torch.cuda.synchronize()
  h = x.double() @ w0.double() + b0.double()
  h = h * torch.sigmoid(h)
  y = torch.nn.functional.layer_norm(h @ w1.double() + b1.double(), (512,), sc.double(), of.double(), 1e-5)
  err = float((out.cpu().double() - y).abs().max() / y.abs().max())
  assert err < 2 * TOL[prec], err


@pytest.mark.parametrize("prec", ["fp32_simt", "bf16x3"])
def test_mixed_image_and_gathered_segments_with_residual_image(prec):
  """[image segment | gathered fp32 segment], LayerNorm + residual, result delivered as
  fp32 AND as an operand image (which must include the residual)."""
  lib = _native.lib()
  dev = torch.device("cuda:0")
  rows = 1000
  g = torch.Generator().manual_seed(9)
  a0 = torch.randn(rows, 512, generator=g)
  tab = torch.randn(222, 512, generator=g)
  idx = torch.randint(0, 222, (rows,), generator=g, dtype=torch.int32)
  w = torch.randn(1024, 512, generator=g) / np.sqrt(1024)
  bias, sc, of = 0.1 * torch.randn(512, generator=g), 1 + 0.1 * torch.randn(512, generator=g), 0.1 * torch.randn(512, generator=g)
  res = torch.randn(rows, 512, generator=g)
  img, wf = _pack(lib, w.numpy(), 1024, 512, dev)
  a0d, tabd, idxd, bd, scd, ofd, resd = (t.to(dev) for t in (a0, tab, idx, bias, sc, of, res))
  st = torch.cuda.current_stream().cuda_stream
  a0img = torch.zeros(lib.gcb_a_image_bytes(rows, 512), dtype=torch.uint8, device=dev)
  _native.check(lib.gcb_rows_to_image(a0d.data_ptr(), 512, 1, rows, 512, a0img.data_ptr(), st), "to_image")
  out = torch.empty(rows, 512, device=dev)
  oimg = torch.zeros(lib.gcb_a_image_bytes(rows, 512), dtype=torch.uint8, device=dev)
  d = _native.LayerDesc()
  d.rows, d.n, d.n_valid, d.nseg = rows, 512, 512, 2
  d.seg[0].img, d.seg[0].k = a0img.data_ptr(), 512
  d.seg[1].table, d.seg[1].idx, d.seg[1].ld, d.seg[1].k, d.seg[1].k_valid, d.seg[1].fan = \
      tabd.data_ptr(), idxd.data_ptr(), 512, 512, 512, 1
  d.w_packed, d.w_f32, d.bias = img.data_ptr(), wf.data_ptr(), bd.data_ptr()
  d.ln_scale, d.ln_offset = scd.data_ptr(), ofd.data_ptr()
  d.residual, d.ld_res, d.out, d.ld_out, d.out_img = resd.data_ptr(), 512, out.data_ptr(), 512, oimg.data_ptr()
  d.precision = _native.PRECISIONS[prec]
  _native.check(lib.gcb_layer_forward(C.byref(d), st), "layer")
  torch.cuda.synchronize()
  z = torch.cat([a0.double(), tab.double()[idx.long()]], 1)
  y = torch.nn.functional.layer_norm(z @ w.double() + bias.double(), (512,), sc.double(), of.double(), 1e-5)
  want = y + res.double()
  assert float((out.cpu().double() - want).abs().max() / want.abs().max()) < 2 * TOL[prec]
  # decode the output image and compare with the fp32 output (bf16 hi+lo ~ 2^-17 relative)
  blocks = oimg.cpu().numpy().view(np.uint16).reshape(-1, 32, 2, 2112)   # tile, kstep, hi|lo, halfwords
  def part(p):
    x = blocks[:, :, p, :].astype(np.uint32) << 16
    x = x.view(np.float32).reshape(-1, 32, 2, 1056)[..., :1024].reshape(-1, 32, 2, 128, 8)
    return x.transpose(0, 3, 1, 2, 4).reshape(-1, 512)                   # [tile*128, 512]
  dec = (part(0) + part(1))[:rows]
  np.testing.assert_allclose(dec, out.cpu().numpy(), rtol=2e-5, atol=2e-5)


def test_rows_to_image_fan_in():
  lib = _native.lib()
  dev = torch.device("cuda:0")
  rows, fan, k = 301, 3, 512
  src = torch.randn(rows * fan, 516, device=dev)
  img = torch.zeros(lib.gcb_a_image_bytes(rows, k), dtype=torch.uint8, device=dev)
  _native.check(lib.gcb_rows_to_image(src.data_ptr(), 516, fan, rows, k, img.data_ptr(),
                                      torch.cuda.current_stream().cuda_stream), "to_image")
  torch.cuda.synchronize()
  blocks = img.cpu().numpy().view(np.uint16).reshape(-1, 32, 2, 2112)
  def part(p):
    x = blocks[:, :, p, :].astype(np.uint32) << 16
    x = x.view(np.float32).reshape(-1, 32, 2, 1056)[..., :1024].reshape(-1, 32, 2, 128, 8)
    return x.transpose(0, 3, 1, 2, 4).reshape(-1, 512)
  dec = part(0) + part(1)
  want = src[:, :k].view(rows, fan, k).sum(1).cpu().numpy()
  np.testing.assert_allclose(dec[:rows], want, rtol=2e-5, atol=2e-5)
  assert np.all(dec[rows:] == 0)


def test_zero_rows_is_a_noop():
  lib = _native.lib()
  d = _native.LayerDesc()
  t = torch.zeros(16, 16, device="cuda:0")
  d.rows, d.n, d.n_valid, d.nseg = 0, 512, 512, 1
  d.seg[0].table, d.seg[0].ld, d.seg[0].k, d.seg[0].k_valid, d.seg[0].fan = t.data_ptr(), 16, 16, 16, 1
  d.w_packed, d.bias, d.out, d.ld_out = t.data_ptr(), t.data_ptr(), t.data_ptr(), 512
  assert lib.gcb_layer_forward(C.byref(d), None) == 0


def test_tensor_path_matches_simt_arm_selftest():
  lib = _native.lib()
  for prec, tol in (("bf16x3", 3e-5), ("bf16", 2e-2)):
    err = C.c_float(-1)
    assert lib.gcb_selftest_layer(3000, 1024, 512, _native.PRECISIONS[prec], C.byref(err)) == 0
    assert 0 <= err.value < tol


# The tests above run at the library's default cluster size of 2 (the N-split schedule for
# n = 512).  Clusters of 1 and 4 take the unsplit schedule: each CTA owns its tiles and runs
# both 256-column units, the weight stream is multicast to 4 CTAs, and some clusters have
# idle CTAs.  The fp32 CUDA-core arm has no clusters, so only the tensor-core precisions repeat.
@pytest.mark.parametrize("cluster", [1, 4], indirect=True)
@pytest.mark.parametrize("rows", RAGGED_ROWS)
def test_ragged_row_counts_at_cluster_size(rows, cluster):
  test_ragged_row_counts(rows)


@pytest.mark.parametrize("cluster", [1, 4], indirect=True)
def test_padded_inputs_and_narrow_output_at_cluster_size(cluster):
  test_padded_inputs_and_narrow_output("bf16x3")


@pytest.mark.parametrize("cluster", [1, 4], indirect=True)
@pytest.mark.parametrize("prec", ["bf16x3", "bf16"])
@pytest.mark.parametrize("rows", [700, 128 * 148 + 77])
def test_gathered_pre_activation_addends_at_cluster_size(prec, rows, cluster):
  test_gathered_pre_activation_addends(prec, rows)


@pytest.mark.parametrize("cluster", [1, 4], indirect=True)
@pytest.mark.parametrize("prec", ["bf16x3", "bf16"])
@pytest.mark.parametrize("rows", [1, 333, 128 * 148 * 2 + 5])
def test_operand_image_chain_at_cluster_size(prec, rows, cluster):
  test_operand_image_chain(prec, rows)
