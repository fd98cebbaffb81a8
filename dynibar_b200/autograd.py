"""Training backward (row f2): `torch.autograd.Function`s over the CUDA forward/backward kernels of every stage
of the path, so that `render_ray.render_rays_mono(..., is_train=True)` is differentiable end to end
(parameters of MotionMLP / DynibarDynamic / DynibarStatic, the source feature maps).

  * `composite`         raw2outputs (ibrnet/render_ray.py:214-330): gradients of rgb / rgb_static / rgb_dy / depth /
                        alpha_dy / weights_dy / weights_st / alpha / weights w.r.t. raw_dy, raw_st.
  * `project_gather`    Projector.compute_with_motions (ibrnet/projection.py:103-176): gradient of rgb_feat w.r.t.
                        the source feature maps and the motion-displaced points (ray_diff and mask are detached /
                        non-differentiable, as in the reference).

  * `motion_mlp`        MotionMLP.forward (ibrnet/mlp_network.py:605-618): gradients w.r.t. every parameter of the
                        module and w.r.t. the xyzt rows (fp32 GEMMs, csrc/motion_train.cu).

  * `net_dynamic` / `net_static`   DynibarDynamic.forward / DynibarStatic.forward (mlp_network.py:236-316,
                        :423-527) incl. the ray transformer: gradients w.r.t. every parameter, the gathered
                        rgb_feat and (dynamic) the sample points (csrc/nets_train.cu, fp32).
  * `composite_vanilla` raw2outputs_vanilla (render_ray.py:134-211).
                        The two compositors are also the evaluation path's: under no_grad only their forward runs.
  * `traj_combine`      compute_traj_pts and the displacements built from it (render_ray.py:361-369, :462-500).
  * `optical_flow`      compute_optical_flow (render_ray.py:333-358).

tests/test_backward_gpu.py and tests/test_train_gpu.py check them -- and the whole training forward/backward --
against torch autograd through the oracle's restatement of the same functions.
"""

from collections import OrderedDict

import torch

from dynibar_b200._lib import lib, ptr, f32c, check, stream, dev_of, Args


class _Composite(torch.autograd.Function):
  @staticmethod
  def forward(ctx, raw_dy, raw_st, z_vals, mask_dy, mask_st, min_dy, min_st):
    R, S = z_vals.shape
    dev = dev_of(z_vals)
    V_dy, V_st = mask_dy.shape[2], mask_st.shape[2]
    rays = torch.empty(R, 11, device=dev)
    samp = torch.empty(5, R, S, device=dev)
    rd, rs, zz = f32c(raw_dy), f32c(raw_st), f32c(z_vals)
    A = Args()
    with torch.cuda.device(dev):
      check(lib.dyn_composite(ptr(rd), ptr(rs), ptr(zz), A(mask_dy), V_dy, int(min_dy), A(mask_st), V_st, int(min_st),
                              R, S, ptr(rays), ptr(samp), stream()))
    ctx.save_for_backward(rd, rs, zz)
    ctx.mark_non_differentiable(rays[:, 10])
    return rays, samp

  @staticmethod
  def backward(ctx, g_rays, g_samp):
    rd, rs, zz = ctx.saved_tensors
    R, S = zz.shape
    g_dy, g_st = torch.empty_like(rd), torch.empty_like(rs)
    gr = f32c(g_rays) if g_rays is not None else torch.zeros(R, 11, device=zz.device)
    gs = f32c(g_samp) if g_samp is not None else None
    with torch.cuda.device(zz.device):
      check(lib.dyn_composite_backward(ptr(rd), ptr(rs), ptr(zz), ptr(gr), ptr(gs) if gs is not None else None,
                                       R, S, ptr(g_dy), ptr(g_st), stream()))
    return g_dy, g_st, None, None, None, None, None


def composite(raw_dy, raw_st, z_vals, mask_dy, mask_st, min_views_dy=1, min_views_st=1):
  """raw2outputs, differentiable w.r.t. raw_dy / raw_st -> the reference's 11-key dict.  mask_* [R,S,V(,1)]: a
  sample counts when more than min_views_* of its V views see it."""
  rays, samp = _Composite.apply(raw_dy, raw_st, z_vals, mask_dy, mask_st, min_views_dy, min_views_st)
  return OrderedDict([
      ("rgb", rays[:, 0:3]), ("rgb_static", rays[:, 3:6]), ("rgb_dy", rays[:, 6:9]),
      ("depth", rays[:, 9]), ("alpha_dy", samp[0]), ("weights_dy", samp[1]),
      ("weights_st", samp[2]), ("alpha", samp[3]), ("weights", samp[4]),
      ("mask", rays[:, 10].detach() > 0.5), ("z_vals", z_vals),
  ])


class _ProjectGather(torch.autograd.Function):
  @staticmethod
  def forward(ctx, xyz_st, xyz, featmaps, query_camera, train_imgs, train_cameras):
    from dynibar_b200.projection import project_gather
    rgb_feat, ray_diff, mask = project_gather(xyz_st, xyz, query_camera, train_imgs, train_cameras, featmaps)
    ctx.has_xyz = xyz is not None
    ctx.save_for_backward(f32c(xyz_st), f32c(xyz) if xyz is not None else f32c(xyz_st), f32c(featmaps),
                          f32c(train_imgs))
    ctx.cams = train_cameras.detach().float().cpu().contiguous()
    ctx.mark_non_differentiable(ray_diff, mask)
    return rgb_feat, ray_diff, mask

  @staticmethod
  def backward(ctx, g_feat, _g_rd, _g_mask):
    xyz_st, xyz, fm, imgs = ctx.saved_tensors
    R, S = xyz_st.shape[:2]
    _, V, H, W, _ = imgs.shape
    _, Cc, h, w = fm.shape
    need_maps, need_xyz = ctx.needs_input_grad[2], ctx.needs_input_grad[1] and ctx.has_xyz
    if not (need_maps or need_xyz):
      return None, None, None, None, None, None
    g_maps = torch.empty_like(fm) if need_maps else None
    g_xyz = torch.empty_like(xyz) if need_xyz else None
    gf = f32c(g_feat)
    with torch.cuda.device(fm.device):
      check(lib.dyn_project_gather_backward(ptr(xyz_st), ptr(xyz) if ctx.has_xyz else None, ptr(imgs),
                                            ctx.cams.data_ptr(), ptr(fm), ptr(gf),
                                            V, R, S, H, W, Cc, h, w,
                                            ptr(g_maps) if need_maps else None,
                                            ptr(g_xyz) if need_xyz else None, stream()))
    return None, g_xyz, g_maps, None, None, None


def project_gather(xyz_st, xyz, query_camera, train_imgs, train_cameras, featmaps):
  """Differentiable Projector.compute_with_motions -> (rgb_feat, ray_diff, mask)."""
  return _ProjectGather.apply(xyz_st, xyz, featmaps, query_camera, train_imgs, train_cameras)


class _MotionMLP(torch.autograd.Function):
  @staticmethod
  def forward(ctx, xyzt, module, prec, *params):
    from dynibar_b200 import weights
    dev = dev_of(xyzt)
    net = weights.packed_of(module, dev, level=1 if prec else 0)
    ctx.prec = prec
    x = f32c(xyzt.detach()).reshape(-1, 4)
    N = x.shape[0]
    out = torch.empty(N, 3 * net.num_basis, device=dev)
    nbytes = int(lib.dyn_motion_train_workspace_bytes(N))
    saved = torch.empty(max(nbytes, 16), dtype=torch.uint8, device=dev)
    with torch.cuda.device(dev):
      check(lib.dyn_motion_mlp_train_forward(net.handle, ptr(x), N, ptr(out), saved.data_ptr(), nbytes, prec,
                                             stream()))
    ctx.net, ctx.ws, ctx.nbytes, ctx.x = net, saved, nbytes, x
    ctx.in_shape = xyzt.shape
    ctx.shapes = [p.shape for p in params]
    return out.reshape(xyzt.shape[:-1] + (out.shape[-1],))

  @staticmethod
  def backward(ctx, g):
    net, x = ctx.net, ctx.x
    N = x.shape[0]
    gc = f32c(g).reshape(N, -1)
    d_params = torch.zeros(net.blob.numel(), device=x.device)
    d_x = torch.empty_like(x) if ctx.needs_input_grad[0] else None
    with torch.cuda.device(x.device):
      check(lib.dyn_motion_mlp_backward(net.handle, ptr(x), ptr(gc), N, ctx.ws.data_ptr(), ctx.nbytes,
                                        ptr(d_params), ptr(d_x) if d_x is not None else None, ctx.prec, stream()))
    return ((d_x.reshape(ctx.in_shape) if d_x is not None else None, None, None)
            + tuple(_split_param_grads(d_params, ctx.shapes)))


def _prec_code(precision):
  """None -> the library-wide setting of render_ray (`set_precision` / `precision_scope`)."""
  from dynibar_b200 import render_ray
  return render_ray._prec() if precision is None else render_ray._PREC[precision]


def motion_mlp(module, xyzt, precision=None):
  """Differentiable MotionMLP.forward on [...,4] rows; honours `sf_mag_div` like render_ray.motion_mlp_forward.
  precision "bf16": the products run on tcgen05 (bf16 operands, fp32 accumulation / master weights)."""
  from dynibar_b200 import render_ray, weights
  out = _MotionMLP.apply(xyzt, module, _prec_code(precision), *weights.de_parallel(module).parameters())
  return render_ray._sf_mag_div(module, out)


def _split_param_grads(d_params, shapes):
  """Flat blob gradient -> per-parameter tensors (state_dict order == parameters() order == the blob's order)."""
  grads, o = [], 0
  for shp in shapes:
    n = 1
    for d in shp:
      n *= d
    grads.append(d_params[o:o + n].reshape(shp))
    o += n
  assert o == d_params.numel()
  return grads


class _NetDynamic(torch.autograd.Function):
  @staticmethod
  def forward(ctx, pts, rgb_feat, ray_dir, mask, time, module, prec, *params):
    from dynibar_b200 import weights, _lib
    dev = dev_of(pts)
    net = weights.packed_of(module, dev, level=1 if prec else 0)
    ctx.prec = prec
    R, S, V = rgb_feat.shape[:3]
    p, f, rd, mk = f32c(pts), f32c(rgb_feat), f32c(ray_dir), f32c(mask)
    raw = torch.empty(R, S, 4, device=dev)
    nbytes = int(lib.dyn_net_train_workspace_bytes(_lib.NET_DYNAMIC, R, S, V))
    saved = torch.empty(max(nbytes, 16), dtype=torch.uint8, device=dev)
    with torch.cuda.device(dev):
      check(lib.dyn_net_dynamic_train_forward(net.handle, ptr(p), ptr(f), ptr(rd), ptr(mk), float(time), R, S, V,
                                              ptr(raw), saved.data_ptr(), nbytes, prec, stream()))
    ctx.net, ctx.ws, ctx.nbytes, ctx.p, ctx.mk, ctx.dims = net, saved, nbytes, p, mk, (R, S, V)
    ctx.shapes = [q.shape for q in params]
    return raw

  @staticmethod
  def backward(ctx, g_raw):
    from dynibar_b200 import _lib
    net, (R, S, V) = ctx.net, ctx.dims
    dev = ctx.p.device
    g = f32c(g_raw)
    d_params = torch.zeros(net.blob.numel(), device=dev)
    d_feat = torch.empty(R, S, V, 35, device=dev) if ctx.needs_input_grad[1] else None
    d_pts = torch.empty(R, S, 3, device=dev) if ctx.needs_input_grad[0] else None
    sbytes = int(lib.dyn_net_backward_scratch_bytes(_lib.NET_DYNAMIC, R, S, V))
    scratch = _lib.workspace.get(sbytes, dev, slot=2)
    with torch.cuda.device(dev):
      check(lib.dyn_net_dynamic_backward(net.handle, ptr(ctx.p), ptr(ctx.mk), R, S, V, ptr(g), ctx.ws.data_ptr(),
                                         ctx.nbytes, scratch.data_ptr(), sbytes, ptr(d_params),
                                         ptr(d_feat) if d_feat is not None else None,
                                         ptr(d_pts) if d_pts is not None else None, ctx.prec, stream()))
    ctx.ws = None
    return (d_pts, d_feat, None, None, None, None, None) + tuple(_split_param_grads(d_params, ctx.shapes))


def net_dynamic(module, pts, rgb_feat, ray_dir, mask, time, precision=None):
  """Differentiable DynibarDynamic.forward -> raw [R,S,4].  precision "fp32": SIMT products; "bf16": the large
  products on tcgen05 (bf16 operands, fp32 accumulation, master weights and gradients); glue always fp32."""
  from dynibar_b200 import weights
  m = weights.de_parallel(module)
  t = float(time.reshape(-1)[0]) if torch.is_tensor(time) else float(time)
  return _NetDynamic.apply(pts, rgb_feat, ray_dir, mask, t, module, _prec_code(precision), *m.parameters())


class _NetStatic(torch.autograd.Function):
  @staticmethod
  def forward(ctx, pts, ref_rays, src_rays, rgb_feat, ray_diff, mask, module, prec, *params):
    from dynibar_b200 import weights, _lib
    dev = dev_of(pts)
    net = weights.packed_of(module, dev, level=1 if prec else 0)
    ctx.prec = prec
    R, S, V = rgb_feat.shape[:3]
    f, rd, mk = f32c(rgb_feat), f32c(ray_diff), f32c(mask)
    raw = torch.empty(R, S, 4, device=dev)
    nbytes = int(lib.dyn_net_train_workspace_bytes(_lib.NET_STATIC, R, S, V))
    saved = torch.empty(max(nbytes, 16), dtype=torch.uint8, device=dev)
    A = Args()
    with torch.cuda.device(dev):
      check(lib.dyn_net_static_train_forward(net.handle, A(pts), A(ref_rays), A(src_rays), ptr(f), ptr(rd), ptr(mk),
                                             R, S, V, ptr(raw), saved.data_ptr(), nbytes, prec, stream()))
    ctx.net, ctx.ws, ctx.nbytes, ctx.f, ctx.rd, ctx.dims = net, saved, nbytes, f, rd, (R, S, V)
    ctx.shapes = [q.shape for q in params]
    return raw

  @staticmethod
  def backward(ctx, g_raw):
    from dynibar_b200 import _lib
    net, (R, S, V) = ctx.net, ctx.dims
    dev = ctx.f.device
    g = f32c(g_raw)
    d_params = torch.zeros(net.blob.numel(), device=dev)
    d_feat = torch.empty(R, S, V, 35, device=dev) if ctx.needs_input_grad[3] else None
    sbytes = int(lib.dyn_net_backward_scratch_bytes(_lib.NET_STATIC, R, S, V))
    scratch = _lib.workspace.get(sbytes, dev, slot=2)
    with torch.cuda.device(dev):
      check(lib.dyn_net_static_backward(net.handle, ptr(ctx.f), ptr(ctx.rd), R, S, V, ptr(g), ctx.ws.data_ptr(),
                                        ctx.nbytes, scratch.data_ptr(), sbytes, ptr(d_params),
                                        ptr(d_feat) if d_feat is not None else None, ctx.prec, stream()))
    ctx.ws = None
    return (None, None, None, d_feat, None, None, None, None) + tuple(_split_param_grads(d_params, ctx.shapes))


def net_static(module, pts, ref_rays, src_rays, rgb_feat, ray_diff, mask, precision=None):
  """Differentiable DynibarStatic.forward -> raw [R,S,4] (precision: see net_dynamic)."""
  from dynibar_b200 import weights
  m = weights.de_parallel(module)
  return _NetStatic.apply(pts, ref_rays, src_rays, rgb_feat, ray_diff, mask, module, _prec_code(precision),
                          *m.parameters())


class _CompositeVanilla(torch.autograd.Function):
  @staticmethod
  def forward(ctx, raw, z_vals, mask, min_views):
    R, S = z_vals.shape
    dev = dev_of(z_vals)
    V = mask.shape[2]
    rays = torch.empty(R, 5, device=dev)
    samp = torch.empty(2, R, S, device=dev)
    rw, zz = f32c(raw), f32c(z_vals)
    with torch.cuda.device(dev):
      check(lib.dyn_composite_vanilla(ptr(rw), ptr(zz), ptr(f32c(mask)), V, int(min_views), R, S, ptr(rays),
                                      ptr(samp), stream()))
    ctx.save_for_backward(rw, zz)
    ctx.mark_non_differentiable(rays[:, 4])
    return rays, samp

  @staticmethod
  def backward(ctx, g_rays, g_samp):
    rw, zz = ctx.saved_tensors
    R, S = zz.shape
    g_raw = torch.empty_like(rw)
    gr = f32c(g_rays) if g_rays is not None else torch.zeros(R, 5, device=zz.device)
    gs = f32c(g_samp) if g_samp is not None else None
    with torch.cuda.device(zz.device):
      check(lib.dyn_composite_vanilla_backward(ptr(rw), ptr(zz), ptr(gr), ptr(gs) if gs is not None else None,
                                               R, S, ptr(g_raw), stream()))
    return g_raw, None, None, None


def composite_vanilla(raw, z_vals, mask, min_views=1):
  """raw2outputs_vanilla, differentiable w.r.t. raw -> the reference's 6-key dict (mask: see composite)."""
  rays, samp = _CompositeVanilla.apply(raw, z_vals, mask, min_views)
  return OrderedDict([
      ("rgb", rays[:, 0:3]), ("depth", rays[:, 3]), ("weights", samp[0]),
      ("mask", rays[:, 4].detach() > 0.5), ("alpha", samp[1]), ("z_vals", z_vals),
  ])


class _TrajCombine(torch.autograd.Function):
  @staticmethod
  def forward(ctx, coeff, D, base):
    dev = dev_of(coeff)
    R, S = coeff.shape[:2]
    n, nb = D.shape
    c, Dd = f32c(coeff), f32c(D)
    b = f32c(base) if base is not None else None
    out = torch.empty(n, R, S, 3, device=dev)
    with torch.cuda.device(dev):
      check(lib.dyn_traj_combine(ptr(c), ptr(Dd), ptr(b) if b is not None else None, n, nb, R * S, ptr(out),
                                 stream()))
    ctx.D, ctx.dims = Dd, (n, nb, R, S)
    return out

  @staticmethod
  def backward(ctx, g):
    n, nb, R, S = ctx.dims
    go = f32c(g)
    need_c, need_b = ctx.needs_input_grad[0], ctx.needs_input_grad[2]
    if not (need_c or need_b):
      return None, None, None
    g_c = torch.empty(R, S, 3 * nb, device=go.device) if need_c else None
    g_b = torch.empty(R, S, 3, device=go.device) if need_b else None
    with torch.cuda.device(go.device):
      check(lib.dyn_traj_combine_backward(ptr(go), ptr(ctx.D), n, nb, R * S, ptr(g_c) if need_c else None,
                                          ptr(g_b) if need_b else None, stream()))
    return g_c, None, g_b


def traj_combine(coeff, D, base=None):
  """out[i] = (base or 0) + sum_k coeff[..., axis * nb + k] * D[i, k] -> [n,R,S,3]; D [n,nb] on the device."""
  return _TrajCombine.apply(coeff, D, base)


class _OpticalFlow(torch.autograd.Function):
  @staticmethod
  def forward(ctx, weights, pts_seq, src_cameras, uv_grid):
    dev = dev_of(weights)
    R, S = weights.shape
    n = pts_seq.shape[0]
    w, ps = f32c(weights), f32c(pts_seq)
    cams = src_cameras.detach().float().cpu().contiguous().reshape(-1, 34)[:n].contiguous()
    flows = torch.empty(n, R, 2, device=dev)
    A = Args()
    with torch.cuda.device(dev):
      check(lib.dyn_flow_sceneflow(ptr(w), ptr(ps), cams.data_ptr(), A(uv_grid), None, None, 0, 1, 0, 0, n, R, S,
                                   ptr(flows), None, stream()))
    ctx.save_for_backward(w, ps)
    ctx.cams = cams
    return flows

  @staticmethod
  def backward(ctx, g):
    w, ps = ctx.saved_tensors
    R, S = w.shape
    n = ps.shape[0]
    gf = f32c(g)
    g_w = torch.empty_like(w) if ctx.needs_input_grad[0] else None
    g_p = torch.empty_like(ps) if ctx.needs_input_grad[1] else None
    if g_w is None and g_p is None:
      return None, None, None, None
    with torch.cuda.device(w.device):
      check(lib.dyn_flow_backward(ptr(w), ptr(ps), ctx.cams.data_ptr(), ptr(gf), n, R, S,
                                  ptr(g_w) if g_w is not None else None, ptr(g_p) if g_p is not None else None,
                                  stream()))
    return g_w, g_p, None, None


def optical_flow(weights, pts_seq, src_cameras, uv_grid):
  """Differentiable compute_optical_flow -> [n,R,2] for the n views of pts_seq."""
  return _OpticalFlow.apply(weights, pts_seq, src_cameras, uv_grid)
