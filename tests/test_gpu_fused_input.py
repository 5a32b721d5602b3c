"""The 16-bit network input `x` written by the fused kernels, channel by channel, against the CPU oracle.

Three writers fill `x` (include/mpx.h): mpx_render_crop_fused (single-view samples: the whole pixel vector
[crop rgb(d) | render rgb, normals(, depth) | zero pad]), and mpx_roi_align_fused followed by mpx_raster_render_fused
(multi-view samples: the crop in channels 0..c_in-1, view slot v at ch_offset + v * ch_per_view).  The reference input is
built from the oracle alone -- RefRenderer, lib3d_ref.crop_images, lib3d_ref.normalize_depth -- concatenated in the
reference's order and converted to the 16-bit type as the kernels convert (fp16: clamped to +-65504 first, which is what
the saturating conversion does).  Both sides get the same fp32 poses, intrinsics, boxes, image indices and
depth-normalisation z, so no geometry rounding enters the comparison.

Bounds:
  * render channels (rgb, normals, normalised render depth): equal.  The rasteriser is bit-exact against the oracle for
    identical inputs, depth_norm divides with the IEEE quotient as torch does on the CPU, and a saturating conversion
    equals clamp-then-convert;
  * crop rgb: |got - want| <= 1 ulp of the 16-bit type at |want| plus the fp32 roi_align bound of
    tests/test_gpu_kernels.py (atol 2e-5, rtol 1e-5: fma contraction moves sample coordinates by an ulp);
  * crop depth: the same with atol 2e-4 (the depth map has steep gradients) scaled by the normalisation's slope, except
    where the 0.99 validity threshold flips: that fraction stays below 1e-3;
  * NaN: at the same positions on both sides;
  * channels a writer does not own: `x` is prefilled with a sentinel; the fused crop overwrites all c_pad channels (the pad
    reads +0), the other two writers leave every channel outside their slots bit for bit as it was.
"""
import pytest
import torch

from megapose6d_b200 import _abi, lib3d, load_model, procedural
from megapose6d_b200.renderer import DEPTH_NORM_SHIFT, RASTER_POINT_LIGHTS, BatchRenderer
from oracle import lib3d_ref as L
from oracle import pipeline_ref
from tests import helpers
from tests import test_gpu_variants as variants

pytestmark = pytest.mark.gpu
DEV = "cuda"
ACT = _abi.act_dtype() if torch.cuda.is_available() else torch.float16  # the library's 16-bit type
KIND_NAMES = {0: "tCR_scale_clamp_center", 1: "tCR_scale", 2: "tCR_center_clamp", 3: "none"}
SENTINEL = -3.140625  # exact in fp16 and bf16
N_VIEWS = 54          # views rendered per size (27 views x 2 samples is the largest case)
N_SAMPLES = 40
PATHS = {"scatter": (7, 18), "strips": (2, 18), "tiled": (7, 40), "untiled": (3, 40)}  # raster mode, views
SIZES = {"224x224": (224, 224), "64x96": (64, 96), "64x968": (64, 968)}  # 64x968: h + w > 1024, no collapsed crop tables


# ------------------------------------------------------------------------------------------------------------------------
# inputs (identical fp32 tensors for both sides) and the oracle, computed once per size
# ------------------------------------------------------------------------------------------------------------------------
def _poses(n):
    """Poses of tests/test_gpu_kernels.py: test_raster_big_batch_bit_exact_vs_oracle: near plane, out of frustum, NaN."""
    TCO = torch.from_numpy(procedural.random_poses(n, 121, z_range=(0.25, 0.9))).float()
    TCO[3, 2, 3] = 0.12
    TCO[4, 0, 3] = 0.35
    TCO[7, 1, 1] = float("nan")
    TCO[9, 2, 3] = 0.06   # straddles the near plane
    TCO[11, 2, 3] = 0.02  # the eye inside the mesh
    return TCO


def _boxes(n, b):
    """One box kind per sample: inside, partly outside, minified (bins > 2.67 px: uncollapsed roi_align), sub-pixel,
    image index out of range (the crop must be zero)."""
    kinds = torch.tensor([[100.0, 80, 420, 320], [-40, -30, 200, 150], [-100, -100, 800, 700], [300, 200, 300.5, 200.2],
                          [120, 90, 400, 330]])
    i = torch.arange(n)
    boxes = kinds[i % 5] + (i // 5).float().unsqueeze(1) * torch.tensor([3.25, -2.5, 1.75, 4.0])
    im_idx = (i % 2).to(torch.int32)
    im_idx[i % 5 == 4] = torch.where((i[i % 5 == 4] // 5) % 2 == 0, b, -1).to(torch.int32)
    return boxes, im_idx


def _K(n, h, w):
    f = 1000.0 * h / 224
    K = torch.tensor([[f, 0, w / 2], [0, f, h / 2], [0, 0, 1]]).repeat(n, 1, 1)
    K[5] = torch.tensor([[0.3 * f, 0, w / 2 - 9.7], [0, 0.31 * f, h / 2 - 1.1], [0, 0, 1]])
    return K


class _Inputs:
    def __init__(self):
        self.ds, images, _ = helpers.make_scene(3, seed=11, with_depth=True)
        self.images = torch.cat((images, torch.flip(images, dims=[-1])))  # two frames: im_idx matters
        self.b = self.images.shape[0]
        self.rm = helpers.ref_meshes_from_dataset(self.ds)
        self.renderer = BatchRenderer(object_dataset=self.ds)
        self.labels = [self.ds[i % 3].label for i in range(N_VIEWS)]
        self.lab = self.renderer.mesh_db.label_ids(self.labels, DEV)
        self.TCO = _poses(N_VIEWS)
        self.boxes, self.im_idx = _boxes(N_SAMPLES, self.b)
        self.z = torch.from_numpy(procedural.random_poses(N_SAMPLES, 5, z_range=(0.4, 0.9))[:, 2, 3]).float()
        self.nhwc4 = lib3d.image_to_nhwc4(self.images.cuda())
        self._renders, self._crops = {}, {}

    def K(self, size):
        return _K(N_VIEWS, *size)

    def renders(self, size):
        """Oracle renders of all N_VIEWS views: rgb under ambient and under point lights, normals, depth."""
        if size not in self._renders:
            rr = pipeline_ref.RefRenderer(self.rm)
            amb = rr.render(self.labels, self.TCO, self.K(size), None, size, render_depth=True, render_normals=True)
            pt = rr.render(self.labels, self.TCO, self.K(size), None, size, point_lights=True)
            self._renders[size] = dict(rgb_amb=amb["rgbs"], rgb_pt=pt["rgbs"], normals=amb["normals"], depth=amb["depths"])
        return self._renders[size]

    def crops(self, size, n, c_in):
        """Oracle crops (fp32, depth masked, not normalised) of samples 0..n-1; an out-of-range image index crops zeros.
        roi_align treats channels independently: the rgb of the 4-channel crop is the 3-channel crop."""
        if size not in self._crops:
            ok = (self.im_idx >= 0) & (self.im_idx < self.b)
            boxes5 = torch.cat((torch.where(ok, self.im_idx, 0).float().unsqueeze(1), self.boxes), dim=1)
            crop = L.crop_images(self.images, boxes5, size)
            crop[~ok] = 0.0
            self._crops[size] = crop
        return self._crops[size][:n, :c_in]


@pytest.fixture(scope="module")
def inputs():
    return _Inputs()


@pytest.fixture
def raster_mode():
    """Sets the raster kernel selection (include/mpx.h mpx_raster_set_mode) for one test and restores the default."""
    yield lambda mode: _abi.lib().mpx_raster_set_mode(mode)
    _abi.lib().mpx_raster_set_mode(7)


# ------------------------------------------------------------------------------------------------------------------------
# reference input and the comparison
# ------------------------------------------------------------------------------------------------------------------------
def _to_act(t):
    """fp32 -> the 16-bit type as the kernels convert: fp16 saturates at +-65504 (cvt.rn.satfinite, the same as clamping
    first), bf16 rounds to nearest (its range is fp32's)."""
    if ACT == torch.float16:
        fi = torch.finfo(ACT)
        t = t.clamp(-fi.max, fi.max)
    return t.to(ACT).float()


def _ulp(v):
    """Spacing of the 16-bit type at |v| (v already representable)."""
    fi = torch.finfo(ACT)
    _, e = torch.frexp(v.abs())
    tiny = torch.full_like(v, fi.smallest_normal * fi.eps)  # subnormal spacing
    return torch.where(v == 0, tiny, torch.maximum(torch.pow(2.0, (e - 1).float()) * fi.eps, tiny))


def _tcr(z):
    t = torch.zeros(z.shape[0], 3)
    t[:, 2] = z
    return t


def _norm(depth, z, kind):
    return L.normalize_depth(depth, _tcr(z), KIND_NAMES[kind])


def _unpack(x, n, h, w, c_pad):
    """[n, h/2, w/2, 4*c_pad] (channel (dy*2+dx)*c_pad + c) -> [n, c_pad, h, w] on the host."""
    return x.view(n, h // 2, w // 2, 2, 2, c_pad).permute(0, 5, 1, 3, 2, 4).reshape(n, c_pad, h, w).cpu()


def _where(mask, ch0=0):
    """Count and first position of a mask over channels ch0.. of [n, c, h, w]."""
    idx = mask.nonzero()
    if not idx.numel():
        return "none"
    s, c, i, j = idx[0].tolist()
    return f"{idx.shape[0]} positions, first (sample, channel, row, col) = ({s}, {c + ch0}, {i}, {j})"


def _assert_exact(got, want, what, ch0):
    gn, wn = got.isnan(), want.isnan()
    assert torch.equal(gn, wn), f"{what}: NaN positions differ at {_where(gn != wn, ch0)}"
    bad = (got != want) & ~gn
    assert not bad.any(), \
        f"{what}: values differ at {_where(bad, ch0)}, got {got[bad][:4].tolist()} want {want[bad][:4].tolist()}"


def _assert_crop(got, want32, what, atol, ch0, scale=None, max_frac=0.0):
    want = _to_act(want32)
    gn, wn = got.isnan(), want.isnan()
    tol = _ulp(want) + atol * (scale if scale is not None else 1.0) + 1e-5 * want.abs()
    ok = (gn & wn) | (~gn & ~wn & ((got - want).abs() <= tol))
    frac = (~ok).float().mean().item()
    assert frac <= max_frac, (f"{what}: {frac:.2e} of the values off by more than 1 ulp + fp32 bound, {_where(~ok, ch0)}, "
                              f"got {got[~ok][:4].tolist()} want {want[~ok][:4].tolist()}")


def _depth_slope(z, kind):
    """|d normalised / d depth| per sample, [n, 1, 1, 1]: the fp32 crop error scales with it."""
    s = torch.ones_like(z)
    if kind in (0, 1):
        s = 1.0 / z.abs().clamp_min(1e-3)
    return torch.nan_to_num(s, nan=1.0).view(-1, 1, 1, 1)


def _render_want(orc, views, cpv, point, z_view, kind):
    parts = [orc["rgb_pt" if point else "rgb_amb"][views]]
    if cpv >= 6:
        parts.append(orc["normals"][views])
    if cpv in (4, 7):
        parts.append(_norm(orc["depth"][views], z_view, kind))
    return torch.cat(parts, dim=1)


def _check_input(x, c_pad, crop, c_in, z, kind, renders, rest, what=""):
    """x against [crop (c_in channels, reference-normalised) | renders | rest] where rest is 'zero' or 'sentinel'."""
    n, _, h, w = crop.shape
    got = _unpack(x, n, h, w, c_pad).float()
    bits = _unpack(x.view(torch.int16), n, h, w, c_pad)
    k = renders.shape[1]
    _assert_exact(got[:, c_in:c_in + k], _to_act(renders), f"{what}render channels {c_in}..{c_in + k - 1}", c_in)
    _assert_crop(got[:, :3], crop[:, :3], f"{what}crop rgb", atol=2e-5, ch0=0)
    if c_in == 4:
        _assert_crop(got[:, 3:4], _norm(crop[:, 3:4], z, kind), f"{what}crop depth", atol=2e-4, ch0=3,
                     scale=_depth_slope(z, kind), max_frac=1e-3)
    tail = bits[:, c_in + k:]
    want_bits = 0 if rest == "zero" else torch.tensor(SENTINEL, dtype=ACT).view(torch.int16).item()
    assert (tail == want_bits).all(), \
        f"{what}channels {c_in + k}..{c_pad - 1} were not left {rest}: {_where(tail != want_bits, c_in + k)}"


def _sentinel_x(n, h, w, c_pad):
    return torch.full((n, h // 2, w // 2, 4 * c_pad), SENTINEL, device=DEV, dtype=ACT)


def _flags(cpv, kind, point=None):
    point = cpv in (3, 4) if point is None else point  # what the predictor does: normals-free renders are lit
    return (RASTER_POINT_LIGHTS if point else 0) | (kind << DEPTH_NORM_SHIFT)


# ------------------------------------------------------------------------------------------------------------------------
# mpx_render_crop_fused
# ------------------------------------------------------------------------------------------------------------------------
def _layouts():
    out = []
    for c_in in (3, 4):
        for cpv in (3, 4, 6, 7):
            has_depth = c_in == 4 or cpv in (4, 7)
            for kind in ((0, 1, 2, 3) if has_depth else (3,)):
                out.append((c_in, cpv, kind))
    return out


def _crop_fused_cases():
    cases = []
    for size, paths in (("224x224", list(PATHS)), ("64x96", ["scatter", "tiled"]), ("64x968", ["scatter", "tiled"])):
        for path in paths:
            for c_in, cpv, kind in _layouts():
                cases.append(pytest.param(size, path, c_in, cpv, kind, 16, None,
                                          id=f"{size}-{path}-cin{c_in}-cpv{cpv}-kind{kind}"))
    for path in PATHS:
        cases.append(pytest.param("224x224", path, 4, 7, 0, 32, None, id=f"224x224-{path}-cin4-cpv7-kind0-cpad32"))
        cases.append(pytest.param("224x224", path, 3, 3, 3, 16, False, id=f"224x224-{path}-cin3-cpv3-ambient"))
        cases.append(pytest.param("64x96", path, 3, 6, 3, 16, True, id=f"64x96-{path}-cin3-cpv6-point-lights"))
    return cases


@pytest.mark.parametrize("size,path,c_in,cpv,kind,c_pad,point", _crop_fused_cases())
def test_render_crop_fused_vs_oracle(inputs, raster_mode, size, path, c_in, cpv, kind, c_pad, point):
    h, w = SIZES[size]
    mode, n = PATHS[path]
    raster_mode(mode)
    point = cpv in (3, 4) if point is None else point
    x = _sentinel_x(n, h, w, c_pad)
    z = inputs.z[:n]
    inputs.renderer.render_crop_fused(inputs.lab[:n], inputs.TCO[:n].cuda(), inputs.K((h, w))[:n].cuda(), (h, w),
                                      inputs.nhwc4, inputs.im_idx[:n].cuda(), inputs.boxes[:n].cuda(), c_in, x, c_pad, cpv,
                                      z.cuda(), _flags(cpv, kind, point))
    torch.cuda.synchronize()
    want = _render_want(inputs.renders((h, w)), slice(0, n), cpv, point, z, kind)
    _check_input(x, c_pad, inputs.crops((h, w), n, c_in), c_in, z, kind, want, rest="zero")


# ------------------------------------------------------------------------------------------------------------------------
# mpx_roi_align_fused + mpx_raster_render_fused
# ------------------------------------------------------------------------------------------------------------------------
MULTIVIEW = [(1, 12, 7), (2, 20, 7), (2, 20, 3), (4, 4, 7), (4, 10, 3), (27, 2, 7), (27, 2, 3)]  # vps, samples, mode


def _multiview_cases():
    cases = []
    for size, runs in (("224x224", MULTIVIEW), ("64x968", [(2, 20, 7), (4, 4, 7)])):
        for vps, n, mode in runs:
            for c_in in (3, 4):
                for cpv in (3, 4, 6, 7):
                    kind = (cpv + 2 * c_in + vps) % 4  # every kind appears for every views_per_sample
                    path = "scatter" if n * vps * 8 <= 144 else ("untiled" if mode == 3 else "tiled")
                    cases.append(pytest.param(size, vps, n, mode, c_in, cpv, kind,
                                              id=f"{size}-vps{vps}-n{n}-{path}-cin{c_in}-cpv{cpv}-kind{kind}"))
    return cases


def _multiview_write(inputs, x, size, vps, n, c_in, cpv, kind, c_pad, z):
    h, w = size
    im_idx, boxes, z = inputs.im_idx[:n].cuda(), inputs.boxes[:n].cuda(), z.cuda()  # alive until the kernels have run
    _abi.check(_abi.lib().mpx_roi_align_fused(
        _abi.ptr(inputs.nhwc4), inputs.b, inputs.nhwc4.shape[1], inputs.nhwc4.shape[2], _abi.ptr(im_idx), _abi.ptr(boxes),
        n, c_in, h, w, _abi.ptr(x), c_pad, _abi.ptr(z), kind, _abi.stream_ptr()))
    torch.cuda.synchronize()
    sentinel = torch.tensor(SENTINEL, dtype=ACT, device=DEV)
    rest = x.view(n, h // 2, w // 2, 4, c_pad)[..., c_in:]
    assert (rest.view(torch.int16) == sentinel.view(torch.int16)).all(), "roi_align_fused wrote outside channels 0..c_in-1"
    nv = n * vps
    inputs.renderer.render_fused(inputs.lab[:nv], inputs.TCO[:nv].cuda(), inputs.K(size)[:nv].cuda(), vps, size, x, c_pad,
                                 c_in, cpv, z, _flags(cpv, kind))
    torch.cuda.synchronize()


@pytest.mark.parametrize("size,vps,n,mode,c_in,cpv,kind", _multiview_cases())
def test_multiview_fused_vs_oracle(inputs, raster_mode, size, vps, n, mode, c_in, cpv, kind):
    h, w = SIZES[size]
    raster_mode(mode)
    c_pad = (c_in + vps * cpv + 15) // 16 * 16
    z = inputs.z[:n]
    x = _sentinel_x(n, h, w, c_pad)
    _multiview_write(inputs, x, (h, w), vps, n, c_in, cpv, kind, c_pad, z)
    nv = n * vps
    want = _render_want(inputs.renders((h, w)), slice(0, nv), cpv, cpv in (3, 4), z.repeat_interleave(vps), kind)
    want = want.view(n, vps * want.shape[1], h, w)  # [crop | view0 | view1 | ...]
    _check_input(x, c_pad, inputs.crops((h, w), n, c_in), c_in, z, kind, want, rest="sentinel")


# ------------------------------------------------------------------------------------------------------------------------
# depth normalisation at its edges: z = 1e-7 (|d / z| beyond the 16-bit range), 0 (0 / 0 on the background), < 0, NaN
# ------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("writer", ["render_crop_fused", "roi_align_fused+render_fused"])
@pytest.mark.parametrize("kind", [0, 1, 2, 3])
def test_depth_norm_edges(inputs, raster_mode, writer, kind):
    raster_mode(7)
    size = SIZES["64x96"]
    h, w = size
    n, c_pad, c_in, cpv = 8, 16, 4, 7
    z = torch.tensor([1e-7, 0.0, -0.5, float("nan"), 1e-7, 0.0, -0.5, float("nan")])
    x = _sentinel_x(n, h, w, c_pad)
    if writer == "render_crop_fused":
        inputs.renderer.render_crop_fused(inputs.lab[:n], inputs.TCO[:n].cuda(), inputs.K(size)[:n].cuda(), size,
                                          inputs.nhwc4, inputs.im_idx[:n].cuda(), inputs.boxes[:n].cuda(), c_in, x, c_pad,
                                          cpv, z.cuda(), _flags(cpv, kind))
        torch.cuda.synchronize()
        rest = "zero"
    else:
        _multiview_write(inputs, x, size, 1, n, c_in, cpv, kind, c_pad, z)
        rest = "sentinel"
    want = _render_want(inputs.renders(size), slice(0, n), cpv, False, z, kind)
    _check_input(x, c_pad, inputs.crops(size, n, c_in), c_in, z, kind, want, rest=rest)


# ------------------------------------------------------------------------------------------------------------------------
# the predictor's wiring: which writer, flags, ch_offset, kind and ch_per_view each configuration uses
# ------------------------------------------------------------------------------------------------------------------------
RELEASED = {"coarse": ("coarse-rgb-906902141", helpers.COARSE_CFG, 5),
            "refiner_rgb": ("refiner-rgb-653307694", helpers.REFINER_CFG, 6),
            "refiner_rgbd": ("refiner-rgbd-288182519", helpers.REFINER_RGBD_CFG, 7)}


@pytest.fixture(scope="module")
def predictor_scene():
    ds, images, K = helpers.make_scene(2, seed=8, with_depth=True)
    return ds, images, K, helpers.ref_meshes_from_dataset(ds)


def _model(predictor_scene, tmp_path, name):
    """(PosePredictor, oracle RefPosePredictor) for a released configuration or a test_gpu_variants.VARIANTS entry."""
    ds, images, K, rm = predictor_scene
    if name in RELEASED:
        run_id, cfg, seed = RELEASED[name]
        sd = helpers.make_state_dict(cfg, seed)
        load_model.write_run(tmp_path, run_id, sd)
        other = "refiner-rgb-653307694" if name == "coarse" else "coarse-rgb-906902141"
        other_cfg = helpers.REFINER_CFG if name == "coarse" else helpers.COARSE_CFG
        load_model.write_run(tmp_path, other, helpers.make_state_dict(other_cfg, 1))
        coarse_id, refiner_id = (run_id, other) if name == "coarse" else (other, run_id)
        coarse, refiner, _ = load_model.load_pose_models(coarse_id, refiner_id, ds, models_root=tmp_path)
        model = coarse if name == "coarse" else refiner
        return model, pipeline_ref.RefPosePredictor(sd, cfg, rm, pipeline_ref.RefRenderer(rm))
    model, oracle, _, _ = variants._variant_models(predictor_scene, tmp_path, dict(variants.VARIANTS[name]),
                                                   seed=20 + len(name))
    return model, oracle


@pytest.mark.parametrize("name", list(RELEASED) + list(variants.VARIANTS))
def test_predictor_writes_the_oracle_input(predictor_scene, tmp_path, name):
    ds, images, K, rm = predictor_scene
    model, oracle = _model(predictor_scene, tmp_path, name)
    model.use_cuda_graphs = False
    c_in = 4 if oracle.input_depth else 3
    imgs = images[:, :c_in].contiguous()
    n = 3
    labels = [ds[i % 2].label for i in range(n)]
    TCO = torch.from_numpy(procedural.random_poses(n, 19, z_range=(0.4, 0.8))).float()
    Kn = K.repeat(n, 1, 1)
    it = model(images=imgs.cuda(), K=Kn.cuda(), labels=labels, TCO=TCO.cuda(), n_iterations=1,
               batch_im_ids=torch.zeros(n, dtype=torch.long))["iteration=1"]
    torch.cuda.synchronize()
    h, w = model.render_size
    x = model._x_cache[(n, h, w)]
    c_pad = model.backbone.c_pad
    # the oracle's input from the product's own crop boxes, view cameras and tCR of this iteration
    boxes5 = torch.cat((torch.zeros(n, 1), it.boxes_crop.cpu()), dim=1)
    crop = L.crop_images(imgs, boxes5, (h, w))
    renders = oracle.render_images_multiview(labels, it.TCV_O_input.cpu(), it.KV_crop.cpu())
    tCR = it.tCR.cpu()
    _, renders = oracle.normalize_images(crop, renders, tCR)
    kind = {v: k for k, v in KIND_NAMES.items()}[oracle.norm_type] if oracle.input_depth or oracle.render_depth else 3
    _check_input(x, c_pad, crop, c_in, tCR[:, 2], kind, renders, rest="zero", what=f"{name}: ")


# ------------------------------------------------------------------------------------------------------------------------
# layouts the writers must refuse: nonzero return with a message, nothing launched, x untouched
# ------------------------------------------------------------------------------------------------------------------------
def test_fused_writers_reject_bad_layouts(inputs):
    lib = _abi.lib()
    r = inputs.renderer
    n, h, w, c_pad = 4, 64, 96, 16
    x = _sentinel_x(n, h + 2, w, 48)  # room for every layout below
    before = x.clone()
    tensors = dict(lab=inputs.lab, TCO=inputs.TCO[:n].cuda(), K=inputs.K((h, w))[:n].cuda(), boxes=inputs.boxes[:n].cuda(),
                   im_idx=inputs.im_idx[:n].cuda(), z=inputs.z[:n].cuda())
    args = {k: _abi.ptr(t) for k, t in tensors.items()}
    img = (_abi.ptr(inputs.nhwc4), inputs.b, inputs.nhwc4.shape[1], inputs.nhwc4.shape[2])
    s = _abi.stream_ptr()

    def render_fused(vps, hh, c_pad_, ch_offset, cpv):
        ws = r.workspace(hh, w, DEV)
        return lib.mpx_raster_render_fused(r.mesh_db.handle, args["lab"], args["TCO"], args["K"], n, vps, hh, w, 0,
                                           _abi.ptr(x), c_pad_, ch_offset, cpv, args["z"], _abi.ptr(ws), ws.numel(), s)

    def crop_fused(c_in, c_pad_, cpv, byte_offset=0, hh=h):
        ws = r.workspace(hh, w, DEV)
        return lib.mpx_render_crop_fused(r.mesh_db.handle, args["lab"], args["TCO"], args["K"], n, hh, w, 0, *img,
                                         args["im_idx"], args["boxes"], c_in, _abi.ptr(x) + byte_offset, c_pad_, cpv,
                                         args["z"], _abi.ptr(ws), ws.numel(), s)

    def roi_fused(c, c_pad_, kind, hh=h):
        return lib.mpx_roi_align_fused(*img, args["im_idx"], args["boxes"], n, c, hh, w, _abi.ptr(x), c_pad_, args["z"], kind,
                                       s)

    cases = [
        ("ch_per_view = 5", lambda: render_fused(1, h, c_pad, 3, 5), "ch_per_view must be"),
        ("ch_per_view = 5, fused crop", lambda: crop_fused(3, c_pad, 5), "ch_per_view must be"),
        ("ch_offset + vps * cpv = c_pad + 1", lambda: render_fused(2, h, c_pad, 3, 7), "do not fit"),
        ("c_in + cpv = c_pad + 1, fused crop", lambda: crop_fused(4, 10, 7), "do not fit"),
        ("odd h", lambda: render_fused(1, h - 1, c_pad, 3, 6), "even resolution"),
        ("odd h, fused crop", lambda: crop_fused(3, c_pad, 6, hh=h - 1), "even resolution"),
        ("odd h, roi_align_fused", lambda: roi_fused(3, c_pad, 0, hh=h - 1), "even size"),
        ("fused crop with c_pad = 48", lambda: crop_fused(3, 48, 6), "fused crop layout unsupported"),
        ("x misaligned by 2 bytes, fused crop", lambda: crop_fused(3, c_pad, 6, byte_offset=2), "16-byte aligned"),
        ("roi_align_fused c > c_pad", lambda: roi_fused(4, 3, 0), "c=4 > c_pad=3"),
        ("roi_align_fused kind 4", lambda: roi_fused(4, c_pad, 4), "depth_norm_kind=4"),
    ]
    for what, call, msg in cases:
        launches = lib.mpx_launch_count()
        rc = call()
        torch.cuda.synchronize()
        err = (lib.mpx_last_error() or b"").decode()
        assert rc != 0, f"{what}: accepted"
        assert msg in err, f"{what}: message {err!r}"
        assert lib.mpx_launch_count() == launches, f"{what}: launched a kernel"
        assert torch.equal(x.view(torch.int16), before.view(torch.int16)), f"{what}: x was written"
