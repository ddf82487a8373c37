"""-m gpu: SAM2ImagePredictor.predict / predict_batch with point, box and mask prompts, and the kernel that makes their
full-resolution output (ops.upsample_select).

* the kernel, bit for bit, against the numpy oracle and ops.upsample_bilinear of the gathered planes, for every candidate
  selection, ragged and tiny frame sizes, thresholds hit exactly, and an output past 2^31 bytes;
* predict against the upstream restatement in oracle/sam2_ref/image_predict.py for each prompt kind (the decoder's
  token counts 6, 8, 9..16 and > 16), both output modes, both coordinate conventions, square and non-square images;
* predict_batch against per-image predict (bit for bit) and the oracle, and upstream's asserts;
* the hole / sprinkle fill options against the oracle's fill given our own low-res logits.
Hiera-tiny is random-initialised and conditioned as in tests/test_gpu_configs.py.
"""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
REL_TOL = 2e-2  # BASELINE.json north_star: bf16 embeddings / logits within 2e-2 relative error


def rel_l2(a, b):
    a, b = torch.as_tensor(a).double(), torch.as_tensor(b).double()
    return ((a - b).norm() / (b.norm() + 1e-12)).item()


def _conditioned(sd):
    """As tests/test_gpu_configs.py: realistic mask-logit range and well-separated IoU / object-score heads."""
    sd = dict(sd)
    for k in list(sd):
        if "output_hypernetworks_mlps" in k and ".layers.2." in k:
            sd[k] = sd[k] * 30.0
    sd["sam_mask_decoder.iou_prediction_head.layers.2.bias"] = torch.tensor([0.0, -1.0, 1.0, 0.0])
    sd["sam_mask_decoder.pred_obj_score_head.layers.2.bias"] = torch.tensor([1.5])
    return sd


# ------------------------------------------------------------------------------------------------- 1. the kernel
def _planes(P, thr, seed):
    g = torch.Generator().manual_seed(seed)
    planes = torch.randn(P, 4, 256, 256, generator=g) * 4.0
    planes[:, :, 100:140, 50:90] = thr  # up-sampled values exactly at the threshold
    planes[:, :, 0:3, :] = thr
    return planes.cuda().contiguous()


def _gather(planes, sel, cpp):
    if cpp == 3:
        return planes[:, 1:4].contiguous()
    if sel is not None:
        return planes[torch.arange(planes.shape[0], device="cuda"), sel.long()].unsqueeze(1).contiguous()
    return planes[:, 0:1].contiguous()


SIZES = [(1, 1), (1, 517), (255, 256), (256, 256), (300, 517), (927, 1000), (2085, 1111)]


@pytest.mark.parametrize("hw", SIZES)
@pytest.mark.parametrize("mode", ["multi", "sel", "token0"])
@pytest.mark.parametrize("thr", [0.0, 0.5, -1.0])
def test_upsample_select_bit_exact(hw, mode, thr):
    from oracle import amg_post_ref as R
    from saber_b200 import ops
    H, W = hw
    cpp = 3 if mode == "multi" else 1
    P = {1: 65, 255: 65, 256: 17, 300: 7, 927: 2, 2085: 1}[H]
    planes = _planes(P, thr, seed=H + W)
    sel = torch.randint(0, 4, (P,), dtype=torch.int32, device="cuda") if mode == "sel" else None
    g = _gather(planes, sel, cpp)
    want = ops.upsample_bilinear(g, H, W)
    logits = ops.upsample_select(planes, sel, cpp, H, W, thr, logits=True)
    masks = ops.upsample_select(planes, sel, cpp, H, W, thr)
    assert logits.shape == masks.shape == (P, cpp, H, W) and masks.dtype == torch.bool and logits.dtype == torch.float32
    assert torch.equal(logits, want)
    assert torch.equal(masks, want > thr)
    k = max(1, min(P, 4_000_000 // (cpp * H * W)))  # the numpy oracle on the first k candidates
    ref = R.upsample_bilinear(g[:k].cpu().numpy(), (H, W))
    np.testing.assert_array_equal(logits[:k].cpu().numpy(), ref)
    np.testing.assert_array_equal(masks[:k].cpu().numpy(), ref > np.float32(thr))
    if H * W > 1:
        assert masks.any() and not masks.all()


@pytest.mark.parametrize("P", [1, 2, 3, 33, 64, 65])
def test_upsample_select_prompt_counts(P):
    from saber_b200 import ops
    planes = _planes(P, 0.0, seed=P)
    sel = torch.randint(0, 4, (P,), dtype=torch.int32, device="cuda")
    for cpp, s in ((3, None), (1, sel), (1, None)):
        want = ops.upsample_bilinear(_gather(planes, s, cpp), 300, 517)
        assert torch.equal(ops.upsample_select(planes, s, cpp, 300, 517, 0.0), want > 0.0)
        assert torch.equal(ops.upsample_select(planes, s, cpp, 300, 517, 0.0, logits=True), want)


def test_upsample_select_past_2_31():
    """43 prompts x 3 masks x 4096^2 bool = 2.16e9 bytes: the last candidate and sampled rows of others."""
    from saber_b200 import ops
    P, H, W = 43, 4096, 4096
    planes = _planes(P, 0.0, seed=7)
    masks = ops.upsample_select(planes, None, 3, H, W, 0.0)
    assert masks.numel() > 2 ** 31
    want_last = ops.upsample_bilinear(planes[P - 1:P, 3:4].contiguous(), H, W) > 0.0
    assert torch.equal(masks[P - 1, 2:3], want_last[0])
    rng = np.random.default_rng(0)
    for p in rng.choice(P, 6, replace=False):
        want = ops.upsample_bilinear(planes[p:p + 1, 1:4].contiguous(), H, W) > 0.0
        rows = torch.as_tensor(rng.choice(H, 64, replace=False), device="cuda")
        assert torch.equal(masks[p][:, rows], want[0][:, rows])


# --------------------------------------------------------------------------------------------- 2. predict vs oracle
@pytest.fixture(scope="module")
def models():
    from oracle.sam2_ref.sam2_base import SAM2Base
    from saber_b200.sam2 import arch
    from saber_b200.sam2.build_sam import build_sam2
    sd = _conditioned(arch.random_state_dict("tiny", seed=0))
    orc = SAM2Base("tiny", dynamic_multimask_via_stability=True)
    orc.load_state_dict(sd, strict=True)
    orc = orc.cuda().eval()
    ours = build_sam2("tiny", None, device="cuda", state_dict=sd, apply_postprocessing=True)
    return ours, orc


def _image(hw, seed, uint8=False):
    rng = np.random.default_rng(seed)
    H, W = hw
    yy, xx = np.mgrid[0:H, 0:W].astype(np.float32)
    img = 0.5 + 0.3 * np.sin(xx / 23.0)[..., None] * np.cos(yy / 17.0)[..., None] + 0.1 * rng.normal(size=(H, W, 3))
    img = np.clip(img, 0, 1).astype(np.float32)
    return (img * 255).astype(np.uint8) if uint8 else img


IMAGES = {"square": (512, 512), "wide": (300, 517)}


@pytest.fixture(scope="module")
def predictors(models):
    from oracle.sam2_ref.image_predict import SAM2ImagePredictor as OraclePredictor
    from saber_b200.sam2.sam2_image_predictor import SAM2ImagePredictor
    ours, orc = models
    out = {}
    for name, hw in IMAGES.items():
        img = _image(hw, seed=hw[1])
        a, b = SAM2ImagePredictor(ours), OraclePredictor(orc)
        a.set_image(img)
        b.set_image(img)
        # a mask prompt: the previous call's best low-res logits
        _, iou, low = a.predict(point_coords=np.array([[hw[1] * 0.4, hw[0] * 0.5]]), point_labels=np.array([1]))
        out[name] = (a, b, hw, low[np.argmax(iou)][None])
    return out


def _prompts(kind, hw, prev):
    """Prompt keywords in original-image pixels."""
    H, W = hw
    rng = np.random.default_rng(len(kind))
    pts = lambda n: np.stack([rng.uniform(0.1, 0.9, n) * W, rng.uniform(0.1, 0.9, n) * H], 1).astype(np.float32)
    box = np.array([0.2 * W, 0.25 * H, 0.7 * W, 0.8 * H], np.float32)
    if kind == "point":
        return dict(point_coords=pts(1), point_labels=np.array([1]))
    if kind == "points_neg":
        return dict(point_coords=pts(3), point_labels=np.array([1, 0, 1]))
    if kind == "many_points":  # 12 points + pad: 19 decoder tokens
        return dict(point_coords=pts(12), point_labels=(np.arange(12) % 3 != 2).astype(np.int32))
    if kind == "box":
        return dict(box=box)
    if kind == "box_points":
        return dict(box=box, point_coords=pts(2), point_labels=np.array([1, 0]))
    if kind == "n_boxes":
        xy = rng.uniform(0, 0.5, (4, 2)) * [W, H]
        return dict(box=np.concatenate([xy, xy + rng.uniform(0.2, 0.45, (4, 2)) * [W, H]], 1).astype(np.float32))
    if kind == "mask":  # no sparse prompt: 6 decoder tokens
        return dict(mask_input=prev)
    if kind == "points_prev":
        return dict(point_coords=pts(2), point_labels=np.array([1, 1]), mask_input=prev)
    raise KeyError(kind)


def _normalised(kw, hw):
    """The same prompts for normalize_coords=False: coordinates already in [0, 1]."""
    H, W = hw
    kw = dict(kw)
    if "point_coords" in kw:
        kw["point_coords"] = kw["point_coords"] / np.array([W, H], np.float32)
    if "box" in kw:
        kw["box"] = kw["box"] / np.array([W, H, W, H], np.float32)
    return kw


KINDS = ["point", "points_neg", "many_points", "box", "box_points", "n_boxes", "mask", "points_prev"]


@pytest.mark.parametrize("image", list(IMAGES))
@pytest.mark.parametrize("normalize", [True, False])
@pytest.mark.parametrize("multimask", [True, False])
@pytest.mark.parametrize("kind", KINDS)
def test_predict_matches_oracle(predictors, kind, multimask, normalize, image):
    ours, orc, hw, prev = predictors[image]
    kw = _prompts(kind, hw, prev)
    if not normalize:
        kw = _normalised(kw, hw)
    kw.update(multimask_output=multimask, normalize_coords=normalize)
    logits, iou, low = ours.predict(return_logits=True, **kw)
    r_logits, r_iou, r_low = orc.predict(return_logits=True, **kw)
    masks, iou_m, low_m = ours.predict(**kw)
    r_masks, _, _ = orc.predict(**kw)
    for a, b in ((logits, r_logits), (iou, r_iou), (low, r_low), (masks, r_masks)):
        assert a.shape == b.shape and a.dtype == b.dtype == np.float32, (a.shape, b.shape, a.dtype, b.dtype)
    C = 3 if multimask else 1
    lead = (4,) if kind == "n_boxes" else ()
    assert logits.shape == lead + (C,) + hw and low.shape == lead + (C, 256, 256) and iou.shape == lead + (C,)
    assert rel_l2(iou, r_iou) < REL_TOL
    assert rel_l2(low, r_low) < REL_TOL
    assert rel_l2(logits, r_logits) < REL_TOL
    np.testing.assert_array_equal(masks, (logits > ours.mask_threshold).astype(np.float32))
    np.testing.assert_array_equal(iou_m, iou)
    np.testing.assert_array_equal(low_m, low)


# ------------------------------------------------------------------------------------------------ 3. predict_batch
def test_predict_batch(models):
    from oracle.sam2_ref.image_predict import SAM2ImagePredictor as OraclePredictor
    from saber_b200.sam2.sam2_image_predictor import SAM2ImagePredictor
    ours, orc = models
    hws = [(300, 517), (512, 512), (411, 290)]
    imgs = [_image(hws[0], 1), _image(hws[1], 2, uint8=True), _image(hws[2], 3)]
    kws = [_prompts("point", hws[0], None), _prompts("box", hws[1], None), _prompts("box_points", hws[2], None)]
    batch = dict(point_coords_batch=[k.get("point_coords") for k in kws],
                 point_labels_batch=[k.get("point_labels") for k in kws], box_batch=[k.get("box") for k in kws])
    a, b, single = SAM2ImagePredictor(ours), OraclePredictor(orc), SAM2ImagePredictor(ours)
    a.set_image_batch(imgs)
    b.set_image_batch(imgs)
    for return_logits in (True, False):
        got = a.predict_batch(return_logits=return_logits, **batch)
        want = b.predict_batch(return_logits=return_logits, **batch)
        for i, (img, kw) in enumerate(zip(imgs, kws)):
            single.set_image(img)
            one = single.predict(return_logits=return_logits, **kw)
            for g, o, w in zip((got[0][i], got[1][i], got[2][i]), one, (want[0][i], want[1][i], want[2][i])):
                np.testing.assert_array_equal(g, o)
                assert g.shape == w.shape and g.dtype == w.dtype
            if return_logits:
                for g, w in zip((got[0][i], got[1][i], got[2][i]), (want[0][i], want[1][i], want[2][i])):
                    assert rel_l2(g, w) < REL_TOL
    with pytest.raises(AssertionError):  # one box list entry short of the image count
        a.predict_batch(box_batch=batch["box_batch"][:2])
    with pytest.raises(AssertionError):  # not in batched mode
        single.predict_batch(**batch)


# ------------------------------------------------------------------------------------------------- 4. fill options
@pytest.mark.parametrize("multimask", [True, False])
def test_predict_fill_options(models, multimask):
    from oracle.sam2_ref.small_regions import fill_holes_and_sprinkles
    from saber_b200 import ops
    from saber_b200.sam2.sam2_image_predictor import SAM2ImagePredictor
    ours, _ = models
    hw = (300, 517)
    img = _image(hw, 5)
    plain, filled = SAM2ImagePredictor(ours), SAM2ImagePredictor(ours, max_hole_area=8, max_sprinkle_area=8)
    plain.set_image(img)
    filled.set_image(img)
    kw = dict(_prompts("box_points", hw, None), multimask_output=multimask)
    masks, iou, low = filled.predict(**kw)
    m0, i0, low0 = plain.predict(**kw)
    np.testing.assert_array_equal(low, low0)
    np.testing.assert_array_equal(iou, i0)
    # the raw (unclamped) decoder planes of the same prompt, selected as predict selects them
    _, coords, labels, box = plain._prep_prompts(kw["point_coords"], kw["point_labels"], kw["box"], None, True)
    dec, tok = ours.decoder, plain._features.tok
    c = torch.cat([box.reshape(-1, 2, 2), coords], 1).contiguous()
    l = torch.cat([torch.tensor([[2, 3]], dtype=torch.int32, device="cuda"), labels], 1).contiguous()
    out = dec.forward(tok["embed"][:4096], tok["s0"][:65536], tok["s1"][:16384], dec.prompt_tokens(c, l), None,
                      multimask_output=multimask)
    if multimask:
        raw = out["masks"][:, 1:4]
    elif out.get("sel_idx") is not None:
        raw = out["masks"][torch.arange(1, device="cuda"), out["sel_idx"].long()].unsqueeze(1)
    else:
        raw = out["masks"][:, 0:1]
    want = ops.upsample_bilinear(fill_holes_and_sprinkles(raw, 0.0, 8, 8).contiguous(), *hw) > 0.0
    np.testing.assert_array_equal(masks, want.squeeze(0).cpu().numpy().astype(np.float32))
    assert not np.array_equal(masks, m0)


# ------------------------------------------------------------------------------------------ 5. the torch-level API
def test_predict_with_boxes_equals_predict(predictors, models):
    from saber_b200.sam2.sam2_image_predictor import SAM2ImagePredictor
    ours, _, hw, _ = predictors["wide"]
    kw = _prompts("box", hw, None)
    for multimask in (True, False):
        for return_logits in (True, False):
            want = ours.predict(multimask_output=multimask, return_logits=return_logits, **kw)
            _, _, _, box = ours._prep_prompts(None, None, kw["box"], None, True)
            masks, iou, low = ours._predict(None, None, boxes=box, multimask_output=multimask,
                                            return_logits=return_logits)
            assert masks.dtype == (torch.float32 if return_logits else torch.bool)
            np.testing.assert_array_equal(masks.squeeze(0).float().cpu().numpy(), want[0])
            np.testing.assert_array_equal(iou.squeeze(0).cpu().numpy(), want[1])
            np.testing.assert_array_equal(low.squeeze(0).cpu().numpy(), want[2])
    unset = SAM2ImagePredictor(models[0])
    with pytest.raises(RuntimeError, match="An image must be set"):
        unset.predict(box=kw["box"])
    with pytest.raises(RuntimeError, match="An image must be set"):
        unset._predict(None, None, boxes=torch.zeros(1, 4, device="cuda"))
