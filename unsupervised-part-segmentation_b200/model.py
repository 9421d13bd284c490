"""Drop-in for the module-level helpers of the reference's model files
(cub/code/SB_model48i/model.py, pennaction/code/SB_model48i/model.py,
deepfashion/code/SB_model48c/model.py) that sit on the part-disentanglement path."""
import torch

from . import nn, ops
from . import tps as _tps

PARTS_DIM = 3      # cub/code/SB_model48i/model.py:12
FEATURE_DIM = 4    # cub/code/SB_model48i/model.py:13


def categorical_kl(probs):
    """cub/code/SB_model48i/model.py:21-25 — reduce_mean over pixels of sum_k p*log(K*p + 1e-20)."""
    return ops.categorical_kl(probs)


def weak_cross_entropy(log_probs, entropy_func="cross_entropy"):
    """cub/code/SB_model48i/model.py:667-681 — reduce_mean of softmax_cross_entropy_with_logits_v2 between the part
    logits and their own straight-through hard assignment ("cross_entropy") or their softmax ("entropy")."""
    if entropy_func == "cross_entropy":
        return ops.weak_xent(log_probs, 0)
    elif entropy_func == "entropy":
        return ops.weak_xent(log_probs, 1)
    raise ValueError("unkown entropy_func")


def mask_parts(image, mask):
    """cub/code/SB_model48i/model.py:176-187 — [B,H,W,3],[B,H,W,parts] -> [B,H,W,parts,3]."""
    bs, h, w, n_features = image.shape
    mshape = list(mask.shape)
    assert mshape[0] == bs and mshape[1] == h and mshape[2] == w, mshape
    return ops.mask_parts(image, mask, False)


def mask_parts_partmajor(image, mask):
    """mask_parts followed by nn.apply_partwise's fold (cub/code/nn.py:100-103) in one pass:
    [B,H,W,3],[B,H,W,parts] -> [parts*B,H,W,3] with row k*B+b."""
    bs, h, w, _ = image.shape
    mshape = list(mask.shape)
    assert mshape[0] == bs and mshape[1] == h and mshape[2] == w, mshape
    return ops.mask_parts(image, mask, True)


def encode_parts(part_image, encoder):
    """cub/code/SB_model48i/model.py:214-222 — [B,H,W,parts,3] -> [B,parts,features]."""
    b, h, w, parts, channels = part_image.shape
    part_encodings = nn.apply_partwise(part_image, encoder)
    part_encodings = part_encodings.reshape(b, parts, -1)
    out_shape = list(part_encodings.shape)
    assert out_shape[0] == b and out_shape[1] == parts
    return part_encodings


def unpool_features(feature_vectors, mask, reshape=False):
    """cub/code/SB_model48i/model.py:225-249 ; deepfashion/code/foo.py:462-498 (`reshape`).
    feature_vectors [B,parts,F], mask [B,h,w,parts] -> [B,h,w,parts,F]."""
    bs, h, w, n_parts = mask.shape
    fshape = list(feature_vectors.shape)
    assert len(fshape) == 3, fshape
    assert fshape[0] == bs and fshape[1] == n_parts, fshape
    out = ops.part_unpool(feature_vectors, mask)
    if reshape:
        out = out.reshape(bs, h, w, n_parts * fshape[2])
    return out


def inject_features(feature_vectors, mask):
    """tf.concat([tf.reduce_sum(unpool_features(f, m), 3), m], 3) — the three lines at
    cub/code/SB_model48i/model.py:482-484 (and :493-500) without the [B,h,w,parts,F]
    intermediate: -> [B,h,w,F+parts]."""
    bs, h, w, n_parts = mask.shape
    fshape = list(feature_vectors.shape)
    assert len(fshape) == 3, fshape
    assert fshape[0] == bs and fshape[1] == n_parts, fshape
    return ops.part_inject(feature_vectors, mask)


def inject_conv2d(feature_vectors, mask, V, b):
    """The decoder's first layer on the injected part map, without the map: the three lines at
    cub/code/SB_model48i/model.py:482-484 followed by hourglass_model's `nn.conv2d(x, config[0])`
    (model.py:96; `dd`, :485; cub/code/nn.py:617-664 — 3x3, stride 1, SAME, + bias).
    feature_vectors [B,parts,F], mask [B,h,w,parts], V [3,3,F+parts,Co] (TensorFlow HWIO), b [Co] -> [B,h,w,Co].
    Equals nn.conv2d(inject_features(feature_vectors, mask)); differentiable in all four arguments."""
    bs, h, w, n_parts = mask.shape
    fshape = list(feature_vectors.shape)
    assert len(fshape) == 3, fshape
    assert fshape[0] == bs and fshape[1] == n_parts, fshape
    vshape = list(V.shape)
    assert vshape[:3] == [3, 3, fshape[2] + n_parts], vshape
    assert list(b.shape) == [vshape[3]], b.shape
    G = ops.inject_conv_table(feature_vectors, V.reshape(9, vshape[2], vshape[3]))
    return ops.inject_conv_apply(mask, G, b)


def decode_conv2d(logits, feature_vectors, V, b):
    """The decode side of the step with the first decoder layer folded in (model.py:426,434-436,447,470-473,482-485):
    m0 = softmax(logits); labels = argmax(m0); mask = ST(hard_max(m0)); h = inject_conv2d(feature_vectors, mask, V, b).
    Returns (m0, labels int64, mask, h); the backward runs the conv backward, the straight-through estimator and the
    softmax backward in one kernel."""
    bs, h, w, n_parts = logits.shape
    fshape = list(feature_vectors.shape)
    assert len(fshape) == 3, fshape
    assert fshape[0] == bs and fshape[1] == n_parts, fshape
    vshape = list(V.shape)
    assert vshape[:3] == [3, 3, fshape[2] + n_parts], vshape
    assert list(b.shape) == [vshape[3]], b.shape
    G = ops.inject_conv_table(feature_vectors, V.reshape(9, vshape[2], vshape[3]))
    return ops.decode_conv(logits, G, b)


def _noise_args(noise_seed):
    """noise_seed (None, an int in [0, 2**64) or a one-element int64 CUDA tensor) -> the ops' (noise, seed, seed_value)."""
    if noise_seed is None:
        return ops.NOISE_NONE, None, 0
    if isinstance(noise_seed, torch.Tensor):
        return ops.NOISE_DEVICE, noise_seed, 0
    return ops.NOISE_INT, None, ops._seed_i64(noise_seed)


def part_encode(logits1, image1, noise_seed=None, noise_level=1.0, sample_offset=0):
    """The encode side of the step (model.py:428-430,453-455,478 and the pooling tail of e_alpha, :50-52) in one kernel:
    m1 = softmax(logits1); mask = ST(hard_max(m1)); parts = mask_parts(image1, mask) folded part-major
    (nn.apply_partwise, cub/code/nn.py:100-103); pooled = mean over pixels of mask * image1.
    logits1 [B,h,w,parts], image1 [B,h,w,3] (the warped view 1) -> (m1, parts [parts*B,h,w,3] with row k*B+b,
    pooled [B,parts,3]).  Differentiable in logits1, and in image1 when it requires grad.
    noise_seed: l1 are the means of MeanFieldDistribution and the kernel softmaxes the sample
    logits1 + noise_level * eps (model.py:420-421), eps drawn on the device from the seed (draw 1, pixel
    (sample_offset + b) * h*w + p, as PartStep.forward).  An int is passed by value; a one-element int64 CUDA tensor is
    read by the kernel, which is what a captured CUDA graph needs (an int raises during capture)."""
    bs, h, w, n_parts = logits1.shape
    ishape = list(image1.shape)
    assert ishape == [bs, h, w, 3], ishape
    noise, seed, seed_value = _noise_args(noise_seed)
    return ops.part_encode(logits1, image1, noise, seed, seed_value, float(noise_level), int(sample_offset))


def part_decode(logits0, feature_vectors, noise_seed=None, noise_level=1.0, sample_offset=0):
    """The decode side of the step (model.py:426,434-436,447,470,482-484) in one kernel: m0 = softmax(logits0);
    labels = argmax(m0); mask = ST(hard_max(m0)); inj = concat(sum_k unpool_features(feature_vectors, mask), mask).
    logits0 [B,h,w,parts], feature_vectors [B,parts,F] (e_alpha's output) -> (m0, labels int64 [B,h,w],
    inj [B,h,w,F+parts]).  Differentiable in logits0 and feature_vectors.  noise_seed, noise_level, sample_offset as in
    part_encode (draw 0)."""
    bs, h, w, n_parts = logits0.shape
    fshape = list(feature_vectors.shape)
    assert len(fshape) == 3, fshape
    assert fshape[0] == bs and fshape[1] == n_parts, fshape
    noise, seed, seed_value = _noise_args(noise_seed)
    return ops.part_decode(logits0, feature_vectors, noise, seed, seed_value, float(noise_level), int(sample_offset))


def parts_conv2d(image, mask, V, b):
    """The appearance encoder's first layer on the masked part images, without the part images:
    `mask_parts(image, mask)` (cub/code/SB_model48i/model.py:176-187, :478) folded part-major by
    `nn.apply_partwise` (cub/code/nn.py:100-103) and fed to encoder_model's `nn.conv2d(x, config[0])`
    (model.py:40; cub/code/nn.py:617-664).  image [B,h,w,3], mask [B,h,w,parts], V [3,3,3,Co], b [Co]
    -> [parts*B,h,w,Co] (row k*B+b), what the rest of `e_alpha` consumes inside apply_partwise.  Differentiable in
    mask, V and b (the image gets no gradient: the reference's inputs are placeholders)."""
    bs, h, w, n_features = image.shape
    mshape = list(mask.shape)
    assert mshape[0] == bs and mshape[1] == h and mshape[2] == w, mshape
    vshape = list(V.shape)
    assert vshape[:3] == [3, 3, n_features], vshape
    assert list(b.shape) == [vshape[3]], b.shape
    return ops.parts_conv(image, mask, V.reshape(9, n_features, vshape[3]), b)


def images_from_uint8(images):
    """The host-side normalisation of the reference's data pipeline, moved onto the device:
    `o.astype(np.float32) * 2.0 / 255.0 - 1.0` (cub/code/data/data.py:134,152;
    pennaction/code/data/data.py:134,152).  uint8 CUDA tensor of any shape -> fp32, bit-identical
    to the numpy expression.  Lets a step's views cross PCIe as bytes."""
    return ops.views_u8_to_f32(images)


def make_tps(views, tps_parameters, generator=None):
    """TrainModel.make_tps — cub/code/SB_model48i/model.py:282-311 (3 views; the target view
    re-uses the first-half parameters) / pennaction/code/SB_model48i/model.py:281-303 (2 views)."""
    bs = views[0].shape[0]
    img_batch = torch.cat(list(views[:2]), dim=0)
    bs_doubled = img_batch.shape[0]
    tps_param_dict = _tps.tps_parameters(bs_doubled, generator=generator, device=img_batch.device,
                                         **tps_parameters)
    coord, vector = _tps.make_input_tps_param(tps_param_dict)
    t_images, t_mesh = _tps.ThinPlateSpline(img_batch, coord, vector, img_batch.shape[1], img_batch.shape[-1])
    augmented_views = list(torch.split(t_images, bs, dim=0))
    if len(views) > 2:
        t_images, t_mesh = _tps.ThinPlateSpline(views[2], coord[:bs], vector[:bs], views[2].shape[1],
                                                views[2].shape[-1])
        augmented_views.append(t_images)
    return augmented_views
