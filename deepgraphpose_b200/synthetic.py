"""Seeded synthetic weights and video for the DGP hot path (no network, no checkpoints).

Weights use the reference's TF variable names and layouts so that a real DLC/DGP
snapshot converted to a ``{name: ndarray}`` dict loads through the same entry point
(slim names: /root/reference/src/DeepLabCut/deeplabcut/pose_estimation_tensorflow/nnet/pose_net.py:18-26,50-52;
restore scopes: /root/reference/src/deepgraphpose/models/fitdgp.py:689-696).
"""
import numpy as np

# (scope, base_depth, num_units, stride) -- slim resnet_v1_50
RESNET50_BLOCKS = (("block1", 64, 3, 2), ("block2", 128, 4, 2), ("block3", 256, 6, 2), ("block4", 512, 3, 1))
# units per block of slim resnet_v1_50 / _101 / _152 (DLC's net_type); channels, strides and dilation are the same
BLOCK_UNITS = {"resnet_50": (3, 4, 6, 3), "resnet_101": (3, 4, 23, 3), "resnet_152": (3, 8, 36, 3)}
NET_TYPES = tuple(BLOCK_UNITS)
# Scale of the last BN gamma of every bottleneck (see make_weights).  Chosen with the fp32 oracle so that the deeper nets'
# part_pred logits have the spread of the ResNet-50 set: std of the logits of seed 0, nj 4, on a 235x301 synthetic frame is
# 4.10 at depth 50 (0.25), 4.07 at depth 101 (0.145) and 4.13 at depth 152 (0.14); at 0.25 the deeper nets reach 17 / 37
# and saturate the sigmoid on 82 / 92 % of the map.
CONV3_GAMMA_SCALE = {"resnet_50": 0.25, "resnet_101": 0.145, "resnet_152": 0.14}


def net_scope(net_type):
    """slim scope of the backbone variables: 'resnet_50' -> 'resnet_v1_50'."""
    if net_type not in BLOCK_UNITS:
        raise ValueError("net_type must be one of %s (got %r)" % (", ".join(NET_TYPES), net_type))
    return "resnet_v1_" + net_type.split("_")[1]


def net_blocks(net_type="resnet_50"):
    """(scope, base_depth, num_units, stride) of the four blocks of slim resnet_v1_<depth>."""
    net_scope(net_type)
    return tuple((name, base, n, stride) for (name, base, _, stride), n in zip(RESNET50_BLOCKS, BLOCK_UNITS[net_type]))


def net_type_of(variables):
    """net_type ('resnet_50' / 'resnet_101' / 'resnet_152') of a {tf_var_name: array} dict, from its backbone scope."""
    scopes = sorted({k.split("/", 1)[0] for k in variables if k.startswith("resnet_v1_")})
    if len(scopes) != 1:
        raise ValueError("the weights must hold exactly one backbone scope out of resnet_v1_50, resnet_v1_101, resnet_v1_152 "
                         "(found %s)" % (", ".join(scopes) if scopes else "none"))
    net_type = "resnet_" + scopes[0][len("resnet_v1_"):]
    net_scope(net_type)
    return net_type


def conv_specs(net_type="resnet_50"):
    """(scope, kh, kw, cin, cout) of every conv of slim resnet_v1_<depth> in execution order (53 / 104 / 155 convs)."""
    prefix = net_scope(net_type)
    specs = [(prefix + "/conv1", 7, 7, 3, 64)]
    cin = 64
    for name, base, units, _ in net_blocks(net_type):
        for u in range(units):
            scope = "%s/%s/unit_%d/bottleneck_v1" % (prefix, name, u + 1)
            depth = base * 4
            if cin != depth:
                specs.append((scope + "/shortcut", 1, 1, cin, depth))
            specs.append((scope + "/conv1", 1, 1, cin, base))
            specs.append((scope + "/conv2", 3, 3, base, base))
            specs.append((scope + "/conv3", 1, 1, base, depth))
            cin = depth
    return specs


def resnet50_conv_specs():
    """Yield (scope, kh, kw, cin, cout) for the 53 convs of slim resnet_v1_50 in execution order."""
    return conv_specs("resnet_50")


def make_weights(nj, seed=0, location_refinement=True, bn_random=True, head_gain=1.0, trained_like=False, net_type="resnet_50"):
    """Random-init weights of the DLC pose net on slim resnet_v1_<depth> (``net_type`` resnet_50 / resnet_101 /
    resnet_152), TF names -> float32 ndarrays.

    conv: He-normal (fan-in) HWIO; BN: gamma~U(.5,1.5), beta~N(0,.1), mean~N(0,.1), var~U(.5,1.5)
    (``bn_random=False`` gives the TF initial values gamma=1, beta=0, mean=0, var=1 of config (a)).
    The last BN of every bottleneck gets gamma scaled by CONV3_GAMMA_SCALE[net_type] (0.25 for the 16 units of ResNet-50,
    less for the 33 / 50 units of the deeper nets) so the residual stream stays O(1) (otherwise logits saturate the sigmoid
    and every parity test degenerates to ties).  ResNet-50 draws the same random stream whatever the other nets draw.
    Heads: xavier-uniform ``[3,3,cout,2048]`` scaled so logits have std ~3, zero bias.

    ``trained_like=True`` gives the second weight set of the parity tests, shaped like a fine-tuned DLC snapshot rather than
    a fresh initialisation: (i) an ImageNet-style BatchNorm spectrum -- in every bottleneck's last BN 15 % of the channels
    carry a near-zero gamma (10^U(-5,-2)) and 2 % exactly 0 (resnet_v1_50.ckpt, the reference's starting point, README.md:52,
    has many such channels; they are what a division by gamma cannot differentiate), (ii) peaked scoremaps -- part_pred
    gain x2 with bias -4, so the sigmoid map is ~0 background with a few confident peaks instead of a flat 0.5 field.
    """
    rng = np.random.default_rng(seed)
    W = {}
    gamma_scale = CONV3_GAMMA_SCALE[net_type]
    for scope, kh, kw, cin, cout in conv_specs(net_type):
        fan_in = kh * kw * cin
        gain = np.sqrt(2.0 / fan_in)
        if scope.endswith("/conv1") and cin == 3:
            gain *= 0.02  # pixels are fed as 0..255 (std ~50): fold a unit-variance input scaling into conv1
        W[scope + "/weights"] = (rng.standard_normal((kh, kw, cin, cout)) * gain).astype(np.float32)
        if bn_random:
            g = rng.uniform(0.5, 1.5, cout)
            b = rng.normal(0.0, 0.1, cout)
            m = rng.normal(0.0, 0.1, cout)
            v = rng.uniform(0.5, 1.5, cout)
        else:
            g, b, m, v = np.ones(cout), np.zeros(cout), np.zeros(cout), np.ones(cout)
        if scope.endswith("/conv3"):
            g = g * gamma_scale
            if trained_like:
                u = rng.uniform(size=cout)
                tiny = 10.0 ** rng.uniform(-5.0, -2.0, cout)
                g = np.where(u < 0.15, tiny, g)
                g = np.where(u < 0.02, 0.0, g)
        W[scope + "/BatchNorm/gamma"] = g.astype(np.float32)
        W[scope + "/BatchNorm/beta"] = b.astype(np.float32)
        W[scope + "/BatchNorm/moving_mean"] = m.astype(np.float32)
        W[scope + "/BatchNorm/moving_variance"] = v.astype(np.float32)
    heads = [("part_pred", nj)]
    if location_refinement:
        heads.append(("locref_pred", 2 * nj))
    for name, cout in heads:
        fan_in, fan_out = 9 * 2048, 9 * cout
        lim = np.sqrt(6.0 / (fan_in + fan_out))
        w = rng.uniform(-lim, lim, (3, 3, cout, 2048)) * head_gain
        b = np.zeros(cout)
        if trained_like and name == "part_pred":
            w, b = w * 2.0, b - 4.0
        W["pose/%s/block4/weights" % name] = w.astype(np.float32)
        W["pose/%s/block4/biases" % name] = b.astype(np.float32)
    return W


def make_video(T, H, W, nj, seed=1234, blob_sigma=6.0):
    """Synthetic uint8 RGB video (T,H,W,3): smooth background + nj bright blobs on random walks."""
    rng = np.random.default_rng(seed)
    ys = np.arange(H, dtype=np.float32)[:, None]
    xs = np.arange(W, dtype=np.float32)[None, :]
    coarse = rng.uniform(0, 255, (H // 32 + 2, W // 32 + 2, 3)).astype(np.float32)
    iy = np.minimum((ys / 32).astype(np.int64), coarse.shape[0] - 2)
    ix = np.minimum((xs / 32).astype(np.int64), coarse.shape[1] - 2)
    fy = (ys / 32 - iy)[..., None]
    fx = (xs / 32 - ix)[..., None]
    bg = (coarse[iy, ix] * (1 - fy) * (1 - fx) + coarse[iy + 1, ix] * fy * (1 - fx)
          + coarse[iy, ix + 1] * (1 - fy) * fx + coarse[iy + 1, ix + 1] * fy * fx)
    pos = np.stack([rng.uniform(0.2 * H, 0.8 * H, nj), rng.uniform(0.2 * W, 0.8 * W, nj)], 1)
    vel = rng.normal(0, 1.0, (nj, 2))
    colors = rng.uniform(128, 255, (nj, 3)).astype(np.float32)
    frames = np.empty((T, H, W, 3), np.uint8)
    tracks = np.empty((T, nj, 2), np.float32)
    for t in range(T):
        vel = 0.9 * vel + rng.normal(0, 0.7, (nj, 2))
        pos = pos + vel
        pos[:, 0] = np.clip(pos[:, 0], 8, H - 9)
        pos[:, 1] = np.clip(pos[:, 1], 8, W - 9)
        img = bg.copy()
        for j in range(nj):
            g = np.exp(-((ys - pos[j, 0]) ** 2 + (xs - pos[j, 1]) ** 2) / (2 * blob_sigma ** 2))[..., None]
            img = img * (1 - g) + colors[j] * g
        frames[t] = np.clip(img + rng.normal(0, 2.0, img.shape), 0, 255).astype(np.uint8)
        tracks[t] = pos
    return frames, tracks


def chain_skeleton(nj):
    return [(i, i + 1) for i in range(nj - 1)]


def dense_skeleton(nj):
    return [(i, j) for i in range(nj) for j in range(i + 1, nj)]


def make_training_batch(nt, H, W, nj, vis_frames, nan_joints=(), seed=0):
    """Synthetic fit_dgp batch in the reference's feed_dict contract (fitdgp.py:797-815, dataset.py:187-239): labels of the
    visible frames in scoremap (row, col) units with NaN for missing joints, marker index vectors
    (marker = frame_in_batch * nj + joint; NaN-labelled joints of visible frames move to the hidden list), and the
    positions of the visible frames in the batch (the locref maps are then built by the coord2map feeder).
    Returns (labels (n_vis,nj,2) float64, feed dict)."""
    rng = np.random.default_rng(seed)
    vis = np.asarray(sorted(vis_frames), dtype=np.int64)
    hid = np.array([t for t in range(nt) if t not in set(vis.tolist())], dtype=np.int64)
    labels = np.stack([rng.uniform(1, H - 2, (len(vis), nj)), rng.uniform(1, W - 2, (len(vis), nj))], axis=2)
    for (i, j) in nan_joints:
        labels[i, j, :] = np.nan
    nan_ind = sorted(int(nj * vis[i] + j) for (i, j) in nan_joints)
    hidden = np.sort(np.concatenate([(hid[:, None] * nj + np.arange(nj)[None, :]).reshape(-1), np.asarray(nan_ind, dtype=np.int64)]))
    vm0 = np.sort((vis[:, None] * nj + np.arange(nj)[None, :]).reshape(-1))
    visible = np.setdiff1d(vm0, nan_ind)
    feed = {"targets": labels, "visible_marker_pl": visible.astype(np.int64), "hidden_marker_pl": hidden.astype(np.int64),
            "visible_marker_in_targets_pl": np.nonzero(np.isin(vm0, visible))[0], "nt_batch_pl": nt,
            "visible_frame_within_batch": vis.tolist()}
    return labels, feed
