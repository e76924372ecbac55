"""Shared by the CPU and GPU parity tests: cases of tests/golden/model_zoo.npz and model_full.npz."""
ZOO_CASES = ["double_filters", "triple_filters", "half_filters", "depth_ver_1", "depth_ver_2", "depth_ver_3",
             "depth_ver_4", "rgb_base_model", "rgb_silu_model"]
ZOO_MODEL = {"rgb_base_model": "base_model", "rgb_silu_model": "silu_model"}


def zoo_inputs(z, case):
    """Inputs of a model_zoo.npz / model_full.npz case, regenerated from the seeds in its cfg row (the fixtures hold
    no images, labels or weights)."""
    import yogo_b200
    from tools.synth import synth_fill_model, synth_images, synth_labels

    ch, N, H, W, K, seed, ostride = (int(v) for v in z[case + ".cfg"])
    name = ZOO_MODEL.get(case, case[5:] if case.startswith("full_") else case)
    net = yogo_b200.YOGO((H, W), 0.0425, 0.0555, 7, is_rgb=ch == 3, model_func=yogo_b200.get_model_func(name))
    synth_fill_model(net, seed)
    img = synth_images(N, H, W, seed=seed, channels=ch)
    lab = synth_labels(N, net.Sy, net.Sx, 7, K, seed=seed + 100)
    return name, net, img, lab, ostride


def grad_sample(g, n):
    """The `n` elements of the flat gradient `g` that a model_zoo.npz / model_full.npz case stores: every
    ceil(size / 4096)-th, and of those every second one where the fixture keeps half (make_golden.py, `shrink`)."""
    g = g[:: max(1, -(-g.size // 4096))]
    return g if g.size == n else g[::2]
