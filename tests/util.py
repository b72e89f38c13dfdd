"""Shared helpers of the parity tests: run the CUDA path / the oracle on the same inputs."""
import numpy as np

from oracle import softras as osr


def run_oracle(fv, tex, params, grad=None, rows=None):
    out = osr.forward(fv, tex, params, rows=rows)
    if grad is not None:
        out["grad_faces"], out["grad_textures"] = osr.backward(fv, tex, out, grad, params, accumulate_double=True, rows=rows)
    return out


def run_cuda(fv, tex, params, grad=None, device="cuda:0", want_faces_info=True):
    """Through the public torch API -> ctypes -> C ABI -> sm_100a kernels."""
    import torch
    from jrender_b200 import SoftRasterizeFunction
    dev = torch.device(device)
    fvt = torch.from_numpy(np.ascontiguousarray(fv)).to(dev).requires_grad_(grad is not None)
    txt = torch.from_numpy(np.ascontiguousarray(tex)).to(dev).requires_grad_(grad is not None)
    fn = SoftRasterizeFunction(
        image_size=params["image_size"], near=params["near"], far=params["far"], fill_back=params["fill_back"],
        eps=params["eps"], sigma_val=params["sigma_val"], dist_func=params["dist_func"], dist_eps=params["dist_eps"],
        gamma_val=params["gamma_val"], aggr_func_rgb=params["aggr_func_rgb"], aggr_func_alpha=params["aggr_func_alpha"],
        texture_type=params["texture_type"], max_faces_per_pixel_for_grad=params["max_faces_per_pixel_for_grad"])
    fn.return_faces_info = want_faces_info
    soft_colors, aggrs_info, ids = fn.raw(fvt, txt)
    from jrender_b200.softras import pad_face_ids
    ids = pad_face_ids(ids)   # the library terminates the per-pixel lists with one -1; the reference pads all K slots
    out = dict(soft_colors=soft_colors.detach().cpu().numpy(), aggrs_info=aggrs_info.cpu().numpy(),
               faces_id_buffer=ids.cpu().numpy())
    if want_faces_info:
        out["faces_info"] = fn.save_vars[3].cpu().numpy()
    if grad is not None:
        soft_colors.backward(torch.from_numpy(np.ascontiguousarray(grad)).to(dev))
        out["grad_faces"] = fvt.grad.cpu().numpy()
        out["grad_textures"] = txt.grad.cpu().numpy()
    torch.cuda.synchronize()
    return out


def sorted_ids(ids):
    """[B,K,H,W] -> per-pixel ascending id sets with -1 (empty) moved last."""
    a = ids.astype(np.int64).copy()
    a[a < 0] = np.iinfo(np.int32).max
    a.sort(axis=1)
    return a


def rel_err(a, b):
    """max |a-b| / max(|b|, tiny): scale-relative error of a whole tensor."""
    denom = max(float(np.abs(b).max()), 1e-30)
    return float(np.abs(a.astype(np.float64) - b.astype(np.float64)).max()) / denom


def large_softras_inputs(nfaces, H):
    """Inputs of tests/test_softras_gpu.py::test_against_reference_kernels_on_gpu: UV sphere, one image, seeded gradient."""
    from jrender_b200 import workloads as wl
    fv, tex = wl.make_scene(nfaces, batch=1)
    return fv, tex, np.random.default_rng(2).uniform(-1, 1, (1, 4, H, H)).astype(np.float32)


def c4_inputs():
    """Inputs of tests/test_nmr_gpu.py::test_c4_against_reference_kernels_on_gpu (BASELINE config C4, one image)."""
    faces, tex = nmr_scene(39200, batch=1, ts=2)
    g = np.random.default_rng(0).uniform(-1, 1, (1, 1024, 1024, 3)).astype(np.float32)
    ga = np.random.default_rng(1).uniform(-1, 1, (1, 1024, 1024)).astype(np.float32)
    return faces, tex, g, ga


# Reference outputs at C3 / C4 sizes are tens of MB, so tests/golden/refsample_*.npz keep a stratified sample of them.
# Where the reference output is trivial (a pixel no face reaches, a face without gradient) only a bitmask is stored and
# the product is compared there exactly.  The rest is split by where the product disagreed with the reference when the
# fixture was made (FMA contraction in the reference build flips top-K membership and depth ties there): each stratum
# is sampled at a fixed seed and every sampled value carries the weight (stratum size / sample size) that makes the
# weighted sums unbiased estimates of the sums over the whole image / all faces, for any product.
def input_sums(*arrays):
    """sum |x| per input in float64: tells a changed input generator from ulp-level drift."""
    return np.array([np.abs(a).sum(dtype=np.float64) for a in arrays])


def _stratified_sample(strata, seed):
    """strata: [(mask, n)] of disjoint masks -> ascending positions and their weights."""
    rng = np.random.default_rng(seed)
    pos, w = [np.zeros(0, np.int64)], [np.zeros(0)]
    for mask, n in strata:
        idx = np.flatnonzero(mask)
        k = min(n, idx.size)
        if k:
            pos.append(rng.choice(idx, k, replace=False))
            w.append(np.full(k, idx.size / k))
    pos, w = np.concatenate(pos), np.concatenate(w)
    order = np.argsort(pos)
    return pos[order].astype(np.int32), w[order]


def _grad_fixture(ref, got, n_worst, n_rest, seed):
    """Faces with a zero reference gradient: bitmask.  The n_worst faces where `got` differed most from the reference:
    all stored.  The other faces: n_rest sampled."""
    nf = ref["grad_faces"].shape[1]
    nonzero = (ref["grad_faces"][0].reshape(nf, -1) != 0).any(1) | (ref["grad_textures"][0].reshape(nf, -1) != 0).any(1)
    fix = dict(faces_nonzero=np.packbits(nonzero))
    score = np.zeros(nf)
    for k in ("grad_faces", "grad_textures"):
        a = ref[k][0]
        fix[k + "_abs_sum"] = np.abs(a[np.isfinite(a)]).sum(dtype=np.float64)
        score += np.nan_to_num(np.abs(a - got[k][0]).reshape(nf, -1).sum(1), nan=np.inf) / fix[k + "_abs_sum"]
    worst = np.zeros(nf, bool)
    worst[np.flatnonzero(nonzero)[np.argsort(-score[nonzero], kind="stable")[:n_worst]]] = True
    fix["faces"], fix["face_weights"] = _stratified_sample([(worst, n_worst), (nonzero & ~worst, n_rest)], seed)
    for k in ("grad_faces", "grad_textures"):
        fix[k] = ref[k][0][fix["faces"]]
    return fix


def _grad_rel_l1(fix, got):
    """sum |ref - got| / sum |ref| over the finite entries of grad_faces and grad_textures."""
    nf = got["grad_faces"].shape[1]
    nonzero = np.unpackbits(fix["faces_nonzero"], count=nf).astype(bool)
    res = {}
    for k in ("grad_faces", "grad_textures"):
        b = got[k][0]
        zero = np.abs(b[~nonzero])
        d = np.abs(fix[k] - b[fix["faces"]]).reshape(fix["faces"].size, -1)
        d = np.where(np.isfinite(d), d, 0.0).sum(1)
        res[k] = (zero[np.isfinite(zero)].sum(dtype=np.float64) + (fix["face_weights"] * d).sum()) / fix[k + "_abs_sum"]
    return res


def softras_fixture(ref, got, n_pixels, n_worst_faces, n_faces, seed=0):
    """Stratified sample of batch-1 SoftRas reference outputs; `got`: the product's outputs on the same inputs."""
    K = ref["faces_id_buffer"].shape[1]
    ids = ref["faces_id_buffer"][0].reshape(K, -1)
    colors = ref["soft_colors"][0].reshape(4, -1)
    covered = (ids >= 0).any(0)
    assert not colors[:, ~covered].any()          # a pixel no face reaches keeps colour and alpha 0
    differ = ~(np.sort(ids, 0) == np.sort(got["faces_id_buffer"][0].reshape(K, -1), 0)).all(0) | \
        (np.abs(colors - got["soft_colors"][0].reshape(4, -1)).max(0) > 2e-3)
    pixels, w = _stratified_sample([(covered & differ, n_pixels // 2), (covered & ~differ, n_pixels // 2)], seed)
    ids_s = np.sort(ids[:, pixels].T, 1)
    return dict(covered=np.packbits(covered), pixels=pixels, pixel_weights=w,
                faces_id_buffer=ids_s.astype(np.int16 if ids_s.max() < 32767 else np.int32), soft_colors=colors[:, pixels].T,
                **_grad_fixture(ref, got, n_worst_faces, n_faces, seed))


def softras_stats(fix, got):
    """Estimates, over the whole image, of: the fraction of pixels with the reference's top-K id set (`same`), the
    fraction with a colour channel off by more than 2e-3 and the mean of that per-pixel max difference; and the
    gradients' relative L1 difference."""
    K = got["faces_id_buffer"].shape[1]
    ids = got["faces_id_buffer"][0].reshape(K, -1)
    colors = got["soft_colors"][0].reshape(4, -1)
    npix = ids.shape[1]
    covered = np.unpackbits(fix["covered"], count=npix).astype(bool)
    px, w = fix["pixels"], fix["pixel_weights"]
    d_out = np.abs(colors[:, ~covered]).max(0)
    d_in = np.abs(colors[:, px].T - fix["soft_colors"]).max(1)
    differ_in = ~(np.sort(ids[:, px].T, 1) == fix["faces_id_buffer"]).all(1)
    res = dict(same=1 - ((ids[:, ~covered] >= 0).any(0).sum() + (w * differ_in).sum()) / npix,
               color_frac=((d_out > 2e-3).sum() + (w * (d_in > 2e-3)).sum()) / npix,
               color_mean=(d_out.sum(dtype=np.float64) + (w * d_in).sum()) / npix)
    res.update(_grad_rel_l1(fix, got))
    return res


def nmr_fixture(ref, got, n_pixels, n_worst_faces, n_faces, far, seed=0):
    """Stratified sample of batch-1 NMR reference outputs (background colour 0); `got`: the product's outputs."""
    fim = ref["face_index_map"].reshape(-1)
    depth = ref["depth_map"].reshape(-1)
    rgb = ref["rgb_map"].reshape(-1, 3)
    covered = fim >= 0
    assert (depth[~covered] == np.float32(far)).all() and not rgb[~covered].any()
    differ = (fim != got["face_index_map"].reshape(-1)) | (np.abs(depth - got["depth_map"].reshape(-1)) > 1e-4) | \
        (np.abs(rgb - got["rgb_map"].reshape(-1, 3)).max(1) > 2e-3)
    pixels, w = _stratified_sample([(covered & differ, n_pixels // 2), (covered & ~differ, n_pixels // 2)], seed)
    return dict(covered=np.packbits(covered), pixels=pixels, pixel_weights=w, face_index_map=fim[pixels],
                depth_map=depth[pixels], rgb_map=rgb[pixels], **_grad_fixture(ref, got, n_worst_faces, n_faces, seed))


def nmr_stats(fix, got, far):
    """Estimates, over the whole image, of: the fraction of pixels with the reference's face index (`same`); over those
    pixels, the fraction of depths off by more than 1e-4 and of colour channels off by more than 2e-3; the largest such
    differences (over the uncovered pixels and the sample); and the gradients' relative L1 difference."""
    fim = got["face_index_map"].reshape(-1)
    depth = got["depth_map"].reshape(-1)
    rgb = got["rgb_map"].reshape(-1, 3)
    covered = np.unpackbits(fix["covered"], count=fim.size).astype(bool)
    out_same = fim[~covered] < 0
    dd_out = np.abs(depth[~covered][out_same] - np.float32(far))
    dc_out = np.abs(rgb[~covered][out_same])
    px = fix["pixels"]
    same = fim[px] == fix["face_index_map"]
    w = fix["pixel_weights"] * same
    dd_in = np.abs(depth[px] - fix["depth_map"])
    dc_in = np.abs(rgb[px] - fix["rgb_map"])
    n_same = out_same.sum() + w.sum()
    res = dict(same=n_same / fim.size,
               depth_frac=((dd_out > 1e-4).sum() + (w * (dd_in > 1e-4)).sum()) / n_same,
               depth_max=max(dd_out.max(initial=0.0), dd_in[same].max(initial=0.0)),
               color_frac=((dc_out > 2e-3).sum() + (w * (dc_in > 2e-3).sum(1)).sum()) / (3 * n_same),
               color_max=max(dc_out.max(initial=0.0), dc_in[same].max(initial=0.0)))
    res.update(_grad_rel_l1(fix, got))
    return res


def nmr_scene(num_faces=280, batch=1, ts=2, fill_back=True, seed=1):
    from jrender_b200 import workloads as wl
    return wl.nmr_scene(num_faces, batch=batch, ts=ts, fill_back=fill_back, seed=seed)


def run_nmr_cuda(faces, textures, image_size, near=0.1, far=100.0, eps=1e-3, background_color=(0, 0, 0),
                 flags=(True, True, True), grads=None, device="cuda:0"):
    """Through jrender_b200.n3mr.RasterizeFunction -> ctypes -> C ABI.  grads = (g_rgb, g_alpha, g_depth)."""
    import torch
    from jrender_b200.n3mr import RasterizeFunction
    dev = torch.device(device)
    fc = torch.from_numpy(np.ascontiguousarray(faces)).to(dev).requires_grad_(grads is not None)
    tx = torch.from_numpy(np.ascontiguousarray(textures)).to(dev).requires_grad_(grads is not None) if flags[0] else None
    fn = RasterizeFunction(image_size, near, far, eps, background_color, *flags)
    rgb, alpha, depth = fn(fc, tx)
    sv = fn.save_vars
    out = dict(face_index_map=sv[2].cpu().numpy(), weight_map=sv[3].cpu().numpy(), depth_map=sv[4].cpu().numpy())
    if flags[0]:
        out.update(rgb_map=rgb.detach().cpu().numpy(), sampling_index_map=sv[8].cpu().numpy(), sampling_weight_map=sv[9].cpu().numpy())
    if flags[1]:
        out["alpha_map"] = alpha.detach().cpu().numpy()
    if flags[2]:
        out["face_inv_map"] = sv[7].cpu().numpy()
    if grads is not None:
        outs, gs = [], []
        for o, g, f in zip((rgb, alpha, depth), grads, flags):
            if f:
                outs.append(o)
                gs.append(torch.from_numpy(np.ascontiguousarray(g)).to(dev))
        torch.autograd.backward(outs, gs)
        out["grad_faces"] = fc.grad.cpu().numpy()
        if flags[0]:
            out["grad_textures"] = tx.grad.cpu().numpy()
    torch.cuda.synchronize()
    return out
