"""Seeded synthetic descriptor sets of the reference's feature types (SURVEY.md 8d).

Layouts mirror PCL's point structs as the reference hands them to the matcher
(`&cloud.points[0]`, stride `sizeof(FeatureT)`, include/matching.h:553-560):
    FPFH  = pcl::FPFHSignature33  : float histogram[33]                -> 132 B / row
    RoPS  = pcl::Histogram<135>   : float histogram[135]               -> 540 B / row
    SHOT  = pcl::SHOT352          : float descriptor[352]; float rf[9] -> 1444 B / row
    USC   = pcl::UniqueShapeContext1960 : float descriptor[1960]; float rf[9] -> 7876 B / row
The generators return the AoS buffer (float32 [n, stride/4]); the descriptor is
columns [0, dim).  The value statistics are stand-ins of the descriptors' shape (sign, sparsity,
normalisation), not measured from PCL's estimators.
"""
import numpy as np

SEED = 566  # echoes `#define SEED 566ul`, include/common.h:25

DESCRIPTORS = {
    # name: (dim, row stride in floats)
    "fpfh": (33, 33),
    "rops": (135, 135),
    "shot": (352, 361),
    "usc": (1960, 1969),
}


def _prototype_rows(rng, n, dim, n_proto, make_proto, noise):
    protos = make_proto(rng, n_proto, dim)
    which = rng.integers(0, n_proto, size=n)
    rows = protos[which] + noise(rng, n, dim)
    return rows


def _fpfh_like(rng, n, dim=33):
    """3 sub-histograms x 11 bins, each non-negative and summing to 100 (PCL FPFH
    convention); rows cluster around n/64 prototypes."""
    n_proto = max(n // 64, 4)
    protos = rng.gamma(0.5, 1.0, size=(n_proto, 3, 11)).astype(np.float32)
    which = rng.integers(0, n_proto, size=n)
    rows = protos[which] * (1.0 + 0.35 * rng.standard_normal((n, 3, 11)).astype(np.float32)) \
        + 0.02 * rng.gamma(0.5, 1.0, size=(n, 3, 11)).astype(np.float32)
    rows = np.abs(rows)
    rows *= (100.0 / np.maximum(rows.sum(axis=2, keepdims=True), 1e-12))
    return rows.reshape(n, 33).astype(np.float32)


def _shot_like(rng, n, dim=352):
    """32 volumes x 11 bins, non-negative, ~70 % zeros, unit L2 norm (PCL SHOT
    convention); rows cluster around n/64 prototypes."""
    n_proto = max(n // 64, 4)
    protos = rng.gamma(0.6, 1.0, size=(n_proto, dim)).astype(np.float32)
    protos *= (rng.random((n_proto, dim)) < 0.3)
    which = rng.integers(0, n_proto, size=n)
    rows = protos[which]
    rows = rows * (1.0 + 0.3 * rng.standard_normal((n, dim)).astype(np.float32))
    extra = rng.gamma(0.6, 1.0, size=(n, dim)).astype(np.float32) * (rng.random((n, dim)) < 0.02)
    rows = np.abs(rows) + 0.25 * extra
    nrm = np.sqrt((rows.astype(np.float64) ** 2).sum(axis=1, keepdims=True))
    rows = rows / np.maximum(nrm, 1e-12)
    return rows.astype(np.float32)


def _rops_like(rng, n, dim=135):
    n_proto = max(n // 64, 4)
    protos = rng.standard_normal((n_proto, dim)).astype(np.float32)
    which = rng.integers(0, n_proto, size=n)
    return (protos[which] + 0.3 * rng.standard_normal((n, dim)).astype(np.float32)).astype(np.float32)


def _usc_like(rng, n, dim=1960):
    """Shape-context-like histogram: non-negative, ~85 % zeros, bin weights growing along
    the row (outer shells hold more points); rows cluster around n/64 prototypes."""
    n_proto = max(n // 64, 4)
    shell = np.linspace(0.5, 2.0, dim).astype(np.float32)
    protos = rng.gamma(0.5, 1.0, size=(n_proto, dim)).astype(np.float32) * shell
    protos *= (rng.random((n_proto, dim)) < 0.15)
    which = rng.integers(0, n_proto, size=n)
    rows = protos[which] * (1.0 + 0.25 * rng.standard_normal((n, dim)).astype(np.float32))
    extra = rng.gamma(0.5, 1.0, size=(n, dim)).astype(np.float32) * (rng.random((n, dim)) < 0.01)
    return (np.abs(rows) + 0.5 * extra).astype(np.float32)


_GEN = {"fpfh": _fpfh_like, "shot": _shot_like, "rops": _rops_like, "usc": _usc_like}


def to_aos(rows, stride_floats, rng=None):
    """Embed dense rows [n, dim] in an AoS buffer [n, stride_floats]; the tail (SHOT's
    rf[9]) is filled with junk the matcher must ignore."""
    n, dim = rows.shape
    if stride_floats == dim:
        return np.ascontiguousarray(rows, np.float32)
    buf = np.empty((n, stride_floats), np.float32)
    buf[:, :dim] = rows
    buf[:, dim:] = 7.0 if rng is None else rng.standard_normal((n, stride_floats - dim))
    return buf


def make_pair(descriptor, n_src, n_tgt, seed=SEED, nan_frac=0.001, distractor_frac=0.3, noise=0.05):
    """(src_aos, tgt_aos, dim): target = noisy permutation of (part of) the source set plus
    `distractor_frac` unrelated rows, so mutual/ratio filters keep a non-trivial fraction;
    `nan_frac` of the rows on each side carry a NaN (invalid descriptor, include/common.h:409)."""
    dim, stride = DESCRIPTORS[descriptor]
    rng_s = np.random.default_rng([seed, 0])
    rng_t = np.random.default_rng([seed, 1])
    gen = _GEN[descriptor]
    src = gen(rng_s, n_src, dim)
    n_dis = int(round(distractor_frac * n_tgt))
    n_cpy = n_tgt - n_dis
    pick = rng_t.integers(0, n_src, size=n_cpy) if n_cpy > n_src else rng_t.permutation(n_src)[:n_cpy]
    scale = float(np.sqrt((src.astype(np.float64) ** 2).sum(1).mean() / dim))
    tgt_c = src[pick] + (noise * scale) * rng_t.standard_normal((n_cpy, dim)).astype(np.float32)
    if descriptor in ("fpfh", "shot", "usc"):
        tgt_c = np.abs(tgt_c)
    tgt = np.concatenate([tgt_c, gen(rng_t, n_dis, dim)], axis=0) if n_dis else tgt_c
    tgt = tgt[rng_t.permutation(n_tgt)].astype(np.float32)
    for a, rng in ((src, rng_s), (tgt, rng_t)):
        n_bad = int(round(nan_frac * a.shape[0]))
        if n_bad:
            r = rng.choice(a.shape[0], size=n_bad, replace=False)
            c = rng.integers(0, dim, size=n_bad)
            a[r, c] = np.nan
    return to_aos(src, stride, rng_s), to_aos(tgt, stride, rng_t), dim


def make_pair_torch(descriptor, n_src, n_tgt, device, seed=SEED, nan_frac=0.001, distractor_frac=0.3,
                    noise=0.05):
    """Same recipe generated with torch on `device` (bench sizes: 500k x 352 takes too long
    in numpy).  Returns dense AoS float32 tensors [n, stride_floats] and dim."""
    import torch
    dim, stride = DESCRIPTORS[descriptor]
    g = torch.Generator(device=device)
    g.manual_seed(seed)

    def gamma_like(shape, expo):
        # cheap heavy-tailed non-negative draw: |N(0,1)|^expo
        return torch.randn(shape, generator=g, device=device).abs_().pow_(expo)

    def gen(n):
        n_proto = max(n // 64, 4)
        which = torch.randint(0, n_proto, (n,), generator=g, device=device)
        if descriptor == "fpfh":
            protos = gamma_like((n_proto, 33), 3.0)
            rows = protos[which] * (1.0 + 0.35 * torch.randn((n, 33), generator=g, device=device))
            rows = rows.abs_() + 0.02 * gamma_like((n, 33), 3.0)
            rows = rows.view(n, 3, 11)
            rows = rows * (100.0 / rows.sum(dim=2, keepdim=True).clamp_min(1e-12))
            return rows.reshape(n, 33).contiguous()
        if descriptor == "shot":
            protos = gamma_like((n_proto, dim), 2.5)
            protos = protos * (torch.rand((n_proto, dim), generator=g, device=device) < 0.3)
            rows = protos[which]
            rows = rows * (1.0 + 0.3 * torch.randn((n, dim), generator=g, device=device))
            rows = rows.abs_()
            extra = gamma_like((n, dim), 2.5) * (torch.rand((n, dim), generator=g, device=device) < 0.02)
            rows = rows + 0.25 * extra
            return rows / rows.norm(dim=1, keepdim=True).clamp_min(1e-12)
        if descriptor == "usc":
            shell = torch.linspace(0.5, 2.0, dim, device=device)
            protos = gamma_like((n_proto, dim), 2.5) * shell
            protos = protos * (torch.rand((n_proto, dim), generator=g, device=device) < 0.15)
            rows = protos[which] * (1.0 + 0.25 * torch.randn((n, dim), generator=g, device=device))
            extra = gamma_like((n, dim), 2.5) * (torch.rand((n, dim), generator=g, device=device) < 0.01)
            return rows.abs_() + 0.5 * extra
        protos = torch.randn((n_proto, dim), generator=g, device=device)
        return protos[which] + 0.3 * torch.randn((n, dim), generator=g, device=device)

    src = gen(n_src)
    n_dis = int(round(distractor_frac * n_tgt))
    n_cpy = n_tgt - n_dis
    if n_cpy > n_src:
        pick = torch.randint(0, n_src, (n_cpy,), generator=g, device=device)
    else:
        pick = torch.randperm(n_src, generator=g, device=device)[:n_cpy]
    scale = float(src.pow(2).sum(1).mean().div(dim).sqrt())
    tgt = src[pick] + (noise * scale) * torch.randn((n_cpy, dim), generator=g, device=device)
    if descriptor in ("fpfh", "shot", "usc"):
        tgt = tgt.abs_()
    if n_dis:
        tgt = torch.cat([tgt, gen(n_dis)], dim=0)
    tgt = tgt[torch.randperm(n_tgt, generator=g, device=device)].contiguous()
    for a in (src, tgt):
        n_bad = int(round(nan_frac * a.shape[0]))
        if n_bad:
            r = torch.randperm(a.shape[0], generator=g, device=device)[:n_bad]
            c = torch.randint(0, dim, (n_bad,), generator=g, device=device)
            a[r, c] = float("nan")

    def aos(rows):
        if stride == dim:
            return rows.float().contiguous()
        buf = torch.full((rows.shape[0], stride), 7.0, device=device, dtype=torch.float32)
        buf[:, :dim] = rows
        return buf

    return aos(src), aos(tgt), dim
