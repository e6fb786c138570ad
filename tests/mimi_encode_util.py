"""Shared checks of the Mimi encoder tests: the latent bar and the margin rule for codes."""
import numpy as np


def check_latent(name, got, want, rel):
    got, want = np.asarray(got, dtype=np.float32), np.asarray(want, dtype=np.float32)
    assert got.shape == want.shape, (name, got.shape, want.shape)
    assert np.isfinite(got).all(), f"{name}: non-finite latent"
    scale = float(np.abs(want).max())
    err = float(np.abs(got - want).max())
    print(f"{name}: latent max abs error {err:.3g} (scale {scale:.3g}, rel {err / scale:.2g})")
    assert err <= rel * scale, f"{name}: latent max abs error {err:.3g} vs scale {scale:.3g}"


def check_codes(name, got, want, gap, margin=1e-3):
    """Margin rule: frame by frame, codebook by codebook, a code may differ from the reference only where the reference's
    relative gap between its two nearest codebook rows is below `margin`; after the first difference in a frame its residual
    has diverged and the rest of that frame is not compared.  Returns the share of frames that are identical."""
    got, want, gap = np.asarray(got), np.asarray(want), np.asarray(gap)
    assert got.shape == want.shape, (name, got.shape, want.shape)
    n_q, T = want.shape
    same = 0
    for t in range(T):
        for q in range(n_q):
            if got[q, t] != want[q, t]:
                assert gap[q, t] < margin, f"{name}: frame {t} codebook {q}: {got[q, t]} vs {want[q, t]}, gap {gap[q, t]:.3g}"
                break
        else:
            same += 1
    share = same / max(T, 1)
    print(f"{name}: {same} / {T} frames identical ({100 * share:.1f} %)")
    return share


def oracle_gaps(orc, z, codes):
    """[n_q, T] relative top-2 gaps in fp64 along the oracle's own residual path (z [1, dim, T], codes [1, n_q, T])."""
    import torch
    import torch.nn.functional as F

    d, sd = orc.d, orc.sd
    gaps, q = [], 0
    for prefix, n in (("quantizer.semantic_residual_vector_quantizer", 1), ("quantizer.acoustic_residual_vector_quantizer", d.n_q - 1)):
        r = F.conv1d(z, sd[f"{prefix}.input_proj.weight"])[0].t()
        for i in range(n):
            emb = sd[f"{prefix}.layers.{i}.codebook.embed_sum"] / torch.clamp(sd[f"{prefix}.layers.{i}.codebook.cluster_usage"], min=d.cb_eps)[:, None]
            dist = torch.cdist(r.double(), emb.double()).sort(dim=-1).values
            gaps.append(((dist[:, 1] - dist[:, 0]) / dist[:, 0].clamp(min=1e-300)).numpy())
            r = r - emb[codes[0, q]]
            q += 1
    return np.stack(gaps)
